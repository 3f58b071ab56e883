// Value head, reward cosine, A2C loss (+ gradient seeds), token-stream construction.
//   value head   models.py:175-178 : linear2(linear1(cat(features, h))) with no activation in between,
//                so it is evaluated in collapsed form  v = w_eff . [f, h] + b_eff,
//                w_eff = W2 W1 (1024), b_eff = W2 b1 + b2; the gradients of W1, b1, W2, b2 are
//                reconstructed exactly from g = sum dv * [f, h] and sum dv (rank-1 structure).
//   reward       trainers.py:117-120 : cos(visual_embed(f), semantic_embed(h)), F.normalize eps 1e-12.
//   loss         trainers.py:471-475 : adv = values - rewards; mean(-logp*adv) + 0.5*mean(adv^2)
//                (optionally - entropy_coef * mean(policy entropy): the entropy bonus, off by default).
#include "common.cuh"

namespace {
constexpr int H = ICRL_H;

// w_eff[j] = sum_i W2[i] W1[i][j]; b_eff = sum_i W2[i] b1[i] + b2
__global__ void pack_value_head_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                       const float* __restrict__ W2, const float* __restrict__ b2,
                                       float* __restrict__ w_eff, float* __restrict__ b_eff) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 2 * H) {
    float acc = 0.f;
    for (int i = 0; i < H; ++i) acc = fmaf(W2[i], W1[(size_t)i * 2 * H + j], acc);
    w_eff[j] = acc;
  }
  if (j == 0) {
    float acc = 0.f;
    for (int i = 0; i < H; ++i) acc = fmaf(W2[i], b1[i], acc);
    b_eff[0] = acc + b2[0];
  }
}

// one warp per (s,b): values[b][s] = w_eff[:512].f[b] + w_eff[512:].h_take[s][b] + b_eff
__global__ void value_head_fwd_kernel(int B, int S, const float* __restrict__ features, const float* __restrict__ h_take,
                                      const float* __restrict__ w_eff, const float* __restrict__ b_eff,
                                      float* __restrict__ values) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * S) return;
  const int s = warp / B, b = warp % B;
  const float* f = features + (size_t)b * H;
  const float* h = h_take + (size_t)warp * H;
  float acc = 0.f;
  for (int k = lane; k < H; k += 32) acc = fmaf(w_eff[k], f[k], acc);
  for (int k = lane; k < H; k += 32) acc = fmaf(w_eff[H + k], h[k], acc);
  acc = warp_sum(acc);
  if (lane == 0) values[(size_t)b * S + s] = acc + b_eff[0];
}

// dh_take[s][b][k] = dv_sb[s][b] * w_eff[512 + k]
__global__ void value_head_dh_kernel(long long rows, const float* __restrict__ dv_sb, const float* __restrict__ w_eff,
                                     float* __restrict__ dh_take) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * H) return;
  dh_take[i] = dv_sb[i / H] * w_eff[H + (int)(i % H)];
}

// g (1024) = sum dv*[f,h]; sdv = sum dv.
//   dW1[i][j] = W2[i] g[j]; db1[i] = W2[i] sdv; dW2[i] = W1[i,:].g + b1[i] sdv; db2 = sdv
__global__ void value_head_grads_kernel(const float* __restrict__ g, const float* __restrict__ sdv,
                                        const float* __restrict__ W1, const float* __restrict__ b1,
                                        const float* __restrict__ W2, float* __restrict__ dW1, float* __restrict__ db1,
                                        float* __restrict__ dW2, float* __restrict__ db2) {
  const int i = blockIdx.x;                    // 512 blocks, one per hidden row of linear1
  const float w2 = W2[i], sd = sdv[0];
  __shared__ float red[8];
  float acc = 0.f;
  for (int j = threadIdx.x; j < 2 * H; j += blockDim.x) {
    const float gj = g[j];
    dW1[(size_t)i * 2 * H + j] = w2 * gj;
    acc = fmaf(W1[(size_t)i * 2 * H + j], gj, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    dW2[i] = t + b1[i] * sd;
    db1[i] = w2 * sd;
    if (i == 0) db2[0] = sd;
  }
}

// one warp per (s,b): rewards[b][s] = <ve[b]/max(|ve[b]|,eps), se[s][b]/max(|se|,eps)>
__global__ void reward_cosine_kernel(int B, int S, const float* __restrict__ ve, const float* __restrict__ se,
                                     float* __restrict__ rewards) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * S) return;
  const int s = warp / B, b = warp % B;
  const float* v = ve + (size_t)b * H;
  const float* e = se + (size_t)warp * H;
  float nv = 0.f, ne = 0.f;
  for (int k = lane; k < H; k += 32) { nv = fmaf(v[k], v[k], nv); ne = fmaf(e[k], e[k], ne); }
  nv = fmaxf(sqrtf(warp_sum(nv)), 1e-12f);
  ne = fmaxf(sqrtf(warp_sum(ne)), 1e-12f);
  float dot = 0.f;
  for (int k = lane; k < H; k += 32) dot = fmaf(v[k] / nv, e[k] / ne, dot);
  dot = warp_sum(dot);
  if (lane == 0) rewards[(size_t)b * S + s] = dot;
}

// Single block.  out[0] = loss, out[1] = mean reward, out[2] = mean advantage (all scaled by inv_denom
// = 1/(B_global*S); for a data-parallel shard these are partial sums to be all-reduced).
//   dL/dvalues = (adv - logp) * inv_denom   (written [S][B] for the chain backward)
//   dL/dlogp   = -adv * inv_denom           (written [B][S])
// entropy != NULL ([B][S], the policy's entropy per sampled step): the entropy bonus -entropy_coef * mean(H) is added
// to out[0] and out[3] = mean entropy (scaled by inv_denom like the others); the gradient seeds do not change.
__global__ void a2c_loss_kernel(int B, int S, const float* __restrict__ values, const float* __restrict__ rewards,
                                const float* __restrict__ logp, float inv_denom, float* __restrict__ out,
                                float* __restrict__ dv_sb, float* __restrict__ dlogp, float* __restrict__ sum_dv,
                                const float* __restrict__ entropy, float entropy_coef) {
  __shared__ double red[5][32];
  double l = 0.0, r = 0.0, a = 0.0, d = 0.0, e = 0.0;
  const int n = B * S;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int b = i / S, s = i % S;
    const float adv = values[i] - rewards[i];
    const float lp = logp[i];
    l += (double)(-lp * adv) + 0.5 * (double)(adv * adv);
    r += (double)rewards[i];
    a += (double)adv;
    const float dv = (adv - lp) * inv_denom;
    d += (double)dv;
    if (dv_sb) dv_sb[(size_t)s * B + b] = dv;
    if (dlogp) dlogp[i] = -adv * inv_denom;
    if (entropy) e += (double)entropy[i];
  }
  l = warp_sum_d(l); r = warp_sum_d(r); a = warp_sum_d(a); d = warp_sum_d(d); e = warp_sum_d(e);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][w] = l; red[1][w] = r; red[2][w] = a; red[3][w] = d; red[4][w] = e; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    l = lane < nw ? red[0][lane] : 0.0; r = lane < nw ? red[1][lane] : 0.0;
    a = lane < nw ? red[2][lane] : 0.0; d = lane < nw ? red[3][lane] : 0.0;
    e = lane < nw ? red[4][lane] : 0.0;
    l = warp_sum_d(l); r = warp_sum_d(r); a = warp_sum_d(a); d = warp_sum_d(d); e = warp_sum_d(e);
    if (lane == 0) {
      if (entropy) {
        out[0] = (float)((l - (double)entropy_coef * e) * (double)inv_denom);
        out[3] = (float)(e * (double)inv_denom);
      } else {
        out[0] = (float)(l * (double)inv_denom);
      }
      out[1] = (float)(r * (double)inv_denom);
      out[2] = (float)(a * (double)inv_denom);
      if (sum_dv) sum_dv[0] = (float)d;
    }
  }
}

// Token stream of the batch-as-time chains (models.py:133/226 called per column, state carried):
// block s = columns 0..p0+s-1+extra of tokcm ([col][B] int32), rows in order.  take[t] = s*B + b when
// stream position t is row b's output at rollout step s (last column of block s), else -1.
__global__ void build_stream_kernel(int B, int p0, int S, int extra, const int* __restrict__ tokcm,
                                    int* __restrict__ stream, int* __restrict__ take, int* __restrict__ take_pos) {
  const int s = blockIdx.y;
  const int n = p0 + s + extra;
  // block start = B * sum_{q<s} (p0 + q + extra)
  const long long start = (long long)B * ((long long)s * (p0 + extra) + (long long)s * (s - 1) / 2);
  const long long len = (long long)n * B;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
    stream[start + i] = tokcm[i];
    const long long last = (long long)(n - 1) * B;
    const int tk = i >= last ? (int)(s * B + (i - last)) : -1;
    if (take) take[start + i] = tk;
    if (tk >= 0 && take_pos) take_pos[tk] = (int)(start + i);
  }
}

// The same streams for `shards` contiguous row shards of Bs = B / shards rows, each an independent chain:
// shard k's arrays start at k * stride (stride = T_shard + 1; the padding entry gets token 0 / take -1);
// take holds GLOBAL rows s*B + b, take_pos GLOBAL stash rows k * stride + position.
__global__ void build_stream_sharded_kernel(int B, int Bs, int p0, int S, int extra, long long stride,
                                            const int* __restrict__ tokcm, int* __restrict__ stream,
                                            int* __restrict__ take, int* __restrict__ take_pos) {
  const int s = blockIdx.y, k = blockIdx.z;
  const int n = p0 + s + extra;
  const long long start = (long long)Bs * ((long long)s * (p0 + extra) + (long long)s * (s - 1) / 2);
  const long long len = (long long)n * Bs;
  const long long base = (long long)k * stride;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i / Bs), bl = (int)(i % Bs);
    const int row = k * Bs + bl;
    stream[base + start + i] = tokcm[(long long)col * B + row];
    const int tk = col == n - 1 ? s * B + row : -1;
    if (take) take[base + start + i] = tk;
    if (tk >= 0 && take_pos) take_pos[tk] = (int)(base + start + i);
  }
  if (s == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    stream[base + stride - 1] = 0;
    if (take) take[base + stride - 1] = -1;
  }
}

// Value chain of one beam step of the look-ahead decoder (trainers.py:87-92): for candidate c and word i (block
// s = c*k + i, the reference's call order) the n prefix columns cand_tok[c] ([K][n][B]) and the word column
// words[c][b][i] ([K][B][k]), rows in order.  take_pos[s*B + b] = stream position of row b of the word column.
__global__ void lookahead_stream_kernel(int B, int n, int k, const int* __restrict__ cand_tok, const int* __restrict__ words,
                                        int* __restrict__ stream, int* __restrict__ take_pos) {
  const int s = blockIdx.y, c = s / k, i = s % k;
  const long long len = (long long)(n + 1) * B;
  const long long start = (long long)s * len;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < len; p += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(p / B), b = (int)(p % B);
    if (col < n) {
      stream[start + p] = cand_tok[((long long)c * n + col) * B + b];
    } else {
      stream[start + p] = words[((long long)c * B + b) * k + i];
      take_pos[(long long)s * B + b] = (int)(start + p);
    }
  }
}

// One block per child s = c*k + i: child[s][b] = parent[c][b] - (0.6 V + 0.4 log(top)) in the reference's operation
// order (trainers.py:92, fp32, every product and sum rounded on its own), means[s] = the batch mean of child[s].
__global__ void lookahead_score_kernel(int B, int K, int k, const float* __restrict__ parent, const float* __restrict__ values,
                                       const float* __restrict__ top_val, float* __restrict__ child, float* __restrict__ means) {
  const int s = blockIdx.x, c = s / k, i = s % k, S = K * k;
  __shared__ double red[32];
  double acc = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float v = values[(size_t)b * S + s];
    const float t = top_val[((size_t)c * B + b) * k + i];
    const float x = __fsub_rn(parent[(size_t)c * B + b], __fadd_rn(__fmul_rn(0.6f, v), __fmul_rn(0.4f, logf(t))));
    child[(size_t)s * B + b] = x;
    acc += (double)x;
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
    acc = warp_sum_d(acc);
    if (threadIdx.x == 0) means[s] = (float)(acc / B);
  }
}

// dst[r] = src[idx[r] + row_offset]  (rows of H floats)
__global__ void gather_rows_kernel(long long R, const float* __restrict__ src, const int* __restrict__ idx,
                                   long long row_offset, float* __restrict__ dst) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * (H / 4)) return;
  const long long r = i / (H / 4);
  const int q = (int)(i % (H / 4));
  reinterpret_cast<float4*>(dst)[i] =
      reinterpret_cast<const float4*>(src)[((long long)idx[r] + row_offset) * (H / 4) + q];
}

// table[v][j] += b_ih[j] + (j < fold ? b_hh[j] : 0)   (applied after the E * W_ih^T GEMM)
__global__ void add_gate_bias_kernel(int V, int G, int fold, const float* __restrict__ b_ih,
                                     const float* __restrict__ b_hh, float* __restrict__ table) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)V * G) return;
  const int j = (int)(i % G);
  table[i] += b_ih[j] + (j < fold ? b_hh[j] : 0.f);
}

// torch.optim.Adam (trainers.py:378, default betas / eps, no weight decay, no amsgrad) on flat arrays, in the order of
// torch's own kernel: m = lerp(m, g, 1-b1); v = b2 v + (1-b2) g^2; p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps).
__global__ void adam_flat_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, float one_minus_b1, float b2, float one_minus_b2, float step_size,
                                 float bc2_sqrt, float eps) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = m[i] + one_minus_b1 * (gi - m[i]);
    const float vi = b2 * v[i] + one_minus_b2 * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] = p[i] - step_size * (mi / (sqrtf(vi) / bc2_sqrt + eps));
  }
}

}  // namespace

int icrl_adam_flat_impl(cudaStream_t st, long long n, float* p, const float* g, float* m, float* v, float lr, float b1,
                        float b2, float eps, int step) {
  const double bc1 = 1.0 - pow((double)b1, step), bc2 = 1.0 - pow((double)b2, step);
  adam_flat_kernel<<<(int)min((long long)148 * 8, (n + 255) / 256), 256, 0, st>>>(
      n, p, g, m, v, 1.f - b1, b2, 1.f - b2, (float)((double)lr / bc1), (float)sqrt(bc2), eps);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_pack_value_head_impl(cudaStream_t st, const float* W1, const float* b1, const float* W2, const float* b2,
                              float* w_eff, float* b_eff) {
  pack_value_head_kernel<<<8, 128, 0, st>>>(W1, b1, W2, b2, w_eff, b_eff);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_value_head_fwd_impl(cudaStream_t st, int B, int S, const float* features, const float* h_take,
                             const float* w_eff, const float* b_eff, float* values) {
  value_head_fwd_kernel<<<icrl_cdiv((long long)B * S * 32, 256), 256, 0, st>>>(B, S, features, h_take, w_eff, b_eff, values);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_value_head_dh_impl(cudaStream_t st, long long rows, const float* dv_sb, const float* w_eff, float* dh_take) {
  value_head_dh_kernel<<<icrl_cdiv(rows * H, 256), 256, 0, st>>>(rows, dv_sb, w_eff, dh_take);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_value_head_grads_impl(cudaStream_t st, const float* g, const float* sdv, const float* W1, const float* b1,
                               const float* W2, float* dW1, float* db1, float* dW2, float* db2) {
  value_head_grads_kernel<<<H, 256, 0, st>>>(g, sdv, W1, b1, W2, dW1, db1, dW2, db2);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_reward_cosine_impl(cudaStream_t st, int B, int S, const float* ve, const float* se, float* rewards) {
  reward_cosine_kernel<<<icrl_cdiv((long long)B * S * 32, 256), 256, 0, st>>>(B, S, ve, se, rewards);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_a2c_loss_impl(cudaStream_t st, int B, int S, const float* values, const float* rewards, const float* logp,
                       float inv_denom, float* out3, float* dv_sb, float* dlogp, float* sum_dv, const float* entropy,
                       float entropy_coef) {
  a2c_loss_kernel<<<1, 1024, 0, st>>>(B, S, values, rewards, logp, inv_denom, out3, dv_sb, dlogp, sum_dv, entropy,
                                      entropy_coef);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_build_stream_impl(cudaStream_t st, int B, int p0, int S, int extra, const int* tokcm, int* stream, int* take,
                           int* take_pos) {
  dim3 grid(icrl_cdiv((long long)(p0 + S + extra) * B, 256 * 4), S);
  build_stream_kernel<<<grid, 256, 0, st>>>(B, p0, S, extra, tokcm, stream, take, take_pos);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_build_stream_sharded_impl(cudaStream_t st, int B, int p0, int S, int extra, int shards, const int* tokcm,
                                   int* stream, int* take, int* take_pos) {
  const int Bs = B / shards;
  const long long T = (long long)Bs * ((long long)S * (p0 + extra) + (long long)S * (S - 1) / 2);
  dim3 grid(icrl_cdiv((long long)(p0 + S + extra) * Bs, 256 * 4), S, shards);
  build_stream_sharded_kernel<<<grid, 256, 0, st>>>(B, Bs, p0, S, extra, T + 1, tokcm, stream, take, take_pos);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_lookahead_stream_impl(cudaStream_t st, int B, int n, int K, int k, const int* cand_tok, const int* words, int* stream,
                               int* take_pos) {
  dim3 grid(icrl_cdiv((long long)(n + 1) * B, 256 * 4), K * k);
  lookahead_stream_kernel<<<grid, 256, 0, st>>>(B, n, k, cand_tok, words, stream, take_pos);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_lookahead_score_impl(cudaStream_t st, int B, int K, int k, const float* parent, const float* values, const float* top_val,
                              float* child, float* means) {
  lookahead_score_kernel<<<K * k, 256, 0, st>>>(B, K, k, parent, values, top_val, child, means);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_gather_rows_impl(cudaStream_t st, long long R, const float* src, const int* idx, long long row_offset,
                          float* dst) {
  gather_rows_kernel<<<icrl_cdiv(R * (H / 4), 256), 256, 0, st>>>(R, src, idx, row_offset, dst);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_add_gate_bias_impl(cudaStream_t st, int V, int G, int fold, const float* b_ih, const float* b_hh,
                            float* table) {
  add_gate_bias_kernel<<<icrl_cdiv((long long)V * G, 256), 256, 0, st>>>(V, G, fold, b_ih, b_hh, table);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}
