// Policy-side elementwise / row kernels of the rollout:
//   LSTM cell update and its backward (models.py:80; gate order i,f,g,o),
//   softmax -> numpy-semantics inverse-CDF sampling or greedy argmax -> log-prob
//   (trainers.py:444-458, :69), softmax backward, and the gate-table gradient scatter.
#include <cuda_fp16.h>
#include "common.cuh"

namespace {

constexpr int H = ICRL_H;

// gates_pre = gpre[b] (h_{t-1} W_hh^T) + table[tok[b]] (W_ih E[tok] + b_ih + b_hh)
__global__ void lstm_pointwise_fwd_kernel(int B, const float* __restrict__ gpre, const float* __restrict__ table,
                                          const int* __restrict__ tok, const float* __restrict__ c_prev,
                                          float* __restrict__ gates_act, float* __restrict__ c_out,
                                          float* __restrict__ h_out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx % H;
  const float* g = gpre + (size_t)b * 4 * H;
  const float* t = table + (size_t)tok[b] * 4 * H;
  const float i = sigmoidf_acc(g[u] + t[u]);
  const float f = sigmoidf_acc(g[H + u] + t[H + u]);
  const float gg = tanhf(g[2 * H + u] + t[2 * H + u]);
  const float o = sigmoidf_acc(g[3 * H + u] + t[3 * H + u]);
  const float c = f * c_prev[idx] + i * gg;
  float* ga = gates_act + (size_t)b * 4 * H;
  ga[u] = i; ga[H + u] = f; ga[2 * H + u] = gg; ga[3 * H + u] = o;
  c_out[idx] = c;
  h_out[idx] = o * tanhf(c);
}

// dh = dh_rec + dh_add; writes pre-activation gate gradients and dc for the previous step (in place).
__global__ void lstm_pointwise_bwd_kernel(int B, const float* __restrict__ dh_rec, const float* __restrict__ dh_add,
                                          float* __restrict__ dc, const float* __restrict__ gates_act,
                                          const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                          float* __restrict__ dgpre) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx % H;
  const float* ga = gates_act + (size_t)b * 4 * H;
  const float i = ga[u], f = ga[H + u], g = ga[2 * H + u], o = ga[3 * H + u];
  float dh = dh_rec ? dh_rec[idx] : 0.f;
  if (dh_add) dh += dh_add[idx];
  const float tc = tanhf(c_cur[idx]);
  const float dct = dc[idx] + dh * o * (1.f - tc * tc);
  float* dg = dgpre + (size_t)b * 4 * H;
  dg[u] = dct * g * i * (1.f - i);
  dg[H + u] = dct * c_prev[idx] * f * (1.f - f);
  dg[2 * H + u] = dct * i * (1.f - g * g);
  dg[3 * H + u] = dh * tc * o * (1.f - o);
  dc[idx] = dct * f;
}

// One warp per row.  softmax in f32 as torch does it (exp(x - max) * (1 / sum), trainers.py:444);
// sampling = numpy's RandomState.choice: cdf = cumsum(float64(p)); cdf /= cdf[-1];
// index = #(cdf <= u)  (searchsorted side='right', trainers.py:449).  Greedy = first argmax of the
// logits (trainers.py:69).  log-prob = log(p[a]) in f32 (trainers.py:458), not log-softmax.
__global__ void softmax_sample_kernel(int B, int V, const float* __restrict__ logits, int ldl,
                                      const double* __restrict__ uniforms, int greedy, const long long* __restrict__ forced,
                                      int* __restrict__ tok_next,
                                      long long* __restrict__ tokens_out, float* __restrict__ logp_out, int S, int s,
                                      float* __restrict__ probs_out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  const float* x = logits + (size_t)warp * ldl;
  const int per = (V + 31) / 32;                 // contiguous chunk per lane
  const int beg = min(V, lane * per), end = min(V, beg + per);
  float mx = -INFINITY;
  int amax = V;
  for (int v = beg; v < end; ++v) {
    const float xv = x[v];
    if (xv > mx) { mx = xv; amax = v; }
  }
  // warp argmax with smallest-index tie break
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, amax, o);
    if (om > mx || (om == mx && oa < amax)) { mx = om; amax = oa; }
  }
  float lsum = 0.f;
  for (int v = beg; v < end; ++v) lsum += expf(x[v] - mx);
  const float inv = 1.0f / warp_sum(lsum);
  int a;
  if (forced) {
    a = (int)forced[(size_t)warp * S + s];
  } else if (greedy) {
    a = amax;
  } else {
    double loc = 0.0;
    for (int v = beg; v < end; ++v) loc += (double)(expf(x[v] - mx) * inv);
    // exclusive prefix of lane totals
    double pre = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(0xffffffffu, pre, o);
      if (lane >= o) pre += t;
    }
    const double total = __shfl_sync(0xffffffffu, pre, 31);
    double run = pre - loc;
    const double u = uniforms[warp];
    int cnt = 0;
    for (int v = beg; v < end; ++v) {
      run += (double)(expf(x[v] - mx) * inv);
      cnt += (run / total <= u) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    a = min(cnt, V - 1);
  }
  if (probs_out)
    for (int v = beg; v < end; ++v) probs_out[(size_t)warp * V + v] = expf(x[v] - mx) * inv;
  if (lane == 0) {
    tok_next[warp] = a;
    tokens_out[(size_t)warp * S + s] = a;
    logp_out[(size_t)warp * S + s] = logf(expf(x[a] - mx) * inv);
  }
}

// In place: row r = s*B + b of z (logits) becomes dL/dlogits = dlogp[b][s] * (onehot(a) - softmax(z)).
// entropy != NULL (entropy [B][S] of policy_entropy_kernel) adds the entropy bonus's term scale * p (log p + H), with
// log p = (z - max) - log(sum) so that it stays finite where p underflows to zero.
__global__ void softmax_bwd_kernel(int B, int S, int V, float* __restrict__ z, int ldl,
                                   const long long* __restrict__ tokens_out, const float* __restrict__ dlogp,
                                   const float* __restrict__ entropy, float scale) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * S) return;
  const int s = warp / B, b = warp % B;
  float* x = z + (size_t)warp * ldl;
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, x[v]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int v = lane; v < V; v += 32) sum += expf(x[v] - mx);
  const float tot = warp_sum(sum);
  const float inv = 1.0f / tot;
  const float d = dlogp[(size_t)b * S + s];
  const int a = (int)tokens_out[(size_t)b * S + s];
  if (entropy) {
    const float h = entropy[(size_t)b * S + s], lsum = logf(tot);
    for (int v = lane; v < V; v += 32) {
      const float p = expf(x[v] - mx) * inv;
      x[v] = d * ((v == a ? 1.f : 0.f) - p) + scale * p * ((x[v] - mx) - lsum + h);
    }
    return;
  }
  for (int v = lane; v < V; v += 32) {
    const float p = expf(x[v] - mx) * inv;
    x[v] = d * ((v == a ? 1.f : 0.f) - p);
  }
}

// One warp per row r = s*B + b of the logits stash (row stride ldl, the V real columns only): entropy[b][s] =
// -sum p log p = log(sum) - sum e (z - max) / sum with e = exp(z - max), the max / exp / sum of softmax_bwd_kernel.
// A column whose e underflows to zero adds nothing (also for z = -inf).
__global__ void policy_entropy_kernel(int B, int S, int V, const float* __restrict__ logits, int ldl,
                                      float* __restrict__ entropy) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * S) return;
  const int s = warp / B, b = warp % B;
  const float* x = logits + (size_t)warp * ldl;
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, x[v]);
  mx = warp_max(mx);
  float sum = 0.f, t = 0.f;
  for (int v = lane; v < V; v += 32) {
    const float y = x[v] - mx, e = expf(y);
    sum += e;
    if (e > 0.f) t = fmaf(e, y, t);
  }
  const float tot = warp_sum(sum);
  t = warp_sum(t);
  if (lane == 0) entropy[(size_t)b * S + s] = logf(tot) - t / tot;
}

// Weighted cross entropy of the policy's supervised pretraining (trainers.py:202-257).  One warp per row r = s*B + b of
// the teacher-forced logits stash z [S][B][V]: for s < n[b], with p = softmax(z) (the max / exp / sum of
// softmax_bwd_kernel), ce[r] = log(sum exp(z - max)) - (z[t] - max) -- finite where p[t] underflows, unlike log(p[t]) --
// and dz[r][v] = w[b] (p[v] - [v == t]), t = target[b][s]; rows with s >= n[b] get ce = 0 and dz = 0.  Columns V..ldz-1
// of dz are written zero.  z is read only, so the backward can be re-run from it.
__global__ void policy_xent_kernel(int B, int S, int V, const float* __restrict__ z, const long long* __restrict__ target,
                                   const int* __restrict__ n_rows, const double* __restrict__ w_rows, float* __restrict__ dz,
                                   int ldz, float* __restrict__ ce) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * S) return;
  const int s = warp / B, b = warp % B;
  float* d = dz + (size_t)warp * ldz;
  if (s >= n_rows[b]) {
    for (int v = lane; v < ldz; v += 32) d[v] = 0.f;
    if (lane == 0) ce[warp] = 0.f;
    return;
  }
  const float* x = z + (size_t)warp * V;
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, x[v]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int v = lane; v < V; v += 32) sum += expf(x[v] - mx);
  const float tot = warp_sum(sum);
  const float inv = 1.0f / tot;
  const int t = (int)target[(size_t)b * S + s];
  const float w = (float)w_rows[b];
  for (int v = lane; v < V; v += 32) d[v] = w * (expf(x[v] - mx) * inv - (v == t ? 1.f : 0.f));
  for (int v = V + lane; v < ldz; v += 32) d[v] = 0.f;
  if (lane == 0) ce[warp] = logf(tot) - (x[t] - mx);
}

// Single block: loss = sum_r w[r % B] ce[r] in double, in a fixed order (no atomics), as a2c_loss_kernel sums.
__global__ void xent_loss_kernel(int B, int n, const float* __restrict__ ce, const double* __restrict__ w_rows,
                                 float* __restrict__ loss) {
  __shared__ double red[32];
  double l = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) l += w_rows[i % B] * (double)ce[i];
  l = warp_sum_d(l);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[w] = l;
  __syncthreads();
  if (w == 0) {
    l = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.0;
    l = warp_sum_d(l);
    if (lane == 0) loss[0] = (float)l;
  }
}

// The same with 16-byte vector reductions (red.global.add.v4.f32, sm_90+): a quarter of the instructions and of the L2
// atomic transactions of the scalar form (1.6 G atomics per step at B = 4096: 3.9 ms, 6.5 % of the step).  C % 4 == 0.
__global__ void scatter_add_rows_v4_kernel(long long R, int C4, const float4* __restrict__ src, const int* __restrict__ idx,
                                           float* __restrict__ dst) {
  const long long total = R * C4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C4;
    const int c = (int)(i % C4);
    const float4 v = __ldg(src + i);
    float* d = dst + ((size_t)idx[r] * C4 + c) * 4;
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(d), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  }
}

// The same for the rows of a batch-as-time token stream (build_stream_kernel, heads.cu): block s of the stream holds the
// columns 0 .. p0+s+extra-1 of the [col][B] token matrix, so the token at (col, b) is consumed once in every block that
// contains column col.  Those positions are summed in registers first -- one vector reduction per (col, b) instead of
// one per stream position: B * n_col * C/4 of them instead of T * C/4 (10 times fewer at 19 rollout steps), which turns
// the scatter from atomic-throughput-bound into a streaming read of src.  The kernel also returns the column |max| of
// src (the weight-gradient GEMM's per-column scale: wgrad_tc.cu) from the values it has in registers anyway.
// blockDim.x = C/4; thread c owns the 4 adjacent columns src.col(c) .. +3 of every row.
struct RowsF32 {                              // src [T][C] fp32
  const float4* src;
  __device__ float4 load(long long pos, int c) const { return __ldg(src + pos * blockDim.x + c); }
  __device__ int col(int c) const { return 4 * c; }
};
struct GatePairs {                            // the chain backward's [2][rows][2048] fp16 pairs (icrl_gate_pair_col order)
  const uint2* hi;                            // 4 halves per thread and row
  long long plane;                            // rows * 512
  const float* inv_scale;
  __device__ float4 load(long long pos, int c) const {
    const uint2 h = __ldg(hi + pos * 512 + c), l = __ldg(hi + plane + pos * 512 + c);
    const float2 h01 = __half22float2(*reinterpret_cast<const __half2*>(&h.x)), h23 = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
    const float2 l01 = __half22float2(*reinterpret_cast<const __half2*>(&l.x)), l23 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
    const float s = __ldg(inv_scale), li = 1.f / 2048.f;
    return make_float4(fmaf(l01.x, li, h01.x) * s, fmaf(l01.y, li, h01.y) * s, fmaf(l23.x, li, h23.x) * s, fmaf(l23.y, li, h23.y) * s);
  }
  __device__ int col(int c) const { return icrl_gate_pair_natural(4 * c); }
};
template <class Src>
__global__ void scatter_add_stream_kernel(int B, int p0, int S, int extra, const Src src, const int* __restrict__ tok_stream,
                                          float* __restrict__ dst, unsigned* __restrict__ colmax) {
  const int C = 4 * blockDim.x, c = threadIdx.x;
  const int n_col = p0 + S - 1 + extra;
  const long long rows = (long long)n_col * B;
  float4 mx = make_float4(0.f, 0.f, 0.f, 0.f);
  auto take = [&](float4& acc, const float4 v) {
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    mx.x = fmaxf(mx.x, fabsf(v.x)); mx.y = fmaxf(mx.y, fabsf(v.y)); mx.z = fmaxf(mx.z, fabsf(v.z)); mx.w = fmaxf(mx.w, fabsf(v.w));
  };
  for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
    const int col = (int)(r / B), b = (int)(r % B);
    const int s0 = max(0, col - p0 - extra + 1);                       // first block with more than `col` columns
    // stream position of (col, b) in block s: B * (s * (p0 + extra) + s (s - 1) / 2) + col * B + b
    auto pos = [&](int s) { return (long long)B * ((long long)s * (p0 + extra) + (long long)s * (s - 1) / 2 + col) + b; };
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = s0;
    for (; s + 3 < S; s += 4) {
      const float4 v0 = src.load(pos(s), c), v1 = src.load(pos(s + 1), c);
      const float4 v2 = src.load(pos(s + 2), c), v3 = src.load(pos(s + 3), c);
      take(acc, v0); take(acc, v1); take(acc, v2); take(acc, v3);
    }
    for (; s < S; ++s) take(acc, src.load(pos(s), c));
    float* d = dst + (size_t)tok_stream[pos(s0)] * C + src.col(c);
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(d), "f"(acc.x), "f"(acc.y), "f"(acc.z), "f"(acc.w) : "memory");
  }
  if (colmax) {                                                        // non-negative floats order like their bit patterns
    const int c0 = src.col(c);
    atomicMax(colmax + c0, __float_as_uint(mx.x));
    atomicMax(colmax + c0 + 1, __float_as_uint(mx.y));
    atomicMax(colmax + c0 + 2, __float_as_uint(mx.z));
    atomicMax(colmax + c0 + 3, __float_as_uint(mx.w));
  }
}

// dst[idx[r]][c] += src[r][c]   (gate-table gradient: rows that consumed the same token accumulate)
__global__ void scatter_add_rows_kernel(long long R, int C, const float* __restrict__ src, const int* __restrict__ idx,
                                        float* __restrict__ dst) {
  const long long total = R * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i % C);
    atomicAdd(dst + (size_t)idx[r] * C + c, src[i]);
  }
}

// out[c] = sum_r w[r] * X[r % row_mod][c]  (w may be null => 1).  Stage 1 writes per-chunk partials.
__global__ void wcolsum_stage1_kernel(long long R, int C, const float* __restrict__ X, const float* __restrict__ w,
                                      long long row_mod, long long rows_per_chunk, float* __restrict__ partial) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const long long r0 = (long long)blockIdx.y * rows_per_chunk, r1 = min(R, r0 + rows_per_chunk);
  float acc = 0.f;
  for (long long r = r0; r < r1; ++r) {
    const float xv = X[(size_t)(r % row_mod) * C + c];
    acc += w ? w[r] * xv : xv;
  }
  partial[(size_t)blockIdx.y * C + c] = acc;
}
__global__ void wcolsum_stage2_kernel(int C, int chunks, const float* __restrict__ partial, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float acc = 0.f;
  for (int k = 0; k < chunks; ++k) acc += partial[(size_t)k * C + c];
  out[c] = acc;
}

// Order of the row top-k: larger value first, equal values by lower index; a NaN ranks above every number (torch.topk).
__device__ __forceinline__ bool topk_before(float va, int ia, float vb, int ib) {
  const bool na = va != va, nb = vb != vb;
  if (na || nb) return na && (!nb || ia < ib);
  return va > vb || (va == vb && ia < ib);
}

// One warp per row: k rounds, each the warp-wide first element (in topk_before order) that ranks after the previous pick.
__global__ void topk_rows_kernel(int R, int V, int k, const float* __restrict__ x, float* __restrict__ top_val,
                                 int* __restrict__ top_idx) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= R) return;
  const float* xr = x + (size_t)row * V;
  float pv = 0.f;
  int pi = -1;
  for (int r = 0; r < k; ++r) {
    float bv = 0.f;
    int bi = -1;
    for (int j = lane; j < V; j += 32) {
      const float v = xr[j];
      if (pi >= 0 && !topk_before(pv, pi, v, j)) continue;
      if (bi < 0 || topk_before(v, j, bv, bi)) { bv = v; bi = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || topk_before(ov, oi, bv, bi))) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
      top_val[(size_t)row * k + r] = bv;
      top_idx[(size_t)row * k + r] = bi;
    }
    pv = bv;
    pi = bi;
  }
}

}  // namespace

int icrl_topk_rows(cudaStream_t st, int R, int V, int k, const float* x, float* top_val, int* top_idx) {
  ICRL_REQUIRE(R > 0 && k >= 1 && k <= 16 && k <= V, "row top-k needs 1 <= k <= min(16, V)");
  topk_rows_kernel<<<icrl_cdiv((long long)R * 32, 256), 256, 0, st>>>(R, V, k, x, top_val, top_idx);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_lstm_pointwise_fwd(cudaStream_t st, int B, const float* gpre, const float* table, const int* tok,
                            const float* c_prev, float* gates_act, float* c_out, float* h_out) {
  lstm_pointwise_fwd_kernel<<<icrl_cdiv((long long)B * H, 256), 256, 0, st>>>(B, gpre, table, tok, c_prev, gates_act,
                                                                             c_out, h_out);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_lstm_pointwise_bwd(cudaStream_t st, int B, const float* dh_rec, const float* dh_add, float* dc,
                            const float* gates_act, const float* c_prev, const float* c_cur, float* dgpre) {
  lstm_pointwise_bwd_kernel<<<icrl_cdiv((long long)B * H, 256), 256, 0, st>>>(B, dh_rec, dh_add, dc, gates_act, c_prev,
                                                                             c_cur, dgpre);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_softmax_sample(cudaStream_t st, int B, int V, const float* logits, int ldl, const double* uniforms, int greedy,
                        const long long* forced, int* tok_next, long long* tokens_out, float* logp_out, int S, int s, float* probs_out) {
  softmax_sample_kernel<<<icrl_cdiv((long long)B * 32, 128), 128, 0, st>>>(B, V, logits, ldl, uniforms, greedy, forced, tok_next,
                                                                          tokens_out, logp_out, S, s, probs_out);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_softmax_bwd(cudaStream_t st, int B, int S, int V, float* z, int ldl, const long long* tokens_out,
                     const float* dlogp, const float* entropy, float scale) {
  softmax_bwd_kernel<<<icrl_cdiv((long long)B * S * 32, 128), 128, 0, st>>>(B, S, V, z, ldl, tokens_out, dlogp, entropy,
                                                                           scale);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_policy_entropy_impl(cudaStream_t st, int B, int S, int V, const float* logits, int ldl, float* entropy) {
  policy_entropy_kernel<<<icrl_cdiv((long long)B * S * 32, 128), 128, 0, st>>>(B, S, V, logits, ldl, entropy);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_policy_xent_impl(cudaStream_t st, int B, int S, int V, const float* logits, const long long* targets,
                          const int* n_rows, const double* w_rows, float* dz, int ldz, float* ce, float* loss) {
  policy_xent_kernel<<<icrl_cdiv((long long)B * S * 32, 128), 128, 0, st>>>(B, S, V, logits, targets, n_rows, w_rows, dz, ldz,
                                                                           ce);
  ICRL_LAUNCH_CHECK();
  xent_loss_kernel<<<1, 1024, 0, st>>>(B, B * S, ce, w_rows, loss);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

int icrl_scatter_add_rows(cudaStream_t st, long long R, int C, const float* src, const int* idx, float* dst) {
  const long long total = R * C;
  const int blocks = (int)min((long long)148 * 16, (total + 255) / 256);
  if (C % 4 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    scatter_add_rows_v4_kernel<<<blocks, 256, 0, st>>>(R, C / 4, reinterpret_cast<const float4*>(src), idx, dst);
    ICRL_LAUNCH_CHECK();
    return ICRL_OK;
  }
  scatter_add_rows_kernel<<<blocks, 256, 0, st>>>(R, C, src, idx, dst);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// src [T][C] rows of the stream of icrl_build_stream(B, p0, S, extra); colmax (nullable): C words, zeroed here.
int icrl_scatter_add_stream(cudaStream_t st, int B, int p0, int S, int extra, int C, const float* src, const int* tok_stream,
                            float* dst, unsigned* colmax) {
  ICRL_REQUIRE(B >= 1 && p0 >= 1 && S >= 1 && extra >= 0, "bad stream shape");
  ICRL_REQUIRE(C % 4 == 0 && C / 4 <= 1024 && (C / 4) % 32 == 0, "scatter_add_stream: C must be a multiple of 128, at most 4096");
  ICRL_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, "unaligned rows");
  if (colmax) ICRL_CUDA(cudaMemsetAsync(colmax, 0, (size_t)C * sizeof(unsigned), st));
  const long long rows = (long long)(p0 + S - 1 + extra) * B;
  const int blocks = (int)min((long long)148 * 4, rows);
  scatter_add_stream_kernel<<<blocks, C / 4, 0, st>>>(B, p0, S, extra, RowsF32{reinterpret_cast<const float4*>(src)}, tok_stream,
                                                      dst, colmax);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// The same with src = the chain backward's gate-gradient pairs (planes [2][pair_rows][2048], icrl_gate_pair_col order,
// values (hi + lo'/2048) * *inv_scale); dst [V][2048] in natural column order.
int icrl_scatter_add_stream_pairs(cudaStream_t st, int B, int p0, int S, int extra, const void* pairs, long long pair_rows,
                                  const float* inv_scale, const int* tok_stream, float* dst) {
  ICRL_REQUIRE(B >= 1 && p0 >= 1 && S >= 1 && extra >= 0, "bad stream shape");
  ICRL_REQUIRE(((reinterpret_cast<uintptr_t>(pairs) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, "unaligned rows");
  const long long rows = (long long)(p0 + S - 1 + extra) * B;
  const int blocks = (int)min((long long)148 * 4, rows);
  const GatePairs src{reinterpret_cast<const uint2*>(pairs), pair_rows * 512, inv_scale};
  scatter_add_stream_kernel<<<blocks, 512, 0, st>>>(B, p0, S, extra, src, tok_stream, dst, nullptr);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// partial must hold chunks*C floats with chunks = icrl_wcolsum_chunks(R)
int icrl_wcolsum_chunks(long long R) { return (int)min((long long)296, (R + 63) / 64); }

int icrl_wcolsum(cudaStream_t st, long long R, int C, const float* X, const float* w, long long row_mod,
                 float* partial, float* out) {
  const int chunks = icrl_wcolsum_chunks(R);
  const long long rpc = (R + chunks - 1) / chunks;
  dim3 grid(icrl_cdiv(C, 128), chunks);
  wcolsum_stage1_kernel<<<grid, 128, 0, st>>>(R, C, X, w, row_mod > 0 ? row_mod : R, rpc, partial);
  ICRL_LAUNCH_CHECK();
  wcolsum_stage2_kernel<<<icrl_cdiv(C, 128), 128, 0, st>>>(C, chunks, partial, out);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}
