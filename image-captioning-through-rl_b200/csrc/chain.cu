// Serial-chain kernels for the reference's batch-as-time value (LSTM) and reward (GRU) RNNs.
//
// The reference feeds each caption COLUMN of B rows to a non-batch_first RNN, i.e. seq_len = B,
// batch = 1, and carries the hidden state between calls (models.py:133, 226; reset once per
// minibatch, trainers.py:495-496).  A minibatch is therefore ONE strictly serial recurrence over
// T = B * sum_s (p0 + s [+1]) tokens.  It is latency bound: each step is a batch-1 GEMV against
// W_hh followed by the cell update, and step t+1 cannot start before all of h_t exists.
//
// Design (grid-persistent, cooperative launch, one chain = 64 CTAs x 8 warps):
//   * warp w of CTA c owns hidden unit u = 8c + w: its NG gate rows of W_hh (NG x 512 floats) live
//     in REGISTERS for the whole kernel (64 regs/lane for the LSTM, 48 for the GRU); the input half
//     W_ih E[tok] + b is a precomputed gate table gathered by token id (prefetched one step ahead).
//   * per step every CTA needs all 512 h values.  They are exchanged through L2 as 64-bit
//     {float value, uint32 step tag} words (single-copy atomic, no fences, no flags): the producer
//     lane stores one word, consumers poll the words themselves.  Double buffered by step parity.
//   * the backward kernel exchanges dh_t the same way (512 words per step); every CTA rebuilds all
//     2048 gate gradients from it, and warp u holds column u of W_hh (2048 floats, 64 regs/lane) to
//     compute dh_{t-1}[u].
//   * every spin is bounded (watchdog) and checks a global abort word, so a scheduling failure
//     returns ICRL_ERR_WATCHDOG instead of hanging the GPU.
//   * batched kernels (second half of the file): the same CTAs advance K = 2, 4 or 8 independent row shards of the
//     batch from zero state in lockstep ("chain shards", the numbers of K data-parallel ranks), sharing the
//     register-resident weights and one exchange round trip.
#include <cooperative_groups.h>
#include "common.cuh"

namespace {

constexpr int H = ICRL_H;
constexpr int UNITS = 8;              // hidden units (= warps) per CTA
constexpr int CHAIN_CTAS = H / UNITS; // 64 CTAs per chain
constexpr int THREADS = UNITS * 32;
constexpr unsigned SPIN_LIMIT = 1u << 22;

// Activations on the serial critical path.  The accurate forms (expf, IEEE division, branchy tanhf)
// cost 466 cycles per LSTM step, the SFU forms 180 (scripts/xchg_bench.cu, measured on B200).  The SFU
// forms have abs error ~1e-7 on the O(1) gate values; the recurrence is contractive, so the values
// stay within the 1e-5 parity budget (checked by tests/test_gpu_parity.py at B=256, 48,640 steps).
#ifndef ICRL_CHAIN_ACT
#define ICRL_CHAIN_ACT 1
#endif
__device__ __forceinline__ float act_sigmoid(float x) {
#if ICRL_CHAIN_ACT
  return __fdividef(1.0f, 1.0f + __expf(-x));            // MUFU.EX2 + MUFU.RCP
#else
  return sigmoidf_acc(x);
#endif
}
__device__ __forceinline__ float act_tanh(float x) {
#if ICRL_CHAIN_ACT
  return 1.0f - 2.0f * __fdividef(1.0f, 1.0f + __expf(2.0f * x));
#else
  return tanhf(x);
#endif
}

__device__ __forceinline__ void ld_tagged2(const unsigned long long* p, unsigned long long& a, unsigned long long& b) {
  asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p));
}
// A fence after the publishing store shortens the isolated two-CTA ping-pong (968 -> 821 cycles one way,
// scripts/chain_micro.cu) but LENGTHENS the real step (B=256: fwd 69.7 -> 76.2 ms, bwd 66.8 -> 81.2 ms): the
// warp reconverges behind the fenced lane and its next poll issues late.  Kept as a build switch, off.
#ifndef ICRL_CHAIN_FENCE
#define ICRL_CHAIN_FENCE 0
#endif
__device__ __forceinline__ void st_tagged(unsigned long long* p, float v, unsigned tag) {
  const unsigned long long w = ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(v);
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
#if ICRL_CHAIN_FENCE
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
#endif
}

struct ChainFwdArgs {
  const int* stream;          // [T] token ids
  int T;
  const float* table;         // [V][NG*H]  W_ih E[v] + b_ih (+ b_hh where it folds)
  const float* w_hh;          // [NG*H][H]
  const float* b_hn;          // GRU: [H] hidden bias of the n gate (kept inside r*(.)); LSTM: unused
  const float* h0;            // [H] or null (zeros)
  const float* c0;            // [H] or null (LSTM)
  float* stash_h;             // [(T+1)][H]; row 0 = initial h, row t+1 = h_t
  float* stash_c;             // LSTM: [(T+1)][H] or null
  float* stash_gates;         // [T][4H] or null.  LSTM: activated i,f,g,o.  GRU: r, z, n, W_hn h + b_hn
  float* h_out;               // [H] final h or null
  float* c_out;               // [H] final c or null
  unsigned long long* xchg;   // [2][H] tagged exchange words, zeroed before launch
  int* abort_flag;            // global abort word, zeroed before launch
};

// Fetch the full exchanged vector of step `tag` (N floats, N = NV * THREADS * 2) into smem.
template <int NV>
__device__ __forceinline__ bool fetch_exchange(const unsigned long long* buf, unsigned tag, float* sm,
                                               volatile int* abort_flag) {
  bool ok = true;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int e = (v * THREADS + threadIdx.x) * 2;
    unsigned long long a, b;
    unsigned spins = 0;
    while (true) {
      ld_tagged2(buf + e, a, b);
      if ((unsigned)(a >> 32) == tag && (unsigned)(b >> 32) == tag) break;
      if (++spins >= SPIN_LIMIT || ((spins & 1023u) == 0 && *abort_flag != 0)) { ok = false; break; }
    }
    reinterpret_cast<float2*>(sm)[v * THREADS + threadIdx.x] =
        make_float2(__uint_as_float((unsigned)a), __uint_as_float((unsigned)b));
  }
  return ok;
}

// transposed butterfly: v[0..NB) per lane in, afterwards lane l holds in v[0] the warp-wide sum of element
// b = l >> (5 - log2 NB)
template <int NB>
__device__ __forceinline__ float reduce_transposed(float (&v)[NB], int lane) {
  int o = 16;
#pragma unroll
  for (int n = NB; n > 1; n >>= 1, o >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = upper ? v[i] : v[i + n / 2];
      const float keep = upper ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  for (; o > 0; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
  return v[0];
}

// Batched form: all NV polls are in flight before the first tag is examined (one L2 round trip for the whole
// batch instead of one per vector); only words that had not arrived yet are polled again.
template <int NV>
__device__ __forceinline__ void exchange_issue(const unsigned long long* buf, unsigned long long (&a)[NV],
                                               unsigned long long (&b)[NV]) {
#pragma unroll
  for (int v = 0; v < NV; ++v) ld_tagged2(buf + (v * THREADS + threadIdx.x) * 2, a[v], b[v]);
}
// Poll in ROUNDS: every word that has not arrived is re-read in the same round (one L2 round trip per round).
// Re-polling word by word costs one round trip per word, because the first sample of every later word was
// taken before the data existed: measured 1,705 / 2,593 / 5,574 cycles of wait at NV = 2 / 4 / 8.
template <int NV>
__device__ __forceinline__ bool exchange_complete(const unsigned long long* buf, unsigned tag, float* sm,
                                                  volatile int* abort_flag, unsigned long long (&a)[NV],
                                                  unsigned long long (&b)[NV]) {
  unsigned pending = (1u << NV) - 1u, spins = 0;
  bool ok = true;
  while (true) {
#pragma unroll
    for (int v = 0; v < NV; ++v)
      if ((pending >> v & 1u) && (unsigned)(a[v] >> 32) == tag && (unsigned)(b[v] >> 32) == tag) pending &= ~(1u << v);
    if (pending == 0) break;
    if (++spins >= SPIN_LIMIT || ((spins & 1023u) == 0 && *abort_flag != 0)) { ok = false; break; }
#pragma unroll
    for (int v = 0; v < NV; ++v)
      if (pending >> v & 1u) ld_tagged2(buf + (v * THREADS + threadIdx.x) * 2, a[v], b[v]);
  }
#pragma unroll
  for (int v = 0; v < NV; ++v)
    reinterpret_cast<float2*>(sm)[v * THREADS + threadIdx.x] =
        make_float2(__uint_as_float((unsigned)a[v]), __uint_as_float((unsigned)b[v]));
  return ok;
}
template <int NV>
__device__ __forceinline__ bool fetch_exchange_all(const unsigned long long* buf, unsigned tag, float* sm,
                                                   volatile int* abort_flag) {
  unsigned long long a[NV], b[NV];
  exchange_issue<NV>(buf, a, b);
  return exchange_complete<NV>(buf, tag, sm, abort_flag, a, b);
}

template <int NG>   // 4 = LSTM (i,f,g,o), 3 = GRU (r,z,n)
__device__ void chain_fwd_body(const ChainFwdArgs& p, int cta) {
  __shared__ __align__(16) float sh_h[2][H];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = cta * UNITS + warp;

  float w[NG][16];
#pragma unroll
  for (int g = 0; g < NG; ++g)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 t = *reinterpret_cast<const float4*>(p.w_hh + (size_t)(g * H + unit) * H + 128 * j + 4 * lane);
      w[g][4 * j + 0] = t.x; w[g][4 * j + 1] = t.y; w[g][4 * j + 2] = t.z; w[g][4 * j + 3] = t.w;
    }
  const float bhn = (NG == 3) ? p.b_hn[unit] : 0.f;
  float c = (NG == 4 && p.c0) ? p.c0[unit] : 0.f;
  float hprev = p.h0 ? p.h0[unit] : 0.f;
  if (lane == 0) {
    p.stash_h[unit] = hprev;
    if (NG == 4 && p.stash_c) p.stash_c[unit] = c;
  }
  // step-0 vector straight from h0
  for (int i = threadIdx.x; i < H; i += THREADS) sh_h[0][i] = p.h0 ? p.h0[i] : 0.f;

  // token / gate-table prefetch pipeline (tokens are known up front)
  int tok_next = p.T > 1 ? p.stream[1] : 0;
  float xg[NG];
  {
    const int tok0 = p.stream[0];
#pragma unroll
    for (int g = 0; g < NG; ++g) xg[g] = p.table[(size_t)tok0 * (NG * H) + g * H + unit];
  }

  for (int t = 0; t < p.T; ++t) {
    const int buf = t & 1;
    bool ok = true;
    if (t > 0) ok = fetch_exchange<1>(p.xchg + (size_t)((t - 1) & 1) * H, (unsigned)t, sh_h[buf], p.abort_flag);
    if (__syncthreads_or(!ok)) {
      if (threadIdx.x == 0) atomicExch(p.abort_flag, 1);
      return;
    }
    // prefetch next step's gate-table entries and the token after it
    float xg_n[NG];
    {
      const int tk = tok_next;
      if (t + 1 < p.T) {
#pragma unroll
        for (int g = 0; g < NG; ++g) xg_n[g] = p.table[(size_t)tk * (NG * H) + g * H + unit];
      } else {
#pragma unroll
        for (int g = 0; g < NG; ++g) xg_n[g] = 0.f;
      }
      tok_next = (t + 2 < p.T) ? p.stream[t + 2] : 0;
    }
    // batch-1 GEMV: NG rows x 512, weights in registers, h from smem
    float acc[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) acc[g] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 hv = *reinterpret_cast<const float4*>(&sh_h[buf][128 * j + 4 * lane]);
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        acc[g] = fmaf(w[g][4 * j + 0], hv.x, acc[g]);
        acc[g] = fmaf(w[g][4 * j + 1], hv.y, acc[g]);
        acc[g] = fmaf(w[g][4 * j + 2], hv.z, acc[g]);
        acc[g] = fmaf(w[g][4 * j + 3], hv.w, acc[g]);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int g = 0; g < NG; ++g) acc[g] += __shfl_xor_sync(0xffffffffu, acc[g], o);

    float hnew;
    if constexpr (NG == 4) {
      const float i = act_sigmoid(acc[0] + xg[0]);
      const float f = act_sigmoid(acc[1] + xg[1]);
      const float g = act_tanh(acc[2] + xg[2]);
      const float o = act_sigmoid(acc[3 % NG] + xg[3 % NG]);
      c = f * c + i * g;
      hnew = o * act_tanh(c);
      if (p.stash_gates) {
        const float sel = lane == 0 ? i : (lane == 1 ? f : (lane == 2 ? g : o));
        if (lane < 4) p.stash_gates[(size_t)t * 4 * H + lane * H + unit] = sel;
      }
      if (p.stash_c && lane == 4) p.stash_c[(size_t)(t + 1) * H + unit] = c;
    } else {
      const float r = act_sigmoid(acc[0] + xg[0]);
      const float z = act_sigmoid(acc[1] + xg[1]);
      const float anh = acc[2] + bhn;
      const float n = act_tanh(xg[2] + r * anh);
      hnew = (1.f - z) * n + z * hprev;
      if (p.stash_gates && lane < 4) {                 // training stash of the reward GRU: r, z, n, W_hn h + b_hn
        const float sel = lane == 0 ? r : (lane == 1 ? z : (lane == 2 ? n : anh));
        p.stash_gates[(size_t)t * 4 * H + lane * H + unit] = sel;
      }
    }
    hprev = hnew;
    if (lane == 8) st_tagged(p.xchg + (size_t)buf * H + unit, hnew, (unsigned)(t + 1));
    if (lane == 5) p.stash_h[(size_t)(t + 1) * H + unit] = hnew;
#pragma unroll
    for (int g = 0; g < NG; ++g) xg[g] = xg_n[g];
  }
  if (lane == 0) {
    if (p.h_out) p.h_out[unit] = hprev;
    if (NG == 4 && p.c_out) p.c_out[unit] = c;
  }
}

__global__ void __launch_bounds__(THREADS, 1) chain_lstm_fwd_kernel(ChainFwdArgs a) { chain_fwd_body<4>(a, blockIdx.x); }
__global__ void __launch_bounds__(THREADS, 1) chain_gru_fwd_kernel(ChainFwdArgs a) { chain_fwd_body<3>(a, blockIdx.x); }
// value LSTM chain on CTAs 0..63 and reward GRU chain on CTAs 64..127 of one cooperative launch
__global__ void __launch_bounds__(THREADS, 1) chains_fwd_fused_kernel(ChainFwdArgs lstm, ChainFwdArgs gru) {
  if (blockIdx.x < CHAIN_CTAS) chain_fwd_body<4>(lstm, blockIdx.x);
  else chain_fwd_body<3>(gru, blockIdx.x - CHAIN_CTAS);
}

struct ChainBwdArgs {
  int T;
  const float* w_hh;          // [4H][H]
  const float* stash_gates;   // [T][4H] activated i,f,g,o
  const float* stash_c;       // [(T+1)][H]
  const int* take;            // [T]  row of dh_take injected at step t, or -1
  const float* dh_take;       // [S*B][H] dL/dh at the take positions (from the value head)
  float* dgates;              // [T][4H] pre-activation gate gradients (output, feeds dW_hh / table grads)
  unsigned long long* xchg;   // [2][H] tagged dh words
  int* abort_flag;
  const float* dh_init;       // [H] dL/dh_T flowing in from a later call that consumed the carried state, or null
  const float* dc_init;       // [H] dL/dc_T, or null
  float* dh0_out;             // [H] dL/dh_0 (gradient of the incoming hidden state), or null
  float* dc0_out;             // [H] dL/dc_0, or null
};

// Backward recurrence.  What crosses CTAs per step is dh_t (512 floats, the same volume and pattern as
// the forward kernel): every CTA redundantly turns dh_t into all 2048 gate gradients (two hidden units
// per thread; the stashed activations are prefetched a step ahead, dc is carried in registers), and warp
// w of CTA c then computes dh_{t-1}[u] = W_hh[:,u] . dgates_t for its unit u = 8c + w from column u of
// W_hh held in registers (64 per lane), adds the value-head gradient injected at take positions, and
// publishes it as one tagged word.
__global__ void __launch_bounds__(THREADS, 1) chain_lstm_bwd_kernel(ChainBwdArgs p) {
  __shared__ __align__(16) float sh_dg[2][4 * H];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cta = blockIdx.x;
  const int unit = cta * UNITS + warp;
  const int pu = 2 * threadIdx.x;                              // this thread's two pointwise units
  const bool owner = (pu >= cta * UNITS) && (pu < cta * UNITS + UNITS);

  // dh_{t-1}[u] = sum_j W_hh[j][u] dg[j] for the CTA's 8 units u.  The 2048 j are split over the 8 warps (warp w:
  // j in [256w, 256w+256), lane: 8 consecutive j) so that every dg value is read from shared memory by ONE lane
  // (the earlier warp-per-unit mapping had all 8 warps read all 2048 values: 64 KB of LDS per step, ~500 cycles).
  // wl[i][k] = W_hh[256w + 8 lane + k][8 cta + i]
  __shared__ float sh_part[UNITS][UNITS];                      // [warp][unit] partial sums
  float wl[UNITS][8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float* src = p.w_hh + (size_t)(256 * warp + 8 * lane + k) * H + cta * UNITS;
    const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
    wl[0][k] = x0.x; wl[1][k] = x0.y; wl[2][k] = x0.z; wl[3][k] = x0.w;
    wl[4][k] = x1.x; wl[5][k] = x1.y; wl[6][k] = x1.z; wl[7][k] = x1.w;
  }

  float2 dc = p.dc_init ? *reinterpret_cast<const float2*>(p.dc_init + pu) : make_float2(0.f, 0.f);
  auto load_step = [&](int t, float2& gi, float2& gf, float2& gg, float2& go, float2& cc, float2& cp) {
    const float* ga = p.stash_gates + (size_t)t * 4 * H + pu;
    gi = *reinterpret_cast<const float2*>(ga);
    gf = *reinterpret_cast<const float2*>(ga + H);
    gg = *reinterpret_cast<const float2*>(ga + 2 * H);
    go = *reinterpret_cast<const float2*>(ga + 3 * H);
    cc = *reinterpret_cast<const float2*>(p.stash_c + (size_t)(t + 1) * H + pu);
    cp = *reinterpret_cast<const float2*>(p.stash_c + (size_t)t * H + pu);
  };
  float2 gi, gf, gg, go, cc, cp;
  load_step(p.T - 1, gi, gf, gg, go, cc, cp);
  // dh of the last step is the injected head gradient only
  float2 dh = make_float2(0.f, 0.f);
  {
    const int tk = p.take[p.T - 1];
    if (tk >= 0) dh = *reinterpret_cast<const float2*>(p.dh_take + (size_t)tk * H + pu);
    if (p.dh_init) { dh.x += p.dh_init[pu]; dh.y += p.dh_init[pu + 1]; }
  }
  int tk_prev = p.T > 1 ? p.take[p.T - 2] : -1;                // injection for the dh this warp publishes

  for (int it = 0; it < p.T; ++it) {
    const int t = p.T - 1 - it;
    const int buf = it & 1;
    bool ok = true;
    unsigned long long a = 0, b = 0;
    const unsigned long long* src = p.xchg + (size_t)((it - 1) & 1) * H + pu;
    if (it > 0) ld_tagged2(src, a, b);                         // first poll in flight while the coefficients are computed
    // everything that does not depend on dh
    const float tcx = act_tanh(cc.x), tcy = act_tanh(cc.y);
    const float kcx = go.x * (1.f - tcx * tcx), kcy = go.y * (1.f - tcy * tcy);
    const float kox = tcx * go.x * (1.f - go.x), koy = tcy * go.y * (1.f - go.y);
    const float kix = gg.x * gi.x * (1.f - gi.x), kiy = gg.y * gi.y * (1.f - gi.y);
    const float kfx = cp.x * gf.x * (1.f - gf.x), kfy = cp.y * gf.y * (1.f - gf.y);
    const float kgx = gi.x * (1.f - gg.x * gg.x), kgy = gi.y * (1.f - gg.y * gg.y);
    const float inj = tk_prev >= 0 ? p.dh_take[(size_t)tk_prev * H + unit] : 0.f;
    float2 ngi = gi, ngf = gf, ngg = gg, ngo = go, ncc = cc, ncp = cp;
    if (t > 0) load_step(t - 1, ngi, ngf, ngg, ngo, ncc, ncp);
    tk_prev = t > 1 ? p.take[t - 2] : -1;

    if (it > 0) {
      unsigned spins = 0;
      while (!((unsigned)(a >> 32) == (unsigned)it && (unsigned)(b >> 32) == (unsigned)it)) {
        if (++spins >= SPIN_LIMIT || ((spins & 1023u) == 0 && *(volatile int*)p.abort_flag != 0)) { ok = false; break; }
        ld_tagged2(src, a, b);
      }
      dh = make_float2(__uint_as_float((unsigned)a), __uint_as_float((unsigned)b));
    }
    const float dctx = dc.x + dh.x * kcx, dcty = dc.y + dh.y * kcy;
    dc = make_float2(dctx * gf.x, dcty * gf.y);
    const float2 d_i = make_float2(dctx * kix, dcty * kiy), d_f = make_float2(dctx * kfx, dcty * kfy);
    const float2 d_g = make_float2(dctx * kgx, dcty * kgy), d_o = make_float2(dh.x * kox, dh.y * koy);
    *reinterpret_cast<float2*>(&sh_dg[buf][pu]) = d_i;
    *reinterpret_cast<float2*>(&sh_dg[buf][H + pu]) = d_f;
    *reinterpret_cast<float2*>(&sh_dg[buf][2 * H + pu]) = d_g;
    *reinterpret_cast<float2*>(&sh_dg[buf][3 * H + pu]) = d_o;
    if (owner) {
      float* out = p.dgates + (size_t)t * 4 * H + pu;
      *reinterpret_cast<float2*>(out) = d_i;
      *reinterpret_cast<float2*>(out + H) = d_f;
      *reinterpret_cast<float2*>(out + 2 * H) = d_g;
      *reinterpret_cast<float2*>(out + 3 * H) = d_o;
    }
    if (__syncthreads_or(!ok)) {
      if (threadIdx.x == 0) atomicExch(p.abort_flag, 1);
      return;
    }
    if (t > 0 || p.dh0_out) {
      const float4 d0 = *reinterpret_cast<const float4*>(&sh_dg[buf][256 * warp + 8 * lane]);
      const float4 d1 = *reinterpret_cast<const float4*>(&sh_dg[buf][256 * warp + 8 * lane + 4]);
      float part[UNITS];
#pragma unroll
      for (int i = 0; i < UNITS; ++i) {
        float a = wl[i][0] * d0.x;
        a = fmaf(wl[i][1], d0.y, a); a = fmaf(wl[i][2], d0.z, a); a = fmaf(wl[i][3], d0.w, a);
        a = fmaf(wl[i][4], d1.x, a); a = fmaf(wl[i][5], d1.y, a); a = fmaf(wl[i][6], d1.z, a); a = fmaf(wl[i][7], d1.w, a);
        part[i] = a;
      }
      const float ps = reduce_transposed<UNITS>(part, lane);      // lane l: unit l >> 2, summed over the warp's 256 j
      if ((lane & 3) == 0) sh_part[warp][lane >> 2] = ps;
      __syncthreads();
      if (lane < UNITS) {
        float rec = sh_part[lane][warp];                           // this warp finishes unit `warp`
        rec += __shfl_xor_sync(0xffu, rec, 1);
        rec += __shfl_xor_sync(0xffu, rec, 2);
        rec += __shfl_xor_sync(0xffu, rec, 4);
        if (lane == 0) {
          if (t > 0) st_tagged(p.xchg + (size_t)buf * H + unit, rec + inj, (unsigned)(it + 1));
          else p.dh0_out[unit] = rec;
        }
      }
    }
    gi = ngi; gf = ngf; gg = ngg; go = ngo; cc = ncc; cp = ncp;
  }
  if (p.dc0_out && owner) *reinterpret_cast<float2*>(p.dc0_out + pu) = dc;
}


// ------------------------------------------------------------------------------------------------------
// Batched chains: NB independent recurrences ("chain shards": row shards of the minibatch, each starting
// from zero state = the reference run on that shard, which is also what each data-parallel rank computes,
// SURVEY.md 8e/H6) advance in lockstep on the same CTAs.  They share W_hh in registers, and one L2 exchange
// round trip now carries NB hidden vectors, so the latency that bounds the single chain is amortised:
// the step becomes FMA-bound instead of exchange-bound.
// All per-step arrays of a shard use the same row stride (T + 1): stream [NB][stride], stash_h / stash_c
// [NB][stride][H], stash_gates / dgates [NB][stride][4H] (row T unused / zero), take [NB][stride].

constexpr int NB_MAX = 8;         // shards per launch: the exchange areas are sized for it

struct ChainFwdBatchArgs {
  const int* stream;          // [NB][stride]
  int T;
  long long stride;           // rows per shard (T + 1)
  const float* table;         // [V][NG*H]
  const float* w_hh;          // [NG*H][H]
  const float* b_hn;          // GRU only
  float* stash_h;             // [NB][stride][H]; row 0 = 0, row t+1 = h_t
  float* stash_c;             // LSTM: [NB][stride][H] or null
  float* stash_gates;         // LSTM: [NB][stride][4H] or null
  unsigned long long* xchg;   // [2][NB][H] tagged words, zeroed before launch
  int* abort_flag;
  long long* prof;            // debug: {exchange wait, GEMV + reduce, pointwise + publish} cycles of CTA 0 thread 0, T
};

// (Tried and dropped for this exchange, both slower at NB = 8: a unit-major word layout [unit][NB], 393 -> 426 ms, and
// plain data + one release flag per unit polled with acquire loads, 393 -> 508 ms: the release store waits for the
// warp's stash writes.)
template <int NG, int NB>
__device__ void chain_fwd_batched_body(const ChainFwdBatchArgs& p, int cta, float* sh_h /* [2][NB][H] */) {
  constexpr int GL = 32 / NB;                          // lanes per shard group after the transposed reduction
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = cta * UNITS + warp;
  const int b = lane / GL, sub = lane % GL;            // this lane's shard for the pointwise stage
  const int* my_stream = p.stream + (size_t)b * p.stride;

  float w[NG][16];
#pragma unroll
  for (int g = 0; g < NG; ++g)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 t = *reinterpret_cast<const float4*>(p.w_hh + (size_t)(g * H + unit) * H + 128 * j + 4 * lane);
      w[g][4 * j + 0] = t.x; w[g][4 * j + 1] = t.y; w[g][4 * j + 2] = t.z; w[g][4 * j + 3] = t.w;
    }
  const float bhn = (NG == 3) ? p.b_hn[unit] : 0.f;
  float c = 0.f, hprev = 0.f, xg[NG];
  if (sub == 0) {
    p.stash_h[(size_t)b * p.stride * H + unit] = 0.f;
    if (NG == 4 && p.stash_c) p.stash_c[(size_t)b * p.stride * H + unit] = 0.f;
  }
  int tok_next = p.T > 1 ? my_stream[1] : 0;
  {
    const int tok0 = my_stream[0];
#pragma unroll
    for (int g = 0; g < NG; ++g) xg[g] = p.table[(size_t)tok0 * (NG * H) + g * H + unit];
  }
  for (int i = threadIdx.x; i < 2 * NB * H; i += THREADS) sh_h[i] = 0.f;      // step-0 vectors: zero state

  long long prof_wait = 0, prof_gemv = 0, prof_rest = 0;
  const bool prof = p.prof != nullptr && cta == 0 && threadIdx.x == 0;
  for (int t = 0; t < p.T; ++t) {
    const long long c0 = prof ? clock64() : 0;
    const int buf = t & 1;
    float* hb = sh_h + (size_t)buf * NB * H;
    bool ok = true;
    if (t > 0) ok = fetch_exchange_all<NB>(p.xchg + (size_t)((t - 1) & 1) * NB * H, (unsigned)t, hb, p.abort_flag);
    if (__syncthreads_or(!ok)) {
      if (threadIdx.x == 0) atomicExch(p.abort_flag, 1);
      return;
    }
    const long long c1 = prof ? clock64() : 0;
    float xg_n[NG];
    {
      const int tk = tok_next;
      if (t + 1 < p.T) {
#pragma unroll
        for (int g = 0; g < NG; ++g) xg_n[g] = p.table[(size_t)tk * (NG * H) + g * H + unit];
      } else {
#pragma unroll
        for (int g = 0; g < NG; ++g) xg_n[g] = 0.f;
      }
      tok_next = (t + 2 < p.T) ? my_stream[t + 2] : 0;
    }
    // batch-NB GEMV: NG rows x 512 against NB hidden vectors, weights in registers
    float acc[NG][NB];
#pragma unroll
    for (int g = 0; g < NG; ++g)
#pragma unroll
      for (int v = 0; v < NB; ++v) acc[g][v] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int v = 0; v < NB; ++v) {
        const float4 hv = *reinterpret_cast<const float4*>(&hb[v * H + 128 * j + 4 * lane]);
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          acc[g][v] = fmaf(w[g][4 * j + 0], hv.x, acc[g][v]);
          acc[g][v] = fmaf(w[g][4 * j + 1], hv.y, acc[g][v]);
          acc[g][v] = fmaf(w[g][4 * j + 2], hv.z, acc[g][v]);
          acc[g][v] = fmaf(w[g][4 * j + 3], hv.w, acc[g][v]);
        }
      }
    }
    float sum[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) sum[g] = reduce_transposed<NB>(acc[g], lane);
    const long long c2 = prof ? clock64() : 0;

    const size_t row = (size_t)b * p.stride + t;       // this shard's row of the per-step arrays
    float hnew;
    if constexpr (NG == 4) {
      const float i = act_sigmoid(sum[0] + xg[0]);
      const float f = act_sigmoid(sum[1] + xg[1]);
      const float g = act_tanh(sum[2] + xg[2]);
      const float o = act_sigmoid(sum[3 % NG] + xg[3 % NG]);
      c = f * c + i * g;
      hnew = o * act_tanh(c);
      if (p.stash_gates) {                             // the GL lanes of a shard share the four stores
        if constexpr (GL >= 4) {
          if (sub < 4) p.stash_gates[row * 4 * H + sub * H + unit] = sub == 0 ? i : (sub == 1 ? f : (sub == 2 ? g : o));
        } else {
          p.stash_gates[row * 4 * H + sub * H + unit] = sub == 0 ? i : f;
          p.stash_gates[row * 4 * H + (2 + sub) * H + unit] = sub == 0 ? g : o;
        }
      }
      if (p.stash_c && sub == 4 % GL) p.stash_c[(row + 1) * H + unit] = c;
    } else {
      const float r = act_sigmoid(sum[0] + xg[0]);
      const float z = act_sigmoid(sum[1] + xg[1]);
      const float n = act_tanh(xg[2] + r * (sum[2] + bhn));
      hnew = (1.f - z) * n + z * hprev;
    }
    hprev = hnew;
    if (sub == 6 % GL) st_tagged(p.xchg + ((size_t)buf * NB + b) * H + unit, hnew, (unsigned)(t + 1));
    if (sub == 5 % GL) p.stash_h[(row + 1) * H + unit] = hnew;
#pragma unroll
    for (int g = 0; g < NG; ++g) xg[g] = xg_n[g];
    if (prof) { const long long c3 = clock64(); prof_wait += c1 - c0; prof_gemv += c2 - c1; prof_rest += c3 - c2; }
  }
  if (prof) { p.prof[0] = prof_wait; p.prof[1] = prof_gemv; p.prof[2] = prof_rest; p.prof[3] = p.T; }
}

template <int NB>
__global__ void __launch_bounds__(THREADS, 1) chains_fwd_fused_batched_kernel(ChainFwdBatchArgs lstm, ChainFwdBatchArgs gru) {
  extern __shared__ __align__(16) float sh_dyn[];
  if (blockIdx.x < CHAIN_CTAS) chain_fwd_batched_body<4, NB>(lstm, blockIdx.x, sh_dyn);
  else chain_fwd_batched_body<3, NB>(gru, blockIdx.x - CHAIN_CTAS, sh_dyn);
}

struct ChainBwdBatchArgs {
  int T;
  long long stride;
  const float* w_hh;          // [4H][H]
  const float* stash_gates;   // [shards][stride][4H]
  const float* stash_c;       // [shards][stride][H]
  const int* take;            // [shards][stride]
  const float* dh_take;       // [S*B][H]
  float* dgates;              // [shards][stride][4H]; row T of every shard is zeroed by the launcher
  unsigned long long* xchg;   // [2][shards][H]
  int shards;                 // total shards = gridDim.x / CHAIN_CTAS * NB
  int* abort_flag;
  long long* prof;            // debug: cycles of CTA 0 thread 0 {coefficients + requests, poll wait, gate gradients + stores,
                              // barrier, contraction + reduce, barrier + publish}, then T
};

// Backward recurrence of NB shards per 64-CTA group (see chain_lstm_bwd_kernel for the single-chain scheme).  The stash
// rows of the next step are requested before this step's gate gradients are computed, so they land under its arithmetic.
template <int NB, bool PROF>
__global__ void __launch_bounds__(THREADS, 1) chain_lstm_bwd_batched_kernel(ChainBwdBatchArgs p) {
  extern __shared__ __align__(16) float sh_dyn[];      // [2][NB][4H]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int group = blockIdx.x / CHAIN_CTAS, cta = blockIdx.x % CHAIN_CTAS;
  const int sb = group * NB;                           // first shard of this group
  const int unit = cta * UNITS + warp;
  const int pu = 2 * threadIdx.x;
  const bool owner = (pu >= cta * UNITS) && (pu < cta * UNITS + UNITS);
  const int myb = (lane >> 3) < NB ? (lane >> 3) : 0;  // shard whose dh lane 8*myb publishes

  // contraction split over the warps as in chain_lstm_bwd_kernel: wl[i][k] = W_hh[256w + 8 lane + k][8 cta + i]
  __shared__ float sh_part[UNITS][NB * UNITS];         // [warp][shard * 8 + unit]
  float wl[UNITS][8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float* src = p.w_hh + (size_t)(256 * warp + 8 * lane + k) * H + cta * UNITS;
    const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
    wl[0][k] = x0.x; wl[1][k] = x0.y; wl[2][k] = x0.z; wl[3][k] = x0.w;
    wl[4][k] = x1.x; wl[5][k] = x1.y; wl[6][k] = x1.z; wl[7][k] = x1.w;
  }

  float2 dc[NB], gi[NB], gf[NB], gg[NB], go[NB], cc[NB], cp[NB];
  auto load_step = [&](int shard, int t, float2& a_i, float2& a_f, float2& a_g, float2& a_o, float2& a_cc, float2& a_cp) {
    const float* ga = p.stash_gates + ((size_t)shard * p.stride + t) * 4 * H + pu;
    const float* ca = p.stash_c + ((size_t)shard * p.stride + t) * H + pu;
    a_i = *reinterpret_cast<const float2*>(ga);
    a_f = *reinterpret_cast<const float2*>(ga + H);
    a_g = *reinterpret_cast<const float2*>(ga + 2 * H);
    a_o = *reinterpret_cast<const float2*>(ga + 3 * H);
    a_cc = *reinterpret_cast<const float2*>(ca + H);
    a_cp = *reinterpret_cast<const float2*>(ca);
  };
#pragma unroll
  for (int v = 0; v < NB; ++v) dc[v] = make_float2(0.f, 0.f);
  int tk_prev = p.T > 1 ? p.take[(size_t)(sb + myb) * p.stride + p.T - 2] : -1;
#pragma unroll
  for (int v = 0; v < NB; ++v) load_step(sb + v, p.T - 1, gi[v], gf[v], gg[v], go[v], cc[v], cp[v]);
  unsigned long long pa[NB], pb[NB];                   // polled dh words
  const bool prof = PROF && blockIdx.x == 0 && threadIdx.x == 0;       // PROF: the cycle-split build of the kernel
  long long pr[PROF ? 6 : 1] = {};

  for (int it = 0; it < p.T; ++it) {
    const int t = p.T - 1 - it;
    const long long k0 = prof ? clock64() : 0;
    float* dgb = sh_dyn + (it & 1) * NB * 4 * H;
    bool ok = true;
    const unsigned long long* src = p.xchg + ((size_t)((it - 1) & 1) * p.shards + sb) * H + pu;
    if (it > 0) {
#pragma unroll
      for (int v = 0; v < NB; ++v) ld_tagged2(src + (size_t)v * H, pa[v], pb[v]);
    }
    // coefficients that do not depend on dh
    float2 kc[NB], ko[NB], ki[NB], kf[NB], kg[NB], fgate[NB], dh[NB];
#pragma unroll
    for (int v = 0; v < NB; ++v) {
      const float tcx = act_tanh(cc[v].x), tcy = act_tanh(cc[v].y);
      kc[v] = make_float2(go[v].x * (1.f - tcx * tcx), go[v].y * (1.f - tcy * tcy));
      ko[v] = make_float2(tcx * go[v].x * (1.f - go[v].x), tcy * go[v].y * (1.f - go[v].y));
      ki[v] = make_float2(gg[v].x * gi[v].x * (1.f - gi[v].x), gg[v].y * gi[v].y * (1.f - gi[v].y));
      kf[v] = make_float2(cp[v].x * gf[v].x * (1.f - gf[v].x), cp[v].y * gf[v].y * (1.f - gf[v].y));
      kg[v] = make_float2(gi[v].x * (1.f - gg[v].x * gg[v].x), gi[v].y * (1.f - gg[v].y * gg[v].y));
      fgate[v] = gf[v];
    }
    const float inj = tk_prev >= 0 ? p.dh_take[(size_t)tk_prev * H + unit] : 0.f;
    tk_prev = t > 1 ? p.take[(size_t)(sb + myb) * p.stride + t - 2] : -1;
    const long long k1 = prof ? clock64() : 0;
    if (it == 0) {                                     // the recurrence starts with the gradient injected at the last position
#pragma unroll
      for (int v = 0; v < NB; ++v) {
        dh[v] = make_float2(0.f, 0.f);
        const int tk = p.take[(size_t)(sb + v) * p.stride + p.T - 1];
        if (tk >= 0) dh[v] = *reinterpret_cast<const float2*>(p.dh_take + (size_t)tk * H + pu);
      }
    } else {
      unsigned pending = (1u << NB) - 1u, spins = 0;   // rounds: all missing words are re-read together
      while (true) {
#pragma unroll
        for (int v = 0; v < NB; ++v)
          if ((pending >> v & 1u) && (unsigned)(pa[v] >> 32) == (unsigned)it && (unsigned)(pb[v] >> 32) == (unsigned)it)
            pending &= ~(1u << v);
        if (pending == 0) break;
        if (++spins >= SPIN_LIMIT || ((spins & 1023u) == 0 && *(volatile int*)p.abort_flag != 0)) { ok = false; break; }
#pragma unroll
        for (int v = 0; v < NB; ++v)
          if (pending >> v & 1u) ld_tagged2(src + (size_t)v * H, pa[v], pb[v]);
      }
#pragma unroll
      for (int v = 0; v < NB; ++v) dh[v] = make_float2(__uint_as_float((unsigned)pa[v]), __uint_as_float((unsigned)pb[v]));
    }
    const long long k2 = prof ? clock64() : 0;
    if (t > 0) {                                       // the next step's stash rows
#pragma unroll
      for (int v = 0; v < NB; ++v) load_step(sb + v, t - 1, gi[v], gf[v], gg[v], go[v], cc[v], cp[v]);
    }
#pragma unroll
    for (int v = 0; v < NB; ++v) {
      const float dctx = dc[v].x + dh[v].x * kc[v].x, dcty = dc[v].y + dh[v].y * kc[v].y;
      dc[v] = make_float2(dctx * fgate[v].x, dcty * fgate[v].y);
      const float2 d_i = make_float2(dctx * ki[v].x, dcty * ki[v].y), d_f = make_float2(dctx * kf[v].x, dcty * kf[v].y);
      const float2 d_g = make_float2(dctx * kg[v].x, dcty * kg[v].y), d_o = make_float2(dh[v].x * ko[v].x, dh[v].y * ko[v].y);
      float* sd = dgb + v * 4 * H + pu;
      *reinterpret_cast<float2*>(sd) = d_i;
      *reinterpret_cast<float2*>(sd + H) = d_f;
      *reinterpret_cast<float2*>(sd + 2 * H) = d_g;
      *reinterpret_cast<float2*>(sd + 3 * H) = d_o;
      if (owner) {
        float* out = p.dgates + ((size_t)(sb + v) * p.stride + t) * 4 * H + pu;
        *reinterpret_cast<float2*>(out) = d_i;
        *reinterpret_cast<float2*>(out + H) = d_f;
        *reinterpret_cast<float2*>(out + 2 * H) = d_g;
        *reinterpret_cast<float2*>(out + 3 * H) = d_o;
      }
    }
    const long long k3 = prof ? clock64() : 0;
    if (__syncthreads_or(!ok)) {
      if (threadIdx.x == 0) atomicExch(p.abort_flag, 1);
      return;
    }
    const long long k4 = prof ? clock64() : 0;
    long long k5 = k4;
    if (t > 0) {
      float part[NB * UNITS];
#pragma unroll
      for (int v = 0; v < NB; ++v) {
        const float4 d0 = *reinterpret_cast<const float4*>(&dgb[v * 4 * H + 256 * warp + 8 * lane]);
        const float4 d1 = *reinterpret_cast<const float4*>(&dgb[v * 4 * H + 256 * warp + 8 * lane + 4]);
#pragma unroll
        for (int i = 0; i < UNITS; ++i) {
          float a = wl[i][0] * d0.x;
          a = fmaf(wl[i][1], d0.y, a); a = fmaf(wl[i][2], d0.z, a); a = fmaf(wl[i][3], d0.w, a);
          a = fmaf(wl[i][4], d1.x, a); a = fmaf(wl[i][5], d1.y, a); a = fmaf(wl[i][6], d1.z, a); a = fmaf(wl[i][7], d1.w, a);
          part[v * UNITS + i] = a;
        }
      }
      constexpr int R = NB * UNITS;                     // 8, 16 or 32 values: lane l ends with element l >> (5 - log2 R)
      const float ps = reduce_transposed<R>(part, lane);
      if ((lane & (32 / R - 1)) == 0) sh_part[warp][lane / (32 / R)] = ps;
      k5 = prof ? clock64() : 0;
      __syncthreads();
      if (lane < R) {
        float r = sh_part[lane & 7][(lane >> 3) * UNITS + warp];   // lane 8v + w': warp w' partial of (shard v, unit `warp`)
        r += __shfl_xor_sync((unsigned)((1ull << R) - 1), r, 1);
        r += __shfl_xor_sync((unsigned)((1ull << R) - 1), r, 2);
        r += __shfl_xor_sync((unsigned)((1ull << R) - 1), r, 4);
        if ((lane & 7) == 0) st_tagged(p.xchg + ((size_t)(it & 1) * p.shards + sb + (lane >> 3)) * H + unit, r + inj, (unsigned)(it + 1));
      }
    }
    if constexpr (PROF) {
      if (prof) {
        const long long k6 = clock64();
        pr[0] += k1 - k0; pr[1] += k2 - k1; pr[2] += k3 - k2; pr[3] += k4 - k3; pr[4] += k5 - k4; pr[5] += k6 - k5;
      }
    }
  }
  if constexpr (PROF) {
    if (prof) {
#pragma unroll
      for (int i = 0; i < 6; ++i) p.prof[i] = pr[i];
      p.prof[6] = p.T;
    }
  }
}

struct ChainGruBwdArgs {
  int T;
  const float* w_hh;          // [3H][H]
  const float* stash_gates;   // [T][4H]: r, z, n, a_nh = W_hn h_{t-1} + b_hn
  const float* stash_h;       // [(T+1)][H]; row t = h_{t-1}
  const int* take;            // [T]
  const float* dh_take;       // [rows][H]
  float* dgh;                 // [T][3H] hidden-side pre-activation gradients (da_r, da_z, da_nh): feeds dW_hh, db_hn
  float* dgx;                 // [T][3H] input-side gradients (da_r, da_z, da_n): feeds the gate table, W_ih, E, b_ih
  unsigned long long* xchg;   // [2][H]
  int* abort_flag;
  const float* dh_init;       // [H] or null
  float* dh0_out;             // [H] or null
};

// BPTT through the reward GRU chain (the reference trains it in train_reward_network, trainers.py:260-309; the
// A2C step keeps it frozen).  h_t = (1-z) n + z h_{t-1}, n = tanh(x_n + r a_nh):
//   da_n = dh (1-z)(1-n^2), da_nh = da_n r, da_r = da_n a_nh r(1-r), da_z = dh (h_{t-1} - n) z(1-z),
//   dh_{t-1} = dh z + W_hh^T (da_r, da_z, da_nh).
// Same scheme as chain_lstm_bwd_kernel: dh_t crosses CTAs as tagged words, every CTA rebuilds all 1536 gate
// gradients, the contraction over them is split across the warps (192 each, 6 per lane).
__global__ void __launch_bounds__(THREADS, 1) chain_gru_bwd_kernel(ChainGruBwdArgs p) {
  __shared__ __align__(16) float sh_dg[2][3 * H];
  __shared__ float sh_direct[2][H];
  __shared__ float sh_part[UNITS][UNITS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cta = blockIdx.x;
  const int unit = cta * UNITS + warp;
  const int pu = 2 * threadIdx.x;
  const bool owner = (pu >= cta * UNITS) && (pu < cta * UNITS + UNITS);

  float wl[UNITS][6];                                  // wl[i][k] = W_hh[192 warp + 6 lane + k][8 cta + i]
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const float* src = p.w_hh + (size_t)(192 * warp + 6 * lane + k) * H + cta * UNITS;
    const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
    wl[0][k] = x0.x; wl[1][k] = x0.y; wl[2][k] = x0.z; wl[3][k] = x0.w;
    wl[4][k] = x1.x; wl[5][k] = x1.y; wl[6][k] = x1.z; wl[7][k] = x1.w;
  }
  auto load_step = [&](int t, float2& r, float2& z, float2& n, float2& a, float2& hp) {
    const float* ga = p.stash_gates + (size_t)t * 4 * H + pu;
    r = *reinterpret_cast<const float2*>(ga);
    z = *reinterpret_cast<const float2*>(ga + H);
    n = *reinterpret_cast<const float2*>(ga + 2 * H);
    a = *reinterpret_cast<const float2*>(ga + 3 * H);
    hp = *reinterpret_cast<const float2*>(p.stash_h + (size_t)t * H + pu);
  };
  float2 r, z, n, a, hp;
  load_step(p.T - 1, r, z, n, a, hp);
  float2 dh = make_float2(0.f, 0.f);
  {
    const int tk = p.take[p.T - 1];
    if (tk >= 0) dh = *reinterpret_cast<const float2*>(p.dh_take + (size_t)tk * H + pu);
    if (p.dh_init) { dh.x += p.dh_init[pu]; dh.y += p.dh_init[pu + 1]; }
  }
  int tk_prev = p.T > 1 ? p.take[p.T - 2] : -1;

  for (int it = 0; it < p.T; ++it) {
    const int t = p.T - 1 - it;
    const int buf = it & 1;
    bool ok = true;
    unsigned long long wa = 0, wb = 0;
    const unsigned long long* src = p.xchg + (size_t)((it - 1) & 1) * H + pu;
    if (it > 0) ld_tagged2(src, wa, wb);
    const float knx = (1.f - z.x) * (1.f - n.x * n.x), kny = (1.f - z.y) * (1.f - n.y * n.y);
    const float khx = knx * r.x, khy = kny * r.y;
    const float krx = knx * a.x * r.x * (1.f - r.x), kry = kny * a.y * r.y * (1.f - r.y);
    const float kzx = (hp.x - n.x) * z.x * (1.f - z.x), kzy = (hp.y - n.y) * z.y * (1.f - z.y);
    const float2 zz = z;
    const float inj = tk_prev >= 0 ? p.dh_take[(size_t)tk_prev * H + unit] : 0.f;
    if (t > 0) load_step(t - 1, r, z, n, a, hp);
    tk_prev = t > 1 ? p.take[t - 2] : -1;
    if (it > 0) {
      unsigned spins = 0;
      while (!((unsigned)(wa >> 32) == (unsigned)it && (unsigned)(wb >> 32) == (unsigned)it)) {
        if (++spins >= SPIN_LIMIT || ((spins & 1023u) == 0 && *(volatile int*)p.abort_flag != 0)) { ok = false; break; }
        ld_tagged2(src, wa, wb);
      }
      dh = make_float2(__uint_as_float((unsigned)wa), __uint_as_float((unsigned)wb));
    }
    const float2 d_r = make_float2(dh.x * krx, dh.y * kry), d_z = make_float2(dh.x * kzx, dh.y * kzy);
    const float2 d_h = make_float2(dh.x * khx, dh.y * khy), d_n = make_float2(dh.x * knx, dh.y * kny);
    *reinterpret_cast<float2*>(&sh_dg[buf][pu]) = d_r;
    *reinterpret_cast<float2*>(&sh_dg[buf][H + pu]) = d_z;
    *reinterpret_cast<float2*>(&sh_dg[buf][2 * H + pu]) = d_h;
    *reinterpret_cast<float2*>(&sh_direct[buf][pu]) = make_float2(dh.x * zz.x, dh.y * zz.y);
    if (owner) {
      float* oh = p.dgh + (size_t)t * 3 * H + pu;
      float* ox = p.dgx + (size_t)t * 3 * H + pu;
      *reinterpret_cast<float2*>(oh) = d_r;          *reinterpret_cast<float2*>(ox) = d_r;
      *reinterpret_cast<float2*>(oh + H) = d_z;      *reinterpret_cast<float2*>(ox + H) = d_z;
      *reinterpret_cast<float2*>(oh + 2 * H) = d_h;  *reinterpret_cast<float2*>(ox + 2 * H) = d_n;
    }
    if (__syncthreads_or(!ok)) {
      if (threadIdx.x == 0) atomicExch(p.abort_flag, 1);
      return;
    }
    if (t > 0 || p.dh0_out) {
      const float2 q0 = *reinterpret_cast<const float2*>(&sh_dg[buf][192 * warp + 6 * lane]);
      const float2 q1 = *reinterpret_cast<const float2*>(&sh_dg[buf][192 * warp + 6 * lane + 2]);
      const float2 q2 = *reinterpret_cast<const float2*>(&sh_dg[buf][192 * warp + 6 * lane + 4]);
      float part[UNITS];
#pragma unroll
      for (int i = 0; i < UNITS; ++i) {
        float acc = wl[i][0] * q0.x;
        acc = fmaf(wl[i][1], q0.y, acc); acc = fmaf(wl[i][2], q1.x, acc); acc = fmaf(wl[i][3], q1.y, acc);
        acc = fmaf(wl[i][4], q2.x, acc); acc = fmaf(wl[i][5], q2.y, acc);
        part[i] = acc;
      }
      const float ps = reduce_transposed<UNITS>(part, lane);
      if ((lane & 3) == 0) sh_part[warp][lane >> 2] = ps;
      __syncthreads();
      if (lane < UNITS) {
        float rec = sh_part[lane][warp];
        rec += __shfl_xor_sync(0xffu, rec, 1);
        rec += __shfl_xor_sync(0xffu, rec, 2);
        rec += __shfl_xor_sync(0xffu, rec, 4);
        if (lane == 0) {
          rec += sh_direct[buf][unit];
          if (t > 0) st_tagged(p.xchg + (size_t)buf * H + unit, rec + inj, (unsigned)(it + 1));
          else p.dh0_out[unit] = rec;
        }
      }
    }
  }
}

int coop_launch(const void* fn, int grid, void** args, cudaStream_t st) {
  int dev = 0, coop = 0, sms = 0, per_sm = 0;
  ICRL_CUDA(cudaGetDevice(&dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  ICRL_REQUIRE(coop, "device lacks cooperative launch");
  ICRL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ICRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, THREADS, 0));
  ICRL_REQUIRE(per_sm * sms >= grid, "chain grid is not co-resident on this device");
  ICRL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(THREADS), args, 0, st));
  return ICRL_OK;
}

}  // namespace

int icrl_chain_ctas() { return CHAIN_CTAS; }

static ChainFwdArgs make_fwd(const int* stream, int T, const float* table, const float* w_hh, const float* b_hn,
                             const float* h0, const float* c0, float* stash_h, float* stash_c, float* stash_gates,
                             float* h_out, float* c_out, unsigned long long* xchg, int* abort_flag) {
  ChainFwdArgs a;
  a.stream = stream; a.T = T; a.table = table; a.w_hh = w_hh; a.b_hn = b_hn; a.h0 = h0; a.c0 = c0;
  a.stash_h = stash_h; a.stash_c = stash_c; a.stash_gates = stash_gates; a.h_out = h_out; a.c_out = c_out;
  a.xchg = xchg; a.abort_flag = abort_flag;
  return a;
}

// sync_state layout (device, caller-owned, >= icrl_chain_sync_bytes(), zeroed once by the caller):
// [0,64) sticky abort word (+pad; cleared only by icrl_chain_check), then exchange buffers
// (re-zeroed before every launch): lstm fwd, gru fwd, lstm bwd, 2 * NB_MAX * H 64-bit words each.
size_t icrl_chain_sync_bytes_impl() { return 64 + sizeof(unsigned long long) * 3 * (2 * NB_MAX * H); }

static int* sync_abort(void* s) { return reinterpret_cast<int*>(s); }
static unsigned long long* sync_xchg(void* s, int which) {
  unsigned long long* base = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(s) + 64);
  return base + (size_t)which * (2 * NB_MAX * H);
}

int icrl_chain_lstm_fwd_impl(cudaStream_t st, const int* stream, int T, const float* table, const float* w_hh,
                             const float* h0, const float* c0, float* stash_h, float* stash_c, float* stash_gates,
                             float* h_out, float* c_out, void* sync_state) {
  ICRL_REQUIRE(T > 0 && stash_h, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainFwdArgs a = make_fwd(stream, T, table, w_hh, nullptr, h0, c0, stash_h, stash_c, stash_gates, h_out, c_out,
                            sync_xchg(sync_state, 0), sync_abort(sync_state));
  void* args[] = {&a};
  return coop_launch((const void*)chain_lstm_fwd_kernel, CHAIN_CTAS, args, st);
}

int icrl_chain_gru_fwd_impl(cudaStream_t st, const int* stream, int T, const float* table, const float* w_hh,
                            const float* b_hn, const float* h0, float* stash_h, float* h_out, void* sync_state,
                            float* stash_gates) {
  ICRL_REQUIRE(T > 0 && stash_h, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainFwdArgs a = make_fwd(stream, T, table, w_hh, b_hn, h0, nullptr, stash_h, nullptr, stash_gates, h_out, nullptr,
                            sync_xchg(sync_state, 1), sync_abort(sync_state));
  void* args[] = {&a};
  return coop_launch((const void*)chain_gru_fwd_kernel, CHAIN_CTAS, args, st);
}

int icrl_chains_fwd_fused_impl(cudaStream_t st, const int* v_stream, int v_T, const float* v_table,
                               const float* v_w_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                               const int* r_stream, int r_T, const float* r_table, const float* r_w_hh,
                               const float* r_b_hn, float* r_stash_h, void* sync_state) {
  ICRL_REQUIRE(v_T > 0 && r_T > 0, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainFwdArgs a = make_fwd(v_stream, v_T, v_table, v_w_hh, nullptr, nullptr, nullptr, v_stash_h, v_stash_c,
                            v_stash_gates, nullptr, nullptr, sync_xchg(sync_state, 0), sync_abort(sync_state));
  ChainFwdArgs b = make_fwd(r_stream, r_T, r_table, r_w_hh, r_b_hn, nullptr, nullptr, r_stash_h, nullptr, nullptr,
                            nullptr, nullptr, sync_xchg(sync_state, 1), sync_abort(sync_state));
  void* args[] = {&a, &b};
  return coop_launch((const void*)chains_fwd_fused_kernel, 2 * CHAIN_CTAS, args, st);
}

int icrl_chain_lstm_bwd_impl(cudaStream_t st, int T, const float* w_hh, const float* stash_gates, const float* stash_c,
                             const int* take, const float* dh_take, float* dgates, void* sync_state, const float* dh_init,
                             const float* dc_init, float* dh0_out, float* dc0_out) {
  ICRL_REQUIRE(T > 0, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainBwdArgs a;
  a.T = T; a.w_hh = w_hh; a.stash_gates = stash_gates; a.stash_c = stash_c; a.take = take; a.dh_take = dh_take;
  a.dgates = dgates; a.xchg = sync_xchg(sync_state, 2); a.abort_flag = sync_abort(sync_state);
  a.dh_init = dh_init; a.dc_init = dc_init; a.dh0_out = dh0_out; a.dc0_out = dc0_out;
  void* args[] = {&a};
  return coop_launch((const void*)chain_lstm_bwd_kernel, CHAIN_CTAS, args, st);
}

int icrl_chain_gru_bwd_impl(cudaStream_t st, int T, const float* w_hh, const float* stash_gates, const float* stash_h,
                            const int* take, const float* dh_take, float* dgh, float* dgx, void* sync_state,
                            const float* dh_init, float* dh0_out) {
  ICRL_REQUIRE(T > 0, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainGruBwdArgs a;
  a.T = T; a.w_hh = w_hh; a.stash_gates = stash_gates; a.stash_h = stash_h; a.take = take; a.dh_take = dh_take;
  a.dgh = dgh; a.dgx = dgx; a.xchg = sync_xchg(sync_state, 2); a.abort_flag = sync_abort(sync_state);
  a.dh_init = dh_init; a.dh0_out = dh0_out;
  void* args[] = {&a};
  return coop_launch((const void*)chain_gru_bwd_kernel, CHAIN_CTAS, args, st);
}

// Reads the abort word (synchronises the stream).  Returns ICRL_ERR_WATCHDOG if a chain gave up.
int icrl_chain_check_impl(cudaStream_t st, void* sync_state) {
  int flag = 0;
  ICRL_CUDA(cudaMemcpyAsync(&flag, sync_state, sizeof(int), cudaMemcpyDeviceToHost, st));
  ICRL_CUDA(cudaStreamSynchronize(st));
  if (flag != 0) {
    ICRL_CUDA(cudaMemsetAsync(sync_state, 0, 64, st));
    icrl_set_error("serial-chain watchdog tripped: a CTA waited > %u polls for its peers", SPIN_LIMIT);
    return ICRL_ERR_WATCHDOG;
  }
  return ICRL_OK;
}


// ---- batched launchers (nb chain shards; see the kernels above)
static long long* g_chain_prof = nullptr;      // icrl_chain_set_profile: 16 device int64 (LSTM, GRU forward shard kernels [0..7]; backward [8..14])
void icrl_chain_set_profile_impl(long long* buf) { g_chain_prof = buf; }
static int coop_launch_smem(const void* fn, int grid, void** args, size_t smem, cudaStream_t st) {
  int dev = 0, sms = 0, per_sm = 0;
  ICRL_CUDA(cudaGetDevice(&dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ICRL_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ICRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, THREADS, smem));
  ICRL_REQUIRE(per_sm * sms >= grid, "chain grid is not co-resident on this device");
  ICRL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(THREADS), args, smem, st));
  return ICRL_OK;
}

// `nb` = 2, 4 or 8 independent row shards, v_T / r_T steps each, arrays of shard k at row k * (T + 1).
int icrl_chains_fwd_fused_batched_impl(cudaStream_t st, int nb, const int* v_stream, int v_T, const float* v_table,
                                       const float* v_w_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                                       const int* r_stream, int r_T, const float* r_table, const float* r_w_hh,
                                       const float* r_b_hn, float* r_stash_h, void* sync_state) {
  ICRL_REQUIRE(nb == 2 || nb == 4 || nb == 8, "chain shards per launch must be 2, 4 or 8");
  ICRL_REQUIRE(v_T > 0 && r_T > 0, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  ChainFwdBatchArgs a, b;
  a.stream = v_stream; a.T = v_T; a.stride = (long long)v_T + 1; a.table = v_table; a.w_hh = v_w_hh; a.b_hn = nullptr;
  a.stash_h = v_stash_h; a.stash_c = v_stash_c; a.stash_gates = v_stash_gates; a.xchg = sync_xchg(sync_state, 0);
  a.abort_flag = sync_abort(sync_state); a.prof = g_chain_prof;
  b.stream = r_stream; b.T = r_T; b.stride = (long long)r_T + 1; b.table = r_table; b.w_hh = r_w_hh; b.b_hn = r_b_hn;
  b.stash_h = r_stash_h; b.stash_c = nullptr; b.stash_gates = nullptr; b.xchg = sync_xchg(sync_state, 1);
  b.abort_flag = sync_abort(sync_state); b.prof = g_chain_prof ? g_chain_prof + 4 : nullptr;
  const size_t smem = (size_t)2 * nb * H * sizeof(float);      // [2][shards][H]
  void* args[] = {&a, &b};
  const void* fn = nb == 2 ? (const void*)chains_fwd_fused_batched_kernel<2>
                 : nb == 4 ? (const void*)chains_fwd_fused_batched_kernel<4>
                           : (const void*)chains_fwd_fused_batched_kernel<8>;
  return coop_launch_smem(fn, 2 * CHAIN_CTAS, args, smem, st);
}

// shards = 2, 4 or 8 total; they are split over two 64-CTA groups (1, 2 or 4 shards per group).
int icrl_chain_lstm_bwd_batched_impl(cudaStream_t st, int shards, int T, const float* w_hh, const float* stash_gates,
                                     const float* stash_c, const int* take, const float* dh_take, float* dgates,
                                     void* sync_state) {
  ICRL_REQUIRE(shards == 2 || shards == 4 || shards == 8, "chain shards must be 2, 4 or 8");
  ICRL_REQUIRE(T > 0, "empty chain");
  ICRL_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(sync_state) + 64, 0, icrl_chain_sync_bytes_impl() - 64, st));
  const long long stride = (long long)T + 1;
  for (int k = 0; k < shards; ++k)                      // padding row T of every shard (feeds the weight-gradient GEMM)
    ICRL_CUDA(cudaMemsetAsync(dgates + ((size_t)k * stride + T) * 4 * H, 0, 4 * H * sizeof(float), st));
  ChainBwdBatchArgs a;
  a.T = T; a.stride = stride; a.w_hh = w_hh; a.stash_gates = stash_gates; a.stash_c = stash_c; a.take = take;
  a.dh_take = dh_take; a.dgates = dgates; a.xchg = sync_xchg(sync_state, 2); a.shards = shards;
  a.abort_flag = sync_abort(sync_state);
  a.prof = g_chain_prof ? g_chain_prof + 8 : nullptr;
  void* args[] = {&a};
  // two 64-CTA groups of shards / 2 shards each (8 shards: 113.8 ms per launch at B = 2048, measured); a kernel step costs
  // about 1.0 us of fixed work (poll round trip, two barriers, butterfly, publish) plus 0.32 us per shard
  const int nb = shards / 2;
  const void* fn = shards == 2 ? (const void*)chain_lstm_bwd_batched_kernel<1, false>
                 : shards == 4 ? (const void*)chain_lstm_bwd_batched_kernel<2, false>
                 : a.prof      ? (const void*)chain_lstm_bwd_batched_kernel<4, true>
                               : (const void*)chain_lstm_bwd_batched_kernel<4, false>;
  const size_t smem = (size_t)2 * nb * 4 * H * sizeof(float);
  return coop_launch_smem(fn, 2 * CHAIN_CTAS, args, smem, st);
}
