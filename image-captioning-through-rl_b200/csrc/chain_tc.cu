// Chain pieces on tcgen05 (sm_100a): the value-LSTM / reward-GRU batch-as-time recurrences of the reference
// (models.py:130-135, 223-228: seq = B, batch = 1, hidden state carried across calls; trainers.py:479 for the backward)
// advanced as HUNDREDS of lockstep pieces of the ONE carried-state chain.
//
// Why this is a GEMM.  chain.cu walks the chain position by position (latency floor ~1.3 us per position) or as <= 32
// lockstep pieces on CUDA cores.  With P pieces in lockstep, one kernel step is  H_prev [P x 512] . W_hh^T [512 x G]
// (G = 2048 LSTM, 1536 GRU) followed by the pointwise cell update -- exactly the shape decode.cu already runs on
// tcgen05 with the policy's batch rows in the M dimension.  Here the M rows are PIECES of one chain: piece k covers
// stream positions [k*seg, (k+1)*seg + warm); pieces k >= 1 start from zero state, discard their first `warm` positions
// (nothing is stored for them) and by then carry the single chain's state to float rounding because the gated
// recurrence contracts state differences.  That is CHECKED on every launch, never assumed: the state each piece
// reaches at the end of (and half-way through) its warm-up is compared with the state the preceding pieces stored at
// the same positions (chain_tc_check_*), and the engine re-runs with a longer warm-up when the check fails.
//
// Decomposition (forward).  A cluster of 8 CTAs owns 128 pieces for the whole launch and never talks to another
// cluster.  CTA r owns hidden units [64r, 64r+64): NG*64 gate columns (W_hh rows permuted at pack time), i.e. the
// N-slice of the step GEMM; K = 512.  Per step: TMA ring (4 stages of 32-wide K blocks; the A tile = fp16 split of
// h_{t-1} of the 128 pieces is fetched in 16-row slices and multicast to the whole cluster, the B tile = this CTA's
// W_hh slice comes from L2) -> tcgen05.mma (M=128, N=NG*64; three products hi*hi -> main accumulator, hi*lo' + lo'*hi
// -> correction accumulator, f32 in tensor memory: fp32-grade, see decode.cu) -> epilogue warps: gate-table rows of
// the consumed tokens and the carried c (LSTM) / h (GRU) gathered into a swizzled shared-memory tile with cp.async,
// cell update thread-per-row, coalesced stores of the backward stash (live positions only), of the carried state and
// of the fp16 split of h_t for the next step -> cluster barrier.
//
// Backward (LSTM).  Mirrored: piece k walks positions (k+1)*seg + warm - 1 down to k*seg, pieces other than the last
// start with dh = dc = 0 and discard the gate gradients of their first `warm` steps (injections at take positions inside
// the window are applied).  Step GEMM: dh_{t-1} [P x 512] = dgates_t [P x 2048] . W_hh [2048 x 512], cut over the
// cluster as 2 K halves x 4 column quarters (see BwdCfg; A = fp16 split of the gate gradients of all 8 CTAs, exchanged
// through L2 and TMA-multicast to the 4 CTAs of a K half; B = W_hh^T slice; partial sums swapped through DSMEM); each
// CTA owns the cell arithmetic of 64 hidden units.  Gate gradients span many orders of magnitude, so the exchanged copy is
// scaled by a power of two derived from max |dL/dh_take| (fp16 keeps 22 bits down to 2^-18 of that maximum; overflow
// is detected and reported).  The gate gradients of live positions go to the parameter-gradient contractions as that
// same scaled split, in planes [2][rows][2048] with the columns of icrl_gate_pair_col (the policy's BPTT writes fp32).
#include "tc_ptx.cuh"
#include "internal.h"

using namespace icrl_tc;

namespace {

constexpr int H = ICRL_H;
constexpr int CL = 8;                       // CTAs per cluster
constexpr int BM = 128;                     // pieces per cluster (MMA M)
constexpr int UN = H / CL;                  // 64 hidden units per CTA
constexpr int BK = 32, UMMA_K = 16;         // 64-byte K rows (SWIZZLE_64B)
constexpr int A_TILE = BM * BK * 2;         // 8 KB
constexpr int A_SLICE_ROWS = BM / CL;       // 16 rows fetched (and multicast) per CTA
constexpr int A_SLICE = A_SLICE_ROWS * BK * 2;
constexpr int EPI_WARPS = 8, EPI_WARP0 = 4;
constexpr int THREADS = 32 * (EPI_WARP0 + EPI_WARPS);      // 384
constexpr float LO_INV = 1.f / 2048.f;
constexpr int CORR = 256;                   // forward: TMEM column of the correction accumulator

// Publishing the per-step exchange (fp16 split of h / of the gate gradients, written with ordinary global stores) to the
// TMA loads of the other CTAs of the cluster: fence.proxy.async (generic -> async proxy) on both sides of a cluster
// barrier whose arrive is a RELEASE and whose wait is an ACQUIRE at cluster scope.  An extra __threadfence() (gpu-scope
// fence, as decode.cu issues) costs ~2.5 K cycles per step and is not required by the memory model; build with
// -DICRL_TC_GPU_FENCE=1 to restore it.
#ifndef ICRL_TC_GPU_FENCE
#define ICRL_TC_GPU_FENCE 0
#endif
__device__ __forceinline__ void publish_exchange() {
#if ICRL_TC_GPU_FENCE
  __threadfence();
#endif
  fence_proxy_async();
  __syncwarp();
  cluster_arrive();
}

// ------------------------------------------------------------------------------------------------ forward
constexpr int F_STAGES = 4, F_KB = H / BK;  // 16 K blocks per step
template <int NG> struct FwdCfg {
  static constexpr int GN = NG * UN;                        // 256 / 192 gate columns per CTA
  static constexpr int B_TILE = GN * BK * 2;                // 16 / 12 KB
  static constexpr int STAGE = 2 * A_TILE + 2 * B_TILE;     // 48 / 40 KB
  static constexpr int NARR = NG == 4 ? 6 : 4;              // staging arrays of [32 rows][32 units] f32 per epilogue warp
  static constexpr int GST_WARP = NARR * 4096;
  static constexpr int SMEM = F_STAGES * STAGE + 256 + 1024;
  static_assert(EPI_WARPS * GST_WARP <= F_STAGES * STAGE, "epilogue staging lives inside the (idle) TMA ring");
};

struct FwdArgs {
  int P, Ppad, steps, warm, cp_half;
  long long seg;
  const int* stream;       // [P*seg + warm]
  const float* table;      // [V][NG*512]
  const float* b_hn;       // GRU: [512]
  float* stash_h;          // [(P*seg + warm + 1)][512]; row 0 = zeros (set by the launcher)
  float* stash_c;          // LSTM
  float* stash_g;          // LSTM: [P*seg + warm][2048] activated i,f,g,o (nullable)
  float* state;            // [Ppad][512] carried c (LSTM) / h (GRU), zeroed by the launcher
  __half* hparts;          // [2 buffers][2 parts][Ppad][512]; buffer 0 zeroed by the launcher
  float* wstate;           // [2 checkpoints][P][2][512]: (h, c) of piece k after step cp_half (0) / warm-1 (1)
  float main_gain;         // 1 + compensation of the tensor core's truncating accumulation (see g_tc_bias)
  int tma_store;           // the stash of the live positions leaves through TMA tensor stores (maps in FwdMaps)
  long long* prof;         // optional: cycle sums of CTA 0's first epilogue warp {acc wait, gather, cell, store, barrier}, steps
};

// fp32 stash arrays as 3-D tensors {column, step j of a piece, piece}: row (k * seg + j [+ 1]) of the array, i.e. strides
// (4 B, row, seg rows).  The epilogue's staging tiles ([32 pieces][32 units] f32, 16-byte chunk c of row r at
// r*128 + ((c ^ (r & 7)) << 4)) ARE the 128B-swizzled box {32, 1, 32} of these maps, so a tile leaves with one instruction.
struct FwdMaps {
  CUtensorMap h, w;        // operands: fp16 split of h (A, multicast slices), packed W_hh (B)
  CUtensorMap sg, sc, sh;  // stores: stash_g [..][2048], stash_c / stash_h [..][512] (both based at row 1)
};

template <int NG>
__device__ __forceinline__ void chain_tc_fwd_body(const FwdMaps& maps, const FwdArgs& p, const int cluster) {
  const CUtensorMap& map_h = maps.h;
  const CUtensorMap& map_w = maps.w;
  using C = FwdCfg<NG>;
  constexpr int GN = C::GN, B_TILE = C::B_TILE, STAGE = C::STAGE, STAGES = F_STAGES;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + STAGES * STAGE);
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * STAGES + 2);
  const unsigned bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[STAGES]);
  const unsigned bar_acc_full = smem_u32(&bars[2 * STAGES]), bar_acc_empty = smem_u32(&bars[2 * STAGES + 1]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned rank = cluster_rank();
  const int m0 = cluster * BM;
  const int P = p.P, Ppad = p.Ppad, steps = p.steps;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, CL); }
    mbar_init(bar_acc_full, 1);
    mbar_init(bar_acc_empty, EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_h) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  cluster_arrive();                      // every CTA's mbarriers are initialised before anyone multicasts into them
  cluster_wait();

  if (warp == 2 || warp == 3) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    for (int j = 0; j < steps; ++j) { cluster_arrive(); cluster_wait(); }
  } else if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    unsigned it = 0;
    for (int j = 0; j < steps; ++j) {
      if (lane == 0) {
        const int arow = ((j & 1) * 2) * Ppad + m0;
        for (int kb = 0; kb < F_KB; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_empty + 8 * s, ((it / STAGES) & 1u) ^ 1u);
          const unsigned full = bar_full + 8 * s;
          mbar_expect_tx(full, 2 * A_TILE + 2 * B_TILE);
          const unsigned base = smem_u32(smem + s * STAGE);
          tma_load_2d_mcast(base + rank * A_SLICE, &map_h, kb * BK, arow + (int)rank * A_SLICE_ROWS, full, 0xFF);
          tma_load_2d_mcast(base + A_TILE + rank * A_SLICE, &map_h, kb * BK, arow + Ppad + (int)rank * A_SLICE_ROWS, full, 0xFF);
          tma_load_3d(base + 2 * A_TILE, &map_w, kb * BK, (int)rank * GN, 0, full);      // hi at +0, lo' at +B_TILE
        }
      }
      __syncwarp();
      cluster_arrive();
      cluster_wait();                    // h_j of all 8 CTAs is in global memory
      if (lane == 0) fence_proxy_async();
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (warp-uniform loops, elect.sync)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    unsigned it = 0;
    for (int j = 0; j < steps; ++j) {
      if (j > 0) mbar_wait(bar_acc_empty, (unsigned)(j - 1) & 1u);        // previous epilogue drained TMEM
      tc_fence_after();
      for (int kb = 0; kb < F_KB; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(bar_full + 8 * s, (it / STAGES) & 1u);
        tc_fence_after();
        const unsigned base = smem_u32(smem + s * STAGE);
        const unsigned long long dA0 = smem_desc_sw64(base), dA1 = smem_desc_sw64(base + A_TILE);
        const unsigned long long dB0 = smem_desc_sw64(base + 2 * A_TILE), dB1 = smem_desc_sw64(base + 2 * A_TILE + B_TILE);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {                          // +2 = 32 bytes (16 fp16 along K) in 16-byte units
            tc_mma(tmem_base, dA0 + 2 * k, dB0 + 2 * k, idesc_f16_m128(GN), (kb | k) != 0);          // hi  * hi  -> main
            tc_mma(tmem_base + CORR, dA0 + 2 * k, dB1 + 2 * k, idesc_f16_m128(GN), (kb | k) != 0);   // hi  * lo' -> correction
            tc_mma(tmem_base + CORR, dA1 + 2 * k, dB0 + 2 * k, idesc_f16_m128(GN), 1u);              // lo' * hi  -> correction
          }
          tc_commit_mcast(bar_empty + 8 * s, 0xFF);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(bar_acc_full);
      __syncwarp();
      cluster_arrive();
      cluster_wait();
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int ew = warp - EPI_WARP0;
    const int q = warp & 3;                    // TMEM lane quarter this warp may read
    const int ch = ew >> 2;                    // unit half
    const int k_own = m0 + 32 * q + lane;      // this thread's piece (row of the cluster tile)
    const bool valid = k_own < P;
    const unsigned tq = tmem_base + ((unsigned)(32 * q) << 16);
    unsigned char* gst = smem + ew * C::GST_WARP;
    const int ucol0 = (int)rank * UN + 32 * ch;
    const long long seg = p.seg;
    int tok = valid ? p.stream[(long long)k_own * seg] : 0;
    const float mg = p.main_gain;
    const float k0 = -mg * L2E, k1 = -LO_INV * L2E;            // accumulators -> exponent of a sigmoid gate
    // The stash of a live step already holds the state the next step carries (row pos + 1 of stash_c / stash_h), so live
    // steps skip the separate state store (32 KB of the ~32 B/clk an SM can push towards L2); not with the TMA store path,
    // whose writes travel through the async proxy.
    const bool stash_carry = !p.tma_store;
    const float* carry_stash = NG == 4 ? p.stash_c : p.stash_h;
    const bool prof = p.prof != nullptr && cluster == 0 && rank == 0 && ew == 0 && lane == 0;
    long long pr[5] = {0, 0, 0, 0, 0};

    for (int j = 0; j < steps; ++j) {
      const long long t0 = prof ? clock64() : 0;
      const int tok_n = (valid && j + 1 < steps) ? p.stream[(long long)k_own * seg + j + 1] : 0;
      mbar_wait(bar_acc_full, (unsigned)j & 1u);
      tc_fence_after();
      const long long t1 = prof ? clock64() : 0;
      // (L) gate-table rows of the consumed tokens (arrays 0..NG-1) and the carried state (array NG) -> staging,
      //     8 lanes per row; element (row, 16-byte chunk c) lives at row*128 + ((c ^ (row & 7)) << 4).
      {
        const int c4 = lane & 7;
#pragma unroll
        for (int i8 = 0; i8 < 8; ++i8) {
          const int r = i8 * 4 + (lane >> 3);
          const int tokr = __shfl_sync(0xffffffffu, tok, r);
          const int kr = m0 + 32 * q + r;
          if (kr < P) {
            const unsigned dst = smem_u32(gst) + (unsigned)(r * 128 + ((c4 ^ (r & 7)) << 4));
            const float* tsrc = p.table + (size_t)tokr * (NG * H) + ucol0 + c4 * 4;
#pragma unroll
            for (int a = 0; a < NG; ++a) cp_async16(dst + a * 4096, tsrc + a * H);
            // carried state (c of the LSTM, h of the GRU): the stash row the previous step wrote when that step was live
            // (this very thread wrote these 16 bytes), else the state array
            const bool prev_live = stash_carry && j >= 1 && (kr == 0 || j - 1 >= p.warm);
            const float* ssrc = prev_live ? carry_stash + ((size_t)kr * seg + j) * H : p.state + (size_t)kr * H;
            cp_async16(dst + NG * 4096, ssrc + ucol0 + c4 * 4);
          }
        }
        cp_async_wait_all();
        __syncwarp();
      }
      const long long t2 = prof ? clock64() : 0;
      // (C) cell update, one row per lane, in place on the staging tile
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float acc[NG][8], cor[NG][8];
#pragma unroll
        for (int g = 0; g < NG; ++g)
          tmem_ld8x2(tq + (unsigned)(g * UN + 32 * ch + 8 * c8), tq + (unsigned)(CORR + g * UN + 32 * ch + 8 * c8), acc[g], cor[g]);
        unsigned char* e0 = gst + lane * 128 + (((2 * c8) ^ (lane & 7)) << 4);
        unsigned char* e1 = gst + lane * 128 + (((2 * c8 + 1) ^ (lane & 7)) << 4);
        float tin[NG + 1][8];
#pragma unroll
        for (int a = 0; a < NG + 1; ++a) {
          const float4 u0 = *reinterpret_cast<const float4*>(e0 + a * 4096);
          const float4 u1 = *reinterpret_cast<const float4*>(e1 + a * 4096);
          tin[a][0] = u0.x; tin[a][1] = u0.y; tin[a][2] = u0.z; tin[a][3] = u0.w;
          tin[a][4] = u1.x; tin[a][5] = u1.y; tin[a][6] = u1.z; tin[a][7] = u1.w;
        }
        if constexpr (NG == 4) {
          float gi[8], gf[8], gg[8], go[8], cn[8], hn[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // sigmoid(x) = 1 / (1 + 2^(-x log2 e)), tanh(x) = 1 - 2 / (1 + 2^(2x log2 e)): the exponent of each gate comes
            // straight out of the FMAs that combine main accumulator (x bias compensation), correction accumulator and
            // gate-table entry (the log2 e factors are folded into their coefficients), the exponents are clamped where both
            // functions are saturated to the last float bit, and the four denominators share ONE reciprocal (their
            // product stays below 6e34): 7 MUFU and ~49 instructions per cell instead of 10 and 64.
            const float yi = clamp_sat(fmaf(tin[0][i], -L2E, fmaf(cor[0][i], k1, acc[0][i] * k0)));
            const float yf = clamp_sat(fmaf(tin[1][i], -L2E, fmaf(cor[1][i], k1, acc[1][i] * k0)));
            const float yg = clamp_sat(fmaf(tin[2][i], 2.f * L2E, fmaf(cor[2][i], -2.f * k1, acc[2][i] * (-2.f * k0))));
            const float yo = clamp_sat(fmaf(tin[3 % NG][i], -L2E, fmaf(cor[3 % NG][i], k1, acc[3 % NG][i] * k0)));
            const float di = 1.f + ex2_ftz(yi), df = 1.f + ex2_ftz(yf), dg = 1.f + ex2_ftz(yg), dz = 1.f + ex2_ftz(yo);
            const float pif = di * df, pgo = dg * dz;
            const float r = rcp_ftz(pif * pgo);
            const float rif = r * pgo, rgo = r * pif;            // 1 / (di df), 1 / (dg dz)
            gi[i] = rif * df;
            gf[i] = rif * di;
            gg[i] = fmaf(-2.f, rgo * dz, 1.f);
            go[i] = rgo * dg;
            cn[i] = fmaf(gf[i], tin[NG][i], gi[i] * gg[i]);
            hn[i] = go[i] * tanh_lean(cn[i]);
          }
          *reinterpret_cast<float4*>(e0) = make_float4(gi[0], gi[1], gi[2], gi[3]);
          *reinterpret_cast<float4*>(e1) = make_float4(gi[4], gi[5], gi[6], gi[7]);
          *reinterpret_cast<float4*>(e0 + 4096) = make_float4(gf[0], gf[1], gf[2], gf[3]);
          *reinterpret_cast<float4*>(e1 + 4096) = make_float4(gf[4], gf[5], gf[6], gf[7]);
          *reinterpret_cast<float4*>(e0 + 2 * 4096) = make_float4(gg[0], gg[1], gg[2], gg[3]);
          *reinterpret_cast<float4*>(e1 + 2 * 4096) = make_float4(gg[4], gg[5], gg[6], gg[7]);
          *reinterpret_cast<float4*>(e0 + 3 * 4096) = make_float4(go[0], go[1], go[2], go[3]);
          *reinterpret_cast<float4*>(e1 + 3 * 4096) = make_float4(go[4], go[5], go[6], go[7]);
          *reinterpret_cast<float4*>(e0 + 4 * 4096) = make_float4(cn[0], cn[1], cn[2], cn[3]);
          *reinterpret_cast<float4*>(e1 + 4 * 4096) = make_float4(cn[4], cn[5], cn[6], cn[7]);
          *reinterpret_cast<float4*>(e0 + (C::NARR - 1) * 4096) = make_float4(hn[0], hn[1], hn[2], hn[3]);
          *reinterpret_cast<float4*>(e1 + (C::NARR - 1) * 4096) = make_float4(hn[4], hn[5], hn[6], hn[7]);
        } else {
          // GRU (gate order r, z, n): n = tanh(x_n + r * (W_hn h + b_hn)), h' = (1 - z) n + z h   (models.py:215)
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.b_hn + ucol0 + 8 * c8));
          const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.b_hn + ucol0 + 8 * c8 + 4));
          const float bh[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          float hn[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // r, z share one reciprocal; exponents straight out of the FMAs (see the LSTM cell)
            const float yr = clamp_sat(fmaf(tin[0][i], -L2E, fmaf(cor[0][i], k1, acc[0][i] * k0)));
            const float yz = clamp_sat(fmaf(tin[1][i], -L2E, fmaf(cor[1][i], k1, acc[1][i] * k0)));
            const float dr = 1.f + ex2_ftz(yr), dzz = 1.f + ex2_ftz(yz);
            const float rr = rcp_ftz(dr * dzz);
            const float r = rr * dzz, z = rr * dr;
            const float n = tanh_lean(fmaf(r, fmaf(cor[2][i], LO_INV, acc[2][i] * mg) + bh[i], tin[2][i]));
            hn[i] = fmaf(z, tin[NG][i] - n, n);                  // (1 - z) n + z h
          }
          *reinterpret_cast<float4*>(e0 + NG * 4096) = make_float4(hn[0], hn[1], hn[2], hn[3]);
          *reinterpret_cast<float4*>(e1 + NG * 4096) = make_float4(hn[4], hn[5], hn[6], hn[7]);
        }
      }
      __syncwarp();
      const long long t3 = prof ? clock64() : 0;
      // (S) one pass over the staged results.  What the next step needs: the fp16 split of h (read by every CTA of the
      // cluster through TMA) and the carried state.  The backward stash of the live positions: from the end of the warm-up
      // on every piece is live (before that only piece 0); with the TMA path each staging tile leaves as ONE tensor store
      // (pieces past P are clipped by the map).  The joint checkpoints at the two checkpoint steps.
      const bool tma_path = p.tma_store && j >= p.warm;
      if (tma_path) {
        fence_proxy_async_smem();                // this thread's staging writes -> visible to the async proxy
        __syncwarp();
        if (lane == 0) {
          const int k0 = m0 + 32 * q;
          if constexpr (NG == 4) {
            if (p.stash_g) {
#pragma unroll
              for (int a = 0; a < 4; ++a) tma_store_3d(&maps.sg, smem_u32(gst + a * 4096), a * H + ucol0, j, k0);
            }
            tma_store_3d(&maps.sc, smem_u32(gst + 4 * 4096), ucol0, j, k0);
          }
          tma_store_3d(&maps.sh, smem_u32(gst + (C::NARR - 1) * 4096), ucol0, j, k0);
          tma_store_commit();
        }
      }
      {
        const int c4 = lane & 7;
        const bool cp_full = j == p.warm - 1, cp_half = j == p.cp_half;
#pragma unroll
        for (int i8 = 0; i8 < 8; ++i8) {
          const int r = i8 * 4 + (lane >> 3);
          const int kr = m0 + 32 * q + r;
          if (kr < P) {
            const unsigned char* e = gst + r * 128 + ((c4 ^ (r & 7)) << 4);
            const size_t pos = (size_t)kr * seg + j;
            const bool live = !tma_path && (kr == 0 || j >= p.warm);
            const bool cp = kr >= 1 && (cp_full || cp_half);
            const int uc = ucol0 + c4 * 4;
            const float4 h4 = *reinterpret_cast<const float4*>(e + (C::NARR - 1) * 4096);
            uint2 hi, lo;
            split4_f16(h4, hi, lo);
            __half* hp = p.hparts + ((size_t)(((j + 1) & 1) * 2) * Ppad + kr) * H + uc;
            *reinterpret_cast<uint2*>(hp) = hi;
            *reinterpret_cast<uint2*>(hp + (size_t)Ppad * H) = lo;
            if constexpr (NG == 4) {
              const float4 cn4 = *reinterpret_cast<const float4*>(e + 4 * 4096);
              if (!(stash_carry && live)) *reinterpret_cast<float4*>(p.state + (size_t)kr * H + uc) = cn4;
              if (live) {
                if (p.stash_g) {
                  float* gs = p.stash_g + pos * (4 * H) + uc;
#pragma unroll
                  for (int a = 0; a < 4; ++a) *reinterpret_cast<float4*>(gs + a * H) = *reinterpret_cast<const float4*>(e + a * 4096);
                }
                *reinterpret_cast<float4*>(p.stash_c + (pos + 1) * H + uc) = cn4;
              }
              if (cp) *reinterpret_cast<float4*>(p.wstate + ((size_t)((cp_full ? 1 : 0) * P + kr) * 2 + 1) * H + uc) = cn4;
            } else {
              if (!(stash_carry && live)) *reinterpret_cast<float4*>(p.state + (size_t)kr * H + uc) = h4;
            }
            if (live) *reinterpret_cast<float4*>(p.stash_h + (pos + 1) * H + uc) = h4;
            if (cp) *reinterpret_cast<float4*>(p.wstate + ((size_t)((cp_full ? 1 : 0) * P + kr) * 2) * H + uc) = h4;
          }
        }
      }
      if (tma_path && lane == 0) tma_store_wait_read();     // the staging tiles have been read: the ring may be refilled
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty);
      const long long t4 = prof ? clock64() : 0;
      publish_exchange();                      // the h split -> visible to the peers' TMA loads
      cluster_wait();
      tok = tok_n;
      if (prof) { const long long t5 = clock64(); pr[0] += t1 - t0; pr[1] += t2 - t1; pr[2] += t3 - t2; pr[3] += t4 - t3; pr[4] += t5 - t4; }
    }
    if (prof) {
#pragma unroll
      for (int i = 0; i < 5; ++i) p.prof[i] = pr[i];
      p.prof[5] = steps;
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_arrive();                          // nobody leaves while a peer may still multicast into its shared memory
  cluster_wait();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

template <int NG>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS, 1)
chain_tc_fwd_kernel(const __grid_constant__ FwdMaps maps, const FwdArgs p) {
  chain_tc_fwd_body<NG>(maps, p, blockIdx.x / CL);
}

// Value LSTM and reward GRU forward chains in ONE launch: clusters [0, clusters_v) walk the value chain, the rest the
// reward chain.  The two recurrences are independent given the tokens; side by side each gets half of the co-resident
// clusters, i.e. half the pieces of twice the length -- but the discarded warm-up is paid once in wall time instead of
// twice, which is what bounds the step when a rank holds few rows (512 rows per rank at 8 GPUs: 51 live + 160..256
// warm-up positions per piece).
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS, 1)
chains_tc_fwd_fused_kernel(const __grid_constant__ FwdMaps maps_v, const FwdArgs pv, const __grid_constant__ FwdMaps maps_r,
                           const FwdArgs pr, const int clusters_v) {
  const int cluster = blockIdx.x / CL;
  if (cluster < clusters_v) chain_tc_fwd_body<4>(maps_v, pv, cluster);
  else chain_tc_fwd_body<3>(maps_r, pr, cluster - clusters_v);
}

// ------------------------------------------------------------------------------------------------ backward (LSTM)
// The step GEMM dh_{t-1} [128 x 512] = dgates_t [128 x 2048] . W_hh [2048 x 512] is cut over the cluster's 8 CTAs as
// 2 K halves x 4 column quarters (N = 128, K = 1024 per CTA; rank = 4 * (K half) + quarter): per step a CTA ingests
// 0.5 MB of exchanged gate gradients (TMA-multicast among the 4 CTAs of its K half) + 0.5 MB of W_hh^T, and the two
// CTAs that share a column quarter swap the 64 columns of their partial sums the other one owns through DSMEM (32 KB per
// CTA per step, st.async into the partner's receive buffer, one mbarrier per step).
//
// What bounds the GEMM part of a step is the SHARED-MEMORY bandwidth of the SM (128 B/clk): operand reads of the MMAs
// plus the TMA writes of the fill.  Measured against that model (cycles from the GEMM's first load to its last MMA):
//   8 column slices (N = 64, K = 2048), 3 MMAs per K step:        2.3 MB read + 1.5 MB fill -> 29.7 K  (28.6 K measured)
//   2 K halves x 4 quarters (N = 128, K = 1024), 3 MMAs:           1.5 MB      + 1.0 MB      -> 19.5 K  (19.4 K measured)
//   the same, A_hi x [B_hi | B_lo] as ONE N = 256 MMA (below):     1.25 MB     + 1.0 MB      -> 17.6 K
// The two parts of W_hh^T of a stage are adjacent in shared memory (rows 0..127 hi, 128..255 lo' of one K-major tile),
// so main and the first correction term come from one instruction into adjacent accumulator columns; A_lo x B_hi
// accumulates onto the correction columns.  (Two alternating sets of 128 pieces per cluster -- the GEMM of one under
// the epilogue of the other -- were built and measured: 35.4 K cycles per set and step against 38.8 K, because the
// epilogue's staging traffic then competes for the same shared-memory bandwidth; with twice the warm-ups to pay it
// loses below ~14,000 rows and was removed.)
struct BwdCfg {
  static constexpr int STAGES = 6;
  static constexpr int KB = 2 * H / BK;                       // 32 K blocks per step and CTA
  static constexpr int NCOL = 2 * UN;                         // 128 output columns per CTA
  static constexpr int B_TILE = NCOL * BK * 2;                // 8 KB
  static constexpr int STAGE = 2 * A_TILE + 2 * B_TILE;       // 32 KB
  static constexpr int GROUP = 4;                             // CTAs that share (and multicast) an A tile
  static constexpr int SLICE_ROWS = BM / GROUP;               // 32 rows fetched per CTA
  static constexpr int SLICE = SLICE_ROWS * BK * 2;
  static constexpr int XBUF = BM * UN * 4;                    // 32 KB receive buffer of the partner's partial sums
  static constexpr int TMEM_COLS = 2 * NCOL, CORR = NCOL;
  static constexpr int SMEM = STAGES * STAGE + XBUF + 256 + 1024;
};
// chain_tc_bwd_kernel: per epilogue warp one staging buffer of 6 arrays of [32 rows][32 units] f32 (gates i,f,g,o, c_t,
// c_{t-1}): 128-byte row segments in both directions.  What a gather or a store pass costs is the NUMBER of row segments it
// touches (~2-3 cycles each, LSU and TMA engine alike: 3,072 segments of 64 bytes per step took 8.9 K cycles to request with
// cp.async and 11.3 K as TMA boxes -- both measured -- against 2.4 K for the forward's 1,280 segments of 128 bytes), so the
// tile is as wide as the 32 units a warp owns.  The injected dL/dh rows (one position in ten) travel through registers.
constexpr int B_GST_WARP = 6 * 4096;
static_assert(EPI_WARPS * B_GST_WARP <= BwdCfg::STAGES * BwdCfg::STAGE, "epilogue staging lives inside the (idle) TMA ring");
static_assert(BwdCfg::SMEM <= 232448, "shared memory budget");

struct BwdArgs {
  int P, Ppad, steps, warm, cp_half;
  // Row of the per-position arrays that piece (= MMA row) k works on at local time t: k * stride_k + t * stride_t.
  // Chain pieces: (seg, 1).  The policy's BPTT runs on the same kernel with the batch rows as "pieces", the cell steps
  // as time and the rollout's [step][row] arrays: (1, B), warm = 0, no checkpoints, and dL/dh0 written at the end.
  long long stride_k, stride_t;
  const float* stash_g;    // [rows][2048] activated i,f,g,o
  const float* stash_c;    // [rows + stride_t][512]: c after the cell of row r lives at row r + stride_t
  const int* take;         // [rows] row of dh_take injected at the position, or -1
  const float* dh_take;    // [take_rows][512]
  float* dgates;           // [rows][2048] fp32 pre-activation gate gradients of the live positions (policy BPTT), or null
  __half* dg_pair;         // or [2][pair_rows][2048]: their scaled fp16 split, columns in icrl_gate_pair_col order
  long long pair_rows;
  float* dg_inv_scale;     // device word: 1 / scale of dg_pair (written when dg_pair is set)
  __half* dgx;             // [2 buffers][2 parts][Ppad][2048] scaled fp16 split of the gate gradients (exchange)
  const float* dh_max;     // device word: max |dh_take| (scale of the recurrence)
  float* bstate;           // [2 checkpoints][2 sides][P][2][512] (dh, dc) at the joints (null: no checkpoints)
  float* dh0_out;          // [P][512] dL/dh entering local time 0 (one more contraction after the last step), or null
  float* overflow;         // device word: set to 1 when a scaled gate gradient left the fp16 range
  float main_gain;
  long long* prof;
};

// power-of-two scale S with max|dh_take| * S in [8, 16): fp16 then holds 22 bits of every gate gradient down to
// 2^-18 of that maximum and has 2^12 of headroom above it.
__device__ __forceinline__ float bwd_scale(float m) {
  if (!(m > 0.f) || !isfinite(m)) return 1.f;
  int ex;
  frexpf(m, &ex);                              // m = f * 2^ex, f in [0.5, 1)
  ex = 4 - ex;
  ex = ex > 100 ? 100 : (ex < -100 ? -100 : ex);
  return ldexpf(1.f, ex);
}

__device__ __forceinline__ void st_global_v8(__half* dst, const uint2* v) {      // 32 bytes, 32-byte aligned
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(v[0].x), "r"(v[0].y), "r"(v[1].x),
               "r"(v[1].y), "r"(v[2].x), "r"(v[2].y), "r"(v[3].x), "r"(v[3].y) : "memory");
}

__device__ __forceinline__ unsigned mapa_u32(unsigned addr, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_v4(unsigned raddr, const float* v, unsigned rbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(raddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "r"(rbar) : "memory");
}

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS, 1)
chain_tc_bwd_kernel(const __grid_constant__ CUtensorMap map_dg, const __grid_constant__ CUtensorMap map_w, const BwdArgs p) {
  using Cfg = BwdCfg;
  constexpr int STAGES = Cfg::STAGES, STAGE = Cfg::STAGE, B_KB = Cfg::KB, B_CORR = Cfg::CORR, BB_TILE = Cfg::B_TILE;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char* xbuf = smem + STAGES * STAGE;       // [128 rows][16 chunks of 4 floats], chunk c of row r at c ^ (r & 7)
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(xbuf + Cfg::XBUF);
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * STAGES + 3);
  const unsigned bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[STAGES]);
  const unsigned bar_acc_full = smem_u32(&bars[2 * STAGES]), bar_acc_empty = smem_u32(&bars[2 * STAGES + 1]);
  const unsigned bar_x = smem_u32(&bars[2 * STAGES + 2]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned rank = cluster_rank();
  // rank = 4 * (K half) + (column quarter); the CTA contracts K half kh for the 128 columns of quarter nq and owns
  // (cell arithmetic, stores) the 64 columns [128 nq + 64 kh, +64) of them
  const int kh = (int)(rank >> 2), nq = (int)(rank & 3);
  const int ub = 128 * nq + 64 * kh;                                // first hidden unit this CTA owns
  const int own_c = 64 * kh;                                        // its column in this CTA's accumulators
  const unsigned short grp_mask = (unsigned short)(0xF << (4 * kh));
  const int m0 = (blockIdx.x / CL) * BM;
  const int P = p.P, Ppad = p.Ppad, steps = p.steps;
  const int iters = steps + (p.dh0_out ? 1 : 0);       // one more contraction when dL/dh0 is wanted

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, Cfg::GROUP); }
    mbar_init(bar_acc_full, 1);
    mbar_init(bar_acc_empty, EPI_WARPS);
    mbar_init(bar_x, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dg) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  cluster_arrive();
  cluster_wait();

  if (warp == 2 || warp == 3) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    for (int it = 0; it < iters; ++it) { cluster_arrive(); cluster_wait(); }
  } else if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (no GEMM before the first step)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    unsigned n = 0;
    for (int it = 0; it < iters; ++it) {
      if (it > 0 && lane == 0) {
        const int arow = ((it & 1) * 2) * Ppad + m0;
        for (int kb = 0; kb < B_KB; ++kb, ++n) {
          const int s = n % STAGES;
          mbar_wait(bar_empty + 8 * s, ((n / STAGES) & 1u) ^ 1u);
          const unsigned full = bar_full + 8 * s;
          mbar_expect_tx(full, 2 * A_TILE + 2 * BB_TILE);
          const unsigned base = smem_u32(smem + s * STAGE);
          const int kc = (kh * B_KB + kb) * BK;
          tma_load_2d_mcast(base + nq * Cfg::SLICE, &map_dg, kc, arow + nq * Cfg::SLICE_ROWS, full, grp_mask);
          tma_load_2d_mcast(base + A_TILE + nq * Cfg::SLICE, &map_dg, kc, arow + Ppad + nq * Cfg::SLICE_ROWS, full, grp_mask);
          tma_load_3d(base + 2 * A_TILE, &map_w, kc, nq * Cfg::NCOL, 0, full);            // hi at +0, lo' at +BB_TILE
        }
      }
      __syncwarp();
      cluster_arrive();
      cluster_wait();                    // the gate gradients of this step (all 8 CTAs) are in global memory
      if (lane == 0) fence_proxy_async();
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    unsigned n = 0;
    for (int it = 0; it < iters; ++it) {
      if (it > 0) {
        mbar_wait(bar_acc_empty, (unsigned)(it - 1) & 1u);
        tc_fence_after();
        for (int kb = 0; kb < B_KB; ++kb, ++n) {
          const int s = n % STAGES;
          mbar_wait(bar_full + 8 * s, (n / STAGES) & 1u);
          tc_fence_after();
          const unsigned base = smem_u32(smem + s * STAGE);
          const unsigned long long dA0 = smem_desc_sw64(base), dA1 = smem_desc_sw64(base + A_TILE);
          const unsigned long long dB0 = smem_desc_sw64(base + 2 * A_TILE);      // 256 rows: hi, then lo' at +BB_TILE
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              // [main | correction] = A_hi x [B_hi | B_lo'] in one N = 256 instruction, then correction += A_lo' x B_hi
              tc_mma(tmem_base, dA0 + 2 * k, dB0 + 2 * k, idesc_f16_m128(2 * Cfg::NCOL), (kb | k) != 0);
              tc_mma(tmem_base + B_CORR, dA1 + 2 * k, dB0 + 2 * k, idesc_f16_m128(Cfg::NCOL), 1u);
            }
            tc_commit_mcast(bar_empty + 8 * s, grp_mask);
          }
          __syncwarp();
        }
        if (elect_one()) tc_commit(bar_acc_full);
      }
      __syncwarp();
      cluster_arrive();
      cluster_wait();
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int ew = warp - EPI_WARP0;
    const int q = warp & 3;
    const int ch = ew >> 2;
    const int k_own = m0 + 32 * q + lane;
    const bool valid = k_own < P;
    const unsigned tq = tmem_base + ((unsigned)(32 * q) << 16);
    unsigned char* gst = smem + ew * B_GST_WARP;
    const long long sk = p.stride_k, stt = p.stride_t;
    const float S = bwd_scale(*p.dh_max), invS = 1.f / S;
    if (p.dg_pair && blockIdx.x == 0 && ew == 0 && lane == 0) *p.dg_inv_scale = invS;
    const float mg = p.main_gain;
    float dc[4][8];                            // carried dL/dc of this thread's piece: [8-unit group][unit]
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int i = 0; i < 8; ++i) dc[a][i] = 0.f;
    float ovf = 0.f;
    int tk = valid ? p.take[(long long)k_own * sk + (long long)(steps - 1) * stt] : -1;
    const bool prof = p.prof != nullptr && blockIdx.x == 0 && ew == 0 && lane == 0;
    long long pr[5] = {0, 0, 0, 0, 0}, pr_issue = 0, pr_xwait = 0;
    const int half_ref_it = steps - 1 - (p.warm - 1 - p.cp_half);      // reference side of the half-way checkpoint
    // K split: receive buffer of the partner CTA (rank ^ 4) and this thread's row in it / in the own one
    const int xrow = (32 * q + lane) * 256, xsw = lane & 7;
    const unsigned x_remote = mapa_u32(smem_u32(xbuf), rank ^ 4u), x_rbar = mapa_u32(bar_x, rank ^ 4u);
    bool x_have = false;                       // whether this iteration has partial sums to add (it > 0)
    auto load_partner = [&](int c8, float* xr) {       // c8: 8-unit group 0..3 of this warp's 32 units
      if (x_have) {
        const float4 a = *reinterpret_cast<const float4*>(xbuf + xrow + (((8 * ch + 2 * c8) ^ xsw) << 4));
        const float4 b = *reinterpret_cast<const float4*>(xbuf + xrow + (((8 * ch + 2 * c8 + 1) ^ xsw) << 4));
        xr[0] = a.x; xr[1] = a.y; xr[2] = a.z; xr[3] = a.w; xr[4] = b.x; xr[5] = b.y; xr[6] = b.z; xr[7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) xr[i] = 0.f;
      }
    };

    const int ucolw = ub + 32 * ch;              // first of this warp's 32 units
    // (L) stash of position t: activated gates (arrays 0..3), c_t (4), c_{t-1} (5), 8 lanes per row (128 bytes); element
    //     (row, 16-byte chunk c) lives at row*128 + ((c ^ (row & 7)) << 4).  Requested as soon as the ring is idle (the
    //     step's MMAs have completed), before the partial-sum swap, so that the rows travel while that is under way.
    auto issue_gather = [&](int t) {
      const int c4 = lane & 7;
#pragma unroll
      for (int i8 = 0; i8 < 8; ++i8) {
        const int r = i8 * 4 + (lane >> 3);
        const int kr = m0 + 32 * q + r;
        if (kr < P) {
          const size_t pos = (size_t)kr * sk + (size_t)t * stt;
          const unsigned dst = smem_u32(gst) + (unsigned)(r * 128 + ((c4 ^ (r & 7)) << 4));
          const float* gsrc = p.stash_g + pos * (4 * H) + ucolw + c4 * 4;
#pragma unroll
          for (int a = 0; a < 4; ++a) cp_async16(dst + a * 4096, gsrc + a * H);
          cp_async16(dst + 4 * 4096, p.stash_c + (pos + stt) * H + ucolw + c4 * 4);
          cp_async16(dst + 5 * 4096, p.stash_c + pos * H + ucolw + c4 * 4);
        }
      }
    };

    for (int it = 0; it < iters; ++it) {
      const long long t0 = prof ? clock64() : 0;
      const int t = steps - 1 - it;
      x_have = it > 0;
      const int tk_n = (valid && t > 0) ? p.take[(long long)k_own * sk + (long long)(t - 1) * stt] : -1;
      long long tgi = 0;
      if (it == 0) issue_gather(t);
      if (it > 0) {
        mbar_wait(bar_acc_full, (unsigned)(it - 1) & 1u);
        tc_fence_after();
        if (it < steps) {
          const long long g0 = prof ? clock64() : 0;
          issue_gather(t);
          if (prof) tgi = clock64() - g0;
        }
        {
          // the 64 columns of this CTA's partial sums that the partner (other K half, same column quarter) owns: this
          // thread's row, its 32-column half, combined main + correction, straight into the partner's receive buffer
          if (ew == 0 && lane == 0) mbar_expect_tx(bar_x, Cfg::XBUF);
          const int pc = 64 * (1 - kh) + 32 * ch;
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            float rec[8], cor[8], v[8];
            tmem_ld8x2(tq + (unsigned)(pc + 8 * j8), tq + (unsigned)(B_CORR + pc + 8 * j8), rec, cor);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = fmaf(cor[i], LO_INV, rec[i] * mg);
            st_async_v4(x_remote + (unsigned)(xrow + (((8 * ch + 2 * j8) ^ xsw) << 4)), v, x_rbar);
            st_async_v4(x_remote + (unsigned)(xrow + (((8 * ch + 2 * j8 + 1) ^ xsw) << 4)), v + 4, x_rbar);
          }
        }
      }
      bool x_ready = it == 0;
      if (it == steps) {
        if (!x_ready) { mbar_wait(bar_x, (unsigned)(it - 1) & 1u); x_ready = true; }
        // the extra iteration: dL/dh entering local time 0 = the contraction of the last step's gate gradients
#pragma unroll
        for (int ps = 0; ps < 2; ++ps) {
          const int ucolp = ub + 32 * ch + 16 * ps;
#pragma unroll
          for (int c8 = 0; c8 < 2; ++c8) {
            float rec[8], cor[8], xr[8];
            tmem_ld8x2(tq + (unsigned)(own_c + 32 * ch + 16 * ps + 8 * c8), tq + (unsigned)(B_CORR + own_c + 32 * ch + 16 * ps + 8 * c8), rec, cor);
            load_partner(2 * ps + c8, xr);
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = (fmaf(cor[i], LO_INV, rec[i] * mg) + xr[i]) * invS;
            *reinterpret_cast<float4*>(gst + lane * 64 + (((2 * c8) ^ ((lane >> 1) & 3)) << 4)) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4*>(gst + lane * 64 + (((2 * c8 + 1) ^ ((lane >> 1) & 3)) << 4)) = make_float4(o[4], o[5], o[6], o[7]);
          }
          __syncwarp();
          const int c4 = lane & 3;
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4) {
            const int r = i4 * 8 + (lane >> 2);
            const int kr = m0 + 32 * q + r;
            if (kr < P)
              *reinterpret_cast<float4*>(p.dh0_out + (size_t)kr * H + ucolp + c4 * 4) =
                  *reinterpret_cast<const float4*>(gst + r * 64 + ((c4 ^ ((r >> 1) & 3)) << 4));
          }
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty);
        cluster_arrive();
        cluster_wait();
        break;
      }
      const long long t1 = prof ? clock64() : 0;
      const bool w_full = it == p.warm - 1, w_half = it == p.cp_half;            // warm-up side records (pieces < P-1)
      const bool r_full = it == steps - 1, r_half = p.cp_half >= 0 && it == half_ref_it;   // reference side (pieces >= 1)
      const bool cp_it = p.bstate != nullptr && (w_full || w_half || r_full || r_half);
      long long tg = 0, tc = 0, ts = 0;
      // injected dL/dh of this thread's own row (one position in ten): 8 units at a time, one group ahead of its use
      const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool has_inj = valid && tk >= 0;
      const float4* inj_src = reinterpret_cast<const float4*>(p.dh_take + (size_t)(has_inj ? tk : 0) * H + ucolw);
      float4 nx0 = has_inj ? __ldg(inj_src) : zero4, nx1 = has_inj ? __ldg(inj_src + 1) : zero4;
      const long long t2 = prof ? clock64() : 0;
      if (!x_ready) mbar_wait(bar_x, (unsigned)(it - 1) & 1u);
      const long long u0 = prof ? clock64() : 0;
      cp_async_wait_all();
      __syncwarp();
      const long long u1 = prof ? clock64() : 0;
      if (prof) { pr_issue += tgi; pr_xwait += u0 - t2; tg += u1 - u0; }
      // (C) gate gradients, one row per lane, in place on the staging tile
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float rec[8], cor[8], xr[8];
        const float4 inj0 = nx0, inj1 = nx1;
        if (c8 < 3 && has_inj) { nx0 = __ldg(inj_src + 2 * (c8 + 1)); nx1 = __ldg(inj_src + 2 * (c8 + 1) + 1); }
        load_partner(c8, xr);
        if (it > 0) {
          tmem_ld8x2(tq + (unsigned)(own_c + 32 * ch + 8 * c8), tq + (unsigned)(B_CORR + own_c + 32 * ch + 8 * c8), rec, cor);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) { rec[i] = 0.f; cor[i] = 0.f; }
        }
        unsigned char* e0 = gst + lane * 128 + (((2 * c8) ^ (lane & 7)) << 4);
        unsigned char* e1 = gst + lane * 128 + (((2 * c8 + 1) ^ (lane & 7)) << 4);
        float tin[6][8];
        const float injv[8] = {inj0.x, inj0.y, inj0.z, inj0.w, inj1.x, inj1.y, inj1.z, inj1.w};
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          const float4 v0 = *reinterpret_cast<const float4*>(e0 + a * 4096);
          const float4 v1 = *reinterpret_cast<const float4*>(e1 + a * 4096);
          tin[a][0] = v0.x; tin[a][1] = v0.y; tin[a][2] = v0.z; tin[a][3] = v0.w;
          tin[a][4] = v1.x; tin[a][5] = v1.y; tin[a][6] = v1.z; tin[a][7] = v1.w;
        }
        float d_i[8], d_f[8], d_g[8], d_o[8], dhv[8], dci[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float gi = tin[0][i], gf = tin[1][i], gg = tin[2][i], go = tin[3][i], cc = tin[4][i], cp = tin[5][i];
          const float dh = (fmaf(cor[i], LO_INV, rec[i] * mg) + xr[i]) * invS + injv[i];
          const float tcv = tanh_lean(cc);
          const float dct = dc[c8][i] + dh * (go * (1.f - tcv * tcv));
          dhv[i] = dh;
          dci[i] = dc[c8][i];
          d_o[i] = dh * (tcv * go * (1.f - go));
          d_i[i] = dct * (gg * gi * (1.f - gi));
          d_f[i] = dct * (cp * gf * (1.f - gf));
          d_g[i] = dct * (gi * (1.f - gg * gg));
          dc[c8][i] = dct * gf;
          ovf = fmaxf(ovf, fmaxf(fmaxf(fabsf(d_i[i]), fabsf(d_f[i])), fmaxf(fabsf(d_g[i]), fabsf(d_o[i]))));
        }
        *reinterpret_cast<float4*>(e0) = make_float4(d_i[0], d_i[1], d_i[2], d_i[3]);
        *reinterpret_cast<float4*>(e1) = make_float4(d_i[4], d_i[5], d_i[6], d_i[7]);
        *reinterpret_cast<float4*>(e0 + 4096) = make_float4(d_f[0], d_f[1], d_f[2], d_f[3]);
        *reinterpret_cast<float4*>(e1 + 4096) = make_float4(d_f[4], d_f[5], d_f[6], d_f[7]);
        *reinterpret_cast<float4*>(e0 + 2 * 4096) = make_float4(d_g[0], d_g[1], d_g[2], d_g[3]);
        *reinterpret_cast<float4*>(e1 + 2 * 4096) = make_float4(d_g[4], d_g[5], d_g[6], d_g[7]);
        *reinterpret_cast<float4*>(e0 + 3 * 4096) = make_float4(d_o[0], d_o[1], d_o[2], d_o[3]);
        *reinterpret_cast<float4*>(e1 + 3 * 4096) = make_float4(d_o[4], d_o[5], d_o[6], d_o[7]);
        if (cp_it) {                             // (dh, dc) entering the step: only the joint checkpoints read them
          *reinterpret_cast<float4*>(e0 + 4 * 4096) = make_float4(dhv[0], dhv[1], dhv[2], dhv[3]);
          *reinterpret_cast<float4*>(e1 + 4 * 4096) = make_float4(dhv[4], dhv[5], dhv[6], dhv[7]);
          *reinterpret_cast<float4*>(e0 + 5 * 4096) = make_float4(dci[0], dci[1], dci[2], dci[3]);
          *reinterpret_cast<float4*>(e1 + 5 * 4096) = make_float4(dci[4], dci[5], dci[6], dci[7]);
        }
      }
      __syncwarp();
      const long long u2 = prof ? clock64() : 0;
      // (S) one pass over the staged gate gradients, 8 lanes per row: the scaled fp16 split (the next step's A operand of
      //     every CTA of the cluster), the live positions' gate gradients (parameter-gradient contractions), the joint
      //     checkpoints
      {
        const int c4 = lane & 7;
#pragma unroll
        for (int i8 = 0; i8 < 8; ++i8) {
          const int r = i8 * 4 + (lane >> 3);
          const int kr = m0 + 32 * q + r;
          if (kr < P) {
            const size_t pos = (size_t)kr * sk + (size_t)t * stt;
            const unsigned char* e = gst + r * 128 + ((c4 ^ (r & 7)) << 4);
            const bool live = kr == P - 1 || it >= p.warm;
            const int uc = ucolw + c4 * 4;
            __half* xp = p.dgx + ((size_t)((((it + 1) & 1) * 2) * Ppad + kr)) * (4 * H) + uc;
            uint2 hi[4], lo[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
              const float4 d = *reinterpret_cast<const float4*>(e + a * 4096);
              split4_f16(make_float4(d.x * S, d.y * S, d.z * S, d.w * S), hi[a], lo[a]);
              *reinterpret_cast<uint2*>(xp + a * H) = hi[a];
              *reinterpret_cast<uint2*>(xp + (size_t)Ppad * (4 * H) + a * H) = lo[a];
              if (live && p.dgates) *reinterpret_cast<float4*>(p.dgates + pos * (4 * H) + a * H + uc) = d;
            }
            if (live && p.dg_pair) {
              // the same split for the parameter-gradient contractions: this lane's 4 units of all 4 gates are 16
              // adjacent columns (icrl_gate_pair_col), one 32-byte store per plane -- 4 row segments of 128 bytes per
              // warp and row, as many as the fp32 values would cost
              __half* pp = p.dg_pair + pos * (4 * H) + icrl_gate_pair_col(uc);
              st_global_v8(pp, hi);
              st_global_v8(pp + (size_t)p.pair_rows * (4 * H), lo);
            }
            if (cp_it) {
              const float4 dh4 = *reinterpret_cast<const float4*>(e + 4 * 4096);
              const float4 dc4 = *reinterpret_cast<const float4*>(e + 5 * 4096);
              if (kr < P - 1 && (w_full || w_half)) {
                float* bs = p.bstate + ((size_t)(((w_full ? 1 : 0) * 2 + 0) * P + kr) * 2) * H + uc;
                *reinterpret_cast<float4*>(bs) = dh4;
                *reinterpret_cast<float4*>(bs + H) = dc4;
              }
              if (kr >= 1 && (r_full || r_half)) {
                float* bs = p.bstate + ((size_t)(((r_full ? 1 : 0) * 2 + 1) * P + kr) * 2) * H + uc;
                *reinterpret_cast<float4*>(bs) = dh4;
                *reinterpret_cast<float4*>(bs + H) = dc4;
              }
            }
          }
        }
      }
      __syncwarp();                            // the next step's gather overwrites the staging tile
      if (prof) { const long long u3 = clock64(); tc += u2 - u1; ts += u3 - u2; }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty);
      const long long t4 = prof ? clock64() : 0;
      publish_exchange();
      cluster_wait();
      tk = tk_n;
      if (prof) { const long long t5 = clock64(); pr[0] += t1 - t0 - tgi; pr[1] += tg; pr[2] += tc; pr[3] += ts; pr[4] += t5 - t4; }
    }
    if (valid && !(ovf * S < 30000.f)) *p.overflow = 1.f;       // also catches NaN
    if (prof) {
#pragma unroll
      for (int i = 0; i < 5; ++i) p.prof[i] = pr[i];
      p.prof[5] = steps;
      p.prof[6] = pr_issue;                    // gather requests
      p.prof[7] = pr_xwait;                    // wait for the partner's partial sums
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_arrive();
  cluster_wait();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ packing / checks
// LSTM / GRU forward operand: [2 parts][NG*512][512], row (r*GN + g*64 + jj) = W_hh row (g*512 + r*64 + jj).
// LSTM backward operand:      [2 parts][512][2048],   row n (hidden unit), column k (gate row): W_hh[k][n].
__global__ void pack_chain_tc_kernel(int NG, const float* __restrict__ W_hh, __half* __restrict__ fwd, __half* __restrict__ bwd) {
  const long long n_f = (long long)NG * H * H;
  const long long total = n_f + (bwd ? n_f : 0);
  const int GN = NG * UN;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float v;
    __half *hi, *lo;
    if (i < n_f) {
      const int prow = (int)(i / H), k = (int)(i % H);
      const int r = prow / GN, g = (prow % GN) / UN, jj = prow % UN;
      v = W_hh[(size_t)(g * H + r * UN + jj) * H + k];
      hi = fwd + i;
      lo = fwd + n_f + i;
    } else {
      const long long e = i - n_f;
      const int n = (int)(e / (NG * H)), k = (int)(e % (NG * H));
      v = W_hh[(size_t)k * H + n];
      hi = bwd + e;
      lo = bwd + n_f + e;
    }
    const __half h = __float2half_rn(v);
    *hi = h;
    *lo = __float2half_rn((v - __half2float(h)) * 2048.f);
  }
}

// integer max of the bit pattern: non-negative floats order like their patterns, a NaN has the largest one
__device__ __forceinline__ void err_max_bits(float* slot, int bits) { atomicMax(reinterpret_cast<int*>(slot), bits); }

// Block (k-1, cp): state piece k reached after step cp_half (cp = 0) / warm-1 (cp = 1) against the stash row the
// preceding pieces wrote for the same position.  err[0] = max |dh| (full), err[1] = max |dc| / max(1, |c|) (full),
// err[2], err[3] = the same half-way through the warm-up.
__global__ void chain_tc_check_fwd_kernel(int P, long long seg, int warm, int cp_half, const float* wstate,
                                          const float* stash_h, const float* stash_c, float* err) {
  const int k = blockIdx.x + 1, cp = blockIdx.y, u = threadIdx.x;
  const int j = cp ? warm - 1 : cp_half;
  if (j < 0) return;
  const size_t row = (size_t)k * seg + j + 1;
  const float* w = wstate + ((size_t)(cp * P + k) * 2) * H;
  int ih = __float_as_int(fabsf(w[u] - stash_h[row * H + u])), ic = 0;
  if (stash_c) {
    const float ct = stash_c[row * H + u];
    ic = __float_as_int(fabsf(w[H + u] - ct) / fmaxf(1.f, fabsf(ct)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ih = max(ih, __shfl_xor_sync(0xffffffffu, ih, o));
    ic = max(ic, __shfl_xor_sync(0xffffffffu, ic, o));
  }
  if ((threadIdx.x & 31) == 0) {
    err_max_bits(err + (cp ? 0 : 2), ih);
    if (stash_c) err_max_bits(err + (cp ? 1 : 3), ic);
  }
}

// Block (k, cp): (dh, dc) piece k carried at the joint (cp = 1: position (k+1)*seg, its last warm-up step; cp = 0:
// half-way through the warm-up) against what piece k+1 computed at the same position, relative to max |dh_take|.
// err[0] = dh (full), err[1] = dc (full), err[2], err[3] = half-way; err[4] = max |dh_take| (read only).
__global__ void chain_tc_check_bwd_kernel(int P, int cp_half, const float* bstate, float* err) {
  const int k = blockIdx.x, cp = blockIdx.y, u = threadIdx.x;
  if (cp == 0 && cp_half < 0) return;
  const float m = err[4];
  const float inv = m > 0.f ? 1.f / m : 1.f;
  const float* a = bstate + ((size_t)((cp * 2 + 0) * P + k) * 2) * H;
  const float* b = bstate + ((size_t)((cp * 2 + 1) * P + k + 1) * 2) * H;
  int ih = __float_as_int(fabsf(a[u] - b[u]) * inv), ic = __float_as_int(fabsf(a[H + u] - b[H + u]) * inv);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ih = max(ih, __shfl_xor_sync(0xffffffffu, ih, o));
    ic = max(ic, __shfl_xor_sync(0xffffffffu, ic, o));
  }
  if ((threadIdx.x & 31) == 0) {
    err_max_bits(err + (cp ? 0 : 2), ih);
    err_max_bits(err + (cp ? 1 : 3), ic);
  }
}

__global__ void absmax_kernel(long long n, const float* __restrict__ x, float* out) {
  int m = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = max(m, __float_as_int(fabsf(x[i])));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) err_max_bits(out, m);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_fn(EncodeTiledFn* out) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void* q = nullptr;
    ICRL_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres));
    ICRL_REQUIRE(q && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  *out = fn;
  return ICRL_OK;
}

// fp16 [rows][cols] row-major, box {32, box_rows}, 64B swizzle
int make_map_2d(CUtensorMap* map, const void* ptr, long long cols, long long rows, int box_rows) {
  EncodeTiledFn fn;
  int rc = encode_fn(&fn);
  if (rc) return rc;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    icrl_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld, cols %lld)", (int)r, rows, cols);
    return ICRL_ERR_CUDA;
  }
  return ICRL_OK;
}

// fp16 [2 parts][rows][cols], box {32, box_rows, 2}
int make_map_3d(CUtensorMap* map, const void* ptr, long long cols, long long rows, int box_rows) {
  EncodeTiledFn fn;
  int rc = encode_fn(&fn);
  if (rc) return rc;
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, 2};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows * cols * 2};
  const cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 2};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    icrl_set_error("cuTensorMapEncodeTiled (3-D) failed with CUresult %d (rows %lld, cols %lld)", (int)r, rows, cols);
    return ICRL_ERR_CUDA;
  }
  return ICRL_OK;
}

// fp32 [..][cols] stash array as {column, step of a piece, piece}: strides (4 B, cols * 4 B, seg * cols * 4 B), box
// {box_cols, 1, 32} with the swizzle whose span equals the box row (32 floats: 128B, 16 floats: 64B).  Returns
// ICRL_ERR_CUDA when the driver refuses the (overlapping) strides; callers then keep the per-thread stores.
int make_map_stash(CUtensorMap* map, const float* base, int cols, long long steps, long long seg, int P, int box_cols) {
  EncodeTiledFn fn;
  int rc = encode_fn(&fn);
  if (rc) return rc;
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)steps, (cuuint64_t)P};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)seg * cols * 4};
  const cuuint32_t box[3] = {(cuuint32_t)box_cols, 1, 32};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? ICRL_OK : ICRL_ERR_CUDA;
}

int cp_half_of(int warm) { return warm >= 8 ? warm / 2 - 1 : -1; }

}  // namespace

// Compensation of the tensor core's truncating accumulation.  tcgen05.mma truncates (round toward zero) each time it adds
// into a tensor-memory accumulator: measured -1.5e-8 .. -1.8e-8 of the accumulator per MMA (scripts/tc_accuracy_probe.py,
// scripts/debug_bias.py).  The main accumulator of a step sums K / 16 instructions, so its expected relative loss is
// (K / 16) * 1.8e-8: 5.8e-7 forward (K = 512), 2.3e-6 backward (K = 2048) -- a SYSTEMATIC bias toward zero, unlike the
// unbiased round-to-nearest of the fp32 FMA chains.  Uncompensated it leaves mean(h_tc - h_serial) * sign(h) = -3.3e-7
// after 200 optimizer steps (values 1.1e-5 off at |v| ~ 8, gradients 4e-4 of max where the advantage cancels);
// multiplying the main accumulator by 1 + that expectation zeroes the mean (-5e-8 .. +8e-8 between 4.8e-7 and 7.2e-7) and
// leaves the random part (~1.6 ulp, below the 512-term FMA chain's own rounding noise).  icrl_chain_tc_set_bias
// overrides the two factors (experiments).
static float g_tc_bias[2] = {32 * 1.8e-8f, 128 * 1.8e-8f};
void icrl_chain_tc_set_bias_impl(float fwd, float bwd) { g_tc_bias[0] = fwd; g_tc_bias[1] = bwd; }
// icrl_chain_tc_set_tma_store: stash stores through TMA tensor stores (1) or per-thread vector stores (0, default).
// Measured at B = 4096: no gain (forward 18.5 vs 17.7 ms) -- the store phase is not bound by instruction issue but by the
// L2: every cluster writes its 240 KB of stash per CTA in the same window (29 MB per kernel step chip-wide, on top of
// 92 MB of operand fill and 20 MB of gathers: 141 MB per step = 22 K cycles at the measured 6.3 KB/clk L2 cap, against
// a step of 35 K).  Kept as a switch.
static int g_tc_tma_store = 0;
void icrl_chain_tc_set_tma_store_impl(int on) { g_tc_tma_store = on; }
// (Tried and removed: a second backward kernel sized for two co-resident CTAs per SM -- 3-stage ring, 8-unit staging
// passes, dL/dc in shared memory, 80 registers, 106 KB -- so that one cluster's epilogue would run under the operand fill of
// the cluster sharing its SMs.  It was correct, but the driver grants a tcgen05 kernel ONE CTA per SM whatever its
// footprint (cudaOccupancyMaxActiveBlocksPerMultiprocessor = 1 at 0 bytes of dynamic shared memory, 384 threads x 80
// registers; registers are granted per 4 warps, setmaxnreg does not raise ptxas' allocation above the launch-bounds cap), so
// the second cluster never shared the SMs and the leaner kernel was simply slower: 23.8 vs 16.4 ms at B = 4096.)
static long long* g_chain_tc_prof = nullptr;      // icrl_chain_tc_set_profile: 24 device int64 (forward [0..5], backward [8..13], fused reward chain [16..21])
void icrl_chain_tc_set_profile_impl(long long* buf) { g_chain_tc_prof = buf; }

// Co-resident clusters of 8 CTAs x 128 pieces (a cluster cannot span GPCs: 15-16 clusters on a B200).
int icrl_chain_tc_max_pieces_impl() {
  static int cached = 0;
  if (cached) return cached;
  int n = 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CL * 64);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = FwdCfg<4>::SMEM;
  cudaLaunchAttribute at;
  at.id = cudaLaunchAttributeClusterDimension;
  at.val.clusterDim.x = CL; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  cfg.attrs = &at;
  cfg.numAttrs = 1;
  cudaError_t e = cudaFuncSetAttribute(chain_tc_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<4>::SMEM);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, (void*)chain_tc_fwd_kernel<4>, &cfg);
  if (e != cudaSuccess || n < 1) { cudaGetLastError(); n = 12; }
  cached = n * BM;
  return cached;
}

// pieces of the backward recurrence that are co-resident: the same clusters as the forward kernels (one CTA per SM)
int icrl_chain_tc_bwd_max_pieces_impl() { return icrl_chain_tc_max_pieces_impl(); }

size_t icrl_chain_tc_weight_halves_impl(int kind) { return kind == 0 ? (size_t)4 * 4 * H * H : (size_t)2 * 3 * H * H; }

int icrl_pack_chain_tc_weights_impl(cudaStream_t st, int kind, const float* W_hh, void* packed) {
  ICRL_REQUIRE(kind == 0 || kind == 1, "kind: 0 = LSTM, 1 = GRU");
  __half* fwd = reinterpret_cast<__half*>(packed);
  const int NG = kind == 0 ? 4 : 3;
  __half* bwd = kind == 0 ? fwd + (size_t)2 * NG * H * H : nullptr;
  pack_chain_tc_kernel<<<148 * 4, 256, 0, st>>>(NG, W_hh, fwd, bwd);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

static int pad_pieces(int P) { return icrl_cdiv(P, BM) * BM; }

// one launch's scratch: the backward exchange buffer is the largest user (fp16 [2][2][Ppad][2048])
size_t icrl_chain_tc_ws_bytes_impl(int pieces) { return (size_t)4 * pad_pieces(pieces) * 4 * H * sizeof(__half); }
size_t icrl_chain_tc_cp_floats_impl(int pieces) { return (size_t)2 * 2 * pieces * 2 * H; }

// argument block, tensor maps and scratch initialisation of one forward chain launch
static int fwd_setup(cudaStream_t st, int kind, int P, long long seg, int warm, const int* stream, const float* table,
                     const void* packed, const float* b_hn, float* stash_h, float* stash_c, float* stash_g, void* ws,
                     float* cp_state, float* err, FwdArgs* a, FwdMaps* m) {
  CUtensorMap* mh = &m->h;
  CUtensorMap* mw = &m->w;
  ICRL_REQUIRE(kind == 0 || kind == 1, "kind: 0 = LSTM, 1 = GRU");
  ICRL_REQUIRE(P >= 2 && seg >= 1 && warm >= 1, "chain pieces need P >= 2, seg >= 1, warm >= 1");
  ICRL_REQUIRE((long long)P * seg + warm < (1ll << 31), "token stream longer than 2^31");
  ICRL_REQUIRE(stream && table && packed && stash_h && ws && cp_state && err, "null argument");
  ICRL_REQUIRE(kind == 1 ? b_hn != nullptr : stash_c != nullptr, "LSTM needs stash_c, GRU needs b_hn");
  const int Ppad = pad_pieces(P);
  __half* hparts = reinterpret_cast<__half*>(ws);
  float* state = reinterpret_cast<float*>(hparts + (size_t)4 * Ppad * H);
  ICRL_CUDA(cudaMemsetAsync(hparts, 0, (size_t)4 * Ppad * H * sizeof(__half) + (size_t)Ppad * H * sizeof(float), st));
  ICRL_CUDA(cudaMemsetAsync(stash_h, 0, H * sizeof(float), st));
  if (stash_c) ICRL_CUDA(cudaMemsetAsync(stash_c, 0, H * sizeof(float), st));
  a->P = P; a->Ppad = Ppad; a->steps = (int)(seg + warm); a->warm = warm; a->cp_half = cp_half_of(warm); a->seg = seg;
  a->stream = stream; a->table = table; a->b_hn = b_hn; a->stash_h = stash_h; a->stash_c = stash_c; a->stash_g = stash_g;
  a->state = state; a->hparts = hparts; a->wstate = cp_state; a->prof = g_chain_tc_prof; a->main_gain = 1.f + g_tc_bias[0];
  int rc;
  if ((rc = make_map_2d(mh, hparts, H, (long long)4 * Ppad, A_SLICE_ROWS))) return rc;
  // the stash stores as TMA tensor stores (g_tc_tma_store: experiment switch); a refused encode keeps the per-thread stores
  a->tma_store = 0;
  if (g_tc_tma_store) {
    const long long steps = seg + warm;
    int ok = make_map_stash(&m->sh, stash_h + H, H, steps, seg, P, 32) == ICRL_OK;
    if (kind == 0) {
      ok = ok && make_map_stash(&m->sc, stash_c + H, H, steps, seg, P, 32) == ICRL_OK;
      if (stash_g) ok = ok && make_map_stash(&m->sg, stash_g, 4 * H, steps, seg, P, 32) == ICRL_OK;
      else m->sg = m->sh;
    } else {
      m->sc = m->sh; m->sg = m->sh;
    }
    a->tma_store = ok ? 1 : 0;
  }
  if (!a->tma_store) { m->sh = *mh; m->sc = *mh; m->sg = *mh; }       // defined contents for the unused maps
  if (kind == 0) return make_map_3d(mw, packed, H, 4 * H, FwdCfg<4>::GN);
  return make_map_3d(mw, packed, H, 3 * H, FwdCfg<3>::GN);
}

int icrl_chain_tc_fwd_impl(cudaStream_t st, int kind, int P, long long seg, int warm, const int* stream,
                           const float* table, const void* packed, const float* b_hn, float* stash_h, float* stash_c,
                           float* stash_g, void* ws, float* cp_state, float* err) {
  FwdArgs a;
  FwdMaps m;
  int rc = fwd_setup(st, kind, P, seg, warm, stream, table, packed, b_hn, stash_h, stash_c, stash_g, ws, cp_state, err, &a, &m);
  if (rc) return rc;
  const int grid = CL * (a.Ppad / BM);
  if (kind == 0) {
    ICRL_CUDA(cudaFuncSetAttribute(chain_tc_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<4>::SMEM));
    chain_tc_fwd_kernel<4><<<dim3(grid), dim3(THREADS), FwdCfg<4>::SMEM, st>>>(m, a);
  } else {
    ICRL_CUDA(cudaFuncSetAttribute(chain_tc_fwd_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<3>::SMEM));
    chain_tc_fwd_kernel<3><<<dim3(grid), dim3(THREADS), FwdCfg<3>::SMEM, st>>>(m, a);
  }
  ICRL_LAUNCH_CHECK();
  chain_tc_check_fwd_kernel<<<dim3(P - 1, 2), H, 0, st>>>(P, seg, warm, a.cp_half, cp_state, stash_h, kind == 0 ? stash_c : nullptr, err);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

namespace {
// Piece 0 of an LSTM launch starts from (h0, c0) instead of zeros: what fwd_setup zeroed for it is overwritten with the
// state itself -- the fp16 hi/lo' split of h0 in row 0 of hparts buffer 0 (the A operand of kernel step 0, split exactly as
// the epilogue splits h for the next step), c0 in row 0 of the carried state, and stash rows 0.  A null pointer is zeros.
__global__ void chain_tc_seed_kernel(int Ppad, const float* __restrict__ h0, const float* __restrict__ c0, __half* hparts,
                                     float* state, float* stash_h, float* stash_c) {
  const int u = 4 * threadIdx.x;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 h4 = h0 ? *reinterpret_cast<const float4*>(h0 + u) : z;
  const float4 c4 = c0 ? *reinterpret_cast<const float4*>(c0 + u) : z;
  uint2 hi, lo;
  split4_f16(h4, hi, lo);
  *reinterpret_cast<uint2*>(hparts + u) = hi;
  *reinterpret_cast<uint2*>(hparts + (size_t)Ppad * H + u) = lo;
  *reinterpret_cast<float4*>(state + u) = c4;
  *reinterpret_cast<float4*>(stash_h + u) = h4;
  *reinterpret_cast<float4*>(stash_c + u) = c4;
}
}  // namespace

int icrl_chain_tc_lstm_fwd_from_impl(cudaStream_t st, int P, long long seg, int warm, const int* stream, const float* table,
                                     const void* packed, const float* h0, const float* c0, float* stash_h, float* stash_c,
                                     float* stash_g, void* ws, float* cp_state, float* err) {
  ICRL_REQUIRE(((reinterpret_cast<uintptr_t>(h0) | reinterpret_cast<uintptr_t>(c0)) & 15) == 0, "h0 / c0 must be 16-byte aligned");
  FwdArgs a;
  FwdMaps m;
  int rc = fwd_setup(st, 0, P, seg, warm, stream, table, packed, nullptr, stash_h, stash_c, stash_g, ws, cp_state, err, &a, &m);
  if (rc) return rc;
  if (h0 || c0) {
    chain_tc_seed_kernel<<<1, H / 4, 0, st>>>(a.Ppad, h0, c0, a.hparts, a.state, stash_h, stash_c);
    ICRL_LAUNCH_CHECK();
  }
  ICRL_CUDA(cudaFuncSetAttribute(chain_tc_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<4>::SMEM));
  chain_tc_fwd_kernel<4><<<dim3(CL * (a.Ppad / BM)), dim3(THREADS), FwdCfg<4>::SMEM, st>>>(m, a);
  ICRL_LAUNCH_CHECK();
  chain_tc_check_fwd_kernel<<<dim3(P - 1, 2), H, 0, st>>>(P, seg, warm, a.cp_half, cp_state, stash_h, stash_c, err);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// Both forward chains in one launch (chains_tc_fwd_fused_kernel): value LSTM with Pv pieces, reward GRU with Pr pieces.
int icrl_chains_tc_fwd_fused_impl(cudaStream_t st, int Pv, long long seg_v, int warm_v, const int* v_stream,
                                  const float* v_table, const void* v_packed, float* v_stash_h, float* v_stash_c,
                                  float* v_stash_g, void* v_ws, float* v_cp, float* v_err, int Pr, long long seg_r,
                                  int warm_r, const int* r_stream, const float* r_table, const void* r_packed,
                                  const float* r_b_hn, float* r_stash_h, void* r_ws, float* r_cp, float* r_err) {
  FwdArgs av, ar;
  FwdMaps mv, mr;
  int rc;
  if ((rc = fwd_setup(st, 0, Pv, seg_v, warm_v, v_stream, v_table, v_packed, nullptr, v_stash_h, v_stash_c, v_stash_g, v_ws,
                      v_cp, v_err, &av, &mv))) return rc;
  if ((rc = fwd_setup(st, 1, Pr, seg_r, warm_r, r_stream, r_table, r_packed, r_b_hn, r_stash_h, nullptr, nullptr, r_ws, r_cp,
                      r_err, &ar, &mr))) return rc;
  ar.prof = g_chain_tc_prof ? g_chain_tc_prof + 16 : nullptr;          // reward chain: slots [16..21]
  const int cv = av.Ppad / BM, cr = ar.Ppad / BM;
  constexpr int SMEM = FwdCfg<4>::SMEM > FwdCfg<3>::SMEM ? FwdCfg<4>::SMEM : FwdCfg<3>::SMEM;
  ICRL_CUDA(cudaFuncSetAttribute(chains_tc_fwd_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
  chains_tc_fwd_fused_kernel<<<dim3(CL * (cv + cr)), dim3(THREADS), SMEM, st>>>(mv, av, mr, ar, cv);
  ICRL_LAUNCH_CHECK();
  chain_tc_check_fwd_kernel<<<dim3(Pv - 1, 2), H, 0, st>>>(Pv, seg_v, warm_v, av.cp_half, v_cp, v_stash_h, v_stash_c, v_err);
  ICRL_LAUNCH_CHECK();
  chain_tc_check_fwd_kernel<<<dim3(Pr - 1, 2), H, 0, st>>>(Pr, seg_r, warm_r, ar.cp_half, r_cp, r_stash_h, nullptr, r_err);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

namespace {
int launch_bwd(cudaStream_t st, const __half* dgx, const __half* whhT, int Ppad, BwdArgs* a) {
  using Cfg = BwdCfg;
  // truncation bias of the tensor-core accumulation: g_tc_bias[1] is quoted for 128 chained MMAs (K = 2048); each K half
  // chains 64
  a->main_gain = 1.f + 0.5f * g_tc_bias[1];
  CUtensorMap mg, mw;
  int rc;
  if ((rc = make_map_2d(&mg, dgx, 4 * H, (long long)4 * Ppad, Cfg::SLICE_ROWS))) return rc;
  if ((rc = make_map_3d(&mw, whhT, 4 * H, H, Cfg::NCOL))) return rc;
  ICRL_CUDA(cudaFuncSetAttribute(chain_tc_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
  chain_tc_bwd_kernel<<<dim3(CL * (Ppad / BM)), dim3(THREADS), Cfg::SMEM, st>>>(mg, mw, *a);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}
}  // namespace

int icrl_chain_tc_lstm_bwd_impl(cudaStream_t st, int P, long long seg, int warm, const void* packed,
                                const float* stash_g, const float* stash_c, const int* take, const float* dh_take,
                                long long take_rows, void* dg_pair, long long pair_rows, float* dg_inv_scale, void* ws,
                                float* cp_state, float* err) {
  ICRL_REQUIRE(P >= 2 && seg >= 1 && warm >= 1, "chain pieces need P >= 2, seg >= 1, warm >= 1");
  ICRL_REQUIRE(packed && stash_g && stash_c && take && dh_take && dg_pair && dg_inv_scale && ws && cp_state && err, "null argument");
  ICRL_REQUIRE(pair_rows >= P * seg + warm && (reinterpret_cast<uintptr_t>(dg_pair) & 31) == 0, "gate-gradient pairs: too few rows or unaligned");
  const int Ppad = pad_pieces(P);
  __half* dgx = reinterpret_cast<__half*>(ws);
  const __half* whhT = reinterpret_cast<const __half*>(packed) + (size_t)2 * 4 * H * H;
  // err[4] = max |dh_take| (scale of the recurrence), err[5] = overflow flag
  ICRL_CUDA(cudaMemsetAsync(err + 4, 0, 2 * sizeof(float), st));
  absmax_kernel<<<148 * 2, 256, 0, st>>>(take_rows * H, dh_take, err + 4);
  ICRL_LAUNCH_CHECK();
  BwdArgs a;
  a.P = P; a.Ppad = Ppad; a.steps = (int)(seg + warm); a.warm = warm; a.cp_half = cp_half_of(warm);
  a.stride_k = seg; a.stride_t = 1; a.dh0_out = nullptr;
  a.stash_g = stash_g; a.stash_c = stash_c; a.take = take; a.dh_take = dh_take; a.dgates = nullptr; a.dgx = dgx;
  a.dg_pair = reinterpret_cast<__half*>(dg_pair); a.pair_rows = pair_rows; a.dg_inv_scale = dg_inv_scale;
  a.dh_max = err + 4; a.bstate = cp_state; a.overflow = err + 5; a.prof = g_chain_tc_prof ? g_chain_tc_prof + 8 : nullptr;
  int rc;
  if ((rc = launch_bwd(st, dgx, whhT, Ppad, &a))) return rc;
  chain_tc_check_bwd_kernel<<<dim3(P - 1, 2), H, 0, st>>>(P, a.cp_half, cp_state, err);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// ---- the policy's BPTT on the same kernel (trainers.py:479 through PolicyNetwork's LSTM, models.py:80): rows of the batch in
// the MMA M dimension, n_cell serial cell steps, the rollout's [step][row] stash, dL/dh injected at the sampled steps.
namespace {
__global__ void policy_take_kernel(int B, int n_cell, int p0, int* take) {
  const long long n = (long long)B * n_cell;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i / B), k = (int)(i % B);
    take[i] = t >= p0 - 1 ? (t - (p0 - 1)) * B + k : -1;
  }
}
}  // namespace

size_t icrl_policy_bptt_tc_ws_bytes_impl(int B, int n_cell) {
  return icrl_chain_tc_ws_bytes_impl(B) + (size_t)B * n_cell * sizeof(int) + 256;
}

// packed: icrl_pack_chain_tc_weights(kind 0) of the policy's W_hh.  Gs [n_cell][B][2048], Cs [(n_cell+1)][B][512],
// dHv [S][B][512] (S = n_cell - p0 + 1), DG [n_cell][B][2048] out, dh0 [B][512] out, err: 8 floats (err[4] = max |dHv|,
// err[5] = 1 on fp16 overflow of the exchange).
int icrl_policy_bptt_tc_impl(cudaStream_t st, int B, int n_cell, int p0, const void* packed, const float* Gs,
                             const float* Cs, const float* dHv, float* DG, float* dh0, void* ws, float* err) {
  ICRL_REQUIRE(B >= 1 && n_cell >= 1 && p0 >= 1 && n_cell >= p0, "bad rollout shape");
  ICRL_REQUIRE(packed && Gs && Cs && dHv && DG && dh0 && ws && err, "null argument");
  const int Ppad = pad_pieces(B);
  __half* dgx = reinterpret_cast<__half*>(ws);
  int* take = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + ((icrl_chain_tc_ws_bytes_impl(B) + 255) / 256) * 256);
  const __half* whhT = reinterpret_cast<const __half*>(packed) + (size_t)2 * 4 * H * H;
  const int S = n_cell - p0 + 1;
  ICRL_CUDA(cudaMemsetAsync(err + 4, 0, 2 * sizeof(float), st));
  absmax_kernel<<<148 * 2, 256, 0, st>>>((long long)S * B * H, dHv, err + 4);
  ICRL_LAUNCH_CHECK();
  policy_take_kernel<<<148, 256, 0, st>>>(B, n_cell, p0, take);
  ICRL_LAUNCH_CHECK();
  BwdArgs a;
  a.P = B; a.Ppad = Ppad; a.steps = n_cell; a.warm = 0; a.cp_half = -1;
  a.stride_k = 1; a.stride_t = B; a.dh0_out = dh0;
  a.stash_g = Gs; a.stash_c = Cs; a.take = take; a.dh_take = dHv; a.dgates = DG; a.dgx = dgx;
  a.dg_pair = nullptr; a.pair_rows = 0; a.dg_inv_scale = nullptr;
  a.dh_max = err + 4; a.bstate = nullptr; a.overflow = err + 5; a.prof = nullptr;
  int rc;
  if ((rc = launch_bwd(st, dgx, whhT, Ppad, &a))) return rc;
  return ICRL_OK;
}
