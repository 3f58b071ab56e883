// Weight-gradient contraction of the value chain on tcgen05 (SURVEY.md K14):
//   dW_hh[m][n] = sum_t dgates[t][m] * h_prev[t][n],   M = 2048, N = 512, K = T (number of serial steps, up to ~10^6).
// The operands are time-major ([T][M], [T][N]): the MMA reads them MN-major as they lie, as fp16 pairs x*s = hi + lo'/2048
// (22 mantissa bits) in planes [2][T][C].  The chain backward writes the gate gradients in that form itself
// (chain_tc.cu, pass (S): one power-of-two scale per launch, columns in the order of icrl_gate_pair_col); fp32 operands
// go through one elementwise pre-pass first:
//   1. column |max| of A over t  -> a power-of-two scale per row m of the result (gradients are ~1e-4 .. 1e-12 and
//      would fall into fp16 subnormals / underflow; h is in (-1, 1) and needs none)
//   2. split: [T][C] fp32 -> [2][T][C] fp16 (same layout, no transpose)
// GEMM: 128x128 tiles, split-K over gridDim.z, 3-stage TMA ring of 64-deep K blocks (SW128 boxes of 64 columns x 64 rows;
// rows past T are zero-filled by the tensor map), 2 MMAs per K step (hi * [hi | lo'] -> [main | correction], lo'*hi ->
// correction accumulator).  Because the tensor core truncates on every accumulate (gemm_tc.cu header), a TMEM accumulator
// only ever sums 512 K elements: after 8 K blocks the epilogue warps add main + correction/2048 into fp32 REGISTERS (round
// to nearest) while the MMAs continue in the second accumulator set.  Each split writes its partial tile; a last kernel
// sums the splits, undoes the scale and puts the rows in natural order.
#include <cuda.h>
#include <cuda_fp16.h>
#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 64, UMMA_K = 16, STAGES = 3;
constexpr int OP_TILE = 2 * BM * BK * 2;                   // hi + lo' of one operand: 32 KB
constexpr int STAGE_BYTES = 2 * OP_TILE;                   // 64 KB
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
constexpr int FLUSH_KB = 8;                                // K blocks per TMEM accumulation (512 K elements)
constexpr int TMEM_COLS = 512;                             // 2 sets x (main 128 + correction 128)
constexpr int THREADS = 192;
constexpr int CLN = 4;                                      // CTAs of a cluster: the 4 N tiles of one (M tile, split) share A
constexpr int A_SLICE_ROWS = BK / 2, A_SLICE = 64 * A_SLICE_ROWS * 2;    // 64 columns x 32 K rows = 4 KB per part and CTA
static_assert(CLN * A_SLICE == OP_TILE / 2, "the 4 CTAs of a cluster fetch one quarter of the A tile each");
constexpr float LO_INV = 1.f / 2048.f;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  for (unsigned spins = 0; spins < (1u << 27); ++spins) {
    unsigned ok;
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
  }
  __trap();
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_3d_mcast(unsigned dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned bar,
                                                  unsigned short mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_commit_mcast(unsigned bar, unsigned short mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ unsigned cluster_rank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
  unsigned pred;
  asm volatile("{\n.reg .pred P1;\nelect.sync _|P1, 0xffffffff;\nselp.u32 %0, 1, 0, P1;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(unsigned bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma(unsigned tmem_d, unsigned long long da, unsigned long long db, unsigned idesc,
                                       unsigned accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc),
      "r"(accumulate) : "memory");
}
// MN-major, 128B swizzle: atoms of 64 MN elements (128 bytes) x 8 K rows; LBO = 8 KB from one 64-column box to the next
// along MN, SBO = 1 KB from one group of 8 K rows to the next.  A K step of 16 advances the start by 2 KB.
constexpr unsigned BOX_BYTES = 64 * BK * 2;                // 64 columns x 64 K rows: 8 KB
__device__ __forceinline__ unsigned long long smem_desc(unsigned addr) {
  return (unsigned long long)((addr & 0x3FFFF) >> 4) | ((unsigned long long)(BOX_BYTES >> 4) << 16) | (64ull << 32) |
         (1ull << 46) | (2ull << 61);
}
constexpr unsigned long long DESC_K_STEP = UMMA_K * 128 / 16;
// F32 accumulate, fp16 x fp16, A and B MN-major (bits 15, 16), N = 128 / 256, M = 128
constexpr unsigned IDESC = (1u << 4) | (1u << 15) | (1u << 16) | ((unsigned)(BN >> 3) << 17) | ((unsigned)(BM >> 4) << 24);
constexpr unsigned IDESC2 = (1u << 4) | (1u << 15) | (1u << 16) | ((unsigned)(2 * BN >> 3) << 17) | ((unsigned)(BM >> 4) << 24);

__device__ __forceinline__ void tmem_ld32x2(unsigned ta, unsigned tb, float* a, float* b) {
  unsigned r[64];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%64];\n"
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, "
      "%47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%65];\n"
      "tcgen05.wait::ld.sync.aligned;\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]),
        "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]),
        "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]),
        "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]),
        "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(ta), "r"(tb)
      : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[32 + i]); }
}

// ------------------------------------------------------------------------------------------------ pre-passes
__global__ void col_absmax_kernel(long long T, int C, const float* __restrict__ X, int ldx, unsigned* __restrict__ mx) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const long long per = (T + gridDim.y - 1) / gridDim.y;
  const long long t0 = (long long)blockIdx.y * per, t1 = min(T, t0 + per);
  float m = 0.f;
  for (long long t = t0; t < t1; ++t) m = fmaxf(m, fabsf(X[(size_t)t * ldx + c]));
  atomicMax(mx + c, __float_as_uint(m));               // non-negative floats order like their bit patterns
}

// out [2][T][C] fp16 (hi plane, then lo' plane) <- X [T][C] fp32 (row stride ldx), elementwise and in place of the
// layout: x * s = hi + lo'/2048 with s = 2^-e for max|X[:,c]| in [2^(e-1), 2^e) (null mx: s = 1), inv_scale[c] = 2^e.
// Four columns per thread (C % 4 == 0); float4 loads when vec (ldx % 4 == 0 and a 16-byte aligned X).
__global__ void __launch_bounds__(256) split_kernel(long long T, int C, const float* __restrict__ X, int ldx, int vec,
                                                    const unsigned* __restrict__ mx, __half* __restrict__ out,
                                                    float* __restrict__ inv_scale) {
  const int C4 = C / 4;
  const long long total = T * C4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long t = i / C4;
    const int c = 4 * (int)(i - t * C4);
    const float* x = X + (size_t)t * ldx + c;
    float4 v = vec ? __ldg(reinterpret_cast<const float4*>(x)) : make_float4(__ldg(x), __ldg(x + 1), __ldg(x + 2), __ldg(x + 3));
    if (mx) {
      float s[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float m = __uint_as_float(mx[c + j]);
        int e = 0;
        if (m > 0.f) frexpf(m, &e);
        s[j] = exp2f((float)-e);
        if (t == 0) inv_scale[c + j] = exp2f((float)e);
      }
      v = make_float4(v.x * s[0], v.y * s[1], v.z * s[2], v.w * s[3]);
    }
    uint2 hi, lo;
    icrl_tc::split4_f16(v, hi, lo);
    *reinterpret_cast<uint2*>(out + (size_t)t * C + c) = hi;
    *reinterpret_cast<uint2*>(out + (size_t)(T + t) * C + c) = lo;
  }
}

// ------------------------------------------------------------------------------------------------ GEMM
// map_a / map_b: 3-D {columns, T, 2 parts}; boxes of 64 columns x 32 (A) / 64 (B) K rows.  partial [gridDim.z][M][N].
// Stage: A_hi [2 boxes of 64 columns][64 K], A_lo' likewise, then B as [hi, lo'][2 boxes][64 K], so that the four
// B boxes are the 256 columns [B_hi | B_lo'] of one instruction.
// The 4 CTAs of a cluster (the N tiles of one M tile and split) consume the same A tile: each fetches a quarter of it
// (one column box, one half of its K rows) and TMA-multicasts it to all four, so A crosses L2 -> SM once per cluster instead of once per CTA and the four
// stay in lockstep (a ring stage is refilled only after all four have consumed it).  (Also sharing the B tile between two
// M tiles -- clusters of 4 x 2 -- was measured and is slower: the 128 CTAs of the value chain's contraction are 16 clusters
// of 8, of which a B200 holds 15 at a time, so the last cluster runs as a second wave.)
__global__ void __cluster_dims__(CLN, 1, 1) __launch_bounds__(THREADS, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int M, int N,
             int kb_total, float* __restrict__ partial) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + STAGES * STAGE_BYTES);
  // bars: full[3], empty[3], acc_full[2], acc_empty[2]
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * STAGES + 4);
  const unsigned bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[STAGES]);
  const unsigned bar_acc_full = smem_u32(&bars[2 * STAGES]), bar_acc_empty = smem_u32(&bars[2 * STAGES + 2]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  // this split's K blocks
  const int per = (kb_total + gridDim.z - 1) / gridDim.z;
  const int kb0 = blockIdx.z * per, kb1 = min(kb_total, kb0 + per);
  const int nkb = max(kb1 - kb0, 0);
  const int nchunk = (nkb + FLUSH_KB - 1) / FLUSH_KB;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, CLN); }
    for (int s = 0; s < 2; ++s) { mbar_init(bar_acc_full + 8 * s, 1); mbar_init(bar_acc_empty + 8 * s, 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;
  const unsigned rank = cluster_rank();
  cluster_sync_all();                                       // every CTA's barriers exist before a peer multicasts into it

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES;
        mbar_wait(bar_empty + 8 * s, ((unsigned)(i / STAGES) & 1u) ^ 1u);      // all 4 CTAs have consumed the stage
        const unsigned full = bar_full + 8 * s;
        mbar_expect_tx(full, STAGE_BYTES);
        const unsigned base = smem_u32(smem + s * STAGE_BYTES);
        const unsigned a_dst = base + rank * A_SLICE;      // box rank >> 1, K rows [32 (rank & 1), +32)
        const int a_col = m0 + 64 * (int)(rank >> 1), a_k = (kb0 + i) * BK + A_SLICE_ROWS * (int)(rank & 1);
        tma_load_3d_mcast(a_dst, &map_a, a_col, a_k, 0, full, (unsigned short)0xF);
        tma_load_3d_mcast(a_dst + OP_TILE / 2, &map_a, a_col, a_k, 1, full, (unsigned short)0xF);
#pragma unroll
        for (int pb = 0; pb < 4; ++pb)                      // [hi, lo'] x [columns n0 .. +63, n0 + 64 .. +127]
          tma_load_3d(base + OP_TILE + pb * BOX_BYTES, &map_b, n0 + 64 * (pb & 1), (kb0 + i) * BK, pb >> 1, full);
      }
    }
  } else if (warp == 1) {
    for (int c = 0; c < nchunk; ++c) {
      const int set = c & 1;
      if (c >= 2) mbar_wait(bar_acc_empty + 8 * set, (unsigned)((c >> 1) - 1) & 1u);     // the flush of chunk c-2 drained this set
      tc_fence_after();
      const unsigned acc_main = tmem_base + (unsigned)set * 2 * BN, acc_corr = acc_main + BN;
      const int i0 = c * FLUSH_KB, i1 = min(nkb, i0 + FLUSH_KB);
      for (int i = i0; i < i1; ++i) {
        const int s = i % STAGES;
        mbar_wait(bar_full + 8 * s, (unsigned)(i / STAGES) & 1u);
        tc_fence_after();
        const unsigned base = smem_u32(smem + s * STAGE_BYTES);
        const unsigned long long dA0 = smem_desc(base), dA1 = smem_desc(base + OP_TILE / 2);
        const unsigned long long dB0 = smem_desc(base + OP_TILE);       // 256 columns: hi, then lo' (adjacent)
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const unsigned first = (i == i0 && k == 0) ? 0u : 1u;
            // [main | correction] = A_hi x [B_hi | B_lo'] in ONE N = 256 instruction (A_hi is read from shared memory once
            // instead of twice: operand reads + TMA fill bound this kernel, chain_tc.cu BwdCfg), then correction += A_lo' x B_hi
            tc_mma(acc_main, dA0 + DESC_K_STEP * k, dB0 + DESC_K_STEP * k, IDESC2, first);
            tc_mma(acc_corr, dA1 + DESC_K_STEP * k, dB0 + DESC_K_STEP * k, IDESC, 1u);
          }
          tc_commit_mcast(bar_empty + 8 * s, (unsigned short)0xF);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(bar_acc_full + 8 * set);
      __syncwarp();
    }
  } else {
    const int q = warp & 3;                                   // TMEM lane quarter of this warp
    const int row = m0 + 32 * q + lane;
    float acc[BN];
#pragma unroll
    for (int i = 0; i < BN; ++i) acc[i] = 0.f;
    for (int c = 0; c < nchunk; ++c) {
      const int set = c & 1;
      mbar_wait(bar_acc_full + 8 * set, (unsigned)(c >> 1) & 1u);
      tc_fence_after();
      const unsigned tl = tmem_base + ((unsigned)(32 * q) << 16) + (unsigned)set * 2 * BN;
#pragma unroll
      for (int g = 0; g < BN / 32; ++g) {
        float mv[32], cv[32];
        tmem_ld32x2(tl + 32 * g, tl + BN + 32 * g, mv, cv);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[32 * g + i] += fmaf(cv[i], LO_INV, mv[i]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * set);
    }
    if (row < M) {
      float* dst = partial + ((size_t)blockIdx.z * M + row) * N + n0;
#pragma unroll
      for (int i = 0; i < BN; i += 4)
        if (n0 + i + 3 < N) *reinterpret_cast<float4*>(dst + i) = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                       // nobody leaves while a peer may still multicast into it
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// C[row(m)][n] = inv_scale[m * scale_stride] * sum_s partial[s][m][n]; row(m) = m, or the natural gate column of stored
// column m for operands in the chain backward's order (permuted)
__global__ void wgrad_reduce_kernel(int M, int N, int S, const float* __restrict__ partial, const float* __restrict__ inv_scale,
                                    int scale_stride, int permuted, float* __restrict__ C, int ldc) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * N) return;
  const int m = (int)(i / N), n = (int)(i % N);
  float s = 0.f;
  for (int k = 0; k < S; ++k) s += partial[((size_t)k * M + m) * N + n];
  C[(size_t)(permuted ? icrl_gate_pair_natural(m) : m) * ldc + n] = s * inv_scale[(size_t)m * scale_stride];
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// planes [2][plane_rows][C] fp16, of which rows [0, T) are read; box: 64 columns x box_k rows of one plane
int make_map(CUtensorMap* map, const void* ptr, int C, long long T, long long plane_rows, int box_k) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void* q = nullptr;
    ICRL_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres));
    ICRL_REQUIRE(q && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, 2};
  const cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)plane_rows * C * 2};
  const cuuint32_t box[3] = {64, (cuuint32_t)box_k, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    icrl_set_error("cuTensorMapEncodeTiled (wgrad) failed with CUresult %d (C %d, T %lld)", (int)r, C, T);
    return ICRL_ERR_CUDA;
  }
  return ICRL_OK;
}

struct Ws {                                  // workspace of icrl_wgrad_tc_ws_bytes_impl(M, N, T, splits)
  __half* a;                                 // [2][T][M]
  __half* b;                                 // [2][T][N]
  float* partial;                            // [splits][M][N]
  unsigned* mx;                              // [M] column maxima of A
  float* inv_scale;                          // [M]
};
Ws carve(void* ws, int M, int N, long long T, int splits) {
  Ws w;
  w.a = reinterpret_cast<__half*>(ws);
  w.b = w.a + (size_t)2 * M * T;
  w.partial = reinterpret_cast<float*>(w.b + (size_t)2 * N * T);
  w.mx = reinterpret_cast<unsigned*>(w.partial + (size_t)splits * M * N);
  w.inv_scale = reinterpret_cast<float*>(w.mx + M);
  return w;
}

int split(cudaStream_t st, long long T, int C, const float* X, int ldx, const unsigned* mx, __half* out, float* inv_scale) {
  const int vec = ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0;
  const int blocks = (int)min((long long)148 * 8, (T * (C / 4) + 255) / 256);
  split_kernel<<<blocks, 256, 0, st>>>(T, C, X, ldx, vec, mx, out, inv_scale);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

// partial sums of A^T B for A planes [2][a_rows][M] and the B planes in the workspace, then the reduction into C
int contract(cudaStream_t st, int M, int N, long long T, const __half* a, long long a_rows, const Ws& w, int splits,
             const float* inv_scale, int scale_stride, int permuted, float* C, int ldc) {
  static bool attr_set = false;
  if (!attr_set) {
    ICRL_CUDA(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set = true;
  }
  CUtensorMap ma, mb;
  int rc;
  if ((rc = make_map(&ma, a, M, T, a_rows, A_SLICE_ROWS))) return rc;
  if ((rc = make_map(&mb, w.b, N, T, T, BK))) return rc;
  dim3 grid(N / BN, M / BM, splits);
  wgrad_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(ma, mb, M, N, icrl_cdiv(T, BK), w.partial);
  ICRL_LAUNCH_CHECK();
  wgrad_reduce_kernel<<<icrl_cdiv((long long)M * N, 256), 256, 0, st>>>(M, N, splits, w.partial, inv_scale, scale_stride,
                                                                        permuted, C, ldc);
  ICRL_LAUNCH_CHECK();
  return ICRL_OK;
}

}  // namespace

// workspace bytes for icrl_wgrad_tc_impl
size_t icrl_wgrad_tc_ws_bytes_impl(int M, int N, long long T, int splits) {
  return (size_t)4 * T * (M + N)             // hi + lo' of both operands, fp16
         + (size_t)splits * M * N * 4        // partial tiles
         + (size_t)M * 8 + 1024;             // column maxima + inverse scales (+ alignment)
}

// C [M][ldc] = A^T B with A [T][lda] (M columns used, scaled per column), B [T][ldb] (N columns used).
// The B operand's pre-pass alone (split into the workspace of the same M, N, T, splits): B is often final long before A
// (the value chain's h stash exists after the forward), so a caller can run this on another stream beside whatever
// produces A and then pass b_packed = 1 to the contraction.
int icrl_wgrad_tc_pack_b_impl(cudaStream_t st, int M, int N, long long T, const float* B, int ldb, void* ws, size_t ws_bytes,
                              int splits) {
  ICRL_REQUIRE(M % BM == 0 && N % (BN * CLN) == 0 && T > 0 && splits >= 1, "wgrad_tc needs M a multiple of 128, N of 512");
  ICRL_REQUIRE(ws && ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(M, N, T, splits), "wgrad_tc workspace too small");
  return split(st, T, N, B, ldb, nullptr, carve(ws, M, N, T, splits).b, nullptr);
}

// colmax (nullable): M words holding the bit patterns of max_t |A[t][m]| when the caller has them already (the gate-table
// scatter reads all of A and returns them: icrl_scatter_add_stream); otherwise a pre-pass over A computes them.
// b_packed: the B operand already lies in the workspace (icrl_wgrad_tc_pack_b_impl).
int icrl_wgrad_tc_impl(cudaStream_t st, int M, int N, long long T, const float* A, int lda, const float* B, int ldb,
                       float* C, int ldc, void* ws, size_t ws_bytes, int splits, const unsigned* colmax, int b_packed) {
  ICRL_REQUIRE(M % BM == 0 && N % (BN * CLN) == 0 && T > 0 && splits >= 1, "wgrad_tc needs M a multiple of 128, N of 512");
  ICRL_REQUIRE(ws && ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(M, N, T, splits), "wgrad_tc workspace too small");
  const Ws w = carve(ws, M, N, T, splits);
  const unsigned* mx = colmax;
  if (!mx) {
    ICRL_CUDA(cudaMemsetAsync(w.mx, 0, (size_t)M * sizeof(unsigned), st));
    dim3 grid(icrl_cdiv(M, 128), (unsigned)min((long long)592, (T + 255) / 256));
    col_absmax_kernel<<<grid, 128, 0, st>>>(T, M, A, lda, w.mx);
    ICRL_LAUNCH_CHECK();
    mx = w.mx;
  }
  int rc;
  if ((rc = split(st, T, M, A, lda, mx, w.a, w.inv_scale))) return rc;
  if (!b_packed && (rc = split(st, T, N, B, ldb, nullptr, w.b, nullptr))) return rc;
  return contract(st, M, N, T, w.a, T, w, splits, w.inv_scale, 1, 0, C, ldc);
}

// dW_hh [2048][ldc] from the chain backward's gate-gradient pairs: planes [2][pair_rows][2048] in the column order of
// icrl_gate_pair_col, scaled by the power of two whose inverse is the device word *inv_scale; B [T][ldb] as above.
int icrl_wgrad_tc_gate_pairs_impl(cudaStream_t st, int N, long long T, const void* pairs, long long pair_rows,
                                  const float* inv_scale, const float* B, int ldb, float* C, int ldc, void* ws,
                                  size_t ws_bytes, int splits, int b_packed) {
  constexpr int M = 4 * ICRL_H;
  ICRL_REQUIRE(N % (BN * CLN) == 0 && T > 0 && T <= pair_rows && splits >= 1, "wgrad_tc gate pairs: bad shape");
  ICRL_REQUIRE(pairs && inv_scale && (reinterpret_cast<uintptr_t>(pairs) & 15) == 0, "wgrad_tc gate pairs: bad pointer");
  ICRL_REQUIRE(ws && ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(M, N, T, splits), "wgrad_tc workspace too small");
  const Ws w = carve(ws, M, N, T, splits);
  int rc;
  if (!b_packed && (rc = split(st, T, N, B, ldb, nullptr, w.b, nullptr))) return rc;
  return contract(st, M, N, T, reinterpret_cast<const __half*>(pairs), pair_rows, w, splits, inv_scale, 0, 1, C, ldc);
}
