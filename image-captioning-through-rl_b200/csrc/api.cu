// extern "C" surface of libicrl_b200.so (declared in include/icrl_b200.h) and the per-phase drivers
// that sequence the kernels of the policy rollout and the parameter-gradient contractions.
#include <stdarg.h>
#include <string.h>
#include "../../include/icrl_b200.h"
#include "internal.h"

static thread_local char g_err[512] = "";

void icrl_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

#define TRY(x)                     \
  do {                             \
    int rc__ = (x);                \
    if (rc__ != ICRL_OK) return rc__; \
  } while (0)

static inline cudaStream_t S_(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline void bump(int* l, int n) { if (l) *l += n; }
constexpr int H = ICRL_H;

extern "C" {

const char* icrl_last_error(void) { return g_err; }
int icrl_version(void) { return 100; }

int icrl_device_info(int* out4) {
  int dev = 0;
  ICRL_CUDA(cudaGetDevice(&dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&out4[0], cudaDevAttrMultiProcessorCount, dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&out4[1], cudaDevAttrComputeCapabilityMajor, dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&out4[2], cudaDevAttrComputeCapabilityMinor, dev));
  ICRL_CUDA(cudaDeviceGetAttribute(&out4[3], cudaDevAttrCooperativeLaunch, dev));
  return ICRL_OK;
}

int icrl_gemm_f32(void* stream, int transA, int transB, int M, int N, int K, const float* A, int lda,
                  const float* B, int ldb, float* C, int ldc, const float* bias, float beta, float* ws,
                  size_t ws_bytes, int* launches) {
  return icrl_gemm_f32_impl(S_(stream), transA, transB, M, N, K, A, lda, B, ldb, C, ldc, bias, beta, ws, ws_bytes,
                            launches);
}

int icrl_pack_gate_table(void* stream, int V, int G, int fold, int D, const float* E, const float* W_ih,
                         const float* b_ih, const float* b_hh, float* table, int* launches) {
  // table = E [V][D] * W_ih^T ([G][D], K contiguous); D = embedding width (512, or that of frozen pretrained vectors)
  ICRL_REQUIRE(D > 0, "embedding width");
  TRY(icrl_gemm_f32_impl(S_(stream), 0, 1, V, G, D, E, D, W_ih, D, table, G, nullptr, 0.f, nullptr, 0, launches));
  TRY(icrl_add_gate_bias_impl(S_(stream), V, G, fold, b_ih, b_hh, table));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_pack_value_head(void* stream, const float* W1, const float* b1, const float* W2, const float* b2,
                         float* w_eff, float* b_eff, int* launches) {
  TRY(icrl_pack_value_head_impl(S_(stream), W1, b1, W2, b2, w_eff, b_eff));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_policy_rollout_fwd(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                            const float* W_cnn, const float* b_cnn, const float* table, const float* W_hh,
                            const float* W_v, const float* b_v, const double* uniforms, const long long* forced,
                            int* tokcm, long long* tokens_out, float* logp, float* Hs, float* Cs, float* Gs, float* logits,
                            float* gpre, int* launches) {
  ICRL_REQUIRE(B > 0 && V > 0 && p0 >= 1 && S >= 1, "bad rollout shape");
  ICRL_REQUIRE(greedy || uniforms || forced, "sampling needs uniforms");
  cudaStream_t st = S_(stream);
  const int n_cell = p0 - 1 + S;
  const size_t BH = (size_t)B * H;
  // h0 = cnn2linear(features), c0 = 0   (models.py:75-78)
  TRY(icrl_gemm_f32_impl(st, 0, 1, B, H, H, features, H, W_cnn, H, Hs, H, b_cnn, 0.f, nullptr, 0, launches));
  ICRL_CUDA(cudaMemsetAsync(Cs, 0, BH * sizeof(float), st));
  for (int j = 0; j < n_cell; ++j) {
    // recurrent half of the gates: h_{j-1} W_hh^T ; input half comes from the gate table
    TRY(icrl_gemm_f32_impl(st, 0, 1, B, 4 * H, H, Hs + j * BH, H, W_hh, H, gpre, 4 * H, nullptr, 0.f, nullptr, 0,
                           launches));
    TRY(icrl_lstm_pointwise_fwd(st, B, gpre, table, tokcm + (size_t)j * B, Cs + j * BH, Gs + (size_t)j * B * 4 * H,
                                Cs + (j + 1) * BH, Hs + (j + 1) * BH));
    bump(launches, 1);
    const int s = j - (p0 - 1);
    if (s >= 0) {
      float* lg = logits + (size_t)s * B * V;
      TRY(icrl_gemm_f32_impl(st, 0, 1, B, V, H, Hs + (j + 1) * BH, H, W_v, H, lg, V, b_v, 0.f, nullptr, 0, launches));
      TRY(icrl_softmax_sample(st, B, V, lg, V, (greedy || !uniforms) ? nullptr : uniforms + (size_t)s * B, greedy, forced,
                              tokcm + (size_t)(p0 + s) * B, tokens_out, logp, S, s, nullptr));
      bump(launches, 1);
    }
  }
  return ICRL_OK;
}

int icrl_split_bf16x3(void* stream, long long n, const float* x, void* parts, int* launches) {
  TRY(icrl_split_bf16x3_impl(S_(stream), n, x, parts));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_gemm_bf16x3(void* stream, int M, int N, int K, const void* a_parts, const void* b_parts, float* C, int ldc,
                     const float* bias, int* launches) {
  TRY(icrl_gemm_bf16x3_impl(S_(stream), M, N, K, a_parts, b_parts, C, ldc, bias));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_policy_rollout_fwd_tc(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                               const float* W_cnn, const float* b_cnn, const float* table, const void* whh_parts,
                               const void* wv_parts, const float* b_v, const double* uniforms,
                               const long long* forced, int* tokcm, long long* tokens_out, float* logp, float* Hs,
                               float* Cs, float* Gs, float* logits, float* gpre, void* h_parts, int* launches) {
  ICRL_REQUIRE(B > 0 && V > 0 && p0 >= 1 && S >= 1, "bad rollout shape");
  ICRL_REQUIRE(greedy || uniforms || forced, "sampling needs uniforms");
  cudaStream_t st = S_(stream);
  const int n_cell = p0 - 1 + S;
  const size_t BH = (size_t)B * H;
  TRY(icrl_gemm_f32_impl(st, 0, 1, B, H, H, features, H, W_cnn, H, Hs, H, b_cnn, 0.f, nullptr, 0, launches));
  ICRL_CUDA(cudaMemsetAsync(Cs, 0, BH * sizeof(float), st));
  TRY(icrl_split_bf16x3_impl(st, (long long)BH, Hs, h_parts));
  bump(launches, 1);
  for (int j = 0; j < n_cell; ++j) {
    TRY(icrl_gemm_bf16x3_impl(st, B, 4 * H, H, h_parts, whh_parts, gpre, 4 * H, nullptr));
    TRY(icrl_lstm_pointwise_fwd(st, B, gpre, table, tokcm + (size_t)j * B, Cs + j * BH, Gs + (size_t)j * B * 4 * H,
                                Cs + (j + 1) * BH, Hs + (j + 1) * BH));
    TRY(icrl_split_bf16x3_impl(st, (long long)BH, Hs + (j + 1) * BH, h_parts));
    bump(launches, 3);
    const int s = j - (p0 - 1);
    if (s >= 0) {
      float* lg = logits + (size_t)s * B * V;
      TRY(icrl_gemm_bf16x3_impl(st, B, V, H, h_parts, wv_parts, lg, V, b_v));
      TRY(icrl_softmax_sample(st, B, V, lg, V, (greedy || !uniforms) ? nullptr : uniforms + (size_t)s * B, greedy, forced,
                              tokcm + (size_t)(p0 + s) * B, tokens_out, logp, S, s, nullptr));
      bump(launches, 2);
    }
  }
  return ICRL_OK;
}

int icrl_decode_set_profile(void* buf) { icrl_decode_set_profile_impl(reinterpret_cast<long long*>(buf)); return ICRL_OK; }

size_t icrl_wgrad_tc_ws_bytes(int M, int N, long long T, int splits) { return icrl_wgrad_tc_ws_bytes_impl(M, N, T, splits); }

int icrl_wgrad_tc(void* stream, int M, int N, long long T, const float* A, int lda, const float* B, int ldb, float* C,
                  int ldc, void* ws, size_t ws_bytes, int splits, int* launches) {
  TRY(icrl_wgrad_tc_impl(S_(stream), M, N, T, A, lda, B, ldb, C, ldc, ws, ws_bytes, splits));
  bump(launches, 5);
  return ICRL_OK;
}

int icrl_wgrad_tc_pack_b(void* stream, int M, int N, long long T, const float* B, int ldb, void* ws, size_t ws_bytes,
                         int splits, int* launches) {
  TRY(icrl_wgrad_tc_pack_b_impl(S_(stream), M, N, T, B, ldb, ws, ws_bytes, splits));
  bump(launches, 1);
  return ICRL_OK;
}

size_t icrl_decode_weight_halves(void) { return icrl_decode_weight_halves_impl(); }

int icrl_pack_decode_weights(void* stream, int V, const float* W_hh, const float* W_v, void* packed, int* launches) {
  TRY(icrl_pack_decode_weights_impl(S_(stream), V, W_hh, W_v, packed));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_policy_rollout_fwd_fused(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                                  const float* W_cnn, const float* b_cnn, const float* table, const void* packed,
                                  const float* b_v, const double* uniforms, const long long* forced, int* tokcm,
                                  long long* tokens_out, float* logp, float* Hs, float* Cs, float* Gs, float* logits,
                                  float* last_logits, void* hparts, int* launches) {
  cudaStream_t st = S_(stream);
  // h0 = cnn2linear(features), c0 = 0   (models.py:75-78)
  TRY(icrl_gemm_f32_impl(st, 0, 1, B, H, H, features, H, W_cnn, H, Hs, H, b_cnn, 0.f, nullptr, 0, launches));
  ICRL_CUDA(cudaMemsetAsync(Cs, 0, (size_t)B * H * sizeof(float), st));
  TRY(icrl_policy_decode_impl(st, B, V, p0, S, greedy, table, packed, b_v, uniforms, forced, tokcm, tokens_out, logp,
                              Hs, Cs, Gs, logits, last_logits, hparts));
  bump(launches, 2);                       // h split + the persistent decode kernel
  return ICRL_OK;
}

// ---- direction-agnostic teacher-forced LSTM sequence (bidirectional policy variant, models.py:59-78: each direction
//      is one call; the caller reverses the token columns for the reverse direction).
int icrl_lstm_seq_fwd(void* stream, int B, int n, const float* h0, const int* tokcm, const float* table,
                      const float* W_hh, float* Hs, float* Cs, float* Gs, float* gpre, int* launches) {
  ICRL_REQUIRE(B > 0 && n > 0, "bad sequence shape");
  cudaStream_t st = S_(stream);
  const size_t BH = (size_t)B * H;
  ICRL_CUDA(cudaMemcpyAsync(Hs, h0, BH * sizeof(float), cudaMemcpyDeviceToDevice, st));
  ICRL_CUDA(cudaMemsetAsync(Cs, 0, BH * sizeof(float), st));
  for (int j = 0; j < n; ++j) {
    TRY(icrl_gemm_f32_impl(st, 0, 1, B, 4 * H, H, Hs + j * BH, H, W_hh, H, gpre, 4 * H, nullptr, 0.f, nullptr, 0, launches));
    TRY(icrl_lstm_pointwise_fwd(st, B, gpre, table, tokcm + (size_t)j * B, Cs + j * BH, Gs + (size_t)j * B * 4 * H,
                                Cs + (j + 1) * BH, Hs + (j + 1) * BH));
    bump(launches, 1);
  }
  return ICRL_OK;
}

// dH [n][B][512] = dL/d(h after cell j).  Outputs (overwritten): dh0 [B][512], dE [V][D] (nullable), dW_ih [2048][D],
// dW_hh [2048][512], db_ih, db_hh [2048].  Workspaces as icrl_policy_rollout_bwd.
int icrl_lstm_seq_bwd(void* stream, int B, int n, int V, int D, const int* tokcm, const float* Hs, const float* Cs,
                      const float* Gs, const float* dH, const float* W_hh, const float* E, const float* W_ih, float* DG,
                      float* dh, float* dc, float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes,
                      float* dh0, float* dE, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh, int* launches) {
  ICRL_REQUIRE(B > 0 && n > 0, "bad sequence shape");
  cudaStream_t st = S_(stream);
  const size_t BH = (size_t)B * H;
  float* dh_cur = dh;
  float* dh_nxt = dh + BH;
  ICRL_CUDA(cudaMemsetAsync(dh_cur, 0, BH * sizeof(float), st));
  ICRL_CUDA(cudaMemsetAsync(dc, 0, BH * sizeof(float), st));
  for (int j = n - 1; j >= 0; --j) {
    float* dg = DG + (size_t)j * B * 4 * H;
    TRY(icrl_lstm_pointwise_bwd(st, B, dh_cur, dH + (size_t)j * BH, dc, Gs + (size_t)j * B * 4 * H, Cs + j * BH,
                                Cs + (j + 1) * BH, dg));
    bump(launches, 1);
    TRY(icrl_gemm_f32_impl(st, 0, 0, B, H, 4 * H, dg, 4 * H, W_hh, H, dh_nxt, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
    float* t = dh_cur; dh_cur = dh_nxt; dh_nxt = t;
  }
  ICRL_CUDA(cudaMemcpyAsync(dh0, dh_cur, BH * sizeof(float), cudaMemcpyDeviceToDevice, st));
  const long long nB = (long long)n * B;
  TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, H, (int)nB, DG, 4 * H, Hs, H, dW_hh, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  ICRL_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * 4 * H * sizeof(float), st));
  TRY(icrl_scatter_add_rows(st, nB, 4 * H, DG, tokcm, dtable));
  bump(launches, 1);
  TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, D, V, dtable, 4 * H, E, D, dW_ih, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  if (dE) TRY(icrl_gemm_f32_impl(st, 0, 0, V, D, 4 * H, dtable, 4 * H, W_ih, D, dE, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  TRY(icrl_wcolsum(st, V, 4 * H, dtable, nullptr, 0, colsum_ws, db_ih));
  bump(launches, 2);
  ICRL_CUDA(cudaMemcpyAsync(db_hh, db_ih, 4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return ICRL_OK;
}

size_t icrl_colsum_ws_floats(long long rows, int cols) { return (size_t)icrl_wcolsum_chunks(rows) * cols; }

}  // extern "C"

// tc_packed != NULL: the serial part (step 4) runs as ONE launch of the tcgen05 chain-backward kernel (chain_tc.cu).
static int policy_rollout_bwd_common(void* stream, int B, int V, int p0, int S, int D, const float* features, const float* E,
                            const float* W_ih, const float* W_hh, const float* W_v, const int* tokcm,
                            const long long* tokens_out, const float* dlogp, const float* Hs, const float* Cs,
                            const float* Gs, float* logits, float* dHv, float* DG, float* dh, float* dc,
                            float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE,
                            float* dW_cnn, float* db_cnn, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh,
                            float* dW_v, float* db_v, const void* tc_packed, void* tc_ws, float* tc_err, int ldz,
                            int* launches) {
  // ldz: row stride of `logits` / dL/dlogits.  tc path: ldz = ICRL_VPAD (1024) with zero padding columns, so that the two
  // vocabulary-sized contractions run on tcgen05 as well (dW_v: K = S*B on wgrad_tc; dHv: bf16x3 GEMM with K = ldz).
  cudaStream_t st = S_(stream);
  const int n_cell = p0 - 1 + S;
  const size_t BH = (size_t)B * H;
  const int SB = S * B;
  // 1. dL/dlogits in place (log(softmax(z))[a] backward); dlogp == NULL: `logits` already holds dL/dlogits
  if (dlogp) {
    TRY(icrl_softmax_bwd(st, B, S, V, logits, ldz, tokens_out, dlogp));
    bump(launches, 1);
  }
  const float* dZ = logits;
  const float* Hsel = Hs + (size_t)p0 * BH;          // h after cell step p0-1+s, s = 0..S-1
  const bool tc_vocab = tc_packed && ldz == ICRL_VPAD && V <= ICRL_VPAD &&
                        gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(ICRL_VPAD, H, SB, 2);
  if (tc_vocab) {
    char* w2 = reinterpret_cast<char*>(tc_ws) + ((icrl_policy_bptt_tc_ws_bytes_impl(B, n_cell) + 255) / 256) * 256;
    void* zparts = w2;                                               // [3][SB][1024] bf16
    void* wvT = w2 + (size_t)3 * SB * ICRL_VPAD * 2;                 // [3][512][1024] bf16
    float* dWv_tmp = reinterpret_cast<float*>(reinterpret_cast<char*>(wvT) + (size_t)3 * H * ICRL_VPAD * 2);   // [1024][512]
    float* dbv_tmp = dWv_tmp + (size_t)ICRL_VPAD * H;                // [1024]
    // 2. vocab projection gradients: dW_v = dZ^T Hsel (K = S*B) on wgrad_tc, rows >= V of the padded result dropped
    TRY(icrl_wgrad_tc_impl(st, ICRL_VPAD, H, SB, dZ, ldz, Hsel, H, dWv_tmp, H, gemm_ws, gemm_ws_bytes, 2));
    ICRL_CUDA(cudaMemcpyAsync(dW_v, dWv_tmp, (size_t)V * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    TRY(icrl_wcolsum(st, SB, ICRL_VPAD, dZ, nullptr, 0, colsum_ws, dbv_tmp));
    ICRL_CUDA(cudaMemcpyAsync(db_v, dbv_tmp, (size_t)V * sizeof(float), cudaMemcpyDeviceToDevice, st));
    bump(launches, 7);
    // 3. dL/dh from the vocab path, all steps at once: dHv = dZ W_v as a 3-part bf16 split product (fp32-grade)
    TRY(icrl_split_bf16x3_impl(st, (long long)SB * ICRL_VPAD, dZ, zparts));
    TRY(icrl_pack_transposed_bf16x3_impl(st, V, H, ICRL_VPAD, W_v, wvT));
    TRY(icrl_gemm_bf16x3_impl(st, SB, H, ICRL_VPAD, zparts, wvT, dHv, H, nullptr));
    bump(launches, 3);
  } else {
    // 2. vocab projection gradients
    TRY(icrl_gemm_f32_impl(st, 1, 0, V, H, SB, dZ, ldz, Hsel, H, dW_v, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
    if (ldz == V) {
      TRY(icrl_wcolsum(st, SB, V, dZ, nullptr, 0, colsum_ws, db_v));
    } else {
      float* tmp = colsum_ws + (size_t)icrl_wcolsum_chunks(SB) * ldz;
      TRY(icrl_wcolsum(st, SB, ldz, dZ, nullptr, 0, colsum_ws, tmp));
      ICRL_CUDA(cudaMemcpyAsync(db_v, tmp, (size_t)V * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    bump(launches, 2);
    // 3. dL/dh from the vocab path, all steps at once
    TRY(icrl_gemm_f32_impl(st, 0, 0, SB, H, V, dZ, ldz, W_v, H, dHv, H, nullptr, 0.f, nullptr, 0, launches));
  }
  // 4. BPTT
  float* dh_cur = dh;
  float* dh_nxt = dh + BH;
  if (tc_packed) {
    TRY(icrl_policy_bptt_tc_impl(st, B, n_cell, p0, tc_packed, Gs, Cs, dHv, DG, dh_cur, tc_ws, tc_err));
    bump(launches, 3);                     // |dHv| maximum, the injection map, the persistent cluster kernel
  } else {
    ICRL_CUDA(cudaMemsetAsync(dh_cur, 0, BH * sizeof(float), st));
    ICRL_CUDA(cudaMemsetAsync(dc, 0, BH * sizeof(float), st));
    for (int j = n_cell - 1; j >= 0; --j) {
      const int s = j - (p0 - 1);
      float* dg = DG + (size_t)j * B * 4 * H;
      TRY(icrl_lstm_pointwise_bwd(st, B, dh_cur, s >= 0 ? dHv + (size_t)s * BH : nullptr, dc,
                                  Gs + (size_t)j * B * 4 * H, Cs + j * BH, Cs + (j + 1) * BH, dg));
      bump(launches, 1);
      TRY(icrl_gemm_f32_impl(st, 0, 0, B, H, 4 * H, dg, 4 * H, W_hh, H, dh_nxt, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
      float* t = dh_cur; dh_cur = dh_nxt; dh_nxt = t;
    }
  }
  // dh_cur = dL/dh0
  // 5. recurrent weight gradient: DG^T [2048 x nB] * H_prev [nB x 512]
  const long long nB = (long long)n_cell * B;
  if (gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(4 * H, H, nB, 2)) {       // tcgen05 (wgrad_tc.cu) when the workspace allows
    TRY(icrl_wgrad_tc_impl(st, 4 * H, H, nB, DG, 4 * H, Hs, H, dW_hh, H, gemm_ws, gemm_ws_bytes, 2));
    bump(launches, 5);
  } else {
    TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, H, (int)nB, DG, 4 * H, Hs, H, dW_hh, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes,
                           launches));
  }
  // 6. gate-table gradient, then its factors
  ICRL_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * 4 * H * sizeof(float), st));
  TRY(icrl_scatter_add_rows(st, nB, 4 * H, DG, tokcm, dtable));
  bump(launches, 1);
  TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, D, V, dtable, 4 * H, E, D, dW_ih, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  if (dE)                                            // null: frozen pretrained embedding (models.py:61-63)
    TRY(icrl_gemm_f32_impl(st, 0, 0, V, D, 4 * H, dtable, 4 * H, W_ih, D, dE, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  TRY(icrl_wcolsum(st, V, 4 * H, dtable, nullptr, 0, colsum_ws, db_ih));
  bump(launches, 2);
  ICRL_CUDA(cudaMemcpyAsync(db_hh, db_ih, 4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // 7. cnn2linear
  TRY(icrl_gemm_f32_impl(st, 1, 0, H, H, B, dh_cur, H, features, H, dW_cnn, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  TRY(icrl_wcolsum(st, B, H, dh_cur, nullptr, 0, colsum_ws, db_cnn));
  bump(launches, 2);
  return ICRL_OK;
}

extern "C" {

int icrl_policy_rollout_bwd(void* stream, int B, int V, int p0, int S, int D, const float* features, const float* E,
                            const float* W_ih, const float* W_hh, const float* W_v, const int* tokcm,
                            const long long* tokens_out, const float* dlogp, const float* Hs, const float* Cs,
                            const float* Gs, float* logits, float* dHv, float* DG, float* dh, float* dc,
                            float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE,
                            float* dW_cnn, float* db_cnn, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh,
                            float* dW_v, float* db_v, int* launches) {
  return policy_rollout_bwd_common(stream, B, V, p0, S, D, features, E, W_ih, W_hh, W_v, tokcm, tokens_out, dlogp, Hs, Cs, Gs,
                                   logits, dHv, DG, dh, dc, dtable, colsum_ws, gemm_ws, gemm_ws_bytes, dE, dW_cnn, db_cnn, dW_ih,
                                   dW_hh, db_ih, db_hh, dW_v, db_v, nullptr, nullptr, nullptr, V, launches);
}

size_t icrl_policy_bwd_tc_ws_bytes(int B, int S, int n_cell) {
  const size_t SB = (size_t)S * B;
  return ((icrl_policy_bptt_tc_ws_bytes_impl(B, n_cell) + 255) / 256) * 256 + 3 * SB * ICRL_VPAD * 2 + (size_t)3 * H * ICRL_VPAD * 2 +
         (size_t)ICRL_VPAD * H * 4 + ICRL_VPAD * 4 + 256;
}
int icrl_vocab_pad(void) { return ICRL_VPAD; }

int icrl_policy_rollout_bwd_tc(void* stream, int B, int V, int p0, int S, int D, const float* features, const float* E,
                               const float* W_ih, const float* W_hh, const float* W_v, const int* tokcm,
                               const long long* tokens_out, const float* dlogp, const float* Hs, const float* Cs,
                               const float* Gs, float* logits, float* dHv, float* DG, float* dh, float* dc,
                               float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE,
                               float* dW_cnn, float* db_cnn, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh,
                               float* dW_v, float* db_v, const void* tc_packed, void* tc_ws, float* tc_err, int ldz,
                               int* launches) {
  ICRL_REQUIRE(tc_packed && tc_ws && tc_err, "the tcgen05 BPTT needs the packed W_hh, its workspace and the error words");
  ICRL_REQUIRE(ldz >= V, "row stride of the logits");
  return policy_rollout_bwd_common(stream, B, V, p0, S, D, features, E, W_ih, W_hh, W_v, tokcm, tokens_out, dlogp, Hs, Cs, Gs,
                                   logits, dHv, DG, dh, dc, dtable, colsum_ws, gemm_ws, gemm_ws_bytes, dE, dW_cnn, db_cnn, dW_ih,
                                   dW_hh, db_ih, db_hh, dW_v, db_v, tc_packed, tc_ws, tc_err, ldz, launches);
}

long long icrl_stream_len(int B, int p0, int S, int extra) {
  return (long long)B * ((long long)S * (p0 + extra) + (long long)S * (S - 1) / 2);
}

int icrl_build_stream(void* stream, int B, int p0, int S, int extra, const int* tokcm, int* stream_out, int* take,
                      int* take_pos, int* launches) {
  ICRL_REQUIRE(icrl_stream_len(B, p0, S, extra) < (1ll << 31), "token stream longer than 2^31");
  TRY(icrl_build_stream_impl(S_(stream), B, p0, S, extra, tokcm, stream_out, take, take_pos));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_build_stream_sharded(void* stream, int B, int p0, int S, int extra, int shards, const int* tokcm,
                              int* stream_out, int* take, int* take_pos, int* launches) {
  ICRL_REQUIRE(shards >= 1 && B % shards == 0, "the batch must split evenly into chain shards");
  ICRL_REQUIRE(icrl_stream_len(B / shards, p0, S, extra) + 1 < (1ll << 31) / shards, "token stream longer than 2^31");
  TRY(icrl_build_stream_sharded_impl(S_(stream), B, p0, S, extra, shards, tokcm, stream_out, take, take_pos));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chains_fwd_fused_sharded(void* stream, int shards, const int* v_stream, int v_T, const float* v_table,
                                  const float* v_W_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                                  const int* r_stream, int r_T, const float* r_table, const float* r_W_hh,
                                  const float* r_b_hn, float* r_stash_h, void* sync_state, int* launches) {
  TRY(icrl_chains_fwd_fused_batched_impl(S_(stream), shards, v_stream, v_T, v_table, v_W_hh, v_stash_h, v_stash_c,
                                         v_stash_gates, r_stream, r_T, r_table, r_W_hh, r_b_hn, r_stash_h, sync_state));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_lstm_bwd_sharded(void* stream, int shards, int T, const float* W_hh, const float* stash_gates,
                                const float* stash_c, const int* take, const float* dh_take, float* dgates,
                                void* sync_state, int* launches) {
  TRY(icrl_chain_lstm_bwd_batched_impl(S_(stream), shards, T, W_hh, stash_gates, stash_c, take, dh_take, dgates,
                                       sync_state));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_tc_max_pieces(void) { return icrl_chain_tc_max_pieces_impl(); }
size_t icrl_chain_tc_weight_halves(int kind) { return icrl_chain_tc_weight_halves_impl(kind); }
size_t icrl_chain_tc_ws_bytes(int pieces) { return icrl_chain_tc_ws_bytes_impl(pieces); }
size_t icrl_chain_tc_cp_floats(int pieces) { return icrl_chain_tc_cp_floats_impl(pieces); }
int icrl_chain_tc_set_tma_store(int on) { icrl_chain_tc_set_tma_store_impl(on); return ICRL_OK; }
int icrl_chain_tc_bwd_max_pieces(void) { return icrl_chain_tc_bwd_max_pieces_impl(); }
int icrl_chain_tc_set_bias(float fwd, float bwd) { icrl_chain_tc_set_bias_impl(fwd, bwd); return ICRL_OK; }
int icrl_chain_tc_set_profile(void* buf) { icrl_chain_tc_set_profile_impl(reinterpret_cast<long long*>(buf)); return ICRL_OK; }

int icrl_pack_chain_tc_weights(void* stream, int kind, const float* W_hh, void* packed, int* launches) {
  TRY(icrl_pack_chain_tc_weights_impl(S_(stream), kind, W_hh, packed));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_tc_fwd(void* stream, int kind, int pieces, long long seg, int warm, const int* tok_stream,
                      const float* table, const void* packed, const float* b_hn, float* stash_h, float* stash_c,
                      float* stash_gates, void* ws, float* cp_state, float* err, int* launches) {
  TRY(icrl_chain_tc_fwd_impl(S_(stream), kind, pieces, seg, warm, tok_stream, table, packed, b_hn, stash_h, stash_c,
                             stash_gates, ws, cp_state, err));
  bump(launches, 2);                       // the persistent cluster kernel + the joint check
  return ICRL_OK;
}

int icrl_chains_tc_fwd_fused(void* stream, int v_pieces, long long v_seg, int v_warm, const int* v_stream,
                             const float* v_table, const void* v_packed, float* v_stash_h, float* v_stash_c,
                             float* v_stash_gates, void* v_ws, float* v_cp_state, float* v_err, int r_pieces, long long r_seg,
                             int r_warm, const int* r_stream, const float* r_table, const void* r_packed, const float* r_b_hn,
                             float* r_stash_h, void* r_ws, float* r_cp_state, float* r_err, int* launches) {
  TRY(icrl_chains_tc_fwd_fused_impl(S_(stream), v_pieces, v_seg, v_warm, v_stream, v_table, v_packed, v_stash_h, v_stash_c,
                                    v_stash_gates, v_ws, v_cp_state, v_err, r_pieces, r_seg, r_warm, r_stream, r_table,
                                    r_packed, r_b_hn, r_stash_h, r_ws, r_cp_state, r_err));
  bump(launches, 3);                       // one persistent cluster kernel for both chains + the two joint checks
  return ICRL_OK;
}

int icrl_chain_tc_lstm_bwd(void* stream, int pieces, long long seg, int warm, const void* packed,
                           const float* stash_gates, const float* stash_c, const int* take, const float* dh_take,
                           long long take_rows, void* dg_pairs, long long pair_rows, float* dg_inv_scale, void* ws,
                           float* cp_state, float* err, int* launches) {
  TRY(icrl_chain_tc_lstm_bwd_impl(S_(stream), pieces, seg, warm, packed, stash_gates, stash_c, take, dh_take, take_rows,
                                  dg_pairs, pair_rows, dg_inv_scale, ws, cp_state, err));
  bump(launches, 3);                       // |dh_take| maximum, the persistent cluster kernel, the joint check
  return ICRL_OK;
}

int icrl_chain_tc_lstm_fwd_from(void* stream, int pieces, long long seg, int warm, const int* tok_stream, const float* table,
                                const void* packed, const float* h0, const float* c0, float* stash_h, float* stash_c,
                                float* stash_gates, void* ws, float* cp_state, float* err, int* launches) {
  TRY(icrl_chain_tc_lstm_fwd_from_impl(S_(stream), pieces, seg, warm, tok_stream, table, packed, h0, c0, stash_h, stash_c,
                                       stash_gates, ws, cp_state, err));
  bump(launches, (h0 || c0) ? 3 : 2);      // the state seed, the persistent cluster kernel, the joint check
  return ICRL_OK;
}

// ---- value-guided look-ahead decoder (trainers.py:73-105)
int icrl_lookahead_stream(void* stream, int B, int n, int K, int k, const int* cand_tok, const int* words, int* tok_stream,
                          int* take_pos, int* launches) {
  ICRL_REQUIRE(B > 0 && n >= 1 && K >= 1 && k >= 1, "bad look-ahead shape");
  ICRL_REQUIRE((long long)K * k * (n + 1) * B < (1ll << 31), "token stream longer than 2^31");
  TRY(icrl_lookahead_stream_impl(S_(stream), B, n, K, k, cand_tok, words, tok_stream, take_pos));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_lookahead_policy_step(void* stream, int R, int V, int k, int first, const float* features, const float* W_cnn,
                               const float* b_cnn, const float* table, const int* parent, const float* h_in, const float* c_in,
                               const int* tok, const void* whh_parts, const void* wv_parts, const float* b_v, float* h_out,
                               float* c_out, float* logits, float* top_val, int* top_idx, void* ws, int* launches) {
  ICRL_REQUIRE(R > 0 && V > 0 && k >= 1 && k <= 16 && k <= V, "bad beam-step shape (1 <= k <= min(16, V))");
  ICRL_REQUIRE(first ? features != nullptr : (parent && h_in && c_in), "the first step needs the features, later ones the parents");
  cudaStream_t st = S_(stream);
  const size_t RH = (size_t)R * H;
  float* h_prev = reinterpret_cast<float*>(ws);
  float* c_prev = h_prev + RH;
  float* gpre = c_prev + RH;
  float* gates = gpre + 4 * RH;
  void* h_parts = gates + 4 * RH;
  float* lg = logits ? logits : reinterpret_cast<float*>(reinterpret_cast<char*>(h_parts) + 3 * RH * 2);
  if (first) {
    // h0 = cnn2linear(features), c0 = 0 (models.py:75-78), as icrl_policy_rollout_fwd_tc starts
    TRY(icrl_gemm_f32_impl(st, 0, 1, R, H, H, features, H, W_cnn, H, h_prev, H, b_cnn, 0.f, nullptr, 0, launches));
    ICRL_CUDA(cudaMemsetAsync(c_prev, 0, RH * sizeof(float), st));
  } else {
    TRY(icrl_gather_rows_impl(st, R, h_in, parent, 0, h_prev));
    TRY(icrl_gather_rows_impl(st, R, c_in, parent, 0, c_prev));
    bump(launches, 2);
  }
  // one decode step of icrl_policy_rollout_fwd_tc for R rows, then the top-k of every row's logits
  TRY(icrl_split_bf16x3_impl(st, (long long)RH, h_prev, h_parts));
  TRY(icrl_gemm_bf16x3_impl(st, R, 4 * H, H, h_parts, whh_parts, gpre, 4 * H, nullptr));
  TRY(icrl_lstm_pointwise_fwd(st, R, gpre, table, tok, c_prev, gates, c_out, h_out));
  TRY(icrl_split_bf16x3_impl(st, (long long)RH, h_out, h_parts));
  TRY(icrl_gemm_bf16x3_impl(st, R, V, H, h_parts, wv_parts, lg, V, b_v));
  TRY(icrl_topk_rows(st, R, V, k, lg, top_val, top_idx));
  bump(launches, 6);
  return ICRL_OK;
}

int icrl_lookahead_score(void* stream, int B, int K, int k, const float* parent_score, const float* values, const float* top_val,
                         float* child_score, float* means, int* launches) {
  ICRL_REQUIRE(B > 0 && K >= 1 && k >= 1, "bad look-ahead shape");
  TRY(icrl_lookahead_score_impl(S_(stream), B, K, k, parent_score, values, top_val, child_score, means));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_set_profile(void* buf) { icrl_chain_set_profile_impl(reinterpret_cast<long long*>(buf)); return ICRL_OK; }

size_t icrl_chain_sync_bytes(void) { return icrl_chain_sync_bytes_impl(); }

int icrl_chain_lstm_fwd(void* stream, const int* tok_stream, int T, const float* table, const float* W_hh,
                        const float* h0, const float* c0, float* stash_h, float* stash_c, float* stash_gates,
                        float* h_out, float* c_out, void* sync_state, int* launches) {
  TRY(icrl_chain_lstm_fwd_impl(S_(stream), tok_stream, T, table, W_hh, h0, c0, stash_h, stash_c, stash_gates, h_out,
                               c_out, sync_state));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_gru_fwd(void* stream, const int* tok_stream, int T, const float* table, const float* W_hh,
                       const float* b_hn, const float* h0, float* stash_h, float* h_out, void* sync_state,
                       float* stash_gates, int* launches) {
  TRY(icrl_chain_gru_fwd_impl(S_(stream), tok_stream, T, table, W_hh, b_hn, h0, stash_h, h_out, sync_state, stash_gates));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chains_fwd_fused(void* stream, const int* v_stream, int v_T, const float* v_table, const float* v_W_hh,
                          float* v_stash_h, float* v_stash_c, float* v_stash_gates, const int* r_stream, int r_T,
                          const float* r_table, const float* r_W_hh, const float* r_b_hn, float* r_stash_h,
                          void* sync_state, int* launches) {
  TRY(icrl_chains_fwd_fused_impl(S_(stream), v_stream, v_T, v_table, v_W_hh, v_stash_h, v_stash_c, v_stash_gates,
                                 r_stream, r_T, r_table, r_W_hh, r_b_hn, r_stash_h, sync_state));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_lstm_bwd(void* stream, int T, const float* W_hh, const float* stash_gates, const float* stash_c,
                        const int* take, const float* dh_take, float* dgates, void* sync_state, const float* dh_init,
                        const float* dc_init, float* dh0_out, float* dc0_out, int* launches) {
  TRY(icrl_chain_lstm_bwd_impl(S_(stream), T, W_hh, stash_gates, stash_c, take, dh_take, dgates, sync_state, dh_init,
                               dc_init, dh0_out, dc0_out));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_gru_bwd(void* stream, int T, const float* W_hh, const float* stash_gates, const float* stash_h,
                       const int* take, const float* dh_take, float* dgh, float* dgx, void* sync_state,
                       const float* dh_init, float* dh0_out, int* launches) {
  TRY(icrl_chain_gru_bwd_impl(S_(stream), T, W_hh, stash_gates, stash_h, take, dh_take, dgh, dgx, sync_state, dh_init,
                              dh0_out));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_reward_chain_param_grads(void* stream, int T, int V, int D, const int* tok_stream, const float* dgh, const float* dgx,
                                  const float* stash_h, const float* E, const float* W_ih, float* dtable,
                                  float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE, float* dW_ih,
                                  float* dW_hh, float* db_ih, float* db_hh, int* launches) {
  cudaStream_t st = S_(stream);
  const int G = 3 * H;
  // dW_hh = sum_t (da_r, da_z, da_nh)_t (x) h_{t-1}
  TRY(icrl_gemm_f32_impl(st, 1, 0, G, H, T, dgh, G, stash_h, H, dW_hh, H, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  // gate-table gradient from the input-side gradients, then its factors
  ICRL_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * G * sizeof(float), st));
  TRY(icrl_scatter_add_rows(st, T, G, dgx, tok_stream, dtable));
  bump(launches, 1);
  TRY(icrl_gemm_f32_impl(st, 1, 0, G, D, V, dtable, G, E, D, dW_ih, D, nullptr, 0.f, nullptr, 0, launches));
  if (dE) TRY(icrl_gemm_f32_impl(st, 0, 0, V, D, G, dtable, G, W_ih, D, dE, D, nullptr, 0.f, nullptr, 0, launches));
  TRY(icrl_wcolsum(st, V, G, dtable, nullptr, 0, colsum_ws, db_ih));
  // b_hh: the r,z rows are folded into the table (same gradient as b_ih); b_hn sits inside r*(.) -> column sums of da_nh
  float* tmp = colsum_ws + (size_t)icrl_wcolsum_chunks(T > V ? T : V) * G;
  TRY(icrl_wcolsum(st, T, G, dgh, nullptr, 0, colsum_ws, tmp));
  bump(launches, 4);
  ICRL_CUDA(cudaMemcpyAsync(db_hh, db_ih, 2 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  ICRL_CUDA(cudaMemcpyAsync(db_hh + 2 * H, tmp + 2 * H, H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return ICRL_OK;
}

int icrl_linear_bwd(void* stream, int M, int N, int K, const float* x, const float* W, const float* dy, float* dx,
                    float* dW, float* db, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, int* launches) {
  cudaStream_t st = S_(stream);
  if (dx) TRY(icrl_gemm_f32_impl(st, 0, 0, M, K, N, dy, N, W, K, dx, K, nullptr, 0.f, nullptr, 0, launches));
  TRY(icrl_gemm_f32_impl(st, 1, 0, N, K, M, dy, N, x, K, dW, K, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  TRY(icrl_wcolsum(st, M, N, dy, nullptr, 0, colsum_ws, db));
  bump(launches, 2);
  return ICRL_OK;
}

int icrl_adam_flat(void* stream, long long n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                   float lr, float beta1, float beta2, float eps, int step, int* launches) {
  ICRL_REQUIRE(n > 0 && step >= 1, "bad Adam arguments");
  TRY(icrl_adam_flat_impl(S_(stream), n, params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_chain_check(void* stream, void* sync_state) { return icrl_chain_check_impl(S_(stream), sync_state); }

int icrl_gather_rows(void* stream, long long R, const float* src, const int* idx, long long row_offset, float* dst,
                     int* launches) {
  TRY(icrl_gather_rows_impl(S_(stream), R, src, idx, row_offset, dst));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_value_head_fwd(void* stream, int B, int S, const float* features, const float* h_take, const float* w_eff,
                        const float* b_eff, float* values, int* launches) {
  TRY(icrl_value_head_fwd_impl(S_(stream), B, S, features, h_take, w_eff, b_eff, values));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_value_head_bwd(void* stream, int B, int S, const float* features, const float* h_take, const float* dv_sb,
                        const float* sum_dv, const float* W1, const float* b1, const float* W2, const float* w_eff,
                        float* dh_take, float* dW1, float* db1, float* dW2, float* db2, float* ws, int* launches) {
  cudaStream_t st = S_(stream);
  const long long SB = (long long)S * B;
  float* g = ws;                  // [1024] = sum dv * [f, h]
  float* part = ws + 2 * H;
  TRY(icrl_wcolsum(st, SB, H, features, dv_sb, B, part, g));          // row r = s*B+b -> features[b]
  TRY(icrl_wcolsum(st, SB, H, h_take, dv_sb, 0, part, g + H));
  TRY(icrl_value_head_grads_impl(st, g, sum_dv, W1, b1, W2, dW1, db1, dW2, db2));
  TRY(icrl_value_head_dh_impl(st, SB, dv_sb, w_eff, dh_take));
  bump(launches, 6);
  return ICRL_OK;
}

// dW_ih = dtable^T E, dE = dtable W_ih (when dE is set), db_ih = db_hh = column sums of dtable
static int gate_table_grads(cudaStream_t st, int V, int D, const float* dtable, const float* E, const float* W_ih,
                            float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE, float* dW_ih, float* db_ih,
                            float* db_hh, int* launches) {
  TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, D, V, dtable, 4 * H, E, D, dW_ih, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  if (dE)
    TRY(icrl_gemm_f32_impl(st, 0, 0, V, D, 4 * H, dtable, 4 * H, W_ih, D, dE, D, nullptr, 0.f, gemm_ws, gemm_ws_bytes, launches));
  TRY(icrl_wcolsum(st, V, 4 * H, dtable, nullptr, 0, colsum_ws, db_ih));
  bump(launches, 2);
  ICRL_CUDA(cudaMemcpyAsync(db_hh, db_ih, 4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return ICRL_OK;
}

int icrl_value_chain_param_grads(void* stream, int T, int V, int D, const int* tok_stream, const float* dgates,
                                 const float* stash_h, const float* E, const float* W_ih, float* dtable,
                                 float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE, float* dW_ih,
                                 float* dW_hh, float* db_ih, float* db_hh, int B, int p0, int S, int h_packed,
                                 int* launches) {
  cudaStream_t st = S_(stream);
  // Gate-table gradient: dtable[token] += dgates of every position that consumed the token.  When the caller names the
  // stream's shape (B > 0: tok_stream = icrl_build_stream(B, p0, S, extra 0)) the positions of one (column, row) are
  // summed before the reduction and the column maxima of dgates come back for the contraction below.
  unsigned* colmax = nullptr;
  ICRL_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * 4 * H * sizeof(float), st));
  if (B > 0) {
    ICRL_REQUIRE(T == icrl_stream_len(B, p0, S, 0), "T is not the length of the (B, p0, S) stream");
    colmax = reinterpret_cast<unsigned*>(colsum_ws);             // consumed by the split below, before colsum_ws is reused
    TRY(icrl_scatter_add_stream(st, B, p0, S, 0, 4 * H, dgates, tok_stream, dtable, colmax));
  } else {
    TRY(icrl_scatter_add_rows(st, T, 4 * H, dgates, tok_stream, dtable));
  }
  bump(launches, 1);
  // dW_hh = sum_t dgates_t (x) h_{t-1};  stash_h row t = h_{t-1}.  With a workspace of icrl_wgrad_tc_ws_bytes(2048, 512,
  // T, 2) bytes the contraction runs on tcgen05 (wgrad_tc.cu), otherwise on the fp32 SIMT GEMM.
  ICRL_REQUIRE(!h_packed || gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(4 * H, H, T, 2), "h_packed needs the wgrad_tc workspace");
  if (gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(4 * H, H, T, 2)) {
    TRY(icrl_wgrad_tc_impl(st, 4 * H, H, T, dgates, 4 * H, stash_h, H, dW_hh, H, gemm_ws, gemm_ws_bytes, 2, colmax, h_packed));
    bump(launches, (colmax ? 4 : 5) - (h_packed ? 1 : 0));
  } else {
    TRY(icrl_gemm_f32_impl(st, 1, 0, 4 * H, H, T, dgates, 4 * H, stash_h, H, dW_hh, H, nullptr, 0.f, gemm_ws,
                           gemm_ws_bytes, launches));
  }
  return gate_table_grads(st, V, D, dtable, E, W_ih, colsum_ws, gemm_ws, gemm_ws_bytes, dE, dW_ih, db_ih, db_hh, launches);
}

int icrl_value_chain_param_grads_pairs(void* stream, int T, int V, int D, const int* tok_stream, const void* dg_pairs,
                                       long long pair_rows, const float* dg_inv_scale, const float* stash_h, const float* E,
                                       const float* W_ih, float* dtable, float* colsum_ws, float* gemm_ws,
                                       size_t gemm_ws_bytes, float* dE, float* dW_ih, float* dW_hh, float* db_ih,
                                       float* db_hh, int B, int p0, int S, int h_packed, int* launches) {
  cudaStream_t st = S_(stream);
  ICRL_REQUIRE(B > 0 && T == icrl_stream_len(B, p0, S, 0), "T is not the length of the (B, p0, S) stream");
  ICRL_REQUIRE(gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes_impl(4 * H, H, T, 2), "gate-gradient pairs need the wgrad_tc workspace");
  ICRL_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * 4 * H * sizeof(float), st));
  TRY(icrl_scatter_add_stream_pairs(st, B, p0, S, 0, dg_pairs, pair_rows, dg_inv_scale, tok_stream, dtable));
  TRY(icrl_wgrad_tc_gate_pairs_impl(st, H, T, dg_pairs, pair_rows, dg_inv_scale, stash_h, H, dW_hh, H, gemm_ws, gemm_ws_bytes,
                                    2, h_packed));
  bump(launches, 3 - (h_packed ? 1 : 0));
  return gate_table_grads(st, V, D, dtable, E, W_ih, colsum_ws, gemm_ws, gemm_ws_bytes, dE, dW_ih, db_ih, db_hh, launches);
}

int icrl_reward_cosine_fwd(void* stream, int B, int S, const float* ve, const float* se, float* rewards,
                           int* launches) {
  TRY(icrl_reward_cosine_impl(S_(stream), B, S, ve, se, rewards));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_a2c_loss_fwd_bwd(void* stream, int B, int S, const float* values, const float* rewards, const float* logp,
                          float inv_denom, float* out3, float* dv_sb, float* dlogp, float* sum_dv, int* launches) {
  TRY(icrl_a2c_loss_impl(S_(stream), B, S, values, rewards, logp, inv_denom, out3, dv_sb, dlogp, sum_dv));
  bump(launches, 1);
  return ICRL_OK;
}

// ---- entropy bonus (new; the reference's loss has none)
int icrl_policy_entropy(void* stream, int B, int S, int V, const float* logits, int ldl, float* entropy, int* launches) {
  ICRL_REQUIRE(B > 0 && S > 0 && V > 0 && ldl >= V, "bad entropy shape (B, S, V > 0, ldl >= V)");
  ICRL_REQUIRE(logits && entropy, "the entropy pass needs the logits and the output");
  TRY(icrl_policy_entropy_impl(S_(stream), B, S, V, logits, ldl, entropy));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_a2c_loss_entropy_fwd_bwd(void* stream, int B, int S, const float* values, const float* rewards, const float* logp,
                                  const float* entropy, float entropy_coef, float inv_denom, float* out4, float* dv_sb,
                                  float* dlogp, float* sum_dv, int* launches) {
  ICRL_REQUIRE(entropy && out4, "the entropy loss needs the entropy and four output words");
  TRY(icrl_a2c_loss_impl(S_(stream), B, S, values, rewards, logp, inv_denom, out4, dv_sb, dlogp, sum_dv, entropy,
                         entropy_coef));
  bump(launches, 1);
  return ICRL_OK;
}

int icrl_softmax_entropy_bwd(void* stream, int B, int S, int V, float* z, int ldz, const long long* tokens_out,
                             const float* dlogp, const float* entropy, float scale, int* launches) {
  ICRL_REQUIRE(B > 0 && S > 0 && V > 0 && ldz >= V, "bad logits shape (B, S, V > 0, ldz >= V)");
  ICRL_REQUIRE(z && tokens_out && dlogp && entropy, "the softmax backward needs z, the tokens, dL/dlogp and the entropy");
  TRY(icrl_softmax_bwd(S_(stream), B, S, V, z, ldz, tokens_out, dlogp, entropy, scale));
  bump(launches, 1);
  return ICRL_OK;
}

// ---- policy pretraining loss (trainers.py:202-257)
int icrl_policy_xent_fwd_bwd(void* stream, int B, int S, int V, const float* logits, const long long* targets,
                             const int* n_rows, const double* w_rows, float* dz, int ldz, float* ce, float* loss,
                             int* launches) {
  ICRL_REQUIRE(B > 0 && S > 0 && V > 0 && ldz >= V, "bad logits shape (B, S, V > 0, ldz >= V)");
  ICRL_REQUIRE(logits && targets && n_rows && w_rows && dz && ce && loss, "null argument");
  ICRL_REQUIRE(dz != logits, "dL/dlogits is written out of place: the logits stay intact for a re-run");
  TRY(icrl_policy_xent_impl(S_(stream), B, S, V, logits, targets, n_rows, w_rows, dz, ldz, ce, loss));
  bump(launches, 2);
  return ICRL_OK;
}

}  // extern "C"
