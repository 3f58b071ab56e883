// Internal (non-exported) entry points shared between the translation units.
#pragma once
#include "common.cuh"

int icrl_gemm_f32_impl(cudaStream_t st, int transA, int transB, int M, int N, int K, const float* A, int lda,
                       const float* B, int ldb, float* C, int ldc, const float* bias, float beta, float* ws,
                       size_t ws_bytes, int* launches);
int icrl_lstm_pointwise_fwd(cudaStream_t st, int B, const float* gpre, const float* table, const int* tok,
                            const float* c_prev, float* gates_act, float* c_out, float* h_out);
int icrl_lstm_pointwise_bwd(cudaStream_t st, int B, const float* dh_rec, const float* dh_add, float* dc,
                            const float* gates_act, const float* c_prev, const float* c_cur, float* dgpre);
int icrl_softmax_sample(cudaStream_t st, int B, int V, const float* logits, int ldl, const double* uniforms, int greedy,
                        const long long* forced, int* tok_next, long long* tokens_out, float* logp_out, int S, int s, float* probs_out);
// entropy (nullable, [B][S]): add the entropy bonus's term scale * p (log p + H) to dL/dlogits
int icrl_softmax_bwd(cudaStream_t st, int B, int S, int V, float* z, int ldl, const long long* tokens_out,
                     const float* dlogp, const float* entropy = nullptr, float scale = 0.f);
int icrl_policy_entropy_impl(cudaStream_t st, int B, int S, int V, const float* logits, int ldl, float* entropy);
int icrl_policy_xent_impl(cudaStream_t st, int B, int S, int V, const float* logits, const long long* targets,
                          const int* n_rows, const double* w_rows, float* dz, int ldz, float* ce, float* loss);
int icrl_topk_rows(cudaStream_t st, int R, int V, int k, const float* x, float* top_val, int* top_idx);
int icrl_scatter_add_rows(cudaStream_t st, long long R, int C, const float* src, const int* idx, float* dst);
int icrl_scatter_add_stream(cudaStream_t st, int B, int p0, int S, int extra, int C, const float* src, const int* tok_stream,
                            float* dst, unsigned* colmax);
int icrl_scatter_add_stream_pairs(cudaStream_t st, int B, int p0, int S, int extra, const void* pairs, long long pair_rows,
                                  const float* inv_scale, const int* tok_stream, float* dst);
int icrl_wcolsum_chunks(long long R);
int icrl_wcolsum(cudaStream_t st, long long R, int C, const float* X, const float* w, long long row_mod,
                 float* partial, float* out);

int icrl_pack_value_head_impl(cudaStream_t st, const float* W1, const float* b1, const float* W2, const float* b2,
                              float* w_eff, float* b_eff);
int icrl_value_head_fwd_impl(cudaStream_t st, int B, int S, const float* features, const float* h_take,
                             const float* w_eff, const float* b_eff, float* values);
int icrl_value_head_dh_impl(cudaStream_t st, long long rows, const float* dv_sb, const float* w_eff, float* dh_take);
int icrl_value_head_grads_impl(cudaStream_t st, const float* g, const float* sdv, const float* W1, const float* b1,
                               const float* W2, float* dW1, float* db1, float* dW2, float* db2);
int icrl_reward_cosine_impl(cudaStream_t st, int B, int S, const float* ve, const float* se, float* rewards);
int icrl_a2c_loss_impl(cudaStream_t st, int B, int S, const float* values, const float* rewards, const float* logp,
                       float inv_denom, float* out3, float* dv_sb, float* dlogp, float* sum_dv,
                       const float* entropy = nullptr, float entropy_coef = 0.f);
int icrl_build_stream_impl(cudaStream_t st, int B, int p0, int S, int extra, const int* tokcm, int* stream, int* take,
                           int* take_pos);
int icrl_gather_rows_impl(cudaStream_t st, long long R, const float* src, const int* idx, long long row_offset,
                          float* dst);
int icrl_lookahead_stream_impl(cudaStream_t st, int B, int n, int K, int k, const int* cand_tok, const int* words, int* stream,
                               int* take_pos);
int icrl_lookahead_score_impl(cudaStream_t st, int B, int K, int k, const float* parent, const float* values, const float* top_val,
                              float* child, float* means);
int icrl_add_gate_bias_impl(cudaStream_t st, int V, int G, int fold, const float* b_ih, const float* b_hh,
                            float* table);

size_t icrl_chain_sync_bytes_impl();
int icrl_chain_lstm_fwd_impl(cudaStream_t st, const int* stream, int T, const float* table, const float* w_hh,
                             const float* h0, const float* c0, float* stash_h, float* stash_c, float* stash_gates,
                             float* h_out, float* c_out, void* sync_state);
int icrl_chain_gru_fwd_impl(cudaStream_t st, const int* stream, int T, const float* table, const float* w_hh,
                            const float* b_hn, const float* h0, float* stash_h, float* h_out, void* sync_state,
                            float* stash_gates = nullptr);
int icrl_chain_gru_bwd_impl(cudaStream_t st, int T, const float* w_hh, const float* stash_gates, const float* stash_h,
                            const int* take, const float* dh_take, float* dgh, float* dgx, void* sync_state,
                            const float* dh_init, float* dh0_out);
int icrl_chains_fwd_fused_impl(cudaStream_t st, const int* v_stream, int v_T, const float* v_table,
                               const float* v_w_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                               const int* r_stream, int r_T, const float* r_table, const float* r_w_hh,
                               const float* r_b_hn, float* r_stash_h, void* sync_state);
int icrl_chain_lstm_bwd_impl(cudaStream_t st, int T, const float* w_hh, const float* stash_gates, const float* stash_c,
                             const int* take, const float* dh_take, float* dgates, void* sync_state, const float* dh_init,
                             const float* dc_init, float* dh0_out, float* dc0_out);
int icrl_chain_check_impl(cudaStream_t st, void* sync_state);

int icrl_split_bf16x3_impl(cudaStream_t st, long long n, const float* x, void* parts);
int icrl_gemm_bf16x3_impl(cudaStream_t st, int M, int N, int K, const void* a_parts, const void* b_parts, float* C,
                          int ldc, const float* bias);

size_t icrl_decode_weight_halves_impl();
int icrl_pack_decode_weights_impl(cudaStream_t st, int V, const float* W_hh, const float* W_v, void* packed);
int icrl_policy_decode_impl(cudaStream_t st, int B, int V, int p0, int S, int greedy, const float* table,
                            const void* packed, const float* b_v, const double* uniforms, const long long* forced,
                            int* tokcm, long long* tokens_out, float* logp, float* Hs, float* Cs, float* Gs,
                            float* logits, float* last_logits, void* hparts);
void icrl_decode_set_profile_impl(long long* buf);
int icrl_build_stream_sharded_impl(cudaStream_t st, int B, int p0, int S, int extra, int shards, const int* tokcm,
                                   int* stream, int* take, int* take_pos);
int icrl_chains_fwd_fused_batched_impl(cudaStream_t st, int nb, const int* v_stream, int v_T, const float* v_table,
                                       const float* v_w_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                                       const int* r_stream, int r_T, const float* r_table, const float* r_w_hh,
                                       const float* r_b_hn, float* r_stash_h, void* sync_state);
int icrl_chain_lstm_bwd_batched_impl(cudaStream_t st, int shards, int T, const float* w_hh, const float* stash_gates,
                                     const float* stash_c, const int* take, const float* dh_take, float* dgates,
                                     void* sync_state);
void icrl_chain_set_profile_impl(long long* buf);
size_t icrl_wgrad_tc_ws_bytes_impl(int M, int N, long long T, int splits);
int icrl_wgrad_tc_impl(cudaStream_t st, int M, int N, long long T, const float* A, int lda, const float* B, int ldb,
                       float* C, int ldc, void* ws, size_t ws_bytes, int splits, const unsigned* colmax = nullptr,
                       int b_packed = 0);
int icrl_wgrad_tc_gate_pairs_impl(cudaStream_t st, int N, long long T, const void* pairs, long long pair_rows,
                                  const float* inv_scale, const float* B, int ldb, float* C, int ldc, void* ws,
                                  size_t ws_bytes, int splits, int b_packed);
int icrl_wgrad_tc_pack_b_impl(cudaStream_t st, int M, int N, long long T, const float* B, int ldb, void* ws, size_t ws_bytes,
                              int splits);
int icrl_adam_flat_impl(cudaStream_t st, long long n, float* p, const float* g, float* m, float* v, float lr, float b1,
                        float b2, float eps, int step);

// chain_tc.cu: chain pieces on tcgen05
void icrl_chain_tc_set_profile_impl(long long* buf);
void icrl_chain_tc_set_bias_impl(float fwd, float bwd);
int icrl_chain_tc_max_pieces_impl();
size_t icrl_chain_tc_weight_halves_impl(int kind);
int icrl_pack_chain_tc_weights_impl(cudaStream_t st, int kind, const float* W_hh, void* packed);
size_t icrl_chain_tc_ws_bytes_impl(int pieces);
size_t icrl_chain_tc_cp_floats_impl(int pieces);
int icrl_chain_tc_fwd_impl(cudaStream_t st, int kind, int P, long long seg, int warm, const int* stream,
                           const float* table, const void* packed, const float* b_hn, float* stash_h, float* stash_c,
                           float* stash_g, void* ws, float* cp_state, float* err);
int icrl_chain_tc_lstm_fwd_from_impl(cudaStream_t st, int P, long long seg, int warm, const int* stream, const float* table,
                                     const void* packed, const float* h0, const float* c0, float* stash_h, float* stash_c,
                                     float* stash_g, void* ws, float* cp_state, float* err);
int icrl_chain_tc_lstm_bwd_impl(cudaStream_t st, int P, long long seg, int warm, const void* packed,
                                const float* stash_g, const float* stash_c, const int* take, const float* dh_take,
                                long long take_rows, void* dg_pair, long long pair_rows, float* dg_inv_scale, void* ws,
                                float* cp_state, float* err);
size_t icrl_policy_bptt_tc_ws_bytes_impl(int B, int n_cell);
int icrl_policy_bptt_tc_impl(cudaStream_t st, int B, int n_cell, int p0, const void* packed, const float* Gs,
                             const float* Cs, const float* dHv, float* DG, float* dh0, void* ws, float* err);
int icrl_pack_transposed_bf16x3_impl(cudaStream_t st, int rows, int cols, int Kp, const float* W, void* parts);
int icrl_chains_tc_fwd_fused_impl(cudaStream_t st, int Pv, long long seg_v, int warm_v, const int* v_stream,
                                  const float* v_table, const void* v_packed, float* v_stash_h, float* v_stash_c,
                                  float* v_stash_g, void* v_ws, float* v_cp, float* v_err, int Pr, long long seg_r,
                                  int warm_r, const int* r_stream, const float* r_table, const void* r_packed,
                                  const float* r_b_hn, float* r_stash_h, void* r_ws, float* r_cp, float* r_err);
void icrl_chain_tc_set_tma_store_impl(int on);
int icrl_chain_tc_bwd_max_pieces_impl();
