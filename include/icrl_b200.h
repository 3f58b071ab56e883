/* icrl_b200 -- C ABI of the B200-native A2C caption-training hot path.
 *
 * The reference (pratikpv/image-captioning-through-rl) has no FFI layer: its operator API is the
 * Python surface of models.py plus five trainers.py call sites (SURVEY.md section 8b).  This header
 * is the boundary the drop-in Python modules (image-captioning-through-rl_b200/models.py,
 * trainers.py, engine.py) bind with ctypes.  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types.
 *   - every function returns 0 on success or an ICRL_ERR_* code; icrl_last_error() gives the text.
 *   - all buffers are caller-owned DEVICE pointers (fp32 unless stated); the library never allocates
 *     persistent memory.  Row-major everywhere.  H = 512 is fixed (models.py:41,160,250).
 *   - `stream` is a cudaStream_t passed as void*; launches are asynchronous on it.  The only calls
 *     that synchronise are icrl_chain_check and icrl_device_info.
 *   - `launches` (nullable) is incremented by the number of kernels the call launched.
 *   - token matrices: `tokcm` is int32 [n_cols][B] (column-major captions: the order in which the
 *     reference feeds columns to its RNNs); `tokens_out` is int64 [B][S] like the reference's actions.
 */
#ifndef ICRL_B200_H
#define ICRL_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICRL_OK 0
#define ICRL_ERR_ARG 1
#define ICRL_ERR_CUDA 2
#define ICRL_ERR_WATCHDOG 3

const char* icrl_last_error(void);
int icrl_version(void);
/* out[0]=SM count, out[1]=cc major, out[2]=cc minor, out[3]=cooperative launch supported */
int icrl_device_info(int* out4);

/* ---- dense contraction (replaces the cuBLAS sgemm calls behind nn.Linear / nn.LSTM input projections,
 *      models.py:75, 82, 177-178, 259-260).  C = beta*C + bias + op(A) op(B); see gemm_simt.cu for op().
 *      ws/ws_bytes: optional split-K workspace. */
int icrl_gemm_f32(void* stream, int transA, int transB, int M, int N, int K, const float* A, int lda,
                  const float* B, int ldb, float* C, int ldc, const float* bias, float beta, float* ws,
                  size_t ws_bytes, int* launches);

/* ---- tensor-core contraction (tcgen05, sm_100a): C[M][ldc] = A B^T + bias, fp32-grade: each fp32 operand is
 *      split into three bf16 parts (icrl_split_bf16x3: parts is bf16 [3][n], x ~= p0 + p1 + p2) and the six
 *      products with i + j <= 2 are accumulated in f32 in tensor memory.  a_parts [3][M][K], b_parts [3][N][K];
 *      K % 64 == 0. */
int icrl_split_bf16x3(void* stream, long long n, const float* x, void* parts, int* launches);
int icrl_gemm_bf16x3(void* stream, int M, int N, int K, const void* a_parts, const void* b_parts, float* C, int ldc,
                     const float* bias, int* launches);

/* ---- weight packing, once per optimizer step (new; the reference recomputes these products at every
 *      RNN step).  table[v][:] = W_ih E[v] + b_ih + (b_hh for the first `fold` gate rows).
 *      LSTM: G = 2048, fold = 2048.  GRU: G = 1536, fold = 1024 (b_hn stays inside r*(.), models.py:215).
 *      D = embedding width: E [V][D], W_ih [G][D] (512, or the width of frozen pretrained vectors, models.py:61-63).
 *      The same D is passed to the three parameter-gradient entry points, whose dE may be NULL (frozen embedding). */
int icrl_pack_gate_table(void* stream, int V, int G, int fold, int D, const float* E, const float* W_ih,
                         const float* b_ih, const float* b_hh, float* table, int* launches);
/* value head linear2(linear1(.)) has no activation (models.py:177-178): w_eff = W2 W1 (1024), b_eff (1). */
int icrl_pack_value_head(void* stream, const float* W1, const float* b1, const float* W2, const float* b2,
                         float* w_eff, float* b_eff, int* launches);

/* ---- policy rollout (replaces PolicyNetwork.forward re-run per step + softmax + np.random.choice +
 *      log-prob gather: models.py:71-84, 286; trainers.py:441-458; greedy: trainers.py:57-70).
 *      n_cell = p0 - 1 + S LSTM cell steps; the last S are followed by vocab projection + sampling.
 *      uniforms: float64 [S][B] (the doubles np.random.choice would draw), ignored when greedy != 0.
 *      forced: nullable int64 [B][S]; when given, these actions are taken instead (teacher forcing for
 *      parity checks) while log-probs / stash are still computed.
 *      tokcm: in: columns 0..p0-1 hold the prefix; out: columns p0..p0+S-1 hold the sampled tokens.
 *      Stash (for backward): Hs,Cs [(n_cell+1)][B][512], Gs [n_cell][B][2048], logits [S][B][V].
 *      gpre: workspace [B][2048]. */
int icrl_policy_rollout_fwd(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                            const float* W_cnn, const float* b_cnn, const float* table, const float* W_hh,
                            const float* W_v, const float* b_v, const double* uniforms, const long long* forced,
                            int* tokcm, long long* tokens_out, float* logp, float* Hs, float* Cs, float* Gs, float* logits,
                            float* gpre, int* launches);
/*      Same rollout with the two per-step GEMMs (h W_hh^T and h W_v^T) on the tcgen05 pipe.  Extra operands:
 *      3-part bf16 splits of W_hh ([3][2048][512]) and W_v ([3][V][512]) (icrl_split_bf16x3, once per optimizer
 *      step) and scratch h_parts [3][B][512] bf16. */
int icrl_policy_rollout_fwd_tc(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                               const float* W_cnn, const float* b_cnn, const float* table, const void* whh_parts,
                               const void* wv_parts, const float* b_v, const double* uniforms,
                               const long long* forced, int* tokcm, long long* tokens_out, float* logp, float* Hs,
                               float* Cs, float* Gs, float* logits, float* gpre, void* h_parts, int* launches);

/* ---- weight-gradient contraction on tcgen05 (wgrad_tc.cu): C [M][ldc] = A^T B for time-major fp32 operands A [T][lda]
 *      (M columns), B [T][ldb] (N columns); M a multiple of 128, N of 512 (the 4 N tiles of an M tile form a cluster
 *      that shares the A tile by TMA multicast).  Operands are scaled per A column and split into fp16
 *      pairs [2][T][C] by an elementwise pre-pass and read MN-major by the MMA; f32 accumulation in TMEM is flushed to
 *      registers every 512 K elements.
 *      ws: icrl_wgrad_tc_ws_bytes(M, N, T, splits) device bytes.  icrl_value_chain_param_grads takes this path by
 *      itself when its gemm_ws is at least icrl_wgrad_tc_ws_bytes(2048, 512, T, 2) bytes. */
size_t icrl_wgrad_tc_ws_bytes(int M, int N, long long T, int splits);
int icrl_wgrad_tc(void* stream, int M, int N, long long T, const float* A, int lda, const float* B, int ldb, float* C,
                  int ldc, void* ws, size_t ws_bytes, int splits, int* launches);
/*      The B operand's pre-pass alone, into the workspace of the same (M, N, T, splits): for callers whose B is final before
 *      A (the value chain's h stash exists after the forward) and who want it off the critical path, on another stream;
 *      icrl_value_chain_param_grads(..., h_packed = 1) then skips it. */
int icrl_wgrad_tc_pack_b(void* stream, int M, int N, long long T, const float* B, int ldb, void* ws, size_t ws_bytes,
                         int splits, int* launches);

/*      The same rollout as ONE persistent kernel (decode.cu): clusters of 8 CTAs own 128 rows each for all
 *      timesteps; gate and vocab GEMMs on tcgen05 (2-part fp16 split, 3 MMAs, f32 accumulation in TMEM) with the
 *      cell update, softmax, inverse-CDF sampling / argmax and log-prob fused into their epilogues.
 *      packed: icrl_decode_weight_halves() fp16 values written by icrl_pack_decode_weights (once per optimizer
 *      step; needs V <= 1024, V % 4 == 0).  hparts: scratch, 4*B*512 fp16.  Gs / logits may be null (inference:
 *      no backward stash); last_logits (nullable) [B][V] receives the logits of the final step. */
size_t icrl_decode_weight_halves(void);
/*      Debug aid: when buf != NULL, CTA 0 of later icrl_policy_rollout_fwd_fused launches writes clock64 stamps of
 *      its phases to buf[n_cell][16] (device int64); NULL switches it off. */
int icrl_decode_set_profile(void* buf);
int icrl_pack_decode_weights(void* stream, int V, const float* W_hh, const float* W_v, void* packed, int* launches);
int icrl_policy_rollout_fwd_fused(void* stream, int B, int V, int p0, int S, int greedy, const float* features,
                                  const float* W_cnn, const float* b_cnn, const float* table, const void* packed,
                                  const float* b_v, const double* uniforms, const long long* forced, int* tokcm,
                                  long long* tokens_out, float* logp, float* Hs, float* Cs, float* Gs, float* logits,
                                  float* last_logits, void* hparts, int* launches);

/* ---- policy backward through time (replaces autograd over the S prefix re-runs, trainers.py:479).
 *      dlogp [B][S]; when dlogp is NULL, `logits` must already hold dL/dlogits [S][B][V] (module-level autograd).
 *      logits is overwritten with dL/dlogits.  Workspaces: dHv [S*B][512],
 *      DG [n_cell*B][2048], dh [2][B][512], dc [B][512], dtable [V][2048], colsum_ws
 *      [icrl_colsum_ws_floats(max(S*B, V), 2048)], gemm_ws/gemm_ws_bytes.  Gradients are OVERWRITTEN. */
int icrl_policy_rollout_bwd(void* stream, int B, int V, int p0, int S, int D, const float* features, const float* E,
                            const float* W_ih, const float* W_hh, const float* W_v, const int* tokcm,
                            const long long* tokens_out, const float* dlogp, const float* Hs, const float* Cs,
                            const float* Gs, float* logits, float* dHv, float* DG, float* dh, float* dc,
                            float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE,
                            float* dW_cnn, float* db_cnn, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh,
                            float* dW_v, float* db_v, int* launches);
/* The same backward with its contractions on tcgen05: the n_cell serial cell-backward steps ([B x 2048] . W_hh each) as ONE
 * launch of the chain-backward kernel (chain_tc.cu: batch rows in the MMA M dimension, 128 per cluster of 8 CTAs), and --
 * when the logits are handed over with row stride ldz = icrl_vocab_pad() (1024; columns >= V zero) -- dW_v = dZ^T H
 * (K = S*B, wgrad_tc) and dHv = dZ W_v (3-part bf16 split).  tc_packed: icrl_pack_chain_tc_weights(kind 0) of the policy's
 * W_hh; tc_ws: icrl_policy_bwd_tc_ws_bytes(B, S, p0 - 1 + S) bytes; tc_err: 8 floats (tc_err[4] = max |dL/dh| injected,
 * tc_err[5] = 1 when the fp16 exchange overflowed: re-run with icrl_policy_rollout_bwd). */
size_t icrl_policy_bwd_tc_ws_bytes(int B, int S, int n_cell);
int icrl_vocab_pad(void);
int icrl_policy_rollout_bwd_tc(void* stream, int B, int V, int p0, int S, int D, const float* features, const float* E,
                               const float* W_ih, const float* W_hh, const float* W_v, const int* tokcm,
                               const long long* tokens_out, const float* dlogp, const float* Hs, const float* Cs,
                               const float* Gs, float* logits, float* dHv, float* DG, float* dh, float* dc,
                               float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE,
                               float* dW_cnn, float* db_cnn, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh,
                               float* dW_v, float* db_v, const void* tc_packed, void* tc_ws, float* tc_err, int ldz,
                               int* launches);
size_t icrl_colsum_ws_floats(long long rows, int cols);
/* ---- teacher-forced LSTM sequence, one direction (bidirectional policy variant, models.py:59-78; for the reverse
 *      direction the caller passes the token columns reversed).  Cell j consumes tokcm[j][:]; Hs/Cs [(n+1)][B][512]
 *      (row 0 = h0 / 0), Gs [n][B][2048]; gpre: workspace [B][2048].
 *      Backward: dH [n][B][512] = dL/d(h after cell j); outputs overwritten: dh0 [B][512], dE [V][D] (nullable),
 *      dW_ih [2048][D], dW_hh [2048][512], db_ih, db_hh [2048]; DG [n*B][2048], dh [2][B][512], dc [B][512],
 *      dtable [V][2048], colsum_ws / gemm_ws as icrl_policy_rollout_bwd. */
int icrl_lstm_seq_fwd(void* stream, int B, int n, const float* h0, const int* tokcm, const float* table,
                      const float* W_hh, float* Hs, float* Cs, float* Gs, float* gpre, int* launches);
int icrl_lstm_seq_bwd(void* stream, int B, int n, int V, int D, const int* tokcm, const float* Hs, const float* Cs,
                      const float* Gs, const float* dH, const float* W_hh, const float* E, const float* W_ih, float* DG,
                      float* dh, float* dc, float* dtable, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes,
                      float* dh0, float* dE, float* dW_ih, float* dW_hh, float* db_ih, float* db_hh, int* launches);

/* ---- token streams of the batch-as-time chains (models.py:166-169, 253-255).  Block s = columns
 *      0..p0+s-1+extra (extra = 0 value net, 1 reward net; for GetRewards on whole captions use
 *      p0 = L, S = 1, extra = 0).  T = icrl_stream_len(B,p0,S,extra).  stream int32 [T];
 *      take int32 [T] (row s*B+b or -1); take_pos int32 [S*B] (stream position of each output). */
long long icrl_stream_len(int B, int p0, int S, int extra);
int icrl_build_stream(void* stream, int B, int p0, int S, int extra, const int* tokcm, int* stream_out, int* take,
                      int* take_pos, int* launches);

/* ---- serial chains (replace the seq=B,batch=1 nn.LSTM / nn.GRU calls with carried hidden_cell,
 *      models.py:130-135, 223-228).  Cooperative launches of 64 (single) or 128 (fused) CTAs.
 *      sync_state: icrl_chain_sync_bytes() device bytes, zeroed once by the caller.
 *      h0/c0 [512] nullable (= init_hidden zeros, models.py:122-128); h_out/c_out [512] nullable
 *      (the carried hidden_cell after the call).  stash_h [(T+1)][512] (row 0 = h0, row t+1 = h_t);
 *      LSTM training stash: stash_c [(T+1)][512], stash_gates [T][2048] (nullable for inference). */
size_t icrl_chain_sync_bytes(void);
int icrl_chain_lstm_fwd(void* stream, const int* tok_stream, int T, const float* table, const float* W_hh,
                        const float* h0, const float* c0, float* stash_h, float* stash_c, float* stash_gates,
                        float* h_out, float* c_out, void* sync_state, int* launches);
/* stash_gates (nullable) [T][2048]: r, z, n, W_hn h + b_hn per step -- only for training the reward network. */
int icrl_chain_gru_fwd(void* stream, const int* tok_stream, int T, const float* table, const float* W_hh,
                       const float* b_hn, const float* h0, float* stash_h, float* h_out, void* sync_state,
                       float* stash_gates, int* launches);
/* BPTT through the reward GRU chain (train_reward_network, trainers.py:260-309; the A2C step keeps the reward net
 * frozen).  dgh [T][1536] = hidden-side gate gradients (da_r, da_z, da_nh), dgx [T][1536] = input-side
 * (da_r, da_z, da_n); dh_init / dh0_out as in icrl_chain_lstm_bwd. */
int icrl_chain_gru_bwd(void* stream, int T, const float* W_hh, const float* stash_gates, const float* stash_h,
                       const int* take, const float* dh_take, float* dgh, float* dgx, void* sync_state,
                       const float* dh_init, float* dh0_out, int* launches);
/* reward-chain parameter gradients (overwritten); colsum_ws: icrl_colsum_ws_floats(max(T,V), 1536) + 1536 floats. */
int icrl_reward_chain_param_grads(void* stream, int T, int V, int D, const int* tok_stream, const float* dgh, const float* dgx,
                                  const float* stash_h, const float* E, const float* W_ih, float* dtable,
                                  float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE, float* dW_ih,
                                  float* dW_hh, float* db_ih, float* db_hh, int* launches);
/* backward of y = x W^T + b (nn.Linear; visual_embed / semantic_embed, models.py:259-260): dx [M][K] (nullable),
 * dW [N][K], db [N] (overwritten); colsum_ws: icrl_colsum_ws_floats(M, N) floats. */
int icrl_linear_bwd(void* stream, int M, int N, int K, const float* x, const float* W, const float* dy, float* dx,
                    float* dW, float* db, float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, int* launches);
/* value LSTM chain and reward GRU chain side by side in one launch (both from zero state) */
int icrl_chains_fwd_fused(void* stream, const int* v_stream, int v_T, const float* v_table, const float* v_W_hh,
                          float* v_stash_h, float* v_stash_c, float* v_stash_gates, const int* r_stream, int r_T,
                          const float* r_table, const float* r_W_hh, const float* r_b_hn, float* r_stash_h,
                          void* sync_state, int* launches);
/* BPTT through the value chain (replaces autograd through the carried-state LSTM, trainers.py:479):
 * dgates [T][2048] = dL/d(pre-activation gates); dh_take [S*B][512] injected at take[t] >= 0.
 * The reference carries hidden_cell WITH its autograd history from one call to the next (models.py:133), so a
 * segment's backward may receive dL/d(final h, c) from the call that consumed its state (dh_init, dc_init [512],
 * nullable = zero) and must hand dL/d(initial h, c) to the call before it (dh0_out, dc0_out [512], nullable). */
int icrl_chain_lstm_bwd(void* stream, int T, const float* W_hh, const float* stash_gates, const float* stash_c,
                        const int* take, const float* dh_take, float* dgates, void* sync_state, const float* dh_init,
                        const float* dc_init, float* dh0_out, float* dc0_out, int* launches);
/* ---- chain shards (new; the reference has no equivalent).  The batch is cut into `shards` (2, 4 or 8) contiguous
 *      row shards and the value / reward recurrences of every shard start from zero state: exactly the reference
 *      run on `shards` minibatches of B/shards rows with the gradients averaged, i.e. what `shards` data-parallel
 *      ranks compute (SURVEY.md 8e).  The shards advance in lockstep on the same CTAs, sharing W_hh in registers, so
 *      one exchange round trip carries `shards` hidden vectors.  Layout: every per-step array of shard k starts at
 *      row k * (T + 1) with T = icrl_stream_len(B / shards, p0, S, extra); take holds global rows s*B + b and take_pos
 *      global stash rows, so heads, loss and the parameter-gradient entry points are used unchanged with
 *      T_total = shards * (T + 1). */
int icrl_build_stream_sharded(void* stream, int B, int p0, int S, int extra, int shards, const int* tokcm,
                              int* stream_out, int* take, int* take_pos, int* launches);
int icrl_chains_fwd_fused_sharded(void* stream, int shards, const int* v_stream, int v_T, const float* v_table,
                                  const float* v_W_hh, float* v_stash_h, float* v_stash_c, float* v_stash_gates,
                                  const int* r_stream, int r_T, const float* r_table, const float* r_W_hh,
                                  const float* r_b_hn, float* r_stash_h, void* sync_state, int* launches);
int icrl_chain_lstm_bwd_sharded(void* stream, int shards, int T, const float* W_hh, const float* stash_gates,
                                const float* stash_c, const int* take, const float* dh_take, float* dgates,
                                void* sync_state, int* launches);
/* ---- chain pieces on tcgen05 (chain_tc.cu; the default engine).  The same ONE carried-state chain
 *      (models.py:130-135 value LSTM, :223-228 reward GRU; backward of trainers.py:479) advanced as `pieces` lockstep
 *      pieces, 128 per cluster of 8 CTAs: one kernel step is the contraction H_prev [pieces x 512] . W_hh^T on the
 *      tensor cores (fp16 hi/lo' split, three products, f32 accumulation in tensor memory: fp32-grade) with the cell
 *      update in its epilogue.  Piece k covers positions [k*seg, (k+1)*seg + warm) of the stream; pieces k >= 1 start
 *      from zero state and discard their first `warm` positions; the backward recurrence is mirrored (piece k walks
 *      (k+1)*seg + warm - 1 down to k*seg; all but the last start with dh = dc = 0 and discard `warm` steps).
 *      Array sizes: streams / take pieces*seg + warm entries (the tail past the chain padded with token 0 / -1),
 *      stash_gates the same number of rows, stash_h / stash_c one row more (row 0 is zeroed by the call); any
 *      pieces >= 2, seg >= 1 is accepted.  CHECKED, not assumed: after every launch err[] holds running maxima (zero
 *      to re-arm) of the state differences at the joints -- forward err[0] = max |dh| and err[1] = max |dc| / max(1, |c|) at the end
 *      of the warm-up, err[2], err[3] the same half-way through it (the slope gives the contraction rate the caller
 *      sizes the next warm-up with); backward err[0..3] = |d(dh)|, |d(dc)| at the joints (end / half-way) relative to
 *      err[4] = max |dh_take|, err[5] = 1 when a scaled gate gradient left the fp16 range of the exchange.
 *      kind: 0 = LSTM (stash_c, stash_gates = activated i,f,g,o), 1 = GRU (b_hn [512]; stash_c, stash_gates NULL).
 *      packed: icrl_pack_chain_tc_weights (icrl_chain_tc_weight_halves(kind) fp16 values; after every optimizer step).
 *      ws: icrl_chain_tc_ws_bytes(pieces) bytes of scratch per launch; cp_state: icrl_chain_tc_cp_floats(pieces)
 *      floats (joint checkpoints).  icrl_chain_tc_max_pieces(): pieces that are co-resident on the device. */
int icrl_chain_tc_max_pieces(void);
size_t icrl_chain_tc_weight_halves(int kind);
size_t icrl_chain_tc_ws_bytes(int pieces);
size_t icrl_chain_tc_cp_floats(int pieces);
int icrl_pack_chain_tc_weights(void* stream, int kind, const float* W_hh, void* packed, int* launches);
int icrl_chain_tc_fwd(void* stream, int kind, int pieces, long long seg, int warm, const int* tok_stream,
                      const float* table, const void* packed, const float* b_hn, float* stash_h, float* stash_c,
                      float* stash_gates, void* ws, float* cp_state, float* err, int* launches);
/* Value LSTM and reward GRU forward chains in ONE launch: the co-resident clusters are split between the two independent
 * recurrences (v_pieces + r_pieces <= icrl_chain_tc_max_pieces(), each rounded up to whole clusters of 128), so the discarded
 * warm-up is paid once in wall time instead of twice.  Arguments as two icrl_chain_tc_fwd calls (kind 0, then kind 1). */
int icrl_chains_tc_fwd_fused(void* stream, int v_pieces, long long v_seg, int v_warm, const int* v_stream,
                             const float* v_table, const void* v_packed, float* v_stash_h, float* v_stash_c,
                             float* v_stash_gates, void* v_ws, float* v_cp_state, float* v_err, int r_pieces, long long r_seg,
                             int r_warm, const int* r_stream, const float* r_table, const void* r_packed, const float* r_b_hn,
                             float* r_stash_h, void* r_ws, float* r_cp_state, float* r_err, int* launches);
int icrl_chain_tc_lstm_bwd(void* stream, int pieces, long long seg, int warm, const void* packed,
                           const float* stash_gates, const float* stash_c, const int* take, const float* dh_take,
                           long long take_rows, void* dg_pairs, long long pair_rows, float* dg_inv_scale, void* ws,
                           float* cp_state, float* err, int* launches);
/* LSTM pieces from a carried state: icrl_chain_tc_fwd(kind 0) with piece 0 starting from h0 / c0 [512] (16-byte aligned;
 * NULL = zeros; both NULL gives icrl_chain_tc_fwd's output bit for bit).  Stash row 0 holds (h0, c0); the state after the
 * chain's T live positions is stash row T. */
int icrl_chain_tc_lstm_fwd_from(void* stream, int pieces, long long seg, int warm, const int* tok_stream, const float* table,
                                const void* packed, const float* h0, const float* c0, float* stash_h, float* stash_c,
                                float* stash_gates, void* ws, float* cp_state, float* err, int* launches);
/*      The gate gradients of the live positions come out as the fp16 pairs the recurrence itself runs on: dg_pairs =
 *      [2][pair_rows][2048] halves (hi plane, then lo' plane; pair_rows >= pieces * seg + warm, 32-byte aligned), value =
 *      (hi + lo'/2048) * *dg_inv_scale (one power of two per launch, written to the device word dg_inv_scale), columns of
 *      each block of 32 hidden units in the order [unit quad][gate][unit of the quad] (natural a*512 + u -> stored
 *      128 (u / 32) + 16 ((u % 32) / 4) + 4 a + u % 4).  icrl_value_chain_param_grads_pairs consumes them. */
/* Debug aid: buf != NULL (24 device int64): cycle sums of cluster 0 / CTA 0's first epilogue warp, forward [0..5] =
 * {accumulator wait, gather, cell update, stores, cluster barrier, steps}, backward [8..13] likewise, [16..21] the reward
 * chain's first cluster when the forward launch is fused. */
int icrl_chain_tc_set_profile(void* buf);
/* Experiment knob: relative compensation (1 + x) applied to the main tensor-memory accumulator of the forward / backward
 * chain kernels (the tensor core truncates on every accumulate; DESIGN 4.1).  Default 5.76e-7, 2.3e-6 = 1.8e-8 per
 * accumulating MMA instruction. */
int icrl_chain_tc_set_bias(float fwd, float bwd);
/* Pieces of the backward recurrence that are co-resident (same clusters as the forward). */
int icrl_chain_tc_bwd_max_pieces(void);
/* Experiment knob: 1 = the forward stash of the live positions leaves through TMA tensor stores, 0 (default) = per-thread
 * vector stores (measured equal: the store phase is L2-bound, not issue-bound). */
int icrl_chain_tc_set_tma_store(int on);
/* Debug aid: when buf != NULL (16 device int64), CTA 0 / thread 0 of the sharded chain kernels accumulates its
 * cycles per phase: [0..3] value LSTM forward {exchange wait, GEMV + reduce, pointwise + publish, T}, [4..7] reward GRU
 * forward, [8..14] backward {coefficients + requests, poll wait, gate gradients + stores, barrier, contraction + reduce,
 * barrier + publish, T} (the backward runs a separately compiled, instrumented build of the kernel). */
int icrl_chain_set_profile(void* buf);
/* synchronises `stream`; ICRL_ERR_WATCHDOG if any chain launch since the last check gave up waiting */
int icrl_chain_check(void* stream, void* sync_state);
/* dst[r][:] = src[idx[r] + row_offset][:]  (rows of 512 floats; h at the take positions) */
int icrl_gather_rows(void* stream, long long R, const float* src, const int* idx, long long row_offset, float* dst,
                     int* launches);

/* ---- heads and loss.
 *      value head (models.py:175-178): values [B][S] from h_take [S][B][512]. */
int icrl_value_head_fwd(void* stream, int B, int S, const float* features, const float* h_take, const float* w_eff,
                        const float* b_eff, float* values, int* launches);
/*      value head backward: dv_sb [S][B], sum_dv [1] -> dh_take [S*B][512] and the four head gradients
 *      (overwritten).  ws: >= 1024 + icrl_colsum_ws_floats(S*B, 512) floats. */
int icrl_value_head_bwd(void* stream, int B, int S, const float* features, const float* h_take, const float* dv_sb,
                        const float* sum_dv, const float* W1, const float* b1, const float* W2, const float* w_eff,
                        float* dh_take, float* dW1, float* db1, float* dW2, float* db2, float* ws, int* launches);
/*      value-chain parameter gradients from the chain backward's dgates (overwritten):
 *      dW_hh = dgates^T h_prev, gate-table scatter, dW_ih = dtable^T E, dE = dtable W_ih, db = colsum.
 *      B > 0: tok_stream is the stream icrl_build_stream(B, p0, S, extra 0) built (T = icrl_stream_len(B, p0, S, 0)); the
 *      scatter then sums the positions that consumed the same (column, row) token before one vector reduction each
 *      (ten times fewer reductions at 19 rollout steps) and hands the column maxima of dgates to the contraction.
 *      B = 0: any token stream of T positions (one reduction per position).
 *      h_packed = 1: gemm_ws already holds the fp16 split of stash_h (icrl_wgrad_tc_pack_b(2048, 512, T, ...)). */
int icrl_value_chain_param_grads(void* stream, int T, int V, int D, const int* tok_stream, const float* dgates,
                                 const float* stash_h, const float* E, const float* W_ih, float* dtable,
                                 float* colsum_ws, float* gemm_ws, size_t gemm_ws_bytes, float* dE, float* dW_ih,
                                 float* dW_hh, float* db_ih, float* db_hh, int B, int p0, int S, int h_packed,
                                 int* launches);
/*      The same from icrl_chain_tc_lstm_bwd's gate-gradient pairs (dg_pairs, pair_rows, dg_inv_scale as written there)
 *      instead of fp32 dgates; the contraction reads them as they lie.  Needs B > 0 (the stream's shape) and the wgrad_tc
 *      workspace (gemm_ws_bytes >= icrl_wgrad_tc_ws_bytes(2048, 512, T, 2)). */
int icrl_value_chain_param_grads_pairs(void* stream, int T, int V, int D, const int* tok_stream, const void* dg_pairs,
                                       long long pair_rows, const float* dg_inv_scale, const float* stash_h, const float* E,
                                       const float* W_ih, float* dtable, float* colsum_ws, float* gemm_ws,
                                       size_t gemm_ws_bytes, float* dE, float* dW_ih, float* dW_hh, float* db_ih,
                                       float* db_hh, int B, int p0, int S, int h_packed, int* launches);
/*      reward (models.py:259-260 + GetRewards trainers.py:117-120): rewards [B][S] = cos(ve[b], se[s][b]). */
int icrl_reward_cosine_fwd(void* stream, int B, int S, const float* ve, const float* se, float* rewards,
                           int* launches);
/*      A2C loss (trainers.py:471-475) and its gradient seeds.  inv_denom = 1/(B_global*S).
 *      out3 = {loss, mean reward, mean advantage} (partial sums for a data-parallel shard);
 *      dv_sb [S][B] = dL/dvalues, dlogp [B][S] = dL/dlogp, sum_dv [1]  (all nullable). */
int icrl_a2c_loss_fwd_bwd(void* stream, int B, int S, const float* values, const float* rewards, const float* logp,
                          float inv_denom, float* out3, float* dv_sb, float* dlogp, float* sum_dv, int* launches);

/* ---- entropy bonus (new; the reference's loss, trainers.py:471-475, has none): the A3C regulariser
 *      loss = reference loss - entropy_coef * mean_{b,s} H[b][s],  H = -sum_j p_j log p_j of the softmax the rollout
 *      sampled step s of row b from.  Off (no call) reproduces the reference.
 *      Policy entropy over the logits stash of the rollout (icrl_policy_rollout_fwd*: logits [S][B][ldl], the V real
 *      columns summed): entropy [B][S] (the layout of logp), same max / exp / sum arithmetic as the softmax backward.
 *      One warp per row; reads S*B*V*4 bytes once. */
int icrl_policy_entropy(void* stream, int B, int S, int V, const float* logits, int ldl, float* entropy, int* launches);
/*      icrl_a2c_loss_fwd_bwd with the entropy bonus: out4 = {loss - entropy_coef * mean entropy, mean reward,
 *      mean advantage, mean entropy} (partial sums scaled by inv_denom); dv_sb, dlogp, sum_dv bit-identical to
 *      icrl_a2c_loss_fwd_bwd's (the bonus does not depend on values, rewards or log-probs). */
int icrl_a2c_loss_entropy_fwd_bwd(void* stream, int B, int S, const float* values, const float* rewards, const float* logp,
                                  const float* entropy, float entropy_coef, float inv_denom, float* out4, float* dv_sb,
                                  float* dlogp, float* sum_dv, int* launches);
/*      Step 1 of icrl_policy_rollout_bwd[_tc] with the bonus (logits backward of trainers.py:458 plus the entropy term):
 *      z [S][B][ldz] (the logits) becomes, in place,
 *        dL/dz = dlogp[b][s] (onehot(a) - p) + scale * p (log p + H[b][s]),  scale = entropy_coef * inv_denom.
 *      Columns >= V are not touched (the zero padding of ldz = icrl_vocab_pad() stays zero).  Then call
 *      icrl_policy_rollout_bwd[_tc] with dlogp = NULL. */
int icrl_softmax_entropy_bwd(void* stream, int B, int S, int V, float* z, int ldz, const long long* tokens_out,
                             const float* dlogp, const float* entropy, float scale, int* launches);

/* ---- policy pretraining loss (train_policy_network, trainers.py:202-257): teacher-forced logits [S][B][V] of
 *      icrl_policy_rollout_fwd* with forced tokens, targets [B][S] int64 (the forced tokens, captions[:, 1:1+S]).
 *      Row b counts its first n_rows[b] <= S positions with weight w_rows[b] (f64; the reference's
 *      caplen_b / (B * n_b)):
 *        loss[0] = sum_b w_b sum_{s < n_b} CE(z[s][b], t[b][s]),  CE = log(sum exp(z - max)) - (z_t - max),
 *      summed in double in a fixed order; ce [S*B] f32 holds the per-row CE terms (zero past n_b).
 *      dz [S*B][ldz] (out of place; the logits are not modified):
 *        dz[s*B+b][v] = w_b (softmax(z)[v] - [v == t]) for s < n_b, 0 for s >= n_b and for the columns V..ldz-1.
 *      Then call icrl_policy_rollout_bwd_tc with dlogp = NULL, logits = dz and this ldz (or icrl_policy_rollout_bwd with
 *      ldz = V). */
int icrl_policy_xent_fwd_bwd(void* stream, int B, int S, int V, const float* logits, const long long* targets,
                             const int* n_rows, const double* w_rows, float* dz, int ldz, float* ce, float* loss,
                             int* launches);

/* ---- value-guided look-ahead decoder (GenerateCaptionsWithActorCriticLookAhead, trainers.py:73-105).  K candidate
 *      caption batches of B rows and n columns each are expanded by their k best words per beam step.
 *      Stream: cand_tok [K][n][B] int32 (each candidate's columns), words [K][B][k] int32 -> the value chain of the step,
 *      K*k blocks of (n+1)*B positions in the reference's call order (block c*k + i = candidate c's n columns, then its
 *      word column i), and take_pos [K*k][B] = stream position of each row of the word column (for icrl_gather_rows). */
int icrl_lookahead_stream(void* stream, int B, int n, int K, int k, const int* cand_tok, const int* words, int* tok_stream,
                          int* take_pos, int* launches);
/*      Policy beam step for R rows (R = K*B): each row's (h, c) is gathered from row parent[r] of h_in / c_in [*][512]
 *      (first != 0: the initial state cnn2linear(features [R][512]), c = 0; parent, h_in, c_in unused), one LSTM cell
 *      consumes tok [R] (gate table `table`, W_hh as the icrl_split_bf16x3 parts whh_parts) into h_out / c_out [R][512],
 *      logits = h_out W_v^T + b_v (wv_parts) go to `logits` [R][V] (nullable) and their top k <= 16 (descending, equal
 *      values by lower index) to top_val [R][k] f32 / top_idx [R][k] int32.  ws: R * (46*512 + 4*V) bytes. */
int icrl_lookahead_policy_step(void* stream, int R, int V, int k, int first, const float* features, const float* W_cnn,
                               const float* b_cnn, const float* table, const int* parent, const float* h_in, const float* c_in,
                               const int* tok, const void* whh_parts, const void* wv_parts, const float* b_v, float* h_out,
                               float* c_out, float* logits, float* top_val, int* top_idx, void* ws, int* launches);
/*      Scores: child_score [K*k][B] = parent_score [K][B] - (0.6 values + 0.4 log(top_val)) in fp32 and the reference's
 *      operation order (values [B][K*k] of icrl_value_head_fwd with S = K*k; a negative logit gives NaN as there), and
 *      means [K*k] = each child's batch mean (the reference's sort key). */
int icrl_lookahead_score(void* stream, int B, int K, int k, const float* parent_score, const float* values, const float* top_val,
                         float* child_score, float* means, int* launches);

/* ---- optimizer (replaces torch.optim.Adam.step over the 18 tensors, trainers.py:378, 480; SURVEY 8f row 4): one
 *      kernel over the flat parameter / gradient buckets, torch's default Adam (betas 0.9/0.999, eps 1e-8, no weight
 *      decay); `step` is the 1-based step count. */
int icrl_adam_flat(void* stream, long long n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                   float lr, float beta1, float beta2, float eps, int step, int* launches);

#ifdef __cplusplus
}
#endif
#endif /* ICRL_B200_H */
