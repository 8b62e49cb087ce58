/*
 * seqrec_b200 -- C-ABI of the B200-native next-item training / scoring hot path.
 *
 * The reference (efikarra/seq-recommendations) has no FFI of its own: its hot path is everything Keras/Theano
 * executes under `self.model.fit(...)` / `self.model.predict(...)` (model.py:181, model.py:195).  The entry points
 * below are what a binding for that path would call; each cites the reference construct it replaces.  The Python
 * host (`seq_recommendations_b200/engine.py`) binds them with ctypes -- see INTEGRATION.md for the stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates); nothing is allocated here
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); calls are asynchronous
 *   - return value: 0 on success, a negative cudaError_t on launch/config failure, -1000-x for argument errors
 *   - token order is TIME-MAJOR: token n = t*B + b, ids/targets/mask are [T][B]; pad tokens have mask 0
 *   - weights keep the Keras layouts: W_in (F, G*H), U (H, G*H), b (G*H), W_out (H, V), b_out (V), row-major fp32
 *   - gate order along G*H:  LSTM i,f,c,o   GRU z,r,h   simpleRNN h
 */
#ifndef SEQREC_B200_H_
#define SEQREC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { SEQREC_CELL_SIMPLE = 0, SEQREC_CELL_LSTM = 1, SEQREC_CELL_GRU = 2 };
enum { SEQREC_ACT_RELU = 0, SEQREC_ACT_TANH = 1, SEQREC_ACT_LINEAR = 2 };

/* library / device sanity: returns the compute capability major*10+minor of the current device, or <0 */
int seqrec_device_cc(void);
/* ABI version of this header */
int seqrec_abi_version(void);
/* number of kernels this library has launched since load (or since the last call with reset != 0) */
int seqrec_launch_count(int reset);

/* ---- batch formatting on the device (the step before the hot path; preprocessor.py:67-94 + Keras pad_sequences with
 * padding='pre', truncating='pre').  Ragged input: items (flat int32) and offsets (n_seqs+1, int64); sequence i of length
 * L gives the pairs (s[j], s[j+1]); its last min(L-1, T) pairs fill the right end of row i of ids_bt / tgt_bt (n_seqs, T),
 * the rest is pad = -1.  No (N,T,V) one-hot ever exists. */
int seqrec_pad_sequences(const int32_t* items, const int64_t* offsets, int32_t* ids_bt, int32_t* tgt_bt, int64_t n_seqs,
                         int T, void* stream);

/* ---- history features on the device (datasets.py:97-113 build_xs, consumed as c = xs[:-1] by
 * FullModelPreprocessor.transform_data, preprocessor.py:71,89,92): c (n_seqs, T, V) float32, c[b,t,v] = number of times
 * (freq != 0) or whether (freq == 0) item v occurred among s[0..j] of sequence b, where input position j lands on column t
 * of the left-padded / left-truncated row (truncated positions still count); pad columns are 0.  table (may be NULL):
 * value transform indexed by the count, table_len entries (the drivers' np.log(x + 1), experiments_server.py:35-36).
 * An item outside [0, V) sets bit 0 of err[0] (int32, may be NULL; the reference raises IndexError). */
int seqrec_history_features(const int32_t* items, const int64_t* offsets, float* c, int64_t n_seqs, int T, int V,
                            int freq, const float* table, int table_len, int32_t* err, void* stream);

/* ---- batch format (preprocessor.py:67-94, model.py:335 Masking) ------------------------------------------------
 * (B,T) batch-major ids/targets (pad = negative) -> time-major ids/targets/mask; counts valid tokens into
 * n_valid[0] (int32, must be zeroed by the caller).  Range check: an input id >= n_in, or a target outside [0, n_items)
 * on a valid step, turns the token into a pad and sets bit 0 / bit 1 of err[0] (int32, may be NULL; the reference raises
 * IndexError in np_utils.to_categorical, preprocessor.py:75-78) -- no kernel ever indexes a table with such an id. */
int seqrec_format_batch(const int32_t* ids_bt, const int32_t* tgt_bt, int32_t* ids_tb, int32_t* tgt_tb,
                        uint8_t* mask_tb, int32_t* n_valid, int B, int T, int n_in, int n_items, int32_t* err,
                        void* stream);

/* ---- K1: one-hot x input-kernel == row gather (model.py:360-364 LSTM on the masked one-hot input) ---------------
 * xp[n,:] = (mask[n] ? in_scale[n]*W_in[ids[n],:] : 0) + b.   in_scale may be NULL (no y->z dropout). */
int seqrec_gather_rows(const float* W_in, const float* b, const int32_t* ids, const uint8_t* mask,
                       const float* in_scale, float* xp, int64_t n_tokens, int V, int GH, void* stream);

/* ---- K7: dense one_hot^T . dxp of Theano == scatter-add (SURVEY D3) ----------------------------------------------
 * dW_in[ids[n],:] += in_scale[n]*dxp[n,:] for valid tokens, warp-aggregated atomics.  Rows touched for the first time
 * are appended to rows[] (count in n_rows[0]) using the flag array touched[V]; dW_in and touched must be all-zero
 * on entry for untouched rows (the row-sparse optimizer restores that invariant). */
int seqrec_scatter_add_rows(const float* dxp, const int32_t* ids, const uint8_t* mask, const float* in_scale,
                            float* dW_in, int32_t* touched, int32_t* rows, int32_t* n_rows, int64_t n_tokens,
                            int V, int GH, void* stream);

/* union row marking for data-parallel runs: claims every valid id of ids[] in touched[] / rows[] without adding */
int seqrec_mark_rows(const int32_t* ids, const uint8_t* mask, int32_t* touched, int32_t* rows, int32_t* n_rows,
                     int64_t n_tokens, int V, void* stream);

/* ---- K2: dense-feature input projection (RNNBaseline with [onehot || xs], model.py:245-255) ----------------------
 * C[M,N] (+)= A[M,K] . Bm[K,N] (+ bias[N]); plain fp32 SIMT GEMM for the small feature widths of that model. */
int seqrec_gemm_nn(const float* A, const float* Bm, const float* bias, float* C, int M, int N, int K,
                   int accumulate, void* stream);
/* K2 on the tcgen05 tensor cores (csrc/gemm_tc.cu): C[M,N] (+)= A[M,K] . Bt[N,K]^T (+ bias[N]), fp32 C (leading dimension
 * ldc).  A (M, K; ld lda) and Bt (N, K; ld ldb) are K-major bf16 hi/lo pairs staged by seqrec_split_bf16 (lda, ldb
 * multiples of 8; lo may be NULL when x3 == 0).  x3 != 0: 3-pass split product, ~2^-16 relative (fp32-grade).  Serves
 * the dense half of the input projection (x_to_z: model.py:354-358; RNNBaseline with [onehot || xs]: model.py:245-255)
 * and, with the operands staged transposed, the products of the x_to_y / y_to_y branches and their gradients. */
int seqrec_gemm_tc(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                   const float* bias, float* C, int64_t M, int N, int K, int64_t lda, int64_t ldb, int64_t ldc,
                   int accumulate, int x3, void* stream);
/* C[M,N] += A[K,M]^T . Bm[K,N]  (weight gradients: dW = X^T . dY), atomics over K-splits; C must be pre-zeroed */
int seqrec_gemm_tn_atomic(const float* A, const float* Bm, float* C, int M, int N, int K, void* stream);

/* ---- K3: recurrent scan forward (Theano K.rnn with mask; model.py:345-352) --------------------------------------
 * xg: in = xp [T][B][G*H], out = post-activation gates (in place).  hout [T][B][H]; cst [T][B][H] (LSTM cell
 * state; scratch for GRU backward).  Masked steps hold state and repeat the previous output. */
int seqrec_rnn_forward(int cell, int act, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                       int T, int B, int H, void* stream);

/* seqrec_rnn_forward from an initial state: h0 (B,H) and c0 (B,H, LSTM only) fp32, either may be NULL (= zeros;
 * then the result is bit-identical to seqrec_rnn_forward).  The final state is hout[T-1] (and cst[T-1] for LSTM): every family
 * (generic, register-resident and tensor-core scans) writes the held h and c on masked steps, so an all-pad row ends
 * bit for bit where it started.  A scan continued from hout[T-1] / cst[T-1] of an earlier call gives bit-identical
 * results to one call over both chunks at the same B (the per-step arithmetic does not depend on t).  c0 for a
 * GRU / SimpleRNN cell is an argument error.  Inference only: there is no backward from a non-zero state. */
int seqrec_rnn_forward_state(int cell, int act, float* xg, const float* U, const float* h0, const float* c0,
                             const uint8_t* mask, float* hout, float* cst, int T, int B, int H, void* stream);

/* ---- K4: recurrent scan backward (Theano scan gradient) ----------------------------------------------------------
 * dhout [T][B][H] = dLoss/dHout.  xg: in = saved gates, out = dxp (pre-activation gradients, in place).
 * U (H, G*H) and Ut = U^T (G*H, H).  For GRU, cst receives r*h_{t-1} (operand of dU's candidate block). */
int seqrec_rnn_backward(int cell, int act, float* xg, const float* U, const float* Ut, const uint8_t* mask,
                        const float* hout, float* cst, const float* dhout, int T, int B, int H, void* stream);
/* ---- K3 / K4 with Keras `recurrent_dropout` (model.py:346, :351; tune_params.py:83, tune_params_msnbc.py:54,77) ----
 * rec_mask (G, B, H): one inverted-dropout mask per gate block, constant over time; gate block g multiplies h_{t-1}
 * by rec_mask[g] before its recurrent product (GRU candidate: r * h_{t-1} * rec_mask[2]).  Same buffers and contracts
 * as seqrec_rnn_forward / seqrec_rnn_backward / seqrec_rnn_weight_grad; always the generic fp32 scan.  scratch: T*B*H
 * floats. */
int seqrec_rnn_forward_rd(int cell, int act, float* xg, const float* U, const float* rec_mask, const uint8_t* mask,
                          float* hout, float* cst, int T, int B, int H, void* stream);
int seqrec_rnn_backward_rd(int cell, int act, float* xg, const float* Ut, const float* rec_mask, const uint8_t* mask,
                           const float* hout, float* cst, const float* dhout, int T, int B, int H, void* stream);
int seqrec_rnn_weight_grad_rd(int cell, const float* dxp, const float* hout, const float* cst, const float* rec_mask,
                              float* scratch, float* dU, float* db, int T, int B, int H, void* stream);
/* 1 when seqrec_rnn_backward reads Ut for this (cell, H); 0 when the register-resident scan (GRU / SimpleRNN with
 * H <= 128, U held in registers for all T steps) serves it from U and Ut may be NULL */
int seqrec_rnn_needs_ut(int cell, int H);
/* ---- K3 on the tcgen05 tensor cores (csrc/rnn_tc.cu): same contract as seqrec_rnn_forward for LSTM / GRU with
 * H = 128 or 256.  A cluster of H/32 CTAs owns 64 batch rows for all T steps; each CTA keeps its slice of the
 * recurrent kernel in shared memory as a bf16 hi/lo operand (3-pass split products, fp32 accumulate in TMEM) and the
 * new hidden state is all-gathered through distributed shared memory every step.
 * Ut_hi / Ut_lo = seqrec_split_bf16(U, transpose = 1): U^T (G*H, H) as bf16 hi / lo, leading dimension H. */
int seqrec_rnn_tc_applicable(int cell, int H);
/* how many clusters of that scan (64 batch rows each) the current device keeps resident at once
 * (cudaOccupancyMaxActiveClusters): a batch of more than 64 x this many rows runs in waves; < 0 on error */
int seqrec_rnn_tc_max_clusters(int cell, int H);
int seqrec_rnn_tc_forward(int cell, int act, float* xg, const uint16_t* Ut_hi, const uint16_t* Ut_lo,
                          const uint8_t* mask, float* hout, float* cst, int T, int B, int H, void* stream);
/* seqrec_rnn_tc_forward from an initial state, with the contract of seqrec_rnn_forward_state (h0 / c0 16-byte
 * aligned).  Every CTA builds the h_{-1} operand from h0 with the same bf16 hi/lo split the scan applies to its own
 * h_t, so continuing from hout[T-1] is bit-identical to one longer scan. */
int seqrec_rnn_tc_forward_state(int cell, int act, float* xg, const uint16_t* Ut_hi, const uint16_t* Ut_lo,
                                const float* h0, const float* c0, const uint8_t* mask, float* hout, float* cst,
                                int T, int B, int H, void* stream);
/* K4 on the tensor cores, same contract as seqrec_rnn_backward: each CTA forms the K-split partial product of ITS gate
 * columns with U[:, cols] (bf16 hi/lo, resident in shared memory) and dL/dh_{t-1} is reduce-scattered through
 * distributed shared memory.  U_hi / U_lo = seqrec_split_bf16(U, transpose = 0): (H, G*H), leading dimension G*H. */
int seqrec_rnn_tc_backward(int cell, int act, float* xg, const uint16_t* U_hi, const uint16_t* U_lo,
                           const uint8_t* mask, const float* hout, float* cst, const float* dhout, int T, int B, int H,
                           void* stream);
/* diagnostics (scripts/time_rnn.py): device buffer of 64 x 8 clock64() stamps written by CTA 0 of the tensor-core scans
 * at their protocol points; NULL switches the capture off (the default) */
int seqrec_rnn_tc_debug_buffer(long long* dev_buf);
/* dU (H,G*H) += sum_t hprev_t^T . dxp_t (GRU candidate block uses cst = r*hprev);  db (G*H) += sum_n dxp[n,:].
 * dU and db must be pre-zeroed. */
int seqrec_rnn_weight_grad(int cell, const float* dxp, const float* hout, const float* cst, float* dU, float* db,
                           int T, int B, int H, void* stream);
/* the same gradient as one split-K tcgen05 GEMM over all tokens (csrc/wgrad_tc.cu; LSTM / GRU, H = 128 or 256):
 * dxp_hi/lo (N, G*H), h_hi/lo (N, H) and -- GRU only -- c_hi/c_lo (N, H) are the seqrec_split_bf16 images of dxp, hout
 * and cst; both operands are consumed token-major (MN-major UMMA operands), 3-pass split products, fp32 accumulate.
 * db is summed from the fp32 dxp. */
int seqrec_rnn_weight_grad_tc(int cell, const float* dxp, const uint16_t* dxp_hi, const uint16_t* dxp_lo,
                              const uint16_t* h_hi, const uint16_t* h_lo, const uint16_t* c_hi, const uint16_t* c_lo,
                              float* dU, float* db, int T, int B, int H, void* stream);
/* out (cols, rows) = in (rows, cols)^T */
int seqrec_transpose(const float* in, float* out, int rows, int cols, void* stream);

/* ---- K5: TimeDistributed(Dense) + softmax + categorical_crossentropy, never materialising (N,V)
 *          (model.py:382-384, :397; experiments_methods.py:42) -----------------------------------------------------
 * Per token: running max m and sum-exp s over the vocabulary and the target logit zy.  With V split over `splits`
 * partial ranges (or GPUs) the partial (m,s) live in ws_m/ws_s [splits][N]; seqrec_ce_finalize merges them.
 * hscale: optional inverted-dropout factors (N,H) applied to hout (z->y Dropout, model.py:371-372). */
int seqrec_ce_forward(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                      const int32_t* tgt, float* ws_m, float* ws_s, float* zy, int64_t n_tokens, int H, int V,
                      int v_begin, int v_end, int ldw, int splits, void* stream);
/* merge partial stats; ce[n] = -log(clip(exp(zy-m)/s, 1e-7, 1-1e-7))*mask; py[n] = clipped prob (model.py:108-110);
 * coef[n] = mask * [clip inactive] (to be scaled by 1/n_valid); loss_sum[0] = sum ce (deterministic single block) */
int seqrec_ce_finalize(const float* ws_m, const float* ws_s, const float* zy, const uint8_t* mask, float* m_out,
                       float* s_out, float* ce, float* py, float* coef, float* loss_sum, int64_t n_tokens,
                       int splits, void* stream);
/* seqrec_ce_finalize plus the masked mean Keras reports (weighted loss / number of unmasked steps, training.py
 * `_weighted_masked_objective` as used by model.py:397): n_valid[0] = unmasked tokens (int32, device);
 * n_valid_f[0] = (float)n_valid (the denominator the optimiser divides the un-normalised gradients by -- summed over
 * ranks in a data-parallel step), loss_mean[0] = loss_sum / n_valid.  n_tokens_dev (may be NULL): compacted token axis --
 * the number of tokens to process is read on the device and n_tokens is only the upper bound (splits must be 1). */
int seqrec_ce_finalize_mean(const float* ws_m, const float* ws_s, const float* zy, const uint8_t* mask, float* m_out,
                            float* s_out, float* ce, float* py, float* coef, float* loss_sum, const int32_t* n_valid,
                            float* n_valid_f, float* loss_mean, int64_t n_tokens, int splits,
                            const int32_t* n_tokens_dev, void* stream);

/* ---- K6: backward of K5 with recomputed logits ------------------------------------------------------------------
 * dlogit[n,v] = (exp(z-m)/s - [v==tgt]) * coef[n] * inv_nvalid[0];
 * dh (N,H) = dlogit . W_out^T (times hscale), dW_out (H,V) += hs^T . dlogit, db_out (V) += sum_n dlogit.
 * dW_out / db_out must be pre-zeroed; dh is overwritten (or accumulated when accumulate_dh != 0). */
int seqrec_ce_backward(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                       const int32_t* tgt, const float* m, const float* s, const float* coef,
                       const float* inv_nvalid, float* dh, float* dW_out, float* db_out, int64_t n_tokens, int H,
                       int V, int v_begin, int v_end, int ldw, int accumulate_dh, void* stream);

/* ---- K5/K6 on the tcgen05 tensor cores (csrc/ce_tc.cu) ----------------------------------------------------------
 * Operands are bf16 hi/lo pairs staged by seqrec_split_bf16 (lo pointers may be NULL when x3 == 0 = single-pass bf16):
 *   A  = hs            (N, Hk)   hs = hout (x dropout factors), Hk = H padded to a multiple of 64 with zeros
 *   Ht = hs^T          (Hk, Np)  Np = N padded to a multiple of 8
 *   Bt = W_out^T       (V, Hk)
 *   W  = W_out         (Hk, Vp)  Vp = V padded to a multiple of 8
 * x3 != 0 selects the 3-pass split product (fp32-grade, ~2^-16 relative); Hk <= 256.  b_out (V, may be NULL) is the
 * output bias, db_out (V, pre-zeroed, may be NULL) receives its gradient.  dh is overwritten unless accumulate_dh != 0; dW_out must be pre-zeroed (both leave
 * the SM through vector reductions).  ws_m / ws_s as in seqrec_ce_forward; the target logit comes from
 * seqrec_target_logit (exact fp32 dot product). */
int seqrec_ce_tc_forward(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                         const float* b_out, float* ws_m, float* ws_s, int64_t n_tokens, int Hk, int V, int v_begin,
                         int v_end, int x3, void* stream);
/* rows of ws_m / ws_s (partials per token) seqrec_ce_tc_forward writes for this problem size: the kernels run as a
 * persistent grid whose CTAs own balanced contiguous runs of (token tile, item tile) pairs, so a token tile's
 * vocabulary reduction is split over a few CTAs; pass the value as `splits` to seqrec_ce_finalize */
int seqrec_ce_tc_partials(int64_t n_tokens, int v_begin, int v_end);
int seqrec_ce_tc_backward(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Ht_hi, const uint16_t* Ht_lo,
                          const uint16_t* Bt_hi, const uint16_t* Bt_lo, const uint16_t* W_hi, const uint16_t* W_lo,
                          const int32_t* tgt, const float* m, const float* s, const float* coef,
                          const float* inv_nvalid, const float* hscale, float* dh, float* dW_out, int64_t n_tokens,
                          int H, int Hk, int V, int Vp, int64_t Np, int v_begin, int v_end, int ldw,
                          int accumulate_dh, int x3, const float* b_out, float* db_out, const int32_t* n_tokens_dev,
                          void* stream);
/* ---- rank of the true next item (Recall@k / MRR@k / NDCG@k without the logits) ------------------------------------
 * For a token with target y >= 0 and logits z (bias included):
 *     rank = 1 + #{v != y : z_v > z_y} + #{v < y : z_v == z_y}
 * i.e. the 1-based position of y in the stable descending order, ties to the lower item id (the order of seqrec_topk:
 * rank <= k <=> y is the top-k entry rank-1).  Pads (y < 0) have rank 0.
 * seqrec_ce_tc_forward_rank is seqrec_ce_tc_forward (same operands, same ws_m / ws_s partials, bit for bit) that also
 * counts, per token, the items of [v_begin, v_end) that precede y against the reference logit ref[n] (the exact fp32
 * target logit of seqrec_target_logit; the tensor-core logits are compared with it, so the count is exact outside a
 * band of the split-product error around z_y).  tgt holds GLOBAL item ids: item v of this launch is id_offset + v, so
 * a vocabulary shard (id_offset = its first item) counts its items under the catalog-wide tie rule.
 * Both rank entry points ADD their count to rank[n] with integer atomics (deterministic): the caller initialises
 * rank[] -- 0 to receive the bare count (vocabulary shards, whose counts are then summed), or 1 on valid tokens and 0
 * on pads to receive the 1-based rank directly (what the engine does; the +1 is never added by these kernels). */
int seqrec_ce_tc_forward_rank(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                              const float* b_out, float* ws_m, float* ws_s, const float* ref, const int32_t* tgt,
                              int id_offset, int32_t* rank, int64_t n_tokens, int Hk, int V, int v_begin, int v_end,
                              int x3, void* stream);
/* the same count on the exact-fp32 SIMT logits of seqrec_ce_forward (hout (N,H), W_out (H, ldw), b_out may be NULL).
 * ref NULL: z_y is computed with the same arithmetic as every z_v (an item whose W_out column equals the target's ties
 * exactly and the tie rule decides); every target must then lie in this launch's items. */
int seqrec_target_rank(const float* hout, const float* W_out, const float* b_out, const float* ref, const int32_t* tgt,
                       int id_offset, int32_t* rank, int64_t n_tokens, int H, int V, int v_begin, int v_end, int ldw,
                       void* stream);

/* ---- K5 + K6 (dH half) from ONE logits pass (csrc/ce_tc.cu, TS_FUSED) -----------------------------------------
 * The softmax is evaluated against a per-token REFERENCE logit ref[n] (the exact fp32 target logit from
 * seqrec_target_logit) instead of the running row maximum -- exp(z - ref) needs no rescaling (ref is one of the row's
 * logits; fp32 carries e^88 without loss of relative precision), so every CTA that shares a token tile accumulates
 *     acc[n,:] += sum_v exp(z[n,v] - ref[n]) . W_out[:,v]          s[n] += sum_v exp(z[n,v] - ref[n])
 * against the same reference and both leave through reductions: acc (N,H) and s (N) must be ZERO on entry.
 * Then seqrec_ce_finalize(ws_m = ref, ws_s = s, splits = 1) gives loss / clip coefficient, and seqrec_ce_dh_finish
 *     dh[n,:] = coef[n] . (acc[n,:] / s[n] - W_out[:, tgt[n]]) (. hscale[n,:])          (dh may alias acc)
 * (tgt[n] < 0: no one-hot term -- the target belongs to another item shard; coef[n] == 0: zeros).  With the
 * item-stationary dW kernel (seqrec_ce_tc_backward with dh = NULL, m = ref) a training step issues 4 logits-sized GEMMs
 * for 3 algorithmic ones instead of 5.  Operands as for seqrec_ce_tc_backward. */
int seqrec_ce_tc_fused(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                       const uint16_t* W_hi, const uint16_t* W_lo, const float* ref, const uint8_t* mask,
                       const float* b_out, float* acc, float* s, int64_t n_tokens, int H, int Hk, int V, int Vp,
                       int v_begin, int v_end, int x3, const int32_t* n_tokens_dev, void* stream);
int seqrec_ce_dh_finish(const float* acc, float* dh, const float* s, const float* coef, const int32_t* tgt,
                        const uint16_t* Bt_hi, const uint16_t* Bt_lo, const float* hscale, int64_t n_tokens, int H,
                        int Hk, const int32_t* orig, const int32_t* n_tokens_dev, void* stream);

/* ---- token compaction: pad tokens carry neither loss nor gradient, so the logits kernels of a training step run on
 * the VALID tokens only (a quarter fewer rows in all three logits GEMMs at the synthetic BASELINE workloads, whose
 * lengths are uniform in [T/2, T]).  orig[c] = time-major index of the c-th valid token in ascending order, tgt_c[c] =
 * its target, count[0] = number of valid tokens; block_counts: scratch of ceil(n_tokens / 256) int32.  The kernels
 * above take the count as `n_tokens_dev` (read on the device; their n_tokens argument is then the upper bound the TMA
 * descriptors are built for) and `orig` where a compacted row maps back to a row of hout / dh; mask may then be NULL.
 * seqrec_split_bf16_both_rows stages the compacted operand rows: output row r < n_rows[0] is source row orig[r]. */
int seqrec_compact_tokens(const uint8_t* mask, const int32_t* tgt, int64_t n_tokens, int32_t* orig, int32_t* tgt_c,
                          int32_t* count, int32_t* block_counts, void* stream);
int seqrec_split_bf16_both_rows(const float* src, const float* scale, const int32_t* orig, const int32_t* n_rows,
                                uint16_t* hi, uint16_t* lo, uint16_t* hi_t, uint16_t* lo_t, int64_t max_rows,
                                int64_t cols, int64_t ld_out, int64_t ld_t, void* stream);
int seqrec_target_logit(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                        const int32_t* tgt, float* zy, int64_t n_tokens, int H, int ldw, const int32_t* orig,
                        const int32_t* n_tokens_dev, void* stream);

/* ---- K9: scoring (model.py:194-195 predict; model.py:106-112 consumer) ------------------------------------------
 * full probabilities, batch-major (B,T,V) float32, for catalogs small enough to materialise */
int seqrec_predict_probs(const float* hout, const float* W_out, const float* b_out, const float* m, const float* s,
                         float* probs_btv, int T, int B, int H, int V, void* stream);
/* top-k item ids (and their probabilities) per token row; ties broken by the lower item id.  rows index hout. */
int seqrec_topk(const float* hout, const float* W_out, const float* b_out, const float* m, const float* s,
                int32_t* topk_ids, float* topk_p, int64_t n_rows, int H, int V, int k, void* stream);

/* top-k on the tcgen05 tensor cores (csrc/ce_tc.cu): logits tiles as in seqrec_ce_tc_forward; every epilogue thread
 * keeps a private top-k list of its (row, column-half) stream, a second kernel merges the lists of a row (value
 * descending, lower item id first on ties).  ws_v / ws_i: seqrec_ce_tc_partials(n_rows, 0, V) * n_rows * k elements.
 * k <= 32. */
int seqrec_topk_tc(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                   const float* b_out, const float* m, const float* s, float* ws_v, int32_t* ws_i, int32_t* topk_ids,
                   float* topk_p, int64_t n_rows, int Hk, int V, int k, int x3, void* stream);

/* merge of n_lists candidate lists per row -- cand_v / cand_i [n_lists][.][k] with `list_stride` elements between the
 * lists of a row -- into the row's top k: value descending, lower item id first on ties (the stable-argsort order of
 * the oracle).  Ends the vocabulary-parallel ranking (one list per item shard).  n_lists * k <= 384. */
int seqrec_topk_merge(const float* cand_v, const int32_t* cand_i, int n_lists, int64_t list_stride,
                      int32_t* topk_ids, float* topk_p, int64_t n_rows, int k, void* stream);

/* ---- candidate scoring (csrc/candidates.cu): a given list of C item ids per row (id < 0 = pad) ---------------------
 * z[n, j] = sum_h hout[n, h] . Wt[c - id_offset, h] (+ b_out[c - id_offset]) for c = cand[n * cand_ld + j], with the
 * arithmetic of seqrec_target_logit (bit-equal to its zy for target c).  Wt (v_local, H) is the item-major copy of
 * W_out (seqrec_transpose).  A pad, or an id outside [id_offset, id_offset + v_local) (another vocabulary shard's
 * item), writes 0.0f: summed over the shards, exactly one addend is non-zero.  z is (n_rows, C); any C >= 1 and H. */
#define SEQREC_MAX_CANDIDATES 1024
int seqrec_candidate_logits(const float* hout, const float* Wt, const float* b_out, const int32_t* cand,
                            int64_t cand_ld, float* z, int64_t n_rows, int C, int H, int id_offset, int v_local,
                            void* stream);
/* order of the candidates of each row from their logits z (n_rows, C) and ids cand (n_rows, C): score descending, then
 * lower item id, then lower list position; pads last, reported as id -1 with score 0.  Positions < k go to out_ids /
 * out_scores (n_rows, k); scores are z, or exp(z - m[n]) / s[n] when m and s are given.  out_ids NULL: no order.
 * tgt / zy / rank (n_rows each): rank[n] = 1 + #{j : cand_j >= 0, cand_j != y, z_j > zy[n] or (z_j == zy[n] and
 * cand_j < y)} for y = tgt[n] >= 0, 0 for y < 0.  tgt NULL: no rank. */
int seqrec_candidate_order(const float* z, const int32_t* cand, int C, int64_t n_rows, const float* m, const float* s,
                           int k, int32_t* out_ids, float* out_scores, const float* zy, const int32_t* tgt,
                           int32_t* rank, void* stream);

/* ---- sampled softmax with log-Q correction (csrc/sampled.cu) -----------------------------------------------------
 * A training step draws S item ids with replacement from q and scores every token against its target y and those S
 * shared items: with log Q(v) = log(S q(v)) and o_v = h . W_out[:, v] + b_out[v],
 *     l_0 = o_y - log Q(y),  l_j = o_{s_j} - log Q(s_j) (removed where s_j == y),  loss = -l_0 + log sum_j exp(l_j).
 * seqrec_sample_items: ids (S,) from draw i = state[0] + i of r_i = splitmix64(splitmix64(seed) ^ i): column
 * c = ((r >> 32) * V) >> 32, kept if (uint32)r < thr[c], else alias[c] (a Vose alias table; thr and alias NULL =
 * uniform).  state (2 x uint64) as for seqrec_dropout_mask_dev: advanced by S when the launch completes. */
#define SEQREC_MAX_SAMPLED 32768
int seqrec_sample_items(int32_t* ids, int S, const uint32_t* thr, const int32_t* alias, int V, uint64_t seed,
                        uint64_t* state, void* stream);
/* W_S (H, S) = W_out[:, ids] (W_out leading dimension ldw) and bias_S[j] = b_out[ids[j]] (b_out may be NULL = 0) minus
 * logQ[ids[j]]; logQ (V,) = log(S q(v)).  A strided gather: S*H 32-byte sectors read. */
int seqrec_gather_columns(const float* W_out, int64_t ldw, const float* b_out, const float* logQ, const int32_t* ids,
                          int S, int H, float* W_S, float* bias_S, void* stream);
/* one panel of materialised sampled logits Z (n_rows, S), Z = o + b - log Q of the sampled columns.  Per row n with
 * target y = tgt[n] and mask[n] != 0: l_0 = zy[n] - logQ[y] (zy: the exact fp32 target logit, bias included), columns
 * with ids[j] == y removed; ce[n] (may be NULL) = the row's loss, Z[n, j] <- p_j (0 on removed columns),
 * g_tgt[n] = p_0 - 1.  Pad rows: Z, ce and g_tgt become 0.  loss_part[0] = sum of the rows' losses, deterministic (no
 * float atomics).  S <= SEQREC_MAX_SAMPLED: the ids are held in shared memory for the accidental-hit test. */
int seqrec_sampled_softmax_rows(float* Z, int S, const int32_t* ids, const float* zy, const int32_t* tgt,
                                const float* logQ, const uint8_t* mask, float* ce, float* g_tgt, float* loss_part,
                                int64_t n_rows, void* stream);
/* the target column of each token: dh[n,:] += g_tgt[n] W_out[:, y_n], dW_out[:, y_n] += g_tgt[n] hs[n,:] (hs = hout, times
 * hscale when not NULL) and db_out[y_n] += g_tgt[n]; dh, dW_out, db_out may each be NULL (frozen weights); pads
 * (y_n < 0) are skipped.  Atomics. */
int seqrec_target_columns(const float* hout, const float* hscale, const float* W_out, int64_t ldw, const int32_t* tgt,
                          const float* g_tgt, float* dh, float* dW_out, float* db_out, int64_t n_tokens, int H,
                          void* stream);
/* dW_out[:, ids[j]] += dW_S[:, j] (dW_S (H, S)) and db_out[ids[j]] += db_S[j]; duplicate ids add up (atomics).  dW_out
 * or db_out may be NULL. */
int seqrec_scatter_add_columns(const float* dW_S, const float* db_S, const int32_t* ids, int S, int H, float* dW_out,
                               int64_t ldw, float* db_out, void* stream);

/* ---- history-feature / skip branches (csrc/dense_ops.cu): RNNFullModel's x_to_z / x_to_y / y_to_y (model.py:354-358,
 * :376-392) and NoRecurrenceModel (model.py:264-319).  logits z = hs.W + x.B + A[y_{t-1}] (+ biases) carry per-(token,
 * item) terms; the reference runs these models on small catalogs ((V,V) transition kernel A), so Z (N,V) is materialised.
 * Z[n,:] += (ids[n] >= 0 ? table[ids[n],:] : 0) + bias      (one-hot . A == row lookup; table or bias may be NULL) */
int seqrec_add_rows(float* Z, const float* table, const float* bias, const int32_t* ids, int64_t n_tokens, int V,
                    void* stream);
/* per-row max m, sum-exp s and target logit zy (may be NULL) of materialised logits; feed seqrec_ce_finalize, splits 1 */
int seqrec_softmax_rows_stats(const float* Z, const int32_t* tgt, float* m, float* s, float* zy, int64_t n_tokens,
                              int V, void* stream);
/* Z <- (exp(Z - m)/s - onehot(tgt)) * coef, in place (un-normalised, like K6; rows with coef == 0 become zeros) */
int seqrec_softmax_rows_dlogit(float* Z, const int32_t* tgt, const float* m, const float* s, const float* coef,
                               int64_t n_tokens, int V, void* stream);
/* rank[n] (overwritten) = the 1-based rank of tgt[n] in row n of materialised logits Z (n_rows, V), 0 for pads; the
 * reference value is Z[n, tgt[n]] itself, so ties are exact (definition at seqrec_ce_tc_forward_rank) */
int seqrec_rows_rank(const float* Z, const int32_t* tgt, int32_t* rank, int64_t n_rows, int V, void* stream);
/* model.predict from materialised time-major logits (T,B,V): batch-major probabilities (B,T,V) */
int seqrec_softmax_rows_probs(const float* Z, const float* m, const float* s, float* probs_btv, int T, int B, int V,
                              void* stream);
/* C[M,N] (=|+=) A[M,K] . Bm[N,K]^T   (fp32 SIMT; dH = dZ . W^T) */
int seqrec_gemm_nt(const float* A, const float* Bm, float* C, int M, int N, int K, int lda, int ldb, int ldc,
                   int accumulate, void* stream);
/* out[c] += sum_r in[r,c]   (bias gradients; out pre-zeroed) */
int seqrec_colsum(const float* in, float* out, int64_t rows, int cols, int ld, void* stream);
/* OnlyNonZeroDiagonal(dim, skip_rows) (model.py:48-66): zero the off-diagonal entries of the (dim, dim) block below the
 * first skip_rows rows of the (skip_rows + dim, dim) kernel W; Keras applies it to the updated weights */
int seqrec_diag_constraint(float* W, int skip_rows, int dim, void* stream);

/* ---- scoring metrics on the device (csrc/likelihood.cu): P (n_seqs, T) per-step probabilities p(true next item),
 * right-aligned (a sequence of L steps fills the last L columns); lengths (n_seqs, may be NULL = whole rows);
 * skip_first drops the first step of every window (count_first_prob=False of the reference).
 * utils.py:166-178 compute_likelihood: out2[0] += sum over sequences of mean_t -log(clip(p, 1e-7, 1-1e-7)),
 * out2[1] += sequences with a non-empty window (out2 pre-zeroed; the metric is out2[0] / out2[1]). */
int seqrec_likelihood(const float* P, const int32_t* lengths, int64_t n_seqs, int T, int skip_first, double* out2,
                      void* stream);
/* utils.py:145-163 compute_likelihood_cut (ValLossHistoryCut, model.py:106-112): per sequence the first
 * ceil(train_percent*L) steps and the last floor((1-train_percent)*L) steps; out4 = {sum, count} of the train parts,
 * {sum, count} of the val parts (pre-zeroed). */
int seqrec_likelihood_cut(const float* P, const int32_t* lengths, int64_t n_seqs, int T, int skip_first,
                          double train_percent, double* out4, void* stream);

/* ranking metrics from per-token ranks (n, 0 = pad): for q < n_ks, out[3q..3q+2] += {#(rank <= ks[q]), sum 1/rank,
 * sum 1/log2(rank+1)} over the ranks <= ks[q]; out[3 n_ks..3 n_ks+2] += the same sums over every rank > 0 (the first is
 * the number of scored tokens, the second the uncut MRR sum).  ks: n_ks int32 on the device, each >= 1; out (3 n_ks + 3
 * doubles) pre-zeroed.  Recall@k = out[3q] / n, MRR@k = out[3q+1] / n, NDCG@k = out[3q+2] / n. */
int seqrec_rank_metrics(const int32_t* rank, int64_t n, const int32_t* ks, int n_ks, double* out, void* stream);

/* ---- K8: global-norm clip + Adagrad (experiments_methods.py:41) or Adam -----------------------------------------
 * sumsq[0] (double, pre-zeroed) += sum g^2 */
int seqrec_sumsq(const float* g, int64_t n, double* sumsq, void* stream);
int seqrec_sumsq_rows(const float* g, const int32_t* rows, const int32_t* n_rows, int GH, int max_rows,
                      double* sumsq, void* stream);
/* The stored gradient g may be UN-normalised (a sum over tokens): gdenom[0] (device float, NULL = 1) is the global number
 * of unmasked steps the Keras objective divides by.  g' = g / gdenom; norm = sqrt(sumsq) / gdenom;
 * scale = (norm >= clipnorm) ? clipnorm/norm : 1 (clipnorm <= 0: no clip); a += (g'*scale)^2;
 * p -= lr*g'*scale/(sqrt(a)+eps) */
int seqrec_adagrad(float* p, const float* g, float* a, int64_t n, float lr, float eps, float clipnorm,
                   const double* sumsq, const float* gdenom, void* stream);
/* row-sparse variant over the touched rows; also re-zeroes those rows of g and their touched flags */
int seqrec_adagrad_rows(float* p, float* g, float* a, const int32_t* rows, const int32_t* n_rows, int32_t* touched,
                        int GH, int max_rows, float lr, float eps, float clipnorm, const double* sumsq,
                        const float* gdenom, void* stream);
/* Keras 2.0.x Adam with the same clip and 1/gdenom factor: g' = g * scale (scale as for seqrec_adagrad);
 * k = iterations[0] (device int64: updates applied before this one, advanced by the caller after the step, so a
 * launch captured in a CUDA graph uses the current k at every replay; never written here);
 * lr_e = lr / (1 + decay*k); lr_t = lr_e * sqrt(1 - beta_2^(k+1)) / (1 - beta_1^(k+1)) (double, once per block);
 * m = beta_1*m + (1-beta_1)*g'; v = beta_2*v + (1-beta_2)*g'^2; p -= lr_t * m / (sqrt(v) + eps) */
int seqrec_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta_1, float beta_2,
                float eps, float decay, float clipnorm, const double* sumsq, const float* gdenom,
                const int64_t* iterations, void* stream);
/* the same update over EVERY row of an (F, GH) table (dense semantics: untouched rows take g' = 0, their m and v
 * decay and p still moves); the gradient row is read only where touched[row] != 0, and those rows of g and their
 * touched flags are re-zeroed */
int seqrec_adam_table(float* p, float* g, float* m, float* v, int32_t* touched, int64_t F, int GH, float lr,
                      float beta_1, float beta_2, float eps, float decay, float clipnorm, const double* sumsq,
                      const float* gdenom, const int64_t* iterations, void* stream);

/* ---- Dropout (model.py:362-363, :371-372): inverted-dropout factors from a counter-based RNG ---------------------
 * out[i] = (u_i >= rate) ? 1/(1-rate) : 0 */
int seqrec_dropout_mask(float* out, int64_t n, float rate, uint64_t seed, uint64_t offset, void* stream);
/* the same factors with the stream position on the device: state[0] = offset of the next draw (advanced by n when the
 * launch completes), state[1] = internal ticket (0 between launches).  Lets a captured training step draw new factors
 * at every graph replay. */
int seqrec_dropout_mask_dev(float* out, int64_t n, float rate, uint64_t seed, uint64_t* state, void* stream);

/* ---- bf16 hi/lo operand staging for the tensor-core logits kernels ----------------------------------------------
 * src (rows, cols) fp32 (optionally times scale (rows, cols)) -> hi, lo bf16 with hi+lo ~= src to 16 mantissa bits.
 * transpose != 0 writes (cols, rows).  ld_out = leading dimension (elements) of the outputs. */
int seqrec_split_bf16(const float* src, const float* scale, uint16_t* hi, uint16_t* lo, int64_t rows, int64_t cols,
                      int64_t ld_out, int transpose, void* stream);

/* the same with BOTH layouts from one read of src: hi/lo (rows, cols; leading dimension ld_out) and hi_t/lo_t
 * (cols, rows; leading dimension ld_t) */
int seqrec_split_bf16_both(const float* src, const float* scale, uint16_t* hi, uint16_t* lo, uint16_t* hi_t,
                           uint16_t* lo_t, int64_t rows, int64_t cols, int64_t ld_out, int64_t ld_t, void* stream);

/* split + column sums in one pass: hi/lo (rows, cols) and colsum[c] += sum_r src[r,c] (colsum pre-zeroed, may be NULL);
 * feeds the dU GEMM (dxp operand) and db from one read of dxp */
int seqrec_split_bf16_colsum(const float* src, uint16_t* hi, uint16_t* lo, float* colsum, int64_t rows, int cols,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEQREC_B200_H_ */
