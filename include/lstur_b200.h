/*
 * lstur_b200.h — C ABI of the B200-native LSTUR training/scoring hot path.
 *
 * Drop-in boundary for the path named in BASELINE.json (SURVEY.md §8b).  The
 * reference (nvagus/mnexp) is pure Python on Keras/TensorFlow: it has no FFI
 * of its own; its "operator API" for this path is the set of Keras layer call
 * sites in task/paper.py / task/cook.py / models.py.  Each entry point below
 * names the reference call site(s) it replaces.  The Python shim
 * (mnexp_b200/task/paper.py) implements the reference's model-builder surface
 * on top of these calls via ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions: every pointer is a DEVICE pointer owned by the caller (any
 * allocator), row-major, fp32 / int32 unless stated; `ld*` are leading
 * dimensions in elements; all work is enqueued on `stream`; return value is
 * LSTUR_OK or a negative LSTUR_ERR_* with text in lstur_last_error().  No
 * global state besides the thread-local error string; one plan per
 * stream/rank.  There is no CPU fallback.
 */
#ifndef LSTUR_B200_H_
#define LSTUR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define LSTUR_OK 0
#define LSTUR_ERR_ARG (-1)
#define LSTUR_ERR_CUDA (-2)
#define LSTUR_ERR_UNSUPPORTED (-3)
#define LSTUR_ERR_WORKSPACE (-4)

#define LSTUR_GEMM_RELU 1
#define LSTUR_GEMM_ACCUM 2
#define LSTUR_GEMM_PRECISE 4 /* lstur_gemm_tc only: 3-term fp16 split (~fp32 accuracy) */

/* user-encoder architectures (SURVEY.md §9.9; task/paper.py:596-626, task/cook.py:146-168) */
#define LSTUR_ARCH_INI 0       /* paper 'igru' / cook 'ingru': GRU(initial_state=user_emb) — LSTUR-ini  */
#define LSTUR_ARCH_CON_DENSE 1 /* paper 'gru': Dense([GRU ‖ user_emb])                    — LSTUR-con  */
#define LSTUR_ARCH_CON_CAT 2   /* paper 'ngru','hgru','dgru' / cook 'igru': [GRU ‖ user_emb]           */
#define LSTUR_ARCH_NOID 3      /* paper 'nigru' / cook 'gru': GRU only                                 */
#define LSTUR_ARCH_ADD 4       /* paper 'pgru' / cook 'agru': GRU + user_emb                           */
#define LSTUR_ARCH_VO 5        /* 'vo': user_emb only                                                  */
#define LSTUR_ARCH_AVG 6       /* paper 'niavg': GlobalAveragePoolingMaskSupport of the history (models.py:422-441) */
#define LSTUR_ARCH_INI_CAT 8   /* Seq2VecPaperId 'iigru': [GRU(initial_state=user_emb) ‖ user_emb2], task/paper.py:338-343 */
#define LSTUR_ARCH_INI_CON 7   /* paper 'iigru': Dense([GRU(initial_state=user_emb) ‖ user_emb2]), task/paper.py:614-619;
                                  the two tables are the column halves of one (n_users, Ue = G + U2) table */
#define LSTUR_ARCH_AVG_CAT 9   /* cook 'iavg': [GlobalAveragePoolingMaskSupport(history) ‖ user_emb], task/cook.py:155-157 */
#define LSTUR_ARCH_ATT 10      /* Seq2VecPaper 'att': SimpleAttentionMaskSupport(Masking(history)), task/paper.py:206-208 */
#define LSTUR_ARCH_ATT_CAT 11  /* cook 'iatt': [SimpleAttentionMaskSupport(history) ‖ user_emb], task/cook.py:158-160 */
#define LSTUR_ARCH_INI_ADD 12  /* cook 'inagru': GRU(initial_state=user_emb) + user_emb2, task/cook.py:177-183 (Ue = 2G) */
#define LSTUR_ARCH_ATT_PAIR 13 /* cook 'atgru', task/cook.py:184-190 as written: the 2G entries of [GRU ; user_emb] are 2G
                                  one-feature steps (expand_dims(x, -1), concatenate(axis=-2)); Masking() +
                                  SimpleAttentionMaskSupport (kernel (1,1)) pool them into ONE scalar per user (U = 1) */
#define LSTUR_ARCH_ALPHA 14    /* cook 'algru': models.AlphaAdd([GRU, user_emb]) = alpha h + (1 - alpha) u, task/cook.py:191-193,
                                  models.py:540-554 (alpha constrained to [0, 1] after every update) */
#define LSTUR_ARCH_LSTM_CAT 15 /* cook 'ilstm': [keras.layers.LSTM(history) ‖ user_emb], task/cook.py:161-163 */

#define LSTUR_SCORE_DOT 0      /* task/paper.py:446-447 */
#define LSTUR_SCORE_DNN 1      /* Dense(Hs, relu)([u ‖ d]) -> Dense(1), task/paper.py:448-451 */
#define LSTUR_SCORE_DDOT 2     /* tanh Dense(Hs) on both sides, then dot, task/paper.py:452-455 */
#define LSTUR_SCORE_DDOT_LINEAR 3 /* cook flavour: linear Dense(Hs) on both sides, task/cook.py:206-209 */

#define LSTUR_LOSS_SOFTMAX_CE 0   /* (1+K)-way softmax + categorical cross-entropy, task/paper.py:460-464, 657 */
#define LSTUR_LOSS_WEIGHTED_BCE 1 /* sigmoid + Seq2Vec.loss, task/paper.py:222-256, task/seq2vec.py:213-216     */

#define LSTUR_ACT_HARD_SIGMOID 0 /* Keras <= 2.2.x GRU recurrent_activation default */
#define LSTUR_ACT_SIGMOID 1      /* Keras >= 2.3 */

#define LSTUR_PREC_FP32 0    /* FFMA everywhere: verification mode, ~1e-6 of the oracle */
#define LSTUR_PREC_BF16_TC 1 /* title Conv1D on tcgen05 (bf16 in, fp32 accumulate in TMEM) */
#define LSTUR_PREC_FP16_TC 2 /* same instruction and rate with fp16 operands: 8x smaller rounding error */

const char* lstur_last_error(void);
const char* lstur_version(void);
/* number of kernels this library has launched so far in this process (bench.py "gpu_launches") */
unsigned long long lstur_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Fine-grained operators (each validated against oracle/ in tests/)
 * ---------------------------------------------------------------------------------------- */

/* Window.get_title(): np.stack([docs[i].title ...]) task/seq2vec.py:25-30; candidates
 * task/paper.py:538-541.  tokens[n,:] = doc_tokens[doc_ids[n],:]; ids outside [0,n_docs) read doc 0. */
int lstur_token_gather(int N, int L, int n_docs, const int* doc_tokens, const int* doc_ids, int* tokens,
                       cudaStream_t stream);

/* keras Embedding(mask_zero=False) + Dropout, task/paper.py:132-138,142,147, into the zero-haloed
 * title buffer Xp (N, L+KS-1, E) consumed by the fp32 conv GEMM. */
int lstur_embed_gather_pad(int N, int L, int E, int V, int KS, const float* word_emb, const int* tokens, float* Xp,
                           float dropout, unsigned seed, cudaStream_t stream);

/* Tensor-core news encoder (tcgen05/TMEM): Embedding + Dropout + Conv1D(F,3,'same',relu) + pad mask + Masking +
 * Dropout + SimpleAttentionMaskSupport in ONE kernel (task/paper.py:141-158, models.py:474-489).
 * emb_16: (V, lstur_tc_padded_e(E)) 16-bit table from lstur_pack_word_emb_16; wimg: lstur_tc_wimg_elems(E,F)
 * 16-bit elements from lstur_pack_conv_w_tc.  c_out_16 (n_titles,L,F) receives the attention input (saved for
 * backward).  fp16 != 0: IEEE half operands (10-bit mantissa, meets the 1e-3 parity bound); 0: bfloat16. */
int lstur_tc_set_trace(void* dev_buf);   /* profiling hook: clock64 stamps of CTA 0's warp roles; NULL disables */
int lstur_tc_supported(int L, int E, int F, int KS);
int lstur_tc_slot(int L);                /* rows of a title slot in the tensor-core kernels: 32 (L <= 31) or 64 (L <= 63) */
int lstur_tc_padded_e(int E);
long long lstur_tc_wimg_elems(int E, int F);
int lstur_pack_word_emb_16(long long V, int E, const float* word_emb, void* emb_16, int fp16, cudaStream_t stream);
int lstur_pack_conv_w_tc(int E, int F, const float* conv_w, void* wimg, int fp16, cudaStream_t stream);
int lstur_news_conv_tc_fwd(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                           const void* wimg, const float* conv_b, const float* att_w, const float* att_b,
                           void* c_out_16, float* pooled, float* att_a, float* att_wt, float dropout, unsigned seed,
                           int fp16, int max_ctas, cudaStream_t stream);

/* Title compaction (lstur_compact_titles): the news encoder of an all-pad title — every token 0, i.e. the left padding of
 * a short click history (task/seq2vec.py:23,46-49) — is identically zero in value and in gradient (pad mask,
 * task/paper.py:150-155), so the plan runs the tensor-core kernels over the ascending list of live titles only:
 * n_live (1), live_idx (N: original index of every live title), tokens_c (N,L: their tokens); scratch holds
 * lstur_compact_titles_scratch_ints(N) ints.  The
 * kernels below take the live count as a device scalar (n_titles_dev, NULL = all n_titles) and, where a tensor outside the
 * encoder is touched (pooled rows, d_pooled rows), the original title index (title_idx, NULL = identity). */
long long lstur_compact_titles_scratch_ints(int N);
int lstur_compact_titles(int N, int L, const int* tokens, int* scratch, int* live_idx, int* n_live, int* tokens_c,
                         cudaStream_t stream);

/* Same kernels with the X-dropout keep bits handed from the forward to the weight-gradient kernel (one byte per 16-byte
 * piece of an embedding row, lstur_tc_xmask_bytes) instead of replaying the dropout hash there; NULL = replay. */
size_t lstur_tc_xmask_bytes(int n_titles, int L, int E);
int lstur_news_conv_tc_fwd_m(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                             const void* wimg, const float* conv_b, const float* att_w, const float* att_b,
                             void* c_out_16, float* pooled, float* att_a, float* att_wt, float dropout, unsigned seed,
                             int fp16, int max_ctas, void* xmask_out, const int* n_titles_dev, const int* title_idx,
                             cudaStream_t stream);
int lstur_conv_wgrad_tc_m(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                          const void* dpre_img, float* d_conv_w, float dropout, unsigned seed, int fp16,
                          void* partial_ws, size_t partial_bytes, const void* xmask, float dpre_scale,
                          const int* n_titles_dev, cudaStream_t stream);
/* Conv1D INPUT gradient on tcgen05 (word-table training: Embedding(trainable=True), task/paper.py:132-138, main.py:36):
 * dx16 (n_titles, L, lstur_tc_padded_e(E)) 16-bit rows = out_scale * sum_j sum_f dPre[m+1-j, f] * conv_w[j, e, f], from
 * the dPre image of lstur_attn_pool_bwd_img (its img_scale multiplies through) and the transposed, tap-reversed weight
 * image of lstur_pack_conv_w_dgrad_tc (lstur_tc_wimg_dgrad_elems 16-bit elements). */
long long lstur_tc_wimg_dgrad_elems(int E, int F);
int lstur_pack_conv_w_dgrad_tc(int E, int F, const float* conv_w, void* wimg_d, int fp16, cudaStream_t stream);
int lstur_conv_dgrad_tc(int n_titles, int L, int E, int F, const void* dpre_img, const void* wimg_d, void* dx16,
                        float out_scale, int fp16, int max_ctas, const int* n_titles_dev, cudaStream_t stream);

/* Backward of the tensor-core news encoder: attention/ReLU/mask backward emitting dPre as 16-bit K-block images
 * (lstur_attn_pool_bwd_img; the image holds img_scale * dPre — a power-of-two loss scale that keeps the gradients of a
 * large-batch mean out of fp16's subnormal range), then the Conv1D weight gradient on tcgen05 (lstur_conv_wgrad_tc;
 * lstur_conv_wgrad_tc_m takes the image's scale as dpre_scale and divides it out). */
int lstur_attn_pool_bwd_img(int fp16, int N, int L, int F, const void* Cd_16, const float* a_in, const float* w_in,
                            const float* d_pooled, long long lddp, const float* att_w, void* dpre_img, float dropout,
                            float img_scale, float* d_att_w, float* d_conv_b, float* d_att_b, int accumulate,
                            float* partials, size_t partial_bytes, const int* n_titles_dev, const int* title_idx,
                            cudaStream_t stream);
size_t lstur_tc_dpre_img_bytes(int n_titles, int L, int F);
size_t lstur_tc_wgrad_partial_bytes(int n_titles, int E, int F);
int lstur_conv_wgrad_tc(int n_titles, int L, int E, int F, int V, const int* tokens, const void* emb_16,
                        const void* dpre_img, float* d_conv_w, float dropout, unsigned seed, int fp16,
                        void* partial_ws, size_t partial_bytes, cudaStream_t stream);

/* C[M,N] (+)= op(A).op(B) + bias, optional ReLU: keras Dense / Conv1D-as-GEMM / all weight gradients. */
size_t lstur_gemm_f32_workspace_bytes(int M, int N, int K, int* splits_out);
int lstur_gemm_f32(int transA, int transB, int M, int N, int K, const float* A, long long lda, const float* B,
                   long long ldb, float* C, long long ldc, const float* bias, int flags, void* workspace,
                   size_t workspace_bytes, cudaStream_t stream);

/* Same contract on the tensor cores (tcgen05, operands rounded to fp16 while staged, fp32 accumulate). */
size_t lstur_gemm_tc_workspace_bytes(int M, int N, int K);
int lstur_gemm_tc(int transA, int transB, int M, int N, int K, const float* A, long long lda, const float* B,
                  long long ldb, float* C, long long ldc, const float* bias, int flags, void* workspace,
                  size_t workspace_bytes, cudaStream_t stream);
/* TN product over a list of reduction rows: C[M,N] = sum_{k in k_rows[0..*k_count)} A[k,:M]^T B[k,:N] (A, B stored [K,.];
 * k_rows ascending device ints, k_count a device scalar <= K).  Used for the weight gradients of the step, whose
 * reduction rows — (user, step) rows of the GRU tensors, title rows of the Dense — are identically zero where the
 * history is padding: the same sum over half the rows. */
int lstur_gemm_tc_tn_rows(int M, int N, int K, const float* A, long long lda, const float* B, long long ldb, float* C,
                          long long ldc, const int* k_rows, const int* k_count, void* workspace, size_t workspace_bytes,
                          cudaStream_t stream);
/* NN / NT product over a list of rows: C[m,:] = A[m,:K] . op(B) (+ bias) (relu) for m in m_rows[0..*m_count) only (A stored
 * [M,K]); the other rows of C are left untouched.  The dense layers of the step run over (user, step) / title rows half of
 * which are padding: their result is never read (or is a constant the caller fills in). */
int lstur_gemm_tc_mrows(int transB, int M, int N, int K, const float* A, long long lda, const float* B, long long ldb, float* C,
                        long long ldc, const float* bias, int flags, const int* m_rows, const int* m_count, void* workspace,
                        size_t workspace_bytes, cudaStream_t stream);

/* pad mask + Masking + Dropout + models.SimpleAttentionMaskSupport (task/paper.py:150-158, models.py:474-489). */
int lstur_attn_pool_fwd(int N, int L, int F, float* C, long long title_stride, const int* tokens, const float* att_w,
                        const float* att_b, float* pooled, long long ldp, float* a_out, float* w_out, float dropout,
                        unsigned seed, cudaStream_t stream);
int lstur_attn_bwd_grid(int N);
int lstur_attn_pool_bwd(int N, int L, int Lrows, int F, const float* Cd, long long title_stride, const float* a_in,
                        const float* w_in, const float* d_pooled, long long lddp, const float* att_w, float* dPre,
                        long long dpre_title_stride, float dropout, float* d_att_w, float* d_conv_b, float* d_att_b,
                        int accumulate, float* partials, size_t partial_bytes, cudaStream_t stream);
int lstur_colsum(long long rows, int cols, const float* in, long long ld, float* out, int accumulate,
                 float* workspace, size_t workspace_bytes, cudaStream_t stream);

/* models.ComputeMasking(0) + multiply Lambda + Masking() (models.py:25-27, task/paper.py:644-645, 592). */
int lstur_hist_mask_apply(int rows, int L, int D, const int* tokens, float* H, long long ldh, float* hm, float* gm,
                          cudaStream_t stream);

/* user-ID Embedding lookup (task/paper.py:589-591), optional per-row scale (cook id_keep, task/cook.py:141-142). */
int lstur_row_gather(int B, int D, int n_rows, const float* table, const int* ids, const float* scale, float* out,
                     long long ldo, cudaStream_t stream);

/* keras GRU recurrence (task/paper.py:596-613); XW = H.Wx + b is a GEMM done by the caller.  lstur_gru_fwd/bwd run the
 * cluster kernels when lstur_gru_cluster_supported(), else the streaming kernels, which ignore row_order. */
int lstur_transpose(int rows, int cols, const float* in, float* out, cudaStream_t stream);
int lstur_gru_fwd(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                  const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH, float* HP,
                  float* RH, const int* row_order, cudaStream_t stream);
int lstur_gru_bwd(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                  const float* HP, const float* WhT, int rec_act, const float* dhT, long long lddh, float* dA,
                  float* dh0, long long lddh0, const int* row_order, cudaStream_t stream);
/* The two implementations behind lstur_gru_fwd/bwd.  _cluster: recurrent weights resident in the shared memory of a
 * thread-block cluster for the whole launch, state exchanged through distributed shared memory (gru_cl.cu);
 * row_order (B) optionally permutes the batch rows inside the kernel (length-sorted tiles skip padded steps) or NULL.
 * _streaming: weights streamed from L2 every step (any G <= 1024). */
int lstur_gru_cluster_supported(int B, int W, int G);
int lstur_gru_fwd_cluster(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                          const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH,
                          float* HP, float* RH, const int* row_order, cudaStream_t stream);
int lstur_gru_bwd_cluster(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                          const float* HP, const float* WhT, int rec_act, const float* dhT, long long lddh, float* dA,
                          float* dh0, long long lddh0, const int* row_order, cudaStream_t stream);
/* Tensor-core recurrence (tcgen05, fp16 hi/lo 3-term split, fp32 accumulate): same arguments and saved tensors as
 * lstur_gru_fwd_cluster.  Used by the plan in the tensor-core precision modes when lstur_gru_tc_supported(). */
int lstur_gru_tc_supported(int B, int W, int G);
int lstur_gru_fwd_tc(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                     const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH,
                     float* HP, float* RH, const int* row_order, cudaStream_t stream);
/* BPTT on the tensor cores; takes Wh itself (not its transpose).  Weights enter as fp16 (like the other backward
 * GEMMs of the tensor-core modes), the exchanged gradients as fp16 hi + lo under a power-of-two scale that follows the
 * cluster-wide max |d h|.  db_partial (optional, lstur_gru_tc_db_rows(B) x 3G): partial column sums of dA (the bias
 * gradient) per (32-row tile, 8-row group); their column sum over all rows is sum_{b,t} dA[b,t,:]. */
int lstur_gru_tc_db_rows(int B);
int lstur_gru_bwd_tc(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                     const float* HP, const float* Wh, int rec_act, const float* dhT, long long lddh, float* dA,
                     float* dh0, long long lddh0, const int* row_order, float* db_partial, cudaStream_t stream);
int lstur_gru_fwd_streaming(int B, int W, int G, const float* XW, const float* gm, const float* h0, long long ldh0,
                            const float* Wh, int rec_act, float* hT, long long ldo, float* Z, float* R, float* HH,
                            float* HP, float* RH, cudaStream_t stream);
int lstur_gru_bwd_streaming(int B, int W, int G, const float* gm, const float* Z, const float* R, const float* HH,
                            const float* HP, const float* WhT, int rec_act, const float* dhT, long long lddh,
                            float* dA, float* dh0, long long lddh0, cudaStream_t stream);

/* dot scorer + softmax + categorical_crossentropy fwd(+bwd) (task/paper.py:446-447, 460-464, 657);
 * sigmoid test head (task/paper.py:661-665). */
int lstur_score_softmax_ce(int B, int C, int D, const float* u, long long ldu, const float* d, long long ldd,
                           const float* label, float* logits, float* probs, float* loss_rows, float* loss_mean,
                           float* du, long long lddu, float* dd, long long lddd, float grad_scale,
                           cudaStream_t stream);
int lstur_score_sigmoid(long long n_pairs, int C, int D, const float* u, long long ldu, const float* d, long long ldd,
                        float* out, int apply_sigmoid, cudaStream_t stream);
/* Ragged test head over impressions of different sizes: out[j] = sigmoid(u[pair_row[j]] . d[pair_doc[j]]) (d[j] when
 * pair_doc is NULL), one warp per pair.  lstur_csr_rows: CSR offsets (n_rows + 1) -> row_of[j - offsets[0]] = the row
 * whose range [offsets[r], offsets[r+1]) holds j. */
int lstur_score_sigmoid_ragged(long long n_pairs, int D, const int* pair_row, const float* u, long long ldu,
                               const int* pair_doc, const float* d, long long ldd, float* out, cudaStream_t stream);
int lstur_csr_rows(int n_rows, const int* offsets, int* row_of, cudaStream_t stream);

/* Device-side sample assembly: train_gen / valid_gen + Window + Impression.negative_samples (task/paper.py:7-18,
 * 387-441, 669-694; task/seq2vec.py:17-53).  Every user's clicks form one stream (stream_docs[stream_off[u] ..
 * stream_off[u+1])); a sample s is a click c = sample_click[s] (global stream index); idx (B) picks the batch's samples.
 *   user_out (B)          click_user[c]
 *   hist_doc_out (B,W)    the W stream entries before hist_end, left-padded with 0 (bit-exact with Window);
 *                         hist_end = sample_hist_end[s], or c when sample_hist_end is NULL (the training rule).
 *                         click_time non-NULL (int32 seconds since the Days Window's zero, 2000-01-01): a slot j keeps
 *                         its doc only if click_time[j] + expire_seconds >= click_time[c] (64-bit sum), else doc 0.
 *   cand_doc_out (B,1+K)  [the click, K negatives drawn with replacement from neg_docs[neg_off[c] .. neg_off[c+1])]:
 *                         negative k of row b = neg_docs[n0 + rng_u32(seed, (row0 + b) * K + k) % n]. */
int lstur_assemble_samples(int B, int W, int K, const int* sample_click, const int* sample_hist_end, const int* idx,
                           const int* click_user, const int* click_time, long long expire_seconds, const int* stream_off,
                           const int* stream_docs, const int* neg_off, const int* neg_docs, unsigned seed, long long row0,
                           int* user_out, int* hist_doc_out, int* cand_doc_out, cudaStream_t stream);
/* lstur_assemble_samples(sample_hist_end = NULL, click_time = NULL, row0 = 0): training samples, no time window. */
int lstur_assemble_batch(int B, int W, int K, const int* sample_click, const int* idx, const int* click_user,
                         const int* stream_off, const int* stream_docs, const int* neg_off, const int* neg_docs,
                         unsigned seed, int* user_out, int* hist_doc_out, int* cand_doc_out, cudaStream_t stream);

/* Pieces of the 'dnn' / 'ddot' scorers (task/paper.py:448-455) and of 'niavg' (models.py:422-441) around the GEMMs:
 * pair rows [u[b] ‖ d[(b,c)]] (b = i / C, or pair_row[i] when pair_row is non-NULL) and their gradient split (du summed over the C candidates in a fixed order), the output
 * Dense(1), its backward (dhid, and dl*hid whose column sums are d w2), tanh and its backward, the masked mean. */
int lstur_pair_concat(long long n_pairs, int C, int U, int D, const float* u, long long ldu, const float* d,
                      long long ldd, float* out, const int* pair_row, cudaStream_t stream);
int lstur_pair_split(int B, int C, int U, int D, const float* dcat, float* du, long long lddu, float* dd, long long lddd,
                     cudaStream_t stream);
int lstur_rowdot_bias(long long n, int H, const float* h, const float* w, const float* bias, float* out,
                      cudaStream_t stream);
int lstur_dnn_out_bwd(long long n, int H, const float* hid, const float* w2, const float* dlogit, float* dhid,
                      float* whid, cudaStream_t stream);
/* Sigmoid-family head (Seq2VecPaper / Seq2VecPaperDot / Seq2VecPaperId): p = sigmoid(score) and the weighted binary
 * cross-entropy Seq2Vec.loss (task/seq2vec.py:213-216); dscores (optional) = grad_scale * dL_i/dscore_i with grad_scale
 * = 1/global batch.  lstur_dot_score_bwd: backward of score[(b,c)] = u[b] . d[(b,c)]. */
int lstur_bce_loss(long long n, const float* scores, const float* label, float gain, int negative_samples, float* probs,
                   float* loss_rows, float* loss_mean, float* dscores, float grad_scale, cudaStream_t stream);
int lstur_dot_score_bwd(int B, int C, int D, const float* u, long long ldu, const float* d, long long ldd,
                        const float* dscores, float* du, long long lddu, float* dd, long long lddd, cudaStream_t stream);
int lstur_fill(long long n, float v, float* x, cudaStream_t stream);
int lstur_tanh_fwd(long long n, float* x, cudaStream_t stream);
int lstur_tanh_bwd(long long n, const float* y, float* g, cudaStream_t stream);
int lstur_masked_mean_fwd(int B, int W, int D, const float* H, const float* mask, float* out, long long ldo,
                          cudaStream_t stream);
int lstur_masked_mean_bwd(int B, int W, int D, const float* dout, long long ldd, const float* mask, const float* keep,
                          float* dH, cudaStream_t stream);

/* models.SimpleAttentionMaskSupport over a sequence of W vectors per row (models.py:474-489; history pooling of
 * Seq2VecPaper 'att' task/paper.py:206-208 and cook 'iatt' / 'atgru' task/cook.py:158-160,184-190):
 * a = tanh(H.att_w + att_b); e = exp(a) * mask; w = e / (sum e + 1e-7); out = sum_t w_t H_t.  H (B,W,D) contiguous; a_out /
 * w_out (B,W) saved for backward (may be NULL).  Backward: dH = keep * (w dout + d pre att_w) (keep NULL = 1) and per-row
 * partials (B, D+1) = [d att_w | d att_b] to be column-summed (lstur_colsum) in a fixed order. */
int lstur_seq_attn_fwd(int B, int W, int D, const float* H, const float* mask, const float* att_w, const float* att_b,
                       float* out, long long ldo, float* a_out, float* w_out, cudaStream_t stream);
int lstur_seq_attn_bwd(int B, int W, int D, const float* H, const float* att_w, const float* a_in, const float* w_in,
                       const float* dout, long long ldd, const float* keep, float* dH, float* partial,
                       cudaStream_t stream);
/* key[b] = first unmasked step of row b (W if none).  Sorting the batch rows by this key (lstur_sort_unique_i32 ->
 * sorted_pos) gives the `row_order` of the recurrence kernels: rows of similar history length share a 32-row tile, and
 * a tile skips every step at which all of its rows are masked (left-padded histories, task/seq2vec.py:23,46-49). */
int lstur_first_live_step(int B, int W, const float* mask, int* key, cudaStream_t stream);
/* out[r,:cols] = bias (or 0 when NULL) for the rows with flags[r] == want: the rows a row-listed GEMM
 * (lstur_gemm_tc_mrows) leaves out get their constant result — Dense(0) = bias for an all-pad title. */
int lstur_fill_rows_where(int rows, int cols, const int* flags, int want, const float* bias, float* out, long long ld,
                          cudaStream_t stream);
/* keras Masking(): mask[r] = any_k(x[r,k] != 0) */
int lstur_rows_nonzero(long long rows, int D, const float* x, long long ld, float* mask, cudaStream_t stream);
/* y[r,:] = ay * y[r,:] + ax * x[r,:] on strided rows (keras.layers.add of cook 'inagru', task/cook.py:183) */
int lstur_add_rows(int rows, int D, float ax, const float* x, long long ldx, float ay, float* y, long long ldy,
                   cudaStream_t stream);
/* models.AlphaAdd (models.py:540-554): out = alpha a + (1 - alpha) b with a learned scalar alpha (device pointer);
 * backward writes d a, d b and row_partial[r] = sum_k dout (a - b) (column-sum it for d alpha). */
int lstur_alpha_add_fwd(int rows, int D, const float* alpha, const float* a, long long lda, const float* b, long long ldb,
                        float* out, long long ldo, cudaStream_t stream);
int lstur_alpha_add_bwd(int rows, int D, const float* alpha, const float* a, long long lda, const float* b, long long ldb,
                        const float* dout, long long ldd, float* da, long long ldda, float* db, long long lddb,
                        float* row_partial, cudaStream_t stream);
/* softmax + keras.losses.categorical_crossentropy against integer class labels (= one-hot targets): the auxiliary
 * vertical classifier of Seq2VecPaperSoftmaxDaysIdVertSup (task/paper.py:899-902, 973-990) and the vertical model of
 * ...VertAlt (:1128-1136).  logits (n, n_classes); probs / loss_rows / loss_mean / dlogits optional;
 * dlogits = scale * dL_row/dlogits (zero through a saturated clip, like Keras). */
int lstur_softmax_ce_labels(long long n, int n_classes, const float* logits, const int* label, float* probs,
                            float* loss_rows, float* loss_mean, float* dlogits, float scale, cudaStream_t stream);
/* g[i] = 0 where y[i] <= 0: backward of a relu Dense given its output y */
int lstur_relu_bwd(long long n, const float* y, float* g, cudaStream_t stream);
/* keras.constraints.MinMaxNorm(lo, hi) on a vector of independent scalars (AlphaAdd.alpha, models.py:545), applied after
 * the optimizer update: w <- w * clip(|w|, lo, hi) / (1e-7 + |w|). */
int lstur_minmaxnorm(int n, float lo, float hi, float* w, cudaStream_t stream);
/* keras.layers.LSTM(G)(Masking()(history)) of cook 'ilstm' (task/cook.py:161-163): recurrent part.  XW (B,W,4G) = H.Wx + b
 * precomputed, gate order i,f,c,o; masked steps carry (h, c); output = last h.  SI..STC (B,W,G) saved gates / previous
 * cell / previous state / tanh(c') (all NULL for inference).  Backward yields dA (B,W,4G), zero on masked steps; WhT is
 * Wh transposed (4G, G). */
int lstur_lstm_fwd(int B, int W, int G, const float* XW, const float* gm, const float* Wh, int rec_act, float* hT,
                   long long ldo, float* SI, float* SF, float* SG, float* SO, float* SCP, float* SHP, float* STC,
                   cudaStream_t stream);
int lstur_lstm_bwd(int B, int W, int G, const float* gm, const float* SI, const float* SF, const float* SG,
                   const float* SO, const float* SCP, const float* STC, const float* WhT, int rec_act, const float* dhT,
                   long long lddh, float* dA, cudaStream_t stream);

/* Per-impression AUC / nDCG@10 / nDCG@5 / MRR (Seq2VecPaperSoftmax.callback, task/paper.py:497-524; utils.py:106-124;
 * sklearn roc_auc_score): offsets (n_impr+1) index scores / labels; out (n_impr, 4); ties ordered by descending index. */
int lstur_ranking_metrics(int n_impr, const int* offsets, const float* scores, const float* labels, float* out,
                          cudaStream_t stream);

/* keras.optimizers.Adam (task/paper.py:656): dense, and row-sparse for embedding tables. */
int lstur_adam_dense(long long n, float* p, const float* g, float* m, float* v, float lr, int t, float beta1,
                     float beta2, float eps, float grad_scale, cudaStream_t stream);
int lstur_adam_rows(int max_rows, const int* n_rows_dev, int D, const int* rows, const float* g_rows, float* p,
                    float* m, float* v, float lr, int t, float beta1, float beta2, float eps, float grad_scale,
                    cudaStream_t stream);

/* Embedding backward = index dedup + segment-sorted scatter-add (deterministic). */
int lstur_sort_unique_i32(int n, const int* keys, int* sorted_pos, int* uniq, int* seg_start, int* inverse,
                          int* n_uniq, cudaStream_t stream);
int lstur_segment_sum_rows(int n, int D, const int* n_uniq, const int* seg_start, const int* sorted_pos,
                           const float* src, long long lds, float* out, cudaStream_t stream);
int lstur_rows_add(int max_rows, const int* n_rows_dev, int D, const int* rows, const float* g_rows, float* table,
                   cudaStream_t stream);
/* Word-table gradient (keras Embedding(trainable=True) backward, task/paper.py:132-138): d_word_emb (V,E) is overwritten
 * with sum over token positions p of scale * dX[p,:] * xdrop[p,:] grouped by tokens[p] — stable radix sort of the
 * positions by token + fixed-tree segment sums, no floating-point atomics (bit-reproducible).  E % 4 == 0, E <= 512.
 * _16: dX as the 16-bit rows of lstur_conv_dgrad_tc, xmask = the forward's keep bytes (or NULL);
 * _f32: dXp (n_titles, L+KS-1, E) = gradient of the zero-haloed title buffer of lstur_embed_gather_pad, whose dropout
 * stream (dropout, seed) is replayed. */
size_t lstur_word_grad_workspace_bytes(long long n_pos, int V, int E);
int lstur_word_grad_scatter_16(int n_titles, int L, int E, int V, const int* tokens, const void* dx16, int fp16,
                               float scale, const void* xmask, float* d_word_emb, void* workspace,
                               size_t workspace_bytes, const int* n_titles_dev, cudaStream_t stream);
int lstur_word_grad_scatter_f32(int n_titles, int L, int KS, int E, int V, const int* tokens, const float* dXp,
                                float dropout, unsigned seed, float scale, float* d_word_emb, void* workspace,
                                size_t workspace_bytes, cudaStream_t stream);
int lstur_axpby(long long n, float a, const float* x, float b, float* y, cudaStream_t stream);

/* Cook.get_doc_encoder concat (task/cook.py:99-113): doc_vec[n, col0 .. col0+dv) = vert_emb[doc_vert[doc_ids[n]]],
 * doc_vec[n, col0+dv .. +ds) = subvert_emb[doc_subvert[doc_ids[n]]]; the looked-up ids are kept in title_vert /
 * title_subvert (n) for the backward.  lstur_small_table_grad is the Embedding backward of such a small table:
 * d_table[r, :] = sum over titles n with ids[n] == r of d_doc_vec[n, col0 .. col0+dim), two-stage, fixed order. */
int lstur_vert_concat(int n, int D, int col0, int dv, int ds, int n_docs, int n_vert, int n_subvert, const int* doc_ids,
                      const int* doc_vert, const int* doc_subvert, const float* vert_emb, const float* subvert_emb,
                      float* doc_vec, int* title_vert, int* title_subvert, cudaStream_t stream);
size_t lstur_small_table_grad_workspace_bytes(int n_rows, int dim);
int lstur_small_table_grad(int n, int D, int col0, int dim, int n_rows, const int* ids, const float* d_doc_vec,
                           float* d_table, float* workspace, size_t workspace_bytes, cudaStream_t stream);
/* x[b, 0..D) *= scale[b]  (backward of the user-vector multiplier: dgru whole-vector dropout, cook id_keep) */
int lstur_scale_rows(int B, int D, const float* scale, float* x, long long ld, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------
 * Whole-path plan: Seq2VecPaperSoftmaxId._build_model (task/paper.py:635-665) /
 * Cook._build_model (task/cook.py:214-277) as one forward / backward / update sequence.
 * ---------------------------------------------------------------------------------------- */
typedef struct lstur_config {
  int B, W, C, L;      /* rows per rank, window_size, 1+negative_samples, title_shape        */
  int E, F, KS;        /* textual_embedding_dim, title_filter_shape = (F, KS)                 */
  int use_dense;       /* 1: Dense(F->Dd) after pooling (paper.py:159); 0: cook.py            */
  int Dd;              /* title-vector dim: user_embedding_dim if use_dense else F            */
  int dv, ds;          /* vertical / subvertical embedding dims, 0 = off (cook.py:99-113)     */
  int G, Ue, U;        /* GRU units, user-embedding dim, user-vector dim                      */
  int arch, score_model, rec_act, precision;
  int V, n_users, n_docs;
  float dropout;
  int save_for_backward; /* 0: inference plan (smaller workspace)                            */
  int n_vert, n_subvert; /* rows of the vertical / subvertical tables (16 / 307, utils.py:153-228) */
  int Hs;                /* hidden width of the 'dnn' / 'ddot' scorers (= user_embedding_dim), 0 for 'dot'   */
  int loss_model;        /* LSTUR_LOSS_SOFTMAX_CE | LSTUR_LOSS_WEIGHTED_BCE (then C == 1 and label is required) */
  int bce_neg;           /* negative_samples of the weighted BCE (task/seq2vec.py:213-216)                   */
  float gain;            /* its positive-class gain                                                           */
  int trainable_word_emb; /* textual_embedding_trainable (task/paper.py:136, main.py:36): lstur_backward_w also yields d word_emb */
  /* Seq2VecPaperSoftmaxDaysIdVertSup (task/paper.py:948-990): TimeDistributed vertical classifier Dense(aux_hidden, relu) ->
   * Dense(aux_nv, softmax) over the W + C news vectors of every row, loss = CE + aux_gain * mean CE_vertical; 0 = off.
   * Labels: the batch's hist_vert / cand_vert ids (or doc_vert[hist_doc / cand_doc]). */
  int aux_nv, aux_hidden;
  float aux_gain;
  /* Seq2VecPaperSoftmaxDaysIdVertAlt (task/paper.py:1128-1136): Dense(cls_nv, softmax) on the doc_encoder output, trained by
   * lstur_title_cls_forward / lstur_title_cls_backward on (title, vertical) batches; 0 = off */
  int cls_nv;
} lstur_config;

typedef struct lstur_weights {
  const float* dense;      /* flat dense parameters, layout from lstur_plan_dense_offset()    */
  const float* word_emb;   /* (V,E)                                                            */
  const float* user_emb;   /* (n_users,Ue) or NULL                                             */
  const int* doc_tokens;   /* (n_docs,L) or NULL when batches carry tokens                     */
  const int* doc_vert;     /* (n_docs) or NULL                                                 */
  const int* doc_subvert;  /* (n_docs) or NULL                                                 */
} lstur_weights;

typedef struct lstur_batch {
  const int* user;       /* (B)                                                                */
  const int* hist_doc;   /* (B,W) doc ids, left-padded with 0 — or NULL if hist_tok given      */
  const int* cand_doc;   /* (B,C) doc ids, positive first                                      */
  const int* hist_tok;   /* (B,W,L) tokens (reference data protocol, task/paper.py:538-541)    */
  const int* cand_tok;   /* (B,C,L)                                                            */
  const float* label;    /* (B,C) one-hot or NULL (= positive at column 0, task/paper.py:529)  */
  const float* user_scale; /* (B) multiplier on the user embedding or NULL (dgru / id_keep)    */
  /* cook .npz protocol (task/cook.py:14-17): vertical / subvertical ids per title slot next to the tokens, instead of
   * doc ids + the doc_vert / doc_subvert tables; all four or none */
  const int* hist_vert;    /* (B,W) */
  const int* hist_subvert; /* (B,W) */
  const int* cand_vert;    /* (B,C) */
  const int* cand_subvert; /* (B,C) */
  /* two-table archs (cook 'inigru' / 'inagru', task/cook.py:169-183: each id embedding has its OWN Dropout(1 - id_keep)
   * layer): multiplier of the second table's columns; NULL = user_scale applies to the whole row */
  const float* user_scale2; /* (B) */
} lstur_batch;

typedef struct lstur_plan lstur_plan;

int lstur_plan_create(const lstur_config* cfg, lstur_plan** out);
void lstur_plan_destroy(lstur_plan* plan);
/* The 16-bit operand copy of the word table is packed once and reused while the table is frozen (reference default,
 * main.py:36); call this after writing word_emb so the next lstur_forward re-packs it. */
int lstur_plan_invalidate_tables(lstur_plan* plan);
size_t lstur_plan_workspace_bytes(const lstur_plan* plan);
long long lstur_plan_dense_count(const lstur_plan* plan);
/* name in {conv_w, conv_b, att_w, att_b, dense_w, dense_b, vert_emb, subvert_emb, gru_wx, gru_wh, gru_b,
 * con_w, con_b}; returns LSTUR_ERR_ARG if the tensor does not exist in this configuration. */
int lstur_plan_dense_offset(const lstur_plan* plan, const char* name, long long* offset, long long* count);
/* named views into the workspace after forward/backward (for tests and the Python shim):
 * tokens, pooled, doc_vec, hist_mask, user_vec, logits, probs, loss, d_user_rows, user_rows, n_user_rows */
int lstur_plan_view(const lstur_plan* plan, void* workspace, const char* name, void** ptr, long long* count);

/* Measurement hook: record the two CUDA events (cudaEvent_t) around one kernel of the step. */
#define LSTUR_PROBE_NONE 0
#define LSTUR_PROBE_CONV_FWD 1
#define LSTUR_PROBE_CONV_WGRAD 2
#define LSTUR_PROBE_GATHER 3
#define LSTUR_PROBE_GRU_FWD 4
#define LSTUR_PROBE_CONV_DGRAD 5
#define LSTUR_PROBE_SCATTER 6
#define LSTUR_PROBE_ATTN_BWD 7
#define LSTUR_PROBE_GRU_BWD 8
int lstur_plan_set_probe(lstur_plan* plan, int probe_id, void* start_event, void* stop_event);
/* Data-parallel overlap: `event` (cudaEvent_t) is recorded by lstur_backward as soon as every gradient except the
 * title-encoder bucket — the first lstur_plan_dense_head_count() floats of the arena: conv_w, conv_b, att_w, att_b — and
 * the user-row gradients are final; the exchange of the rest can then run on another stream under the ~2 ms of
 * attention backward + conv weight gradient that remain. */
#define LSTUR_EVENT_TAIL_GRADS_READY 1
int lstur_plan_set_event(lstur_plan* plan, int which, void* event);
long long lstur_plan_dense_head_count(const lstur_plan* plan);
int lstur_stream_wait_event(cudaStream_t stream, void* event);
int lstur_event_record(void* event, cudaStream_t stream);
int lstur_event_create(void** ev);
int lstur_event_destroy(void* ev);
int lstur_event_elapsed_ms(void* start_event, void* stop_event, float* ms);

int lstur_forward(const lstur_plan* plan, const lstur_weights* w, const lstur_batch* b, void* workspace,
                  int training, unsigned seed, cudaStream_t stream);
/* Vertical model of Seq2VecPaperSoftmaxDaysIdVertAlt (task/paper.py:1128-1136; plan with cls_nv > 0):
 * Dense(cls_nv, softmax)(doc_encoder(title)) + categorical cross-entropy on n <= B*(W+C) titles.  tokens (n,L), labels (n)
 * device ints.  Workspace views afterwards: vc_probs (n, cls_nv), vc_loss_rows (n), vc_loss (1).  The backward fills the
 * whole dense-gradient arena (zero outside vcls_w / vcls_b and the title-encoder tensors) and word_grad when the word table
 * trains; grad_scale = 1 / (global number of titles). */
int lstur_title_cls_forward(const lstur_plan* plan, const lstur_weights* w, void* workspace, int n, const int* tokens,
                            const int* labels, int training, unsigned seed, cudaStream_t stream);
int lstur_title_cls_backward(const lstur_plan* plan, const lstur_weights* w, void* workspace, float* dgrad,
                             float* word_grad, float grad_scale, cudaStream_t stream);
/* dense_grad (dense_count floats) is overwritten.  User-embedding gradient is left as unique rows in the
 * workspace (views user_rows / d_user_rows / n_user_rows).  grad_scale multiplies d(loss): 1/global_batch. */
int lstur_backward(const lstur_plan* plan, const lstur_weights* w, const lstur_batch* b, void* workspace,
                   float* dense_grad, float grad_scale, cudaStream_t stream);
/* Same, for a plan with trainable_word_emb: word_grad (V,E) is overwritten with the dense gradient of the word table
 * (conv input gradient + segment-sorted scatter-add; rows of tokens absent from the batch are zero). */
int lstur_backward_w(const lstur_plan* plan, const lstur_weights* w, const lstur_batch* b, void* workspace,
                     float* dense_grad, float* word_grad, float grad_scale, cudaStream_t stream);

/* Decomposed inference (task/test_pipeline.py:37-211; BASELINE config 4): encode documents once, then run the user
 * encoder and scorer against the cached vectors.  lstur_encode_docs handles n <= B*(W+C) documents per call
 * (doc_ids on the device, weights->doc_tokens required); lstur_forward_docvecs gathers history / candidate vectors from
 * doc_vec_table (n_rows, ld == document-vector width) — an all-zero row (unknown / pad document) is a masked history
 * slot — and leaves probs / logits / user_vec in the workspace like lstur_forward. */
int lstur_encode_docs(const lstur_plan* plan, const lstur_weights* weights, void* workspace, int n, const int* doc_ids,
                      float* doc_vec_out, long long ldo, cudaStream_t stream);
/* The same encoder on explicit token rows (n, L) instead of document ids: `doc_encoder.predict(titles)`, the layer
 * TestPipeline fetches with get_layer('doc_encoder') (task/test_pipeline.py:27-35, task/paper.py:160). */
int lstur_encode_titles(const lstur_plan* plan, const lstur_weights* weights, void* workspace, int n, const int* tokens,
                        float* doc_vec_out, long long ldo, cudaStream_t stream);
int lstur_forward_docvecs(const lstur_plan* plan, const lstur_weights* weights, const lstur_batch* batch, void* workspace,
                          const float* doc_vec_table, long long ld, int n_rows, cudaStream_t stream);
/* Ranking of whole impressions (the evaluation pass of Seq2VecPaperSoftmax.callback, task/paper.py:497-524) against
 * cached document vectors doc_vec_table (n_rows, document-vector width), on an inference plan (save_for_backward = 0).
 * Impression i: user[i], history hist_doc[i, 0..W), candidates cand_doc[cand_off[i] .. cand_off[i+1]).
 * scores_out[j] = sigmoid(score(user vector of j's impression, doc_vec_table[cand_doc[j]])) with the plan's scorer ('dot',
 * 'dnn', 'ddot'): the test head's value, as LsturEngine.score_sigmoid after lstur_forward.  The user encoder runs once per
 * impression, on chunks of at most B impressions and B*C pairs; an impression of more than B*C candidates is
 * LSTUR_ERR_ARG.  A history slot is masked when its document's title is all zero tokens (weights->doc_tokens required),
 * as lstur_forward masks it; a candidate keeps its row of the table.  cand_off (n_impr + 1 ints) is HOST memory: the
 * chunks are cut on the host and each chunk's offsets copied to the device.  Every other array is on the device. */
int lstur_score_impressions(const lstur_plan* plan, const lstur_weights* weights, void* workspace, int n_impr,
                            const int* user, const int* hist_doc, const int* cand_off, const int* cand_doc,
                            const float* doc_vec_table, int n_rows, float* scores_out, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LSTUR_B200_H_ */
