/* srfrd_b200.h -- C ABI of libsrfrd_b200.so: the B200 (sm_100a) kernels behind the SRFRD hot path.
 *
 * The reference (oss0430/SRFRD) has no native code and no FFI: every native instruction on its hot
 * path is reached through torch.nn modules.  Each entry point below therefore cites the reference
 * *Python* lines whose ATen/cuBLAS/cuDNN launches it replaces ("replaces: file:line", paths relative
 * to the upstream checkout).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into memory owned by the caller (torch-allocated); the
 *     library never allocates, frees or retains device memory between calls;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - return 0 = ok; non-zero = error, message via srfrd_last_error() (thread-local);
 *     invalid shapes / alignment are rejected before any launch.  There is NO CPU fallback;
 *   - activations are bf16 row-major with an explicit leading dimension (elements); ids are int64
 *     (the reference feeds torch.LongTensor, trainer.py:29); parameters, statistics, logits,
 *     gradients of parameters and the final hidden state are fp32;
 *   - "T" = B*L tokens, "H" = encoder width, "D" = item-table width, "F" = fake-embedding width.
 */
#ifndef SRFRD_B200_H
#define SRFRD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRFRD_ABI_VERSION 10
#if defined(__GNUC__)
#define SRFRD_API __attribute__((visibility("default")))
#else
#define SRFRD_API
#endif

SRFRD_API const char* srfrd_last_error(void);
SRFRD_API int srfrd_abi_version(void);
/* 0 if the current device is an sm_100 part; error otherwise (called once by the Python loader). */
SRFRD_API int srfrd_device_check(void);

/* ---- K1: embedding gather + positional add + fake concat / user-label add + pad mask + LayerNorm ----
 * replaces: SRFR_model.py:17-34 (SRFR_Embedding.forward), :98-99 (pad mask), :111 (first attention LN);
 *           :411-424 (SRFU_Embedding.forward); :620-628 (SASRec.log2feats head).
 * mode 0: x = E[seq]*item_scale + P[l]                         (SASRec, item_scale = sqrt(D))
 * mode 1: x = [E[seq] + P[l] || Fe[aux_ids[t]]]                (SRFR/SRFRN; aux_ids NULL -> all 0)
 * mode 2: x = E[seq] + P[l] + Ul[aux_ids[b]]                   (SRFU_*; aux_ids = per-sequence labels)
 * then x *= (seq != 0); optional outputs: x0_bf16 (T, ldx), x0_f32 (T, H) [bit-identical to torch],
 * q_bf16 = LayerNorm(x) (T, ldx) with stats (T, 2) = {mean, rstd} when ln_w != NULL. */
SRFRD_API int srfrd_embed_ln_fwd(const float* item_table, int64_t n_rows, int D, const float* pos_table,
                       const float* aux_table, int64_t n_aux, int F, int mode, const int64_t* seq,
                       const int64_t* aux_ids, int64_t B, int L, float item_scale, const float* ln_w,
                       const float* ln_b, float eps, void* x0_bf16, float* x0_f32, void* q_bf16, float* stats,
                       int ldx, float drop_p, uint64_t drop_seed, uint32_t drop_stream, const float* drop_step,
                       void* stream);

/* SRFU_B/F/R.get_Labels -- replaces SRFR_model.py:546-570.  kind 0 = B, 1 = F, 2 = R,
 * 3 = the truncating variant SRFRN.predict uses (SRFR_model.py:244). */
SRFRD_API int srfrd_srfu_labels(const int64_t* fake_ids, int64_t B, int L, int kind, int64_t* labels, void* stream);

/* K5: gradient of the input-sequence lookups into the item table (and fake / user-label table).
 * replaces: the embedding_dense_backward launches autograd issues for SRFR_model.py:22,31 / :415,421. */
SRFRD_API int srfrd_embed_bwd(const void* dx0_bf16, int ldx, const int64_t* seq, const int64_t* aux_ids, int64_t B, int L,
                    int D, int F, int mode, float item_scale, float* d_item, float* d_aux, void* stream);

/* ---- LayerNorm (eps 1e-8 in the reference, SRFR_model.py:77,80,86) ----
 * fwd: y[t] = LN(x[t*row_stride + row_offset]); row_stride/offset select e.g. only the last position.
 * bwd: dx = LN'(dy) (+ add) (* (row_ids != 0)); dw/db accumulated with atomics. */
SRFRD_API int srfrd_layernorm_fwd(const void* x_bf16, int ldx, const float* w, const float* b, float eps, void* y_bf16,
                        float* y_f32, int ldy, float* stats, int64_t T, int H, int64_t row_stride,
                        int64_t row_offset, void* stream);
SRFRD_API int srfrd_layernorm_bwd(const void* dy_bf16, const float* dy_f32, int lddy, const void* x_bf16, int ldx,
                        const float* stats, const float* w, const void* add_bf16, int ldadd,
                        const int64_t* row_ids, void* dx_bf16, int lddx, float* dw, float* db, int64_t T, int H,
                        void* stream);

/* ---- tcgen05 GEMMs ----
 * replaces: the cuBLAS / cuDNN launches behind nn.MultiheadAttention's in/out projections
 * (SRFR_model.py:83,112), PointWiseFeedForward's two 1x1 Conv1d (:41,44,47-51) and last_conv (:76,123),
 * plus their autograd backward. */
typedef struct {
  const float* bias;       /* [N] or NULL */
  const void* residual;    /* bf16 [M, ldr] or NULL: added after bias/dropout/relu/gate */
  const void* gate;        /* bf16 [M, ldg] or NULL: v *= (gate > 0)   (ReLU backward) */
  const int64_t* row_ids;  /* [M] or NULL: v *= (row_ids[m] != 0)       (pad re-mask) */
  void* out_bf16;          /* [M, ldc] or NULL */
  float* out_f32;          /* [M, ldc] or NULL */
  int ldr, ldg, ldc;
  int relu;
  float drop_p;            /* 0 = no dropout; keep = hash(drop_seed ^ step, drop_stream, m*N+n) >= p */
  uint32_t drop_stream;
  uint64_t drop_seed;
  const float* drop_step;  /* device scalar mixed into the seed (the Adam step counter) or NULL: lets a
                              captured CUDA graph draw a fresh mask on every replay */
  /* Optional fused LayerNorm of the result row (the LayerNorm that follows the residual add in the reference,
   * SRFR_model.py:113-118 / :100-104): ln_out[m, :] = LN(bf16(out[m, :])) * ln_w + ln_b, ln_stats[m] = (mean, rstd).
   * Needs residual, out_bf16, N <= 128 and N a multiple of 16; NULL ln_out = off. */
  void* ln_out_bf16;       /* [M, ld_ln] or NULL */
  const float* ln_w;       /* [N] */
  const float* ln_b;       /* [N] */
  float* ln_stats;         /* [M, 2] or NULL */
  int ld_ln;
  float ln_eps;
} srfrd_gemm_epilogue_t;

/* C[M,N] = epilogue(A[M,K] . B[N,K]^T), A and B bf16 K-major. */
SRFRD_API int srfrd_gemm_tn(const void* A_bf16, int lda, const void* B_bf16, int ldb, int M, int N, int K,
                  const srfrd_gemm_epilogue_t* ep, void* stream);
/* The tile / pipeline plan srfrd_gemm_tn would use for a shape, without launching anything (no device needed): out[11] =
 * {block_n, n_tiles, stages, kgroup (K blocks per stage), b_resident, nacc (TMEM accumulator stages), nbuf (tile buffers),
 *  buf_blocks, dynamic shared memory bytes, second MMA issuer active, K blocks}.  Used by the CPU tests to check the host
 * logic for every shape and to feed the pipeline-protocol model check with the real configurations. */
SRFRD_API int srfrd_gemm_tn_plan(int M, int N, int K, int has_aux, int bf16_out, int fused_ln, int* out);
/* dW[Mo,No] += sum_t dY[t,Mo] * X[t,No]  (fp32 atomics into dW; split over tokens).
 * dbias (nullable): dbias[Mo] += sum_t dY[t,Mo], from one extra N=16 MMA per K step against an all-ones operand. */
/* profiling experiments only: with SRFRD_GEMM_DEBUG=5 gemm_tn records a clock64 timeline of CTA 0 (32 x 16 int64). */
SRFRD_API int srfrd_gemm_debug_read(long long* host_dst);
/* same for attention_fwd with SRFRD_ATTN_DEBUG=5 (16 x 16 int64). */
SRFRD_API int srfrd_attn_debug_read(long long* host_dst);

SRFRD_API int srfrd_gemm_wgrad(const void* dY_bf16, int lda, const void* X_bf16, int ldb, int64_t T, int Mo, int No,
                     float* dW, int ldw, float* dbias, void* stream);
/* SIMT cross-check used by the GPU tests only. */
SRFRD_API int srfrd_gemm_ref(const void* A, int lda, const void* B, int ldb, float* C, int ldc, int M, int N, int K,
                   int a_mn_major, int b_mn_major, void* stream);

/* out[n] += sum_m X[m, n]   (bias gradients; positional-table gradient through the (B, L*ld) view) */
SRFRD_API int srfrd_colsum(const void* X_bf16, int64_t M, int N, int64_t ld, float* out, void* stream);
/* out[(n / seg_in) * seg_out + n % seg_in] += in[n] for n % seg_in < seg_out; `in` is consumed (zeroed) */
SRFRD_API int srfrd_add_segments(float* in, int64_t n, int seg_in, int seg_out, float* out, void* stream);

/* out = keep(seed ^ step, stream_id, m*N+n) ? x / (1-p) : 0  -- re-applies a forward dropout mask to a
 * gradient (same hash as the forward kernels, nothing is stored). */
SRFRD_API int srfrd_dropout_apply(const void* x_bf16, int ldx, void* out_bf16, int ldo, int64_t M, int N, float drop_p,
                        uint64_t seed, uint32_t stream_id, const float* drop_step, void* stream);

/* fp32 master weights -> bf16 GEMM operands (W and W^T), one launch for the whole table of matrices. */
typedef struct {
  const float* src; int src_ld;   /* (rows, cols) fp32 */
  void* dst; int dst_ld;          /* bf16 (rows, cols) or NULL */
  void* dst_t; int dst_t_ld;      /* bf16 (cols, rows) or NULL */
  int rows, cols;
  int dst_is_f32;                 /* 1: dst is fp32 (zero-padded shadow of a bias / LayerNorm vector), dst_t unused */
} srfrd_cast_desc_t;
SRFRD_API int srfrd_cast_weights(const srfrd_cast_desc_t* descs_dev, int n, void* stream);
/* hi[r] = bf16(src[row_index ? row_index[r] : r]); lo = bf16(src - hi) (lo, row_index may be NULL).
 * With row_index this is the candidate-row gather of predict() (SRFR_model.py:148). */
SRFRD_API int srfrd_f32_to_bf16_split(const float* src, int64_t src_ld, const int64_t* row_index, void* hi, void* lo,
                            int64_t rows, int cols, int dst_ld, void* stream);

/* ---- causal self-attention ----
 * replaces: F.multi_head_attention_forward need_weights branch reached from SRFR_model.py:112
 * (q scaling, baddbmm, softmax, dropout, bmm) and its backward.  k and v share ldkv.
 * tcgen05 kernels for maxlen <= 128 (one 128-token window of whole sequences per tile) and for 128 < maxlen <= 256
 * (two query tiles per sequence); SIMT otherwise.  `stats` (fp32, 4 per (token, head): max * scale * log2e, 1 / sum,
 * delta, -) is written by the forward when non-NULL; the backward of maxlen > 128 needs it together with the forward
 * output `o` (FlashAttention-2 style independent tile pairs); both may be NULL for maxlen <= 128. */
SRFRD_API int srfrd_attention_fwd(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo,
                        float* stats, int64_t B, int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id,
                        const float* drop_step, void* stream);
SRFRD_API int srfrd_attention_bwd(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v, int ldkv,
                        const void* o, int ldo, float* stats, void* dq, int lddq, void* dk, void* dv, int lddkv, int64_t B,
                        int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id, const float* drop_step,
                        void* stream);

/* ---- K4: pos/neg scoring + (discriminator-weighted) BCE ----
 * replaces: SRFR_model.py:129-136 (SRFRN :225-233, SASRec :657-661) and trainer.py:31-38.
 * fake_table != NULL selects SRFRN rows E[id] || Fe[fake_id].
 * score_loss_fused: z+- (optional out), loss_acc[0] += sum w+ softplus(-z+), loss_acc[1] += sum w- softplus(z-),
 *   dz+ = w+ (sigmoid(z+) - 1) / norm[0], dz- = w- sigmoid(z-) / norm[1], dh = dz+ E[pos] + dz- E[neg],
 *   d_item[pos] += dz+ h, d_item[neg] += dz- h (row 0 never written: padding_idx).  w NULL -> 1[pos != 0]
 *   which reproduces trainer.py:36-38 exactly. */
SRFRD_API int srfrd_score_fwd(const float* h, int ldh, const float* item_table, const float* fake_table, const int64_t* pos,
                    const int64_t* neg, const int64_t* prs, const int64_t* nrs, int64_t T, int D, int F, float* zp,
                    float* zn, void* stream);
SRFRD_API int srfrd_score_bwd(const float* h, int ldh, const float* item_table, const float* fake_table, const int64_t* pos,
                    const int64_t* neg, const int64_t* prs, const int64_t* nrs, const float* dzp, const float* dzn,
                    int64_t T, int D, int F, float* dh, int lddh, float* d_item, float* d_fake, void* stream);
SRFRD_API int srfrd_score_loss_fused(const float* h, int ldh, const float* item_table, const float* fake_table,
                           const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                           const float* w_pos, const float* w_neg, const float* norm, int64_t T, int D, int F,
                           float* zp, float* zn, float* loss_acc, float* dh, int lddh, float* d_item, float* d_fake,
                           void* stream);
SRFRD_API int srfrd_weight_sums(const int64_t* pos, const float* w_pos, const float* w_neg, int64_t T, float* out2,
                      void* stream);
/* loss = acc2[0] / norm2[0] + acc2[1] / norm2[1]; the accumulators are consumed (zeroed for the next step). */
SRFRD_API int srfrd_loss_finalize(float* acc2, const float* norm2, float* loss, void* stream);

/* ---- K7: Adam(lr, betas, eps), dense, torch.optim.Adam arithmetic (trainer.py:390) ----
 * state3 = {step, 1-beta1^step, 1-beta2^step} lives on the device (CUDA-graph replayable). */
SRFRD_API int srfrd_adam_tick(float* state3, float beta1, float beta2, void* stream);
SRFRD_API int srfrd_adam_step(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                    const float* state3, int zero_grad, void* stream);

/* The tail of a training step in ONE launch: srfrd_adam_tick + srfrd_adam_step + srfrd_loss_finalize (acc2 nullable).
 * state8 = {step, 1-beta1^step, 1-beta2^step, uint32 step bits (seed of dropout / sampler), int scratch counter, -, -, -}:
 * every block derives the new state from the old one, the last block to finish publishes it.
 * Optional l2_emb regulariser (replaces: trainer.py:31-39, loss += l2_emb * torch.norm(param) for every parameter):
 * l2_seg = the device segment table of srfrd_param_l2, l2_coef / l2_reg its outputs.  Each element's gradient becomes
 * g + l2_coef[t] * p (t = the tensor holding it, p before this update) and loss[0] gains l2_reg[0]; needs acc2 and
 * n % 4 == 0.  l2_seg = NULL (l2_n_seg, l2_coef, l2_reg ignored) is the plain step. */
SRFRD_API int srfrd_adam_step_fused(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                          float eps, float* state8, int zero_grad, float* acc2, const float* norm2, float* loss,
                          void* stream, const int64_t* l2_seg, int l2_n_seg, const float* l2_coef, const float* l2_reg);

/* ---- l2_emb regulariser: per-tensor L2 norms of the flat parameter buffer (replaces: trainer.py:37-39) ----
 * seg = {offset, numel} per parameter tensor (int64 pairs, offsets 4-aligned and increasing, the gaps between tensors
 * are never read), at most 256 tensors.  Writes coef[t] = l2 / ||p_t|| (0 when ||p_t|| == 0, as torch's gradient of the
 * norm of a zero tensor is 0) and reg[0] = l2 * sum_t ||p_t||.  The buffer is cut into fixed 8192-float chunks that do
 * not cross tensors; sums of squares are accumulated and reduced in fp64 in a fixed order (no float atomics), so the
 * outputs are bit-identical across launches and ranks.  srfrd_param_l2_plan (host arithmetic on a HOST copy of seg)
 * returns the chunk count; ws = n_chunks + 1 doubles, zero-initialised once (word 0 is a counter the kernel leaves 0). */
SRFRD_API int srfrd_param_l2_plan(const int64_t* seg_host, int n_seg, int64_t* n_chunks);
SRFRD_API int srfrd_param_l2(const float* p, const int64_t* seg, int n_seg, int64_t n_chunks, float l2, float* coef,
                   float* reg, double* ws, void* stream);

/* ---- K8/K9: full-catalogue scoring fused with a streaming per-row top-k, 1 <= k <= SRFRD_TOPK_KMAX ----
 * replaces: SRFR_model.py:144-152 predict() called with label = arange(1, N+1) + the double argsort of
 * utils.py:591, i.e. rank by (score desc, item id asc).
 * List length rule: every list below is L = max(k, 10) entries long -- the (U, chunks, L) partial lists, the packed
 * wire row of 2L words and the input lists of srfrd_merge_topk / srfrd_merge_topk_packed.  k <= 10 runs the top-10
 * kernels (a smaller k is the prefix of the top-10, exact under the tie-break); k > 10 runs their k-list variants,
 * which only the unit form serves (n_split * D <= 256) and whose per-row lists must fit shared memory: the plan refuses
 * a k above srfrd_catalogue_topk_kmax(D, n_split) (64 at D = 64 and at D = 128 with one split, 48 at D = 256).
 * feats: bf16 (n_split stacked blocks of u_pad rows, D); table: bf16 (n_rows, D); candidates are local
 * rows [row_lo, n_rows) with global id = id_base + row.  Writes (U, chunks, L) partial lists whose chunk 0 holds each
 * user's exact local top-k, sorted, (-inf, -1) past the end, the other chunks emptied (ids -1); srfrd_merge_topk reduces
 * them (also used for the cross-GPU merge).  For k > 10 the merge inputs must be such sorted lists. */
#define SRFRD_TOPK_KMAX 64
SRFRD_API int srfrd_catalogue_topk_plan(int64_t U, int64_t n_rows, int64_t row_lo, int D, int n_split, int* chunks_out,
                                        int k);
/* largest k the plan accepts for this width and split (10 where only the tile form runs) */
SRFRD_API int srfrd_catalogue_topk_kmax(int D, int n_split, int* kmax_out);
SRFRD_API int srfrd_catalogue_topk(const void* feats_bf16, int64_t U, int64_t u_pad, int n_split, const void* table_bf16,
                         int64_t n_rows, int64_t row_lo, int64_t id_base, int D, int ld_feats, int ld_table,
                         int chunks, float* part_scores, int* part_ids, float* packed_out, void* stream, int k);
SRFRD_API int srfrd_merge_topk(const float* scores, const int* ids, int64_t U, int nlists, int k, float* out_scores,
                     int64_t* out_ids, void* stream);
/* Row-sharded scoring: packed_out (nullable, (U, 2L) fp32 words) receives each user's final local list as L fp32 scores
 * followed by L int32 global ids -- 8L B per user (80 B at k <= 10), the send buffer of ONE all-gather;
 * srfrd_merge_topk_packed merges the gathered (nlists, U, 2L) buffer (list l of user u at word (l * U + u) * 2L) into the
 * global top-k, identical on every rank. */
SRFRD_API int srfrd_merge_topk_packed(const float* packed, int64_t U, int nlists, int k, float* out_scores,
                            int64_t* out_ids, void* stream);
/* K8 rank form: exact full-catalogue rank of each user's held-out item (the reference's evaluation protocol,
 * utils.py:589-591, with every item as a candidate).  rank_out[u] (int32, zeroed by the call) receives the number of
 * local rows r in [row_lo, n_rows), global id i = id_base + r, i != target_ids[u], with score(u, i) > score(u, t) or
 * score(u, i) == score(u, t) and i < t.  Item scores are the streaming kernel's tensor-core scores (same operands and
 * splits as srfrd_catalogue_topk); score(u, t) is computed with SIMT fmaf from target_rows_bf16 (U rows of D bf16,
 * leading dimension ld_target: the target's row, passed in because under row sharding it usually lives on another
 * rank) in the order of the top-k re-scoring, and written to target_scores (nullable, fp32 (U,)).  The target is
 * excluded by id, never by score.  Row shards' counts add up to the global rank (one integer all-reduce).  Only the unit
 * form serves ranks (n_split * D <= 256); the tile form is refused before any launch.  Shape, alignment and null checks
 * as srfrd_catalogue_topk. */
SRFRD_API int srfrd_catalogue_rank(const void* feats_bf16, int64_t U, int64_t u_pad, int n_split,
                                   const void* table_bf16, int64_t n_rows, int64_t row_lo, int64_t id_base,
                                   int D, int ld_feats, int ld_table,
                                   const void* target_rows_bf16, int ld_target, const int64_t* target_ids,
                                   float* target_scores, int* rank_out, void* stream);

/* ---- full-catalogue softmax cross-entropy (opt-in training objective; no reference counterpart) ----
 * The logits are predict()'s (SRFR_model.py:144-152 with label = arange(1, N+1)) at every h row with a loss term:
 * z_rj = <h_r, E_j>, j = 1..N (row 0, the pad item, is never a candidate); loss = sum_r w_r (LSE_j z_rj - z_r,pos) / norm[0],
 * dh_r = (w_r / norm[0]) (sum_j p_rj E_j - E_pos),  dE_j = sum_r (w_r / norm[0]) (p_rj - 1[j = pos_r]) h_r,  dE_0 = 0.
 * The (rows, N) logits never reach memory.  Operands: h_bf16 (cap_rows, ldh) and table_bf16 ((n_items + 1), ldt) bf16
 * K-major rows padded with zeros to Dp columns (a multiple of 16, at most 256), 16-byte aligned with ld % 8 == 0;
 * fp32 accumulation and LSE; probabilities enter the second tcgen05 product as bf16.
 * Rows: rows = cap_rows, or min(cap_rows, rows_dev[0]) read on the device (packed token layout).  h row r belongs to
 * dense token row_tok[r] (-1: none; NULL: identity); pos / w_pos are indexed by the dense token.  A row carries a loss
 * term when its token exists, 1 <= pos <= n_items and its weight (w_pos, or 1 when w_pos is NULL) is non-zero.
 * srfrd_catalogue_ce_plan: host only; the shared-memory bytes, ring stages and TMEM columns of the kernels (any pointer
 * may be NULL); refuses a Dp the kernels cannot serve. */
SRFRD_API int srfrd_catalogue_ce_plan(int Dp, int64_t* smem_bytes, int* ring_stages, int* tmem_cols);
/* Pass 1: lse[r] (fp32, natural log) for r < rows, and loss_acc[0] += sum_r w_r (lse_r - z_r,pos) -- the unnormalised
 * loss; the read-out of srfrd_adam_step_fused / srfrd_dp_adam_step / srfrd_loss_finalize divides it by norm[0]. */
SRFRD_API int srfrd_catalogue_ce_fwd(const void* h_bf16, int ldh, const void* table_bf16, int ldt, int64_t n_items, int Dp,
                                     const int64_t* pos, const float* w_pos, const int* row_tok, const int* rows_dev,
                                     int64_t cap_rows, float* lse, float* loss_acc, void* stream);
/* Passes 2 and 3 from pass 1's lse; norm[0] is read on the device (0 -> every gradient is 0).  dh (nullable): rows
 * r < rows, first D columns, written (zero rows for rows without a loss term).  d_item (nullable, (n_items + 1, ldd)
 * fp32): dE added to the first D columns of rows 1..n_items; each item tile is owned by one CTA, so the result is
 * deterministic and needs no atomics. */
SRFRD_API int srfrd_catalogue_ce_bwd(const void* h_bf16, int ldh, const void* table_bf16, int ldt, int64_t n_items, int Dp,
                                     int D, const int64_t* pos, const float* w_pos, const float* norm, const int* row_tok,
                                     const int* rows_dev, int64_t cap_rows, const float* lse, float* dh, int lddh,
                                     float* d_item, int ldd, void* stream);

/* ---- on-device batch sampler (next row 8f #1) ----
 * replaces: WarpSampler_fr / sample_function_fr (utils.py:14-90) and the seven LongTensor.to(device) copies per
 * step (trainer.py:29).  CSR training interactions (offsets int64 (usernum+1), items int32, labels int8 {1 fake,
 * 2 real}, p_fake fp32 or NULL), `eligible` = 0-based rows of users with > 1 train item (utils.py:25).  Writes the
 * reference's batch layout: right-aligned, left-padded int64 (B, L) arrays seq / rsq / pos / prs / neg / nrs, the
 * chosen 1-based user ids (B) and, if w_pos != NULL, the discriminator weights of row L (policy 0 none, 1 mask,
 * 2 soft).  `step` (device fp32 counter, may be NULL) is mixed into the seed so graph replays draw new batches. */
SRFRD_API int srfrd_sample_batch(const int64_t* offsets, const int* items, const int8_t* labels, const float* p_fake,
                       const int* eligible, int n_eligible, int itemnum, int B, int L, int policy, uint64_t seed,
                       const float* step, int64_t* users, int64_t* seq, int64_t* rsq, int64_t* pos, int64_t* prs,
                       int64_t* neg, int64_t* nrs, float* w_pos, void* stream);

/* ---- sampled-candidate evaluation (row A10 / next row 8f #2) ----
 * replaces: the per-user loop of evaluation() / evaluation_with_label() (utils.py:558-597, :650-720): the rejection
 * draw of 100 negatives (utils.py:578-583), the batch-1 predict() call (utils.py:589 -> SRFR_model.py:144-152) and the
 * double argsort (utils.py:591).
 * sample_candidates: cand[u, 0] = target[users0[u]], cand[u, 1..C) = uniform ids in 1..itemnum not in the user's TRAIN
 *   row of the CSR (offsets, items).
 * candidate_rank: logits[u, c] = <feats[u, :D], E[cand[u, c]]> (+ <feats[u, D:D+F], Fe[user_label[u]]> when fake_table
 *   != NULL: SRFRN rows, SRFR_model.py:244-257); rank[u] = #{c >= 1 : logits[u, c] > logits[u, 0]}.  Ids outside
 *   [0, n_rows) are clamped to row 0 and *err_flag (nullable device int) is set to 1 (the reference raises IndexError).
 * add_user_term: logits[u, 0..I) += <feats_tail[u, 0..F), Fe[label[u]]>  (the same SRFRN term for predict()). */
SRFRD_API int srfrd_sample_candidates(const int64_t* offsets, const int* items, const int* users0, const int* target,
                            int64_t U, int itemnum, int C, uint64_t seed, int64_t* cand, void* stream);
SRFRD_API int srfrd_candidate_rank(const float* feats, int ldf, const float* item_table, int64_t n_rows, int D,
                         const int64_t* cand, int64_t U, int C, const float* fake_table, int F,
                         const int64_t* user_label, float* logits, int ldl, int* rank, int* err_flag, void* stream);
SRFRD_API int srfrd_add_user_term(float* logits, int ldl, int64_t U, int I, const float* feats_tail, int ldf,
                        const float* fake_table, const int64_t* label, int F, void* stream);

/* ---- packed token layout: do not compute padding (SRFR_model.py:98-99, :113, :121) ----
 * The sampler's batches are mostly pad slots (88 % at C2).  A pad slot enters the encoder as x = 0 and is re-zeroed after
 * every block; with no key-padding mask it still is a key / value (k = b_k, v = b_v), identical for every pad of a
 * sequence.  The packed layout keeps per sequence ONE pad-representative row followed by the kept tokens (input id != 0,
 * or `keep` id != 0) in position order, rounded up with filler rows to a multiple of 128.  Attention weights the
 * representative's key column by the number of dropped pads before the query's position, which reproduces the dense
 * result exactly (forward and backward).  All maps are built on the device (srfrd_pack_plan; the row count is data
 * dependent and the step runs inside a CUDA graph); rows[0] is the dynamic row count every other kernel reads. */
typedef struct {
  int* rows;        /* [4] device: {M = rows incl. filler (multiple of 128), T' = real rows, attention tiles, 0} */
  int* cnt;         /* [B] scratch: kept tokens per sequence */
  int* seq_first;   /* [B + 1] first packed row of each sequence (its pad representative); [B] = T' */
  int* tok_row;     /* [B * L] packed row of each dense token, -1 = dropped pad */
  int* row_tok;     /* [cap] dense token (b * L + l) of each packed row, -1 = pad representative / filler row */
  int64_t* row_ids; /* [cap] input item id of the row, 0 for representative / kept pad / filler rows: the pad mask */
  int* row_info;    /* [cap][4] {first row of the row's sequence, one past its last row, float bits of the pad column's
                       weight for this row, position l}; 16-byte aligned */
  int* tile_row0;   /* [B + 130] first row of each attention tile (whole sequences, <= 128 rows); entry [tiles] = M */
  int* last_row;    /* [B] packed row that holds position L - 1 of each sequence (its representative if that slot is a pad) */
  int64_t cap;      /* capacity in rows, >= roundup(B * (L + 1), 128) */
} srfrd_pack_t;
/* seq, keep: (B, L) int64 (keep nullable).  B <= 16384; the attention tile plan is built only when L + 1 <= 128
 * (longer sequences use the row maps with the dense-layout attention kernels, see srfrd_unpack_rows). */
SRFRD_API int srfrd_pack_plan(const int64_t* seq, const int64_t* keep, int64_t B, int L, const srfrd_pack_t* pk, void* stream);
/* Dynamic row count for the row-wise entry points: after srfrd_set_row_limit(rows_dev), srfrd_gemm_tn (M), srfrd_gemm_wgrad
 * (T), srfrd_layernorm_fwd / _bwd (T) and srfrd_dropout_apply (M) launched from THIS host thread treat their row argument
 * as a capacity and process min(argument, *rows_dev) rows, *rows_dev being read on the device when the kernel runs
 * (a multiple of 128 for the GEMMs).  NULL restores static counts.  Thread-local; captured into CUDA graphs by value. */
SRFRD_API int srfrd_set_row_limit(const int* rows_dev);
/* K1 on the packed layout: output row t holds dense token row_tok[t] (id 0 -> a zero row).  Widths multiples of 8. */
SRFRD_API int srfrd_embed_ln_fwd_packed(const float* item_table, int64_t n_rows, int D, const float* pos_table,
                              const float* aux_table, int64_t n_aux, int F, int mode, const int64_t* seq,
                              const int64_t* aux_ids, int64_t B, int L, float item_scale, const float* ln_w,
                              const float* ln_b, float eps, void* x0_bf16, void* q_bf16, float* stats, int ldx,
                              float drop_p, uint64_t drop_seed, uint32_t drop_stream, const float* drop_step,
                              const int* row_tok, const int* rows_dev, int64_t cap_rows, void* stream);
/* y[t] = LN(x[row_index[t]]) for t < n (fp32 out): the final LayerNorm of each sequence's last position only. */
SRFRD_API int srfrd_layernorm_fwd_rows(const void* x_bf16, int ldx, const float* w, const float* b, float eps, float* y_f32,
                             int ldy, const int* row_index, int64_t n, int H, void* stream);
/* Causal attention over packed rows (tcgen05; L + 1 <= 128, head width a multiple of 16, one head or 64-column heads). */
SRFRD_API int srfrd_attention_packed_supported(int L, int H, int heads);
/* Whether the packed kernels can fold the attention out-projection in (SRFR_model.py:112-113, the out_proj of
 * F.multi_head_attention_forward): bit 0 forward, bit 1 backward.  Needs one head of at most 128 columns. */
SRFRD_API int srfrd_attention_packed_oproj_supported(int L, int H, int heads);
/* Trailing arguments (wo NULL: plain attention, o only): fused out-projection, residual add and LayerNorm, each row
 * exactly what srfrd_gemm_tn(o, wo, bias = bo, residual = res, ln_out = y, ...) computes:
 *     r = o wo^T + bo + res,   y = LayerNorm(r) * ln_w + ln_b,   ln_stats = (mean, rstd) per row     (bo, ln_stats nullable)
 * wo: the [H, H] weight (rows = output features, K-major), ldw its row pitch.  o is still written. */
SRFRD_API int srfrd_attention_fwd_packed(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo,
                               const srfrd_pack_t* pk, int L, int H, int heads, float drop_p, uint64_t seed,
                               uint32_t stream_id, const float* drop_step, void* stream, const void* wo, int ldw,
                               const float* bo, const void* res, int ldres, const float* ln_w, const float* ln_b,
                               float ln_eps, float* ln_stats, void* r, int ldr, void* y, int ldy);
/* Trailing arguments (dr NULL: dout is read): dout = dr woT^T is computed in the kernel (what srfrd_gemm_tn(dr, woT)
 * writes) and dout / lddo are ignored.  woT: the transposed [H, H] out-projection weight, ldw its row pitch. */
SRFRD_API int srfrd_attention_bwd_packed(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v,
                               int ldkv, void* dq, int lddq, void* dk, void* dv, int lddkv, const srfrd_pack_t* pk,
                               int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id,
                               const float* drop_step, void* stream, const void* dr, int lddr, const void* woT, int ldw);
/* K4 on the packed layout: h / dh are packed rows; ids, weights stay (B * L) dense and are reached through row_tok. */
SRFRD_API int srfrd_score_loss_fused_packed(const float* h, int ldh, const float* item_table, const float* fake_table,
                                  const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                                  const float* w_pos, const float* w_neg, const float* norm, int D, int F,
                                  float* loss_acc, float* dh, int lddh, float* d_item, float* d_fake,
                                  const int* row_tok, const int* rows_dev, int64_t cap_rows, void* stream);
/* K5 on the packed layout (+ the positional-table gradient, which the dense path takes from srfrd_colsum). */
SRFRD_API int srfrd_embed_bwd_packed(const void* dx0_bf16, int ldx, const int64_t* seq, const int64_t* aux_ids,
                           const int* row_tok, const int* rows_dev, int64_t cap_rows, int L, int D, int F, int mode,
                           float item_scale, float* d_item, float* d_aux, float* d_pos, void* stream);

/* Two chained GEMMs with square weights (N = K <= 128, multiple of 16) in ONE launch:
 *   mid = stage1(A W1^T):  + bias1, dropout (drop1), ReLU (relu1), gate (v = gate > 0 ? v : 0)       -> mid_out (bf16)
 *   out = stage2(mid W2^T): + bias2, dropout (drop2), + residual, * (row_ids != 0)                    -> out (bf16)
 *   optional ln_out = LayerNorm(out) * ln_w + ln_b with ln_stats = (mean, rstd)
 * replaces: PointWiseFeedForward's two 1x1 Conv1d (SRFR_model.py:41,44,47-51) in the forward (residual = A, the FFN input)
 * and their data-gradient pair in the backward (gate = h1, residual = the incoming gradient), i.e. two srfrd_gemm_tn
 * launches; the intermediate tile goes from epilogue 1 to MMA 2 through shared memory.  Honours srfrd_set_row_limit. */
typedef struct {
  const float* bias1; const float* bias2;     /* [N] or NULL */
  const void* gate; int ldg;                  /* bf16 [M, ldg] or NULL */
  int relu1;
  float drop1_p, drop2_p; uint32_t drop1_stream, drop2_stream; uint64_t drop_seed; const float* drop_step;
  const void* residual; int ldr;              /* bf16 [M, ldr]; NULL + residual_is_a = 1 (or == A): the A operand itself */
  int residual_is_a;
  const int64_t* row_ids;                     /* [M] or NULL */
  void* mid_out; int ldm;                     /* bf16 [M, ldm] */
  void* out; int ldc;                         /* bf16 [M, ldc] */
  void* ln_out; int ld_ln; const float* ln_w; const float* ln_b; float* ln_stats; float ln_eps;   /* ln_out NULL = off */
} srfrd_mlp2_t;
SRFRD_API int srfrd_mlp2_tn(const void* A_bf16, int lda, const void* W1_bf16, int ldw1, const void* W2_bf16, int ldw2, int M, int N,
                  const srfrd_mlp2_t* ep, void* stream);

/* Dead query tiles of the hybrid layout (maxlen > 128: srfrd_attention_fwd / _bwd run on the dense (B, L) tensors between
 * srfrd_unpack_rows / srfrd_pack_rows).  A 128-position query tile of a sequence whose positions are all dropped padding
 * produces outputs nobody reads (srfrd_pack_rows takes zeros for the representative's o / dq) and has dO = 0, so every
 * (query tile, key tile) pair with such a query tile contributes exactly nothing (SRFR_model.py:98-99, :121 re-mask those
 * rows).  srfrd_attention_live_items derives from the pack plan's tok_row (B * L) the first live query tile of every
 * sequence (q_lo, B ints) and the list of live (sequence, head, query tile) items (items, up to B * heads * ceil(L / 128)
 * ints; n_live[0] = their number).  After srfrd_set_attention_live(q_lo, items, n_live, tok_row) the maxlen > 128 attention
 * kernels launched from THIS host thread skip the dead tiles (forward and dQ: listed items only; dK / dV: pair loops
 * start at the first live query tile; the delta pre-pass writes 0 for dropped pad slots, whose dO is zero, without reading
 * them); four NULLs restore the full loops.  Thread-local; captured into CUDA
 * graphs by value.  Only valid while nothing reads the dense o / dq rows of dropped pad slots. */
SRFRD_API int srfrd_attention_live_items(const int* tok_row, int64_t B, int L, int heads, int* q_lo, int* items, int* n_live,
                               void* stream);
SRFRD_API int srfrd_set_attention_live(const int* q_lo, const int* items, const int* n_live, const int* tok_row);

/* Packed <-> dense row movement for sequence lengths whose attention kernels work on the dense (B, L) layout
 * (128 < maxlen <= 256): the row-wise bulk of a block runs on packed rows, attention on dense tensors.
 * unpack: dense[t] = packed[tok_row[t]]; a dropped pad slot takes its sequence's pad-representative row (mode 0: q, k, v)
 *         or zeros (mode 1: dO).   pack: packed[r] = dense[row_tok[r]]; representative rows take zeros (mode 0: o, dq) or
 *         the sum over the sequence's dropped pad slots (mode 1: dk, dv); filler rows zeros.  Up to 3 tensors per call. */
typedef struct {
  const void* src; int ld_s;   /* bf16 rows: packed (unpack) / dense (pack) */
  void* dst; int ld_d;         /* bf16 rows: dense (unpack) / packed (pack) */
  int W;                       /* columns, multiple of 8 */
  int mode;
} srfrd_repack_part_t;
SRFRD_API int srfrd_unpack_rows(const srfrd_repack_part_t* parts, int n_parts, const srfrd_pack_t* pk, int64_t B, int L,
                      void* stream);
SRFRD_API int srfrd_pack_rows(const srfrd_repack_part_t* parts, int n_parts, const srfrd_pack_t* pk, int64_t B, int L,
                    void* stream);

/* ---- data-parallel gradient exchange fused with Adam over NVLink peer memory (SURVEY.md 8e) ----
 * One launch per rank: reduce-scatter (rank r sums slice r of every rank's gradient bucket through peer pointers),
 * torch.optim.Adam arithmetic on that slice with the rank's own slice of the moments, all-gather (the new parameters are
 * written into every rank's parameter buffer, every rank's gradient slice is zeroed), loss read-out (rank 0 reduces the
 * two accumulators in the bucket's tail [n, n+1] and writes the loss to param[n] of every rank), entry / exit barriers
 * through release / acquire flags in each rank's signal words.  grad / param / signal pointer arrays are DEVICE arrays of
 * `world` peer-mapped pointers (torch.distributed._symmetric_memory buffer_ptrs_dev); buckets and parameter buffers hold
 * n + 4 floats; local4 = 4 zero-initialised device words (epoch, grid barrier).  Replaces an NCCL all-reduce of the bucket
 * followed by srfrd_adam_step_fused on every rank; with world == 1 it is the same arithmetic as srfrd_adam_step_fused.
 * l2_seg / l2_n_seg / l2_coef / l2_reg: the optional l2_emb term of srfrd_adam_step_fused, added once to the SUMMED
 * gradient of the owned slice (the slice is cut on float4 boundaries, not tensors); rank 0 adds l2_reg[0] to the loss. */
SRFRD_API int srfrd_dp_adam_step(float* const* grad_ptrs_dev, float* const* param_ptrs_dev, uint32_t* const* signal_ptrs_dev,
                       int rank, int world, int64_t n, float* m, float* v, float lr, float beta1, float beta2, float eps,
                       float* state8, const float* norm2, uint32_t* local4, void* stream, const int64_t* l2_seg,
                       int l2_n_seg, const float* l2_coef, const float* l2_reg);

#ifdef __cplusplus
}
#endif
#endif /* SRFRD_B200_H */
