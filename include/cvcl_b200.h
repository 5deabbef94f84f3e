/* cvcl_b200.h -- C ABI of libcvcl_b200.so: the B200 (sm_100a) implementation of the CVCL
 * contrastive image-utterance hot path of wkvong/multimodal-baby.
 *
 * The reference has no FFI for this path: its boundary is the Python class API of
 * multimodal/multimodal.py (MultiModalModel) whose arithmetic is dispatched to ATen.  Each
 * entry point below replaces the ATen op sequence of the cited reference lines; the Python
 * host (multimodal-baby_b200/) binds them with ctypes and registers them as torch.library ops.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated; the caller (torch) owns all memory,
 *     the library never allocates, frees or synchronises; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*), and is CUDA-graph capturable;
 *   - matrices are row-major; `ld*` are leading dimensions in ELEMENTS; bf16 operands that feed
 *     the tensor-core GEMMs must be 16-byte aligned with ld % 8 == 0 (TMA requirement);
 *   - token ids / lengths are int64 exactly as the reference's collate produces them
 *     (multimodal_data_module.py:98-109);
 *   - return 0 on success, <0 on error (CVCL_ERR_*); cvcl_last_error() gives the thread-local
 *     message.  Unsupported requests are errors, never fallbacks.  There is no CPU path.
 */
#ifndef CVCL_B200_H
#define CVCL_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVCL_ABI_VERSION 6
#define CVCL_OK 0
#define CVCL_ERR_INVALID (-1)
#define CVCL_ERR_UNSUPPORTED (-2)
#define CVCL_ERR_CUDA (-3)

int cvcl_abi_version(void);
const char* cvcl_last_error(void);
/* number of CUDA kernels this library has launched so far in the process (host-side counter). */
unsigned long long cvcl_launch_count(void);

/* Page-locked host staging memory for the per-step H2D copy (staging.PinnedBatchStager); write_combined != 0:
 * cudaHostAllocWriteCombined -- the CPU only writes it, the DMA engine never has to snoop CPU caches.  NULL on
 * failure (cvcl_last_error). */
void* cvcl_host_alloc(size_t bytes, int write_combined);
int cvcl_host_free(void* p);

/* ---- K1 text encoder, embedding branch ------------------------------------------------
 * replaces TextEncoder.forward (multimodal.py:496-503,575-584) + F.normalize (:743).
 * per_token = 0 (flat): feat[b] = normalise(sum_l table[ids[b,l]] / len[b]).
 * per_token = 1 (spatial): tok[b,l] = normalise(table[ids[b,l]]) (:498) and
 *   feat[b] = sum_l tok[b,l] * pool_scale / len[b] (the text factor of the "mean"
 *   similarity, :765-770).  Any output pointer may be NULL.  *status is set to 1 if an id is
 *   outside [0,V) (the reference raises IndexError). */
int cvcl_text_encoder_fwd(const int64_t* ids, const int64_t* lens, const float* table,
                          int B, int L, int E, int V, int normalize, int per_token, float pool_scale,
                          float* feat_f32, void* feat_bf16, int ld_bf16,
                          float* inv_norm, float* tok_f32, void* tok_bf16, int* status, void* stream);

/* text_outputs = embedding(ids) (multimodal.py:496,575-584): [n_tok, E] fp32 row gather. */
int cvcl_embedding_gather(const int64_t* ids, const float* table, float* out, int n_tok, int E, int V,
                          void* stream);

/* autograd of nn.Embedding(padding_idx=0): dtable[ids[b,l]] += g[b] (flat, g [B,E]) or
 * += g[b*L+l] (per_token, g [B*L,E]); row 0 untouched.  dtable must be pre-zeroed. */
int cvcl_embedding_scatter_add(const int64_t* ids, const float* g, float* dtable, int B, int L, int E,
                               int V, int per_token, void* stream);

/* spatial text backward: F.normalize backward per token + scatter-add (dtok [B*L,E] and/or
 * dpool [B,E], either may be NULL). */
int cvcl_text_token_bwd(const int64_t* ids, const int64_t* lens, const float* table, const float* dtok,
                        const float* dpool, float pool_scale, float* dtable, int B, int L, int E, int V,
                        int normalize, void* stream);

/* ---- casts / transposes feeding the GEMMs ------------------------------------------------
 * src [batch][R][C] (fp32, or bf16 if src_is_bf16) -> dst [batch][R][C] bf16 and/or
 * dst_t [batch][C][R] bf16.  bs_* are batch strides in elements. */
int cvcl_cast_transpose(const void* src, int src_is_bf16, void* dst, void* dst_t, int batch, int R, int C,
                        int64_t ld_src, int64_t ld_dst, int64_t ld_t, int64_t bs_src, int64_t bs_dst,
                        int64_t bs_t, void* stream);

/* stand-alone backward of the flat text encoder (encode_text differentiated on its own):
 * dm = F.normalize-backward(g [B,E]; feat, inv_norm) / len, then the embedding scatter-add. */
int cvcl_embedding_bag_bwd(const int64_t* ids, const int64_t* lens, const float* g, const float* feat,
                           const float* inv_norm, int normalize, float* dtable, int B, int L, int E, int V,
                           void* stream);

/* stand-alone F.normalize backward on rows (autograd of multimodal.py:736,743):
 * du = (g - feat <feat,g>) * inv_norm -> fp32 [M,E] / bf16 [M,ld] / bf16^T [E,ld_t] / dbias += sum. */
int cvcl_rownorm_bwd(const float* g, const float* feat, const float* inv_norm, int M, int E, int normalize,
                     float* du_f32, void* du_bf16, int ld, void* du_bf16_t, int ld_t, float* dbias,
                     void* stream);

/* sum over the H*W locations of a [B,HW,E] fp32 map: image factor of the spatial "mean"
 * similarity (multimodal.py:765-770). */
int cvcl_spatial_pool(const float* src, int B, int HW, int E, float* out_f32, void* out_bf16, int ld,
                      void* out_bf16_t, int ld_t, void* stream);
/* C [M,N] fp32 = A [M,K] . W[N,K]^T + bias [N], fp32 operands and fp32 FMA accumulation (no tensor cores): the
 * exact-mode projection head of the evaluation path (reference fc in fp32, multimodal.py:186-192, called per trial
 * from eval.py:196-214).  K % 4 == 0. */
int cvcl_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias, int M, int N, int K,
                    float* C, int ldc, void* stream);

/* The two other evaluation forms of the reference, both "normalise, all-pairs cosine, arg-max" in fp32:
 *   - n-category classification of a frame (multimodal_saycam_data_module.py:545-606: image vs every category text,
 *     argmax over the categories): normalize_rows (frames, texts) -> linear_f32 (scores) -> row_argmax;
 *   - cosine nearest-neighbour search between two feature sets (analysis_cvcl/duplicates.py:561-607: F.normalize +
 *     F.cosine_similarity + np.argmax/np.max per evaluation frame), chunked over the keys with `merge`.
 * normalize_rows: dst[m,:] = src[m,:] / max(||src[m,:]||, 1e-12).  row_argmax: first maximum of each row of
 * scores [M,N] (leading dimension ld) and its index + col0; merge != 0 folds it into the (best, arg) of earlier,
 * lower-index column chunks. */
int cvcl_normalize_rows_f32(const float* src, float* dst, long long M, int E, void* stream);
int cvcl_row_argmax_f32(const float* scores, long long ld, long long M, int N, int col0, int merge, float* best,
                        int* arg, void* stream);

/* Cross-modal retrieval selection (image->text and text->image recall@K, median rank): for each of the M full query
 * rows of scores [M,N] (leading dimension ld), row m being query q0 + m, orders the N keys as
 * torch.sort(row, descending=True, stable=True) does (a NaN above every number, -0 == +0, equal values by ascending
 * key index) and writes
 *   topk_idx [M,k] int32 / topk_val [M,k] fp32   the first k keys of that order and their scores;
 *   rank [M] int32                               the 0-based position of the query's first positive, -1 without one.
 * Positives: with q_group [Nq] and k_group [N] (int64), the keys n with k_group[n] == q_group[q0 + m]; with both NULL
 * (pair mode), the key n == q0 + m.  1 <= k <= min(64, N).  One block per row; the row is read once, and a second
 * time only when the first positive lies outside the top-k.  No atomics on global data (a replay is bit-identical). */
int cvcl_rank_topk_f32(const float* scores, long long ld, long long M, int N, long long q0, const int64_t* q_group,
                       const int64_t* k_group, int k, int* topk_idx, float* topk_val, int* rank, void* stream);

/* its backward: dst [B,HW,E] fp32 = g [B,E] broadcast over the locations (autograd of the sum, multimodal.py:765). */
int cvcl_spatial_pool_bwd(const float* g, int B, int HW, int E, float* dst, void* stream);

/* generic C [M,N] fp32 = alpha * A . B^T on the tcgen05 engine (bf16 operands, fp32 accumulate).
 * a_mn = 0: A stored [M,K] (K-major);  a_mn = 1: A stored [K,M] (MN-major, i.e. the transposed
 * matrix is read in place through an MN-major UMMA descriptor).  Same for B ([N,K] / [K,N]). */
int cvcl_gemm_f32out(const void* A, int lda, int a_mn, const void* B, int ldb, int b_mn, int M, int N, int K,
                     float alpha, float* C, int ldc, void* stream);

/* ---- K2 projection head + L2 normalise -----------------------------------------------------
 * replaces model.fc / the 1x1 conv (multimodal.py:181-192, applied at :101) + F.normalize (:736).
 * x [M,K] bf16 (M = B, or B*49 NHWC rows), w [E,K] bf16, bias [E] fp32.  tcgen05 GEMM, bias +
 * full-row norm in the epilogue (cluster of ceil(E/128) CTAs shares the row sum of squares);
 * the bf16 feature tile leaves through a TMA store. */
int cvcl_head_proj_norm_fwd(const void* x, int ldx, const void* w, int ldw, const float* bias,
                            int M, int E, int K, int normalize,
                            float* out_f32, int ld_f32, void* out_bf16, int ld_bf16,
                            float* inv_norm, void* stream);

/* ---- K3+K4 similarity GEMM fused with the symmetric InfoNCE statistics ----------------------
 * replaces multimodal.py:755 (match), :783-787 (logit_scale) and :801-818 (cross-entropy both
 * ways, argmax accuracy, entropy) without materialising the logits.
 * Direction 0 (image->text): rows img_q [M0,E] against txt_k [N0,E]; direction 1 (text->image):
 * rows txt_q [M1,E] against img_k [N1,E].  On one GPU img_q == img_k and txt_q == txt_k; on a
 * shard the *_q are the local pairs and the *_k the all-gathered features, and diag_off is the
 * column offset of the local block (SURVEY 8e).  log_scale = s = -log(temperature).
 * out5 = {loss, image_accuracy, text_accuracy, image_entropy, text_entropy}, each a partial
 * sum scaled by inv_rows = 1/B_global (sum over ranks gives the global value). */
size_t cvcl_sim_workspace_bytes(int M0, int N0, int M1, int N1);
int cvcl_sim_infonce_fwd(const void* img_q, const void* txt_k, const void* txt_q, const void* img_k,
                         int ld, int M0, int N0, int M1, int N1, int E, float log_scale,
                         int diag_off, float inv_rows, void* workspace,
                         float* lse0, float* lse1, int* argmax0, int* argmax1, float* out5,
                         int unit_norm, void* stream);
/* unit_norm != 0: the caller promises unit-norm feature rows (F.normalize, multimodal.py:736/743).  Large square
 * single-device problems (queries = keys, >= 4096 pairs, a multiple of 256, exp(s) <= 32) then take ONE similarity
 * pass for both directions (multimodal.py:755 computes `match` once): row statistics per thread, column statistics
 * through a transposed butterfly over the lanes, one exp per element against the fixed reference exp(s). */

/* materialised logits for the forward() API (multimodal.py:783-794):
 * lpi [Ni,Nt] = exp(s) * img . txt^T ; lpt [Nt,Ni] (either may be NULL). */
int cvcl_sim_logits_fwd(const void* img, const void* txt, int ld, int Ni, int Nt, int E, float log_scale,
                        float* lpi, float* lpt, void* stream);

/* ---- K5 backward --------------------------------------------------------------------------
 * (a) dL/dlogits tiles from recomputed logits: Gs0 [M0, N0] (rows = local images) and
 *     Gs1 [M1, N1] (rows = local texts), bf16, = exp(s) * coef * (softmax_row + softmax_col) with
 *     coef = upstream / (2 B_global), diagonal included.  The -2*I term of
 *     G = (softmax_row + softmax_col - 2 I)/(2B) is NOT in the bf16 matrix (it would dominate the
 *     rounding error): gdiag0 [M0] (gdiag1 [M1]) receives, per row m, G_ii - bf16(Gs[m, m + diag_off])
 *     in fp32, with G_ii = w (expm1(S_ii - lse_q) + expm1(S_ii - lse_k)), w = exp(s) coef; (b) adds
 *     gdiag[m] times the positive.  (When a pair is confident, w (P_row + P_col) and -2w nearly cancel;
 *     the bf16 rounding of the first would otherwise be the whole gradient of the row.)
 *     lse_k0 [N0] = column LSEs seen by direction 0 (= all-gathered lse1), lse_k1 [N1] likewise.
 *     Gs1 and gdiag1 may be NULL (single GPU: the dT GEMM reads Gs0 transposed in place, and its
 *     diagonal is the same element, so it uses gdiag0).
 *     *dscale += sum G * logits (the logit_scale gradient, multimodal.py:711-715,783-787). */
int cvcl_sim_infonce_bwd_g(const void* img_q, const void* txt_k, const void* txt_q, const void* img_k,
                           int ld, int M0, int N0, int M1, int N1, int E, float log_scale, int diag_off,
                           float coef, const float* lse_q0, const float* lse_k0, const float* lse_q1,
                           const float* lse_k1, void* Gs0, int ldg0, void* Gs1, int ldg1, float* gdiag0,
                           float* gdiag1, float* dscale, void* stream);
/* (b) dFeat = Gs . other + diag_coef[m] * diag_feat[m + diag_off] (diag_coef [M] = the gdiag of (a):
 *     the diagonal of G in fp32; diag_feat [diag_rows,E] bf16 may be NULL, and with it diag_coef),
 *     followed by the F.normalize backward in the
 *     epilogue (feat [M,E] bf16 + inv_norm).  Gs is [M,Kc] (gs_transposed = 0) or stored [Kc,M]
 *     (gs_transposed = 1: the other orientation is read in place, MN-major); other is the [Kc,E] bf16
 *     feature matrix as stored.  Exactly one output: out_f32 [M,E] (scaled by 1/row_len if given:
 *     d mean-embedding) or out_bf16 [M,E] (operand of the weight-gradient GEMM); dbias [E] += column
 *     sums (nullable). */
int cvcl_feat_grad_norm_bwd(const void* Gs, int ldg, int gs_transposed, const void* other, int ld_other,
                            int M, int E, int Kc, const void* feat_bf16, int ld_feat, const float* inv_norm,
                            int normalize, const int64_t* row_len, const void* diag_feat, int ld_diag,
                            int diag_rows, int diag_off, const float* diag_coef, float* out_f32, int ld_f32,
                            void* out_bf16, int ld_bf16, float* dbias, void* stream);
/* same, with an optional fp32 scratch acc_scratch [M,E]: when the contraction is long (Kc >= 1536, the
 * sharded global batch) and the output has few tiles, the GEMM is split over the contraction into
 * acc_scratch (or into out_f32 itself when that is the output) with fp32 vector atomics, and a
 * warp-per-row pass applies the diagonal term, the normalise backward, 1/len and the bias sums. */
int cvcl_feat_grad_norm_bwd_ws(const void* Gs, int ldg, int gs_transposed, const void* other, int ld_other,
                               int M, int E, int Kc, const void* feat_bf16, int ld_feat, const float* inv_norm,
                               int normalize, const int64_t* row_len, const void* diag_feat, int ld_diag,
                               int diag_rows, int diag_off, const float* diag_coef, float* out_f32, int ld_f32,
                               void* out_bf16, int ld_bf16, float* dbias, float* acc_scratch, void* stream);
/* (c) dW [E,K] = sum_m du[m,:]^T x[m,:]  (autograd of nn.Linear / 1x1 conv weight); du [M,E] and
 *     x [M,K] bf16 as stored (both read MN-major). */
int cvcl_head_weight_grad(const void* du, int ld_du, const void* x, int ld_x, int E, int K, int M,
                          float* dW, int ld_dw, void* stream);

/* ---- fused flat train step: K1 .. K5 sequenced in one call ----------------------------------
 * replaces MultiModalModel.calculate_contrastive_loss (multimodal.py:796-822) + loss.backward()
 * for embedding_type = "flat".  x [B,K] trunk-boundary features (fp32 or bf16), w/bias/table the
 * fp32 master parameters.  Outputs: out5 (see above), dW [E,K], dbias [E], dtable [V,E], dscale [1]
 * (all fp32, overwritten), optional img/txt features fp32 [B,E].  Gradients are d(loss)/d(param)
 * for upstream = 1.  Workspace from cvcl_flat_step_workspace_bytes. */
size_t cvcl_flat_step_workspace_bytes(int B, int L, int E, int K, int V);
/* byte offsets of the blocks a finished cvcl_flat_contrastive_step leaves in its workspace (tests read them):
 * out[0..11] = img16, txt16 [B,E] bf16, invn_i, invn_t, lse0, lse1 [B] fp32, G0 [B, ldB] bf16, du16 [B,E] bf16,
 * dm [B,E] fp32 (d mean-embedding), gdiag [B] fp32, ldB, bytes. */
int cvcl_flat_step_layout(int B, int L, int E, int K, int V, long long* out, int n);
int cvcl_flat_contrastive_step(const void* x, int x_is_bf16, const int64_t* ids, const int64_t* lens,
                               const float* w, const float* bias, const float* table,
                               int B, int L, int E, int K, int V, int normalize, float log_scale,
                               int need_grads, void* workspace,
                               float* out5, float* img_feat_f32, float* txt_feat_f32,
                               float* dW, float* dbias, float* dtable, float* dscale,
                               int* status, void* stream);

/* ---- fused flat train step as ONE persistent kernel ---------------------------------------------
 * Same contract as cvcl_flat_contrastive_step (multimodal.py:796-822 + loss.backward()), executed by a
 * single cooperative launch (one CTA per SM, grid-wide barriers between the phases; csrc/fused_step.cuh):
 * no weight cast, no memsets, the logits tile stays in TMEM from the statistics to dL/dlogits.
 * x16 [B,K] and w16 [E,K] are bf16 (the caller keeps a bf16 shadow of the fp32 master weight: refreshed by
 * cvcl_adamw_step's bf16_shadow output, or cast once after loading); bias/table fp32 masters.
 * log_scale_dev (nullable) is a DEVICE scalar s = -log(temperature): when given it is read by the kernel
 * (trainable temperature without a host sync, multimodal.py:711-715) and log_scale is ignored.
 * Shapes covered: E in {128,256,384,512}, K % 64 == 0, B <= 1024, L <= 256 (cvcl_flat_fused_supported); anything
 * else returns CVCL_ERR_UNSUPPORTED (callers then use cvcl_flat_contrastive_step).
 * workspace: cvcl_flat_fused_workspace_bytes bytes, 256-byte aligned, its first 1024 bytes zeroed ONCE before
 * the first call (the kernel leaves them reusable); one step in flight per workspace.
 * phase_limit: 0 = whole step; k = 1..5 leaves after phase k, 100 = six grid barriers only (measurement /
 * debugging; outputs then partial).  No atomics on data: every reduction is a fixed-order sum and the
 * embedding gradient is the GEMM  d table = C^T . dm  against the token-count matrix C[b,v], so the step
 * is bit-reproducible (the reference's embedding_dense_backward on CUDA is not). */
int cvcl_flat_fused_supported(int B, int L, int E, int K, int V);
size_t cvcl_flat_fused_workspace_bytes(int B, int L, int E, int K, int V);
/* byte offsets of the workspace blocks (tests / tools): out[0..13] = ctrl, hpart, img16, txt16, invn, part, diag,
 * lse, rb_part, dspart, dqpart, du16, dbpart, total; out[14..19] = Bp, KS, nPart, dw_bn, grid, nCB;
 * out[20..24] = dm16, cmat, QS, Vp, gdiag.  ctrl + 128 holds 48 globaltimer stamps (ns) of CTA 0: [0] start,
 * [k] after grid barrier k, [15] end, [16..28] inside the phases (csrc/fused_step.cuh: CVCL_STAMP). */
int cvcl_flat_fused_layout(int B, int L, int E, int K, int V, long long* out, int n);
int cvcl_flat_step_fused(const void* x16, const void* w16, const int64_t* ids, const int64_t* lens,
                         const float* bias, const float* table, int B, int L, int E, int K, int V,
                         int normalize, float log_scale, const float* log_scale_dev, int need_grads,
                         void* workspace, float* out5, float* img_feat_f32, float* txt_feat_f32,
                         float* dW, float* dbias, float* dtable, float* dscale, int* status, int phase_limit,
                         void* stream);

/* The same kernel with the batch sharded by pairs over `world` ranks of one NVLink domain (SURVEY 8e): rank r owns
 * pairs [r*B, r*B + B) of the global batch of world*B pairs, the head / embedding parameters are replicated.
 * All peer_* arguments are HOST arrays of `world` device pointers into peer-mapped symmetric memory, entry p =
 * rank p's buffer: gathered text / image features [world*B, E] bf16, gathered softmax partials
 * (cvcl_flat_fused_sharded_part_bytes(B, world) bytes: (max, sum) pairs [2 directions][2*nCB][world*B]), 32 flag
 * words (zero before first use).  `epoch` is a LOCAL device word, zero before first use.  The phases that produce
 * features and softmax partials store them straight into every rank's gathered buffers (posted stores over NVLink) and the
 * grid barrier that follows also spans the ranks (flag words, st.release.sys / ld.acquire.sys): no exchange
 * kernel, no NCCL.  Gradient sum: with peer_stats / peer_scratch (HOST arrays of `world` device pointers: rank p's
 * block [out5(8) | ds(4) | db(E) | d table(V*E) | dW(E*K)] floats and rank p's scratch of
 * cvcl_flat_fused_sharded_scratch_bytes(...) bytes, both in symmetric memory) and reduce_floats > 0 (8 = the five
 * scalars only, or 8 + 4 + E + V*E + E*K), the kernel sums the block over the ranks itself: every 128 x 128 tile of
 * dW / d table is owned by rank (tile % world); the tile GEMMs store their partial tiles straight into the owner's
 * scratch (TMA store over NVLink), the owner adds the partials in rank order (bit-identical on every rank) and
 * stores the sum into every rank's block; scalars and d bias go one-shot.  out5, dscale, dbias, dtable, dW must
 * then be this rank's pointers INTO peer_stats[rank] at those offsets.  The closing cross-rank barrier fences the
 * reuse of every exchange buffer by the next step.  With reduce_floats = 0 (tables may
 * be null) the outputs are this rank's PARTIAL sums (out5 scaled by 1/(world*B)) and the caller sums them
 * (cvcl_peer_allreduce_push_f32), which is then also the fence.  Every rank must call with the same shapes.
 * world = 1 is allowed (nothing crosses a link). */
int cvcl_flat_fused_sharded_supported(int B, int L, int E, int K, int V, int world);
size_t cvcl_flat_fused_sharded_workspace_bytes(int B, int L, int E, int K, int V, int world);
size_t cvcl_flat_fused_sharded_part_bytes(int B, int world);
size_t cvcl_flat_fused_sharded_scratch_bytes(int B, int L, int E, int K, int V, int world);
int cvcl_flat_step_fused_sharded(const void* x16, const void* w16, const int64_t* ids, const int64_t* lens,
                                 const float* bias, const float* table, int B, int L, int E, int K, int V,
                                 int normalize, float log_scale, const float* log_scale_dev, int need_grads,
                                 void* workspace, float* out5, float* img_feat_f32, float* txt_feat_f32,
                                 float* dW, float* dbias, float* dtable, float* dscale, int* status, int phase_limit,
                                 int world, int rank, void* const* peer_txt_all, void* const* peer_img_all,
                                 void* const* peer_part_all, void* const* peer_flags, unsigned int* epoch,
                                 void* const* peer_stats, void* const* peer_scratch, long long reduce_floats,
                                 void* stream);

/* ---- K6 spatial "max" similarity --------------------------------------------------------------
 * replaces multimodal.py:771-780 (einsum 'iehw,tle->itlhw' + amax over (h,w) + sum over l / len)
 * without materialising the [B,B,L,H,W] tensor.  tok [Bt*L, E] bf16 (per-token normalised text
 * features), img [Bi*HW, E] bf16 (NHWC location features).  match [Bi,Bt] fp32; the argmax
 * location per (i,t,l) is saved as uint8 in both [Bi, Bt*L] and [Bt*L, Bi] layouts. */
int cvcl_spatial_max_fwd(const void* tok, const void* img, const int64_t* lens, int Bt, int L, int Bi, int HW,
                         int E, float* match, unsigned char* amax_it, unsigned char* amax_ti, void* stream);
/* autograd of the above: dtok [Bt*L,E] and dimg [Bi*HW,E] fp32 (either may be NULL) from
 * gmatch = dL/dmatch [Bi,Bt].  With a workspace (cvcl_spatial_max_bwd_workspace_bytes, 256-byte aligned) the saved
 * arg-max is expanded into the bf16 matrix P[(t,l),(i,hw)] = [hw = argmax] * g[i,t]/len[t] over the REAL token rows
 * only (pad positions are dropped; their count stays on the device and bounds the GEMMs from there, no sync) and both
 * gradients run as tcgen05 GEMMs (dtok = P.img, dimg = P^T.tok, P^T read in place MN-major);
 * workspace = NULL selects the SIMT gather form (ids [Bt*L], nullable, lets pad tokens be skipped). */
size_t cvcl_spatial_max_bwd_workspace_bytes(int Bt, int L, int Bi, int HW, int E);
int cvcl_spatial_max_bwd(const float* gmatch, const int64_t* lens, const int64_t* ids,
                         const unsigned char* amax_it, const unsigned char* amax_ti, const void* tok,
                         const void* img, int Bt, int L, int Bi, int HW, int E, float* dtok, float* dimg,
                         void* workspace, void* stream);
/* symmetric InfoNCE statistics (multimodal.py:801-818) from a materialised match [B,B] fp32 and
 * their backward: dmatch = exp(s) * G, *dscale += sum G * logits.  workspace as for K3+K4. */
int cvcl_match_infonce_fwd(const float* match, int B, float log_scale, float inv_rows, void* workspace,
                           float* lse0, float* lse1, int* argmax0, int* argmax1, float* out5, void* stream);
int cvcl_match_infonce_bwd(const float* match, int B, float log_scale, float coef, const float* lse0,
                           const float* lse1, float* dmatch, float* dscale, void* stream);
/* One rank's share of the same loss when the batch is sharded over a process group (multimodal.py:771-822 on the
 * global batch; rank r owns pairs [r*b, (r+1)*b), N = world*b, diag_off = r*b): the row block match_r [b,N] (local
 * images x all texts) gives the image->text CE of the local images, the column block match_c [N,b] (all images x
 * local texts) the text->image CE of the local texts.  out5 = partial sums scaled by inv_rows = 1/N (summed over the
 * ranks by the caller); lse0 / argmax0 [b] per local image, lse1 / argmax1 [b] per local text; workspace
 * cvcl_sim_workspace_bytes(b, N, b, N).  b = N, diag_off = 0, match_r = match_c is cvcl_match_infonce_fwd.
 * Backward: dmatch_r = exp(s) G_r, dmatch_c = exp(s) G_c with the gathered LSEs of all ranks (lse1_all, lse0_all
 * [N]); *dscale = sum G_r * logits over the row block (the caller sums it over the ranks), written in a fixed
 * summation order through the workspace (cvcl_match_infonce_block_bwd_workspace_bytes, 256-byte aligned). */
int cvcl_match_infonce_block_fwd(const float* match_r, const float* match_c, int b, int N, int diag_off,
                                 float log_scale, float inv_rows, void* workspace, float* lse0, float* lse1,
                                 int* argmax0, int* argmax1, float* out5, void* stream);
size_t cvcl_match_infonce_block_bwd_workspace_bytes(int b, int N);
int cvcl_match_infonce_block_bwd(const float* match_r, const float* match_c, int b, int N, int diag_off,
                                 float log_scale, float coef, const float* lse0, const float* lse1_all,
                                 const float* lse0_all, const float* lse1, float* dmatch_r, float* dmatch_c,
                                 float* dscale, void* workspace, void* stream);

/* ---- all-gather over NVLink peer memory (the exchange step of the sharded loss, SURVEY 8e) ------
 * peer_ptrs: HOST array of `world` device pointers, entry r = rank r's block (symmetric memory, peer
 * mapped).  Copies `bytes_per_rank` bytes from every rank except skip_rank (-1: none) to
 * dst + r * dst_stride_bytes with 16-byte loads from the peer pointers.  The caller orders it after a
 * cross-rank barrier (torch symmetric-memory barrier). */
int cvcl_p2p_gather(const void* const* peer_ptrs, int world, int skip_rank, long long bytes_per_rank, void* dst,
                    long long dst_stride_bytes, void* stream);

/* ---- collectives over NVLink peer memory with in-kernel cross-rank barriers (SURVEY 8e) ---------
 * The exchange steps and the gradient sum of the sharded step as single kernels instead of NCCL
 * calls.  Every rank passes the same HOST tables of `world` device pointers: peer_data[r] = rank r's
 * block and peer_flags[r] = rank r's flag area for THIS call site ("channel"), both in peer-mapped
 * symmetric memory.  A channel's flag area holds cvcl_peer_flag_words() uint32 words, zeroed once
 * before first use (followed by any cross-rank barrier); `epoch` is a LOCAL uint32 array of
 * cvcl_peer_max_blocks() words, zeroed once; `status` (local int, nullable) becomes non-zero if a
 * barrier did not complete within timeout_ms (0 = 10 minutes), after which the kernel traps (or, with
 * CVCL_PEER_NO_TRAP or'ed into timeout_ms, continues: probe mode, results undefined).  All ranks
 * must issue the same sequence of calls per channel with the same sizes.  Graph capturable.
 *   allgather    : barrier, then dst[s*dst_seg_stride + r*seg_bytes ..] <- segment s (at
 *                  s*src_seg_stride) of rank r's block, for all r (including the caller's own) and s.
 *                  The blocks may be overwritten again only after a later barrier / all-reduce.
 *   allreduce_f32: in-place sum over ranks of n floats (n % 4 == 0, world in {1,2,4,8}); slice r is
 *                  summed by rank r in rank order and written to every rank: bit-identical results on
 *                  all ranks, independent of timing.
 *   barrier      : barrier only.
 *   allgather_push / allreduce_push_f32: the same results with PUSH traffic only (posted stores over
 *                  NVLink, no load round trips): allgather_push stores the caller's block `src` into slot
 *                  `rank` of every rank's gathered buffer peer_dst[p] and then barriers; allreduce_push
 *                  scatters slice p of the caller's buffer into rank p's scratch block
 *                  (cvcl_peer_allreduce_scratch_bytes, peer-mapped), barriers, sums its own slice locally
 *                  in rank order, stores the sum into every rank's buffer, barriers.  Both are launched
 *                  with programmatic dependent launch (their launch overlaps the tail of the previous kernel). */
#define CVCL_PEER_NO_TRAP 0x80000000u
size_t cvcl_peer_flag_words(void);
int cvcl_peer_max_blocks(void);
int cvcl_peer_allgather(void* const* peer_data, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                        int rank, long long seg_bytes, int nseg, long long src_seg_stride_bytes, void* dst,
                        long long dst_seg_stride_bytes, unsigned int timeout_ms, void* stream);
int cvcl_peer_allreduce_f32(void* const* peer_data, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                            int rank, long long n, unsigned int timeout_ms, void* stream);
int cvcl_peer_allgather_push(void* const* peer_dst, void* const* peer_flags, unsigned int* epoch, int* status, int world,
                             int rank, const void* src, long long seg_bytes, int nseg, long long src_seg_stride_bytes,
                             long long dst_seg_stride_bytes, unsigned int timeout_ms, void* stream);
size_t cvcl_peer_allreduce_scratch_bytes(long long n, int world);
int cvcl_peer_allreduce_push_f32(void* const* peer_data, void* const* peer_scratch, void* const* peer_flags,
                                 unsigned int* epoch, int* status, int world, int rank, long long n,
                                 unsigned int timeout_ms, void* stream);
int cvcl_peer_barrier(void* const* peer_flags, unsigned int* epoch, int* status, int world, int rank,
                      unsigned int timeout_ms, void* stream);

/* ---- fused AdamW for the head parameters (SURVEY 8f item 2) -------------------------------------
 * replaces torch.optim.AdamW.step (multimodal_lit.py:112-128) for one fp32 tensor of n elements:
 * p *= 1 - lr*wd; m = lerp(m, g, 1-beta1); v = beta2*v + (1-beta2)*g^2;
 * p -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps).   g is read as g*grad_scale.
 * bf16_shadow (nullable): refreshed bf16 copy of p (the operand the head GEMM consumes). */
int cvcl_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                    float beta2, float eps, float weight_decay, int step, float grad_scale, void* bf16_shadow,
                    void* stream);

/* the same update for `count` (<= 8) tensors in ONE launch with the step number kept on the DEVICE
 * (step_dev[0] = completed steps, incremented by the kernel; ticket[0] = 0 on entry): the launch can be
 * captured in a CUDA graph and replayed, which makes a whole train step -- cvcl_flat_step_fused + this --
 * one graph.  All arrays are HOST arrays of `count` entries; p/g/m/v/bf16_shadow entries are device pointers
 * (bf16_shadow, or single entries of it, may be NULL). */
int cvcl_adamw_multi_step(int count, float* const* p, const float* const* g, float* const* m, float* const* v,
                          const long long* n, void* const* bf16_shadow, const float* lr, const float* weight_decay,
                          float beta1, float beta2, float eps, float grad_scale, int* step_dev,
                          unsigned int* ticket, void* stream);

/* ---- Grad-CAM attention maps for the flat head (SURVEY 8f item 4) ---------------------------------
 * replaces multimodal/attention_maps.py:111-165 (gradCAM: forward through layer4 -> avgpool -> fc,
 * F.normalize, output.backward(target), alpha = grad.mean((2,3)), clamp(sum_c act*alpha, 0)) for the
 * saliency layer the reference uses (layer4).  The head is linear in the pooled activation, so the
 * gradient is computed in closed form: no trunk backward.  fp32 end to end.
 * act [N,K,HW] (NCHW layer4 activation, HW <= 64), w [E,K], bias [E] (nullable), target [N,E] ->
 * cam [N,HW].  workspace: cvcl_gradcam_workspace_bytes(N,K,E), 16-byte aligned. */
size_t cvcl_gradcam_workspace_bytes(int N, int K, int E);
int cvcl_gradcam_flat(const float* act, const float* w, const float* bias, const float* target, int N, int K, int HW,
                      int E, int normalize, void* workspace, float* cam, void* stream);
/* F.interpolate(mode="bicubic", align_corners=False) of [N,h,w] fp32 maps to [N,H,W]
 * (attention_maps.py:158-163). */
int cvcl_bicubic_upsample(const float* in, int N, int h, int w, int H, int W, float* out, void* stream);

/* ---- K7 n-way evaluation (fp32, bit-exact argmax contract) -----------------------------------
 * replaces the per-trial loop of eval.py:196-214 / multimodal_lit.py:466-511.
 * img [n_trials*n_way, E] fp32 embeddings (target first), txt [C,E] fp32 label embeddings,
 * txt_index [n_trials] (NULL = identity).  pred [n_trials] int32; logits [n_trials,n_way] optional. */
int cvcl_eval_nway_fwd(const float* img, const float* txt, const int* txt_index, int n_trials, int n_way,
                       int E, int normalize, float log_scale, int* pred, float* logits, void* stream);

/* ---- spatial-embedding evaluation (fp32 SIMT) ------------------------------------------------
 * The batched form of the per-trial loop (eval.py:196-214, multimodal_lit.py:466-511) and of the n-category
 * classification (multimodal_saycam_data_module.py:545-606) for embedding_type = "spatial".
 *
 * conv1x1: the 1x1-conv head (multimodal.py:181-185, applied at :101) in fp32 with fp32 FMA accumulation, the
 * same arithmetic class as cvcl_linear_f32.  x [B,K,HW] is the layer4 map as the trunk emits it (NCHW, read in
 * place), w [E,K] (16-byte aligned), bias [E] (nullable) -> out [B*HW, E] NHWC rows:
 * out[b*HW + p, e] = bias[e] + sum_k w[e,k] x[b,k,p].  K % 4 == 0. */
int cvcl_conv1x1_f32(const float* x, const float* w, const float* bias, int B, int K, int HW, int E, float* out,
                     void* stream);
/* spatial "max" logits (multimodal.py:771-780, then :783-787):
 *   out = exp(log_scale) * (sum_{l < len[c]} max_p <img[m,p,:], tok[c,l,:]>) / len[c]
 * img [M,HW,E] fp32 normalised location features (NHWC rows), tok [C,L,E] fp32 per-token text features, lens [C].
 * Trial mode (n_way >= 1, M a multiple of n_way): image m is scored against label txt_index[m / n_way] (NULL =
 * identity, then C >= M / n_way), out [M]; a label index outside [0, C) gives NaN.  Category mode (n_way = 0):
 * every image against all C labels, out [M, C].  Each image block is read from HBM once; no atomics (a replay is
 * bit-identical).  HW <= 256; the HW x E block must fit in shared memory (49 x 1024 does). */
int cvcl_spatial_max_scores_f32(const float* img, const float* tok, const int64_t* lens, const int* txt_index, int M,
                                int HW, int E, int C, int L, int n_way, float log_scale, float* out, void* stream);

/* ---- text-to-location attention maps for spatial embeddings (fp32 SIMT) -------------------------
 * The per-location terms of the spatial similarity (multimodal.py:771-780) before its max / mean reductions; the
 * reference returns no such tensor, these are the summands of its own forward.  Image m is paired with label
 * c = txt_index[m] (NULL = identity, then C >= M):
 *   token_maps[m,l,p] = <img[m,p,:], tok[c,l,:]>                          for l < len[c]; exactly 0 for l >= len[c]
 *   utt_maps[m,p]     = (sum_{l < len[c]} token_maps[m,l,p]) / len[c]     (position order; len 0 gives NaN)
 *   token_argmax[m,l] = first p attaining max_p token_maps[m,l,p] (a NaN wins), -1 for l >= len[c]
 * img [M,HW,E] fp32 normalised location features (NHWC rows), tok [C,L,E] fp32 per-token text features, lens [C];
 * token_maps [M,L,HW] and token_argmax [M,L] are nullable, utt_maps [M,HW].  Match units (no exp(s)).  A label
 * index outside [0, C) gives NaN maps and arg-max -1.  The dots are bit-identical to the ones
 * cvcl_spatial_max_scores_f32 takes the maximum of in trial mode; no atomics (a replay is bit-identical).
 * HW <= 256; the HW x E block must fit in shared memory (49 x 1024 does). */
int cvcl_spatial_attention_f32(const float* img, const float* tok, const int64_t* lens, const int* txt_index, int M,
                               int HW, int E, int C, int L, float* token_maps, float* utt_maps, int* token_argmax,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CVCL_B200_H */
