/* cor_b200.h -- C ABI of libcor_b200.so: B200 (sm_100a) kernels for CORE's region pooling,
 * scoring and loss path.
 *
 * The reference (wangtong627/COR) has no FFI: the boundary it exposes for this path is a set of
 * Python names (SURVEY.md 8b).  Each entry point below names the reference call site whose
 * arithmetic it replaces; cor_b200 (Python, ctypes) binds them with ctypes and re-exposes the reference's
 * Python signatures on top.  All pointers are DEVICE pointers unless marked host; all tensors
 * are dense row-major ("contiguous" in torch terms); `stream` is a cudaStream_t passed as
 * void*.  Every function returns 0 on success or a negative COR_E* code and leaves a message
 * retrievable with cor_last_error().  There is no CPU fallback anywhere in the library.
 */
#ifndef COR_B200_H_
#define COR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COR_ABI_VERSION 3

/* element types */
#define COR_F32 0
#define COR_BF16 1
#define COR_U8 2

/* status codes */
#define COR_OK 0
#define COR_EINVAL (-1)   /* bad argument (shape, dtype, alignment) */
#define COR_ECUDA (-2)    /* CUDA runtime error, see cor_last_error() */
#define COR_EARCH (-3)    /* device is not sm_100 */
#define COR_EUNSUP (-4)   /* valid request this build cannot serve (message says which) */

/* weight transforms applied to the resampled mask / map (pool kernels) */
#define COR_W_PLAIN 0     /* MaskedPooling: w = r                 (mask_adapter.py:22)   */
#define COR_W_CLAMP 1     /* mask_pooling:  w = clamp(r, 0, 1)    (loss_func.py:49)      */
#define COR_W_SIGMOID 2   /* MaskAdapterPooling tail: softmax(logsigmoid(x)) == sigmoid(x)/sum
                             (mask_adapter.py:71)                                        */

typedef void* cor_stream_t;

int cor_abi_version(void);
const char* cor_last_error(void);
/* Fills SM count and compute capability of the current device; COR_EARCH if it is not 10.x. */
int cor_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Mask resample + sums.  Replaces F.interpolate(mask, size=(h,w), mode="bilinear",
 * align_corners=False) at mask_adapter.py:19-20, loss_func.py:46-47, and the full-resolution
 * validity sums at loss_func.py:73-74 and :103-107, in ONE pass over the masks.
 *   masks    [n_masks, Hm, Wm]  f32 / bf16 / u8 (u8 value v means v * mask_scale)
 *   w_f32    [n_masks, ldw] resampled values r (no transform), or NULL
 *   w_bf16   transform(r) rounded to bf16 (tensor-core operand), or NULL; row of mask n starts at
 *            element (n / group) * group_stride + (n % group) * ldw  (group <= 0: plain [n_masks, ldw])
 *   stats    [n_masks, 4] f32:  {sum(mask), sum(1-mask), sum_p transform(r), sum_p bf16(transform(r))}
 *   work     scratch of cor_mask_prep_work_bytes() bytes
 * ---------------------------------------------------------------------------------------- */
size_t cor_mask_prep_work_bytes(int n_masks, int Hm, int Wm, int h, int w);
int cor_mask_prep(const void* masks, int mask_dtype, float mask_scale, int n_masks, int Hm, int Wm,
                  int h, int w, int transform, float* w_f32, void* w_bf16, long long ldw,
                  int group, long long group_stride, float* stats, void* work, cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Region pooling, streaming (CUDA-core, exact fp32) variant: any number of rows R, best for
 * small R (the reference's M=1 and the MaskAdapter tail's 8 maps).  Replaces the mul/sum chain
 * at mask_adapter.py:22-23, loss_func.py:50-52 and the bmm at mask_adapter.py:72-75.
 *   feat   [B, C, P]  f32 / bf16
 *   wts    [B, R, ldw] f32 raw resampled values; transform applied on the fly
 *   fg_sum [B, R, C]  = sum_p w * F ;  bg_sum [B, R, C] = sum_p (1-w) * F (or NULL)
 * ---------------------------------------------------------------------------------------- */
int cor_pool_stream_fwd(const void* feat, int feat_dtype, const float* wts, long long ldw, int B, int C,
                        int P, int R, int transform, float* fg_sum, float* bg_sum, cor_stream_t stream);

/* Tensor-core (tcgen05 / TMEM, TMA-staged) variant for bf16 features and many masks:
 *   feat [B, C, P] bf16 (P % 64 == 0, C % 128 == 0), wts [B, Rp, P] bf16 with Rp % 16 == 0 and
 *   16 <= Rp <= 256; one row of wts may be all ones so that its pooled sum is sum_p F (background
 *   by subtraction).  Split-K over the mask pixels: writes ksplit = cor_pool_umma_ksplit(B,C,P)
 *   fp32 partial tiles part [ksplit, B, Rp, C]; cor_rows_finalize sums them in fixed order.      */
int cor_pool_umma_ksplit(int B, int C, int P);
size_t cor_pool_umma_work_bytes(int B, int C, int P, int Rp);   /* bytes of `part` */
int cor_pool_umma_fwd(const void* feat_bf16, const void* wts_bf16, int B, int C, int P, int Rp,
                      float* part, cor_stream_t stream);

/* Row epilogue: divide by the denominator, optional group mean, optional L2-normalise
 * (loss_func.py:51-53; mask_adapter.py:23, :77-79).  One row = one (image, mask).
 *   sums: row i lives at (i / rows_per_image) * img_stride + (i % rows_per_image) * C floats, and is
 *         the fixed-order sum of nsplit partial copies split_stride floats apart (nsplit <= 1: none);
 *   den [rows_in] (stride den_stride floats); eps added to den;
 *   group G >= 1: output row j = mean of input rows j*G .. j*G+G-1 after division;
 *   out_f32 [rows_in/G, C] ; out_bf16 same shape or NULL ; inv_norm [rows_in/G] (1/max(|p|,1e-12)
 *   when normalize, else 1) saved for backward.  If all_sum != NULL the row is the BACKGROUND
 *   (all_sum[b] - sums[row]) / (p_total - den + eps), all_sum[b] at b * img_stride floats (+ splits). */
int cor_rows_finalize(const float* sums, int rows_per_image, long long img_stride, int nsplit, long long split_stride,
                      const float* den, int den_stride, float eps, int rows_in, int C, int G, int normalize,
                      const float* all_sum, float p_total, float* out_f32, void* out_bf16, float* inv_norm,
                      cor_stream_t stream);

/* Backward of cor_rows_finalize: g_out [rows_out, C] -> g_sums [rows_in, C], the gradient w.r.t. the
 * sum row the epilogue consumed (for bg_from_all rows: w.r.t. the background sum all - fg). */
int cor_rows_finalize_bwd(const float* g_out, const float* out_f32, const float* inv_norm, const float* den,
                          int den_stride, float eps, int rows_in, int C, int G, int normalize, int bg_from_all,
                          float p_total, float* g_sums, cor_stream_t stream);

/* Backward of the pooling contraction w.r.t. the features:
 *   g_feat[b,c,p] = sum_r g_fg[b,r,c] * w[b,r,p] + g_bg[b,r,c] * (1 - w[b,r,p])   (g_bg may be NULL) */
int cor_pool_bwd_feat(const float* g_fg, const float* g_bg, const float* wts, long long ldw, int B, int C, int P,
                      int R, int transform, void* g_feat, int feat_dtype, cor_stream_t stream);

/* Same contraction on tcgen05 tensor cores (bf16 operands built in shared memory from the fp32 inputs,
 * fp32 accumulate in TMEM); write-bound.  cor_pool_bwd_umma_ok() says whether a shape is served
 * (C % 128 == 0, P % 256 == 0, R (+1 with g_bg) <= 256); otherwise use cor_pool_bwd_feat. */
int cor_pool_bwd_umma_ok(int B, int C, int P, int R, int has_bg);
int cor_pool_bwd_umma(const float* g_fg, const float* g_bg, const float* wts, long long ldw, int B, int C, int P,
                      int R, int transform, void* g_feat, int feat_dtype, cor_stream_t stream);

/* Backward w.r.t. the (sigmoid) maps of the MaskAdapter tail (mask_adapter.py:71-79):
 *   g_x[b,r,p] = s(1-s)/den_r * ( sum_c g_sum... ) -- see DESIGN.md; g_pooled is d/d(pooled row). */
int cor_pool_bwd_maps(const void* feat, int feat_dtype, const float* maps, long long ldw, const float* g_pooled,
                      const float* pooled, const float* den, int B, int C, int P, int R, float* g_maps,
                      cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Foreground / background cosine losses (loss_func.py:59-126) on already pooled unit rows.
 *   fg_rows, bg_rows [n, C] f32 (row i of image i), comb [n, C] f32, stats [n,4] from mask_prep
 *   (validity = sum(mask) > 0, sum(1-mask) > 0), strides in floats between consecutive samples.
 *   bg_mode 0: the reference's broadcast form (loss_func.py:120-123); 1: paired cosine.
 *   out[0]=fg loss, out[1]=bg loss, out[2]=#valid fg, out[3]=#valid bg.
 * Backward writes g_fg_rows, g_bg_rows [n, C] and g_comb [n, C] for upstream scalars g[0], g[1]
 * (device pointer to 2 floats). */
size_t cor_fgbg_aux_floats(int n, int C);   /* floats of `aux` scratch kept from forward to backward */
int cor_fgbg_loss_fwd(const float* fg_rows, long long fg_stride, const float* bg_rows, long long bg_stride,
                      const float* comb, long long comb_stride, const float* stats, long long stats_stride,
                      int n, int C, int bg_mode, float* out4, float* aux, cor_stream_t stream);
/* Upstream gradients: d/d fg-loss = g2[0] * gw_fg, d/d bg-loss = g2[g2_stride] * gw_bg (g2_stride 0 lets one
 * device scalar feed both).  g_fg_rows / g_comb are written (or, with *_accumulate, added to) at the given
 * row strides, so a caller can fold these gradients straight into larger gradient buffers. */
int cor_fgbg_loss_bwd(const float* fg_rows, long long fg_stride, const float* bg_rows, long long bg_stride,
                      const float* comb, long long comb_stride, int n, int C, int bg_mode, const float* out4,
                      const float* aux, const float* g2, long long g2_stride, float gw_fg, float gw_bg,
                      float* g_fg_rows, long long gfg_stride, int fg_accumulate,
                      float* g_bg_rows, long long gbg_stride, float* g_comb, long long gcomb_stride,
                      int comb_accumulate, cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * The fused step's region tail in one launch each way (csrc/step_tail.cu; cor_b200/region.py, one rank, bg_mode 0):
 * B <= 16 triplets with M candidate masks each, C % 8 == 0, C <= 256; query b's target is region row b*M.
 *   cor_step_tail_fwd: the pooling GEMM's split-K partials part [nsplit][B][Rp][C] (row M of each image = the all-ones
 *     weight row) -> unit rows fg [B*M, C] f32 + bf16 + inv_fg [B*M] (= cor_rows_finalize), background rows of the
 *     ground-truth masks bg [B, C] + inv_bg [B], the InfoNCE of every query against all B*M rows (lse [B], nce [1],
 *     tgt_logit [B]), the fg / bg losses out4 [4] + aux (= cor_fgbg_loss_fwd, bg_mode 0) and
 *     total = seg[0] + w_fg * out4[0] + w_bg * out4[1] + w_nce * nce (= cor_infonce_tail).  stats [B*M, 4] from
 *     cor_mask_prep; queries [B, C] bf16, comb [B, C] f32 (the same queries).
 *   cor_step_tail_bwd: for upstream scalar *g_loss, the InfoNCE + fg-loss gradient of every region row taken back
 *     through the row epilogue, cast to bf16 into a16 [B][Kp][C] (rows M..Kp-1 zeroed: the K-padded operand of the
 *     pooling-backward GEMM; NULL = not wanted) and the gradient of the queries g_queries [B, C] f32 (NULL = not wanted).
 *   work: cor_step_tail_work_bytes() bytes; counter: cor_step_tail_counter_words() u32 words, zero before the first
 *   launch and left zero by every launch (graph-replayable).  Deterministic.
 * ---------------------------------------------------------------------------------------- */
int cor_step_tail_counter_words(void);
size_t cor_step_tail_work_bytes(int B, int M, int C);
int cor_step_tail_fwd(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                      const float* stats, const void* queries_bf16, const float* comb, const long long* targets, float inv_tau,
                      const float* seg, float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16, float* inv_fg, float* bg,
                      float* inv_bg, float* fgbg_out4, float* aux, float* lse, float* nce, float* tgt_logit, float* total,
                      void* work, unsigned* counter, cor_stream_t stream);
int cor_step_tail_bwd(const void* regions_bf16, const void* queries_bf16, const long long* targets, const float* lse, int B, int M,
                      int C, float inv_tau, const float* g_loss, float w_nce, const float* fg, const float* inv_fg,
                      const float* stats, const float* comb, const float* fgbg_out4, const float* aux, float w_fg, float w_bg,
                      void* a16, int Kp, float* g_queries, void* work, unsigned* counter, cor_stream_t stream);
/* Extend cor_step_tail_fwd / _bwd: the logit scale s = 1/tau is read from device memory (logit_scale, one f32; a CUDA
 * graph that captured the call picks up a new value at every replay).  _bwd also writes d total / d s to g_logit_scale
 * (one f32; NULL = not wanted): w_nce * g_loss[0] * mean_q sum_r (softmax(s S_q)_r - [r == t(q)]) S_qr, folded in a fixed
 * order by the dQ CTAs (which then run even when g_queries is NULL). */
int cor_step_tail_fwd_ls(const float* part, int nsplit, long long split_stride, int Rp, int B, int M, int C, float p_total,
                         const float* stats, const void* queries_bf16, const float* comb, const long long* targets,
                         const float* logit_scale, const float* seg, float w_fg, float w_bg, float w_nce, float* fg, void* fg_bf16,
                         float* inv_fg, float* bg, float* inv_bg, float* fgbg_out4, float* aux, float* lse, float* nce,
                         float* tgt_logit, float* total, void* work, unsigned* counter, cor_stream_t stream);
int cor_step_tail_bwd_ls(const void* regions_bf16, const void* queries_bf16, const long long* targets, const float* lse, int B,
                         int M, int C, const float* logit_scale, const float* g_loss, float w_nce, const float* fg,
                         const float* inv_fg, const float* stats, const float* comb, const float* fgbg_out4, const float* aux,
                         float w_fg, float w_bg, void* a16, int Kp, float* g_queries, float* g_logit_scale, void* work,
                         unsigned* counter, cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Segmentation loss (loss_func.py:5-32) with the target resample of trainer_v3_g.py:67 fused in.
 *   pred [N, H, W] f32/bf16 logits; mask [N, Hm, Wm] f32/bf16/u8 (resampled to HxW if sizes differ)
 *   Per sample, from ONE pass over (pred, mask), seven terms (t = target, p = sigmoid(pred),
 *   w = 1 + 5|boxmean31(t) - t|, sm = dice_smooth):
 *     COR_SEG_WBCE  sum(w bce)/sum(w)                               loss_func.py:21-22
 *     COR_SEG_WIOU  1 - (sum(ptw) + 1e-6)/(sum((p+t)w) - sum(ptw) + 1e-6)   loss_func.py:25-29
 *     COR_SEG_DICE  1 - (2 sum(pt) + sm)/(sum(p) + sum(t) + sm)     [Class N: names only in the reference's stale .pyc]
 *     COR_SEG_BCE   mean(bce)                                       [Class N]
 *     COR_SEG_IOU   1 - (sum(pt) + 1e-6)/(sum(p) + sum(t) - sum(pt) + 1e-6)   [Class N]
 *     COR_SEG_WDICE 1 - (2 sum(ptw) + sm)/(sum((p+t)w) + sm)        [Class N]
 *     COR_SEG_FOCAL mean(a_t (1 - p_t)^gamma bce)                   [Class N; evaluated only when focal_gamma >= 0]
 *   loss = mean_n sum_k coef7[k] term_k[n]; coef7 is a HOST array of COR_SEG_NTERMS floats, NULL = {1, 1, 0, ...}
 *   (= wbce_with_wiou_loss, loss_func.py:31).
 *   out8 [8]: {loss, dice, focal, wbce, wiou, bce, iou, wdice}, each the mean over samples;
 *   per_sample [N, cor_seg_loss_npartials()] partial sums saved for backward;
 *   t_save, w_save [N,H,W] f32 (resampled target, edge weight) or NULL when no backward is needed.
 *   Kernels: a TMA-streamed row-strip kernel when the mask is at the logit size or at exactly 4x it (W <= 256,
 *   W % 16 == 0, 16-byte aligned), a 64x64 tile kernel otherwise -- and for small batches of 2/4-byte 4x masks, where it measures
 *   faster (COR_SEG_STRIP=0 forces the tile kernel, =2 the strip kernel wherever it applies).
 * ---------------------------------------------------------------------------------------- */
enum { COR_SEG_WBCE = 0, COR_SEG_WIOU = 1, COR_SEG_DICE = 2, COR_SEG_BCE = 3, COR_SEG_IOU = 4, COR_SEG_WDICE = 5, COR_SEG_FOCAL = 6,
       COR_SEG_NTERMS = 7 };
int cor_seg_loss_npartials(void);
size_t cor_seg_loss_work_bytes(int N, int H, int W);
int cor_seg_loss_fwd(const void* pred, int pred_dtype, const void* mask, int mask_dtype, float mask_scale,
                     int N, int H, int W, int Hm, int Wm, long long mask_nstride /* elements between samples; <=0: Hm*Wm */,
                     const float* coef7, float focal_alpha, float focal_gamma, float dice_smooth, float* out8,
                     float* per_sample, float* t_save, float* w_save, void* work, cor_stream_t stream);
int cor_seg_loss_bwd(const void* pred, int pred_dtype, const float* t_save, const float* w_save,
                     const float* per_sample, int N, int H, int W, const float* coef7, float dice_smooth, float focal_alpha,
                     float focal_gamma, const float* g_loss, void* g_pred, int g_dtype, cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Region x query similarity and InfoNCE (Class N: no reference implementation; nearest call
 * site F.cosine_similarity at loss_func.py:84,123 computes only the diagonal).
 *   regions [Nr, D] bf16 unit rows, queries [Nq, D] bf16 unit rows, D % 8 == 0.
 *   S [Nq, Nr] f32 or NULL; lse [Nq] (log-sum-exp of S/tau over regions) or NULL.
 * cor_sim_stream_*: CUDA-core streaming kernels, HBM-bound regime (few queries).
 * cor_sim_umma_fwd: tcgen05/TMEM GEMM (many queries).  It takes S or lse, not both (COR_EINVAL): S comes from a kernel
 *   with both operands in shared memory, lse from one that holds the queries in tensor memory and folds the
 *   log-sum-exp into its epilogue.  cor_sim_stream_fwd serves both in one pass.
 * ---------------------------------------------------------------------------------------- */
size_t cor_sim_work_bytes(int Nq, int Nr, int D);
int cor_sim_stream_fwd(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau,
                       float* S, float* lse, void* work, cor_stream_t stream);
int cor_sim_umma_fwd(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau,
                     float* S, float* lse, void* work, cor_stream_t stream);
/* As cor_sim_{stream,umma}_fwd asked for lse only, but the log-sum-exp partials stay in `work`, laid out
 * [ceil(Nq / *qt)][*nparts][*qt][2] (running max, sum), for cor_infonce_tail to merge.  engine: 0 = stream, 1 = umma. */
int cor_sim_lse_parts(int engine, const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau,
                      void* work, int* nparts, int* qt, cor_stream_t stream);
/* The tail of the fused step in ONE launch: merge of those partials -> lse [Nq]; tgt_logit and nce as cor_infonce_fwd;
 * and, when total != NULL, total = seg[0] + w_fg * fgbg[0] + w_bg * fgbg[1] + w_nce * nce (utils/trainer_v3_g.py:67-73
 * plus the Class-N term). */
int cor_infonce_tail(const float* lse_part, int nparts, int qt, const void* regions, const void* queries,
                     const long long* targets, int Nr, int Nq, int D, float inv_tau, float* lse, float* nce,
                     float* tgt_logit, const float* seg, const float* fgbg, float w_fg, float w_bg, float w_nce,
                     float* total, cor_stream_t stream);
/* loss = mean_q (lse[q] - S[q, target[q]] / tau); tgt_logit [Nq] is S[q,target[q]] (f32). */
int cor_infonce_fwd(const void* regions, const void* queries, const long long* targets, const float* lse,
                    int Nr, int Nq, int D, float inv_tau, float* loss, float* tgt_logit, cor_stream_t stream);
/* g_regions [Nr, D] f32 and/or g_queries [Nq, D] f32 (either may be NULL) for upstream scalar *g_loss * g_mul.
 * A rank of a data-parallel job can call it twice -- (all regions, its queries) -> g_queries and
 * (its regions, all queries; g_mul = world size) -> g_regions -- so that the backward needs no collective. */
int cor_infonce_bwd(const void* regions, const void* queries, const long long* targets, const float* lse,
                    int Nr, int Nq, int D, float inv_tau, const float* g_loss, float g_mul, float* g_regions,
                    float* g_queries, void* work, cor_stream_t stream);
/* InfoNCE backward for MANY queries on tcgen05 tensor cores (csrc/nce_bwd_umma.cu): dQ = P R and dR = P^T Q with
 * P = (exp(S/tau - lse) - onehot(target)) * g_loss[0] * g_mul / (tau * Nq) formed tile by tile in registers and fed back
 * to the tensor cores through shared memory -- neither S nor P is ever written to global memory and no library GEMM
 * is involved.  regions [Nr,D], queries [Nq,D] bf16, D in {64,128,192,256}; g_regions [Nr,D] / g_queries [Nq,D] f32
 * (either may be NULL); work: cor_infonce_bwd_umma_work_bytes() bytes (fp32 split partials, folded in fixed order). */
size_t cor_infonce_bwd_umma_work_bytes(int Nq, int Nr, int D);
int cor_infonce_bwd_umma(const void* regions, const void* queries, int Nr, int Nq, int D, float inv_tau, const float* lse,
                         const long long* targets, const float* g_loss, float g_mul, float* g_regions, float* g_queries,
                         void* work, cor_stream_t stream);

/* Learnable temperature: the entries above with the logit scale s (= 1/tau) read from device memory instead of the
 * float inv_tau.  logit_scale: one f32 on the device, positive; read once per CTA when the kernel runs, so a captured
 * CUDA graph picks up a new value at every replay.  S, lse and every coefficient are those of the float entries at
 * inv_tau = *logit_scale (bit-equal for the same f32 value).  Same arguments otherwise, same kernels, same launches.
 * The backward entries also write g_logit_scale (one f32 on the device; NULL = not wanted):
 *   d loss / d s = g_loss[0] * g_mul * mean_q sum_r (exp(s S[q,r] - lse[q]) - [r == target(q)]) S[q,r]
 * from per-query partials folded in a fixed order (no float atomics, no host synchronisation: deterministic and
 * graph-capturable).
 *   cor_sim_stream_fwd_ls, cor_sim_umma_fwd_ls, cor_sim_lse_parts_ls, cor_infonce_tail_ls, cor_infonce_fwd_ls: as the
 *     entries without the suffix.
 *   cor_infonce_bwd_ls: extends cor_infonce_bwd.  The gradient comes from the (regions, queries) pair of the call, so a
 *     data-parallel rank asks for it on its (all regions, its queries) call; g_logit_scale needs `work`.
 *   cor_infonce_bwd_umma_ls: extends cor_infonce_bwd_umma.  The dQ launch forms the partials; with g_logit_scale but
 *     no g_queries it still runs (the whole dQ GEMM, result not stored), plus one single-CTA fold launch.
 * ---------------------------------------------------------------------------------------- */
int cor_sim_stream_fwd_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                          float* S, float* lse, void* work, cor_stream_t stream);
int cor_sim_umma_fwd_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                        float* S, float* lse, void* work, cor_stream_t stream);
int cor_sim_lse_parts_ls(int engine, const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                         void* work, int* nparts, int* qt, cor_stream_t stream);
int cor_infonce_tail_ls(const float* lse_part, int nparts, int qt, const void* regions, const void* queries,
                        const long long* targets, int Nr, int Nq, int D, const float* logit_scale, float* lse, float* nce,
                        float* tgt_logit, const float* seg, const float* fgbg, float w_fg, float w_bg, float w_nce,
                        float* total, cor_stream_t stream);
int cor_infonce_fwd_ls(const void* regions, const void* queries, const long long* targets, const float* lse,
                       int Nr, int Nq, int D, const float* logit_scale, float* loss, float* tgt_logit, cor_stream_t stream);
int cor_infonce_bwd_ls(const void* regions, const void* queries, const long long* targets, const float* lse,
                       int Nr, int Nq, int D, const float* logit_scale, const float* g_loss, float g_mul, float* g_regions,
                       float* g_queries, float* g_logit_scale, void* work, cor_stream_t stream);
int cor_infonce_bwd_umma_ls(const void* regions, const void* queries, int Nr, int Nq, int D, const float* logit_scale,
                            const float* lse, const long long* targets, const float* g_loss, float g_mul, float* g_regions,
                            float* g_queries, float* g_logit_scale, void* work, cor_stream_t stream);

/* Top-k retrieval: per query the k best regions under (score desc, index asc), where score is the
 * canonical value fl32(sum in fp64 of exact bf16 products).  S is the (tensor-core) prefilter
 * matrix from cor_sim_*; the top (k + slack) prefilter candidates are re-scored exactly.
 *   idx [Nq, k] int64, score [Nq, k] f32. */
int cor_topk(const float* S, const void* regions, const void* queries, int Nr, int Nq, int D, int k,
             long long* idx, float* score, cor_stream_t stream);

/* Row-wise L2 normalise x / max(|x|, 1e-12) (support_branch.py:85, cir_feature_fuse.py:59):
 *   x [n, D] f32/bf16 -> y_f32 and/or y_bf16. */
int cor_l2_normalize(const void* x, int x_dtype, int n, int D, float* y_f32, void* y_bf16, float* inv_norm,
                     cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Validation post-process (trainer_v3_g.py:226-231; vailder.py:427-430,473): bilinear resize of
 * the logits to HoxWo, sigmoid, per-sample min-max stretch (+1e-8), optional binarise (>0.5)*255
 * and the soft metrics of trainer_v3_g.py:381-443 against gt [N,Ho,Wo] (f32/u8) if given.
 *   post [N,Ho,Wo] f32 or NULL; hard [N,Ho,Wo] u8 or NULL; metrics [N,5] {dice,mae,iou,mdice,miou}.
 * ---------------------------------------------------------------------------------------- */
size_t cor_val_post_work_bytes(int N, int Ho, int Wo);
int cor_val_post(const void* pred, int pred_dtype, int N, int H, int W, int Ho, int Wo,
                 int post_first /* 0: resize logits, then sigmoid + min-max (trainer_v3_g.py:226-231);
                                   1: sigmoid + min-max at the logit size, then resize the map (vailder.py:427-430,466) */,
                 float* post,
                 uint8_t* hard, const void* gt, int gt_dtype, float gt_scale, float* metrics, void* work,
                 cor_stream_t stream);

/* Soft metrics of utils/trainer_v3_g.py:381-443 on an already post-processed map: pred [N, total] f32, gt [N, total]
 * f32 / u8 -> metrics [N,5] {dice, mae, iou, mdice, miou}; work: cor_val_post_work_bytes(N, ...) bytes. */
int cor_soft_metrics(const float* pred, const void* gt, int gt_dtype, float gt_scale, int N, long long total,
                     float smooth, float* metrics, void* work, cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * General bf16 GEMM on tcgen05 tensor cores with a fused epilogue (csrc/gemm_umma.cu): the building block of the
 * learned modules either side of the region path -- the 1x1 convolutions / point-wise MLPs of GenerateMaskAdapterMap
 * (lib/support_model/mask_adapter.py:97-223) and the linear layers of the composed-query head
 * (lib/support_model/cir_feature_fuse.py:20-43, lib/support_branch.py:47-54), forward and backward.
 *   C[b][m][n] = epi( alpha * sum_k A[b](m,k) B[b](n,k) ),  epi: + bias[n]; (pre = v, bf16, optional); act; * emul[b][m][n]
 *   (dropout mask, optional); * colscale[n]; + residual[b][m][n]; store f32 / bf16 with row pitch ldc.
 *   Operand orientation (x_mn): 0 = K-major, stored [rows][K]; 1 = MN-major, stored [K][rows].  Both are 2-D bf16 tensors of
 *   x_rows_total rows (K-major: x_rows_total x K; MN-major: x_rows_total x rows, x_rows_total = batch * K); batch entry b
 *   starts at row b * x_batch_rows (0 = the operand is shared by every batch entry).  Row pitches must be multiples of 16 B.
 *   ksplit: 0 = automatic split-K when there are few output tiles (weight-gradient GEMMs), >0 forces it; split partials are
 *   folded in fixed order.  work: cor_gemm_bf16_work_bytes() bytes.
 * ---------------------------------------------------------------------------------------- */
enum { COR_ACT_NONE = 0, COR_ACT_RELU = 1, COR_ACT_GELU = 2, COR_ACT_SIGMOID = 3 };
size_t cor_gemm_bf16_work_bytes(int M, int N, int K, int batch, int ksplit);
int cor_gemm_bf16(const void* A, int a_mn, long long a_rows_total, long long a_batch_rows, const void* B, int b_mn,
                  long long b_rows_total, long long b_batch_rows, int M, int N, int K, int batch, float alpha, const float* bias,
                  int act, const float* emul, const float* colscale, const void* residual, int res_dtype, long long ldr, void* C,
                  int c_dtype, long long ldc, void* pre_bf16, int ksplit, void* work, cor_stream_t stream);

/* Operand prep and epilogue backward for cor_gemm_bf16 (csrc/ew.cu).
 *   cor_cast_cat_bf16: out[r] = bf16(concat(a[r][0:c0], b[r][0:c1])) (b NULL, c1 = 0: a plain cast) -- torch.cat at
 *                      cir_feature_fuse.py:49,54 fused with the operand cast.
 *   cor_act_bwd: dz = dy * emul * colscale * act'(.) as bf16 [M,N]; db[n] = sum_m dz; dcolscale[n] = sum_m dy * emul * pre
 *                (rows in chunk order: deterministic).  y_f32 = activation output before mask / scale (relu, sigmoid),
 *                pre_bf16 = pre-activation saved by the GEMM (gelu; the un-scaled linear output for a column scale).
 *                work: cor_act_bwd_work_bytes(M, N) bytes when db or dcolscale is requested. */
int cor_cast_cat_bf16(const float* a, int c0, const float* b, int c1, long long rows, void* out_bf16, cor_stream_t stream);
/* out[b][r][:] = bf16(src[b][r][:]) for r < rows, zeros up to rows_padded: a K-padded MN-major GEMM operand (the pooling
 * backward d feat[b] = gs[b]^T w[b] as one batched cor_gemm_bf16, cor_b200/region.py). cols % 4 == 0. */
int cor_cast_pad_rows_bf16(const float* src, int batch, int rows, int rows_padded, int cols, void* out_bf16, cor_stream_t stream);
size_t cor_act_bwd_work_bytes(long long M, int N);
int cor_act_bwd(const void* dy, int dy_dtype /* f32 or bf16 */, const float* y_f32, const void* pre_bf16, const float* emul,
                const float* colscale, int act,
                long long M, int N, void* dz_bf16, float* db, float* dcolscale, void* work, cor_stream_t stream);

/* Row-wise LayerNorm (+ optional GELU) over channels-last rows, forward and backward (csrc/ln_rows.cu): the norms of the
 * MaskAdapter map generator (lib/support_model/mask_adapter.py:83-94, :171-173, :200-209, :240-251).
 *   y = act((x - mean) * rstd * weight + bias), x [rows, C] f32, C <= 1024; y f32 or bf16; stats [rows, 2] = {mean, rstd}.
 *   bwd: dx [rows, C], dweight / dbias [C]; work: cor_ln_rows_work_bytes(rows, C). */
size_t cor_ln_rows_work_bytes(long long rows, int C);
int cor_ln_rows_fwd(const float* x, const float* weight, const float* bias, long long rows, int C, float eps, int act,
                    void* y, int y_dtype, float* stats, cor_stream_t stream);
int cor_ln_rows_bwd(const void* dy, int dy_dtype /* f32 or bf16 */, const float* x, const float* weight, const float* bias, const float* stats,
                    long long rows, int C, int act, float* dx, float* dweight, float* dbias, void* work, cor_stream_t stream);

/* Channels-first LayerNorm over a few channels (+ GELU), x [N][C][P] f32, C <= 32 (csrc/ln_rows.cu): the two
 * normalisations of mask_downscaling (lib/support_model/mask_adapter.py:128-142, LayerNorm(channels_first) :240-251 -
 * mean / pow / sqrt over dim 1 as separate element-wise launches in the reference), one launch forward, one backward
 * (+ the fold of the affine gradients).  work: cor_ln_cf_work_bytes(N, C, P). */
size_t cor_ln_cf_work_bytes(long long N, int C, long long P);
int cor_ln_cf_fwd(const float* x, const float* weight, const float* bias, long long N, int C, long long P, float eps, int act,
                  float* y, cor_stream_t stream);
int cor_ln_cf_bwd(const float* dy, const float* x, const float* weight, const float* bias, long long N, int C, long long P, float eps,
                  int act, float* dx, float* dweight, float* dbias, void* work, cor_stream_t stream);

/* Depth-wise 7x7 convolution (padding 3, stride 1) on channels-last maps [n][h][w][C] f32 (csrc/dwconv.cu): the spatial
 * step of the ConvNeXt blocks (lib/support_model/mask_adapter.py:196-199).  weight [C][49] (nn.Conv2d's [C,1,7,7]), bias [C] or
 * NULL; flip = 1 applies the kernel rotated by 180 degrees = the gradient w.r.t. the input when `in` is d out.
 * cor_dwconv7_cl_wgrad: dweight [C][49] and dbias [C] (may be NULL) from (in, d out); work: cor_dwconv7_work_bytes().
 * C % 32 == 0; the row band + halo of 32 channels must fit shared memory (w <= ~300). */
size_t cor_dwconv7_work_bytes(int n, int h, int w, int C);
int cor_dwconv7_cl(const float* in, const float* weight, const float* bias, float* out, int n, int h, int w, int C, int flip,
                   cor_stream_t stream);
int cor_dwconv7_cl_wgrad(const float* in, const float* dout, float* dweight, float* dbias, int n, int h, int w, int C, void* work,
                         cor_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Mask-logit producer (SURVEY.md 8f rank 3): the hypernetwork product of the SAM decoder,
 *   masks[b, t, p] = sum_c hyper_in[b, t0 + t, c] * upscaled[b, c, p]     lib/sam_model/mask_decoder.py:135-137
 * for the T consumed tokens only (the reference computes all four and slices, :97-102), written in the dtype the
 * segmentation-loss kernel reads.  hyper [B, T_all, C] f32, up [B, C, P] f32/bf16, out [B, T, P] f32/bf16;
 * T <= 4, C <= 64, P % 4 == 0.  Backward in one pass over `up` and the logit gradient g [B, T, P]:
 * d_up [B, C, P] (dtype of up; may be NULL) and d_hyper [B, T_all, C] f32 (zero rows for unused tokens);
 * work: cor_hyper_logits_work_bytes() bytes of per-CTA partials, folded in fixed order.
 * ---------------------------------------------------------------------------------------- */
size_t cor_hyper_logits_work_bytes(int B, int T, int C, long long P);
int cor_hyper_logits_fwd(const float* hyper, const void* up, int up_dtype, void* out, int out_dtype, int B, int T_all, int t0,
                         int T, int C, long long P, cor_stream_t stream);
int cor_hyper_logits_bwd(const float* hyper, const void* up, int up_dtype, const void* g, int g_dtype, void* d_up,
                         float* d_hyper, int B, int T_all, int t0, int T, int C, long long P, void* work, cor_stream_t stream);

/* Pooling tail of MaskAdapterPooling on the tensor cores (csrc/adapter_tail.cu; lib/support_model/mask_adapter.py:62-79:
 * softmax over pixels of logsigmoid(maps), mask_weights @ feat^T, mean over the num_output_maps maps of a mask).  The mean
 * and the per-map normalisation fold into one weight row per mask, Wq[b,q,p] = (1/G) sum_j sigmoid(maps[b,qG+j,p]) / den,
 * so the pooling is ONE batched cor_gemm_bf16 (out[b] = Wq[b] feat[b]^T).  These two entries are its element-wise ends:
 *   cor_adapter_tail_weights: maps [B][R][P] f32 -> wq [B][Qp][P] bf16 (rows q >= R/G untouched: the caller zeroes them
 *                             once so that Qp, a multiple of 64, can serve as a GEMM K extent in the backward), den [B*R].
 *   cor_adapter_tail_bwd:     gwq [B][R/G][P] f32 (= g_out[b] feat[b], a GEMM) -> gmaps [B][R][P] f32. */
int cor_adapter_tail_weights(const float* maps, int B, int R, int P, int G, int Qp, void* wq_bf16, float* den, cor_stream_t stream);
int cor_adapter_tail_bwd(const float* maps, const float* den, const float* gwq, int B, int R, int P, int G, float* gmaps,
                         cor_stream_t stream);

/* ----------------------------------------------------------------------------------------------
 * (e) Multi-GPU exchange over NVLink peer memory (one process per GPU, one node) - the B200-native replacement of
 * the all-gather of the region rows and the reduce-scatter of their gradient around the similarity stage
 * (SURVEY.md §8e; the reference gathers nothing: its loss is per-sample, utils/trainer_v3_g.py:67-73, and its
 * multi-GPU plumbing is accelerate/DDP, utils/trainer_v3_g.py:46-57).
 *   cor_peer_alloc/free: a zero-filled cudaMalloc region on `device`; cor_peer_export: its 64-byte CUDA IPC handle;
 *   cor_peer_open/close: map a peer's region into this process (peer access enabled lazily).
 *   flags: every rank sets aside cor_peer_flag_bytes() of its region (zeroed), peers signal into it; state:
 *   cor_peer_state_bytes() of LOCAL zeroed memory (epoch + CTA counter per channel, then one error word).
 *   Waits last at most COR_PEER_TIMEOUT_S seconds (environment, default 600, 0 = unbounded); an expired wait does not
 *   trap: it stores 0x80000000|epoch in state[cor_peer_error_word()] and the kernel carries on with stale data, so
 *   the host must check that word before trusting a step (cor_b200.peer.PeerExchange.check()).
 *   peer_src / peer_flags: DEVICE arrays [world] of pointers (entry `rank` = the local buffer).
 *   cor_peer_gather_rows:  all[p*bytes : (p+1)*bytes] = peer_src[p][0 : bytes]   for every rank p
 *   cor_peer_reduce_rows:  out[i] = sum_p peer_src[p][rank*floats + i], p ascending (deterministic)
 *   cor_peer_signal:    "my buffer for the next epoch of `channel` is ready" - one tiny CTA right after the producer
 *                       kernel; exactly one per exchange, BEFORE it (what runs in between hides the rank skew)
 *   cor_peer_wait_exit: "every peer has finished reading what my last exchange on `channel` published" - needed
 *                       before the producer only when no exchange on the other channel ran since (cor_b200/peer.py)
 *   The exchanges wait for all peers' signal, pull, and post their own exit flag.  Epochs live in device memory:
 *   graph-capturable; every rank must issue the same sequence.
 * ---------------------------------------------------------------------------------------------- */
int cor_peer_max_world(void);
size_t cor_peer_flag_bytes(void);
size_t cor_peer_state_bytes(void);
int cor_peer_error_word(void);   /* index (in u32 words) of the error word inside `state`: non-zero = a wait expired */
int cor_peer_alloc(int device, size_t bytes, void** ptr);
int cor_peer_free(void* ptr);
int cor_peer_export(void* ptr, unsigned char* handle64);
int cor_peer_open(int device, const unsigned char* handle64, void** ptr);
int cor_peer_close(void* ptr);
int cor_peer_signal(void* const* peer_flags, void* state, int rank, int world, int channel, cor_stream_t stream);
int cor_peer_wait_exit(void* const* peer_flags, void* state, int rank, int world, int channel, cor_stream_t stream);
int cor_peer_gather_rows(const void* const* peer_src, void* all, long long bytes_per_rank, void* const* peer_flags, void* state,
                         int rank, int world, int channel, cor_stream_t stream);
int cor_peer_reduce_rows(const void* const* peer_src, float* out, long long floats_per_rank, void* const* peer_flags, void* state,
                         int rank, int world, int channel, cor_stream_t stream);
/* Fused all-gather + similarity for a rank's few (<= 16) queries: ONE kernel pulls every peer's region rows over NVLink
 * once, writes them into the local gathered buffer `all` [world*n_local][D] bf16 (rank-major, what cor_peer_gather_rows
 * produces) and, while a row is in registers, scores it against `queries` [Nq][D] bf16 -- leaving the log-sum-exp partials
 * `part` [*nparts][16][2] in the layout cor_infonce_tail consumes (same as cor_sim_lse_parts, qt = 16).  Same flag protocol
 * as cor_peer_gather_rows (enter barrier on `channel`, exit flag).  D % 8 == 0, D <= 256.
 * part: cor_peer_gather_sim_work_bytes() bytes. */
size_t cor_peer_gather_sim_work_bytes(void);
int cor_peer_gather_sim(const void* const* peer_src, void* all, long long n_local, int D, const void* queries, int Nq, float inv_tau,
                        float* part, int* nparts, void* const* peer_flags, void* state, int rank, int world, int channel,
                        cor_stream_t stream);
/* Extends cor_peer_gather_sim: the logit scale is read from device memory (logit_scale, one f32), as the _ls InfoNCE entries. */
int cor_peer_gather_sim_ls(const void* const* peer_src, void* all, long long n_local, int D, const void* queries, int Nq,
                           const float* logit_scale, float* part, int* nparts, void* const* peer_flags, void* state, int rank, int world,
                           int channel, cor_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* COR_B200_H_ */
