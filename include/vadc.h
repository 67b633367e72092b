/* vadc.h — C ABI of libvadc.so: the B200 (sm_100a) kernels behind the
 * clustering / memory / loss / scoring hot path of
 * Bun-TianYi/Video-anomaly-detection-guided-by-clustering-learning.
 *
 * The reference has no FFI layer (it is a pure PyTorch program; SURVEY.md §8b),
 * so every entry point below names the reference Python symbol (file:line,
 * relative to the reference root) whose arithmetic it replaces.  The host-side
 * mirror classes in video-anomaly-detection-guided-by-clustering-learning_b200/
 * bind these with ctypes; INTEGRATION.md shows the binding a reference
 * maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless marked host; all float tensors
 *    are fp32, contiguous, 16-byte aligned; labels / indices are int64.
 *  - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream()).
 *  - functions never allocate, never synchronise the stream and never throw.
 *    Scratch memory is caller-provided: ask the matching *_workspace_bytes().
 *  - return value: 0 on success, a negative VADC_ERR_* code otherwise
 *    (vadc_error_string() gives the text; the Python wrapper raises
 *    RuntimeError with it, mirroring the reference's exception-only error
 *    convention).
 */
#ifndef VADC_H_
#define VADC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VADC_OK 0
#define VADC_ERR_BAD_SHAPE (-1)      /* a size is <= 0 or violates a stated constraint   */
#define VADC_ERR_NULL_POINTER (-2)   /* a required pointer is NULL                        */
#define VADC_ERR_MISALIGNED (-3)     /* a pointer is not 16-byte aligned                  */
#define VADC_ERR_WORKSPACE (-4)      /* workspace too small                               */
#define VADC_ERR_CUDA (-5)           /* a CUDA call / launch failed (see vadc_last_cuda_error) */
#define VADC_ERR_UNSUPPORTED (-6)    /* shape outside what this kernel variant supports   */
#define VADC_ERR_NO_DEVICE (-7)      /* no sm_100 device                                  */

/* implementation selector for ops that have more than one kernel family */
#define VADC_IMPL_AUTO 0             /* tcgen05 path when the shape fits, else SIMT      */
#define VADC_IMPL_SIMT 1             /* fp32 CUDA-core kernels (any shape)               */
#define VADC_IMPL_TCGEN05 2          /* tcgen05/TMEM/TMA kernel; VADC_ERR_UNSUPPORTED if the shape does not fit */

/* pixel-loss reductions (vadc_pixel_loss*) */
#define VADC_LOSS_L1_MEAN 0          /* Recon_Loss: mean |x-t|      loss_tool/Recon_Loss.py:23-32 */
#define VADC_LOSS_MSE_MEAN 1         /* mean (x-t)^2                main.py:191                    */
#define VADC_LOSS_E4_NORM 2          /* sqrt(sum (x-t)^4)           main_predict.py:273-275        */

const char* vadc_version(void);
const char* vadc_error_string(int code);
const char* vadc_last_cuda_error(void);              /* text of the last CUDA failure on this thread */
int vadc_device_ok(void);                            /* 1 if the current device is sm_100          */
/* number of kernel launches this library has issued in this process (bench.py's gpu_launches) */
unsigned long long vadc_launch_count(void);
/* The kernel-variant switches (VADC_BWD_IMPL, VADC_NO_TC_GEMM, ... — A/B runs and debugging) are environment
 * variables read once per process at their first use; call this after changing one of them at run time. */
int vadc_refresh_env(void);

/* Measurement aid: with timing enabled, CUDA events are recorded on the launching stream immediately around
 * the two dominant kernels (slot 0: the fused K = 32 cluster forward of vadc_cluster_fwd, slot 1: the fused
 * tcgen05 cluster backward of vadc_cluster_bwd), up to 256 launches per slot.  vadc_timing_read synchronises on
 * the recorded events and returns the mean kernel duration; enabling resets the counters.  Do not enable while
 * a stream is being captured into a CUDA graph. */
int vadc_timing_enable(int on);
int vadc_timing_read(int slot, float* mean_ms, int* count);

/* ------------------------------------------------------------------------ *
 * C1 + L1: EuclidDistance_Assign_Module.forward   model/cluster.py:81-99
 *          NegSoftAssign.forward                   model/cluster.py:48-55
 *          torch.norm(x_distance * x_assign)       model/backbone.py:98
 *
 * x [N,C] tokens (channel-last 'B D H W C' flattened), centers [K,C].
 *   feature = LayerNorm_C(x)                        [N,C]
 *   D       = sqrt(max(0,|f|^2+|c|^2-2 f.c^T))      [N,K]   (torch.cdist, mm form)
 *   label   = argmin_k D (first minimum)            [N] int64
 *   A       = exp(-alpha (D - min_k D)) / sum_k     [N,K]
 *   x_rec   = A @ centers                           [N,C]
 *   mu,rstd = LayerNorm statistics                  [N] each (saved for the backward)
 *   rowstats = per-token sums the backward's closed-form LayerNorm statistics use, [N,4]:
 *              |f|^2, sum_c f gamma, sum_c f gamma xhat, 0   (may be NULL: not produced)
 *   loss_sq = sum (D*A)^2                           [1]     (sqrt of it is the cluster loss)
 * Constraints: 1 <= C <= 4096 (VADC_ERR_UNSUPPORTED above), K % 4 == 0.  Any C: rows of C % 4 != 0 are read without
 * assuming 16-byte alignment (the base pointers still need it); the tensor-core contractions run over C rounded up to 8
 * with zero padding.  The same holds for vadc_cluster_fwd_padded and vadc_cluster_bwd.
 * ------------------------------------------------------------------------ */
size_t vadc_cluster_fwd_workspace_bytes(int64_t N, int C, int K, int impl);
int vadc_cluster_fwd(const float* x, const float* ln_w, const float* ln_b,
                     const float* centers, int64_t N, int C, int K,
                     float alpha, float eps,
                     float* D, float* A, float* x_rec, float* feature,
                     int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq,
                     void* workspace, size_t workspace_bytes, int impl, void* stream);

/* PosSoftAssign.forward / NegSoftAssign.forward  model/cluster.py:27-55, stand-alone:
 * y = exp(a (x - ext)) / sum over the last axis of x [rows,K]; a = +alpha with
 * ext = max (Pos) or a = -alpha with ext = min (Neg).  _bwd: gx = a y (g - sum g y). */
int vadc_soft_assign(const float* x, int64_t rows, int K, float signed_alpha, float* y, void* stream);
int vadc_soft_assign_bwd(const float* y, const float* g, int64_t rows, int K, float signed_alpha,
                         float* gx, void* stream);

/* EuclidDistance_Assign_Module.self_similarity   model/cluster.py:77-79
 * Space_...Module.self_similarity                 model/cluster.py:124-125
 * batched torch.cdist(a, b): a [nb,R,C], b [nb,P,C] -> out [nb,R,P]. */
size_t vadc_cdist_workspace_bytes(int nb, int64_t R, int64_t P, int C);
int vadc_cdist(const float* a, const float* b, int nb, int64_t R, int64_t P, int C,
               float* out, void* workspace, size_t workspace_bytes, void* stream);
/* Its backward (torch.cdist's gradient, ATen's _euclidean_dist_backward), per batch:
 *   r = g / dist (0 where dist == 0), ga = a rowsum(r) - r b, gb = b colsum(r) - r^T a.
 * a [nb,R,C], b [nb,P,C], dist [nb,R,P] (vadc_cdist's output), g [nb,R,P] -> ga [nb,R,C], gb [nb,P,C];
 * either output may be NULL (not computed).  self != 0: a == b (b may be NULL), R == P, ga receives the whole
 * gradient of cdist(a, a) and gb must be NULL; the diagonal is skipped (its exact contribution is 0).  Empty problems
 * (nb, R or P == 0) write zero gradients.  nb <= 65535.  Deterministic; no allocation, no synchronisation. */
size_t vadc_cdist_bwd_workspace_bytes(int nb, int64_t R, int64_t P, int C);
int vadc_cdist_bwd(const float* a, const float* b, const float* dist, const float* g, int nb, int64_t R, int64_t P,
                   int C, int self, float* ga, float* gb, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * C2: autograd of C1 — the reference's "centroid update" (SURVEY.md D4):
 *     loss.backward()  main_predict.py:296, through cluster.py:84-95.
 *
 * Inputs saved by the forward: x, mu, rstd, rowstats (NULL allowed: slower kernel), feature, D, A.  Upstream grads
 * (each may be NULL = zero): gD, gA [N,K]; gR (x_rec) , gF (feature) [N,C].
 * Fused loss gradient (optional): if g_loss_sq != NULL (device scalar, the
 * upstream gradient of the forward's loss_sq = sum (D*A)^2) its contribution
 * is added in-kernel (gD += 2 g D A^2, gA += 2 g D^2 A) without materialising
 * two [N,K] tensors.  The caller derives g_loss_sq from whatever it did with
 * loss_sq (local sqrt, or all-reduce over ranks then sqrt: SURVEY.md §8e).
 * Outputs: gx [N,C]; gcenters [K,C]; g_ln_w, g_ln_b [C] (overwritten, not
 * accumulated).  Shapes as vadc_cluster_fwd: 1 <= C <= 4096, K % 4 == 0.
 * ------------------------------------------------------------------------ */
size_t vadc_cluster_bwd_workspace_bytes(int64_t N, int C, int K);
int vadc_cluster_bwd(const float* x, const float* mu, const float* rstd, const float* rowstats,
                     const float* feature, const float* ln_w, const float* ln_b,
                     const float* centers,
                     const float* D, const float* A,
                     const float* gD, const float* gA, const float* gR, const float* gF,
                     const float* g_loss_sq,
                     int64_t N, int C, int K, float alpha,
                     float* gx, float* gcenters, float* g_ln_w, float* g_ln_b,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * C3 + L1: Space_EuclidDistance_Assign_Module.forward  model/cluster.py:127-149
 *          torch.norm(xf_distance * xf_assign)          model/backbone.py:94
 *
 * x [M*P, C] tokens (M = B*D clips-frames, P = H*W), centers [C,K,P].
 *   Ds [M,C,K] ('B D C CN'), As [M,C,K], mu/rstd [M*P], loss_sq [1];
 *   selfdist [C,K,K] = cdist(centers, centers) (model/cluster.py:134), or NULL to skip it.
 * zt_state (vadc_space_cluster_saved_bytes bytes, 16-byte aligned) keeps the
 * LayerNorm output in the transposed layout [C,M,P] the batched cdist consumes,
 * for the backward: opaque to the caller — the three bf16 operand terms of the
 * tensor-core contractions (their exact sum is the fp32 value) where those run,
 * plain fp32 otherwise.  The forward and its backward must run under the same
 * environment (no vadc_refresh_env in between).
 * ------------------------------------------------------------------------ */
size_t vadc_space_cluster_saved_bytes(int64_t M, int P, int C, int K);
size_t vadc_space_cluster_fwd_workspace_bytes(int64_t M, int P, int C, int K);
int vadc_space_cluster_fwd(const float* x, const float* ln_w, const float* ln_b,
                           const float* centers, int64_t M, int P, int C, int K,
                           float alpha, float eps,
                           float* Ds, float* As, float* selfdist, void* zt_state, float* mu, float* rstd,
                           float* loss_sq,
                           void* workspace, size_t workspace_bytes, void* stream);

/* Any cluster_num (the reference's constructors take any: model/cluster.py:58-75, :102-122): the kernels address rows
 * of K fp32 values with 128-bit accesses, so K % 4 == 0 is required; for other sizes the HOST pads the centroids with
 * K - K_valid trailing rows (any finite values; the Python wrapper uses zeros) and calls these entry points, which exclude
 * the padding from argmin / softmin / loss (A is exactly 0 there, D holds the finite distance to the padding row).  The
 * backward entry points need no change: A = 0 makes every gradient through a padded column 0. */
int vadc_cluster_fwd_padded(const float* x, const float* ln_w, const float* ln_b, const float* centers,
                            int64_t N, int C, int K, int K_valid, float alpha, float eps,
                            float* D, float* A, float* x_rec, float* feature, int64_t* label,
                            float* mu, float* rstd, float* rowstats, float* loss_sq,
                            void* workspace, size_t workspace_bytes, void* stream);
int vadc_space_cluster_fwd_padded(const float* x, const float* ln_w, const float* ln_b,
                                  const float* centers, int64_t M, int P, int C, int K, int K_valid,
                                  float alpha, float eps,
                                  float* Ds, float* As, float* selfdist, void* zt_state, float* mu, float* rstd,
                                  float* loss_sq,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* autograd of C3 (main_predict.py:296). gD/gA [M,C,K] may be NULL; optional
 * fused loss gradient as in vadc_cluster_bwd.  Outputs gx [M*P,C],
 * gcenters [C,K,P], g_ln_w, g_ln_b [C]. */
size_t vadc_space_cluster_bwd_workspace_bytes(int64_t M, int P, int C, int K);
int vadc_space_cluster_bwd(const float* x, const float* mu, const float* rstd,
                           const void* zt_state, const float* ln_w, const float* ln_b,
                           const float* centers,
                           const float* Ds, const float* As,
                           const float* gD, const float* gA,
                           const float* g_loss_sq,
                           int64_t M, int P, int C, int K, float alpha,
                           float* gx, float* gcenters, float* g_ln_w, float* g_ln_b,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * L2 / L3: pixel losses as single-pass reductions.
 *   Recon_Loss.forward                     loss_tool/Recon_Loss.py:23-32
 *   torch.mean(MSELoss(none)(r,t))         main.py:191
 *   torch.norm(MSELoss(none)(r,t))         main_predict.py:273-275
 * x, t: n floats.  n_pad extra elements of x (at x_pad) are compared with 0
 * (Recon_Loss zero-pads the target on D; NULL/0 when no padding).  out[0] =
 * the loss value; out[1] = the raw sum (for a cross-rank all-reduce).
 * ------------------------------------------------------------------------ */
size_t vadc_pixel_loss_workspace_bytes(int64_t n);
int vadc_pixel_loss(const float* x, const float* t, int64_t n,
                    const float* x_pad, int64_t n_pad, int mode, float* out,
                    void* workspace, size_t workspace_bytes, void* stream);
/* d loss / d x  (gout: upstream scalar grad on device; out_fwd: the `out` of the forward) */
int vadc_pixel_loss_bwd(const float* x, const float* t, int64_t n, int mode,
                        const float* gout, const float* out_fwd, int64_t n_total,
                        float* gx, void* stream);

/* ------------------------------------------------------------------------ *
 * E1: per-frame reconstruction error
 *   tool/evaluate.py:175-179, tool/contrast_evaluae.py:232-236,
 *   tool/predict_evaluae.py:228-234, main_predict.py:420-423
 * recon, clip [B,Cc,T,H*W] -> mse [B,T] (mean over Cc,H,W) and, if
 * psnr != NULL, psnr [B,T] = 10 log10(1/mse) in float64 (misc/utils.py:124-128).
 * ------------------------------------------------------------------------ */
size_t vadc_frame_mse_workspace_bytes(int B, int T, int64_t HW, int Cc);
int vadc_frame_mse(const float* recon, const float* clip, int B, int Cc, int T, int64_t HW,
                   float* mse, double* psnr,
                   void* workspace, size_t workspace_bytes, void* stream);
/* The same reduction over strided views (strides in ELEMENTS along batch, channel, frame; the H*W plane itself is
 * contiguous): clip batches are taken out of a device-resident video without a copy — consecutive clips
 * (tool/contrast_evaluae.py:185-203), clips that overlap by all but one frame (tool/predict_evaluae.py:185-203,
 * main_predict.py:401-404) — and single frames of a reconstruction (recon[:, :, 0], main_predict.py:417-420). */
int vadc_frame_mse_strided(const float* recon, int64_t recon_stride_b, int64_t recon_stride_c, int64_t recon_stride_t,
                           const float* clip, int64_t clip_stride_b, int64_t clip_stride_c, int64_t clip_stride_t,
                           int B, int Cc, int T, int64_t HW, float* mse, double* psnr,
                           void* workspace, size_t workspace_bytes, void* stream);

/* E3: anomly_score  misc/utils.py:131-135 — per-video 1 - minmax(psnr).
 * psnr [total] float64, seg_offsets [n_videos+1] int64 (device) -> score [total]
 * float64.  A constant segment yields NaN (the reference raises
 * ZeroDivisionError; the Python wrapper turns NaN segments into that). */
int vadc_minmax_score(const double* psnr, const int64_t* seg_offsets, int n_videos,
                      double* score, void* stream);

/* ------------------------------------------------------------------------ *
 * M1-M5: Memory  model/Memory.py:62-261
 * ------------------------------------------------------------------------ */
/* F.normalize(query, dim=1) + permute(0,2,3,1)  Memory.py:148-149
 * query [B,d,HW] -> q [B*HW, d] */
size_t vadc_memory_prepare_query_workspace_bytes(int B, int64_t HW);
int vadc_memory_prepare_query(const float* query, int B, int d, int64_t HW, float* q,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Backward of Memory.forward with respect to `query` (autograd of Memory.py:145-175; keys are
 * constants there: every use is .detach()ed or un-graded).  What reaches the query: the first d
 * channels of g_updated_query [B,2d,HW] (cat :256; the read softmax is detached :255),
 * g_gather * d MSELoss(q, keys[top1]) (:245), g_spread * d TripletMarginLoss(margin=1,p=2,eps=1e-6)
 * (q, keys[top1], keys[top2]) (:229), all pulled back through F.normalize(query, dim=1) (:148).
 * g_updated_query / g_gather / g_spread / top2 may each be NULL (term absent; g_gather and g_spread
 * are device scalars).  query, g_query [B,d,HW]. */
int vadc_memory_query_bwd(const float* query, const float* keys, const int64_t* top1,
                          const int64_t* top2, const float* g_updated_query,
                          const float* g_gather, const float* g_spread, int B, int d,
                          int64_t HW, int m, float* g_query, void* stream);

/* The same with g_qhat [B,d,HW] (may be NULL): a gradient with respect to the normalised query q-hat (in the query's
 * layout) added to what is pulled back through F.normalize, in the same single pass — the share of the returned score
 * matrices (vadc_memory_scores_bwd). */
int vadc_memory_query_bwd_ex(const float* query, const float* keys, const int64_t* top1,
                             const int64_t* top2, const float* g_updated_query,
                             const float* g_gather, const float* g_spread, const float* g_qhat, int B, int d,
                             int64_t HW, int m, float* g_query, void* stream);

/* get_score  Memory.py:133-143 (+ the top-1 / top-2 of score_memory that
 * gather_loss :241, spread_loss :223 and update :185 take with torch.topk):
 *   logits = q keys^T [N,m]; score_query = softmax over N; score_memory =
 *   softmax over m; colmax[m] = max_n logits; colsum[m] = sum_n exp(logit-colmax);
 *   top1/top2 [N] int64.
 * score_memory_terms (optional, 4*N*m bytes, 16-byte aligned, or NULL): the operand terms of score_memory for the
 * read contraction, written in the softmax pass; hand the same buffer to vadc_memory_read to skip its split pass. */
size_t vadc_memory_score_workspace_bytes(int64_t N, int m, int d);
int vadc_memory_score(const float* q, const float* keys, int64_t N, int m, int d,
                      float* score_query, float* score_memory,
                      float* colmax, float* colsum, int64_t* top1, int64_t* top2,
                      void* score_memory_terms,
                      void* workspace, size_t workspace_bytes, void* stream);

/* read  Memory.py:249-261: updated_query [N,2d] = cat(q, score_memory @ keys); score_memory holds softmax weights
 * (values in [0, 1]: the fp16 x2 operand terms scale them by 2^13) */
size_t vadc_memory_read_workspace_bytes(int64_t N, int m, int d);
int vadc_memory_read(const float* q, const float* score_memory, const void* score_memory_terms,
                     const float* keys,
                     int64_t N, int m, int d, float* updated_query,
                     void* workspace, size_t workspace_bytes, void* stream);

/* gather_loss Memory.py:233-247 (out[0]) and spread_loss :214-231 (out[1],
 * TripletMarginLoss(margin=1,p=2,eps=1e-6)); top2 == NULL skips spread. */
size_t vadc_memory_losses_workspace_bytes(int64_t N, int d);
int vadc_memory_losses(const float* q, const float* keys, const int64_t* top1, const int64_t* top2,
                       int64_t N, int m, int d, float* out,
                       void* workspace, size_t workspace_bytes, void* stream);

/* update + get_update_query  Memory.py:177-204, :94-131:
 *   u_i = sum_{n: top1[n]=i} (score_query[n,i] / max_n score_query[:,i]) q_n
 *   updated_memory = F.normalize(u + keys, dim=1)
 * The python loop over m with nonzero() is replaced by a segmented sum. */
size_t vadc_memory_update_workspace_bytes(int64_t N, int m, int d);
int vadc_memory_update(const float* q, const float* keys, const float* score_query,
                       const int64_t* top1, int64_t N, int m, int d,
                       float* query_update, float* updated_memory,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Global-batch memory under data parallelism (SURVEY 8e): softmax(score, dim=0) (Memory.py:140) and
 * max_n score_query[:, i] (:108) span ALL tokens of the batch.  With the tokens sharded over ranks:
 *   colmax_global = all-reduce MAX of vadc_memory_score's colmax;
 *   contrib = colsum_local * exp(colmax_local - colmax_global)   (vadc_memory_dp_contrib), S = all-reduce SUM;
 *   global score_query = local score_query * contrib / S         (vadc_scale_columns, in place);
 *   this rank's share of the update sums = local query_update * exp(colmax_local - colmax_global)
 *   (vadc_memory_dp_scale_update, in place), all-reduce SUM, then
 *   updated_memory = F.normalize(query_update + keys, dim=1)     (vadc_memory_finish_update; Memory.py:193). */
int vadc_memory_dp_contrib(const float* colmax_local, const float* colsum_local,
                           const float* colmax_global, int m, float* contrib, void* stream);
int vadc_scale_columns(float* x, const float* num, const float* den, int64_t N, int m, void* stream);
int vadc_memory_dp_scale_update(float* query_update, const float* colmax_local,
                                const float* colmax_global, int m, int d, void* stream);
int vadc_memory_finish_update(const float* query_update, const float* keys, int m, int d,
                              float* updated_memory, void* stream);

/* MemoryLoss  Memory.py:52-59: sum |K K^T/2 + 1/2 - I| / (m (m-1)) -> out[0] */
size_t vadc_memory_separateness_workspace_bytes(int m, int d);
int vadc_memory_separateness(const float* keys, int m, int d, float* out,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Backward of read with respect to the memory items (autograd of Memory.py:255, keys learnable):
 *   g_keys [m,d] = score_memory^T G_r,  G_r[b*HW + hw, c] = g_updated_query[b, d + c, hw]
 * score_memory [B*HW, m] as returned by vadc_memory_score; g_updated_query [B,2d,HW] (only channels d..2d-1 are
 * read).  g_keys is overwritten.  Split-K over the tokens on the tcgen05 GEMM, the partials summed in a fixed order
 * (bit-identical across launches); operand terms as in vadc_memory_read (VADC_MEMORY_TERMS=3: bf16 x3).
 * Under a token-sharded global batch the result is this rank's share; the sum over ranks is the full gradient.
 * d >= 8 (VADC_ERR_UNSUPPORTED otherwise). */
size_t vadc_memory_keys_bwd_workspace_bytes(int B, int d, int64_t HW, int m);
int vadc_memory_keys_bwd(const float* score_memory, const float* g_updated_query, int B, int d, int64_t HW,
                         int m, float* g_keys, void* workspace, size_t workspace_bytes, void* stream);

/* Backward through the two score matrices Memory.forward returns (get_score, Memory.py:133-143: s = q-hat K^T,
 * score_query sq = softmax(s, dim=0), score_memory sm = softmax(s, dim=1)), given their gradients Gq, Gm [N,m]:
 *   coldot c_i = sum_n Gq[n,i] sq[n,i]                     (vadc_memory_score_coldot; over ALL tokens of the batch:
 *                                                           under a token-sharded global batch, all-reduce SUM it)
 *   r_n = sum_i Gm[n,i] sm[n,i],  g_s = sq (Gq - 1 c^T) + sm (Gm - r 1^T)
 *   g_qhat [B,d,HW] = g_s K   (overwritten; in the query's layout: hand it to vadc_memory_query_bwd_ex)
 *   g_keys [m,d]   += g_s^T q-hat   (accumulated: added, in a fixed order, to what g_keys holds, e.g. the result of
 *                                    vadc_memory_keys_bwd; bit-identical across launches)
 * The column dots are a two-level reduction in a fixed order (no atomics).  g_s is formed in one pass and written
 * directly as the operand terms of both contractions on the tcgen05 GEMM (g_qhat: one GEMM with rows = tokens;
 * g_keys: split-K over the tokens with the q-hat terms written from query and its norms).  Precision as the module's
 * forward: fp16 x2 with power-of-two scales from the measured bounds of Gq, Gm, c and K (no host sync), or
 * VADC_MEMORY_TERMS=3: bf16 x3.  Either gradient may be NULL (Gq also needs score_query and coldot, Gm needs
 * score_memory), but not both; one of g_qhat / g_keys may be NULL.  query [B,d,HW], keys [m,d] as in the forward.
 * d >= 8 (VADC_ERR_UNSUPPORTED otherwise). */
size_t vadc_memory_score_coldot_workspace_bytes(int64_t N, int m);
int vadc_memory_score_coldot(const float* score_query, const float* g_score_query, int64_t N, int m,
                             float* coldot, void* workspace, size_t workspace_bytes, void* stream);
size_t vadc_memory_scores_bwd_workspace_bytes(int B, int d, int64_t HW, int m);
int vadc_memory_scores_bwd(const float* query, const float* keys, const float* score_query,
                           const float* score_memory, const float* g_score_query, const float* g_score_memory,
                           const float* coldot, int B, int d, int64_t HW, int m, float* g_qhat, float* g_keys,
                           void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the stand-alone methods (get_score :133-143, read :249-261, gather_loss :233-247, spread_loss :214-231),
 * which take the query channel-last, [B,h,w,d] flattened to q [N,d], and do not normalise it.
 *
 * vadc_memory_scores_bwd_rows: the channel-last twin of vadc_memory_scores_bwd, with s = q K^T for q as passed:
 *   g_q_rows [N,d] = g_s K      (overwritten; one GEMM with rows = channels, stored one 128-byte line of a row per warp)
 *   g_keys [m,d]  += g_s^T q    (accumulated in a fixed order, bit-identical across launches; split-K over the tokens,
 *                                the operand terms of q written in one transposing pass)
 * coldot from vadc_memory_score_coldot.  Precision as vadc_memory_scores_bwd, except that in fp16 x2 q is scaled by the
 * power of two of its measured bound (no host sync).  Either gradient may be NULL (Gq also needs score_query and
 * coldot, Gm needs score_memory), but not both; one of g_q_rows / g_keys may be NULL.  d >= 8 (VADC_ERR_UNSUPPORTED
 * otherwise). */
size_t vadc_memory_scores_bwd_rows_workspace_bytes(int64_t N, int d, int m);
int vadc_memory_scores_bwd_rows(const float* q, const float* keys, const float* score_query,
                                const float* score_memory, const float* g_score_query, const float* g_score_memory,
                                const float* coldot, int64_t N, int d, int m, float* g_q_rows, float* g_keys,
                                void* workspace, size_t workspace_bytes, void* stream);

/* vadc_memory_rows_bwd: the query gradient of read / gather_loss / spread_loss, channel-last and without the
 * normalisation (the counterpart of vadc_memory_query_bwd_ex), one per-token pass:
 *   g_query[n,c] = g_updated_query[b,c,hw] + g_q_rows[n,c] + g_gather 2 (q - keys[top1]) / (N d)
 *                + g_spread / N (TripletMarginLoss(margin=1,p=2,eps=1e-6) gradient of (q, keys[top1], keys[top2]))
 * with n = b HW + hw.  q, g_q_rows, g_query [N,d]; g_updated_query [B,2d,HW] (only channels 0..d-1 are read).  Each
 * term may be NULL, but not all of them; g_gather and g_spread are device scalars; the gather term needs top1, the
 * spread term top1 and top2.  g_q_rows may be g_query (updated in place).  No workspace. */
int vadc_memory_rows_bwd(const float* q, const float* keys, const int64_t* top1, const int64_t* top2,
                         const float* g_updated_query, const float* g_gather, const float* g_spread,
                         const float* g_q_rows, int B, int d, int64_t HW, int m, float* g_query, void* stream);

/* vadc_memory_prepare_query_bwd: backward of vadc_memory_prepare_query (F.normalize(query, dim=1) + permute, :148-149):
 *   g_x[b,:,hw] = (g - q-hat (q-hat . g)) / max(|x|, 1e-12),  q-hat = x / max(|x|, 1e-12),  x = query[b,:,hw]
 * (q-hat . g taken as 0 where |x| < 1e-12: the clamp is a constant).  g [B,HW,d] channel-last, query and g_x [B,d,HW];
 * one pass.  No workspace. */
int vadc_memory_prepare_query_bwd(const float* g, const float* query, int B, int d, int64_t HW, float* g_x,
                                  void* stream);

/* Backward of MemoryLoss  Memory.py:52-59 with respect to keys [m,d]; g_out is a device scalar:
 *   S = K K^T/2 + 1/2 - I (recomputed as vadc_memory_separateness does), G = sgn(S) with sgn(0) = 0,
 *   g_keys = g_out / (m (m-1)) * (G + G^T)/2 K   (G is symmetric bit for bit).  g_keys is overwritten. */
size_t vadc_memory_separateness_bwd_workspace_bytes(int m, int d);
int vadc_memory_separateness_bwd(const float* keys, const float* g_out, int m, int d, float* g_keys,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * Debug / self-test: one CTA runs out[128,N] = A * B on tcgen05 (TMEM
 * accumulator, SWIZZLE_128B shared-memory operands).  mode bit0: B is [Kd,N]
 * (MN-major) instead of [N,Kd]; bit1: bf16 inputs (kind::f16) instead of tf32;
 * bit2: A is [Kd,128] (MN-major) instead of [128,Kd].  Used by the tests to
 * pin the descriptor encodings the fused kernels rely on.
 * ------------------------------------------------------------------------ */
int vadc_debug_umma(const float* A, const float* B, float* out, int N, int Kd, int mode, void* stream);
/* self-test of the TMA-fed tcgen05 GEMM (three-term bf16 split, six products): out [M,N] = A [M,Kd] . B^T with
 * B [N,Kd] (b_mn = 0) or B [Kd,N] (b_mn = 1). */
size_t vadc_debug_tc_gemm_workspace_bytes(int64_t M, int64_t N, int64_t Kd);
int vadc_debug_tc_gemm(const float* A, const float* B, int64_t M, int64_t N, int64_t Kd, int b_mn,
                       float* out, void* workspace, size_t workspace_bytes, void* stream);
/* issue-rate micro-benchmark of one tcgen05.mma shape (bf16, shared-memory operands): `reps` x 8
 * instructions back to back; out[0] = cycles until the commit arrives, out[1] = cycles to issue. */
int vadc_debug_umma_bench(int M, int N, int a_mn, int b_mn, int reps, long long* out, void* stream);

/* ------------------------------------------------------------------------ *
 * §8f-2: the consumer of x_rec — LayerNorm(C) (model/backbone.py:120) + the decoder's entry timedebd =
 * ConvTranspose3d(C, C, kernel (2,1,1), stride (2,1,1)) (model/swin_decoder_predict.py:593-594, :599-602) on the
 * channel-last tokens: ONE GEMM [N, C] x [C, 2C] whose epilogue scatters the column halves to output frames 2d, 2d+1.
 * x [N, C] (N = frames * HW tokens, frame-major), out [2N, C] channel-last.
 * wt [2C, C]: wt[j*C + co, ci] = W[ci, co, j] (forward operand);  wk [C, 2C]: wk[ci, j*C + co] = W[ci, co, j] (backward);
 * gwk is d/d wk in wk's arrangement.  mu, rstd [N] are saved for the backward.
 * ------------------------------------------------------------------------ */
size_t vadc_norm_timedebd_workspace_bytes(int64_t N, int C);
int vadc_norm_timedebd_fwd(const float* x, const float* ln_w, const float* ln_b, const float* wt, const float* bias,
                           int64_t N, int C, int64_t HW, float eps, float* out, float* mu, float* rstd,
                           void* workspace, size_t workspace_bytes, void* stream);
int vadc_norm_timedebd_bwd(const float* x, const float* mu, const float* rstd, const float* ln_w, const float* ln_b,
                           const float* wk, const float* gout, int64_t N, int C, int64_t HW, float eps,
                           float* gx, float* g_ln_w, float* g_ln_b, float* gwk, float* gbias,
                           void* workspace, size_t workspace_bytes, void* stream);

/* predict mode (model/swin_decoder_predict.py:591-592): timedebd = Conv3d(C, C, kernel (2,1,1), stride (2,1,1)).
 * x [N,C] channel-last tokens of an EVEN number of frames (HW tokens each); wk [C, 2C], wk[co, j*C + ci] =
 * weight[co, ci, j]; out [N/2, C] channel-last (frame pairs merged).  Backward: gout [N/2, C] -> gx [N,C], g_ln_w/b [C],
 * gwk [C, 2C] (same arrangement as wk), gbias [C].  Workspace: vadc_norm_timedebd_workspace_bytes(N, C). */
int vadc_norm_timeconv_fwd(const float* x, const float* ln_w, const float* ln_b, const float* wk, const float* bias,
                           int64_t N, int C, int64_t HW, float eps, float* out, float* mu, float* rstd,
                           void* workspace, size_t workspace_bytes, void* stream);
int vadc_norm_timeconv_bwd(const float* x, const float* mu, const float* rstd, const float* ln_w, const float* ln_b,
                           const float* wk, const float* gout, int64_t N, int C, int64_t HW, float eps,
                           float* gx, float* g_ln_w, float* g_ln_b, float* gwk, float* gbias,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * SURVEY 8f-3: the encoder's downsample stage as a producer of channel-last tokens
 *   nn.Sequential(Conv3d(Cin, Cout, kernel (1,2,2), stride (1,2,2)), GELU)   model/swin_transformer.py:575-585
 *   followed by 'n c d h w -> n d h w c'                                      swin_transformer.py:745, model/backbone.py:82
 * x [B,Cin,D,2H,2W] contiguous (channel-first); weight [Cout, Cin*4] = Conv3d.weight.reshape(Cout, -1); bias [Cout].
 * out [B,D,H,W,Cout] channel-last = gelu(conv(x)) (exact erf GELU); pre (same shape, or NULL for inference) keeps the
 * pre-activation the backward needs.  Backward: gout [B,D,H,W,Cout] -> gx [B,Cin,D,2H,2W], gweight [Cout,Cin*4], gbias.
 * vadc_downsample_gelu_supported: 1 when the shape runs here (Cin even, Cout % 8 == 0, TMA row pitches); the entry
 * points return VADC_ERR_UNSUPPORTED otherwise.
 * ------------------------------------------------------------------------ */
int vadc_downsample_gelu_supported(int B, int Cin, int D, int H, int W, int Cout);
size_t vadc_downsample_gelu_workspace_bytes(int B, int Cin, int D, int H, int W, int Cout);
int vadc_downsample_gelu_fwd(const float* x, const float* weight, const float* bias,
                             int B, int Cin, int D, int H, int W, int Cout,
                             float* out, float* pre,
                             void* workspace, size_t workspace_bytes, void* stream);
int vadc_downsample_gelu_bwd(const float* x, const float* weight, const float* pre, const float* gout,
                             int B, int Cin, int D, int H, int W, int Cout,
                             float* gx, float* gweight, float* gbias,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * §8e: one-shot all-reduce(sum) of small fp32 messages over NVLink peer memory — replaces the two latency-bound
 * collectives per training step that utils/distritributed_model.py's gloo DDP (main_predict.py:171) implies for this
 * path: the scalar sum (D*A)^2 (backbone.py:98, full-batch norm) and [g cluster_center | g gamma | g beta].
 * peer_blocks_dev: DEVICE array of `world` pointers, one symmetric block per rank: 256 zero-initialised uint32 flag words
 * followed by 2 * capacity floats, allocated and exchanged once by the host (torch.distributed._symmetric_memory).
 * Up to four tensors are reduced IN PLACE in one launch; the sum runs in rank order on every rank (bit-identical
 * results).  Every rank must call with the same sizes in the same order.
 * ------------------------------------------------------------------------ */
int vadc_oneshot_allreduce(const void* peer_blocks_dev, int rank, int world,
                           int64_t capacity, float* t0, int64_t n0, float* t1, int64_t n1, float* t2, int64_t n2,
                           float* t3, int64_t n3, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VADC_H_ */
