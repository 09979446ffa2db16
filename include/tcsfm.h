/* tcsfm.h -- C ABI of the fused sm_100a inverse-warp + SSIM/L1 photometric-loss path.
 *
 * The reference (utiasSTARS/tightly-coupled-SfM) is pure Python/PyTorch and has no
 * FFI of its own; its "operator API" for this path is a handful of Python callables.
 * Each entry point below names the reference callable (file:line, relative to the
 * reference root) whose arithmetic it replaces.  The Python drop-ins in
 * tightly-coupled-sfm_b200/{stn,losses,train_mono,pft}.py bind these symbols with
 * ctypes and keep the reference's call signatures (see INTEGRATION.md).
 *
 * Conventions
 *  - plain C: device pointers + sizes, no C++/torch types.  All tensors are fp32.
 *  - images are [B,C,H,W] views with unit W stride and H stride == W; batch and
 *    channel strides (in elements) are passed explicitly so that channel slices of
 *    a 6-channel stack (train_mono.py:69 passes imgs[:,3:6]) need no copy.
 *    depth / mask / per-pixel outputs are contiguous [B,1,H,W].
 *  - kinv is K^-1 as [B,9] row-major, proj is K @ [R|t] as [B,12] row-major
 *    (models/stn.py:257,262); they are produced by the caller so that their bits
 *    are the reference's.
 *  - every launch goes to `stream` (a cudaStream_t passed as void*); no host
 *    synchronisation, no allocation, no global state besides the last-error string.
 *    Buffers documented as "accumulated" are zeroed by the library on `stream`.
 *  - return value: 0 on success, non-zero on error (message via tcsfm_last_error()).
 */
#ifndef TCSFM_H_
#define TCSFM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCSFM_ABI_VERSION 21

/* ---- flags ------------------------------------------------------------------ */
/* Arithmetic flavour.  Eager PyTorch rounds after every operator, but a few ATen
 * operators differ between devices (SURVEY.md App. B): CUDA divides by a Python
 * scalar by multiplying with its fp32 reciprocal and takes mean(dim) as
 * sum * (1/n); the CPU kernels divide.  Flavour 0 reproduces the CUDA operators
 * (the reference's production path), flavour 1 the CPU ones (used to compare
 * bit-for-bit against CPU-generated golden vectors). */
#define TCSFM_ARITH_CPU        (1 << 0)
/* eager PyTorch's projection bmm `rot @ cam` (models/stn.py:210) runs a different cuBLAS kernel for
 * batch 1 while m*n*k = 9*H*W <= 2^21: (a0*b0 + a1*b1) + a2*b2 with every product and sum rounded,
 * instead of the k-ascending FMA chain.  (`K^-1 @ grid`, stn.py:47, keeps the FMA chain because
 * torch.inverse returns K^-1 column-major; profiles/r01_probe_bmm*.json, r01_probe_b1_calls.json.)
 * Set by the Python layer when the reference would have issued such a call. */
#define TCSFM_ARITH_BMM_NOFMA  (1 << 6)
/* "fast" arithmetic of the fused pair loss: geometry, bilinear sample, validity mask, the L1 term and the auto-mask
 * comparison of losses.py:158 keep the exact roundings selected above; the 3x3 SSIM statistics, the SSIM ratio and the
 * depth-inconsistency ratio are evaluated with separable sums, fused multiply-adds and approximate reciprocals
 * (tolerance level: loss 1e-5, gradients 1e-4 of the reference; BASELINE.json north_star).  The workspace then has the
 * layout / size tcsfm_pair_ws_floats() reports. */
#define TCSFM_ARITH_FAST       (1 << 7)
/* pair-loss configuration (losses.py:65-73,151-183 config keys) */
#define TCSFM_AUTO_MASK        (1 << 1)   /* with_auto_mask   */
#define TCSFM_SSIM             (1 << 2)   /* l_ssim           */
#define TCSFM_DEPTH_MASK       (1 << 3)   /* with_depth_mask  */
#define TCSFM_DEPTH_CONSIST    (1 << 4)   /* l_depth_consist  */
/* backward only: several groups write into the same gradient buffers (e.g. the target
 * depth is `tgt_depth` of the forward pairs and `ref_depth` of the inverse pairs).  All
 * depth-gradient writes become atomic adds and the CALLER zeroes g_tgt_depth / g_ref_depth. */
#define TCSFM_SHARED_GRADS     (1 << 5)

const char* tcsfm_last_error(void);
int tcsfm_abi_version(void);

/* ---- inverse_warp2 (models/stn.py:234-273; pixel2cam :33-48, cam2pixel2 :198-231,
 *      F.grid_sample bilinear/zeros/align_corners=False :266,271) ------------------
 * out_img [B,3,H,W], out_valid / out_proj_depth / out_comp_depth [B,1,H,W]
 * (any output pointer may be NULL to skip it). */
int tcsfm_warp_fwd(const float* img, int64_t img_sb, int64_t img_sc,
                   const float* depth, const float* ref_depth,
                   const float* kinv, const float* proj,
                   float* out_img, float* out_valid, float* out_proj_depth, float* out_comp_depth,
                   const float* tgt, int64_t tgt_sb, int64_t tgt_sc, float* out_stack,
                   int B, int H, int W, int flags, void* stream);
/* Optional fused glue of solve_pose_iteratively (train_mono.py:74-76,102-104): when `out_stack`
 * [B,6,H,W] is given, the kernel also writes the next pose-network input
 * [ tgt * valid_mask | projected_img ] (tgt is the [B,3,H,W] view of the reconstruction target). */

/* Backward of the above (the autograd replay of stn.py:257-271).  g_out_* are the
 * upstream gradients (NULL = zero).  g_depth is overwritten; g_ref_depth [B,1,H,W],
 * g_proj [B,12] and the optional g_img [B,3,H,W] (contiguous) are accumulated
 * (scatter / reduction).  NULL output pointers are skipped. */
int tcsfm_warp_bwd(const float* img, int64_t img_sb, int64_t img_sc,
                   const float* depth, const float* ref_depth,
                   const float* kinv, const float* proj,
                   const float* g_out_img, const float* g_out_proj_depth, const float* g_out_comp_depth,
                   const float* g_out_stack,
                   float* g_depth, float* g_ref_depth, float* g_proj, float* g_img,
                   int B, int H, int W, int flags, void* stream);
/* g_out_stack [B,6,H,W] (NULL = none): upstream gradient of `out_stack`; its channels 3:6 add to
 * g_out_img. */

/* ---- SSIM_Loss.forward (losses.py:27-41) and its backward ---------------------
 * x, y, out, g_out, g_x, g_y are contiguous [N,H,W] planes (N = B*C).
 * g_x / g_y may be NULL. */
int tcsfm_ssim_fwd(const float* x, const float* y, float* out,
                   int N, int H, int W, int flags, void* stream);
int tcsfm_ssim_bwd(const float* x, const float* y, const float* g_out, float* g_x, float* g_y,
                   int N, int H, int W, int flags, void* stream);
/* SSIM_Loss(x, y).mean() as one launch each way (the depth-initialisation term of the PFT loss,
 * optimization_experiments/optimizer.py:89-90): out_mean[1] is zeroed and accumulated; g_mean[1] is the
 * device scalar upstream of the mean. */
int tcsfm_ssim_mean_fwd(const float* x, const float* y, float* out_mean, int N, int H, int W, int flags, void* stream);
int tcsfm_ssim_mean_bwd(const float* x, const float* y, const float* g_mean, float* g_x, float* g_y,
                        int N, int H, int W, int flags, void* stream);

/* ---- Compute_Loss.compute_pairwise_loss (losses.py:151-183) fused with
 *      mean_on_mask's sums (losses.py:142-149) --------------------------------------
 * One launch evaluates n_groups independent pair groups (e.g. the 2*S
 * direction/source combinations of Compute_Loss.forward, losses.py:99-127), each a
 * batch of B pairs at HxW.  Host array of descriptors; all pointers inside are
 * device pointers. */
typedef struct tcsfm_pair_group {
    const float* tgt_img;   int64_t tgt_sb, tgt_sc;   /* reconstruction target [B,3,H,W]  */
    const float* ref_img;   int64_t ref_sb, ref_sc;   /* image that is sampled [B,3,H,W]  */
    const float* tgt_depth;                           /* depth of the target   [B,1,H,W]  */
    const float* ref_depth;                           /* depth that is sampled [B,1,H,W]  */
    const float* kinv;                                /* [B,9]   */
    const float* proj;                                /* [B,12]  */
    /* forward outputs */
    float* diff_img;        /* [B,1,H,W] per-pixel photometric error (losses.py:167,174); may be NULL */
    float* mask;            /* [B,1,H,W] final valid_mask (auto*valid or valid, :158-162); required by bwd */
    float* sums;            /* [4] accumulated: sum(diff*mask), sum(mask), sum(diff_depth*mask), 0 */
    float* coef;            /* [B,P,H,W] workspace, P = tcsfm_pair_coef_planes(): SSIM adjoint coefficients saved
                               by the forward for the backward; NULL = inference only (no backward) */
    /* backward inputs */
    const float* g_diff;    /* upstream grad of diff_img [B,1,H,W], may be NULL */
    const float* g_scalars; /* device [2]: upstream grads of l_reprojection and l_depth, may be NULL */
    /* per-pixel min over competing groups (losses.py:129-132): this group's diff_img is entry
     * `min_index` of `min_count` maps spaced `min_stride` floats apart from `min_base`; the
     * upstream gradient *g_min goes to the arg-min map (lowest index on ties).  NULL = unused. */
    const float* min_base;  int64_t min_stride;  int32_t min_count, min_index;
    const float* g_min;
    /* backward outputs */
    float* g_tgt_depth;     /* [B,1,H,W] overwritten */
    float* g_ref_depth;     /* [B,1,H,W] accumulated; may be NULL when no depth term is active */
    float* g_proj;          /* [B,12] accumulated */
} tcsfm_pair_group;

int tcsfm_pair_coef_planes(void);
/* floats of workspace per pair (one batch element of one group) for the arithmetic selected in `flags`:
 * coef of a group is [B, tcsfm_pair_ws_floats(H, W, flags)], 16-byte aligned. */
int64_t tcsfm_pair_ws_floats(int H, int W, int flags);
int tcsfm_pair_loss_fwd(const tcsfm_pair_group* groups, int n_groups,
                        int B, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
int tcsfm_pair_loss_bwd(const tcsfm_pair_group* groups, int n_groups,
                        int B, int H, int W, float w_l1, float w_ssim, int flags, void* stream);

/* ---- the `return_errors` photometric block of solve_pose_iteratively (train_mono.py:84-92),
 *      also compute_photometric_error (optimization_experiments/helpers.py:12-18) ----------
 * For N stacked pairs: tgt / src are [N,3,H,W] views (channel slices of the 6-channel stack),
 * rec [N,3,H,W], proj_depth / comp_depth [N,1,H,W] contiguous (the outputs of inverse_warp2).
 *   auto_err  = mean_c(w_l1 * clamp|tgt - src| + w_ssim * SSIM(tgt, src))
 *   diff      = mean_c(w_l1 * clamp|rec - tgt| + w_ssim * SSIM(tgt, rec))
 *   auto_mask = diff < auto_err            weight = 1 - clamp(|cd - pd| / (cd + pd), 0, 1)
 * coef [N,P,H,W], P = tcsfm_photo_coef_planes(), is the workspace the backward needs (NULL for
 * inference).  The backward returns the gradients w.r.t. rec and the two depths. */
int tcsfm_photo_coef_planes(void);
int tcsfm_photo_fwd(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb, int64_t src_sc,
                    const float* rec, const float* proj_depth, const float* comp_depth,
                    float* auto_err, float* diff, float* auto_mask, float* weight, float* coef,
                    const float* valid,
                    int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
/* `valid` [N,1,H,W] (may be NULL): inverse_warp2's valid_mask; when given auto_mask comes out already
 * multiplied by it (helpers.py:18 returns auto_mask * valid_mask). */
int tcsfm_photo_bwd(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* rec,
                    const float* proj_depth, const float* comp_depth, const float* coef,
                    const float* g_diff, const float* g_weight, float* g_rec, float* g_pd, float* g_cd,
                    int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);

/* ---- compute_photometric_error (optimization_experiments/helpers.py:8-23) for N pose hypotheses of ONE frame
 *      pair, reduced to the loss-surface value of plot_loss_surface.py:11-87 -----------------------------------
 * tgt / src are [1,3,H,W] views (channel strides given; the *_pairs forms below take B pairs with batch strides),
 * tgt_depth / src_depth [1,1,H,W] contiguous, kinv [9], proj [N,12] (hypothesis n's K @ [R|t], as
 * tcsfm_pose_proj_fwd forms it).  For each
 * n, with the warp of tcsfm_warp_fwd under proj[n] and the maps of tcsfm_photo_fwd (valid folded into the mask):
 *   sums[n] = ( sum((diff * mask) * weight), sum(mask) )
 * The per-pixel products carry the eager expression's roundings; the sums are added in a fixed order (the same
 * inputs give the same bits on every call).  The optional maps rec [N,3,H,W] and diff / mask / weight [N,1,H,W]
 * (NULL = not written) are those of a batch-1 compute_photometric_error call with the same `flags`.
 * scratch [H,W] and partials [tcsfm_photo_sweep_partial_floats(N, H, W)]: workspace, overwritten.
 * Three launches on `stream`. */
int64_t tcsfm_photo_sweep_partial_floats(int N, int H, int W);
int tcsfm_photo_sweep(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                      const float* tgt_depth, const float* src_depth, const float* kinv, const float* proj,
                      float* scratch, float* partials, float* sums,
                      float* rec, float* diff, float* mask, float* weight,
                      int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
/* The same sums, and the pose gradient of every hypothesis's loss_n = sums[n][0] / sums[n][1]:
 *   g_proj[n] = d loss_n / d proj[n]   [N,12], already divided by sums[n][1] (NaN where it is 0)
 * The mask (a comparison and the valid mask) and sums[n][1] carry no gradient; the gradient flows through diff (the
 * warped image, over each pixel's 3x3 SSIM window with reflection padding) and through weight (the computed depth and
 * the sampled source depth).  sums[n] has the bits tcsfm_photo_sweep gives.  partials
 * [tcsfm_photo_sweep_grad_partial_floats(N, H, W)]: workspace, overwritten.  Three launches on `stream`; the forward
 * is recomputed inside each CTA, so no workspace grows with N * H * W. */
int64_t tcsfm_photo_sweep_grad_partial_floats(int N, int H, int W);
int tcsfm_photo_sweep_grad(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                           const float* tgt_depth, const float* src_depth, const float* kinv, const float* proj,
                           float* scratch, float* partials, float* sums, float* g_proj,
                           int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
/* Multi-start refinement: `steps` Adam updates of each of the N poses [N,6] (in place, un-negated like the `pose` of
 * compute_photometric_error) on its loss_n = sums[n][0] / sums[n][1] above.  K [9] is the intrinsics; K[R|t] of every
 * pose is formed as tcsfm_pose_proj_fwd(poses, -1, K, 1, proj, N, pose_flags) forms it.  For t = 1 .. steps, with
 *   c1 = lr / (1 - beta1^t),  c2 = sqrt(1 - beta2^t)
 * and b1 = beta1, a1 = 1 - beta1, b2 = beta2, a2 = 1 - beta2, e = eps, each computed in double and rounded to fp32 once,
 * and g the pose gradient of tcsfm_photo_sweep_grad + tcsfm_pose_proj_bwd (sign -1), every column updates as
 *   m = b1*m + a1*g;  v = b2*v + a2*(g*g);  p = p - c1*(m / (sqrt(v)/c2 + e))
 * with every operation rounded to fp32 (m = v = 0 at t = 1).  A pose whose sums[n][1] is 0 is not updated.
 *   loss [(steps+1)*N]: row k = loss_n at the poses after k updates (NaN where no pixel is valid);
 *   best_loss [N], best_step [N], best_pose [N,6]: the smallest finite loss of row n's history, the first k that
 *   reaches it and the pose there (NaN, -1 and the starting pose when there is none).
 * Workspace, overwritten: m, v [N,6], proj [N,12], scratch [H,W], partials [tcsfm_photo_sweep_grad_partial_floats(N, H,
 * W)].  2*steps + 4 launches on `stream`; no allocation, no synchronisation, the same bits on every call. */
int tcsfm_photo_refine(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                       const float* tgt_depth, const float* src_depth, const float* kinv, const float* K,
                       float* poses, float* m, float* v, float* proj, float* scratch, float* partials,
                       float* loss, float* best_loss, int* best_step, float* best_pose,
                       int N, int H, int W, int steps, double lr, double beta1, double beta2, double eps,
                       float w_l1, float w_ssim, int flags, int pose_flags, void* stream);

/* The three calls above for B frame pairs of N hypotheses each, in one call with the same launch count whatever B is.
 * tgt / src are [B,3,H,W] views: pair b's channel c starts b * *_sb + c * *_sc floats after the pointer (any
 * *_sb >= 0, so channel slices of a [B,6,H,W] stack need no copy); tgt_depth / src_depth [B,1,H,W] contiguous,
 * kinv [B,9] and K [B,9] (refine); scratch [B,H,W].  Hypotheses are pair-major: row h = b * N + n of proj, sums,
 * g_proj, the maps, poses, m, v, best_loss, best_step and best_pose is start n of pair b, and the loss history is
 * [(steps+1)*B*N].  Every row holds the bits the single-pair call on pair b with those N rows gives.  partials:
 * tcsfm_photo_sweep_partial_floats / tcsfm_photo_sweep_grad_partial_floats of B * N. */
int tcsfm_photo_sweep_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb,
                            int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                            const float* proj, float* scratch, float* partials, float* sums,
                            float* rec, float* diff, float* mask, float* weight,
                            int B, int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
int tcsfm_photo_sweep_grad_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb,
                                 int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                                 const float* proj, float* scratch, float* partials, float* sums, float* g_proj,
                                 int B, int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream);
int tcsfm_photo_refine_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb,
                             int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                             const float* K, float* poses, float* m, float* v, float* proj, float* scratch,
                             float* partials, float* loss, float* best_loss, int* best_step, float* best_pose,
                             int B, int N, int H, int W, int steps, double lr, double beta1, double beta2, double eps,
                             float w_l1, float w_ssim, int flags, int pose_flags, void* stream);

/* ---- DepthOptimizer.compute_optimization_loss (optimization_experiments/optimizer.py:45-86): the
 *      reduction of the error maps of solve_pose_iteratively(return_errors=True) to the PFT loss --------
 * The maps are the two halves of the stacked [2*S*B,1,H,W] outputs (train_mono.py:94-100): forward half
 * (target <- source j: rows j*B .. j*B+B-1) f_diff, f_valid, f_aerr (auto_mask_error), f_weight; inverse half
 * i_diff, i_valid, i_auto (auto_mask), i_weight; n = H*W.
 *   TCSFM_PFT_ARGMIN       options['diff_img_argmin']: per-pixel min over the S sources (first index on ties),
 *                          valid = clamp(sum_j valid_j, 0, 1) [* (min diff < min auto_err) with AUTOMASK],
 *                          sum(diff_min * valid * f_weight[0:B]) / sum(valid)          (optimizer.py:49-69);
 *                          without it 0.25 * sum(f_diff * f_valid * f_weight) / sum(f_valid)       (:71-73)
 *   TCSFM_PFT_AUTOMASK     options['automasking']
 *   TCSFM_PFT_INVERSE      options['l_inverse_reconstruction']: + 0.25 * sum(i_diff * i_valid * i_weight [* i_auto])
 *                          / sum(i_valid [* i_auto])                                                (:75-81)
 *   TCSFM_PFT_DEPTH_CONSIST options['l_depth_consist']: + w_depth * mean(1 - f_weight) [+ w_depth * mean(1 - i_weight)]
 * sums [8] workspace (zeroed by the forward, read by the backward); loss [1].  The backward writes the
 * gradients w.r.t. diff_img and weight_mask of both halves (every element, no accumulation); the masks and
 * auto_mask_error are comparisons and carry none. */
#define TCSFM_PFT_ARGMIN         (1 << 0)
#define TCSFM_PFT_AUTOMASK       (1 << 1)
#define TCSFM_PFT_INVERSE        (1 << 2)
#define TCSFM_PFT_DEPTH_CONSIST  (1 << 3)
int tcsfm_pft_reduce_fwd(const float* f_diff, const float* f_valid, const float* f_aerr, const float* f_weight,
                         const float* i_diff, const float* i_valid, const float* i_auto, const float* i_weight,
                         int B, int S, int64_t n, int flags, float w_depth, float* sums, float* loss, void* stream);
int tcsfm_pft_reduce_bwd(const float* f_diff, const float* f_valid, const float* f_aerr, const float* f_weight,
                         const float* i_diff, const float* i_valid, const float* i_auto, const float* i_weight,
                         int B, int S, int64_t n, int flags, float w_depth, const float* sums, const float* g_loss,
                         float* g_f_diff, float* g_f_weight, float* g_i_diff, float* g_i_weight, void* stream);

/* ---- get_smooth_loss (losses.py:43-61): edge-aware smoothness of the mean-normalised disparity --
 * disp [B,1,H,W] contiguous, img [B,3,H,W] view; workspace: 2*B+2 floats kept between forward and
 * backward; out / g_out: device scalars; g_disp [B,1,H,W]. */
int tcsfm_smooth_fwd(const float* disp, const float* img, int64_t img_sb, int64_t img_sc,
                     float* workspace, float* out, int B, int H, int W, void* stream);
int tcsfm_smooth_bwd(const float* disp, const float* img, int64_t img_sb, int64_t img_sc,
                     float* workspace, const float* g_out, float* g_disp, int B, int H, int W, void* stream);

/* ---- data format at the host boundary: the reference's loader turns uint8 frames into float tensors on the host
 *      (utils/custom_transforms.py:74: torch.from_numpy(im).float() / 255) and ships fp32 to the GPU.  dst[i] =
 *      float(src[i]) / 255 with the same IEEE division, so frames can cross the host link as bytes. */
int tcsfm_u8_to_float(const unsigned char* src, float* dst, int64_t n, void* stream);

/* K^-1 of B row-major 3x3 fp32 matrices -> row-major [B,9], with the bits of `intrinsics.inverse()` on CUDA
 * (models/stn.py:257: cuBLAS batched LU + triangular solves, ten launches) in one launch; the arithmetic ordering was
 * matched bit for bit on probed inverses (tools/probe_kinv.py, tools/match_kinv.py). */
int tcsfm_intrinsics_inverse(const float* K, float* kinv, int B, void* stream);

/* The glue on either side of the pair kernels of one frame (Compute_Loss.forward, losses.py:86-122) as one launch each:
 * prologue = tcsfm_disp_to_depth_fwd of `count` (<= 4) maps of n elements + tcsfm_pose_proj_fwd of n_groups (<= 8) pose
 * tensors [B, >= 6] read in place through a pointer table (row stride `pose_stride` floats; proj [n_groups*B,3,4]);
 * with `kinv` != NULL the prologue also writes K^-1 [B,9] (tcsfm_intrinsics_inverse);
 * epilogue = the two chain rules (g_pose [n_groups*B,6]). */
int tcsfm_frame_prologue(const float* const* disp, float* const* depth, int count, int64_t n, float min_disp, float range,
                         const float* const* pose, int n_groups, int pose_stride, float sign, const float* K, int B,
                         float* proj, float* kinv, int flags, void* stream);
int tcsfm_frame_epilogue(const float* const* g_depth, const float* const* depth, float* const* g_disp, int count, int64_t n,
                         float range, const float* const* pose, int n_groups, int pose_stride, float sign,
                         const float* K, int B, const float* g_proj, float* g_pose, void* stream);

/* ---- glue of Compute_Loss.forward (losses.py:75-140) ----------------------------
 * pose [N,6] (times `sign`; every call site passes -pose) -> K @ [Rx Ry Rz | t] as [N,12]
 * (models/stn.py:81-116,143-158,262); row i uses K[i % Bk].  Bit-identical to the eager
 * CUDA operators: the k-ascending FMA chain of the batched SGEMM when the reference's calls
 * have batch >= 2, the non-fused batch-1 kernel with TCSFM_ARITH_BMM_NOFMA in `flags`.  The
 * backward maps grad(K[R|t]) to the 6-DoF pose gradient. */
int tcsfm_pose_proj_fwd(const float* pose, float sign, const float* K, int Bk, float* proj, int N, int flags,
                        void* stream);
int tcsfm_pose_proj_bwd(const float* pose, float sign, const float* K, int Bk, const float* g_proj,
                        float* g_pose, int N, void* stream);

/* disp_to_depth (utils/learning_helpers.py:77-86) for `count` <= 4 maps of n floats in one launch:
 * depth = 1 / (min_disp + range * disp), range = max_disp - min_disp; pointer tables are HOST
 * arrays of device pointers.  Backward: g_disp = -g_depth * depth^2 * range. */
int tcsfm_disp_to_depth_fwd(const float* const* disp, float* const* depth, int count, int64_t n,
                            float min_disp, float range, void* stream);
int tcsfm_disp_to_depth_bwd(const float* const* g_depth, const float* const* depth, float* const* g_disp, int count,
                            int64_t n, float range, void* stream);

/* The same with the nearest-neighbour upsample of a lower pyramid scale folded in
 * (F.interpolate(disp, (H, W), mode='nearest') then disp_to_depth, losses.py:86-88,102-104): disp
 * [B,1,h,w] -> depth [B,1,H,W] with ATen's index rule; the backward sums the gradients of the
 * full-resolution pixels that read each low-resolution one: g_disp [B,1,h,w]. */
int tcsfm_disp_upsample_to_depth_fwd(const float* const* disp, float* const* depth, int count, int B, int h, int w,
                                     int H, int W, float min_disp, float range, void* stream);
int tcsfm_disp_upsample_to_depth_bwd(const float* const* g_depth, const float* const* depth, float* const* g_disp,
                                     int count, int B, int h, int w, int H, int W, float range, void* stream);

typedef struct tcsfm_frame_cfg {
    int32_t n_groups;       /* pair groups of the launch, in the reference's evaluation order      */
    int32_t role[8];        /* 0 = inverse reconstruction (scalar, x w_inverse), 1 = forward (min)  */
    float   w_inverse;      /* 0.3, losses.py:116                                                   */
    float   w_depth;        /* l_depth_consist_weight if l_depth_consist else 0, losses.py:114,121  */
    int64_t n_min_pixels;   /* B*H*W: the mean of losses.py:132                                     */
} tcsfm_frame_cfg;

/* out_sum[0] = sum_i min_j base[j*stride + i], j < count, i < n  (losses.py:129-131).  With `cfg` != NULL the
 * launch also does tcsfm_frame_finalize(sums, out_sum, cfg, out, total): the last block to add its partial sum
 * computes the loss terms; ticket [1]: scratch.  With `cfg` == NULL, ticket, sums, out and total are ignored. */
int tcsfm_min_reduce(const float* base, int64_t stride, int count, int64_t n, float* out_sum, int* ticket,
                     const float* sums, const tcsfm_frame_cfg* cfg, float* out, float* total, void* stream);

/* The same minimum over the diff_img of `groups` (the competing forward groups in candidate order, forward fields
 * filled), with its near-ties re-decided:
 * every block takes the min of its pixels, keeps in shared memory those whose two smallest candidates differ by less
 * than `band` (or involve a NaN) and overwrites their diff_img entries in every group with the value the exact
 * arithmetic gives, so that the arg-min routing of the backward (torch.min, first index on ties) is the reference's
 * even when the maps were produced by TCSFM_ARITH_FAST.  out_sum [1]: sum over the B*H*W pixels of the min over the
 * groups' diff_img (values as the forward produced them); counters [2]: (number of pixels re-evaluated, scratch).
 * With `cfg` != NULL the last block to finish also does tcsfm_frame_finalize(sums, out_sum, cfg, out_terms,
 * out_total).  Replaces torch.min(reconstruction_errors, 1)[0] of losses.py:129-131 under the fast arithmetic. */
int tcsfm_pair_min_resolve(const tcsfm_pair_group* groups, int n_groups, int B, int H, int W,
                           float w_l1, float w_ssim, int flags, float band, float* out_sum, int* counters,
                           const float* sums, const tcsfm_frame_cfg* cfg, float* out_terms, float* out_total,
                           void* stream);


/* out[3] = (l_reconstruct_inverse, l_reconstruct_forward, l_depth) of one scale, from the pair
 * kernels' sums [G,4] and the min-reduce sum (mean_on_mask's 10000-pixel rule on the device).
 * total[1] (may be NULL) = (out[0] + out[1]) + out[2], the order Compute_Loss.forward adds the
 * terms into losses['total'] (losses.py:134-138). */
int tcsfm_frame_finalize(const float* sums, const float* min_sum, const tcsfm_frame_cfg* cfg, float* out, float* total,
                         void* stream);
/* Upstream gradients of the three terms (g_out[3], may be NULL) and of their sum (g_total[1],
 * may be NULL) -> g_scalars [G,2] and g_min [1], the upstream scalars tcsfm_pair_loss_bwd consumes.
 * With `zero` != NULL the launch also zero-fills it (n_zero floats, 16-byte aligned, n_zero % 4 == 0): the
 * accumulated depth-gradient buffer of the shared-gradient backward pair launch.  NULL = no fill. */
int tcsfm_frame_bwd_prepare(const float* g_out, const float* g_total, const tcsfm_frame_cfg* cfg, float* g_scalars,
                            float* g_min, float* zero, int64_t n_zero, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TCSFM_H_ */
