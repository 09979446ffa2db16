"""Drop-ins for the loss half of the reference's per-frame test-time optimisation
(PFT): ``DepthOptimizer.compute_optimization_loss`` (optimization_experiments/
optimizer.py:29-97) and ``compute_photometric_error`` (optimization_experiments/
helpers.py:8-23).  The optimisation driver itself (deep copies of the depth net,
Adam, plotting; optimizer.py:136-297) is the reference's harness and calls these.
``photometric_loss_surface`` evaluates ``compute_photometric_error`` for N pose hypotheses of one pair in one call
(the loss-surface plots, plot_loss_surface.py:11-87); ``photometric_loss_surface_and_grad`` also returns the pose
gradient of every hypothesis's loss, and ``refine_pose_hypotheses`` descends the surface from every hypothesis.  Given
poses [B,N,6] all three do the same for B frame pairs of N hypotheses each, in one call.
"""
import math
import numbers

import torch

from . import _cabi, _raw, ops, stn
from .losses import get_smooth_loss
from .stn import inverse_warp2


def _stacked(fwd_data, inv_data, key):
    """The [2*S*B,1,H,W] tensor whose two halves are fwd_data[key] / inv_data[key].  The dictionaries
    solve_pose_iteratively returns hold slices of one stacked tensor (train_mono.py:94-100): then the base is
    used as it is (no copy, and the gradient flows straight into it); anything else is concatenated once."""
    f, i = fwd_data[key], inv_data[key]
    base = f._base
    if (base is not None and base is i._base and base.is_contiguous() and f.shape == i.shape
            and base.shape[0] == 2 * f.shape[0] and base.shape[1:] == f.shape[1:]
            and f.data_ptr() == base.data_ptr() and i.data_ptr() == base.data_ptr() + f.numel() * f.element_size()):
        return base
    return torch.cat([f, i], 0)


def _pft_flags(options):
    flags = 0
    if options['diff_img_argmin'] == True:             # noqa: E712 -- the reference compares with ==
        flags |= _cabi.PFT_ARGMIN
    if options['automasking'] == True:                 # noqa: E712
        flags |= _cabi.PFT_AUTOMASK
    if options['l_inverse_reconstruction'] == True:    # noqa: E712
        flags |= _cabi.PFT_INVERSE
    if options['l_depth_consist'] == True:             # noqa: E712
        flags |= _cabi.PFT_DEPTH_CONSIST
    return flags


def compute_optimization_loss(options, target_img, target_disparity, init_disparity, fwd_data, inv_data,
                              ssim_loss=None):
    """optimizer.py:45-97 without the plotting branches.  `init_disparity` is the reference's
    ``self.target_disparity`` (the un-optimised prediction).

    The reconstruction and depth-consistency terms (optimizer.py:45-86: per-pixel min over the sources,
    valid-mask union, auto-mask, the masked weighted means and the two (1 - weight).mean() terms) are one
    fused launch forward and one backward (csrc/pft_kernels.cu); the depth-initialisation term is the fused
    SSIM-mean pair; no full-image PyTorch operator runs here."""
    bsz = target_img.shape[0]
    n_src = options['num_source_imgs']
    if fwd_data['diff_img'].shape[0] != n_src * bsz or inv_data['diff_img'].shape[0] != n_src * bsz:
        raise ValueError("compute_optimization_loss: the error maps must hold num_source_imgs * batch pairs")
    maps = [_stacked(fwd_data, inv_data, k) for k in ('diff_img', 'valid_mask', 'auto_mask_error', 'auto_mask', 'weight_mask')]
    w_depth = float(options['l_depth_consist_weight']) if options['l_depth_consist'] == True else 0.0   # noqa: E712
    loss = ops.PftReduceFn.apply(*maps, bsz, n_src, _pft_flags(options), w_depth)
    if options['diff_img_argmin'] != True:   # noqa: E712 -- only the arg-min term keeps the channel dim (optimizer.py:69)
        loss = loss.reshape(())
    if options['l_depth_init'] == True:   # noqa: E712
        loss = loss + options['l_depth_init_weight'] * ops.SsimMeanFn.apply(target_disparity, init_disparity.detach()).reshape(())
    if options['l_smooth'] == True:   # noqa: E712
        loss = loss + options['l_smooth_weight'] * get_smooth_loss(target_disparity, target_img)
    if options['l_pose_consist'] == True:   # noqa: E712
        loss = loss + 0.1 * (fwd_data['poses'] + inv_data['poses']).abs().mean()
    return loss


def compute_photometric_error(target_img, source_img, target_depth, source_depth, pose, intrinsics):
    """helpers.py:8-23: single-pair forward error maps for the loss-surface plots (one warp
    launch + one photometric launch)."""
    img_rec, valid_mask, projected_depth, computed_depth = inverse_warp2(
        source_img, target_depth, source_depth, -pose, intrinsics, 'zeros')
    # auto_mask * valid_mask (helpers.py:18) comes out of the photometric launch itself
    _, diff_img, masked, weight_mask = ops.PhotoErrorFn.apply(
        target_img.detach(), source_img.detach(), img_rec, projected_depth, computed_depth, 0.15, 0.85, valid_mask)
    return {'diff_img': diff_img, 'img_rec': img_rec, 'valid_mask': masked,
            'weight_mask': weight_mask, 'poses': pose}


def photometric_loss_surface(target_img, source_img, target_depth, source_depth, poses, intrinsics, return_maps=False):
    """compute_photometric_error (helpers.py:8-23) of one frame pair under N pose hypotheses, reduced per hypothesis to
    the loss-surface value sum(diff_img * valid_mask * weight_mask) / sum(valid_mask) of plot_loss_surface.py:11-87.

    target_img / source_img [1,3,H,W] (may be channel slices), target_depth / source_depth [1,1,H,W], poses [N,6] or
    [N,8] (columns 0:6, un-negated like `pose` of compute_photometric_error), intrinsics [1,3,3].  Returns
    {'loss': [N], 'error_sum': [N], 'valid_sum': [N]}; with return_maps=True also 'diff_img', 'img_rec', 'valid_mask'
    and 'weight_mask' stacked over the N hypotheses.  The maps are bit-identical to N batch-1 calls of
    compute_photometric_error; the sums are added in a fixed order (deterministic), loss = error_sum / valid_sum
    (NaN where no pixel is valid).  Six launches whatever N is: K^-1, K @ [R|t] of every hypothesis, the three of
    tcsfm_photo_sweep and the division.  Forward only.

    B frame pairs of N hypotheses each: poses [B,N,6] or [B,N,8], target_img / source_img [B,3,H,W] (may be channel
    slices), depths [B,1,H,W], intrinsics [B,3,3].  The outputs gain the leading B ([B,N] sums, [B,N,C,H,W] maps),
    and row (b, n) holds the bits of the single-pair call on pair b with poses[b].  One more launch, for the rows of
    K, whatever B is."""
    ops._require_cuda(target_img, source_img, target_depth, source_depth, poses, intrinsics)
    if torch.is_grad_enabled() and any(t.requires_grad for t in (target_img, source_img, target_depth, source_depth,
                                                                     poses, intrinsics)):
        raise NotImplementedError("photometric_loss_surface is forward only: no gradient of the surface is implemented "
                                  "(photometric_loss_surface_and_grad returns the pose gradient)")
    _check_surface_args(target_img, poses, source_img, target_depth, source_depth, intrinsics)
    h, w = target_img.shape[2], target_img.shape[3]
    kinv = stn.inverse_intrinsics(intrinsics)
    with ops._guard(poses):
        proj = _surface_projections(*_hypothesis_rows(poses, intrinsics)).view(poses.shape[:-1] + (3, 4))
        sums, maps = _raw.photo_sweep(ops.lib(), target_img, source_img, target_depth, source_depth, kinv, proj,
                                      0.15, 0.85, ops.arith_flags(1, h, w), want_maps=return_maps)
    out = {'loss': sums[..., 0] / sums[..., 1], 'error_sum': sums[..., 0], 'valid_sum': sums[..., 1]}
    if return_maps:
        out['img_rec'], out['diff_img'], out['valid_mask'], out['weight_mask'] = maps
    return out


def photometric_loss_surface_and_grad(target_img, source_img, target_depth, source_depth, poses, intrinsics):
    """photometric_loss_surface's 'loss', 'error_sum' and 'valid_sum' (the same bits) plus 'pose_grad', the shape of
    `poses`: row n is d loss[n] / d poses[n] as autograd gives it for the batch-1 expression
    sum(diff_img * valid_mask * weight_mask) / sum(valid_mask) of compute_photometric_error(..., poses[n:n+1], ...).
    The masks carry no gradient; the target image, the depths and the intrinsics get none; columns 6: of [N,8] poses
    are 0; a row with no valid pixel is NaN.

    Functional, not autograd: no graph is recorded and the outputs do not require grad (inputs that require grad are
    read as values).  Seven launches whatever N is: K^-1, K @ [R|t] of every hypothesis, the three of
    tcsfm_photo_sweep_grad (the forward is recomputed inside each CTA, so no workspace grows with N * H * W), the chain
    rule to the pose and the division; [N,8] poses add one for the zero columns.

    B frame pairs as in photometric_loss_surface (poses [B,N,6|8]): [B,N] sums and pose_grad [B,N,6|8], row (b, n)
    with the bits of the single-pair call on pair b; one more launch, for the rows of K."""
    ops._require_cuda(target_img, source_img, target_depth, source_depth, poses, intrinsics)
    _check_surface_args(target_img, poses, source_img, target_depth, source_depth, intrinsics)
    h, w = target_img.shape[2], target_img.shape[3]
    with torch.no_grad(), ops._guard(poses):
        kinv = stn.inverse_intrinsics(intrinsics)
        rows, k_rows = _hypothesis_rows(poses, intrinsics)
        proj = _surface_projections(rows, k_rows).view(poses.shape[:-1] + (3, 4))
        sums, g_proj = _raw.photo_sweep_grad(ops.lib(), target_img, source_img, target_depth, source_depth, kinv, proj,
                                             0.15, 0.85, ops.arith_flags(1, h, w))
        pose_grad = _raw.pose_proj_bwd(ops.lib(), rows[:, 0:6], k_rows, -1.0, g_proj.view(-1, 3, 4))
        pose_grad = pose_grad.view(poses.shape[:-1] + (6,))
        if poses.shape[-1] > 6:
            pose_grad = torch.nn.functional.pad(pose_grad, (0, poses.shape[-1] - 6))
        return {'loss': sums[..., 0] / sums[..., 1], 'error_sum': sums[..., 0], 'valid_sum': sums[..., 1],
                'pose_grad': pose_grad}


def refine_pose_hypotheses(target_img, source_img, target_depth, source_depth, poses, intrinsics,
                           steps=50, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
    """Multi-start photometric pose refinement: `steps` Adam updates of every hypothesis of photometric_loss_surface,
    each on its own loss sum(diff_img * valid_mask * weight_mask) / sum(valid_mask), in one call.

    The arguments are photometric_loss_surface's (poses [N,6] or [N,8], un-negated; columns 6: are carried through).
    The update is Adam without weight decay, per column: for step t the scalars b1 = beta1, a1 = 1 - beta1,
    b2 = beta2, a2 = 1 - beta2, eps, c1 = lr / (1 - beta1**t) and c2 = sqrt(1 - beta2**t) are formed in double and
    rounded to fp32 once; with g the pose_grad photometric_loss_surface_and_grad gives at the current pose,
        m = b1*m + a1*g;  v = b2*v + a2*(g*g);  p = p - c1*(m / (sqrt(v)/c2 + eps))
    each operation rounded to fp32 (m = v = 0 at first).  A hypothesis with no valid pixel at its current pose is not
    updated (its gradient is NaN), so it keeps that pose and a NaN loss from then on.

    Returns {'poses': the poses after `steps` updates, 'loss': [steps+1, N] (row k at the poses after k updates),
    'best_loss': [N] the smallest finite loss of each column (NaN if none), 'best_step': [N] int64 the first row that
    reaches it (-1 if none), 'best_pose': the pose there (the starting pose if none)}.

    Functional, not autograd: no graph is recorded, inputs that require grad are read as values and `poses` is not
    written.  2 * steps + 6 launches for [N,6] poses: K^-1, the 2 * steps + 4 of tcsfm_photo_refine (the auto-mask
    error, K[R|t] of the starting poses, per step the fused forward + adjoint and the update, then the last
    evaluation) and best_step's int64 copy; [N,8] poses add two for their columns 6:.  No host work between the
    steps, the same bits on every call, and capturable in a CUDA graph.

    B frame pairs as in photometric_loss_surface (poses [B,N,6|8], each pair descending with its own intrinsics), with
    the same launch count: 'poses' and 'best_pose' [B,N,6|8], 'loss' [steps+1,B,N], 'best_loss' and 'best_step'
    [B,N]; entry (b, n) has the bits of the single-pair call on pair b with poses[b]."""
    ops._require_cuda(target_img, source_img, target_depth, source_depth, poses, intrinsics)
    _check_surface_args(target_img, poses, source_img, target_depth, source_depth, intrinsics)
    steps, lr, beta1, beta2, eps = _check_adam_args(steps, lr, betas, eps)
    h, w = target_img.shape[2], target_img.shape[3]
    with torch.no_grad(), ops._guard(poses):
        kinv = stn.inverse_intrinsics(intrinsics)
        final, loss, best_loss, best_step, best_pose = _raw.photo_refine(
            ops.lib(), target_img, source_img, target_depth, source_depth, kinv, intrinsics, poses[..., 0:6], steps, lr,
            beta1, beta2, eps, 0.15, 0.85, ops.arith_flags(1, h, w), ops.pose_flags(1))
        if poses.shape[-1] > 6:
            final = torch.cat([final, poses[..., 6:]], -1)
            best_pose = torch.cat([best_pose, poses[..., 6:]], -1)
        return {'poses': final, 'loss': loss, 'best_loss': best_loss, 'best_step': best_step.long(),
                'best_pose': best_pose}


def _check_adam_args(steps, lr, betas, eps):
    """(steps, lr, beta1, beta2, eps) as int and floats, or ValueError."""
    if isinstance(steps, bool) or not isinstance(steps, numbers.Integral) or steps < 0:
        raise ValueError("refine_pose_hypotheses: steps must be an int >= 0, got %r" % (steps,))
    try:
        lr, eps = float(lr), float(eps)
        beta1, beta2 = (float(b) for b in betas)
    except (TypeError, ValueError):
        raise ValueError("refine_pose_hypotheses: lr and eps must be numbers and betas a pair of numbers, got lr=%r "
                         "betas=%r eps=%r" % (lr, betas, eps)) from None
    for name, x in (("lr", lr), ("eps", eps)):
        if not (math.isfinite(x) and x > 0):
            raise ValueError("refine_pose_hypotheses: %s must be finite and > 0, got %r" % (name, x))
    for x in (beta1, beta2):
        if not 0.0 <= x < 1.0:
            raise ValueError("refine_pose_hypotheses: each beta must be in [0, 1), got %r" % (betas,))
    return int(steps), lr, beta1, beta2, eps


def _check_surface_args(target_img, poses, source_img, target_depth, source_depth, intrinsics):
    """poses [N,6|8]: one frame pair (batch-1 inputs); poses [B,N,6|8]: B pairs, whose inputs must all have batch B."""
    if poses.dim() == 3:
        b = poses.shape[0]
        if b < 1 or poses.shape[1] < 1 or poses.shape[2] not in (6, 8):
            raise ValueError("photometric_loss_surface: poses must be [B,N,6] or [B,N,8] with B, N >= 1, got %s"
                             % list(poses.shape))
        for t, c, name in ((target_img, 3, "target_img"), (source_img, 3, "source_img"),
                           (target_depth, 1, "target_depth"), (source_depth, 1, "source_depth")):
            if t.dim() != 4 or t.shape[0] != b or t.shape[1] != c:
                raise ValueError("photometric_loss_surface: %s must be [B,%d,H,W] with the B = %d of poses [B,N,%d], "
                                 "got %s" % (name, c, b, poses.shape[2], list(t.shape)))
        if tuple(intrinsics.shape) != (b, 3, 3):
            raise ValueError("photometric_loss_surface: intrinsics must be [B,3,3] with the B = %d of poses, got %s"
                             % (b, list(intrinsics.shape)))
        return
    if target_img.dim() != 4 or target_img.shape[0] != 1:
        raise ValueError("photometric_loss_surface: one frame pair (batch 1) per call, or pass poses [B,N,6] for B "
                         "pairs, got target_img %s" % list(target_img.shape))
    if poses.dim() != 2 or poses.shape[0] < 1 or poses.shape[1] not in (6, 8):
        raise ValueError("photometric_loss_surface: poses must be [N,6] or [N,8] with N >= 1, got %s" % list(poses.shape))


def _hypothesis_rows(poses, intrinsics):
    """(pose rows [R,6|8], intrinsics [R,3,3] or [1,3,3]) with row r the intrinsics of pose row r: the rows of
    [B,N,6|8] poses are pair-major, so pair b's K is repeated N times."""
    if poses.dim() == 3:
        b, n = poses.shape[0], poses.shape[1]
        return poses.reshape(b * n, poses.shape[2]), intrinsics[:, None].expand(b, n, 3, 3).reshape(b * n, 3, 3)
    return poses, intrinsics


def _surface_projections(poses, intrinsics):
    """K @ [R|t] of -pose for every hypothesis, as the batch-1 call of compute_photometric_error forms it: with the
    batch-1 rounding of the pose algebra (and, in the sweep, the batch-1 warp arithmetic) whatever N is."""
    if intrinsics.is_cuda:
        return _raw.pose_proj_fwd(ops.lib(), poses[:, 0:6], intrinsics, -1.0, ops.pose_flags(1))
    # CPU tensors (test builds): the eager operators stn.projection_matrices takes there
    return intrinsics @ stn.pose_vec2mat(-poses[:, 0:6])
