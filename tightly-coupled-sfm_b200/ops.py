"""Autograd operators over the CUDA C ABI (hand-written backward kernels).

Every operator requires CUDA tensors and the built library; there is no CPU or
eager-PyTorch fallback (a missing library or a CPU tensor raises).
"""
import contextlib

import torch

from . import _cabi, _raw
from ._lib import lib

# Arithmetic flavour handed to the kernels: 0 reproduces eager PyTorch's CUDA
# operators (the reference's production path); tests flip this to
# _cabi.ARITH_CPU to compare bit-for-bit with CPU-generated golden vectors.
ARITH_FLAGS = 0


# SSIM arithmetic of the fused pair loss: "exact" keeps every rounding step of eager PyTorch (bit-identical
# diff_img / SSIM maps); "fast" (when the library provides it) keeps geometry, warp, L1 and every mask bit-exact
# and evaluates the 3x3 SSIM statistics at tolerance level (loss <= 1e-5, gradients <= 1e-4 of the reference).
PAIR_ARITHMETIC = "exact"
PAIR_ARITHMETICS = ("exact", "fast")
# diagnostics: the device-side near-tie count ([1] int32) of the most recent fast-arithmetic frame loss
LAST_TIE_COUNT = None


def set_arithmetic(mode):
    global PAIR_ARITHMETIC
    if mode not in PAIR_ARITHMETICS:
        raise NotImplementedError("pair-loss arithmetic %r is not available (have %s)" % (mode, ", ".join(PAIR_ARITHMETICS)))
    PAIR_ARITHMETIC = mode


def arith_flags(batch, height, width):
    """Arithmetic flavour of a launch standing in for reference calls with `batch` pairs: eager
    CUDA bmm runs a non-fused kernel for batch 1 while m*n*k = 9*H*W <= 2^21 (bisected on the
    B200: last non-fused size 233016, tools/probe_bmm_b1_bisect.py; include/tcsfm.h)."""
    flags = ARITH_FLAGS
    if not (flags & _cabi.ARITH_CPU) and batch == 1 and 9 * height * width <= (1 << 21):
        flags |= _cabi.ARITH_BMM_NOFMA
    return flags


def pair_flags(batch, height, width):
    """arith_flags plus the SSIM arithmetic selected for the fused pair loss."""
    flags = arith_flags(batch, height, width)
    if PAIR_ARITHMETIC == "fast":
        flags |= _cabi.ARITH_FAST
    return flags


def pose_flags(ref_batch):
    """The 3x3 products of the pose algebra (m*n*k <= 36) always take the non-fused cuBLAS kernel
    at batch 1 (tools/probe_b1_pose.py)."""
    if not (ARITH_FLAGS & _cabi.ARITH_CPU) and ref_batch == 1:
        return _cabi.ARITH_BMM_NOFMA
    return 0


def _guard(t):
    """Makes the tensor's GPU current for the launch (the C ABI launches on the
    current device / the stream it is handed)."""
    return torch.cuda.device(t.device) if t.is_cuda else contextlib.nullcontext()


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("tcsfm_b200 operators run on CUDA tensors only (got a %s tensor); "
                               "there is no CPU fallback" % t.device.type)


class InverseWarp2Fn(torch.autograd.Function):
    """(img, depth, ref_depth, kinv, proj[, stack_target]) -> (projected_img, valid_mask,
    projected_depth, computed_depth[, stack]); kernels: csrc/warp_kernels.cu.  With a
    `stack_target` (the [B,3,H,W] reconstruction target) the forward also emits the next
    pose-network input [target * valid_mask | projected_img] of train_mono.py:74-76."""

    @staticmethod
    def forward(ctx, img, depth, ref_depth, kinv, proj, stack_target=None, need_depths=True):
        # need_depths=False: projected_depth / computed_depth come back as None and are neither computed nor
        # stored (solve_pose_iteratively only consumes the last iteration's, train_mono.py:69,80 vs :91)
        _require_cuda(img, depth, ref_depth, kinv, proj, stack_target)
        ctx.set_materialize_grads(False)
        ctx.flags = arith_flags(img.shape[0], img.shape[2], img.shape[3])
        with _guard(img):
            outs = _raw.warp_fwd(lib(), img, depth, ref_depth, kinv, proj, ctx.flags, need_depths=need_depths,
                                 stack_target=stack_target)
        ctx.save_for_backward(img, depth, ref_depth, kinv, proj)
        ctx.mark_non_differentiable(outs[1])
        return outs

    @staticmethod
    def backward(ctx, g_img, g_valid, g_pd, g_cd, g_stack=None):
        img, depth, ref_depth, kinv, proj = ctx.saved_tensors
        need_img = ctx.needs_input_grad[0]
        need_ref = ctx.needs_input_grad[2] and g_pd is not None      # ref_depth only feeds projected_depth
        with _guard(img):
            g_depth, g_ref, g_proj, g_src = _raw.warp_bwd(
                lib(), img, depth, ref_depth, kinv, proj, g_img, g_pd, g_cd, ctx.flags,
                need_img_grad=need_img, need_ref_depth_grad=need_ref, g_stack=g_stack)
        return g_src, g_depth, g_ref, None, g_proj, None, None


class SsimFn(torch.autograd.Function):
    """SSIM dissimilarity map of two [B,C,H,W] tensors; kernels: csrc/ssim_kernels.cu."""

    @staticmethod
    def forward(ctx, x, y):
        _require_cuda(x, y)
        with _guard(x):
            out = _raw.ssim_fwd(lib(), x, y, ARITH_FLAGS)
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, y = ctx.saved_tensors
        with _guard(x):
            g_x, g_y = _raw.ssim_bwd(lib(), x, y, g_out, ctx.needs_input_grad[0], ctx.needs_input_grad[1], ARITH_FLAGS)
        return g_x, g_y


class SsimMeanFn(torch.autograd.Function):
    """mean(SSIM dissimilarity map) of two [B,C,H,W] tensors as a [1] tensor: one launch forward (no
    map in HBM), one backward (the depth-initialisation term of the PFT loss, optimizer.py:89-90)."""

    @staticmethod
    def forward(ctx, x, y):
        _require_cuda(x, y)
        with _guard(x):
            out = _raw.ssim_mean_fwd(lib(), x, y, ARITH_FLAGS)
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, y = ctx.saved_tensors
        with _guard(x):
            g_x, g_y = _raw.ssim_mean_bwd(lib(), x, y, g_out, ctx.needs_input_grad[0], ctx.needs_input_grad[1], ARITH_FLAGS)
        return g_x, g_y


class PftReduceFn(torch.autograd.Function):
    """(diff_img, valid_mask, auto_mask_error, auto_mask, weight_mask) stacked [2*S*B,1,H,W] -> the
    reconstruction + depth-consistency part of the PFT loss (optimizer.py:45-86) as a [1] tensor;
    kernels: csrc/pft_kernels.cu.  Differentiable w.r.t. diff_img and weight_mask."""

    @staticmethod
    def forward(ctx, diff, valid, auto_err, auto_mask, weight, bsz, n_src, flags, w_depth):
        _require_cuda(diff, valid, auto_err, auto_mask, weight)
        with _guard(diff):
            loss, sums, maps = _raw.pft_reduce_fwd(lib(), diff, valid, auto_err, auto_mask, weight, bsz, n_src, flags, w_depth)
        ctx.save_for_backward(sums, *maps)
        ctx.cfg = (bsz, n_src, flags, w_depth)
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        sums, maps = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        with _guard(sums):
            g_diff, g_weight = _raw.pft_reduce_bwd(lib(), maps, sums, g_loss, *ctx.cfg)
        return g_diff, None, None, None, g_weight, None, None, None, None


class PairLossFn(torch.autograd.Function):
    """G independent groups of B pairs in one launch (csrc/pair_kernels.cu).

    apply(cfg, n_groups, kinv [B,3,3], proj [G*B,3,4], *tensors) with tensors = for
    each group (tgt_img, ref_img, tgt_depth, ref_depth).  Returns
    (diff [G,B,1,H,W], mask [G,B,1,H,W], l_reprojection [G], l_depth [G])."""

    @staticmethod
    def forward(ctx, cfg, n_groups, kinv, proj, *tensors):
        w_l1, w_ssim, flags = cfg
        _require_cuda(kinv, proj, *tensors)
        kinv, proj = kinv.contiguous(), proj.contiguous()
        b = kinv.shape[0]
        groups = []
        for i in range(n_groups):
            t = tensors[4 * i:4 * i + 4]
            groups.append({"tgt_img": t[0], "ref_img": t[1], "tgt_depth": t[2], "ref_depth": t[3],
                           "kinv": kinv, "proj": proj[i * b:(i + 1) * b]})
        flags = flags | pair_flags(b, tensors[0].shape[2], tensors[0].shape[3])
        with _guard(kinv):
            batch = _raw.PairBatch(groups)
            want_grad = any(ctx.needs_input_grad)
            diff, mask, sums, coef = _raw.pair_loss_fwd(lib(), batch, w_l1, w_ssim, flags, want_grad=want_grad)
        # mean_on_mask (losses.py:142-149) without the host round trip
        enough = sums[:, 1] > 10000
        zero = torch.zeros_like(sums[:, 0])
        l_rep = torch.where(enough, sums[:, 0] / sums[:, 1], zero)
        l_dep = torch.where(enough, sums[:, 2] / sums[:, 1], zero)
        ctx.batch, ctx.cfg, ctx.flags, ctx.n_groups = batch, (w_l1, w_ssim), flags, n_groups
        if want_grad:
            ctx.save_for_backward(mask, sums, coef)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(mask)
        return diff, mask, l_rep, l_dep

    @staticmethod
    def backward(ctx, g_diff, g_mask, g_lrep, g_ldep):
        mask, sums, coef = ctx.saved_tensors
        g_scalars = None
        if g_lrep is not None or g_ldep is not None:
            z = torch.zeros_like(sums[:, 0])
            g_scalars = torch.stack([g_lrep if g_lrep is not None else z,
                                     g_ldep if g_ldep is not None else z], dim=1)
        need_ref = (ctx.flags & (_cabi.DEPTH_MASK | _cabi.DEPTH_CONSIST)) != 0
        with _guard(mask):
            g_td, g_rd, g_proj = _raw.pair_loss_bwd(lib(), ctx.batch, mask, sums, coef, g_diff, g_scalars,
                                                    ctx.cfg[0], ctx.cfg[1], ctx.flags, need_ref)
        grads = [None, None, None, g_proj.reshape(-1, 3, 4)]
        for i in range(ctx.n_groups):
            grads += [None, None, g_td[i], g_rd[i] if need_ref else None]
        return tuple(grads)


class DispToDepthFn(torch.autograd.Function):
    """depth = 1 / (min_disp + (max_disp - min_disp) * disp) (utils/learning_helpers.py:77-86) as one launch
    each way; bit-identical to the eager expression (rounded product, rounded sum, IEEE reciprocal)."""

    @staticmethod
    def forward(ctx, disp, min_disp, max_disp):
        _require_cuda(disp)
        with _guard(disp):
            depth = _raw.disp_to_depth_fwd(lib(), [disp], min_disp, max_disp - min_disp)[0]
        ctx.save_for_backward(depth)
        ctx.disp_range = max_disp - min_disp
        return depth

    @staticmethod
    def backward(ctx, g_depth):
        (depth,) = ctx.saved_tensors
        with _guard(depth):
            g = _raw.disp_to_depth_bwd(lib(), [g_depth.contiguous()], [depth], ctx.disp_range)[0]
        return g, None, None


class PoseProjFn(torch.autograd.Function):
    """pose [N,6] (multiplied by `sign`), K [Bk,3,3] -> K @ [Rx Ry Rz | t] as [N,3,4]
    (csrc/frame_kernels.cu); one launch forward, one backward."""

    @staticmethod
    def forward(ctx, pose, K, sign, ref_batch=None):
        # ref_batch: batch size of the reference's own `intrinsics @ pose_vec2mat(pose)` calls this
        # launch stands in for (cuBLAS rounds batch-1 products differently)
        _require_cuda(pose, K)
        flags = pose_flags(pose.shape[0] if ref_batch is None else ref_batch)
        with _guard(pose):
            proj = _raw.pose_proj_fwd(lib(), pose, K, sign, flags)
        ctx.save_for_backward(pose, K)
        ctx.sign = sign
        return proj

    @staticmethod
    def backward(ctx, g_proj):
        pose, K = ctx.saved_tensors
        with _guard(pose):
            g_pose = _raw.pose_proj_bwd(lib(), pose, K, ctx.sign, g_proj)
        return g_pose, None, None, None


class FrameLossFn(torch.autograd.Function):
    """The reconstruction terms of one scale of Compute_Loss.forward (losses.py:86-132) as one
    autograd node: disp_to_depth, pose -> K[R|t], the pair kernel over all direction/source
    groups, min-reprojection reduce and the mean-on-mask finalize forward; prepare, the pair
    kernel, the pose chain rule and the depth -> disparity chain rule backward.

    apply(meta, kinv, K, *poses, *images, *disps) -> (terms [3], total [1]):
    terms = (l_reconstruct_inverse, l_reconstruct_forward, l_depth) before the division by
    num_scales, total = (terms[0] + terms[1]) + terms[2] as Compute_Loss.forward adds them
    (losses.py:134-138).  A loss built on `total` alone costs no slice / add kernels.
    meta: dict(w_l1, w_ssim, flags, w_inverse, w_depth, min_depth, max_depth, n_img,
    groups=[(role, tgt_img, ref_img, tgt_disp, ref_disp)]) with indices into `images` /
    `disps`; one pose [B,6] per group (un-negated); role 0 = inverse, 1 = forward."""

    @staticmethod
    def forward(ctx, meta, kinv, K, *tensors):
        _require_cuda(kinv, K, *tensors)
        groups = meta["groups"]
        g, b = len(groups), K.shape[0]
        poses_in, images, disps = tensors[:g], tensors[g:g + meta["n_img"]], tensors[g + meta["n_img"]:]
        flags = meta["flags"] | pair_flags(b, images[0].shape[2], images[0].shape[3])
        min_disp, max_disp = 1 / meta["max_depth"], 1 / meta["min_depth"]      # learning_helpers.py:82-83
        with _guard(K):
            want_kinv = kinv is None               # models/stn.py:257: computed here, once, and handed back in meta["kinv"]
            if not want_kinv:
                kinv = kinv.contiguous()
            # disparities of a lower pyramid scale arrive at their own resolution: the nearest upsample of
            # losses.py:86-87,102-103 happens inside the disp -> depth kernel
            full_hw = tuple(images[0].shape[-2:])
            rows = _raw.pose_rows(poses_in)
            glued = (rows is not None and len(disps) <= 4 and tuple(disps[0].shape[-2:]) == full_hw
                     and all(d.shape == disps[0].shape for d in disps))
            if glued:
                # full-resolution disparities, poses readable in place: disp -> depth and pose -> K[R|t] in one launch
                poses, pose_stride = rows
                fused_kinv = want_kinv and K.is_cuda
                depths, proj, k_out = _raw.frame_prologue(lib(), disps, min_disp, max_disp - min_disp, poses, pose_stride, K, -1.0,
                                                          pose_flags(b), want_kinv=fused_kinv)
                if fused_kinv:
                    kinv, want_kinv = k_out, False
            else:
                depths = []
                for i in range(0, len(disps), 4):
                    depths += _raw.disp_to_depth_fwd(lib(), disps[i:i + 4], min_disp, max_disp - min_disp, out_hw=full_hw)
                poses, pose_stride = [torch.cat([p[:, 0:6] for p in poses_in], 0)], 6
                proj = _raw.pose_proj_fwd(lib(), poses[0], K, -1.0, pose_flags(b))
            if want_kinv:       # CPU tensors (test builds) take torch's LAPACK inverse, whose bits the CPU goldens carry
                kinv = _raw.intrinsics_inverse(lib(), K.detach()) if K.is_cuda else torch.linalg.inv_ex(K.detach())[0].contiguous()
            meta["kinv"] = kinv
            specs = [{"tgt_img": images[ti], "ref_img": images[ri], "tgt_depth": depths[td], "ref_depth": depths[rd],
                      "kinv": kinv, "proj": proj[i * b:(i + 1) * b]} for i, (_, ti, ri, td, rd) in enumerate(groups)]
            batch = _raw.PairBatch(specs)
            want_grad = any(ctx.needs_input_grad)
            if meta.get("kinv_ready") is not None:         # K^-1 was forked onto a side stream (stn.inverse_intrinsics_forked)
                torch.cuda.current_stream(K.device).wait_event(meta["kinv_ready"])
            diff, mask, sums, coef = _raw.pair_loss_fwd(lib(), batch, meta["w_l1"], meta["w_ssim"], flags, want_grad=want_grad)
            fwd_idx = [i for i, grp in enumerate(groups) if grp[0] == 1]
            step = fwd_idx[1] - fwd_idx[0] if len(fwd_idx) > 1 else 1
            if any(fwd_idx[k + 1] - fwd_idx[k] != step for k in range(len(fwd_idx) - 1)):
                raise ValueError("forward groups must be evenly spaced")
            n_px = diff[0].numel()
            cfg = _raw.make_frame_cfg([grp[0] for grp in groups], meta["w_inverse"], meta["w_depth"], n_px)
            # the per-pixel min over the forward groups and the loss assembly are one launch (the last block of the reduce
            # finalises); terms / total are two separate tensors (not views of one buffer): callers may add to `total` in place
            if fwd_idx and (flags & _cabi.ARITH_FAST) and len(fwd_idx) > 1:
                # tolerance-level diff values: the near-ties of the per-pixel min are kept in shared memory and re-decided
                # with the exact arithmetic right away
                global LAST_TIE_COUNT
                _, LAST_TIE_COUNT, terms, total = _raw.pair_min_resolve(lib(), batch, fwd_idx, meta["w_l1"], meta["w_ssim"], flags,
                                                                        sums=sums, cfg=cfg)
            elif fwd_idx:
                _, terms, total = _raw.min_reduce(lib(), diff[fwd_idx[0]], step * n_px, len(fwd_idx), n_px, sums=sums, cfg=cfg)
            else:
                terms, total = _raw.frame_finalize(lib(), sums, None, cfg)
        if want_grad:
            ctx.save_for_backward(mask, sums, coef, diff, K, *depths, *poses)
            ctx.n_depths, ctx.glued, ctx.pose_stride = len(depths), glued, pose_stride
            ctx.batch, ctx.cfg, ctx.meta, ctx.flags = batch, cfg, meta, flags
            ctx.min_info = (fwd_idx, step * n_px)
            ctx.disp_range = max_disp - min_disp
            ctx.disp_hw = tuple(disps[0].shape[-2:])
            ctx.set_materialize_grads(False)
        return terms, total

    @staticmethod
    def backward(ctx, g_terms, g_total):
        if g_terms is None and g_total is None:
            return (None,) * (3 + len(ctx.meta["groups"]) + ctx.meta["n_img"] + ctx.n_depths)
        mask, sums, coef, diff, K = ctx.saved_tensors[:5]
        depths = list(ctx.saved_tensors[5:5 + ctx.n_depths])
        poses = list(ctx.saved_tensors[5 + ctx.n_depths:])
        meta, groups = ctx.meta, ctx.meta["groups"]
        g, b = len(groups), K.shape[0]
        fwd_idx, stride = ctx.min_info
        need_ref = (ctx.flags & (_cabi.DEPTH_MASK | _cabi.DEPTH_CONSIST)) != 0
        with _guard(K):
            g_depths = torch.empty((len(depths),) + tuple(depths[0].shape), dtype=torch.float32, device=K.device)
            g_scalars, g_min = _raw.frame_bwd_prepare(lib(), g_terms, g_total, ctx.cfg, zero=g_depths)    # also zeroes g_depths
            min_pos = [fwd_idx.index(i) if i in fwd_idx else -1 for i in range(g)]
            min_first = diff[fwd_idx[0]] if fwd_idx else None
            g_proj = _raw.pair_loss_bwd_shared(
                lib(), ctx.batch, mask, sums, coef, g_scalars, g_min, (min_first, stride, min_pos, len(fwd_idx)),
                g_depths, [grp[3] for grp in groups], [grp[4] for grp in groups],
                meta["w_l1"], meta["w_ssim"], ctx.flags, need_ref, zeroed=True)
            if ctx.glued:                       # the two chain rules behind the pair kernel in one launch
                g_disps, g_pose = _raw.frame_epilogue(lib(), [g_depths[j] for j in range(len(depths))], depths, ctx.disp_range,
                                                      poses, ctx.pose_stride, K, -1.0, g_proj.reshape(-1, 3, 4))
            else:
                g_pose = _raw.pose_proj_bwd(lib(), poses[0], K, -1.0, g_proj.reshape(-1, 3, 4))
                g_disps = []
                for i in range(0, len(depths), 4):
                    g_disps += _raw.disp_to_depth_bwd(lib(), [g_depths[j] for j in range(i, min(i + 4, len(depths)))],
                                                      depths[i:i + 4], ctx.disp_range, disp_hw=ctx.disp_hw)
        g_poses = tuple(g_pose[i * b:(i + 1) * b] for i in range(g))
        return (None, None, None) + g_poses + (None,) * meta["n_img"] + tuple(g_disps)


class PhotoErrorFn(torch.autograd.Function):
    """(tgt, src, rec, projected_depth, computed_depth) -> (auto_mask_error, diff_img, auto_mask,
    weight_mask) of train_mono.py:84-92 in one launch; backward w.r.t. rec and the depths in one."""

    @staticmethod
    def forward(ctx, tgt, src, rec, proj_depth, comp_depth, w_l1, w_ssim, valid=None):
        _require_cuda(tgt, src, rec, proj_depth, comp_depth, valid)
        want_grad = any(ctx.needs_input_grad[2:5])
        with _guard(rec):
            auto_err, diff, auto_mask, weight, coef = _raw.photo_fwd(lib(), tgt, src, rec, proj_depth, comp_depth,
                                                                     w_l1, w_ssim, ARITH_FLAGS, want_grad, valid=valid)
        if want_grad:
            ctx.save_for_backward(tgt, rec, proj_depth, comp_depth, coef)
            ctx.weights = (w_l1, w_ssim)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(auto_err, auto_mask)
        return auto_err, diff, auto_mask, weight

    @staticmethod
    def backward(ctx, g_auto_err, g_diff, g_auto_mask, g_weight):
        tgt, rec, proj_depth, comp_depth, coef = ctx.saved_tensors
        with _guard(rec):
            g_rec, g_pd, g_cd = _raw.photo_bwd(lib(), tgt, rec, proj_depth, comp_depth, coef, g_diff, g_weight,
                                               ctx.weights[0], ctx.weights[1], ARITH_FLAGS)
        return None, None, g_rec, g_pd, g_cd, None, None, None


class SmoothLossFn(torch.autograd.Function):
    """get_smooth_loss(disp, img) (losses.py:43-61) -> scalar; kernels: csrc/smooth_kernels.cu."""

    @staticmethod
    def forward(ctx, disp, img):
        _require_cuda(disp, img)
        with _guard(disp):
            out, ws = _raw.smooth_fwd(lib(), disp, img)
        ctx.save_for_backward(disp, img, ws)
        return out

    @staticmethod
    def backward(ctx, g_out):
        disp, img, ws = ctx.saved_tensors
        with _guard(disp):
            g_disp = _raw.smooth_bwd(lib(), disp, img, ws, g_out)
        return g_disp, None
