"""Tensor-level marshalling onto the C ABI (include/tcsfm.h).

These helpers take torch tensors, allocate the outputs with torch's allocator and
pass raw pointers + the current CUDA stream to the library.  They are device
agnostic on purpose (the test-only CUDA emulator drives the same code with host
pointers); the public operators in ``ops.py`` are the ones that insist on CUDA.
"""
import ctypes as C

import torch

from . import _cabi, _timing
from ._cabi import PairGroup


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t):
    if t.is_cuda:
        return torch.cuda.current_stream(t.device).cuda_stream
    return None


def _call(lib, fn, name, is_cuda, *args, launches=1):
    """fn(*args), one entry point of `lib`: timed as `name` while a kernel timer is recording (CUDA calls only), its
    return code checked, and the `launches` kernels it issues added to the launch count."""
    with _timing.launch(name, is_cuda):
        rc = fn(*args)
    _cabi.check(lib, rc)
    _timing.count_launch(launches)


def _f32c(t, name):
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, t.dtype))
    return t.contiguous()


def image_view(img, name="img"):
    """(tensor, batch stride, channel stride) of a [B,C,H,W] fp32 view whose rows
    are dense; other layouts (never produced by the reference's callers) are
    copied once."""
    if img.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, img.dtype))
    b, c, h, w = img.shape
    ok = img.stride(3) == 1 and img.stride(2) == w
    if b > 1 and img.stride(0) < 0 or c > 1 and img.stride(1) < 0:
        ok = False
    if not ok:
        img = img.contiguous()
    return img, (img.stride(0) if b > 1 else c * h * w), (img.stride(1) if c > 1 else h * w)


def _expect(t, shape, name):
    """The kernels index raw pointers: a wrongly shaped tensor would be read out of bounds, so every
    marshalling helper checks the shapes the reference's own operators would have rejected."""
    if t is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (name, list(shape), list(t.shape)))


def warp_fwd(lib, img, depth, ref_depth, kinv, proj, flags=0, need_depths=True, stack_target=None):
    """stack_target: optional [B,3,H,W] view of the reconstruction target; when given the kernel
    also writes the next pose-network input [target * valid | projected_img] ([B,6,H,W])."""
    b, _, h, w = img.shape
    _expect(img, (b, 3, h, w), "img")
    _expect(depth, (b, 1, h, w), "depth")
    _expect(ref_depth, (b, 1, h, w), "ref_depth")
    _expect(kinv, (b, 3, 3), "kinv")
    _expect(proj, (b, 3, 4), "proj")
    _expect(stack_target, (b, 3, h, w), "stack_target")
    img, sb, sc = image_view(img)
    depth, ref_depth = _f32c(depth, "depth"), _f32c(ref_depth, "ref_depth")
    kinv, proj = _f32c(kinv, "kinv"), _f32c(proj, "proj")
    out_img = torch.empty((b, 3, h, w), dtype=torch.float32, device=img.device)
    out_valid = torch.empty((b, 1, h, w), dtype=torch.float32, device=img.device)
    out_pd = torch.empty_like(out_valid) if need_depths else None
    out_cd = torch.empty_like(out_valid) if need_depths else None
    tgt, tsb, tsc, stack = None, 0, 0, None
    if stack_target is not None:
        tgt, tsb, tsc = image_view(stack_target, "stack_target")
        stack = torch.empty((b, 6, h, w), dtype=torch.float32, device=img.device)
    _call(lib, lib.tcsfm_warp_fwd, "warp_fwd", img.is_cuda,
          _ptr(img), sb, sc, _ptr(depth), _ptr(ref_depth), _ptr(kinv), _ptr(proj),
          _ptr(out_img), _ptr(out_valid), _ptr(out_pd), _ptr(out_cd),
          _ptr(tgt), tsb, tsc, _ptr(stack), b, h, w, flags, _stream(img))
    if stack_target is not None:
        return out_img, out_valid, out_pd, out_cd, stack
    return out_img, out_valid, out_pd, out_cd


def warp_bwd(lib, img, depth, ref_depth, kinv, proj, g_img, g_pd, g_cd, flags=0,
             need_img_grad=False, need_ref_depth_grad=True, g_stack=None):
    b, _, h, w = img.shape
    _expect(img, (b, 3, h, w), "img")
    _expect(depth, (b, 1, h, w), "depth")
    _expect(ref_depth, (b, 1, h, w), "ref_depth")
    _expect(kinv, (b, 3, 3), "kinv")
    _expect(proj, (b, 3, 4), "proj")
    _expect(g_img, (b, 3, h, w), "g_img")
    _expect(g_pd, (b, 1, h, w), "g_pd")
    _expect(g_cd, (b, 1, h, w), "g_cd")
    _expect(g_stack, (b, 6, h, w), "g_stack")
    img, sb, sc = image_view(img)
    depth, ref_depth = _f32c(depth, "depth"), _f32c(ref_depth, "ref_depth")
    kinv, proj = _f32c(kinv, "kinv"), _f32c(proj, "proj")
    g_img, g_pd, g_cd = _f32c(g_img, "g_img"), _f32c(g_pd, "g_pd"), _f32c(g_cd, "g_cd")
    g_stack = _f32c(g_stack, "g_stack")
    dev = img.device
    g_depth = torch.empty((b, 1, h, w), dtype=torch.float32, device=dev)
    g_ref = torch.empty((b, 1, h, w), dtype=torch.float32, device=dev) if need_ref_depth_grad else None
    g_proj = torch.empty((b, 3, 4), dtype=torch.float32, device=dev)
    g_src = torch.empty((b, 3, h, w), dtype=torch.float32, device=dev) if need_img_grad else None
    _call(lib, lib.tcsfm_warp_bwd, "warp_bwd", img.is_cuda,
          _ptr(img), sb, sc, _ptr(depth), _ptr(ref_depth), _ptr(kinv), _ptr(proj),
          _ptr(g_img), _ptr(g_pd), _ptr(g_cd), _ptr(g_stack),
          _ptr(g_depth), _ptr(g_ref), _ptr(g_proj), _ptr(g_src),
          b, h, w, flags, _stream(img))
    return g_depth, g_ref, g_proj, g_src


def ssim_fwd(lib, x, y, flags=0):
    x, y = _f32c(x, "x"), _f32c(y, "y")
    if x.shape != y.shape or x.dim() != 4:
        raise ValueError("ssim: x and y must be [B,C,H,W] of equal shape")
    b, c, h, w = x.shape
    out = torch.empty_like(x)
    _call(lib, lib.tcsfm_ssim_fwd, "ssim_fwd", x.is_cuda, _ptr(x), _ptr(y), _ptr(out), b * c, h, w, flags, _stream(x))
    return out


def ssim_bwd(lib, x, y, g_out, need_x=True, need_y=True, flags=0):
    x, y, g_out = _f32c(x, "x"), _f32c(y, "y"), _f32c(g_out, "g_out")
    b, c, h, w = x.shape
    g_x = torch.empty_like(x) if need_x else None
    g_y = torch.empty_like(x) if need_y else None
    _call(lib, lib.tcsfm_ssim_bwd, "ssim_bwd", x.is_cuda,
          _ptr(x), _ptr(y), _ptr(g_out), _ptr(g_x), _ptr(g_y), b * c, h, w, flags, _stream(x))
    return g_x, g_y


def ssim_mean_fwd(lib, x, y, flags=0):
    """mean(SSIM_Loss(x, y)) as a [1] tensor, one launch (no map is written)."""
    x, y = _f32c(x, "x"), _f32c(y, "y")
    if x.shape != y.shape or x.dim() != 4:
        raise ValueError("ssim: x and y must be [B,C,H,W] of equal shape")
    b, c, h, w = x.shape
    out = torch.empty((1,), dtype=torch.float32, device=x.device)
    _call(lib, lib.tcsfm_ssim_mean_fwd, "ssim_mean_fwd", x.is_cuda, _ptr(x), _ptr(y), _ptr(out), b * c, h, w, flags, _stream(x))
    return out


def ssim_mean_bwd(lib, x, y, g_mean, need_x=True, need_y=True, flags=0):
    x, y, g_mean = _f32c(x, "x"), _f32c(y, "y"), _f32c(g_mean, "g_mean")
    b, c, h, w = x.shape
    g_x = torch.empty_like(x) if need_x else None
    g_y = torch.empty_like(x) if need_y else None
    _call(lib, lib.tcsfm_ssim_mean_bwd, "ssim_mean_bwd", x.is_cuda,
          _ptr(x), _ptr(y), _ptr(g_mean), _ptr(g_x), _ptr(g_y), b * c, h, w, flags, _stream(x))
    return g_x, g_y


def intrinsics_inverse(lib, K):
    """K^-1 [B,3,3] (row-major, contiguous) of fp32 matrices [B,3,3] with the bits of K.inverse() on CUDA, one launch."""
    _expect(K, (K.shape[0], 3, 3), "intrinsics")
    K = _f32c(K, "intrinsics")
    out = torch.empty_like(K)
    _call(lib, lib.tcsfm_intrinsics_inverse, "intrinsics_inverse", K.is_cuda, _ptr(K), _ptr(out), K.shape[0], _stream(K))
    return out


def u8_to_float(lib, src, out=None):
    """float(src) / 255 (the loader's conversion, utils/custom_transforms.py:74) of a uint8 tensor; `out`: optional
    preallocated fp32 tensor of the same shape (e.g. the static input buffer of a CUDA graph)."""
    if src.dtype != torch.uint8:
        raise TypeError("u8_to_float expects a uint8 tensor, got %s" % src.dtype)
    src = src.contiguous()
    if out is None:
        out = torch.empty(src.shape, dtype=torch.float32, device=src.device)
    elif out.dtype != torch.float32 or out.shape != src.shape or not out.is_contiguous():
        raise ValueError("u8_to_float: `out` must be a contiguous fp32 tensor of the input's shape")
    _call(lib, lib.tcsfm_u8_to_float, "u8_to_float", src.is_cuda, _ptr(src), _ptr(out), src.numel(), _stream(src))
    return out


class PairBatch:
    """Host-side descriptor array for one multi-group pair-loss launch; keeps every
    tensor it points at alive."""

    def __init__(self, groups):
        # groups: list of dicts with tgt_img, ref_img, tgt_depth, ref_depth, kinv, proj
        self.n = len(groups)
        self.arr = (PairGroup * self.n)()
        self.keep = []
        first = groups[0]["tgt_img"]
        self.b, _, self.h, self.w = first.shape
        self.device = first.device
        for i, g in enumerate(groups):
            if g["tgt_img"].shape != first.shape or g["ref_img"].shape != first.shape:
                raise ValueError("all pair groups of one launch must share [B,3,H,W]")
            _expect(first, (self.b, 3, self.h, self.w), "tgt_img")
            _expect(g["tgt_depth"], (self.b, 1, self.h, self.w), "tgt_depth")
            _expect(g.get("ref_depth"), (self.b, 1, self.h, self.w), "ref_depth")
            _expect(g["kinv"], (self.b, 3, 3), "kinv")
            _expect(g["proj"], (self.b, 3, 4), "proj")
            tgt, tsb, tsc = image_view(g["tgt_img"], "tgt_img")
            ref, rsb, rsc = image_view(g["ref_img"], "ref_img")
            td, rd = _f32c(g["tgt_depth"], "tgt_depth"), _f32c(g.get("ref_depth"), "ref_depth")
            kinv, proj = _f32c(g["kinv"], "kinv"), _f32c(g["proj"], "proj")
            self.keep.append((tgt, ref, td, rd, kinv, proj))
            a = self.arr[i]
            a.tgt_img, a.tgt_sb, a.tgt_sc = _ptr(tgt), tsb, tsc
            a.ref_img, a.ref_sb, a.ref_sc = _ptr(ref), rsb, rsc
            a.tgt_depth, a.ref_depth, a.kinv, a.proj = _ptr(td), _ptr(rd), _ptr(kinv), _ptr(proj)

    def stream(self):
        return _stream(self.keep[0][0])


def pair_loss_fwd(lib, batch, w_l1, w_ssim, flags, want_diff=True, want_grad=True):
    """Returns (diff [G,B,1,H,W] or None, mask [G,B,1,H,W], sums [G,4], coef workspace or None)."""
    g, b, h, w, dev = batch.n, batch.b, batch.h, batch.w, batch.device
    diff = torch.empty((g, b, 1, h, w), dtype=torch.float32, device=dev) if want_diff else None
    mask = torch.empty((g, b, 1, h, w), dtype=torch.float32, device=dev)
    sums = torch.empty((g, 4), dtype=torch.float32, device=dev)
    # workspace the forward leaves for the backward (layout private to the arithmetic flavour in `flags`)
    coef = torch.empty((g, b, lib.tcsfm_pair_ws_floats(h, w, flags)), dtype=torch.float32, device=dev) if want_grad else None
    for i in range(g):
        a = batch.arr[i]
        a.diff_img = _ptr(diff[i]) if want_diff else None
        a.mask = _ptr(mask[i])
        a.sums = _ptr(sums[i])
        a.coef = _ptr(coef[i]) if want_grad else None
    _call(lib, lib.tcsfm_pair_loss_fwd, "pair_loss_fwd", dev.type == "cuda",
          batch.arr, g, b, h, w, w_l1, w_ssim, flags, batch.stream())
    return diff, mask, sums, coef


def pair_loss_bwd(lib, batch, mask, sums, coef, g_diff, g_scalars, w_l1, w_ssim, flags, need_ref_depth_grad):
    """g_diff: [G,B,1,H,W] or None; g_scalars: [G,2] or None.
    Returns (g_tgt_depth [G,B,1,H,W], g_ref_depth [G,B,1,H,W] or None, g_proj [G,B,3,4])."""
    g, b, h, w, dev = batch.n, batch.b, batch.h, batch.w, batch.device
    g_diff, g_scalars = _f32c(g_diff, "g_diff"), _f32c(g_scalars, "g_scalars")
    g_td = torch.empty((g, b, 1, h, w), dtype=torch.float32, device=dev)
    g_rd = torch.empty((g, b, 1, h, w), dtype=torch.float32, device=dev) if need_ref_depth_grad else None
    g_proj = torch.empty((g, b, 3, 4), dtype=torch.float32, device=dev)
    for i in range(g):
        a = batch.arr[i]
        a.mask, a.sums, a.coef = _ptr(mask[i]), _ptr(sums[i]), _ptr(coef[i])
        a.g_diff = _ptr(g_diff[i]) if g_diff is not None else None
        a.g_scalars = _ptr(g_scalars[i]) if g_scalars is not None else None
        a.g_tgt_depth = _ptr(g_td[i])
        a.g_ref_depth = _ptr(g_rd[i]) if need_ref_depth_grad else None
        a.g_proj = _ptr(g_proj[i])
    _call(lib, lib.tcsfm_pair_loss_bwd, "pair_loss_bwd", dev.type == "cuda",
          batch.arr, g, b, h, w, w_l1, w_ssim, flags, batch.stream())
    return g_td, g_rd, g_proj


# ---------------------------------------------------------------------------
# glue kernels of Compute_Loss.forward (csrc/frame_kernels.cu)
# ---------------------------------------------------------------------------

def pose_proj_fwd(lib, pose, K, sign, flags=0):
    """pose [N,6], K [Bk,3,3] -> K @ [R|t] as [N,3,4] (row i uses K[i % Bk])."""
    pose, K = _f32c(pose, "pose"), _f32c(K, "K")
    n = pose.shape[0]
    proj = torch.empty((n, 3, 4), dtype=torch.float32, device=pose.device)
    _call(lib, lib.tcsfm_pose_proj_fwd, "pose_proj_fwd", pose.is_cuda,
          _ptr(pose), sign, _ptr(K), K.shape[0], _ptr(proj), n, flags, _stream(pose))
    return proj


def pose_proj_bwd(lib, pose, K, sign, g_proj):
    pose, K, g_proj = _f32c(pose, "pose"), _f32c(K, "K"), _f32c(g_proj, "g_proj")
    n = pose.shape[0]
    g_pose = torch.empty((n, 6), dtype=torch.float32, device=pose.device)
    _call(lib, lib.tcsfm_pose_proj_bwd, "pose_proj_bwd", pose.is_cuda,
          _ptr(pose), sign, _ptr(K), K.shape[0], _ptr(g_proj), _ptr(g_pose), n, _stream(pose))
    return g_pose


def min_reduce(lib, first, stride, count, n, sums=None, cfg=None):
    """sum_i min_j first.flatten()[j*stride + i] as [1]; `first` is the first competing map.  With `sums` [G,4] and
    `cfg` the launch also finalises the frame: the return value gains (terms [3], total [1]) like frame_finalize."""
    dev = first.device
    out = torch.empty((1,), dtype=torch.float32, device=dev)
    ticket = terms = total = None
    if cfg is not None:
        ticket = torch.empty((1,), dtype=torch.int32, device=dev)
        terms = torch.empty((3,), dtype=torch.float32, device=dev)
        total = torch.empty((1,), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_min_reduce, "min_reduce", first.is_cuda,
          _ptr(first), stride, count, n, _ptr(out), _ptr(ticket), _ptr(sums) if cfg is not None else None,
          C.byref(cfg) if cfg is not None else None, _ptr(terms), _ptr(total), _stream(first))
    if cfg is not None:
        return out, terms, total
    return out


TIE_BAND = 2e-4     # |second smallest - smallest| below which the per-pixel min is re-decided with the exact arithmetic


def pair_min_resolve(lib, batch, group_ids, w_l1, w_ssim, flags, sums=None, cfg=None):
    """Per-pixel min over the listed groups' diff_img with its near-ties re-decided, one launch: returns (sum [1] of that
    min, tie_count int32 [1]); the groups' diff_img entries at the near-tie pixels now hold the exact arithmetic's
    values.  With `sums` [G,4] and `cfg` the launch also finalises the frame: the return value gains (terms [3],
    total [1]) like frame_finalize."""
    sub = (PairGroup * len(group_ids))(*[batch.arr[i] for i in group_ids])
    dev = batch.device
    out = torch.empty((1,), dtype=torch.float32, device=dev)
    counters = torch.empty((2,), dtype=torch.int32, device=dev)
    terms = total = None
    if cfg is not None:
        terms = torch.empty((3,), dtype=torch.float32, device=dev)
        total = torch.empty((1,), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_pair_min_resolve, "pair_min_resolve", dev.type == "cuda",
          sub, len(group_ids), batch.b, batch.h, batch.w, w_l1, w_ssim, flags, TIE_BAND,
          _ptr(out), _ptr(counters), _ptr(sums) if cfg is not None else None,
          C.byref(cfg) if cfg is not None else None, _ptr(terms), _ptr(total), batch.stream())
    if cfg is not None:
        return out, counters[0:1], terms, total
    return out, counters[0:1]


def make_frame_cfg(roles, w_inverse, w_depth, n_min_pixels):
    cfg = _cabi.FrameCfg()
    cfg.n_groups = len(roles)
    for i, r in enumerate(roles):
        cfg.role[i] = r
    cfg.w_inverse, cfg.w_depth, cfg.n_min_pixels = w_inverse, w_depth, n_min_pixels
    return cfg


def frame_finalize(lib, sums, min_sum, cfg):
    """-> terms [3] = (l_reconstruct_inverse, l_reconstruct_forward, l_depth), total [1] = their sum."""
    out = torch.empty((3,), dtype=torch.float32, device=sums.device)
    total = torch.empty((1,), dtype=torch.float32, device=sums.device)
    _call(lib, lib.tcsfm_frame_finalize, "frame_finalize", sums.is_cuda,
          _ptr(sums), _ptr(min_sum), C.byref(cfg), _ptr(out), _ptr(total), _stream(sums))
    return out, total


def frame_bwd_prepare(lib, g_terms, g_total, cfg, zero=None):
    """Upstream of the three terms ([3] or None) and of their sum ([1] or None).  `zero`: a contiguous fp32 buffer the
    same launch fills with zeros (the accumulated depth gradients of the backward pair launch)."""
    ref = g_terms if g_terms is not None else g_total
    g_terms = None if g_terms is None else _f32c(g_terms, "g_terms")
    g_total = None if g_total is None else _f32c(g_total, "g_total")
    g_scalars = torch.empty((cfg.n_groups, 2), dtype=torch.float32, device=ref.device)
    g_min = torch.empty((1,), dtype=torch.float32, device=ref.device)
    if zero is not None and not (zero.numel() % 4 == 0 and zero.data_ptr() % 16 == 0 and zero.is_contiguous()):
        zero.zero_()            # the launch fills 16-byte aligned float4s only
        zero = None
    _call(lib, lib.tcsfm_frame_bwd_prepare, "frame_bwd_prepare", ref.is_cuda,
          _ptr(g_terms), _ptr(g_total), C.byref(cfg), _ptr(g_scalars), _ptr(g_min),
          _ptr(zero), zero.numel() if zero is not None else 0, _stream(ref))
    return g_scalars, g_min


def pair_loss_bwd_shared(lib, batch, mask, sums, coef, g_scalars, g_min, min_info, g_depths, tgt_idx, ref_idx,
                         w_l1, w_ssim, flags, need_ref_depth_grad, zeroed=False):
    """Backward of a multi-group launch whose groups share depth tensors: every group adds into
    g_depths[tgt_idx[i]] / g_depths[ref_idx[i]] (zero-initialised here unless `zeroed`).  min_info =
    (first diff map, stride, [group index -> position or -1], count).  Returns g_proj [G,B,3,4]."""
    g, b, h, w, dev = batch.n, batch.b, batch.h, batch.w, batch.device
    g_proj = torch.empty((g, b, 3, 4), dtype=torch.float32, device=dev)
    if not zeroed:
        g_depths.zero_()
    min_first, min_stride, min_pos, min_count = min_info
    for i in range(g):
        a = batch.arr[i]
        a.mask, a.sums, a.coef = _ptr(mask[i]), _ptr(sums[i]), _ptr(coef[i])
        a.g_diff = None
        a.g_scalars = _ptr(g_scalars[i])
        a.g_tgt_depth = _ptr(g_depths[tgt_idx[i]])
        a.g_ref_depth = _ptr(g_depths[ref_idx[i]]) if need_ref_depth_grad else None
        a.g_proj = _ptr(g_proj[i])
        if min_pos[i] >= 0:
            a.min_base, a.min_stride, a.min_count, a.min_index = _ptr(min_first), min_stride, min_count, min_pos[i]
            a.g_min = _ptr(g_min)
        else:
            a.min_base, a.g_min = None, None
    _call(lib, lib.tcsfm_pair_loss_bwd, "pair_loss_bwd", dev.type == "cuda",
          batch.arr, g, b, h, w, w_l1, w_ssim, flags | _cabi.SHARED_GRADS, batch.stream())
    return g_proj


# ---------------------------------------------------------------------------
# photometric error maps of solve_pose_iteratively(return_errors=True) (csrc/photo_kernels.cu)
# ---------------------------------------------------------------------------

def photo_fwd(lib, tgt, src, rec, proj_depth, comp_depth, w_l1, w_ssim, flags=0, want_grad=True, valid=None):
    """valid: optional inverse_warp2 valid_mask [N,1,H,W]; when given the returned auto_mask is already
    multiplied by it (helpers.py:18)."""
    n, _, h, w = rec.shape
    _expect(valid, (n, 1, h, w), "valid")
    valid = _f32c(valid, "valid")
    for t, name in ((tgt, "tgt"), (src, "src"), (rec, "rec")):
        _expect(t, (n, 3, h, w), name)
    _expect(proj_depth, (n, 1, h, w), "proj_depth")
    _expect(comp_depth, (n, 1, h, w), "comp_depth")
    tgt, tsb, tsc = image_view(tgt, "tgt")
    src, ssb, ssc = image_view(src, "src")
    rec, pd, cd = _f32c(rec, "rec"), _f32c(proj_depth, "proj_depth"), _f32c(comp_depth, "comp_depth")
    dev = rec.device
    outs = [torch.empty((n, 1, h, w), dtype=torch.float32, device=dev) for _ in range(4)]
    coef = torch.empty((n, lib.tcsfm_photo_coef_planes(), h, w), dtype=torch.float32, device=dev) if want_grad else None
    _call(lib, lib.tcsfm_photo_fwd, "photo_fwd", rec.is_cuda,
          _ptr(tgt), tsb, tsc, _ptr(src), ssb, ssc, _ptr(rec), _ptr(pd), _ptr(cd),
          _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[2]), _ptr(outs[3]), _ptr(coef), _ptr(valid),
          n, h, w, w_l1, w_ssim, flags, _stream(rec))
    return outs[0], outs[1], outs[2], outs[3], coef


def photo_bwd(lib, tgt, rec, proj_depth, comp_depth, coef, g_diff, g_weight, w_l1, w_ssim, flags=0):
    n, _, h, w = rec.shape
    tgt, tsb, tsc = image_view(tgt, "tgt")
    rec, pd, cd = _f32c(rec, "rec"), _f32c(proj_depth, "proj_depth"), _f32c(comp_depth, "comp_depth")
    g_diff, g_weight = _f32c(g_diff, "g_diff"), _f32c(g_weight, "g_weight")
    dev = rec.device
    g_rec = torch.empty((n, 3, h, w), dtype=torch.float32, device=dev)
    g_pd = torch.empty((n, 1, h, w), dtype=torch.float32, device=dev)
    g_cd = torch.empty((n, 1, h, w), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_photo_bwd, "photo_bwd", rec.is_cuda,
          _ptr(tgt), tsb, tsc, _ptr(rec), _ptr(pd), _ptr(cd), _ptr(coef), _ptr(g_diff), _ptr(g_weight),
          _ptr(g_rec), _ptr(g_pd), _ptr(g_cd), n, h, w, w_l1, w_ssim, flags, _stream(rec))
    return g_rec, g_pd, g_cd


def _pairs(b, tgt, src, tgt_depth, src_depth, kinv, *expect):
    """Checks and marshals the b frame pairs of the photo_sweep family: tgt / src [b,3,H,W] views, depths [b,1,H,W]
    and kinv [b,3,3].  `expect` holds (tensor, shape, name) checks of the caller's other arguments, made after these
    and before any conversion.  Returns (tgt, its batch and channel strides, src, its batch and channel strides,
    tgt_depth, src_depth, kinv)."""
    h, w = tgt.shape[-2], tgt.shape[-1]
    _expect(tgt, (b, 3, h, w), "tgt")
    _expect(src, (b, 3, h, w), "src")
    _expect(tgt_depth, (b, 1, h, w), "tgt_depth")
    _expect(src_depth, (b, 1, h, w), "src_depth")
    _expect(kinv, (b, 3, 3), "kinv")
    for t, shape, name in expect:
        _expect(t, shape, name)
    tgt, tsb, tsc = image_view(tgt, "tgt")
    src, ssb, ssc = image_view(src, "src")
    return (tgt, tsb, tsc, src, ssb, ssc, _f32c(tgt_depth, "tgt_depth"), _f32c(src_depth, "src_depth"),
            _f32c(kinv, "kinv"))


def _hypotheses(rows, tail):
    """(pairs b, hypotheses per pair n, the leading shape) of `rows`, which is [N] + tail for one pair or [B,N] + tail
    for B pairs."""
    if rows.dim() == len(tail) + 2:
        return rows.shape[0], rows.shape[1], tuple(rows.shape[:2])
    return 1, rows.shape[0], (rows.shape[0],)


def photo_sweep(lib, tgt, src, tgt_depth, src_depth, kinv, proj, w_l1, w_ssim, flags=0, want_maps=False):
    """compute_photometric_error of ONE pair (tgt / src [1,3,H,W] views, depths [1,1,H,W], kinv [1,3,3]) under each of
    the N projections proj [N,3,4], three launches.  Returns (sums [N,2] = (sum(diff * mask * weight), sum(mask)),
    maps) with maps = (rec [N,3,H,W], diff, mask, weight [N,1,H,W]) when `want_maps`, else None.
    With proj [B,N,3,4]: B pairs (tgt / src [B,3,H,W] views, depths [B,1,H,W], kinv [B,3,3]), still three launches;
    the outputs gain the leading B ([B,N,2], [B,N,3,H,W], [B,N,1,H,W])."""
    b, n, lead = _hypotheses(proj, (3, 4))
    h, w = tgt.shape[-2], tgt.shape[-1]
    tgt, tsb, tsc, src, ssb, ssc, td, sd, kinv = _pairs(b, tgt, src, tgt_depth, src_depth, kinv,
                                                        (proj, lead + (3, 4), "proj"))
    proj = _f32c(proj, "proj")
    dev = tgt.device
    scratch = torch.empty((b, h, w), dtype=torch.float32, device=dev)
    partials = torch.empty((lib.tcsfm_photo_sweep_partial_floats(b * n, h, w),), dtype=torch.float32, device=dev)
    sums = torch.empty(lead + (2,), dtype=torch.float32, device=dev)
    maps = None
    if want_maps:
        maps = (torch.empty(lead + (3, h, w), dtype=torch.float32, device=dev),) + \
            tuple(torch.empty(lead + (1, h, w), dtype=torch.float32, device=dev) for _ in range(3))
    rec, diff, mask, weight = maps if want_maps else (None,) * 4
    _call(lib, lib.tcsfm_photo_sweep_pairs, "photo_sweep", tgt.is_cuda,
          _ptr(tgt), tsb, tsc, _ptr(src), ssb, ssc, _ptr(td), _ptr(sd), _ptr(kinv), _ptr(proj),
          _ptr(scratch), _ptr(partials), _ptr(sums), _ptr(rec), _ptr(diff), _ptr(mask), _ptr(weight),
          b, n, h, w, w_l1, w_ssim, flags, _stream(tgt), launches=3)
    return sums, maps


def photo_sweep_grad(lib, tgt, src, tgt_depth, src_depth, kinv, proj, w_l1, w_ssim, flags=0):
    """photo_sweep's sums plus g_proj [N,3,4] = d (sums[n,0] / sums[n,1]) / d proj[n], three launches; proj [B,N,3,4]
    takes B pairs as photo_sweep does (sums [B,N,2], g_proj [B,N,3,4])."""
    b, n, lead = _hypotheses(proj, (3, 4))
    h, w = tgt.shape[-2], tgt.shape[-1]
    tgt, tsb, tsc, src, ssb, ssc, td, sd, kinv = _pairs(b, tgt, src, tgt_depth, src_depth, kinv,
                                                        (proj, lead + (3, 4), "proj"))
    proj = _f32c(proj, "proj")
    dev = tgt.device
    scratch = torch.empty((b, h, w), dtype=torch.float32, device=dev)
    partials = torch.empty((lib.tcsfm_photo_sweep_grad_partial_floats(b * n, h, w),), dtype=torch.float32, device=dev)
    sums = torch.empty(lead + (2,), dtype=torch.float32, device=dev)
    g_proj = torch.empty(lead + (3, 4), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_photo_sweep_grad_pairs, "photo_sweep_grad", tgt.is_cuda,
          _ptr(tgt), tsb, tsc, _ptr(src), ssb, ssc, _ptr(td), _ptr(sd), _ptr(kinv), _ptr(proj),
          _ptr(scratch), _ptr(partials), _ptr(sums), _ptr(g_proj),
          b, n, h, w, w_l1, w_ssim, flags, _stream(tgt), launches=3)
    return sums, g_proj


def photo_refine(lib, tgt, src, tgt_depth, src_depth, kinv, K, poses, steps, lr, beta1, beta2, eps, w_l1, w_ssim,
                 flags=0, pose_flags=0):
    """`steps` Adam updates of each starting pose poses [N,6] on its photo_sweep loss, 2 * steps + 4 launches.  Returns
    (poses [N,6] after the updates, loss [steps+1,N], best_loss [N], best_step int32 [N], best_pose [N,6]); `poses`
    itself is not written.  poses [B,N,6] with K [B,3,3] take B pairs as photo_sweep does, with the same launch count;
    the outputs gain B after their step dimension ([B,N,6], [steps+1,B,N], [B,N])."""
    b, n, lead = _hypotheses(poses, (6,))
    h, w = tgt.shape[-2], tgt.shape[-1]
    tgt, tsb, tsc, src, ssb, ssc, td, sd, kinv = _pairs(b, tgt, src, tgt_depth, src_depth, kinv,
                                                        (K, (b, 3, 3), "K"), (poses, lead + (6,), "poses"))
    K = _f32c(K, "K")
    out = _f32c(poses, "poses").clone()
    dev = tgt.device
    m = torch.empty(lead + (6,), dtype=torch.float32, device=dev)
    v = torch.empty(lead + (6,), dtype=torch.float32, device=dev)
    proj = torch.empty(lead + (3, 4), dtype=torch.float32, device=dev)
    scratch = torch.empty((b, h, w), dtype=torch.float32, device=dev)
    partials = torch.empty((lib.tcsfm_photo_sweep_grad_partial_floats(b * n, h, w),), dtype=torch.float32, device=dev)
    loss = torch.empty((steps + 1,) + lead, dtype=torch.float32, device=dev)
    best_loss = torch.empty(lead, dtype=torch.float32, device=dev)
    best_step = torch.empty(lead, dtype=torch.int32, device=dev)
    best_pose = torch.empty(lead + (6,), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_photo_refine_pairs, "photo_refine", tgt.is_cuda,
          _ptr(tgt), tsb, tsc, _ptr(src), ssb, ssc, _ptr(td), _ptr(sd), _ptr(kinv), _ptr(K),
          _ptr(out), _ptr(m), _ptr(v), _ptr(proj), _ptr(scratch), _ptr(partials),
          _ptr(loss), _ptr(best_loss), _ptr(best_step), _ptr(best_pose),
          b, n, h, w, steps, lr, beta1, beta2, eps, w_l1, w_ssim, flags, pose_flags, _stream(tgt),
          launches=2 * steps + 4)
    return out, loss, best_loss, best_step, best_pose


def _ptr_table(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def disp_to_depth_fwd(lib, disps, min_disp, disp_range, out_hw=None):
    """disps: list of <= 4 equally shaped fp32 maps [B,1,h,w] -> list of depth maps (one launch).
    With out_hw = (H, W) != (h, w) the nearest-neighbour upsample of losses.py:86-87 is folded in:
    the depths come out at [B,1,H,W]."""
    disps = [_f32c(d, "disp") for d in disps]
    b, h, w = disps[0].shape[0], disps[0].shape[-2], disps[0].shape[-1]
    if any(d.shape != disps[0].shape for d in disps):
        raise ValueError("disp_to_depth_fwd: the maps of one launch must share a shape")
    if out_hw is None or tuple(out_hw) == (h, w):
        depths = [torch.empty_like(d) for d in disps]
        _call(lib, lib.tcsfm_disp_to_depth_fwd, "disp_to_depth_fwd", disps[0].is_cuda,
              _ptr_table(disps), _ptr_table(depths), len(disps), disps[0].numel(), min_disp, disp_range, _stream(disps[0]))
    else:
        if disps[0].dim() != 4 or disps[0].shape[1] != 1:
            raise ValueError("disp_to_depth_fwd: upsampling expects [B,1,h,w] maps")
        big_h, big_w = int(out_hw[0]), int(out_hw[1])
        depths = [torch.empty((b, 1, big_h, big_w), dtype=torch.float32, device=d.device) for d in disps]
        _call(lib, lib.tcsfm_disp_upsample_to_depth_fwd, "disp_to_depth_fwd", disps[0].is_cuda,
              _ptr_table(disps), _ptr_table(depths), len(disps), b, h, w, big_h, big_w, min_disp, disp_range,
              _stream(disps[0]))
    return depths


def disp_to_depth_bwd(lib, g_depths, depths, disp_range, disp_hw=None):
    """Gradients w.r.t. the disparities; disp_hw = (h, w) of the disparity maps when they were
    upsampled by disp_to_depth_fwd (the gradient comes out at that resolution)."""
    g_depths = [_f32c(g, "g_depth") for g in g_depths]
    b, big_h, big_w = depths[0].shape[0], depths[0].shape[-2], depths[0].shape[-1]
    if disp_hw is None or tuple(disp_hw) == (big_h, big_w):
        g_disps = [torch.empty_like(d) for d in depths]
        _call(lib, lib.tcsfm_disp_to_depth_bwd, "disp_to_depth_bwd", depths[0].is_cuda,
              _ptr_table(g_depths), _ptr_table(depths), _ptr_table(g_disps), len(depths), depths[0].numel(), disp_range,
              _stream(depths[0]))
    else:
        h, w = int(disp_hw[0]), int(disp_hw[1])
        g_disps = [torch.empty((b, 1, h, w), dtype=torch.float32, device=d.device) for d in depths]
        _call(lib, lib.tcsfm_disp_upsample_to_depth_bwd, "disp_to_depth_bwd", depths[0].is_cuda,
              _ptr_table(g_depths), _ptr_table(depths), _ptr_table(g_disps), len(depths), b, h, w, big_h, big_w, disp_range,
              _stream(depths[0]))
    return g_disps


def pose_rows(poses):
    """The pose tensors of a frame's groups as (list of fp32 tensors readable in place, row stride in floats), or None
    when they do not share a layout (the caller then concatenates them)."""
    if not poses or len(poses) > 8:
        return None
    stride = poses[0].stride(0)
    for p in poses:
        if p.dtype != torch.float32 or p.dim() != 2 or p.shape[1] < 6 or p.stride(1) != 1 or p.stride(0) != stride \
                or p.shape[0] != poses[0].shape[0] or stride < 6:
            return None
    return list(poses), stride


def frame_prologue(lib, disps, min_disp, disp_range, poses, pose_stride, K, sign, flags, want_kinv=False):
    """disp -> depth of <= 4 equally shaped maps, pose -> K[R|t] of the groups' pose tensors and (want_kinv) K^-1 as
    ONE launch.  Returns (depths, proj [G*B,3,4], kinv [B,3,3] or None)."""
    disps = [_f32c(d, "disp") for d in disps]
    if any(d.shape != disps[0].shape for d in disps):
        raise ValueError("frame_prologue: the maps of one launch must share a shape")
    K = _f32c(K, "K")
    b = K.shape[0]
    _expect(K, (b, 3, 3), "K")
    if any(p.shape[0] != b for p in poses) or disps[0].shape[0] != b:
        raise ValueError("frame_prologue: poses / disparities / intrinsics disagree on the batch size")
    depths = [torch.empty_like(d) for d in disps]
    proj = torch.empty((len(poses) * b, 3, 4), dtype=torch.float32, device=K.device)
    kinv = torch.empty((b, 3, 3), dtype=torch.float32, device=K.device) if want_kinv else None
    _call(lib, lib.tcsfm_frame_prologue, "frame_prologue", K.is_cuda,
          _ptr_table(disps), _ptr_table(depths), len(disps), disps[0].numel(), min_disp, disp_range,
          _ptr_table(poses), len(poses), pose_stride, sign, _ptr(K), b, _ptr(proj), _ptr(kinv), flags, _stream(K))
    return depths, proj, kinv


def frame_epilogue(lib, g_depths, depths, disp_range, poses, pose_stride, K, sign, g_proj):
    """The chain rules of frame_prologue as ONE launch: (g_disps, g_pose [G*B,6])."""
    g_depths = [_f32c(g, "g_depth") for g in g_depths]
    K, g_proj = _f32c(K, "K"), _f32c(g_proj, "g_proj")
    b = K.shape[0]
    _expect(g_proj, (len(poses) * b, 3, 4), "g_proj")
    if any(p.shape[0] != b for p in poses) or any(g.shape != d.shape for g, d in zip(g_depths, depths)):
        raise ValueError("frame_epilogue: poses / gradients disagree with the forward's shapes")
    g_disps = [torch.empty_like(d) for d in depths]
    g_pose = torch.empty((len(poses) * b, 6), dtype=torch.float32, device=K.device)
    _call(lib, lib.tcsfm_frame_epilogue, "frame_epilogue", K.is_cuda,
          _ptr_table(g_depths), _ptr_table(depths), _ptr_table(g_disps), len(depths), depths[0].numel(), disp_range,
          _ptr_table(poses), len(poses), pose_stride, sign, _ptr(K), b, _ptr(g_proj), _ptr(g_pose), _stream(K))
    return g_disps, g_pose


def smooth_fwd(lib, disp, img):
    disp = _f32c(disp, "disp")
    img, sb, sc = image_view(img, "img")
    b, _, h, w = disp.shape
    ws = torch.empty((2 * b + 2,), dtype=torch.float32, device=disp.device)
    out = torch.empty((), dtype=torch.float32, device=disp.device)
    _call(lib, lib.tcsfm_smooth_fwd, "smooth_fwd", disp.is_cuda,
          _ptr(disp), _ptr(img), sb, sc, _ptr(ws), _ptr(out), b, h, w, _stream(disp), launches=3)
    return out, ws


def smooth_bwd(lib, disp, img, ws, g_out):
    disp, g_out = _f32c(disp, "disp"), _f32c(g_out, "g_out")
    img, sb, sc = image_view(img, "img")
    b, _, h, w = disp.shape
    g_disp = torch.empty_like(disp)
    _call(lib, lib.tcsfm_smooth_bwd, "smooth_bwd", disp.is_cuda,
          _ptr(disp), _ptr(img), sb, sc, _ptr(ws), _ptr(g_out), _ptr(g_disp), b, h, w, _stream(disp), launches=2)
    return g_disp


# ---------------------------------------------------------------------------
# PFT loss reduction (csrc/pft_kernels.cu; optimization_experiments/optimizer.py:45-86)
# ---------------------------------------------------------------------------

def _halves(t, split, name):
    """(forward half, inverse half) pointers of a stacked [2*S*B,1,H,W] map."""
    t = _f32c(t, name)
    return t, t.data_ptr(), t.data_ptr() + split * t[0].numel() * 4


def pft_reduce_fwd(lib, diff, valid, auto_err, auto_mask, weight, bsz, n_src, flags, w_depth):
    """The maps are the stacked [2*S*B,1,H,W] outputs of solve_pose_iteratively(return_errors=True)
    (forward half first).  Returns (loss [1], sums [8])."""
    split = bsz * n_src
    n = diff[0].numel()
    for t, name in ((diff, "diff_img"), (valid, "valid_mask"), (auto_err, "auto_mask_error"), (auto_mask, "auto_mask"),
                    (weight, "weight_mask")):
        _expect(t, (2 * split,) + tuple(diff.shape[1:]), name)
    keep = [_halves(t, split, name) for t, name in ((diff, "diff"), (valid, "valid"), (auto_err, "auto_err"),
                                                     (auto_mask, "auto_mask"), (weight, "weight"))]
    (_, d_f, d_i), (_, v_f, v_i), (_, a_f, _), (_, _, m_i), (_, w_f, w_i) = keep
    dev = diff.device
    sums = torch.empty((8,), dtype=torch.float32, device=dev)
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    _call(lib, lib.tcsfm_pft_reduce_fwd, "pft_reduce_fwd", diff.is_cuda,
          d_f, v_f, a_f, w_f, d_i, v_i, m_i, w_i, bsz, n_src, n, flags, w_depth, _ptr(sums), _ptr(loss), _stream(diff))
    return loss, sums, [k[0] for k in keep]


def pft_reduce_bwd(lib, maps, sums, g_loss, bsz, n_src, flags, w_depth):
    """maps: the contiguous tensors the forward used.  Returns (g_diff, g_weight), each [2*S*B,1,H,W]."""
    diff, valid, auto_err, auto_mask, weight = maps
    split = bsz * n_src
    n = diff[0].numel()
    half = split * n * 4
    g_loss = _f32c(g_loss, "g_loss")
    g_diff, g_weight = torch.empty_like(diff), torch.empty_like(weight)
    _call(lib, lib.tcsfm_pft_reduce_bwd, "pft_reduce_bwd", diff.is_cuda,
          diff.data_ptr(), valid.data_ptr(), auto_err.data_ptr(), weight.data_ptr(),
          diff.data_ptr() + half, valid.data_ptr() + half, auto_mask.data_ptr() + half, weight.data_ptr() + half,
          bsz, n_src, n, flags, w_depth, _ptr(sums), _ptr(g_loss),
          g_diff.data_ptr(), g_weight.data_ptr(), g_diff.data_ptr() + half, g_weight.data_ptr() + half, _stream(diff))
    return g_diff, g_weight
