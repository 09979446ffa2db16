"""The hand-written backward kernels against a float64 evaluation of the oracle, region by region.

Every case runs one operation three times on the same device: through the public drop-in API (the CUDA kernels, or
their emulator build where there is no GPU), through the oracle in fp32 (eager PyTorch: the reference's own
arithmetic), and through the oracle in float64 with float64 inputs and upstream gradients.  Each gradient is then
compared with the float64 one separately on each region of the image where the kernels branch:

- ``border``: rows and columns 0, 1, H-2, H-1 (the reflection duplicates of the SSIM adjoints, the edge taps of the
  bilinear scatter);
- ``corners``: the four corner pixels;
- ``seams`` (64x16-tiled kernels): x mod 64 in {0, 63} or y mod 16 in {0, 15}, the halo cells of a tile;
- ``partial_tile`` (when W % 64 or H % 16 is not 0): the last, partly filled tile column and row;
- ``chunk_edges`` / ``tail_chunk`` (warp backward, one thread block per kWarpThreads * kWarpBwdPix = 1024 pixels):
  the first and last warp of every chunk, and the last, partial chunk;
- ``interior``: everything off the border and the seams.

A global rel-L2 sees an error of relative size e on a fraction f of the pixels as about e * sqrt(f), so one wrong
column or corner passes a loose global tolerance.  Per region the bounds are

    ||kernel - f64||  <= RATIO_L2  * max(||eager fp32 - f64||,  rel_eager * ||f64||)     + FLOOR * ||f64||
    max|kernel - f64| <= RATIO_MAX * max(max|eager fp32 - f64|, maxrel_eager * max|f64|) + FLOOR * max|f64|

with norms and maxima over the region, and rel_eager / maxrel_eager the eager errors over the whole tensor relative
to its norm / largest entry.  The second term matters only in regions of a few entries (the corners, a 2x2 image),
where eager's error is a sample of a handful of roundings and can be several times below its typical size by luck:
a defect confined to one region still stands out against the whole tensor's eager error.  When the whole image has
fewer than FEW_PIXELS pixels (the 2x2 and 3x5 cases) that estimate is a handful of roundings too: the SSIM-mean
gradient of a 2x2 image (y = 0.9 x + 0.02, so the statistics cancel) has a kernel / eager ratio between 0.8 and 6.1
over twelve seeds while the kernel's own error stays in eager's range (7e-7 to 2e-5 of the gradient's norm).  Those
images get RATIO_FEW for both bounds; a missing reflection duplicate moves them by more than 1e3.

Pixels where the fp32 and float64 references take different discrete decisions follow a different branch of the
adjoint in the two, so they are excluded, together with every gradient entry they feed: the valid mask, the
out-of-view overwrite, the floor cell of the bilinear sample and the z clamp of the warp (the pixel and the four
taps of both cells); the clamp(0, 1) of L1 and SSIM, abs at 0 and the depth-ratio clamp (the pixel, and the 3x3
window of an SSIM output); the sign of a neighbour difference of the smoothness term (both pixels).  The excluded
fraction must stay below MAX_EXCLUDED.  Nothing is excluded by the size of its gradient.

Calibration: the largest kernel / eager ratio over all regions and cases, eager's error taken as in the bounds above
(the kernels compute in fp32 with approximate reciprocals on the gradient path, eager with IEEE division):

    emulator (x86-64, ARITH_CPU flavour):  rel-L2 ratio 1.52, max ratio 2.10; images under 16 pixels 5.91 / 6.08

RATIO_L2 = 2 and RATIO_MAX = 4 leave room for other seeds without hiding a wrong region: a dropped reflection
duplicate, a skipped tile column, a dropped scatter tap or a reversed tie rule moves a region's error by orders of
magnitude.
"""
import os

import pytest
import torch
import torch.nn.functional as F

from emu_lib import emu
from oracle import ref_torch as O
from tcsfm_b200 import _cabi, losses, ops, pft, stn, synth, train_mono

RATIO_L2 = 2.0
RATIO_MAX = 4.0
FEW_PIXELS = 16
RATIO_FEW = 8.0
FLOOR = 1e-7
# The smoothness gradient is scaled as a whole by 1 / mean(disp), and the kernel forms the mean from an fp32 sum of
# block partials added with atomics, where eager reduces pairwise.  At 16x376x1242 that leaves a uniform 3.4e-7
# (every region alike) against eager's 1.2e-7; a few ulps of the sum, so the term gets a floor of four ulps.
SMOOTH_FLOOR = 4 * 2.0 ** -23
MAX_EXCLUDED = 1e-3
WARP_CHUNK = 256 * 4          # kWarpThreads * kWarpBwdPix of csrc/warp_kernels.cu
REPORT = os.environ.get("TCSFM_F64_REPORT")   # a file to append every region's figures to


@pytest.fixture()
def emu_ops(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)


# ---------------------------------------------------------------------------------------------------- the helper
def regions(h, w, tiled=False, chunk=None):
    """Boolean [H,W] masks of the regions that exist at this shape; each one is non-empty."""
    y = torch.arange(h).view(h, 1)
    x = torch.arange(w).view(1, w)
    out = {"border": ((y < 2) | (y >= h - 2)) | ((x < 2) | (x >= w - 2)),
           "corners": ((y == 0) | (y == h - 1)) & ((x == 0) | (x == w - 1))}
    interior = ~out["border"]
    if tiled:
        seams = ((x % 64 == 0) | (x % 64 == 63)) | ((y % 16 == 0) | (y % 16 == 15))
        out["seams"] = seams.expand(h, w)
        interior = interior & ~seams
        if w % 64 or h % 16:
            out["partial_tile"] = ((x >= w // 64 * 64) & (w % 64 != 0)) | ((y >= h // 16 * 16) & (h % 16 != 0))
    if chunk:
        flat = y * w + x
        out["chunk_edges"] = (flat % chunk < 32) | (flat % chunk >= chunk - 32)
        if (h * w) % chunk:
            out["tail_chunk"] = flat >= (h * w) // chunk * chunk
    if h > 4 and w > 4:
        out["interior"] = interior
    for name, m in out.items():
        assert m.any(), "region %s is empty at %dx%d" % (name, h, w)
    return out


def run(fn, inputs, leaves, upstream, dtype):
    """fn(dict of tensors) -> tuple of outputs; the gradients of sum(output * upstream) w.r.t. `leaves`, with every
    floating-point input and upstream tensor converted to `dtype`."""
    x = {k: v.detach().to(dtype).requires_grad_(k in leaves) if torch.is_tensor(v) and v.is_floating_point() else v
         for k, v in inputs.items()}
    outs = fn(x)
    total = sum((o * u.to(dtype)).sum() for o, u in zip(outs, upstream) if o is not None and u is not None)
    total.backward()
    return {k: x[k].grad for k in leaves}


def compare(tag, name, got, e32, r64, regs, keep=None, floor=FLOOR):
    """Asserts the per-region bounds of the module docstring for one gradient tensor.  `regs`: region masks that
    broadcast against it; `keep`: entries left after the discontinuity exclusion (broadcasts too)."""
    r64 = r64.detach()
    got = torch.zeros_like(r64) if got is None else got.detach().to(r64.dtype)
    e32 = torch.zeros_like(r64) if e32 is None else e32.detach().to(r64.dtype)
    kept = torch.ones_like(r64, dtype=torch.bool) if keep is None else keep.to(r64.device).expand_as(r64)
    whole = r64[kept], e32[kept] - r64[kept]
    rel_e = whole[1].norm().item() / max(whole[0].norm().item(), 1e-300)
    maxrel_e = whole[1].abs().max().item() / max(whole[0].abs().max().item(), 1e-300)
    for rname, m in regs.items():
        m = m.to(r64.device).expand_as(r64) & kept
        assert m.any(), (tag, name, rname, "nothing left after the exclusion")
        ref = r64[m]
        dk, de = got[m] - ref, e32[m] - ref
        assert torch.isfinite(dk).all(), (tag, name, rname, "non-finite kernel gradient")
        l2k, l2e, l2r = dk.norm().item(), de.norm().item(), ref.norm().item()
        mk, me, mr = dk.abs().max().item(), de.abs().max().item(), ref.abs().max().item()
        l2e, me = max(l2e, rel_e * l2r), max(me, maxrel_e * mr)
        line = "%s %s %s: rel-L2 kernel %.3e eager %.3e (ratio %.2f), max kernel %.3e eager %.3e (ratio %.2f)" % (
            tag, name, rname, l2k / max(l2r, 1e-300), l2e / max(l2r, 1e-300), l2k / max(l2e, 1e-300),
            mk / max(mr, 1e-300), me / max(mr, 1e-300), mk / max(me, 1e-300))
        if REPORT:
            with open(REPORT, "a") as f:
                f.write(line + "\n")
        few = r64.dim() == 4 and r64.shape[-2] * r64.shape[-1] < FEW_PIXELS
        assert l2k <= (RATIO_FEW if few else RATIO_L2) * l2e + floor * l2r, line
        assert mk <= (RATIO_FEW if few else RATIO_MAX) * me + floor * mr, line


def excluded_fraction_ok(tag, *keeps):
    for keep in keeps:
        frac = 1.0 - keep.float().mean().item()
        assert frac <= MAX_EXCLUDED, (tag, "excluded fraction %.2e" % frac)


def dilate3(bad):
    """[...,H,W] bool -> every pixel within the 3x3 window of a bad one (the reflected cells of a window are inside it)."""
    shape = bad.shape
    t = bad.reshape(-1, 1, shape[-2], shape[-1]).double()
    return (F.max_pool2d(t, 3, 1, 1) > 0).reshape(shape)


def ssim_raw(x, y):
    """(1 - SSIM) / 2 before the clamp: the op sequence of O.ssim_dissimilarity, so fp32 rounds as eager does."""
    x = F.pad(x, (1, 1, 1, 1), mode="reflect")
    y = F.pad(y, (1, 1, 1, 1), mode="reflect")
    mu_x, mu_y = F.avg_pool2d(x, 3, 1), F.avg_pool2d(y, 3, 1)
    sigma_x = F.avg_pool2d(x ** 2, 3, 1) - mu_x ** 2
    sigma_y = F.avg_pool2d(y ** 2, 3, 1) - mu_y ** 2
    sigma_xy = F.avg_pool2d(x * y, 3, 1) - mu_x * mu_y
    num = (2 * mu_x * mu_y + O.SSIM_C1) * (2 * sigma_xy + O.SSIM_C2)
    den = (mu_x ** 2 + mu_y ** 2 + O.SSIM_C1) * (sigma_x + sigma_y + O.SSIM_C2)
    return (1 - num / den) / 2


def clamp_branch(v):
    """The branch torch.clamp(v, 0, 1)'s backward takes: 0 below, 1 inside (bounds included), 2 above."""
    return torch.where(v < 0, 0, torch.where(v <= 1, 1, 2))


def ssim_flips(x, y):
    """SSIM outputs whose clamp takes another branch in fp32 than in float64 ([N,C,H,W] bool)."""
    return clamp_branch(ssim_raw(x.float(), y.float())) != clamp_branch(ssim_raw(x.double(), y.double()))


# ---------------------------------------------------------------------------------------------------- warp
def warp_decisions(depth, pose, K, dtype):
    """The discrete choices of inverse_warp2 per target pixel [B,H,W]: z clamp, out-of-view overwrite per axis (the
    valid mask follows from the two) and the floor cell of the bilinear sample (O.project_normalised's arithmetic)."""
    d, p, k = depth.detach().to(dtype), pose.detach().to(dtype), K.detach().to(dtype)
    b, _, h, w = d.shape
    cam = O.backproject(d.squeeze(1), k.inverse())
    proj = k @ O.pose_to_matrix(p[:, 0:6])
    pc = proj[:, :, :3] @ cam.reshape(b, 3, -1)
    pc = pc + proj[:, :, -1:]
    z = pc[:, 2].clamp(min=1e-3)
    xn = 2 * (pc[:, 0] / z) / (w - 1) - 1
    yn = 2 * (pc[:, 1] / z) / (h - 1) - 1
    xm, ym = (xn > 1) | (xn < -1), (yn > 1) | (yn < -1)
    xn, yn = torch.where(xm, torch.full_like(xn, 2), xn), torch.where(ym, torch.full_like(yn, 2), yn)
    ix, iy = ((xn + 1) * w - 1) / 2, ((yn + 1) * h - 1) / 2
    out = {"z": pc[:, 2] >= 1e-3, "xm": xm, "ym": ym, "x0": ix.floor().long(), "y0": iy.floor().long()}
    return {key: v.reshape(b, h, w) for key, v in out.items()}


def warp_exclusions(depth, pose, K):
    """(target pixels, source pixels) to keep, [B,1,H,W] each: a target pixel whose decisions differ between fp32
    and float64 is dropped from g_depth, and the four taps of both of its cells from g_img / g_ref_depth."""
    a, c = warp_decisions(depth, pose, K, torch.float32), warp_decisions(depth, pose, K, torch.float64)
    bad = torch.zeros_like(a["z"])
    for key in a:
        bad |= a[key] != c[key]
    b, h, w = bad.shape
    src_bad = torch.zeros(b * h * w, dtype=torch.bool, device=bad.device)
    bidx = torch.arange(b, device=bad.device).view(b, 1, 1).expand(b, h, w)
    for dec in (a, c):
        for dy in (0, 1):
            for dx in (0, 1):
                xs, ys = dec["x0"] + dx, dec["y0"] + dy
                hit = bad & (xs >= 0) & (xs < w) & (ys >= 0) & (ys < h)
                src_bad[(bidx * h * w + ys * w + xs)[hit]] = True
    return ~bad.unsqueeze(1), ~src_bad.view(b, 1, h, w)


def warp_scene(b, h, w, mode, seed, device):
    """make_frames plus a pose that puts part of the image out of view ("wide") or behind the camera ("behind")."""
    fr = synth.make_frames(b, h, w, seed=seed, yaw=0.02, device=device, intrinsics=synth.scaled_intrinsics(h, w))
    pose = -fr["poses"][0]
    if mode == "wide":          # a band of about 13 % of every image leaves the view on one side
        pose = pose + torch.tensor([0.04, 0.0, 0.0, 0.0, 0.06, 0.0], device=device)
    elif mode == "behind":      # the camera moves past the nearest points: ~0.5 % behind it (z clamp), ~75 % out of view
        pose = pose + torch.tensor([0.0, 0.0, -0.1, 0.0, 0.0, 0.0], device=device)
    return fr, pose.contiguous()


def check_warp(b, h, w, mode, entry, device, seed=3):
    """stn.inverse_warp2 / inverse_warp2_stacked -> InverseWarp2Fn -> warp_bwd_kernel: g_depth, g_ref_depth, g_img and
    the pose (through K @ [R|t]).  The image is the channel slice [:, 3:6] of a six-channel stack, as the callers pass
    it; `entry` "stacked" / "stacked_nodepth" also takes the fused next pose-net input with need_depths True / False."""
    fr, pose = warp_scene(b, h, w, mode, seed, device)
    six = torch.cat([fr["target"], fr["sources"][0]], 1)
    inputs = {"six": six, "depth": fr["depths"][0], "ref_depth": fr["depths"][1], "pose": pose, "K": fr["K"],
              "tgt": fr["target"]}
    gen = torch.Generator().manual_seed(seed + 7)
    up = [torch.randn(b, c, h, w, generator=gen).to(device) for c in (3, 1, 1, 6)]
    need_depths = entry != "stacked_nodepth"

    def kernel(x):
        if entry == "plain":
            pim, _, pd, cd = stn.inverse_warp2(x["six"][:, 3:6], x["depth"], x["ref_depth"], x["pose"], x["K"])
            return pim, pd, cd
        kinv = stn.inverse_intrinsics(x["K"])
        pim, _, pd, cd, stack = stn.inverse_warp2_stacked(x["six"][:, 3:6], x["depth"], x["ref_depth"], x["pose"], x["K"],
                                                          kinv, x["tgt"], need_depths=need_depths)
        return pim, pd, cd, stack

    def oracle(x):
        pim, valid, pd, cd = O.inverse_warp2(x["six"][:, 3:6], x["depth"], x["ref_depth"], x["pose"], x["K"])
        if entry == "plain":
            return pim, pd, cd
        stack = torch.cat([x["tgt"] * valid, pim], 1)
        return (pim, pd, cd, stack) if need_depths else (pim, None, None, stack)

    leaves = ("six", "depth", "ref_depth", "pose") if need_depths else ("six", "depth", "pose")
    got = run(kernel, inputs, leaves, up, torch.float32)
    e32 = run(oracle, inputs, leaves, up, torch.float32)
    r64 = run(oracle, inputs, leaves, up, torch.float64)
    keep_t, keep_s = warp_exclusions(fr["depths"][0], pose, fr["K"])
    tag = "warp %dx%dx%d %s %s" % (b, h, w, mode, entry)
    excluded_fraction_ok(tag, keep_t, keep_s)
    plane = regions(h, w)
    compare(tag, "g_depth", got["depth"], e32["depth"], r64["depth"], regions(h, w, chunk=WARP_CHUNK), keep_t)
    compare(tag, "g_img", got["six"], e32["six"], r64["six"], plane, keep_s)
    if need_depths:
        compare(tag, "g_ref_depth", got["ref_depth"], e32["ref_depth"], r64["ref_depth"], plane, keep_s)
    compare(tag, "g_pose", got["pose"], e32["pose"], r64["pose"], {"all": torch.ones((), dtype=torch.bool)})


EMU_WARP = [(1, 2, 2, "fwd", "plain"), (1, 3, 5, "fwd", "plain"), (2, 17, 65, "wide", "plain"),
            (2, 33, 130, "behind", "plain"), (1, 16, 64, "wide", "plain"), (2, 33, 130, "wide", "stacked"),
            (2, 17, 65, "behind", "stacked_nodepth"), (1, 33, 130, "wide", "stacked")]


@pytest.mark.parametrize("case", EMU_WARP, ids=lambda c: "%dx%dx%d-%s-%s" % c)
def test_warp_backward_vs_f64(emu_ops, case):
    check_warp(*case, device="cpu")


GPU_WARP = [(6, 192, 640, "wide", "plain"), (1, 192, 640, "wide", "plain"), (16, 376, 1242, "behind", "plain"),
            (1, 376, 1242, "behind", "plain"), (24, 50, 77, "wide", "stacked"), (1, 50, 77, "wide", "stacked_nodepth"),
            (6, 511, 513, "behind", "stacked_nodepth"), (2, 720, 1280, "wide", "stacked")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_WARP, ids=lambda c: "%dx%dx%d-%s-%s" % c)
def test_warp_backward_vs_f64_cuda(case):
    check_warp(*case, device="cuda:0")


# ---------------------------------------------------------------------------------------------------- photo
def check_photo(b, h, w, device, seed=5):
    """train_mono.photometric_error_maps -> PhotoErrorFn -> photo_bwd_kernel: g_rec, g_pd, g_cd.  The inputs are one
    warp of a stacked batch (so the projected depth is 0 on the out-of-view band, as in solve_pose_iteratively)."""
    fr, pose = warp_scene(b, h, w, "wide", seed, device)
    imgs = torch.cat([fr["target"], fr["sources"][0]], 1)
    with torch.no_grad():
        rec, _, pd, cd = O.inverse_warp2(imgs[:, 3:6], fr["depths"][0], fr["depths"][1], pose, fr["K"])
    gen = torch.Generator().manual_seed(seed + 1)
    up = [torch.rand(b, 1, h, w, generator=gen).to(device), torch.randn(b, 1, h, w, generator=gen).to(device)]
    inputs = {"imgs": imgs, "rec": rec, "pd": pd, "cd": cd}
    leaves = ("rec", "pd", "cd")

    def kernel(x):
        _, diff, _, weight = train_mono.photometric_error_maps(x["imgs"], x["rec"], x["pd"], x["cd"])
        return diff, weight

    def oracle(x):
        _, diff, _, weight = O.pft_error_maps(x["imgs"], x["rec"], x["pd"], x["cd"])
        return diff, weight

    got = run(kernel, inputs, leaves, up, torch.float32)
    e32 = run(oracle, inputs, leaves, up, torch.float32)
    r64 = run(oracle, inputs, leaves, up, torch.float64)
    # decisions: SSIM clamp (3x3 window of g_rec), L1 clamp and sign (the pixel), depth-ratio clamp and sign (the pixel)
    tgt = imgs[:, 0:3]
    bad = dilate3(ssim_flips(tgt, rec).any(1, keepdim=True))
    d32, d64 = rec.float() - tgt.float(), rec.double() - tgt.double()
    bad |= ((torch.sign(d32) != torch.sign(d64)) | (clamp_branch(d32.abs()) != clamp_branch(d64.abs()))).any(1, keepdim=True)
    r32 = (cd - pd).abs() / (cd + pd)
    r64_ = (cd.double() - pd.double()).abs() / (cd.double() + pd.double())
    bad_w = (clamp_branch(r32) != clamp_branch(r64_)) | (torch.sign(cd - pd) != torch.sign(cd.double() - pd.double()))
    tag = "photo %dx%dx%d" % (b, h, w)
    excluded_fraction_ok(tag, ~bad, ~bad_w)
    reg = regions(h, w, tiled=True)
    compare(tag, "g_rec", got["rec"], e32["rec"], r64["rec"], reg, ~bad)
    compare(tag, "g_pd", got["pd"], e32["pd"], r64["pd"], reg, ~bad_w)
    compare(tag, "g_cd", got["cd"], e32["cd"], r64["cd"], reg, ~bad_w)


EMU_SHAPES = [(1, 2, 2), (1, 3, 5), (2, 17, 65), (2, 33, 130), (1, 16, 64)]
GPU_SHAPES = [(6, 192, 640), (16, 376, 1242), (24, 50, 77), (6, 511, 513), (2, 720, 1280)]


@pytest.mark.parametrize("shape", EMU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_photo_backward_vs_f64(emu_ops, shape):
    check_photo(*shape, device="cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", GPU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_photo_backward_vs_f64_cuda(shape):
    check_photo(*shape, device="cuda:0")


# ---------------------------------------------------------------------------------------------------- SSIM
def ssim_inputs(b, c, h, w, kind, device, seed):
    """'textured': two independent images; 'smooth': a smooth disparity map and 0.9 of it + 0.02 (the depth-init
    term of the PFT loss: variances of ~1e-5 out of E[x^2] - mu^2, where fp32 eager itself is ~6e-4 off float64)."""
    gen = torch.Generator().manual_seed(seed)
    if kind == "textured":
        x, y = torch.rand(b, c, h, w, generator=gen), torch.rand(b, c, h, w, generator=gen)
    else:
        x = synth.make_frames(b, h, w, seed=seed)["disps"][0].repeat(1, c, 1, 1)
        y = x * 0.9 + 0.02
    return x.to(device), y.to(device)


def check_ssim(b, c, h, w, kind, mean, device, seed=9):
    """losses.SSIM_Loss -> SsimFn -> ssim_bwd_kernel (g_x, g_y), or ops.SsimMeanFn -> ssim_mean_bwd (g_x, y detached
    as in the depth-init term)."""
    x, y = ssim_inputs(b, c, h, w, kind, device, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    if mean:
        up = [torch.full((1,), 0.37).to(device)]
        leaves = ("x",)
        kernel = lambda v: (ops.SsimMeanFn.apply(v["x"], v["y"]),)              # noqa: E731
        oracle = lambda v: (O.ssim_dissimilarity(v["x"], v["y"]).mean().reshape(1),)   # noqa: E731
    else:
        up = [torch.randn(b, c, h, w, generator=gen).to(device)]
        leaves = ("x", "y")
        kernel = lambda v: (losses.SSIM_Loss()(v["x"], v["y"]),)                 # noqa: E731
        oracle = lambda v: (O.ssim_dissimilarity(v["x"], v["y"]),)               # noqa: E731
    inputs = {"x": x, "y": y}
    got = run(kernel, inputs, leaves, up, torch.float32)
    e32 = run(oracle, inputs, leaves, up, torch.float32)
    r64 = run(oracle, inputs, leaves, up, torch.float64)
    keep = ~dilate3(ssim_flips(x, y))
    tag = "ssim%s %dx%dx%dx%d %s" % ("_mean" if mean else "", b, c, h, w, kind)
    excluded_fraction_ok(tag, keep)
    reg = regions(h, w, tiled=True)
    for k in leaves:
        compare(tag, "g_" + k, got[k], e32[k], r64[k], reg, keep)


@pytest.mark.parametrize("mean", [False, True], ids=["map", "mean"])
@pytest.mark.parametrize("kind", ["textured", "smooth"])
@pytest.mark.parametrize("shape", EMU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_ssim_backward_vs_f64(emu_ops, shape, kind, mean):
    b, h, w = shape
    check_ssim(b, 3 if kind == "textured" else 1, h, w, kind, mean, device="cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("mean", [False, True], ids=["map", "mean"])
@pytest.mark.parametrize("kind", ["textured", "smooth"])
@pytest.mark.parametrize("shape", GPU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_ssim_backward_vs_f64_cuda(shape, kind, mean):
    b, h, w = shape
    check_ssim(b, 3 if kind == "textured" else 1, h, w, kind, mean, device="cuda:0")


# ---------------------------------------------------------------------------------------------------- smoothness
def check_smooth(b, h, w, device, img_slice=False, seed=4):
    """losses.get_smooth_loss -> SmoothLossFn -> smooth_* (the two-pass mean normalisation).  The loss is an L1 norm of
    neighbour differences of the normalised disparity.  Exact ties between neighbours are placed on purpose: their
    difference is 0 in every precision and abs at 0 has no gradient, so the kernel must give none either (nvcc's FMA
    contraction of n(p) - d(q) / m once turned them into a rounding residue with a full-size sign).  A pair whose
    difference changes sign between fp32 and float64, or is not 0 but within the fp32 rounding of the normalisation
    (4 ulp, where the kernel's rounded reciprocal may decide it differently from eager's division), takes another
    branch of abs; both of its pixels are excluded."""
    fr = synth.make_frames(b, h, w, seed=seed, device=device)
    img = torch.cat([fr["sources"][0], fr["target"]], 1)[:, 3:6] if img_slice else fr["target"]
    gen = torch.Generator().manual_seed(seed)
    disp = fr["disps"][0].cpu()
    disp[..., :, 1:] = torch.where(torch.rand(b, 1, h, w - 1, generator=gen) < 0.03, disp[..., :, :-1], disp[..., :, 1:])
    disp[..., 1:, :] = torch.where(torch.rand(b, 1, h - 1, w, generator=gen) < 0.03, disp[..., :-1, :], disp[..., 1:, :])
    fr["disps"][0] = disp.to(device)
    inputs = {"disp": fr["disps"][0], "img": img}
    up = [torch.full((), 1.7).to(device)]
    got = run(lambda x: (losses.get_smooth_loss(x["disp"], x["img"]),), inputs, ("disp",), up, torch.float32)
    e32 = run(lambda x: (O.smooth_loss(x["disp"], x["img"]),), inputs, ("disp",), up, torch.float32)
    r64 = run(lambda x: (O.smooth_loss(x["disp"], x["img"]),), inputs, ("disp",), up, torch.float64)

    def norm(dtype):
        d = fr["disps"][0].to(dtype)
        return d / (d.mean(2, True).mean(3, True) + 1e-7)
    n32, n64 = norm(torch.float32), norm(torch.float64)
    bad = torch.zeros_like(n64, dtype=torch.bool)
    for dim in (2, 3):
        a32, a64 = n32.diff(dim=dim), n64.diff(dim=dim)
        band = 4 * torch.finfo(torch.float32).eps * torch.maximum(n64.narrow(dim, 0, a64.shape[dim]).abs(),
                                                                  n64.narrow(dim, 1, a64.shape[dim]).abs())
        flip = (torch.sign(a32) != torch.sign(a64)) | ((a64 != 0) & (a64.abs() <= band))
        lo = bad.narrow(dim, 0, flip.shape[dim])
        hi = bad.narrow(dim, 1, flip.shape[dim])
        lo |= flip
        hi |= flip
    tag = "smooth %dx%dx%d%s" % (b, h, w, " slice" if img_slice else "")
    excluded_fraction_ok(tag, ~bad)
    compare(tag, "g_disp", got["disp"], e32["disp"], r64["disp"], regions(h, w), ~bad, floor=SMOOTH_FLOOR)


@pytest.mark.parametrize("shape", EMU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_smooth_backward_vs_f64(emu_ops, shape):
    check_smooth(*shape, device="cpu", img_slice=shape[1] == 33)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", GPU_SHAPES, ids=lambda s: "%dx%dx%d" % s)
def test_smooth_backward_vs_f64_cuda(shape):
    check_smooth(*shape, device="cuda:0", img_slice=shape[0] == 6)


# ---------------------------------------------------------------------------------------------------- PFT reduction
PFT_VARIANTS = [
    {},
    {"diff_img_argmin": False},
    {"automasking": False},
    {"l_inverse_reconstruction": False},
    {"l_depth_consist": False},
    {"diff_img_argmin": False, "automasking": False, "l_depth_consist": False},
    {"l_depth_init": False, "l_smooth": True, "l_pose_consist": True},
]
PFT_OPTIONS = {"num_source_imgs": 2, "diff_img_argmin": True, "automasking": True, "l_inverse_reconstruction": True,
               "l_depth_consist": True, "l_depth_consist_weight": 0.15, "l_depth_init": True,
               "l_depth_init_weight": 0.1, "l_smooth": False, "l_smooth_weight": 0.05, "l_pose_consist": False,
               "plotting": False, "epochs": 20}


def check_pft(b, h, w, n_src, variant, device, seed=0):
    """pft.compute_optimization_loss with leaf maps (slices of one stack, the zero-copy path) -> PftReduceFn ->
    pft_reduce_bwd_kernel (g_diff, g_weight), plus the depth-init SSIM mean / smoothness term (g_tdisp).  Exact ties
    between sources are placed on purpose: torch.min routes the gradient to the first index holding the minimum.
    The maps are fp32 values, so every comparison of the reduction decides identically in fp32 and float64."""
    opts = dict(PFT_OPTIONS, num_source_imgs=n_src, **PFT_VARIANTS[variant])
    gen = torch.Generator().manual_seed(1000 * n_src + 10 * variant + seed)
    rows = 2 * n_src * b
    diff = torch.rand(rows, 1, h, w, generator=gen)
    for j in range(1, n_src):            # ties with source 0, and (3 sources) between sources 1 and 2
        sl = slice(j * b, (j + 1) * b)
        diff[sl] = torch.where(torch.rand(b, 1, h, w, generator=gen) < 0.3, diff[0:b], diff[sl])
        if j == 2:
            diff[sl] = torch.where(torch.rand(b, 1, h, w, generator=gen) < 0.3, diff[b:2 * b], diff[sl])
    aerr = torch.rand(rows, 1, h, w, generator=gen)
    aerr[0:b] = torch.where(torch.rand(b, 1, h, w, generator=gen) < 0.05, diff[0:b], aerr[0:b])   # ties with the min
    inputs = {"diff": diff, "valid": (torch.rand(rows, 1, h, w, generator=gen) < 0.8).float(), "aerr": aerr,
              "amask": (torch.rand(rows, 1, h, w, generator=gen) < 0.7).float(),
              "weight": torch.rand(rows, 1, h, w, generator=gen), "target": torch.rand(b, 3, h, w, generator=gen),
              "tdisp": synth.make_frames(b, h, w, seed=seed + 3)["disps"][0],
              "poses": torch.randn(rows, 3, 6, generator=gen) * 0.01}
    inputs = {k: v.to(device) for k, v in inputs.items()}
    split = n_src * b

    def with_fn(fn):
        def call(x):
            data = [{}, {}]
            for key, name in (("diff_img", "diff"), ("valid_mask", "valid"), ("auto_mask_error", "aerr"),
                              ("auto_mask", "amask"), ("weight_mask", "weight"), ("poses", "poses")):
                data[0][key], data[1][key] = x[name][:split], x[name][split:]
            return (fn(opts, x["target"], x["tdisp"], x["tdisp"].detach() * 0.9 + 0.02, data[0], data[1]),)
        return call

    leaves = ("diff", "weight", "tdisp")
    up = [torch.full((), 0.8).to(device)]
    got = run(with_fn(pft.compute_optimization_loss), inputs, leaves, up, torch.float32)
    e32 = run(with_fn(O.pft_window_loss), inputs, leaves, up, torch.float32)
    r64 = run(with_fn(O.pft_window_loss), inputs, leaves, up, torch.float64)
    tag = "pft %dx%dx%d S=%d variant %d" % (b, h, w, n_src, variant)
    reg = regions(h, w)
    compare(tag, "g_diff", got["diff"], e32["diff"], r64["diff"], reg)
    compare(tag, "g_weight", got["weight"], e32["weight"], r64["weight"], reg)
    if opts["l_depth_init"] or opts["l_smooth"]:
        td = inputs["tdisp"]
        keep = ~dilate3(ssim_flips(td, td * 0.9 + 0.02)) if opts["l_depth_init"] else None
        if keep is not None:
            excluded_fraction_ok(tag, keep)
        compare(tag, "g_tdisp", got["tdisp"], e32["tdisp"], r64["tdisp"], reg, keep,
                floor=SMOOTH_FLOOR if opts["l_smooth"] else FLOOR)


@pytest.mark.parametrize("n_src", [1, 2, 3])
@pytest.mark.parametrize("variant", range(len(PFT_VARIANTS)))
def test_pft_reduce_backward_vs_f64(emu_ops, n_src, variant):
    check_pft(2, 17, 65, n_src, variant, device="cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6, 192, 640, 2), (16, 376, 1242, 1), (24, 50, 77, 3)],
                         ids=lambda s: "%dx%dx%d-S%d" % s)
@pytest.mark.parametrize("variant", range(len(PFT_VARIANTS)))
def test_pft_reduce_backward_vs_f64_cuda(shape, variant):
    b, h, w, n_src = shape
    check_pft(b, h, w, n_src, variant, device="cuda:0")


# ---------------------------------------------------------------------------------------------------- chain rules
def check_chain_rules(n, device, seed=2):
    """ops.PoseProjFn (pose -> K @ [Rx Ry Rz | t], the sign folded in) and ops.DispToDepthFn (losses.disp_to_depth on
    CUDA tensors): g_pose and g_disp."""
    gen = torch.Generator().manual_seed(seed)
    pose = (torch.randn(n, 6, generator=gen) * torch.tensor([0.3, 0.3, 0.5, 0.1, 0.2, 0.1])).to(device)
    K = synth.scaled_intrinsics(192, 640).unsqueeze(0).repeat(n, 1, 1).to(device)
    up = [torch.randn(n, 3, 4, generator=gen).to(device)]
    inputs = {"pose": pose, "K": K}
    got = run(lambda x: (ops.PoseProjFn.apply(x["pose"], x["K"], -1.0),), inputs, ("pose",), up, torch.float32)
    e32 = run(lambda x: (x["K"] @ O.pose_to_matrix(-x["pose"]),), inputs, ("pose",), up, torch.float32)
    r64 = run(lambda x: (x["K"] @ O.pose_to_matrix(-x["pose"]),), inputs, ("pose",), up, torch.float64)
    compare("pose_proj n=%d" % n, "g_pose", got["pose"], e32["pose"], r64["pose"], {"all": torch.ones((), dtype=torch.bool)})

    h, w = 33, 130
    disp = synth.make_frames(n, h, w, seed=seed)["disps"][0].to(device)
    up = [torch.randn(n, 1, h, w, generator=gen).to(device)]
    lo, hi = synth.KITTI_DEPTH_RANGE
    got = run(lambda x: (ops.DispToDepthFn.apply(x["disp"], 1 / hi, 1 / lo),), {"disp": disp}, ("disp",), up, torch.float32)
    e32 = run(lambda x: (O.disp_to_depth(x["disp"], lo, hi)[1],), {"disp": disp}, ("disp",), up, torch.float32)
    r64 = run(lambda x: (O.disp_to_depth(x["disp"], lo, hi)[1],), {"disp": disp}, ("disp",), up, torch.float64)
    compare("disp_to_depth %dx%dx%d" % (n, h, w), "g_disp", got["disp"], e32["disp"], r64["disp"], regions(h, w))


@pytest.mark.parametrize("n", [1, 5])
def test_chain_rules_vs_f64(emu_ops, n):
    check_chain_rules(n, device="cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 24])
def test_chain_rules_vs_f64_cuda(n):
    check_chain_rules(n, device="cuda:0")
    # losses.disp_to_depth takes the kernel on CUDA fp32 tensors
    disp = torch.rand(n, 1, 40, 56, device="cuda:0")
    assert torch.equal(losses.disp_to_depth(disp, 0.06, 2.67)[1], O.disp_to_depth(disp, 0.06, 2.67)[1])
