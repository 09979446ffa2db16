"""Parity of the CUDA path (through the drop-in API -> ctypes -> C ABI ->
sm_100a kernels) against the oracle and the reference-generated golden vectors.

Tolerances (BASELINE.json north_star): loss <= 1e-5 relative, gradients <= 1e-4
relative (rel-L2), validity masks bit-exact.  Two arbiters are used:
  * golden fixtures / CPU oracle with the kernels' CPU arithmetic flavour;
  * the oracle run with eager PyTorch on the same GPU (the reference's production
    path) with the default CUDA flavour.
Nothing here reads /root/reference."""
import ctypes
import os

import pytest
import torch

import goldens
from goldens import Golden, rel_l2
from oracle import ref_torch as O
from tcsfm_b200 import _cabi, _lib, losses, ops, stn, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def leaf(t):
    return t.clone().detach().requires_grad_(True)


@pytest.fixture()
def cpu_flavour(monkeypatch):
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)


def test_native_library_is_loaded():
    lib = _lib.lib()
    assert lib.tcsfm_abi_version() == _cabi.ABI_VERSION
    with open("/proc/self/maps") as f:
        assert "libtcsfm_b200.so" in f.read()


# ---------------------------------------------------------------- golden vectors
# The fixtures were produced by the reference on a CPU, so K^-1 and K[R|t] are formed
# on the CPU here as well (CUDA's sin/cos/inverse differ from the CPU's in the last
# bit, which moves coordinates by ~1e-5 px); the kernels then run with the CPU
# arithmetic flavour and must reproduce the fixture masks bit for bit.
def cpu_projection(g, pose_key="in/pose0", sign=-1.0):
    cpu = Golden(g.name, "cpu")
    p0 = (sign * cpu.t(pose_key)).clone().requires_grad_(True)
    kinv, proj = stn.projection_matrices(p0, cpu.t("in/K"))
    return p0, kinv.to(DEV), proj.to(DEV)


@pytest.mark.parametrize("case", goldens.CASES)
def test_warp_vs_golden(cpu_flavour, case):
    g = Golden(case, DEV)
    fr = g.frames()
    p0, kinv, proj = cpu_projection(g)
    d0, d1 = leaf(fr["depths"][0]), leaf(fr["depths"][1])
    pim, vm, pd, cd = ops.InverseWarp2Fn.apply(fr["sources"][0], d0, d1, kinv, proj)
    assert torch.equal(vm, g.t("warp/valid_mask"))
    assert torch.equal(cd, g.t("warp/computed_depth"))
    assert (pim - g.t("warp/projected_img")).abs().max() < 1e-6
    assert (pd - g.t("warp/projected_depth")).abs().max() < 1e-6
    ((pim * g.t("in/g_img")).sum() + (pd * g.t("in/g_pd")).sum() + (cd * g.t("in/g_cd")).sum()).backward()
    assert rel_l2(d0.grad, g.t("warp/g_depth")) < 1e-4
    assert rel_l2(d1.grad, g.t("warp/g_ref_depth")) < 1e-4
    assert rel_l2(p0.grad, g.t("warp/g_pose").cpu()) < 1e-4


@pytest.mark.parametrize("case", goldens.CASES)
def test_ssim_vs_golden(cpu_flavour, case):
    g = Golden(case, DEV)
    x, y = leaf(g.t("in/target")), leaf(g.t("in/source0"))
    s = losses.SSIM_Loss()(x, y)
    assert torch.equal(s, g.t("ssim/map"))
    (s * g.t("in/g_img")).sum().backward()
    assert rel_l2(x.grad, g.t("ssim/g_x")) < 1e-4 and rel_l2(y.grad, g.t("ssim/g_y")) < 1e-4


@pytest.mark.parametrize("case", goldens.CASES)
@pytest.mark.parametrize("tag", ["train", "full", "noauto"])
def test_pairwise_vs_golden(cpu_flavour, case, tag):
    g = Golden(case, DEV)
    fr = g.frames()
    cfg = goldens.PAIR_CFGS[tag]
    p0, kinv, proj = cpu_projection(g)
    d0, d1 = leaf(fr["depths"][0]), leaf(fr["depths"][1])
    diff, vmask, l_rep, l_dep = ops.PairLossFn.apply((0.15, 0.85, losses._pair_flags(cfg)), 1, kinv, proj,
                                                     fr["target"], fr["sources"][0], d0, d1)
    diff, vmask, l_rep, l_dep = diff[0], vmask[0], l_rep[0], l_dep[0]
    assert torch.equal(vmask, g.t("pair_%s/valid_mask" % tag))
    assert torch.equal(diff, g.t("pair_%s/diff_img" % tag))
    ref_l = float(g.t("pair_%s/l_reprojection" % tag))
    assert abs(float(l_rep.detach()) - ref_l) <= 1e-5 * max(abs(ref_l), 1e-12)
    obj = l_rep + (diff * g.t("in/g_diff")).sum()
    if cfg["l_depth_consist"]:
        ref_d = float(g.t("pair_%s/l_depth" % tag))
        assert abs(float(l_dep.detach()) - ref_d) <= 1e-5 * max(abs(ref_d), 1e-12)
        obj = obj + 0.5 * l_dep
    obj.backward()
    assert rel_l2(d0.grad, g.t("pair_%s/g_depth" % tag)) < 1e-4
    assert rel_l2(p0.grad, g.t("pair_%s/g_pose" % tag).cpu()) < 1e-4
    if tag != "train":
        assert rel_l2(d1.grad, g.t("pair_%s/g_ref_depth" % tag)) < 1e-4


# ------------------------------------------------- same-device eager oracle, full sizes
SHAPES = [(4, 192, 640, 0.01, synth.KITTI_DEPTH_RANGE), (4, 256, 320, 0.04, synth.SCANNET_DEPTH_RANGE),
          (2, 256, 448, 0.02, synth.SCANNET_DEPTH_RANGE), (2, 376, 1242, 0.02, synth.KITTI_DEPTH_RANGE),
          (3, 50, 77, 0.08, synth.KITTI_DEPTH_RANGE)]


def frames(b, h, w, yaw, rng, seed=21):
    return synth.make_frames(b, h, w, seed=seed, yaw=yaw, depth_range=rng, device=DEV,
                             intrinsics=synth.scaled_intrinsics(h, w))


@pytest.mark.parametrize("shape", SHAPES)
def test_warp_vs_eager_cuda(shape):
    b, h, w, yaw, rng = shape
    fr = frames(b, h, w, yaw, rng)
    six = torch.cat([fr["target"], fr["sources"][0]], 1)           # callers pass imgs[:,3:6]
    up = [torch.randn(b, c, h, w, device=DEV) for c in (3, 1, 1)]
    res = []
    for fn in (O.inverse_warp2, stn.inverse_warp2):
        d0, d1, p0 = leaf(fr["depths"][0]), leaf(fr["depths"][1]), leaf(-fr["poses"][0])
        pim, vm, pd, cd = fn(six[:, 3:6], d0, d1, p0, fr["K"], 'zeros')
        ((pim * up[0]).sum() + (pd * up[1]).sum() + (cd * up[2]).sum()).backward()
        res.append((pim, vm, pd, cd, d0.grad, d1.grad, p0.grad))
    ref, got = res
    assert torch.equal(got[1], ref[1]), "valid mask differs on %d px" % int((got[1] != ref[1]).sum())
    assert torch.equal(got[3], ref[3])                               # computed depth, bit for bit
    assert torch.equal(got[0], ref[0]) and torch.equal(got[2], ref[2])      # warped image / depth, bit for bit
    assert rel_l2(got[4], ref[4]) < 1e-4
    assert rel_l2(got[5], ref[5]) < 1e-4
    assert rel_l2(got[6], ref[6]) < 1e-4


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("tag", ["train", "full"])
def test_compute_loss_vs_eager_cuda(shape, tag):
    b, h, w, yaw, rng = shape
    fr = frames(b, h, w, yaw, rng)
    cfg = dict(goldens.LOSS_CFGS[tag], min_depth=rng[0], max_depth=rng[1])
    res = []
    for impl in ("oracle", "cuda"):
        disps = [leaf(d) for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        dl = [[disps[0]], [disps[1]], [disps[2]]]
        if impl == "oracle":
            out = O.compute_loss(cfg, fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        else:
            out = losses.Compute_Loss(cfg)(fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        out["total"].sum().backward()
        res.append((out, disps, poses, poses_inv))
    (ro, rd, rp, rpi), (go, gd, gp, gpi) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)
    def grad(t):
        return t.grad if t.grad is not None else torch.zeros_like(t)
    for j in range(3):
        assert rel_l2(grad(gd[j]), grad(rd[j])) < 1e-4, ("disp", j, rel_l2(grad(gd[j]), grad(rd[j])))
    for j in range(2):
        assert rel_l2(grad(gp[j]), grad(rp[j])) < 1e-4, ("pose", j, rel_l2(grad(gp[j]), grad(rp[j])))
        assert rel_l2(grad(gpi[j]), grad(rpi[j])) < 1e-4, ("pose_inv", j, rel_l2(grad(gpi[j]), grad(rpi[j])))


@pytest.mark.parametrize("shape", [(16, 256, 320), (4, 256, 448), (3, 90, 130)])
@pytest.mark.parametrize("tag", ["train", "full"])
def test_compute_loss_single_source_vs_eager_cuda(shape, tag):
    """Config 3 (ScanNet pairs, S = 1): the per-pixel min-reprojection runs over one candidate."""
    b, h, w = shape
    fr = synth.make_frames(b, h, w, n_src=1, seed=31, depth_range=synth.SCANNET_DEPTH_RANGE, device=DEV,
                           intrinsics=synth.scaled_intrinsics(h, w, synth.SCANNET_K, (256, 320)))
    cfg = dict(goldens.LOSS_CFGS[tag], min_depth=synth.SCANNET_DEPTH_RANGE[0], max_depth=synth.SCANNET_DEPTH_RANGE[1])
    res = []
    for impl in ("oracle", "cuda"):
        disps = [[leaf(d)] for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        args = (fr["sources"], fr["target"], [poses, poses_inv], disps, fr["K"])
        out = O.compute_loss(cfg, *args) if impl == "oracle" else losses.Compute_Loss(cfg)(*args)
        out["total"].sum().backward()
        res.append((out, [d[0] for d in disps] + poses + poses_inv))
    (ro, rl), (go, gl) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)
    for i, (a, bb) in enumerate(zip(gl, rl)):
        ga = a.grad if a.grad is not None else torch.zeros_like(a)
        gb = bb.grad if bb.grad is not None else torch.zeros_like(bb)
        assert rel_l2(ga, gb) < 1e-4, (i, tuple(a.shape), rel_l2(ga, gb))


@pytest.mark.parametrize("shape", [(1, 1080, 1920), (2, 720, 1280), (48, 64, 96)])
def test_compute_loss_large_frames_and_batches_vs_eager_cuda(shape):
    """Frame sizes / batch sizes well outside the benchmark configurations (2 Mpx frames, B = 48)."""
    b, h, w = shape
    fr = frames(b, h, w, 0.0, synth.KITTI_DEPTH_RANGE, seed=17)
    cfg = dict(goldens.LOSS_CFGS["full"], min_depth=synth.KITTI_DEPTH_RANGE[0], max_depth=synth.KITTI_DEPTH_RANGE[1])
    res = []
    for impl in ("oracle", "cuda"):
        disps = [[leaf(d)] for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        args = (fr["sources"], fr["target"], [poses, poses_inv], disps, fr["K"])
        out = O.compute_loss(cfg, *args) if impl == "oracle" else losses.Compute_Loss(cfg)(*args)
        out["total"].sum().backward()
        res.append((out, [d[0] for d in disps] + poses + poses_inv))
    (ro, rl), (go, gl) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)
    for i, (a, bb) in enumerate(zip(gl, rl)):
        ga = a.grad if a.grad is not None else torch.zeros_like(a)
        gb = bb.grad if bb.grad is not None else torch.zeros_like(bb)
        assert rel_l2(ga, gb) < 1e-4, (i, tuple(a.shape), rel_l2(ga, gb))


@pytest.mark.parametrize("shape", [(4, 192, 640), (3, 90, 130)])
def test_compute_loss_three_sources_vs_eager_cuda(shape):
    """Three source frames: six pair groups per launch, three-way per-pixel min-reprojection."""
    b, h, w = shape
    fr = synth.make_frames(b, h, w, n_src=3, seed=41, depth_range=synth.KITTI_DEPTH_RANGE, device=DEV,
                           intrinsics=synth.scaled_intrinsics(h, w))
    cfg = dict(goldens.LOSS_CFGS["full"], min_depth=synth.KITTI_DEPTH_RANGE[0], max_depth=synth.KITTI_DEPTH_RANGE[1])
    res = []
    for impl in ("oracle", "cuda"):
        disps = [[leaf(d)] for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        args = (fr["sources"], fr["target"], [poses, poses_inv], disps, fr["K"])
        out = O.compute_loss(cfg, *args) if impl == "oracle" else losses.Compute_Loss(cfg)(*args)
        out["total"].sum().backward()
        res.append((out, [d[0] for d in disps] + poses + poses_inv))
    (ro, rl), (go, gl) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)
    for i, (a, bb) in enumerate(zip(gl, rl)):
        ga = a.grad if a.grad is not None else torch.zeros_like(a)
        gb = bb.grad if bb.grad is not None else torch.zeros_like(bb)
        assert rel_l2(ga, gb) < 1e-4, (i, tuple(a.shape), rel_l2(ga, gb))


@pytest.mark.parametrize("hw", [(192, 640), (376, 1242), (100, 333)])
def test_compute_loss_four_scales_vs_eager_cuda(hw):
    """Config 5 (num_scales = 4): the lower-scale disparities arrive at their own resolution and are
    nearest-upsampled inside the disp -> depth kernel; loss 1e-5, gradients (also of the low-resolution
    disparities) 1e-4 against the reference's interpolate + disp_to_depth on the same GPU."""
    h, w = hw
    fr = frames(2, h, w, 0.0, synth.KITTI_DEPTH_RANGE, seed=11)
    cfg = dict(goldens.LOSS_CFGS["full"], num_scales=4, min_depth=synth.KITTI_DEPTH_RANGE[0], max_depth=synth.KITTI_DEPTH_RANGE[1])
    pyramid = [[d] + [torch.nn.functional.avg_pool2d(d, 2 ** sc, ceil_mode=True) for sc in range(1, 4)] for d in fr["disps"]]
    res = []
    for impl in ("oracle", "cuda"):
        disps = [[leaf(t) for t in per_frame] for per_frame in pyramid]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        args = (fr["sources"], fr["target"], [poses, poses_inv], disps, fr["K"])
        out = O.compute_loss(cfg, *args) if impl == "oracle" else losses.Compute_Loss(cfg)(*args)
        out["total"].sum().backward()
        res.append((out, [t for per_frame in disps for t in per_frame] + poses + poses_inv))
    (ro, rl), (go, gl) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)
    for i, (a, bb) in enumerate(zip(gl, rl)):
        ga = a.grad if a.grad is not None else torch.zeros_like(a)
        gb = bb.grad if bb.grad is not None else torch.zeros_like(bb)
        assert ga.shape == gb.shape and rel_l2(ga, gb) < 1e-4, (i, tuple(a.shape), rel_l2(ga, gb))


@pytest.mark.parametrize("shape", SHAPES[:3])
def test_pair_masks_bit_exact_vs_eager_cuda(shape):
    b, h, w, yaw, rng = shape
    fr = frames(b, h, w, yaw, rng, seed=5)
    for tag in ("train", "full", "noauto"):
        cfg = goldens.PAIR_CFGS[tag]
        for j in range(2):
            args = (fr["target"], fr["sources"][j], fr["depths"][0], fr["depths"][1 + j], -fr["poses"][j], fr["K"])
            ref = O.pairwise_loss(cfg, *args)
            got = losses.Compute_Loss(cfg).compute_pairwise_loss(*args, 5)
            assert torch.equal(got[3], ref[3]), (tag, j, int((got[3] != ref[3]).sum()))
            assert torch.equal(got[2], ref[2])                               # diff_img, bit for bit


# ------------------------------------------------- size-independent properties, config-2 size
def test_properties_full_size():
    b, h, w = 8, 192, 640
    fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=0)
    cfg = goldens.FULL_CFG
    mod = losses.Compute_Loss(cfg)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], -fr["poses"][0], fr["K"])
    l_rep, l_dep, diff, mask, _ = mod.compute_pairwise_loss(*args, 5)
    # masks are 0/1, the reported means are the masked means of the returned maps
    assert set(torch.unique(mask).tolist()) <= {0.0, 1.0}
    assert mask.sum() > 10000
    ref_mean = (diff.double() * mask.double()).sum() / mask.double().sum()
    assert abs(float(l_rep) - float(ref_mean)) <= 1e-5 * float(ref_mean)
    assert (diff >= 0).all() and (diff <= 1).all()
    # determinism of the forward, linearity of the backward in the upstream gradient
    l2, _, diff2, mask2, _ = mod.compute_pairwise_loss(*args, 5)
    assert torch.equal(diff, diff2) and torch.equal(mask, mask2)
    d0 = leaf(fr["depths"][0])
    u, v = torch.randn_like(diff), torch.randn_like(diff)
    outs = []
    for up in (u, v, 2 * u - 3 * v):
        d0.grad = None
        _, _, dd, _, _ = mod.compute_pairwise_loss(fr["target"], fr["sources"][0], d0, fr["depths"][1], -fr["poses"][0], fr["K"], 5)
        (dd * up).sum().backward()
        outs.append(d0.grad.clone())
    assert rel_l2(outs[2], 2 * outs[0] - 3 * outs[1]) < 1e-5
    # fully out-of-view pose: empty mask -> the <=10000 rule returns exactly 0 and a zero gradient
    far = fr["poses"][0].clone()
    far[:, 0] = 1.0e4
    d0.grad = None
    l_far, _, _, m_far, _ = mod.compute_pairwise_loss(fr["target"], fr["sources"][0], d0, fr["depths"][1], far, fr["K"], 5)
    assert float(m_far.sum()) == 0 and float(l_far) == 0
    l_far.backward()
    assert float(d0.grad.abs().max()) == 0


def test_edge_cases_identity_and_clamped_depth():
    b, h, w = 2, 64, 96
    fr = frames(b, h, w, 0.0, synth.KITTI_DEPTH_RANGE, seed=3)
    zero_pose = torch.zeros(b, 6, device=DEV)
    a = O.inverse_warp2(fr["sources"][0], fr["depths"][0], fr["depths"][1], zero_pose, fr["K"])
    g = stn.inverse_warp2(fr["sources"][0], fr["depths"][0], fr["depths"][1], zero_pose, fr["K"])
    assert torch.equal(a[1], g[1]) and (a[0] - g[0]).abs().max() < 1e-6
    # points behind the camera: Z is clamped to 1e-3 (models/stn.py:218) and gets no gradient
    back = zero_pose.clone()
    back[:, 2] = -10.0
    d0r, d0g = leaf(fr["depths"][0]), leaf(fr["depths"][0])
    a = O.inverse_warp2(fr["sources"][0], d0r, fr["depths"][1], back, fr["K"])
    g = stn.inverse_warp2(fr["sources"][0], d0g, fr["depths"][1], back, fr["K"])
    assert torch.equal(a[1], g[1]) and torch.equal(a[3], g[3]) and float(g[3].max()) == pytest.approx(1e-3)
    a[3].sum().backward()
    g[3].sum().backward()
    assert torch.equal(d0r.grad, d0g.grad)


def test_pose_proj_bit_exact_vs_eager_cuda():
    """tcsfm_pose_proj_fwd reproduces `intrinsics @ pose_vec2mat(-pose)` (models/stn.py:259-262)
    bit for bit on the same GPU (sinf/cosf of the CUDA math library, k-ascending FMA chains)."""
    from tcsfm_b200 import _raw
    gen = torch.Generator().manual_seed(0)
    for n, bk in ((32, 8), (2, 2), (24, 6), (4096, 8), (1, 1)):
        pose = (0.3 * torch.randn(n, 6, generator=gen)).to(DEV)
        pose[0, 3:] = 0.0
        K = (torch.tensor(synth.KITTI_K).repeat(bk, 1, 1) + 0.01 * torch.rand(bk, 3, 3, generator=gen)).to(DEV)
        ref = K.repeat(n // bk, 1, 1) @ stn.pose_vec2mat(-pose)
        got = _raw.pose_proj_fwd(_lib.lib(), pose, K, -1.0, ops.pose_flags(n))
        assert torch.equal(got, ref), (n, int((got != ref).sum()))
        p = leaf(pose)
        gp = torch.randn(n, 3, 4, device=DEV)
        (K.repeat(n // bk, 1, 1) @ stn.pose_vec2mat(-p)).backward(gp)
        g_pose = _raw.pose_proj_bwd(_lib.lib(), pose, K, -1.0, gp)
        assert rel_l2(g_pose, p.grad) < 1e-5


def test_pft_window_trajectory_vs_oracle():
    """Four optimisation epochs of a PFT window (stand-in networks) through the fused path and
    through the oracle on the same GPU: loss trajectory within 1e-4 (SURVEY.md §4 integration)."""
    from tcsfm_b200 import pft_driver

    class OracleBackend:
        solve_pose_iteratively = staticmethod(O.iterative_pose)
        compute_optimization_loss = staticmethod(
            lambda opts, tgt, disp, init, fwd, inv: O.pft_window_loss(opts, tgt, disp, init, fwd, inv))
        disp_to_depth = staticmethod(O.disp_to_depth)

    b, h, w = 3, 96, 160
    fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=8)
    depth_net = synth.TinyDepthNet(seed=1).to(DEV)
    pose_net = synth.TinyPoseNet(seed=1).to(DEV)
    opts = {"epochs": 4}
    got = pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, iterations=3)
    ref = pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, iterations=3,
                                     backend=OracleBackend)
    assert got["losses"].shape == (4,)
    assert torch.allclose(got["losses"], ref["losses"], rtol=1e-4, atol=0), (got["losses"], ref["losses"])
    assert (got["disparity"] - ref["disparity"]).abs().max() < 1e-4


@pytest.mark.parametrize("hw", [(192, 640), (256, 320), (344, 677), (511, 513), (512, 512), (376, 1242)])
def test_batch_one_is_bit_exact_too(hw):
    """With batch 1 eager PyTorch's k=3 bmm switches kernels at 9*H*W <= 2^21 (no FMA below); the
    operators pick the matching arithmetic so masks stay bit-exact and gradients tight."""
    h, w = hw
    fr = frames(1, h, w, 0.02, synth.KITTI_DEPTH_RANGE, seed=13)
    args = (fr["sources"][0], fr["depths"][0], fr["depths"][1], -fr["poses"][0], fr["K"])
    ref, got = O.inverse_warp2(*args), stn.inverse_warp2(*args)
    for a, b_ in zip(got, ref):
        assert torch.equal(a, b_), (hw, int((a != b_).sum()))
    cfg = goldens.FULL_CFG
    res = []
    for impl in ("oracle", "cuda"):
        disps = [leaf(d) for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        dl = [[disps[0]], [disps[1]], [disps[2]]]
        if impl == "oracle":
            out = O.compute_loss(cfg, fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        else:
            out = losses.Compute_Loss(cfg)(fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        out["total"].sum().backward()
        res.append((out, disps, poses))
    (ro, rd, rp), (go, gd, gp) = res
    assert abs(float(go["total"].detach()) - float(ro["total"].detach())) <= 1e-5 * abs(float(ro["total"].detach()))
    for j in range(3):
        assert rel_l2(gd[j].grad, rd[j].grad) < 1e-4, (hw, j, rel_l2(gd[j].grad, rd[j].grad))


def test_pft_window_cuda_graph_matches_eager():
    """The whole optimisation epoch (stand-in networks + fused path + backward + Adam) replayed as
    a CUDA graph gives the same loss trajectory as eager execution."""
    from tcsfm_b200 import pft_driver
    b, h, w = 2, 64, 96
    fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=9)
    depth_net, pose_net = synth.TinyDepthNet(seed=3).to(DEV), synth.TinyPoseNet(seed=3).to(DEV)
    opts = {"epochs": 7}
    eager = pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, iterations=3)
    graph = pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, iterations=3,
                                       cuda_graph=True)
    assert graph["losses"].shape == eager["losses"].shape == (7,)
    assert torch.allclose(graph["losses"], eager["losses"], rtol=1e-4, atol=0), (graph["losses"], eager["losses"])


@pytest.mark.parametrize("depth_range", [synth.KITTI_DEPTH_RANGE, (0.1, 10.0)])
def test_disp_to_depth_vs_eager_cuda(depth_range):
    """disp_to_depth (utils/learning_helpers.py:77-86) as called per frame and epoch by PFT: both outputs bit-identical
    to the eager expression, gradient (through the depth and through the scaled disparity) within 1e-6."""
    fr = frames(6, 192, 640, 0.01, depth_range, seed=8)
    d_ref, d_got = leaf(fr["disps"][0]), leaf(fr["disps"][0])
    s_ref, z_ref = O.disp_to_depth(d_ref, *depth_range)
    s_got, z_got = losses.disp_to_depth(d_got, *depth_range)
    assert torch.equal(s_ref, s_got) and torch.equal(z_ref, z_got)
    g = torch.randn_like(z_ref)
    (z_ref * g + 0.3 * s_ref).sum().backward()
    (z_got * g + 0.3 * s_got).sum().backward()
    assert rel_l2(d_got.grad, d_ref.grad) < 1e-6, rel_l2(d_got.grad, d_ref.grad)


@pytest.mark.parametrize("shape", [(8, 192, 640), (3, 50, 77)])
def test_smooth_loss_vs_eager_cuda(shape):
    """get_smooth_loss (losses.py:43-61): value within 1e-5 of eager PyTorch; gradient within 1e-4
    away from the discontinuities.  The loss is an L1 norm of neighbour differences of the
    mean-normalised disparity: its gradient is sign(n_p - n_q), so a pair of neighbours that agree
    to the last few ulps flips by O(1) on any re-rounding of the mean (the reference's own
    fp32-vs-fp64 gradient differs the same way).  Such pairs are excluded from the comparison."""
    b, h, w = shape
    fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=4)
    d_ref, d_got = leaf(fr["disps"][0]), leaf(fr["disps"][0])
    six = torch.cat([fr["sources"][0], fr["target"]], 1)
    ref = O.smooth_loss(d_ref, six[:, 3:6])
    got = losses.get_smooth_loss(d_got, six[:, 3:6])
    assert abs(float(got.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach()))
    ref.backward()
    got.backward()
    d = fr["disps"][0].double()
    n = d / (d.mean(dim=(2, 3), keepdim=True) + 1e-7)
    tie = torch.zeros_like(n, dtype=torch.bool)
    near_x = (n[..., :, :-1] - n[..., :, 1:]).abs() < 1e-5
    near_y = (n[..., :-1, :] - n[..., 1:, :]).abs() < 1e-5
    tie[..., :, :-1] |= near_x
    tie[..., :, 1:] |= near_x
    tie[..., :-1, :] |= near_y
    tie[..., 1:, :] |= near_y
    assert tie.float().mean() < 0.01
    keep = ~tie
    assert rel_l2(d_got.grad[keep], d_ref.grad[keep]) < 1e-4
    # and the discontinuities do not dominate: the full gradient still agrees to a few 1e-3
    assert rel_l2(d_got.grad, d_ref.grad) < 2e-2


def test_pft_window_runner_reuses_graphs():
    """WindowRunner (graphs captured once, replayed for every later window) == optimize_window per window."""
    from tcsfm_b200 import pft_driver
    b, h, w = 2, 64, 96
    depth_net, pose_net = synth.TinyDepthNet(seed=5).to(DEV), synth.TinyPoseNet(seed=5).to(DEV)
    opts = {"epochs": 6}
    runner = pft_driver.WindowRunner(depth_net, pose_net, opts, iterations=3)
    for seed in (20, 21, 22):
        fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=seed)
        got = runner(fr["target"], fr["sources"], fr["K"])
        ref = pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, iterations=3)
        assert torch.allclose(got["losses"], ref["losses"], rtol=1e-4, atol=0), (seed, got["losses"], ref["losses"])
        assert (got["disparity"] - ref["disparity"]).abs().max() < 1e-4


@pytest.mark.parametrize("seed", list(range(40)))
def test_randomised_sweep_vs_eager_cuda(seed):
    """Random shapes (not multiples of the 64x16 tile), intrinsics, poses (up to ~10 deg and large
    translations: wide out-of-view bands, points behind the camera), depth ranges and batch sizes:
    every forward output bit for bit, gradients (incl. the sampled image's) within 1e-4."""
    gen = torch.Generator().manual_seed(1234 + seed)
    b = int(torch.randint(1, 5, (1,), generator=gen))
    h = int(torch.randint(18, 200, (1,), generator=gen))
    w = int(torch.randint(18, 300, (1,), generator=gen))
    fr = synth.make_frames(b, h, w, seed=100 + seed, yaw=0.02, device=DEV, intrinsics=synth.scaled_intrinsics(h, w))
    K = fr["K"].clone()
    K[:, 0, 0] *= float(0.6 + 0.8 * torch.rand(1, generator=gen))
    K[:, 1, 1] *= float(0.6 + 0.8 * torch.rand(1, generator=gen))
    K[:, 0, 1] = float(2.0 * torch.rand(1, generator=gen))                     # skew: K^-1 without exact zeros
    scale = torch.tensor([0.05, 0.05, 0.3, 0.05, 0.18, 0.05])
    pose = (torch.randn(b, 6, generator=gen) * scale).to(DEV)
    if seed % 3 == 0:
        pose[:, 2] = -3.0                                                       # many points behind the camera
    depth_scale = float(0.2 + 3.0 * torch.rand(1, generator=gen))
    src = leaf(fr["sources"][0])
    up = [torch.randn(b, c, h, w, device=DEV) for c in (3, 1, 1)]
    res = []
    for fn in (O.inverse_warp2, stn.inverse_warp2):
        s_ = leaf(src)
        d0, d1, p0 = leaf(fr["depths"][0] * depth_scale), leaf(fr["depths"][1] * depth_scale), leaf(pose)
        pim, vm, pd, cd = fn(s_, d0, d1, p0, K, 'zeros')
        ((pim * up[0]).sum() + (pd * up[1]).sum() + (cd * up[2]).sum()).backward()
        res.append((pim, vm, pd, cd, d0.grad, d1.grad, p0.grad, s_.grad))
    ref, got = res
    for i in range(4):
        assert torch.equal(got[i], ref[i]), (seed, i, int((got[i] != ref[i]).sum()))
    for i in range(4, 8):
        assert rel_l2(got[i], ref[i]) < 1e-4, (seed, i, rel_l2(got[i], ref[i]))
    cfg = goldens.FULL_CFG if seed % 2 else goldens.TRAIN_CFG
    args = (fr["target"], fr["sources"][0], fr["depths"][0] * depth_scale, fr["depths"][1] * depth_scale, pose, K)
    pr = O.pairwise_loss(cfg, *args)
    pg = losses.Compute_Loss(cfg).compute_pairwise_loss(*args, 5)
    assert torch.equal(pg[3], pr[3]) and torch.equal(pg[2], pr[2]), (seed, int((pg[3] != pr[3]).sum()))


# ------------------------------------------------- PFT block (train_mono.py:84-92, optimizer.py:45-97, helpers.py:8-23)
def _pft_stack(b, h, w, rng, seed, n_src=2):
    """The stacked tensors solve_pose_iteratively builds (train_mono.py:54-67) and one warp of them."""
    fr = frames(b, h, w, 0.02, rng, seed=seed) if n_src == 2 else \
        synth.make_frames(b, h, w, n_src=n_src, seed=seed, yaw=0.02, depth_range=rng, device=DEV,
                          intrinsics=synth.scaled_intrinsics(h, w))
    tgt = fr["target"].repeat(n_src, 1, 1, 1)
    src = torch.cat(fr["sources"], 0)
    imgs = torch.cat([torch.cat([tgt, src], 1), torch.cat([src, tgt], 1)], 0)
    td = fr["depths"][0].repeat(n_src, 1, 1, 1)
    sd = torch.cat(fr["depths"][1:], 0)
    depth, ref_depth = torch.cat([td, sd], 0), torch.cat([sd, td], 0)
    poses = torch.cat(list(fr["poses"]) + list(fr["poses_inv"]), 0)
    K = fr["K"].repeat(2 * n_src, 1, 1)
    with torch.no_grad():
        rec, valid, pd, cd = O.inverse_warp2(imgs[:, 3:6], depth, ref_depth, -poses, K, 'zeros')
    return fr, imgs, rec, valid, pd, cd


@pytest.mark.parametrize("shape", [(6, 192, 640, synth.KITTI_DEPTH_RANGE), (16, 256, 320, synth.SCANNET_DEPTH_RANGE),
                                   (2, 50, 77, synth.KITTI_DEPTH_RANGE)])
def test_photo_error_maps_bit_exact_vs_eager_cuda(shape):
    """tcsfm_photo_fwd: auto_mask_error, diff_img, auto_mask, weight_mask of train_mono.py:84-92 at the stacked
    batch 2*S*B (24 at 192x640, 32 at 256x320), bit for bit against eager PyTorch on the same GPU; tcsfm_photo_bwd:
    gradients w.r.t. the reconstruction and the two depths within 1e-4."""
    from tcsfm_b200 import train_mono
    b, h, w, rng = shape
    n_src = 2 if h != 256 else 1
    _, imgs, rec, _, pd, cd = _pft_stack(b, h, w, rng, seed=31, n_src=n_src)
    up_d, up_w = torch.rand_like(pd), torch.randn_like(pd)
    res = []
    for fn in (O.pft_error_maps, train_mono.photometric_error_maps):
        r, p, c = leaf(rec), leaf(pd), leaf(cd)
        aerr, diff, amask, weight = fn(imgs, r, p, c)
        ((diff * up_d).sum() + (weight * up_w).sum()).backward()
        res.append((aerr, diff, amask, weight, r.grad, p.grad, c.grad))
    ref, got = res
    for name, a, b_ in zip(("auto_mask_error", "diff_img", "auto_mask", "weight_mask"), got[:4], ref[:4]):
        assert torch.equal(a.reshape(b_.shape), b_), (name, int((a.reshape(b_.shape) != b_).sum()))
    assert not got[2].requires_grad
    for name, a, b_ in zip(("g_rec", "g_proj_depth", "g_comp_depth"), got[4:], ref[4:]):
        assert rel_l2(a, b_) < 1e-4, (name, rel_l2(a, b_))


@pytest.mark.parametrize("shape", [(6, 192, 640, synth.KITTI_DEPTH_RANGE, 2), (16, 256, 320, synth.SCANNET_DEPTH_RANGE, 1),
                                   (3, 96, 160, synth.KITTI_DEPTH_RANGE, 3)])
@pytest.mark.parametrize("variant", [{}, {"diff_img_argmin": False}, {"automasking": False, "l_depth_consist": False},
                                     {"l_inverse_reconstruction": False}])
def test_compute_optimization_loss_vs_eager_cuda(shape, variant):
    """solve_pose_iteratively(return_errors=True) + compute_optimization_loss (optimizer.py:45-97) through the
    fused kernels (warp + stack, photometric maps, tcsfm_pft_reduce, SSIM mean) against the oracle on the same
    GPU: PFT auto-mask / valid masks bit-exact, loss within 1e-5, gradients w.r.t. the depths within 1e-4."""
    from tcsfm_b200 import pft, train_mono
    b, h, w, rng, n_src = shape
    fr = synth.make_frames(b, h, w, n_src=n_src, seed=17, yaw=0.01, depth_range=rng, device=DEV,
                           intrinsics=synth.scaled_intrinsics(h, w))
    net = synth.TinyPoseNet(seed=5).to(DEV)
    opts = dict(goldens.PFT_OPTIONS, num_source_imgs=n_src, **variant)
    res = []
    for impl in ("oracle", "cuda"):
        dl = [leaf(d) for d in fr["depths"]]
        tdisp = leaf(fr["disps"][0])
        if impl == "oracle":
            poses, poses_inv, out = O.iterative_pose(3, dl, net, fr["target"], fr["sources"], fr["K"], return_errors=True)
            loss = O.pft_window_loss(opts, fr["target"], tdisp, fr["disps"][0] * 0.9 + 0.02, out["fwd"], out["inv"])
        else:
            poses, poses_inv, out = train_mono.solve_pose_iteratively(3, dl, net, fr["target"], fr["sources"], fr["K"],
                                                                      return_errors=True)
            loss = pft.compute_optimization_loss(opts, fr["target"], tdisp, fr["disps"][0] * 0.9 + 0.02,
                                                 out["fwd"], out["inv"])
        loss.sum().backward()
        res.append((loss.detach(), out, [d.grad for d in dl], tdisp.grad, poses, poses_inv))
    ref, got = res
    for side in ("fwd", "inv"):
        for k in ("valid_mask", "auto_mask"):
            assert torch.equal(got[1][side][k], ref[1][side][k]), (side, k)
        for k in ("diff_img", "weight_mask", "auto_mask_error", "img_rec"):
            assert torch.equal(got[1][side][k], ref[1][side][k]), (side, k)
    assert got[0].shape == ref[0].shape
    assert abs(float(got[0]) - float(ref[0])) <= 1e-5 * abs(float(ref[0])), (float(got[0]), float(ref[0]))
    for j in range(1 + n_src):
        assert rel_l2(got[2][j], ref[2][j]) < 1e-4, (j, rel_l2(got[2][j], ref[2][j]))
    # the depth-init term is SSIM on two smooth, 0.9-correlated maps: the reference's own fp32 gradient is
    # ~6e-4 from its fp64 evaluation there (test_ssim_gradient_noise_floor_on_gpu)
    assert rel_l2(got[3], ref[3]) < 5e-4
    for a, b_ in zip(got[4] + got[5], ref[4] + ref[5]):
        assert torch.equal(a, b_)


@pytest.mark.parametrize("hw", [(192, 640), (256, 320), (50, 77)])
def test_compute_photometric_error_vs_eager_cuda(hw):
    """helpers.py:8-23 at batch 1 (the loss-surface sweeps): every returned map bit for bit."""
    from tcsfm_b200 import pft
    h, w = hw
    fr = frames(1, h, w, 0.02, synth.KITTI_DEPTH_RANGE, seed=23)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], fr["poses"][0], fr["K"])
    with torch.no_grad():
        ref, got = O.photometric_error(*args), pft.compute_photometric_error(*args)
    for k in ("diff_img", "img_rec", "valid_mask", "weight_mask"):
        assert torch.equal(got[k], ref[k]), (k, int((got[k] != ref[k]).sum()))


@pytest.mark.parametrize("shape", [(8, 3, 192, 640), (4, 1, 256, 320), (2, 3, 51, 67)])
def test_ssim_vs_eager_cuda(shape):
    """Standalone SSIM_Loss with the CUDA arithmetic flavour against eager PyTorch on the same device: the map bit
    for bit, gradients w.r.t. both arguments within 1e-4 on textured inputs."""
    gen = torch.Generator(device=DEV).manual_seed(3)
    x = torch.rand(shape, device=DEV, generator=gen)
    y = (x + 0.1 * torch.randn(shape, device=DEV, generator=gen)).clamp(0, 1)
    up = torch.randn(shape, device=DEV, generator=gen)
    res = []
    for fn in (O.ssim_dissimilarity, losses.SSIM_Loss()):
        xx, yy = leaf(x), leaf(y)
        out = fn(xx, yy)
        (out * up).sum().backward()
        res.append((out, xx.grad, yy.grad))
    ref, got = res
    assert torch.equal(got[0], ref[0]), int((got[0] != ref[0]).sum())
    assert rel_l2(got[1], ref[1]) < 1e-4 and rel_l2(got[2], ref[2]) < 1e-4
    mean = ops.SsimMeanFn.apply(x, y)
    assert abs(float(mean) - float(ref[0].mean())) <= 1e-6 * float(ref[0].mean())


def test_ssim_gradient_noise_floor_on_gpu():
    """On smooth, highly correlated inputs (the disparity-init term, optimizer.py:89-90) the kernel's gradient is
    closer to the reference's fp32 autograd than that is to its own fp64 evaluation (the documented exception
    to the 1e-4 gradient tolerance)."""
    g = Golden("mid_b2_64x96", DEV)
    x = g.frames()["disps"][0]
    y = x * 0.9 + 0.02
    gout = torch.full_like(x, 0.1 / x.numel())

    def ref(dtype):
        xx = x.to(dtype).clone().requires_grad_(True)
        (O.ssim_dissimilarity(xx, y.to(dtype)) * gout.to(dtype)).sum().backward()
        return xx.grad
    r32, r64 = ref(torch.float32), ref(torch.float64)
    xx = leaf(x)
    (losses.SSIM_Loss()(xx, y) * gout).sum().backward()
    assert rel_l2(xx.grad, r32) < rel_l2(r32, r64)
    assert rel_l2(xx.grad, r64) < 1.5 * rel_l2(r32, r64)


def test_graph_replay_follows_changed_intrinsics():
    """K^-1 is recomputed inside every call (models/stn.py:257), so a captured step replayed after the static K
    buffer was overwritten gives the eager result for the new K (round-1 finding: a memoised K^-1 was baked in)."""
    b, h, w = 2, 96, 160
    fr = frames(b, h, w, 0.01, synth.KITTI_DEPTH_RANGE, seed=3)
    mod = losses.Compute_Loss(goldens.FULL_CFG)
    K = fr["K"].clone()
    disps = [leaf(d) for d in fr["disps"]]
    poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]

    def step():
        for t in disps:
            t.grad = None
        out = mod(fr["sources"], fr["target"], [poses, poses_inv], [[d] for d in disps], K)
        out["total"].backward()
        return out["total"]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_total = step()
    K2 = fr["K"].clone()
    K2[:, 0, 0] *= 1.07
    K2[:, 1, 2] += 3.0
    K.copy_(K2)
    graph.replay()
    got, got_grad = static_total.detach().clone(), disps[0].grad.clone()
    ref = step()
    # (the masked sums are accumulated with atomics: equal up to their run-to-run rounding order)
    assert abs(float(got) - float(ref)) <= 2e-6 * abs(float(ref)), (float(got), float(ref))
    assert rel_l2(got_grad, disps[0].grad) < 1e-5
    stale = O.compute_loss(goldens.FULL_CFG, fr["sources"], fr["target"], [fr["poses"], fr["poses_inv"]],
                           [[d.detach()] for d in fr["disps"]], fr["K"])
    assert abs(float(got) - float(stale["total"])) > 1e-4 * abs(float(got)), "the changed K must change the loss"
    fresh = [leaf(d) for d in fr["disps"]]
    out = O.compute_loss(goldens.FULL_CFG, fr["sources"], fr["target"], [fr["poses"], fr["poses_inv"]],
                         [[d] for d in fresh], K2)
    assert abs(float(got) - float(out["total"])) <= 1e-5 * abs(float(out["total"]))


# ------------------------------------------------- "fast" SSIM arithmetic (TCSFM_ARITH_FAST, csrc/pair_fast_kernels.cu)
@pytest.fixture()
def fast_arith():
    ops.set_arithmetic("fast")
    yield
    ops.set_arithmetic("exact")


FAST_SHAPES = [(8, 192, 640, 0.01, synth.KITTI_DEPTH_RANGE, 2),       # BASELINE config 2
               (16, 256, 320, 0.04, synth.SCANNET_DEPTH_RANGE, 1),    # config 3
               (2, 376, 1242, 0.02, synth.KITTI_DEPTH_RANGE, 2),      # config 5 resolution
               (4, 256, 448, 0.02, synth.SCANNET_DEPTH_RANGE, 1),
               (3, 51, 77, 0.08, synth.KITTI_DEPTH_RANGE, 3),         # odd sizes, three sources
               (1, 192, 640, 0.02, synth.KITTI_DEPTH_RANGE, 2)]       # batch 1: the non-fused cuBLAS flavour


@pytest.mark.parametrize("shape", FAST_SHAPES)
@pytest.mark.parametrize("tag", ["train", "full"])
def test_fast_compute_loss_vs_eager_cuda(fast_arith, shape, tag):
    """North-star tolerances for the fast flavour: every loss term within 1e-5, gradients within 1e-4 (rel-L2) of the
    reference's eager CUDA path."""
    b, h, w, yaw, rng, n_src = shape
    fr = synth.make_frames(b, h, w, n_src=n_src, seed=21, yaw=yaw, depth_range=rng, device=DEV,
                           intrinsics=synth.scaled_intrinsics(h, w))
    cfg = dict(goldens.LOSS_CFGS[tag], min_depth=rng[0], max_depth=rng[1])
    res = []
    for impl in ("oracle", "cuda"):
        disps = [leaf(d) for d in fr["disps"]]
        poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
        dl = [[d] for d in disps]
        if impl == "oracle":
            out = O.compute_loss(cfg, fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        else:
            out = losses.Compute_Loss(cfg)(fr["sources"], fr["target"], [poses, poses_inv], dl, fr["K"])
        out["total"].sum().backward()
        res.append((out, disps, poses, poses_inv))
    (ro, rd, rp, rpi), (go, gd, gp, gpi) = res
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, bb = float(go[k].detach()), float(ro[k].detach())
        assert abs(a - bb) <= 1e-5 * max(abs(bb), 1e-12), (k, a, bb)

    def grad(t):
        return t.grad if t.grad is not None else torch.zeros_like(t)
    for j in range(1 + n_src):
        assert rel_l2(grad(gd[j]), grad(rd[j])) < 1e-4, ("disp", j, rel_l2(grad(gd[j]), grad(rd[j])))
    for j in range(n_src):
        assert rel_l2(grad(gp[j]), grad(rp[j])) < 1e-4, ("pose", j, rel_l2(grad(gp[j]), grad(rp[j])))
        assert rel_l2(grad(gpi[j]), grad(rpi[j])) < 1e-4, ("pose_inv", j, rel_l2(grad(gpi[j]), grad(rpi[j])))


@pytest.mark.parametrize("shape", FAST_SHAPES)
def test_fast_pair_masks_bit_exact_vs_eager_cuda(fast_arith, shape):
    """The fast flavour keeps geometry, warp, L1 and the auto-mask comparison bit-exact: valid / auto masks identical
    to eager PyTorch on the same GPU; diff_img at the reference's own fp32 noise floor."""
    b, h, w, yaw, rng, _ = shape
    fr = frames(b, h, w, yaw, rng, seed=5)
    for tag in ("train", "full", "noauto"):
        cfg = goldens.PAIR_CFGS[tag]
        for tgt, ref, td, rd, pose in ((fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], -fr["poses"][0]),
                                       (fr["sources"][1], fr["target"], fr["depths"][2], fr["depths"][0], -fr["poses_inv"][1])):
            _, _, rdiff, rmask, _ = O.pairwise_loss(cfg, tgt, ref, td, rd, pose, fr["K"])
            _, _, gdiff, gmask, _ = losses.Compute_Loss(cfg).compute_pairwise_loss(tgt, ref, td, rd, pose, fr["K"], 0)
            assert torch.equal(gmask, rmask), (tag, int((gmask != rmask).sum()))
            assert rel_l2(gdiff, rdiff) < 5e-5, (tag, rel_l2(gdiff, rdiff))


def test_fast_randomised_sweep_vs_eager_cuda(fast_arith):
    """Random shapes, skewed intrinsics, depth scales and poses (incl. points behind the camera) through the fast
    flavour: masks bit-exact, loss 1e-5, gradients 1e-4."""
    gen = torch.Generator().manual_seed(1234)
    for it in range(12):
        b = int(torch.randint(1, 5, (1,), generator=gen))
        h = int(torch.randint(20, 200, (1,), generator=gen))
        w = int(torch.randint(20, 300, (1,), generator=gen))
        fr = frames(b, h, w, float(torch.rand(1, generator=gen)) * 0.1, synth.KITTI_DEPTH_RANGE, seed=100 + it)
        fr["K"][:, 0, 1] = float(torch.rand(1, generator=gen)) * 2.0          # skew
        cfg = goldens.FULL_CFG
        res = []
        for impl in ("oracle", "cuda"):
            disps = [leaf(d) for d in fr["disps"]]
            dl = [[d] for d in disps]
            args = (fr["sources"], fr["target"], [fr["poses"], fr["poses_inv"]], dl, fr["K"])
            out = O.compute_loss(cfg, *args) if impl == "oracle" else losses.Compute_Loss(cfg)(*args)
            out["total"].sum().backward()
            res.append((float(out["total"].detach()), [d.grad for d in disps]))
        assert abs(res[1][0] - res[0][0]) <= 1e-5 * abs(res[0][0]), (it, b, h, w, res[1][0], res[0][0])
        for j in range(3):
            assert rel_l2(res[1][1][j], res[0][1][j]) < 1e-4, (it, b, h, w, j, rel_l2(res[1][1][j], res[0][1][j]))


def test_graphed_train_step_matches_eager():
    """training.FlatGradTrainer: forward+backward and Adam replayed as CUDA graphs give the losses and parameters of the
    eager run_train_step on the same sequence of minibatches; building the trainer does not change the parameters."""
    from tcsfm_b200 import training
    cfg = training.default_config(num_scales=2, iterations=2, full_profile=True)
    data = [synth.make_frames(2, 96, 160, seed=40 + s, device=DEV) for s in range(3)]
    step_a, optim_a = training.make_step(cfg, seed=1, device=DEV, padded=False)
    step_b, optim_b = training.make_step(cfg, seed=1, device=DEV, padded=False, capturable=True)
    trainer = training.FlatGradTrainer(step_b, optim_b, data[0])
    for p, q in zip(step_a.parameters(), step_b.parameters()):
        assert torch.equal(p, q)
    for fr in data:
        ta = training.run_train_step(step_a, optim_a, fr)
        tb = trainer.run(fr).clone()
        assert torch.allclose(ta, tb, rtol=2e-5, atol=0), (ta, tb)
    # (Adam's first updates are lr * sign-like: a gradient that rounds differently near zero moves a single weight by
    # up to 2 lr, so the parameters are compared in the mean)
    for p, q in zip(step_a.parameters(), step_b.parameters()):
        assert float((p - q).abs().mean()) < 2e-5, float((p - q).abs().mean())


def test_min_resolve_restores_the_reference_routing():
    """tcsfm_pair_min_resolve (per-pixel min + exact re-evaluation of its near-ties, ties kept in shared memory) at
    config 2 re-evaluates exactly the near-ties found on the host from the forward's maps: their values become the
    exact kernels', every other value is left as it was, the arg-min over the sources is the exact arithmetic's
    everywhere, and the sum is the one of the maps as the forward produced them."""
    from tcsfm_b200 import _raw
    L = _lib.lib()
    fr = frames(8, 192, 640, 0.01, synth.KITTI_DEPTH_RANGE, seed=31)
    flags = _cabi.SSIM | _cabi.AUTO_MASK | _cabi.DEPTH_MASK | _cabi.DEPTH_CONSIST

    def forward(fl):
        groups = []
        for j in range(2):
            kinv, proj = stn.projection_matrices(-fr["poses"][j], fr["K"])
            groups.append({"tgt_img": fr["target"], "ref_img": fr["sources"][j], "tgt_depth": fr["depths"][0],
                           "ref_depth": fr["depths"][1 + j], "kinv": kinv, "proj": proj})
        batch = _raw.PairBatch(groups)
        diff, _, _, _ = _raw.pair_loss_fwd(L, batch, 0.15, 0.85, fl)
        return batch, diff

    _, d_exact = forward(flags)
    fast = flags | _cabi.ARITH_FAST
    batch, d = forward(fast)
    before = d.clone()
    # the kernel's rule in fp32: a NaN in either candidate, or the two closer than the band
    a, b = before.reshape(2, -1)
    band = torch.tensor(_raw.TIE_BAND, dtype=torch.float32, device=a.device)
    ties = a.isnan() | b.isnan() | ~(torch.maximum(a, b) - torch.minimum(a, b) >= band)
    min_sum, tie_count = _raw.pair_min_resolve(L, batch, [0, 1], 0.15, 0.85, fast)
    assert int(tie_count) == int(ties.sum()) > 0
    for j in range(2):
        assert torch.equal(d[j].flatten()[ties], d_exact[j].flatten()[ties])
        assert torch.equal(d[j].flatten()[~ties], before[j].flatten()[~ties])
    assert torch.equal(torch.min(d.reshape(2, -1), 0)[1], torch.min(d_exact.reshape(2, -1), 0)[1])
    want = float(torch.min(before.reshape(2, -1), 0)[0].sum())
    assert abs(float(min_sum) - want) <= 1e-5 * abs(want)


def test_intrinsics_inverse_bit_exact_vs_torch_cuda():
    """stn.inverse_intrinsics (one launch of the library's batched 3x3 LU) against torch.linalg.inv_ex and
    torch.inverse on the same GPU, 50 000 matrices per family: bit for bit."""
    g = torch.Generator().manual_seed(5)
    n = 50000
    fx = 200 + 1000 * torch.rand(n, generator=g)
    kitti = torch.zeros(n, 3, 3)
    kitti[:, 0, 0], kitti[:, 1, 1] = fx, fx * (0.9 + 0.2 * torch.rand(n, generator=g))
    kitti[:, 0, 2], kitti[:, 1, 2], kitti[:, 2, 2] = 100 + 600 * torch.rand(n, generator=g), 50 + 300 * torch.rand(n, generator=g), 1.0
    skew = kitti.clone()
    skew[:, 0, 1] = 5 * torch.randn(n, generator=g)
    fams = {"kitti": kitti, "skew": skew, "lower": kitti.transpose(1, 2).contiguous(),
            "dense": torch.randn(n, 3, 3, generator=g) + 3 * torch.eye(3),
            "scaled": torch.randn(n, 3, 3, generator=g) * torch.tensor([300.0, 30.0, 1.0]).view(1, 3, 1),
            "perm": torch.randn(n, 3, 3, generator=g)[:, [2, 0, 1]]}
    for name, k in fams.items():
        k = k.to(DEV)
        got = stn.inverse_intrinsics(k)
        want = torch.linalg.inv_ex(k)[0]
        assert got.is_contiguous() and got.shape == (n, 3, 3)
        bad = (got.view(torch.int32) != want.contiguous().view(torch.int32)).flatten(1).any(1)
        assert int(bad.sum()) == 0, (name, int(bad.sum()))
        assert torch.equal(got[:256], torch.inverse(k[:256]))
    one = stn.inverse_intrinsics(fams["kitti"][:1].to(DEV))                      # batch 1
    assert torch.equal(one, torch.inverse(fams["kitti"][:1].to(DEV)))
