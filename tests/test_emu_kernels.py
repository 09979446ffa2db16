"""Kernel logic checked on the CPU through the test-only CUDA emulator build
(tests/emu): same csrc/*.cu sources, same C ABI, host pointers.  Compared with the
oracle and the reference-generated golden vectors using the CPU arithmetic
flavour, so masks and forward values must match bit for bit."""
import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden, rel_l2
from oracle import ref_torch as O
from tcsfm_b200 import _cabi, _raw, stn, synth

CPU = _cabi.ARITH_CPU


def same(a, b):
    return torch.equal(a.detach().float(), b.detach().float())


def cfg_flags(cfg):
    f = CPU | _cabi.SSIM
    if cfg["with_auto_mask"]:
        f |= _cabi.AUTO_MASK
    if cfg["with_depth_mask"]:
        f |= _cabi.DEPTH_MASK
    if cfg["l_depth_consist"]:
        f |= _cabi.DEPTH_CONSIST
    return f


@pytest.mark.parametrize("case", goldens.CASES)
def test_warp_fwd_bwd_vs_golden(case):
    g = Golden(case)
    fr = g.frames()
    pose = -fr["poses"][0]
    kinv, proj = stn.projection_matrices(pose, fr["K"])
    out_img, valid, pd, cd = _raw.warp_fwd(emu(), fr["sources"][0], fr["depths"][0], fr["depths"][1], kinv, proj, CPU)
    assert same(valid, g.t("warp/valid_mask"))
    assert same(cd, g.t("warp/computed_depth"))
    assert rel_l2(out_img, g.t("warp/projected_img")) < 1e-6
    assert rel_l2(pd, g.t("warp/projected_depth")) < 1e-6
    # backward: grad wrt proj is mapped to the pose by autograd of the tiny algebra
    p0 = pose.clone().requires_grad_(True)
    _, proj_t = stn.projection_matrices(p0, fr["K"])
    g_depth, g_ref, g_proj, g_src = _raw.warp_bwd(emu(), fr["sources"][0], fr["depths"][0], fr["depths"][1], kinv, proj,
                                                  g.t("in/g_img"), g.t("in/g_pd"), g.t("in/g_cd"), CPU, need_img_grad=True)
    proj_t.backward(g_proj)
    assert rel_l2(g_depth, g.t("warp/g_depth")) < 2e-5
    assert rel_l2(g_ref, g.t("warp/g_ref_depth")) < 2e-5
    assert rel_l2(p0.grad, g.t("warp/g_pose")) < 2e-4
    # grad wrt the sampled image against oracle autograd
    src = fr["sources"][0].clone().requires_grad_(True)
    pim, _, _, _ = O.inverse_warp2(src, fr["depths"][0], fr["depths"][1], pose, fr["K"])
    (pim * g.t("in/g_img")).sum().backward()
    assert rel_l2(g_src, src.grad) < 2e-5


def test_warp_strided_channel_slice():
    fr = synth.make_frames(2, 20, 70, seed=5)
    six = torch.cat([fr["target"], fr["sources"][0]], 1)
    pose = -fr["poses"][0]
    kinv, proj = stn.projection_matrices(pose, fr["K"])
    a = _raw.warp_fwd(emu(), six[:, 3:6], fr["depths"][0], fr["depths"][1], kinv, proj, CPU)
    b = _raw.warp_fwd(emu(), fr["sources"][0], fr["depths"][0], fr["depths"][1], kinv, proj, CPU)
    for x, y in zip(a, b):
        assert same(x, y)


@pytest.mark.parametrize("case", goldens.CASES)
def test_ssim_vs_golden(case):
    g = Golden(case)
    x, y = g.t("in/target"), g.t("in/source0")
    out = _raw.ssim_fwd(emu(), x, y, CPU)
    assert same(out, g.t("ssim/map"))
    g_x, g_y = _raw.ssim_bwd(emu(), x, y, g.t("in/g_img"), True, True, CPU)
    assert rel_l2(g_x, g.t("ssim/g_x")) < 2e-5
    assert rel_l2(g_y, g.t("ssim/g_y")) < 2e-5


@pytest.mark.parametrize("hw", [(2, 2), (3, 5), (17, 65), (16, 64), (33, 130)])
def test_ssim_odd_sizes_vs_oracle(hw):
    h, w = hw
    gen = torch.Generator().manual_seed(h * 100 + w)
    x = torch.rand(2, 1, h, w, generator=gen).requires_grad_(True)
    y = torch.rand(2, 1, h, w, generator=gen).requires_grad_(True)
    gout = torch.randn(2, 1, h, w, generator=gen)
    ref = O.ssim_dissimilarity(x, y)
    (ref * gout).sum().backward()
    out = _raw.ssim_fwd(emu(), x.detach(), y.detach(), CPU)
    assert same(out, ref)
    g_x, g_y = _raw.ssim_bwd(emu(), x.detach(), y.detach(), gout, True, True, CPU)
    assert rel_l2(g_x, x.grad) < 2e-5 and rel_l2(g_y, y.grad) < 2e-5


def run_pair(fr, cfg, g_diff, lrep_w=1.0, ldep_w=0.5):
    pose = -fr["poses"][0]
    p0 = pose.clone().requires_grad_(True)
    kinv, proj = stn.projection_matrices(p0, fr["K"])
    flags = cfg_flags(cfg)
    batch = _raw.PairBatch([{"tgt_img": fr["target"], "ref_img": fr["sources"][0], "tgt_depth": fr["depths"][0],
                             "ref_depth": fr["depths"][1], "kinv": kinv.detach(), "proj": proj.detach()}])
    diff, mask, sums, coef = _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, flags)
    g_scalars = torch.tensor([[lrep_w, ldep_w if cfg["l_depth_consist"] else 0.0]])
    need_ref = cfg["with_depth_mask"] or cfg["l_depth_consist"]
    g_td, g_rd, g_proj = _raw.pair_loss_bwd(emu(), batch, mask, sums, coef, g_diff.unsqueeze(0), g_scalars, 0.15, 0.85, flags, need_ref)
    proj.backward(g_proj[0])
    return diff[0], mask[0], sums[0], g_td[0], (g_rd[0] if need_ref else None), p0.grad


@pytest.mark.parametrize("case", goldens.CASES)
@pytest.mark.parametrize("tag", ["train", "full", "noauto"])
def test_pair_loss_vs_golden(case, tag):
    g = Golden(case)
    fr = g.frames()
    cfg = goldens.PAIR_CFGS[tag]
    diff, mask, sums, g_td, g_rd, g_pose = run_pair(fr, cfg, g.t("in/g_diff"))
    assert same(mask, g.t("pair_%s/valid_mask" % tag))
    ref_diff = g.t("pair_%s/diff_img" % tag)
    assert (diff - ref_diff).abs().max().item() < 2e-6
    n_mask = float(mask.sum())
    assert float(sums[1]) == n_mask
    l_rep = float(sums[0] / sums[1]) if n_mask > 10000 else 0.0
    assert abs(l_rep - float(g.t("pair_%s/l_reprojection" % tag))) <= 1e-5 * max(abs(l_rep), 1e-12)
    if cfg["l_depth_consist"]:
        l_dep = float(sums[2] / sums[1]) if n_mask > 10000 else 0.0
        assert abs(l_dep - float(g.t("pair_%s/l_depth" % tag))) <= 1e-5 * max(abs(l_dep), 1e-12)
    assert rel_l2(g_td, g.t("pair_%s/g_depth" % tag)) < 1e-4
    if g_rd is not None:
        assert rel_l2(g_rd, g.t("pair_%s/g_ref_depth" % tag)) < 1e-4
    assert rel_l2(g_pose, g.t("pair_%s/g_pose" % tag)) < 1e-3


def test_pair_loss_multi_group_and_partial_tiles():
    """Two groups in one launch (forward + inverse direction) on a size that is not
    a multiple of the 64x16 tile, against the oracle."""
    fr = synth.make_frames(2, 37, 150, seed=9)
    cfg = goldens.FULL_CFG
    flags = cfg_flags(cfg)
    K = fr["K"]
    specs = [(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], -fr["poses"][0]),
             (fr["sources"][0], fr["target"], fr["depths"][1], fr["depths"][0], -fr["poses_inv"][0])]
    groups = []
    for tgt, ref, td, rd, pose in specs:
        kinv, proj = stn.projection_matrices(pose, K)
        groups.append({"tgt_img": tgt, "ref_img": ref, "tgt_depth": td, "ref_depth": rd, "kinv": kinv, "proj": proj})
    batch = _raw.PairBatch(groups)
    diff, mask, sums, coef = _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, flags)
    gen = torch.Generator().manual_seed(3)
    g_diff = torch.randn(2, 2, 1, 37, 150, generator=gen)
    g_td, g_rd, g_proj = _raw.pair_loss_bwd(emu(), batch, mask, sums, coef, g_diff, None, 0.15, 0.85, flags, True)
    for i, (tgt, ref, td, rd, pose) in enumerate(specs):
        td_l, rd_l = td.clone().requires_grad_(True), rd.clone().requires_grad_(True)
        _, _, rdiff, rmask, _ = O.pairwise_loss(cfg, tgt, ref, td_l, rd_l, pose, K)
        assert same(mask[i], rmask)
        assert (diff[i] - rdiff).abs().max().item() < 2e-6
        (rdiff * g_diff[i]).sum().backward()
        assert rel_l2(g_td[i], td_l.grad) < 1e-4
        assert rel_l2(g_rd[i], rd_l.grad) < 1e-4


def test_bad_arguments_return_errors():
    fr = synth.make_frames(1, 8, 8, seed=0)
    kinv, proj = stn.projection_matrices(-fr["poses"][0], fr["K"])
    with pytest.raises(RuntimeError, match="bad shape"):
        _raw.ssim_fwd(emu(), torch.rand(1, 1, 1, 8), torch.rand(1, 1, 1, 8))
    batch = _raw.PairBatch([{"tgt_img": fr["target"], "ref_img": fr["sources"][0], "tgt_depth": fr["depths"][0],
                             "ref_depth": None, "kinv": kinv, "proj": proj}])
    with pytest.raises(RuntimeError, match="ref_depth"):
        _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, CPU | _cabi.SSIM | _cabi.DEPTH_MASK)
    with pytest.raises(RuntimeError, match="TCSFM_SSIM"):
        _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, CPU)
    # in-kernel offsets inside one batch element are 32-bit: a channel stride that cannot be is refused
    import ctypes
    grp = _cabi.PairGroup()
    dummy = torch.zeros(64)
    for name in ("tgt_img", "ref_img", "tgt_depth", "kinv", "proj", "sums"):
        setattr(grp, name, dummy.data_ptr())
    grp.tgt_sc, grp.ref_sc = 64, 1 << 31
    rc = emu().tcsfm_pair_loss_fwd(ctypes.byref(grp), 1, 1, 8, 8, 0.15, 0.85, CPU | _cabi.SSIM, None)
    assert rc != 0 and b"channel stride out of range" in emu().tcsfm_last_error()
    # the frame-level upstream needs at least one of its two gradient pointers
    cfg = _raw.make_frame_cfg([0, 1], 0.3, 0.14, 64)
    rc = emu().tcsfm_frame_bwd_prepare(None, None, ctypes.byref(cfg), dummy.data_ptr(), dummy.data_ptr(), None, 0, None)
    assert rc != 0 and b"tcsfm_frame_bwd_prepare" in emu().tcsfm_last_error()


def test_pose_proj_fwd_bwd_vs_torch():
    gen = torch.Generator().manual_seed(0)
    pose = (0.2 * torch.randn(12, 6, generator=gen)).requires_grad_(True)
    K = torch.tensor(synth.KITTI_K).repeat(4, 1, 1) + 0.01 * torch.rand(4, 3, 3, generator=gen)
    ref = K.repeat(3, 1, 1) @ stn.pose_vec2mat(-pose)
    got = _raw.pose_proj_fwd(emu(), pose.detach(), K, -1.0, 0)
    assert (got - ref).abs().max() < 1e-4 * ref.abs().max()
    gp = torch.randn(12, 3, 4, generator=gen)
    ref.backward(gp)
    g_pose = _raw.pose_proj_bwd(emu(), pose.detach(), K, -1.0, gp)
    assert rel_l2(g_pose, pose.grad) < 1e-5


def test_min_reduce_and_routing_ties():
    gen = torch.Generator().manual_seed(1)
    stack = torch.rand(3, 2, 1, 9, 11, generator=gen)
    stack[1] = torch.where(torch.rand(2, 1, 9, 11, generator=gen) < 0.3, stack[0], stack[1])   # exact ties
    ref = torch.min(stack.permute(1, 0, 2, 3, 4).reshape(2, 3, 9, 11), 1)[0].sum()
    got = _raw.min_reduce(emu(), stack[0], stack[0].numel(), 3, stack[0].numel())
    assert abs(float(got) - float(ref)) < 1e-4


@pytest.mark.parametrize("hw", [(2, 2), (3, 3), (2, 70), (5, 66), (17, 3), (16, 64), (33, 129)])
def test_pair_and_photo_tiny_and_edge_sizes_vs_oracle(hw):
    """Degenerate / tile-edge image sizes: reflection padding with H or W of 2-3, exactly one tile,
    one pixel past a tile.  Forward bit for bit, gradients within tolerance, against the oracle."""
    h, w = hw
    fr = synth.make_frames(2, h, w, seed=h * 7 + w, intrinsics=synth.scaled_intrinsics(max(h, 8), max(w, 8)))
    cfg = goldens.FULL_CFG
    flags = cfg_flags(cfg)
    pose = -fr["poses"][0]
    kinv, proj = stn.projection_matrices(pose, fr["K"])
    batch = _raw.PairBatch([{"tgt_img": fr["target"], "ref_img": fr["sources"][0], "tgt_depth": fr["depths"][0],
                             "ref_depth": fr["depths"][1], "kinv": kinv, "proj": proj}])
    diff, mask, sums, coef = _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, flags)
    td, rd = fr["depths"][0].clone().requires_grad_(True), fr["depths"][1].clone().requires_grad_(True)
    _, _, rdiff, rmask, _ = O.pairwise_loss(cfg, fr["target"], fr["sources"][0], td, rd, pose, fr["K"])
    # (with fewer than ~16 pixels the CPU BLAS behind the oracle's k=3 bmm rounds differently, so the
    # degenerate sizes are compared to 1e-4 instead of bit for bit)
    exact = h * w >= 16
    assert same(mask[0], rmask)
    assert same(diff[0], rdiff) if exact else (diff[0] - rdiff).abs().max() < 1e-4
    gen = torch.Generator().manual_seed(1)
    g_diff = torch.randn(1, 2, 1, h, w, generator=gen)
    g_td, g_rd, _ = _raw.pair_loss_bwd(emu(), batch, mask, sums, coef, g_diff, None, 0.15, 0.85, flags, True)
    (rdiff * g_diff[0]).sum().backward()
    assert rel_l2(g_td[0], td.grad) < 1e-4 and rel_l2(g_rd[0], rd.grad) < 1e-4
    # PFT photometric block on the same inputs
    rec, _, pd, cd = _raw.warp_fwd(emu(), fr["sources"][0], fr["depths"][0], fr["depths"][1], kinv, proj, CPU)
    six = torch.cat([fr["target"], fr["sources"][0]], 1)
    rec_l = rec.clone().requires_grad_(True)
    ref = O.pft_error_maps(six, rec_l, pd, cd)
    got = _raw.photo_fwd(emu(), six[:, 0:3], six[:, 3:6], rec, pd, cd, 0.15, 0.85, CPU)
    for a, b_ in zip(got[:4], ref):
        assert same(a, b_) if exact else (a - b_).abs().max() < 1e-4
    g1 = torch.randn(2, 1, h, w, generator=gen)
    (ref[1] * g1).sum().backward()
    g_rec, _, _ = _raw.photo_bwd(emu(), six[:, 0:3], rec, pd, cd, got[4], g1, None, 0.15, 0.85, CPU)
    assert rel_l2(g_rec, rec_l.grad) < 1e-4


@pytest.mark.parametrize("shapes", [((47, 155), (376, 1242)), ((12, 20), (24, 40)), ((7, 9), (24, 40)), ((24, 40), (24, 40)),
                                    ((1, 1), (5, 7)), ((94, 310), (376, 1242))])
def test_disp_upsample_to_depth_vs_interpolate(shapes):
    """The nearest upsample folded into disp -> depth (losses.py:86-88): bit for bit the index rule of
    F.interpolate(mode='nearest'), and the gradient of the composed torch expression."""
    (h, w), (big_h, big_w) = shapes
    b = 2 if big_h < 100 else 1
    gen = torch.Generator().manual_seed(h * 1000 + w)
    disps = [torch.rand(b, 1, h, w, generator=gen).requires_grad_(True) for _ in range(3)]
    min_disp, max_disp = 1 / 2.67, 1 / 0.06
    got = _raw.disp_to_depth_fwd(emu(), [d.detach() for d in disps], min_disp, max_disp - min_disp, out_hw=(big_h, big_w))
    g_out = [torch.randn(b, 1, big_h, big_w, generator=gen) for _ in range(3)]
    g_got = _raw.disp_to_depth_bwd(emu(), g_out, got, max_disp - min_disp, disp_hw=(h, w))
    for d, dep, g, gd in zip(disps, got, g_out, g_got):
        up = torch.nn.functional.interpolate(d, (big_h, big_w), mode="nearest")
        ref = 1 / (min_disp + (max_disp - min_disp) * up)
        assert dep.shape == ref.shape and same(dep, ref)
        ref.backward(g)
        assert gd.shape == d.shape and rel_l2(gd, d.grad) < 1e-5


def test_intrinsics_inverse_has_the_bits_of_torch_on_cuda():
    """tcsfm_intrinsics_inverse against inverses that torch.linalg.inv_ex produced on a B200 (tests/golden/probes/
    kinv_cuda_probe.npz: the first 300 matrices of each family of tools/probe_kinv.py -- camera intrinsics, skewed,
    lower-triangular, dense, badly scaled): bit for bit, signs of zeros included."""
    import os
    import numpy as np
    from tcsfm_b200 import _raw
    d = np.load(os.path.join(os.path.dirname(__file__), "golden", "probes", "kinv_cuda_probe.npz"))
    for fam in ("kitti", "skew", "dense", "general", "lower"):
        k = torch.from_numpy(d[fam + "_in"])
        want = torch.from_numpy(d[fam + "_inv"])
        got = _raw.intrinsics_inverse(emu(), k)
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), fam


def test_frame_prologue_and_epilogue_equal_the_separate_launches():
    """tcsfm_frame_prologue (disp -> depth + pose -> K[R|t] + K^-1, poses read in place with a row stride) and
    tcsfm_frame_epilogue (their chain rules) against the single-purpose entry points: identical bits."""
    from tcsfm_b200 import _raw, synth
    fr = synth.make_frames(3, 20, 36, seed=2)
    K = fr["K"]
    wide = [torch.cat([p, torch.zeros(3, 2)], 1) for p in (fr["poses"][0], fr["poses"][1], fr["poses_inv"][0])]   # [B,8] storage
    poses = [w[:, 0:6] for w in wide]
    rows = _raw.pose_rows(poses)
    assert rows is not None and rows[1] == 8
    disps = fr["disps"]
    lo, hi = 1 / synth.KITTI_DEPTH_RANGE[1], 1 / synth.KITTI_DEPTH_RANGE[0]
    depths, proj, kinv = _raw.frame_prologue(emu(), disps, lo, hi - lo, rows[0], rows[1], K, -1.0, 0, want_kinv=True)
    want_d = _raw.disp_to_depth_fwd(emu(), disps, lo, hi - lo)
    want_p = _raw.pose_proj_fwd(emu(), torch.cat(poses, 0).contiguous(), K, -1.0, 0)
    assert all(torch.equal(a, b) for a, b in zip(depths, want_d))
    assert torch.equal(proj, want_p)
    assert torch.equal(kinv, _raw.intrinsics_inverse(emu(), K))
    g_depths = [torch.randn_like(d) for d in depths]
    g_proj = torch.randn_like(proj)
    g_disps, g_pose = _raw.frame_epilogue(emu(), g_depths, depths, hi - lo, rows[0], rows[1], K, -1.0, g_proj)
    want_gd = _raw.disp_to_depth_bwd(emu(), g_depths, depths, hi - lo)
    want_gp = _raw.pose_proj_bwd(emu(), torch.cat(poses, 0).contiguous(), K, -1.0, g_proj)
    assert all(torch.equal(a, b) for a, b in zip(g_disps, want_gd))
    assert torch.equal(g_pose, want_gp)
    # prepare + zero-fill in one launch
    cfg = _raw.make_frame_cfg([0, 1, 0, 1], 0.3, 0.14, 3 * 20 * 36)
    buf = torch.randn(3, 3, 1, 20, 36)
    a = _raw.frame_bwd_prepare(emu(), torch.tensor([0.5, 1.0, 2.0]), torch.tensor([0.25]), cfg, zero=buf)
    b = _raw.frame_bwd_prepare(emu(), torch.tensor([0.5, 1.0, 2.0]), torch.tensor([0.25]), cfg)
    assert float(buf.abs().sum()) == 0.0 and torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
