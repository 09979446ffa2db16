"""The "fast" SSIM arithmetic of the fused pair loss (TCSFM_ARITH_FAST, csrc/pair_fast_kernels.cu) on the
test-only emulator: masks stay bit-exact against the reference-generated fixtures, values / losses /
gradients meet the north-star tolerances (loss 1e-5, gradients 1e-4 rel-L2)."""
import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden, rel_l2
from oracle import ref_torch as O
from tcsfm_b200 import _cabi, _raw, losses, ops, stn, synth

CPU_FAST = _cabi.ARITH_CPU | _cabi.ARITH_FAST


def cfg_flags(cfg):
    flags = _cabi.SSIM | CPU_FAST
    if cfg["with_auto_mask"]:
        flags |= _cabi.AUTO_MASK
    if cfg["with_depth_mask"]:
        flags |= _cabi.DEPTH_MASK
    if cfg["l_depth_consist"]:
        flags |= _cabi.DEPTH_CONSIST
    return flags


def leaf(t):
    return t.clone().detach().requires_grad_(True)


@pytest.fixture()
def emu_fast(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)
    monkeypatch.setattr(ops, "PAIR_ARITHMETIC", "fast")


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
def test_fast_pair_loss_vs_golden(case, tag):
    g = Golden(case)
    fr = g.frames()
    cfg = goldens.PAIR_CFGS[tag]
    diff, mask, sums, g_td, g_rd, g_pose = run_pair(fr, cfg, g.t("in/g_diff"))
    assert torch.equal(mask, g.t("pair_%s/valid_mask" % tag))              # masks: bit-exact
    ref_diff = g.t("pair_%s/diff_img" % tag)
    # per-pixel values sit at the reference's own fp32 noise floor (its fp32 vs fp64 diff_img: 1e-5 .. 2e-5 rel-L2, SURVEY.md 0-6)
    assert rel_l2(diff, ref_diff) < 5e-5, rel_l2(diff, ref_diff)
    assert (diff - ref_diff).abs().max().item() < 2e-4      # cancellation in E[x^2] - mu^2 against C2 = 9e-4
    n_mask = float(mask.sum())
    assert float(sums[1]) == n_mask
    l_rep = float(sums[0] / sums[1]) if n_mask > 0 else 0.0
    ref_rep = float((ref_diff * mask).sum() / mask.sum()) if n_mask > 0 else 0.0
    assert abs(l_rep - ref_rep) <= 1e-5 * max(abs(ref_rep), 1e-12)
    assert rel_l2(g_td, g.t("pair_%s/g_depth" % tag)) < 1e-4, rel_l2(g_td, g.t("pair_%s/g_depth" % tag))
    if g_rd is not None:
        assert rel_l2(g_rd, g.t("pair_%s/g_ref_depth" % tag)) < 1e-4
    assert rel_l2(g_pose, g.t("pair_%s/g_pose" % tag)) < 1e-3


@pytest.mark.parametrize("hw,tile_h", [((37, 150), None), ((33, 65), None), ((2, 2), None), ((3, 64), None), ((64, 3), None),
                                       ((31, 129), None), ((37, 150), 16), ((37, 150), 24), ((49, 65), 24), ((37, 150), 32)])
def test_fast_multi_group_partial_tiles_and_odd_sizes(hw, tile_h, monkeypatch):
    """Forward + inverse direction in one launch on sizes that are not multiples of the 64 x {16, 24, 32} tiles (odd
    heights exercise the last pixel pair of a column), against the oracle; every tile height the host may pick
    (TCSFM_FAST_FH pins it, None = the wave-count rule)."""
    if tile_h is None:
        monkeypatch.delenv("TCSFM_FAST_FH", raising=False)
    else:
        monkeypatch.setenv("TCSFM_FAST_FH", str(tile_h))
    h, w = hw
    fr = synth.make_frames(2, h, w, seed=9)
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
    g_diff = torch.randn(2, 2, 1, h, w, generator=gen)
    g_td, g_rd, g_proj = _raw.pair_loss_bwd(emu(), batch, mask, sums, coef, g_diff, None, 0.15, 0.85, flags, True)
    for i, (tgt, ref, td, rd, pose) in enumerate(specs):
        td_l, rd_l = leaf(td), leaf(rd)
        _, _, rdiff, rmask, _ = O.pairwise_loss(cfg, tgt, ref, td_l, rd_l, pose, K)
        assert torch.equal(mask[i], rmask)
        assert rel_l2(diff[i], rdiff) < 5e-5 and (diff[i] - rdiff).abs().max().item() < 2e-4
        (rdiff * g_diff[i]).sum().backward()
        assert rel_l2(g_td[i], td_l.grad) < 1e-4, rel_l2(g_td[i], td_l.grad)
        assert rel_l2(g_rd[i], rd_l.grad) < 1e-4, rel_l2(g_rd[i], rd_l.grad)


@pytest.mark.parametrize("case", goldens.CASES)
@pytest.mark.parametrize("tag", ["train", "full"])
def test_fast_compute_loss_forward_backward(emu_fast, case, tag):
    g = Golden(case)
    fr = g.frames()
    mod = losses.Compute_Loss(goldens.LOSS_CFGS[tag])
    disps = [leaf(d) for d in fr["disps"]]
    poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
    out = mod(fr["sources"], fr["target"], [poses, poses_inv], [[disps[0]], [disps[1]], [disps[2]]], fr["K"])
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "total"):
        a, b = float(out[k]), float(g.t("loss_%s/%s" % (tag, k)))
        assert abs(a - b) <= 1e-5 * max(abs(b), 1e-12), (k, a, b)
    out["total"].sum().backward()
    for j in range(3):
        ref_g = g.t("loss_%s/g_disp%d" % (tag, j))
        got = disps[j].grad if disps[j].grad is not None else torch.zeros_like(ref_g)
        assert rel_l2(got, ref_g) < 1e-4, (j, rel_l2(got, ref_g))
    for j in range(2):
        for name, lst in (("g_pose%d", poses), ("g_pose_inv%d", poses_inv)):
            ref_g = g.t(("loss_%s/" % tag) + name % j)
            got = lst[j].grad if lst[j].grad is not None else torch.zeros_like(ref_g)
            assert rel_l2(got, ref_g) < 1e-3, (name, j)


def test_fast_three_sources_and_multi_scale(emu_fast):
    fr = synth.make_frames(2, 40, 72, n_src=3, seed=11)
    cfg = dict(goldens.FULL_CFG, num_scales=2)
    low = [torch.nn.functional.avg_pool2d(d, 2) for d in fr["disps"]]
    res = []
    for impl in ("ours", "oracle"):
        disps = [[leaf(d), leaf(l)] for d, l in zip(fr["disps"], low)]
        args = (fr["sources"], fr["target"], [fr["poses"], fr["poses_inv"]], disps, fr["K"])
        out = losses.Compute_Loss(cfg)(*args) if impl == "ours" else O.compute_loss(cfg, *args)
        out["total"].sum().backward()
        res.append((float(out["total"].detach()), [t.grad for ds in disps for t in ds]))
    assert abs(res[0][0] - res[1][0]) <= 1e-5 * abs(res[1][0])
    for a, b in zip(res[0][1], res[1][1]):
        assert rel_l2(a, b) < 1e-4, rel_l2(a, b)


def test_min_resolve_restores_the_reference_routing():
    """tcsfm_pair_min_resolve re-evaluates exactly the near-ties of the per-pixel min, found here on the host from the
    fast flavour's forward maps: afterwards the maps hold the exact kernels' values at those pixels and the forward's
    values everywhere else, and the per-pixel arg-min over the sources is the exact arithmetic's everywhere."""
    fr = synth.make_frames(2, 40, 70, seed=4)
    # make the two sources nearly identical inside a patch so that near-ties are plentiful there
    patch = torch.zeros_like(fr["sources"][0])
    patch[:, :, 8:18, 10:25] = 1.0
    fr["sources"][1] = torch.where(patch > 0, (fr["sources"][0] + 1e-4 * torch.randn_like(fr["sources"][0])).clamp(0, 1),
                                   (fr["sources"][0] * 0.5 + 0.2))
    fr["depths"][2] = fr["depths"][1].clone()
    fr["poses"][1] = fr["poses"][0].clone()
    cfg = goldens.FULL_CFG
    K = fr["K"]

    def forward(flags):
        groups = []
        for j in range(2):
            kinv, proj = stn.projection_matrices(-fr["poses"][j], K)
            groups.append({"tgt_img": fr["target"], "ref_img": fr["sources"][j], "tgt_depth": fr["depths"][0],
                           "ref_depth": fr["depths"][1 + j], "kinv": kinv, "proj": proj})
        batch = _raw.PairBatch(groups)
        diff, mask, sums, coef = _raw.pair_loss_fwd(emu(), batch, 0.15, 0.85, flags)
        return batch, diff

    exact_flags = cfg_flags(cfg) & ~_cabi.ARITH_FAST
    _, d_exact = forward(exact_flags)
    batch, d_fast = forward(cfg_flags(cfg))
    before = d_fast.clone()
    # the kernel's rule in fp32: a NaN in either candidate, or the two closer than the band
    a, b = before.reshape(2, -1)
    band = torch.tensor(_raw.TIE_BAND, dtype=torch.float32)
    ties = a.isnan() | b.isnan() | ~(torch.maximum(a, b) - torch.minimum(a, b) >= band)
    min_sum, tie_count = _raw.pair_min_resolve(emu(), batch, [0, 1], 0.15, 0.85, cfg_flags(cfg))
    assert int(tie_count) == int(ties.sum()) > 0
    for j in range(2):
        assert torch.equal(d_fast[j].flatten()[ties], d_exact[j].flatten()[ties])          # exact values at the ties
        assert torch.equal(d_fast[j].flatten()[~ties], before[j].flatten()[~ties])         # untouched elsewhere
    assert torch.equal(torch.min(d_fast.reshape(2, -1), 0)[1], torch.min(d_exact.reshape(2, -1), 0)[1])
    assert abs(float(min_sum) - float(torch.min(before.reshape(2, -1), 0)[0].sum())) < 1e-3
