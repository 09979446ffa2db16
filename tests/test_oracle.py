"""Pins oracle/ref_torch.py (the CPU restatement) to the reference: bit-for-bit
against the committed golden vectors that the unmodified reference produced; the
stored fresh-input vectors are also checked against the live reference where
TCSFM_REFERENCE_ROOT names a checkout of it."""
import types

import pytest
import torch

import goldens
import refshim
from goldens import Golden
from oracle import ref_torch as O
from tcsfm_b200 import synth


def leaf(t):
    return t.clone().detach().requires_grad_(True)


def same(a, b):
    return torch.equal(a.detach().float().cpu(), b.detach().float().cpu())


def close_scalar(a, b, rtol=2e-6):
    a, b = float(torch.as_tensor(a).sum()), float(torch.as_tensor(b).sum())
    return abs(a - b) <= rtol * max(abs(a), abs(b), 1e-12)


@pytest.fixture(autouse=True)
def _one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)     # fixtures were generated single-threaded
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("case", goldens.CASES)
def test_warp_matches_golden(case):
    g = Golden(case)
    fr = g.frames()
    d0, d1, p0 = leaf(fr["depths"][0]), leaf(fr["depths"][1]), leaf(-fr["poses"][0])
    pim, vm, pd, cd = O.inverse_warp2(fr["sources"][0], d0, d1, p0, fr["K"])
    assert same(vm, g.t("warp/valid_mask"))
    assert same(pim, g.t("warp/projected_img"))
    assert same(pd, g.t("warp/projected_depth"))
    assert same(cd, g.t("warp/computed_depth"))
    ((pim * g.t("in/g_img")).sum() + (pd * g.t("in/g_pd")).sum() + (cd * g.t("in/g_cd")).sum()).backward()
    assert goldens.rel_l2(d0.grad, g.t("warp/g_depth")) < 1e-6
    assert goldens.rel_l2(d1.grad, g.t("warp/g_ref_depth")) < 1e-6
    assert goldens.rel_l2(p0.grad, g.t("warp/g_pose")) < 1e-5


@pytest.mark.parametrize("case", goldens.CASES)
def test_ssim_matches_golden(case):
    g = Golden(case)
    x, y = leaf(g.t("in/target")), leaf(g.t("in/source0"))
    s = O.ssim_dissimilarity(x, y)
    assert same(s, g.t("ssim/map"))
    (s * g.t("in/g_img")).sum().backward()
    assert same(x.grad, g.t("ssim/g_x")) and same(y.grad, g.t("ssim/g_y"))


@pytest.mark.parametrize("case", goldens.CASES)
@pytest.mark.parametrize("tag", ["train", "full", "noauto"])
def test_pairwise_matches_golden(case, tag):
    g = Golden(case)
    fr = g.frames()
    d0, d1, p0 = leaf(fr["depths"][0]), leaf(fr["depths"][1]), leaf(-fr["poses"][0])
    l_rep, l_dep, diff, vmask, _ = O.pairwise_loss(goldens.PAIR_CFGS[tag], fr["target"], fr["sources"][0],
                                                   d0, d1, p0, fr["K"])
    assert same(vmask, g.t("pair_%s/valid_mask" % tag))
    assert same(diff, g.t("pair_%s/diff_img" % tag))
    assert close_scalar(l_rep, g.t("pair_%s/l_reprojection" % tag))
    assert close_scalar(l_dep, g.t("pair_%s/l_depth" % tag))
    obj = l_rep + (diff * g.t("in/g_diff")).sum()
    if torch.is_tensor(l_dep):
        obj = obj + 0.5 * l_dep
    obj.backward()
    assert goldens.rel_l2(d0.grad, g.t("pair_%s/g_depth" % tag)) < 1e-6
    assert goldens.rel_l2(p0.grad, g.t("pair_%s/g_pose" % tag)) < 1e-5


@pytest.mark.parametrize("case", goldens.CASES)
@pytest.mark.parametrize("tag", ["train", "full", "smooth"])
def test_compute_loss_matches_golden(case, tag):
    g = Golden(case)
    fr = g.frames()
    disps = [leaf(d) for d in fr["disps"]]
    poses, poses_inv = [leaf(p) for p in fr["poses"]], [leaf(p) for p in fr["poses_inv"]]
    out = O.compute_loss(goldens.LOSS_CFGS[tag], fr["sources"], fr["target"], [poses, poses_inv],
                         [[disps[0]], [disps[1]], [disps[2]]], fr["K"])
    for k in ("l_reconstruct_inverse", "l_reconstruct_forward", "l_depth", "l_smooth", "total"):
        assert out[k].shape == (1,)
        assert close_scalar(out[k], g.t("loss_%s/%s" % (tag, k))), k
    out["total"].sum().backward()
    for j in range(3):
        ref_g = g.t("loss_%s/g_disp%d" % (tag, j))
        got = disps[j].grad if disps[j].grad is not None else torch.zeros_like(ref_g)
        assert goldens.rel_l2(got, ref_g) < 1e-5


@pytest.mark.parametrize("case", goldens.CASES)
def test_pft_matches_golden(case):
    g = Golden(case)
    fr = g.frames()
    seed = {"small_b2_24x40": 1, "mid_b2_64x96": 2, "yaw_b2_32x48": 3}[case]
    net = synth.TinyPoseNet(seed=seed)
    dl = [leaf(d) for d in fr["depths"]]
    poses, poses_inv, outputs = O.iterative_pose(3, dl, net, fr["target"], fr["sources"], fr["K"], return_errors=True)
    for side in ("fwd", "inv"):
        for k in ("diff_img", "valid_mask", "weight_mask", "auto_mask_error", "auto_mask"):
            assert same(outputs[side][k], g.t("pft/%s/%s" % (side, k))), (side, k)
    for j in range(2):
        assert same(poses[j], g.t("pft/pose%d" % j)) and same(poses_inv[j], g.t("pft/pose_inv%d" % j))
    tdisp = leaf(fr["disps"][0])
    loss = O.pft_window_loss(goldens.PFT_OPTIONS, fr["target"], tdisp, fr["disps"][0] * 0.9 + 0.02,
                             outputs["fwd"], outputs["inv"])
    assert close_scalar(loss, g.t("pft/loss"))
    loss.sum().backward()
    assert goldens.rel_l2(tdisp.grad, g.t("pft/g_tdisp")) < 1e-6
    for j in range(3):
        assert goldens.rel_l2(dl[j].grad, g.t("pft/g_depth%d" % j)) < 1e-5


@pytest.mark.parametrize("case", goldens.CASES)
def test_photometric_error_matches_golden(case):
    g = Golden(case)
    fr = g.frames()
    with torch.no_grad():
        res = O.photometric_error(fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1],
                                  fr["depths"][1][:1], fr["poses"][0][:1], fr["K"][:1])
    for k in ("diff_img", "img_rec", "valid_mask", "weight_mask"):
        assert same(res[k], g.t("photo/%s" % k)), k


def test_oracle_matches_live_reference_on_fresh_inputs():
    """Inputs that none of the golden cases uses (the second source warped with the outer depths, both euler2mat, the
    smoothness loss, the pairwise diff / mask), against the outputs stored in tests/golden/fresh/ (its `source` entry
    names what wrote them; test_fresh_fixture_matches_live_reference checks them against the reference itself)."""
    fr = synth.make_frames(**goldens.FRESH_FRAMES)
    stored = goldens.load_fresh()
    assert goldens.fresh_inputs_digest(fr) == str(stored["in/sha256"]), "the seeded inputs changed"
    for k, v in goldens.fresh_outputs(fr, **goldens.fresh_fns_oracle()).items():
        assert same(v, torch.from_numpy(stored[k])), k


@pytest.mark.skipif(not refshim.reference_available(), reason="needs TCSFM_REFERENCE_ROOT: a checkout of the reference")
def test_fresh_fixture_matches_live_reference():
    ref = refshim.load_reference()
    fr = synth.make_frames(**goldens.FRESH_FRAMES)
    stored = goldens.load_fresh()
    for k, v in goldens.fresh_outputs(fr, **goldens.fresh_fns_reference(ref)).items():
        assert same(v, torch.from_numpy(stored[k])), k
