"""pft.photometric_loss_surface / photometric_loss_surface_and_grad / refine_pose_hypotheses with poses [B,N,6|8], and
tcsfm_photo_sweep_pairs / tcsfm_photo_sweep_grad_pairs / tcsfm_photo_refine_pairs: B frame pairs of N hypotheses each in
one call.  Row (b, n) of every output must have the bits of the single-pair call on pair b with poses[b], which the
sibling test files check against the batch-1 loop, the float64 oracle and torch's Adam.

Emulator tests run everywhere, the others on the GPU."""
import math

import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden
from tcsfm_b200 import _cabi, _raw, ops, pft, synth
from test_photo_sweep import hypotheses, sweep_poses
from test_photo_sweep_grad import same_bits

SURFACE = ("loss", "error_sum", "valid_sum", "diff_img", "img_rec", "valid_mask", "weight_mask")
GRAD = ("loss", "error_sum", "valid_sum", "pose_grad")
REFINE = ("poses", "best_loss", "best_step", "best_pose")


@pytest.fixture()
def emu_ops(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)
    monkeypatch.setattr(pft, "_surface_projections",
                        lambda poses, K: _raw.pose_proj_fwd(ops.lib(), poses[:, 0:6], K, -1.0, ops.pose_flags(1)))


def pair(args, b):
    return tuple(a[b:b + 1] for a in args)


def check_rows(res, ref, keys, b, tag, step_dim=False):
    """Row b of every batched output against the single-pair call's output."""
    for k in keys:
        got = res[k][:, b] if step_dim and k == "loss" else res[k][b]
        assert got.shape == ref[k].shape and got.dtype == ref[k].dtype, (tag, b, k, got.shape, ref[k].shape)
        assert same_bits(got, ref[k]), (tag, b, k)


def check_all(args, poses, K, tag, steps=3):
    """The three batched calls against the single-pair calls, pair by pair."""
    surf = pft.photometric_loss_surface(*args, poses, K, return_maps=True)
    grad = pft.photometric_loss_surface_and_grad(*args, poses, K)
    ref_ = pft.refine_pose_hypotheses(*args, poses, K, steps=steps)
    assert ref_["loss"].shape == (steps + 1,) + tuple(poses.shape[:2])
    for b in range(poses.shape[0]):
        one, Kb = pair(args, b), K[b:b + 1]
        check_rows(surf, pft.photometric_loss_surface(*one, poses[b], Kb, return_maps=True), SURFACE, b, tag)
        check_rows(grad, pft.photometric_loss_surface_and_grad(*one, poses[b], Kb), GRAD, b, tag)
        check_rows(ref_, pft.refine_pose_hypotheses(*one, poses[b], Kb, steps=steps), REFINE + ("loss",), b, tag,
                   step_dim=True)
    return surf, grad, ref_


def golden_args(case):
    fr = Golden(case).frames()
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    B = fr["target"].shape[0]
    poses = torch.stack([hypotheses(fr["poses"][0][b:b + 1]) for b in range(B)])
    return args, poses, fr["K"]


def frames_args(B, h, w, seed=5):
    fr = synth.make_frames(B, h, w, n_src=1, seed=seed)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    return args, torch.stack([hypotheses(fr["poses"][0][b:b + 1]) for b in range(B)]), fr["K"]


# ------------------------------------------------------------------------------------------------ emulator

@pytest.mark.parametrize("case", goldens.CASES)
def test_rows_are_the_single_pair_calls(emu_ops, case):
    args, poses, K = golden_args(case)
    assert poses.shape[0] == 2
    surf, _, _ = check_all(args, poses, K, case)
    assert not same_bits(surf["img_rec"][0], surf["img_rec"][1])


def test_each_pair_uses_its_own_intrinsics(emu_ops):
    """The golden cases share one K between their pairs: only here does a kernel that reads pair 0's K fail."""
    args, poses, K = golden_args(goldens.CASES[0])
    K = K.clone()
    K[1, 0, 0] *= 1.1
    check_all(args, poses, K, "fx*1.1")


def test_channel_slices_of_a_stack(emu_ops):
    args, poses, K = golden_args(goldens.CASES[1])
    stack = torch.cat([args[0], args[1]], 1)
    sliced = (stack[:, 0:3], stack[:, 3:6]) + args[2:]
    assert stack[:, 3:6].stride(0) == 6 * stack.shape[2] * stack.shape[3]
    a = pft.photometric_loss_surface(*sliced, poses, K, return_maps=True)
    b = pft.photometric_loss_surface(*args, poses, K, return_maps=True)
    for k in SURFACE:
        assert same_bits(a[k], b[k]), k
    a, b = pft.photometric_loss_surface_and_grad(*sliced, poses, K), pft.photometric_loss_surface_and_grad(*args, poses, K)
    for k in GRAD:
        assert same_bits(a[k], b[k]), k
    a = pft.refine_pose_hypotheses(*sliced, poses, K, steps=2)
    b = pft.refine_pose_hypotheses(*args, poses, K, steps=2)
    for k in REFINE + ("loss",):
        assert same_bits(a[k], b[k]), k


@pytest.mark.parametrize("hw", [(50, 77), (17, 130)])
def test_partial_tiles(emu_ops, hw):
    args, poses, K = frames_args(3, *hw)
    check_all(args, poses, K, hw)


def test_a_pair_out_of_view_beside_normal_pairs(emu_ops):
    """Every start of pair 1 leaves the view: NaN losses and frozen poses there, finite losses elsewhere."""
    args, poses, K = frames_args(3, 24, 40, seed=7)
    poses = poses[:, :-1].clone()                      # drop hypotheses()' own out-of-view row
    poses[1, :, 0] += 50.0
    _, grad, res = check_all(args, poses, K, "away", steps=3)
    assert torch.isnan(grad["loss"][1]).all() and torch.isnan(grad["pose_grad"][1]).all()
    assert torch.isnan(res["loss"][:, 1]).all() and torch.isnan(res["best_loss"][1]).all()
    assert torch.equal(res["poses"][1], poses[1]) and torch.equal(res["best_pose"][1], poses[1])
    assert res["best_step"][1].tolist() == [-1] * poses.shape[1]
    for b in (0, 2):
        assert torch.isfinite(res["loss"][:, b]).all() and torch.isfinite(grad["pose_grad"][b]).all()
        assert (res["best_step"][b] >= 0).all() and not torch.equal(res["poses"][b], poses[b])


def test_eight_column_poses(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    extra = torch.randn(poses.shape[0], poses.shape[1], 2, generator=torch.Generator().manual_seed(2))
    wide = torch.cat([poses, extra], 2)
    before = wide.clone()
    _, grad, res = check_all(args, wide, K, "[B,N,8]", steps=2)
    assert torch.equal(wide, before)
    assert grad["pose_grad"].shape == wide.shape and torch.equal(grad["pose_grad"][..., 6:], torch.zeros_like(extra))
    assert torch.equal(res["poses"][..., 6:], extra) and torch.equal(res["best_pose"][..., 6:], extra)
    narrow = pft.photometric_loss_surface_and_grad(*args, poses, K)
    assert same_bits(grad["pose_grad"][..., 0:6], narrow["pose_grad"])


def test_one_pair_in_the_batched_form_is_the_single_pair_form(emu_ops):
    args, poses, K = golden_args(goldens.CASES[2])
    one, p, Kb = pair(args, 0), poses[0], K[0:1]
    a = pft.photometric_loss_surface(*one, p[None], Kb, return_maps=True)
    b = pft.photometric_loss_surface(*one, p, Kb, return_maps=True)
    for k in SURFACE:
        assert same_bits(a[k][0], b[k]), k
    a, b = pft.photometric_loss_surface_and_grad(*one, p[None], Kb), pft.photometric_loss_surface_and_grad(*one, p, Kb)
    for k in GRAD:
        assert same_bits(a[k][0], b[k]), k
    a, b = pft.refine_pose_hypotheses(*one, p[None], Kb, steps=2), pft.refine_pose_hypotheses(*one, p, Kb, steps=2)
    for k in REFINE:
        assert same_bits(a[k][0], b[k]), k
    assert same_bits(a["loss"][:, 0], b["loss"])


def test_python_argument_errors(emu_ops):
    args, poses, K = frames_args(2, 16, 24, seed=1)
    fns = (pft.photometric_loss_surface, pft.photometric_loss_surface_and_grad, pft.refine_pose_hypotheses)
    for fn in fns:
        # 2-D poses keep the single-pair rules
        with pytest.raises(ValueError, match="batch 1"):
            fn(*args, poses[0], K)
        for bad in (poses[:, :0], poses[:0], poses[..., :5], torch.zeros(2, 3, 7)):
            with pytest.raises(ValueError, match="poses"):
                fn(*args, bad, K)
        for i in range(4):                               # one input with another B
            bad = list(args)
            bad[i] = bad[i][:1]
            with pytest.raises(ValueError, match="B = 2"):
                fn(*bad, poses, K)
        with pytest.raises(ValueError, match="intrinsics"):
            fn(*args, poses, K[:1])
        with pytest.raises(ValueError, match="target_img"):
            fn(args[0][:, :2], *args[1:], poses, K)
        with pytest.raises(ValueError):                  # another image size
            fn(args[0], args[1][..., :-1], *args[2:], poses, K)
    with pytest.raises(NotImplementedError, match="forward only"):
        pft.photometric_loss_surface(*args, poses.clone().requires_grad_(True), K)
    leaf = poses.clone().requires_grad_(True)
    for fn in fns[1:]:
        res = fn(*args, leaf, K)
        assert all(not v.requires_grad for v in res.values()) and leaf.grad is None
    with pytest.raises(ValueError, match="refine_pose_hypotheses"):
        pft.refine_pose_hypotheses(*args, poses, K, steps=-1)


def test_cpu_tensors_raise():
    args, poses, K = frames_args(2, 16, 24, seed=1)
    for fn in (pft.photometric_loss_surface, pft.photometric_loss_surface_and_grad, pft.refine_pose_hypotheses):
        with pytest.raises(RuntimeError, match="CUDA tensors only"):
            fn(*args, poses, K)


def test_c_abi_argument_errors():
    """Every check fails before a launch: the outputs keep their sentinel."""
    lib = emu()
    h, w, B, n = 8, 8, 2, 2
    hw = h * w
    buf = [torch.zeros(8192) for _ in range(20)]
    p = [t.data_ptr() for t in buf]
    sentinel = buf[12]                                   # sums / g_proj / loss

    def sweep(B=B, N=n, H=h, W=w, tsb=3 * hw, ssb=3 * hw, kinv=p[6], scratch=p[8], **_):
        return lib.tcsfm_photo_sweep_pairs(p[0], tsb, hw, p[1], ssb, hw, p[2], p[3], kinv, p[7], scratch, p[9], p[12],
                                           None, None, None, None, B, N, H, W, 0.15, 0.85, _cabi.ARITH_CPU, None)

    def grad(B=B, N=n, H=h, W=w, tsb=3 * hw, ssb=3 * hw, kinv=p[6], scratch=p[8], **_):
        return lib.tcsfm_photo_sweep_grad_pairs(p[0], tsb, hw, p[1], ssb, hw, p[2], p[3], kinv, p[7], scratch, p[9],
                                                p[13], p[12], B, N, H, W, 0.15, 0.85, _cabi.ARITH_CPU, None)

    def refine(B=B, N=n, H=h, W=w, tsb=3 * hw, ssb=3 * hw, kinv=p[6], scratch=p[8], K=p[5], steps=2):
        return lib.tcsfm_photo_refine_pairs(p[0], tsb, hw, p[1], ssb, hw, p[2], p[3], kinv, K, p[10], p[11], p[14],
                                            p[7], scratch, p[9], p[12], p[15], p[16], p[17], B, N, H, W, steps,
                                            1e-3, 0.9, 0.999, 1e-8, 0.15, 0.85, _cabi.ARITH_CPU, 0, None)

    common = [dict(B=0), dict(B=-1), dict(N=0), dict(tsb=-1), dict(ssb=-hw), dict(kinv=None), dict(scratch=None),
              dict(B=1 << 16, N=1 << 15),                 # B * N overflows int
              dict(B=1 << 15, N=1 << 15, W=70)]           # 2 tiles x 2^30 hypotheses exceed the grid
    for fn, prefix, extra in ((sweep, b"tcsfm_photo_sweep_pairs", []), (grad, b"tcsfm_photo_sweep_grad_pairs", []),
                              (refine, b"tcsfm_photo_refine_pairs",
                               [dict(K=None), dict(steps=-1), dict(B=1 << 10, N=1 << 10, steps=1 << 11)])):
        for bad in common + extra:
            sentinel.fill_(7.0)
            assert fn(**bad) != 0, (prefix, bad)
            assert lib.tcsfm_last_error().startswith(prefix), (bad, lib.tcsfm_last_error())
            assert bool((sentinel == 7.0).all()), (prefix, bad)
        sentinel.fill_(7.0)
        assert fn() == 0 and not bool((sentinel[:B * n] == 7.0).all()), prefix
        assert fn(tsb=0, ssb=0) == 0, prefix          # every pair reads the same images


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


def gpu_pairs(B, h, w, n_line, seed=23):
    """B pairs of the synthetic scene, pair b's fx scaled by 1 + 0.05 b, with sweep_poses of each pair's pose."""
    fr = synth.make_frames(B, h, w, n_src=2, seed=seed, device=DEV, intrinsics=synth.scaled_intrinsics(h, w))
    K = fr["K"].clone()
    K[:, 0, 0] *= 1.0 + 0.05 * torch.arange(B, device=DEV)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = torch.stack([sweep_poses(fr["poses"][0][b:b + 1], n_line) for b in range(B)])
    return args, poses, K


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 192, 640), (2, 376, 1242), (3, 50, 77)])
def test_rows_are_the_single_pair_calls_on_gpu(shape):
    """(192, 640) takes the batch-1 non-fused projection product, (376, 1242) the FMA chain, (50, 77) partial tiles."""
    args, poses, K = gpu_pairs(*shape, n_line=3)
    check_all(args, poses, K, shape, steps=5)


@pytest.mark.gpu
def test_many_pairs_on_gpu():
    """B = 32, N = 9: 288 hypotheses span three blocks of the finish and step kernels.  The ninth start repeats the
    first (padding with duplicate starts) and gets its bits."""
    args, poses, K = gpu_pairs(32, 96, 160, n_line=3, seed=5)
    poses = torch.cat([poses, poses[:, :1]], 1)
    assert poses.shape[:2] == (32, 9)
    _, grad, res = check_all(args, poses, K, "B=32", steps=3)
    assert same_bits(grad["pose_grad"][:, 8], grad["pose_grad"][:, 0]) and same_bits(res["loss"][..., 8], res["loss"][..., 0])


@pytest.mark.gpu
def test_channel_slices_on_gpu():
    args, poses, K = gpu_pairs(3, 96, 160, n_line=3)
    stack = torch.cat([args[0], args[1]], 1)
    a = pft.refine_pose_hypotheses(stack[:, 0:3], stack[:, 3:6], *args[2:], poses, K, steps=3)
    b = pft.refine_pose_hypotheses(*args, poses, K, steps=3)
    for k in REFINE + ("loss",):
        assert same_bits(a[k], b[k]), k


@pytest.mark.gpu
def test_graph_replay_of_the_batched_refine():
    args, poses, K = gpu_pairs(4, 192, 640, n_line=4)
    static = poses.clone()

    def run():
        return pft.refine_pose_hypotheses(*args, static, K, steps=4)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
    new = poses.clone()
    new[..., 2] += 0.01
    new[..., 5] -= 0.003
    static.copy_(new)
    graph.replay()
    torch.cuda.synchronize()
    ref = pft.refine_pose_hypotheses(*args, new, K, steps=4)
    for k in REFINE + ("loss",):
        assert same_bits(out[k], ref[k]), k
    assert not torch.equal(out["loss"], pft.refine_pose_hypotheses(*args, poses, K, steps=4)["loss"])
    assert math.isfinite(float(out["best_loss"][0, 0]))
