"""pft.photometric_loss_surface / tcsfm_photo_sweep: compute_photometric_error (helpers.py:8-23) of one frame pair
under N pose hypotheses in one call.  The maps must be the bits of N batch-1 compute_photometric_error calls; the
sums are checked against the maps.  Emulator tests run everywhere, the others on the GPU."""
import ctypes as C

import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden
from tcsfm_b200 import _cabi, ops, pft, synth

MAPS = ("diff_img", "img_rec", "valid_mask", "weight_mask")


@pytest.fixture()
def emu_ops(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)


def hypotheses(pose, t=(0.02,), yaw=(0.01,)):
    """[N,6]: the pose itself, +- each translation step along z, +- each yaw step, and one pose that sends every
    pixel out of view (last row)."""
    rows = [pose[0].clone()]
    for axis, steps in ((2, t), (4, yaw)):
        for d in steps:
            for s in (1.0, -1.0):
                p = pose[0].clone()
                p[axis] += s * d
                rows.append(p)
    away = pose[0].clone()
    away[0] += 50.0
    rows.append(away)
    return torch.stack(rows)


def loop(args, poses, K):
    """The batch-1 loop the op replaces."""
    return [pft.compute_photometric_error(*args, poses[i:i + 1], K) for i in range(poses.shape[0])]


def check_against_loop(res, refs):
    for i, r in enumerate(refs):
        for k in MAPS:
            assert torch.equal(res[k][i:i + 1], r[k]), (i, k, int((res[k][i:i + 1] != r[k]).sum()))
    check_sums(res, refs)


def check_sums(res, refs):
    for i, r in enumerate(refs):
        vs = r["valid_mask"].sum()
        assert float(res["valid_sum"][i]) == float(vs), i
        exact = float((r["diff_img"] * r["valid_mask"] * r["weight_mask"]).double().sum())
        assert abs(float(res["error_sum"][i]) - exact) <= 2e-6 * abs(exact), (i, float(res["error_sum"][i]), exact)
        if float(vs) == 0:
            assert torch.isnan(res["loss"][i])
        else:
            assert torch.equal(res["loss"][i], res["error_sum"][i] / res["valid_sum"][i])


# ------------------------------------------------------------------------------------------------ emulator

@pytest.mark.parametrize("case", goldens.CASES)
def test_maps_and_sums_match_the_batch1_loop(emu_ops, case):
    fr = Golden(case).frames()
    args = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    K = fr["K"][:1]
    poses = hypotheses(fr["poses"][0][:1])
    with torch.no_grad():
        res = pft.photometric_loss_surface(*args, poses, K, return_maps=True)
        refs = loop(args, poses, K)
    check_against_loop(res, refs)
    assert float(res["valid_sum"][-1]) == 0 and torch.isnan(res["loss"][-1])
    assert float(res["valid_sum"][0]) > 0


def test_sums_are_deterministic(emu_ops):
    fr = Golden(goldens.CASES[0]).frames()
    args = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    poses = hypotheses(fr["poses"][0][:1])
    a = pft.photometric_loss_surface(*args, poses, fr["K"][:1])
    b = pft.photometric_loss_surface(*args, poses, fr["K"][:1])
    for k in ("error_sum", "valid_sum"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("hw", [(50, 77), (17, 130)])
def test_partial_tiles(emu_ops, hw):
    h, w = hw
    fr = synth.make_frames(1, h, w, n_src=1, seed=5)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = hypotheses(fr["poses"][0])
    with torch.no_grad():
        res = pft.photometric_loss_surface(*args, poses, fr["K"], return_maps=True)
        refs = loop(args, poses, fr["K"])
    check_against_loop(res, refs)


def test_c_abi_argument_errors():
    lib = emu()
    h, w, n = 8, 8, 2
    buf = [torch.zeros(4096) for _ in range(12)]
    p = [t.data_ptr() for t in buf]

    def call(N=n, H=h, W=w, tgt=p[0], scratch=p[6]):
        return lib.tcsfm_photo_sweep(tgt, h * w, p[1], h * w, p[2], p[3], p[4], p[5], scratch, p[7], p[8],
                                     None, None, None, None, N, H, W, 0.15, 0.85, _cabi.ARITH_CPU, None)

    for bad in (dict(N=0), dict(N=-3), dict(H=1), dict(W=1), dict(tgt=None), dict(scratch=None)):
        assert call(**bad) != 0, bad
        assert lib.tcsfm_last_error().startswith(b"tcsfm_photo_sweep"), (bad, lib.tcsfm_last_error())
    assert call() == 0
    assert lib.tcsfm_photo_sweep_partial_floats(n, 20, 70) == 2 * n * 2 * 2


def test_python_layer_rejects_bad_inputs(emu_ops):
    fr = synth.make_frames(2, 16, 24, n_src=1, seed=1)
    one = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    K = fr["K"][:1]
    poses = hypotheses(fr["poses"][0][:1])
    with pytest.raises(ValueError, match="batch 1"):
        pft.photometric_loss_surface(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], poses, fr["K"])
    for bad in (poses[:, :5], poses[:, :6].reshape(-1), torch.zeros(0, 6), torch.zeros(3, 7)):
        with pytest.raises(ValueError, match="poses"):
            pft.photometric_loss_surface(*one, bad, K)
    with pytest.raises(NotImplementedError, match="forward only"):
        pft.photometric_loss_surface(*one, poses.clone().requires_grad_(True), K)
    with pytest.raises(NotImplementedError, match="forward only"):
        pft.photometric_loss_surface(one[0], one[1], one[2].clone().requires_grad_(True), one[3], poses, K)
    with torch.no_grad():        # requires_grad inputs are fine where no graph is recorded
        pft.photometric_loss_surface(*one, poses.clone().requires_grad_(True), K)


def test_cpu_tensors_raise():
    fr = synth.make_frames(1, 16, 24, n_src=1, seed=1)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        pft.photometric_loss_surface(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1],
                                     hypotheses(fr["poses"][0]), fr["K"])


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


def gpu_frames(h, w, seed=23, intrinsics=None):
    k = synth.scaled_intrinsics(h, w) if intrinsics is None else intrinsics
    return synth.make_frames(1, h, w, n_src=2, seed=seed, device=DEV, intrinsics=k)


def sweep_poses(pose, n_line):
    """n_line translation and n_line yaw samples of the demo's +-0.05 lines, the pose itself and one out-of-view pose."""
    d = torch.linspace(-0.05, 0.05, n_line, device=pose.device)
    rows = [pose[0].clone()]
    for axis in (2, 4):
        p = pose[0].repeat(n_line, 1)
        p[:, axis] += d
        rows += list(p)
    away = pose[0].clone()
    away[0] += 50.0
    rows.append(away)
    return torch.stack(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(192, 640), (376, 1242), (50, 77)])
def test_maps_bit_identical_on_gpu(hw):
    """(192, 640) takes the batch-1 non-fused projection product, (376, 1242) the FMA chain, (50, 77) partial tiles."""
    from oracle import ref_torch as O
    fr = gpu_frames(*hw)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 7)
    assert poses.shape[0] == 16
    with torch.no_grad():
        res = pft.photometric_loss_surface(*args, poses, fr["K"], return_maps=True)
        refs = loop(args, poses, fr["K"])
        for i in range(poses.shape[0]):
            o = O.photometric_error(*args, poses[i:i + 1], fr["K"])
            for k in MAPS:
                assert torch.equal(res[k][i:i + 1], o[k]), (hw, i, k)
    check_against_loop(res, refs)
    assert float(res["valid_sum"][-1]) == 0 and torch.isnan(res["loss"][-1])


@pytest.mark.gpu
def test_sums_on_the_demo_input():
    """N = 100 hypotheses of the sweep benchmark's input (192x640, KITTI intrinsics, seed 0)."""
    fr = synth.make_frames(1, 192, 640, n_src=2, seed=0, device=DEV, intrinsics=torch.tensor(synth.KITTI_K))
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    d = torch.linspace(-0.05, 0.05, 50, device=DEV)
    poses = fr["poses"][0].repeat(100, 1)
    poses[:50, 2] += d
    poses[50:, 4] += d
    with torch.no_grad():
        res = pft.photometric_loss_surface(*args, poses, fr["K"], return_maps=True)
        refs = loop(args, poses, fr["K"])
    check_against_loop(res, refs)
    again = pft.photometric_loss_surface(*args, poses, fr["K"])
    for k in ("loss", "error_sum", "valid_sum"):
        assert torch.equal(again[k], res[k]), k


@pytest.mark.gpu
def test_channel_slices_give_the_same_bits():
    fr = gpu_frames(96, 160)
    stack = torch.cat([fr["target"], fr["sources"][0]], 1)
    poses = sweep_poses(fr["poses"][0], 3)
    rest = (fr["depths"][0], fr["depths"][1], poses, fr["K"])
    with torch.no_grad():
        a = pft.photometric_loss_surface(stack[:, 0:3], stack[:, 3:6], *rest, return_maps=True)
        b = pft.photometric_loss_surface(stack[:, 0:3].contiguous(), stack[:, 3:6].contiguous(), *rest, return_maps=True)
    for k in MAPS + ("error_sum", "valid_sum"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_graph_replay_with_new_poses():
    fr = gpu_frames(192, 640)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 10)
    static = poses.clone()

    def run():
        return pft.photometric_loss_surface(*args, static, fr["K"], return_maps=True)

    with torch.no_grad():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = run()
        new = poses.clone()
        new[:, 2] += 0.01
        new[:, 5] -= 0.003
        static.copy_(new)
        graph.replay()
        torch.cuda.synchronize()
        ref = pft.photometric_loss_surface(*args, new, fr["K"], return_maps=True)
    for k in MAPS + ("error_sum", "valid_sum"):
        assert torch.equal(out[k], ref[k]), k
    assert not torch.equal(out["error_sum"], pft.photometric_loss_surface(*args, poses, fr["K"])["error_sum"])
