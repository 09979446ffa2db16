"""pft.photometric_loss_surface_and_grad / tcsfm_photo_sweep_grad: the loss surface of N pose hypotheses of one frame
pair and d loss_n / d poses[n] of every hypothesis in one call.

The gradient is checked two ways:

- against the batch-1 loop it replaces: compute_photometric_error of one hypothesis, the masked mean
  sum(diff * valid * weight) / sum(valid) and autograd through the library's own backward kernels.  Each row must
  agree within LOOP_REL of the row's norm (both sides are fp32 sums over every pixel in different orders);
- against float64: the oracle (oracle/ref_torch.photometric_error) evaluated in float64 with the mask of its fp32
  evaluation held constant (the mask is a comparison and carries no gradient).  The kernel's error must stay within
  test_backward_f64's RATIO_L2 / RATIO_MAX of eager fp32's error (test_backward_f64.compare over the [N,6] gradient
  of the hypotheses that see any valid pixel).

Calibration (largest figure over the cases of this file):

    kernel vs the batch-1 loop, relative to the row's norm:  emulator (x86-64, ARITH_CPU flavour) 3.7e-6
    float64 bound, kernel / eager ratio:                    emulator rel-L2 1.01, max 1.00

On the golden case and the 33x130 "wide" scene both fp32 gradients sit about 1e-2 from float64: there the float64 oracle
takes other branches of the clamps and of the floor cell at a few pixels, and both fp32 evaluations share that error
(ratio 1.00).  The "behind" and 17x65 scenes see none (2.4e-5 and 1.2e-5 for both).

Emulator tests run everywhere, the others on the GPU."""
import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden
from oracle import ref_torch as O
from tcsfm_b200 import _cabi, ops, pft, synth
from test_backward_f64 import compare, warp_scene
from test_photo_sweep import gpu_frames, hypotheses, sweep_poses

LOOP_REL = 1e-4
SUMS = ("loss", "error_sum", "valid_sum")


@pytest.fixture()
def emu_ops(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)


def loop_grad(args, poses, K):
    """The batch-1 forward + backward loop the op replaces: [N,6] pose gradients of the masked mean."""
    rows = []
    for i in range(poses.shape[0]):
        p = poses[i:i + 1, 0:6].detach().clone().requires_grad_(True)
        r = pft.compute_photometric_error(*args, p, K)
        ((r["diff_img"] * r["valid_mask"] * r["weight_mask"]).sum() / r["valid_mask"].sum()).backward()
        rows.append(p.grad[0])
    return torch.stack(rows)


def same_bits(a, b):
    """torch.equal, with NaN equal to NaN."""
    return torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num())


def check_against_loop(res, ref, tag):
    got = res["pose_grad"][:, 0:6]
    for i in range(ref.shape[0]):
        if torch.isnan(ref[i]).any():
            assert torch.isnan(got[i]).all() and float(res["valid_sum"][i]) == 0, (tag, i, got[i])
            continue
        g, r = got[i].double(), ref[i].double()
        rel = ((g - r).norm() / r.norm()).item()
        assert rel <= LOOP_REL, (tag, i, rel, got[i].tolist(), ref[i].tolist())


def oracle_grad(args, poses, K, dtype, masks):
    """[N,6] d loss_n / d poses[n] of the oracle in `dtype`, loss_n = sum((diff * mask) * weight) / sum(mask) with the
    mask given (held constant)."""
    rows = []
    for i in range(poses.shape[0]):
        x = [a.detach().to(dtype) for a in args]
        p = poses[i:i + 1].detach().to(dtype).requires_grad_(True)
        r = O.photometric_error(*x, p, K.detach().to(dtype))
        m = masks[i].to(dtype)
        ((r["diff_img"] * m * r["weight_mask"]).sum() / m.sum()).backward()
        rows.append(p.grad[0])
    return torch.stack(rows)


def check_against_f64(res, args, poses, K, tag):
    poses = poses[:, 0:6]
    with torch.no_grad():
        masks = [O.photometric_error(*args, poses[i:i + 1], K)["valid_mask"] for i in range(poses.shape[0])]
    seen = torch.tensor([float(m.sum()) > 0 for m in masks])
    assert seen.sum() >= 2, tag
    idx = seen.nonzero().flatten().tolist()
    e32 = oracle_grad(args, poses[idx], K, torch.float32, [masks[i] for i in idx])
    r64 = oracle_grad(args, poses[idx], K, torch.float64, [masks[i] for i in idx])
    compare(tag, "pose_grad", res["pose_grad"][idx, 0:6], e32, r64, {"all": torch.ones((), dtype=torch.bool)})


def golden_args(case):
    fr = Golden(case).frames()
    args = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    return args, hypotheses(fr["poses"][0][:1]), fr["K"][:1]


def scene_args(h, w, mode, device, seed=3):
    """test_backward_f64's warp scenes: part of the view leaves the image ("wide") or points fall behind the camera
    ("behind").  Their pose is inverse_warp2's argument, the hypotheses are around its negation."""
    fr, pose = warp_scene(1, h, w, mode, seed, device)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    return args, hypotheses(-pose), fr["K"]


# ------------------------------------------------------------------------------------------------ emulator

@pytest.mark.parametrize("case", goldens.CASES)
def test_pose_grad_matches_the_batch1_loop(emu_ops, case):
    args, poses, K = golden_args(case)
    res = pft.photometric_loss_surface_and_grad(*args, poses, K)
    check_against_loop(res, loop_grad(args, poses, K), case)
    assert torch.isnan(res["pose_grad"][-1]).all() and float(res["valid_sum"][-1]) == 0


@pytest.mark.parametrize("hw", [(50, 77), (17, 130)])
def test_partial_tiles(emu_ops, hw):
    fr = synth.make_frames(1, *hw, n_src=1, seed=5)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = hypotheses(fr["poses"][0])
    res = pft.photometric_loss_surface_and_grad(*args, poses, fr["K"])
    check_against_loop(res, loop_grad(args, poses, fr["K"]), hw)


@pytest.mark.parametrize("scene", [("golden",), (33, 130, "wide"), (33, 130, "behind"), (17, 65, "wide")],
                         ids=lambda s: "-".join(map(str, s)))
def test_pose_grad_vs_f64(emu_ops, scene):
    args, poses, K = golden_args(goldens.CASES[0]) if scene == ("golden",) else scene_args(*scene, device="cpu")
    res = pft.photometric_loss_surface_and_grad(*args, poses, K)
    check_against_f64(res, args, poses, K, "sweep grad %s" % (scene,))


def test_sums_are_the_forward_bits(emu_ops):
    for case in goldens.CASES:
        args, poses, K = golden_args(case)
        res = pft.photometric_loss_surface_and_grad(*args, poses, K)
        fwd = pft.photometric_loss_surface(*args, poses, K)
        for k in SUMS:
            assert same_bits(res[k], fwd[k]), (case, k)


def test_pose_grad_is_deterministic(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    a = pft.photometric_loss_surface_and_grad(*args, poses, K)
    b = pft.photometric_loss_surface_and_grad(*args, poses, K)
    assert same_bits(a["pose_grad"], b["pose_grad"])


def test_eight_column_poses(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    wide = torch.cat([poses, torch.randn(poses.shape[0], 2)], 1)
    a = pft.photometric_loss_surface_and_grad(*args, wide, K)
    b = pft.photometric_loss_surface_and_grad(*args, poses, K)
    assert a["pose_grad"].shape == wide.shape
    assert torch.equal(a["pose_grad"][:, 6:], torch.zeros(poses.shape[0], 2))
    assert same_bits(a["pose_grad"][:, 0:6], b["pose_grad"])


def test_c_abi_argument_errors():
    lib = emu()
    h, w, n = 8, 8, 2
    buf = [torch.zeros(4096) for _ in range(12)]
    p = [t.data_ptr() for t in buf]

    def call(N=n, H=h, W=w, tgt=p[0], scratch=p[6], partials=p[7], g_proj=p[9], tsc=h * w):
        return lib.tcsfm_photo_sweep_grad(tgt, tsc, p[1], h * w, p[2], p[3], p[4], p[5], scratch, partials, p[8], g_proj,
                                          N, H, W, 0.15, 0.85, _cabi.ARITH_CPU, None)

    for bad in (dict(N=0), dict(N=-3), dict(H=1), dict(W=1), dict(tgt=None), dict(scratch=None), dict(partials=None),
                dict(g_proj=None), dict(tsc=-1), dict(tsc=1 << 30)):
        assert call(**bad) != 0, bad
        assert lib.tcsfm_last_error().startswith(b"tcsfm_photo_sweep_grad"), (bad, lib.tcsfm_last_error())
    assert call() == 0
    assert lib.tcsfm_photo_sweep_grad_partial_floats(n, 20, 70) == 14 * n * 2 * 2
    assert lib.tcsfm_photo_sweep_grad_partial_floats(0, 20, 70) == 0


def test_python_layer(emu_ops):
    fr = synth.make_frames(2, 16, 24, n_src=1, seed=1)
    one = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    K = fr["K"][:1]
    poses = hypotheses(fr["poses"][0][:1])
    with pytest.raises(ValueError, match="batch 1"):
        pft.photometric_loss_surface_and_grad(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], poses,
                                              fr["K"])
    for bad in (poses[:, :5], poses[:, :6].reshape(-1), torch.zeros(0, 6), torch.zeros(3, 7)):
        with pytest.raises(ValueError, match="poses"):
            pft.photometric_loss_surface_and_grad(*one, bad, K)
    # inputs that require grad are read as values: no graph, outputs that do not require grad
    leaf = poses.clone().requires_grad_(True)
    depth = one[2].clone().requires_grad_(True)
    res = pft.photometric_loss_surface_and_grad(one[0], one[1], depth, one[3], leaf, K)
    ref = pft.photometric_loss_surface_and_grad(*one, poses, K)
    for k, v in res.items():
        assert not v.requires_grad and v.grad_fn is None, k
        assert same_bits(v, ref[k]), k
    assert res["pose_grad"].shape == poses.shape and leaf.grad is None
    # the forward-only surface still refuses them, and says where the gradient is
    with pytest.raises(NotImplementedError, match="forward only"):
        pft.photometric_loss_surface(*one, leaf, K)


def test_cpu_tensors_raise():
    fr = synth.make_frames(1, 16, 24, n_src=1, seed=1)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        pft.photometric_loss_surface_and_grad(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1],
                                              hypotheses(fr["poses"][0]), fr["K"])


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(192, 640), (376, 1242), (50, 77)])
def test_pose_grad_on_gpu(hw):
    """(192, 640) takes the batch-1 non-fused projection product, (376, 1242) the FMA chain, (50, 77) partial tiles."""
    fr = gpu_frames(*hw)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 7)
    res = pft.photometric_loss_surface_and_grad(*args, poses, fr["K"])
    fwd = pft.photometric_loss_surface(*args, poses, fr["K"])
    for k in ("error_sum", "valid_sum"):
        assert torch.equal(res[k], fwd[k]), (hw, k)
    check_against_loop(res, loop_grad(args, poses, fr["K"]), hw)
    check_against_f64(res, args, poses, fr["K"], "sweep grad %dx%d" % hw)
    assert torch.isnan(res["pose_grad"][-1]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["wide", "behind"])
def test_pose_grad_vs_f64_on_gpu(mode):
    args, poses, K = scene_args(192, 640, mode, DEV)
    res = pft.photometric_loss_surface_and_grad(*args, poses, K)
    check_against_loop(res, loop_grad(args, poses, K), mode)
    check_against_f64(res, args, poses, K, "sweep grad 192x640 %s" % mode)


@pytest.mark.gpu
def test_demo_input():
    """N = 100 hypotheses of the sweep benchmark's input (192x640, KITTI intrinsics, seed 0)."""
    fr = synth.make_frames(1, 192, 640, n_src=2, seed=0, device=DEV, intrinsics=torch.tensor(synth.KITTI_K))
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    d = torch.linspace(-0.05, 0.05, 50, device=DEV)
    poses = fr["poses"][0].repeat(100, 1)
    poses[:50, 2] += d
    poses[50:, 4] += d
    res = pft.photometric_loss_surface_and_grad(*args, poses, fr["K"])
    fwd = pft.photometric_loss_surface(*args, poses, fr["K"])
    for k in SUMS:
        assert same_bits(res[k], fwd[k]), k
    check_against_loop(res, loop_grad(args, poses, fr["K"]), "demo")
    again = pft.photometric_loss_surface_and_grad(*args, poses, fr["K"])
    assert torch.equal(again["pose_grad"], res["pose_grad"])


@pytest.mark.gpu
def test_channel_slices_give_the_same_bits():
    fr = gpu_frames(96, 160)
    stack = torch.cat([fr["target"], fr["sources"][0]], 1)
    poses = sweep_poses(fr["poses"][0], 3)[:-1]
    rest = (fr["depths"][0], fr["depths"][1], poses, fr["K"])
    a = pft.photometric_loss_surface_and_grad(stack[:, 0:3], stack[:, 3:6], *rest)
    b = pft.photometric_loss_surface_and_grad(stack[:, 0:3].contiguous(), stack[:, 3:6].contiguous(), *rest)
    for k in SUMS + ("pose_grad",):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_graph_replay_with_new_poses():
    fr = gpu_frames(192, 640)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 10)[:-1]
    static = poses.clone()

    def run():
        return pft.photometric_loss_surface_and_grad(*args, static, fr["K"])

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
    ref = pft.photometric_loss_surface_and_grad(*args, new, fr["K"])
    for k in SUMS + ("pose_grad",):
        assert torch.equal(out[k], ref[k]), k
    assert not torch.equal(out["pose_grad"], pft.photometric_loss_surface_and_grad(*args, poses, fr["K"])["pose_grad"])
