"""pft.refine_pose_hypotheses / tcsfm_photo_refine: Adam descent of the photometric loss surface from N starting poses
of one frame pair in one call.

The reference is the loop a user writes with the library's surface functions: per step
photometric_loss_surface_and_grad, then the update rule of refine_pose_hypotheses as separate torch operators on fp32
tensors (each scalar a 0-d fp32 tensor on the poses' device, so that no division turns into a multiplication by a
reciprocal; the square root taken in float64 and rounded once), a row with valid_sum 0 left as it is;
photometric_loss_surface for the last row of the history; best_* on the host.  The call must give the bits of that loop.

On the emulator the reference forms K[R|t] with the library's pose kernel, as it does on CUDA tensors (the eager CPU
operators of the CPU branch round the pose algebra differently, and the refinement forms K[R|t] on the device).

Emulator tests run everywhere, the others on the GPU."""
import math

import pytest
import torch

import goldens
from emu_lib import emu
from goldens import Golden
from tcsfm_b200 import _cabi, _raw, ops, pft, synth
from test_photo_sweep import gpu_frames, hypotheses, sweep_poses
from test_photo_sweep_grad import same_bits

OUT = ("poses", "loss", "best_loss", "best_step", "best_pose")


@pytest.fixture()
def emu_ops(monkeypatch):
    monkeypatch.setattr(ops, "lib", emu)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "ARITH_FLAGS", _cabi.ARITH_CPU)
    monkeypatch.setattr(pft, "_surface_projections",
                        lambda poses, K: _raw.pose_proj_fwd(ops.lib(), poses[:, 0:6], K, -1.0, ops.pose_flags(1)))


def reference(args, poses, K, steps, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
    """The refinement as a loop of surface calls and torch operators."""
    dev = poses.device

    def f32(x):
        return torch.tensor(x, dtype=torch.float32, device=dev)

    b1, b2 = betas
    p = poses[:, 0:6].clone()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    rows, path = [], [p]
    for t in range(1, steps + 1):
        r = pft.photometric_loss_surface_and_grad(*args, p, K)
        rows.append(r["loss"])
        g = r["pose_grad"]
        c1, c2 = f32(lr / (1 - b1 ** t)), f32(math.sqrt(1 - b2 ** t))
        m_new = f32(b1) * m + f32(1 - b1) * g
        v_new = f32(b2) * v + f32(1 - b2) * (g * g)
        # sqrt through float64: the fp32 square root rounded once, which torch's CPU kernel does not give
        p_new = p - c1 * (m_new / (v_new.double().sqrt().float() / c2 + f32(eps)))
        live = (r["valid_sum"] > 0)[:, None]
        m, v, p = torch.where(live, m_new, m), torch.where(live, v_new, v), torch.where(live, p_new, p)
        path.append(p)
    rows.append(pft.photometric_loss_surface(*args, p, K)["loss"])
    loss = torch.stack(rows)
    n = poses.shape[0]
    best_loss = torch.full((n,), float("nan"), device=dev)
    best_step = torch.full((n,), -1, dtype=torch.int64, device=dev)
    best_pose = poses[:, 0:6].clone()
    host = loss.cpu().tolist()
    for i in range(n):
        for k in range(steps + 1):
            x = host[k][i]
            if math.isfinite(x) and (best_step[i] < 0 or x < best_loss[i].item()):
                best_loss[i], best_step[i], best_pose[i] = loss[k, i], k, path[k][i]
    if poses.shape[1] > 6:
        p = torch.cat([p, poses[:, 6:]], 1)
        best_pose = torch.cat([best_pose, poses[:, 6:]], 1)
    return {"poses": p, "loss": loss, "best_loss": best_loss, "best_step": best_step, "best_pose": best_pose}


def check_same(res, ref, tag):
    for k in OUT:
        assert res[k].shape == ref[k].shape and res[k].dtype == ref[k].dtype, (tag, k, res[k].shape, ref[k].shape)
        assert same_bits(res[k], ref[k]), (tag, k, res[k], ref[k])


def golden_args(case):
    fr = Golden(case).frames()
    args = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    return args, hypotheses(fr["poses"][0][:1]), fr["K"][:1]


def first_frozen_step(loss_col):
    """The first k > 0 with a NaN loss after a finite one, or None."""
    for k in range(1, len(loss_col)):
        if math.isnan(loss_col[k]) and math.isfinite(loss_col[k - 1]):
            return k
    return None


# ------------------------------------------------------------------------------------------------ emulator

@pytest.mark.parametrize("case", goldens.CASES)
def test_matches_the_reference_loop(emu_ops, case):
    args, poses, K = golden_args(case)
    res = pft.refine_pose_hypotheses(*args, poses, K, steps=4)
    check_same(res, reference(args, poses, K, 4), case)
    # the last hypothesis sees no pixel: it keeps its starting pose, has no loss and no best step
    assert torch.equal(res["poses"][-1], poses[-1]) and torch.equal(res["best_pose"][-1], poses[-1])
    assert torch.isnan(res["loss"][:, -1]).all() and int(res["best_step"][-1]) == -1
    assert torch.isnan(res["best_loss"][-1])
    assert not torch.equal(res["poses"][:-1], poses[:-1])


@pytest.mark.parametrize("hw", [(50, 77), (17, 130)])
def test_partial_tiles(emu_ops, hw):
    fr = synth.make_frames(1, *hw, n_src=1, seed=5)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = hypotheses(fr["poses"][0])
    res = pft.refine_pose_hypotheses(*args, poses, fr["K"], steps=3)
    check_same(res, reference(args, poses, fr["K"], 3), hw)


def test_row_that_leaves_the_view_freezes(emu_ops):
    """Starts shifted sideways to the edge of validity (about 0.35 on this case, where a few pixels stay valid): some
    descend back into the view, some leave it after an update or two."""
    args, poses, K = golden_args(goldens.CASES[0])
    starts = poses[0].repeat(6, 1)
    starts[:, 0] += torch.tensor([0.3, 0.32, 0.34, 0.345, -0.3, -0.34])
    steps, lr = 3, 0.01
    res = pft.refine_pose_hypotheses(*args, starts, K, steps=steps, lr=lr)
    check_same(res, reference(args, starts, K, steps, lr=lr), "edge")
    loss = res["loss"].t().tolist()
    assert all(math.isfinite(col[0]) for col in loss), loss
    frozen = [(i, first_frozen_step(col)) for i, col in enumerate(loss) if first_frozen_step(col) is not None]
    assert len(frozen) >= 2 and len(frozen) < len(loss), loss
    for i, k in frozen:
        assert all(math.isnan(x) for x in loss[i][k:]), (i, loss[i])
        assert 0 <= int(res["best_step"][i]) < k
    # a frozen row keeps the pose it reached: one more step does not move it
    more = pft.refine_pose_hypotheses(*args, starts, K, steps=steps + 1, lr=lr)
    for i, _ in frozen:
        assert torch.equal(more["poses"][i], res["poses"][i]), i


def test_zero_steps_evaluates_the_start(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    res = pft.refine_pose_hypotheses(*args, poses, K, steps=0)
    assert res["loss"].shape == (1, poses.shape[0])
    assert same_bits(res["loss"][0], pft.photometric_loss_surface(*args, poses, K)["loss"])
    assert torch.equal(res["poses"], poses) and torch.equal(res["best_pose"], poses)
    assert res["best_step"].tolist() == [0] * (poses.shape[0] - 1) + [-1]
    check_same(res, reference(args, poses, K, 0), "steps=0")


def test_eight_column_poses_and_the_input_is_not_written(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    wide = torch.cat([poses, torch.randn(poses.shape[0], 2, generator=torch.Generator().manual_seed(2))], 1)
    before = wide.clone()
    res = pft.refine_pose_hypotheses(*args, wide, K, steps=2)
    assert torch.equal(wide, before)
    assert res["poses"].shape == wide.shape and res["best_pose"].shape == wide.shape
    assert torch.equal(res["poses"][:, 6:], wide[:, 6:]) and torch.equal(res["best_pose"][:, 6:], wide[:, 6:])
    narrow = pft.refine_pose_hypotheses(*args, poses, K, steps=2)
    for k in OUT:
        assert same_bits(res[k][..., 0:6] if k in ("poses", "best_pose") else res[k], narrow[k]), k


def test_two_calls_give_the_same_bits(emu_ops):
    args, poses, K = golden_args(goldens.CASES[0])
    a = pft.refine_pose_hypotheses(*args, poses, K, steps=2)
    b = pft.refine_pose_hypotheses(*args, poses, K, steps=2)
    for k in OUT:
        assert same_bits(a[k], b[k]), k


def test_one_step_is_adam(emu_ops):
    """The displacement of one step is torch.optim.Adam's, fed the same gradient."""
    args, poses, K = golden_args(goldens.CASES[0])
    lr, betas, eps = 3e-3, (0.8, 0.99), 1e-6
    res = pft.refine_pose_hypotheses(*args, poses, K, steps=1, lr=lr, betas=betas, eps=eps)
    r = pft.photometric_loss_surface_and_grad(*args, poses, K)
    live = (r["valid_sum"] > 0).nonzero().flatten()
    leaf = poses[live].clone().requires_grad_(True)
    opt = torch.optim.Adam([leaf], lr=lr, betas=betas, eps=eps, foreach=False)
    leaf.grad = r["pose_grad"][live].clone()
    opt.step()
    want = (leaf.detach() - poses[live]).double()
    got = (res["poses"][live] - poses[live]).double()
    assert float((got - want).norm()) <= 1e-5 * float(want.norm()), (got, want)


def test_default_lr_descends(emu_ops):
    """From yaw +-0.01 off the pose of the yaw golden case, the default settings end below the start."""
    fr = Golden("yaw_b2_32x48").frames()
    args = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    starts = fr["poses"][0][:1].repeat(2, 1)
    starts[:, 4] += torch.tensor([0.01, -0.01])
    res = pft.refine_pose_hypotheses(*args, starts, fr["K"][:1])
    assert res["loss"].shape == (51, 2)
    assert bool((res["loss"][-1] < res["loss"][0]).all()), res["loss"][[0, -1]]


def test_c_abi_argument_errors():
    lib = emu()
    h, w, n = 8, 8, 2
    buf = [torch.zeros(4096) for _ in range(18)]
    p = [t.data_ptr() for t in buf]

    def call(N=n, H=h, W=w, steps=2, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, **ptrs):
        ptr = {k: p[i] for i, k in enumerate(("tgt", "src", "td", "sd", "kinv", "K", "poses", "m", "v", "proj", "scratch",
                                              "partials", "loss", "best_loss", "best_step", "best_pose"))}
        ptr.update(ptrs)
        return lib.tcsfm_photo_refine(ptr["tgt"], h * w, ptr["src"], h * w, ptr["td"], ptr["sd"], ptr["kinv"], ptr["K"],
                                      ptr["poses"], ptr["m"], ptr["v"], ptr["proj"], ptr["scratch"], ptr["partials"],
                                      ptr["loss"], ptr["best_loss"], ptr["best_step"], ptr["best_pose"],
                                      N, H, W, steps, lr, beta1, beta2, eps, 0.15, 0.85, _cabi.ARITH_CPU, 0, None)

    bad_args = [dict(N=0), dict(H=1), dict(steps=-1), dict(steps=1 << 30, N=4), dict(steps=0x7fffffff),
                dict(lr=0.0), dict(lr=float("inf")), dict(eps=-1.0), dict(eps=float("nan")), dict(beta1=1.0),
                dict(beta2=-0.1)]
    bad_args += [{k: None} for k in ("tgt", "kinv", "K", "poses", "m", "v", "proj", "scratch", "partials", "loss",
                                     "best_loss", "best_step", "best_pose")]
    for bad in bad_args:
        assert call(**bad) != 0, bad
        assert lib.tcsfm_last_error().startswith(b"tcsfm_photo_refine"), (bad, lib.tcsfm_last_error())
    assert call() == 0
    assert call(steps=0) == 0


def test_python_layer(emu_ops):
    fr = synth.make_frames(2, 16, 24, n_src=1, seed=1)
    one = (fr["target"][:1], fr["sources"][0][:1], fr["depths"][0][:1], fr["depths"][1][:1])
    K = fr["K"][:1]
    poses = hypotheses(fr["poses"][0][:1])
    with pytest.raises(ValueError, match="batch 1"):
        pft.refine_pose_hypotheses(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], poses, fr["K"])
    for bad in (poses[:, :5], poses[:, :6].reshape(-1), torch.zeros(0, 6), torch.zeros(3, 7)):
        with pytest.raises(ValueError, match="poses"):
            pft.refine_pose_hypotheses(*one, bad, K)
    for bad in (dict(steps=-1), dict(steps=2.0), dict(steps=True), dict(steps="3"), dict(lr=0), dict(lr=-1e-3),
                dict(lr=float("inf")), dict(lr=float("nan")), dict(lr="fast"), dict(eps=0.0), dict(eps=float("inf")),
                dict(betas=(1.0, 0.999)), dict(betas=(0.9, -0.1)), dict(betas=(0.9,)), dict(betas=(0.9, 0.99, 0.9)),
                dict(betas=0.9), dict(betas=(0.9, float("nan")))):
        with pytest.raises(ValueError, match="refine_pose_hypotheses"):
            pft.refine_pose_hypotheses(*one, poses, K, **bad)
    # inputs that require grad are read as values: no graph, outputs that do not require grad
    leaf = poses.clone().requires_grad_(True)
    depth = one[2].clone().requires_grad_(True)
    res = pft.refine_pose_hypotheses(one[0], one[1], depth, one[3], leaf, K, steps=1)
    ref = pft.refine_pose_hypotheses(*one, poses, K, steps=1)
    for k in OUT:
        assert not res[k].requires_grad and res[k].grad_fn is None, k
        assert same_bits(res[k], ref[k]), k
    assert leaf.grad is None and torch.equal(leaf.detach(), poses)
    assert res["best_step"].dtype == torch.int64


def test_cpu_tensors_raise():
    fr = synth.make_frames(1, 16, 24, n_src=1, seed=1)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        pft.refine_pose_hypotheses(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1],
                                   hypotheses(fr["poses"][0]), fr["K"])


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(192, 640), (376, 1242), (50, 77)])
def test_matches_the_reference_loop_on_gpu(hw):
    """(192, 640) takes the batch-1 non-fused projection product, (376, 1242) the FMA chain, (50, 77) partial tiles."""
    fr = gpu_frames(*hw)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 7)
    res = pft.refine_pose_hypotheses(*args, poses, fr["K"], steps=5)
    check_same(res, reference(args, poses, fr["K"], 5), hw)
    assert torch.isnan(res["loss"][:, -1]).all() and torch.equal(res["poses"][-1], poses[-1])


@pytest.mark.gpu
def test_many_hypotheses_on_gpu():
    """N = 300: the step kernel spans three 128-thread blocks."""
    fr = gpu_frames(96, 160)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 149)
    assert poses.shape[0] == 300
    res = pft.refine_pose_hypotheses(*args, poses, fr["K"], steps=3)
    check_same(res, reference(args, poses, fr["K"], 3), "N=300")


@pytest.mark.gpu
def test_channel_slices_give_the_same_bits():
    fr = gpu_frames(96, 160)
    stack = torch.cat([fr["target"], fr["sources"][0]], 1)
    poses = sweep_poses(fr["poses"][0], 3)
    rest = (fr["depths"][0], fr["depths"][1], poses, fr["K"])
    a = pft.refine_pose_hypotheses(stack[:, 0:3], stack[:, 3:6], *rest, steps=3)
    b = pft.refine_pose_hypotheses(stack[:, 0:3].contiguous(), stack[:, 3:6].contiguous(), *rest, steps=3)
    for k in OUT:
        assert same_bits(a[k], b[k]), k


@pytest.mark.gpu
def test_graph_replay_with_new_starts():
    fr = gpu_frames(192, 640)
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    poses = sweep_poses(fr["poses"][0], 10)
    static = poses.clone()

    def run():
        return pft.refine_pose_hypotheses(*args, static, fr["K"], steps=4)

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
    ref = pft.refine_pose_hypotheses(*args, new, fr["K"], steps=4)
    for k in OUT:
        assert same_bits(out[k], ref[k]), k
    assert not torch.equal(out["loss"], pft.refine_pose_hypotheses(*args, poses, fr["K"], steps=4)["loss"])
