"""Loss-surface sweeps of the demo (plot_loss_surface.py:11-87) two ways on one GPU, printed as one JSON line:

  loop   the batch-1 loop `bench.py --workload sweep` times: one pft.compute_photometric_error call and the masked
         mean (diff_img * valid_mask * weight_mask).sum() / valid_mask.sum() per pose sample;
  batch  one pft.photometric_loss_surface call over all samples.

and, for the pose gradient of every sample (the "grad" section):

  loop   per sample one compute_photometric_error call with a pose that requires grad, the masked mean and
         .backward(), then pose.grad;
  batch  one pft.photometric_loss_surface_and_grad call over all samples (loss and pose_grad).

and, for multi-start refinement, `--refine-steps` Adam steps from every sample (the "refine" section):

  loop   what a user writes with the surface functions: per step pft.photometric_loss_surface_and_grad and
         torch.optim.Adam (defaults) on an [N,6] leaf, the NaN gradients of samples with no valid pixel zeroed, then
         one pft.photometric_loss_surface for the final loss;
  batch  one pft.refine_pose_hypotheses call (the loss history).

The refine section runs N = 8, 100 (the demo's) and 200 (bench.py's); both ways end with the D2H copy of the
[steps+1, N] loss history.  The two do not give the same bits (torch's Adam rounds differently), so no difference is
reported for them.

and, for B frame pairs of N hypotheses each (the "pairs" section), surface and refine:

  loop   a Python loop of B single-pair calls (photometric_loss_surface, or refine_pose_hypotheses with
         `--refine-steps`), the results stacked;
  batch  one call with poses [B,N,6].

B = 4, N = 100 is the demo's four surfaces per epoch; B = 32, N = 8 is config 2's 2*S*B pose / pair combinations of
a minibatch with a few starts each.  The frames are make_frames(B, 192, 640, ...) with the same seed and intrinsics
as above, and each pair's N hypotheses are the two +-0.05 lines of N / 2 samples around its pose.  Both ways give the
same bits ("identical").

Input: what `bench.py --workload sweep` evaluates, make_frames(1, 192, 640, n_src=2, seed=0, KITTI intrinsics) with a
line of forward-translation (pose column 2) and a line of yaw (column 4) samples, linspace(-0.05, 0.05, n) each:
n = 100 (bench.py's default --sweep-evals, N = 200) and n = 50 (the demo's, N = 100).  Both are timed like
main_sweep: wall clock of a whole sweep including the final device-to-host copy, after one warm-up sweep, the two
alternated round by round.  The batched op's device time per call comes from CUDA events around `--device-iters`
back-to-back calls, next to the forward-only call's in the grad section.  The working set (one frame pair, ~2.5 MB) stays in L2, so no HBM roofline fraction is claimed.

Usage: python tools/bench_photo_sweep.py [--rounds R] [--device-iters I] [--refine-steps S] [--refine-iters J]
                                        [--sections surface,grad,refine,pairs]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tcsfm_b200 import pft, synth  # noqa: E402


def card():
    """(name, power limit) of the card, a read-only query."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        idx = torch.cuda.current_device()
        name, power = [s.strip() for s in out[idx].split(",")]
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(), "unknown"


def measure(fr, n, rounds, device_iters):
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    deltas = torch.linspace(-0.05, 0.05, n)
    deltas_dev = deltas.to(fr["K"].device)

    def loop():                                     # bench.py main_sweep's loop body
        vals = []
        with torch.no_grad():
            for axis in (2, 4):
                for d in deltas:
                    pose = fr["poses"][0].clone()
                    pose[:, axis] += d
                    r = pft.compute_photometric_error(*args, pose, fr["K"])
                    vals.append((r["diff_img"] * r["valid_mask"] * r["weight_mask"]).sum() / r["valid_mask"].sum())
        return torch.stack(vals)

    def poses():
        p = fr["poses"][0].repeat(2 * n, 1)
        p[:n, 2] += deltas_dev
        p[n:, 4] += deltas_dev
        return p

    def batch():
        with torch.no_grad():
            return pft.photometric_loss_surface(*args, poses(), fr["K"])["loss"]

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        host = fn().cpu()
        return time.perf_counter() - t0, host

    loop(), batch()                                 # warm-up sweeps
    t_loop, t_batch = [], []
    for _ in range(rounds):
        dt, ref = timed(loop)
        t_loop.append(dt)
        dt, got = timed(batch)
        t_batch.append(dt)
    rel = ((got - ref).abs() / ref.abs()).max().item()

    p = poses()
    with torch.no_grad():
        for _ in range(10):
            pft.photometric_loss_surface(*args, p, fr["K"])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(device_iters):
            pft.photometric_loss_surface(*args, p, fr["K"])
        e1.record()
        torch.cuda.synchronize()
    ms_call = e0.elapsed_time(e1) / device_iters
    evals = 2 * n
    return {"N": evals,
            "loop_evals_per_s": round(evals / statistics.median(t_loop), 1),
            "batch_evals_per_s": round(evals / statistics.median(t_batch), 1),
            "speedup": round(statistics.median(t_loop) / statistics.median(t_batch), 2),
            "loop_ms_per_sweep": [round(t * 1e3, 3) for t in t_loop],
            "batch_ms_per_sweep": [round(t * 1e3, 3) for t in t_batch],
            "batch_device_ms_per_call": round(ms_call, 4),
            "batch_device_us_per_eval": round(ms_call * 1e3 / evals, 3),
            "device_calls_timed": device_iters,
            "max_rel_diff_loss": rel}


def measure_grad(fr, n, rounds, device_iters):
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    deltas = torch.linspace(-0.05, 0.05, n)
    deltas_dev = deltas.to(fr["K"].device)

    def poses():
        p = fr["poses"][0].repeat(2 * n, 1)
        p[:n, 2] += deltas_dev
        p[n:, 4] += deltas_dev
        return p

    def loop():
        grads = []
        for axis in (2, 4):
            for d in deltas:
                pose = fr["poses"][0].clone()
                pose[:, axis] += d
                pose.requires_grad_(True)
                r = pft.compute_photometric_error(*args, pose, fr["K"])
                ((r["diff_img"] * r["valid_mask"] * r["weight_mask"]).sum() / r["valid_mask"].sum()).backward()
                grads.append(pose.grad[0])
        return torch.stack(grads)

    def batch():
        return pft.photometric_loss_surface_and_grad(*args, poses(), fr["K"])["pose_grad"]

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        host = fn().cpu()
        return time.perf_counter() - t0, host

    loop(), batch()                                 # warm-up sweeps
    t_loop, t_batch = [], []
    for _ in range(rounds):
        dt, ref = timed(loop)
        t_loop.append(dt)
        dt, got = timed(batch)
        t_batch.append(dt)
    rel = ((got.double() - ref.double()).norm(dim=1) / ref.double().norm(dim=1)).max().item()

    def device_ms(fn):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(device_iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / device_iters

    p = poses()
    with torch.no_grad():
        ms_grad = device_ms(lambda: pft.photometric_loss_surface_and_grad(*args, p, fr["K"]))
        ms_fwd = device_ms(lambda: pft.photometric_loss_surface(*args, p, fr["K"]))
    evals = 2 * n
    return {"N": evals,
            "loop_evals_per_s": round(evals / statistics.median(t_loop), 1),
            "batch_evals_per_s": round(evals / statistics.median(t_batch), 1),
            "speedup": round(statistics.median(t_loop) / statistics.median(t_batch), 2),
            "loop_ms_per_sweep": [round(t * 1e3, 3) for t in t_loop],
            "batch_ms_per_sweep": [round(t * 1e3, 3) for t in t_batch],
            "grad_device_ms_per_call": round(ms_grad, 4),
            "forward_device_ms_per_call": round(ms_fwd, 4),
            "grad_device_us_per_eval": round(ms_grad * 1e3 / evals, 3),
            "device_calls_timed": device_iters,
            "max_rel_diff_pose_grad": rel}


def measure_refine(fr, n, rounds, steps, device_iters):
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    deltas = torch.linspace(-0.05, 0.05, n, device=fr["K"].device)
    start = fr["poses"][0].repeat(2 * n, 1)
    start[:n, 2] += deltas
    start[n:, 4] += deltas

    def loop():
        leaf = start.clone().requires_grad_(True)
        opt = torch.optim.Adam([leaf], lr=1e-3)
        rows = []
        for _ in range(steps):
            r = pft.photometric_loss_surface_and_grad(*args, leaf, fr["K"])
            rows.append(r["loss"])
            leaf.grad = torch.where((r["valid_sum"] > 0)[:, None], r["pose_grad"], 0.0)
            opt.step()
        rows.append(pft.photometric_loss_surface(*args, leaf.detach(), fr["K"])["loss"])
        return torch.stack(rows)

    def batch():
        return pft.refine_pose_hypotheses(*args, start, fr["K"], steps=steps)["loss"]

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn().cpu()
        return time.perf_counter() - t0

    loop(), batch()                                 # warm-up descents
    t_loop, t_batch = [], []
    for _ in range(rounds):
        t_loop.append(timed(loop))
        t_batch.append(timed(batch))
    with torch.no_grad():
        for _ in range(2):
            batch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(device_iters):
            batch()
        e1.record()
        torch.cuda.synchronize()
    ms_call = e0.elapsed_time(e1) / device_iters
    return {"N": 2 * n, "steps": steps,
            "loop_ms_per_descent": round(statistics.median(t_loop) * 1e3, 3),
            "batch_ms_per_descent": round(statistics.median(t_batch) * 1e3, 3),
            "speedup": round(statistics.median(t_loop) / statistics.median(t_batch), 2),
            "loop_ms_rounds": [round(t * 1e3, 3) for t in t_loop],
            "batch_ms_rounds": [round(t * 1e3, 3) for t in t_batch],
            "batch_device_ms_per_call": round(ms_call, 4),
            "batch_device_ms_per_step": round(ms_call / (steps + 1), 4),
            "device_calls_timed": device_iters}


def measure_pairs(B, n, rounds, steps, device_iters, refine_iters):
    """B pairs of 2 * n hypotheses: a loop of B single-pair calls against one batched call, surface and refine."""
    dev = torch.device("cuda:0")
    fr = synth.make_frames(B, 192, 640, n_src=2, seed=0, device=dev, intrinsics=torch.tensor(synth.KITTI_K))
    args = (fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1])
    K = fr["K"]
    deltas = torch.linspace(-0.05, 0.05, n, device=dev)
    poses = fr["poses"][0][:, None].repeat(1, 2 * n, 1)
    poses[:, :n, 2] += deltas
    poses[:, n:, 4] += deltas

    def pair(b):
        return tuple(a[b:b + 1] for a in args)

    fns = {
        "surface": (lambda: torch.stack([pft.photometric_loss_surface(*pair(b), poses[b], K[b:b + 1])["loss"]
                                         for b in range(B)]),
                    lambda: pft.photometric_loss_surface(*args, poses, K)["loss"], device_iters),
        "refine": (lambda: torch.stack([pft.refine_pose_hypotheses(*pair(b), poses[b], K[b:b + 1], steps=steps)["loss"]
                                        for b in range(B)], 1),
                   lambda: pft.refine_pose_hypotheses(*args, poses, K, steps=steps)["loss"], refine_iters),
    }
    out = {"B": B, "N": 2 * n, "steps": steps}
    with torch.no_grad():
        for name, (loop, batch, iters) in fns.items():
            def timed(fn):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                host = fn().cpu()
                return time.perf_counter() - t0, host

            loop(), batch()                         # warm-up
            t_loop, t_batch = [], []
            for _ in range(rounds):
                dt, ref = timed(loop)
                t_loop.append(dt)
                dt, got = timed(batch)
                t_batch.append(dt)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                batch()
            e1.record()
            torch.cuda.synchronize()
            out[name] = {"loop_ms": round(statistics.median(t_loop) * 1e3, 3),
                         "batch_ms": round(statistics.median(t_batch) * 1e3, 3),
                         "speedup": round(statistics.median(t_loop) / statistics.median(t_batch), 2),
                         "loop_ms_rounds": [round(t * 1e3, 3) for t in t_loop],
                         "batch_ms_rounds": [round(t * 1e3, 3) for t in t_batch],
                         "batch_device_ms_per_call": round(e0.elapsed_time(e1) / iters, 4),
                         "device_calls_timed": iters,
                         "identical": bool(torch.equal(got.isnan(), ref.isnan())
                                           and torch.equal(got.nan_to_num(), ref.nan_to_num()))}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=5, help="alternated loop / batch sweeps per configuration")
    ap.add_argument("--device-iters", type=int, default=200, help="back-to-back calls timed with CUDA events")
    ap.add_argument("--refine-steps", type=int, default=50, help="Adam steps per descent in the refine section")
    ap.add_argument("--refine-iters", type=int, default=20, help="back-to-back refine calls timed with CUDA events")
    ap.add_argument("--sections", default="surface,grad,refine,pairs", help="comma-separated sections to run")
    args = ap.parse_args()
    sections = set(args.sections.split(","))
    if not torch.cuda.is_available():
        sys.exit("bench_photo_sweep.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    fr = synth.make_frames(1, 192, 640, n_src=2, seed=0, device=dev, intrinsics=torch.tensor(synth.KITTI_K))
    name, power = card()
    line = {"metric": "loss-surface evaluations/s (B=1, 192x640, forward only): batch-1 loop vs one batched call",
            "unit": "evals/s", "gpu": name, "power_limit": power, "dtype": "f32", "data": "synthetic",
            "timing": "wall clock of a whole sweep incl. the final D2H, median of alternated rounds; device time from "
                      "CUDA events",
            "note": "working set (one frame pair, ~2.5 MB) is L2-resident: no HBM roofline fraction is claimed"}
    if "surface" in sections:
        line["configs"] = {"bench_sweep_default_100x2": measure(fr, 100, args.rounds, args.device_iters),
                           "demo_50x2": measure(fr, 50, args.rounds, args.device_iters)}
    if "grad" in sections:
        line["grad"] = {"metric": "loss-surface evaluations with the pose gradient per s: batch-1 forward + backward "
                                  "loop vs one photometric_loss_surface_and_grad call",
                        "max_rel_diff": "largest |pose_grad - loop| / |loop| over the rows",
                        "configs": {"bench_sweep_default_100x2": measure_grad(fr, 100, args.rounds, args.device_iters),
                                    "demo_50x2": measure_grad(fr, 50, args.rounds, args.device_iters)}}
    if "refine" in sections:
        line["refine"] = {"metric": "multi-start refinement, ms per descent of N starts: the surface_and_grad + "
                                    "torch.optim.Adam loop vs one refine_pose_hypotheses call",
                          "configs": {"N%d" % (2 * n): measure_refine(fr, n, args.rounds, args.refine_steps,
                                                                      args.refine_iters) for n in (4, 50, 100)}}
    if "pairs" in sections:
        line["pairs"] = {"metric": "B frame pairs of N hypotheses, ms per call: a loop of B single-pair calls vs one "
                                   "call with poses [B,N,6] (surface, and refine with --refine-steps)",
                         "configs": {"B%d_N%d" % (B, 2 * n): measure_pairs(B, n, args.rounds, args.refine_steps,
                                                                             args.device_iters, args.refine_iters)
                                     for B, n in ((4, 50), (32, 4))}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
