#!/usr/bin/env python
"""Benchmark of the warp + SSIM/L1 photometric-loss hot path (BASELINE.json metric:
"warp+SSIM/L1 loss fwd+bwd frames/s at 192x640").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload kitti|scannet] [--dump-outputs DIR]

One *step* = one `Compute_Loss.forward` + `.backward()` over one synthetic minibatch
(config 2 of BASELINE.json: B=8 KITTI-shaped 3-frame snippets at 192x640, forward and
inverse direction for both sources = 32 pair evaluations, SSIM + L1 + auto-mask +
depth-consistency mask/term, gradients to the three disparity maps and four poses).
A *frame* is one target frame (2*S pair evaluations).

Prints ONE JSON line (rank 0).  Multi-GPU (torchrun, one rank per GPU): every rank
processes its own shard of minibatches, no data-path collective (SURVEY.md §8e),
`scaling: weak`; the timed region is bracketed by barrier + synchronize and the
slowest rank's device time is used.

`--impl reference` times the oracle port of the reference's PyTorch CPU path
(oracle/ref_torch.py: the same ATen operators in the same order) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (which may be read-only)
# stdout must carry exactly one JSON line, but NCCL writes its version banner to fd 1: park the
# real stdout and route everything else that lands on fd 1 to stderr
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line_dict):
    os.write(_REAL_STDOUT, (json.dumps(line_dict) + "\n").encode())

PFT_WORKLOADS = {
    # sequential per-frame test-time optimisation (configs 3/4 of BASELINE.json); stand-in networks
    "pft": dict(b=6, h=192, w=640, n_src=2, iterations=4, epochs=20,
                desc="pft_kitti_windows_b6_192x640_4iter_20epochs_standin_nets"),
    "pft-scannet": dict(b=16, h=256, w=320, n_src=1, iterations=4, epochs=20,
                        desc="pft_scannet_pairs_b16_256x320_4iter_20epochs_standin_nets"),
}

WORKLOADS = {
    # name: (B, H, W, n_src, depth_range key, intrinsics)
    "kitti": dict(b=8, h=192, w=640, n_src=2, desc="kitti_triplets_b8_192x640_fwd+inv_ssim_l1_automask_depthconsist"),
    "scannet": dict(b=16, h=256, w=320, n_src=1, desc="scannet_pairs_b16_256x320_fwd+inv_ssim_l1_automask_depthconsist"),
    "scannet448": dict(b=16, h=256, w=448, n_src=1, desc="scannet_pairs_b16_256x448_fwd+inv_ssim_l1_automask_depthconsist"),
    # config 5: the training-step loss path at 4 scales (every scale nearest-upsampled to full
    # resolution, losses.py:86-87) at 376x1242
    "kitti376x4": dict(b=2, h=376, w=1242, n_src=2, scales=4,
                       desc="kitti_triplets_b2_376x1242_4scales_fwd+inv_ssim_l1_automask_depthconsist"),
}
LOSS_CFG = {"l1_weight": 0.15, "l_ssim_weight": 0.85, "l_smooth_weight": 0.05, "num_scales": 1,
            "l_depth_consist_weight": 0.14, "min_depth": 0.06, "max_depth": 2.67, "l_smooth": False,
            "l_reconstruction": True, "l_inverse": True, "l_depth_consist": True,
            "with_auto_mask": True, "l_ssim": True, "with_depth_mask": True}
TRAIN_WORKLOADS = {
    # BASELINE config 5: the training-step loss path at 4 scales up to 376x1242 (every scale nearest-upsampled to full
    # resolution, losses.py:86-87), 4 egomotion iterations, the paper's training flags (run_mono_training.py:50-64)
    "train376x4": dict(b=2, h=376, w=1242, scales=4, iterations=4, full=False,
                       desc="train_step_b2_376x1242_4scales_4iter_standin_nets_adam"),
}
METRIC = "warp+SSIM/L1 loss fwd+bwd frames/s at 192x640"
ARITH_MODES = ("exact", "fast")
# the benchmarked default: the "fast" SSIM arithmetic passes the north-star parity gates on the GPU (loss 1e-5, gradients
# 1e-4, every mask bit-exact; tests/test_gpu_parity.py::test_fast_*); "exact" (bit-identical diff_img as well) is timed in
# the same run and reported under "other_arithmetic"
DEFAULT_ARITH = "fast"
N_INPUT_SETS = 8      # rotating input sets: 8 x ~47 MB > 126 MB of L2, so no step finds its inputs in L2


def make_inputs(wl, seed, device, pin=False, slab=False):
    from tcsfm_b200 import synth
    kitti = wl["h"] in (192, 376)
    rng = synth.KITTI_DEPTH_RANGE if kitti else synth.SCANNET_DEPTH_RANGE
    if wl["h"] == 376:
        base = torch.tensor(synth.KITTI_FULL_K, dtype=torch.float32)
    elif kitti:
        base = torch.tensor(synth.KITTI_K, dtype=torch.float32)
    else:
        base = synth.scaled_intrinsics(wl["h"], wl["w"], synth.SCANNET_K, (256, 320))
    # every input set carries its own intrinsics (focal lengths / principal point jittered by up to 1 %), so a
    # step that reused a stale K^-1 would be caught: K^-1 is recomputed inside every timed step (models/stn.py:257)
    base = base.clone()
    base[0, 0] *= 1.0 + 0.002 * (seed % 5)
    base[1, 1] *= 1.0 + 0.002 * (seed % 3)
    base[0, 2] += 0.25 * (seed % 4)
    fr = synth.make_frames(wl["b"], wl["h"], wl["w"], n_src=wl["n_src"], seed=seed, depth_range=rng, intrinsics=base)
    flat = {"target": fr["target"]}                 # the frames first: they form one contiguous region of a slab
    for j in range(wl["n_src"]):
        flat["source%d" % j] = fr["sources"][j]
    flat["K"] = fr["K"]
    for j in range(wl["n_src"]):
        flat["pose%d" % j] = fr["poses"][j]
        flat["pose_inv%d" % j] = fr["poses_inv"][j]
    for j in range(1 + wl["n_src"]):
        flat["disp%d" % j] = fr["disps"][j]
        for sc in range(1, wl.get("scales", 1)):          # lower-resolution disparities of the other scales
            flat["disp%d_s%d" % (j, sc)] = torch.nn.functional.avg_pool2d(fr["disps"][j], 2 ** sc, ceil_mode=True)
    if slab:
        # one contiguous buffer per minibatch (dataformat.pack_slab): the end-to-end arm moves it with a single copy
        from tcsfm_b200 import dataformat
        return dataformat.pack_slab(flat, device=device, pin=pin)
    if pin:
        return {k: v.pin_memory() for k, v in flat.items()}
    return {k: v.to(device) for k, v in flat.items()}


def run_step(loss_mod, inp, n_src, need_value=False):
    """One training-step loss: forward + backward.  Returns the loss dict (every entry [1]); the gradients are left
    in `.grad` of the disparity / pose tensors of `inp`."""
    n_scales = loss_mod.num_scales
    disps = [inp["disp%d" % j].requires_grad_(True) for j in range(1 + n_src)]
    extra = [[inp["disp%d_s%d" % (j, sc)].requires_grad_(True) for sc in range(1, n_scales)] for j in range(1 + n_src)]
    poses = [inp["pose%d" % j].requires_grad_(True) for j in range(n_src)]
    poses_inv = [inp["pose_inv%d" % j].requires_grad_(True) for j in range(n_src)]
    for t in disps + poses + poses_inv + [e for ex in extra for e in ex]:
        t.grad = None
    out = loss_mod([inp["source%d" % j] for j in range(n_src)], inp["target"], [poses, poses_inv],
                   [[d] + ex for d, ex in zip(disps, extra)], inp["K"])
    out["total"].backward()         # [1]; backward() on it directly, like train_mono.py:193
    return out


def step_outputs(out, inp):
    """Host copies of what one run_step call gave its caller: the loss terms and the gradients of its inputs."""
    arrays = {"loss_" + k: v for k, v in out.items()}
    arrays.update({"grad_" + k: t.grad for k, t in inp.items() if t.grad is not None})
    return {k: v.detach().cpu().numpy() for k, v in arrays.items()}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(arrays, out_dir):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:        # every workload of WORKLOADS stays far below (kitti: 11.8 MB)
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in o.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples if len(s) >= 6 for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_port_throughput(wl, steps, warmup, threads):
    """Times the oracle port of the reference's CPU path (fwd + bwd) on the host cores."""
    from oracle import ref_torch as O
    torch.set_num_threads(threads)
    inp = make_inputs(wl, 0, "cpu")
    n_src = wl["n_src"]

    n_scales = wl.get("scales", 1)
    kitti = wl["h"] in (192, 376)
    from tcsfm_b200 import synth
    rng = synth.KITTI_DEPTH_RANGE if kitti else synth.SCANNET_DEPTH_RANGE
    cfg = dict(LOSS_CFG, num_scales=n_scales, min_depth=rng[0], max_depth=rng[1])

    def step():
        disps = [[inp["disp%d" % j].clone().requires_grad_(True)] +
                 [inp["disp%d_s%d" % (j, sc)].clone().requires_grad_(True) for sc in range(1, n_scales)]
                 for j in range(1 + n_src)]
        poses = [inp["pose%d" % j].clone().requires_grad_(True) for j in range(n_src)]
        poses_inv = [inp["pose_inv%d" % j].clone().requires_grad_(True) for j in range(n_src)]
        out = O.compute_loss(cfg, [inp["source%d" % j] for j in range(n_src)], inp["target"],
                             [poses, poses_inv], disps, inp["K"])
        out["total"].sum().backward()
        return float(out["total"].sum().detach())

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return wl["b"] * steps / dt, dt / steps * 1e3


class Ranks:
    """One process per GPU (torchrun): rank bookkeeping, barrier and max-over-ranks of device times."""

    def __init__(self, need_cuda=True):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        self.dev = None
        if need_cuda:
            torch.cuda.set_device(self.local_rank)
            self.dev = torch.device("cuda", self.local_rank)
            if self.world > 1:
                import torch.distributed as dist
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                dist.init_process_group("nccl", device_id=self.dev)
                self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, *values):
        if self.dist is None:
            return list(values)
        t = torch.tensor(list(values), device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def timed(self, fn, steps):
        """Device time (CUDA events on the launching stream) of `steps` calls, bracketed by barrier +
        synchronize on both sides, max over ranks."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1))[0]

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def pft_measure(R, name, steps, warm, no_graph=False, sequence_frames=0):
    """PFT frames/s on this rank's shard of window minibatches (tcsfm_b200.shard), no communication; a 'step' is one
    window minibatch taken through all optimisation epochs (depth-net -> solve_pose_iteratively -> loss -> backward
    -> Adam; optimizer.py:136-297 with stand-in networks).  Returns the sub-object for the JSON line.

    sequence_frames > 0 additionally runs BASELINE config 4: a whole synthetic sequence of that many frames
    (1591 = KITTI seq 09 -> 795 windows -> 133 minibatches, the last of 3 windows), its minibatches sharded
    contiguously over the ranks -- total work fixed, i.e. strong scaling."""
    from tcsfm_b200 import _timing, pft_driver, shard, synth
    wl = PFT_WORKLOADS[name]
    dev = R.dev
    opts = {"epochs": wl["epochs"], "num_source_imgs": wl["n_src"]}
    rng = synth.KITTI_DEPTH_RANGE if wl["h"] == 192 else synth.SCANNET_DEPTH_RANGE
    base = synth.KITTI_K if wl["h"] == 192 else synth.SCANNET_K

    def frames_for(seed, b=wl["b"]):
        k = torch.tensor(base, dtype=torch.float32)
        k[0, 0] *= 1.0 + 0.002 * (seed % 5)                      # windows do not share intrinsics bit for bit
        return synth.make_frames(b, wl["h"], wl["w"], n_src=wl["n_src"], seed=seed, depth_range=rng, intrinsics=k, device=dev)

    depth_net, pose_net = synth.TinyDepthNet(0).to(dev), synth.TinyPoseNet(0).to(dev)
    total_mbs = steps * R.world
    lo, hi = shard.shard_range(total_mbs, R.rank, R.world)           # this rank's window minibatches
    data = [frames_for(1000 + i) for i in range(lo, hi)]
    host = [{k: ([t.cpu().pin_memory() for t in v] if isinstance(v, list) else v.cpu().pin_memory()) for k, v in d.items()}
            for d in data[:2]]
    runner = None if no_graph else pft_driver.WindowRunner(depth_net, pose_net, opts, wl["iterations"], rng)

    def run(fr):
        if runner is not None:        # epoch graphs captured on the first (warm-up) window, replayed afterwards
            return runner(fr["target"], fr["sources"], fr["K"])
        return pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts,
                                          wl["iterations"], rng)

    for i in range(max(1, warm)):
        run(data[i % len(data)])
    l0 = _timing.LAUNCH_COUNT
    ms = R.timed(lambda i: run(data[i]), len(data))
    launches = _timing.LAUNCH_COUNT - l0

    def e2e_step(i):        # window inputs from pinned host memory, the final loss read back
        h = host[i % len(host)]
        fr = {k: ([t.to(dev, non_blocking=True) for t in v] if isinstance(v, list) else v.to(dev, non_blocking=True))
              for k, v in h.items() if k in ("target", "sources", "K")}
        float(run(fr)["losses"][-1])
    ms_e2e = R.timed(e2e_step, len(data))
    # device time of the library's own launches inside one window minibatch (the hot path proper) against
    # the device time of the whole window, both eager (events recorded during graph capture cannot be timed)
    timer = _timing.KernelTimer()
    torch.cuda.synchronize()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # (one untimed eager window first: the eager path's own lazy initialisations -- cuDNN plans of the stand-in network,
    # allocator growth -- otherwise land in the interval)
    pft_driver.optimize_window(depth_net, pose_net, data[0]["target"], data[0]["sources"], data[0]["K"], opts,
                               wl["iterations"], rng, cuda_graph=False)
    torch.cuda.synchronize()
    w0.record()
    with _timing.record(timer):
        pft_driver.optimize_window(depth_net, pose_net, data[0]["target"], data[0]["sources"], data[0]["K"], opts,
                                   wl["iterations"], rng, cuda_graph=False)
    w1.record()
    ksum = timer.summary()
    eager_window_ms = w0.elapsed_time(w1)
    hot_ms = sum(v["launches"] * v["avg_ms"] for v in ksum.values())
    # the hot path proper: the same epoch body with the (out-of-scope) depth network replaced by leaf disparities --
    # what is left besides the library's kernels is PyTorch glue (tools/profile_pft_hotpath.py)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import profile_pft_hotpath
    proper = profile_pft_hotpath.run(3, wl["b"], wl["h"], wl["w"], wl["n_src"], wl["iterations"], dev, record=True)
    frames = wl["b"] * total_mbs
    h2d = sum(t.numel() * 4 for t in [host[0]["target"], host[0]["K"]] + host[0]["sources"])
    out = {"metric": "PFT frames/s", "value": frames / (ms / 1e3), "unit": "frames/s", "workload": wl["desc"],
           "window_minibatches_per_gpu": steps, "ms_per_window_minibatch": ms / steps, "scaling": "weak",
           "launch": "eager" if no_graph else "epoch CUDA graphs captured on the warm-up window, replayed for every timed window",
           "networks": "stand-in TinyDepthNet/TinyPoseNet (the reference nets are out of scope)",
           "e2e": {"value": frames / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
           "gpu_launches": launches,
           "hot_path": {"ms_per_window_minibatch": hot_ms, "frames_per_s": wl["b"] / (hot_ms / 1e3),
                        "share_of_eager_window_device_time": hot_ms / eager_window_ms,
                        "note": "sum of the library launches' device time (CUDA events) over one eager window minibatch; "
                                "the rest is the stand-in networks, Adam and PyTorch's own glue",
                        "kernels": ksum,
                        "without_depth_net": {k: v for k, v in proper.items() if k != "kernels"}}}
    if sequence_frames:
        mbs = shard.window_minibatches(sequence_frames, stride=2, minibatch=wl["b"])
        s_lo, s_hi = shard.shard_range(len(mbs), R.rank, R.world)
        pool = data + [frames_for(5000 + i) for i in range(max(0, 4 - len(data)))]
        short = {}

        def seq_step(i):
            n_win = len(mbs[s_lo + i])
            if n_win == wl["b"]:
                run(pool[i % len(pool)])
            else:                                               # the ragged last minibatch: eager, its own batch size
                if n_win not in short:
                    short[n_win] = frames_for(7000 + n_win, b=n_win)
                fr = short[n_win]
                pft_driver.optimize_window(depth_net, pose_net, fr["target"], fr["sources"], fr["K"], opts, wl["iterations"], rng)
        ms_seq = R.timed(seq_step, s_hi - s_lo)
        out["sequence"] = {"frames": sequence_frames, "windows": sum(len(m) for m in mbs), "window_minibatches": len(mbs),
                           "minibatches_this_rank": s_hi - s_lo, "seconds": ms_seq / 1e3,
                           "sequence_frames_per_s": sequence_frames / (ms_seq / 1e3),
                           "windows_per_s": sum(len(m) for m in mbs) / (ms_seq / 1e3), "scaling": "strong",
                           "note": "BASELINE config 4: contiguous minibatch ranges per GPU, no inter-GPU traffic"}
    return out


def main_pft(args):
    wl = PFT_WORKLOADS[args.workload]
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        from oracle import ref_torch as O
        from tcsfm_b200 import pft_driver, synth

        class OracleBackend:
            solve_pose_iteratively = staticmethod(O.iterative_pose)
            compute_optimization_loss = staticmethod(O.pft_window_loss)
            disp_to_depth = staticmethod(O.disp_to_depth)
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        rng = synth.KITTI_DEPTH_RANGE if wl["h"] == 192 else synth.SCANNET_DEPTH_RANGE
        base = synth.KITTI_K if wl["h"] == 192 else synth.SCANNET_K
        cpu_opts = {"epochs": 2, "num_source_imgs": wl["n_src"]}
        fr = synth.make_frames(wl["b"], wl["h"], wl["w"], n_src=wl["n_src"], seed=0, depth_range=rng,
                               intrinsics=torch.tensor(base, dtype=torch.float32))
        dn, pn = synth.TinyDepthNet(0), synth.TinyPoseNet(0)
        t0 = time.perf_counter()
        pft_driver.optimize_window(dn, pn, fr["target"], fr["sources"], fr["K"], cpu_opts, wl["iterations"], rng, OracleBackend)
        dt = (time.perf_counter() - t0) * wl["epochs"] / cpu_opts["epochs"]
        fps = wl["b"] / dt
        emit(({"impl": "reference", "metric": "PFT frames/s", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
               "steps": 1, "warmup": 0, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": wl["desc"]},
               "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": "2 of %d epochs of one window minibatch, extrapolated" % wl["epochs"]},
               "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    R = Ranks()
    steps = min(args.steps, 4)
    warm = max(1, min(args.warmup, 1))
    sub = pft_measure(R, args.workload, steps, warm, args.no_graph, sequence_frames=args.sequence_frames)
    R.close()
    if R.rank != 0:
        return
    line = {"metric": sub["metric"], "value": sub["value"], "unit": "frames/s", "n_gpus": R.world, "steps": steps,
            "warmup": warm, "ms_per_step": sub["ms_per_window_minibatch"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": sub["workload"], "window_minibatches_per_gpu": steps, "parallelism": "shard%d" % R.world,
                       "networks": sub["networks"], "launch": sub["launch"]},
            "e2e": sub["e2e"], "gpu_launches": sub["gpu_launches"], "hot_path": sub["hot_path"]}
    if "sequence" in sub:
        line["sequence"] = sub["sequence"]
    emit(line)


def main_sweep(args):
    """Config 1's forward-only part: the loss-surface sweeps of the demo (plot_loss_surface.py:11-87 via
    helpers.compute_photometric_error): batch-1 evaluations of warp + photometric error for a line of
    translation and a line of yaw perturbations.  A launch-latency-bound use of the same kernels."""
    from tcsfm_b200 import pft, synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.sweep_evals
    if args.impl == "reference":
        from oracle import ref_torch as O
        dev, fn = "cpu", O.photometric_error
        torch.set_num_threads(os.cpu_count() or 1)
        n = min(n, 20)
    else:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dev, fn = "cuda", pft.compute_photometric_error
    fr = synth.make_frames(1, 192, 640, n_src=2, seed=0, device=dev, intrinsics=torch.tensor(synth.KITTI_K))
    deltas = torch.linspace(-0.05, 0.05, n)

    def sweep():
        vals = []
        with torch.no_grad():
            for axis in (2, 4):                                 # forward translation, yaw
                for d in deltas:
                    pose = fr["poses"][0].clone()
                    pose[:, axis] += d
                    r = fn(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], pose, fr["K"])
                    vals.append((r["diff_img"] * r["valid_mask"] * r["weight_mask"]).sum() / r["valid_mask"].sum())
        return torch.stack(vals)

    sweep()
    if dev == "cuda":
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = sweep()
    host = out.cpu()
    dt = time.perf_counter() - t0
    line = {"metric": "loss-surface evaluations/s (B=1, 192x640, forward only)", "value": 2 * n / dt, "unit": "evals/s",
            "n_gpus": 1, "steps": 2 * n, "warmup": 2 * n, "ms_per_step": dt / (2 * n) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "demo_loss_surface_sweep_b1_192x640", "launch": "eager, wall clock incl. the final D2H"},
            "e2e": {"value": 2 * n / dt, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4}}
    if args.impl == "reference":
        line["impl"] = "reference"
        line["cpu_baseline"] = {"value": line["value"], "unit": "evals/s", "cores": os.cpu_count(), "kind": "port",
                                "sample": "%d evaluations" % (2 * n)}
    else:
        line["surface_min"] = float(host.min())
    emit(line)


def train_measure(R, steps, warm, wl_name="train376x4"):
    """Training mode (BASELINE config 5): one minibatch of Trainer.forward (train_mono.py:159-194) per step around the
    fused loss at 4 scales, stand-in networks of the reference's parameter volume (15.7 M fp32 = 62.8 MB of
    gradients), Adam; with more than one rank DistributedDataParallel all-reduces the network gradients over NCCL --
    the only collective of the mode.  Reports the step with and without the all-reduce (`no_sync`) and the bare
    all-reduce of the same payload, so the exposed (non-overlapped) NCCL time is visible."""
    from tcsfm_b200 import _timing, synth, training
    wl = TRAIN_WORKLOADS[wl_name]
    dev = R.dev
    cfg = training.default_config(num_scales=wl["scales"], iterations=wl["iterations"], full_profile=wl["full"])
    step, optim = training.make_step(cfg, seed=0, device=dev, padded=True)
    model = training.wrap_ddp(step, dev) if R.dist is not None else step
    k = torch.tensor(synth.KITTI_FULL_K if wl["h"] == 376 else synth.KITTI_K, dtype=torch.float32)
    data = [synth.make_frames(wl["b"], wl["h"], wl["w"], n_src=2, seed=300 + 10 * R.rank + i, intrinsics=k, device=dev)
            for i in range(4)]
    n_params = sum(p.numel() for p in step.parameters())
    for i in range(max(3, warm)):
        training.run_train_step(model, optim, data[i % 4])
    l0 = _timing.LAUNCH_COUNT
    ms_sync = R.timed(lambda i: training.run_train_step(model, optim, data[i % 4], sync=True), steps)
    launches = _timing.LAUNCH_COUNT - l0
    ms_nosync = R.timed(lambda i: training.run_train_step(model, optim, data[i % 4], sync=False), steps)
    out = {"metric": "training-step frames/s (loss at %d scales, %dx%d)" % (wl["scales"], wl["h"], wl["w"]),
           "workload": wl["desc"], "value": wl["b"] * R.world * steps / (ms_sync / 1e3), "unit": "frames/s",
           "batch_per_gpu": wl["b"], "steps": steps, "ms_per_step": ms_sync / steps, "scaling": "weak",
           "ms_per_step_without_allreduce": ms_nosync / steps,
           "exposed_allreduce_ms_per_step": max(0.0, (ms_sync - ms_nosync) / steps),
           "gradient_bytes_per_step": 4 * n_params, "gpu_launches": launches,
           "collective": ("DistributedDataParallel: NCCL all-reduce (mean) of the network gradients, %d ranks" % R.world)
           if R.dist is not None else "none (single rank)",
           "networks": "stand-in depth/pose networks padded to the reference's %d parameters" % n_params,
           "launch": "eager"}
    if R.dist is not None:
        flat = torch.zeros(n_params, device=dev)
        for _ in range(3):
            R.dist.all_reduce(flat)
        ms_ar = R.timed(lambda i: R.dist.all_reduce(flat), 10)
        out["bare_allreduce_ms"] = ms_ar / 10
        out["bare_allreduce_busbw_GBps"] = 4 * n_params * 2 * (R.world - 1) / R.world / (ms_ar / 10 * 1e-3) / 1e9
    # The same step with the host taken out (training.FlatGradTrainer): forward + backward as one CUDA graph, ONE
    # all-reduce of the flat gradient buffer, Adam as a second graph.  This is the mode's headline; the eager numbers
    # above stay in the record as `eager`.
    del model, optim, step
    step_g, optim_g = training.make_step(cfg, seed=0, device=dev, padded=True, capturable=True)
    trainer = training.FlatGradTrainer(step_g, optim_g, data[0], group=R.dist.group.WORLD if R.dist is not None else None)
    for i in range(3):
        trainer.run(data[i % 4])
    g_steps = max(steps, 20)
    ms_g = R.timed(lambda i: trainer.run(data[i % 4], sync=True), g_steps)
    ms_g_nosync = R.timed(lambda i: trainer.run(data[i % 4], sync=False), g_steps)
    eager = {k: out[k] for k in ("value", "ms_per_step", "ms_per_step_without_allreduce", "exposed_allreduce_ms_per_step",
                                 "gpu_launches", "collective", "launch", "steps")}
    out.update({"value": wl["b"] * R.world * g_steps / (ms_g / 1e3), "ms_per_step": ms_g / g_steps, "steps": g_steps,
                "ms_per_step_without_allreduce": ms_g_nosync / g_steps,
                "exposed_allreduce_ms_per_step": max(0.0, (ms_g - ms_g_nosync) / g_steps),
                "launch": "two CUDA graphs per step (forward+backward, Adam), static input buffers",
                "collective": ("one NCCL all-reduce (mean) of the flat %d-byte gradient buffer between the two graphs, %d ranks"
                               % (4 * n_params, R.world)) if R.dist is not None else "none (single rank)",
                "eager": eager})
    return out


def h2d_ceiling(dev, mbytes=512, reps=6):
    """Best-of-`reps` pinned host -> device bandwidth of one large copy (GB/s): the host link's ceiling the end-to-end
    number is read against."""
    src = torch.empty(mbytes << 20, dtype=torch.uint8).pin_memory()
    dst = torch.empty(mbytes << 20, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, (mbytes << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def eager_cuda_measure(wl, sets, cfg, steps):
    """The reference's eager PyTorch path (the oracle's op-for-op restatement: the same ATen CUDA kernels in the same
    order, including mean_on_mask's host synchronisation) on the same B200 -- the bar a user of the reference sees."""
    from oracle import ref_torch as O
    n_src, n_scales = wl["n_src"], wl.get("scales", 1)

    def step(i):
        inp = sets[i % len(sets)]
        disps = [[inp["disp%d" % j].detach().clone().requires_grad_(True)] +
                 [inp["disp%d_s%d" % (j, sc)].detach().clone().requires_grad_(True) for sc in range(1, n_scales)]
                 for j in range(1 + n_src)]
        poses = [inp["pose%d" % j].detach().clone().requires_grad_(True) for j in range(n_src)]
        poses_inv = [inp["pose_inv%d" % j].detach().clone().requires_grad_(True) for j in range(n_src)]
        out = O.compute_loss(cfg, [inp["source%d" % j] for j in range(n_src)], inp["target"], [poses, poses_inv], disps, inp["K"])
        out["total"].sum().backward()
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": wl["b"] / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms, "steps": steps, "kind": "port",
            "what": "oracle/ref_torch.py (the reference's ATen operator sequence) run eagerly on the same GPU, "
                    "CUDA events, inputs resident"}


def base_config(args, wl, world):
    """The `config` object of the JSON line -- identical for the two arms (`--impl ours|reference`)."""
    cfg = {"workload": wl["desc"], "batch_per_gpu": wl["b"],
           "pairs_per_step_per_gpu": 2 * wl["n_src"] * wl["b"] * wl.get("scales", 1),
           "height": wl["h"], "width": wl["w"], "flags": "full (depth-consistency mask + term, auto-mask, SSIM+L1)",
           "parallelism": "shard%d" % max(world, args.gpus),
           "l2": "inputs rotate over %d sets (> L2 capacity), each with its own intrinsics" % N_INPUT_SETS,
           "launch": "eager" if args.no_graph else "cuda-graph replay of the full step (one graph per input set)",
           "arithmetic": args.arith}
    if args.profile == "train":
        cfg["flags"] = "paper training defaults (auto-mask, SSIM+L1; no depth-consistency mask/term)"
    return cfg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 2000 ours, 20 reference arm)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default: 50 ours, 3 reference arm)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="kitti", choices=sorted(WORKLOADS) + sorted(PFT_WORKLOADS) + ["sweep"])
    ap.add_argument("--cpu-steps", type=int, default=None, help="steps of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of replaying CUDA graphs")
    ap.add_argument("--sweep-evals", type=int, default=100, help="workload 'sweep': evaluations per surface")
    ap.add_argument("--profile", default="full", choices=["full", "train"],
                    help="loss flags: 'full' = depth-consistency mask + term on (what PFT uses, 84 B/px/pair), "
                         "'train' = the paper's training defaults (run_mono_training.py:50-64: both off)")
    ap.add_argument("--arith", default=DEFAULT_ARITH, choices=sorted(ARITH_MODES),
                    help="SSIM arithmetic of the pair kernels: 'exact' keeps every rounding step of eager PyTorch; "
                         "'fast' keeps geometry, warp and masks bit-exact and evaluates the SSIM statistics at tolerance level")
    ap.add_argument("--only", default=None, choices=["loss"], help="'loss': skip the pft / train / eager-CUDA sub-benchmarks")
    ap.add_argument("--sequence-frames", type=int, default=0, help="PFT workloads: also time a whole sequence of this many frames")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="loss-step workloads: write what the last timed step returned (loss terms, gradients of the "
                         "disparities and poses; rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    ref_arm = args.impl == "reference"
    if args.dump_outputs and (ref_arm or args.workload not in WORKLOADS):
        ap.error("--dump-outputs needs --impl ours and one of the workloads %s" % ", ".join(sorted(WORKLOADS)))
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.steps is None:
        args.steps = 20 if ref_arm else 2000
    if args.warmup is None:
        args.warmup = 3 if ref_arm else 50
    if args.workload in PFT_WORKLOADS:
        return main_pft(args)
    if args.workload == "sweep":
        return main_sweep(args)
    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1

    if ref_arm:
        # the reference's own CPU implementation of the path (oracle port: the same ATen kernels in the same order),
        # all host threads, the arm's --steps / --warmup honoured as given
        if int(os.environ.get("RANK", "0")) != 0:
            return
        world = int(os.environ.get("WORLD_SIZE", "1"))
        config = base_config(args, wl, world)
        fps, ms = cpu_port_throughput(wl, args.steps, args.warmup, cores)
        line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                 "sample": "%d steps of the same B=%d minibatch, oracle port of the reference's "
                                           "PyTorch CPU path, torch threads=%d" % (args.steps, wl["b"], cores)},
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    R = Ranks()
    rank, world, dev = R.rank, R.world, R.dev
    config = base_config(args, wl, world)

    from tcsfm_b200 import _timing, losses, ops, synth
    ops.set_arithmetic(args.arith)
    kitti = wl["h"] in (192, 376)
    rng = synth.KITTI_DEPTH_RANGE if kitti else synth.SCANNET_DEPTH_RANGE
    flags_cfg = {} if args.profile == "full" else {"l_depth_consist": False, "with_depth_mask": False}
    loss_cfg = dict(LOSS_CFG, num_scales=wl.get("scales", 1), min_depth=rng[0], max_depth=rng[1], **flags_cfg)
    loss_mod = losses.Compute_Loss(loss_cfg)
    n_src = wl["n_src"]
    # sets 0 and 1 double as the device-side staging buffers of the end-to-end arm: each is one slab, mirrored by a
    # pinned host slab of the same layout
    dev_slabs = [make_inputs(wl, 100 * rank + s, dev, slab=True) for s in range(2)]
    sets = [d[1] for d in dev_slabs] + [make_inputs(wl, 100 * rank + s, dev) for s in range(2, N_INPUT_SETS)]
    host_slabs = [make_inputs(wl, 100 * rank + s, dev, pin=True, slab=True) for s in range(2)]
    host_sets = [h[1] for h in host_slabs]

    # The resident-input arm replays one captured CUDA graph per input set (the step has no host-side control flow:
    # the mean-on-mask threshold is decided on the device, K^-1 is computed inside the step without a host check), so
    # the timed region contains exactly the device work of K full steps.
    graphs = None
    if not args.no_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for s_ in sets:
                for _ in range(3):
                    run_step(loss_mod, s_, n_src)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graphs = []
        for s_ in sets:
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_):
                out_ = run_step(loss_mod, s_, n_src)
            graphs.append((g_, out_))

    eager_out = [None]          # without graphs: the loss dict of the latest step

    def step_resident(i):
        if graphs is not None:
            graphs[i % N_INPUT_SETS][0].replay()
        else:
            eager_out[0] = run_step(loss_mod, sets[i % N_INPUT_SETS], n_src)

    # End-to-end arm: every step copies its inputs from pinned host memory and reads the loss back to the host.  Two
    # device-side input buffers are used so that the copy of step i+1 (copy stream) overlaps the compute of step i
    # (graph replay on the main stream); the loss of step i is read on the host while step i+1 runs.
    loss_holder = [0.0]
    e2e = None
    if graphs is not None:
        copy_stream = torch.cuda.Stream()
        e2e = {"in": [graphs[0], graphs[1]], "bufs": [sets[0], sets[1]],
               "h2d_done": [torch.cuda.Event(), torch.cuda.Event()],
               "compute_done": [torch.cuda.Event(), torch.cuda.Event()],
               "loss_host": [torch.zeros(1, pin_memory=True), torch.zeros(1, pin_memory=True)]}
        for ev in e2e["compute_done"]:
            ev.record()

    def step_e2e(i):
        h = host_sets[i % 2]
        if e2e is None:
            inp = {k: v.to(dev, non_blocking=True) for k, v in h.items()}
            loss_holder[0] = float(run_step(loss_mod, inp, n_src)["total"].detach())   # device -> host read of the loss
            return
        k = i % 2
        with torch.cuda.stream(copy_stream), torch.no_grad():
            copy_stream.wait_event(e2e["compute_done"][k])          # buffer k is free again
            dev_slabs[k][0].copy_(host_slabs[i % 2][0], non_blocking=True)    # the whole minibatch: one copy
            e2e["h2d_done"][k].record(copy_stream)
        main = torch.cuda.current_stream()
        main.wait_event(e2e["h2d_done"][k])
        graph_k, loss_k = e2e["in"][k]
        graph_k.replay()
        e2e["loss_host"][k].copy_(loss_k["total"].detach(), non_blocking=True)
        e2e["compute_done"][k].record(main)
        if i > 0:                                                     # read the previous step's loss
            e2e["compute_done"][1 - k].synchronize()
            loss_holder[0] = float(e2e["loss_host"][1 - k])

    for i in range(args.warmup):
        step_resident(i)
    sampler = ClockSampler(R.local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = _timing.LAUNCH_COUNT
    ms_total = R.timed(step_resident, args.steps)
    launches = _timing.LAUNCH_COUNT - launches0
    clocks = sampler.summary() if sampler else None
    if args.dump_outputs and rank == 0:
        # now: the passes below run the step again into the same tensors, one of them with the other arithmetic
        last = (args.steps - 1) % N_INPUT_SETS
        dump_outputs(step_outputs(graphs[last][1] if graphs is not None else eager_out[0], sets[last]), args.dump_outputs)

    # per-launch device time of the library calls, live over a second (eager) pass of the same steps
    # (the device is first parked on a ~2 ms spin so that the whole step is already queued when it starts executing:
    # otherwise each event pair also brackets the host's submission gap, which is 15-20 us per call from Python)
    def step_eager(i):
        torch.cuda._sleep(4_000_000)
        run_step(loss_mod, sets[i % N_INPUT_SETS], n_src)
    eager_steps = min(args.steps, 50)
    l0 = _timing.LAUNCH_COUNT
    timer = _timing.KernelTimer()
    with _timing.record(timer):
        R.timed(step_eager, eager_steps)
    ksum = timer.summary()
    tie_fraction = None
    if args.arith == "fast" and ops.LAST_TIE_COUNT is not None:      # near-ties of the min-reprojection re-evaluated exactly
        tie_fraction = int(ops.LAST_TIE_COUNT) / float(wl["b"] * wl["h"] * wl["w"])
    if graphs is not None:       # launches inside a replayed graph are not seen by the Python counter
        launches = (_timing.LAUNCH_COUNT - l0) // eager_steps * args.steps

    for i in range(min(args.warmup, 5)):
        step_e2e(i)
    e2e_steps = max(5, min(args.steps, 500))
    ms_e2e = R.timed(step_e2e, e2e_steps)
    h2d_peak = h2d_ceiling(dev)
    # Opt-in end-to-end mode: the three frames cross the host link as uint8 (what the loader reads from disk) and are
    # converted on the device with the loader's own arithmetic (tcsfm_u8_to_float == custom_transforms.py:74, bit for
    # bit); disparities / poses / K stay fp32.  Same pipeline as above: copy of step i+1 overlaps compute of step i.
    e2e_u8 = None
    if e2e is not None:
        from tcsfm_b200 import dataformat
        img_keys = [k for k in host_sets[0] if k == "target" or k.startswith("source")]
        # the frames are the leading region of the slab (make_inputs puts them first; the alignment padding between
        # them is zero and converts to zero): one uint8 copy + one conversion launch for all of them, one fp32 copy for
        # the rest
        first_other = next(k for k in host_sets[0] if k not in img_keys)
        n_img = (host_sets[0][first_other].data_ptr() - host_slabs[0][0].data_ptr()) // 4
        assert list(host_sets[0])[:len(img_keys)] == img_keys and n_img >= sum(host_sets[0][k].numel() for k in img_keys)
        host_u8 = [(h[0][:n_img] * 255).round().to(torch.uint8).pin_memory() for h in host_slabs]
        dev_u8 = [torch.empty(n_img, dtype=torch.uint8, device=dev) for _ in range(2)]

        def step_e2e_u8(i):
            k = i % 2
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(e2e["compute_done"][k])
                dev_u8[k].copy_(host_u8[i % 2], non_blocking=True)
                dataformat.images_from_uint8(dev_u8[k], dev_slabs[k][0][:n_img])
                dev_slabs[k][0][n_img:].copy_(host_slabs[i % 2][0][n_img:], non_blocking=True)
                e2e["h2d_done"][k].record(copy_stream)
            main = torch.cuda.current_stream()
            main.wait_event(e2e["h2d_done"][k])
            graph_k, loss_k = e2e["in"][k]
            graph_k.replay()
            e2e["loss_host"][k].copy_(loss_k["total"].detach(), non_blocking=True)
            e2e["compute_done"][k].record(main)
            if i > 0:
                e2e["compute_done"][1 - k].synchronize()
                loss_holder[0] = float(e2e["loss_host"][1 - k])
        for i in range(min(args.warmup, 5)):
            step_e2e_u8(i)
        ms_u8 = R.timed(step_e2e_u8, e2e_steps)
        h2d_u8 = n_img + (host_slabs[0][0].numel() - n_img) * 4
        e2e_u8 = {"value": wl["b"] * world * e2e_steps / (ms_u8 / 1e3), "unit": "frames/s", "h2d_bytes_per_step": h2d_u8,
                  "d2h_bytes_per_step": 4, "ms_per_step": ms_u8 / e2e_steps, "steps": e2e_steps,
                  "note": "opt-in: frames cross the host link as uint8 and are converted on the device exactly like the "
                          "reference's loader does on the host (dataformat.images_from_uint8); images quantised to 8 bits"}
    # restore the resident buffers the e2e arm overwrote (sets 0 and 1 double as its staging buffers)
    with torch.no_grad():
        for k_ in range(2):
            fresh = make_inputs(wl, 100 * rank + k_, dev)
            for name, t in fresh.items():
                sets[k_][name].copy_(t)

    sub = {}
    if args.only is None and args.workload == "kitti":
        # driver-visible numbers for the other two modes of BASELINE.json's metric / configs 3-5
        pft_steps = max(1, min(args.steps, 6))
        sub["pft"] = pft_measure(R, "pft", pft_steps, 2, sequence_frames=1591)
        sub["pft_scannet"] = pft_measure(R, "pft-scannet", pft_steps, 2)
        sub["train_ddp" if world > 1 else "train"] = train_measure(R, max(3, min(args.steps, 10)), 3)
    other = None
    alt = "exact" if args.arith == "fast" else "fast"
    if args.only is None and rank == 0 and args.workload == "kitti" and alt in ops.PAIR_ARITHMETICS:
        # the same workload through the other SSIM arithmetic flavour (both are reported every run): CUDA-graph replay of
        # the full step like the headline, per-launch times of the pair kernels from an eager pass
        ops.set_arithmetic(alt)
        alt_ms = None
        if graphs is not None:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for s_ in sets:
                    for _ in range(3):
                        run_step(loss_mod, s_, n_src)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            alt_graphs = []
            for s_ in sets:
                g_ = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_):
                    run_step(loss_mod, s_, n_src)
                alt_graphs.append(g_)
            for i in range(min(args.warmup, 5)):
                alt_graphs[i % N_INPUT_SETS].replay()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for i in range(args.steps):
                alt_graphs[i % N_INPUT_SETS].replay()
            a1.record()
            torch.cuda.synchronize()
            alt_ms = a0.elapsed_time(a1) / args.steps
        t_alt = _timing.KernelTimer()
        with _timing.record(t_alt):
            for i in range(eager_steps):
                step_eager(i)
        k_alt = t_alt.summary()
        other = {"arithmetic": alt, "launch": config["launch"], "ms_per_step": alt_ms,
                 "value": (wl["b"] / (alt_ms / 1e3)) if alt_ms else None, "unit": "frames/s",
                 "kernels": {k: v for k, v in k_alt.items() if k.startswith("pair_")}}
        ops.set_arithmetic(args.arith)
    eager_cuda = None
    if args.only is None and rank == 0:
        eager_cuda = eager_cuda_measure(wl, sets, loss_cfg, max(20, min(args.steps, 50)))
    R.barrier()
    R.close()
    if rank != 0:
        return

    frames = wl["b"] * world
    value = frames * args.steps / (ms_total / 1e3)
    e2e_value = frames * e2e_steps / (ms_e2e / 1e3)
    h2d = host_slabs[0][0].numel() * host_slabs[0][0].element_size()      # the slab that is copied, padding included
    npx = wl["h"] * wl["w"]
    pairs = 2 * n_src * wl["b"] * wl.get("scales", 1)
    # algorithmic bytes per pixel per pair (SURVEY.md §8d / DESIGN.md): fwd 32 R + 8 W, bwd 36 R + 8 W
    per_launch_pairs = 2 * n_src * wl["b"]
    bytes_per_launch = {"pair_loss_fwd": 40 * npx * per_launch_pairs, "pair_loss_bwd": 44 * npx * per_launch_pairs}
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    dom = max((k for k in ksum if k in bytes_per_launch), key=lambda k: ksum[k]["avg_ms"], default=None)
    roofline = None
    if dom:
        ach = bytes_per_launch[dom] / (ksum[dom]["avg_ms"] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.isfile(tpath) and args.workload == "kitti":
            traffic = json.load(open(tpath)).get(args.arith, {}).get(dom)   # dram read+write per launch, committed ncu capture
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "peak_source": peak_src, "avg_launch_ms": ksum[dom]["avg_ms"],
                    "algorithmic_bytes_per_launch": bytes_per_launch[dom],
                    "step_algorithmic_GBps": 84 * npx * pairs / (ms_total / args.steps * 1e-3) / 1e9,
                    "step_frac": 84 * npx * pairs / (ms_total / args.steps * 1e-3) / 1e9 / peak,
                    "kernels": ksum}
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        csteps = args.cpu_steps or 4
        cfps, cms = cpu_port_throughput(wl, csteps, 1, cores)
        cpu_baseline = {"value": cfps, "unit": "frames/s", "cores": cores, "kind": "port", "ms_per_step": cms,
                        "sample": "%d steps of one B=%d minibatch of the same workload (oracle port of the "
                                  "reference's PyTorch CPU path, torch threads=%d)" % (csteps, wl["b"], cores)}
    metric = METRIC if args.workload == "kitti" else "warp+SSIM/L1 loss fwd+bwd frames/s at %dx%d" % (wl["h"], wl["w"])
    line = {"metric": metric, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "pairs_per_s": value * 2 * n_src, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
                    "h2d_GBps_per_gpu": h2d / (ms_e2e / e2e_steps * 1e-3) / 1e9, "h2d_peak_GBps": h2d_peak},
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "e2e_uint8_images": e2e_u8, "eager_cuda_baseline": eager_cuda, "other_arithmetic": other,
            "tie_fraction": tie_fraction}
    line.update(sub)
    emit(line)


if __name__ == "__main__":
    main()
