"""Generates tests/golden/*.npz and tests/golden/fresh/ from the UNMODIFIED
reference imported on CPU.
Run:  TCSFM_REFERENCE_ROOT=<checkout of the reference> python tests/golden/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md §4/§8c); these
fixtures are the pin for ``oracle/`` and for the CUDA path.  Inputs are stored
next to the outputs of the cases so that they do not depend on RNG
reproducibility; the fresh fixture stores a digest of its seeded inputs instead.

``--fresh-from-oracle`` writes only the fresh fixture, from oracle/ref_torch.py,
for where the reference is not at hand; its ``source`` entry says so.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import goldens  # noqa: E402
import refshim  # noqa: E402
from tcsfm_b200 import synth  # noqa: E402

torch.set_num_threads(1)
ref = None                  # the reference modules, loaded in __main__

TRAIN_CFG = {"l1_weight": 0.15, "l_ssim_weight": 0.85, "l_smooth_weight": 0.05, "num_scales": 1,
             "l_depth_consist_weight": 0.14, "min_depth": 0.06, "max_depth": 2.67, "l_smooth": False,
             "l_reconstruction": True, "l_inverse": True, "l_depth_consist": False,
             "with_auto_mask": True, "l_ssim": True, "with_depth_mask": False}
FULL_CFG = dict(TRAIN_CFG, l_depth_consist=True, with_depth_mask=True)
NOAUTO_CFG = dict(FULL_CFG, with_auto_mask=False)
PFT_OPTIONS = {"num_source_imgs": 2, "diff_img_argmin": True, "automasking": True,
               "l_inverse_reconstruction": True, "l_depth_consist": True, "l_depth_consist_weight": 0.15,
               "l_depth_init": True, "l_depth_init_weight": 0.1, "l_smooth": False, "l_smooth_weight": 0.05,
               "l_pose_consist": False, "plotting": False, "epochs": 20}


def npy(t, like=None):
    if t is None:               # input did not take part in the objective
        t = torch.zeros_like(like)
    return t.detach().cpu().numpy()


def leaf(t):
    return t.clone().detach().requires_grad_(True)


def gen_case(name, b, h, w, seed, yaw):
    out = {}
    fr = synth.make_frames(b, h, w, n_src=2, seed=seed, yaw=yaw)
    gen = torch.Generator().manual_seed(1000 + seed)
    out["in/target"] = npy(fr["target"])
    for j in range(2):
        out["in/source%d" % j] = npy(fr["sources"][j])
        out["in/pose%d" % j] = npy(fr["poses"][j])
        out["in/pose_inv%d" % j] = npy(fr["poses_inv"][j])
    for j in range(3):
        out["in/disp%d" % j] = npy(fr["disps"][j])
    out["in/K"] = npy(fr["K"])
    up = {k: torch.randn(b, c, h, w, generator=gen) for k, c in
          (("g_img", 3), ("g_pd", 1), ("g_cd", 1), ("g_diff", 1))}
    for k, v in up.items():
        out["in/" + k] = npy(v)

    _, depths = zip(*[ref.learning_helpers.disp_to_depth(d, 0.06, 2.67) for d in fr["disps"]])
    K = fr["K"]

    # --- inverse_warp2 (models/stn.py:234) fwd + bwd -------------------------
    ref.stn.pixel_coords = None
    d0, d1, p0 = leaf(depths[0]), leaf(depths[1]), leaf(-fr["poses"][0])
    pim, vm, pd, cd = ref.stn.inverse_warp2(fr["sources"][0], d0, d1, p0, K, "zeros")
    obj = (pim * up["g_img"]).sum() + (pd * up["g_pd"]).sum() + (cd * up["g_cd"]).sum()
    obj.backward()
    out.update({"warp/projected_img": npy(pim), "warp/valid_mask": npy(vm), "warp/projected_depth": npy(pd),
                "warp/computed_depth": npy(cd), "warp/g_depth": npy(d0.grad), "warp/g_ref_depth": npy(d1.grad),
                "warp/g_pose": npy(p0.grad)})

    # --- SSIM (losses.py:27) fwd + bwd --------------------------------------
    x, y = leaf(fr["target"]), leaf(fr["sources"][0])
    s = ref.losses.SSIM_Loss()(x, y)
    (s * up["g_img"]).sum().backward()
    out.update({"ssim/map": npy(s), "ssim/g_x": npy(x.grad), "ssim/g_y": npy(y.grad)})

    # --- compute_pairwise_loss (losses.py:151) under three flag profiles -----
    for tag, cfg in (("train", TRAIN_CFG), ("full", FULL_CFG), ("noauto", NOAUTO_CFG)):
        ref.stn.pixel_coords = None
        loss_mod = ref.losses.Compute_Loss(cfg)
        d0, d1, p0 = leaf(depths[0]), leaf(depths[1]), leaf(-fr["poses"][0])
        l_rep, l_dep, diff, vmask, _ = loss_mod.compute_pairwise_loss(
            fr["target"], fr["sources"][0], d0, d1, p0, K, 5)
        obj = l_rep + (diff * up["g_diff"]).sum()
        if torch.is_tensor(l_dep):
            obj = obj + 0.5 * l_dep
        obj.backward()
        out.update({"pair_%s/l_reprojection" % tag: npy(l_rep),
                    "pair_%s/l_depth" % tag: npy(torch.as_tensor(l_dep, dtype=torch.float32)),
                    "pair_%s/diff_img" % tag: npy(diff), "pair_%s/valid_mask" % tag: npy(vmask),
                    "pair_%s/g_depth" % tag: npy(d0.grad),
                    "pair_%s/g_ref_depth" % tag: npy(d1.grad, d1),
                    "pair_%s/g_pose" % tag: npy(p0.grad)})

    # --- Compute_Loss.forward (losses.py:75) + backward ----------------------
    for tag, cfg in (("train", TRAIN_CFG), ("full", FULL_CFG), ("smooth", dict(TRAIN_CFG, l_smooth=True))):
        ref.stn.pixel_coords = None
        loss_mod = ref.losses.Compute_Loss(cfg)
        disps = [leaf(d) for d in fr["disps"]]
        poses = [leaf(p) for p in fr["poses"]]
        poses_inv = [leaf(p) for p in fr["poses_inv"]]
        losses = loss_mod(fr["sources"], fr["target"], [poses, poses_inv], [[disps[0]], [disps[1]], [disps[2]]], K)
        losses["total"].sum().backward()
        for k, v in losses.items():
            out["loss_%s/%s" % (tag, k)] = npy(v)
        for j in range(3):
            out["loss_%s/g_disp%d" % (tag, j)] = npy(disps[j].grad, disps[j])
        for j in range(2):
            out["loss_%s/g_pose%d" % (tag, j)] = npy(poses[j].grad, poses[j])
            out["loss_%s/g_pose_inv%d" % (tag, j)] = npy(poses_inv[j].grad, poses_inv[j])

    # --- solve_pose_iteratively(return_errors) + compute_optimization_loss ---
    ref.stn.pixel_coords = None
    net = synth.TinyPoseNet(seed=seed)
    dl = [leaf(d) for d in depths]
    poses, poses_inv, outputs = ref.train_mono.solve_pose_iteratively(
        3, dl, net, fr["target"], fr["sources"], K, return_errors=True)
    fake_self = types.SimpleNamespace(options=PFT_OPTIONS, ssim_loss=ref.losses.SSIM_Loss(),
                                      target_disparity=fr["disps"][0] * 0.9 + 0.02)
    tdisp = leaf(fr["disps"][0])
    loss = ref.optimizer.DepthOptimizer.compute_optimization_loss(
        fake_self, 1, 0, fr["target"], tdisp, outputs["fwd"], outputs["inv"])
    loss.sum().backward()
    out["pft/loss"] = npy(loss)
    out["pft/g_tdisp"] = npy(tdisp.grad)
    for j in range(3):
        out["pft/g_depth%d" % j] = npy(dl[j].grad, dl[j])
    for j in range(2):
        out["pft/pose%d" % j] = npy(poses[j])
        out["pft/pose_inv%d" % j] = npy(poses_inv[j])
    for side in ("fwd", "inv"):
        for k in ("diff_img", "valid_mask", "weight_mask", "auto_mask_error", "auto_mask"):
            out["pft/%s/%s" % (side, k)] = npy(outputs[side][k])

    # --- compute_photometric_error (optimization_experiments/helpers.py:8) ---
    ref.stn.pixel_coords = None
    with torch.no_grad():
        res = ref.helpers.compute_photometric_error(fr["target"][:1], fr["sources"][0][:1], depths[0][:1],
                                                    depths[1][:1], fr["poses"][0][:1], K[:1])
    for k in ("diff_img", "img_rec", "valid_mask", "weight_mask"):
        out["photo/%s" % k] = npy(res[k])

    for k in list(out.keys()):       # 0/1 masks are stored as bytes
        if k.endswith("mask") and not k.endswith("weight_mask"):
            assert set(np.unique(out[k]).tolist()) <= {0.0, 1.0}, k
            out[k] = out[k].astype(np.uint8)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def gen_fresh(fns, source):
    fr = synth.make_frames(**goldens.FRESH_FRAMES)
    out = {k: v.numpy() for k, v in goldens.fresh_outputs(fr, **fns).items()}
    for k in out:               # 0/1 masks are stored as bytes
        if k.endswith("valid_mask"):
            assert set(np.unique(out[k]).tolist()) <= {0.0, 1.0}, k
            out[k] = out[k].astype(np.uint8)
    out["in/sha256"] = np.array(goldens.fresh_inputs_digest(fr))
    out["source"] = np.array(source)
    os.makedirs(os.path.dirname(goldens.FRESH_PATH), exist_ok=True)
    np.savez_compressed(goldens.FRESH_PATH, **out)
    print("fresh ->", goldens.FRESH_PATH, "%.1f KB" % (os.path.getsize(goldens.FRESH_PATH) / 1024))


if __name__ == "__main__":
    if sys.argv[1:] == ["--fresh-from-oracle"]:
        gen_fresh(goldens.fresh_fns_oracle(), "oracle/ref_torch.py")
        sys.exit(0)
    ref = refshim.load_reference()
    gen_case("small_b2_24x40", 2, 24, 40, seed=1, yaw=0.01)
    gen_case("mid_b2_64x96", 2, 64, 96, seed=2, yaw=0.01)
    gen_case("yaw_b2_32x48", 2, 32, 48, seed=3, yaw=0.09)     # ~5 deg: large OOB band
    gen_fresh(goldens.fresh_fns_reference(ref), "reference")
