"""Loader for the committed golden fixtures (tests/golden/*.npz, generated from
the unmodified reference by tests/golden/make_golden.py)."""
import glob
import hashlib
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))

TRAIN_CFG = {"l1_weight": 0.15, "l_ssim_weight": 0.85, "l_smooth_weight": 0.05, "num_scales": 1,
             "l_depth_consist_weight": 0.14, "min_depth": 0.06, "max_depth": 2.67, "l_smooth": False,
             "l_reconstruction": True, "l_inverse": True, "l_depth_consist": False,
             "with_auto_mask": True, "l_ssim": True, "with_depth_mask": False}
FULL_CFG = dict(TRAIN_CFG, l_depth_consist=True, with_depth_mask=True)
NOAUTO_CFG = dict(FULL_CFG, with_auto_mask=False)
SMOOTH_CFG = dict(TRAIN_CFG, l_smooth=True)
PAIR_CFGS = {"train": TRAIN_CFG, "full": FULL_CFG, "noauto": NOAUTO_CFG}
LOSS_CFGS = {"train": TRAIN_CFG, "full": FULL_CFG, "smooth": SMOOTH_CFG}
PFT_OPTIONS = {"num_source_imgs": 2, "diff_img_argmin": True, "automasking": True,
               "l_inverse_reconstruction": True, "l_depth_consist": True, "l_depth_consist_weight": 0.15,
               "l_depth_init": True, "l_depth_init_weight": 0.1, "l_smooth": False, "l_smooth_weight": 0.05,
               "l_pose_consist": False, "plotting": False, "epochs": 20}


# Fresh inputs (none of the golden cases): the warp of the second source with the outer depths, both euler2mat, the
# smoothness loss and the pairwise diff_img / valid_mask, stored outside the enumerated CASES.  The inputs are
# regenerated from the seed and checked against a stored digest.
FRESH_FRAMES = dict(b=2, h=40, w=56, n_src=2, seed=11, yaw=0.03)
FRESH_PATH = os.path.join(GOLDEN_DIR, "fresh", "b2_40x56_seed11.npz")


def fresh_inputs_digest(fr):
    h = hashlib.sha256()
    for t in [fr["target"], *fr["sources"], *fr["disps"], *fr["depths"], *fr["poses"], *fr["poses_inv"], fr["K"]]:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def fresh_outputs(fr, inverse_warp2, euler2mat_stn, euler2mat_geometry, smooth_loss, pairwise_loss):
    """The arrays compared on the fresh inputs; each callable has the signature of the reference function it names
    (pairwise_loss: Compute_Loss(FULL_CFG).compute_pairwise_loss without the trailing epoch argument)."""
    out = {}
    warp = inverse_warp2(fr["sources"][1], fr["depths"][0], fr["depths"][2], -fr["poses"][1], fr["K"])
    for k, t in zip(("projected_img", "valid_mask", "projected_depth", "computed_depth"), warp):
        out["warp/" + k] = t
    out["euler2mat/stn"] = euler2mat_stn(fr["poses"][0][:, 3:])
    out["euler2mat/geometry_helpers"] = euler2mat_geometry(fr["poses"][0][:, 3:])
    out["smooth_loss"] = smooth_loss(fr["disps"][0], fr["target"])
    pair = pairwise_loss(fr["target"], fr["sources"][0], fr["depths"][0], fr["depths"][1], -fr["poses"][0], fr["K"])
    out["pair_full/diff_img"], out["pair_full/valid_mask"] = pair[2], pair[3]
    return {k: v.detach().float().cpu() for k, v in out.items()}


def fresh_fns_reference(ref):
    """fresh_outputs' callables from the reference modules (refshim.load_reference())."""
    def warp(*a):
        ref.stn.pixel_coords = None
        return ref.stn.inverse_warp2(*a, "zeros")
    return dict(inverse_warp2=warp, euler2mat_stn=ref.stn.euler2mat, euler2mat_geometry=ref.geometry_helpers.euler2mat,
                smooth_loss=ref.losses.get_smooth_loss,
                pairwise_loss=lambda *a: ref.losses.Compute_Loss(FULL_CFG).compute_pairwise_loss(*a, 5))


def fresh_fns_oracle():
    from oracle import ref_torch as O
    return dict(inverse_warp2=O.inverse_warp2, euler2mat_stn=O.euler_to_matrix, euler2mat_geometry=O.euler_to_matrix,
                smooth_loss=O.smooth_loss, pairwise_loss=lambda *a: O.pairwise_loss(FULL_CFG, *a))


def load_fresh():
    z = np.load(FRESH_PATH)
    return {k: (z[k].astype(np.float32) if z[k].dtype == np.uint8 else z[k]) for k in z.files}


class Golden:
    def __init__(self, name, device="cpu"):
        self.name = name
        self.device = device
        self._z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))

    def __contains__(self, key):
        return key in self._z.files

    def np(self, key):
        return self._z[key]

    def t(self, key):
        a = self._z[key]
        if a.dtype == np.uint8:
            a = a.astype(np.float32)
        return torch.from_numpy(a).to(self.device)

    def frames(self):
        """Inputs in the layout of tcsfm_b200.synth.make_frames."""
        disps = [self.t("in/disp%d" % j) for j in range(3)]
        lo, hi = 0.06, 2.67
        depths = [1 / (1 / hi + (1 / lo - 1 / hi) * d) for d in disps]
        return {"target": self.t("in/target"), "sources": [self.t("in/source%d" % j) for j in range(2)],
                "disps": disps, "depths": depths,
                "poses": [self.t("in/pose%d" % j) for j in range(2)],
                "poses_inv": [self.t("in/pose_inv%d" % j) for j in range(2)], "K": self.t("in/K")}


def rel_l2(a, b):
    a = a.detach().double().flatten().cpu()
    b = b.detach().double().flatten().cpu()
    den = b.norm().item()
    return (a - b).norm().item() / den if den > 0 else (a - b).norm().item()
