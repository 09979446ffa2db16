"""ctypes declarations of the C ABI in include/tcsfm.h (one place, used by the
package loader and by the test-only emulator binding)."""
import ctypes as C

ABI_VERSION = 21

ARITH_CPU = 1 << 0
AUTO_MASK = 1 << 1
SSIM = 1 << 2
DEPTH_MASK = 1 << 3
DEPTH_CONSIST = 1 << 4
SHARED_GRADS = 1 << 5
ARITH_BMM_NOFMA = 1 << 6
ARITH_FAST = 1 << 7

PFT_ARGMIN = 1 << 0
PFT_AUTOMASK = 1 << 1
PFT_INVERSE = 1 << 2
PFT_DEPTH_CONSIST = 1 << 3

_fp = C.c_void_p          # device (or, in the emulator, host) pointer to float
_i64 = C.c_int64


class PairGroup(C.Structure):
    """struct tcsfm_pair_group"""
    _fields_ = [
        ("tgt_img", _fp), ("tgt_sb", _i64), ("tgt_sc", _i64),
        ("ref_img", _fp), ("ref_sb", _i64), ("ref_sc", _i64),
        ("tgt_depth", _fp), ("ref_depth", _fp), ("kinv", _fp), ("proj", _fp),
        ("diff_img", _fp), ("mask", _fp), ("sums", _fp), ("coef", _fp),
        ("g_diff", _fp), ("g_scalars", _fp),
        ("min_base", _fp), ("min_stride", _i64), ("min_count", C.c_int32), ("min_index", C.c_int32), ("g_min", _fp),
        ("g_tgt_depth", _fp), ("g_ref_depth", _fp), ("g_proj", _fp),
    ]


class FrameCfg(C.Structure):
    """struct tcsfm_frame_cfg"""
    _fields_ = [("n_groups", C.c_int32), ("role", C.c_int32 * 8), ("w_inverse", C.c_float), ("w_depth", C.c_float),
                ("n_min_pixels", _i64)]


SIGNATURES = {
    "tcsfm_last_error": (C.c_char_p, []),
    "tcsfm_abi_version": (C.c_int, []),
    "tcsfm_warp_fwd": (C.c_int, [_fp, _i64, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _i64, _i64, _fp,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_warp_bwd": (C.c_int, [_fp, _i64, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_ssim_fwd": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_ssim_bwd": (C.c_int, [_fp, _fp, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_ssim_mean_fwd": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_ssim_mean_bwd": (C.c_int, [_fp, _fp, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_pft_reduce_fwd": (C.c_int, [_fp] * 8 + [C.c_int, C.c_int, _i64, C.c_int, C.c_float, _fp, _fp, C.c_void_p]),
    "tcsfm_pft_reduce_bwd": (C.c_int, [_fp] * 8 + [C.c_int, C.c_int, _i64, C.c_int, C.c_float, _fp, _fp,
                                                    _fp, _fp, _fp, _fp, C.c_void_p]),
    "tcsfm_pair_coef_planes": (C.c_int, []),
    "tcsfm_pair_ws_floats": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "tcsfm_pair_loss_fwd": (C.c_int, [C.POINTER(PairGroup), C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_pair_loss_bwd": (C.c_int, [C.POINTER(PairGroup), C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_coef_planes": (C.c_int, []),
    "tcsfm_photo_fwd": (C.c_int, [_fp, _i64, _i64, _fp, _i64, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp,
                                  C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_bwd": (C.c_int, [_fp, _i64, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp,
                                  C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_sweep_partial_floats": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "tcsfm_photo_sweep": (C.c_int, [_fp, _i64, _fp, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp,
                                    C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_sweep_grad_partial_floats": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "tcsfm_photo_sweep_grad": (C.c_int, [_fp, _i64, _fp, _i64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp,
                                         C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_refine": (C.c_int, [_fp, _i64, _fp, _i64] + [_fp] * 14 +
                           [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                            C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_photo_sweep_pairs": (C.c_int, [_fp, _i64, _i64, _fp, _i64, _i64] + [_fp] * 11 +
                                    [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_sweep_grad_pairs": (C.c_int, [_fp, _i64, _i64, _fp, _i64, _i64] + [_fp] * 8 +
                                         [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "tcsfm_photo_refine_pairs": (C.c_int, [_fp, _i64, _i64, _fp, _i64, _i64] + [_fp] * 14 +
                                 [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double,
                                  C.c_double, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_smooth_fwd": (C.c_int, [_fp, _fp, _i64, _i64, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_smooth_bwd": (C.c_int, [_fp, _fp, _i64, _i64, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_pose_proj_fwd": (C.c_int, [_fp, C.c_float, _fp, C.c_int, _fp, C.c_int, C.c_int, C.c_void_p]),
    "tcsfm_pose_proj_bwd": (C.c_int, [_fp, C.c_float, _fp, C.c_int, _fp, _fp, C.c_int, C.c_void_p]),
    "tcsfm_disp_to_depth_fwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, _i64,
                                          C.c_float, C.c_float, C.c_void_p]),
    "tcsfm_disp_to_depth_bwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                          _i64, C.c_float, C.c_void_p]),
    "tcsfm_disp_upsample_to_depth_fwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int,
                                                   C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p]),
    "tcsfm_disp_upsample_to_depth_bwd": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "tcsfm_min_reduce": (C.c_int, [_fp, _i64, C.c_int, _i64, _fp, _fp, _fp, C.POINTER(FrameCfg), _fp, _fp, C.c_void_p]),
    "tcsfm_u8_to_float": (C.c_int, [_fp, _fp, _i64, C.c_void_p]),
    "tcsfm_intrinsics_inverse": (C.c_int, [_fp, _fp, C.c_int, C.c_void_p]),
    "tcsfm_frame_prologue": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, _i64, C.c_float, C.c_float,
                                       C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_float, _fp, C.c_int, _fp, _fp, C.c_int, C.c_void_p]),
    "tcsfm_frame_epilogue": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, _i64, C.c_float,
                                       C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_float, _fp, C.c_int, _fp, _fp, C.c_void_p]),
    "tcsfm_pair_min_resolve": (C.c_int, [C.POINTER(PairGroup), C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                         C.c_int, C.c_float, _fp, _fp, _fp, C.POINTER(FrameCfg), _fp, _fp, C.c_void_p]),
    "tcsfm_frame_finalize": (C.c_int, [_fp, _fp, C.POINTER(FrameCfg), _fp, _fp, C.c_void_p]),
    "tcsfm_frame_bwd_prepare": (C.c_int, [_fp, _fp, C.POINTER(FrameCfg), _fp, _fp, _fp, _i64, C.c_void_p]),
}


def bind(path):
    """dlopen `path` and attach argtypes/restype for every declared symbol.
    Raises if a symbol is missing or the ABI version differs."""
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if not exported
        fn.restype = res
        fn.argtypes = args
    if lib.tcsfm_abi_version() != ABI_VERSION:
        raise RuntimeError("%s: ABI version %d, expected %d" % (path, lib.tcsfm_abi_version(), ABI_VERSION))
    return lib


def check(lib, rc):
    if rc != 0:
        raise RuntimeError(lib.tcsfm_last_error().decode("utf-8", "replace") or "tcsfm call failed (%d)" % rc)
