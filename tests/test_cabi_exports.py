"""The CUDA C-ABI library loads on a machine without a GPU and exports every symbol
include/tcsfm.h declares (no compute calls here)."""
import os
import re
import subprocess

from tcsfm_b200 import _cabi, _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "tcsfm.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tcsfm_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_header_symbols():
    path = build.build()
    assert os.path.isfile(path)
    lib = _lib.lib()
    syms = header_symbols()
    assert len(syms) >= 8
    for s in syms:
        assert hasattr(lib, s), s
        assert s in _cabi.SIGNATURES, "ctypes binding missing for %s" % s
    assert lib.tcsfm_abi_version() == _cabi.ABI_VERSION
    assert lib.tcsfm_last_error() == b""


def test_library_targets_sm_100a():
    # the cuobjdump of the toolkit that built the library, which need not be on PATH; when nvcc itself was found only
    # through PATH, build._nvcc() returns the bare "nvcc" and cuobjdump is looked up on PATH as well
    cuobjdump = os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_struct_layout_matches_header():
    import ctypes
    # 2 x (pointer + 2 strides) for the images, 15 further pointers, a stride and two int32: 23 x 8 bytes
    assert ctypes.sizeof(_cabi.PairGroup) == 23 * 8
    assert ctypes.sizeof(_cabi.FrameCfg) == 4 + 32 + 4 + 4 + 4 + 8   # incl. 4 bytes of padding before the int64
