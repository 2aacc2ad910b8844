"""TEST INFRASTRUCTURE: ctypes access to the oracle of float level 0 (tests/oracle_float/ibl_float_pack_oracle.cpp):
equirect pack and six-image ingest in rgbe, RGBA32F or RGBA16F, and its binary16 rounding.  Built with g++ into a
temporary directory on first use.  Never imported by datum_b200."""

import ctypes
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "oracle_float", "ibl_float_pack_oracle.cpp")

_lib = None


def oracle():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="datum_float_pack_oracle_"), "libibl_float_pack_oracle.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        # the flags of oracle/Makefile: strict IEEE fp32, no contraction
        subprocess.check_call([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-pthread", "-fPIC", "-shared", "-o", out, SRC])
        lib = ctypes.CDLL(out)
        lib.oracle_float_pack_cube.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        lib.oracle_float_ingest_cube_argb32.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        lib.oracle_half_rn_array.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        _lib = lib
    return _lib


# level 0 of each texel format (0 rgbe, 1 RGBA32F, 2 RGBA16F): numpy dtype and channels per texel
_LEVEL0 = {0: (np.uint32, None), 1: (np.float32, 4), 2: (np.float16, 4)}


def _level0(fmt, texels):
    dtype, channels = _LEVEL0[fmt]
    return np.zeros(texels if channels is None else (texels, channels), dtype)


def pack_cube(fmt, image, width, height):
    """Equirect (H, W, 4) float32 image -> level 0 in format `fmt`: the rgbe oracle's resample and edge blend
    with the texel store of the format.  rgbe: uint32 words; F32 / F16: (texels, 4) float32 / float16."""
    image = np.ascontiguousarray(image, dtype=np.float32)
    out = _level0(fmt, 6 * width * height)
    assert oracle().oracle_float_pack_cube(fmt, image.shape[1], image.shape[0], image.ctypes.data, width, height, out.ctypes.data) == 0
    return out


def ingest_cube_argb32(fmt, faces):
    """(6, H, W) uint32 ARGB32 faces -> level 0 in format `fmt` (srgba, vertical mirror)."""
    faces = np.ascontiguousarray(faces, dtype=np.uint32)
    out = _level0(fmt, faces.size)
    assert oracle().oracle_float_ingest_cube_argb32(fmt, faces.ctypes.data, faces.shape[2], faces.shape[1], out.ctypes.data) == 0
    return out


def half_rn(x):
    """float32 values (finite, non-negative) -> float16 of min(x, 65504) rounded to nearest-even."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.zeros(x.shape, np.uint16)
    oracle().oracle_half_rn_array(x.ctypes.data, x.size, out.ctypes.data)
    return out.view(np.float16)


