"""TEST INFRASTRUCTURE: ctypes access to the float-chain oracle (tests/oracle_float/ibl_float_oracle.cpp),
built with g++ into a temporary directory on first use.  Never imported by datum_b200."""

import ctypes
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "oracle_float", "ibl_float_oracle.cpp")

_lib = None


def oracle():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="datum_float_oracle_"), "libibl_float_oracle.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        # the flags of oracle/Makefile: strict IEEE fp32, no contraction
        subprocess.check_call([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-pthread", "-fPIC", "-shared", "-o", out, SRC])
        lib = ctypes.CDLL(out)
        lib.oracle_prefilter_level_rgba32f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int,
                                                       ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        _lib = lib
    return _lib


def prefilter_level_rgba32f(src, ws, hs, level, levels, samples=1024, row_begin=0, row_end=None, threads=0):
    """fp32 rgb of the (ws/2 x hs/2 x 6) level computed from the RGBA float level `src` (float32, or
    float16 widened exactly); rows outside [row_begin, row_end) stay 0."""
    src = np.ascontiguousarray(src, dtype=np.float32).reshape(-1, 4)
    wd, hd = ws >> 1, hs >> 1
    if row_end is None:
        row_end = 6 * hd
    f32 = np.zeros((6 * hd * wd, 3), np.float32)
    roughness = np.float32(level) / np.float32(levels - 1)
    oracle().oracle_prefilter_level_rgba32f(src.ctypes.data, ws, hs, float(roughness), samples, row_begin, row_end, f32.ctypes.data, threads)
    return f32
