"""Float chains (RGBA32F / RGBA16F) on the CPU: the float oracle pinned to the rgbe oracle, and the host
compilation of the float kernels' record layout and tap arithmetic (tests/emu/prefilter_f_emu.cpp)
against the float oracle.  A check OF the kernel source, not a fallback for it."""

import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import datum_b200
import float_oracle_lib
import float_parity
import oracle_lib
from datum_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_emu = None


def emu():
    """g++ build of tests/emu/prefilter_f_emu.cpp, into a temporary directory."""
    global _emu
    if _emu is None:
        out = os.path.join(tempfile.mkdtemp(prefix="datum_float_emu_"), "libprefilter_f_emu.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                               os.path.join(ROOT, "tests", "emu", "prefilter_f_emu.cpp"),
                               os.path.join(ROOT, "datum_b200", "csrc", "ibl_tables.cpp")])
        lib = ctypes.CDLL(out)
        lib.emu_prefilter_level_float.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_void_p] * 2
        lib.emu_half_to_float.argtypes = [ctypes.c_uint32]
        lib.emu_half_to_float.restype = ctypes.c_float
        lib.emu_float_to_half.argtypes = [ctypes.c_float]
        lib.emu_float_to_half.restype = ctypes.c_uint32
        _emu = lib
    return _emu


def emu_level(fmt, src, ws, hs, level, levels, samples):
    src = np.ascontiguousarray(src)
    n = 6 * (ws >> 1) * (hs >> 1)
    f32 = np.zeros((n, 3), np.float32)
    f16 = np.zeros((n, 4), np.float16) if fmt == datum_b200.FORMAT_F16 else None
    emu().emu_prefilter_level_float(fmt, src.ctypes.data, ws, hs, level, levels, samples, f32.ctypes.data, f16.ctypes.data if f16 is not None else None)
    return f32, f16


@pytest.mark.parametrize("w,h", [(16, 16), (32, 32), (24, 12)])
@pytest.mark.parametrize("samples", [1024, 7])
def test_float_oracle_is_bit_identical_to_the_rgbe_oracle_on_decoded_words(w, h, samples):
    """The float oracle fed the decoded words of an rgbe level gives exactly the fp32 values the rgbe
    oracle hands to rgbe(): the only difference between the two is the texel fetch."""
    words = synth.synthetic_chain(w, h, 1, probe=3, noise=True, sun=True)
    levels = 4
    _, want = oracle_lib.prefilter_level(words, w, h, 1, levels, samples)
    got = float_oracle_lib.prefilter_level_rgba32f(oracle_lib.rgbe_decode_array(words), w, h, 1, levels, samples)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_half_conversions_match_numpy():
    lib = emu()
    halves = np.arange(0, 0x7C00, 7, dtype=np.uint16)
    got = np.array([lib.emu_half_to_float(int(h)) for h in halves], np.float32)
    assert np.array_equal(got, halves.view(np.float16).astype(np.float32))

    rng = np.random.default_rng(5)
    x = np.concatenate([np.exp2(rng.uniform(-30, 17, 4000)), [0.0, 65504.0, 65519.0, 65520.0, 1e9, 2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -26]]).astype(np.float32)
    got = np.array([lib.emu_float_to_half(float(v)) for v in x], np.uint16)
    assert np.array_equal(got, float_parity.round_f16(x).view(np.uint16))


@pytest.mark.parametrize("fmt", [datum_b200.FORMAT_F32, datum_b200.FORMAT_F16])
@pytest.mark.parametrize("w,h,level,levels,samples,sun", [
    (16, 16, 1, 5, 1024, True),
    (16, 16, 3, 5, 64, False),
    (24, 12, 1, 3, 1024, True),     # non-square, not a power of two
    (11, 11, 1, 2, 256, True),      # odd source: the non-projective footprint
    (2, 2, 1, 2, 1024, False),      # smallest legal level: 2x2 -> 1x1
])
def test_emulated_float_level_matches_the_float_oracle(fmt, w, h, level, levels, samples, sun):
    cube = synth.synthetic_cube(w, h, probe=7, noise=True, sun=sun)
    src = cube.astype(np.float16) if fmt == datum_b200.FORMAT_F16 else cube
    f32, f16 = emu_level(fmt, src, w, h, level, levels, samples)
    float_parity.check_float_level(f32, f16, src, w, h, level, levels, samples)
    if f16 is not None:
        assert np.array_equal(f16[:, :3].view(np.uint16), float_parity.round_f16(f32).view(np.uint16))


def test_f16_format_constant():
    assert datum_b200.FORMAT_F16 == 2
    with open(os.path.join(ROOT, "include", "datum_ibl_cuda.h")) as f:
        assert re.search(r"#define DATUM_IBL_FORMAT_F16 2\b", f.read())
