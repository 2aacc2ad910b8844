"""The impulse-response criterion (tests/impulse.py) on the host compilations of the kernel arithmetic: the rgbe
one-sample and pair kernels (tests/emu/prefilter_emu.cpp) against the rgbe oracle, the float kernels
(tests/emu/prefilter_f_emu.cpp) against the float oracle.  Pins the criterion's constants to the kernels' own
arithmetic, on a machine without a GPU."""

import numpy as np
import pytest

import datum_b200
import emu_lib
import float_oracle_lib
import impulse
import oracle_lib
from test_float_chain_cpu import emu_level

# (source size, level, levels, samples, impulses (face, y, x) of channels r, g, b: a face interior, a texel of a
# face edge row or column, a face corner)
CASES = [
    (64, 1, 8, 1024, [(0, 31, 31), (1, 0, 17), (2, 63, 63)]),
    (32, 2, 6, 1024, [(5, 10, 5), (3, 16, 0), (4, 0, 31)]),
    (16, 4, 5, 16, [(3, 7, 7), (2, 0, 9), (1, 15, 0)]),
]


@pytest.mark.parametrize("kernel", ["dn", "dp"])
@pytest.mark.parametrize("ws,level,levels,samples,spots", CASES)
def test_emulated_rgbe_kernels_answer_an_impulse_like_the_oracle(kernel, ws, level, levels, samples, spots):
    src, radiance = impulse.rgbe_source(ws, ws, spots, 1000.0)
    n = 6 * (ws >> 1) ** 2
    words, f32 = np.zeros(n, np.uint32), np.zeros((n, 3), np.float32)
    run = emu_lib.load().emu_prefilter_level_dn if kernel == "dn" else emu_lib.load().emu_prefilter_level_dp
    run(src.ctypes.data, ws, ws, level, levels, samples, 16, words.ctypes.data, f32.ctypes.data)
    _, want = oracle_lib.prefilter_level(src, ws, ws, level, levels, samples)
    print(impulse.check(f32, want, radiance, ws, ws, level, levels, samples))


@pytest.mark.parametrize("fmt", [datum_b200.FORMAT_F32, datum_b200.FORMAT_F16])
@pytest.mark.parametrize("ws,level,levels,samples,spots", CASES)
def test_emulated_float_kernels_answer_an_impulse_like_the_float_oracle(fmt, ws, level, levels, samples, spots):
    dtype = np.float16 if fmt == datum_b200.FORMAT_F16 else np.float32
    src, radiance = impulse.float_source(ws, ws, spots, 1000.0, dtype)
    f32, f16 = emu_level(fmt, src, ws, ws, level, levels, samples)
    want = float_oracle_lib.prefilter_level_rgba32f(src.astype(np.float32), ws, ws, level, levels, samples)
    print(impulse.check(f32, want, radiance, ws, ws, level, levels, samples, got_f16=f16))


def test_lobe_rows_hold_every_nonzero_texel():
    """The row selection of the big GPU levels: outside lobe_rows the oracle's response is exactly 0."""
    ws, level, levels, samples = 64, 1, 8, 1024
    spots = [(4, 31, 31), (4, 0, 40)]
    src, _ = impulse.rgbe_source(ws, ws, spots, 1000.0)
    _, want = oracle_lib.prefilter_level(src, ws, ws, level, levels, samples)
    rows = impulse.lobe_rows(ws, ws, spots, level, levels, samples)
    assert not rows.all()
    nonzero = (want.reshape(6 * (ws >> 1), -1) > 0).any(axis=1)
    assert not np.any(nonzero & ~rows)
    assert impulse.row_runs(np.array([1, 1, 0, 1, 0, 0, 1], bool)) == [(0, 2), (3, 4), (6, 7)]
