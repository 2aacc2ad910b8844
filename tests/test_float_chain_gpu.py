"""GPU parity of the float prefilter chains (RGBA32F / RGBA16F, prefilter_f.cu) through the C ABI, against
the float oracle on the same source level (float_parity.py)."""

import ctypes

import numpy as np
import pytest
import torch

import datum_b200
import float_parity
import oracle_lib
from datum_b200 import synth

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F32, F16 = datum_b200.FORMAT_F32, datum_b200.FORMAT_F16
TORCH_DTYPE = {F32: torch.float32, F16: torch.float16}
NP_DTYPE = {F32: np.float32, F16: np.float16}


@pytest.fixture(scope="module")
def fctx():
    context = datum_b200.IblContext(0)
    yield context
    context.close()


def level_offsets(w, h, levels):
    return datum_b200.level_offsets(w, h, levels)


def source_chain(fmt, w, h, levels, probe=11, noise=True, sun=False):
    """(texels, 4) host chain of the format, level 0 filled from synth.synthetic_cube."""
    offs = level_offsets(w, h, levels)
    chain = np.zeros((offs[-1], 4), NP_DTYPE[fmt])
    cube = synth.synthetic_cube(w, h, probe=probe, noise=noise, sun=sun)
    chain[: offs[1]] = cube.reshape(-1, 4).astype(NP_DTYPE[fmt])
    return chain


def run_chain_device(ctx, fmt, chain, w, h, levels, samples):
    """Chain on the device; returns (chain, fp32 rgb of levels >= 1)."""
    offs = level_offsets(w, h, levels)
    d_chain = torch.from_numpy(chain.copy()).to(DEV)
    d_f32 = torch.zeros(max(1, (offs[-1] - offs[1]) * 3), dtype=torch.float32, device=DEV)
    ctx.buildmips_cube_float_device(fmt, w, h, levels, d_chain, samples, d_f32)
    ctx.synchronize()
    return d_chain.cpu().numpy(), d_f32.cpu().numpy().reshape(-1, 3)


def check_chain_level(fmt, got, got_f32, w, h, levels, samples, level, ranges=None):
    offs = level_offsets(w, h, levels)
    ws, hs = w >> (level - 1), h >> (level - 1)
    src = got[offs[level - 1]:offs[level]]
    out_f32 = got_f32[offs[level] - offs[1]:offs[level + 1] - offs[1]]
    out = got[offs[level]:offs[level + 1]]
    if fmt == F32:
        # the stored level is the fp32 result itself, alpha 1.0
        assert np.array_equal(out[:, :3], out_f32) and np.all(out[:, 3] == 1.0)
    for a, b in ranges or [(0, 6 * (hs >> 1))]:
        float_parity.check_float_level(out_f32, out if fmt == F16 else None, src, ws, hs, level, levels, samples, row_begin=a, row_end=b)


def spot_ranges(hd, rows=4):
    """Top edge of face 0, the seam of faces 0 and 1, the middle of face 2, the bottom edge of face 5."""
    return [(0, rows), (hd - rows // 2, hd + rows // 2), (2 * hd + hd // 2, 2 * hd + hd // 2 + rows), (6 * hd - rows, 6 * hd)]


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("sun", [False, True])
@pytest.mark.parametrize("w,h,levels,samples", [
    (32, 32, 6, 1024),      # all levels down to 1x1 faces
    (64, 64, 7, 1024),
    (128, 128, 8, 1024),
    (64, 64, 4, 4096),
    (16, 16, 5, 16),
    (24, 12, 3, 1024),      # non-square, not a power of two
    (2, 2, 2, 1024),        # smallest legal chain
])
def test_every_float_level_matches_the_float_oracle_on_the_same_source(fctx, fmt, sun, w, h, levels, samples):
    chain = source_chain(fmt, w, h, levels, sun=sun)
    got, got_f32 = run_chain_device(fctx, fmt, chain, w, h, levels, samples)
    offs = level_offsets(w, h, levels)
    assert np.array_equal(got[: offs[1]].view(np.uint8), chain[: offs[1]].view(np.uint8))     # level 0 untouched
    for level in range(1, levels):
        check_chain_level(fmt, got, got_f32, w, h, levels, samples, level)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_baseline_config_2_float_chain_on_spot_rows(fctx, fmt):
    """512^2 faces, 8 levels, 1024 spp: the 4-warp and 8-warp pair kernels with tile queues (levels 1-3,
    spot rows at face edges, a seam and a face centre) and the tail kernel (levels 4-7, complete)."""
    w, levels, samples = 512, 8, 1024
    chain = source_chain(fmt, w, w, levels, probe=0, sun=True)
    got, got_f32 = run_chain_device(fctx, fmt, chain, w, w, levels, samples)
    for level in range(1, levels):
        hd = (w >> (level - 1)) >> 1
        check_chain_level(fmt, got, got_f32, w, w, levels, samples, level, spot_ranges(hd) if level <= 3 else None)


def test_baseline_config_3_level_1_in_f16_on_spot_rows(fctx):
    """2048^2 -> 1024^2 at 4096 spp (12 levels): the sector table read through L1, faces at the
    proj_usable limit.  No sun, like the rgbe chain's test of this launch."""
    w, levels, samples = 2048, 12, 4096
    src = source_chain(F16, w, w, 1, probe=1, sun=False)
    d_src = torch.from_numpy(src).to(DEV)
    n = 6 * (w >> 1) * (w >> 1)
    d_dst = torch.zeros((n, 4), dtype=torch.float16, device=DEV)
    d_f32 = torch.zeros((n, 3), dtype=torch.float32, device=DEV)
    fctx.prefilter_level_float_device(F16, d_src, w, w, 1, levels, samples, 0, 6 * (w >> 1), d_dst, d_f32)
    fctx.synchronize()
    got16, got32 = d_dst.cpu().numpy(), d_f32.cpu().numpy()
    # 4096 samples: the oracle's sequential fp32 sum differs from the kernel's by ~sqrt(4096) * 2^-24 of a
    # texel (3e-5 at most here), which moves about 1 % of the values across a binary16 rounding boundary;
    # they stay within 1 ulp, the identical share is held to 98 % (measured 98.99 %)
    for a, b in spot_ranges(w >> 1, rows=2):
        float_parity.check_float_level(got32, got16, src, w, w, 1, levels, samples, row_begin=a, row_end=b, min_identical=0.98)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_odd_source_at_pair_kernel_slab_sizes(fctx, fmt):
    """101 x 101 -> 50 x 50: 15 000 destination texels, above the tail kernel's slab size, but a source
    the pair kernel cannot address (odd): the tail kernel takes the whole level.  No sun: next to the
    2e4 disc a footprint moved by the reciprocal's two-ulp shrink changes a clean texel by up to 8e-4,
    inside criterion (i) but two binary16 ulps."""
    w, levels, samples = 101, 2, 1024
    src = source_chain(fmt, w, w, 1, probe=4, sun=False)
    d_src = torch.from_numpy(src).to(DEV)
    n = 6 * 50 * 50
    d_dst = torch.zeros((n, 4), dtype=TORCH_DTYPE[fmt], device=DEV)
    d_f32 = torch.zeros((n, 3), dtype=torch.float32, device=DEV)
    fctx.prefilter_level_float_device(fmt, d_src, w, w, 1, levels, samples, 0, 300, d_dst, d_f32)
    fctx.synchronize()
    float_parity.check_float_level(d_f32.cpu().numpy(), d_dst.cpu().numpy() if fmt == F16 else None, src, w, w, 1, levels, samples)


def test_f32_input_up_to_1e12(fctx):
    w, levels, samples = 64, 4, 1024
    chain = source_chain(F32, w, w, levels, probe=2, sun=True)
    chain[:, :3] *= np.float32(1e12) / chain[:, :3].max()
    assert 0.999e12 <= chain[:, :3].max() <= 1.001e12
    got, got_f32 = run_chain_device(fctx, F32, chain, w, w, levels, samples)
    assert np.all(np.isfinite(got_f32))
    for level in range(1, levels):
        check_chain_level(F32, got, got_f32, w, w, levels, samples, level)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_host_entry_equals_device_entry(fctx, fmt):
    w, levels, samples = 64, 5, 256
    chain = source_chain(fmt, w, w, levels, probe=9, sun=True)
    want, _ = run_chain_device(fctx, fmt, chain, w, w, levels, samples)

    pageable = chain.copy()
    fctx.buildmips_cube_float(fmt, w, w, levels, pageable, samples)
    assert np.array_equal(pageable.view(np.uint8), want.view(np.uint8))

    pinned = torch.from_numpy(chain.copy()).pin_memory()
    fctx.buildmips_cube_float(fmt, w, w, levels, pinned, samples)
    assert np.array_equal(pinned.numpy().view(np.uint8), want.view(np.uint8))


def test_bad_input_is_rejected_before_any_launch(fctx):
    w, levels = 16, 3
    n = level_offsets(w, w, levels)[-1]
    launches = fctx.launch_count

    with pytest.raises(ValueError):      # wrong dtype
        fctx.buildmips_cube_float(F16, w, w, levels, np.zeros((n, 4), np.float32))
    with pytest.raises(ValueError):
        fctx.buildmips_cube_float_device(F32, w, w, levels, torch.zeros((n, 4), dtype=torch.float16, device=DEV))
    with pytest.raises(ValueError):      # unknown format
        fctx.buildmips_cube_float(5, w, w, levels, np.zeros((n, 4), np.float32))
    with pytest.raises(ValueError):      # too small
        fctx.buildmips_cube_float(F32, w, w, levels, np.zeros((n - 1, 4), np.float32))
    with pytest.raises(ValueError):      # not on the context's device
        fctx.buildmips_cube_float_device(F32, w, w, levels, torch.zeros((n, 4), dtype=torch.float32))
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            fctx.buildmips_cube_float_device(F32, w, w, levels, torch.zeros((n, 4), dtype=torch.float32, device="cuda:1"))

    # the C ABI's own checks: unknown format, misaligned pointer, rows outside the level, a chain valid_chain rejects
    lib, h = fctx._lib, fctx._handle
    d = torch.zeros((n, 4), dtype=torch.float32, device=DEV)
    p = d.data_ptr()
    assert lib.datum_ibl_buildmips_cube_float_device(h, 3, w, w, levels, 64, ctypes.c_void_p(p), None) != 0
    assert b"format" in lib.datum_ibl_last_error()
    assert lib.datum_ibl_buildmips_cube_float_device(h, F32, w, w, levels, 64, ctypes.c_void_p(p + 8), None) != 0
    assert b"misaligned" in lib.datum_ibl_last_error()
    assert lib.datum_ibl_buildmips_cube_float_device(h, F16, w, w, levels, 64, ctypes.c_void_p(p + 4), None) != 0
    assert lib.datum_ibl_buildmips_cube_float_device(h, F32, w, w, 6, 64, ctypes.c_void_p(p), None) != 0
    assert lib.datum_ibl_prefilter_level_float_device(h, F32, ctypes.c_void_p(p), w, w, 1, levels, 64, 0, 6 * (w >> 1) + 1, ctypes.c_void_p(p), None) != 0
    assert b"row range" in lib.datum_ibl_last_error()
    assert lib.datum_ibl_prefilter_level_float_device(h, F32, None, w, w, 1, levels, 64, 0, 1, ctypes.c_void_p(p), None) != 0

    torch.cuda.synchronize()
    assert fctx.launch_count == launches


def test_sh9_of_an_f16_cube(fctx):
    w = 64
    cube16 = synth.synthetic_cube(w, w, probe=5, noise=True, sun=True).astype(np.float16)
    widened = cube16.astype(np.float32)
    got = fctx.project_sh9(cube16, F16, w, w)
    want = oracle_lib.project_sh9(widened, F32, w, w)
    assert np.abs(got.astype(np.float64) - want).max() <= 1e-4 * np.abs(want).max()
    # the arithmetic after the load is the F32 path's
    assert np.array_equal(got, fctx.project_sh9(widened, F32, w, w))
