"""Batched float bakes (datum_ibl_bake_probes_float): every chain of a batch ends with the bytes of a single
datum_ibl_buildmips_cube_float call on the same level 0, and the batch's SH9 equals project_sh9 of that level 0."""

import ctypes

import numpy as np
import pytest
import torch

import datum_b200
from datum_b200 import synth

pytestmark = pytest.mark.gpu

F32, F16 = datum_b200.FORMAT_F32, datum_b200.FORMAT_F16
NP_DTYPE = {F32: np.float32, F16: np.float16}


@pytest.fixture(scope="module")
def ctx():
    c = datum_b200.IblContext(0)
    yield c
    c.close()


def float_chain(fmt, w, levels, probe, sun=True):
    """(texels, 4) host chain of the format, level 0 from synth.synthetic_cube, the other levels zero."""
    chain = np.zeros((datum_b200.level_offsets(w, w, levels)[-1], 4), NP_DTYPE[fmt])
    chain[: 6 * w * w] = synth.synthetic_cube(w, w, probe=probe, sun=sun).reshape(-1, 4).astype(NP_DTYPE[fmt])
    return chain


def single_calls(ctx, fmt, w, levels, samples, probes):
    out = []
    for p in probes:
        chain = float_chain(fmt, w, levels, p)
        ctx.buildmips_cube_float(fmt, w, w, levels, chain, samples)
        out.append(chain)
    return out


def host_bytes(chain):
    return (chain.numpy() if isinstance(chain, torch.Tensor) else chain).view(np.uint8)


def check_batch(ctx, fmt, w, levels, samples, probes, pinned=False, sh9=True, bake=None):
    want = single_calls(ctx, fmt, w, levels, samples, probes)
    chains = [float_chain(fmt, w, levels, p) for p in probes]
    if pinned:
        chains = [torch.from_numpy(c).pin_memory() for c in chains]
    sh = (bake or ctx.bake_probes_float)(fmt, w, w, levels, chains, samples, sh9=sh9)
    for i, (got, ref) in enumerate(zip(chains, want)):
        assert np.array_equal(host_bytes(got), ref.view(np.uint8)), "probe %d" % i
    if sh9:
        assert sh.shape == (len(probes), 9, 3)
        for i, ref in enumerate(want):
            level0 = np.ascontiguousarray(ref[: 6 * w * w])
            assert np.array_equal(sh[i], ctx.project_sh9(level0, fmt, w, w)), "probe %d" % i
    else:
        assert sh is None
    return want


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("count", [1, 2, 5])
@pytest.mark.parametrize("pinned", [False, True])
def test_float_batch_equals_single_calls(ctx, fmt, count, pinned):
    check_batch(ctx, fmt, 64, 6, 256, list(range(40, 40 + count)), pinned=pinned)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_a_group_of_sixteen_and_a_short_group(ctx, fmt):
    """19 probes of 64^2: one launch per level for 16 of them, then a short group."""
    check_batch(ctx, fmt, 64, 7, 128, list(range(200, 219)), pinned=True)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_a_batch_with_quarter_groups_at_both_ends(ctx, fmt):
    """26 probes of 32^2 down to 1x1 faces: long enough for the short groups at the start and the end."""
    check_batch(ctx, fmt, 32, 6, 64, list(range(300, 326)), pinned=True)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_float_batch_at_the_c4_probe_size(ctx, fmt):
    """BASELINE config 4's unit (256^2 faces, 8 levels, 1024 spp), three probes: the queued 8-warp pair kernel
    (levels 1 and 2), and the tail kernel (levels 3 to 7)."""
    w, levels, samples = 256, 8, 1024
    want = check_batch(ctx, fmt, w, levels, samples, [3, 4, 5], pinned=True, sh9=False)
    # a single call AFTER the batch: the batch's launch shapes must not change the single call's
    again = single_calls(ctx, fmt, w, levels, samples, [3])
    assert np.array_equal(again[0].view(np.uint8), want[0].view(np.uint8))


@pytest.mark.parametrize("fmt", [F32, F16])
def test_probes_with_an_odd_source_level(ctx, fmt):
    """50^2 x 3: level 2 reads a 25^2 source the pair kernel cannot address, so every probe runs alone."""
    check_batch(ctx, fmt, 50, 3, 256, [7, 8, 9])


def test_probes_too_big_to_share_a_launch(ctx):
    """1024^2 probes fill the machine alone (a group of one)."""
    check_batch(ctx, F16, 1024, 4, 64, [1, 2], pinned=True)


def test_rgbe_and_float_batches_share_one_context(ctx):
    """The rgbe and the float batch share the device payloads and the streams of the context."""
    w, levels, samples = 64, 6, 256
    probes = [60, 61, 62]

    def rgbe_batch():
        want = []
        for p in probes:
            bits = synth.synthetic_chain(w, w, levels, probe=p)
            ctx.image_buildmips_cube_ibl(w, w, levels, bits, samples)
            want.append(bits)
        payloads = [synth.synthetic_chain(w, w, levels, probe=p) for p in probes]
        ctx.bake_probes(w, w, levels, payloads, samples)
        for got, ref in zip(payloads, want):
            assert np.array_equal(got, ref)

    rgbe_batch()
    check_batch(ctx, F16, w, levels, samples, probes)
    rgbe_batch()


@pytest.mark.parametrize("devices", [
    [0, 0],
    pytest.param([0, 1], marks=pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")),
])
def test_device_list_bakes_float_batches(ctx, devices):
    with datum_b200.MultiContext(devices) as multi:
        check_batch(ctx, F32, 64, 6, 256, [70, 71, 72, 73, 74], bake=multi.bake_probes_float)
        check_batch(ctx, F16, 64, 6, 256, [75, 76, 77], pinned=True, bake=multi.bake_probes_float)


def test_bad_input_is_rejected_before_any_launch(ctx):
    w, levels = 16, 3
    n = datum_b200.level_offsets(w, w, levels)[-1]
    launches = ctx.launch_count

    assert ctx.bake_probes_float(F32, w, w, levels, [], 64) is None           # empty batch
    assert ctx.bake_probes_float(F32, w, w, levels, [], 64, sh9=True).shape == (0, 9, 3)
    with pytest.raises(ValueError):      # wrong dtype
        ctx.bake_probes_float(F16, w, w, levels, [np.zeros((n, 4), np.float16), np.zeros((n, 4), np.float32)], 64)
    with pytest.raises(ValueError):
        ctx.bake_probes_float(F32, w, w, levels, [torch.zeros((n, 4), dtype=torch.float16)], 64)
    with pytest.raises(ValueError):      # too small
        ctx.bake_probes_float(F32, w, w, levels, [np.zeros((n - 1, 4), np.float32)], 64)
    with pytest.raises(ValueError):      # unknown format
        ctx.bake_probes_float(5, w, w, levels, [np.zeros((n, 4), np.float32)], 64)
    with pytest.raises(datum_b200.IblError):      # samples outside 1..4096
        ctx.bake_probes_float(F32, w, w, levels, [np.zeros((n, 4), np.float32)], 0)
    with pytest.raises(datum_b200.IblError):
        ctx.bake_probes_float(F32, w, w, levels, [np.zeros((n, 4), np.float32)], 4097)
    deep = datum_b200.level_offsets(w, w, 6)[-1]
    with pytest.raises(datum_b200.IblError):      # 16 >> 5 == 0
        ctx.bake_probes_float(F32, w, w, 6, [np.zeros((deep, 4), np.float32)], 64)

    # the C ABI's own checks
    lib, h = ctx._lib, ctx._handle
    chain = np.zeros((n, 4), np.float32)
    ok = (ctypes.c_void_p * 2)(chain.ctypes.data, chain.ctypes.data)
    assert lib.datum_ibl_bake_probes_float(h, 3, 1, w, w, levels, 64, ok, None) != 0
    assert b"format" in lib.datum_ibl_last_error()
    assert lib.datum_ibl_bake_probes_float(h, F32, -1, w, w, levels, 64, ok, None) != 0
    with_null = (ctypes.c_void_p * 2)(chain.ctypes.data, None)
    assert lib.datum_ibl_bake_probes_float(h, F32, 2, w, w, levels, 64, with_null, None) != 0
    assert b"null payload" in lib.datum_ibl_last_error()
    assert lib.datum_ibl_bake_probes_float(h, F32, 1, w, w, levels, 64, None, None) != 0

    torch.cuda.synchronize()
    assert ctx.launch_count == launches
