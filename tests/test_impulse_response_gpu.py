"""Every prefilter kernel path against the oracle on single-texel impulse sources (tests/impulse.py).

On noise or smooth sources one dropped, doubled or misplaced sample moves a texel by about 1e-3 of its value,
the size of the parity tolerance.  With level 0 zero except for one texel per channel it moves a texel by up to a
whole unit u = I / W, while the kernels agree with the oracle to 1e-3 u.  Every case reuses a launch (source size,
level, levels, samples, row range, variant) that another test of the suite runs on noise; the cases at the ends
of the input range change only the impulse's value."""

import numpy as np
import pytest
import torch

import datum_b200
import impulse
import oracle_lib

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F32, F16 = datum_b200.FORMAT_F32, datum_b200.FORMAT_F16
NP_DTYPE = {F32: np.float32, F16: np.float16}
TORCH_DTYPE = {F32: torch.float32, F16: torch.float16}
I = 1000.0


def rgbe_level(ctx, src, ws, hs, level, levels, samples, rows=None):
    """(words, fp32 rgb) of one level through prefilter_level_device, rows [a, b) (default: all)."""
    n = 6 * (ws >> 1) * (hs >> 1)
    a, b = rows or (0, 6 * (hs >> 1))
    d_src = torch.from_numpy(src.view(np.int32)).to(DEV)
    words = torch.zeros(n, dtype=torch.int32, device=DEV)
    f32 = torch.zeros(n * 3, dtype=torch.float32, device=DEV)
    ctx.prefilter_level_device(d_src, ws, hs, level, levels, samples, a, b, words, f32)
    ctx.synchronize()
    return words.cpu().numpy().view(np.uint32), f32.cpu().numpy().reshape(-1, 3)


def float_level(ctx, fmt, src, ws, hs, level, levels, samples):
    """(fp32 rgb, stored texels) of one level through prefilter_level_float_device."""
    n = 6 * (ws >> 1) * (hs >> 1)
    d_dst = torch.zeros((n, 4), dtype=TORCH_DTYPE[fmt], device=DEV)
    d_f32 = torch.zeros((n, 3), dtype=torch.float32, device=DEV)
    ctx.prefilter_level_float_device(fmt, torch.from_numpy(src).to(DEV), ws, hs, level, levels, samples, 0, 6 * (hs >> 1), d_dst, d_f32)
    ctx.synchronize()
    return d_f32.cpu().numpy(), d_dst.cpu().numpy()


def check_rgbe(ctx, ws, hs, level, levels, samples, spots, rows=None, value=I):
    src, radiance = impulse.rgbe_source(ws, hs, spots, value)
    words, got = rgbe_level(ctx, src, ws, hs, level, levels, samples, rows)
    runs = [rows or (0, 6 * (hs >> 1))]
    want = impulse.oracle_rows(False, src, ws, hs, level, levels, samples, runs)
    report = impulse.check(got, want, radiance, ws, hs, level, levels, samples, runs=runs, got_words=words)
    print(report)
    return report, got


def check_float(ctx, fmt, ws, level, levels, samples, spots, value=I):
    src, radiance = impulse.float_source(ws, ws, spots, value, NP_DTYPE[fmt])
    got, stored = float_level(ctx, fmt, src, ws, ws, level, levels, samples)
    if fmt == F32:
        assert np.array_equal(stored[:, :3], got) and np.all(stored[:, 3] == 1.0)
    want = impulse.oracle_rows(True, src, ws, ws, level, levels, samples, [(0, 6 * (ws >> 1))])
    report = impulse.check(got, want, radiance, ws, ws, level, levels, samples, got_f16=stored if fmt == F16 else None)
    print(report)
    return report, got, stored


def lobe_runs(ws, spots, level, levels, samples, block=16, period=384):
    """(oracle row runs, rows that must stay zero) of a big level.  Inside the lobes (impulse.lobe_rows) the oracle
    runs on blocks of `block` rows every `period` rows and on the block around each impulse's own destination row:
    at 2048^2 level 1/12 a lobe reaches 56 degrees, 2000 to 4000 of the 6144 rows, which would take the oracle
    minutes.  Every row outside the lobes must stay zero."""
    hd = ws >> 1
    lobes = impulse.lobe_rows(ws, ws, spots, level, levels, samples)
    pick = np.arange(6 * hd) % period < block
    for face, y, _ in spots:
        row = face * hd + y // 2
        pick[max(0, row - block // 2):row + block // 2] = True
    return impulse.row_runs(lobes & pick), ~lobes


# ---- rgbe chain: prefilter_level_device with d_dst_f32 ------------------------------------------------------

@pytest.mark.parametrize("ws,hs,level,levels,samples,spots", [
    # tail kernel (test_every_level_matches_the_oracle_on_the_same_source, 16^2 x 5 at 16 spp; 24x12 x 3)
    pytest.param(16, 16, 4, 5, 16, [(3, 7, 7), (2, 0, 9), (1, 15, 0)], id="tail-16"),
    pytest.param(24, 12, 1, 3, 1024, [(0, 5, 11), (4, 0, 7), (2, 11, 23)], id="tail-24x12"),
    # pair kernel, 4 warps, tile queues (BASELINE config 2 level 1)
    pytest.param(512, 512, 1, 8, 1024, [(1, 200, 300), (3, 0, 123), (5, 511, 0)], id="pair4-512"),
    # pair kernel, 8 warps (BASELINE config 2 level 2)
    pytest.param(256, 256, 2, 8, 1024, [(2, 100, 77), (0, 255, 40), (4, 0, 255)], id="pair8-256"),
])
def test_rgbe_level_answers_an_impulse_like_the_oracle(ctx, ws, hs, level, levels, samples, spots):
    check_rgbe(ctx, ws, hs, level, levels, samples, spots)


@pytest.mark.parametrize("ws", [1371, 1370])
def test_rgbe_one_sample_handover_answers_an_impulse(ctx, ws):
    """test_pair_kernel_hands_over_when_its_fp32_index_does_not_apply: rows (0, 16) of level 1/3 at 8 spp; 1371
    runs the one-sample kernel, 1370 the pair kernel.  At 8 spp few source texels are read by those rows (the top
    rows of face 0); the impulses sit on texels they read: inside face 0, on its last column, and on the last column
    of face 4 (oracle responses of 0.83 u, 0.14 u and 0.9 u).  No face corner is read there."""
    spots = [(0, 21, 601), (0, 1, ws - 1), (4, 1, ws - 1)]
    report, got = check_rgbe(ctx, ws, ws, 1, 3, 8, spots, rows=(0, 16))
    assert np.all(got.max(axis=0) > 0.1 * impulse.units([I] * 3, 1, 3, 8))


def test_rgbe_config_3_level_1_answers_an_impulse_on_the_lobe_rows(ctx):
    """test_baseline_config_3_level_1_against_the_oracle_on_spot_rows: 2048^2 -> 1024^2 at 4096 spp, the 4096-entry
    table read through L1."""
    ws, level, levels, samples = 2048, 1, 12, 4096
    spots = [(4, 1000, 1030), (3, 2047, 512), (0, 0, 2047)]
    src, radiance = impulse.rgbe_source(ws, ws, spots, I)
    words, got = rgbe_level(ctx, src, ws, ws, level, levels, samples)
    runs, zero = lobe_runs(ws, spots, level, levels, samples)
    want = impulse.oracle_rows(False, src, ws, ws, level, levels, samples, runs)
    print(impulse.check(got, want, radiance, ws, ws, level, levels, samples, runs=runs, got_words=words, zero_rows=zero))


VARIANT_SPOTS = {64: [(0, 31, 31), (1, 0, 17), (2, 63, 63)], 32: [(5, 10, 5), (3, 16, 0), (4, 0, 31)]}


@pytest.mark.parametrize("variant", [0, 51, 52, 53, 54, 66, 67, 70, 71, 72, 73, 80])
@pytest.mark.parametrize("ws,level", [(64, 1), (32, 2)])
def test_every_kernel_variant_answers_an_impulse_like_the_oracle(ctx, variant, ws, level):
    """The shapes of test_kernel_variants_agree (64^2 x 6 levels, 1024 spp), each against the oracle."""
    ctx.set_prefilter_variant(variant)
    try:
        check_rgbe(ctx, ws, ws, level, 6, 1024, VARIANT_SPOTS[ws])
    finally:
        ctx.set_prefilter_variant(0)


def test_row_slabs_answer_an_impulse_like_the_oracle(ctx):
    """The cuts of test_row_slabs_reproduce_the_full_level (64^2 -> 32^2, level 2/7): every slab alone against the
    oracle on its rows, nothing written outside them.  The face-1 impulse sits at destination row 50, a cut; the
    responses of all three cross several cuts."""
    ws, level, levels, samples = 64, 2, 7, 1024
    wd = ws >> 1
    spots = [(1, 36, 20), (3, 0, 30), (0, 0, 63)]
    src, radiance = impulse.rgbe_source(ws, ws, spots, I)
    cuts = [0, 7, 8, 50, 97, 6 * wd]
    for a, b in zip(cuts[:-1], cuts[1:]):
        words, got = rgbe_level(ctx, src, ws, ws, level, levels, samples, (a, b))
        want = impulse.oracle_rows(False, src, ws, ws, level, levels, samples, [(a, b)])
        outside = np.ones(6 * wd, bool)
        outside[a:b] = False
        assert not words.reshape(6 * wd, wd)[outside].any() and not got.reshape(6 * wd, wd, 3)[outside].any()
        print((a, b), impulse.check(got, want, radiance, ws, ws, level, levels, samples, runs=[(a, b)], got_words=words))


BATCH_SPOTS = [
    [(0, 128, 128), (2, 0, 64), (5, 255, 255)],
    [(1, 60, 190), (4, 255, 100), (3, 0, 0)],
    [(5, 128, 30), (0, 77, 0), (2, 255, 0)],
]


def test_rgbe_batch_answers_each_probes_impulses(ctx):
    """test_a_config_4_probe_through_the_batch_entry_against_the_oracle: three probes of 256^2 x 8 levels through
    bake_probes, with impulses at different texels.  Level 1 of each probe against the oracle on its own level 0:
    a response of another probe would be a unit off."""
    w, levels, samples = 256, 8, 1024
    offs = datum_b200.level_offsets(w, w, levels)
    payloads, radiance = [], []
    for spots in BATCH_SPOTS:
        bits = np.zeros(offs[-1], np.uint32)
        bits[: offs[1]], rad = impulse.rgbe_source(w, w, spots, I)
        payloads.append(bits)
        radiance.append(rad)
    ctx.bake_probes(w, w, levels, payloads, samples)
    for bits, rad in zip(payloads, radiance):
        _, want = oracle_lib.prefilter_level(bits[: offs[1]], w, w, 1, levels, samples)
        print(impulse.check(None, want, rad, w, w, 1, levels, samples, got_words=bits[offs[1]:offs[2]]))


def test_rgbe_impulse_at_the_largest_rgbe_value(ctx):
    """Words with the largest exponent and mantissa (test_every_level_matches_the_oracle_on_the_same_source, 64^2 x
    7 levels): every result finite and within the criterion."""
    ws, level, levels, samples = 64, 1, 7, 1024
    spots = [(4, 31, 31), (0, 0, 10), (3, 63, 63)]
    src = np.zeros(6 * ws * ws, np.uint32)
    for c, spot in enumerate(spots):
        src[impulse.texel_index(ws, ws, spot)] = np.uint32(0xF8000000) | np.uint32(0x1FF << (9 * c))
    decoded = oracle_lib.rgbe_decode_array(src)[:, :3]
    radiance = [float(decoded[impulse.texel_index(ws, ws, spot), c]) for c, spot in enumerate(spots)]
    assert np.isfinite(radiance).all() and min(radiance) >= 65408.0
    words, got = rgbe_level(ctx, src, ws, ws, level, levels, samples)
    _, want = oracle_lib.prefilter_level(src, ws, ws, level, levels, samples)
    print(impulse.check(got, want, radiance, ws, ws, level, levels, samples, got_words=words))


# ---- float chains: prefilter_level_float_device, F32 and F16 -------------------------------------------------

@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("ws,level,levels,samples,spots", [
    # tail kernel (test_every_float_level_matches_the_float_oracle_on_the_same_source, 16^2 x 5 at 16 spp)
    pytest.param(16, 4, 5, 16, [(2, 8, 8), (5, 15, 3), (0, 0, 0)], id="tail-16"),
    # pair kernel, 4 and 8 warps (test_baseline_config_2_float_chain_on_spot_rows, levels 1 and 2)
    pytest.param(512, 1, 8, 1024, [(4, 300, 200), (1, 511, 100), (2, 0, 511)], id="pair4-512"),
    pytest.param(256, 2, 8, 1024, [(3, 128, 60), (5, 0, 200), (1, 255, 255)], id="pair8-256"),
    # odd source at pair-kernel slab sizes (test_odd_source_at_pair_kernel_slab_sizes)
    pytest.param(101, 1, 2, 1024, [(0, 50, 50), (4, 100, 33), (3, 0, 100)], id="odd-101"),
])
def test_float_level_answers_an_impulse_like_the_float_oracle(ctx, fmt, ws, level, levels, samples, spots):
    check_float(ctx, fmt, ws, level, levels, samples, spots)


def test_f16_config_3_level_1_answers_an_impulse_on_the_lobe_rows(ctx):
    """test_baseline_config_3_level_1_in_f16_on_spot_rows: 2048^2 -> 1024^2 at 4096 spp in F16."""
    ws, level, levels, samples = 2048, 1, 12, 4096
    spots = [(1, 900, 1100), (5, 0, 700), (2, 2047, 2047)]
    src, radiance = impulse.float_source(ws, ws, spots, I, np.float16)
    got, stored = float_level(ctx, F16, src, ws, ws, level, levels, samples)
    runs, zero = lobe_runs(ws, spots, level, levels, samples)
    want = impulse.oracle_rows(True, src, ws, ws, level, levels, samples, runs)
    print(impulse.check(got, want, radiance, ws, ws, level, levels, samples, runs=runs, got_f16=stored, zero_rows=zero))


@pytest.mark.parametrize("fmt", [F32, F16])
def test_float_batch_answers_each_probes_impulses(ctx, fmt):
    """test_float_batch_at_the_c4_probe_size: three probes of 256^2 x 8 levels through bake_probes_float, level 1 of
    each against the float oracle on its own level 0."""
    w, levels, samples = 256, 8, 1024
    offs = datum_b200.level_offsets(w, w, levels)
    chains, radiance = [], []
    for spots in BATCH_SPOTS:
        chain = np.zeros((offs[-1], 4), NP_DTYPE[fmt])
        chain[: offs[1]], rad = impulse.float_source(w, w, spots, I, NP_DTYPE[fmt])
        chains.append(chain)
        radiance.append(rad)
    ctx.bake_probes_float(fmt, w, w, levels, chains, samples)
    for chain, rad in zip(chains, radiance):
        want = impulse.oracle_rows(True, chain[: offs[1]], w, w, 1, levels, samples, [(0, 6 * (w >> 1))])
        out = chain[offs[1]:offs[2]]
        assert np.all(out[:, 3] == 1.0)
        print(impulse.check(out[:, :3] if fmt == F32 else None, want, rad, w, w, 1, levels, samples, got_f16=out if fmt == F16 else None))


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("ws", [128, 101, 32])
def test_float_peers_world_of_one_answers_an_impulse(ctx, fmt, ws):
    """test_world_of_one_equals_the_device_entry: prefilter_level_float_peers, world 1, level 1/4 at 256 spp."""
    levels, samples = 4, 256
    spots = [(3, ws // 2, ws // 3), (0, ws - 1, ws // 2), (4, 0, ws - 1)]
    src, radiance = impulse.float_source(ws, ws, spots, I, NP_DTYPE[fmt])
    d_src = torch.from_numpy(src).to(DEV)
    n = 6 * (ws >> 1) ** 2
    got = torch.full((n, 4), 7.0, dtype=TORCH_DTYPE[fmt], device=DEV)
    torch.cuda.synchronize()
    ctx.prefilter_level_float_peers(fmt, d_src.data_ptr(), ws, ws, 1, levels, samples, 0, 6 * (ws >> 1), 0, 1, [got.data_ptr()])
    ctx.synchronize()
    out = got.cpu().numpy()
    want = impulse.oracle_rows(True, src, ws, ws, 1, levels, samples, [(0, 6 * (ws >> 1))])
    assert np.all(out[:, 3] == 1.0)
    print(impulse.check(out[:, :3] if fmt == F32 else None, want, radiance, ws, ws, 1, levels, samples, got_f16=out if fmt == F16 else None))


# ---- the ends of the input range ------------------------------------------------------------------------------

def test_f16_impulse_of_65504(ctx):
    """The largest binary16 value on the pair kernel (128^2 -> 64^2, level 1/8): no stored value inf or above
    65504."""
    check_float(ctx, F16, 128, 1, 8, 1024, [(0, 64, 64), (2, 127, 5), (5, 0, 127)], value=65504.0)


def test_f16_impulse_with_a_subnormal_tail(ctx):
    """I = 2^-10 on the tail kernel (64^2 -> 32^2, level 1/7): u is about 1e-6, so most of the response is stored
    as binary16 subnormals (below 2^-14), rounded on the device like float_parity.round_f16."""
    _, _, stored = check_float(ctx, F16, 64, 1, 7, 1024, [(1, 20, 40), (3, 63, 10), (4, 0, 0)], value=2.0 ** -10)
    rgb = stored[:, :3].astype(np.float32)
    assert np.count_nonzero((rgb > 0) & (rgb < 2.0 ** -14)) > 100


def test_f32_impulse_just_below_the_float_chain_limit(ctx):
    """The largest float32 below kFloatChainMaxRadiance (2^52, prefilter_f.h) at 4096 spp (test_every_float_level_...,
    64^2 x 4 levels)."""
    value = float(np.nextafter(np.float32(2.0 ** 52), np.float32(0)))
    _, got, _ = check_float(ctx, F32, 64, 1, 4, 4096, [(5, 31, 31), (2, 0, 31), (1, 63, 0)], value=value)
    assert np.all(np.isfinite(got)) and got.max() > 1e-3 * value     # the largest response is 26 u, 0.6 % of I
