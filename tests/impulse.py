"""Impulse sources and the impulse-response criterion of the prefilter levels (TEST INFRASTRUCTURE).

Level 0 is zero except for up to three texels, one per channel, of radiance I.  Every destination texel of the
next level is then a sum of the weights of the samples whose bilinear footprint touches such a texel, times
I / W, where W is the total NdotL weight of a texel's samples.  One sample dropped, doubled, fetched from the
wrong texel, face or probe, or put in the wrong channel moves a texel by up to a whole unit u = I / W, while
the kernels agree with the oracle to a small fraction of u (on the CPU emulation of the kernels: 2.9e-4 u at
64^2 -> 32^2 level 1/8, 2.1e-5 u at 32^2 -> 16^2 level 2/6, 2.1e-6 u at 16^2 -> 8^2 level 4/5 at 16 spp).

Criterion, per channel c with u_c = I_c / W:
  clean texels   |got - want| <= FLOOR * u_c + REL * |want|;
  edge texels    (samples within 2e-6 of a cube-face boundary, oracle_lib.edge_ambiguous_counts) the looser
                 rule of parity.py: the weight share of those samples times the brightest impulse, plus 1e-3 of
                 the texel's largest channel;
  RGBA16F        every stored half of a clean texel within 1 ulp of float_parity.round_f16(want), or the binary16
                 rounding of a value within the fp32 rule above; alpha 1.0;
  rgbe words     the decoded value under the fp32 rule, widened by one mantissa code of the word's exponent.
Big levels are compared on rows inside the impulses' lobes (lobe_rows); every texel outside them must stay zero.
"""

import numpy as np

import float_oracle_lib
import float_parity
import oracle_lib
import parity
from datum_b200 import synth

FLOOR = 1e-3       # absolute floor, in units u
REL = 2e-5         # of the oracle's value: fp32 sums of up to 4096 samples associated differently


def texel_index(ws, hs, spot):
    face, y, x = spot
    return (face * hs + y) * ws + x


def impulse_rgb(ws, hs, spots, value):
    """(6*hs*ws, 3) float32: zero, except channel c of texel spots[c] = (face, y, x), which is `value`."""
    rgb = np.zeros((6 * hs * ws, 3), np.float32)
    for c, spot in enumerate(spots):
        rgb[texel_index(ws, hs, spot), c] = value
    return rgb


def rgbe_source(ws, hs, spots, value):
    """rgbe level 0 of impulse_rgb (word 0 elsewhere) and the decoded radiance of each impulse."""
    words = oracle_lib.rgbe_encode_array(impulse_rgb(ws, hs, spots, value))
    decoded = oracle_lib.rgbe_decode_array(words)
    return words, [float(decoded[texel_index(ws, hs, spot), c]) for c, spot in enumerate(spots)]


def float_source(ws, hs, spots, value, dtype):
    """(texels, 4) level 0 of the dtype (alpha 1.0) and the stored radiance of each impulse."""
    src = np.zeros((6 * hs * ws, 4), dtype)
    src[:, :3] = impulse_rgb(ws, hs, spots, value).astype(dtype)
    src[:, 3] = 1.0
    return src, [float(src[texel_index(ws, hs, spot), c]) for c, spot in enumerate(spots)]


def units(radiance, level, levels, samples):
    """u_c = I_c / W for each channel (channels without an impulse get the unit of the first)."""
    weight = parity.total_sample_weight(level, levels, samples)
    u = [r / weight for r in radiance]
    return np.array(u + [u[0]] * (3 - len(u)), np.float64)


def max_sample_angle(level, levels, samples):
    """The largest angle between a texel's direction and one of its accepted sample directions (radians)."""
    n = np.array([0.0, 0.0, -1.0], np.float32)
    dirs = np.zeros((samples, 3), np.float32)
    ndotl = np.zeros(samples, np.float32)
    roughness = np.float32(level) / np.float32(levels - 1)
    oracle_lib.oracle().oracle_trace_samples(float(roughness), samples, n.ctypes.data, dirs.ctypes.data, ndotl.ctypes.data)
    cos = -dirs[ndotl > 0, 2].astype(np.float64) / np.linalg.norm(dirs[ndotl > 0].astype(np.float64), axis=1)
    return float(np.arccos(np.clip(cos.min(), -1.0, 1.0)))


def lobe_rows(ws, hs, spots, level, levels, samples, margin_texels=2):
    """Destination rows (bool, 6*hs/2) holding a texel whose direction lies within the largest sample angle plus
    `margin_texels` source texels (2/ws radians each, their largest angular size) of an impulse.  Outside these
    rows no sample of any texel can reach an impulse's bilinear footprint."""
    wd, hd = ws >> 1, hs >> 1
    limit = np.cos(min(np.pi, max_sample_angle(level, levels, samples) + margin_texels * 2.0 / min(ws, hs)))
    dst = synth.cube_directions(wd, hd, dtype=np.float32).reshape(6 * hd, wd, 3)
    rows = np.zeros(6 * hd, bool)
    for face, y, x in spots:
        d = np.zeros(3, np.float32)
        oracle_lib.oracle().oracle_texel_direction(face, x, y, ws, hs, d.ctypes.data)
        rows |= ((dst @ d) >= limit).any(axis=1)
    return rows


def row_runs(rows):
    """[(begin, end)] of the runs of True in a bool row mask."""
    edges = np.flatnonzero(np.diff(np.concatenate([[0], rows.astype(np.int8), [0]])))
    return list(zip(edges[0::2].tolist(), edges[1::2].tolist()))


def oracle_rows(fmt_float, src, ws, hs, level, levels, samples, runs):
    """fp32 rgb of the oracle on the given row runs of the level (rows outside them stay 0).  fmt_float: False for
    an rgbe source (oracle_lib), True for a float source (float_oracle_lib)."""
    want = np.zeros((6 * (ws >> 1) * (hs >> 1), 3), np.float32)
    if fmt_float:
        src = float_parity.widen(src)
    for a, b in runs:
        if fmt_float:
            part = float_oracle_lib.prefilter_level_rgba32f(src, ws, hs, level, levels, samples, a, b)
        else:
            part = oracle_lib.prefilter_level(src, ws, hs, level, levels, samples, a, b)[1]
        sl = slice(a * (ws >> 1), b * (ws >> 1))
        want[sl] = part[sl]
    return want


def check(got_f32, want_f32, radiance, ws, hs, level, levels, samples, runs=None, got_f16=None, got_words=None, zero_rows=None):
    """Impulse-response criterion of one level on the texels of the row runs (default: the whole level).
    got_f32: (texels, 3) fp32 values of the kernel (or None when only stored texels are at hand); want_f32: the
    oracle's, valid on the runs; radiance: the impulses' I_c.  got_f16: stored RGBA16F texels.  got_words: stored
    rgbe words, held to the criterion plus one mantissa code of their shared exponent.  zero_rows: bool mask of
    the rows whose texels must all be <= FLOOR * u_c.  Returns the measured figures (errors in units u); raises
    AssertionError."""
    wd, hd = ws >> 1, hs >> 1
    runs = runs or [(0, 6 * hd)]
    u = units(radiance, level, levels, samples)
    weight = parity.total_sample_weight(level, levels, samples)
    brightest = max(radiance)
    sel = np.zeros(6 * hd * wd, bool)
    edge_counts = np.zeros(6 * hd * wd, np.int32)
    for a, b in runs:
        sel[a * wd:b * wd] = True
        edge_counts += oracle_lib.edge_ambiguous_counts(wd, hd, level, levels, samples, row_begin=a, row_end=b)
    edge = edge_counts[sel] > 0
    clean = ~edge
    want = np.asarray(want_f32, np.float64).reshape(-1, 3)[sel]
    report = {"texels": int(sel.sum()), "edge_fraction": float(edge.mean()), "max_response_u": float((want / u).max())}

    zero = np.repeat(zero_rows, wd) if zero_rows is not None else np.zeros(6 * hd * wd, bool)

    def assert_close(got, what, clean_rule=True, quantum=0.0):
        err = np.abs(got - want)
        report[what + "_max_clean_u"] = float((err[clean] / u).max()) if clean.any() else 0.0
        if clean_rule:
            bad = clean[:, None] & (err > FLOOR * u + REL * np.abs(want) + quantum)
            assert not bad.any(), (what, report, np.argwhere(bad)[:5].tolist())
        if edge.any():
            share = edge_counts[sel][edge] / weight
            allowed = share * brightest + parity.TOL_F32 * want[edge].max(axis=1)
            assert np.all(err[edge].max(axis=1) <= allowed), (what, report)

    if got_f32 is not None:
        got32 = np.asarray(got_f32, np.float64).reshape(-1, 3)
        assert np.all(np.isfinite(got32)), "non-finite fp32 result"
        assert_close(got32[sel], "f32")
        if zero.any():
            outside = np.abs(got32[zero])
            report["zero_rows_max_u"] = float((outside / u).max())
            assert np.all(outside <= FLOOR * u), report
    if got_words is not None:
        words = np.asarray(got_words, np.uint32).reshape(-1)
        decoded = oracle_lib.rgbe_decode_array(words)[:, :3].astype(np.float64)
        assert np.all(np.isfinite(decoded)), "non-finite rgbe word"
        code = oracle_lib.rgbe_decode_array((words & np.uint32(0xF8000000)) | np.uint32(1))[:, :1].astype(np.float64)
        assert_close(decoded[sel], "words", quantum=code[sel])
        if zero.any():
            assert np.all(decoded[zero] <= FLOOR * u), report
    if got_f16 is not None:
        got16 = np.asarray(got_f16, np.float16).reshape(-1, 4)
        assert np.all(np.isfinite(got16.astype(np.float32))) and np.all(got16[:, :3] <= np.float16(65504.0)), "RGBA16F overflow"
        assert np.all(got16[:, 3] == np.float16(1.0)), "output alpha must be 1.0"
        if got_f32 is not None:      # the stored half is the fp32 result rounded as documented
            assert np.array_equal(got16[:, :3].view(np.uint16), float_parity.round_f16(np.asarray(got_f32, np.float32).reshape(-1, 3)).view(np.uint16))
        half = got16[sel][clean][:, :3]
        ulps = np.abs(half.view(np.uint16).astype(np.int64) - float_parity.round_f16(want[clean]).view(np.uint16).astype(np.int64))
        # or the rounding of a value within the fp32 criterion: where the ulp is small against the floor (a tail of
        # the response) the floor decides, not the ulp (2048^2 level 1/12 in F16: 156 ulps, fp32 within 1.01e-3 u)
        tol = FLOOR * u + REL * np.abs(want[clean])
        lo = float_parity.round_f16(want[clean] - tol).astype(np.float64)
        hi = float_parity.round_f16(want[clean] + tol).astype(np.float64)
        near = (lo <= half.astype(np.float64)) & (half.astype(np.float64) <= hi)
        report["f16_max_ulp"] = int(ulps.max()) if ulps.size else 0
        assert np.all((ulps <= 1) | near), report
        if got_f32 is None:          # halves only: the ulp rule above on clean texels, parity.py's on edge texels
            assert_close(got16[sel][:, :3].astype(np.float64), "f16", clean_rule=False)
        if zero.any():
            assert np.all(got16[zero][:, :3].astype(np.float64) <= FLOOR * u), report
    return report
