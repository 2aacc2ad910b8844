"""Parity criteria of the float chains (RGBA32F / RGBA16F), TEST INFRASTRUCTURE.

The criteria of parity.py, taken against the float oracle (float_oracle_lib.prefilter_level_rgba32f) on the
same source level:
  (i)  fp32 values: max relative error per texel channel <= 1e-3 of the texel's largest channel;
       texels that own samples within 2e-6 of a cube-face boundary may be off by the weight share of
       those samples times the brightest radiance of the source level;
  F16  stored binary16 values, clean texels: at most 1 ulp from the oracle's value rounded the way the
       library rounds (min(x, 65504) to nearest-even), >= 99 % identical.
"""

import numpy as np

import float_oracle_lib
import oracle_lib
import parity

TOL_F32 = parity.TOL_F32


def round_f16(f32):
    """The stored value of a RGBA16F chain for an fp32 result."""
    return np.minimum(np.asarray(f32, np.float32), np.float32(65504.0)).astype(np.float16)


def widen(src):
    """A float level as (texels, 4) float32 (binary16 widened exactly)."""
    return np.asarray(src).reshape(-1, 4).astype(np.float32)


def check_float_level(got_f32, got_f16, src, ws, hs, level, levels, samples, row_begin=0, row_end=None, tol=TOL_F32, min_identical=0.99):
    """Compare one level computed from the float level `src` ((texels, 4) float32 or float16) with the
    float oracle on the same source.  got_f32: (texels, 3) fp32 rgb (or None); got_f16: (texels, 4)
    float16 stored texels (or None).  Returns measured figures; raises AssertionError on violation."""
    wd, hd = ws >> 1, hs >> 1
    if row_end is None:
        row_end = 6 * hd
    src32 = widen(src)
    want = float_oracle_lib.prefilter_level_rgba32f(src32, ws, hs, level, levels, samples, row_begin, row_end)
    sl = slice(row_begin * wd, row_end * wd)
    want = want[sl]
    edge_counts = oracle_lib.edge_ambiguous_counts(wd, hd, level, levels, samples, row_begin=row_begin, row_end=row_end)[sl]
    edge = edge_counts > 0
    clean = ~edge

    report = {"level": level, "texels": int(clean.size), "edge_fraction": float(edge.mean())}

    if got_f32 is not None:
        got = np.asarray(got_f32, dtype=np.float64).reshape(-1, 3)[sl]
        rel = oracle_lib.relative_error(got, want)
        report["max_rel_clean"] = float(rel[clean].max()) if clean.any() else 0.0
        report["max_rel_edge"] = float(rel[edge].max()) if edge.any() else 0.0
        assert report["max_rel_clean"] <= tol, report
        if edge.any():
            brightest = float(src32[:, :3].max())
            share = edge_counts[edge] / parity.total_sample_weight(level, levels, samples)
            abs_err = np.abs(got[edge] - want[edge].astype(np.float64)).max(axis=1)
            allowed = share * brightest + tol * want[edge].max(axis=1)
            assert np.all(abs_err <= allowed), report

    if got_f16 is not None:
        got16 = np.asarray(got_f16, dtype=np.float16).reshape(-1, 4)[sl]
        assert np.all(got16[:, 3] == np.float16(1.0)), "output alpha must be 1.0"
        if got_f32 is not None:      # the stored texel is the fp32 result rounded as documented
            assert np.array_equal(got16[:, :3].view(np.uint16), round_f16(np.asarray(got_f32, np.float32).reshape(-1, 3)[sl]).view(np.uint16))
        a = got16[clean][:, :3].view(np.uint16).astype(np.int64)
        b = round_f16(want[clean]).view(np.uint16).astype(np.int64)
        ulps = np.abs(a - b)
        report["f16_identical"] = float((ulps == 0).mean()) if ulps.size else 1.0
        report["f16_max_ulp"] = int(ulps.max()) if ulps.size else 0
        assert report["f16_max_ulp"] <= 1, report
        if clean.sum() >= 512:
            assert report["f16_identical"] >= min_identical, report

    return report
