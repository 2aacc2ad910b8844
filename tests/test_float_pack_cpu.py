"""Level 0 of a float chain on the CPU: the float oracle's restatement of the equirect pack (resample + edge
blend) and of the six-image ingest, pinned to the rgbe oracle through its rgbe instantiation, and its binary16
rounding pinned to numpy's."""

import os

import numpy as np
import pytest

import float_pack_oracle_lib
import oracle_lib

GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ibl_golden.npz"))

RGBE, F32, F16 = 0, 1, 2

# the shapes of test_host_shim.py::test_equirect_pack_matches_oracle: (image width, image height, face width, face height)
SHAPES = [(64, 32, 16, 16), (300, 150, 32, 32), (97, 53, 8, 8), (512, 256, 64, 64), (40, 20, 24, 12)]


def random_equirect(iw, ih, seed):
    rng = np.random.default_rng(seed)
    img = np.ones((ih, iw, 4), np.float32)
    img[..., :3] = (rng.random((ih, iw, 3)) * np.exp2(rng.integers(-3, 6, (ih, iw, 1)))).astype(np.float32)
    return img


def random_faces(h, w, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2**32, (6, h, w), dtype=np.uint64).astype(np.uint32)


def interior(w, h):
    """Texels off each face's outer ring: the edge blend never writes them."""
    mask = np.zeros((6, h, w), bool)
    mask[:, 1:h - 1, 1:w - 1] = True
    return mask.reshape(-1)


def test_rgbe_restatement_of_the_golden_equirect_pack():
    img = GOLDEN["equirect"]
    assert np.array_equal(float_pack_oracle_lib.pack_cube(RGBE, img, 16, 16), oracle_lib.image_pack_cube(img, 16, 16, 1))


@pytest.mark.parametrize("iw,ih,w,h", SHAPES)
def test_rgbe_restatement_of_the_equirect_pack(iw, ih, w, h):
    img = random_equirect(iw, ih, iw)
    assert np.array_equal(float_pack_oracle_lib.pack_cube(RGBE, img, w, h), oracle_lib.image_pack_cube(img, w, h, 1))


@pytest.mark.parametrize("h,w", [(1, 1), (7, 13), (64, 64)])
def test_rgbe_restatement_of_the_ingest(h, w):
    faces = random_faces(h, w, 40 + h)
    assert np.array_equal(float_pack_oracle_lib.ingest_cube_argb32(RGBE, faces), oracle_lib.ingest_cube_argb32(faces))


def test_rgbe_restatement_of_the_golden_ingest_pixels():
    pixels = GOLDEN["ingest_argb"]
    h, w = 7, len(pixels) // 6 // 7
    faces = pixels[: 6 * h * w].reshape(6, h, w)
    assert np.array_equal(float_pack_oracle_lib.ingest_cube_argb32(RGBE, faces), oracle_lib.ingest_cube_argb32(faces))


@pytest.mark.parametrize("iw,ih,w,h", SHAPES[:3])
def test_float_formats_differ_from_rgbe_only_in_the_store(iw, ih, w, h):
    """Off the outer ring (no blend), rgbe(F32 texel) is the rgbe word and the F16 texel is the F32 texel
    rounded; the blend re-reads stored texels, so on the ring each format follows its own values."""
    img = random_equirect(iw, ih, iw + 1)
    words = float_pack_oracle_lib.pack_cube(RGBE, img, w, h)
    f32 = float_pack_oracle_lib.pack_cube(F32, img, w, h)
    f16 = float_pack_oracle_lib.pack_cube(F16, img, w, h)
    inner = interior(w, h)
    assert np.all(f32[:, 3] == 1.0) and np.all(f16[:, 3] == 1.0)
    assert np.array_equal(oracle_lib.rgbe_encode_array(f32[inner, :3]), words[inner])
    assert np.array_equal(f16[inner, :3].view(np.uint16), float_pack_oracle_lib.half_rn(f32[inner, :3]).view(np.uint16))


def test_float_ingest_is_the_linear_table():
    faces = random_faces(9, 5, 3)
    f32 = float_pack_oracle_lib.ingest_cube_argb32(F32, faces)
    f16 = float_pack_oracle_lib.ingest_cube_argb32(F16, faces)
    table = np.array([np.float32(np.float32(c) / np.float32(255.0)) ** np.float32(2.2) for c in range(256)], np.float32)
    mirrored = faces[:, ::-1, :].reshape(-1)
    want = np.stack([(mirrored >> 16) & 255, (mirrored >> 8) & 255, mirrored & 255], -1)
    # the oracle's powf against numpy's: equal to 1 ulp; the identity with the rgbe ingest is exact
    assert np.allclose(f32[:, :3], table[want], rtol=2e-7, atol=0)
    assert np.array_equal(oracle_lib.rgbe_encode_array(f32[:, :3]), oracle_lib.ingest_cube_argb32(faces))
    assert np.array_equal(f16[:, :3].view(np.uint16), float_pack_oracle_lib.half_rn(f32[:, :3]).view(np.uint16))
    assert np.all(f32[:, 3] == 1.0) and np.all(f16[:, 3] == 1.0)


def half_sweep():
    """Every finite non-negative binary16 value, the midpoints between neighbours and one fp32 ulp on either
    side of each, values above 65504, fp32 values in and below the subnormal range, and a seeded sweep."""
    halves = np.arange(0, 0x7C00, dtype=np.uint16).view(np.float16).astype(np.float32)
    mids = ((halves[:-1].astype(np.float64) + halves[1:].astype(np.float64)) / 2).astype(np.float32)   # exact in fp32
    above = np.array([65504.0, 65505.0, 65519.0, 65519.996, 65520.0, 65536.0, 1e5, 1e6, 1e12, 3.4e38], np.float32)
    tiny = np.array([2.0**-24, 2.0**-25, 2.0**-26, 1.5 * 2.0**-25, 2.0**-14, 2.0**-14 - 2.0**-25, 1e-10, 1e-30, 1e-45], np.float32)
    rng = np.random.default_rng(16)
    bits = rng.integers(0, 0x49800000, 200000, dtype=np.uint32)       # fp32 bit patterns from 0 to 2^20
    values = np.concatenate([halves, mids, np.nextafter(mids, np.float32(0)), np.nextafter(mids, np.float32(np.inf)), above, tiny, bits.view(np.float32)])
    return values.astype(np.float32)


def test_oracle_half_rounding_equals_numpy():
    x = half_sweep()
    with np.errstate(over="ignore"):
        want = np.minimum(x, np.float32(65504.0)).astype(np.float16)
    assert np.array_equal(float_pack_oracle_lib.half_rn(x).view(np.uint16), want.view(np.uint16))
