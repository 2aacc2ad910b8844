"""The CPU oracle against the golden vectors generated from the unmodified
reference (tests/golden/make_golden.py) and against known answers.  CPU only."""

import ctypes
import os

import numpy as np
import pytest

import oracle_lib
from datum_b200 import synth

GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ibl_golden.npz"))


def test_codec_encode_matches_reference_words():
    words = oracle_lib.rgbe_encode_array(GOLDEN["codec_rgb"])
    assert np.array_equal(words, GOLDEN["codec_words"])


def test_codec_decode_matches_reference_bits():
    rgba = oracle_lib.rgbe_decode_array(GOLDEN["decode_words"])
    assert np.array_equal(rgba.view(np.uint32), GOLDEN["decode_rgba"].view(np.uint32))


def test_codec_known_answers():
    enc = lambda r, g, b: int(oracle_lib.oracle().oracle_rgbe_encode(r, g, b))
    assert enc(0, 0, 0) == 0                       # max == 0: log2 -> -inf, exponent floor, word 0
    assert enc(1, 1, 1) == 0x84020100              # e = 1, mantissa round(255.5) = 256 (half away from zero)
    assert enc(65408, 0, 0) == enc(1e9, 0, 0)      # value clamp (color.h:156-158)
    assert enc(65408, 0, 0) >> 27 == 31
    assert enc(255.99998, 0, 0) == 0xC00000FF      # log2f rounds up just below 2^8: exponent rolls over
    assert enc(-5.0, 0.5, 0.25) == enc(0.0, 0.5, 0.25)
    rgba = oracle_lib.rgbe_decode_array(np.array([0x84020100], np.uint32))[0]
    assert rgba[0] == np.float32(256 / 511.0 * 2) and rgba[3] == 1.0


def test_numpy_codec_matches_oracle():
    rng = np.random.default_rng(1)
    rgb = (rng.random((5000, 3)) * np.exp2(rng.integers(-18, 17, (5000, 1)))).astype(np.float32)
    assert np.array_equal(synth.rgbe_words(rgb), oracle_lib.rgbe_encode_array(rgb))


def test_srgba_decode_matches_reference():
    out = np.zeros((len(GOLDEN["srgba_argb"]), 4), np.float32)
    for i, w in enumerate(GOLDEN["srgba_argb"]):
        oracle_lib.oracle().oracle_srgba_decode(int(w), out[i].ctypes.data)
    assert np.array_equal(out.view(np.uint32), GOLDEN["srgba_rgba"].view(np.uint32))


def test_six_image_ingest_matches_reference_pixel_arithmetic():
    """oracle_ingest_cube_argb32 == rgbe(srgba(pixel)) of the reference's color.h for every pixel
    (golden composed from the compiled reference), rows mirrored, faces in argument order
    (tools/assetbuilder.cpp:443-462)."""
    pixels, want = GOLDEN["ingest_argb"], GOLDEN["ingest_words"]
    n = (len(pixels) // 6 // 7) * 7                       # 6 faces of 7 x (n/7)... any rectangle will do
    h, w = 7, n // 7
    faces = pixels[: 6 * h * w].reshape(6, h, w)
    got = oracle_lib.ingest_cube_argb32(faces).reshape(6, h, w)
    assert np.array_equal(got, want[: 6 * h * w].reshape(6, h, w)[:, ::-1, :])


def test_face_rotations_match_reference():
    vecs, want = GOLDEN["rotate_in"], GOLDEN["rotate_out"]
    for f in range(6):
        for i, v in enumerate(vecs):
            out = np.zeros(3, np.float32)
            vin = np.ascontiguousarray(v)
            oracle_lib.oracle().oracle_face_rotate(f, vin.ctypes.data, out.ctypes.data)
            assert np.array_equal(out.view(np.uint32), want[f, i].view(np.uint32))


def test_face_rotations_are_the_closed_forms():
    """ibl.cpp:253-261 rotations equal data/convolve.comp:85-100's closed forms up to rounding."""
    d = synth.cube_directions(8, 8)
    for f in range(6):
        for y in (0, 3, 7):
            for x in (0, 5):
                out = np.zeros(3, np.float32)
                oracle_lib.oracle().oracle_texel_direction(f, x, y, 8, 8, out.ctypes.data)
                assert np.allclose(out, d[f, y, x], atol=3e-7)


def test_radical_inverse_known_answers():
    ri = oracle_lib.oracle().oracle_radicalinverse
    assert ri(0) == 0.0 and ri(1) == 0.5 and ri(2) == 0.25 and ri(3) == 0.75
    assert ri(1023) == np.float32(1023 / 1024.0)
    assert ri(4095) == np.float32(4095 / 4096.0)
    assert ri(0x80000000) == np.float32(2.0 ** -32)


@pytest.mark.parametrize("name,w,h,levels", [("chain16_noise", 16, 16, 5), ("chain16_smooth", 16, 16, 5), ("chain32_noise", 32, 32, 6), ("chain24x12", 24, 12, 3)])
def test_chain_is_word_identical_to_reference(name, w, h, levels):
    want = GOLDEN[name]
    bits = np.zeros_like(want)
    bits[: 6 * w * h] = GOLDEN[name + "_level0"]
    oracle_lib.buildmips_cube_ibl(w, h, levels, bits, samples=1024)
    assert np.array_equal(bits, want)


def test_equirect_pack_is_word_identical_to_reference():
    img = GOLDEN["equirect"]
    assert np.array_equal(oracle_lib.image_pack_cube(img, 16, 16, 1), GOLDEN["equirect_cube16"])
    assert np.array_equal(oracle_lib.image_pack_cube_ibl(img, 16, 16, 4), GOLDEN["equirect_chain16"])


def test_luts_are_word_identical_to_reference():
    words, _ = oracle_lib.pack_envbrdf(16, 16, 1024)
    assert np.array_equal(words, GOLDEN["envbrdf16"])
    p = GOLDEN["water_params"]
    water = oracle_lib.pack_watercolor(p[0:3], p[3:6], float(p[6]), p[7:10], float(p[10]), float(p[11]), 16, 16)
    assert np.array_equal(water, GOLDEN["water16"])


# ---- properties of the bake the GPU tests reuse at full size ----

def test_constant_environment_stays_constant():
    w, levels = 16, 5
    offs = [0]
    for i in range(levels):
        offs.append(offs[-1] + 6 * (w >> i) ** 2)
    bits = np.zeros(offs[-1], np.uint32)
    word = oracle_lib.rgbe_encode_array(np.array([[0.75, 0.5, 0.25]], np.float32))[0]
    bits[: offs[1]] = word
    f32 = oracle_lib.buildmips_cube_ibl(w, w, levels, bits, want_f32=True)
    dec = oracle_lib.rgbe_decode_array(np.array([word], np.uint32))[0, :3]
    assert np.allclose(f32, dec[None, :], rtol=1e-5)   # 1024 sequential fp32 adds
    assert oracle_lib.word_stats(bits[offs[1]:], np.full(offs[-1] - offs[1], word, np.uint32))["max_code"] <= 1


def test_sh9_constant_radiance_and_ramp():
    w = 16
    c = np.array([0.5, 1.0, 2.0])
    level0 = np.ones((6, w, w, 4), np.float32)
    level0[..., :3] = c
    sh = oracle_lib.project_sh9(level0, 1, w, w)
    assert np.allclose(sh[0], 0.282095 * 4 * np.pi * c, rtol=1e-12)
    assert np.abs(sh[1:]).max() < 1e-12

    d = synth.cube_directions(w, w)
    level0[..., :3] = d[..., 1:2]            # radiance = dir.y (signed: the projection is linear)
    sh = oracle_lib.project_sh9(level0, 1, w, w)
    others = np.delete(np.arange(9), 1)
    assert abs(sh[1, 0]) > 1.0 and np.abs(sh[others]).max() < 2e-2 * abs(sh[1, 0])


def test_sh9_partials_add_up():
    w = 8
    level0 = synth.synthetic_cube(w, w, probe=5, sun=False)
    full = oracle_lib.sh9_partial(level0, 1, w, w, 0, 6 * w)
    parts = oracle_lib.sh9_partial(level0, 1, w, w, 0, 19) + oracle_lib.sh9_partial(level0, 1, w, w, 19, 6 * w)
    assert np.allclose(full, parts, rtol=1e-12)
    assert np.isclose(full[27], 4 * np.pi, rtol=1e-9)   # the texel solid angles tile the sphere
    words = synth.rgbe_words(level0)
    sh_rgbe = oracle_lib.project_sh9(words, 0, w, w)
    sh_f32 = oracle_lib.project_sh9(level0, 1, w, w)
    assert np.allclose(sh_rgbe, sh_f32, rtol=5e-3, atol=5e-3 * np.abs(sh_f32).max())


def test_irradiance_of_constant_radiance_is_pi_c():
    w = 8
    level0 = np.ones((6, w, w, 4), np.float32)
    level0[..., :3] = [0.2, 0.4, 0.8]
    sh = oracle_lib.project_sh9(level0, 1, w, w)
    normals = synth.cube_directions(4, 4).reshape(-1, 3)
    e = oracle_lib.sh9_irradiance(sh, normals)
    assert np.allclose(e, np.pi * np.array([0.2, 0.4, 0.8]), rtol=1e-5)
