"""Level 0 of RGBA32F / RGBA16F chains from an equirect HDR image and from six ARGB32 face images on the GPU
(datum_ibl_pack_cube_float[_ibl], datum_ibl_ingest_cube_argb32_float[_ibl]), against the float oracle's
restatement of the rgbe pack and ingest (tests/oracle_float/ibl_float_oracle.cpp) and against the rgbe
entries and the float chain entry they build on."""

import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import datum_b200
import float_pack_oracle_lib
import float_parity
import oracle_lib
from test_host_shim import write_hdr

pytestmark = pytest.mark.gpu

F32, F16 = datum_b200.FORMAT_F32, datum_b200.FORMAT_F16
NP_DTYPE = {F32: np.float32, F16: np.float16}
GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ibl_golden.npz"))
SHAPES = [(64, 32, 16, 16), (300, 150, 32, 32), (97, 53, 8, 8), (512, 256, 64, 64), (40, 20, 24, 12)]

# Equirect level 0 against the float oracle (equirect_report), floors set from one run of this file on an NVIDIA
# B200 over the golden image, the five shapes, the 2048x1024 sun image and the 1e12 image:
#   share of texels whose three channels are bit-identical: F32 0.767 .. 0.815 (atan2f / acosf of the device differ
#   from the host's in the last ulp, which moves the bilinear weights), F16 0.982 .. 1.0; floors 0.70 and 0.95;
#   error relative to the texel's largest channel, 0.995-quantile: F32 at most 1.5e-4, F16 0 (every texel but a
#   few within 1 ulp); floor 5e-4, about 3x the largest, 8x tighter than the rgbe test's 4e-3;
#   largest error: F32 7.5e-4, F16 8.5e-4; floor 4e-3, about 5x (no texel gained or lost a box-filter tap).
MIN_IDENTICAL = {F32: 0.70, F16: 0.95}
MAX_Q995 = 5e-4
MAX_REL = 4e-3


@pytest.fixture(scope="module")
def fctx():
    context = datum_b200.IblContext(0)
    yield context
    context.close()


def random_equirect(iw, ih, seed, sun=0.0):
    """The images of test_equirect_pack_matches_oracle, optionally with a bright disc (a sun) of radiance `sun`."""
    rng = np.random.default_rng(seed)
    img = np.ones((ih, iw, 4), np.float32)
    img[..., :3] = (rng.random((ih, iw, 3)) * np.exp2(rng.integers(-3, 6, (ih, iw, 1)))).astype(np.float32)
    if sun:
        yy, xx = np.meshgrid(np.arange(ih), np.arange(iw), indexing="ij")
        disc = (yy - 0.3 * ih) ** 2 + (xx - 0.6 * iw) ** 2 <= (0.012 * iw) ** 2
        img[disc, :3] = np.float32(sun) * np.array([1.0, 0.9, 0.75], np.float32)
    return img


def random_faces(h, w, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2**32, (6, h, w), dtype=np.uint64).astype(np.uint32)


def interior(w, h):
    """Texels off each face's outer ring: the edge blend never writes them."""
    mask = np.zeros((6, h, w), bool)
    mask[:, 1:h - 1, 1:w - 1] = True
    return mask.reshape(-1)


def pack(ctx, fmt, img, w, h):
    out = np.zeros((6 * w * h, 4), NP_DTYPE[fmt])
    ctx.pack_cube_float(fmt, img, w, h, out)
    return out


def ingest(ctx, fmt, faces):
    out = np.zeros((faces.size, 4), NP_DTYPE[fmt])
    ctx.ingest_cube_argb32_float(fmt, faces, out)
    return out


def equirect_report(fmt, got, want):
    """Measured agreement of a device level 0 with the float oracle's.  F16: a texel counts as exact when each
    channel is within 1 ulp of the oracle's half; otherwise its error is that of the closest value rounding to
    the stored half (the rounding of a value that meets the fp32 rule)."""
    got = np.asarray(got).reshape(-1, 4)
    want = np.asarray(want).reshape(-1, 4)
    bits = np.uint16 if fmt == F16 else np.uint32
    identical = np.all(got[:, :3].view(bits) == want[:, :3].view(bits), axis=1)
    want32 = want[:, :3].astype(np.float64)
    scale = np.maximum(want32.max(axis=1), 1e-30)
    if fmt == F32:
        rel = np.abs(got[:, :3].astype(np.float64) - want32).max(axis=1) / scale
    else:
        ulps = np.abs(got[:, :3].view(np.uint16).astype(np.int64) - want[:, :3].view(np.uint16).astype(np.int64))
        g = got[:, :3].astype(np.float64)
        with np.errstate(over="ignore"):                                 # the neighbour above 65504 is inf
            up = np.nextafter(got[:, :3], np.float16(np.inf)).astype(np.float64)
        down = np.nextafter(got[:, :3], np.float16(0)).astype(np.float64)
        reach = np.where(want32 >= g, (up - g) / 2, (g - down) / 2)      # half the gap towards the oracle's value
        rel = (np.maximum(np.abs(g - want32) - reach, 0).max(axis=1)) / scale
        rel[np.all(ulps <= 1, axis=1)] = 0.0
        report_ulps = int(ulps.max())
    report = {"texels": len(got), "identical": float(identical.mean()), "q995": float(np.quantile(rel, 0.995)),
              "q999": float(np.quantile(rel, 0.999)), "max": float(rel.max())}
    if fmt == F16:
        report["max_ulp"] = report_ulps
    print("equirect", "F16" if fmt == F16 else "F32", report)
    return report


def assert_equirect(fmt, got, want):
    report = equirect_report(fmt, got, want)
    assert np.all(np.asarray(got)[:, 3] == 1.0), "alpha must be 1.0"
    assert report["identical"] >= MIN_IDENTICAL[fmt], report
    assert report["q995"] <= MAX_Q995, report
    assert report["max"] <= MAX_REL, report
    return report


# ---- six-image ingest ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("h,w", [(1, 1), (7, 13), (64, 64), (24, 40)])
def test_ingest_is_bit_exact_with_the_float_oracle(fctx, fmt, h, w):
    faces = random_faces(h, w, 40 + h)
    got = ingest(fctx, fmt, faces)
    assert np.array_equal(got.view(np.uint8), float_pack_oracle_lib.ingest_cube_argb32(fmt, faces).view(np.uint8))
    assert np.all(got[:, 3] == 1.0)
    if fmt == F32:
        words = np.zeros(6 * h * w, np.uint32)
        fctx.ingest_cube_argb32(faces, words)
        assert np.array_equal(oracle_lib.rgbe_encode_array(got[:, :3]), words)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_ingest_of_the_golden_pixels(fctx, fmt):
    pixels = GOLDEN["ingest_argb"]
    h, w = 7, len(pixels) // 6 // 7
    faces = pixels[: 6 * h * w].reshape(6, h, w)
    got = ingest(fctx, fmt, faces)
    assert np.array_equal(got.view(np.uint8), float_pack_oracle_lib.ingest_cube_argb32(fmt, faces).view(np.uint8))


# ---- equirect pack ---------------------------------------------------------------------------------------------

def equirect_cases():
    return [("golden", None)] + [("random", s) for s in SHAPES]


def equirect_input(kind, shape):
    if kind == "golden":
        return GOLDEN["equirect"], 16, 16
    iw, ih, w, h = shape
    return random_equirect(iw, ih, iw), w, h


@pytest.mark.parametrize("kind,shape", equirect_cases())
def test_equirect_interior_equals_the_rgbe_pack_and_rounds_to_f16(fctx, kind, shape):
    """Off the outer ring both formats hold exactly what the rgbe resample encodes: rgbe(F32) is its word, and
    F16 is the F32 texel rounded to nearest-even."""
    img, w, h = equirect_input(kind, shape)
    words = np.zeros(6 * w * h, np.uint32)
    fctx.image_pack_cube(img, w, h, words)
    f32, f16 = pack(fctx, F32, img, w, h), pack(fctx, F16, img, w, h)
    inner = interior(w, h)
    assert np.array_equal(oracle_lib.rgbe_encode_array(f32[inner, :3]), words[inner])
    assert np.array_equal(f16[inner, :3].view(np.uint16), float_parity.round_f16(f32[inner, :3]).view(np.uint16))


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("kind,shape", equirect_cases())
def test_equirect_pack_against_the_float_oracle(fctx, fmt, kind, shape):
    img, w, h = equirect_input(kind, shape)
    assert_equirect(fmt, pack(fctx, fmt, img, w, h), float_pack_oracle_lib.pack_cube(fmt, img, w, h))


# ---- chains ----------------------------------------------------------------------------------------------------

def source(kind, w):
    if kind == "equirect":
        return random_equirect(4 * w, 2 * w, 7, sun=200.0)
    return random_faces(w, w, 8)


def level0_entry(ctx, fmt, kind, src, w):
    return pack(ctx, fmt, src, w, w) if kind == "equirect" else ingest(ctx, fmt, src)


def chain_entry(ctx, fmt, kind, src, w, levels, chain, samples):
    if kind == "equirect":
        ctx.pack_cube_float_ibl(fmt, src, w, w, levels, chain, samples)
    else:
        ctx.skybox_float_from_argb32(fmt, src, levels, chain, samples)


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("kind", ["equirect", "faces"])
@pytest.mark.parametrize("pinned", [False, True])
def test_chain_entry_is_level0_entry_then_buildmips(fctx, fmt, kind, pinned):
    w, levels, samples = 64, 5, 256
    src = source(kind, w)
    offs = datum_b200.level_offsets(w, w, levels)
    chain = torch.zeros((offs[-1], 4), dtype=torch.float32 if fmt == F32 else torch.float16)
    if pinned:
        chain = chain.pin_memory()
    chain_entry(fctx, fmt, kind, src, w, levels, chain, samples)
    got = chain.numpy()

    level0 = level0_entry(fctx, fmt, kind, src, w)
    assert np.array_equal(got[: offs[1]].view(np.uint8), level0.view(np.uint8))
    want = np.zeros_like(got)
    want[: offs[1]] = level0
    fctx.buildmips_cube_float(fmt, w, w, levels, want, samples)
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8))


@pytest.mark.parametrize("fmt", [F32, F16])
def test_whole_chain_from_an_equirect_sun_against_the_oracle(fctx, fmt):
    """2048x1024 equirect image with a sun -> 128^2 x 6 chain: level 0 against the float oracle's pack, every
    other level against the float oracle on the chain's own previous level (float_parity)."""
    w, levels, samples = 128, 6, 1024
    img = random_equirect(2048, 1024, 11, sun=5000.0)
    offs = datum_b200.level_offsets(w, w, levels)
    chain = np.zeros((offs[-1], 4), NP_DTYPE[fmt])
    fctx.pack_cube_float_ibl(fmt, img, w, w, levels, chain, samples)
    assert_equirect(fmt, chain[: offs[1]], float_pack_oracle_lib.pack_cube(fmt, img, w, w))
    for level in range(1, levels):
        ws = w >> (level - 1)
        out = chain[offs[level]:offs[level + 1]]
        src = chain[offs[level - 1]:offs[level]]
        float_parity.check_float_level(out[:, :3].astype(np.float32) if fmt == F32 else None, out if fmt == F16 else None,
                                       src, ws, ws, level, levels, samples)


# ---- input range -----------------------------------------------------------------------------------------------

def test_f16_pack_of_a_1e6_sun_clamps(fctx):
    w, levels = 32, 6
    img = random_equirect(256, 128, 3, sun=1e6)
    offs = datum_b200.level_offsets(w, w, levels)
    chain = np.zeros((offs[-1], 4), np.float16)
    fctx.pack_cube_float_ibl(F16, img, w, w, levels, chain, 256)
    assert np.all(np.isfinite(chain.astype(np.float32)))
    assert chain[: offs[1], :3].max() == np.float16(65504.0)
    assert_equirect(F16, chain[: offs[1]], float_pack_oracle_lib.pack_cube(F16, img, w, w))


def test_f32_pack_up_to_1e12(fctx):
    iw, ih, w, h = SHAPES[1]
    img = random_equirect(iw, ih, 5, sun=1.0)
    img[..., :3] *= np.float32(1e12) / img[..., :3].max()
    got = pack(fctx, F32, img, w, h)
    assert np.all(np.isfinite(got))
    assert_equirect(F32, got, float_pack_oracle_lib.pack_cube(F32, img, w, h))


# ---- rejection -------------------------------------------------------------------------------------------------

def test_bad_arguments_are_rejected_before_any_launch(fctx):
    lib, hnd = fctx._lib, fctx._handle
    img = np.ones((8, 16, 4), np.float32)
    faces = np.zeros((6, 4, 4), np.uint32)
    buf = np.zeros((6 * 16 * 16 * 2, 4), np.float32)
    p_img, p_faces, p_buf = img.ctypes.data, faces.ctypes.data, buf.ctypes.data
    launches = fctx.launch_count

    def fails(status, text):
        assert status != 0
        assert text in lib.datum_ibl_last_error(), lib.datum_ibl_last_error()

    fails(lib.datum_ibl_pack_cube_float(hnd, F32, 16, 8, None, 4, 4, p_buf), b"datum_ibl_pack_cube_float: null argument")
    fails(lib.datum_ibl_pack_cube_float(hnd, F32, 16, 8, p_img, 4, 4, None), b"null argument")
    fails(lib.datum_ibl_pack_cube_float(None, F32, 16, 8, p_img, 4, 4, p_buf), b"null argument")
    fails(lib.datum_ibl_pack_cube_float(hnd, 0, 16, 8, p_img, 4, 4, p_buf), b"unknown format 0 (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16)")
    fails(lib.datum_ibl_pack_cube_float(hnd, 3, 16, 8, p_img, 4, 4, p_buf), b"unknown format 3")
    fails(lib.datum_ibl_pack_cube_float(hnd, F16, 0, 8, p_img, 4, 4, p_buf), b"bad image size")
    fails(lib.datum_ibl_pack_cube_float(hnd, F16, 16, 8, p_img, 0, 4, p_buf), b"bad width/height")

    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, F32, 16, 8, None, 16, 16, 3, 64, p_buf), b"datum_ibl_pack_cube_float_ibl: null argument")
    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, 7, 16, 8, p_img, 16, 16, 3, 64, p_buf), b"unknown format 7")
    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, F32, 16, -1, p_img, 16, 16, 3, 64, p_buf), b"bad image size")
    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, F32, 16, 8, p_img, 16, 16, 3, 4097, p_buf), b"bad width/height/levels/samples")
    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, F32, 16, 8, p_img, 16, 16, 3, 0, p_buf), b"bad width/height/levels/samples")
    fails(lib.datum_ibl_pack_cube_float_ibl(hnd, F32, 16, 8, p_img, 16, 16, 6, 64, p_buf), b"bad width/height/levels/samples")

    fails(lib.datum_ibl_ingest_cube_argb32_float(hnd, F16, 4, 4, None, p_buf), b"datum_ibl_ingest_cube_argb32_float: null argument")
    fails(lib.datum_ibl_ingest_cube_argb32_float(hnd, 9, 4, 4, p_faces, p_buf), b"unknown format 9")
    fails(lib.datum_ibl_ingest_cube_argb32_float(hnd, F16, 0, 4, p_faces, p_buf), b"bad width/height")
    fails(lib.datum_ibl_ingest_cube_argb32_float_ibl(hnd, F16, 4, 4, 2, 64, p_faces, None), b"datum_ibl_ingest_cube_argb32_float_ibl: null argument")
    fails(lib.datum_ibl_ingest_cube_argb32_float_ibl(hnd, 0, 4, 4, 2, 64, p_faces, p_buf), b"unknown format 0")
    fails(lib.datum_ibl_ingest_cube_argb32_float_ibl(hnd, F16, 4, 4, 2, 5000, p_faces, p_buf), b"bad width/height/levels/samples")
    fails(lib.datum_ibl_ingest_cube_argb32_float_ibl(hnd, F16, 4, 4, 4, 64, p_faces, p_buf), b"bad width/height/levels/samples")

    # the Python checks: dtype, size, host buffer
    with pytest.raises(ValueError):
        fctx.pack_cube_float(F16, img, 4, 4, np.zeros((96, 4), np.float32))
    with pytest.raises(ValueError):
        fctx.pack_cube_float(F32, img, 4, 4, np.zeros((95, 4), np.float32))
    with pytest.raises(ValueError):
        fctx.pack_cube_float(5, img, 4, 4, np.zeros((96, 4), np.float32))
    with pytest.raises(ValueError):
        fctx.pack_cube_float_ibl(F32, img[..., :3], 4, 4, 2, np.zeros((120, 4), np.float32))
    with pytest.raises(ValueError):
        fctx.skybox_float_from_argb32(F32, faces, 2, torch.zeros((120, 4), dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError):
        fctx.ingest_cube_argb32_float(F32, faces[:5], np.zeros((96, 4), np.float32))
    with pytest.raises(datum_b200.IblError):
        fctx.skybox_float_from_argb32(F32, faces, 2, np.zeros((120, 4), np.float32), samples=5000)

    torch.cuda.synchronize()
    assert fctx.launch_count == launches


# ---- host shim -------------------------------------------------------------------------------------------------

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def float_pack_driver():
    """tests/host/float_pack_driver.cpp linked against the built shim and library, in a temporary directory."""
    from datum_b200 import build as recipe
    recipe.build_all()
    libdir = os.path.join(ROOT, "datum_b200", "lib")
    out = os.path.join(tempfile.mkdtemp(prefix="datum_float_pack_driver_"), "float_pack_driver")
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([gxx, "-std=c++14", "-O2", "-I", os.path.join(ROOT, "datum_b200", "host"), "-o", out,
                           os.path.join(ROOT, "tests", "host", "float_pack_driver.cpp"),
                           "-L", libdir, "-ldatum_ibl_host", "-ldatum_ibl_cuda", "-Wl,-rpath," + libdir])
    return out

@pytest.mark.parametrize("fmt", [F32, F16])
def test_hdr_file_to_float_chain_through_the_host_shim(fctx, float_pack_driver, tmp_path, fmt):
    """load_hdr + image_pack_cube_float_ibl, the .hdr flow of write_skybox_asset producing a float probe."""
    img = random_equirect(96, 48, 21, sun=300.0)[..., :3]
    decoded = write_hdr(str(tmp_path / "env.hdr"), img)
    w, levels = 16, 4
    out = subprocess.run([float_pack_driver, "hdr_float", str(tmp_path / "env.hdr"), str(w), str(w), str(levels), str(fmt), str(tmp_path / "out.bin")],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout
    got = np.frombuffer((tmp_path / "out.bin").read_bytes(), NP_DTYPE[fmt]).reshape(-1, 4)
    want = np.zeros_like(got)
    fctx.pack_cube_float_ibl(fmt, decoded, w, w, levels, want)
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8))
