"""The C++ host shim (datum_b200/host) through the reference's tools/ibl.h signatures,
driven the way tools/assetbuilder.cpp drives them (tests/host/host_driver.cpp), and the
equirect -> cube stage through the C ABI."""

import os
import subprocess

import numpy as np
import pytest

import oracle_lib
from datum_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", "ibl_golden.npz"))
DRIVER = os.path.join(ROOT, "tests", "host", "host_driver")
DRIVER_SRC = os.path.join(ROOT, "tests", "host", "host_driver.cpp")
LIBDIR = os.path.join(ROOT, "datum_b200", "lib")


def build_driver():
    from datum_b200 import build as recipe
    recipe.build_all()
    stale = not os.path.exists(DRIVER) or os.path.getmtime(DRIVER) < max(os.path.getmtime(DRIVER_SRC), os.path.getmtime(os.path.join(LIBDIR, "libdatum_ibl_host.so")))
    if stale:
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([gxx, "-std=c++14", "-O2", "-I", os.path.join(ROOT, "datum_b200", "host"), "-o", DRIVER, DRIVER_SRC,
                               "-L", LIBDIR, "-ldatum_ibl_host", "-ldatum_ibl_cuda", "-Wl,-rpath," + LIBDIR])
    return DRIVER


def run_driver(*args, env=None):
    return subprocess.run([build_driver()] + [str(a) for a in args], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)


def write_hdr(path, image, exposure=None):
    """Radiance new-style RLE writer (test input for load_hdr): (H, W, 3) float32 -> .hdr.
    Returns the image as the loader will decode it, RGBA fp32."""
    h, w, _ = image.shape
    m = image.max(axis=2)
    e = np.where(m > 1e-32, np.floor(np.log2(np.maximum(m, 1e-38))) + 1, -128).astype(np.int32)
    scale = np.where(m > 1e-32, np.exp2(-e.astype(np.float64)) * 256.0, 0.0)
    mant = np.clip(np.floor(image * scale[..., None]), 0, 255).astype(np.uint8)
    expo = np.where(m > 1e-32, e + 128, 0).astype(np.uint8)
    planes = np.concatenate([mant, expo[..., None]], axis=2)      # (H, W, 4)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\n# written by tests/test_host_shim.py\nFORMAT=32-bit_rle_rgbe\n")
        if exposure is not None:
            f.write(("EXPOSURE=%g\n" % exposure).encode())
        f.write(("\n-Y %d +X %d\n" % (h, w)).encode())
        for y in range(h):
            f.write(bytes([2, 2, w >> 8, w & 255]))
            for k in range(4):
                row = planes[y, :, k]
                x = 0
                while x < w:
                    run = 1
                    while x + run < w and run < 127 and row[x + run] == row[x]:
                        run += 1
                    if run >= 4:
                        f.write(bytes([128 + run, int(row[x])]))
                        x += run
                    else:
                        n = min(128, w - x, 16)
                        f.write(bytes([n]) + row[x:x + n].tobytes())
                        x += n
    decoded = np.ones((h, w, 4), np.float32)
    decoded[..., :3] = (mant.astype(np.float32) / np.float32(255.0)) * np.exp2(expo.astype(np.float32) - np.float32(128.0))[..., None]
    return decoded


def test_shim_reports_a_missing_gpu_like_assetbuilder_would():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = run_driver("nogpu")
    assert out.returncode == 1 and "Critical Error" in out.stdout and "no CPU fallback" in out.stdout


@pytest.mark.gpu
def test_buildmips_through_the_reference_signature(ctx, tmp_path):
    w, levels = 64, 7
    bits = synth.synthetic_chain(w, w, levels, probe=31)
    (tmp_path / "in.bin").write_bytes(bits[: 6 * w * w].tobytes())
    out = run_driver("chain", w, w, levels, tmp_path / "in.bin", tmp_path / "out.bin")
    assert out.returncode == 0, out.stdout
    got = np.frombuffer((tmp_path / "out.bin").read_bytes(), np.uint32)
    want = bits.copy()
    ctx.image_buildmips_cube_ibl(w, w, levels, want)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_hdr_file_to_baked_payload(ctx, tmp_path):
    """load_hdr + image_pack_cube_ibl, the flow of tools/assetbuilder.cpp:473-491, on a small cube."""
    rng = np.random.default_rng(5)
    ih, iw = 48, 96
    yy, xx = np.meshgrid(np.arange(ih), np.arange(iw), indexing="ij")
    img = np.stack([0.2 + 0.8 * np.abs(np.sin(0.13 * xx)), 0.1 + 0.9 * (yy / ih), 0.4 + 0.3 * np.cos(0.09 * xx + 0.1 * yy) ** 2], -1)
    img[10:13, 30:34] += 500.0
    img[20:, :8] = 0.25                      # flat region: exercises the RLE runs
    img *= 1.0 + 0.2 * rng.random((ih, iw, 1))
    decoded = write_hdr(str(tmp_path / "env.hdr"), img.astype(np.float32), exposure=1.5)
    w, levels = 16, 4
    out = run_driver("hdr", tmp_path / "env.hdr", w, w, levels, tmp_path / "out.bin")
    assert out.returncode == 0, out.stdout
    assert out.stdout.split()[:3] == [str(iw), str(ih), "1.5"]
    got = np.frombuffer((tmp_path / "out.bin").read_bytes(), np.uint32)

    want0 = oracle_lib.image_pack_cube(decoded, w, w, 1)
    stats = oracle_lib.word_stats(got[: 6 * w * w], want0)
    assert oracle_lib.words_within_one_code(stats, 0.97), stats
    # the chain on top of OUR level 0 equals the plain chain entry point
    chain = np.zeros_like(got)
    chain[: 6 * w * w] = got[: 6 * w * w]
    ctx.image_buildmips_cube_ibl(w, w, levels, chain)
    assert np.array_equal(got, chain)


@pytest.mark.gpu
def test_luts_through_the_reference_signatures(tmp_path):
    out = run_driver("luts", tmp_path / "luts.bin")
    assert out.returncode == 0, out.stdout
    got = np.frombuffer((tmp_path / "luts.bin").read_bytes(), np.uint32)
    want_brdf, _ = oracle_lib.pack_envbrdf(256, 256, 1024)          # assetbuilder.cpp:496-503
    stats = oracle_lib.word_stats(got[: 65536], want_brdf)
    assert oracle_lib.words_within_one_code(stats, 0.98), stats
    want_water = oracle_lib.pack_watercolor([0.0, 0.007, 0.005], [0.1, 0.6, 0.7], 1.0, [0.0, 0.0, 0.0], 0.328, 5.0, 256, 256)
    stats = oracle_lib.word_stats(got[65536:], want_water)
    assert oracle_lib.words_within_one_code(stats, 0.98), stats


@pytest.mark.gpu
def test_equirect_pack_matches_reference_golden(ctx):
    """tools/hdr.cpp:331-359 (resample + edge blend) and tools/ibl.cpp:283-288 against the
    words the unmodified reference produced."""
    img = GOLDEN["equirect"]
    got = np.zeros(6 * 16 * 16, np.uint32)
    ctx.image_pack_cube(img, 16, 16, got)
    stats = oracle_lib.word_stats(got, GOLDEN["equirect_cube16"])
    assert oracle_lib.words_within_one_code(stats, 0.97), stats

    chain = np.zeros(len(GOLDEN["equirect_chain16"]), np.uint32)
    ctx.image_pack_cube_ibl(img, 16, 16, 4, chain)
    assert np.array_equal(chain[: 6 * 256], got)
    dec_got = oracle_lib.rgbe_decode_array(chain)[:, :3].astype(np.float64)
    dec_ref = oracle_lib.rgbe_decode_array(GOLDEN["equirect_chain16"])[:, :3].astype(np.float64)
    rel = np.abs(dec_got - dec_ref).max(axis=1) / np.maximum(dec_ref.max(axis=1), 1e-30)
    assert np.quantile(rel, 0.99) <= 4e-3 and rel.max() <= 1e-1


@pytest.mark.gpu
@pytest.mark.parametrize("iw,ih,w,h", [(64, 32, 16, 16), (300, 150, 32, 32), (97, 53, 8, 8), (512, 256, 64, 64), (40, 20, 24, 12)])
def test_equirect_pack_matches_oracle(ctx, iw, ih, w, h):
    rng = np.random.default_rng(iw)
    img = np.ones((ih, iw, 4), np.float32)
    img[..., :3] = (rng.random((ih, iw, 3)) * np.exp2(rng.integers(-3, 6, (ih, iw, 1)))).astype(np.float32)
    got = np.zeros(6 * w * h, np.uint32)
    ctx.image_pack_cube(img, w, h, got)
    want = oracle_lib.image_pack_cube(img, w, h, 1)
    stats = oracle_lib.word_stats(got, want)
    # atan2f / acosf of the device differ from the host's in the last ulp: a texel whose box
    # filter gains or loses a tap (fp32 loop counter, hdr.cpp:49-51) may differ more
    assert stats["identical"] >= 0.97, stats
    dec_got, dec_want = oracle_lib.rgbe_decode_array(got)[:, :3], oracle_lib.rgbe_decode_array(want)[:, :3]
    rel = oracle_lib.relative_error(dec_got, dec_want)
    assert np.quantile(rel, 0.995) <= 4e-3, float(np.quantile(rel, 0.995))


@pytest.mark.gpu
def test_irradiance_payloads_through_the_host_shim(ctx, tmp_path):
    """SURVEY 8 f4: SH9 as a 3x9 f32 IMAG payload (== Irradiance::L[9][3]) and the irradiance cube as a
    6-layer rgbe IMAG payload, both through the C++ shim, against the fp64 oracle."""
    import datum_b200
    w, iw = 32, 8
    level0 = synth.synthetic_chain(w, w, 1, probe=61, sun=False)
    (tmp_path / "level0.bin").write_bytes(level0.tobytes())
    out = run_driver("irradiance", w, w, iw, iw, tmp_path / "level0.bin", tmp_path / "out.bin")
    assert out.returncode == 0, out.stdout
    raw = (tmp_path / "out.bin").read_bytes()
    assert len(raw) == 27 * 4 + 6 * iw * iw * 4
    sh = np.frombuffer(raw[:108], np.float32).reshape(9, 3)
    want_sh = oracle_lib.project_sh9(level0, datum_b200.FORMAT_RGBE, w, w)
    assert np.abs(sh - want_sh).max() <= 1e-4 * np.abs(want_sh).max()
    cube = np.frombuffer(raw[108:], np.uint32)
    want_words, _ = ctx.sh9_irradiance_cube(sh, iw, iw)
    assert np.array_equal(cube, want_words)

