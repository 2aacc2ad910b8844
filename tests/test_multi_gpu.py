"""Device-list entry points (datum_ibl_multi_*, include/datum_ibl_cuda.h): several GPUs driven from ONE
process, the way a single-process tools/assetbuilder.cpp would use them.

A device may be listed twice (two contexts on one GPU), so the whole exchange path — row slabs, the
prefilter kernel's stores into every payload, the last CTA's arrival signal, the stream memory waits —
runs on a one-GPU box; with two or more GPUs the same tests also run across NVLink."""

import os

import numpy as np
import pytest
import torch

import datum_b200
import oracle_lib
import parity
from datum_b200 import synth
from test_host_shim import run_driver

pytestmark = pytest.mark.gpu


def device_lists():
    """Lists of several distinct GPUs stay in the suite and skip on a box with fewer."""
    gpus = torch.cuda.device_count() if torch.cuda.is_available() else 0
    lists = [[0, 0], [0, 0, 0]]
    for devices in ([0, 1], [0, 1, 2, 3]):
        lists.append(pytest.param(devices, marks=pytest.mark.skipif(gpus < len(devices), reason="needs %d GPUs" % len(devices))))
    return lists


@pytest.mark.parametrize("devices", device_lists())
def test_one_probe_shared_by_a_device_list(ctx, devices):
    """BASELINE config 3's mechanism on a small probe: the chain of a device list against the single-device
    chain (slabs re-cut the tiles: a few same-face sample counts differ, hence the packed-word criterion)
    and, level by level, against the oracle on the same source."""
    w, levels, samples = 192, 7, 256         # 6 * (192 >> L) rows divide by 2 and by 3 at every split level
    offs = datum_b200.level_offsets(w, w, levels)
    bits = synth.synthetic_chain(w, w, levels, probe=81, sun=False)
    want = bits.copy()
    ctx.image_buildmips_cube_ibl(w, w, levels, want, samples)

    with datum_b200.MultiContext(devices) as multi:
        for rep in range(2):                       # twice: the payloads and arrival counters are reused
            got = bits.copy()
            multi.image_buildmips_cube_ibl(w, w, levels, got, samples)
            assert np.array_equal(got[: offs[1]], bits[: offs[1]])
            stats = oracle_lib.word_stats(got[offs[1]:], want[offs[1]:])
            assert oracle_lib.words_within_one_code(stats, 0.995), stats

    for level in range(1, levels):
        ws = w >> (level - 1)
        parity.check_level(got[offs[level]:offs[level + 1]], None, got[offs[level - 1]:offs[level]], ws, ws, level, levels, samples)


def test_device_list_batch_and_projection_equal_one_device(ctx):
    w, levels, samples = 64, 6, 256
    probes = list(range(90, 95))
    want = []
    for p in probes:
        b = synth.synthetic_chain(w, w, levels, probe=p)
        ctx.image_buildmips_cube_ibl(w, w, levels, b, samples)
        want.append(b)
    payloads = [synth.synthetic_chain(w, w, levels, probe=p) for p in probes]
    with datum_b200.MultiContext([0, 0]) as multi:
        sh = multi.bake_probes(w, w, levels, payloads, samples, sh9=True)
        for i in range(len(probes)):
            assert np.array_equal(payloads[i], want[i])
            level0 = np.ascontiguousarray(want[i][: 6 * w * w])
            assert np.array_equal(sh[i], ctx.project_sh9(level0, datum_b200.FORMAT_RGBE, w, w))

        cube = synth.synthetic_cube(96, 96, probe=96)
        got = multi.project_sh9(cube, datum_b200.FORMAT_F32, 96, 96)
        ref = oracle_lib.project_sh9(cube, datum_b200.FORMAT_F32, 96, 96)
        assert np.abs(got - ref).max() <= 1e-4 * np.abs(ref).max()


def test_bad_device_lists_raise():
    with pytest.raises(datum_b200.IblError):
        datum_b200.MultiContext([])
    with pytest.raises(datum_b200.IblError):
        datum_b200.MultiContext([0] * 9)                  # at most 8 GPUs share a probe
    with pytest.raises(datum_b200.IblError):
        datum_b200.MultiContext([0, 4096])


def test_host_shim_uses_the_device_list(ctx, tmp_path):
    """DATUM_IBL_DEVICES in the C++ shim: image_buildmips_cube_ibl (the reference's signature) shares the probe
    between the listed devices once a face reaches DATUM_IBL_SPLIT_MIN_FACE texels."""
    w, levels = 64, 7
    bits = synth.synthetic_chain(w, w, levels, probe=31)
    (tmp_path / "in.bin").write_bytes(bits[: 6 * w * w].tobytes())
    env = dict(os.environ, DATUM_IBL_DEVICES="0,0", DATUM_IBL_SPLIT_MIN_FACE="1")
    out = run_driver("chain", w, w, levels, tmp_path / "in.bin", tmp_path / "out.bin", env=env)
    assert out.returncode == 0, out.stdout
    got = np.frombuffer((tmp_path / "out.bin").read_bytes(), np.uint32)
    want = bits.copy()
    ctx.image_buildmips_cube_ibl(w, w, levels, want)
    offs = datum_b200.level_offsets(w, w, levels)
    assert np.array_equal(got[: offs[1]], want[: offs[1]])
    stats = oracle_lib.word_stats(got[offs[1]:], want[offs[1]:])
    assert oracle_lib.words_within_one_code(stats, 0.995), stats
    # below the threshold the first device bakes alone: bit-identical
    env = dict(os.environ, DATUM_IBL_DEVICES="0,0")
    out = run_driver("chain", w, w, levels, tmp_path / "in.bin", tmp_path / "out2.bin", env=env)
    assert out.returncode == 0, out.stdout
    assert np.array_equal(np.frombuffer((tmp_path / "out2.bin").read_bytes(), np.uint32), want)
