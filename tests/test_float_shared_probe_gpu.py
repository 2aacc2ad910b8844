"""One RGBA16F / RGBA32F probe shared by several GPUs (datum_ibl_prefilter_level_float_peers,
datum_ibl_multi_buildmips_cube_float, dist.PeerChain with a float format).

Slabs re-cut the tiles (and a small slab may take other warps per tile or per texel than the whole level), so a
shared bake is held to the one-device chain by a tolerance, not byte for byte:
  * level 0 byte-identical, and two bakes of one probe give the same bytes on every rank;
  * F32: every channel within 1e-4 of the texel's largest channel; F16: within 1 binary16 ulp, >= 99.5 %
    identical (inputs without the sun);
  * every level passes float_parity.check_float_level against the float oracle on its own source.
A device may be listed twice, so the whole exchange path runs on a one-GPU box too."""

import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import datum_b200
import float_parity
from datum_b200 import dist as ibl_dist
from datum_b200 import synth

pytestmark = pytest.mark.gpu

F32, F16 = datum_b200.FORMAT_F32, datum_b200.FORMAT_F16
NP_DTYPE = {F32: np.float32, F16: np.float16}
TORCH_DTYPE = {F32: torch.float32, F16: torch.float16}
DEV = "cuda:0"


@pytest.fixture(scope="module")
def fctx():
    context = datum_b200.IblContext(0)
    yield context
    context.close()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def device_lists():
    """Lists of several distinct GPUs stay in the suite and skip on a box with fewer."""
    gpus = torch.cuda.device_count() if torch.cuda.is_available() else 0
    lists = [[0, 0], [0, 0, 0]]
    for devices in ([0, 1], [0, 1, 2, 3]):
        lists.append(pytest.param(devices, marks=pytest.mark.skipif(gpus < len(devices), reason="needs %d GPUs" % len(devices))))
    return lists


def float_chain(fmt, w, levels, probe, sun=False):
    """(texels, 4) host chain of the format, level 0 from synth.synthetic_cube, the other levels zero."""
    chain = np.zeros((datum_b200.level_offsets(w, w, levels)[-1], 4), NP_DTYPE[fmt])
    chain[: 6 * w * w] = synth.synthetic_cube(w, w, probe=probe, sun=sun).reshape(-1, 4).astype(NP_DTYPE[fmt])
    return chain


def one_device(ctx, fmt, w, levels, samples, probe):
    chain = float_chain(fmt, w, levels, probe)
    ctx.buildmips_cube_float(fmt, w, w, levels, chain, samples)
    return chain


def check_close(fmt, got, want):
    """The shared bake against the one-device chain: F32 within 1e-4 of each texel's largest channel, F16
    within 1 ulp and >= 99.5 % identical.  Returns the measured figures."""
    if fmt == F32:
        a, b = got[:, :3].astype(np.float64), want[:, :3].astype(np.float64)
        err = np.abs(a - b).max(axis=1)
        scale = np.abs(b).max(axis=1)
        rel = np.where(scale > 0, err / np.where(scale > 0, scale, 1.0), np.where(err > 0, np.inf, 0.0))
        report = {"max_rel": float(rel.max()), "identical": float(np.mean(got[:, :3] == want[:, :3]))}
        assert report["max_rel"] <= 1e-4, report
    else:
        a = got[:, :3].view(np.uint16).astype(np.int64)
        b = want[:, :3].view(np.uint16).astype(np.int64)
        ulps = np.abs(a - b)
        report = {"max_ulp": int(ulps.max()), "identical": float((ulps == 0).mean())}
        assert report["max_ulp"] <= 1 and report["identical"] >= 0.995, report
    assert np.all(got[:, 3] == 1.0)
    return report


def check_levels_against_oracle(fmt, got, w, levels, samples, ranges=None):
    """Every level of a chain against the float oracle on its own source level (ranges: level -> row ranges)."""
    offs = datum_b200.level_offsets(w, w, levels)
    for level in range(1, levels):
        ws = w >> (level - 1)
        src, out = got[offs[level - 1]:offs[level]], got[offs[level]:offs[level + 1]]
        for a, b in (ranges or {}).get(level, [(0, 6 * (ws >> 1))]):
            float_parity.check_float_level(out[:, :3] if fmt == F32 else None, out if fmt == F16 else None, src, ws, ws, level, levels, samples, row_begin=a, row_end=b)


def check_shared_bake(fmt, got, want, chain, w, levels):
    """Level 0 byte-identical to the input, the other levels close to the one-device chain."""
    offs = datum_b200.level_offsets(w, w, levels)
    assert np.array_equal(got[: offs[1]].view(np.uint8), chain[: offs[1]].view(np.uint8))
    return check_close(fmt, got[offs[1]:], want[offs[1]:])


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("devices", device_lists())
def test_one_float_probe_shared_by_a_device_list(fctx, fmt, devices):
    """BASELINE config 3's mechanism on a small float probe: 192^2 faces, 7 levels, 256 spp (6 * (192 >> L) rows
    divide by 2 and by 3 at every split level), baked twice on one MultiContext (payloads and arrival counters
    reused)."""
    w, levels, samples = 192, 7, 256
    want = one_device(fctx, fmt, w, levels, samples, probe=81)

    bakes = []
    with datum_b200.MultiContext(devices) as multi:
        for rep in range(2):
            chain = float_chain(fmt, w, levels, probe=81)
            got = chain.copy()
            multi.buildmips_cube_float(fmt, w, w, levels, got, samples)
            print(devices, check_shared_bake(fmt, got, want, chain, w, levels))
            bakes.append(got)

    assert np.array_equal(bakes[0].view(np.uint8), bakes[1].view(np.uint8))      # deterministic
    check_levels_against_oracle(fmt, bakes[0], w, levels, samples)


@pytest.mark.parametrize("fmt", [F32, F16])
def test_shared_float_probe_with_an_odd_source_level(fctx, fmt):
    """101^2 faces over 3 levels: level 1 reads the odd 101^2 level, which the pair kernel cannot address, so its
    15 000-texel level (two 7 500-texel slabs, pair-kernel slab sizes) runs the shared tail kernel in its
    non-projective form; level 2 (two slabs of 25^2 x 3) runs its projective form."""
    w, levels, samples = 101, 3, 256
    want = one_device(fctx, fmt, w, levels, samples, probe=82)
    chain = float_chain(fmt, w, levels, probe=82)
    got = chain.copy()
    with datum_b200.MultiContext([0, 0]) as multi:
        multi.buildmips_cube_float(fmt, w, w, levels, got, samples)
    print(check_shared_bake(fmt, got, want, chain, w, levels))
    check_levels_against_oracle(fmt, got, w, levels, samples)


def test_baseline_config_3_float_probe_on_two_contexts(fctx):
    """2048^2 faces, 12 levels, 4096 spp in F16 shared by two contexts on one GPU: the whole chain against the
    one-device chain, level 1 on spot rows (face edges, a seam, a face centre) against the oracle."""
    w, levels, samples = 2048, 12, 4096
    chain = float_chain(F16, w, levels, probe=1)
    want = chain.copy()
    fctx.buildmips_cube_float(F16, w, w, levels, want, samples)
    got = torch.from_numpy(chain).pin_memory()
    with datum_b200.MultiContext([0, 0]) as multi:
        multi.buildmips_cube_float(F16, w, w, levels, got, samples)
    got = got.numpy()
    print(check_shared_bake(F16, got, want, chain, w, levels))

    hd = w >> 1
    offs = datum_b200.level_offsets(w, w, levels)
    # 4096 samples: the oracle's sequential sum moves about 1 % of the values across a binary16 rounding
    # boundary (test_float_chain_gpu.py, config 3 level 1): within 1 ulp, 98 % identical
    for a, b in [(0, 2), (hd - 1, hd + 1), (2 * hd + hd // 2, 2 * hd + hd // 2 + 2), (6 * hd - 2, 6 * hd)]:
        float_parity.check_float_level(None, got[offs[1]:offs[2]], got[: offs[1]], w, w, 1, levels, samples, row_begin=a, row_end=b, min_identical=0.98)


# ---- the C ABI directly: two contexts on one GPU, torch buffers as chains and flag blocks --------------

def level_buffers(fmt, w, probe):
    """(source level on the device, host copy, destination texels) of a w x w -> w/2 x w/2 level."""
    src = float_chain(fmt, w, 1, probe)
    return torch.from_numpy(src).to(DEV), src, 6 * (w >> 1) * (w >> 1)


@pytest.mark.parametrize("fmt", [F32, F16])
@pytest.mark.parametrize("w", [128, 101, 32])
def test_world_of_one_equals_the_device_entry(fctx, fmt, w):
    """world 1, no flags: the bytes of prefilter_level_float_device (pair kernel, odd source, tail kernel)."""
    levels, samples = 4, 256
    d_src, _, n = level_buffers(fmt, w, probe=83)
    want = torch.zeros((n, 4), dtype=TORCH_DTYPE[fmt], device=DEV)
    got = torch.full((n, 4), 7.0, dtype=TORCH_DTYPE[fmt], device=DEV)
    fctx.prefilter_level_float_device(fmt, d_src, w, w, 1, levels, samples, 0, 6 * (w >> 1), want)
    torch.cuda.synchronize()
    fctx.prefilter_level_float_peers(fmt, d_src.data_ptr(), w, w, 1, levels, samples, 0, 6 * (w >> 1), 0, 1, [got.data_ptr()])
    fctx.synchronize()
    assert np.array_equal(got.cpu().numpy().view(np.uint8), want.cpu().numpy().view(np.uint8))


@pytest.mark.parametrize("fmt", [F32, F16])
def test_two_ranks_one_with_an_empty_slab(fmt):
    """Two contexts on cuda:0 split a level through the C ABI: first one rank takes every row and the other's
    slab is empty (it still arrives), then the rows are split evenly.  Both chains hold the same bytes; the
    first split equals the one-context level, the even split is within the bounds."""
    w, levels, samples = 128, 4, 256
    a, b = datum_b200.IblContext(0), datum_b200.IblContext(0)
    try:
        for c in (a, b):
            c.set_peer_timeout_ms(10000)           # a defect fails in seconds, not after the default 60 s
        d_src, _, n = level_buffers(fmt, w, probe=84)
        rows = 6 * (w >> 1)
        want = torch.zeros((n, 4), dtype=TORCH_DTYPE[fmt], device=DEV)
        a.prefilter_level_float_device(fmt, d_src, w, w, 1, levels, samples, 0, rows, want)
        a.synchronize()
        want = want.cpu().numpy()

        dst = [torch.zeros((n, 4), dtype=TORCH_DTYPE[fmt], device=DEV) for _ in range(2)]
        flags = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(2)]      # 256-byte flag blocks
        torch.cuda.synchronize()
        dst_addr = [t.data_ptr() for t in dst]
        flag_addr = [t.data_ptr() for t in flags]

        for epoch, (split_a, split_b) in ((1, ((0, rows), (rows, rows))), (2, ((0, rows // 2), (rows // 2, rows)))):
            for t in dst:
                t.zero_()
            torch.cuda.synchronize()
            a.prefilter_level_float_peers(fmt, d_src.data_ptr(), w, w, 1, levels, samples, split_a[0], split_a[1], 0, 2, dst_addr, flag_addr, epoch)
            b.prefilter_level_float_peers(fmt, d_src.data_ptr(), w, w, 1, levels, samples, split_b[0], split_b[1], 1, 2, dst_addr, flag_addr, epoch)
            a.synchronize()
            b.synchronize()
            got = [t.cpu().numpy() for t in dst]
            assert np.array_equal(got[0].view(np.uint8), got[1].view(np.uint8)), epoch
            if epoch == 1:
                assert np.array_equal(got[0].view(np.uint8), want.view(np.uint8))
            else:
                print(check_close(fmt, got[0], want))
    finally:
        a.close()
        b.close()


# ---- two PROCESSES on one GPU: dist.PeerChain with a float format through CUDA IPC ---------------------

def _ipc_worker(rank, world, port, w, levels, samples, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # plumbing only: the 64-byte IPC handles
    try:
        torch.cuda.set_device(0)
        ctx = datum_b200.IblContext(0)
        ctx.set_peer_timeout_ms(30000)
        for fmt in (F32, F16):
            shared = ibl_dist.PeerChain(ctx, w, w, levels, fmt=fmt)
            assert shared.chain.dtype == TORCH_DTYPE[fmt] and shared.chain.shape == (shared.words, 4)
            for probe in (86, 85):
                with torch.cuda.stream(ctx.torch_stream()):
                    shared.chain.copy_(torch.from_numpy(float_chain(fmt, w, levels, probe)), non_blocking=False)
                    shared.bake(samples)
                    fused = shared.chain.clone()
                ctx.synchronize()
            np.save(os.path.join(out_dir, "ipc_chain_%d_%d.npy" % (fmt, rank)), fused.cpu().numpy())
            shared.close()
        ctx.close()
    finally:
        dist.destroy_process_group()


def test_two_processes_on_one_gpu_share_a_float_probe_through_ipc(tmp_path, fctx):
    """dist.PeerChain(fmt=FORMAT_F32 / FORMAT_F16) with both ranks on cuda:0: the chains of the two processes
    are byte-identical and close to the one-device chain."""
    w, levels, samples = 192, 7, 256
    mp.spawn(_ipc_worker, args=(2, free_port(), w, levels, samples, str(tmp_path)), nprocs=2, join=True)

    for fmt in (F32, F16):
        want = one_device(fctx, fmt, w, levels, samples, probe=85)
        a, b = np.load(tmp_path / ("ipc_chain_%d_0.npy" % fmt)), np.load(tmp_path / ("ipc_chain_%d_1.npy" % fmt))
        assert a.dtype == NP_DTYPE[fmt]
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))         # both ranks hold the same complete chain
        print(fmt, check_shared_bake(fmt, a, want, float_chain(fmt, w, levels, probe=85), w, levels))


# ---- bad input: rejected before any launch ----------------------------------------------------------

def test_bad_input_is_rejected_before_any_launch(fctx):
    w, levels, samples = 32, 3, 64
    d_src, _, n = level_buffers(F32, w, probe=87)
    dst = [torch.zeros((n, 4), dtype=torch.float32, device=DEV) for _ in range(2)]
    flags = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(2)]
    torch.cuda.synchronize()
    src, rows = d_src.data_ptr(), 6 * (w >> 1)
    dsts, flag_addr = [t.data_ptr() for t in dst], [t.data_ptr() for t in flags]
    launches = fctx.launch_count

    def rejected(fmt=F32, samples=samples, rank=0, world=2, dst_addr=None, flag_addr=flag_addr, epoch=1, why=""):
        with pytest.raises(datum_b200.IblError, match=why):
            fctx.prefilter_level_float_peers(fmt, src, w, w, 1, levels, samples, 0, rows // 2, rank, world, dst_addr or dsts, flag_addr, epoch)

    rejected(fmt=5, why="unknown format")
    rejected(fmt=datum_b200.FORMAT_RGBE, why="unknown format")
    rejected(samples=4097, why="bad level/levels/samples")
    rejected(dst_addr=[dsts[0], dsts[1] + 8], why="misaligned")       # half an F32 texel
    rejected(fmt=F16, dst_addr=[dsts[0], dsts[1] + 4], why="misaligned")
    rejected(rank=2, why="bad rank/world")
    rejected(world=9, dst_addr=dsts * 4 + dsts[:1], flag_addr=flag_addr * 4 + flag_addr[:1], why="bad rank/world")
    rejected(epoch=0, why="epochs start at 1")
    rejected(dst_addr=[dsts[0], None], why="null pointer for a rank")
    rejected(flag_addr=[flag_addr[0], None], why="null pointer for a rank")

    with datum_b200.MultiContext([0, 0]) as multi:
        texels = datum_b200.level_offsets(w, w, levels)[-1]
        with pytest.raises(ValueError):      # wrong dtype
            multi.buildmips_cube_float(F16, w, w, levels, np.zeros((texels, 4), np.float32), samples)
        with pytest.raises(ValueError):
            multi.buildmips_cube_float(F32, w, w, levels, torch.zeros((texels, 4), dtype=torch.float16), samples)
        with pytest.raises(ValueError):      # too small
            multi.buildmips_cube_float(F32, w, w, levels, np.zeros((texels - 1, 4), np.float32), samples)
        with pytest.raises(ValueError):      # unknown format
            multi.buildmips_cube_float(5, w, w, levels, np.zeros((texels, 4), np.float32), samples)
        with pytest.raises(datum_b200.IblError, match="bad width/height/levels/samples"):
            multi.buildmips_cube_float(F32, w, w, levels, np.zeros((texels, 4), np.float32), 4097)

    torch.cuda.synchronize()
    assert fctx.launch_count == launches
