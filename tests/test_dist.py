"""Multi-rank sharding logic of datum_b200/dist.py.

CPU leg: world_size 2 over gloo, with an ORACLE-backed engine defined here in the
tests (the product engine is CUDA-only), checks partitioning, slab exchange and the
SH9 all-reduce against a single-process bake.  GPU leg: the same through NCCL with
the CUDA engine when two GPUs are visible."""

import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle_lib
from datum_b200 import dist as ibl_dist
from datum_b200 import synth, level_offsets, FORMAT_F32


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class OracleEngine:
    """TEST-ONLY engine: CPU tensors, slabs computed by the oracle."""

    def prefilter_level(self, src, ws, hs, level, levels, samples, row_begin, row_end, dst):
        words, _ = oracle_lib.prefilter_level(src.numpy().view(np.uint32), ws, hs, level, levels, samples, row_begin, row_end, threads=2)
        wd = ws >> 1
        dst[row_begin * wd:row_end * wd] = torch.from_numpy(words.view(np.int32)[row_begin * wd:row_end * wd].copy())

    def sh9_partial(self, level0, fmt, width, height, row_begin, row_end):
        return torch.from_numpy(oracle_lib.sh9_partial(level0.numpy(), fmt, width, height, row_begin, row_end))

    def sh9_finish(self, partial):
        return oracle_lib.sh9_finish(partial.numpy())


def _cpu_worker(rank, world, port, w, levels, samples, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        bits = synth.synthetic_chain(w, w, levels, probe=41)
        chain = torch.from_numpy(bits.view(np.int32).copy())
        ibl_dist.bake_single_probe(OracleEngine(), chain, w, w, levels, samples, min_split_texels=6 * 2 * 2)
        np.save(os.path.join(out_dir, "chain_%d.npy" % rank), chain.numpy().view(np.uint32))

        cube = torch.from_numpy(synth.synthetic_cube(16, 16, probe=42))
        sh = ibl_dist.project_sh9_single_probe(OracleEngine(), cube, FORMAT_F32, 16, 16)
        np.save(os.path.join(out_dir, "sh_%d.npy" % rank), sh)
    finally:
        dist.destroy_process_group()


def test_plan_splits_big_levels_and_replicates_the_tail():
    plan = ibl_dist.plan_single_probe(2048, 2048, 12, 8)       # BASELINE config 3
    assert [s["level"] for s in plan] == list(range(1, 12))
    assert plan[0]["split"] and plan[0]["rows"] == 6 * 1024 and plan[0]["ranges"][7] == (7 * 768, 8 * 768)
    assert all(s["split"] for s in plan[:5]) and not any(s["split"] for s in plan[6:])   # faces <= 32^2: redundant
    for s in plan:
        covered = sorted(set(s["ranges"]))
        assert covered[0][0] == 0 and covered[-1][1] == s["rows"]
    assert not any(s["split"] for s in ibl_dist.plan_single_probe(512, 512, 8, 1))
    # rows not divisible by the world size: computed whole everywhere
    assert not ibl_dist.plan_single_probe(40, 40, 3, 7)[0]["split"]


def test_row_and_probe_sharding_cover_everything_once():
    for rows, world in ((6144, 8), (24, 5), (3, 8), (0, 2)):
        ranges = ibl_dist.split_rows(rows, world)
        assert len(ranges) == world and ranges[0][0] == 0 and ranges[-1][1] == rows
        assert all(a[1] == b[0] for a, b in zip(ranges[:-1], ranges[1:]))
        assert max(e - b for b, e in ranges) - min(e - b for b, e in ranges) <= 1
    owned = [ibl_dist.shard_probes(256, r, 8) for r in range(8)]
    assert sorted(sum(owned, [])) == list(range(256)) and all(len(o) == 32 for o in owned)


def test_two_ranks_reproduce_the_single_process_bake(tmp_path):
    w, levels, samples = 16, 5, 64
    mp.spawn(_cpu_worker, args=(2, free_port(), w, levels, samples, str(tmp_path)), nprocs=2, join=True)

    want = synth.synthetic_chain(w, w, levels, probe=41)
    oracle_lib.buildmips_cube_ibl(w, w, levels, want, samples=samples)
    for rank in range(2):
        got = np.load(tmp_path / ("chain_%d.npy" % rank))
        assert np.array_equal(got, want)                         # every rank ends with the complete chain

    cube = synth.synthetic_cube(16, 16, probe=42)
    want_sh = oracle_lib.project_sh9(cube, FORMAT_F32, 16, 16)
    for rank in range(2):
        assert np.allclose(np.load(tmp_path / ("sh_%d.npy" % rank)), want_sh, rtol=1e-12)


# ---- NCCL leg ------------------------------------------------------------------------

def _gpu_worker(rank, world, port, w, levels, samples, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import datum_b200
        ctx = datum_b200.IblContext(rank)
        engine = ibl_dist.CudaEngine(ctx)
        bits = synth.synthetic_chain(w, w, levels, probe=43)
        chain = engine.words_tensor(bits)
        ibl_dist.bake_single_probe(engine, chain, w, w, levels, samples)
        np.save(os.path.join(out_dir, "chain_%d.npy" % rank), engine.to_numpy_words(chain))

        cube = torch.from_numpy(synth.synthetic_cube(128, 128, probe=44)).to(engine.device)
        sh = ibl_dist.project_sh9_single_probe(engine, cube, FORMAT_F32, 128, 128)
        np.save(os.path.join(out_dir, "sh_%d.npy" % rank), sh)

        # the same probe through peer-mapped payloads: slabs stored into the peer's chain by the
        # kernel epilogue, barrier kernel between levels, no collective; twice, to reuse the chains
        shared = ibl_dist.PeerChain(ctx, w, w, levels)
        for probe in (45, 43):
            with torch.cuda.stream(ctx.torch_stream()):
                shared.chain.copy_(torch.from_numpy(synth.synthetic_chain(w, w, levels, probe=probe).view(np.int32)), non_blocking=False)
                shared.bake(samples)
                fused = shared.chain.clone()
            ctx.synchronize()
        np.save(os.path.join(out_dir, "fused_%d.npy" % rank), fused.cpu().numpy().view(np.uint32))
        shared.close()

        # the projection the same way: partial sums stored into the peer's array by the kernel, barrier kernel
        peer_sh = ibl_dist.PeerSh9(ctx)
        peer_sh.project(torch.from_numpy(synth.synthetic_cube(128, 128, probe=46)).to(engine.device), FORMAT_F32, 128, 128)
        np.save(os.path.join(out_dir, "sh_peer_%d.npy" % rank), peer_sh.project(cube, FORMAT_F32, 128, 128))
        peer_sh.close()
        ctx.close()
    finally:
        dist.destroy_process_group()


# The NCCL leg needs two distinct GPUs (NCCL refuses two ranks on one device): it skips on a one-GPU box,
# where the shared-probe machinery is covered by the IPC test below and by tests/test_multi_gpu.py (two
# contexts on one GPU); every multi-GPU configuration is also run and parity-checked by `bench.py --gpus N`
# (configs C3, C4, C5 of its JSON line).
@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_two_gpus_split_one_probe_over_nccl(tmp_path, ctx):
    w, levels, samples = 256, 9, 256
    mp.spawn(_gpu_worker, args=(2, free_port(), w, levels, samples, str(tmp_path)), nprocs=2, join=True)

    want = synth.synthetic_chain(w, w, levels, probe=43)
    ctx.image_buildmips_cube_ibl(w, w, levels, want, samples)      # single GPU, same kernels
    a, b = np.load(tmp_path / "chain_0.npy"), np.load(tmp_path / "chain_1.npy")
    assert np.array_equal(a, b)                                    # both ranks hold the same complete chain
    # slabs tile the level differently from one full launch (other warp split, other same-face
    # sample counts), so fp32 sums may differ in the last bit: packed-word criterion
    offs = level_offsets(w, w, levels)
    assert np.array_equal(a[: offs[1]], want[: offs[1]])
    stats = oracle_lib.word_stats(a[offs[1]:], want[offs[1]:])
    assert oracle_lib.words_within_one_code(stats, 0.99), stats

    # peer stores: the same slabs, the same kernels -> the same words as the all-gather path
    assert np.array_equal(np.load(tmp_path / "fused_0.npy"), a)
    assert np.array_equal(np.load(tmp_path / "fused_1.npy"), a)

    cube = synth.synthetic_cube(128, 128, probe=44)
    want_sh = oracle_lib.project_sh9(cube, FORMAT_F32, 128, 128)
    for rank in range(2):
        got = np.load(tmp_path / ("sh_%d.npy" % rank))
        assert np.abs(got - want_sh).max() <= 1e-4 * np.abs(want_sh).max()
        peer = np.load(tmp_path / ("sh_peer_%d.npy" % rank))
        assert np.abs(peer - want_sh).max() <= 1e-4 * np.abs(want_sh).max()
    assert np.array_equal(np.load(tmp_path / "sh_peer_0.npy"), np.load(tmp_path / "sh_peer_1.npy"))   # rows added in rank order on every rank


# ---- two PROCESSES sharing one GPU: the IPC path of PeerChain / PeerSh9 on a one-GPU box ----------

def _ipc_worker(rank, world, port, w, levels, samples, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # plumbing only: the 64-byte IPC handles
    try:
        import datum_b200
        torch.cuda.set_device(0)
        ctx = datum_b200.IblContext(0)
        ctx.set_peer_timeout_ms(30000)
        shared = ibl_dist.PeerChain(ctx, w, w, levels)
        for probe in (45, 43):
            with torch.cuda.stream(ctx.torch_stream()):
                shared.chain.copy_(torch.from_numpy(synth.synthetic_chain(w, w, levels, probe=probe).view(np.int32)), non_blocking=False)
                shared.bake(samples)
                fused = shared.chain.clone()
            ctx.synchronize()
        np.save(os.path.join(out_dir, "ipc_chain_%d.npy" % rank), fused.cpu().numpy().view(np.uint32))
        shared.close()

        cube = torch.from_numpy(synth.synthetic_cube(128, 128, probe=44)).to("cuda:0")
        peer_sh = ibl_dist.PeerSh9(ctx)
        peer_sh.project(torch.from_numpy(synth.synthetic_cube(128, 128, probe=46)).to("cuda:0"), FORMAT_F32, 128, 128)
        np.save(os.path.join(out_dir, "ipc_sh_%d.npy" % rank), peer_sh.project(cube, FORMAT_F32, 128, 128))
        peer_sh.close()
        ctx.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_processes_on_one_gpu_share_a_probe_through_ipc(tmp_path, ctx):
    """The multi-process shared-probe path (payloads mapped through CUDA IPC handles, slabs stored into the
    peer's payload by the prefilter kernel, arrival counters + stream waits) with BOTH ranks on cuda:0: what a
    one-GPU box can run of `bench.py --gpus N`'s config 3 / 5 machinery.  Two GPUs run the same through NCCL
    and NVLink in test_two_gpus_split_one_probe_over_nccl."""
    w, levels, samples = 192, 7, 256
    mp.spawn(_ipc_worker, args=(2, free_port(), w, levels, samples, str(tmp_path)), nprocs=2, join=True)

    want = synth.synthetic_chain(w, w, levels, probe=43)
    ctx.image_buildmips_cube_ibl(w, w, levels, want, samples)
    a, b = np.load(tmp_path / "ipc_chain_0.npy"), np.load(tmp_path / "ipc_chain_1.npy")
    assert np.array_equal(a, b)                                    # both ranks hold the same complete chain
    offs = level_offsets(w, w, levels)
    assert np.array_equal(a[: offs[1]], want[: offs[1]])
    stats = oracle_lib.word_stats(a[offs[1]:], want[offs[1]:])
    assert oracle_lib.words_within_one_code(stats, 0.995), stats

    cube = synth.synthetic_cube(128, 128, probe=44)
    want_sh = oracle_lib.project_sh9(cube, FORMAT_F32, 128, 128)
    sh0, sh1 = np.load(tmp_path / "ipc_sh_0.npy"), np.load(tmp_path / "ipc_sh_1.npy")
    assert np.array_equal(sh0, sh1)
    assert np.abs(sh0 - want_sh).max() <= 1e-4 * np.abs(want_sh).max()
