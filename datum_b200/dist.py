"""Multi-GPU sharding of the IBL bake: one process per GPU over torch.distributed.

The reference has no parallelism at all (the bake is a single-threaded triple
loop, tools/ibl.cpp:263-272).  Three ways the path shards (SURVEY.md §8e):

  probes   a batch of independent environment maps: probe p -> rank p % world,
           every rank runs the full chain (+ SH9) locally.  NO collective.
  rows     ONE probe split across ranks: inside a level every output row is
           independent, but level L reads ALL of level L-1 (tools/ibl.cpp:249,
           274), so after each split level the ranks all-gather their row slabs
           (NCCL over NVLink).  Tail levels are cheaper to compute redundantly
           than to exchange.
  sh9      the projection of one probe split by rows: 27 partial sums + the
           weight sum, one all-reduce of 28 doubles, then project.comp:99-105.

The collectives are issued on the bake context's own stream (CudaEngine.stream),
so they are ordered with the kernels without host synchronisation.

`engine` is the object that runs one level slab / one SH9 slab.  The product
engine is CudaEngine (libdatum_ibl_cuda; raises without a GPU).  The CPU tests
pass their own oracle-backed engine over the gloo backend to exercise this
file's partitioning and exchange logic — that engine lives in tests/, not here.
"""

import contextlib

import numpy as np

from . import ibl


def split_rows(rows, world):
    """Contiguous, near-equal row ranges: [(begin, end)] * world (some may be empty)."""
    base, extra = divmod(rows, world)
    ranges, begin = [], 0
    for r in range(world):
        end = begin + base + (1 if r < extra else 0)
        ranges.append((begin, end))
        begin = end
    return ranges


def shard_probes(count, rank, world):
    """Probe ids owned by `rank`: p % world == rank."""
    return list(range(rank, count, world))


# Levels of at most this many texels are computed by every GPU instead of being exchanged.
MIN_SPLIT_TEXELS = 6 * 16 * 16


def plan_single_probe(width, height, levels, world, min_split_texels=MIN_SPLIT_TEXELS):
    """Per level >= 1: how the 6*(h>>L) destination rows are shared.

    A level is split when its row count divides evenly by the world size (equal
    slabs keep the exchange a plain all-gather) and it has more than
    `min_split_texels` texels; otherwise every rank computes it whole."""
    plan = []
    for level in range(1, levels):
        ws, hs = width >> (level - 1), height >> (level - 1)
        wd, hd = ws >> 1, hs >> 1
        rows = 6 * hd
        split = world > 1 and rows % world == 0 and rows * wd > min_split_texels
        plan.append({
            "level": level, "ws": ws, "hs": hs, "wd": wd, "hd": hd, "rows": rows, "split": split,
            "ranges": split_rows(rows, world) if split else [(0, rows)] * world,
        })
    return plan


class CudaEngine:
    """Runs slabs on one GPU through libdatum_ibl_cuda."""

    def __init__(self, ctx):
        import torch
        self.torch = torch
        self.ctx = ctx
        self.device = torch.device("cuda", ctx.device)

    def stream(self):
        return self.torch.cuda.stream(self.ctx.torch_stream())

    def words_tensor(self, bits):
        """uint32 payload (numpy) -> int32 device tensor"""
        return self.torch.from_numpy(np.ascontiguousarray(bits).view(np.int32)).to(self.device)

    def to_numpy_words(self, t):
        self.ctx.synchronize()
        return t.cpu().numpy().view(np.uint32)

    def prefilter_level(self, src, ws, hs, level, levels, samples, row_begin, row_end, dst):
        self.ctx.prefilter_level_device(src, ws, hs, level, levels, samples, row_begin, row_end, dst)

    def sh9_partial(self, level0, fmt, width, height, row_begin, row_end):
        out = self.torch.zeros(28, dtype=self.torch.float64, device=self.device)
        self.ctx.sh9_partial_device(level0, fmt, width, height, row_begin, row_end, out)
        return out

    def sh9_finish(self, partial):
        self.ctx.synchronize()
        return self.ctx.sh9_finish(partial.cpu().numpy())


def _world(group):
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return dist, 0, 1
    return dist, dist.get_rank(group), dist.get_world_size(group)


def bake_single_probe(engine, chain, width, height, levels, samples=1024, group=None, min_split_texels=MIN_SPLIT_TEXELS):
    """tools/ibl.cpp:242-279 for ONE probe shared by all ranks of `group`.

    `chain` is the payload tensor on the engine's device (int32 words, level 0
    filled on every rank); on return every rank holds the complete chain."""
    dist, rank, world = _world(group)
    offs = ibl.level_offsets(width, height, levels)
    plan = plan_single_probe(width, height, levels, world, min_split_texels)

    ctxmgr = engine.stream() if hasattr(engine, "stream") else contextlib.nullcontext()
    with ctxmgr:
        for step in plan:
            level = step["level"]
            src = chain[offs[level - 1]:offs[level]]
            dst = chain[offs[level]:offs[level + 1]]
            begin, end = step["ranges"][rank]

            engine.prefilter_level(src, step["ws"], step["hs"], level, levels, samples, begin, end, dst)

            if step["split"]:
                # equal slabs: one all-gather straight into the level (the local slab is copied
                # first so that input and output of the collective do not alias)
                wd = step["wd"]
                slab = dst[begin * wd:end * wd].clone()
                dist.all_gather_into_tensor(dst, slab, group=group)

    return chain


class _DeviceArray:
    """A range of device memory owned by someone else, for torch.as_tensor (CUDA array interface)."""

    def __init__(self, address, count, typestr="<i4"):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": typestr, "data": (address, False), "version": 3, "strides": None}


class PeerChain:
    """One probe's payload on every GPU of the group, each mapped into every process.

    The payload (and a small flag array) is allocated by libdatum_ibl_cuda
    (datum_ibl_peer_alloc), the 64-byte IPC handles travel once through
    torch.distributed (all_gather_object: plumbing, not data path), and every rank
    maps its peers' allocations.  bake() then needs no collective: the prefilter
    kernel's epilogue stores each slab into all chains over NVLink and a one-CTA
    stream memory wait on the arrival counters separates the levels.

    `fmt`: ibl.FORMAT_RGBE (the default: `chain` is a flat int32 tensor of rgbe
    words) or a float chain's ibl.FORMAT_F32 / ibl.FORMAT_F16 (`chain` is a
    (texels, 4) float32 / float16 tensor, baked without rgbe re-quantisation)."""

    FLAG_BYTES = 256

    _TYPESTR = {ibl.FORMAT_RGBE: "<i4", ibl.FORMAT_F32: "<f4", ibl.FORMAT_F16: "<f2"}

    def __init__(self, ctx, width, height, levels, group=None, fmt=ibl.FORMAT_RGBE):
        import torch
        self.torch = torch
        self.ctx = ctx
        self.group = group
        self.dist, self.rank, self.world = _world(group)
        if self.world > 8:
            raise ValueError("a probe is shared by at most 8 GPUs (one NVSwitch domain)")
        if fmt not in self._TYPESTR:
            raise ValueError("unknown texel format %r" % (fmt,))
        self.width, self.height, self.levels = width, height, levels
        self.fmt = fmt
        self.texel_bytes = ibl.TEXEL_BYTES[fmt]
        self.offs = ibl.level_offsets(width, height, levels)
        self.words = self.offs[-1]          # texels of the chain (rgbe: words)
        self.epoch = 0

        # flags first (256 B), then the chain
        self.local, handle = ctx.peer_alloc(self.FLAG_BYTES + self.texel_bytes * self.words)
        self.bases = [None] * self.world
        self.bases[self.rank] = self.local
        if self.world > 1:
            handles = [None] * self.world
            self.dist.all_gather_object(handles, handle, group=group)
            for r in range(self.world):
                if r != self.rank:
                    self.bases[r] = ctx.peer_open(handles[r])
        if fmt == ibl.FORMAT_RGBE:
            self.chain = torch.as_tensor(_DeviceArray(self.local + self.FLAG_BYTES, self.words), device=torch.device("cuda", ctx.device))
        else:
            self.chain = torch.as_tensor(_DeviceArray(self.local + self.FLAG_BYTES, 4 * self.words, self._TYPESTR[fmt]), device=torch.device("cuda", ctx.device)).view(self.words, 4)

    def chain_address(self, rank):
        return self.bases[rank] + self.FLAG_BYTES

    def barrier(self):
        self.epoch += 1
        self.ctx.peer_barrier(self.rank, self.world, self.bases, self.epoch)

    def bake(self, samples=1024, min_split_texels=MIN_SPLIT_TEXELS):
        """tools/ibl.cpp:242-279 for the probe whose level 0 every rank has put into `self.chain`;
        on return (asynchronously, on the context's stream) every rank holds the whole chain.
        One launch per split level: the kernel stores its slab into every chain, its last CTA tells
        the peers, the stream waits for their arrivals."""
        plan = plan_single_probe(self.width, self.height, self.levels, self.world, min_split_texels)

        # nobody may still be reading the previous probe out of this chain, or lag a whole bake behind
        if self.world > 1:
            self.barrier()

        tb = self.texel_bytes
        for step in plan:
            level = step["level"]
            src = self.chain_address(self.rank) + tb * self.offs[level - 1]
            begin, end = step["ranges"][self.rank]

            if step["split"]:
                self.epoch += 1
                dst = [self.chain_address(r) + tb * self.offs[level] for r in range(self.world)]
                self._level(src, step, level, samples, begin, end, self.rank, self.world, dst, self.bases, self.epoch)
            else:
                dst = self.chain_address(self.rank) + tb * self.offs[level]
                self._level(src, step, level, samples, begin, end, 0, 1, [dst])

        return self.chain

    def _level(self, src, step, level, samples, begin, end, rank, world, dst, flags=None, epoch=0):
        if self.fmt == ibl.FORMAT_RGBE:
            self.ctx.prefilter_level_peers(src, step["ws"], step["hs"], level, self.levels, samples, begin, end, rank, world, dst, flags, epoch)
        else:
            self.ctx.prefilter_level_float_peers(self.fmt, src, step["ws"], step["hs"], level, self.levels, samples, begin, end, rank, world, dst, flags, epoch)

    def close(self):
        self.ctx.synchronize()
        if self.world > 1:
            self.dist.barrier(group=self.group)      # no peer may still be storing into a chain that goes away
        self.chain = None
        for r in range(self.world):
            if r != self.rank and self.bases[r] is not None:
                self.ctx.peer_close(self.bases[r])
        self.ctx.peer_free(self.local)
        self.bases = []


class PeerSh9:
    """SH9 of one cube shared by the GPUs of the group without a collective: every rank's arrays of
    (world x 28) partial sums are mapped into every process; the projection kernel's last block stores
    the slab's sums into row [rank] of all of them, ONE barrier kernel follows, and every rank adds the
    rows in rank order (deterministic, the same bits on every rank).  Two arrays alternate between
    calls: a fast rank may already be storing the next projection while a slow one still reads this
    one, and it cannot get two projections ahead because of the barrier in between."""

    FLAG_BYTES = 256

    def __init__(self, ctx, group=None):
        import torch
        self.torch = torch
        self.ctx = ctx
        self.group = group
        self.dist, self.rank, self.world = _world(group)
        if self.world > 8:
            raise ValueError("a cube is shared by at most 8 GPUs (one NVSwitch domain)")
        self.epoch = 0
        self.array_bytes = 8 * 28 * self.world
        self.local, handle = ctx.peer_alloc(self.FLAG_BYTES + 2 * self.array_bytes)
        self.bases = [None] * self.world
        self.bases[self.rank] = self.local
        if self.world > 1:
            handles = [None] * self.world
            self.dist.all_gather_object(handles, handle, group=group)
            for r in range(self.world):
                if r != self.rank:
                    self.bases[r] = ctx.peer_open(handles[r])
        device = torch.device("cuda", ctx.device)
        self.rows = [torch.as_tensor(_DeviceArray(self.local + self.FLAG_BYTES + k * self.array_bytes, 28 * self.world, "<f8"), device=device).view(self.world, 28) for k in range(2)]

    def enqueue(self, level0, fmt, width, height):
        """ONE launch on the context's stream (the projection kernel's last block stores the rows and
        tells the peers) + the stream's wait for their arrivals; returns the index of the array that
        will hold the rows."""
        begin, end = split_rows(6 * height, self.world)[self.rank]
        self.epoch += 1
        which = self.epoch & 1
        slots = [base + self.FLAG_BYTES + which * self.array_bytes for base in self.bases]
        self.ctx.sh9_partial_peers(level0, fmt, width, height, begin, end, self.rank, self.world, slots, self.bases if self.world > 1 else None, self.epoch)
        return which

    def project(self, level0, fmt, width, height):
        """data/project.comp:23-106; returns float32 [9][3] (the same on every rank)."""
        which = self.enqueue(level0, fmt, width, height)
        self.ctx.synchronize()
        rows = self.rows[which].cpu().numpy()
        total = np.zeros(28, np.float64)
        for r in range(self.world):
            total += rows[r]
        return self.ctx.sh9_finish(total)

    def close(self):
        self.ctx.synchronize()
        if self.world > 1:
            self.dist.barrier(group=self.group)
        self.rows = None
        for r in range(self.world):
            if r != self.rank and self.bases[r] is not None:
                self.ctx.peer_close(self.bases[r])
        self.ctx.peer_free(self.local)
        self.bases = []


def project_sh9_single_probe(engine, level0, fmt, width, height, group=None):
    """data/project.comp:23-106 for ONE level-0 cube shared by all ranks: rows split,
    28 partial sums all-reduced (the only collective), normalised on every rank."""
    dist, rank, world = _world(group)
    begin, end = split_rows(6 * height, world)[rank]

    ctxmgr = engine.stream() if hasattr(engine, "stream") else contextlib.nullcontext()
    with ctxmgr:
        partial = engine.sh9_partial(level0, fmt, width, height, begin, end)
        if world > 1:
            dist.all_reduce(partial, op=dist.ReduceOp.SUM, group=group)

    return engine.sh9_finish(partial)


def bake_probe_batch(ctx, payloads, width, height, levels, samples=1024, group=None, with_sh9=False):
    """A batch of independent probes (BASELINE config 4): this rank bakes payloads[p] for
    p % world == rank, in place, through the reference-facing host entry point.  No
    collective.  Returns {probe id: sh9 or None}."""
    _, rank, world = _world(group)
    results = {}
    for p in shard_probes(len(payloads), rank, world):
        ctx.image_buildmips_cube_ibl(width, height, levels, payloads[p], samples)
        results[p] = ctx.project_sh9(payloads[p][: 6 * width * height], ibl.FORMAT_RGBE, width, height) if with_sh9 else None
    return results
