#!/usr/bin/env python
"""Benchmark of the IBL bake hot path (BASELINE.json: prefiltered texel-samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one GGX-prefilter chain bake of one synthetic HDR environment map
(BASELINE config 2: 512^2 faces, 8 levels, 1024 samples/texel, rgbe payload as
tools/assetbuilder.cpp hands it to image_buildmips_cube_ibl) per GPU.  Probes
are independent units, so N GPUs bake N probes per step with no data-path
collective (weak scaling); the only collectives of the headline are the barrier
and the max-over-ranks of the timings.

Prints ONE JSON line on rank 0.  `value` is timed on the device (CUDA events,
max over ranks) with inputs resident in HBM; `e2e` goes through the reference-
facing entry point image_buildmips_cube_ibl with pinned HOST buffers, host<->device
copies inside the timed region.  `roofline` is the level-1 prefilter launch
(75 % of the work) against the FP32 FMA peak measured in the same process,
`roofline_sh9` the SH9 projection of one 4096^2 RGBA32F cube against the measured
HBM copy bandwidth; `cpu_baseline` is the unmodified reference tools/ibl.cpp
(compiled into oracle/_ref with the reference's own -O2 -ffast-math) on the host cores.

`configs` carries BASELINE.json's other configurations, each with its own parity flags:
  C1  the reference's bundled skybox at native size (512^2 x 8 levels): GPU end to end from the
      ARGB32 pixels, and the unmodified reference's full bake on one host core (N = 1 only);
  C3  ONE 2048^2 x 12-level x 4096-spp probe shared by all N GPUs (rows of every level split,
      slabs exchanged by NVLink peer stores from the kernel epilogue, and by NCCL all-gather);
  C4  256 probes of 256^2 x 8 levels x 1024 spp + SH9, probe p on rank p % N, no collective;
  C5  SH9 of one 4096^2 RGBA32F cube, rows split, 28 partial sums exchanged (NCCL all-reduce
      and peer stores).
  C3_one_process (N > 1)  config 3 again through the device-list entry point: rank 0 alone, after the
      other ranks have left, drives all N GPUs from one process (datum_ibl_multi_*), host buffers in and out.

`--dump-outputs DIR` saves what the last of the K timed steps baked, so that two builds can be compared
output for output: levels 1..7 of its chain (level 0 is the step's input), decoded from the rgbe words to
float32 RGB, one (6, h, w, 3) array per level as DIR/c2_level<L>.npy (DIR/c2_rank<R>_level<L>.npy with
N > 1), 6.3 MB per GPU and at most 64 MiB in all: with more than 10 GPUs a fixed, seeded sample of 10 ranks
saves theirs.  The inputs are seeded, so the same arguments bake the same probe in every run.
"""

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WIDTH, LEVELS, SAMPLES = 512, 8, 1024            # BASELINE.json configs[1]
POOL = 24                                        # distinct probes resident in HBM: 24 x 8.4 MB > 126 MB L2
FLOP_PER_TEXEL_SAMPLE = 85.0                     # SURVEY.md §8d, itemised in DESIGN.md
SH9_BYTES_PER_TEXEL = 16.0                       # SURVEY.md §8d: RGBA32F texel read once
CPU_SAMPLE = (128, 8)                            # CPU legs: one 128^2-face bake with C2's EIGHT levels (the same roughness set) per thread
SUSTAINED_SECONDS = 2.5
DUMP_BYTES = 64 * 2**20                          # --dump-outputs, all ranks together

METRIC = "prefiltered texel-samples/sec"
UNIT = "texel-samples/s"


def texel_samples(width, levels, samples):
    return sum(6 * (width >> i) * (width >> i) for i in range(1, levels)) * samples


def base_config(world):
    """The workload both arms are quoted on (identical in the two JSON lines)."""
    chain_mb = sum(6 * (WIDTH >> i) ** 2 for i in range(LEVELS)) * 4 // 2**20
    return {
        "workload": "C2: synthetic HDR cube map, 512^2 faces x 8 levels x 1024 GGX samples/texel, rgbe payload (one env map per GPU per step)",
        "texel_samples_per_step_per_gpu": texel_samples(WIDTH, LEVELS, SAMPLES),
        "levels": LEVELS, "samples_per_texel": SAMPLES,
        "parallelism": "probe-sharded x%d, no data-path collective" % world,
        "l2": "GPU arm: rotating pool of %d distinct probes per GPU (%d MB) > 126 MB L2, each step bakes the next one; CPU arm: a bounded sample per step (cpu_baseline.sample)" % (POOL, POOL * chain_mb),
    }


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback of B200_PROFILING.md"


def profiled_traffic():
    """dram__bytes_read + write per launch of the two roofline kernels, from the committed ncu
    --set full summaries (profiles/traffic.json names the capture each figure comes from)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


# ---- the reference's own CPU implementation (bounded sample) ---------------------------

def cpu_reference_run(rounds, threads=None, sample=CPU_SAMPLE):
    """`threads` concurrent calls of the UNMODIFIED reference image_buildmips_cube_ibl
    (oracle/_ref, the reference's -O2 -ffast-math flags) on synthetic chains, `rounds` times.
    The reference function is single-threaded and has no global state; using every host core
    means one independent bake per core.  Falls back to the oracle port when oracle/_ref was
    not built.  Returns (texel-samples/s, seconds, info)."""
    import oracle_lib
    from datum_b200 import synth

    threads = threads or os.cpu_count() or 1
    w, levels = sample

    if oracle_lib.have_ref(fast=True):
        lib = oracle_lib.ref(fast=True)
        kind = "reference"

        def bake(bits):
            lib.ref_image_buildmips_cube_ibl(w, w, levels, bits.ctypes.data)
    else:
        kind = "port"

        def bake(bits):
            oracle_lib.buildmips_cube_ibl(w, w, levels, bits, samples=1024, threads=1)

    payloads = [synth.synthetic_chain(w, w, levels, probe=100 + t) for t in range(threads)]

    def worker(bits):
        for _ in range(rounds):
            bake(bits)          # ctypes releases the GIL for the duration of the call

    pool = [threading.Thread(target=worker, args=(p,)) for p in payloads]
    t0 = time.perf_counter()
    for t in pool:
        t.start()
    for t in pool:
        t.join()
    dt = time.perf_counter() - t0

    work = texel_samples(w, levels, 1024) * threads * rounds
    info = {
        "kind": kind,
        "cores": threads,
        "sample": "%d concurrent %s bakes of a %d^2-face %d-level rgbe chain (C2's level count and roughness set, faces 4x smaller) at 1024 spp, x%d rounds (%.3g texel-samples, %.1f s)"
                  % (threads, "unmodified tools/ibl.cpp image_buildmips_cube_ibl" if kind == "reference" else "oracle port", w, levels, rounds, work, dt),
    }
    return work / dt, dt, info


def skybox_native_faces():
    """BASELINE config 1: the reference's bundled data/skybox_*.jpg as decoded 8-bit RGB (committed
    fixture, tests/golden/skybox512.npz) -> (6, 512, 512) ARGB32 pixels in assetbuilder's face order."""
    golden = np.load(os.path.join(ROOT, "tests", "golden", "skybox512.npz"))
    rgb = golden["faces_rgb"].astype(np.uint32)
    return (np.uint32(0xFF000000) | rgb[..., 0] << np.uint32(16) | rgb[..., 1] << np.uint32(8) | rgb[..., 2]).astype(np.uint32), golden


def cpu_c1_native():
    """One FULL bake of config 1 by the unmodified reference on one host core, as shipped
    (tools/assetbuilder.cpp:416-470: ingest, then image_buildmips_cube_ibl(512, 512, 8))."""
    import oracle_lib

    faces, _ = skybox_native_faces()
    w, levels = faces.shape[2], 8
    chain = np.zeros(sum(6 * (w >> i) ** 2 for i in range(levels)), np.uint32)
    t0 = time.perf_counter()
    chain[: 6 * w * w] = oracle_lib.ingest_cube_argb32(faces)
    if oracle_lib.have_ref(fast=True):
        oracle_lib.ref(fast=True).ref_image_buildmips_cube_ibl(w, w, levels, chain.ctypes.data)
        kind = "reference"
    else:
        oracle_lib.buildmips_cube_ibl(w, w, levels, chain, samples=1024, threads=1)
        kind = "port"
    seconds = time.perf_counter() - t0
    return {"kind": kind, "cores": 1, "seconds": seconds, "texel_samples_per_s": texel_samples(w, levels, 1024) / seconds,
            "sample": "the whole of config 1, once: six 512^2 images -> rgbe(srgba()) -> 8-level bake, one thread (the reference is single-threaded, tools/ibl.cpp:263-272)"}, chain


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0

    for _ in range(args.warmup):
        cpu_reference_run(1)

    t0 = time.perf_counter()
    value, dt, info = cpu_reference_run(max(1, args.steps))
    ms_per_step = (time.perf_counter() - t0) * 1e3 / max(1, args.steps)

    info["value"] = value
    info["unit"] = UNIT
    config = base_config(args.gpus)
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- clock sampling during the timed region ---------------------------------------------

class ClockSampler:
    """Polls SM clock and throttle reasons through NVML while the measurement runs."""

    REASONS = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
        0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost",
    }

    def __init__(self, device_index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[device_index]) if visible and visible.split(",")[device_index].isdigit() else device_index
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM))
                util = int(nv.nvmlDeviceGetUtilizationRates(self._handle).gpu)
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle))
                self.samples.append((mhz, util))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        self.samples, self.reasons = [], set()
        self._stop = threading.Event()
        if self._nvml:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
            self._thread = None
        clocks = [m for m, _ in self.samples]
        return {
            "sm_mhz": float(np.median(clocks)) if clocks else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(clocks),
        }


# ---- our arm -------------------------------------------------------------------------------

class Job:
    """Rank plumbing shared by the measurements."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))

        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — datum_b200 has no CPU path to benchmark")

        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)

        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.device)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def _reduce(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX)

    def min_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.MIN)

    def sum_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM)

    def timed(self, stream, fn, reps=3):
        """Best of `reps`: CUDA events on the bake stream around fn(), max over ranks."""
        torch = self.torch
        best = 1e30
        for _ in range(reps):
            self.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                ev0.record()
                fn()
                ev1.record()
            ev1.synchronize()
            best = min(best, self.max_over_ranks(ev0.elapsed_time(ev1)))
        return best


def config_c1(job, ctx):
    """The reference's bundled skybox at native size: GPU end to end from the ARGB32 pixels (ingest +
    bake, copies included) against the unmodified reference's level words (golden), and the
    reference's own full bake on one host core."""
    import datum_b200
    import oracle_lib

    faces, golden = skybox_native_faces()
    w, levels = faces.shape[2], 8
    offs = datum_b200.level_offsets(w, w, levels)
    bits = np.zeros(offs[-1], np.uint32)
    ctx.skybox_from_argb32(faces, levels, bits)
    best = 1e30
    for _ in range(5):
        t0 = time.perf_counter()
        ctx.skybox_from_argb32(faces, levels, bits)
        best = min(best, time.perf_counter() - t0)

    want = golden["levels"]
    stats = oracle_lib.word_stats(bits[offs[1]:], want)
    dec_got = oracle_lib.rgbe_decode_array(bits[offs[1]:])[:, :3].astype(np.float64)
    dec_ref = oracle_lib.rgbe_decode_array(want)[:, :3].astype(np.float64)
    rel = np.abs(dec_got - dec_ref).max(axis=1) / np.maximum(dec_ref.max(axis=1), 1e-30)

    cpu, cpu_chain = cpu_c1_native()
    return {
        "workload": "C1: the reference's bundled skybox, six 512^2 images -> rgbe(srgba()) -> 8 levels x 1024 spp (tools/assetbuilder.cpp:416-470)",
        "gpu_ms_e2e": best * 1e3, "gpu_api": "image_pack_cube_faces_ibl / datum_ibl_ingest_cube_argb32_ibl: pageable host pixels in, baked payload out",
        "gpu_texel_samples_per_s": texel_samples(w, levels, 1024) / best,
        "cpu_baseline_c1": cpu,
        "speedup_vs_reference_one_core": cpu["seconds"] / best,
        "words_identical_to_reference_golden": stats["identical"],
        "value_rel_err_p99": float(np.quantile(rel, 0.99)),
        "level0_identical_to_reference_ingest": bool(np.array_equal(bits[: offs[1]], cpu_chain[: offs[1]])),
        "cpu_run_equals_golden": float((cpu_chain[offs[1]:] == want).mean()),
        "parity_ok": bool(stats["identical"] >= 0.97 and np.quantile(rel, 0.99) <= 4e-3),
    }


def config_c3(job, ctx, engine, stream):
    import datum_b200
    from datum_b200 import dist as ibl_dist
    from datum_b200 import synth

    torch, device, world = job.torch, job.device, job.world
    w, levels, samples = 2048, 12, 4096
    offs = datum_b200.level_offsets(w, w, levels)
    work = texel_samples(w, levels, samples)
    level0 = torch.from_numpy(synth.synthetic_chain(w, w, 1, probe=3).view(np.int32)).to(device)

    alone = torch.zeros(offs[-1], dtype=torch.int32, device=device)
    alone[: offs[1]] = level0
    ms_alone = job.timed(stream, lambda: ctx.buildmips_cube_ibl_device(w, w, levels, alone, samples), reps=2)

    out = {
        "workload": "C3: ONE 2048^2-face x 12-level x 4096-spp probe (3.44e10 texel-samples) shared by %d GPU(s), rows of every level above 6x16^2 texels split" % world,
        "texel_samples": work, "ms_one_gpu": ms_alone, "texel_samples_per_s_one_gpu": work / ms_alone * 1e3,
    }
    if world == 1:
        return out

    shared = ibl_dist.PeerChain(ctx, w, w, levels)
    with torch.cuda.stream(stream):
        shared.chain[: offs[1]] = level0
    ms_peer = job.timed(stream, lambda: shared.bake(samples))
    ctx.synchronize()
    same_peer = job.min_over_ranks(float((shared.chain == alone).float().mean().item()))

    chain = torch.zeros(offs[-1], dtype=torch.int32, device=device)
    chain[: offs[1]] = level0
    ms_nccl = job.timed(stream, lambda: ibl_dist.bake_single_probe(engine, chain, w, w, levels, samples), reps=2)
    ctx.synchronize()
    same_nccl = job.min_over_ranks(float((chain == alone).float().mean().item()))
    peer_equals_nccl = job.min_over_ranks(1.0 if torch.equal(shared.chain, chain) else 0.0) == 1.0
    shared.close()

    out.update({
        "ms": ms_peer, "texel_samples_per_s": work / ms_peer * 1e3, "speedup_vs_one_gpu": ms_alone / ms_peer,
        "exchange": "NVLink peer stores from the prefilter kernel's epilogue + arrival counters (stream memory wait); no collective library call",
        "ms_nccl_all_gather": ms_nccl, "speedup_vs_one_gpu_nccl": ms_alone / ms_nccl,
        "words_identical_to_one_gpu": same_peer, "words_identical_to_one_gpu_nccl": same_nccl,
        "peer_stores_equal_nccl_words": bool(peer_equals_nccl),
        "parity_ok": bool(same_peer >= 0.999 and same_nccl >= 0.999),
    })
    return out


def config_c3_one_process(job, ctx):
    """Config 3 through the device-list entry point: ONE process (this rank, after the others have left)
    drives all the GPUs of the job — what DATUM_IBL_DEVICES gives a single-process assetbuilder.  End to end
    from a pinned host payload: every GPU uploads one slice of level 0 and fetches the rest from its peers, every GPU
    sends one slice of the baked chain back."""
    import datum_b200
    from datum_b200 import synth

    torch, world = job.torch, job.world
    w, levels, samples = 2048, 12, 4096
    offs = datum_b200.level_offsets(w, w, levels)
    source = synth.synthetic_chain(w, w, levels, probe=3)

    alone = torch.from_numpy(source.view(np.int32).copy()).pin_memory()
    ctx.image_buildmips_cube_ibl(w, w, levels, alone, samples)
    t0 = time.perf_counter()
    ctx.image_buildmips_cube_ibl(w, w, levels, alone, samples)
    ms_alone = (time.perf_counter() - t0) * 1e3

    shared = torch.from_numpy(source.view(np.int32).copy()).pin_memory()
    with datum_b200.MultiContext(list(range(world))) as multi:
        multi.image_buildmips_cube_ibl(w, w, levels, shared, samples)         # allocations, tables and peer mappings on every device
        best = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            multi.image_buildmips_cube_ibl(w, w, levels, shared, samples)
            best = min(best, (time.perf_counter() - t0) * 1e3)

    same = float((shared.numpy() == alone.numpy()).mean())
    return {
        "workload": "C3 from ONE process: datum_ibl_multi_buildmips_cube_ibl over devices 0..%d, pinned host payload in and out (100.7 MB up, 33.5 MB down)" % (world - 1),
        "ms_e2e": best, "ms_e2e_one_gpu": ms_alone, "speedup_e2e_vs_one_gpu": ms_alone / best,
        "texel_samples_per_s_e2e": texel_samples(w, levels, samples) / best * 1e3,
        "words_identical_to_one_gpu": same, "parity_ok": bool(same >= 0.999),
    }


def config_c4(job, ctx):
    import datum_b200
    import oracle_lib
    from datum_b200 import dist as ibl_dist
    from datum_b200 import synth

    torch, world, rank = job.torch, job.world, job.rank
    w, levels, samples, probes = 256, 8, 1024, 256
    mine = ibl_dist.shard_probes(probes, rank, world)
    hosts = [synth.synthetic_chain(w, w, levels, probe=1000 + rank * 8 + k) for k in range(8)]
    distinct = [torch.from_numpy(b.view(np.int32).copy()).pin_memory() for b in hosts]
    payloads = [distinct[i % len(distinct)] for i in range(len(mine))]
    work = texel_samples(w, levels, samples) * probes
    ctx.bake_probes(w, w, levels, payloads[:8], samples, sh9=True)
    best, sh = 1e30, None
    for _ in range(3):
        job.barrier()
        t0 = time.perf_counter()
        sh = ctx.bake_probes(w, w, levels, payloads, samples, sh9=True)
        best = min(best, job.max_over_ranks(time.perf_counter() - t0))

    # parity on this rank's first two probes: SH9 against the fp64 oracle, the chain against a single call
    n0 = 6 * w * w
    sh_err = 0.0
    for k in range(2):
        want = oracle_lib.project_sh9(hosts[k][:n0], datum_b200.FORMAT_RGBE, w, w)
        sh_err = max(sh_err, float(np.abs(sh[k] - want).max() / np.abs(want).max()))
    single = hosts[0].copy()
    ctx.image_buildmips_cube_ibl(w, w, levels, single, samples)
    chain_same = bool(np.array_equal(distinct[0].numpy().view(np.uint32), single))
    sh_err = job.max_over_ranks(sh_err)
    chain_same = job.min_over_ranks(1.0 if chain_same else 0.0) == 1.0

    return {
        "workload": "C4: %d probes of %d^2 faces x %d levels x %d spp, prefilter + SH9, probe p on rank p %% %d, one batched host call per rank (pinned payloads, copies included), no collective" % (probes, w, levels, samples, world),
        "probes": probes, "seconds": best, "probes_per_s": probes / best, "probes_per_s_per_gpu": probes / best / world,
        "texel_samples_per_s": work / best,
        "sh9_max_rel_vs_oracle": sh_err, "chain_words_equal_single_call": chain_same,
        "parity_ok": bool(sh_err <= 1e-4 and chain_same),
    }


def oracle_sh9_threads(cube, w, threads):
    """fp64 oracle of data/project.comp over a host cube, row chunks on `threads` host threads."""
    import datum_b200
    import oracle_lib

    chunks = np.linspace(0, 6 * w, threads + 1).astype(int)
    parts = [None] * threads

    def work(i):
        parts[i] = oracle_lib.sh9_partial(cube, datum_b200.FORMAT_F32, w, w, int(chunks[i]), int(chunks[i + 1]))

    pool = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in pool:
        t.start()
    for t in pool:
        t.join()
    return oracle_lib.sh9_finish(np.sum(parts, axis=0))


def config_c5(job, ctx, engine, stream):
    import datum_b200
    from datum_b200 import dist as ibl_dist

    torch, device, world, rank = job.torch, job.device, job.world, job.rank
    dist = job.dist
    w = 4096
    gen = torch.Generator(device=device)
    gen.manual_seed(5)
    cube = torch.rand((6 * w * w, 4), dtype=torch.float32, device=device, generator=gen)
    cube[:, :3] *= torch.exp2(6 * torch.rand((6 * w * w, 1), dtype=torch.float32, device=device, generator=gen) - 3)   # 6 stops of per-texel exposure
    begin, end = ibl_dist.split_rows(6 * w, world)[rank]
    out = torch.zeros(28, dtype=torch.float64, device=device)
    ctx.sh9_partial_device(cube, datum_b200.FORMAT_F32, w, w, begin, end, out)     # builds the solid-angle table
    ctx.synchronize()

    def project():
        ctx.sh9_partial_device(cube, datum_b200.FORMAT_F32, w, w, begin, end, out)
        if world > 1:
            dist.all_reduce(out, op=dist.ReduceOp.SUM)

    ms_kernel = job.timed(stream, lambda: ctx.sh9_partial_device(cube, datum_b200.FORMAT_F32, w, w, begin, end, out), reps=10)
    ms_nccl = job.timed(stream, project, reps=10) if world > 1 else ms_kernel
    sh_nccl = ibl_dist.project_sh9_single_probe(engine, cube, datum_b200.FORMAT_F32, w, w)

    peer_sh = ibl_dist.PeerSh9(ctx)
    ms_peers = job.timed(stream, lambda: peer_sh.enqueue(cube, datum_b200.FORMAT_F32, w, w), reps=10)

    # A single projection timed from a host barrier also carries the launch skew between the ranks (tens of
    # microseconds, as much as the kernel itself at 8 GPUs): K projections queued back to back — the
    # arrival counters keep the ranks in step, the two result arrays alternate — give the per-projection time
    K = 20

    def burst_peers():
        for _ in range(K):
            peer_sh.enqueue(cube, datum_b200.FORMAT_F32, w, w)

    def burst_nccl():
        for _ in range(K):
            project()

    ms_peers_burst = job.timed(stream, burst_peers, reps=3) / K
    ms_nccl_burst = job.timed(stream, burst_nccl, reps=3) / K if world > 1 else ms_peers_burst
    sh_peers = peer_sh.project(cube, datum_b200.FORMAT_F32, w, w)
    peer_sh.close()

    err_nccl = err_peers = None
    if rank == 0:
        want = oracle_sh9_threads(cube.cpu().numpy().reshape(6, w, w, 4), w, max(1, min(32, os.cpu_count() or 1)))
        err_nccl = float(np.abs(sh_nccl - want).max() / np.abs(want).max())
        err_peers = float(np.abs(sh_peers - want).max() / np.abs(want).max())

    rows = end - begin
    hbm, hbm_source = measured_hbm_peak()
    gbs = rows * w * SH9_BYTES_PER_TEXEL / (ms_kernel * 1e-3) / 1e9
    ms = min(ms_nccl, ms_peers)
    return {
        "workload": "C5: SH9 projection (data/project.comp) of one 4096^2-face RGBA32F cube (1.007e8 texels, 1.61 GB), %d rows per GPU on %d GPU(s)" % (rows, world),
        "texels": 6 * w * w, "ms": ms, "texels_per_s": 6 * w * w / ms * 1e3,
        "ms_peer_stores": ms_peers, "ms_nccl_all_reduce": ms_nccl, "ms_kernel_only": ms_kernel,
        "ms_per_projection_back_to_back": min(ms_peers_burst, ms_nccl_burst), "ms_per_projection_back_to_back_peer_stores": ms_peers_burst, "ms_per_projection_back_to_back_nccl": ms_nccl_burst,
        "timing": "ms / ms_peer_stores / ms_nccl_all_reduce: ONE projection from a host barrier (includes the ranks' launch skew); ms_per_projection_back_to_back: %d projections queued back to back, per projection" % K,
        "exchange": "28 doubles per rank: peer stores from the projection kernel's last block + arrival counters, or one NCCL all-reduce",
        "hbm_gb_per_s_per_gpu_kernel": gbs, "hbm_frac_of_measured_kernel": gbs / hbm, "hbm_peak": hbm, "hbm_peak_source": hbm_source,
        "max_rel_vs_oracle": err_peers, "max_rel_vs_oracle_nccl": err_nccl,
        "parity_ok": None if err_peers is None else bool(err_peers <= 1e-4 and err_nccl <= 1e-4),
    }


def dump_ranks(world):
    """The ranks whose chains --dump-outputs saves: all while they fit DUMP_BYTES, else a fixed, seeded sample."""
    per_rank = sum(6 * (WIDTH >> level) ** 2 * 3 * 4 + 128 for level in range(1, LEVELS))   # float32 RGB + .npy header
    keep = DUMP_BYTES // per_rank
    return list(range(world)) if world <= keep else sorted(np.random.default_rng(0).choice(world, keep, replace=False).tolist())


def dump_outputs(directory, chain, rank, world):
    """Levels >= 1 of one baked C2 chain (uint32 rgbe words), decoded to float32 RGB, one .npy per level."""
    import datum_b200
    import oracle_lib

    os.makedirs(directory, exist_ok=True)
    offs = datum_b200.level_offsets(WIDTH, WIDTH, LEVELS)
    prefix = "c2" if world == 1 else "c2_rank%d" % rank
    for level in range(1, LEVELS):
        side = WIDTH >> level
        rgb = oracle_lib.rgbe_decode_array(chain[offs[level]:offs[level + 1]])[:, :3].reshape(6, side, side, 3)
        np.save(os.path.join(directory, "%s_level%d.npy" % (prefix, level)), np.ascontiguousarray(rgb))


def run_ours(args):
    job = Job()
    torch, world, rank, device = job.torch, job.world, job.rank, job.device

    import datum_b200
    from datum_b200 import dist as ibl_dist
    from datum_b200 import synth

    ctx = datum_b200.IblContext(job.local_rank)
    engine = ibl_dist.CudaEngine(ctx)
    stream = ctx.torch_stream()

    w, levels, samples = WIDTH, LEVELS, SAMPLES
    offs = datum_b200.level_offsets(w, w, levels)
    step_work = texel_samples(w, levels, samples)

    # ---- inputs: a pool of distinct probes resident in HBM (larger than L2), pinned and pageable host copies for e2e
    pool_host = [synth.synthetic_chain(w, w, levels, probe=rank * POOL + p) for p in range(POOL)]
    pool_dev = [torch.from_numpy(b.view(np.int32)).to(device) for b in pool_host]
    pinned = [torch.from_numpy(b.view(np.int32).copy()).pin_memory() for b in pool_host[:4]]
    pageable = [b.copy() for b in pool_host[:4]]
    torch.cuda.synchronize()

    fp32_peak = ctx.measure_fp32_peak()

    sampler = ClockSampler(job.local_rank)
    sampler.start()

    # ---- device-resident throughput: W warm-up + K timed steps, CUDA events on the launching stream
    for i in range(args.warmup):
        ctx.buildmips_cube_ibl_device(w, w, levels, pool_dev[i % POOL], samples)
    ctx.synchronize()
    ctx.dominant_kernel_stats(reset=True)
    launches_before = ctx.launch_count

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    job.barrier()
    with torch.cuda.stream(stream):
        ev0.record()
        for i in range(args.steps):
            ctx.buildmips_cube_ibl_device(w, w, levels, pool_dev[(args.warmup + i) % POOL], samples)
        ev1.record()
    ev1.synchronize()
    job.barrier()
    elapsed_ms = job.max_over_ranks(ev0.elapsed_time(ev1))
    launches = ctx.launch_count - launches_before
    dom_n, dom_ms, dom_ts = ctx.dominant_kernel_stats(reset=True)
    if args.dump_outputs and rank in dump_ranks(world):
        last = pool_dev[(args.warmup + args.steps - 1) % POOL].cpu().numpy().view(np.uint32)
        dump_outputs(args.dump_outputs, last, rank, world)

    # ---- end to end through the reference-facing call: pinned host payload in, baked payload out
    def host_loop(payloads):
        for i in range(min(3, max(1, args.warmup))):
            ctx.image_buildmips_cube_ibl(w, w, levels, payloads[i % len(payloads)], samples)
        job.barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            ctx.image_buildmips_cube_ibl(w, w, levels, payloads[i % len(payloads)], samples)
        seconds = job.max_over_ranks(time.perf_counter() - t0)
        job.barrier()
        return seconds

    e2e_s = host_loop(pinned)
    e2e_pageable_s = host_loop(pageable)       # what assetbuilder hands over: a plain std::vector<char> (assetbuilder.cpp:439, 484)

    # ---- the same K bakes as ONE batched call (datum_ibl_bake_probes): copies of probe i+1 / i-1 under the kernels of probe i
    batch = [pinned[i % len(pinned)] for i in range(args.steps)]
    ctx.bake_probes(w, w, levels, batch[: min(12, len(batch))], samples)      # enough payloads for both device buffers of the pipeline to exist
    job.barrier()
    t0 = time.perf_counter()
    ctx.bake_probes(w, w, levels, batch, samples)
    e2e_batch_local = time.perf_counter() - t0
    e2e_batch_s = job.max_over_ranks(e2e_batch_local)
    if world > 1:
        print("bench.py: rank %d e2e_batched %.3f ms per step" % (rank, e2e_batch_local * 1e3 / args.steps), file=sys.stderr, flush=True)
    job.barrier()

    clocks = sampler.stop()

    # ---- sustained: the same device-resident loop for >= 2.5 s, clocks sampled (power-capped steady state)
    sustained_steps = max(args.steps, int(SUSTAINED_SECONDS * 1e3 / (elapsed_ms / args.steps)) + 1)
    sampler.start()
    job.barrier()
    with torch.cuda.stream(stream):
        ev0.record()
        for i in range(sustained_steps):
            ctx.buildmips_cube_ibl_device(w, w, levels, pool_dev[i % POOL], samples)
        ev1.record()
    ev1.synchronize()
    job.barrier()
    sustained_ms = job.max_over_ranks(ev0.elapsed_time(ev1))
    sustained_clocks = sampler.stop()
    sus_n, sus_dom_ms, _ = ctx.dominant_kernel_stats(reset=True)

    total_launches = int(job.sum_over_ranks(launches))

    cpu_info = None
    if world == 1:
        cpu_value, _, cpu_info = cpu_reference_run(rounds=1)
        cpu_info["value"] = cpu_value
        cpu_info["unit"] = UNIT

    configs = {}

    def emit():
        """The ONE JSON line (rank 0)."""
        value = world * step_work * args.steps / (elapsed_ms * 1e-3)
        e2e_value = world * step_work * args.steps / e2e_s

        achieved = FLOP_PER_TEXEL_SAMPLE * dom_ts / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
        traffic = profiled_traffic()
        hbm_peak, hbm_source = measured_hbm_peak()
        pre_traffic = traffic.get("prefilter_level1", {}).get("dram_bytes")

        line = {
            "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": base_config(world),
            "env_maps_per_s": world * args.steps / (elapsed_ms * 1e-3),
            "e2e": {
                "value": e2e_value, "unit": UNIT,
                "h2d_bytes_per_step": offs[1] * 4, "d2h_bytes_per_step": (offs[-1] - offs[1]) * 4,
                "api": "image_buildmips_cube_ibl(width, height, levels, bits) on a pinned host payload",
                "ms_per_step": e2e_s * 1e3 / args.steps,
            },
            "e2e_pageable": {
                "value": world * step_work * args.steps / e2e_pageable_s, "unit": UNIT,
                "api": "the same call on a pageable host payload (what assetbuilder.cpp:439,484 allocates: std::vector<char>)",
                "ms_per_step": e2e_pageable_s * 1e3 / args.steps,
            },
            "e2e_batched": {
                "value": world * step_work * args.steps / e2e_batch_s, "unit": UNIT,
                "api": "bake_probes: %d pinned host payloads in one datum_ibl_bake_probes call per GPU (uploads, kernels, downloads overlapped)" % args.steps,
                "ms_per_step": e2e_batch_s * 1e3 / args.steps,
            },
            "sustained": {
                "value": world * step_work * sustained_steps / (sustained_ms * 1e-3), "unit": UNIT,
                "seconds": sustained_ms * 1e-3, "steps": sustained_steps, "ms_per_step": sustained_ms / sustained_steps,
                "level1_ms_per_launch": sus_dom_ms, "level1_launches_averaged": sus_n,
                "level1_frac_of_fp32_peak": (FLOP_PER_TEXEL_SAMPLE * dom_ts / (sus_dom_ms * 1e-3) / 1e12 / fp32_peak) if sus_dom_ms > 0 and fp32_peak else None,
                "clocks": {"sm_mhz": sustained_clocks["sm_mhz"], "sm_max_mhz": sustained_clocks["sm_max_mhz"], "reasons": sustained_clocks["reasons"], "samples": sustained_clocks["samples"]},
            },
            "gpu_launches": total_launches,
            "roofline": {
                "bound": "fp32", "kernel": "prefilter_dp_kernel (level 1: 512^2 -> 256^2 faces)",
                "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak if fp32_peak else None,
                "peak_source": "FFMA-chain micro-benchmark run in this process (datum_ibl_measure_fp32_peak); MEASURED_PEAKS.json carries no FP32 figure",
                "flop_per_texel_sample": FLOP_PER_TEXEL_SAMPLE, "texel_samples_per_launch": dom_ts,
                "launches_timed": dom_n, "ms_per_launch": dom_ms,
                "whole_step_frac": FLOP_PER_TEXEL_SAMPLE * step_work / (elapsed_ms / args.steps * 1e-3) / 1e12 / fp32_peak if fp32_peak else None,
                "traffic": pre_traffic, "traffic_source": traffic.get("prefilter_level1", {}).get("source"),
                "hbm": {"achieved": (pre_traffic or 0) / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None, "peak": hbm_peak, "unit": "GB/s", "peak_source": hbm_source},
            },
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
            "configs": configs,
        }

        c5 = configs.get("C5", {})
        if world == 1 and "ms_kernel_only" in c5:
            achieved_gbs = SH9_BYTES_PER_TEXEL * c5["texels"] / (c5["ms_kernel_only"] * 1e-3) / 1e9
            line["roofline_sh9"] = {
                "bound": "hbm", "kernel": "sh9 projection of one 4096^2 RGBA32F cube (config C5 on one GPU)",
                "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                "peak_source": hbm_source, "bytes_per_texel": SH9_BYTES_PER_TEXEL, "texels_per_launch": c5["texels"], "ms_per_launch": c5["ms_kernel_only"],
                "traffic": traffic.get("sh9", {}).get("dram_bytes"), "traffic_source": traffic.get("sh9", {}).get("source"),
            }
        if cpu_info is not None:
            line["cpu_baseline"] = cpu_info

        print(json.dumps(line), flush=True)

    # ---- BASELINE.json's other configurations.  Each sits behind its own try (a failure is reported in
    #      the line, not fatal), and the whole stage behind a watchdog: should a rank die inside a
    #      collective, the headline measured above is still printed and every rank leaves.
    stage = {"name": None}

    def give_up():
        if stage["name"]:
            configs.setdefault(stage["name"], {"error": "no result within %d s (watchdog)" % args.configs_timeout})
        if rank == 0:
            emit()
        sys.stdout.flush()
        os._exit(0)

    watchdog = threading.Timer(args.configs_timeout, give_up)
    watchdog.daemon = True

    def attempt(name, fn):
        stage["name"] = name
        try:
            configs[name] = fn()
        except Exception as exc:                      # noqa: BLE001 - reported in the JSON line
            configs[name] = {"error": "rank %d: %s: %s" % (rank, type(exc).__name__, exc)}
            print("bench.py: config %s failed on rank %d: %s: %s" % (name, rank, type(exc).__name__, exc), file=sys.stderr, flush=True)
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
        stage["name"] = None
        torch.cuda.empty_cache()

    if not args.skip_configs:
        watchdog.start()
        attempt("C4", lambda: config_c4(job, ctx))
        attempt("C5", lambda: config_c5(job, ctx, engine, stream))
        attempt("C3", lambda: config_c3(job, ctx, engine, stream))
        if world == 1 and args.steps >= 5:
            attempt("C1", lambda: config_c1(job, ctx))

        # the device-list path on the same GPUs: the other ranks leave first, then this process alone drives all of them
        if world > 1:
            job.barrier()
            job.dist.destroy_process_group()      # every rank together; nothing below is collective
            if rank != 0:
                watchdog.cancel()
                return 0
            time.sleep(1.0)                       # the other processes release their contexts
            attempt("C3_one_process", lambda: config_c3_one_process(job, ctx))
        watchdog.cancel()

    if rank == 0:
        emit()

    if world > 1 and job.dist.is_initialized():
        job.dist.destroy_process_group()
    return 0


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=None, help="timed steps (default 50; 10 for --impl reference, whose step is ~7 s of CPU work)")
    parser.add_argument("--warmup", type=int, default=5, help="untimed steps before the timed ones (the GPU arm runs at least 3: first launches load modules and build sample tables)")
    parser.add_argument("--impl", choices=["ours", "reference"], default="ours")
    parser.add_argument("--skip-configs", action="store_true", help="only the C2 headline (development runs)")
    parser.add_argument("--configs-timeout", type=int, default=480, help="seconds the extra configurations may take before the line is printed without them")
    parser.add_argument("--dump-outputs", metavar="DIR", default=None, help="save the chain levels the last timed step baked as DIR/*.npy (float32)")
    args = parser.parse_args()
    if args.steps is None:
        args.steps = 50 if args.impl == "ours" else 10
    if args.steps < 1:
        parser.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        parser.error("--dump-outputs saves the GPU bake; the reference arm has none")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else max(0, args.warmup)

    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
