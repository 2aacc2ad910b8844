"""Batched bakes against single calls on one GPU: BASELINE config 4's unit (256^2 faces, 8 levels, 1024 spp,
SH9 on) for rgbe, F16 and F32 chains, 64 distinct seeded probes in pinned host memory.

For every format two arms, alternated round by round in one process after a warm-up of every shape:
  batch   one bake_probes / bake_probes_float call over all probes (SH9 of every level 0 included);
  single  one host call per probe (image_buildmips_cube_ibl / buildmips_cube_float), each followed by
          project_sh9 of its level 0, so that both arms compute the same.
Every call is synchronous: a host clock around it measures it end to end, copies included.  Reported per
arm: probes/s and ms per probe, median/min/max over the rounds.  The card's name, power limit and maximum SM
clock are read with nvidia-smi (query only).

    python tools/float_batch_times.py --out DIR [--rounds 5] [--probes 64]

Writes DIR/float_batch_times.json and prints it.
"""

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

import datum_b200
from datum_b200 import synth

W, LEVELS, SAMPLES = 256, 8, 1024
FORMATS = ("rgbe", "f16", "f32")
FMT = {"rgbe": datum_b200.FORMAT_RGBE, "f16": datum_b200.FORMAT_F16, "f32": datum_b200.FORMAT_F32}


def card():
    proc = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    name, power, clock = [f.strip() for f in proc.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def payloads(fmt, probes):
    """Pinned host chains of the format, level 0 from synth.synthetic_cube(probe=p)."""
    offs = datum_b200.level_offsets(W, W, LEVELS)
    out = []
    for p in range(probes):
        cube = synth.synthetic_cube(W, W, probe=p, noise=True, sun=True).reshape(-1, 4)
        if fmt == "rgbe":
            chain = np.zeros(offs[-1], np.uint32)
            chain[: offs[1]] = synth.rgbe_words(cube)
            out.append(torch.from_numpy(chain.view(np.int32)).pin_memory())
        else:
            chain = np.zeros((offs[-1], 4), np.float16 if fmt == "f16" else np.float32)
            chain[: offs[1]] = cube.astype(chain.dtype)
            out.append(torch.from_numpy(chain).pin_memory())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--probes", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("float_batch_times: no CUDA device")

    ctx = datum_b200.IblContext(0)
    chains = {f: payloads(f, args.probes) for f in FORMATS}
    level0 = 6 * W * W

    def batch(f):
        if f == "rgbe":
            ctx.bake_probes(W, W, LEVELS, chains[f], SAMPLES, sh9=True)
        else:
            ctx.bake_probes_float(FMT[f], W, W, LEVELS, chains[f], SAMPLES, sh9=True)

    def single(f):
        for t in chains[f]:
            if f == "rgbe":
                ctx.image_buildmips_cube_ibl(W, W, LEVELS, t, SAMPLES)
                ctx.project_sh9(t[:level0], FMT[f], W, W)
            else:
                ctx.buildmips_cube_float(FMT[f], W, W, LEVELS, t, SAMPLES)
                ctx.project_sh9(t[:level0], FMT[f], W, W)

    arms = {"batch": batch, "single": single}
    for f in FORMATS:                     # warm-up: tables, frames, launch shapes and staging of every shape
        for run in arms.values():
            run(f)

    seconds = {f: {a: [] for a in arms} for f in FORMATS}
    for _ in range(args.rounds):
        for f in FORMATS:
            for a, run in arms.items():
                t0 = time.perf_counter()
                run(f)
                seconds[f][a].append(time.perf_counter() - t0)

    result = {
        "shape": {"width": W, "levels": LEVELS, "samples": SAMPLES, "sh9": True},
        "card": card(),
        "rounds": args.rounds,
        "probes": args.probes,
        "host_memory": "pinned",
        "formats": {},
    }
    for f in FORMATS:
        result["formats"][f] = {}
        for a in arms:
            s = seconds[f][a]
            result["formats"][f][a] = {
                "probes_per_s_median": args.probes / statistics.median(s),
                "probes_per_s_min": args.probes / max(s),
                "probes_per_s_max": args.probes / min(s),
                "ms_per_probe_median": 1e3 * statistics.median(s) / args.probes,
                "ms_per_probe_min": 1e3 * min(s) / args.probes,
                "ms_per_probe_max": 1e3 * max(s) / args.probes,
            }
        result["formats"][f]["batch_over_single_median"] = result["formats"][f]["batch"]["probes_per_s_median"] / result["formats"][f]["single"]["probes_per_s_median"]

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "float_batch_times.json"), "w") as fh:
        json.dump(result, fh, indent=2)
    print(json.dumps(result, indent=2))


if __name__ == "__main__":
    main()
