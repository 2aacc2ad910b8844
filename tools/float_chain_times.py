"""Float chains against the rgbe chain on one GPU: BASELINE config 2 (512^2 faces, 8 levels, 1024 spp) on
device-resident chains, rgbe, F16 and F32 alternated round by round in one process.

For every format: time of a whole chain (CUDA events around each chain call, `--probes` distinct probes
cycled so that the working set exceeds the 126 MB L2), time of the level-1 prefilter launch (the context's
event ring around it), texel-samples/s of the chain, and the share of the measured fp32 FMA peak at 85 flop
per texel-sample.  The card's name, power limit and maximum SM clock are read with nvidia-smi (query only).

    python tools/float_chain_times.py --out DIR [--rounds 5] [--probes 16]

Writes DIR/float_chain_times.json and prints it.
"""

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

import datum_b200
from datum_b200 import synth

W, LEVELS, SAMPLES = 512, 8, 1024
FLOP_PER_TEXEL_SAMPLE = 85
FORMATS = ("rgbe", "f16", "f32")


def card():
    proc = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    name, power, clock = [f.strip() for f in proc.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--probes", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("float_chain_times: no CUDA device")

    ctx = datum_b200.IblContext(0)
    dev = "cuda:0"
    offs = datum_b200.level_offsets(W, W, LEVELS)
    texel_samples = (offs[-1] - offs[1]) * SAMPLES

    # distinct probes per format, level 0 filled, device-resident
    chains = {f: [] for f in FORMATS}
    for p in range(args.probes):
        cube = synth.synthetic_cube(W, W, probe=p, noise=True, sun=True).reshape(-1, 4)
        bits = np.zeros(offs[-1], np.uint32)
        bits[: offs[1]] = synth.rgbe_words(cube)
        chains["rgbe"].append(torch.from_numpy(bits.view(np.int32)).to(dev))
        for f, dtype in (("f16", np.float16), ("f32", np.float32)):
            chain = np.zeros((offs[-1], 4), dtype)
            chain[: offs[1]] = cube.astype(dtype)
            chains[f].append(torch.from_numpy(chain).to(dev))
    working_set = {f: sum(t.numel() * t.element_size() for t in chains[f]) for f in FORMATS}

    def run(f, t):
        if f == "rgbe":
            ctx.buildmips_cube_ibl_device(W, W, LEVELS, t, SAMPLES)
        else:
            ctx.buildmips_cube_float_device(datum_b200.FORMAT_F16 if f == "f16" else datum_b200.FORMAT_F32, W, W, LEVELS, t, SAMPLES)

    stream = ctx.torch_stream()
    chain_ms = {f: [] for f in FORMATS}
    level1_ms = {f: [] for f in FORMATS}

    with torch.cuda.stream(stream):
        for f in FORMATS:
            for _ in range(args.warmup):
                for t in chains[f]:
                    run(f, t)
        stream.synchronize()

        for _ in range(args.rounds):
            for f in FORMATS:
                ctx.dominant_kernel_stats(reset=True)
                events = []
                for t in chains[f]:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    run(f, t)
                    b.record(stream)
                    events.append((a, b))
                stream.synchronize()
                chain_ms[f] += [a.elapsed_time(b) for a, b in events]
                n, ms, _ = ctx.dominant_kernel_stats(reset=True)
                level1_ms[f].append(ms)

    peak = ctx.measure_fp32_peak()
    result = {
        "shape": {"width": W, "levels": LEVELS, "samples": SAMPLES},
        "card": card(),
        "rounds": args.rounds,
        "probes": args.probes,
        "fp32_peak_tflops_measured": peak,
        "flop_per_texel_sample": FLOP_PER_TEXEL_SAMPLE,
        "texel_samples_per_chain": texel_samples,
        "formats": {},
    }
    for f in FORMATS:
        med = statistics.median(chain_ms[f])
        rate = texel_samples / (med * 1e-3)
        result["formats"][f] = {
            "working_set_bytes": working_set[f],
            "chain_ms_median": med,
            "chain_ms_min": min(chain_ms[f]),
            "chain_ms_max": max(chain_ms[f]),
            "level1_launch_ms_median": statistics.median(level1_ms[f]),
            "texel_samples_per_s": rate,
            "fp32_peak_fraction": rate * FLOP_PER_TEXEL_SAMPLE / (peak * 1e12),
        }

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "float_chain_times.json"), "w") as fh:
        json.dump(result, fh, indent=2)
    print(json.dumps(result, indent=2))


if __name__ == "__main__":
    main()
