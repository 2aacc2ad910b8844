"""One BASELINE config 3 probe (2048^2 faces, 12 levels, 4096 spp) shared by the GPUs of a device list, for F16
and F32 chains, with the rgbe chain on the same lists as the reference.

End to end through the device-list entries from pinned host chains: MultiContext.buildmips_cube_float (F16, F32)
and MultiContext.image_buildmips_cube_ibl (rgbe).  A one-device list runs the single-GPU entries
(datum_ibl_buildmips_cube_float, datum_ibl_buildmips_cube_ibl).  Lists: one GPU, then 2, 4 and 8 distinct GPUs as
far as the box has them; a list the box cannot hold is recorded as "not measured".

Every call is synchronous: a host clock around it measures it end to end, uploads and downloads included.  After
a warm-up of every (format, list), rounds alternate over all of them; reported per pair: median/min/max ms over
the rounds.  The shared bakes' last results are also compared with the one-GPU chain of the same format (F32:
largest error relative to the texel's largest channel; F16: largest ulp distance and identical share).  GPU
names, count, power limits and maximum SM clocks are read with nvidia-smi (query only) in the same run.

    python tools/float_shared_probe_times.py --out DIR [--rounds 5]

Writes DIR/r5_float_shared_probe.json and prints it.
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

W, LEVELS, SAMPLES = 2048, 12, 4096
FORMATS = ("rgbe", "f16", "f32")
FMT = {"rgbe": datum_b200.FORMAT_RGBE, "f16": datum_b200.FORMAT_F16, "f32": datum_b200.FORMAT_F32}
LIST_SIZES = (1, 2, 4, 8)


def cards():
    proc = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    out = []
    for line in proc.stdout.strip().splitlines():
        index, name, power, clock = [f.strip() for f in line.split(",")]
        out.append({"index": int(index), "name": name, "power_limit": power, "clocks_max_sm": clock})
    return out


def level0(fmt):
    """Pinned host chain of the format, level 0 from synth.synthetic_cube(probe=3), no sun; the other levels zero."""
    offs = datum_b200.level_offsets(W, W, LEVELS)
    cube = synth.synthetic_cube(W, W, probe=3, noise=True, sun=False).reshape(-1, 4)
    if fmt == "rgbe":
        chain = np.zeros(offs[-1], np.uint32)
        chain[: offs[1]] = synth.rgbe_words(cube)
        return torch.from_numpy(chain.view(np.int32)).pin_memory()
    chain = np.zeros((offs[-1], 4), np.float16 if fmt == "f16" else np.float32)
    chain[: offs[1]] = cube.astype(chain.dtype)
    return torch.from_numpy(chain).pin_memory()


def compare(fmt, got, want):
    """The shared chain against the one-GPU chain, levels >= 1."""
    start = 6 * W * W
    if fmt == "rgbe":
        a, b = got[start:], want[start:]
        return {"identical": float(np.mean(a == b))}
    if fmt == "f32":
        a, b = got[start:, :3].astype(np.float64), want[start:, :3].astype(np.float64)
        scale = np.abs(b).max(axis=1)
        err = np.abs(a - b).max(axis=1)
        rel = err[scale > 0] / scale[scale > 0]
        return {"max_rel_to_texel_max": float(rel.max()) if rel.size else 0.0, "identical": float(np.mean(a == b)),
                "zero_texels_differing": int(np.sum((scale == 0) & (err > 0)))}
    ulps = np.abs(got[start:, :3].view(np.uint16).astype(np.int64) - want[start:, :3].view(np.uint16).astype(np.int64))
    return {"max_ulp": int(ulps.max()), "identical": float((ulps == 0).mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("float_shared_probe_times: no CUDA device")

    gpus = torch.cuda.device_count()
    lists = {n: list(range(n)) for n in LIST_SIZES if n <= gpus}
    multis = {n: datum_b200.MultiContext(devices) for n, devices in lists.items()}
    sources = {f: level0(f) for f in FORMATS}
    chains = {(f, n): sources[f].clone().pin_memory() for f in FORMATS for n in lists}

    def bake(f, n):
        chain = chains[(f, n)]
        if f == "rgbe":
            multis[n].image_buildmips_cube_ibl(W, W, LEVELS, chain, SAMPLES)
        else:
            multis[n].buildmips_cube_float(FMT[f], W, W, LEVELS, chain, SAMPLES)

    for f in FORMATS:                     # warm-up: tables, frames, payloads and launch shapes of every pair
        for n in lists:
            bake(f, n)

    seconds = {(f, n): [] for f in FORMATS for n in lists}
    for _ in range(args.rounds):
        for f in FORMATS:
            for n in lists:
                t0 = time.perf_counter()
                bake(f, n)
                seconds[(f, n)].append(time.perf_counter() - t0)

    result = {
        "shape": {"width": W, "height": W, "levels": LEVELS, "samples": SAMPLES, "sun": False},
        "gpu_count": gpus,
        "cards": cards(),
        "rounds": args.rounds,
        "host_memory": "pinned",
        "method": "host clock around each synchronous call, warm-up of every (format, list), rounds alternating over all of them",
        "formats": {},
    }
    for f in FORMATS:
        entry = {}
        one = seconds[(f, 1)]
        for n in LIST_SIZES:
            key = "gpus_%d" % n
            if n not in lists:
                entry[key] = "not measured"
                continue
            s = seconds[(f, n)]
            entry[key] = {
                "devices": lists[n],
                "ms_median": 1e3 * statistics.median(s),
                "ms_min": 1e3 * min(s),
                "ms_max": 1e3 * max(s),
                "speedup_over_one_gpu_median": statistics.median(one) / statistics.median(s),
            }
            if n > 1:
                entry[key]["against_one_gpu"] = compare(f, chains[(f, n)].numpy(), chains[(f, 1)].numpy())
        result["formats"][f] = entry

    for m in multis.values():
        m.close()

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r5_float_shared_probe.json"), "w") as fh:
        json.dump(result, fh, indent=2)
    print(json.dumps(result, indent=2))


if __name__ == "__main__":
    main()
