"""Equirect HDR image -> probe on one GPU, rgbe against RGBA16F and RGBA32F: a seeded 2048x1024 RGBA fp32
equirect image with a bright sun baked into a 512^2 x 8 chain at 1024 spp by datum_ibl_pack_cube_ibl (rgbe) and
datum_ibl_pack_cube_float_ibl (F16, F32), and the level-0-only entries (datum_ibl_pack_cube,
datum_ibl_pack_cube_float).

End to end as a caller sees it: image and chain in pinned host memory, a host clock around each synchronous call
(upload, resample, edge blend, chain, download).  Every entry is warmed up, then the entries run in alternated
rounds and the medians are reported.  The card's name and power limit are read with nvidia-smi in the same run
(query only).

    python tools/float_pack_times.py --out profiles/r6_float_pack.json [--rounds 15] [--warmup 3]
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

IMG_W, IMG_H = 2048, 1024
W, LEVELS, SAMPLES = 512, 8, 1024


def card():
    proc = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    name, power, clock = [f.strip() for f in proc.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def sun_equirect(seed=6):
    rng = np.random.default_rng(seed)
    img = np.ones((IMG_H, IMG_W, 4), np.float32)
    img[..., :3] = (rng.random((IMG_H, IMG_W, 3)) * np.exp2(rng.integers(-3, 3, (IMG_H, IMG_W, 1)))).astype(np.float32)
    yy, xx = np.meshgrid(np.arange(IMG_H), np.arange(IMG_W), indexing="ij")
    disc = (yy - 0.3 * IMG_H) ** 2 + (xx - 0.6 * IMG_W) ** 2 <= 12.0 ** 2
    img[disc, :3] = np.array([5000.0, 4500.0, 3800.0], np.float32)
    return img


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("float_pack_times: no CUDA device")

    ctx = datum_b200.IblContext(0)
    image = torch.from_numpy(sun_equirect()).pin_memory()
    texels = datum_b200.level_offsets(W, W, LEVELS)[-1]
    buffers = {
        "rgbe": torch.zeros(texels, dtype=torch.int32).pin_memory(),
        "f16": torch.zeros((texels, 4), dtype=torch.float16).pin_memory(),
        "f32": torch.zeros((texels, 4), dtype=torch.float32).pin_memory(),
    }
    fmt = {"f16": datum_b200.FORMAT_F16, "f32": datum_b200.FORMAT_F32}
    lib, h = ctx._lib, ctx._handle
    p_img = image.data_ptr()

    def chain(name):
        p = buffers[name].data_ptr()
        if name == "rgbe":
            return lib.datum_ibl_pack_cube_ibl(h, IMG_W, IMG_H, p_img, W, W, LEVELS, SAMPLES, p)
        return lib.datum_ibl_pack_cube_float_ibl(h, fmt[name], IMG_W, IMG_H, p_img, W, W, LEVELS, SAMPLES, p)

    def level0_only(name):
        p = buffers[name].data_ptr()
        if name == "rgbe":
            return lib.datum_ibl_pack_cube(h, IMG_W, IMG_H, p_img, W, W, p)
        return lib.datum_ibl_pack_cube_float(h, fmt[name], IMG_W, IMG_H, p_img, W, W, p)

    entries = {("chain", f): (lambda f=f: chain(f)) for f in ("rgbe", "f16", "f32")}
    entries.update({("level0", f): (lambda f=f: level0_only(f)) for f in ("rgbe", "f16", "f32")})

    for run in entries.values():
        for _ in range(args.warmup):
            ctx._check(run())

    times = {k: [] for k in entries}
    for _ in range(args.rounds):
        for k, run in entries.items():
            t0 = time.perf_counter()
            status = run()
            times[k].append((time.perf_counter() - t0) * 1e3)
            ctx._check(status)

    result = {
        "what": "equirect %dx%d RGBA fp32 with a sun -> %d^2 x %d chain at %d spp, pinned host image and chain, host clock around each synchronous call"
                % (IMG_W, IMG_H, W, LEVELS, SAMPLES),
        "card": card(),
        "rounds": args.rounds,
        "warmup": args.warmup,
        "entries": {},
    }
    names = {("chain", "rgbe"): "datum_ibl_pack_cube_ibl", ("chain", "f16"): "datum_ibl_pack_cube_float_ibl F16",
             ("chain", "f32"): "datum_ibl_pack_cube_float_ibl F32", ("level0", "rgbe"): "datum_ibl_pack_cube",
             ("level0", "f16"): "datum_ibl_pack_cube_float F16", ("level0", "f32"): "datum_ibl_pack_cube_float F32"}
    for k, v in times.items():
        result["entries"][names[k]] = {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)}

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=2)
    print(json.dumps(result, indent=2))


if __name__ == "__main__":
    main()
