#!/usr/bin/env python3
"""What the denoiser AOVs cost next to the beauty pass: yart_render_aovs against yart_render, per sample per pixel.

    python tools/aov_probe.py --out DIR [--reps 7] [--spp 16] [--scene david] [--width 1920] [--height 1080]

Device planes and a device film (no PCIe copies in the window); times are the library's own CUDA events
(stats.gpu_ms).  Both calls are warmed up, then alternate for --reps repetitions over samples [0, spp); median and
best are reported per spp, with the spread (max - min) / median.  The JSON line goes to DIR/aov_probe.jsonl together
with the card's name, power limit and maximum SM clock."""
import argparse
import importlib
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def stats(xs, spp):
    xs = np.asarray(xs, dtype=np.float64) / spp
    med = float(np.median(xs))
    return {"median_ms_per_spp": med, "best_ms_per_spp": float(xs.min()), "spread": float((xs.max() - xs.min()) / med)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--scene", default="david")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    args = ap.parse_args()
    y = importlib.import_module("yet-another-raytracer_b200")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    preset = y.ScenePreset(args.scene)
    ctx = y.Context(0)
    ctx.set_scene(preset)
    w, h, spp = args.width, args.height, args.spp
    cam = preset.camera(w, h)
    depth = preset.info.max_depth
    film = ctx.film_create(w, h)
    planes = [ctx.film_create(w, h) for _ in range(3)]

    def beauty():
        ctx.film_clear(film, w, h)
        return ctx.render_device(cam, w, h, 0, spp, film, depth, 1)

    def aovs():
        for p in planes:
            ctx.film_clear(p, w, h)
        return ctx.render_aovs_device(cam, w, h, 0, spp, *planes, max_depth=depth, seed=1)

    for _ in range(2):
        beauty()
        aovs()
    b, a, a_trace = [], [], []
    for _ in range(args.reps):
        b.append(beauty().gpu_ms)
        st = aovs()
        a.append(st.gpu_ms)
        a_trace.append(st.trace_ms)
    line = {"scene": args.scene, "width": w, "height": h, "spp": spp, "max_depth": depth, "reps": args.reps,
            "aovs": stats(a, spp), "aovs_closest_hit": stats(a_trace, spp), "render": stats(b, spp),
            "aov_over_render_median": float(np.median(a) / np.median(b)), "gpu": gpu,
            "times": "CUDA events (stats.gpu_ms), device film and planes"}
    print(json.dumps(line))
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "aov_probe.jsonl", "a") as f:
        f.write(json.dumps(line) + "\n")
    for p in [film] + planes:
        ctx.film_destroy(p)
    ctx.close()


if __name__ == "__main__":
    main()
