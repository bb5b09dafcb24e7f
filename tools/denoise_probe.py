#!/usr/bin/env python3
"""What yart_denoise costs and buys.

    python tools/denoise_probe.py --out DIR [--reps 7] [--ref-spp 4096] [--skip-time] [--skip-quality]

Cost: david 1920x1080, device film, planes and output (no PCIe copies in the window), levels 1..5, one beauty sample
and one AOV sample of the same frame, each warmed up and then alternated for --reps repetitions; times are the
library's CUDA events (stats.gpu_ms), median and spread (max - min) / median.
Quality: cornell-box 300x300 and david 480x270 against a --ref-spp render (seed 100): relMSE (tests/denoise_ref.py)
of the noisy and the denoised image at 1..64 spp (seeds 1-3, planes of min(16, spp) samples), a sigma sweep at 16 spp, and how much denoising the reference
itself changes it (over-blur).  One JSON line per part goes to DIR/denoise_probe.jsonl with the card's name, power limit
and maximum SM clock."""
import argparse
import importlib
import itertools
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import denoise_ref  # noqa: E402

SPPS = (1, 2, 4, 8, 16, 32, 64)
SWEEP = {"sigma_color": (0.5, 2.0, 4.0, 8.0, 16.0, 32.0), "sigma_normal": (0.1, 0.3, 1.0), "sigma_depth": (0.05, 0.2, 1.0),
         "levels": (3, 5)}


def spread(xs):
    xs = np.asarray(xs, dtype=np.float64)
    med = float(np.median(xs))
    return {"median_ms": med, "best_ms": float(xs.min()), "spread": float((xs.max() - xs.min()) / med)}


def cost(y, ctx, reps):
    preset = y.ScenePreset("david")
    ctx.set_scene(preset)
    w, h = 1920, 1080
    cam = preset.camera(w, h)
    depth = preset.info.max_depth
    film = ctx.film_create(w, h)
    planes = [ctx.film_create(w, h) for _ in range(3)]
    out = ctx.film_create(w, h)  # (an f32 rgb image fits in a film's bytes)
    ctx.render_device(cam, w, h, 0, 16, film, depth, 1)
    ctx.render_aovs_device(cam, w, h, 0, 16, *planes, max_depth=depth, seed=1)
    scratch = ctx.film_create(w, h)
    beauty = lambda: ctx.render_device(cam, w, h, 0, 1, scratch, depth, 1).gpu_ms  # noqa: E731
    aov = lambda: ctx.render_aovs_device(cam, w, h, 0, 1, scratch, scratch, scratch, max_depth=depth, seed=1).gpu_ms  # noqa: E731
    calls = {"beauty_1spp": beauty, "aov_1spp": aov}
    for L in range(1, 6):
        calls["denoise_L%d" % L] = (lambda L=L: ctx.denoise_device(film, 16, *planes, w, h, rgb_ptr=out, levels=L).gpu_ms)
    for _ in range(2):
        for f in calls.values():
            f()
    times = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():
            times[k].append(f())
    for p in [film, out, scratch] + planes:
        ctx.film_destroy(p)
    res = {k: spread(v) for k, v in times.items()}
    b = res["beauty_1spp"]["median_ms"]
    return {"part": "cost", "scene": "david", "width": w, "height": h, "reps": reps, "times": res,
            "denoise_L5_over_beauty_spp": res["denoise_L5"]["median_ms"] / b,
            "denoise_L5_over_aov_spp": res["denoise_L5"]["median_ms"] / res["aov_1spp"]["median_ms"]}


def quality(y, ctx, scene, w, h, ref_spp):
    preset = y.ScenePreset(scene)
    ctx.set_scene(preset)
    cam = preset.camera(w, h)
    depth = preset.info.max_depth
    ref_film, _ = ctx.render(cam, w, h, 0, ref_spp, depth, 100)
    ref = ctx.film_finalize_linear(ref_film, ref_spp)
    ref_planes, _ = ctx.render_aovs(cam, w, h, 0, 16, depth, 100)
    valid = ref_planes["depth"][..., 2] > 0
    ref_dn = ctx.denoise(ref_film, ref_spp, ref_planes)
    curve = []
    inputs16 = []
    for spp in SPPS:
        noisy, den, t_r, t_a = [], [], [], []
        for seed in (1, 2, 3):
            film, st = ctx.render(cam, w, h, 0, spp, depth, seed)
            planes, sta = ctx.render_aovs(cam, w, h, 0, min(16, spp), depth, seed)
            noisy.append(denoise_ref.rel_mse(ctx.film_finalize_linear(film, spp), ref, valid))
            den.append(denoise_ref.rel_mse(ctx.denoise(film, spp, planes), ref, valid))
            t_r.append(st.gpu_ms)
            t_a.append(sta.gpu_ms)
            if spp == 16:
                inputs16.append((film, planes))
        curve.append({"spp": spp, "relmse_noisy": noisy, "relmse_denoised": den, "render_ms": float(np.median(t_r)),
                      "aov_ms": float(np.median(t_a))})
    sweep = []
    for vals in itertools.product(*SWEEP.values()):
        kw = dict(zip(SWEEP, vals))
        r = [denoise_ref.rel_mse(ctx.denoise(f, 16, p, **kw), ref, valid) for f, p in inputs16]
        blur = denoise_ref.rel_mse(ctx.denoise(ref_film, ref_spp, ref_planes, **kw), ref, valid)
        sweep.append(dict(kw, relmse_denoised_16=r, relmse_ref_denoised=blur))
    return {"part": "quality", "scene": scene, "width": w, "height": h, "ref_spp": ref_spp, "max_depth": depth,
            "relmse_ref_denoised_default": denoise_ref.rel_mse(ref_dn, ref, valid), "curve": curve, "sweep_16spp": sweep,
            "metric": "mean over valid pixels and channels of (x - ref)^2 / (ref^2 + 0.01), linear RGB"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--skip-time", action="store_true")
    ap.add_argument("--skip-quality", action="store_true")
    args = ap.parse_args()
    y = importlib.import_module("yet-another-raytracer_b200")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    ctx = y.Context(0)
    lines = []
    if not args.skip_time:
        lines.append(cost(y, ctx, args.reps))
    if not args.skip_quality:
        lines.append(quality(y, ctx, "cornell-box", 300, 300, args.ref_spp))
        lines.append(quality(y, ctx, "david", 480, 270, args.ref_spp))
    ctx.close()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "denoise_probe.jsonl", "a") as f:
        for line in lines:
            line["gpu"] = gpu
            print(json.dumps(line)[:2000])
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
