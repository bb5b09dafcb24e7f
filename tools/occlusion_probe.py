#!/usr/bin/env python3
"""yart_occluded next to yart_closest_hit(ORDER_NEAR) -- the fastest closest-hit -- in one process, on the same arrays.

    python tools/occlusion_probe.py --out DIR [--reps 7] [--n 16777216]

Times are the library's own CUDA events (stats.gpu_ms).  Every set is warmed up, then the two queries alternate for
--reps repetitions; median and best are reported, and the spread of each as (max - min) / median.  Sets:
  * 16 Mi david uniform / axis / path rays (bench.sweep_rays), mesh target, f64 and f32 records, device arrays;
  * shadow rays of the david preset (tests/occlusion_sets.py), world target, device arrays;
  * host arrays end to end (page-locked f32 records and outputs), uniform set: wall-clock of the whole call.
Each set's occluded fraction is reported too.  JSON lines go to DIR/occlusion_probe.jsonl together with the card's
name, power limit and maximum SM clock."""
import argparse
import importlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import bench  # noqa: E402  (sweep_rays, MeshOnlyScene: the benchmark's own ray sets)
from occlusion_sets import shadow_rays  # noqa: E402

INF = float("inf")


def stats(xs):
    xs = np.asarray(xs, dtype=np.float64)
    med = float(np.median(xs))
    return {"median_ms": med, "best_ms": float(xs.min()), "spread": float((xs.max() - xs.min()) / med)}


def alternate(occ, ch, reps, warm=3):
    for _ in range(warm):
        occ()
        ch()
    a, b = [], []
    for _ in range(reps):
        a.append(occ())
        b.append(ch())
    return stats(a), stats(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--n", type=int, default=1 << 24)
    args = ap.parse_args()
    import torch
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = gpu[0] if gpu else "unknown"
    y = importlib.import_module("yet-another-raytracer_b200")
    ctx = y.Context(0)
    dev = torch.device("cuda", 0)
    lines = []

    def emit(rec):
        rec["card"] = card
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    def device_pair(name, rays, target, t_min, t_max):
        n = len(rays)
        r64 = torch.from_numpy(rays.view(np.uint8)).to(dev)
        r32 = np.empty(n, dtype=y.abi.RAY_F32_DTYPE)
        r32["origin"], r32["direction"] = rays["origin"], rays["direction"]
        r32d = torch.from_numpy(r32.view(np.uint8)).to(dev)
        flags = torch.empty(n, dtype=torch.uint8, device=dev)
        hits = torch.empty(n * 40, dtype=torch.uint8, device=dev)
        for rec, occ, ch in (
                ("f64", lambda: ctx.occluded_device(r64.data_ptr(), n, flags.data_ptr(), target, t_min, t_max).gpu_ms,
                 lambda: ctx.closest_hit_device(r64.data_ptr(), n, hits.data_ptr(), target, t_min, t_max, y.ORDER_NEAR).gpu_ms),
                ("f32", lambda: ctx.occluded_f32_device(r32d.data_ptr(), n, flags.data_ptr(), target, t_min, t_max).gpu_ms,
                 lambda: ctx.closest_hit_f32_device(r32d.data_ptr(), n, hits.data_ptr(), target, t_min, t_max, y.ORDER_NEAR).gpu_ms)):
            so, sc = alternate(occ, ch, args.reps)
            frac = float(flags.float().mean().item())
            emit({"set": name, "records": rec, "arrays": "device", "n": n, "occluded_fraction": frac,
                  "occluded": so, "closest_hit_near": sc, "speedup_median": sc["median_ms"] / so["median_ms"],
                  "occluded_mrays_s": n / so["median_ms"] / 1e3, "closest_hit_mrays_s": n / sc["median_ms"] / 1e3})

    ms = bench.MeshOnlyScene(y, "david")
    for kind in ("uniform", "axis", "path"):
        rays = bench.sweep_rays(y, "david", kind, args.n, ctx)
        ctx.set_scene(ms.desc)
        device_pair("david_" + kind, rays, 0, 0.0, INF)
    preset = y.ScenePreset("david", seed=3)
    ctx.set_scene(preset)
    srays, t_max = shadow_rays(y, ctx, preset, 1920, 1080)
    device_pair("david_preset_shadow", srays, y.TARGET_WORLD, 0.001, t_max)

    # host arrays end to end: page-locked f32 records and outputs, the call's wall-clock (it returns with the results)
    ctx.set_scene(ms.desc)
    rays = bench.sweep_rays(y, "david", "uniform", args.n, ctx)
    r32 = np.empty(len(rays), dtype=y.abi.RAY_F32_DTYPE)
    r32["origin"], r32["direction"] = rays["origin"], rays["direction"]
    flags = np.empty(len(rays), dtype=np.uint8)
    hits = np.empty(len(rays), dtype=y.abi.HIT_F32_DTYPE)
    for a in (r32, flags, hits):
        ctx.host_register(a)
    try:
        def wall(fn):
            t0 = time.perf_counter()
            fn()
            return (time.perf_counter() - t0) * 1e3
        so, sc = alternate(lambda: wall(lambda: ctx.occluded_f32(r32, 0, 0.0, INF, out=flags)),
                           lambda: wall(lambda: ctx.closest_hit_f32(r32, 0, 0.0, INF, y.ORDER_NEAR, hits=hits)), args.reps)
        emit({"set": "david_uniform", "records": "f32", "arrays": "host pinned (wall-clock)", "n": len(rays),
              "occluded_fraction": float(flags.mean()), "occluded": so, "closest_hit_near": sc,
              "speedup_median": sc["median_ms"] / so["median_ms"],
              "occluded_mrays_s": len(rays) / so["median_ms"] / 1e3, "closest_hit_mrays_s": len(rays) / sc["median_ms"] / 1e3})
    finally:
        for a in (r32, flags, hits):
            ctx.host_unregister(a)
    with open(out_dir / "occlusion_probe.jsonl", "a") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
