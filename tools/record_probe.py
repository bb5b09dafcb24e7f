#!/usr/bin/env python3
"""yart_closest_hit_records next to yart_closest_hit in one process, on the same rays: what the whole HitRecord costs.

    python tools/record_probe.py --out DIR [--reps 7] [--n 16777216]

Device arrays: the library's own CUDA events (stats.gpu_ms: traversal + export).  Host arrays: page-locked rays, times
and outputs, the wall-clock of the whole call (it returns with the results).  Every set is warmed up, then the two
calls alternate for --reps repetitions; median and best are reported, and the spread of each as (max - min) / median.
Sets:
  * 16 Mi david uniform and path rays (bench.sweep_rays), mesh target, both orders;
  * next-week-final camera rays with their own times (groups, media, a MovingSphere), world target, both orders
    (yart_closest_hit traces them at time 0; the work is the same but for the one moving object).
JSON lines go to DIR/record_probe.jsonl together with the card's name, power limit and maximum SM clock."""
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
import bench  # noqa: E402  (sweep_rays, MeshOnlyScene: the benchmark's own ray sets)

INF = float("inf")


def stats(xs):
    xs = np.asarray(xs, dtype=np.float64)
    med = float(np.median(xs))
    return {"median_ms": med, "best_ms": float(xs.min()), "spread": float((xs.max() - xs.min()) / med)}


def alternate(rec, ch, reps, warm=3):
    for _ in range(warm):
        rec()
        ch()
    a, b = [], []
    for _ in range(reps):
        a.append(rec())
        b.append(ch())
    return stats(a), stats(b)


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


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

    def pair(name, rays, times, target, t_min, t_max):
        n = len(rays)
        rd = torch.from_numpy(rays.view(np.uint8)).to(dev)
        td = torch.from_numpy(times).to(dev) if times is not None else None
        recs_d = torch.empty(n * 88, dtype=torch.uint8, device=dev)
        hits_d = torch.empty(n * 40, dtype=torch.uint8, device=dev)
        recs = np.empty(n, dtype=y.RECORD_DTYPE)
        hits = np.empty(n, dtype=y.HIT_DTYPE)
        tms = np.ascontiguousarray(times) if times is not None else None
        pinned = [a for a in (rays, tms, recs, hits) if a is not None]
        for order in (y.ORDER_REFERENCE, y.ORDER_NEAR):
            sr, sc = alternate(
                lambda: ctx.closest_hit_records_device(rd.data_ptr(), td.data_ptr() if td is not None else 0, n,
                                                       recs_d.data_ptr(), target, t_min, t_max, order).gpu_ms,
                lambda: ctx.closest_hit_device(rd.data_ptr(), n, hits_d.data_ptr(), target, t_min, t_max, order).gpu_ms,
                args.reps)
            emit({"set": name, "order": order, "arrays": "device (stats.gpu_ms)", "n": n, "times": times is not None,
                  "records": sr, "closest_hit": sc, "cost_median": sr["median_ms"] / sc["median_ms"] - 1.0,
                  "records_mrays_s": n / sr["median_ms"] / 1e3, "closest_hit_mrays_s": n / sc["median_ms"] / 1e3})
        for a in pinned:
            ctx.host_register(a)
        try:
            for order in (y.ORDER_REFERENCE, y.ORDER_NEAR):
                sr, sc = alternate(lambda: wall(lambda: ctx.closest_hit_records(rays, tms, target, t_min, t_max, order, out=recs)),
                                   lambda: wall(lambda: ctx.closest_hit(rays, target, t_min, t_max, order, hits=hits)),
                                   args.reps)
                emit({"set": name, "order": order, "arrays": "host pinned (wall-clock)", "n": n, "times": times is not None,
                      "records": sr, "closest_hit": sc, "rate_ratio_median": sc["median_ms"] / sr["median_ms"],
                      "records_mrays_s": n / sr["median_ms"] / 1e3, "closest_hit_mrays_s": n / sc["median_ms"] / 1e3})
        finally:
            for a in pinned:
                ctx.host_unregister(a)
        # the same answer in both forms
        hits_dev = np.frombuffer(hits_d.cpu().numpy().tobytes(), dtype=y.HIT_DTYPE)
        assert np.array_equal(hits["obj_id"], hits_dev["obj_id"])
        del rd, td, recs_d, hits_d
        torch.cuda.empty_cache()

    ms = bench.MeshOnlyScene(y, "david")
    for kind in ("uniform", "path"):
        rays = bench.sweep_rays(y, "david", kind, args.n, ctx)
        ctx.set_scene(ms.desc)
        pair("david_" + kind, rays, None, 0, 0.0, INF)
        del rays
    preset = y.ScenePreset("next-week-final", seed=1)
    ctx.set_scene(preset)
    w, h, spp = 1024, 1024, 4
    rays, _, times = ctx.camera_rays(preset.camera(w, h), w, h, 0, spp)
    pair("next_week_final_camera_%dx%dx%d" % (w, h, spp), rays, times, y.TARGET_WORLD, 0.001, INF)
    with open(out_dir / "record_probe.jsonl", "a") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
