#!/usr/bin/env python3
"""What YART_FLAG_NEXT_EVENT costs and what it buys, against the flag-off renderer with the unbiased light pick.

    python tools/nee_probe.py --out DIR [--reps 5] [--ref-spp 16384]

Cost: david at 1920x1080 (16 spp per call) and cornell-box at 600x600 (64 spp per call), both estimators alternating
--reps times after a warm-up; the library's own CUDA events (stats.gpu_ms, stats.trace_ms).  Path rays come from
stats.rays; shadow rays from one more run with YART_DEBUG_BOUNCES=1, which prints them per bounce.  The path rays of
the two estimators are the same, so the extra closest-hit time of the shadow passes is trace_ms(on) - trace_ms(off),
and the whole extra cost (passes, k_nee_resolve, the heavier shading) is gpu_ms(on) - gpu_ms(off).

Benefit: relMSE of the Y channel against a --ref-spp flag-off render (seed 1000), at 16 / 64 / 256 spp and seeds
1-3, on cornell-box 300x300 and david 480x270 (smaller frames, so that the reference fits in the run).  For an
unbiased estimator relMSE ~ V / spp; V is fitted from those points, and the time to reach an error e is
ms_per_spp * V / e with ms_per_spp from the full-size cost runs.  The equal-error time ratio on / off does not depend
on e.  (The reference's own noise adds V_ref / ref_spp to every point; at 16k spp it is below 2 % of the 256-spp
error.)

JSON lines go to DIR/r3_nee_probe.jsonl, the first one naming the card, its power limit and maximum SM clock."""
import argparse
import importlib
import json
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
y = importlib.import_module("yet-another-raytracer_b200")

UB, NEE = y.FLAG_UNBIASED_LIGHT_PICK, y.FLAG_NEXT_EVENT
COST = [("david", 1920, 1080, 16), ("cornell-box", 600, 600, 64)]
ERROR = [("cornell-box", 300, 300), ("david", 480, 270)]
ERROR_SPP = (16, 64, 256)
SEEDS = (1, 2, 3)


def shadow_rays(scene, w, h, spp):
    """Total shadow rays of one NEE render, from the per-bounce debug print (a process of its own: the switch is read
    once per process)."""
    code = ("import importlib, sys\nsys.path.insert(0, %r)\ny = importlib.import_module('yet-another-raytracer_b200')\n"
            "p = y.ScenePreset(%r, seed=1)\nc = y.Context(0); c.set_scene(p)\n"
            "c.render(p.camera(%d, %d), %d, %d, 0, %d, seed=1, flags=y.FLAG_NEXT_EVENT)\n") % (str(ROOT), scene, w, h, w, h, spp)
    res = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, YART_DEBUG_BOUNCES="1"), capture_output=True,
                         text=True, check=True)
    return sum(int(m) for m in re.findall(r"shadow rays\s+(\d+)", res.stderr))


def cost(ctx, scene, w, h, spp, reps):
    p = y.ScenePreset(scene, seed=1)
    ctx.set_scene(p)
    cam = p.camera(w, h)
    runs = {UB: [], NEE: []}
    for flags in (UB, NEE):  # warm-up: modules, buffers, occupancy queries
        ctx.render(cam, w, h, 0, spp, seed=1, flags=flags)
    for _ in range(reps):
        for flags in (UB, NEE):
            _, st = ctx.render(cam, w, h, 0, spp, seed=1, flags=flags)
            runs[flags].append(st)
    off, on = runs[UB], runs[NEE]
    med = lambda sts, f: float(np.median([getattr(s, f) for s in sts]))  # noqa: E731
    assert off[0].rays == on[0].rays
    g_off, g_on = med(off, "gpu_ms"), med(on, "gpu_ms")
    t_off, t_on = med(off, "trace_ms"), med(on, "trace_ms")
    spread = lambda sts: float(np.ptp([s.gpu_ms for s in sts]) / np.median([s.gpu_ms for s in sts]))  # noqa: E731
    return {"kind": "cost", "scene": scene, "width": w, "height": h, "spp": spp, "reps": reps,
            "ms_per_spp_off": g_off / spp, "ms_per_spp_on": g_on / spp, "slowdown": g_on / g_off,
            "spread_off": spread(off), "spread_on": spread(on),
            "path_rays": int(on[0].rays), "shadow_rays": shadow_rays(scene, w, h, spp),
            "shadow_pass_share_of_step": (t_on - t_off) / g_on, "nee_share_of_step": (g_on - g_off) / g_on,
            "trace_ms_off": t_off, "trace_ms_on": t_on}


def error(ctx, scene, w, h, ref_spp, ms_per_spp):
    p = y.ScenePreset(scene, seed=1)
    ctx.set_scene(p)
    cam = p.camera(w, h)
    ref, _ = ctx.render(cam, w, h, 0, ref_spp, seed=1000, flags=UB)
    ref = ref[..., 1] / ref_spp
    denom = float((ref ** 2).mean())
    out = {"kind": "equal_error", "scene": scene, "width": w, "height": h, "ref_spp": ref_spp, "seeds": list(SEEDS)}
    v = {}
    for name, flags in (("off", UB), ("on", NEE)):
        pts = {}
        for spp in ERROR_SPP:
            errs = []
            for seed in SEEDS:
                f, _ = ctx.render(cam, w, h, 0, spp, seed=seed, flags=flags)
                errs.append(float(((f[..., 1] / spp - ref) ** 2).mean() / denom))
            pts[spp] = float(np.mean(errs))
        # least squares of relMSE = V / spp through the points
        xs = np.array([1.0 / s for s in ERROR_SPP])
        v[name] = float((xs * np.array([pts[s] for s in ERROR_SPP])).sum() / (xs ** 2).sum())
        out["relmse_" + name] = {str(k): val for k, val in pts.items()}
        out["V_" + name] = v[name]
    out["relmse_ratio_at_equal_spp"] = v["on"] / v["off"]
    out["ms_per_spp_off"], out["ms_per_spp_on"] = ms_per_spp
    out["equal_error_time_ratio"] = (ms_per_spp[1] * v["on"]) / (ms_per_spp[0] * v["off"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ref-spp", type=int, default=16384)
    args = ap.parse_args()
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [{"kind": "card", "card": gpu[0] if gpu else "unknown"}]
    ctx = y.Context(0)
    per_spp = {}
    for scene, w, h, spp in COST:
        r = cost(ctx, scene, w, h, spp, args.reps)
        per_spp[scene] = (r["ms_per_spp_off"], r["ms_per_spp_on"])
        lines.append(r)
        print(json.dumps(r), flush=True)
    for scene, w, h in ERROR:
        r = error(ctx, scene, w, h, args.ref_spp, per_spp[scene])
        lines.append(r)
        print(json.dumps(r), flush=True)
    ctx.close()
    with open(out_dir / "r3_nee_probe.jsonl", "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
