#!/usr/bin/env python3
"""bench.py -- the headline measurement of the path-tracing hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload render|sweep] [--total-spp S]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload `render` (default; BASELINE.json configs[2], the one its `metric` is quoted on): the `david` preset
(david.obj, 46,664 triangles, white Lambertian mesh + a rotated glass instance + 5 sphere lights) at 1920x1080,
max-depth 50.  A STEP is one wavefront pass of the hot path over one batch: 128 samples of every pixel of the frame
= 265 M camera paths, ~947 M world rays, with the scene resident in HBM; K = 8 steps is the whole 1024-spp job.
With N GPUs every rank renders its own sample range each step (scene replicated, WEAK scaling: per-GPU work is
fixed) and the f64 XYZ films are combined inside every step by the library's own collective
(yart_film_reduce: one in-place ncclReduce over NVLink).  After the timed steps the line also carries the STRONG
scaling number `time_to_image`: the fixed 1024-spp frame split over the N ranks, reduced and finalised to RGBA8.
`--total-spp S` makes that fixed job the step itself (scaling "strong").

At N = 1 the line also carries `other_configs`: BASELINE.json's C1 / C2 / C4 / C5 once each (device time).

Workload `sweep` (BASELINE.json configs[4]): 16 Mi incoherent rays against the david / sycee QBVH -- the reference's
bench ray generators (qbvh.rs:949-986): uniform and axis-aligned sets, plus the renderer's own path rays -- in both
traversal orders, Mrays/s against the fetch roofline.

All timing is on the device (CUDA events on the launching stream), max over ranks.  Rank 0 prints ONE JSON line.
`--dump-outputs DIR` makes rank 0 write, after the timed steps, what the timed path computed in its last step as
DIR/<name>.npy (see OutputDump), so that two builds run with the same arguments can be compared output for output.
`--impl reference` times the CPU oracle -- our C++ restatement of the reference's renderer (the Rust original cannot
be built here) -- on all host cores on bounded samples of the same workload.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

SCENE = "david"
WIDTH, HEIGHT, MAX_DEPTH, TOTAL_SPP = 1920, 1080, 50, 1024
SPP_PER_STEP = 128  # one wavefront batch: 265 M paths in flight, 30 GB of path state (of 180 GB)
SEED = 1
METRIC = "Mrays/s (primary+secondary) on david.obj 1920x1080 max-depth 50"
SWEEP_METRIC = "Mrays/s, 16 Mi incoherent closest-hit rays vs the david.obj QBVH (uniform set, near-first order)"
SWEEP_N = 1 << 24
# bytes one ray moves besides node/triangle fetches: 48 B ray + 8 B time + 4 B queue entry read,
# 32 B hit record written (DESIGN.md "Algorithmic bytes")
STREAM_BYTES_PER_RAY = 92
SWEEP_STREAM_BYTES_PER_RAY = 88  # standalone query: 48 B ray in + 40 B hit out
NODE_BYTES, TRI_BYTES = 128, 48
STATE_BYTES_PER_PATH = 112


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """SM clock + clock-event (throttle) reasons during the timed region, one sample per second (B200_PROFILING.md's
    clocks line).  Read through NVML inside this process (pynvml: two light queries per sample); a spawned
    `nvidia-smi --query-gpu=... -lms` is the fallback.  Why not nvidia-smi first: on some boxes each of its queries (it
    also read power.draw) held a driver lock long enough to stall this launch-heavy step -- 1.5 % of a step at 5 Hz on
    one box, 11 % at 1 Hz on another, while the untimed-by-sampler e2e leg of the same run was unaffected."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
    Q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.proc = None
        self.lines = []
        self.sm, self.mx, self.reasons = [], [], set()
        self.handle = None
        self.how = None
        self._stop = threading.Event()
        self._thread = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
            phys = int(vis[self.idx]) if self.idx < len(vis) else self.idx
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def start(self):
        try:
            self.nv, self.handle = self._nvml_handle()
            self._sample_nvml()  # (fails here, not in the thread, if a query is unsupported)
            self.sm, self.mx = [], []
            self.how = "nvml"
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
            return
        except Exception:
            self.handle = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "1000"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi"
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _sample_nvml(self):
        nv, h = self.nv, self.handle
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
        get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        mask = int(get(h))
        for name, bit in self.REASONS:
            if mask & bit:
                self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml()
            except Exception:
                pass
            self._stop.wait(1.0)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.handle is not None:
            self._stop.set()
            self._thread.join(timeout=2.0)
        elif self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            for ln in self.lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 8:
                    continue
                try:
                    self.sm.append(float(f[1]))
                    self.mx.append(float(f[2]))
                except ValueError:
                    continue
                for (name, _), v in zip(self.REASONS, f[4:8]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["neither NVML nor nvidia-smi available"]}
        sm, mx = self.sm, self.mx
        busy = [x for x in sm if x > 0.5 * max(mx + [1.0])] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(self.reasons), "samples": len(sm), "source": self.how}


def warm_up(step, at_least, seconds=0.3):
    """`at_least` untimed calls of a (synchronous) step, and as many more as it takes to keep the GPU busy for `seconds`:
    a 5 ms sweep step after seconds of host-side ray generation starts at idle clocks, and three of them are not
    enough to get back to the boost clock the timed region is then sampled at."""
    t0, n = time.perf_counter(), 0
    while n < at_least or time.perf_counter() - t0 < seconds:
        step()
        n += 1
    return n


def profiled_traffic():
    """DRAM bytes per ray per k_traverse launch from the committed ncu --set full capture (a PROFILED CONSTANT: ncu's
    numbers cannot be taken live inside a bench run).  Newest round first."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            d = json.loads((ROOT / "profiles" / name).read_text())
            return float(d["dram_bytes_per_ray_per_launch"]), "profiles/" + name
        except Exception:
            continue
    return None, None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def load_pkg():
    pkg = importlib.import_module("yet-another-raytracer_b200")
    pkg.load_library()
    return pkg


DUMP_MAX_BYTES = 64 << 20
DUMP_SWEEP_SAMPLE = 1 << 16  # rays per sweep row whose hits are written (a fixed, seeded sample of the 16 Mi)


class OutputDump:
    """--dump-outputs DIR: float32 / float64 arrays as DIR/<name>.npy, at most DUMP_MAX_BYTES in all.

    render: `film` -- the (H, W, 3) f64 XYZ film the timed steps accumulated into, as the caller holds it after the last
            step (with --total-spp: `rgba`, the (H, W, 4) finalised frame the last step read back); `last_step_counts` --
            [rays, paths] of that step.
    sweep:  `<mesh>_<rays>_<order>_hits` per row -- columns t, u, v, prim_id, obj_id, front_face of the hits the last
            timed step wrote for the rays at `sweep_sample_index`; `david_uniform_near_f32_hits` -- t, u, v, prim_id of
            yart_closest_hit_f32 on the same sample.  A miss is stored as the library returns it: t = +inf, ids MISS."""

    def __init__(self, path):
        self.dir = Path(path)
        self.dir.mkdir(parents=True, exist_ok=True)
        self.nbytes = 0

    def write(self, name, array):
        a = np.ascontiguousarray(array)
        if a.dtype not in (np.float32, np.float64):
            raise TypeError("%s: dumps are float32 or float64, not %s" % (name, a.dtype))
        self.nbytes += a.nbytes
        if self.nbytes > DUMP_MAX_BYTES:
            raise RuntimeError("--dump-outputs: %s takes the dump past %d bytes" % (name, DUMP_MAX_BYTES))
        np.save(self.dir / (name + ".npy"), a)


def hit_columns(hits, fields=("t", "u", "v", "prim_id", "obj_id", "front_face")):
    """Hit records -> (n, len(fields)) f64 (the u32 ids are exact in f64)."""
    return np.stack([hits[f].astype(np.float64) for f in fields], axis=1)


# ------------------------------------------------------------------------------------------------
# ray sets of the sweep (shared with the tests)
# ------------------------------------------------------------------------------------------------
def sweep_rays(pkg, mesh_name, kind, n, ctx=None):
    """(n,) RAY_DTYPE array.  uniform / axis: the reference's bench generators (qbvh.rs:949-986) on the mesh AABB
    (tests/raysets.py);  path: the world rays the renderer itself traces in the mesh's preset, in wavefront order
    (yart_dump_path_rays), as many 1920x1080 one-sample batches as it takes."""
    sys.path.insert(0, str(ROOT / "tests"))
    import raysets
    if kind in ("uniform", "axis"):
        m = pkg.TriangleMesh.from_obj(os.path.join(pkg.assets_dir(), mesh_name + ".obj"))
        q = pkg.L4QBVH.from_mesh(m)
        gen = raysets.uniform if kind == "uniform" else raysets.axis
        o, d = gen(n, q.info.bbox_min, q.info.bbox_max)
        return pkg.make_rays(o, d)
    preset = pkg.ScenePreset(mesh_name, seed=SEED)
    ctx.set_scene(preset)
    cam = preset.camera(WIDTH, HEIGHT)
    rays, total = ctx.dump_path_rays(cam, WIDTH, HEIGHT, 0, 16, n, MAX_DEPTH, SEED, batch_spp=1)
    if len(rays) < n:
        raise RuntimeError("only %d path rays" % len(rays))
    return rays


class MeshOnlyScene:
    """A one-mesh scene description (a single un-wrapped MESH object), built through the public ABI structs."""

    def __init__(self, pkg, mesh_name):
        import ctypes as C
        abi = pkg.abi
        self.mesh = pkg.TriangleMesh.from_obj(os.path.join(pkg.assets_dir(), mesh_name + ".obj"))
        self.tex, self.mat, self.obj, self.sd = abi.Texture(), abi.Material(), abi.Object(), abi.SceneDesc()
        self.tex.kind = abi.TEX_SOLID
        self.mat.kind = abi.MAT_LAMBERTIAN
        self.obj.kind, self.obj.cos_theta = abi.OBJ_MESH, 1.0
        self.sd.objects, self.sd.n_objects = C.pointer(self.obj), 1
        self.sd.meshes, self.sd.n_meshes = C.pointer(self.mesh.trimesh), 1
        self.sd.materials, self.sd.n_materials = C.pointer(self.mat), 1
        self.sd.textures, self.sd.n_textures = C.pointer(self.tex), 1
        self.desc = C.pointer(self.sd)


# ------------------------------------------------------------------------------------------------
# the reference arm: the CPU oracle (port of the reference's renderer) on all host cores
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    pkg = load_pkg()
    from oracle import orc
    orc.build()
    cores = os.cpu_count() or 1
    if args.workload == "sweep":
        ms = MeshOnlyScene(pkg, "david")
        scene = orc.Scene(ms)
        rays = sweep_rays(pkg, "david", "uniform", 1 << 21)
        t0 = time.perf_counter()
        scene.closest_hit(rays[:1 << 16], 0, 0.0, float("inf"), pkg.ORDER_REFERENCE, n_threads=cores)
        rate = (1 << 16) / (time.perf_counter() - t0)
        per_step = int(max(1 << 14, min(len(rays), 120.0 * rate / (args.steps + args.warmup))))

        def step(i):
            lo = (i * per_step) % max(1, len(rays) - per_step + 1)
            scene.closest_hit(rays[lo:lo + per_step], 0, 0.0, float("inf"), pkg.ORDER_REFERENCE, n_threads=cores)
            return per_step

        for i in range(args.warmup):
            step(i)
        t0 = time.perf_counter()
        n = sum(step(args.warmup + i) for i in range(args.steps))
        dt = time.perf_counter() - t0
        val = n / dt / 1e6
        sample = "%d of the 16 Mi uniform rays per step, reference (far-first) order" % per_step
        line = {"impl": "reference", "metric": SWEEP_METRIC, "value": val, "unit": "Mrays/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "sweep: 16 Mi uniform rays vs david.obj QBVH (BASELINE configs[4]); CPU arm: " + sample},
                "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "C++ restatement of the reference's L4QBVH::hit (oracle/), -O3 -march=x86-64-v3; the Rust original cannot be built here"}
        print(json.dumps(line), flush=True)
        return 0
    preset = pkg.ScenePreset(SCENE, seed=SEED)  # host-side scene description only; no GPU involved
    scene = orc.Scene(preset)
    cam = preset.camera(WIDTH, HEIGHT)
    film = np.zeros((HEIGHT, WIDTH, 3))
    # size a step so that (K + W) steps take about two minutes: probe the rate on two tiles
    t0 = time.perf_counter()
    _, st = scene.render(cam, WIDTH, HEIGHT, 0, 1, MAX_DEPTH, SEED, 0, cores, film, tiles=(27, 29))
    rate_paths = st.paths / (time.perf_counter() - t0)
    paths_per_tile = (WIDTH // 8) * (HEIGHT // 8)
    budget_s = 120.0
    tiles_per_step = int(max(1, min(64, round(budget_s * rate_paths / (args.steps + args.warmup) / paths_per_tile))))

    def step(i):
        t = (i * tiles_per_step) % 64
        spp0 = (i * tiles_per_step) // 64
        lo, hi = t, min(64, t + tiles_per_step)
        _, s = scene.render(cam, WIDTH, HEIGHT, spp0, spp0 + 1, MAX_DEPTH, SEED, 0, cores, film, tiles=(lo, hi))
        return s.rays, s.paths

    for i in range(args.warmup):
        step(i)
    rays = paths = 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        r, p = step(args.warmup + i)
        rays += r
        paths += p
    dt = time.perf_counter() - t0
    val = rays / dt / 1e6
    sample = "%d of the 64 tiles of one 1920x1080 sample pass per step (%d paths/step), reference traversal order" % (
        tiles_per_step, tiles_per_step * paths_per_tile)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "david 1920x1080 max-depth 50 (BASELINE configs[2]); CPU arm: " + sample,
                   "scene": SCENE, "width": WIDTH, "height": HEIGHT, "max_depth": MAX_DEPTH, "seed": SEED},
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "spp_per_s": paths / dt / (WIDTH * HEIGHT),
        "note": "C++ restatement of the reference (oracle/, g++ -O3 -march=x86-64-v3 -ffp-contract=off, one thread per "
                "tile job), the Rust original cannot be built here",
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# our arm: common set-up
# ------------------------------------------------------------------------------------------------
class Rig:
    """One rank: torch for the device, stream, events and the rendezvous; the library for everything measured."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.rank, self.world, self.local = dist_env()
        if args.gpus != self.world and self.world > 1:
            raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, self.world))
        if self.world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one process per GPU)")
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
                os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self.pkg = load_pkg()
        self.ctx = self.pkg.Context(self.local)
        self.stream = torch.cuda.current_stream()
        self.ctx.set_stream(self.stream.cuda_stream)  # torch events then time exactly the stream the kernels run on
        self.comm = None
        if self.world > 1:
            # the library's own communicator (yart_comm_init_rank); torch.distributed only carries the 128-byte id
            box = [self.pkg.comm_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(box, src=0)
            self.comm = self.pkg.Comm.from_id(self.ctx, box[0], self.rank, self.world)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)

    def reduce_max_sum(self, sums, maxes):
        torch = self.torch
        tot = torch.tensor(sums, dtype=torch.float64, device="cuda")
        tmax = torch.tensor(maxes, dtype=torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(tot)
            self.dist.all_reduce(tmax, op=self.dist.ReduceOp.MAX)
        return tot.tolist(), tmax.tolist()

    def close(self):
        if self.comm is not None:
            self.comm.close()
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()
        self.ctx.close()


def fetch_peaks(ctx):
    """The fetch rooflines of SURVEY.md 8(d), measured live (untimed, ~0.1 s): random whole-line (128 B = one node
    visit) fetches, at FULL occupancy (mode 1: the hardware's roof) and at k_traverse's own occupancy (mode 0)."""
    out = {}
    for name, size in (("l1_resident", 128 * 1024), ("scene_sized_l2_resident", 7_400_000)):
        out[name + "_gbs"] = max(ctx.measure_fetch_peak(size, 4096, 1) for _ in range(3))
        out[name + "_at_kernel_occupancy_gbs"] = max(ctx.measure_fetch_peak(size, 4096, 0) for _ in range(3))
    return out


def other_configs(rig):
    """BASELINE.json's other configs once each, so that the driver's own record carries them (N = 1 only; ~5 s):
    C1 cornell-box 400x400x32, C2 bunny preset 1280x720x256, C4 next-week-final 1920x1080 (16 of its 1024 spp),
    C5 the 16 Mi-ray david sweep (uniform set, both orders).  Device time of the library's own CUDA events; parity of
    every one of them with the oracle is what tests/test_gpu_baseline_configs.py asserts."""
    torch, pkg, ctx = rig.torch, rig.pkg, rig.ctx
    out = {}
    for tag, scene, w, h, spp, note in (("C1", "cornell-box", 400, 400, 32, "the whole config"),
                                        ("C2", "bunny", 1280, 720, 256, "the whole config; sycee.obj stands in for the unshipped bunny.obj"),
                                        ("C4", "next-week-final", 1920, 1080, 16, "16 of the config's 1024 spp")):
        p = pkg.ScenePreset(scene, seed=SEED)
        ctx.set_scene(p)
        cam = p.camera(w, h)
        film = ctx.film_create(w, h)
        ctx.render_device(cam, w, h, 0, min(spp, 4), film, MAX_DEPTH, SEED)  # warm
        ctx.film_clear(film, w, h)
        st = ctx.render_device(cam, w, h, 0, spp, film, MAX_DEPTH, SEED)
        ctx.film_destroy(film)
        out[tag] = {"scene": scene, "width": w, "height": h, "spp": spp, "mrays_per_s": st.rays / st.gpu_ms / 1e3,
                    "ms": st.gpu_ms, "rays_per_sample": st.rays / st.paths, "note": note}
    ms_scene = MeshOnlyScene(pkg, "david")
    ctx.set_scene(ms_scene.desc)
    rays = sweep_rays(pkg, "david", "uniform", SWEEP_N)
    d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()
    d_hits = torch.empty(SWEEP_N * 40, dtype=torch.uint8, device="cuda")
    c5 = {"mesh": "david", "rays": "uniform, 16 Mi (qbvh.rs:973-986)"}
    for order, oname in ((pkg.ORDER_NEAR, "near"), (pkg.ORDER_REFERENCE, "reference")):
        stc = ctx.closest_hit_device(d_rays.data_ptr(), SWEEP_N, d_hits.data_ptr(), 0, 0.0, float("inf"), order, count_visits=True)
        best = min(ctx.closest_hit_device(d_rays.data_ptr(), SWEEP_N, d_hits.data_ptr(), 0, 0.0, float("inf"), order).gpu_ms
                   for _ in range(4))
        bpr = (NODE_BYTES * stc.node_visits + TRI_BYTES * stc.tri_tests) / SWEEP_N + SWEEP_STREAM_BYTES_PER_RAY
        c5[oname] = {"mrays_per_s": SWEEP_N / best / 1e3, "ms": best, "nodes_per_ray": stc.node_visits / SWEEP_N,
                     "tris_per_ray": stc.tri_tests / SWEEP_N, "bytes_per_ray": bpr, "algorithmic_gbs": bpr * SWEEP_N / best / 1e6}
    out["C5"] = c5
    del d_rays, d_hits
    return out


# ------------------------------------------------------------------------------------------------
# our arm: render
# ------------------------------------------------------------------------------------------------
def run_render(args):
    rig = Rig(args)
    torch, pkg, ctx, rank, N = rig.torch, rig.pkg, rig.ctx, rig.rank, rig.world
    sharding = importlib.import_module("yet-another-raytracer_b200.sharding")
    preset = pkg.ScenePreset(SCENE, seed=SEED)
    ctx.set_scene(preset)
    cam = preset.camera(WIDTH, HEIGHT)
    order = pkg.ORDER_NEAR
    K, W = args.steps, args.warmup
    film = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.float64, device="cuda")
    strong_only = args.total_spp > 0
    job_spp = args.total_spp if strong_only else TOTAL_SPP

    def sample_range(step):  # weak scaling: every rank renders its own SPP_PER_STEP samples per step
        return sharding.step_sample_range(step % (1 << 20), rank, N, SPP_PER_STEP)

    def reduce_film():
        if rig.comm is not None:  # the one real exchange step: in-place ncclReduce of the per-rank f64 XYZ films
            rig.comm.film_reduce(film.data_ptr(), WIDTH, HEIGHT, root=0)

    rgba = torch.empty((HEIGHT, WIDTH, 4), dtype=torch.uint8, device="cuda")
    rgba_host = torch.empty((HEIGHT, WIDTH, 4), dtype=torch.uint8).pin_memory()

    def whole_job(spp_total):
        """The fixed job (strong scaling): this rank's share of spp_total samples of every pixel, the film reduce,
        and on the root the finalisation to RGBA8 + its copy to the host.  Returns (rays, paths, launches)."""
        film.zero_()
        lo, hi = sharding.shard_range(0, spp_total, rank, N)
        rays = paths = launches = 0
        if hi > lo:
            st = ctx.render_device(cam, WIDTH, HEIGHT, lo, hi, film.data_ptr(), MAX_DEPTH, SEED, order, SPP_PER_STEP)
            rays, paths, launches = st.rays, st.paths, st.kernel_launches
        reduce_film()
        if rank == 0:
            ctx.film_finalize_device(film.data_ptr(), WIDTH, HEIGHT, spp_total, rgba.data_ptr())
            rgba_host.copy_(rgba, non_blocking=True)
        return rays, paths, launches + 1

    # ---- algorithmic bytes per ray of this workload: visit counts from one untimed counted step ----
    s0, s1 = sample_range(0)
    stc = ctx.render_device(cam, WIDTH, HEIGHT, s0, s1, film.data_ptr(), MAX_DEPTH, SEED, order, SPP_PER_STEP,
                            count_visits=True)
    nodes_per_ray = stc.node_visits / stc.rays
    tris_per_ray = stc.tri_tests / stc.rays
    bytes_per_ray = NODE_BYTES * nodes_per_ray + TRI_BYTES * tris_per_ray + STREAM_BYTES_PER_RAY
    film.zero_()
    for i in range(W):
        if strong_only:
            whole_job(job_spp)
        else:
            s0, s1 = sample_range(i)
            ctx.render_device(cam, WIDTH, HEIGHT, s0, s1, film.data_ptr(), MAX_DEPTH, SEED, order, SPP_PER_STEP)
            reduce_film()
    film.zero_()

    # ---- timed region 1: device-resident (`value`) ----
    sampler = ClockSampler(rig.local) if rank == 0 else None
    if sampler:
        sampler.start()
    ev0, ev1 = rig.event(), rig.event()
    rig.barrier()
    ev0.record(rig.stream)
    rays = paths = launches = trace_launches = 0
    trace_ms = 0.0
    for i in range(K):
        if strong_only:
            r, p, l = whole_job(job_spp)
            rays, paths, launches = rays + r, paths + p, launches + l
        else:
            s0, s1 = sample_range(W + i)
            st = ctx.render_device(cam, WIDTH, HEIGHT, s0, s1, film.data_ptr(), MAX_DEPTH, SEED, order, SPP_PER_STEP)
            reduce_film()
            rays += st.rays
            paths += st.paths
            launches += st.kernel_launches + (1 if rig.comm is not None else 0)
            trace_launches += st.trace_launches
            trace_ms += st.trace_ms
    ev1.record(rig.stream)
    rig.barrier()
    clocks = sampler.stop() if sampler else None
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:  # before the legs below reuse the film
        dump = OutputDump(args.dump_outputs)
        if strong_only:
            dump.write("rgba", rgba_host.numpy().astype(np.float32))
        else:
            dump.write("film", film.cpu().numpy())
        last = (r, p) if strong_only else (st.rays, st.paths)
        dump.write("last_step_counts", np.array(last, dtype=np.float64))

    # ---- timed region 2: end to end through the C ABI with HOST buffers (`e2e`) ----
    K2 = min(K, 8)
    rays2, ms2, luminance = 0, 0.0, None
    film_bytes = HEIGHT * WIDTH * 3 * 8
    if not strong_only:
        host_film = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.float64).pin_memory()
        hf = host_film.numpy()
        ctx.render(cam, WIDTH, HEIGHT, 0, SPP_PER_STEP, MAX_DEPTH, SEED, order, SPP_PER_STEP, film=hf)  # warm the path
        hf[...] = 0.0
        rig.barrier()
        e0, e1 = rig.event(), rig.event()
        e0.record(rig.stream)
        for i in range(K2):
            s0, s1 = sample_range(W + K + i)
            _, st = ctx.render(cam, WIDTH, HEIGHT, s0, s1, MAX_DEPTH, SEED, order, SPP_PER_STEP, film=hf)
            rays2 += st.rays
        e1.record(rig.stream)
        rig.barrier()
        ms2 = e0.elapsed_time(e1)
        luminance = float(hf[..., 1].sum())  # the host-side result the caller reads

    # ---- strong scaling: time to image of the fixed 1024-spp frame over the N ranks ----
    tti = None
    if not strong_only and not args.no_time_to_image:
        whole_job(N * 8)  # warm the shard shapes
        rig.barrier()
        t0, t1 = rig.event(), rig.event()
        t0.record(rig.stream)
        jr, jp, _ = whole_job(TOTAL_SPP)
        t1.record(rig.stream)
        rig.barrier()
        (jr_all, jp_all), (tti_ms,) = rig.reduce_max_sum([jr, jp], [t0.elapsed_time(t1)])
        tti = {"spp": TOTAL_SPP, "seconds": tti_ms * 1e-3, "n_gpus": N, "mrays_per_s": jr_all / tti_ms / 1e3,
               "rays": int(jr_all), "scaling": "strong",
               "what": "the fixed 1920x1080 %d-spp frame: %d samples per GPU, in-place ncclReduce of the f64 film "
                       "(yart_film_reduce), finalisation to RGBA8 and its 8.3 MB copy to the host on rank 0; device "
                       "time, max over ranks" % (TOTAL_SPP, -(-TOTAL_SPP // N))}

    # ---- combine over ranks: totals summed, time = max ----
    (all_rays, all_paths, all_rays2, all_launches), (ms, ms2, trace_ms_max) = rig.reduce_max_sum(
        [rays, paths, rays2, launches], [ms, ms2, trace_ms])
    value = all_rays / ms / 1e3

    cpu_baseline = None
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        from oracle import orc
        orc.build()
        cores = os.cpu_count() or 1
        oscene = orc.Scene(preset)
        ofilm = np.zeros((HEIGHT, WIDTH, 3))
        t0 = time.perf_counter()
        _, ost = oscene.render(cam, WIDTH, HEIGHT, 0, 1, MAX_DEPTH, SEED, 0, cores, ofilm)
        probe = time.perf_counter() - t0  # one full 1920x1080 sample pass
        n_spp = int(max(1, min(32, round(15.0 / max(probe, 1e-3)))))  # ~15 s of CPU work
        t0 = time.perf_counter()
        _, ost = oscene.render(cam, WIDTH, HEIGHT, 1, 1 + n_spp, MAX_DEPTH, SEED, 0, cores, ofilm)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": ost.rays / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                        "sample": "%d spp of the 1920x1080 frame (%d paths, %d rays, %.1f s of the 1024-spp job), "
                                  "C++ restatement of the reference (g++ -O3 -march=x86-64-v3) on %d threads, reference "
                                  "traversal order" % (n_spp, ost.paths, ost.rays, dt, cores)}

    configs = None
    if rank == 0 and N == 1 and not strong_only and not args.no_other_configs:
        configs = other_configs(rig)
        ctx.set_scene(preset)

    if rank == 0:
        peak, peak_src = measured_peaks()
        fp = fetch_peaks(ctx)
        roofline = None
        if not strong_only:
            trace_launches = max(1, trace_launches)
            # closest-hit launches per bounce: one k_traverse per mesh instance (+ one k_analytic per run of analytic
            # objects that k_shade does not take over); david: 2
            passes = max(1, round(trace_launches / float(K * MAX_DEPTH)))
            achieved = bytes_per_ray * rays / (trace_ms * 1e-3) / 1e9 if trace_ms > 0 else None
            traffic_per_ray, traffic_src = profiled_traffic()
            roofline = {
                "bound": "hbm", "kernel": "closest-hit stage: k_traverse, %d launches per bounce (one per mesh instance)" % passes,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": (traffic_per_ray * rays / (trace_launches / float(passes))) if traffic_per_ray else None,
                "traffic_note": "PROFILED CONSTANT, not measured in this run: %s B of DRAM read+write per ray per k_traverse launch "
                                "(ncu --set full capture, %s) x this run's average rays per launch; ~20x below the algorithmic "
                                "bytes because node/triangle fetches are L1/L2 hits" % (traffic_per_ray, traffic_src),
                "fetch_peaks": dict(fp, **{
                    "frac_of_l2_resident_fetch_peak": (achieved / fp["scene_sized_l2_resident_gbs"]) if achieved else None,
                    "frac_of_l1_resident_fetch_peak": (achieved / fp["l1_resident_gbs"]) if achieved else None,
                    "note": "yart_measure_fetch_peak mode 1 (full occupancy; the roof) and mode 0 (k_traverse_lean's 20 warps/SM): every "
                            "lane fetches whole 128-B lines (four LDG.E.256) at independent random positions of an L1-sized / "
                            "scene-sized table"}),
                "peak_source": peak_src, "bytes_per_ray": bytes_per_ray, "nodes_per_ray": nodes_per_ray,
                "tris_per_ray": tris_per_ray, "trace_launches": int(trace_launches),
                "avg_launch_ms": trace_ms / trace_launches, "trace_share_of_step": trace_ms / ms if ms else None,
                "note": "algorithmic bytes = 128 B x nodes + 48 B x triangles visited (counted on this workload, "
                        "equal to the oracle's counts) + 92 B of ray/hit stream; node and triangle fetches are "
                        "served by L1/L2 (the tree is 5.9 MB), so the HBM fraction is a conservative denominator and the "
                        "kernel's real limiter is fetch latency at its occupancy (see fetch_peaks)",
            }
        workload = ("david 1920x1080 max-depth 50, STRONG scaling: the fixed %d-spp frame per step split over %d GPU(s), reduce + "
                    "finalise + readback inside the step" % (job_spp, N)) if strong_only else (
            "david 1920x1080 max-depth 50, %d spp per step per GPU (BASELINE configs[2]; K=%d steps = the 1024-spp job)" % (
                SPP_PER_STEP, TOTAL_SPP // SPP_PER_STEP))
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if strong_only else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": workload, "scene": SCENE, "width": WIDTH, "height": HEIGHT, "max_depth": MAX_DEPTH,
                "spp_per_step": job_spp if strong_only else SPP_PER_STEP,
                "spp_total": job_spp * K if strong_only else SPP_PER_STEP * K * N, "seed": SEED,
                "traversal_order": "near (bit-identical hits)",
                "l2": "inputs larger than L2: %.0f GB of path state streams per step; the 7 MB scene is meant to "
                      "stay L2-resident" % (WIDTH * HEIGHT * SPP_PER_STEP * STATE_BYTES_PER_PATH / 1e9),
                "parallelism": "sample-range sharding x%d, scene replicated, one in-place ncclReduce of the f64 film per step "
                               "(yart_film_reduce, C ABI)" % N,
            },
            "spp_per_s": all_paths / (ms * 1e-3) / (WIDTH * HEIGHT),
            "rays_per_sample": all_rays / max(all_paths, 1),
            "e2e": None if strong_only else {
                "value": all_rays2 / ms2 / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": film_bytes + 224,
                "d2h_bytes_per_step": film_bytes, "steps": K2, "ms_per_step": ms2 / K2,
                "host_result_luminance_sum": luminance},
            "time_to_image": tti,
            "other_configs": configs,
            "gpu_launches": int(all_launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }
        if strong_only:
            line["e2e"] = {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 224, "d2h_bytes_per_step": HEIGHT * WIDTH * 4,
                           "note": "strong-scaling steps ARE end to end: camera + options in, the finalised RGBA8 frame read back "
                                   "to pinned host memory inside every step"}
        print(json.dumps(line), flush=True)
    rig.close()
    return 0


# ------------------------------------------------------------------------------------------------
# our arm: the closest-hit sweep (BASELINE configs[4])
# ------------------------------------------------------------------------------------------------
def run_sweep(args):
    rig = Rig(args)
    torch, pkg, ctx, rank, N = rig.torch, rig.pkg, rig.ctx, rig.rank, rig.world
    K, W = args.steps, args.warmup
    n = SWEEP_N
    lo, hi = importlib.import_module("yet-another-raytracer_b200.sharding").shard_range(0, n, rank, N)
    table, headline = [], None
    d_hits = torch.empty((hi - lo) * 40, dtype=torch.uint8, device="cuda")
    dump = OutputDump(args.dump_outputs) if args.dump_outputs and rank == 0 else None
    if dump is not None:
        sample = np.sort(np.random.default_rng(SEED).choice(hi - lo, min(DUMP_SWEEP_SAMPLE, hi - lo), replace=False))
        dump.write("sweep_sample_index", sample.astype(np.float64))
        d_sample = torch.from_numpy(sample).cuda()
    sampler = ClockSampler(rig.local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches = 0
    for mesh_name in ("david", "sycee"):
        ms_scene = MeshOnlyScene(pkg, mesh_name)
        for kind in ("uniform", "axis", "path"):
            rays = sweep_rays(pkg, mesh_name, kind, n, ctx)  # (the path set needs the preset loaded; re-set the mesh below)
            ctx.set_scene(ms_scene.desc)
            d_rays = torch.from_numpy(rays[lo:hi].view(np.uint8).reshape(-1)).cuda()
            for order, oname in ((pkg.ORDER_NEAR, "near"), (pkg.ORDER_REFERENCE, "reference")):
                stc = ctx.closest_hit_device(d_rays.data_ptr(), hi - lo, d_hits.data_ptr(), 0, 0.0, float("inf"), order,
                                             count_visits=True)
                warm_up(lambda: ctx.closest_hit_device(d_rays.data_ptr(), hi - lo, d_hits.data_ptr(), 0, 0.0, float("inf"), order), W)
                rig.barrier()
                e0, e1 = rig.event(), rig.event()
                e0.record(rig.stream)
                kernel_ms = 0.0
                for _ in range(K):
                    st = ctx.closest_hit_device(d_rays.data_ptr(), hi - lo, d_hits.data_ptr(), 0, 0.0, float("inf"), order)
                    kernel_ms += st.gpu_ms
                    launches += st.kernel_launches
                e1.record(rig.stream)
                rig.barrier()
                if dump is not None:
                    got = d_hits.view(-1, 40)[d_sample].cpu().numpy().reshape(-1).view(pkg.HIT_DTYPE)
                    dump.write("%s_%s_%s_hits" % (mesh_name, kind, oname), hit_columns(got))
                (nodes, tris), (ms, kms) = rig.reduce_max_sum([stc.node_visits, stc.tri_tests], [e0.elapsed_time(e1), kernel_ms])
                bpr = (NODE_BYTES * nodes + TRI_BYTES * tris) / n + SWEEP_STREAM_BYTES_PER_RAY
                row = {"mesh": mesh_name, "rays": kind, "order": oname, "mrays_per_s": n * K / ms / 1e3,
                       "ms_per_step": ms / K, "kernel_ms_per_step": kms / K, "nodes_per_ray": nodes / n, "tris_per_ray": tris / n,
                       "bytes_per_ray": bpr, "algorithmic_gbs": bpr * n * K / (kms * 1e-3) / 1e9}
                table.append(row)
                if (mesh_name, kind, oname) == ("david", "uniform", "near"):
                    headline = dict(row)
                    headline_rays = rays
                    # the f32-record entry point on the same rays rounded to f32 (24 + 16 B per ray instead of 48 + 40)
                    r32 = np.empty(hi - lo, dtype=pkg.abi.RAY_F32_DTYPE)
                    r32["origin"], r32["direction"] = rays["origin"][lo:hi], rays["direction"][lo:hi]
                    d_r32 = torch.from_numpy(r32.view(np.uint8).reshape(-1)).cuda()
                    warm_up(lambda: ctx.closest_hit_f32_device(d_r32.data_ptr(), hi - lo, d_hits.data_ptr(), 0, 0.0, float("inf"), order), W)
                    rig.barrier()
                    f0, f1 = rig.event(), rig.event()
                    f0.record(rig.stream)
                    for _ in range(K):
                        ctx.closest_hit_f32_device(d_r32.data_ptr(), hi - lo, d_hits.data_ptr(), 0, 0.0, float("inf"), order)
                    f1.record(rig.stream)
                    rig.barrier()
                    if dump is not None:
                        got = d_hits[:(hi - lo) * 16].view(-1, 16)[d_sample].cpu().numpy().reshape(-1).view(pkg.abi.HIT_F32_DTYPE)
                        dump.write("david_uniform_near_f32_hits", hit_columns(got, ("t", "u", "v", "prim_id")))
                    _, (fms,) = rig.reduce_max_sum([0.0], [f0.elapsed_time(f1)])
                    headline["f32_records_mrays_per_s"] = n * K / fms / 1e3
                    del d_r32
            del d_rays
    clocks = sampler.stop() if sampler else None

    # ---- e2e: host buffers through the C ABI (805 MB of rays in, 671 MB of hits out per step) ----
    e2e_scene = MeshOnlyScene(pkg, "david")  # (must outlive the call: the description borrows the mesh's arrays)
    ctx.set_scene(e2e_scene.desc)
    K2 = min(K, 4)
    h_rays = torch.from_numpy(headline_rays[lo:hi].view(np.uint8).reshape(-1).copy()).pin_memory()
    h_hits = torch.empty((hi - lo) * 40, dtype=torch.uint8).pin_memory()
    rays_np = h_rays.numpy().view(pkg.RAY_DTYPE)
    hits_np = h_hits.numpy().view(pkg.HIT_DTYPE)
    warm_up(lambda: ctx.closest_hit(rays_np, 0, 0.0, float("inf"), pkg.ORDER_NEAR, hits=hits_np), 1)
    rig.barrier()
    e0, e1 = rig.event(), rig.event()
    e0.record(rig.stream)
    for _ in range(K2):
        ctx.closest_hit(rays_np, 0, 0.0, float("inf"), pkg.ORDER_NEAR, hits=hits_np)
    e1.record(rig.stream)
    rig.barrier()
    _, (ms2,) = rig.reduce_max_sum([0.0], [e0.elapsed_time(e1)])
    hit_rate = float((hits_np["prim_id"] != pkg.MISS).mean())
    # the same through yart_closest_hit_f32: 24 B in + 16 B out per ray
    h_r32 = torch.empty((hi - lo) * 24, dtype=torch.uint8).pin_memory()
    h_h32 = torch.empty((hi - lo) * 16, dtype=torch.uint8).pin_memory()
    r32_np = h_r32.numpy().view(pkg.abi.RAY_F32_DTYPE)
    h32_np = h_h32.numpy().view(pkg.abi.HIT_F32_DTYPE)
    r32_np["origin"], r32_np["direction"] = rays_np["origin"], rays_np["direction"]
    warm_up(lambda: ctx.closest_hit_f32(r32_np, 0, 0.0, float("inf"), pkg.ORDER_NEAR, hits=h32_np), 1)
    rig.barrier()
    g0, g1 = rig.event(), rig.event()
    g0.record(rig.stream)
    for _ in range(K2):
        ctx.closest_hit_f32(r32_np, 0, 0.0, float("inf"), pkg.ORDER_NEAR, hits=h32_np)
    g1.record(rig.stream)
    rig.barrier()
    _, (ms3,) = rig.reduce_max_sum([0.0], [g0.elapsed_time(g1)])

    cpu_baseline = None
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        from oracle import orc
        orc.build()
        cores = os.cpu_count() or 1
        oscene = orc.Scene(e2e_scene)
        t0 = time.perf_counter()
        oscene.closest_hit(headline_rays[:1 << 17], 0, 0.0, float("inf"), pkg.ORDER_REFERENCE, n_threads=cores)
        rate = (1 << 17) / (time.perf_counter() - t0)
        m = int(max(1 << 17, min(n, 12.0 * rate)))
        t0 = time.perf_counter()
        want, _ = oscene.closest_hit(headline_rays[:m], 0, 0.0, float("inf"), pkg.ORDER_REFERENCE, n_threads=cores)
        dt = time.perf_counter() - t0
        same = all(np.array_equal(want[f], hits_np[f][:m]) for f in ("t", "u", "v", "prim_id")) if lo == 0 else None
        cpu_baseline = {"value": m / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                        "sample": "the first %d of the 16 Mi uniform rays (%.1f s), C++ restatement of L4QBVH::hit "
                                  "(g++ -O3 -march=x86-64-v3) on %d threads, reference order" % (m, dt, cores),
                        "gpu_hits_bit_identical_on_sample": same}

    if rank == 0:
        peak, peak_src = measured_peaks()
        fp = fetch_peaks(ctx)
        achieved = headline["algorithmic_gbs"]
        line = {
            "metric": SWEEP_METRIC, "value": headline["mrays_per_s"], "unit": "Mrays/s", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": headline["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "sweep: 16 Mi rays vs the david / sycee QBVH (BASELINE configs[4]); headline = david, uniform set, "
                                   "near-first order; t_min 0, t_max inf as the reference's benches (qbvh.rs:999)",
                       "n_rays": n, "seed_uniform": "0x5EED0001", "seed_axis": "0x5EED0002",
                       "path_set": "the world rays the renderer traces for the mesh's preset at 1920x1080, wavefront order "
                                   "(yart_dump_path_rays), first 16 Mi",
                       "l2": "inputs larger than L2: 805 MB of rays + 671 MB of hits per step; the tree (5.9 MB) stays L2-resident",
                       "parallelism": "ray array sharded x%d, no collective" % N},
            "sweep": table,
            "f32_records": {"mrays_per_s": headline.get("f32_records_mrays_per_s"),
                            "what": "yart_closest_hit_f32 on the same rays rounded to f32: 24 B ray + 16 B hit records instead of "
                                    "48 + 40; the traversal arithmetic is the same f64"},
            "hit_rate": hit_rate,
            "e2e": {"value": n * K2 / ms2 / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": (hi - lo) * 48,
                    "d2h_bytes_per_step": (hi - lo) * 40, "steps": K2, "ms_per_step": ms2 / K2,
                    "note": "pinned host ray / hit arrays through yart_closest_hit, which pipelines upload / kernels / download in "
                            "512 Ki-ray chunks: bound by the 805 MB upload over PCIe",
                    "f32_records": {"value": n * K2 / ms3 / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": (hi - lo) * 24,
                                    "d2h_bytes_per_step": (hi - lo) * 16, "ms_per_step": ms3 / K2,
                                    "what": "the same rays and call shape through yart_closest_hit_f32"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_traverse<NEAR> (one launch per step) + k_export", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "bytes_per_ray": headline["bytes_per_ray"], "nodes_per_ray": headline["nodes_per_ray"],
                         "tris_per_ray": headline["tris_per_ray"],
                         "fetch_peaks": dict(fp, frac_of_l2_resident_fetch_peak=achieved / fp["scene_sized_l2_resident_gbs"],
                                             frac_of_l1_resident_fetch_peak=achieved / fp["l1_resident_gbs"]),
                         "note": "algorithmic bytes = 128 B x nodes + 48 B x triangles visited (counted, equal to the oracle's) + 88 B "
                                 "ray/hit stream, over the library's own CUDA-event time of the query; fetches are L1/L2 hits"},
            "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line), flush=True)
    rig.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="render", choices=["render", "sweep"])
    ap.add_argument("--total-spp", type=int, default=0,
                    help="render: make the step the FIXED job of this many spp split over the GPUs (strong scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-time-to-image", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = (3 if args.total_spp else TOTAL_SPP // SPP_PER_STEP) if args.workload == "render" else 5
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("--dump-outputs: the reference arm sizes its steps from a timing probe, so its outputs differ "
                         "from run to run")
    if args.impl == "reference":
        return run_reference(args)
    return run_sweep(args) if args.workload == "sweep" else run_render(args)


def _keep_stdout_for_the_json_line():
    """Libraries write to file descriptor 1 behind Python's back (NCCL prints its version banner there at the first
    communicator).  The contract is ONE JSON line on stdout: send everything else that lands on fd 1 to stderr and keep
    the real stdout for Python's own prints, which in this script are the JSON lines only."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    _keep_stdout_for_the_json_line()
    sys.exit(main())
