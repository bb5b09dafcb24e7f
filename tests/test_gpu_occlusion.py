"""GPU occlusion queries: yart_occluded / yart_occluded_f32 against the CPU reference of tests/occlusion_ref.cpp and
against the GPU's own yart_closest_hit(..., ORDER_REFERENCE) hit flag -- bit for bit, on every ray."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import occlusion_ref
import raysets
from occlusion_sets import shadow_rays
from scene_fuzz import FuzzScene

pytestmark = pytest.mark.gpu
INF = float("inf")
NT = os.cpu_count()
ROOT = Path(__file__).resolve().parent.parent


def to_f32(yart, rays):
    r32 = np.empty(len(rays), dtype=yart.abi.RAY_F32_DTYPE)
    r32["origin"], r32["direction"] = rays["origin"], rays["direction"]
    return r32


def widen(yart, r32):
    return yart.make_rays(r32["origin"].astype(np.float64), r32["direction"].astype(np.float64))


def assert_same(got, want, what):
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, "%s: %d of %d rays differ, first %d (gpu %s, expected %s)" % (
        what, bad.size, len(want), bad[0], got[bad[0]], want[bad[0]])


def check(yart, ctx, ref, rays, target, t_min, t_max, what, device=True):
    """yart_occluded on host and device arrays == the CPU reference (an occlusion_ref.Scene) == the GPU's closest-hit
    flag (reference order); the same for the f32 records.  Returns the flags."""
    import torch
    want = ref.occluded(rays, target, t_min, t_max, n_threads=NT)
    hits, _ = ctx.closest_hit(rays, target, t_min, t_max, yart.ORDER_REFERENCE)
    assert_same(hits["prim_id"] != yart.MISS, want, what + " (the reference vs the closest-hit flag)")
    got, st = ctx.occluded(rays, target, t_min, t_max)
    assert_same(got, want, what + " host f64")
    assert st.rays == len(rays) and st.node_visits == 0 and st.kernel_launches == st.trace_launches >= 1
    r32 = to_f32(yart, rays)
    w32 = widen(yart, r32)
    t_min32, t_max32 = float(np.float32(t_min)), float(np.float32(t_max))  # (what the f32 entry points receive)
    want32 = ref.occluded(w32, target, t_min32, t_max32, n_threads=NT)
    h32, _ = ctx.closest_hit_f32(r32, target, t_min, t_max, yart.ORDER_REFERENCE)
    assert_same(h32["prim_id"] != yart.MISS, want32, what + " (f32: the reference vs the closest-hit flag)")
    got32, _ = ctx.occluded_f32(r32, target, t_min, t_max)
    assert_same(got32, want32, what + " host f32")
    if device:
        dev = torch.device("cuda", 0)
        rd = torch.from_numpy(rays.view(np.uint8)).to(dev)
        r32d = torch.from_numpy(r32.view(np.uint8)).to(dev)
        out = torch.full((len(rays),), 7, dtype=torch.uint8, device=dev)
        ctx.occluded_device(rd.data_ptr(), len(rays), out.data_ptr(), target, t_min, t_max)
        assert_same(out.cpu().numpy().view(np.bool_), want, what + " device f64")
        out.fill_(7)
        ctx.occluded_f32_device(r32d.data_ptr(), len(rays), out.data_ptr(), target, t_min, t_max)
        assert_same(out.cpu().numpy().view(np.bool_), want32, what + " device f32")
    return got


def mesh_rays(yart, info, n, shift=0):
    o1, d1 = raysets.uniform(n, info.bbox_min, info.bbox_max, raysets.SEED_UNIFORM + shift)
    o2, d2 = raysets.axis(n // 2, info.bbox_min, info.bbox_max, raysets.SEED_AXIS + shift)
    return yart.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]))


@pytest.mark.parametrize("name", ["cube", "sycee", "david"])
def test_mesh_occlusion(yart, orc, ctx, mesh_scene, name):
    _, ms, s = mesh_scene(name)
    ref = occlusion_ref.Scene(ms)
    ctx.set_scene(ms.desc)
    info = s.qbvh_info(0)
    rays = mesh_rays(yart, info, 200000, 31)
    diag = float(np.linalg.norm(np.asarray(info.bbox_max) - np.asarray(info.bbox_min)))
    for t_min in (0.0, 0.001):
        for t_max in (INF, 0.3 * diag):
            got = check(yart, ctx, ref, rays, 0, t_min, t_max, "%s t in (%g, %g)" % (name, t_min, t_max))
            assert got.any()


def test_grid_ties_and_boundaries(yart, orc, ctx):
    pos, nrm, uv, h = raysets.grid_mesh()
    ms = orc.MeshScene(pos, nrm, uv)
    ref = occlusion_ref.Scene(ms)
    ctx.set_scene(ms.desc)
    rays = yart.make_rays(*raysets.grid_tie_rays(h, 20000))
    full, _ = ctx.closest_hit(rays, 0, 0.001, INF, yart.ORDER_REFERENCE)
    at8 = full["t"] == 8.0
    assert at8.sum() > 5000
    for t_max in (8.0, np.nextafter(8.0, INF), INF):
        got = check(yart, ctx, ref, rays, 0, 0.001, t_max, "grid t_max %r" % t_max)
        assert got[at8].all() if t_max > 8.0 else not got[at8].any()


def test_nan_slab_and_degenerate_rays(yart, orc, ctx, mesh_scene):
    _, ms, _ = mesh_scene("sycee")
    ctx.set_scene(ms.desc)
    ray = yart.make_rays([(0, 3, 0), (1, 5, -8)], [(0, -1, 0), (-1, -4.5, 8)])
    got, _ = ctx.occluded(ray, 0, 0.001, INF)
    assert list(got) == [False, True]
    got, _ = ctx.occluded(ray, 0, 0.001, 0.9)
    assert list(got) == [False, False]
    _, ms, _ = mesh_scene("cube")
    ref = occlusion_ref.Scene(ms)
    ctx.set_scene(ms.desc)
    weird = yart.make_rays([(0, 0, 0), (0, 0, 5), (np.nan, 0, 0), (0, 0, 5), (0, 0, 5), (0, 0, np.inf)],
                           [(0, 0, 0), (0, 0, -np.inf), (0, 0, 1), (0, np.nan, -1), (0, 0, -1e-300), (0, 0, -1)])
    for t_min, t_max in ((0.001, INF), (0.0, 4.5)):
        check(yart, ctx, ref, weird, 0, t_min, t_max, "weird rays")


@pytest.mark.parametrize("scene", ["david", "cornell-box", "cornell-box-smoke", "sycee", "three-spheres",
                                   "next-week-final", "random-scene"])
def test_world_presets(yart, orc, ctx, scene):
    preset = yart.ScenePreset(scene, seed=3)
    ref = occlusion_ref.Scene(preset)
    ctx.set_scene(preset)
    cam = preset.camera(96, 64)
    rays, _, _ = orc.camera_rays(cam, 96, 64, 0, 2, seed=5)
    c = np.asarray(preset.info.lookat)
    r = np.linalg.norm(np.asarray(preset.info.lookfrom) - c)
    o, d = raysets.uniform(6000, c - 0.6 * r, c + 0.6 * r, 77)
    rays = np.concatenate([rays, yart.make_rays(o, d)])
    got = check(yart, ctx, ref, rays, yart.TARGET_WORLD, 0.001, INF, scene)
    assert got.mean() > 0.3


@pytest.mark.parametrize("seed", range(40))
def test_random_worlds(yart, orc, ctx, seed):
    sc = FuzzScene(yart, 6100 + seed)
    ref = occlusion_ref.Scene(sc)
    ctx.set_scene(sc.desc)
    rays = yart.make_rays(*sc.rays(30000))
    for t_min, t_max in ((0.001, INF), (0.0, 3.5)):
        check(yart, ctx, ref, rays, yart.TARGET_WORLD, t_min, t_max, "seed %d t in (%g, %g)" % (seed, t_min, t_max),
              device=seed % 4 == 0)


def test_ragged_sizes_and_empty_world(yart, orc, ctx, mesh_scene):
    _, ms, s = mesh_scene("cube")
    ref = occlusion_ref.Scene(ms)
    ctx.set_scene(ms.desc)
    info = s.qbvh_info(0)
    got, st = ctx.occluded(np.empty(0, dtype=yart.RAY_DTYPE), 0)
    assert len(got) == 0 and st.rays == 0 and st.kernel_launches == 0 and st.gpu_ms == 0.0
    for n in (1, 31, 32, 33, 4097):
        o, d = raysets.uniform(n, info.bbox_min, info.bbox_max, 199 + n)
        d[::3] *= -40.0  # some rays leave the cube before they reach it (t_max below)
        check(yart, ctx, ref, yart.make_rays(o, d), 0, 0.001, 0.5, "n=%d" % n)
    # a world with no objects: everything stays 0
    abi = yart.abi
    tex, mat, sd = abi.Texture(), abi.Material(), abi.SceneDesc()
    tex.kind, mat.kind = abi.TEX_SOLID, abi.MAT_LAMBERTIAN
    sd.materials, sd.n_materials = C.pointer(mat), 1
    sd.textures, sd.n_textures = C.pointer(tex), 1
    ctx.set_scene(C.pointer(sd))
    rays = yart.make_rays(*raysets.uniform(1000, [-1, -1, -1], [1, 1, 1], 5))
    got, st = ctx.occluded(rays, yart.TARGET_WORLD)
    assert not got.any() and st.kernel_launches == 0


def test_chunked_host_calls_equal_unchunked(yart, orc, ctx, mesh_scene, monkeypatch):
    _, ms, s = mesh_scene("david")
    ctx.set_scene(ms.desc)
    rays = mesh_rays(yart, s.qbvh_info(0), 300000, 41)
    whole, st1 = ctx.occluded(rays, 0, 0.0, INF)
    whole32, _ = ctx.occluded_f32(to_f32(yart, rays), 0, 0.0, INF)
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", "65536")
    parts, st2 = ctx.occluded(rays, 0, 0.0, INF)
    parts32, _ = ctx.occluded_f32(to_f32(yart, rays), 0, 0.0, INF)
    assert_same(parts, whole, "chunked f64")
    assert_same(parts32, whole32, "chunked f32")
    assert st1.kernel_launches == 1 and st2.kernel_launches == (len(rays) + 65535) // 65536 and st2.gpu_ms > 0.0
    # a pinned caller-owned output array
    out = np.zeros(len(rays), dtype=np.uint8)
    ctx.host_register(out)
    try:
        ctx.occluded(rays, 0, 0.0, INF, out=out)
    finally:
        ctx.host_unregister(out)
    assert_same(out.view(np.bool_), whole, "pinned output")


def test_full_size_david_sweep(yart, orc, ctx, mesh_scene):
    """16 Mi uniform rays against david: the occlusion flag is the closest-hit flag, a rerun is identical, and a
    64 Ki subset equals the oracle."""
    import torch
    _, ms, s = mesh_scene("david")
    ctx.set_scene(ms.desc)
    ref = occlusion_ref.Scene(ms)
    info = s.qbvh_info(0)
    n = 1 << 24
    rays = yart.make_rays(*raysets.uniform(n, info.bbox_min, info.bbox_max))
    hits, _ = ctx.closest_hit(rays, 0, 0.0, INF, yart.ORDER_REFERENCE)
    a, _ = ctx.occluded(rays, 0, 0.0, INF)
    assert_same(a, hits["prim_id"] != yart.MISS, "sweep vs closest-hit flag")
    dev = torch.device("cuda", 0)
    rd = torch.from_numpy(rays.view(np.uint8)).to(dev)
    out = torch.zeros(n, dtype=torch.uint8, device=dev)
    st = ctx.occluded_device(rd.data_ptr(), n, out.data_ptr(), 0, 0.0, INF)
    assert_same(out.cpu().numpy().view(np.bool_), a, "rerun on device arrays")
    assert st.gpu_ms > 0.0 and 0.2 < a.mean() < 0.95
    idx = np.random.Generator(np.random.Philox(4)).choice(n, 1 << 16, replace=False)
    assert_same(a[idx], ref.occluded(rays[idx], 0, 0.0, INF, n_threads=NT), "subset vs the reference")


def test_shadow_rays_on_the_david_preset(yart, orc, ctx):
    preset = yart.ScenePreset("david", seed=3)
    ref = occlusion_ref.Scene(preset)
    ctx.set_scene(preset)
    rays, t_max = shadow_rays(yart, ctx, preset, 96, 96)
    got = check(yart, ctx, ref, rays, yart.TARGET_WORLD, 0.001, t_max, "david shadow rays")
    assert 0.02 < got.mean() < 0.98


def test_argument_errors(yart, ctx, mesh_scene):
    lib = yart.load_library()
    rays = np.zeros(4, dtype=yart.RAY_DTYPE)
    out = np.zeros(4, dtype=np.uint8)
    fresh = yart.Context(0)
    try:  # no scene
        assert lib.yart_occluded(fresh._h, 0, rays.ctypes.data, 4, 0.0, INF, 0, out.ctypes.data, None) == -1
        assert b"no scene" in lib.yart_last_error(fresh._h)
    finally:
        fresh.close()
    _, ms, _ = mesh_scene("cube")
    ctx.set_scene(ms.desc)

    def call(target=0, r=rays.ctypes.data, n=4, flags=0, o=out.ctypes.data, fn=lib.yart_occluded):
        return fn(ctx._h, target, r, n, 0.0, INF, flags, o, None)

    assert call(r=None) == -1 and call(o=None) == -1
    assert call(n=0xFFFFFFF1) == -1
    assert call(target=7) == -1 and b"target" in lib.yart_last_error(ctx._h)
    assert call(flags=yart.FLAG_COUNT_VISITS) == -1 and call(flags=64) == -1
    assert b"YART_FLAG_DEVICE_PTRS" in lib.yart_last_error(ctx._h)
    assert call(flags=yart.FLAG_DEVICE_PTRS, r=(1 << 40) + 8) == -1 and b"aligned" in lib.yart_last_error(ctx._h)
    assert call(flags=yart.FLAG_DEVICE_PTRS, r=(1 << 40) + 4, fn=lib.yart_occluded_f32) == -1
    st = yart.abi.Stats()
    st.rays = 99
    assert lib.yart_occluded(ctx._h, 0, None, 0, 0.0, INF, 0, None, C.byref(st)) == 0 and st.rays == 0
    assert call() == 0


def test_the_occlusion_kernels_under_bounds_checks(yart, ctx):
    """k_occlude and k_analytic_occluded through the bounds-checked library (the checked build's traps stand in for
    a memory checker), in a fresh process as tests/test_gpu_bounds.py runs the other kernels."""
    checked = ROOT / "yet-another-raytracer_b200" / "libyart_b200_checked.so"
    assert checked.exists(), "run __graft_entry__.build() first"
    code = (
        "import importlib, sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import raysets\n"
        "from scene_fuzz import FuzzScene\n"
        "y = importlib.import_module('yet-another-raytracer_b200')\n"
        "ctx = y.Context(0)\n"
        "for name in ('david', 'cornell-box-smoke', 'next-week-final'):\n"
        "    p = y.ScenePreset(name, seed=2); ctx.set_scene(p)\n"
        "    rays, _, _ = ctx.camera_rays(p.camera(48, 32), 48, 32, 0, 1)\n"
        "    a, _ = ctx.occluded(rays, y.TARGET_WORLD, 0.001, float('inf'))\n"
        "    h, _ = ctx.closest_hit(rays, y.TARGET_WORLD, 0.001, float('inf'), 0)\n"
        "    assert (a == (h['prim_id'] != y.MISS)).all(), name\n"
        "    if name == 'david': ctx.occluded(rays, 0, 0.0, float('inf'))\n"
        "sc = FuzzScene(y, 4100); ctx.set_scene(sc.desc)\n"
        "ctx.occluded(y.make_rays(*sc.rays(20000)), y.TARGET_WORLD, 0.0, 3.5)\n"
        "print('occlusion exercise done')\n"
    ) % (str(ROOT), str(ROOT / "tests"))
    env = dict(os.environ, YART_LIB_PATH=str(checked))
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    out = res.stdout + res.stderr
    assert "YART_CHECK failed" not in out, out[-2000:]
    assert res.returncode == 0 and "occlusion exercise done" in out, out[-2000:]
