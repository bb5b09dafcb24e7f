#!/usr/bin/env python3
"""A small, fast exercise of every kernel and every scene feature (SURVEY.md section 4, item 6).

Run against the bounds-checked library (build.py --bounds-check) it plays the part of a memcheck run:
    YART_LIB_PATH=yet-another-raytracer_b200/libyart_b200_checked.so python tools/exercise_kernels.py
Any index outside its array traps and the next call raises.  tests/test_gpu_bounds.py runs exactly this.
"""
import importlib, sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import raysets
y = importlib.import_module("yet-another-raytracer_b200")
ctx = y.Context(0)
for scene, w, h, spp in (("david", 48, 32, 2), ("cornell-box-smoke", 32, 32, 2), ("next-week-final", 32, 24, 2), ("earth", 24, 16, 2)):
    p = y.ScenePreset(scene, seed=2)
    ctx.set_scene(p)
    cam = p.camera(w, h)
    film, st = ctx.render(cam, w, h, 0, spp, 50, 1)
    ctx.render(cam, w, h, 0, spp, 50, 1, flags=y.FLAG_NEXT_EVENT)
    rgba = ctx.film_finalize(film, spp)
    rays, _, _ = ctx.camera_rays(cam, w, h, 0, 1)
    for order in (0, 1):
        ctx.closest_hit(rays, y.TARGET_WORLD, 0.001, float("inf"), order, count_visits=True)
    ctx.occluded(rays, y.TARGET_WORLD, 0.001, float("inf"))  # k_occlude + k_analytic_occluded
    print(scene, st.rays, int(rgba.sum()))
p = y.ScenePreset("david"); ctx.set_scene(p)
o, d = raysets.uniform(20000, [-60, 0, -90], [70, 200, 60])
rays = y.make_rays(o, d)
weird = y.make_rays([(0, 0, 0), (0, 0, 5), (np.nan, 0, 0), (0, 0, 5)], [(0, 0, 0), (0, 0, -np.inf), (0, 0, 1), (0, 1e-320, -1)])
for r in (rays, weird, rays[:1], rays[:33]):
    for order in (0, 1):
        ctx.closest_hit(r, 0, 0.0, float("inf"), order)
    ctx.occluded(r, 0, 0.0, float("inf"))
# round-2 entry points: f32 records, sampling flags, path-ray dump, device films + a one-rank communicator
r32 = np.empty(len(rays), dtype=y.abi.RAY_F32_DTYPE)
r32["origin"], r32["direction"] = rays["origin"], rays["direction"]
for order in (0, 1):
    ctx.closest_hit_f32(r32, 0, 0.0, float("inf"), order)
    ctx.closest_hit_f32(r32[:33], y.TARGET_WORLD, 0.001, float("inf"), order)
ctx.occluded_f32(r32, 0, 0.0, float("inf"))
cam = p.camera(48, 32)
flags = y.FLAG_UNBIASED_LIGHT_PICK | y.FLAG_RUSSIAN_ROULETTE | y.FLAG_DEPTH_ZERO_BLACK
ctx.render(cam, 48, 32, 0, 3, 50, 1, flags=flags)
ctx.render(cam, 48, 32, 0, 3, 50, 1, flags=flags | y.FLAG_NEXT_EVENT)  # k_shade<true>, shadow passes, k_nee_resolve
ctx.render(cam, 48, 32, 0, 3, 5, 1, batch_spp=2)
dumped, n = ctx.dump_path_rays(cam, 48, 32, 0, 2, 1 << 16)
assert n == len(dumped) > 48 * 32 * 2
film = ctx.film_create(48, 32)
ctx.render_device(cam, 48, 32, 0, 2, film, 50, 1)
comm = y.Comm.from_id(ctx, y.comm_unique_id(), 0, 1)
comm.film_reduce(film, 48, 32, 0)
comm.close()
assert ctx.film_read(film, 48, 32).sum() > 0
ctx.film_destroy(film)
# random scene descriptions and triangle soups (tests/scene_fuzz.py): wrappers, groups, media, degenerate triangles
from scene_fuzz import FuzzScene, fuzz_soup, fuzz_mesh_rays
import ctypes as C


def soup_scene(pos, nrm, uv):
    abi = y.abi
    tm, keep = y.trimesh_from_arrays(pos, nrm, uv)
    tex, mat, obj, sd = abi.Texture(), abi.Material(), abi.Object(), abi.SceneDesc()
    tex.kind, mat.kind = abi.TEX_SOLID, abi.MAT_LAMBERTIAN
    obj.kind, obj.cos_theta = abi.OBJ_MESH, 1.0
    sd.objects, sd.n_objects = C.pointer(obj), 1
    sd.meshes, sd.n_meshes = C.pointer(tm), 1
    sd.materials, sd.n_materials = C.pointer(mat), 1
    sd.textures, sd.n_textures = C.pointer(tex), 1
    return C.pointer(sd), (tm, keep, tex, mat, obj, sd)


for seed in range(6):
    sc = FuzzScene(y, 4000 + seed)
    ctx.set_scene(sc.desc)
    o, d = sc.rays(20000)
    for order in (0, 1):
        ctx.closest_hit(y.make_rays(o, d), y.TARGET_WORLD, 0.001, float("inf"), order, count_visits=bool(order))
    ctx.render(sc.camera(32, 24), 32, 24, 0, 3, 12, 1, flags=flags if seed % 2 else 0)
    ctx.render(sc.camera(32, 24), 32, 24, 0, 3, 12, 1, flags=y.FLAG_NEXT_EVENT)
for seed, n_tris in ((1, 6), (2, 33), (3, 1000)):
    pos, nrm, uv = fuzz_soup(seed, n_tris)
    desc, keep = soup_scene(pos, nrm, uv)
    ctx.set_scene(desc)
    o, d = fuzz_mesh_rays(seed, pos, 20000)
    for order in (0, 1):
        ctx.closest_hit(y.make_rays(o, d), 0, 0.0, float("inf"), order)
print("exercise done")
