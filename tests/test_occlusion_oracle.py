"""CPU side of the occlusion queries: the reference of tests/occlusion_ref.cpp -- an early-exit restatement (t_max fixed,
the first accepted triangle / the first object that hits ends the ray) -- must equal the hit flag of the CPU oracle's
orc_closest_hit in the reference's order.  That equality is the contract of yart_occluded, and the GPU tests compare
against this reference."""
import os

import numpy as np
import pytest

import occlusion_ref
import raysets
from scene_fuzz import FuzzScene

INF = float("inf")
NT = os.cpu_count()


def closest_flag(yart, s, rays, target, t_min, t_max):
    hits, _ = s.closest_hit(rays, target, t_min, t_max, yart.ORDER_REFERENCE, n_threads=NT)
    return hits["prim_id"] != yart.MISS


def assert_same(got, want, what):
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, "%s: %d of %d rays differ, first %d (occluded %s, closest-hit flag %s)" % (
        what, bad.size, len(want), bad[0], got[bad[0]], want[bad[0]])


@pytest.mark.parametrize("name", ["cube", "sycee", "david"])
def test_mesh_occlusion_equals_the_closest_hit_flag(yart, orc, mesh_scene, name):
    _, ms, s = mesh_scene(name)
    ref = occlusion_ref.Scene(ms)
    info = s.qbvh_info(0)
    o1, d1 = raysets.uniform(20000, info.bbox_min, info.bbox_max, raysets.SEED_UNIFORM + 21)
    o2, d2 = raysets.axis(10000, info.bbox_min, info.bbox_max, raysets.SEED_AXIS + 21)
    rays = yart.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]))
    diag = float(np.linalg.norm(np.asarray(info.bbox_max) - np.asarray(info.bbox_min)))
    for t_min in (0.0, 0.001):
        for t_max in (INF, 0.3 * diag):
            want = closest_flag(yart, s, rays, 0, t_min, t_max)
            assert_same(ref.occluded(rays, 0, t_min, t_max, n_threads=NT), want, "%s t in (%g, %g)" % (name, t_min, t_max))
            assert want.any()


def test_grid_ties_at_the_t_max_boundary(yart, orc):
    """Integer height field: rays whose closest hit is an exact t = 8 tie.  The reference's `t_max > t` is strict, so a
    t_max of exactly 8 must leave them unoccluded and one ulp more must occlude them."""
    pos, nrm, uv, h = raysets.grid_mesh()
    ms = orc.MeshScene(pos, nrm, uv)
    s, ref = orc.Scene(ms), occlusion_ref.Scene(ms)
    rays = yart.make_rays(*raysets.grid_tie_rays(h, 20000))
    full, _ = s.closest_hit(rays, 0, 0.001, INF, yart.ORDER_REFERENCE)
    at8 = full["t"] == 8.0
    assert at8.sum() > 5000
    for t_max in (8.0, np.nextafter(8.0, INF)):
        got = ref.occluded(rays, 0, 0.001, t_max)
        assert_same(got, closest_flag(yart, s, rays, 0, 0.001, t_max), "grid t_max %r" % t_max)
        assert got[at8].all() if t_max > 8.0 else not got[at8].any()


def test_nan_slab_and_degenerate_rays(yart, orc, mesh_scene):
    _, ms, s = mesh_scene("sycee")
    ref = occlusion_ref.Scene(ms)
    ray = yart.make_rays([(0, 3, 0), (1, 5, -8)], [(0, -1, 0), (-1, -4.5, 8)])
    assert list(ref.occluded(ray, 0, 0.001, INF)) == [False, True]  # the reference's NaN-slab miss; a hit at t = 0.947
    assert list(ref.occluded(ray, 0, 0.001, 0.9)) == [False, False]
    _, ms, s = mesh_scene("cube")
    ref = occlusion_ref.Scene(ms)
    weird = yart.make_rays([(0, 0, 0), (0, 0, 5), (np.nan, 0, 0), (0, 0, 5), (0, 0, 5), (0, 0, np.inf)],
                           [(0, 0, 0), (0, 0, -np.inf), (0, 0, 1), (0, np.nan, -1), (0, 0, -1e-300), (0, 0, -1)])
    for t_min, t_max in ((0.001, INF), (0.0, 4.5)):
        assert_same(ref.occluded(weird, 0, t_min, t_max), closest_flag(yart, s, weird, 0, t_min, t_max), "weird rays")


@pytest.mark.parametrize("seed", range(24))
def test_random_worlds(yart, orc, seed):
    """Random worlds (tests/scene_fuzz.py): instances, spheres, rects, boxes, loose triangles, media, groups."""
    sc = FuzzScene(yart, 6000 + seed)
    s, ref = orc.Scene(sc), occlusion_ref.Scene(sc)
    rays = yart.make_rays(*sc.rays(8000))
    for t_min, t_max in ((0.001, INF), (0.0, 3.5)):
        want = closest_flag(yart, s, rays, yart.TARGET_WORLD, t_min, t_max)
        assert_same(ref.occluded(rays, yart.TARGET_WORLD, t_min, t_max, n_threads=NT), want, "seed %d" % seed)


@pytest.mark.parametrize("scene", ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light",
                                   "cornell-box", "cornell-box-smoke", "next-week-final", "teapot", "bunny",
                                   "three-spheres", "sycee", "david"])
def test_presets_world(yart, orc, scene):
    preset = yart.ScenePreset(scene, seed=3)
    s, ref = orc.Scene(preset), occlusion_ref.Scene(preset)
    cam = preset.camera(48, 32)
    rays, _, _ = orc.camera_rays(cam, 48, 32, 0, 1, seed=5)
    c = np.asarray(preset.info.lookat)
    r = np.linalg.norm(np.asarray(preset.info.lookfrom) - c)
    o, d = raysets.uniform(3000, c - 0.6 * r, c + 0.6 * r, 78)
    rays = np.concatenate([rays, yart.make_rays(o, d)])
    want = closest_flag(yart, s, rays, yart.TARGET_WORLD, 0.001, INF)
    assert_same(ref.occluded(rays, yart.TARGET_WORLD, 0.001, INF, n_threads=NT), want, scene)
