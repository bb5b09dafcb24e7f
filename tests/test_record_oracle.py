"""CPU side of the hit records: the reference of tests/record_ref.cpp -- the whole HitRecord the CPU oracle's world.hit
builds, for rays with their own time -- must carry exactly orc_closest_hit's t, ids and front_face, and its other fields
must be what an independent restatement gives: p = ray.at(t), the mesh's interpolated normal and uvs, a group member's
material, a moving sphere's normal about center(time).  The GPU tests compare yart_closest_hit_records against it."""
import os

import numpy as np
import pytest

import raysets
import record_ref
from record_sets import SmallWorld, leaf_kinds, ray_at
from scene_fuzz import FuzzScene

INF = float("inf")
NT = os.cpu_count()
PRESETS = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
           "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]


def assert_ids_match(yart, rec, hits, what):
    for f in ("t", "obj_id", "prim_id", "front_face"):
        a, b = rec[f], hits[f]
        bad = np.flatnonzero(~((a == b) | ((a != a) & (b != b))))
        assert bad.size == 0, "%s: %s differs on %d of %d rays, first %d: record %r hit %r" % (
            what, f, bad.size, len(rec), bad[0], rec[bad[0]], hits[bad[0]])
    miss = hits["obj_id"] == yart.MISS
    assert (rec["material"][miss] == yart.MISS).all() and (rec["normal"][miss] == 0).all()


def preset_rays(yart, orc, preset, n_uniform=3000):
    cam = preset.camera(48, 32)
    rays, _, _ = orc.camera_rays(cam, 48, 32, 0, 1, seed=5)
    c = np.asarray(preset.info.lookat)
    r = np.linalg.norm(np.asarray(preset.info.lookfrom) - c)
    o, d = raysets.uniform(n_uniform, c - 0.6 * r, c + 0.6 * r, 78)
    return np.concatenate([rays, yart.make_rays(o, d)])


@pytest.mark.parametrize("scene", PRESETS)
def test_presets_ids_equal_the_closest_hit(yart, orc, scene):
    preset = yart.ScenePreset(scene, seed=3)
    s, ref = orc.Scene(preset), record_ref.Scene(preset)
    rays = preset_rays(yart, orc, preset)
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        hits, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order, n_threads=NT)
        rec = ref.records(rays, None, yart.TARGET_WORLD, 0.001, INF, order, n_threads=NT)
        assert_ids_match(yart, rec, hits, "%s order %d" % (scene, order))
        assert (rec["obj_id"] != yart.MISS).any()


@pytest.mark.parametrize("seed", range(40))
def test_random_worlds_ids_equal_the_closest_hit(yart, orc, seed):
    """Random worlds (tests/scene_fuzz.py): instances, spheres, rects, boxes, loose triangles, media, groups, wrappers."""
    sc = FuzzScene(yart, 1000 + seed)
    s, ref = orc.Scene(sc), record_ref.Scene(sc)
    rays = yart.make_rays(*sc.rays(6000))
    n_plain = 0
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        for t_min, t_max in ((0.001, INF), (0.0, 3.5)):
            hits, _ = s.closest_hit(rays, yart.TARGET_WORLD, t_min, t_max, order, n_threads=NT)
            rec = ref.records(rays, None, yart.TARGET_WORLD, t_min, t_max, order, n_threads=NT)
            assert_ids_match(yart, rec, hits, "seed %d order %d" % (seed, order))
            # p = ray.at(t) exactly wherever no RotateY / Translate moved it (a medium's p is on the world ray)
            kind, medium, wrap = leaf_kinds(yart.abi, sc.desc, rec, yart.TARGET_WORLD)
            plain = (kind >= 0) & (medium | ((wrap & (yart.abi.WRAP_ROTATE_Y | yart.abi.WRAP_TRANSLATE)) == 0))
            n_plain += plain.sum()
            assert np.array_equal(rec["p"][plain], ray_at(rays[plain], rec["t"][plain]))
    assert n_plain > 0


@pytest.mark.parametrize("name", ["cube", "sycee", "david"])
def test_mesh_records_equal_an_independent_interpolation(yart, orc, mesh_scene, name):
    """Mesh target: the normal and u, v follow from the trimesh (f64 normals, f32 uvs widened), the oracle's
    barycentrics and the face-orientation rule of qbvh.rs:452-489 (front face when d . n <= 0, normal flipped
    otherwise); p = ray.at(t); no material."""
    _, ms, s = mesh_scene(name)
    ref = record_ref.Scene(ms)
    info = s.qbvh_info(0)
    o1, d1 = raysets.uniform(20000, info.bbox_min, info.bbox_max, raysets.SEED_UNIFORM + 5)
    o2, d2 = raysets.axis(10000, info.bbox_min, info.bbox_max, raysets.SEED_AXIS + 5)
    rays = yart.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]))
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        hits, _ = s.closest_hit(rays, 0, 0.001, INF, order, n_threads=NT)
        rec = ref.records(rays, None, 0, 0.001, INF, order, n_threads=NT)
        assert_ids_match(yart, rec, hits, "%s order %d" % (name, order))
        hit = np.flatnonzero(hits["prim_id"] != yart.MISS)
        assert hit.size > 1000 and (rec["material"] == yart.MISS).all()
        tri = hits["prim_id"][hit]
        u, v = hits["u"][hit][:, None], hits["v"][hit][:, None]
        w = 1.0 - hits["u"][hit] - hits["v"][hit]
        w = w[:, None]
        n = ms.normals[tri]
        uv = ms.uvs[tri].astype(np.float64)
        outward = n[:, 0] * w + n[:, 1] * u + n[:, 2] * v
        d = rays["direction"][hit]
        ff = (d[:, 0] * outward[:, 0] + d[:, 1] * outward[:, 1] + d[:, 2] * outward[:, 2]) <= 0.0
        sign = np.where(ff, 1.0, -1.0)[:, None]
        assert np.array_equal(rec["front_face"][hit], ff.astype(np.uint32))
        assert np.array_equal(rec["normal"][hit], sign * outward)
        assert np.array_equal(rec["u"][hit], uv[:, 0, 0] * w[:, 0] + uv[:, 1, 0] * u[:, 0] + uv[:, 2, 0] * v[:, 0])
        assert np.array_equal(rec["v"][hit], uv[:, 0, 1] * w[:, 0] + uv[:, 1, 1] * u[:, 0] + uv[:, 2, 1] * v[:, 0])
        assert np.array_equal(rec["p"][hit], ray_at(rays[hit], rec["t"][hit]))


def test_group_hits_carry_the_members_material(yart, orc):
    world = SmallWorld(yart.abi)
    ref = record_ref.Scene(world)
    rays = world.group_rays()
    rec = ref.records(rays)
    on_group = rec["obj_id"] == 0
    assert on_group.sum() > 100 and len(set(rec["prim_id"][on_group])) == 3
    assert np.array_equal(rec["material"][on_group], rec["prim_id"][on_group])  # member i has material i; the group 3
    # each member's normal is (p - centre) / radius, radius 1
    centres = np.asarray(world.GROUP_CENTRES)[rec["prim_id"][on_group]]
    assert np.array_equal(rec["normal"][on_group], rec["p"][on_group] - centres)


def test_moving_sphere_normal_follows_the_centre_at_the_rays_time(yart, orc):
    world = SmallWorld(yart.abi)
    ref = record_ref.Scene(world)
    rays = world.moving_rays()
    (c0, c1, radius) = world.MOVING
    for time in (0.0, 0.5, 1.0):
        times = np.full(len(rays), time)
        rec = ref.records(rays, times)
        hit = rec["obj_id"] == 1
        centre = np.asarray(c0) + ((time - 0.0) / (1.0 - 0.0)) * (np.asarray(c1) - np.asarray(c0))  # sphere.rs:149-152
        assert np.array_equal(hit, np.abs(rays["origin"][:, 0] - centre[0]) < np.sqrt(radius ** 2 - 0.1 ** 2))
        outward = (rec["p"][hit] - centre) / radius
        assert np.array_equal(rec["normal"][hit], outward)  # rays enter from outside: front face, outward normal
        assert (rec["front_face"][hit] == 1).all() and (rec["material"][hit] == 4).all()
    # times NULL is time 0
    assert np.array_equal(ref.records(rays).view(np.uint8), ref.records(rays, np.zeros(len(rays))).view(np.uint8))
