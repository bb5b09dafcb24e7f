"""Fuzz parity: random scene descriptions (tests/scene_fuzz.py) through the CUDA path and the oracle.
Closest hits must agree bit for bit; small renders must agree like the preset renders do."""
import ctypes as C
import os

import numpy as np
import pytest

from scene_fuzz import FuzzScene
from test_gpu_render import compare_films

pytestmark = pytest.mark.gpu
INF = float("inf")
HIT_FIELDS = ("t", "u", "v", "prim_id", "obj_id", "front_face")


@pytest.mark.parametrize("seed", range(40))
def test_random_scene_world_closest_hit_is_bit_exact(yart, orc, ctx, seed):
    sc = FuzzScene(yart, 1000 + seed)
    s = orc.Scene(sc)
    ctx.set_scene(sc.desc)
    o, d = sc.rays(60000)
    rays = yart.make_rays(o, d)
    for t_min, t_max in ((0.001, INF), (0.0, 3.5)):
        want, _ = s.closest_hit(rays, yart.TARGET_WORLD, t_min, t_max, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
        for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
            got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, t_min, t_max, order)
            # a hit inside a ConstantMedium is t1 + (-1/density) * ln(xi) / |d| (hittable.rs:293-300): CUDA's log and glibc's
            # differ in the last bit now and then, so those t's are compared to 1e-12 (as in test_world_closest_hit_*)
            medium = np.array([bool(sc.sd.objects[i].wrap & yart.abi.WRAP_MEDIUM) for i in range(sc.n_objects)] + [False])
            in_medium = medium[np.minimum(want["obj_id"], sc.n_objects)] & (want["prim_id"] != yart.MISS)
            for f in HIT_FIELDS:
                same = (got[f] == want[f]) | ((got[f] != got[f]) & (want[f] != want[f]))
                if f == "t":
                    with np.errstate(invalid="ignore"):  # (inf - inf on the misses)
                        same |= in_medium & (np.abs(got[f] - want[f]) <= 1e-12 * np.abs(want[f]))
                bad = np.flatnonzero(~same)
                assert bad.size == 0, "seed %d order %d field %s: %d of %d rays differ, first %d: gpu %r oracle %r (object kind %s)" % (
                    seed, order, f, bad.size, len(rays), bad[0], got[bad[0]], want[bad[0]],
                    sc.sd.objects[int(want["obj_id"][bad[0]]) % max(sc.n_objects, 1)].kind)


@pytest.mark.parametrize("seed", range(20))
def test_random_scene_render_matches_the_oracle(yart, orc, ctx, seed):
    sc = FuzzScene(yart, 2000 + seed)
    s = orc.Scene(sc)
    ctx.set_scene(sc.desc)
    w, h, spp, depth = 48, 32, 6, 12
    cam = sc.camera(w, h)
    want, st_w = s.render(cam, w, h, 0, spp, max_depth=depth, seed=5, n_threads=os.cpu_count())
    for order in (yart.ORDER_NEAR, yart.ORDER_REFERENCE):
        got, st = ctx.render(cam, w, h, 0, spp, max_depth=depth, seed=5, order=order)
        compare_films(got, want, "fuzz scene %d order %d" % (seed, order), 0.99)
        assert abs(int(st.rays) - int(st_w.rays)) <= max(8, st_w.rays // 200)


def test_coincident_meshes_first_in_list_order_wins(yart, orc, ctx):
    """Exact ties between objects (three copies of one cube): the first in list order keeps the hit in both traversal
    orders and in every kernel variant (lean near-first, classic reference-order, classic near-first when counting)."""
    import ctypes as C
    abi = yart.abi
    mesh = yart.TriangleMesh.from_obj(os.path.join(yart.assets_dir(), "cube.obj"))
    tex, mat = abi.Texture(), abi.Material()
    tex.kind, mat.kind = abi.TEX_SOLID, abi.MAT_LAMBERTIAN
    objs = (abi.Object * 3)()
    for o in objs:
        o.kind, o.cos_theta = abi.OBJ_MESH, 1.0
    sd = abi.SceneDesc()
    sd.objects, sd.n_objects = C.cast(objs, C.POINTER(abi.Object)), 3
    sd.meshes, sd.n_meshes = C.pointer(mesh.trimesh), 1
    sd.materials, sd.n_materials = C.pointer(mat), 1
    sd.textures, sd.n_textures = C.pointer(tex), 1
    ctx.set_scene(C.pointer(sd))
    s = orc.Scene(C.pointer(sd))
    rng = np.random.default_rng(5)
    d = rng.normal(size=(50000, 3))
    o = -4.0 * d / np.linalg.norm(d, axis=1, keepdims=True) + rng.uniform(-0.3, 0.3, size=(50000, 3))
    rays = yart.make_rays(o, d)
    want, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
    hit = want["prim_id"] != yart.MISS
    assert hit.mean() > 0.5 and (want["obj_id"][hit] == 0).all()
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        for count in (False, True):
            got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order, count_visits=count)
            assert got.tobytes() == want.tobytes(), (order, count)


@pytest.mark.parametrize("seed", range(8))
def test_random_scene_sampling_flags_and_f32_records(yart, orc, ctx, seed):
    sc = FuzzScene(yart, 3000 + seed)
    s = orc.Scene(sc)
    ctx.set_scene(sc.desc)
    w, h, spp, depth = 40, 32, 6, 10
    cam = sc.camera(w, h)
    flags = yart.FLAG_UNBIASED_LIGHT_PICK | yart.FLAG_RUSSIAN_ROULETTE | yart.FLAG_DEPTH_ZERO_BLACK
    want, _ = s.render(cam, w, h, 0, spp, max_depth=depth, seed=9, n_threads=os.cpu_count(), flags=flags)
    got, _ = ctx.render(cam, w, h, 0, spp, max_depth=depth, seed=9, flags=flags)
    compare_films(got, want, "fuzz scene %d with all sampling flags" % seed, 0.99)
    # f32 records: the f64 query on the widened rays, rounded
    o, d = sc.rays(30000)
    r32 = np.empty(len(o), dtype=yart.abi.RAY_F32_DTYPE)
    r32["origin"], r32["direction"] = o.astype(np.float32), d.astype(np.float32)
    r64 = yart.make_rays(r32["origin"].astype(np.float64), r32["direction"].astype(np.float64))
    t_min = 2.0 ** -10  # (a float: the f32 entry point takes t_min as one, and a medium's entry clamp shows the difference)
    ref, _ = ctx.closest_hit(r64, yart.TARGET_WORLD, t_min, INF, yart.ORDER_NEAR)
    got32, _ = ctx.closest_hit_f32(r32, yart.TARGET_WORLD, t_min, INF, yart.ORDER_NEAR)
    assert np.array_equal(got32["prim_id"], ref["prim_id"])
    hit = ref["prim_id"] != yart.MISS
    for f in ("t", "u", "v"):
        assert np.array_equal(got32[f][hit], ref[f][hit].astype(np.float32)), f


@pytest.mark.parametrize("seed,n_tris", [(s, n) for s, n in enumerate([5, 6, 7, 8, 9, 12, 13, 16, 17, 31, 33, 64, 100, 257, 1000, 3001, 20000, 4, 11, 500])])
def test_random_soup_build_and_closest_hit(yart, orc, ctx, seed, n_tris):
    """Random triangle soups: device-built tree == host-built tree byte for byte, and L4QBVH::hit bit-exact against the
    oracle (both orders, with and without visit counting, two [t_min, t_max] windows)."""
    from scene_fuzz import fuzz_soup, fuzz_mesh_rays
    from test_gpu_build import assert_same_tree
    pos, nrm, uv = fuzz_soup(seed, n_tris)
    t, keep = yart.trimesh_from_arrays(pos, nrm, uv)
    if n_tris <= 4:  # L4QBVH::new yields no nodes (SURVEY A-17): refused by both builders
        with pytest.raises(yart.YartError):
            yart.L4QBVH(t, keepalive=keep, ctx=ctx)
        with pytest.raises(yart.YartError):
            yart.L4QBVH(t, keepalive=keep)
        return
    assert_same_tree(yart, ctx, t, keep)
    ms = orc.MeshScene(pos, nrm, uv)
    s = orc.Scene(ms)
    ctx.set_scene(ms.desc)
    o, d = fuzz_mesh_rays(seed, pos, 40000)
    rays = yart.make_rays(o, d)
    for t_min, t_max in ((0.001, INF), (0.0, 2.0)):
        wants = {}
        for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
            want, cnt = wants[order] = s.closest_hit(rays, 0, t_min, t_max, order, n_threads=os.cpu_count())
            for count in (False, True):
                got, st = ctx.closest_hit(rays, 0, t_min, t_max, order, count_visits=count)
                for f in ("t", "u", "v", "prim_id"):
                    same = (got[f] == want[f]) | ((got[f] != got[f]) & (want[f] != want[f]))
                    bad = np.flatnonzero(~same)
                    assert bad.size == 0, "soup %d (%d tris) order %d count %s window (%g, %g) field %s: %d rays differ, first %d: ray %r gpu %r oracle %r" % (
                        seed, n_tris, order, count, t_min, t_max, f, bad.size, bad[0], rays[bad[0]], got[bad[0]], want[bad[0]])
                if count:
                    assert (st.node_visits, st.tri_tests) == (cnt.node_visits, cnt.tri_tests), order
        # Near-first against the reference order (yart.h, YART_ORDER_NEAR): identical except where a ray passes within
        # rounding of a vertex / edge that lies ON a box face -- there each order culls the box the other one enters, and
        # the two answers are members of the same near-tie set.  These soups aim a third of their rays at such points.
        ref, near = wants[yart.ORDER_REFERENCE][0], wants[yart.ORDER_NEAR][0]
        diff = np.flatnonzero((ref["t"] != near["t"]) | (ref["prim_id"] != near["prim_id"]))
        assert diff.size <= 0.002 * len(rays)
        assert ((ref["prim_id"][diff] != yart.MISS) & (near["prim_id"][diff] != yart.MISS)).all()
        if t_min > 0.0:  # (with t_min = 0 the soups' degenerate triangles give spurious t = +-0 "hits" in the reference's
            #             Moller-Trumbore, and which order meets them first is arbitrary -- both sides still agree bit for bit above)
            assert (np.abs(ref["t"][diff] - near["t"][diff]) <= 1e-12 * np.abs(ref["t"][diff])).all()


@pytest.mark.parametrize("seed", range(6))
def test_film_finalize_on_random_films_with_special_values(yart, orc, ctx, seed):
    """yart_film_finalize (main.rs:710-718, color.rs:92-107) on films with NaN, +-inf, negatives, zeros, huge and tiny
    values, widths that are / are not multiples of 8, several spp."""
    g = np.random.default_rng(seed)
    h, w = int(g.integers(8, 50)), int(g.integers(8, 70))
    film = g.random((h, w, 3)) * float(g.choice([0.01, 1.0, 30.0, 1e6]))
    special = g.random((h, w, 3)) < 0.05
    film[special] = g.choice([np.nan, np.inf, -np.inf, -1.0, 0.0, -0.0, 1e300, 1e-300, 5e-324], size=int(special.sum()))
    spp = int(g.choice([1, 3, 64, 1024]))
    a = ctx.film_finalize(film, spp)
    b = orc.film_finalize(film, spp)
    # pow() may differ in the last bit; a u8 can flip only when 256 * c sits within 1e-13 of an integer
    assert (a != b).sum() <= 1, np.argwhere(a != b)[:5]


def test_bad_render_options_and_wild_cameras_fail_cleanly(yart, orc, ctx):
    """The reference panics on nonsense; behind a C ABI nonsense must come back as YART_ERR_INVALID (or as a finite
    film), and the context must stay usable."""
    sc = FuzzScene(yart, 4242)
    ctx.set_scene(sc.desc)
    cam = sc.camera(32, 24)
    good, _ = ctx.render(cam, 32, 24, 0, 2, max_depth=8, seed=1)
    bad = [dict(width=0), dict(width=1), dict(height=0), dict(height=1), dict(sample_begin=5, sample_end=2), dict(max_depth=0),
           dict(order=7), dict(width=70000, height=70000)]
    for kw in bad:
        a = dict(width=32, height=24, sample_begin=0, sample_end=2, max_depth=8, order=yart.ORDER_NEAR)
        a.update(kw)
        film = np.zeros((max(a["height"], 1) if a["height"] < 1000 else 1, max(a["width"], 1) if a["width"] < 1000 else 1, 3))
        st = yart.abi.Stats()
        o = ctx._opts(a["width"], a["height"], a["sample_begin"], a["sample_end"], a["max_depth"], 1, a["order"], 0, 0)
        rc = yart.load_library().yart_render(ctx._h, C.byref(cam), C.byref(o), film.ctypes.data, C.byref(st))
        assert rc == -1, kw
    # cameras with NaN / inf / zero-length view directions: every sample is sanitised (main.rs:448-459), never a crash
    g = np.random.default_rng(1)
    for trial in range(8):
        wild = sc.camera(32, 24)
        field = ["lookfrom", "lookat", "vup"][trial % 3]
        getattr(wild, field)[int(g.integers(0, 3))] = float(g.choice([np.nan, np.inf, -np.inf, 1e308]))
        if trial == 6:
            for k in range(3):
                wild.lookat[k] = wild.lookfrom[k]
        if trial == 7:
            wild.vfov_degrees, wild.aperture = 0.0, np.nan
        film, st = ctx.render(wild, 32, 24, 0, 2, max_depth=8, seed=1)
        assert np.isfinite(film).all() and st.paths == 32 * 24 * 2
        # (no comparison with the oracle here: what an all-NaN ray "hits" inside a BVH group depends on the tree's shape
        # in the reference itself -- bvh.rs:151-215 culls with NaN comparisons -- and is unspecified in include/yart.h)
    again, _ = ctx.render(cam, 32, 24, 0, 2, max_depth=8, seed=1)
    assert np.array_equal(good, again)


@pytest.mark.parametrize("seed", range(16))
def test_rays_with_nan_inf_and_zero_components(yart, orc, ctx, seed):
    """Rays the renderer can produce after a degenerate scatter (unit_vector of a zero vector is NaN, vec3.rs:204-212):
    the reference's answer is whatever its all-false NaN comparisons give -- a still sphere or a rect "hits" at t = NaN
    (sphere.rs:54-64, aarect.rs), the mesh ignores NaN slabs (qbvh.rs:495-519).  Same on the GPU, bit for bit.
    (Scenes without BVH groups: there the reference's own answer depends on its tree, see include/yart.h.)"""
    sc = FuzzScene(yart, 5000 + seed, allow_groups=False)
    s = orc.Scene(sc)
    ctx.set_scene(sc.desc)
    g = np.random.default_rng(seed)
    o, d = sc.rays(6000)
    m = g.random(o.shape) < 0.15
    o[m] = g.choice([np.nan, np.inf, -np.inf], size=int(m.sum()))
    m = g.random(d.shape) < 0.15
    d[m] = g.choice([np.nan, np.inf, -np.inf, 0.0, -0.0], size=int(m.sum()))
    o[:200], d[:200] = np.nan, np.nan                     # all-NaN rays
    d[200:400] = 0.0                                      # zero directions
    rays = yart.make_rays(o, d)
    want, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order)
        for f in HIT_FIELDS:
            same = (got[f] == want[f]) | ((got[f] != got[f]) & (want[f] != want[f]))
            bad = np.flatnonzero(~same)
            assert bad.size == 0, "seed %d order %d field %s: %d rays differ, first %d: ray %r gpu %r oracle %r" % (
                seed, order, f, bad.size, bad[0], rays[bad[0]], got[bad[0]], want[bad[0]])


@pytest.mark.parametrize("scene,seed", [("random-scene", 2), ("random-scene", 3), ("random-scene", 77), ("next-week-final", 2),
                                        ("next-week-final", 5), ("two-perlin-spheres", 9), ("simple-light", 4), ("cornell-box-smoke", 3)])
def test_seeded_presets_with_other_seeds(yart, orc, ctx, scene, seed):
    """The presets whose content depends on the scene seed (sphere fields, box heights, Perlin tables, medium draws) with
    seeds the other tests do not use: world closest hit bit-exact in both orders, a small render like the others."""
    preset = yart.ScenePreset(scene, seed=seed)
    s = orc.Scene(preset)
    ctx.set_scene(preset)
    w, h = 64, 40
    cam = preset.camera(w, h)
    rays, _, _ = ctx.camera_rays(cam, w, h, 0, 4, seed=seed)
    sd = preset.desc.contents
    medium = np.array([bool(sd.objects[i].wrap & yart.abi.WRAP_MEDIUM) for i in range(sd.n_objects)] + [False])
    want, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
    in_medium = medium[np.minimum(want["obj_id"], sd.n_objects)] & (want["prim_id"] != yart.MISS)
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order)
        for f in HIT_FIELDS:
            same = (got[f] == want[f]) | ((got[f] != got[f]) & (want[f] != want[f]))
            if f == "t":
                with np.errstate(invalid="ignore"):
                    same |= in_medium & (np.abs(got[f] - want[f]) <= 1e-12 * np.abs(want[f]))
            assert same.all(), (scene, seed, order, f, int((~same).sum()))
    want_film, st_w = s.render(cam, w, h, 0, 4, max_depth=20, seed=seed, n_threads=os.cpu_count())
    got_film, st = ctx.render(cam, w, h, 0, 4, max_depth=20, seed=seed)
    compare_films(got_film, want_film, "%s seed %d" % (scene, seed), 0.97)
