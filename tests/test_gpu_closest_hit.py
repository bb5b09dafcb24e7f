"""GPU parity, closest hit: yart_closest_hit (CUDA, through the C ABI) against the CPU oracle on
the same rays.  The bar is bit-exact: t, barycentrics, primitive id, object id and front_face
must be IDENTICAL -- the kernel does the reference's f64 arithmetic in the reference's order on
losslessly stored f32 geometry (north_star asks for exact prim id and 1e-5 relative t).
"""
import os

import numpy as np
import pytest

import raysets

pytestmark = pytest.mark.gpu
INF = float("inf")
FIELDS = ("t", "u", "v", "prim_id", "obj_id", "front_face")


def assert_same_hits(a, b, what=""):
    for f in FIELDS:
        if not np.array_equal(a[f], b[f]):
            bad = np.nonzero(a[f] != b[f])[0]
            raise AssertionError("%s: field %s differs on %d of %d rays, first %d: %r vs %r" %
                                 (what, f, len(bad), len(a), bad[0], a[bad[0]], b[bad[0]]))


def mesh_rays(orc, info, n, seed_shift=0):
    o1, d1 = raysets.uniform(n, info.bbox_min, info.bbox_max, raysets.SEED_UNIFORM + seed_shift)
    o2, d2 = raysets.axis(n // 2, info.bbox_min, info.bbox_max, raysets.SEED_AXIS + seed_shift)
    return orc.abi.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]))


@pytest.mark.parametrize("name,n", [("cube", 20000), ("sycee", 200000), ("david", 200000)])
def test_mesh_closest_hit_is_bit_exact(yart, orc, ctx, mesh_scene, name, n):
    _, ms, s = mesh_scene(name)
    ctx.set_scene(ms.desc)
    rays = mesh_rays(orc, s.qbvh_info(0), n)
    for t_min in (0.0, 0.001):
        want, cnt = s.closest_hit(rays, 0, t_min, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
        for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
            got, st = ctx.closest_hit(rays, 0, t_min, INF, order)
            assert_same_hits(got, want, "%s order %d t_min %g" % (name, order, t_min))
            assert st.rays == len(rays) and st.kernel_launches == 2 and st.gpu_ms > 0.0  # k_traverse + k_export
        assert (want["prim_id"] != yart.MISS).sum() > len(rays) // 20


def test_visit_counters_match_the_oracle(yart, orc, ctx, mesh_scene):
    """The roofline's algorithmic bytes come from these counts: the kernel must visit exactly the
    nodes and triangles the oracle's traversal visits."""
    _, ms, s = mesh_scene("david")
    ctx.set_scene(ms.desc)
    rays = mesh_rays(orc, s.qbvh_info(0), 50000)
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        _, cnt = s.closest_hit(rays, 0, 0.0, INF, order, n_threads=os.cpu_count())
        _, st = ctx.closest_hit(rays, 0, 0.0, INF, order, count_visits=True)
        assert st.node_visits == cnt.node_visits and st.tri_tests == cnt.tri_tests


def test_equal_t_ties_and_reference_quirks(yart, orc, ctx):
    """Integer height field: thousands of exact equal-t ties, flat leaves the reference never
    enters (strict tfar > tnear) and axis-parallel rays whose slabs are 0*inf = NaN."""
    pos, nrm, uv, h = raysets.grid_mesh()
    ms = orc.MeshScene(pos, nrm, uv)
    s = orc.Scene(ms)
    ctx.set_scene(ms.desc)
    o, d = raysets.grid_tie_rays(h, 20000)
    rays = orc.abi.make_rays(o, d)
    want, _ = s.closest_hit(rays, 0, 0.001, INF, yart.ORDER_REFERENCE)
    bf, ties = s.brute_force_hit(rays, 0, 0.001)
    assert ((ties > 1) & (want["t"] == bf["t"])).sum() > 2000
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, _ = ctx.closest_hit(rays, 0, 0.001, INF, order)
        assert_same_hits(got, want, "grid order %d" % order)


def test_sycee_axis_ray_through_shared_vertex(yart, orc, ctx, mesh_scene):
    _, ms, s = mesh_scene("sycee")
    ctx.set_scene(ms.desc)
    ray = orc.abi.make_rays([(0, 3, 0), (1, 5, -8)], [(0, -1, 0), (-1, -4.5, 8)])
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, _ = ctx.closest_hit(ray, 0, 0.001, INF, order)
        assert got[0]["prim_id"] == yart.MISS and got[0]["t"] == INF  # the reference's NaN-slab miss
        assert got[1]["prim_id"] == 6044 and abs(got[1]["t"] - 0.947010155709422) < 1e-14


def test_ragged_and_empty_inputs(yart, orc, ctx, mesh_scene):
    _, ms, s = mesh_scene("cube")
    ctx.set_scene(ms.desc)
    info = s.qbvh_info(0)
    empty = np.empty(0, dtype=yart.RAY_DTYPE)
    got, st = ctx.closest_hit(empty, 0)
    assert len(got) == 0 and st.rays == 0
    for n in (1, 31, 32, 33, 4097):
        o, d = raysets.uniform(n, info.bbox_min, info.bbox_max, 99 + n)
        rays = orc.abi.make_rays(o, d)
        want, _ = s.closest_hit(rays, 0, 0.001, INF, 0)
        got, _ = ctx.closest_hit(rays, 0, 0.001, INF, yart.ORDER_NEAR)
        assert_same_hits(got, want, "n=%d" % n)
    # degenerate rays: zero direction, NaN, infinities -> same answer as the oracle (all misses or not)
    weird = orc.abi.make_rays([(0, 0, 0), (0, 0, 5), (np.nan, 0, 0), (0, 0, 5), (0, 0, 5)],
                              [(0, 0, 0), (0, 0, -np.inf), (0, 0, 1), (0, np.nan, -1), (0, 0, -1e-300)])
    want, _ = s.closest_hit(weird, 0, 0.001, INF, 0)
    for order in (0, 1):
        got, _ = ctx.closest_hit(weird, 0, 0.001, INF, order)
        assert_same_hits(got, want, "weird rays")
    # a finite t_max cuts hits off exactly like the oracle
    o, d = raysets.uniform(5000, info.bbox_min, info.bbox_max, 5)
    rays = orc.abi.make_rays(o, d)
    want, _ = s.closest_hit(rays, 0, 0.25, 0.9, 0)
    got, _ = ctx.closest_hit(rays, 0, 0.25, 0.9, 1)
    assert_same_hits(got, want, "t window")


def test_error_behaviour(yart, ctx, mesh_scene):
    _, ms, _ = mesh_scene("cube")
    ctx.set_scene(ms.desc)
    rays = np.zeros(4, dtype=yart.RAY_DTYPE)
    with pytest.raises(yart.YartError) as e:
        ctx.closest_hit(rays, 7)  # no such mesh
    assert e.value.code == -1


@pytest.mark.parametrize("scene", ["david", "cornell-box", "cornell-box-smoke", "sycee", "three-spheres",
                                   "next-week-final", "random-scene"])
def test_world_closest_hit_is_bit_exact(yart, orc, ctx, scene):
    """HittableList::hit over whole presets: instances, spheres, rects, boxes, loose triangles,
    constant media (Philox draw inside the intersection), BVH groups."""
    preset = yart.ScenePreset(scene, seed=3)
    s = orc.Scene(preset)
    ctx.set_scene(preset)
    w, h = 96, 64
    cam = preset.camera(w, h)
    rays, _, _ = orc.camera_rays(cam, w, h, 0, 2, seed=5)
    # add incoherent rays from inside the scene's extent
    c = np.asarray(preset.info.lookat)
    r = np.linalg.norm(np.asarray(preset.info.lookfrom) - c)
    o, d = raysets.uniform(6000, c - 0.6 * r, c + 0.6 * r, 77)
    rays = np.concatenate([rays, orc.abi.make_rays(o, d)])
    want, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, 0, n_threads=os.cpu_count())
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order)
        if scene in ("cornell-box-smoke", "next-week-final"):
            # ConstantMedium takes log() of a uniform draw: CUDA's log may differ from glibc's in the
            # last bit, so t inside a medium is compared to 1e-12 relative, everything else exactly
            med = np.array([bool(preset.desc.contents.objects[int(i)].wrap & 8) if i != yart.MISS else False
                            for i in want["obj_id"]])
            assert np.array_equal(got["obj_id"], want["obj_id"])
            assert_same_hits(got[~med], want[~med], scene)
            assert np.allclose(got["t"][med], want["t"][med], rtol=1e-12, atol=0)
        else:
            assert_same_hits(got, want, "%s order %d" % (scene, order))
    assert (want["obj_id"] != yart.MISS).mean() > 0.3


def test_full_size_sweep_properties(yart, orc, ctx, mesh_scene):
    """BASELINE config 5 at full size (16 Mi rays vs david): too big for the oracle in seconds, so
    check size-independent properties: both traversal orders agree bit for bit, a second run is
    identical (idempotence / no races), hits lie inside the mesh AABB, and a 64 Ki-ray random
    subset equals the oracle."""
    _, ms, s = mesh_scene("david")
    ctx.set_scene(ms.desc)
    info = s.qbvh_info(0)
    n = 1 << 24
    o, d = raysets.uniform(n, info.bbox_min, info.bbox_max)
    rays = orc.abi.make_rays(o, d)
    a, st = ctx.closest_hit(rays, 0, 0.0, INF, yart.ORDER_REFERENCE)
    b, _ = ctx.closest_hit(rays, 0, 0.0, INF, yart.ORDER_NEAR)
    c, _ = ctx.closest_hit(rays, 0, 0.0, INF, yart.ORDER_NEAR)
    assert_same_hits(a, b, "orders")
    assert_same_hits(b, c, "rerun")
    hit = a["prim_id"] != yart.MISS
    assert 0.2 < hit.mean() < 0.95
    p = o[hit] + a["t"][hit, None] * d[hit]
    lo, hi = np.asarray(info.bbox_min), np.asarray(info.bbox_max)
    assert (p >= lo - 1e-6).all() and (p <= hi + 1e-6).all()
    assert a["prim_id"][hit].max() < info.n_tris
    idx = np.random.Generator(np.random.Philox(3)).choice(n, 1 << 16, replace=False)
    want, _ = s.closest_hit(rays[idx], 0, 0.0, INF, 0, n_threads=os.cpu_count())
    assert_same_hits(a[idx], want, "subset")


def test_fetch_peak_diagnostic(yart, ctx):
    """yart_measure_fetch_peak (the L1 / L2 fetch roofline of SURVEY.md 8(d)): sane numbers, loud argument errors."""
    l1 = ctx.measure_fetch_peak(128 * 1024, 1024, 0)
    l2 = ctx.measure_fetch_peak(7_400_000, 1024, 0)
    assert 1000.0 < l2 < 40000.0 and 1000.0 < l1 < 40000.0 and l1 > 0.9 * l2
    # modes 2 / 3: four lanes per line (one 256-bit load each) -- far fewer L1 wavefronts per line, a much higher roof
    quad = ctx.measure_fetch_peak(7_400_000, 1024, 2)
    assert quad > 1.5 * l2 and ctx.measure_fetch_peak(7_400_000, 1024, 3) > 1.5 * l2
    with pytest.raises(yart.YartError):
        ctx.measure_fetch_peak(1 << 20, 1024, 4)
    with pytest.raises(yart.YartError):
        ctx.measure_fetch_peak(64, 1024, 0)
    with pytest.raises(yart.YartError):
        ctx.measure_fetch_peak(1 << 20, 0, 0)
