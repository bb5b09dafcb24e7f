"""GPU parity, hit records: yart_closest_hit_records against the CPU reference of tests/record_ref.cpp (the oracle's own
world.hit HitRecord, rays at their own time) and against the library's own yart_closest_hit.  Every field is
bit-identical except those a libm call produces (tests/record_sets.py: sphere u, v; a constant medium's t and p)."""
import ctypes as C
import os

import numpy as np
import pytest

import raysets
import record_ref
from record_sets import SmallWorld, assert_records_match
from scene_fuzz import FuzzScene

pytestmark = pytest.mark.gpu
INF = float("inf")
NT = os.cpu_count()
ORDERS = (0, 1)
PRESETS = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
           "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]


def assert_same_as_closest_hit(yart, rec, hits, what):
    """With times NULL: t, obj_id, prim_id, front_face are yart_closest_hit's, bit for bit."""
    for f in ("t", "obj_id", "prim_id", "front_face"):
        assert rec[f].tobytes() == hits[f].tobytes(), "%s: %s differs from yart_closest_hit" % (what, f)


@pytest.mark.parametrize("name,n", [("cube", 20000), ("sycee", 100000), ("david", 100000)])
def test_mesh_targets(yart, orc, ctx, mesh_scene, name, n):
    _, ms, s = mesh_scene(name)
    ctx.set_scene(ms.desc)
    ref = record_ref.Scene(ms)
    info = s.qbvh_info(0)
    o1, d1 = raysets.uniform(n, info.bbox_min, info.bbox_max, raysets.SEED_UNIFORM + 9)
    o2, d2 = raysets.axis(n // 2, info.bbox_min, info.bbox_max, raysets.SEED_AXIS + 9)
    rays = yart.make_rays(np.concatenate([o1, o2]), np.concatenate([d1, d2]))
    want = ref.records(rays, None, 0, 0.001, INF, yart.ORDER_REFERENCE, n_threads=NT)
    assert (want["obj_id"] != yart.MISS).sum() > len(rays) // 20
    for order in ORDERS:
        got, st = ctx.closest_hit_records(rays, None, 0, 0.001, INF, order)
        assert_records_match(yart.abi, ms.desc, rays, got, want, 0, "%s order %d" % (name, order))
        assert (got["material"] == yart.MISS).all()
        assert st.rays == len(rays) and st.kernel_launches == 2 and st.trace_launches == 1 and st.gpu_ms > 0.0
        hits, _ = ctx.closest_hit(rays, 0, 0.001, INF, order)
        assert_same_as_closest_hit(yart, got, hits, "%s order %d" % (name, order))


def test_mesh_ties_and_boundaries(yart, orc, ctx):
    """Integer height field: exact equal-t ties, flat leaves, NaN slabs; and the t_max boundary of the strict test."""
    pos, nrm, uv, h = raysets.grid_mesh()
    ms = orc.MeshScene(pos, nrm, uv)
    ctx.set_scene(ms.desc)
    ref = record_ref.Scene(ms)
    rays = yart.make_rays(*raysets.grid_tie_rays(h, 20000))
    for t_max in (INF, 8.0, np.nextafter(8.0, INF)):
        want = ref.records(rays, None, 0, 0.001, t_max, yart.ORDER_REFERENCE)
        for order in ORDERS:
            got, _ = ctx.closest_hit_records(rays, None, 0, 0.001, t_max, order)
            assert_records_match(yart.abi, ms.desc, rays, got, want, 0, "grid t_max %r order %d" % (t_max, order))


@pytest.mark.parametrize("scene", PRESETS)
def test_presets_camera_rays_with_their_times(yart, orc, ctx, scene):
    """The renderer's own camera rays, each at the time yart_generate_camera_rays drew for it, over the whole world."""
    preset = yart.ScenePreset(scene, seed=3)
    ctx.set_scene(preset)
    ref = record_ref.Scene(preset)
    cam = preset.camera(96, 64)
    rays, _, times = ctx.camera_rays(cam, 96, 64, 0, 2, seed=5)
    assert times.min() >= 0.0 and times.max() <= 1.0 and times.std() > 0.1
    want = ref.records(rays, times, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=NT)
    assert (want["obj_id"] != yart.MISS).any()
    for order in ORDERS:
        got, _ = ctx.closest_hit_records(rays, times, yart.TARGET_WORLD, 0.001, INF, order)
        assert_records_match(yart.abi, preset.desc, rays, got, want, yart.TARGET_WORLD, "%s order %d" % (scene, order))


@pytest.mark.parametrize("scene", PRESETS)
def test_presets_path_rays(yart, orc, ctx, scene):
    """yart_dump_path_rays sets (every bounce's rays), times NULL; and yart_closest_hit's answer on them."""
    preset = yart.ScenePreset(scene, seed=3)
    ctx.set_scene(preset)
    ref = record_ref.Scene(preset)
    cam = preset.camera(64, 48)
    rays, _ = ctx.dump_path_rays(cam, 64, 48, 0, 2, 1 << 17, max_depth=8)
    want = ref.records(rays, None, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=NT)
    for order in ORDERS:
        got, _ = ctx.closest_hit_records(rays, None, yart.TARGET_WORLD, 0.001, INF, order)
        assert_records_match(yart.abi, preset.desc, rays, got, want, yart.TARGET_WORLD, "%s order %d" % (scene, order))
        hits, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order)
        assert_same_as_closest_hit(yart, got, hits, "%s order %d" % (scene, order))


@pytest.mark.parametrize("seed", range(40))
def test_random_worlds(yart, orc, ctx, seed):
    """Random worlds (tests/scene_fuzz.py), rays at random times, two t windows."""
    sc = FuzzScene(yart, 1000 + seed)
    ctx.set_scene(sc.desc)
    ref = record_ref.Scene(sc)
    rays = yart.make_rays(*sc.rays(20000))
    times = np.random.default_rng(seed).uniform(0.0, 1.0, len(rays))
    for t_min, t_max in ((0.001, INF), (0.0, 3.5)):
        want = ref.records(rays, times, yart.TARGET_WORLD, t_min, t_max, yart.ORDER_REFERENCE, n_threads=NT)
        for order in ORDERS:
            got, _ = ctx.closest_hit_records(rays, times, yart.TARGET_WORLD, t_min, t_max, order)
            assert_records_match(yart.abi, sc.desc, rays, got, want, yart.TARGET_WORLD, "seed %d order %d" % (seed, order))
    got, _ = ctx.closest_hit_records(rays, None, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR)
    hits, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR)
    assert_same_as_closest_hit(yart, got, hits, "seed %d" % seed)


@pytest.mark.parametrize("scene", ["next-week-final", "random-scene"])
def test_non_zero_times(yart, orc, ctx, scene):
    """Rays at time 1 and at random times equal the reference's at those times; on next-week-final, whose MovingSphere
    is in view, some of them hit other things than at time 0."""
    preset = yart.ScenePreset(scene, seed=3)
    ctx.set_scene(preset)
    ref = record_ref.Scene(preset)
    cam = preset.camera(160, 120)
    rays, _, _ = ctx.camera_rays(cam, 160, 120, 0, 1, seed=5)
    at0, _ = ctx.closest_hit_records(rays, None, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR)
    for times in (np.ones(len(rays)), np.random.default_rng(4).uniform(0.0, 1.0, len(rays))):
        want = ref.records(rays, times, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=NT)
        got, _ = ctx.closest_hit_records(rays, times, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR)
        assert_records_match(yart.abi, preset.desc, rays, got, want, yart.TARGET_WORLD, scene)
        if scene == "next-week-final":
            moved = (got["t"] != at0["t"]) | (got["obj_id"] != at0["obj_id"])
            kinds = [preset.desc.contents.objects[int(i)].kind for i in np.concatenate([got["obj_id"], at0["obj_id"]])[
                np.concatenate([moved, moved])] if i != yart.MISS]
            assert moved.sum() > 10 and yart.abi.OBJ_MOVING_SPHERE in kinds


def test_small_world_groups_and_a_moving_sphere(yart, orc, ctx):
    world = SmallWorld(yart.abi)
    ctx.set_scene(world.desc)
    ref = record_ref.Scene(world)
    rays = np.concatenate([world.group_rays(), world.moving_rays()])
    for time in (0.0, 0.37, 1.0):
        times = np.full(len(rays), time)
        want = ref.records(rays, times)
        got, _ = ctx.closest_hit_records(rays, times)
        assert_records_match(yart.abi, world.desc, rays, got, want, yart.TARGET_WORLD, "time %g" % time)
        on_group = got["obj_id"] == 0
        assert on_group.sum() > 100 and np.array_equal(got["material"][on_group], got["prim_id"][on_group])
        assert ((got["obj_id"] == 1) & (got["material"] == 4)).sum() > 20


def test_host_device_and_chunked_arrays(yart, orc, ctx, monkeypatch):
    """Device arrays, host arrays in one piece, ragged host chunks with and without times, a pinned output array."""
    import torch
    preset = yart.ScenePreset("next-week-final", seed=1)
    ctx.set_scene(preset)
    cam = preset.camera(320, 240)
    rays, _, times = ctx.camera_rays(cam, 320, 240, 0, 3)          # 230,400 rays through groups, media, a moving sphere
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", str(1 << 30))
    whole_t, st_w = ctx.closest_hit_records(rays, times, order=yart.ORDER_NEAR, count_visits=True)
    whole_0, _ = ctx.closest_hit_records(rays, None, order=yart.ORDER_NEAR)
    assert whole_t.tobytes() != whole_0.tobytes()
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", "4099")              # 57 ragged chunks
    parts_t, st_p = ctx.closest_hit_records(rays, times, order=yart.ORDER_NEAR, count_visits=True)
    parts_0, _ = ctx.closest_hit_records(rays, None, order=yart.ORDER_NEAR)
    assert parts_t.tobytes() == whole_t.tobytes() and parts_0.tobytes() == whole_0.tobytes()
    assert (st_p.rays, st_p.node_visits, st_p.tri_tests) == (st_w.rays, st_w.node_visits, st_w.tri_tests)
    n_chunks = (len(rays) + 4098) // 4099
    assert st_p.kernel_launches - st_p.trace_launches == n_chunks and st_w.kernel_launches - st_w.trace_launches == 1
    out = np.zeros(len(rays), dtype=yart.RECORD_DTYPE)
    ctx.host_register(out)
    try:
        ctx.closest_hit_records(rays, times, order=yart.ORDER_NEAR, out=out)
    finally:
        ctx.host_unregister(out)
    assert out.tobytes() == whole_t.tobytes()
    dev = torch.device("cuda", 0)
    rd = torch.from_numpy(rays.view(np.uint8)).to(dev)
    td = torch.from_numpy(times).to(dev)
    od = torch.zeros(len(rays) * 88, dtype=torch.uint8, device=dev)
    st = ctx.closest_hit_records_device(rd.data_ptr(), td.data_ptr(), len(rays), od.data_ptr(), order=yart.ORDER_NEAR)
    assert od.cpu().numpy().tobytes() == whole_t.tobytes() and st.gpu_ms > 0.0
    ctx.closest_hit_records_device(rd.data_ptr(), 0, len(rays), od.data_ptr(), order=yart.ORDER_NEAR)
    assert od.cpu().numpy().tobytes() == whole_0.tobytes()


def test_ragged_sizes_empty_input_and_an_empty_world(yart, orc, ctx, mesh_scene):
    _, ms, s = mesh_scene("cube")
    ctx.set_scene(ms.desc)
    ref = record_ref.Scene(ms)
    info = s.qbvh_info(0)
    got, st = ctx.closest_hit_records(np.empty(0, dtype=yart.RAY_DTYPE), target=0)
    assert len(got) == 0 and st.rays == 0 and st.kernel_launches == 0
    for n in (1, 31, 32, 33, 4097):
        rays = yart.make_rays(*raysets.uniform(n, info.bbox_min, info.bbox_max, 99 + n))
        got, _ = ctx.closest_hit_records(rays, None, 0, 0.001, INF, yart.ORDER_NEAR)
        assert_records_match(yart.abi, ms.desc, rays, got, ref.records(rays, None, 0), 0, "n=%d" % n)
    empty = yart.abi.SceneDesc()
    ctx.set_scene(C.pointer(empty))
    rays = yart.make_rays(*raysets.uniform(100, [-1, -1, -1], [1, 1, 1], 3))
    got, _ = ctx.closest_hit_records(rays, np.ones(100))
    assert np.isinf(got["t"]).all() and (got["obj_id"] == yart.MISS).all() and (got["material"] == yart.MISS).all()
    assert (got["prim_id"] == yart.MISS).all() and (got["p"] == 0).all() and (got["normal"] == 0).all()


def test_argument_errors(yart, ctx, mesh_scene):
    lib = yart.load_library()
    rays = np.zeros(4, dtype=yart.RAY_DTYPE)
    times = np.zeros(4)
    out = np.zeros(4, dtype=yart.RECORD_DTYPE)
    fresh = yart.Context(0)
    try:  # no scene
        assert lib.yart_closest_hit_records(fresh._h, 0, rays.ctypes.data, None, 4, 0.0, INF, 0, 0, out.ctypes.data, None) == -1
        assert b"no scene" in lib.yart_last_error(fresh._h)
    finally:
        fresh.close()
    _, ms, _ = mesh_scene("cube")
    ctx.set_scene(ms.desc)

    def call(target=0, r=rays.ctypes.data, t=times.ctypes.data, n=4, order=0, flags=0, o=out.ctypes.data):
        return lib.yart_closest_hit_records(ctx._h, target, r, t, n, 0.0, INF, order, flags, o, None)

    assert call(r=None) == -1 and call(o=None) == -1
    assert call(n=0xFFFFFFF1) == -1
    assert call(target=7) == -1 and b"target" in lib.yart_last_error(ctx._h)
    assert call(order=2) == -1
    for bad in (4, 8, 16, 32, 64, 1 << 31):
        assert call(flags=bad) == -1
    assert b"YART_FLAG_DEVICE_PTRS" in lib.yart_last_error(ctx._h)
    D = yart.FLAG_DEVICE_PTRS
    assert call(flags=D, r=(1 << 40) + 8) == -1 and b"aligned" in lib.yart_last_error(ctx._h)
    assert call(flags=D, r=1 << 40, o=(1 << 40) + 4) == -1 and b"aligned" in lib.yart_last_error(ctx._h)
    assert call(flags=D, r=1 << 40, o=1 << 41, t=(1 << 42) + 4) == -1 and b"time" in lib.yart_last_error(ctx._h)
    st = yart.abi.Stats()
    st.rays = 99
    assert lib.yart_closest_hit_records(ctx._h, 0, None, None, 0, 0.0, INF, 0, 0, None, C.byref(st)) == 0 and st.rays == 0
    assert call() == 0 and call(t=None) == 0 and call(flags=yart.FLAG_COUNT_VISITS) == 0
