"""GPU tests of the round-2 additions to the C ABI: sampling flags (vs the oracle's mirror), yart_closest_hit_f32,
device-resident films + the NCCL communicator (yart_comm_*, yart_film_reduce), scene validation, memory-bounded
batches."""
import ctypes as C
import os
import subprocess
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

import raysets
from test_gpu_render import compare_films

pytestmark = pytest.mark.gpu
INF = float("inf")
ROOT = Path(__file__).resolve().parent.parent


# ---------------------------------------------------------------------------------------------------------
# sampling flags
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene,depth", [("cornell-box", 50), ("david", 50), ("cornell-box", 4)])
def test_sampling_flags_match_the_oracle(yart, orc, ctx, scene, depth):
    preset = yart.ScenePreset(scene, seed=1)
    s = orc.Scene(preset)
    ctx.set_scene(preset)
    w = h = 64
    cam = preset.camera(w, h)
    base, st0 = ctx.render(cam, w, h, 0, 8, max_depth=depth, seed=3)
    again, _ = ctx.render(cam, w, h, 0, 8, max_depth=depth, seed=3, flags=0)
    assert np.array_equal(base, again)
    combos = [yart.FLAG_UNBIASED_LIGHT_PICK, yart.FLAG_RUSSIAN_ROULETTE, yart.FLAG_DEPTH_ZERO_BLACK,
              yart.FLAG_UNBIASED_LIGHT_PICK | yart.FLAG_RUSSIAN_ROULETTE | yart.FLAG_DEPTH_ZERO_BLACK]
    for flags in combos:
        want, st_w = s.render(cam, w, h, 0, 8, max_depth=depth, seed=3, n_threads=os.cpu_count(), flags=flags)
        for order in (yart.ORDER_NEAR, yart.ORDER_REFERENCE):
            got, st = ctx.render(cam, w, h, 0, 8, max_depth=depth, seed=3, order=order, flags=flags)
            compare_films(got, want, "%s depth %d flags %d order %d" % (scene, depth, flags, order), 0.97)
            assert abs(int(st.rays) - int(st_w.rays)) <= max(4, st_w.rays // 500)
        if flags == yart.FLAG_RUSSIAN_ROULETTE and depth == 50:
            assert st.rays < st0.rays
        if flags == yart.FLAG_UNBIASED_LIGHT_PICK and scene == "cornell-box" and depth == 50:
            assert got[..., 1].sum() < 0.85 * base[..., 1].sum()


# ---------------------------------------------------------------------------------------------------------
# f32 ray records
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["sycee", "david"])
def test_closest_hit_f32_equals_the_f64_query_on_widened_rays(yart, orc, ctx, mesh_scene, name):
    _, ms, s = mesh_scene(name)
    ctx.set_scene(ms.desc)
    info = s.qbvh_info(0)
    o, d = raysets.uniform(300000, info.bbox_min, info.bbox_max, 31)
    r32 = np.empty(len(o), dtype=yart.abi.RAY_F32_DTYPE)
    r32["origin"], r32["direction"] = o.astype(np.float32), d.astype(np.float32)
    r64 = orc.abi.make_rays(r32["origin"].astype(np.float64), r32["direction"].astype(np.float64))
    want, _ = s.closest_hit(r64, 0, 0.001, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())  # the ORACLE on the widened rays
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got, st = ctx.closest_hit_f32(r32, 0, 0.001, INF, order)
        assert np.array_equal(got["prim_id"], want["prim_id"])
        hit = want["prim_id"] != yart.MISS
        assert np.array_equal(got["t"][hit], want["t"][hit].astype(np.float32))
        assert np.array_equal(got["u"][hit], want["u"][hit].astype(np.float32))
        assert np.array_equal(got["v"][hit], want["v"][hit].astype(np.float32))
        assert np.isinf(got["t"][~hit]).all() and st.rays == len(r32)
    # ragged sizes, the world target, and an unaligned-size tail
    for n in (1, 33, 4099):
        g, _ = ctx.closest_hit_f32(r32[:n], yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR)
        assert np.array_equal(g["prim_id"], want["prim_id"][:n])
    empty, st = ctx.closest_hit_f32(r32[:0], 0)
    assert len(empty) == 0 and st.rays == 0


# ---------------------------------------------------------------------------------------------------------
# device films + communicator
# ---------------------------------------------------------------------------------------------------------
def test_device_film_round_trip_and_single_rank_comm(yart, ctx):
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    w = h = 64
    cam = preset.camera(w, h)
    want, _ = ctx.render(cam, w, h, 0, 6, seed=2)
    film = ctx.film_create(w, h)
    try:
        assert not ctx.film_read(film, w, h).any()  # zeroed on creation
        ctx.render_device(cam, w, h, 0, 6, film, seed=2)
        assert np.array_equal(ctx.film_read(film, w, h), want)
        comm = yart.Comm.from_id(ctx, yart.comm_unique_id(), 0, 1)  # a one-rank group: the reduce is the identity
        info = comm.info()
        assert info["n_ranks"] == 1 and info["n_local"] == 1 and info["nccl_version"] >= 20000
        comm.film_reduce(film, w, h, root=0)
        assert np.array_equal(ctx.film_read(film, w, h), want)
        comm.film_reduce(film, w, h, root=-1)  # all-reduce flavour
        assert np.array_equal(ctx.film_read(film, w, h), want)
        with pytest.raises(yart.YartError):
            comm.film_reduce(film, w, h, root=3)
        comm.close()
        ctx.film_clear(film, w, h)
        assert not ctx.film_read(film, w, h).any()
        # the same GPU twice is refused (one rank per GPU), loudly
        with pytest.raises(yart.YartError):
            yart.Comm.from_contexts([ctx, ctx])
    finally:
        ctx.film_destroy(film)


def test_n_gpu_film_equals_one_gpu_film(yart):
    """SURVEY.md 8(e) on hardware: N contexts in one process (one host thread each), every GPU renders its sample
    range of every pixel, one in-place ncclReduce -- the root's film equals the 1-GPU film to f64-sum tolerance.
    Needs >= 2 visible GPUs (`gpurun --gpus 2`); the one-rank path is covered by the test above."""
    if yart.device_count() < 2:
        pytest.skip("one GPU visible: the N-GPU equality needs `gpurun --gpus 2` (see profiles/r2_multi_gpu_film_equality.txt)")
    sh = __import__("importlib").import_module("yet-another-raytracer_b200.sharding")
    n = min(yart.device_count(), 4)
    preset = yart.ScenePreset("david", seed=1)
    w, h, spp = 320, 184, 37  # (37 does not divide evenly: ragged shards)
    ctxs = [yart.Context(i) for i in range(n)]
    for c in ctxs:
        c.set_scene(preset)
    cam = preset.camera(w, h)
    single, st1 = ctxs[0].render(cam, w, h, 0, spp, seed=5)
    films = [c.film_create(w, h) for c in ctxs]
    comm = yart.Comm.from_contexts(ctxs)
    assert comm.info()["n_ranks"] == n
    errs = []

    def work(r):
        try:
            lo, hi = sh.shard_range(0, spp, r, n)
            ctxs[r].render_device(cam, w, h, lo, hi, films[r], seed=5)
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    threads = [threading.Thread(target=work, args=(r,)) for r in range(n)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errs, errs
    comm.film_reduce(films, w, h, root=0)
    got = ctxs[0].film_read(films[0], w, h)
    err = np.abs(got - single).max() / np.abs(single).max()
    print("N=%d GPUs: max |film_N - film_1| / max|film| = %.3g" % (n, err))
    assert err <= 1e-13 and got.sum() > 0
    other = ctxs[1].film_read(films[1], w, h)   # a non-root keeps its partial sum
    assert other.sum() < got.sum()
    comm.close()
    for c, f in zip(ctxs, films):
        c.film_destroy(f)
        c.close()


# ---------------------------------------------------------------------------------------------------------
# validation: a bad descriptor is YART_ERR_INVALID, never a wild device load
# ---------------------------------------------------------------------------------------------------------
def test_set_scene_rejects_malformed_descriptions(yart, ctx):
    abi = yart.abi

    def scene(objects, materials, textures, groups=(), images=()):
        sd = abi.SceneDesc()
        keep = []
        for field, cls, items in (("objects", abi.Object, objects), ("materials", abi.Material, materials),
                                  ("textures", abi.Texture, textures), ("groups", abi.Group, groups), ("images", abi.Image, images)):
            arr = (cls * max(len(items), 1))(*items)
            keep.append(arr)
            setattr(sd, field, C.cast(arr, C.POINTER(cls)))
            setattr(sd, "n_" + field, len(items))
        return sd, keep

    def sphere(material):
        o = abi.Object()
        o.kind, o.material, o.cos_theta = abi.OBJ_SPHERE, material, 1.0
        o.p[3] = 1.0
        return o

    lam, tex = abi.Material(), abi.Texture()
    lam.kind, tex.kind = abi.MAT_LAMBERTIAN, abi.TEX_SOLID
    ok, keep = scene([sphere(0)], [lam], [tex])
    ctx.set_scene(C.pointer(ok))
    cases = {}
    cases["object material out of range"] = scene([sphere(5)], [lam], [tex])
    member = sphere(7)                                    # group member with a missing material (ADVICE r1)
    members = (abi.Object * 1)(member)
    g = abi.Group()
    g.members, g.n_members = C.cast(members, C.POINTER(abi.Object)), 1
    grp = abi.Object()
    grp.kind, grp.index, grp.cos_theta = abi.OBJ_GROUP, 0, 1.0
    cases["group member material out of range"] = scene([grp], [lam], [tex], groups=[g])
    img_tex = abi.Texture()
    img_tex.kind, img_tex.image = abi.TEX_IMAGE, 0
    pixels = (C.c_uint8 * 12)()
    for wd, ht, ptr in ((0, 2, pixels), (2, 0, pixels), (2, 2, None)):   # empty images under a TEX_IMAGE
        im = abi.Image()
        im.width, im.height = wd, ht
        im.rgb8 = C.cast(ptr, C.POINTER(C.c_uint8)) if ptr is not None else None
        cases["image %dx%d %s" % (wd, ht, "null" if ptr is None else "data")] = scene([sphere(0)], [lam], [img_tex], images=[im])
    bad_tex = abi.Material()
    bad_tex.kind, bad_tex.texture = abi.MAT_LAMBERTIAN, 9
    cases["material texture out of range"] = scene([sphere(0)], [bad_tex], [tex])
    nullptr_objs, k2 = scene([sphere(0)], [lam], [tex])
    nullptr_objs.objects = None                            # count 1, pointer null
    cases["null objects pointer"] = (nullptr_objs, k2)
    g2 = abi.Group()
    g2.members, g2.n_members = None, 3
    cases["null group members"] = scene([grp], [lam], [tex], groups=[g2])
    for what, (sd, _keep) in cases.items():
        with pytest.raises(yart.YartError) as e:
            ctx.set_scene(C.pointer(sd))
        assert e.value.code == -1, what
        # and nothing half-built stays behind: a query now fails cleanly instead of touching freed tables
        with pytest.raises(yart.YartError):
            ctx.closest_hit(np.zeros(1, dtype=yart.RAY_DTYPE))
    ctx.set_scene(C.pointer(ok))  # the context is still usable
    hits, _ = ctx.closest_hit(yart.make_rays([(0, 0, -5)], [(0, 0, 1)]))
    assert hits[0]["t"] == 4.0


def test_stand_in_meshes_are_announced(yart, tmp_path):
    for name in ("bunny", "teapot"):
        p = yart.ScenePreset(name)
        assert "stands in" in p.note and name + ".obj" in p.note
    assert yart.ScenePreset("david").note == ""
    code = ("import importlib, sys\nsys.path.insert(0, %r)\ny = importlib.import_module('yet-another-raytracer_b200')\n"
            "try:\n    y.ScenePreset('bunny')\nexcept y.YartError as e:\n    print('code', e.code, e)\n") % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, YART_STRICT_ASSETS="1"), capture_output=True, text=True)
    assert "code -4" in out.stdout and "Failed to load OBJ file" in out.stdout, out.stdout + out.stderr


# ---------------------------------------------------------------------------------------------------------
# memory-bounded batches
# ---------------------------------------------------------------------------------------------------------
def test_small_state_budget_gives_the_same_film(yart, ctx, tmp_path):
    """The wavefront batch is sized from free device memory; forcing a 2 MB state budget (YART_TUNE_STATE_MB, read
    once per process) cuts the frame into pixel chunks and sample batches -- the film must not change."""
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    w = h = 96
    want, st = ctx.render(preset.camera(w, h), w, h, 0, 5, seed=6)
    code = ("import importlib, sys, numpy as np\nsys.path.insert(0, %r)\n"
            "y = importlib.import_module('yet-another-raytracer_b200')\np = y.ScenePreset('cornell-box', seed=1)\n"
            "c = y.Context(0); c.set_scene(p)\nf, st = c.render(p.camera(96, 96), 96, 96, 0, 5, seed=6)\n"
            "np.save(%r, f); print('launches', st.kernel_launches)\n") % (str(ROOT), str(tmp_path / "f.npy"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, YART_TUNE_STATE_MB="2"), capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert np.array_equal(np.load(tmp_path / "f.npy"), want)
    assert int(out.stdout.split("launches")[1]) > st.kernel_launches  # it really ran in more, smaller batches


def test_render_reports_nomem_instead_of_a_raw_cuda_error(yart, ctx):
    """Hog the device (torch caching allocator) until less than the margin is free: yart_render must return
    YART_ERR_NOMEM with a message, and work again once the memory is back."""
    import torch
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    w = h = 64
    cam = preset.camera(w, h)
    c2 = yart.Context(0)  # a fresh context: it holds no state buffers yet, so only FREE memory counts for it
    c2.set_scene(preset)
    free, total = torch.cuda.mem_get_info(0)
    hog = torch.empty(free - (96 << 20), dtype=torch.uint8, device="cuda:0")
    try:
        with pytest.raises(yart.YartError) as e:
            c2.render(cam, w, h, 0, 1, seed=1)
        assert e.value.code == -3 and "free device memory" in str(e.value)
    finally:
        del hog
        torch.cuda.empty_cache()
    film, st = c2.render(cam, w, h, 0, 1, seed=1)
    assert st.paths == w * h and film.sum() > 0
    c2.close()


# ---------------------------------------------------------------------------------------------------------
# the renderer's own ray distribution
# ---------------------------------------------------------------------------------------------------------
def test_dump_path_rays_is_what_the_renderer_traces(yart, orc, ctx):
    """yart_dump_path_rays: every world.hit ray of the paths, bounce by bounce.  Bounce 1 must be exactly the camera
    rays (as a set: queue order is not pixel order), the count must equal the render's ray count, and tracing the dumped
    rays -- a large set of REAL secondary rays, origins on surfaces -- must agree with the oracle bit for bit."""
    preset = yart.ScenePreset("david", seed=1)
    s = orc.Scene(preset)
    ctx.set_scene(preset)
    w, h, spp = 160, 96, 3
    cam = preset.camera(w, h)
    _, st = ctx.render(cam, w, h, 0, spp, seed=4)
    rays, n = ctx.dump_path_rays(cam, w, h, 0, spp, 1 << 20, seed=4)
    assert n == st.rays == len(rays)
    prim, _, _ = orc.camera_rays(cam, w, h, 0, spp, seed=4)
    key = lambda r: np.sort(np.ascontiguousarray(r).view([("", "<f8")] * 6).reshape(-1))  # noqa: E731
    assert np.array_equal(key(rays[:w * h * spp]), key(prim))
    # the oracle's own dump of the same samples: the same number of rays (up to a rare last-bit path flip), and most of
    # them IDENTICAL bit for bit -- a bounce sampled through CUDA's sin / cos may differ from glibc's in the last bit of
    # its direction, and every later ray of that path inherits the difference (measured: 87 % identical)
    odump = s.dump_path_rays(cam, w, h, 0, spp, 1 << 20, seed=4)
    assert abs(len(odump) - n) <= max(4, n // 1000)
    common = np.intersect1d(key(rays), key(odump))
    assert len(common) >= 0.7 * n
    # capped output: the count is still the total
    few, n2 = ctx.dump_path_rays(cam, w, h, 0, spp, 1000, seed=4)
    assert n2 == n and len(few) == 1000
    assert np.isin(key(few), key(rays[:w * h * spp])).all()  # (queue order within a bounce is not reproducible run to run)
    # batches of one sample: same rays, grouped sample by sample
    by1, n3 = ctx.dump_path_rays(cam, w, h, 0, spp, 1 << 20, seed=4, batch_spp=1)
    assert n3 == n and np.array_equal(key(by1), key(rays))
    want, _ = s.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE, n_threads=os.cpu_count())
    for order in (yart.ORDER_NEAR, yart.ORDER_REFERENCE):
        got, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, order)
        for f in ("t", "u", "v", "prim_id", "obj_id", "front_face"):
            assert np.array_equal(got[f], want[f]), f
    assert (want["obj_id"] != yart.MISS).mean() > 0.4


# ---------------------------------------------------------------------------------------------------------
# the one-process multi-GPU renderer and the CLI additions
# ---------------------------------------------------------------------------------------------------------
def test_multi_gpu_renderer_progressive_and_against_single_context(yart, ctx):
    """sharding.MultiGpuRenderer on every visible GPU (1 on the default box, 2+ under `gpurun --gpus N`): chained
    sample ranges with a read-out in between give the film of one uninterrupted single-context render."""
    import importlib
    sh = importlib.import_module("yet-another-raytracer_b200.sharding")
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    w = h = 72
    cam = preset.camera(w, h)
    want, st = ctx.render(cam, w, h, 0, 11, seed=8)
    n = min(yart.device_count(), 4)
    mg = sh.MultiGpuRenderer(yart, range(n))
    try:
        mg.set_scene(preset)
        sts = mg.render(cam, w, h, 0, 4, seed=8)
        part = mg.film()                                  # reduce #1: the root keeps the total, the others restart at 0
        first, _ = ctx.render(cam, w, h, 0, 4, seed=8)
        assert np.allclose(part, first, rtol=1e-13, atol=1e-13 * np.abs(first).max())
        sts += mg.render(cam, w, h, 4, 11, seed=8)
        got = mg.film()                                   # reduce #2 adds only what came since
        assert sum(s.paths for s in sts) == st.paths
        if n == 1:
            assert np.array_equal(got, want)              # one GPU: the very same additions in the same order
        assert np.allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max())
        rgba = mg.finalize(11)
        assert (np.abs(rgba.astype(int) - ctx.film_finalize(want, 11).astype(int)) <= 1).all()
        # resuming from a host film
        mg.load_film(first)
        mg.render(cam, w, h, 4, 11, seed=8)
        assert np.allclose(mg.film(), want, rtol=1e-13, atol=1e-13 * np.abs(want).max())
    finally:
        mg.close()


def test_cli_sampling_flags_gpus_and_checkpoint_guard(yart, tmp_path):
    import importlib
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    from PIL import Image
    base = ["--scene", "cornell-box", "--width", "64", "--seed", "3", "--samples", "16"]
    a, b, c, ck = (str(tmp_path / n) for n in ("a.png", "b.png", "c.png", "ck.npz"))
    assert cli.main(base + ["--output", a, "--checkpoint", ck]) == 0
    assert cli.main(base + ["--output", b, "--unbiased-light-pick"]) == 0
    ia, ib = np.asarray(Image.open(a)).astype(float), np.asarray(Image.open(b)).astype(float)
    assert ib[..., :3].mean() < 0.9 * ia[..., :3].mean()   # the unbiased pick is visibly darker (SURVEY A-2)
    # --gpus: as many as are visible (1 on the default box) must give the same picture up to the last bit of a sum
    n = min(yart.device_count(), 2)
    assert cli.main(base + ["--output", c, "--gpus", str(n)]) == 0
    ic = np.asarray(Image.open(c)).astype(float)
    assert np.abs(ic - ia).max() <= 1
    with pytest.raises(SystemExit):
        cli.main(base + ["--output", c, "--gpus", "99"])
    # ADVICE r1: a checkpoint holding MORE samples than asked for must not be divided by the smaller count
    with pytest.raises(SystemExit) as e:
        cli.main(["--scene", "cornell-box", "--width", "64", "--seed", "3", "--samples", "8", "--output", c,
                  "--checkpoint", ck, "--resume"])
    assert "already holds 16" in str(e.value)
    # and a checkpoint made with another estimator is refused
    with pytest.raises(SystemExit):
        cli.main(base + ["--output", c, "--checkpoint", ck, "--resume", "--russian-roulette"])


def test_new_entry_points_edge_cases(yart, orc, ctx, mesh_scene):
    """Degenerate inputs through the round-2 entry points: weird f32 rays, zero-capacity dumps, argument errors."""
    _, ms, s = mesh_scene("cube")
    ctx.set_scene(ms.desc)
    weird = np.zeros(6, dtype=yart.abi.RAY_F32_DTYPE)
    weird["origin"] = [(0, 0, 0), (0, 0, 5), (np.nan, 0, 0), (0, 0, 5), (0, 0, 5), (0.25, 0.5, 5)]
    weird["direction"] = [(0, 0, 0), (0, 0, -np.inf), (0, 0, 1), (0, np.nan, -1), (0, 0, -1e-38), (0, 0, -1)]
    wide = orc.abi.make_rays(weird["origin"].astype(np.float64), weird["direction"].astype(np.float64))
    want, _ = s.closest_hit(wide, 0, 0.001, INF, 0)
    for order in (0, 1):
        got, _ = ctx.closest_hit_f32(weird, 0, 0.001, INF, order)
        assert np.array_equal(got["prim_id"], want["prim_id"])
        hit = want["prim_id"] != yart.MISS
        assert np.array_equal(got["t"][hit], want["t"][hit].astype(np.float32)) and hit[5]
    with pytest.raises(yart.YartError) as e:
        ctx.closest_hit_f32(weird, 9)                      # no such mesh
    assert e.value.code == -1
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    cam = preset.camera(32, 32)
    none, n = ctx.dump_path_rays(cam, 32, 32, 0, 2, 0)   # capacity 0: only the count comes back
    _, st = ctx.render(cam, 32, 32, 0, 2)
    assert len(none) == 0 and n == st.rays
    same, _ = ctx.render(cam, 32, 32, 0, 2, flags=1 << 20)  # unknown flag bits are ignored, not misread
    base, _ = ctx.render(cam, 32, 32, 0, 2)
    assert np.array_equal(same, base)
    film = ctx.film_create(32, 32)
    comm = yart.Comm.from_id(ctx, yart.comm_unique_id(), 0, 1)
    with pytest.raises(yart.YartError):
        comm.film_reduce([0], 32, 32, 0)                    # null film
    with pytest.raises(yart.YartError):
        comm.film_reduce(film, 0, 32, 0)                    # empty frame
    comm.close()
    ctx.film_destroy(film)
    with pytest.raises(yart.YartError):
        yart.Comm.from_id(ctx, yart.comm_unique_id(), 2, 2)  # rank out of range


def _rank_process(rank, world, id_path, out_path):
    """One process per GPU, no torch.distributed: the 128-byte NCCL id travels through a file."""
    import importlib
    import time
    sys.path.insert(0, str(ROOT))
    y = importlib.import_module("yet-another-raytracer_b200")
    sh = importlib.import_module("yet-another-raytracer_b200.sharding")
    ctx = y.Context(rank)
    if rank == 0:
        tmp = id_path + ".tmp"
        with open(tmp, "wb") as f:
            f.write(y.comm_unique_id())
        os.replace(tmp, id_path)
    else:
        for _ in range(600):
            if os.path.exists(id_path):
                break
            time.sleep(0.05)
    uid = open(id_path, "rb").read()
    comm = y.Comm.from_id(ctx, uid, rank, world)
    preset = y.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    w = h = 96
    cam = preset.camera(w, h)
    film = ctx.film_create(w, h)
    lo, hi = sh.shard_range(0, 9, rank, world)
    ctx.render_device(cam, w, h, lo, hi, film, seed=12)
    comm.film_reduce(film, w, h, root=0)
    if rank == 0:
        np.save(out_path, ctx.film_read(film, w, h))
    else:
        ctx.synchronize()
    comm.close()
    ctx.film_destroy(film)
    ctx.close()


def test_one_process_per_gpu_comm_from_id(yart, ctx, tmp_path):
    """The torchrun shape without torch: N processes, one GPU each, yart_comm_unique_id -> a file -> yart_comm_init_rank,
    sample-range shards, yart_film_reduce; rank 0's film equals the single-GPU film."""
    if yart.device_count() < 2:
        pytest.skip("one GPU visible: needs `gpurun --gpus 2` (the single-rank form of from_id is tested above)")
    import multiprocessing as mp
    world = 2
    id_path, out_path = str(tmp_path / "nccl_id.bin"), str(tmp_path / "film.npy")
    procs = [mp.get_context("spawn").Process(target=_rank_process, args=(r, world, id_path, out_path)) for r in range(world)]
    [p.start() for p in procs]
    [p.join(300) for p in procs]
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    preset = yart.ScenePreset("cornell-box", seed=1)
    ctx.set_scene(preset)
    want, _ = ctx.render(preset.camera(96, 96), 96, 96, 0, 9, seed=12)
    got = np.load(out_path)
    assert np.allclose(got, want, rtol=1e-13, atol=1e-13 * np.abs(want).max()) and got.sum() > 0


# ---------------------------------------------------------------------------------------------------------
# host-buffer queries run as a chunk pipeline (upload / kernels / download overlapped): same answers as one piece
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene", ["cornell-box-smoke", "david"])
def test_chunked_host_queries_equal_the_unchunked_ones(yart, ctx, scene, monkeypatch):
    preset = yart.ScenePreset(scene, seed=1)
    ctx.set_scene(preset)
    cam = preset.camera(320, 240)
    rays, _, _ = ctx.camera_rays(cam, 320, 240, 0, 3)          # 230,400 rays; the smoke scene draws random numbers per ray
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", str(1 << 30))
    whole, st_w = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR, count_visits=True)
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", "4099")           # 57 ragged chunks
    parts, st_p = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_NEAR, count_visits=True)
    assert whole.tobytes() == parts.tobytes()
    assert (st_p.rays, st_p.node_visits, st_p.tri_tests) == (st_w.rays, st_w.node_visits, st_w.tri_tests)
    assert st_p.kernel_launches > st_w.kernel_launches
    r32 = np.empty(len(rays), dtype=yart.abi.RAY_F32_DTYPE)
    r32["origin"], r32["direction"] = rays["origin"], rays["direction"]
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", str(1 << 30))
    whole32, _ = ctx.closest_hit_f32(r32, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE)
    monkeypatch.setenv("YART_TUNE_HOST_CHUNK", "70001")
    parts32, _ = ctx.closest_hit_f32(r32, yart.TARGET_WORLD, 0.001, INF, yart.ORDER_REFERENCE)
    assert whole32.tobytes() == parts32.tobytes()


def test_host_register_pins_caller_arrays(yart, ctx, mesh_scene):
    """yart_host_register / yart_host_unregister: a host that does not link CUDA page-locks its own arrays."""
    _, ms, _ = mesh_scene("cube")
    ctx.set_scene(ms.desc)
    rng = np.random.default_rng(2)
    rays = yart.make_rays(rng.uniform(-3, 3, size=(200000, 3)), rng.normal(size=(200000, 3)))
    hits = np.empty(len(rays), dtype=yart.HIT_DTYPE)
    want, _ = ctx.closest_hit(rays, 0, 0.001, INF, yart.ORDER_NEAR)
    ctx.host_register(rays)
    ctx.host_register(hits)
    try:
        got, _ = ctx.closest_hit(rays, 0, 0.001, INF, yart.ORDER_NEAR, hits=hits)
        assert got.tobytes() == want.tobytes()
        with pytest.raises(yart.YartError) as e:   # registering the same range twice is refused, not fatal
            ctx.host_register(rays)
        assert e.value.code == -1
    finally:
        ctx.host_unregister(hits)
        ctx.host_unregister(rays)
    with pytest.raises(yart.YartError):            # and so is unlocking what is not locked
        ctx.host_unregister(rays)
    got, _ = ctx.closest_hit(rays, 0, 0.001, INF, yart.ORDER_NEAR)  # the context is still usable
    assert got.tobytes() == want.tobytes()
