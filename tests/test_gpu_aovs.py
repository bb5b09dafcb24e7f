"""yart_render_aovs and yart_film_finalize_linear on the GPU.

Every plane of every (pixel, sample) must equal the CPU reference (tests/aov_ref.cpp) bit for bit, except where a
libm-perturbed build of that reference (tests/perturbed_oracle.py's variants) also changes it: sphere u, v feeding an
image texel, a checker's sin, marble noise, a medium's log.  On media-free scenes the planes must also follow, in
numpy, from yart_closest_hit_records on yart_generate_camera_rays' rays with their times."""
import ctypes as C
import importlib
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import aov_ref
import perturbed_oracle
from scene_fuzz import FuzzScene

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
SEED = 9
PRESETS = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
           "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]
MEDIA = ("cornell-box-smoke", "next-week-final")
PLANES = aov_ref.PLANES


def same(a, b):
    return (a == b) | ((a != a) & (b != b))


def differs(p, q):
    """(h, w) mask of pixels where any plane of p differs from q's."""
    return np.any([~same(p[k], q[k]).all(axis=2) for k in PLANES], axis=0)


def check_parity(ctx, scene, w, h, ns, what):
    """Sample by sample, both orders: GPU == reference except where a libm variant of the reference moves the sample.
    Returns the number of excused (pixel, sample)s."""
    ctx.set_scene(scene.desc)
    cam = scene.camera(w, h)
    base = aov_ref.Scene(scene)
    variants = None
    excused = 0
    for order in (0, 1):
        whole = {k: np.zeros((h, w, 3)) for k in PLANES}
        for s in range(ns):
            got, st = ctx.render_aovs(cam, w, h, s, s + 1, seed=SEED, order=order)
            want = base.planes(cam, w, h, s, s + 1, seed=SEED, order=order)
            bad = differs(got, want)
            if bad.any():
                if variants is None:
                    variants = [aov_ref.Scene(scene, d) for d in perturbed_oracle.VARIANTS.values()]
                sensitive = np.zeros((h, w), bool)
                for v in variants:
                    sensitive |= differs(v.planes(cam, w, h, s, s + 1, seed=SEED, order=order), want)
                left = bad & ~sensitive
                if left.any():
                    y, x = np.argwhere(left)[0]
                    raise AssertionError("%s order %d: (pixel %d,%d, sample %d) unexcused: %d of %d mismatches; gpu %r ref %r" % (
                        what, order, x, y, s, left.sum(), bad.sum(), {k: got[k][y, x] for k in PLANES},
                        {k: want[k][y, x] for k in PLANES}))
                excused += int(bad.sum())
            for k in PLANES:
                whole[k] += got[k]
        # one call over all samples adds them in the same order as the per-sample calls above
        got, st = ctx.render_aovs(cam, w, h, 0, ns, seed=SEED, order=order)
        assert not differs(got, whole).any(), what
        n_rendered = int((got["depth"][..., 2] > 0).sum())
        assert st.paths == st.rays == n_rendered * ns and st.max_bounce == 1 and st.trace_launches >= 1
    return excused


@pytest.mark.parametrize("name", PRESETS)
def test_presets_match_the_reference(yart, ctx, name):
    preset = yart.ScenePreset(name, seed=3)
    n = check_parity(ctx, preset, 48, 32, 4, name)
    print("%s: %d excused (pixel, sample)s" % (name, n))


@pytest.mark.parametrize("seed", range(20))
def test_fuzz_worlds_match_the_reference(yart, ctx, seed):
    """Random worlds: wrappers, groups, media, moving spheres, image / checker / noise textures."""
    sc = FuzzScene(yart, 7000 + seed)
    check_parity(ctx, sc, 40, 24, 3, "fuzz %d" % seed)


@pytest.mark.parametrize("name", [p for p in PRESETS if p not in MEDIA])
def test_per_sample_planes_follow_from_the_closest_hit_records(yart, ctx, name):
    """1-spp calls against yart_closest_hit_records on the camera rays with their times: normal and distance exactly."""
    preset = yart.ScenePreset(name, seed=3)
    ctx.set_scene(preset)
    w, h = 48, 32
    cam = preset.camera(w, h)
    tiles = np.outer(perturbed_oracle.covered(h), perturbed_oracle.covered(w))
    for order in (0, 1):
        for s in (0, 3):
            got, _ = ctx.render_aovs(cam, w, h, s, s + 1, seed=SEED, order=order)
            rays, _, times = ctx.camera_rays(cam, w, h, s, s + 1, seed=SEED)
            rec, _ = ctx.closest_hit_records(rays, times, yart.TARGET_WORLD, 0.001, float("inf"), order)
            normal, depth = aov_ref.normal_depth_from_records(rec, rays)
            normal, depth = normal.reshape(h, w, 3), depth.reshape(h, w, 3)
            assert (got["normal"][tiles] == normal[tiles]).all(), (name, order, s)
            assert (got["depth"][tiles] == depth[tiles]).all(), (name, order, s)
            for k in PLANES:
                assert (got[k][~tiles] == 0).all()


def test_david_light_spheres_are_in_the_planes(yart, ctx):
    """The spheres after david's meshes are left to k_shade by yart_render; the AOV passes must trace them."""
    preset = yart.ScenePreset("david", seed=3)
    sd = preset.desc.contents
    lights = [i for i in range(sd.n_objects) if sd.objects[i].kind == yart.abi.OBJ_SPHERE]
    assert lights and lights[-1] == sd.n_objects - 1
    ctx.set_scene(preset)
    w, h = 32, 32
    ref = aov_ref.Scene(preset)
    for i in lights:
        cam = preset.camera(w, h, vfov=2.0)
        cam.lookat[:] = list(sd.objects[i].p[:3])
        got, _ = ctx.render_aovs(cam, w, h, 0, 2, seed=SEED)
        samples = ref.samples(cam, w, h, 0, 2, seed=SEED)
        tiles = np.outer(perturbed_oracle.covered(h), perturbed_oracle.covered(w))
        on = np.isin(samples["rec"]["obj_id"], lights).all(axis=2) & tiles  # (two of them coincide)
        assert on.sum() > 0.5 * tiles.sum(), i
        assert (got["albedo"][on] > 0).all() and (got["depth"][on][:, 1] == 2).all()
        assert not differs(got, ref.planes(cam, w, h, 0, 2, seed=SEED)).any(), i


def test_chained_ranges_and_batch_sizes_give_the_same_bits(yart, ctx):
    preset = yart.ScenePreset("cornell-box-smoke", seed=3)
    ctx.set_scene(preset)
    w, h, ns = 64, 48, 7
    cam = preset.camera(w, h)
    one, _ = ctx.render_aovs(cam, w, h, 0, ns, seed=SEED)
    for batch in (1, 2, 3, 7):
        got, _ = ctx.render_aovs(cam, w, h, 0, ns, seed=SEED, batch_spp=batch)
        assert not differs(got, one).any(), batch
    chained, _ = ctx.render_aovs(cam, w, h, 0, 2, seed=SEED)
    ctx.render_aovs(cam, w, h, 2, 5, seed=SEED, planes=chained, batch_spp=2)
    ctx.render_aovs(cam, w, h, 5, ns, seed=SEED, planes=chained)
    assert not differs(chained, one).any()
    # sampling flags change nothing, and the beauty call's max_depth is accepted
    flags = yart.FLAG_UNBIASED_LIGHT_PICK | yart.FLAG_RUSSIAN_ROULETTE | yart.FLAG_DEPTH_ZERO_BLACK | yart.FLAG_NEXT_EVENT
    got, _ = ctx.render_aovs(cam, w, h, 0, ns, max_depth=3, seed=SEED, flags=flags)
    assert not differs(got, one).any()
    # null planes are skipped, the others unchanged
    for k in PLANES:
        only, _ = ctx.render_aovs(cam, w, h, 0, ns, seed=SEED, planes={k: np.zeros((h, w, 3))})
        assert list(only) == [k] and (only[k] == one[k]).all(), k


def test_device_planes_equal_host_planes(yart, ctx):
    preset = yart.ScenePreset("next-week-final", seed=3)
    ctx.set_scene(preset)
    w, h = 48, 32
    cam = preset.camera(w, h)
    host, _ = ctx.render_aovs(cam, w, h, 0, 3, seed=SEED)
    ptr = {k: ctx.film_create(w, h) for k in PLANES}
    try:
        ctx.render_aovs_device(cam, w, h, 0, 1, ptr["albedo"], ptr["normal"], ptr["depth"], seed=SEED)
        ctx.render_aovs_device(cam, w, h, 1, 3, ptr["albedo"], ptr["normal"], ptr["depth"], seed=SEED)
        for k in PLANES:
            assert (ctx.film_read(ptr[k], w, h) == host[k]).all(), k
        ctx.film_clear(ptr["depth"], w, h)
        ctx.render_aovs_device(cam, w, h, 0, 3, depth_ptr=ptr["depth"], seed=SEED)  # albedo, normal null
        assert (ctx.film_read(ptr["depth"], w, h) == host["depth"]).all()
        with pytest.raises(yart.YartError) as e:
            ctx.render_aovs_device(cam, w, h, 0, 1, depth_ptr=ptr["depth"] + 4, seed=SEED)  # misaligned
        assert e.value.code == yart.abi.YART_ERR_INVALID
    finally:
        for p in ptr.values():
            ctx.film_destroy(p)


def test_argument_errors(yart, ctx):
    preset = yart.ScenePreset("cornell-box", seed=3)
    ctx.set_scene(preset)
    cam = preset.camera(16, 16)
    lib = yart.load_library()
    o = ctx._opts(16, 16, 0, 1, 50, 1, 0, 0, 0)
    st = yart.abi.Stats()
    assert lib.yart_render_aovs(ctx._h, C.byref(cam), C.byref(o), C.byref(yart.abi.AovPlanes()), C.byref(st)) == yart.abi.YART_ERR_INVALID
    assert lib.yart_render_aovs(ctx._h, C.byref(cam), C.byref(o), None, None) == yart.abi.YART_ERR_INVALID
    buf = np.zeros((16, 16, 3))
    planes = yart.abi.AovPlanes(None, None, buf.ctypes.data)
    for field, value in (("max_depth", 0), ("width", 1), ("sample_end", 0)):
        bad = ctx._opts(16, 16, 1, 2, 50, 1, 0, 0, 0)
        setattr(bad, field, value)
        assert lib.yart_render_aovs(ctx._h, C.byref(cam), C.byref(bad), C.byref(planes), None) == yart.abi.YART_ERR_INVALID, field
    assert lib.yart_render_aovs(ctx._h, C.byref(cam), C.byref(o), C.byref(planes), None) == yart.abi.YART_OK
    assert buf[..., 2].max() == 1
    empty = ctx._opts(16, 16, 3, 3, 50, 1, 0, 0, 0)
    assert lib.yart_render_aovs(ctx._h, C.byref(cam), C.byref(empty), C.byref(planes), C.byref(st)) == yart.abi.YART_OK
    assert buf[..., 2].max() == 1 and st.rays == 0
    rgb = np.zeros((16, 16, 3), np.float32)
    assert lib.yart_film_finalize_linear(ctx._h, None, 16, 16, 1, 0, rgb.ctypes.data) == yart.abi.YART_ERR_INVALID
    assert lib.yart_film_finalize_linear(ctx._h, buf.ctypes.data, 16, 16, 0, 0, rgb.ctypes.data) == yart.abi.YART_ERR_INVALID


def test_render_is_untouched_by_an_aov_call(yart, ctx):
    preset = yart.ScenePreset("cornell-box-smoke", seed=3)
    ctx.set_scene(preset)
    w, h = 48, 32
    cam = preset.camera(w, h)
    plain, _ = ctx.render(cam, w, h, 0, 2, 50, SEED)
    ctx.render(cam, w, h, 2, 4, 50, SEED, film=plain)
    mixed, _ = ctx.render(cam, w, h, 0, 2, 50, SEED)
    ctx.render_aovs(cam, w, h, 0, 4, seed=SEED)
    ctx.render(cam, w, h, 2, 4, 50, SEED, film=mixed)
    assert (plain == mixed).all()


def linear_numpy(film, spp):
    mul, den = 720.0 - 360.0, 106.856895 * float(spp)
    c = [film[..., k] * mul / den for k in range(3)]
    r = 2.6896552 * c[0] - 1.2758621 * c[1] - 0.4137931 * c[2]
    g = -1.0221082 * c[0] + 1.9782866 * c[1] + 0.0438216 * c[2]
    b = 0.0612245 * c[0] - 0.2244898 * c[1] + 1.1632653 * c[2]
    h, w = film.shape[:2]
    tiles = np.outer(perturbed_oracle.covered(h), perturbed_oracle.covered(w))
    return np.where(tiles[..., None], np.stack([r, g, b], axis=2), 0.0).astype(np.float32)


def test_film_finalize_linear_is_the_numpy_expression(yart, ctx):
    preset = yart.ScenePreset("cornell-box", seed=3)
    ctx.set_scene(preset)
    w, h = 64, 40
    film, _ = ctx.render(preset.camera(w, h), w, h, 0, 3, 50, SEED)
    film[0, 0] = [1e300, -1e300, np.nan]  # (outside the tiles: 0 whatever the film holds)
    film[h // 2, w // 2] = [-5.0, 1e-310, 7.0]
    for spp in (1, 3, 1000):
        got = ctx.film_finalize_linear(film, spp)
        assert got.dtype == np.float32 and got.shape == (h, w, 3)
        assert same(got, linear_numpy(film, spp)).all(), spp
    d_film, d_out = ctx.film_create(w, h), ctx.film_create(w, h)  # (the f32 image fits in a film's bytes)
    try:
        ctx.render_device(preset.camera(w, h), w, h, 0, 3, d_film, 50, SEED)
        film = ctx.film_read(d_film, w, h)
        lib = yart.load_library()
        assert lib.yart_film_finalize_linear(ctx._h, C.c_void_p(d_film), w, h, 3, yart.FLAG_DEVICE_PTRS,
                                             C.c_void_p(d_out)) == 0
        got = ctx.film_read(d_out, w, h).view(np.float32).reshape(-1)[:h * w * 3].reshape(h, w, 3)
        assert (got == linear_numpy(film, 3)).all()
    finally:
        ctx.film_destroy(d_film)
        ctx.film_destroy(d_out)


def expected_files(yart, ctx, scene, w, h, spp, aov_spp, seed, max_depth):
    preset = yart.ScenePreset(scene, seed=seed)
    ctx.set_scene(preset)
    cam = preset.camera(w, h)
    film, _ = ctx.render(cam, w, h, 0, spp, max_depth, seed)
    planes, _ = ctx.render_aovs(cam, w, h, 0, aov_spp, max_depth, seed)
    m = yart.aov_means(planes)
    return {"color": ctx.film_finalize_linear(film, spp), "albedo": m["albedo"].astype(np.float32),
            "normal": m["normal"].astype(np.float32), "depth": m["depth"].astype(np.float32)}


def test_python_cli_writes_the_context_aovs(yart, ctx, tmp_path):
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    out = str(tmp_path / "cb.png")
    assert cli.main(["--scene", "cornell-box", "--width", "64", "--height", "48", "--samples", "3", "--max-depth", "10",
                     "--aovs", "--aov-samples", "2", "--output", out]) == 0
    want = expected_files(yart, ctx, "cornell-box", 64, 48, 3, 2, 1, 10)
    paths = cli.aov_paths(out)
    assert os.path.exists(out)
    for k, img in want.items():
        assert (cli.read_pfm(paths[k]) == img).all(), k
    assert (want["depth"] > 0).any() and (want["albedo"] > 0).any()


def test_native_host_writes_the_context_aovs(yart, ctx, assets, tmp_path):
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    exe = ROOT / "yet-another-raytracer_b200" / "yart"
    out = str(tmp_path / "dv.png")
    r = subprocess.run([str(exe), "--scene", "david", "--width", "64", "--height", "48", "--samples", "20", "--max-depth", "8",
                        "--aovs", "--output", out, "--assets", assets], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    want = expected_files(yart, ctx, "david", 64, 48, 20, 16, 1, 8)  # --aov-samples defaults to min(16, --samples)
    paths = cli.aov_paths(out)
    for k, img in want.items():
        assert (cli.read_pfm(paths[k]) == img).all(), k
