"""yart_denoise on the GPU: bit parity with tests/denoise_ref.py, the RGBA8 display rule, host and device arrays,
argument errors, the render it leaves alone, the image quality it buys, both command lines and the memory a context
gives back."""
import ctypes as C
import importlib
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import denoise_ref

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
PLANES = ("albedo", "normal", "depth")

# relMSE (denoise_ref.rel_mse) bounds against a 4096-spp reference, set from tools/denoise_probe.py with margin
# (DESIGN section 6): denoised 16 spp <= DENOISED_OVER_NOISY x the noisy 16 spp; the denoised reference moves by
# <= OVERBLUR_OVER_NOISY x the noisy 16-spp error.
DENOISED_OVER_NOISY = 0.4
OVERBLUR_OVER_NOISY = 0.25


def synthetic(seed, h, w):
    """A film and planes as render_aovs could sum them, with extreme but finite magnitudes: 0..5 samples a pixel (0 =
    invalid), some of which hit; films spanning 1e-300..1e100 and exact zeros."""
    rng = np.random.default_rng(seed)
    samples = rng.integers(0, 6, (h, w)).astype(np.float64)
    hits = np.floor(samples * rng.uniform(0, 1.2, (h, w))).clip(0, samples)
    depth = np.stack([hits * rng.uniform(0.01, 1e3, (h, w)) * 10.0 ** rng.integers(-3, 4, (h, w)), hits, samples], axis=2)
    albedo = rng.uniform(0, 1, (h, w, 3)) * samples[..., None]
    normal = rng.normal(size=(h, w, 3))
    normal = normal / np.linalg.norm(normal, axis=2, keepdims=True) * samples[..., None]
    film = rng.uniform(-0.2, 1.0, (h, w, 3)) * 10.0 ** rng.integers(-300, 101, (h, w, 1))
    film[rng.uniform(size=(h, w)) < 0.1] = 0.0
    return film, {"albedo": albedo, "normal": normal, "depth": depth}


def check_parity(ctx, film, spp, planes, **kw):
    got = ctx.denoise(film, spp, planes, **kw)
    with np.errstate(over="ignore"):  # (f64 values past the f32 range round to inf on both sides)
        want = denoise_ref.denoise(film, spp, planes, **kw).astype(np.float32)
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), "%d of %d values differ, first at %s: %r vs %r" % (
        bad.sum(), bad.size, np.argwhere(bad)[0], got[bad][0], want[bad][0])
    return got


@pytest.mark.parametrize("h,w", [(1, 1), (5, 7), (37, 61), (3, 20), (20, 6)])
def test_synthetic_inputs_match_the_reference(yart, ctx, h, w):
    film, planes = synthetic(h * 100 + w, h, w)
    for levels in (0, 1, 3):
        check_parity(ctx, film, 3, planes, levels=levels)
    check_parity(ctx, film, 1, planes, sigma_color=3.0, sigma_normal=0.05, sigma_depth=0.7)


def test_every_level_count_matches_the_reference(yart, ctx):
    film, planes = synthetic(7, 40, 52)
    for levels in range(1, 11):
        check_parity(ctx, film, 5, planes, levels=levels)
        check_parity(ctx, film, 5, planes, levels=levels, sigma_color=1e3, sigma_normal=2.0, sigma_depth=1e-3)


PRESETS = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
           "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]


@pytest.mark.parametrize("name", PRESETS)
def test_presets_match_the_reference(yart, ctx, name):
    preset = yart.ScenePreset(name, seed=3)
    ctx.set_scene(preset)
    w, h, spp = 48, 32, 3
    cam = preset.camera(w, h)
    film, _ = ctx.render(cam, w, h, 0, spp, 50, 1)
    planes, _ = ctx.render_aovs(cam, w, h, 0, 2, 50, 1)
    got = check_parity(ctx, film, spp, planes)
    assert (got[planes["depth"][..., 2] > 0] != 0).any()


def test_preset_list_is_covered(yart):
    assert PRESETS == yart.SCENE_NAMES


def test_rgba8_is_the_display_rule_of_the_reference(yart, ctx):
    preset = yart.ScenePreset("cornell-box", seed=3)
    ctx.set_scene(preset)
    w, h = 64, 48
    cam = preset.camera(w, h)
    film, _ = ctx.render(cam, w, h, 0, 4, 50, 1)
    planes, _ = ctx.render_aovs(cam, w, h, 0, 4, 50, 1)
    for f, p in ((film, planes), synthetic(11, 29, 33)):
        hh, ww = f.shape[:2]
        rgb, rgba = ctx.denoise(f, 4, p, rgba=True)
        want, v = denoise_ref.display_rgba(denoise_ref.denoise(f, 4, p), p["depth"])
        near = np.zeros((hh, ww, 4), bool)
        near[..., :3] = np.abs(v - np.round(v)) < 1e-9  # CUDA's pow against numpy's may move such a byte by one
        assert (rgba[~near] == want[~near]).all()
        assert (np.abs(rgba.astype(int) - want)[near] <= 1).all()
        assert rgb.dtype == np.float32 and rgba.dtype == np.uint8 and rgba.shape == (hh, ww, 4)


def test_device_arrays_give_the_host_bits_and_inputs_stay(yart, ctx):
    film, planes = synthetic(3, 30, 41)
    h, w = film.shape[:2]
    copies = (film.copy(), {k: v.copy() for k, v in planes.items()})
    rgb, rgba = ctx.denoise(film, 2, planes, levels=4, rgba=True)
    assert (film == copies[0]).all() and all((planes[k] == copies[1][k]).all() for k in PLANES)
    import torch
    dev = {k: torch.from_numpy(np.ascontiguousarray(arr)).cuda() for k, arr in [("film", film)] + list(planes.items())}
    out = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    out8 = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ptrs = [dev[k].data_ptr() for k in PLANES]
    st = ctx.denoise_device(dev["film"].data_ptr(), 2, *ptrs, w, h, rgb_ptr=out.data_ptr(), rgba_ptr=out8.data_ptr(),
                            levels=4)
    assert (out.cpu().numpy() == rgb).all() and (out8.cpu().numpy() == rgba).all()
    assert st.kernel_launches == 4 + 2 and st.gpu_ms > 0
    assert (dev["film"].cpu().numpy() == film).all()
    assert all((dev[k].cpu().numpy() == planes[k]).all() for k in PLANES)
    only8 = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    ctx.denoise_device(dev["film"].data_ptr(), 2, *ptrs, w, h, rgba_ptr=only8.data_ptr(), levels=4)
    assert (only8.cpu().numpy() == rgba).all()
    with pytest.raises(yart.YartError) as e:  # a misaligned f64 array
        ctx.denoise_device(dev["film"].data_ptr() + 4, 2, *ptrs, w, h, rgb_ptr=out.data_ptr())
    assert e.value.code == yart.abi.YART_ERR_INVALID


def test_argument_errors(yart, ctx):
    film, planes = synthetic(5, 8, 8)
    lib = yart.load_library()
    arrs = {k: np.ascontiguousarray(v) for k, v in planes.items()}
    full = yart.abi.AovPlanes(arrs["albedo"].ctypes.data, arrs["normal"].ctypes.data, arrs["depth"].ctypes.data)
    rgb = np.zeros((8, 8, 3), np.float32)
    st = yart.abi.Stats()

    def call(film_p=film.ctypes.data, spp=1, ap=full, w=8, h=8, opts=None, out=rgb.ctypes.data, out8=None):
        return lib.yart_denoise(ctx._h, film_p, spp, None if ap is None else C.byref(ap), w, h,
                                None if opts is None else C.byref(opts), out, out8, C.byref(st))

    E = yart.abi.YART_ERR_INVALID
    assert call() == yart.abi.YART_OK and st.kernel_launches == 5 + 2
    assert (rgb == ctx.denoise(film, 1, planes)).all()  # NULL opts = the defaults
    assert lib.yart_denoise(None, film.ctypes.data, 1, C.byref(full), 8, 8, None, rgb.ctypes.data, None, None) == E
    assert call(film_p=None) == E
    assert call(spp=0) == E
    assert call(ap=None) == E
    for k in PLANES:
        part = yart.abi.AovPlanes(full.albedo, full.normal, full.depth)
        setattr(part, k, None)
        assert call(ap=part) == E, k
    assert call(out=None) == E
    assert call(w=0) == E and call(h=0) == E
    assert call(w=1 << 16, h=1 << 16) == E  # width * height >= 2^32
    for opts in (yart.abi.DenoiseOpts(11, 0, 0, 0, 0), yart.abi.DenoiseOpts(0, 2, 0, 0, 0),
                 yart.abi.DenoiseOpts(0, 64, 0, 0, 0), yart.abi.DenoiseOpts(0, 0, float("nan"), 0, 0),
                 yart.abi.DenoiseOpts(0, 0, 0, float("inf"), 0), yart.abi.DenoiseOpts(0, 0, 0, 0, -float("inf"))):
        assert call(opts=opts) == E, (opts.levels, opts.flags)
    assert call(opts=yart.abi.DenoiseOpts(10, 0, -1.0, 0.0, -5.0)) == yart.abi.YART_OK


def test_render_is_untouched_by_a_denoise_call(yart, ctx):
    preset = yart.ScenePreset("cornell-box-smoke", seed=3)
    ctx.set_scene(preset)
    w, h = 48, 32
    cam = preset.camera(w, h)
    plain, _ = ctx.render(cam, w, h, 0, 2, 50, 1)
    ctx.render(cam, w, h, 2, 4, 50, 1, film=plain)
    mixed, _ = ctx.render(cam, w, h, 0, 2, 50, 1)
    planes, _ = ctx.render_aovs(cam, w, h, 0, 2, seed=1)
    ctx.denoise(mixed, 2, planes, rgba=True)
    ctx.render(cam, w, h, 2, 4, 50, 1, film=mixed)
    assert (plain == mixed).all()


@pytest.mark.parametrize("scene,w,h", [("cornell-box", 300, 300), ("david", 480, 270)])
def test_denoising_16_spp_reduces_the_error(yart, ctx, scene, w, h):
    preset = yart.ScenePreset(scene)
    ctx.set_scene(preset)
    cam = preset.camera(w, h)
    depth = preset.info.max_depth
    ref_film, _ = ctx.render(cam, w, h, 0, 4096, depth, 100)
    ref = ctx.film_finalize_linear(ref_film, 4096)
    ref_planes, _ = ctx.render_aovs(cam, w, h, 0, 16, depth, 100)
    valid = ref_planes["depth"][..., 2] > 0
    blur = denoise_ref.rel_mse(ctx.denoise(ref_film, 4096, ref_planes), ref, valid)
    for seed in (1, 2, 3):
        film, _ = ctx.render(cam, w, h, 0, 16, depth, seed)
        planes, _ = ctx.render_aovs(cam, w, h, 0, 16, depth, seed)
        noisy = denoise_ref.rel_mse(ctx.film_finalize_linear(film, 16), ref, valid)
        den = denoise_ref.rel_mse(ctx.denoise(film, 16, planes), ref, valid)
        assert den <= DENOISED_OVER_NOISY * noisy, (seed, den, noisy)
        assert blur <= OVERBLUR_OVER_NOISY * noisy, (seed, blur, noisy)


def expected_denoised(yart, ctx, scene, w, h, spp, aov_spp, seed, max_depth):
    preset = yart.ScenePreset(scene, seed=seed)
    ctx.set_scene(preset)
    cam = preset.camera(w, h)
    film, _ = ctx.render(cam, w, h, 0, spp, max_depth, seed)
    planes, _ = ctx.render_aovs(cam, w, h, 0, aov_spp, max_depth, seed)
    return ctx.denoise(film, spp, planes, rgba=True)


def read_png(path):
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGBA"))


def test_python_cli_writes_the_context_denoise(yart, ctx, tmp_path):
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    args = ["--scene", "cornell-box", "--width", "64", "--height", "48", "--samples", "3", "--max-depth", "10"]
    plain = str(tmp_path / "plain.png")
    assert cli.main(args + ["--output", plain]) == 0
    out = str(tmp_path / "cb.png")
    assert cli.main(args + ["--denoise", "--aov-samples", "2", "--output", out]) == 0
    assert Path(plain).read_bytes() == Path(out).read_bytes()
    rgb, rgba = expected_denoised(yart, ctx, "cornell-box", 64, 48, 3, 2, 1, 10)
    paths = cli.denoised_paths(out)
    assert (cli.read_pfm(paths["pfm"]) == rgb).all()
    assert (read_png(paths["png"]) == rgba).all()


def test_native_host_writes_the_context_denoise(yart, ctx, assets, tmp_path):
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    exe = ROOT / "yet-another-raytracer_b200" / "yart"
    args = ["--scene", "david", "--width", "64", "--height", "48", "--samples", "20", "--max-depth", "8", "--assets", assets]
    plain, out = str(tmp_path / "plain.png"), str(tmp_path / "dv.png")
    for extra, path in (([], plain), (["--denoise"], out)):
        r = subprocess.run([str(exe)] + args + extra + ["--output", path], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
    assert Path(plain).read_bytes() == Path(out).read_bytes()
    rgb, rgba = expected_denoised(yart, ctx, "david", 64, 48, 20, 16, 1, 8)  # --aov-samples defaults to min(16, --samples)
    paths = cli.denoised_paths(out)
    assert (cli.read_pfm(paths["pfm"]) == rgb).all()
    assert (read_png(paths["png"]) == rgba).all()


def test_closing_a_context_frees_the_denoise_scratch(yart):
    """1920 x 1080 pixels hold about 250 MB of scratch and staging; five contexts, each closed after two calls, leave
    free memory where it was."""
    import torch
    film, planes = synthetic(9, 1080, 1920)

    def one(w, h):
        ctx = yart.Context(0)
        try:
            for _ in range(2):
                ctx.denoise(film[:h, :w], 2, {k: v[:h, :w] for k, v in planes.items()}, rgba=True)
        finally:
            ctx.close()

    one(16, 16)  # module loading and other once-per-process device allocations
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info(0)
    for _ in range(5):
        one(1920, 1080)
    free_after, _ = torch.cuda.mem_get_info(0)
    assert free_before - free_after < (64 << 20), "closed contexts kept %.0f MiB" % ((free_before - free_after) / (1 << 20))
