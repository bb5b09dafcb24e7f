"""YART_FLAG_NEXT_EVENT on the GPU: next-event estimation with MIS, against its CPU reference tests/nee_ref.cpp
(tests/test_next_event.py checks that reference against the CPU oracle), against the flag-off estimator it must agree with in
expectation, and against its own purpose: less noise at equal samples."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import nee_ref
from test_gpu_render import compare_films

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _setup(yart, orc, ctx, name):
    preset = yart.ScenePreset(name, seed=1)
    ctx.set_scene(preset)
    return preset, orc.Scene(preset)


@pytest.mark.parametrize("scene,w,spp,depth", [("cornell-box", 64, 8, 50), ("cornell-box", 64, 8, 4), ("david", 64, 8, 50),
                                               ("next-week-final", 48, 6, 50)])
def test_next_event_matches_the_cpu_reference(yart, orc, ctx, scene, w, spp, depth):
    """next-week-final has lights and constant media: its shadow rays draw their free paths from their own stream."""
    preset, _ = _setup(yart, orc, ctx, scene)
    s = nee_ref.Scene(preset)
    cam = preset.camera(w, w)
    for flags in (yart.FLAG_NEXT_EVENT, yart.FLAG_NEXT_EVENT | yart.FLAG_RUSSIAN_ROULETTE | yart.FLAG_DEPTH_ZERO_BLACK):
        want, st_w = s.render(cam, w, w, 0, spp, max_depth=depth, seed=3, n_threads=os.cpu_count(), flags=flags)
        for order in (yart.ORDER_NEAR, yart.ORDER_REFERENCE):
            got, st = ctx.render(cam, w, w, 0, spp, max_depth=depth, seed=3, order=order, flags=flags)
            compare_films(got, want, "%s depth %d flags %d order %d" % (scene, depth, flags, order), 0.97)
            assert abs(int(st.rays) - int(st_w.rays)) <= max(4, st_w.rays // 500)


def test_path_rays_and_counts_are_those_of_the_unbiased_pick(yart, orc, ctx):
    preset, _ = _setup(yart, orc, ctx, "cornell-box")
    w = h = 48
    cam = preset.camera(w, h)
    ub = yart.FLAG_UNBIASED_LIGHT_PICK
    a, n_a = ctx.dump_path_rays(cam, w, h, 0, 2, 1 << 20, seed=5, flags=ub)
    b, n_b = ctx.dump_path_rays(cam, w, h, 0, 2, 1 << 20, seed=5, flags=ub | yart.FLAG_NEXT_EVENT)
    assert n_a == n_b and len(a) == n_a
    # (within a bounce the order is the queue's, which warp-aggregated atomics decide: compare as sets)
    key = lambda r: np.lexsort(np.concatenate([r["origin"], r["direction"]], axis=1).T)  # noqa: E731
    assert np.array_equal(a[key(a)], b[key(b)])
    fa, st_a = ctx.render(cam, w, h, 0, 4, seed=5, flags=ub)
    fb, st_b = ctx.render(cam, w, h, 0, 4, seed=5, flags=ub | yart.FLAG_NEXT_EVENT)
    fc, st_c = ctx.render(cam, w, h, 0, 4, seed=5, flags=yart.FLAG_NEXT_EVENT)
    assert st_a.rays == st_b.rays == st_c.rays and st_a.paths == st_b.paths
    assert np.array_equal(fb, fc)  # NEXT_EVENT implies the unbiased pick
    assert not np.array_equal(fa, fb)
    assert st_b.trace_launches > st_a.trace_launches  # the shadow passes are closest-hit launches too


def _chunk_means(ctx, cam, w, h, spp, chunks, flags, seed):
    """(chunks, H, W) per-pixel mean Y of `chunks` independent sample ranges of spp samples each."""
    out = []
    for k in range(chunks):
        f, _ = ctx.render(cam, w, h, k * spp, (k + 1) * spp, seed=seed, flags=flags)
        out.append(f[..., 1] / spp)
    return np.stack(out)


@pytest.mark.parametrize("scene", ["cornell-box", "david", "teapot"])
def test_converges_to_the_flag_off_image(yart, orc, ctx, scene):
    """Frame and quadrant luminance agree with the flag-off unbiased render within 4 sigma, sigma from the variance
    of independent sample batches per pixel (pixels are independent)."""
    preset, _ = _setup(yart, orc, ctx, scene)
    w = h = 96
    cam = preset.camera(w, h)
    a = _chunk_means(ctx, cam, w, h, 64, 24, yart.FLAG_UNBIASED_LIGHT_PICK, 11)
    b = _chunk_means(ctx, cam, w, h, 64, 24, yart.FLAG_NEXT_EVENT, 11)
    regions = {"frame": (slice(0, h), slice(0, w))}
    for i in range(2):
        for j in range(2):
            regions["q%d%d" % (i, j)] = (slice(i * h // 2, (i + 1) * h // 2), slice(j * w // 2, (j + 1) * w // 2))
    for k, (r, c) in regions.items():
        sa, sb = a[:, r, c].sum(axis=(1, 2)), b[:, r, c].sum(axis=(1, 2))
        sd = np.sqrt(sa.var(ddof=1) / len(sa) + sb.var(ddof=1) / len(sb))
        print(scene, k, sa.mean(), sb.mean(), sd)
        assert abs(sa.mean() - sb.mean()) <= 4.0 * sd, (scene, k, sa.mean(), sb.mean(), sd)


# relMSE(NEE) / relMSE(flag off) on cornell-box 96x96 at 64 spp, seeds 1-3: 0.970 on the first B200 measurement
# (NVIDIA B200, 1000 W power limit).  The mixture already sends half the diffuse rays toward the lights, so the gain is
# small (DESIGN.md section 6); the bound keeps a margin of two points.
CORNELL_RELMSE_RATIO_MAX = 0.99


def test_next_event_has_lower_error_at_equal_samples(yart, orc, ctx):
    preset, _ = _setup(yart, orc, ctx, "cornell-box")
    w = h = 96
    cam = preset.camera(w, h)
    ref, _ = ctx.render(cam, w, h, 0, 8192, seed=1000, flags=yart.FLAG_UNBIASED_LIGHT_PICK)
    ref = ref[..., 1] / 8192
    denom = (ref ** 2).mean()

    def relmse(flags, seed):
        f, _ = ctx.render(cam, w, h, 0, 64, seed=seed, flags=flags)
        return float(((f[..., 1] / 64 - ref) ** 2).mean() / denom)

    off = [relmse(yart.FLAG_UNBIASED_LIGHT_PICK, s) for s in (1, 2, 3)]
    on = [relmse(yart.FLAG_NEXT_EVENT, s) for s in (1, 2, 3)]
    ratio = np.mean(on) / np.mean(off)
    print("relMSE off", off, "on", on, "ratio", ratio)
    assert ratio < CORNELL_RELMSE_RATIO_MAX


def test_small_state_budget_gives_the_same_film(yart, orc, ctx, tmp_path):
    """Pixel-chunked batches (a 2 MB state budget, YART_TUNE_STATE_MB, read once per process) render the same NEE
    film: the light-sample sums and shadow queues are per batch."""
    preset, _ = _setup(yart, orc, ctx, "cornell-box")
    want, st = ctx.render(preset.camera(96, 96), 96, 96, 0, 5, seed=6, flags=yart.FLAG_NEXT_EVENT)
    code = ("import importlib, sys, numpy as np\nsys.path.insert(0, %r)\n"
            "y = importlib.import_module('yet-another-raytracer_b200')\np = y.ScenePreset('cornell-box', seed=1)\n"
            "c = y.Context(0); c.set_scene(p)\nf, st = c.render(p.camera(96, 96), 96, 96, 0, 5, seed=6, flags=y.FLAG_NEXT_EVENT)\n"
            "np.save(%r, f); print('launches', st.kernel_launches)\n") % (str(ROOT), str(tmp_path / "f.npy"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, YART_TUNE_STATE_MB="2"), capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert np.array_equal(np.load(tmp_path / "f.npy"), want)
    assert int(out.stdout.split("launches")[1]) > st.kernel_launches


def test_flag_off_render_after_a_next_event_render_is_unchanged(yart, orc, ctx):
    preset, _ = _setup(yart, orc, ctx, "david")
    cam = preset.camera(64, 64)
    a, st_a = ctx.render(cam, 64, 64, 0, 4, seed=2)
    ctx.render(cam, 64, 64, 0, 4, seed=2, flags=yart.FLAG_NEXT_EVENT)
    b, st_b = ctx.render(cam, 64, 64, 0, 4, seed=2)
    assert np.array_equal(a, b) and st_a.rays == st_b.rays and st_a.kernel_launches == st_b.kernel_launches
