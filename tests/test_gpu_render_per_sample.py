"""Per-sample render parity: every (pixel, sample) the GPU renders against the same path of the CPU oracle (or of
tests/nee_ref.cpp with YART_FLAG_NEXT_EVENT), to 1e-9 of the pixel's largest channel.

Both sides draw the same Philox numbers and do the same f64 arithmetic in the same order, so the only legitimate
disagreement is a path that crosses a branch on a last-bit difference between CUDA's sin/cos/acos/atan2/log and
glibc's, or a path whose value amplifies such a difference.  tests/perturbed_oracle.py excuses a mismatch only when
a variant of the reference with its transcendentals moved by a few ulp also flips that sample, or moves it by at
least a tenth of the GPU's deviation, and the oracle's rays of that path get bit-identical closest hits on the GPU;
anything else fails and names the pixel, the sample and the path's object and material kinds.  Excused samples
are capped per case, and each sample range's ray count must match the reference's up to max_depth + 1 rays per
excused sample (and per 5,000 paths: a flip between two paths that both end at zero changes no pixel).

Measured on an NVIDIA B200 (1000 W power limit), mismatched / excused samples per case: david 64x64 at 4 spp, 1 / 1
in each traversal order; david 1920x1080 at 2 spp, 9 / 9 of 4,147,200 paths (one of them a 20-bounce path that lands
1.4e-9 away without a branch flip); the other 83 of the 86 gate runs 0 / 0.  The
file runs in about 20 s.  The caps are ten times the worst count: 10 excused samples per small case, 90 for the
full frame.
"""
import pytest

import perturbed_oracle as po
from scene_fuzz import FuzzScene

pytestmark = pytest.mark.gpu

ALL_PRESETS = ["cornell-box", "david", "bunny", "next-week-final", "cornell-box-smoke", "random-scene", "two-spheres",
               "two-perlin-spheres", "earth", "simple-light", "three-spheres", "sycee", "teapot"]


@pytest.fixture(scope="module", autouse=True)
def variants(orc):
    po.build_all()


def gate(yart, ctx, scene, cam, w, h, samples, depth, seed=7, flags=0, order=None, what="", cap=10):
    """Render each sample of `samples` on the GPU and check it against the reference, sample by sample."""
    order = yart.ORDER_NEAR if order is None else order
    ctx.set_scene(scene.desc if isinstance(scene, FuzzScene) else scene)

    def render(s):
        return ctx.render(cam, w, h, s, s + 1, max_depth=depth, seed=seed, order=order, flags=flags)

    def closest_hit(rays, o):
        return ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, float("inf"), o)[0]

    rep = po.per_sample_gate(scene, cam, w, h, samples, depth, seed, flags, order, render, closest_hit,
                             what=what or "order %d flags %d depth %d" % (order, flags, depth))
    print("PER-SAMPLE", rep.summary(), [(m["x"], m["y"], m["sample"], m["path"][:3]) for m in rep.mismatches][:4])
    rep.check(cap)
    return rep


@pytest.mark.parametrize("scene", ALL_PRESETS)
def test_presets(yart, ctx, scene):
    preset = yart.ScenePreset(scene, seed=2)
    w = h = 64 if scene in ("cornell-box", "david", "sycee", "teapot", "bunny") else 48
    orders = [yart.ORDER_NEAR] + ([yart.ORDER_REFERENCE] if scene in ("cornell-box", "david", "next-week-final") else [])
    for order in orders:
        gate(yart, ctx, preset, preset.camera(w, h), w, h, range(4), 50, order=order, what="%s order %d" % (scene, order))


@pytest.mark.parametrize("depth", [3, 1])
def test_short_paths(yart, ctx, depth):
    """Depth exhaustion returns 1.0 (main.rs:544-546) at depth 3; depth 1 is the camera ray's hit alone."""
    preset = yart.ScenePreset("david", seed=2)
    gate(yart, ctx, preset, preset.camera(48, 48), 48, 48, range(4), depth, what="david depth %d" % depth)


FLAG_SETS = {"unbiased-pick": 4, "roulette": 8, "depth-zero-black": 16, "all-three": 4 | 8 | 16}


@pytest.mark.parametrize("flag_set", list(FLAG_SETS))
@pytest.mark.parametrize("scene", ["cornell-box", "david"] + ["fuzz-%d" % s for s in range(8)])
def test_sampling_flags(yart, ctx, scene, flag_set):
    flags = FLAG_SETS[flag_set]
    if scene.startswith("fuzz"):
        sc = FuzzScene(yart, 3000 + int(scene[5:]))
        w, h, depth = 40, 32, 10
    else:
        sc = yart.ScenePreset(scene, seed=2)
        w, h, depth = 48, 48, 50
    gate(yart, ctx, sc, sc.camera(w, h), w, h, range(4), depth, flags=flags, what="%s %s" % (scene, flag_set))


@pytest.mark.parametrize("seed", range(20))
def test_fuzz_scenes(yart, ctx, seed):
    sc = FuzzScene(yart, 2000 + seed)
    gate(yart, ctx, sc, sc.camera(48, 32), 48, 32, range(4), 12, what="fuzz scene %d" % seed)


@pytest.mark.parametrize("scene", ["cornell-box", "david", "next-week-final"])
def test_next_event(yart, ctx, scene):
    preset = yart.ScenePreset(scene, seed=1)
    w = 48
    for flags in (yart.FLAG_NEXT_EVENT, yart.FLAG_NEXT_EVENT | yart.FLAG_RUSSIAN_ROULETTE | yart.FLAG_DEPTH_ZERO_BLACK):
        gate(yart, ctx, preset, preset.camera(w, w), w, w, range(4), 50, flags=flags, what="%s NEE flags %d" % (scene, flags))


def test_odd_frame_size(yart, ctx):
    """43x29: the reference renders 8x8 tiles of 5x3 pixels; every other pixel stays 0 on both sides."""
    preset = yart.ScenePreset("cornell-box", seed=2)
    gate(yart, ctx, preset, preset.camera(43, 29), 43, 29, range(4), 50, what="cornell-box 43x29")


def test_full_frame(yart, ctx):
    """david at 1920x1080, samples 0 and 1, depth 50: every one of the 4,147,200 paths."""
    preset = yart.ScenePreset("david", seed=2)
    gate(yart, ctx, preset, preset.camera(1920, 1080), 1920, 1080, range(2), 50, what="david 1920x1080", cap=90)
