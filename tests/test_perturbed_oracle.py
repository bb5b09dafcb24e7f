"""The excuse mechanism of the per-sample render gate (tests/perturbed_oracle.py), on the CPU alone: the libm
perturbation hook changes nothing when it moves nothing, each perturbation changes some samples (so check (a) is not
vacuous), a libm the gate never saw is excused wherever it changes a sample (recall), and a small error in one
sample is not (precision)."""
import os

import numpy as np
import pytest

import perturbed_oracle as po
from scene_fuzz import FuzzScene

abi = po.abi
ALL_PRESETS = ["cornell-box", "david", "bunny", "next-week-final", "cornell-box-smoke", "random-scene", "two-spheres",
               "two-perlin-spheres", "earth", "simple-light", "three-spheres", "sycee", "teapot"]


@pytest.fixture(scope="module", autouse=True)
def variants(orc):
    po.build_all()


def _render(L, scene, cam, w, h, s0, s1, depth, flags=0, order=abi.ORDER_REFERENCE):
    return po.orc.Scene(scene, L).render(cam, w, h, s0, s1, max_depth=depth, seed=3, order=order,
                                          n_threads=os.cpu_count(), flags=flags)


@pytest.mark.parametrize("scene", ["cornell-box", "earth", "next-week-final", "two-perlin-spheres"])
def test_identity_hook_is_bit_exact(yart, orc, scene):
    preset = yart.ScenePreset(scene, seed=2)
    cam = preset.camera(32, 32)
    want, st_w = _render(orc.lib(), preset, cam, 32, 32, 0, 3, 50)
    got, st = _render(po.variant_lib("oracle", po.IDENTITY), preset, cam, 32, 32, 0, 3, 50)
    assert got.tobytes() == want.tobytes() and st.rays == st_w.rays
    s = orc.Scene(preset)
    for p in (0, 33, 500):
        a = s.sample(cam, 32, 32, p, 1, max_depth=50, seed=3)
        b = po.orc.Scene(preset, po.variant_lib("oracle", po.IDENTITY)).sample(cam, 32, 32, p, 1, max_depth=50, seed=3)
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1]
    nee = po.nee_ref.Scene(preset).render(cam, 32, 32, 0, 2, max_depth=20, seed=3, n_threads=os.cpu_count())[0]
    nee_id = po.nee_ref.Scene(preset, po.variant_lib("nee", po.IDENTITY)).render(
        cam, 32, 32, 0, 2, max_depth=20, seed=3, n_threads=os.cpu_count())[0]
    assert nee.tobytes() == nee_id.tobytes()


@pytest.mark.parametrize("name", list(po.VARIANTS))
def test_each_perturbation_changes_samples(yart, orc, name):
    """Every variant moves pixel values on each libm-heavy scene (image texture through acos/atan2, Perlin marble
    through sin, media through log), and flips a david sample past the gate's tolerance (a cosine-sampling branch:
    about one sample in 70,000 flips)."""
    lib = po.variant_lib("oracle", po.VARIANTS[name])
    for scene in ("earth", "two-perlin-spheres", "next-week-final"):
        preset = yart.ScenePreset(scene, seed=2)
        cam = preset.camera(48, 48)
        want, _ = _render(orc.lib(), preset, cam, 48, 48, 0, 4, 50)
        got, _ = _render(lib, preset, cam, 48, 48, 0, 4, 50)
        assert (got != want).any(axis=-1).sum() > 100, (name, scene)
    preset = yart.ScenePreset("david", seed=2)
    cam = preset.camera(96, 96)
    want, _ = _render(orc.lib(), preset, cam, 96, 96, 0, 8, 50)
    got, _ = _render(lib, preset, cam, 96, 96, 0, 8, 50)
    assert po.mismatched(got, want).any(), name


def _recall(scene, cam, w, h, samples, depth, flags=0, order=abi.ORDER_REFERENCE, what=""):
    held = po.orc.Scene(scene, po.variant_lib("oracle", po.HELD_OUT))
    held_nee = po.nee_ref.Scene(scene, po.variant_lib("nee", po.HELD_OUT)) if flags & abi.FLAG_NEXT_EVENT else None
    replay = po.orc.Scene(scene)

    def render(s):
        side = held_nee or held
        return side.render(cam, w, h, s, s + 1, max_depth=depth, seed=3, order=order, n_threads=os.cpu_count(),
                           flags=flags)

    rep = po.per_sample_gate(scene, cam, w, h, samples, depth, 3, flags, order, render,
                             lambda rays, o: replay.closest_hit(rays, order=o)[0], what=what)
    rep.check(cap=10 ** 9)  # (the recall tests bound nothing: each excused sample is what they look for)
    return rep


@pytest.mark.parametrize("scene", ALL_PRESETS)
def test_recall_on_presets(yart, orc, scene):
    """A held-out seeded libm stands in for the GPU: every sample it changes must be excused by the other variants."""
    preset = yart.ScenePreset(scene, seed=2)
    cam = preset.camera(40, 40)
    rep = _recall(preset, cam, 40, 40, range(4), 50, what=scene)
    print(rep.summary())


@pytest.mark.parametrize("scene", ["david", "next-week-final"])
def test_recall_where_the_held_out_libm_flips_a_sample(yart, orc, scene):
    """Frames where the held-out variant does flip samples past the tolerance: they are found and excused."""
    preset = yart.ScenePreset(scene, seed=2)
    cam = preset.camera(96, 96)
    rep = _recall(preset, cam, 96, 96, range(8), 50, what=scene)
    assert len(rep.mismatches) >= 1, rep.summary()


@pytest.mark.parametrize("seed", range(6))
def test_recall_on_fuzz_scenes(yart, orc, seed):
    sc = FuzzScene(yart, 2000 + seed)
    cam = sc.camera(40, 32)
    flags = abi.FLAG_UNBIASED_LIGHT_PICK | abi.FLAG_RUSSIAN_ROULETTE if seed % 2 else 0
    print(_recall(sc, cam, 40, 32, range(3), 12, flags=flags, what="fuzz %d" % seed).summary())


@pytest.mark.parametrize("scene", ["cornell-box", "next-week-final"])
def test_recall_with_next_event(yart, orc, scene):
    preset = yart.ScenePreset(scene, seed=1)
    cam = preset.camera(32, 32)
    print(_recall(preset, cam, 32, 32, range(3), 50, flags=abi.FLAG_NEXT_EVENT, what=scene).summary())


def test_precision_a_small_error_on_a_glass_path_is_not_excused(yart, orc):
    """Scale one sample of a pixel whose path goes through glass by (1 + 1e-6) in an otherwise exact film: the gate
    names it, as a dielectric path, and excuses nothing."""
    preset = yart.ScenePreset("three-spheres", seed=2)
    w = h = 32
    cam = preset.camera(w, h)
    s = orc.Scene(preset)
    sd = preset.desc.contents
    mask = po.covered(h)[:, None] & po.covered(w)[None, :]
    target = None
    for p in np.flatnonzero(mask.ravel()):
        if not s.sample(cam, w, h, int(p), 1, max_depth=50, seed=3)[0].any():
            continue
        hits, _ = s.closest_hit(s.sample_path(cam, w, h, int(p), 1, max_depth=50, seed=3))
        path = [po.describe_hit(sd, hh) for hh in hits]
        if any("dielectric" in d for d in path):
            target = (int(p) // w, int(p) % w)
            break
    assert target is not None

    def render(smp):
        film, st = s.render(cam, w, h, smp, smp + 1, max_depth=50, seed=3, n_threads=os.cpu_count())
        if smp == 1:
            film[target] *= 1.0 + 1e-6
        return film, st

    rep = po.per_sample_gate(preset, cam, w, h, range(3), 50, 3, 0, abi.ORDER_REFERENCE, render,
                             lambda rays, o: s.closest_hit(rays, order=o)[0], what="precision")
    assert [(m["y"], m["x"], m["sample"]) for m in rep.mismatches] == [target + (1,)]
    assert not rep.mismatches[0]["excused"] and rep.mismatches[0]["clean"]
    assert any("dielectric" in d for d in rep.mismatches[0]["path"])
    with pytest.raises(AssertionError, match="dielectric"):
        rep.check(cap=0)


def test_a_libm_amplifying_path_is_excused_in_proportion(yart, orc):
    """A sample the B200 rendered 1.44e-9 away from the oracle (NVIDIA B200, david 1920x1080, seed 7, near-first
    order, pixel (873, 730), sample 1): 20 bounces, no branch differs, and the perturbed variants move it by
    1.1e-10 to 9.4e-10.  It is excused; the same pixel 1e-7 away, a hundred times what the variants show, is not."""
    preset = yart.ScenePreset("david", seed=2)
    w, h = 1920, 1080
    cam = preset.camera(w, h)
    s = orc.Scene(preset)
    judge = po.Judge(preset, cam, w, h, 50, 7, 0, abi.ORDER_NEAR, lambda rays, o: s.closest_hit(rays, order=o)[0])
    want = po.sanitized(s.sample(cam, w, h, 730 * w + 873, 1, max_depth=50, seed=7, order=abi.ORDER_NEAR)[0])
    assert want.tolist() == [0.02022987938098004, 0.004173977864026143, 0.11612006417720729]
    b200 = np.array([0.0202298793518048, 0.004173977858006492, 0.1161200640097406])
    m = judge.judge(873, 730, 1, b200, want)
    assert m["clean"] and m["sensitive"] and m["excused"], m
    assert m["path"][-1] == "sphere/diffuse-light(solid)" and len(m["path"]) == 21
    assert po.TOL < po.deviation(b200, want) < 10 * po.TOL and m["libm_deviation"] < po.TOL
    m = judge.judge(873, 730, 1, want * (1.0 + 1e-7), want)
    assert m["clean"] and not m["sensitive"] and not m["excused"]
