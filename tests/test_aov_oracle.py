"""CPU side of the denoiser AOVs: the reference of tests/aov_ref.cpp must see, for every camera sample, exactly the hit
record tests/record_ref.cpp builds for the oracle's camera rays with their times; its albedo must be the RGB the
oracle's texture_value reflects; its normal and depth follow from the record by the rules of include/yart.h; its planes
are the per-sample values summed in sample order.  Also the CLI's PFM writer and the new flags.  The GPU tests
(tests/test_gpu_aovs.py) compare yart_render_aovs against this reference."""
import importlib
import os
import sys
from pathlib import Path

import numpy as np
import pytest

import aov_ref
import perturbed_oracle
import record_ref
from scene_fuzz import FuzzScene

ROOT = Path(__file__).resolve().parent.parent
NT = os.cpu_count()
PRESETS = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
           "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]


def has_media(desc):
    sd = desc.contents
    return any(sd.objects[i].wrap & 8 for i in range(sd.n_objects))


def same(a, b):
    return (a == b) | ((a != a) & (b != b))


@pytest.mark.parametrize("scene", [p for p in PRESETS if p not in ("cornell-box-smoke", "next-week-final")])
def test_sample_records_are_the_world_records_of_the_camera_rays(yart, orc, scene):
    """Media-free presets: record_ref draws media from another Philox stream, so only there do the two coincide."""
    preset = yart.ScenePreset(scene, seed=3)
    assert not has_media(preset.desc)
    w, h, ns = 40, 24, 2
    cam = preset.camera(w, h)
    rays, _, times = orc.camera_rays(cam, w, h, 1, 1 + ns, seed=7)
    ref, rr = aov_ref.Scene(preset), record_ref.Scene(preset)
    for order in (yart.ORDER_REFERENCE, yart.ORDER_NEAR):
        got = ref.samples(cam, w, h, 1, 1 + ns, seed=7, order=order).reshape(-1)
        want = rr.records(rays, times, yart.TARGET_WORLD, 0.001, float("inf"), order, n_threads=NT)
        for f in want.dtype.names:
            assert same(got["rec"][f], want[f]).all(), "%s order %d: field %s" % (scene, order, f)
        normal, depth = aov_ref.normal_depth_from_records(want, rays)
        assert (got["normal"] == normal).all() and (got["depth"] == depth).all(), scene
        assert (got["albedo"] >= 0).all() and (got["albedo"] <= 1).all()
        miss = want["obj_id"] == yart.MISS
        bg = np.clip(np.asarray(preset.desc.contents.background_rgb), 0, 1)
        assert (got["albedo"][miss] == bg).all()


def test_media_samples_hit_inside_the_medium(yart):
    """next-week-final's fog: some first hits are medium hits, with normal 0 and a positive distance."""
    preset = yart.ScenePreset("next-week-final", seed=3)
    ref = aov_ref.Scene(preset)
    s = ref.samples(preset.camera(48, 32), 48, 32, 0, 2).reshape(-1)
    sd = preset.desc.contents
    medium = np.array([bool(sd.objects[o].wrap & 8) if o != yart.MISS else False for o in s["rec"]["obj_id"]])
    assert medium.any()
    assert (s["normal"][medium] == 0).all() and (s["depth"][medium, 0] > 0).all()


def textures_of(desc):
    sd = desc.contents
    return [(i, sd.textures[i]) for i in range(sd.n_textures)]


@pytest.mark.parametrize("source", PRESETS + ["fuzz%d" % k for k in range(10)])
def test_texture_rgb_reflects_to_texture_value(yart, source):
    """rgb_reflect(texture_rgb) == texture_value: solid, checker and image exactly, noise as rgb_reflect(white) * s."""
    scene = FuzzScene(yart, 3000 + int(source[4:])) if source.startswith("fuzz") else yart.ScenePreset(source, seed=3)
    ref = aov_ref.Scene(scene)
    sd = scene.desc.contents
    r = np.random.default_rng(11)
    for i, t in textures_of(scene.desc):
        if t.kind == yart.abi.TEX_IMAGE and not sd.images[t.image].rgb8:
            continue  # (texture_value returns 1.0 without a spectrum; the albedo is white)
        for _ in range(40):
            p, u, v, wl = r.uniform(-6, 6, 3), r.uniform(-0.1, 1.1), r.uniform(-0.1, 1.1), r.uniform(360, 720)
            rgb = ref.texture_rgb(i, p, u, v)
            want = ref.texture_value(i, wl, p, u, v)
            if t.kind == yart.abi.TEX_NOISE:
                assert rgb[0] == rgb[1] == rgb[2]
                got = ref.rgb_reflect(np.ones(3), wl) * rgb[0]
            else:
                got = ref.rgb_reflect(rgb, wl)
            assert got == want, (source, i, t.kind, p, u, v, wl)


def test_planes_are_per_sample_values_summed_in_order(yart):
    preset = yart.ScenePreset("cornell-box-smoke", seed=3)
    ref = aov_ref.Scene(preset)
    w, h = 40, 24
    cam = preset.camera(w, h)
    s = ref.samples(cam, w, h, 0, 4)
    planes = ref.planes(cam, w, h, 0, 4)
    for k in aov_ref.PLANES:
        acc = np.zeros((h, w, 3))
        for j in range(4):
            acc = acc + s[k][:, :, j]
        rendered = planes["depth"][..., 2] > 0
        assert (planes[k][rendered] == acc[rendered]).all(), k
        assert (planes[k][~rendered] == 0).all(), k
    assert (planes["depth"][..., 2] == 4)[rendered].all()
    assert (rendered == np.outer(perturbed_oracle.covered(h), perturbed_oracle.covered(w))).all()
    chained = ref.planes(cam, w, h, 0, 1)
    ref.planes(cam, w, h, 1, 4, planes=chained)
    for k in aov_ref.PLANES:
        assert (chained[k] == planes[k]).all(), k
    only = ref.planes(cam, w, h, 0, 4, planes={"normal": np.zeros((h, w, 3))})
    assert list(only) == ["normal"] and (only["normal"] == planes["normal"]).all()


def cli():
    if str(ROOT) not in sys.path:
        sys.path.insert(0, str(ROOT))
    return importlib.import_module("yart_cli")


def test_pfm_round_trip(tmp_path):
    c = cli()
    r = np.random.default_rng(2)
    for shape in ((5, 7, 3), (4, 9)):
        img = r.standard_normal(shape).astype(np.float32)
        path = str(tmp_path / "x.pfm")
        c.write_pfm(path, img)
        raw = open(path, "rb").read()
        assert raw.startswith(b"PF\n7 5\n-1.0\n" if len(shape) == 3 else b"Pf\n9 4\n-1.0\n")
        back = c.read_pfm(path)
        assert back.dtype == np.float32 and back.shape == shape and (back == img).all()
        # rows are stored bottom to top
        assert np.frombuffer(raw[-img[0].nbytes:], dtype="<f4").tolist() == img[0].reshape(-1).tolist()


def test_cli_parses_the_aov_flags(yart):
    c = cli()
    ap = c.build_parser(yart.SCENE_NAMES)
    a = ap.parse_args(["--scene", "david", "--aovs", "--aov-samples", "8"])
    assert a.aovs and a.aov_samples == 8
    a = ap.parse_args(["--scene", "david"])
    assert not a.aovs and a.aov_samples is None
    with pytest.raises(SystemExit):
        ap.parse_args(["--scene", "david", "--aov-samples", "0"])
    assert c.aov_paths("out/david.png") == {k: "out/david.%s.pfm" % k for k in ("color", "albedo", "normal", "depth")}


def test_aov_means():
    y = importlib.import_module("yet-another-raytracer_b200")
    depth = np.array([[[6.0, 2.0, 4.0], [0.0, 0.0, 3.0], [0.0, 0.0, 0.0]]])
    albedo = np.array([[[2.0, 1.0, 0.0], [3.0, 3.0, 3.0], [0.0, 0.0, 0.0]]])
    m = y.aov_means({"albedo": albedo, "depth": depth})
    assert m["depth"].tolist() == [[3.0, 0.0, 0.0]]
    assert m["albedo"].tolist() == [[[0.5, 0.25, 0.0], [1.0, 1.0, 1.0], [0.0, 0.0, 0.0]]]
    assert "normal" not in m
