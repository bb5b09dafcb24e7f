"""CPU checks of tests/denoise_ref.py, the numpy statement of yart_denoise that tests/test_gpu_denoise.py holds the
library to, and of the --denoise flags of both command lines."""
import importlib
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import denoise_ref

ROOT = Path(__file__).resolve().parent.parent


def flat_inputs(h, w, spp=4, samples=4.0, film_value=(1.0, 2.0, 3.0), albedo=(0.5, 0.5, 0.5), normal=(0.0, 1.0, 0.0),
                dist=3.0):
    """Planes as render_aovs sums them (`samples` samples a pixel, all hitting at `dist`) and a constant film."""
    film = np.broadcast_to(np.asarray(film_value, float), (h, w, 3)).copy()
    planes = {"albedo": np.broadcast_to(np.asarray(albedo) * samples, (h, w, 3)).copy(),
              "normal": np.broadcast_to(np.asarray(normal) * samples, (h, w, 3)).copy(),
              "depth": np.broadcast_to(np.array([dist * samples, samples, samples]), (h, w, 3)).copy()}
    return film, spp, planes


def test_constant_image_on_flat_guides_stays_constant():
    film, spp, planes = flat_inputs(23, 31)
    want = denoise_ref.film_linear(film, spp) / (0.5 + 1 / 128) * (0.5 + 1 / 128)
    for levels in (1, 3, 5, 10):
        out = denoise_ref.denoise(film, spp, planes, levels=levels)
        assert np.abs(out - want).max() <= 1e-15 * np.abs(want).max(), levels


def test_invalid_pixels_output_zero_and_never_leak():
    rng = np.random.default_rng(5)
    film, spp, planes = flat_inputs(20, 24)
    film += rng.uniform(0, 1, film.shape)
    invalid = rng.uniform(size=(20, 24)) < 0.3
    planes["depth"][invalid] = 0.0
    out = denoise_ref.denoise(film, spp, planes)
    assert (out[invalid] == 0).all() and (out[~invalid] != 0).all()
    # whatever the film and the other planes hold at invalid pixels changes nothing
    film2 = film.copy()
    film2[invalid] = 1e6
    planes2 = {k: v.copy() for k, v in planes.items()}
    planes2["albedo"][invalid] = 7.0
    planes2["normal"][invalid] = -3.0
    assert (denoise_ref.denoise(film2, spp, planes2) == out).all()


def test_normal_and_hit_edges_do_not_bleed():
    """Left half: bright, normal +y; right half: 1000x darker, normal +x; below row 10 the right half is a miss.  With a
    colour term too wide to stop anything, the normal edge keeps the bright side out of the dark one, and the hit/miss
    edge is not crossed at all."""
    h, w = 24, 32
    film, spp, planes = flat_inputs(h, w, film_value=(8.0, 8.0, 8.0))
    film *= np.random.default_rng(1).uniform(0.5, 1.5, (h, w, 1))  # noise for the filter to remove
    right = np.zeros((h, w), bool)
    right[:, w // 2:] = True
    film[right] *= 1e-3
    planes["normal"][right] = [4.0, 0.0, 0.0]
    miss = right.copy()
    miss[:10] = False
    planes["depth"][miss] = [0.0, 0.0, 4.0]
    planes["normal"][miss] = 0.0
    wide = {"sigma_color": 1e6}
    out = denoise_ref.denoise(film, spp, planes, **wide)
    lin = denoise_ref.film_linear(film, spp)
    assert out[right].mean() < 1.02 * lin[right].mean()  # (a 0.002 % leak of the bright side would add 2 %)
    assert out[~right].std() < 0.5 * lin[~right].std()  # the filter did smooth
    film_far = film.copy()
    film_far[~miss] *= 1e4  # everything that hits changes ...
    out_far = denoise_ref.denoise(film_far, spp, planes, **wide)
    assert (out_far[miss] == out[miss]).all()  # ... and the misses do not notice


def test_levels_and_defaults_resolve_as_documented():
    assert denoise_ref.resolve() == (5, 8.0, 0.3, 0.05)
    assert denoise_ref.resolve(3, -1.0, 0.0, 2.0) == (3, 8.0, 0.3, 2.0)
    assert denoise_ref.resolve(10)[0] == 10
    for bad in ({"levels": 11}, {"sigma_color": float("nan")}, {"sigma_depth": float("inf")}):
        with pytest.raises(ValueError):
            denoise_ref.resolve(**bad)
    film, spp, planes = flat_inputs(9, 11)
    film = film * np.random.default_rng(2).uniform(0.5, 1.5, film.shape)
    assert (denoise_ref.denoise(film, spp, planes) == denoise_ref.denoise(film, spp, planes, 5, 8.0, 0.3, 0.05)).all()
    assert not (denoise_ref.denoise(film, spp, planes, 1) == denoise_ref.denoise(film, spp, planes, 2)).all()


def test_display_rule_zeroes_invalid_pixels():
    out = np.array([[[0.5, -1.0, 2.0], [0.0, 0.0, 0.0]]])
    depth = np.array([[[1.0, 1.0, 1.0], [0.0, 0.0, 0.0]]])
    rgba, _ = denoise_ref.display_rgba(out, depth)
    assert rgba[0, 0, 1] == 0 and rgba[0, 0, 2] == 255 and rgba[0, 0, 3] == 255 and (rgba[0, 1] == 0).all()


def test_cli_parses_the_denoise_flag(yart):
    sys.path.insert(0, str(ROOT))
    cli = importlib.import_module("yart_cli")
    ap = cli.build_parser(yart.SCENE_NAMES)
    a = ap.parse_args(["--scene", "david", "--denoise", "--aov-samples", "4"])
    assert a.denoise and a.aov_samples == 4 and not a.aovs
    assert not ap.parse_args(["--scene", "david"]).denoise
    assert cli.denoised_paths("out/david.png") == {"png": "out/david.denoised.png", "pfm": "out/david.denoised.pfm"}


def test_native_host_accepts_the_denoise_flag(yart, assets):
    exe = ROOT / "yet-another-raytracer_b200" / "yart"
    r = subprocess.run([str(exe), "--scene", "david", "--denoise", "--dry-run", "--assets", assets], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr
