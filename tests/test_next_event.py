"""YART_FLAG_NEXT_EVENT (next-event estimation with MIS) in its CPU reference, tests/nee_ref.cpp: the estimator the
CUDA path is compared with in tests/test_gpu_next_event.py, checked here against the unchanged CPU oracle.

The flag changes how light is collected, never which path rays are traced, so ray counts are equal to the flag-off
render with the unbiased light pick (which NEXT_EVENT implies).  Its expectation is that render's too; the tests
bound the difference by four standard deviations derived from the per-pixel sample variance.  The sanitiser's clamp
of a sample's Y at 20 is nonlinear and would make the two expectations differ, so the comparisons run where it
(almost) never engages, and the tests check that it does not.
"""
import os

import re
from pathlib import Path

import numpy as np

import nee_ref
import refpins

NEXT_EVENT = 32


def _scene(yart, orc, name, flags=0):
    """The NEE reference for NEXT_EVENT renders, the oracle for everything else."""
    preset = yart.ScenePreset(name, seed=1)
    return preset, (nee_ref.Scene(preset) if flags & NEXT_EVENT else orc.Scene(preset))


def _render(yart, orc, name, w, h, spp, flags, depth=50, seed=1):
    preset, s = _scene(yart, orc, name, flags)
    return s.render(preset.camera(w, h), w, h, 0, spp, max_depth=depth, seed=seed, n_threads=os.cpu_count(), flags=flags)


def _per_sample(yart, orc, name, w, h, spp, flags, depth=50, seed=1):
    """(spp, H, W, 3) sanitised samples, one render call per sample index, and the total ray count."""
    preset, s = _scene(yart, orc, name, flags)
    cam = preset.camera(w, h)
    out, rays = [], 0
    for k in range(spp):
        f, st = s.render(cam, w, h, k, k + 1, max_depth=depth, seed=seed, n_threads=os.cpu_count(), flags=flags)
        out.append(f)
        rays += int(st.rays)
    return np.stack(out), rays


def test_the_flag_is_the_headers(yart):
    header = (Path(__file__).resolve().parent.parent / "include" / "yart.h").read_text()
    assert int(re.search(r"YART_FLAG_NEXT_EVENT = (\d+)u", header).group(1)) == yart.FLAG_NEXT_EVENT == NEXT_EVENT


def test_no_lights_means_no_change(yart, orc):
    """Without a lights list there is nothing to sample: the film is the unbiased-pick film bit for bit."""
    for name, w, h, spp in (("cornell-box-smoke", 32, 32, 4), ("random-scene", 32, 24, 4)):
        a, st_a = _render(yart, orc, name, w, h, spp, yart.FLAG_UNBIASED_LIGHT_PICK)
        b, st_b = _render(yart, orc, name, w, h, spp, NEXT_EVENT)
        assert np.array_equal(a, b), name
        assert st_a.rays == st_b.rays


def test_lights_change_the_film_but_not_the_rays(yart, orc):
    for name in ("cornell-box", "sycee"):
        a, st_a = _render(yart, orc, name, 32, 32, 4, NEXT_EVENT)
        c, st_c = _render(yart, orc, name, 32, 32, 4, yart.FLAG_UNBIASED_LIGHT_PICK)
        assert not np.array_equal(a, c) and st_a.rays == st_c.rays


def _mean_and_sigma(a, b):
    """a, b: (spp, n) per-sample values of n statistics.  Pixels are independent, samples of a pixel i.i.d.:
    the sum over a region has variance sum(var_pixel) / spp per sample mean."""
    ma, mb = a.mean(axis=0), b.mean(axis=0)
    sa, sb = a.var(axis=0, ddof=1) / a.shape[0], b.var(axis=0, ddof=1) / b.shape[0]
    return ma, mb, np.sqrt(sa + sb)


def _region_sums(samples, regions):
    """(spp, len(regions) + 1): Y summed over the whole frame and over each region (40 x 40 block coordinates)."""
    y = samples[..., 1]
    h, w = y.shape[1:]
    cols = [y.sum(axis=(1, 2))]
    for r, c in regions.values():
        rs = slice(r.start * h // 40, r.stop * h // 40)
        cs = slice(c.start * w // 40, c.stop * w // 40)
        cols.append(y[:, rs, cs].sum(axis=(1, 2)))
    return np.stack(cols, axis=1)


def test_same_expectation_as_the_unbiased_pick(yart, orc):
    regions = {k: refpins.CORNELL_REGIONS[k] for k in ("back wall", "floor", "ceiling", "green wall")}
    for name, w, h, spp, regs in (("cornell-box", 96, 96, 48, regions), ("sycee", 64, 64, 24, {})):
        a, rays_a = _per_sample(yart, orc, name, w, h, spp, yart.FLAG_UNBIASED_LIGHT_PICK)
        b, rays_b = _per_sample(yart, orc, name, w, h, spp, NEXT_EVENT)
        assert rays_a == rays_b, name  # the same path rays
        for s in (a, b):  # the clamp (Y > 20 -> 20) must be (nearly) idle for the expectations to be comparable
            assert (s[..., 1] >= 20.0 * (1 - 1e-9)).mean() < 1e-3, name
        ra, rb = _region_sums(a, regs), _region_sums(b, regs)
        ma, mb, sd = _mean_and_sigma(ra, rb)
        labels = ["frame"] + list(regs)
        print(name, {k: (round(float(x), 2), round(float(y), 2), round(float(z), 3)) for k, x, y, z in zip(labels, ma, mb, sd)})
        for k, x, y, z in zip(labels, ma, mb, sd):
            assert abs(x - y) <= 4.0 * z, (name, k, x, y, z)
        # and light sampling pays: the per-sample variance of the frame's Y is lower with it
        if name == "cornell-box":
            assert b[..., 1].var(axis=0).sum() < a[..., 1].var(axis=0).sum()


def test_a_light_sample_is_never_taken_at_max_depth(yart, orc):
    """At depth 1 the only hit is the camera ray's: no light sample pairs with it, so the film is the flag-off one
    (the continuation's emission weight only matters at the next hit, which is never traced)."""
    a, _ = _render(yart, orc, "cornell-box", 32, 32, 4, yart.FLAG_UNBIASED_LIGHT_PICK, depth=1)
    b, _ = _render(yart, orc, "cornell-box", 32, 32, 4, NEXT_EVENT, depth=1)
    assert np.array_equal(a, b)
    c, _ = _render(yart, orc, "cornell-box", 32, 32, 4, yart.FLAG_UNBIASED_LIGHT_PICK, depth=2)
    d, _ = _render(yart, orc, "cornell-box", 32, 32, 4, NEXT_EVENT, depth=2)
    assert not np.array_equal(c, d)
