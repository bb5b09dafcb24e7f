"""The per-sample render gate, and the variants of the CPU oracle and the next-event reference it uses (test
infrastructure only).

The renderer and the oracle consume the same Philox draws and do the same f64 arithmetic in the same order, so one
path of one (pixel, sample) agrees to the last few bits, except where a transcendental differs in its last bits
(CUDA's sin/cos/acos/atan2/log against glibc's) and the path crosses a branch on that difference.  `per_sample_gate`
renders each sample index on its own on both sides, compares every pixel, and excuses a mismatch only if

  (a) it is libm-sensitive: some variant of the reference whose transcendentals are moved by a few ulp
      (YART_ORACLE_LIBM_PERTURB, oracle/yart_oracle.cpp) computes a different value for that (pixel, sample), and
  (b) it is traversal-clean: the oracle's rays of that path get bit-identical closest hits from the side under test
      (both traversal orders; a hit inside a medium, whose t goes through log, to 1e-12).

The variants are compiled like tests/nee_ref.py's library: digest-named in the temporary directory, never in the tree.
"""
import importlib
import os
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
if str(HERE) not in sys.path:
    sys.path.insert(0, str(HERE))
abi = importlib.import_module("yet-another-raytracer_b200._abi")
from oracle import orc  # noqa: E402
import nee_ref  # noqa: E402

# -D switches of each variant: a constant move of every result, or a seeded per-call move in [-2, 2] ulp (CUDA
# documents 2 ulp for double sin/cos/acos/atan2, 1 ulp for log)
IDENTITY = {"YART_ORACLE_LIBM_PERTURB": 0}
VARIANTS = {
    "+1ulp": {"YART_ORACLE_LIBM_PERTURB": 1},
    "-1ulp": {"YART_ORACLE_LIBM_PERTURB": -1},
    "seeded": {"YART_ORACLE_LIBM_PERTURB": 2, "YART_ORACLE_LIBM_SEED": 1},
}
# a libm the gate never uses: tests/test_perturbed_oracle.py treats it as the side under test
HELD_OUT = {"YART_ORACLE_LIBM_PERTURB": 2, "YART_ORACLE_LIBM_SEED": 0x5eed}

ORACLE_SOURCES = [ROOT / "oracle" / "yart_oracle.cpp", ROOT / "oracle" / "yart_oracle.h", ROOT / "include" / "yart.h",
                  ROOT / "include" / "yart_rng.h", ROOT / "include" / "yart_spectral_tables.h"]
ORACLE_FLAGS = [f for f in nee_ref.FLAGS if f != "-fvisibility=hidden"]  # (the flags of oracle/Makefile)
TOL = 1e-9
LIBM_GAIN = 10
ZERO_FLIP_PATHS = 5000

_libs = {}


def _defines(d):
    return ["-D%s=%d" % kv for kv in sorted(d.items())]


def _build(kind, defines):
    d = _defines(defines)
    if kind == "oracle":
        return orc.load(nee_ref.compile_shared("oracle_libm", ROOT / "oracle" / "yart_oracle.cpp", ORACLE_SOURCES,
                                               ORACLE_FLAGS + d))
    return nee_ref.load(nee_ref.compile_shared("nee_ref_libm", HERE / "nee_ref.cpp", nee_ref.SOURCES, nee_ref.FLAGS + d))


def variant_lib(kind, defines):
    """The library of `kind` ("oracle" or "nee") built with the perturbation `defines`."""
    key = (kind, tuple(sorted(defines.items())))
    if key not in _libs:
        _libs[key] = _build(kind, defines)
    return _libs[key]


def build_all():
    """Build every variant of both references (in parallel: each is a full compile of the oracle)."""
    jobs = [(k, d) for k in ("oracle", "nee") for d in [IDENTITY, HELD_OUT] + list(VARIANTS.values())]
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
        list(ex.map(lambda kd: variant_lib(*kd), jobs))


def covered(n):
    """Pixels along an axis of n that the reference's 8x8 tiling renders: n//8 from n*col//8 (main.rs:643-646)."""
    m = np.zeros(n, bool)
    for col in range(8):
        m[n * col // 8: n * col // 8 + n // 8] = True
    return m


def sanitized(xyz):
    out = np.empty(3)
    orc.lib().orc_sanitize_sample_xyz(np.ascontiguousarray(xyz, dtype=np.float64).ctypes.data, out.ctypes.data)
    return out


def deviation(got, want):
    """Per pixel: the largest channel difference over the pixel's largest channel (on either side); 0 where both
    are 0, inf where a value is not finite."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        scale = np.maximum(np.abs(got).max(axis=-1), np.abs(want).max(axis=-1))
        d = np.abs(got - want).max(axis=-1) / scale
    d = np.where(scale == 0, 0.0, d)
    return np.where(np.isfinite(d), d, np.inf)


def mismatched(got, want):
    """Per pixel: some channel differs by more than TOL times the pixel's largest channel (on either side)."""
    return deviation(got, want) > TOL


_OBJ = {abi.OBJ_SPHERE: "sphere", abi.OBJ_MOVING_SPHERE: "moving-sphere", abi.OBJ_XY_RECT: "xy-rect",
        abi.OBJ_XZ_RECT: "xz-rect", abi.OBJ_YZ_RECT: "yz-rect", abi.OBJ_BOX: "box", abi.OBJ_TRIANGLE: "triangle",
        abi.OBJ_MESH: "mesh", abi.OBJ_GROUP: "group"}
_MAT = {abi.MAT_NONE: "none", abi.MAT_LAMBERTIAN: "lambertian", abi.MAT_METAL: "metal", abi.MAT_DIELECTRIC: "dielectric",
        abi.MAT_DIFFUSE_LIGHT: "diffuse-light", abi.MAT_ISOTROPIC: "isotropic"}
_TEX = {abi.TEX_SOLID: "solid", abi.TEX_CHECKER: "checker", abi.TEX_NOISE: "noise", abi.TEX_IMAGE: "image"}


def describe_hit(sd, hit):
    """"object-kind/material-kind(texture-kind)" of a world hit, e.g. "sphere/dielectric" or "medium box/isotropic"."""
    if hit["prim_id"] == abi.MISS:
        return "miss"
    o = sd.objects[int(hit["obj_id"])]
    if o.kind == abi.OBJ_GROUP:
        o = sd.groups[o.index].members[int(hit["prim_id"])]
    m = sd.materials[o.material]
    tex = "(%s)" % _TEX.get(sd.textures[m.texture].kind, "?") if m.kind in (abi.MAT_LAMBERTIAN, abi.MAT_DIFFUSE_LIGHT) else ""
    return "%s%s/%s%s" % ("medium " if o.wrap & abi.WRAP_MEDIUM else "", _OBJ.get(o.kind, "?"), _MAT.get(m.kind, "?"), tex)


def same_hits(sd, got, want):
    """Closest hits bit for bit, except t inside a ConstantMedium to 1e-12 (as the world closest-hit tests)."""
    medium = np.array([bool(sd.objects[i].wrap & abi.WRAP_MEDIUM) for i in range(sd.n_objects)] + [False])
    in_medium = medium[np.minimum(want["obj_id"], sd.n_objects)] & (want["prim_id"] != abi.MISS)
    ok = np.ones(len(want), bool)
    for f in ("t", "u", "v", "prim_id", "obj_id", "front_face"):
        same = (got[f] == want[f]) | ((got[f] != got[f]) & (want[f] != want[f]))
        if f == "t":
            with np.errstate(invalid="ignore"):
                same |= in_medium & (np.abs(got[f] - want[f]) <= 1e-12 * np.abs(want[f]))
        ok &= same
    return bool(ok.all())


class Report:
    """What per_sample_gate found.  `mismatches`: one dict per mismatched (pixel, sample); `problems`: the failures
    that are not mismatches (uncovered pixels, ray counts)."""

    def __init__(self, what):
        self.what, self.mismatches, self.problems, self.n_samples = what, [], [], 0

    @property
    def excused(self):
        return [m for m in self.mismatches if m["excused"]]

    @property
    def unexcused(self):
        return [m for m in self.mismatches if not m["excused"]]

    def summary(self):
        return "%s: %d samples, %d mismatched, %d excused" % (self.what, self.n_samples, len(self.mismatches),
                                                               len(self.excused))

    def check(self, cap):
        """Fail on any unexcused mismatch, on more than `cap` excused ones, or on a problem."""
        lines = []
        for m in self.unexcused[:8]:
            lines.append("  pixel (%d, %d) sample %d: NOT EXCUSED; first hit %s; path %s; gpu %r oracle %r (deviation %.3g, "
                         "largest under a perturbed libm %.3g); libm-sensitive %s, traversal-clean %s" % (
                             m["x"], m["y"], m["sample"], m["path"][0] if m["path"] else "?", " -> ".join(m["path"]),
                             m["got"].tolist(), m["want"].tolist(), deviation(m["got"], m["want"]), m["libm_deviation"],
                             m["sensitive"], m["clean"]))
        assert not self.unexcused, "%s; %d unexcused:\n%s" % (self.summary(), len(self.unexcused), "\n".join(lines))
        assert not self.problems, "%s:\n  %s" % (self.summary(), "\n  ".join(self.problems))
        assert len(self.excused) <= cap, "%s: more than %d excused samples" % (self.summary(), cap)


class Judge:
    """Decides one mismatched (pixel, sample) of a scene and render settings: `judge(x, y, s, got, want)` returns the
    Report entry, with checks (a) and (b) done.  `closest_hit(rays, order) -> hits` is the side under test's world
    query.  (per_sample_gate uses one per case; a test can also ask about a single sample.)"""

    def __init__(self, scene, cam, w, h, depth, seed, flags, order, closest_hit, variants=None, n_threads=None):
        self.scene, self.cam, self.w, self.h, self.depth, self.seed = scene, cam, w, h, depth, seed
        self.flags, self.order, self.closest_hit = flags, order, closest_hit
        self.n_threads = n_threads or os.cpu_count()
        self.variants = list((variants or VARIANTS).values())
        self.nee = bool(flags & abi.FLAG_NEXT_EVENT)
        self.sd = getattr(scene, "desc", scene).contents
        self.replay = orc.Scene(scene)  # NEE paths are the unbiased pick's paths (tests/test_gpu_next_event.py)
        self.replay_flags = (flags & ~abi.FLAG_NEXT_EVENT) | (abi.FLAG_UNBIASED_LIGHT_PICK if self.nee else 0)
        self._var_scenes, self._var_films = None, {}

    def variant_values(self, x, y, s):
        """The sanitised value of (x, y, s) under each perturbed variant."""
        if self._var_scenes is None:
            kind = "nee" if self.nee else "oracle"
            cls = nee_ref.Scene if self.nee else orc.Scene
            self._var_scenes = [cls(self.scene, variant_lib(kind, d)) for d in self.variants]
        out = []
        for i, vs in enumerate(self._var_scenes):
            if self.nee:  # (the next-event reference renders whole frames only)
                if (i, s) not in self._var_films:
                    self._var_films[(i, s)] = vs.render(self.cam, self.w, self.h, s, s + 1, max_depth=self.depth,
                                                        seed=self.seed, order=self.order, n_threads=self.n_threads,
                                                        flags=self.flags)[0]
                out.append(self._var_films[(i, s)][y, x])
            else:
                out.append(sanitized(vs.sample(self.cam, self.w, self.h, y * self.w + x, s, max_depth=self.depth,
                                               seed=self.seed, order=self.order, flags=self.flags)[0]))
        return out

    def judge(self, x, y, s, got, want):
        x, y, s = int(x), int(y), int(s)
        # (a) A variant flips the sample past the tolerance too (a branch taken on a last-bit difference), or the
        # sample is so libm-sensitive that a few ulp move it by at least 1/LIBM_GAIN of the deviation seen.  The
        # second case is a path whose value amplifies ulp differences without a branch: on david 1920x1080 a path of
        # 20 bounces ending on the sphere light moves by 1e-10 to 4e-9 under +-1 and +-2 ulp, and the B200's value
        # of it sits 1.4e-9 from the oracle's (tests/test_perturbed_oracle.py keeps that sample).
        devs = [deviation(v, want) for v in self.variant_values(x, y, s)]
        sensitive = max(devs) > TOL or max(devs) >= deviation(got, want) / LIBM_GAIN
        # (b) the oracle's rays of this path get the same closest hits from the side under test
        rays = self.replay.sample_path(self.cam, self.w, self.h, y * self.w + x, s, max_depth=self.depth,
                                       seed=self.seed, order=self.order, flags=self.replay_flags)
        want_hits = {o: self.replay.closest_hit(rays, order=o)[0] for o in (abi.ORDER_REFERENCE, abi.ORDER_NEAR)}
        clean = all(same_hits(self.sd, self.closest_hit(rays, o), want_hits[o]) for o in want_hits)
        path = [describe_hit(self.sd, hh) for hh in want_hits[abi.ORDER_REFERENCE]]
        return dict(x=x, y=y, sample=s, got=np.array(got, dtype=np.float64), want=np.array(want, dtype=np.float64),
                    sensitive=sensitive, clean=clean, excused=sensitive and clean, path=path, libm_deviation=max(devs))


def per_sample_gate(scene, cam, w, h, samples, depth, seed, flags, order, render, closest_hit, what="",
                    variants=None, n_threads=None):
    """Compare `render(s) -> (film, stats)`, the side under test rendering samples [s, s+1), with the reference
    (the oracle, or tests/nee_ref.cpp when `flags` has FLAG_NEXT_EVENT) for each s in `samples`.
    `closest_hit(rays, order) -> hits` is the side under test's world query, for check (b).  `variants`: the
    perturbation defines used for check (a) (default VARIANTS).  Returns a Report."""
    n_threads = n_threads or os.cpu_count()
    judge = Judge(scene, cam, w, h, depth, seed, flags, order, closest_hit, variants, n_threads)
    base = nee_ref.Scene(scene) if judge.nee else judge.replay
    mask = covered(h)[:, None] & covered(w)[None, :]
    rep = Report(what)
    for s in samples:
        rep.n_samples += int(mask.sum())
        want, st_w = base.render(cam, w, h, s, s + 1, max_depth=depth, seed=seed, order=order, n_threads=n_threads,
                                 flags=flags)
        got, st = render(s)
        for name, f in (("side under test", got), ("reference", want)):
            if not (f[~mask] == 0).all():
                rep.problems.append("sample %d: the %s wrote %d pixels outside the reference's tiles" % (
                    s, name, int((f[~mask] != 0).any(axis=-1).sum())))
        n_excused = 0
        for y, x in np.argwhere(mismatched(got, want) & mask):
            m = judge.judge(x, y, s, got[y, x], want[y, x])
            n_excused += m["excused"]
            rep.mismatches.append(m)
        # A libm flip between two paths that both end at zero (a miss on a black background, say) changes the
        # ray count and not the film: the held-out variant does that on david 96x96 in 4 of 8 sample ranges, by 1-5
        # rays.  So each range may also lose or gain max_depth + 1 rays per ZERO_FLIP_PATHS paths (and at least once).
        slack = n_excused + 1 + int(mask.sum()) // ZERO_FLIP_PATHS
        if abs(int(st.rays) - int(st_w.rays)) > slack * (depth + 1):
            rep.problems.append("sample %d: %d rays against the reference's %d with %d excused samples" % (
                s, st.rays, st_w.rays, n_excused))
        if st.paths != st_w.paths:
            rep.problems.append("sample %d: %d paths against the reference's %d" % (s, st.paths, st_w.paths))
    return rep
