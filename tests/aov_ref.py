"""ctypes binding of tests/aov_ref.cpp, the CPU reference of yart_render_aovs (test infrastructure only).

The library is compiled on first use with the oracle's flags into the temporary directory (tests/nee_ref.py's
compile_shared: digest-named, never in the tree).  `lib(defines)` builds a libm-perturbed variant
(YART_ORACLE_LIBM_PERTURB, tests/perturbed_oracle.py) of the same file."""
import ctypes as C
import importlib
import os
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
for p in (ROOT, HERE):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))
abi = importlib.import_module("yet-another-raytracer_b200._abi")
import nee_ref  # noqa: E402

SOURCES = [HERE / "aov_ref.cpp"] + nee_ref.SOURCES[1:]
FLAGS = nee_ref.FLAGS
# one (pixel, sample) of aovref_samples
SAMPLE_DTYPE = np.dtype([("rec", abi.RECORD_DTYPE), ("albedo", "<f8", 3), ("normal", "<f8", 3), ("depth", "<f8", 3)])
PLANES = ("albedo", "normal", "depth")

_libs = {}


def lib(defines=None):
    """The reference library; `defines` ({name: int}) selects a libm-perturbed variant."""
    key = tuple(sorted((defines or {}).items()))
    if key in _libs:
        return _libs[key]
    d = ["-D%s=%d" % kv for kv in key]
    stem = "aov_ref" + "".join("_%s%d" % (k.rsplit("_", 1)[-1].lower(), v) for k, v in key)
    L = C.CDLL(str(nee_ref.compile_shared(stem, HERE / "aov_ref.cpp", SOURCES, FLAGS + d)))
    vp, P = C.c_void_p, C.POINTER
    L.aovref_last_error.restype, L.aovref_last_error.argtypes = C.c_char_p, []
    L.aovref_scene_create.restype, L.aovref_scene_create.argtypes = C.c_int, [P(abi.SceneDesc), P(vp)]
    L.aovref_scene_free.restype, L.aovref_scene_free.argtypes = None, [vp]
    L.aovref_sample_bytes.restype, L.aovref_sample_bytes.argtypes = C.c_uint32, []
    L.aovref_samples.restype = C.c_int
    L.aovref_samples.argtypes = [vp, P(abi.Camera), P(abi.RenderOpts), vp, C.c_int]
    L.aovref_planes.restype = C.c_int
    L.aovref_planes.argtypes = [vp, P(abi.Camera), P(abi.RenderOpts), vp, vp, vp, C.c_int]
    L.aovref_texture_rgb.restype = None
    L.aovref_texture_rgb.argtypes = [vp, C.c_uint32, vp, C.c_double, C.c_double, vp]
    L.aovref_texture_value.restype = C.c_double
    L.aovref_texture_value.argtypes = [vp, C.c_uint32, C.c_double, vp, C.c_double, C.c_double]
    L.aovref_rgb_reflect.restype, L.aovref_rgb_reflect.argtypes = C.c_double, [vp, C.c_double]
    assert L.aovref_sample_bytes() == SAMPLE_DTYPE.itemsize
    _libs[key] = L
    return L


def normal_depth_from_records(rec, rays):
    """include/yart.h's normal and depth rules, restated in numpy from the record and the camera ray."""
    n = rec["normal"]
    length = np.sqrt(n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1] + n[:, 2] * n[:, 2])
    hit = rec["obj_id"] != abi.MISS
    ok = hit & (length > 0) & np.isfinite(length)
    with np.errstate(invalid="ignore", divide="ignore"):
        normal = np.where(ok[:, None], n / np.where(ok, length, 1.0)[:, None], 0.0)
    d = rays["direction"]
    dist = np.where(hit, rec["t"] * np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]), 0.0)
    depth = np.stack([dist, hit.astype(float), np.ones(len(rec))], axis=1)
    return normal, depth


def opts(w, h, sample_begin, sample_end, seed=1, order=abi.ORDER_REFERENCE):
    o = abi.RenderOpts()
    o.width, o.height, o.sample_begin, o.sample_end = w, h, sample_begin, sample_end
    o.max_depth, o.order, o.batch_spp, o.flags, o.seed = 50, order, 0, 0, seed
    return o


class Scene:
    """The reference's view of a scene description (a ctypes POINTER(SceneDesc) or an object with a `.desc`)."""

    def __init__(self, scene, defines=None):
        self._keep = scene
        self.L = lib(defines)
        self._h = C.c_void_p()
        self._check(self.L.aovref_scene_create(getattr(scene, "desc", scene), C.byref(self._h)))

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("aov reference error %d: %s" % (rc, self.L.aovref_last_error().decode()))

    def samples(self, cam, w, h, sample_begin, sample_end, seed=1, order=abi.ORDER_REFERENCE, n_threads=None):
        """(h, w, n_samples) SAMPLE_DTYPE: every pixel's first-hit record and plane contributions, tiles or not."""
        out = np.empty((h, w, sample_end - sample_begin), dtype=SAMPLE_DTYPE)
        o = opts(w, h, sample_begin, sample_end, seed, order)
        self._check(self.L.aovref_samples(self._h, C.byref(cam), C.byref(o), out.ctypes.data, n_threads or os.cpu_count()))
        return out

    def planes(self, cam, w, h, sample_begin, sample_end, seed=1, order=abi.ORDER_REFERENCE, planes=None, n_threads=None):
        """The planes yart_render_aovs adds for these samples (added to `planes` if given, like the library)."""
        if planes is None:
            planes = {k: np.zeros((h, w, 3)) for k in PLANES}
        ptr = [planes[k].ctypes.data if k in planes else None for k in PLANES]
        o = opts(w, h, sample_begin, sample_end, seed, order)
        self._check(self.L.aovref_planes(self._h, C.byref(cam), C.byref(o), *ptr, n_threads or os.cpu_count()))
        return planes

    def texture_rgb(self, tex, p, u, v):
        p = np.ascontiguousarray(p, dtype=np.float64)
        out = np.empty(3)
        self.L.aovref_texture_rgb(self._h, tex, p.ctypes.data, u, v, out.ctypes.data)
        return out

    def texture_value(self, tex, wl, p, u, v):
        p = np.ascontiguousarray(p, dtype=np.float64)
        return self.L.aovref_texture_value(self._h, tex, wl, p.ctypes.data, u, v)

    def rgb_reflect(self, rgb, wl):
        rgb = np.ascontiguousarray(rgb, dtype=np.float64)
        return self.L.aovref_rgb_reflect(rgb.ctypes.data, wl)

    def __del__(self):
        if getattr(self, "_h", None):
            self.L.aovref_scene_free(self._h)
            self._h = None
