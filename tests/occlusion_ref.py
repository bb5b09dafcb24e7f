"""ctypes binding of tests/occlusion_ref.cpp, the CPU reference of the occlusion queries (test infrastructure only).

The library is compiled on first use with the CPU oracle's own flags (oracle/Makefile) into a per-user directory under
the system's temporary directory, named by a digest of its sources, so the repository tree stays read-only."""
import ctypes as C
import hashlib
import importlib
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
abi = importlib.import_module("yet-another-raytracer_b200._abi")

SOURCES = [HERE / "occlusion_ref.cpp", ROOT / "oracle" / "yart_oracle.cpp", ROOT / "oracle" / "yart_oracle.h",
           ROOT / "include" / "yart.h", ROOT / "include" / "yart_rng.h", ROOT / "include" / "yart_spectral_tables.h"]
FLAGS = ["-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-march=x86-64-v3", "-pthread",
         "-fvisibility=hidden", "-shared"]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    cxx = os.environ.get("CXX", "g++")
    h = hashlib.sha256(" ".join([cxx] + FLAGS).encode())
    for f in SOURCES:
        h.update(f.read_bytes())
    out_dir = Path(tempfile.gettempdir()) / ("yart_occlusion_ref_%d" % os.getuid())
    out_dir.mkdir(exist_ok=True)
    so = out_dir / ("occlusion_ref_%s.so" % h.hexdigest()[:16])
    if not so.exists():
        tmp = so.with_suffix(".tmp%d.so" % os.getpid())
        res = subprocess.run([cxx] + FLAGS + ["-o", str(tmp), str(HERE / "occlusion_ref.cpp")], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("occlusion reference build failed:\n" + res.stdout + res.stderr)
        os.replace(tmp, so)  # (atomic: parallel test workers may build it at the same time)
    L = C.CDLL(str(so))
    vp = C.c_void_p
    L.occref_last_error.restype, L.occref_last_error.argtypes = C.c_char_p, []
    L.occref_scene_create.restype, L.occref_scene_create.argtypes = C.c_int, [C.POINTER(abi.SceneDesc), C.POINTER(vp)]
    L.occref_scene_free.restype, L.occref_scene_free.argtypes = None, [vp]
    L.occref_occluded.restype = C.c_int
    L.occref_occluded.argtypes = [vp, C.c_uint32, vp, C.c_uint64, C.c_double, C.c_double, vp, C.c_int]
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise RuntimeError("occlusion reference error %d: %s" % (rc, lib().occref_last_error().decode()))


class Scene:
    """The reference's view of a scene description (a ctypes POINTER(SceneDesc) or an object with a `.desc`)."""

    def __init__(self, scene):
        self._keep = scene
        self._h = C.c_void_p()
        _check(lib().occref_scene_create(getattr(scene, "desc", scene), C.byref(self._h)))

    def occluded(self, rays, target=abi.TARGET_WORLD, t_min=0.001, t_max=float("inf"), n_threads=1):
        """A bool per ray: True where orc_closest_hit(..., ORDER_REFERENCE) reports a hit."""
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_DTYPE)
        out = np.empty(rays.shape[0], dtype=np.uint8)
        _check(lib().occref_occluded(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, out.ctypes.data,
                                     n_threads))
        return out.view(np.bool_)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.occref_scene_free(self._h)
            self._h = None
