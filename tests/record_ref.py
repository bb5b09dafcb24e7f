"""ctypes binding of tests/record_ref.cpp, the CPU reference of yart_closest_hit_records (test infrastructure only).

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

SOURCES = [HERE / "record_ref.cpp", ROOT / "oracle" / "yart_oracle.cpp", ROOT / "oracle" / "yart_oracle.h",
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
    out_dir = Path(tempfile.gettempdir()) / ("yart_record_ref_%d" % os.getuid())
    out_dir.mkdir(exist_ok=True)
    so = out_dir / ("record_ref_%s.so" % h.hexdigest()[:16])
    if not so.exists():
        tmp = so.with_suffix(".tmp%d.so" % os.getpid())
        res = subprocess.run([cxx] + FLAGS + ["-o", str(tmp), str(HERE / "record_ref.cpp")], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("record reference build failed:\n" + res.stdout + res.stderr)
        os.replace(tmp, so)  # (atomic: parallel test workers may build it at the same time)
    L = C.CDLL(str(so))
    vp = C.c_void_p
    L.recref_last_error.restype, L.recref_last_error.argtypes = C.c_char_p, []
    L.recref_scene_create.restype, L.recref_scene_create.argtypes = C.c_int, [C.POINTER(abi.SceneDesc), C.POINTER(vp)]
    L.recref_scene_free.restype, L.recref_scene_free.argtypes = None, [vp]
    L.recref_records.restype = C.c_int
    L.recref_records.argtypes = [vp, C.c_uint32, vp, vp, C.c_uint64, C.c_double, C.c_double, C.c_uint32, vp, C.c_int]
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise RuntimeError("record reference error %d: %s" % (rc, lib().recref_last_error().decode()))


class Scene:
    """The reference's view of a scene description (a ctypes POINTER(SceneDesc) or an object with a `.desc`)."""

    def __init__(self, scene):
        self._keep = scene
        self._h = C.c_void_p()
        _check(lib().recref_scene_create(getattr(scene, "desc", scene), C.byref(self._h)))

    def records(self, rays, times=None, target=abi.TARGET_WORLD, t_min=0.001, t_max=float("inf"),
                order=abi.ORDER_REFERENCE, n_threads=1):
        """One abi.RECORD_DTYPE record per ray, as the oracle's world.hit (or L4QBVH::hit for a mesh target) builds it."""
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_DTYPE)
        n = rays.shape[0]
        if times is not None:
            times = np.ascontiguousarray(times, dtype=np.float64)
            assert times.shape == (n,)
        out = np.empty(n, dtype=abi.RECORD_DTYPE)
        _check(lib().recref_records(self._h, target, rays.ctypes.data, None if times is None else times.ctypes.data, n,
                                    t_min, t_max, order, out.ctypes.data, n_threads))
        return out

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.recref_scene_free(self._h)
            self._h = None
