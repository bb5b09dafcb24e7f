"""ctypes binding of tests/nee_ref.cpp, the CPU reference of YART_FLAG_NEXT_EVENT (test infrastructure only).

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

SOURCES = [HERE / "nee_ref.cpp", ROOT / "oracle" / "yart_oracle.cpp", ROOT / "oracle" / "yart_oracle.h",
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
    out_dir = Path(tempfile.gettempdir()) / ("yart_nee_ref_%d" % os.getuid())
    out_dir.mkdir(exist_ok=True)
    so = out_dir / ("nee_ref_%s.so" % h.hexdigest()[:16])
    if not so.exists():
        tmp = so.with_suffix(".tmp%d.so" % os.getpid())
        res = subprocess.run([cxx] + FLAGS + ["-o", str(tmp), str(HERE / "nee_ref.cpp")], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("next-event reference build failed:\n" + res.stdout + res.stderr)
        os.replace(tmp, so)  # (atomic: parallel test workers may build it at the same time)
    L = C.CDLL(str(so))
    vp = C.c_void_p
    L.neeref_last_error.restype, L.neeref_last_error.argtypes = C.c_char_p, []
    L.neeref_scene_create.restype, L.neeref_scene_create.argtypes = C.c_int, [C.POINTER(abi.SceneDesc), C.POINTER(vp)]
    L.neeref_scene_free.restype, L.neeref_scene_free.argtypes = None, [vp]
    L.neeref_render.restype = C.c_int
    L.neeref_render.argtypes = [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderOpts), vp, C.POINTER(abi.Stats), C.c_int]
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise RuntimeError("next-event reference error %d: %s" % (rc, lib().neeref_last_error().decode()))


class Scene:
    """The reference's view of a scene description (a ctypes POINTER(SceneDesc) or an object with a `.desc`)."""

    def __init__(self, scene):
        self._keep = scene
        self._h = C.c_void_p()
        _check(lib().neeref_scene_create(getattr(scene, "desc", scene), C.byref(self._h)))

    def render(self, camera, width, height, sample_begin, sample_end, max_depth=50, seed=1, order=abi.ORDER_REFERENCE,
               n_threads=1, flags=abi.FLAG_NEXT_EVENT):
        """(film, stats) like oracle Scene.render, with the next-event estimator (always on; `flags` adds
        YART_FLAG_RUSSIAN_ROULETTE / DEPTH_ZERO_BLACK)."""
        film = np.zeros((height, width, 3), dtype=np.float64)
        o = abi.RenderOpts()
        o.width, o.height, o.sample_begin, o.sample_end = width, height, sample_begin, sample_end
        o.max_depth, o.order, o.batch_spp, o.flags, o.seed = max_depth, order, 0, flags, seed
        st = abi.Stats()
        _check(lib().neeref_render(self._h, C.byref(camera), C.byref(o), film.ctypes.data, C.byref(st), n_threads))
        return film, st

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.neeref_scene_free(self._h)
            self._h = None
