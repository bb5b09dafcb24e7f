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


def compile_shared(stem, source, deps, flags):
    """Compile `source` with `flags` into <tmp>/yart_nee_ref_<uid>/<stem>_<digest>.so, the digest taken over the
    compiler, the flags and `deps`; built once, replaced atomically (parallel test workers may build it at the same
    time).  Returns the path."""
    cxx = os.environ.get("CXX", "g++")
    h = hashlib.sha256(" ".join([cxx] + flags).encode())
    for f in deps:
        h.update(f.read_bytes())
    out_dir = Path(tempfile.gettempdir()) / ("yart_nee_ref_%d" % os.getuid())
    out_dir.mkdir(exist_ok=True)
    so = out_dir / ("%s_%s.so" % (stem, h.hexdigest()[:16]))
    if not so.exists():
        tmp = so.with_suffix(".tmp%d.so" % os.getpid())
        res = subprocess.run([cxx] + flags + ["-o", str(tmp), str(source)], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("%s build failed:\n%s%s" % (stem, res.stdout, res.stderr))
        os.replace(tmp, so)
    return so


def load(path):
    """A build of nee_ref.cpp at `path` (the default one or a variant, tests/perturbed_oracle.py)."""
    L = C.CDLL(str(path))
    vp = C.c_void_p
    L.neeref_last_error.restype, L.neeref_last_error.argtypes = C.c_char_p, []
    L.neeref_scene_create.restype, L.neeref_scene_create.argtypes = C.c_int, [C.POINTER(abi.SceneDesc), C.POINTER(vp)]
    L.neeref_scene_free.restype, L.neeref_scene_free.argtypes = None, [vp]
    L.neeref_render.restype = C.c_int
    L.neeref_render.argtypes = [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderOpts), vp, C.POINTER(abi.Stats), C.c_int]
    return L


def lib():
    global _lib
    if _lib is None:
        _lib = load(compile_shared("nee_ref", HERE / "nee_ref.cpp", SOURCES, FLAGS))
    return _lib


def _check(rc, L=None):
    if rc != 0:
        raise RuntimeError("next-event reference error %d: %s" % (rc, (L or lib()).neeref_last_error().decode()))


class Scene:
    """The reference's view of a scene description (a ctypes POINTER(SceneDesc) or an object with a `.desc`).
    `L`: the library to use (default: lib())."""

    def __init__(self, scene, L=None):
        self._keep = scene
        self._L = L or lib()
        self._h = C.c_void_p()
        _check(self._L.neeref_scene_create(getattr(scene, "desc", scene), C.byref(self._h)), self._L)

    def render(self, camera, width, height, sample_begin, sample_end, max_depth=50, seed=1, order=abi.ORDER_REFERENCE,
               n_threads=1, flags=abi.FLAG_NEXT_EVENT):
        """(film, stats) like oracle Scene.render, with the next-event estimator (always on; `flags` adds
        YART_FLAG_RUSSIAN_ROULETTE / DEPTH_ZERO_BLACK)."""
        film = np.zeros((height, width, 3), dtype=np.float64)
        o = abi.RenderOpts()
        o.width, o.height, o.sample_begin, o.sample_end = width, height, sample_begin, sample_end
        o.max_depth, o.order, o.batch_spp, o.flags, o.seed = max_depth, order, 0, flags, seed
        st = abi.Stats()
        _check(self._L.neeref_render(self._h, C.byref(camera), C.byref(o), film.ctypes.data, C.byref(st), n_threads), self._L)
        return film, st

    def __del__(self):
        if getattr(self, "_h", None) and getattr(self, "_L", None) is not None:
            self._L.neeref_scene_free(self._h)
            self._h = None
