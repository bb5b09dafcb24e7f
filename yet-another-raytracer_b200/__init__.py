"""yet-another-raytracer_b200 -- host-side mirror of the reference's interface over the C ABI.

The product is `libyart_b200.so` (hand-written sm_100a CUDA + a C++ host front end, built by
build.py from csrc/).  This module is the thin ctypes binding used by the tests, bench.py and
the CLI; names follow the reference (TriangleMesh.from_obj, L4QBVH, build_scene_preset,
resolve_dimensions, render ...).  There is no CPU fallback: if the shared library is missing
every entry point raises, and compute calls fail with YART_ERR_CUDA when no B200 is present.

The package name has a hyphen, so import it with
    importlib.import_module("yet-another-raytracer_b200")
"""
import ctypes as C
import gzip
import os
import shutil
from pathlib import Path

import numpy as np

from . import _abi as abi
from ._abi import (FLAG_COUNT_VISITS, FLAG_DEPTH_ZERO_BLACK, FLAG_DEVICE_PTRS, FLAG_NEXT_EVENT, FLAG_RUSSIAN_ROULETTE,
                   FLAG_UNBIASED_LIGHT_PICK, HIT_DTYPE, MISS, ORDER_NEAR, ORDER_REFERENCE, RAY_DTYPE, TARGET_WORLD,
                   make_rays)

PKG_DIR = Path(__file__).resolve().parent
REPO_ROOT = PKG_DIR.parent
LIB_PATH = Path(os.environ.get("YART_LIB_PATH", PKG_DIR / "libyart_b200.so"))  # (override: A/B builds)

SCENE_NAMES = ["random-scene", "two-spheres", "two-perlin-spheres", "earth", "simple-light", "cornell-box",
               "cornell-box-smoke", "next-week-final", "teapot", "bunny", "three-spheres", "sycee", "david"]


BUILDER_HOST, BUILDER_DEVICE = 0, 1


class YartError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("yart error %d: %s" % (code, message))
        self.code = code


_lib = None


def load_library():
    """Load libyart_b200.so (built in-tree by build.py).  Fails loudly when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError("%s is missing: run `python %s` (or __graft_entry__.build()) first; "
                          "there is no Python/CPU fallback" % (LIB_PATH, PKG_DIR / "build.py"))
    lib = C.CDLL(str(LIB_PATH))
    P = C.POINTER
    vp, u32, u64, f64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_double, C.c_int
    sig = {
        "yart_version": (C.c_char_p, []),
        "yart_last_error_global": (C.c_char_p, []),
        "yart_obj_load": (i32, [C.c_char_p, P(vp)]),
        "yart_obj_free": (None, [vp]),
        "yart_obj_trimesh": (i32, [vp, P(abi.Trimesh)]),
        "yart_qbvh_build": (i32, [P(abi.Trimesh), P(vp)]),
        "yart_qbvh_free": (None, [vp]),
        "yart_qbvh_get_info": (i32, [vp, P(abi.QbvhInfo)]),
        "yart_qbvh_nodes": (vp, [vp]),
        "yart_qbvh_tris": (vp, [vp]),
        "yart_qbvh_shade": (vp, [vp]),
        "yart_qbvh_build_device": (i32, [vp, P(abi.Trimesh), P(vp)]),
        "yart_ctx_set_builder": (i32, [vp, u32]),
        "yart_measure_fetch_peak": (i32, [vp, u64, u32, u32, P(f64)]),
        "yart_host_register": (i32, [vp, vp, u64]),
        "yart_host_unregister": (i32, [vp, vp]),
        "yart_preset_build": (i32, [C.c_char_p, C.c_char_p, u64, P(vp)]),
        "yart_preset_free": (None, [vp]),
        "yart_preset_note": (C.c_char_p, [vp]),
        "yart_preset_scene": (P(abi.SceneDesc), [vp]),
        "yart_preset_get_info": (i32, [vp, P(abi.PresetInfo)]),
        "yart_preset_count": (i32, []),
        "yart_preset_name": (C.c_char_p, [i32]),
        "yart_resolve_dimensions": (None, [u32, u32, u32, u32, P(u32), P(u32)]),
        "yart_preset_camera": (i32, [vp, u32, u32, f64, f64, P(abi.Camera)]),
        "yart_device_count": (i32, []),
        "yart_ctx_create": (i32, [i32, P(vp)]),
        "yart_ctx_destroy": (None, [vp]),
        "yart_last_error": (C.c_char_p, [vp]),
        "yart_ctx_set_stream": (i32, [vp, vp]),
        "yart_ctx_synchronize": (i32, [vp]),
        "yart_ctx_set_scene": (i32, [vp, P(abi.SceneDesc)]),
        "yart_closest_hit": (i32, [vp, u32, vp, u64, f64, f64, u32, u32, vp, P(abi.Stats)]),
        "yart_closest_hit_f32": (i32, [vp, u32, vp, u64, C.c_float, C.c_float, u32, u32, vp, P(abi.Stats)]),
        "yart_occluded": (i32, [vp, u32, vp, u64, f64, f64, u32, vp, P(abi.Stats)]),
        "yart_occluded_f32": (i32, [vp, u32, vp, u64, C.c_float, C.c_float, u32, vp, P(abi.Stats)]),
        "yart_render": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, P(abi.Stats)]),
        "yart_film_finalize": (i32, [vp, vp, u32, u32, u32, u32, vp]),
        "yart_generate_camera_rays": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, vp, vp]),
        "yart_dump_path_rays": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, u64, P(u64)]),
        "yart_comm_unique_id": (i32, [vp]),
        "yart_comm_init_rank": (i32, [vp, vp, i32, i32, P(vp)]),
        "yart_comm_init": (i32, [P(vp), i32, P(vp)]),
        "yart_comm_destroy": (None, [vp]),
        "yart_comm_info": (i32, [vp, P(i32), P(i32), P(i32), P(i32)]),
        "yart_comm_last_error": (C.c_char_p, [vp]),
        "yart_film_reduce": (i32, [vp, P(vp), u32, u32, i32]),
        "yart_film_create": (i32, [vp, u32, u32, P(vp)]),
        "yart_film_clear": (i32, [vp, vp, u32, u32]),
        "yart_film_read": (i32, [vp, vp, u32, u32, vp]),
        "yart_film_destroy": (None, [vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "yart_version", "yart_last_error_global", "yart_obj_load", "yart_obj_free", "yart_obj_trimesh", "yart_qbvh_build",
    "yart_qbvh_free", "yart_qbvh_get_info", "yart_qbvh_nodes", "yart_qbvh_tris", "yart_preset_build",
    "yart_preset_free", "yart_preset_scene", "yart_preset_get_info", "yart_preset_count", "yart_preset_name",
    "yart_resolve_dimensions", "yart_preset_camera", "yart_device_count", "yart_ctx_create", "yart_ctx_destroy",
    "yart_last_error", "yart_ctx_set_stream", "yart_ctx_synchronize", "yart_ctx_set_scene", "yart_closest_hit",
    "yart_render", "yart_film_finalize", "yart_generate_camera_rays", "yart_qbvh_shade", "yart_qbvh_build_device",
    "yart_ctx_set_builder", "yart_measure_fetch_peak", "yart_comm_unique_id", "yart_comm_init_rank", "yart_comm_init",
    "yart_comm_destroy", "yart_comm_info", "yart_comm_last_error", "yart_film_reduce", "yart_film_create",
    "yart_film_clear", "yart_film_read", "yart_film_destroy", "yart_preset_note", "yart_closest_hit_f32",
    "yart_dump_path_rays", "yart_host_register", "yart_host_unregister", "yart_occluded", "yart_occluded_f32",
]


def _check_global(rc):
    if rc != 0:
        raise YartError(rc, load_library().yart_last_error_global().decode())


def assets_dir():
    """Directory with cube.obj / david.obj / sycee.obj / earthmap_1024x512.rgb8.

    The repository ships them gzip-compressed under assets/ (they are the reference's own
    input files; /root/reference does not exist on the GPU box); they are unpacked on first use.
    """
    src = REPO_ROOT / "assets"
    dst = src / "_unpacked"
    dst.mkdir(exist_ok=True)
    for gz in sorted(src.glob("*.gz")):
        out = dst / gz.name[:-3]
        if not out.exists() or out.stat().st_mtime < gz.stat().st_mtime:
            tmp = out.with_suffix(out.suffix + ".tmp%d" % os.getpid())
            with gzip.open(gz, "rb") as fi, open(tmp, "wb") as fo:
                shutil.copyfileobj(fi, fo)
            os.replace(tmp, out)
    return str(dst)


class TriangleMesh:
    """`TriangleMesh::from_obj` (reference triangle.rs:110-175) up to the triangle list."""

    def __init__(self, handle):
        self._h = handle
        self.trimesh = abi.Trimesh()
        _check_global(load_library().yart_obj_trimesh(self._h, C.byref(self.trimesh)))

    @classmethod
    def from_obj(cls, path):
        h = C.c_void_p()
        _check_global(load_library().yart_obj_load(str(path).encode(), C.byref(h)))
        return cls(h)

    @property
    def n_tris(self):
        return int(self.trimesh.n_tris)

    def positions(self):
        return np.ctypeslib.as_array(self.trimesh.positions, shape=(self.n_tris, 3, 3)).copy()

    def normals(self):
        return np.ctypeslib.as_array(self.trimesh.normals, shape=(self.n_tris, 3, 3)).copy()

    def uvs(self):
        return np.ctypeslib.as_array(self.trimesh.uvs, shape=(self.n_tris, 3, 2)).copy()

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.yart_obj_free(self._h)
            self._h = None


def trimesh_from_arrays(positions, normals=None, uvs=None):
    """A yart_trimesh view of numpy arrays ((n,3,3) f32 positions, (n,3,3) f64 normals, (n,3,2) f32 uvs).
    Returns (trimesh, keepalive): pass keepalive wherever the view is used."""
    pos = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3, 3)
    n = pos.shape[0]
    nrm = np.ascontiguousarray(np.zeros((n, 3, 3)) if normals is None else normals, dtype=np.float64).reshape(n, 3, 3)
    uv = np.ascontiguousarray(np.zeros((n, 3, 2)) if uvs is None else uvs, dtype=np.float32).reshape(n, 3, 2)
    t = abi.Trimesh()
    t.n_tris = n
    t.positions = pos.ctypes.data_as(C.POINTER(C.c_float))
    t.normals = nrm.ctypes.data_as(C.POINTER(C.c_double))
    t.uvs = uv.ctypes.data_as(C.POINTER(C.c_float))
    return t, (pos, nrm, uv)


class L4QBVH:
    """`L4QBVH::new` (reference qbvh.rs:251-361), flattened into the device layout."""

    def __init__(self, trimesh, keepalive=None, ctx=None):
        """ctx=None: the host builder; ctx=Context: the GPU builder (same tree, byte for byte)."""
        self._keep = keepalive
        self._h = C.c_void_p()
        if ctx is None:
            _check_global(load_library().yart_qbvh_build(C.byref(trimesh), C.byref(self._h)))
        else:
            ctx._check(load_library().yart_qbvh_build_device(ctx._h, C.byref(trimesh), C.byref(self._h)))
        self.info = abi.QbvhInfo()
        _check_global(_lib.yart_qbvh_get_info(self._h, C.byref(self.info)))

    @classmethod
    def from_mesh(cls, mesh, ctx=None):
        return cls(mesh.trimesh, keepalive=mesh, ctx=ctx)

    def shade(self):
        n = self.info.n_tris
        buf = (C.c_char * (n * 96)).from_address(_lib.yart_qbvh_shade(self._h))
        return np.frombuffer(buf, dtype=np.uint8, count=n * 96).reshape(n, 96).copy()

    def nodes(self):
        n = self.info.n_nodes
        buf = (C.c_char * (n * 128)).from_address(_lib.yart_qbvh_nodes(self._h))
        return np.frombuffer(buf, dtype=abi.NODE_DTYPE, count=n).copy()

    def tris(self):
        n = self.info.n_tris
        buf = (C.c_char * (n * 48)).from_address(_lib.yart_qbvh_tris(self._h))
        return np.frombuffer(buf, dtype=abi.TRI_DTYPE, count=n).copy()

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.yart_qbvh_free(self._h)
            self._h = None


def resolve_dimensions(default_width, default_height, width_override=None, height_override=None):
    """`resolve_dimensions` (reference main.rs:166-186)."""
    w, h = C.c_uint32(), C.c_uint32()
    load_library().yart_resolve_dimensions(default_width, default_height, width_override or 0, height_override or 0,
                                           C.byref(w), C.byref(h))
    return int(w.value), int(h.value)


class ScenePreset:
    """`build_scene_preset` (reference main.rs:211-432): world, sampling lights, camera, defaults."""

    def __init__(self, name, assets=None, seed=1):
        self.name = name
        self._h = C.c_void_p()
        _check_global(load_library().yart_preset_build(name.encode(), (assets or assets_dir()).encode(), seed,
                                                       C.byref(self._h)))
        self.info = abi.PresetInfo()
        _check_global(_lib.yart_preset_get_info(self._h, C.byref(self.info)))
        self.desc = _lib.yart_preset_scene(self._h)  # POINTER(SceneDesc), borrowed
        self.note = _lib.yart_preset_note(self._h).decode()  # "" or e.g. "bunny.obj is not shipped ...: sycee.obj stands in"

    def camera(self, width, height, vfov=None, aperture=None):
        cam = abi.Camera()
        _check_global(_lib.yart_preset_camera(self._h, width, height, -1.0 if vfov is None else vfov,
                                              -1.0 if aperture is None else aperture, C.byref(cam)))
        return cam

    def resolve_render_options(self, output=None, width=None, height=None, samples=None, max_depth=None,
                               workers=None, vfov=None, aperture=None):
        """`resolve_render_options` (reference main.rs:188-209)."""
        w, h = resolve_dimensions(self.info.width, self.info.height, width, height)
        return {
            "output_path": output or os.path.join("output", self.info.output_filename.decode()),
            "width": w, "height": h,
            "samples_per_pixel": samples or self.info.samples_per_pixel,
            "max_depth": max_depth or self.info.max_depth,
            "workers": workers or self.info.workers,
            "vfov": self.info.vfov if vfov is None else vfov,
            "aperture": self.info.aperture if aperture is None else aperture,
        }

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.yart_preset_free(self._h)
            self._h = None


def device_count():
    return int(load_library().yart_device_count())


class Context:
    """One GPU.  Not thread-safe; N GPUs = N contexts (one process per GPU in bench.py)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check_global(load_library().yart_ctx_create(device, C.byref(self._h)))
        self.device = device
        self._scene_keep = None

    def _check(self, rc):
        if rc != 0:
            raise YartError(rc, _lib.yart_last_error(self._h).decode())

    def set_scene(self, scene):
        """scene: a ScenePreset or a ctypes pointer to SceneDesc."""
        desc = scene.desc if isinstance(scene, ScenePreset) else scene
        self._scene_keep = scene
        self._check(_lib.yart_ctx_set_scene(self._h, desc))

    def set_builder(self, builder):
        """BUILDER_DEVICE (default) or BUILDER_HOST: which L4QBVH builder set_scene uses for meshes."""
        self._check(_lib.yart_ctx_set_builder(self._h, builder))

    def measure_fetch_peak(self, table_bytes, fetches_per_thread=2048, mode=0):
        """Sustained GB/s of random whole-line (128 B) fetches from a table of this size (roofline denominator)."""
        out = C.c_double()
        self._check(_lib.yart_measure_fetch_peak(self._h, int(table_bytes), int(fetches_per_thread), int(mode), C.byref(out)))
        return float(out.value)

    def set_stream(self, cuda_stream_ptr):
        self._check(_lib.yart_ctx_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def synchronize(self):
        self._check(_lib.yart_ctx_synchronize(self._h))

    def closest_hit(self, rays, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"), order=ORDER_REFERENCE,
                    count_visits=False, hits=None):
        """Batched `Hittable::hit` (reference hittable.rs:24) with host buffers (`hits`: an optional preallocated --
        e.g. pinned -- output array)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        if hits is None:
            hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        assert hits.dtype == HIT_DTYPE and hits.shape == (rays.shape[0],) and hits.flags.c_contiguous
        st = abi.Stats()
        flags = FLAG_COUNT_VISITS if count_visits else 0
        self._check(_lib.yart_closest_hit(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, order, flags,
                                          hits.ctypes.data, C.byref(st)))
        return hits, st

    def closest_hit_f32(self, rays, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"), order=ORDER_REFERENCE,
                        count_visits=False, hits=None):
        """yart_closest_hit_f32 with host buffers: rays is an array of abi.RAY_F32_DTYPE (hits: an optional caller-owned
        output array, e.g. in pinned memory)."""
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_F32_DTYPE)
        if hits is None:
            hits = np.empty(rays.shape[0], dtype=abi.HIT_F32_DTYPE)
        elif hits.dtype != abi.HIT_F32_DTYPE or hits.shape != (rays.shape[0],) or not hits.flags.c_contiguous:
            raise ValueError("hits must be a contiguous abi.HIT_F32_DTYPE array as long as rays")
        st = abi.Stats()
        flags = FLAG_COUNT_VISITS if count_visits else 0
        self._check(_lib.yart_closest_hit_f32(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, order, flags,
                                              hits.ctypes.data, C.byref(st)))
        return hits, st

    def closest_hit_f32_device(self, rays_ptr, n, hits_ptr, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"),
                               order=ORDER_REFERENCE, count_visits=False):
        st = abi.Stats()
        flags = FLAG_DEVICE_PTRS | (FLAG_COUNT_VISITS if count_visits else 0)
        self._check(_lib.yart_closest_hit_f32(self._h, target, C.c_void_p(rays_ptr), n, t_min, t_max, order, flags,
                                              C.c_void_p(hits_ptr), C.byref(st)))
        return st

    def host_register(self, array):
        """Page-lock a numpy array in place (yart_host_register); pair with host_unregister before the array dies."""
        self._check(_lib.yart_host_register(self._h, C.c_void_p(array.ctypes.data), array.nbytes))

    def host_unregister(self, array):
        self._check(_lib.yart_host_unregister(self._h, C.c_void_p(array.ctypes.data)))

    def closest_hit_device(self, rays_ptr, n, hits_ptr, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"),
                           order=ORDER_REFERENCE, count_visits=False):
        """Same with device pointers (e.g. torch tensors' data_ptr()) -- nothing crosses PCIe."""
        st = abi.Stats()
        flags = FLAG_DEVICE_PTRS | (FLAG_COUNT_VISITS if count_visits else 0)
        self._check(_lib.yart_closest_hit(self._h, target, C.c_void_p(rays_ptr), n, t_min, t_max, order, flags,
                                          C.c_void_p(hits_ptr), C.byref(st)))
        return st

    def occluded(self, rays, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"), out=None):
        """Batched occlusion query (yart_occluded) with host buffers: (bool array, stats); True where the ray hits
        anything in (t_min, t_max) -- exactly where closest_hit(..., ORDER_REFERENCE) reports a hit.  `out`: an
        optional preallocated (e.g. pinned) uint8 array as long as rays."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = self._occluded_out(out, rays.shape[0])
        st = abi.Stats()
        self._check(_lib.yart_occluded(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, 0,
                                       out.ctypes.data, C.byref(st)))
        return out.view(np.bool_), st

    def occluded_f32(self, rays, target=TARGET_WORLD, t_min=0.001, t_max=float("inf"), out=None):
        """yart_occluded_f32 with host buffers: rays is an array of abi.RAY_F32_DTYPE."""
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_F32_DTYPE)
        out = self._occluded_out(out, rays.shape[0])
        st = abi.Stats()
        self._check(_lib.yart_occluded_f32(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, 0,
                                           out.ctypes.data, C.byref(st)))
        return out.view(np.bool_), st

    @staticmethod
    def _occluded_out(out, n):
        if out is None:
            return np.empty(n, dtype=np.uint8)
        if out.dtype != np.uint8 or out.shape != (n,) or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous uint8 array as long as rays")
        return out

    def occluded_device(self, rays_ptr, n, out_ptr, target=TARGET_WORLD, t_min=0.001, t_max=float("inf")):
        """Same with device pointers: rays (yart_ray records) and out (n bytes) on this context's GPU."""
        st = abi.Stats()
        self._check(_lib.yart_occluded(self._h, target, C.c_void_p(rays_ptr), n, t_min, t_max, FLAG_DEVICE_PTRS,
                                       C.c_void_p(out_ptr), C.byref(st)))
        return st

    def occluded_f32_device(self, rays_ptr, n, out_ptr, target=TARGET_WORLD, t_min=0.001, t_max=float("inf")):
        st = abi.Stats()
        self._check(_lib.yart_occluded_f32(self._h, target, C.c_void_p(rays_ptr), n, t_min, t_max, FLAG_DEVICE_PTRS,
                                           C.c_void_p(out_ptr), C.byref(st)))
        return st

    def _opts(self, width, height, sample_begin, sample_end, max_depth, seed, order, batch_spp, flags):
        o = abi.RenderOpts()
        o.width, o.height = width, height
        o.sample_begin, o.sample_end = sample_begin, sample_end
        o.max_depth, o.order, o.batch_spp, o.flags, o.seed = max_depth, order, batch_spp, flags, seed
        return o

    def render(self, camera, width, height, sample_begin, sample_end, max_depth=50, seed=1, order=ORDER_NEAR,
               batch_spp=0, film=None, count_visits=False, flags=0):
        """Batched sample loop of `render` (reference main.rs:650-708).  Returns (film, stats);
        film is the (H, W, 3) f64 sum of sanitised XYZ samples (continued if `film` is given;
        pass a pinned buffer for fast host<->device copies)."""
        if film is None:
            film = np.zeros((height, width, 3), dtype=np.float64)
        assert film.dtype == np.float64 and film.shape == (height, width, 3) and film.flags.c_contiguous
        st = abi.Stats()
        o = self._opts(width, height, sample_begin, sample_end, max_depth, seed, order, batch_spp,
                       (FLAG_COUNT_VISITS if count_visits else 0) | flags)
        self._check(_lib.yart_render(self._h, C.byref(camera), C.byref(o), film.ctypes.data, C.byref(st)))
        return film, st

    def render_device(self, camera, width, height, sample_begin, sample_end, film_ptr, max_depth=50, seed=1,
                      order=ORDER_NEAR, batch_spp=0, count_visits=False, flags=0):
        st = abi.Stats()
        o = self._opts(width, height, sample_begin, sample_end, max_depth, seed, order, batch_spp,
                       FLAG_DEVICE_PTRS | (FLAG_COUNT_VISITS if count_visits else 0) | flags)
        self._check(_lib.yart_render(self._h, C.byref(camera), C.byref(o), C.c_void_p(film_ptr), C.byref(st)))
        return st

    def film_finalize(self, film, spp):
        """Per-pixel finalisation (reference main.rs:710-718) -> (H, W, 4) u8."""
        film = np.ascontiguousarray(film, dtype=np.float64)
        h, w = film.shape[:2]
        rgba = np.empty((h, w, 4), dtype=np.uint8)
        self._check(_lib.yart_film_finalize(self._h, film.ctypes.data, w, h, spp, 0, rgba.ctypes.data))
        return rgba

    def film_finalize_device(self, film_ptr, width, height, spp, rgba_ptr):
        """Same with device pointers (film: [h][w][3] f64, rgba: [h][w][4] u8); asynchronous work is synchronised."""
        self._check(_lib.yart_film_finalize(self._h, C.c_void_p(film_ptr), width, height, spp, FLAG_DEVICE_PTRS,
                                            C.c_void_p(rgba_ptr)))

    def camera_rays(self, camera, width, height, sample_begin, sample_end, seed=1):
        n = width * height * (sample_end - sample_begin)
        rays = np.empty(n, dtype=RAY_DTYPE)
        wl = np.empty(n, dtype=np.float64)
        tm = np.empty(n, dtype=np.float64)
        o = self._opts(width, height, sample_begin, sample_end, 1, seed, ORDER_REFERENCE, 0, 0)
        self._check(_lib.yart_generate_camera_rays(self._h, C.byref(camera), C.byref(o), rays.ctypes.data,
                                                   wl.ctypes.data, tm.ctypes.data))
        return rays, wl, tm

    def dump_path_rays(self, camera, width, height, sample_begin, sample_end, cap, max_depth=50, seed=1, batch_spp=0,
                       out_ptr=None, flags=0):
        """Every ray the renderer traces for these samples, in wavefront order (yart_dump_path_rays).  Returns
        (rays[:min(n, cap)], n) with host output, or n alone when out_ptr (a device pointer with room for cap) is given."""
        n = C.c_uint64()
        if out_ptr is not None:
            o = self._opts(width, height, sample_begin, sample_end, max_depth, seed, ORDER_NEAR, batch_spp, FLAG_DEVICE_PTRS | flags)
            self._check(_lib.yart_dump_path_rays(self._h, C.byref(camera), C.byref(o), C.c_void_p(out_ptr), cap, C.byref(n)))
            return int(n.value)
        rays = np.empty(cap, dtype=RAY_DTYPE)
        o = self._opts(width, height, sample_begin, sample_end, max_depth, seed, ORDER_NEAR, batch_spp, flags)
        self._check(_lib.yart_dump_path_rays(self._h, C.byref(camera), C.byref(o), rays.ctypes.data, cap, C.byref(n)))
        return rays[:min(int(n.value), cap)], int(n.value)

    # ---- device-resident films (what the multi-GPU reduce operates on) ----
    def film_create(self, width, height):
        """A zeroed [height][width][3] f64 film on this context's GPU; returns the device pointer (int)."""
        p = C.c_void_p()
        self._check(_lib.yart_film_create(self._h, width, height, C.byref(p)))
        return p.value

    def film_clear(self, film_ptr, width, height):
        self._check(_lib.yart_film_clear(self._h, C.c_void_p(film_ptr), width, height))

    def film_read(self, film_ptr, width, height, out=None):
        if out is None:
            out = np.empty((height, width, 3), dtype=np.float64)
        assert out.dtype == np.float64 and out.shape == (height, width, 3) and out.flags.c_contiguous
        self._check(_lib.yart_film_read(self._h, C.c_void_p(film_ptr), width, height, out.ctypes.data))
        return out

    def film_destroy(self, film_ptr):
        if getattr(self, "_h", None) and _lib is not None and film_ptr:
            _lib.yart_film_destroy(self._h, C.c_void_p(film_ptr))

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.yart_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


COMM_ID_BYTES = 128


def _share_the_python_hosts_nccl():
    """A Python host usually also carries PyTorch, whose libtorch_cuda needs ITS bundled libnccl.so.2 (the
    nvidia-nccl wheel).  If our library bound the system's older copy first, a later `import torch` would fail on
    missing symbols -- so point the library's run-time loader (YART_NCCL_LIB, csrc/device_comm.cu) at the wheel's
    copy when there is one and the user has not chosen otherwise.  (The library itself first reuses any libnccl the
    process has already loaded.)"""
    if os.environ.get("YART_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (spec.submodule_search_locations if spec else []):
            cand = Path(base) / "lib" / "libnccl.so.2"
            if cand.exists():
                os.environ["YART_NCCL_LIB"] = str(cand)
                return
    except Exception:  # noqa: BLE001 -- no wheel: the system library is used
        pass


def comm_unique_id():
    """ncclGetUniqueId through the C ABI: 128 bytes rank 0 ships to the other ranks (any transport)."""
    _share_the_python_hosts_nccl()
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    _check_global(load_library().yart_comm_unique_id(buf))
    return bytes(buf)


class Comm:
    """The multi-GPU group of the C ABI: sample-range sharding + one in-place NCCL reduce of the f64 film
    (the replacement of the reference's tile gather, main.rs:746-760).

    Comm.from_id(ctx, id, rank, n_ranks): one process per GPU;  Comm.from_contexts([ctx0, ctx1, ...]): one process."""

    def __init__(self, handle, contexts):
        self._h = handle
        self.contexts = list(contexts)

    @classmethod
    def from_id(cls, ctx, unique_id, rank, n_ranks):
        assert len(unique_id) == COMM_ID_BYTES
        _share_the_python_hosts_nccl()
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        h = C.c_void_p()
        ctx._check(load_library().yart_comm_init_rank(ctx._h, buf, rank, n_ranks, C.byref(h)))
        return cls(h, [ctx])

    @classmethod
    def from_contexts(cls, contexts):
        _share_the_python_hosts_nccl()
        arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
        h = C.c_void_p()
        _check_global(load_library().yart_comm_init(arr, len(contexts), C.byref(h)))
        return cls(h, contexts)

    def info(self):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _check_global(_lib.yart_comm_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"n_ranks": a.value, "n_local": b.value, "first_local_rank": c.value, "nccl_version": d.value}

    def film_reduce(self, film_ptrs, width, height, root=0):
        """Sum the films onto `root` (root < 0: onto every rank), in place, asynchronous on each context's stream.
        film_ptrs: one device pointer per local rank (an int is accepted for the one-rank-per-process case)."""
        if isinstance(film_ptrs, int):
            film_ptrs = [film_ptrs]
        arr = (C.c_void_p * len(film_ptrs))(*film_ptrs)
        rc = _lib.yart_film_reduce(self._h, arr, width, height, root)
        if rc != 0:
            raise YartError(rc, _lib.yart_comm_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.yart_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()
