"""ctypes binding of the CPU oracle (oracle/yart_oracle.cpp) + an independent numpy OBJ reader.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
PARITY: unpinned by the reference at the level of single hits / samples (the Rust reference cannot be built
here); pinned at image level by digests of the reference's own shipped renders (see yart_oracle.h).
"""
import ctypes as C
import importlib
import subprocess
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
LIB_PATH = HERE / "_build" / "liboracle.so"

if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
abi = importlib.import_module("yet-another-raytracer_b200._abi")  # struct declarations only


def build(force=False):
    """Compile the oracle with the committed Makefile (gcc only, no CUDA)."""
    if force and LIB_PATH.exists():
        LIB_PATH.unlink()
    res = subprocess.run(["make", "-C", str(HERE)], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)
    return str(LIB_PATH)


class QbvhInfo(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("n_leaves", C.c_uint32), ("n_tris", C.c_uint32),
                ("max_stack_seen", C.c_uint32), ("leaves_by_count", C.c_uint32 * 5), ("empty_children", C.c_uint32),
                ("bbox_min", C.c_double * 3), ("bbox_max", C.c_double * 3)]


class Counters(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("node_visits", C.c_uint64), ("leaf_visits", C.c_uint64),
                ("tri_tests", C.c_uint64), ("max_stack", C.c_uint64)]


_lib = None


def lib():
    """The default build, oracle/_build/liboracle.so (built on first use)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            build()
        _lib = load(LIB_PATH)
    return _lib


def load(path):
    """A library of the oracle's API at `path` (the default build or a variant of it, tests/perturbed_oracle.py),
    with its signatures declared."""
    L = C.CDLL(str(path))
    P, vp, u32, u64, f64, i32 = C.POINTER, C.c_void_p, C.c_uint32, C.c_uint64, C.c_double, C.c_int
    sig = {
        "orc_last_error": (C.c_char_p, []),
        "orc_scene_create": (i32, [P(abi.SceneDesc), P(vp)]),
        "orc_scene_free": (None, [vp]),
        "orc_qbvh_info_get": (i32, [vp, u32, P(QbvhInfo)]),
        "orc_qbvh_node": (i32, [vp, u32, u32, vp, vp, vp]),
        "orc_qbvh_tri_order": (i32, [vp, u32, vp]),
        "orc_closest_hit": (i32, [vp, u32, vp, u64, f64, f64, u32, vp, P(Counters), i32]),
        "orc_brute_force_hit": (i32, [vp, u32, vp, u64, f64, f64, vp, vp]),
        "orc_tie_set": (i32, [vp, u32, vp, f64, f64, vp, u32, P(u32)]),
        "orc_render": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, P(abi.Stats), i32]),
        "orc_render_tiles": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, P(abi.Stats), i32, u32, u32]),
        "orc_film_finalize": (i32, [vp, u32, u32, u32, vp]),
        "orc_camera_rays": (i32, [P(abi.Camera), P(abi.RenderOpts), vp, vp, vp]),
        "orc_dump_path_rays": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), vp, u64, P(u64)]),
        "orc_sample": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), u32, u32, vp, P(u32)]),
        "orc_sample_path": (i32, [vp, P(abi.Camera), P(abi.RenderOpts), u32, u32, vp, u64, P(u64)]),
        "orc_sanitize_sample_xyz": (None, [vp, vp]),
        "orc_clamp_display_channel": (C.c_uint8, [f64]),
        "orc_gamma_corrected": (None, [vp, vp]),
        "orc_rgb_reflect": (f64, [vp, f64]),
        "orc_xyz_from_wavelength": (None, [f64, vp]),
        "orc_xyz_into_rgb": (None, [vp, vp]),
        "orc_sellmeier_index": (f64, [P(abi.Material), f64]),
        "orc_push_hit_children": (i32, [vp, P(u32), vp, vp, vp]),
        "orc_philox4x32_10": (None, [vp, vp, vp]),
        "orc_uniform2": (None, [u64, u32, u32, u32, u32, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    return L


def _check(rc, L=None):
    if rc != 0:
        raise RuntimeError("oracle error %d: %s" % (rc, (L or lib()).orc_last_error().decode()))


def _opts(width, height, sample_begin, sample_end, max_depth, seed, order, flags=0):
    o = abi.RenderOpts()
    o.width, o.height = width, height
    o.sample_begin, o.sample_end = sample_begin, sample_end
    o.max_depth, o.order, o.batch_spp, o.flags, o.seed = max_depth, order, 0, flags, seed
    return o


class Scene:
    """The oracle's view of a scene description (a ctypes POINTER(SceneDesc) or a ScenePreset-like
    object with a `.desc`).  `L`: the library to use (default: lib())."""

    def __init__(self, scene, L=None):
        self._keep = scene
        self._L = L or lib()
        desc = getattr(scene, "desc", scene)
        self._h = C.c_void_p()
        self._check(self._L.orc_scene_create(desc, C.byref(self._h)))

    def _check(self, rc):
        _check(rc, self._L)

    def qbvh_info(self, mesh=0):
        info = QbvhInfo()
        self._check(self._L.orc_qbvh_info_get(self._h, mesh, C.byref(info)))
        return info

    def qbvh_node(self, mesh, i):
        boxes = np.empty(24, dtype=np.float64)
        children = np.empty(4, dtype=np.uint32)
        axes = np.empty(3, dtype=np.uint32)
        self._check(self._L.orc_qbvh_node(self._h, mesh, i, boxes.ctypes.data, children.ctypes.data, axes.ctypes.data))
        return boxes, children, axes

    def tri_order(self, mesh=0):
        out = np.empty(self.qbvh_info(mesh).n_tris, dtype=np.uint32)
        self._check(self._L.orc_qbvh_tri_order(self._h, mesh, out.ctypes.data))
        return out

    def closest_hit(self, rays, target=abi.TARGET_WORLD, t_min=0.001, t_max=float("inf"), order=abi.ORDER_REFERENCE,
                    n_threads=1):
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=abi.HIT_DTYPE)
        cnt = Counters()
        self._check(self._L.orc_closest_hit(self._h, target, rays.ctypes.data, rays.shape[0], t_min, t_max, order,
                                            hits.ctypes.data, C.byref(cnt), n_threads))
        return hits, cnt

    def brute_force_hit(self, rays, mesh=0, t_min=0.001, t_max=float("inf")):
        rays = np.ascontiguousarray(rays, dtype=abi.RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=abi.HIT_DTYPE)
        ties = np.empty(rays.shape[0], dtype=np.uint32)
        self._check(self._L.orc_brute_force_hit(self._h, mesh, rays.ctypes.data, rays.shape[0], t_min, t_max,
                                                hits.ctypes.data, ties.ctypes.data))
        return hits, ties

    def tie_set(self, ray, mesh=0, t_min=0.001, t_max=float("inf")):
        ray = np.ascontiguousarray(ray, dtype=abi.RAY_DTYPE).reshape(1)
        ids = np.empty(64, dtype=np.uint32)
        n = C.c_uint32()
        self._check(self._L.orc_tie_set(self._h, mesh, ray.ctypes.data, t_min, t_max, ids.ctypes.data, 64, C.byref(n)))
        return ids[:min(n.value, 64)].copy()

    def render(self, camera, width, height, sample_begin, sample_end, max_depth=50, seed=1, order=abi.ORDER_REFERENCE,
               n_threads=1, film=None, tiles=(0, 64), flags=0):
        if film is None:
            film = np.zeros((height, width, 3), dtype=np.float64)
        st = abi.Stats()
        o = _opts(width, height, sample_begin, sample_end, max_depth, seed, order, flags)
        self._check(self._L.orc_render_tiles(self._h, C.byref(camera), C.byref(o), film.ctypes.data, C.byref(st), n_threads,
                                             tiles[0], tiles[1]))
        return film, st

    def dump_path_rays(self, camera, width, height, sample_begin, sample_end, cap, max_depth=50, seed=1):
        rays = np.empty(cap, dtype=abi.RAY_DTYPE)
        n = C.c_uint64()
        o = _opts(width, height, sample_begin, sample_end, max_depth, seed, abi.ORDER_REFERENCE)
        self._check(self._L.orc_dump_path_rays(self._h, C.byref(camera), C.byref(o), rays.ctypes.data, cap, C.byref(n)))
        return rays[:n.value].copy()

    def sample_path(self, camera, width, height, pixel, sample, max_depth=50, seed=1, order=abi.ORDER_REFERENCE, flags=0):
        rays = np.empty(max_depth + 1, dtype=abi.RAY_DTYPE)
        n = C.c_uint64()
        o = _opts(width, height, sample, sample + 1, max_depth, seed, order, flags)
        self._check(self._L.orc_sample_path(self._h, C.byref(camera), C.byref(o), pixel, sample, rays.ctypes.data, len(rays),
                                            C.byref(n)))
        return rays[:n.value].copy()

    def sample(self, camera, width, height, pixel, sample, max_depth=50, seed=1, order=abi.ORDER_REFERENCE, flags=0):
        """(unsanitised XYZ, ray count) of one (pixel, sample), pixel = y * width + x."""
        xyz = np.empty(3, dtype=np.float64)
        nr = C.c_uint32()
        o = _opts(width, height, sample, sample + 1, max_depth, seed, order, flags)
        self._check(self._L.orc_sample(self._h, C.byref(camera), C.byref(o), pixel, sample, xyz.ctypes.data, C.byref(nr)))
        return xyz, nr.value

    def __del__(self):
        if getattr(self, "_h", None) and getattr(self, "_L", None) is not None:
            self._L.orc_scene_free(self._h)
            self._h = None


def camera_rays(camera, width, height, sample_begin, sample_end, seed=1):
    n = width * height * (sample_end - sample_begin)
    rays = np.empty(n, dtype=abi.RAY_DTYPE)
    wl = np.empty(n, dtype=np.float64)
    tm = np.empty(n, dtype=np.float64)
    o = _opts(width, height, sample_begin, sample_end, 1, seed, 0)
    _check(lib().orc_camera_rays(C.byref(camera), C.byref(o), rays.ctypes.data, wl.ctypes.data, tm.ctypes.data))
    return rays, wl, tm


def film_finalize(film, spp):
    film = np.ascontiguousarray(film, dtype=np.float64)
    h, w = film.shape[:2]
    rgba = np.empty((h, w, 4), dtype=np.uint8)
    _check(lib().orc_film_finalize(film.ctypes.data, w, h, spp, rgba.ctypes.data))
    return rgba


# ------------------------------------------------------------------------------------------
# scene descriptions built in Python (for tests that do not go through a preset)
# ------------------------------------------------------------------------------------------
class MeshScene:
    """A one-mesh scene description (a single un-wrapped MESH object with a Lambertian)."""

    def __init__(self, positions, normals, uvs):
        self.positions = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3, 3)
        self.normals = np.ascontiguousarray(normals, dtype=np.float64).reshape(-1, 3, 3)
        self.uvs = np.ascontiguousarray(uvs, dtype=np.float32).reshape(-1, 3, 2)
        self.trimesh = abi.Trimesh()
        self.trimesh.n_tris = self.positions.shape[0]
        self.trimesh.positions = self.positions.ctypes.data_as(C.POINTER(C.c_float))
        self.trimesh.normals = self.normals.ctypes.data_as(C.POINTER(C.c_double))
        self.trimesh.uvs = self.uvs.ctypes.data_as(C.POINTER(C.c_float))
        self.tex = abi.Texture()
        self.tex.kind = abi.TEX_SOLID
        self.tex.rgb_a[:] = [0.5, 0.5, 0.5]
        self.mat = abi.Material()
        self.mat.kind = abi.MAT_LAMBERTIAN
        self.obj = abi.Object()
        self.obj.kind = abi.OBJ_MESH
        self.obj.cos_theta = 1.0
        self.sd = abi.SceneDesc()
        self.sd.objects, self.sd.n_objects = C.pointer(self.obj), 1
        self.sd.meshes, self.sd.n_meshes = C.pointer(self.trimesh), 1
        self.sd.materials, self.sd.n_materials = C.pointer(self.mat), 1
        self.sd.textures, self.sd.n_textures = C.pointer(self.tex), 1
        self.desc = C.pointer(self.sd)


# ------------------------------------------------------------------------------------------
# independent OBJ reader (numpy / pure Python): pins the product's C++ loader
# ------------------------------------------------------------------------------------------
def load_obj_numpy(path):
    """tobj GPU_LOAD_OPTIONS semantics restated independently of csrc/host_obj.cpp: f32 attributes,
    fan triangulation from the first corner, per-corner v/vt/vn, face-normal / (0,0) fallbacks
    (reference triangle.rs:110-168).  Returns (positions f32 [n,3,3], normals f64 [n,3,3],
    uvs f32 [n,3,2])."""
    v, vt, vn = [], [], []
    tri_v, tri_t, tri_n = [], [], []
    with open(path, "r") as f:
        for line in f:
            s = line.split()
            if not s:
                continue
            if s[0] == "v":
                v.append(s[1:4])
            elif s[0] == "vt":
                vt.append((s[1], s[2] if len(s) > 2 else "0"))
            elif s[0] == "vn":
                vn.append(s[1:4])
            elif s[0] == "f":
                corners = []
                for tok in s[1:]:
                    parts = tok.split("/")
                    iv = int(parts[0])
                    it = int(parts[1]) if len(parts) > 1 and parts[1] else 0
                    inn = int(parts[2]) if len(parts) > 2 and parts[2] else 0
                    fix = lambda i, n: i - 1 if i > 0 else (n + i if i < 0 else -1)
                    corners.append((fix(iv, len(v)), fix(it, len(vt)), fix(inn, len(vn))))
                for k in range(1, len(corners) - 1):
                    for c in (corners[0], corners[k], corners[k + 1]):
                        tri_v.append(c[0])
                        tri_t.append(c[1])
                        tri_n.append(c[2])
    V = np.array(v, dtype=np.float32)  # numpy parses decimal strings correctly rounded to f32
    pos = V[np.array(tri_v)].reshape(-1, 3, 3)
    n = pos.shape[0]
    p64 = pos.astype(np.float64)
    e1, e2 = p64[:, 1] - p64[:, 0], p64[:, 2] - p64[:, 0]
    cx = e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1]
    cy = e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2]
    cz = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
    ln = np.sqrt(cx * cx + cy * cy + cz * cz)
    with np.errstate(invalid="ignore", divide="ignore"):
        face_n = np.stack([cx / ln, cy / ln, cz / ln], axis=1)
    normals = np.repeat(face_n[:, None, :], 3, axis=1)
    tn = np.array(tri_n).reshape(-1, 3)
    if vn:
        N = np.array(vn, dtype=np.float32).astype(np.float64)
        has = tn >= 0
        normals[has] = N[tn[has]]
    uvs = np.zeros((n, 3, 2), dtype=np.float32)
    tt = np.array(tri_t).reshape(-1, 3)
    if vt:
        T = np.array(vt, dtype=np.float32)
        has = tt >= 0
        uvs[has] = T[tt[has]]
    return pos, normals, uvs
