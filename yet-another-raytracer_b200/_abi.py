"""ctypes mirror of include/yart.h (declarations only -- loads nothing).

Kept in one place so the product binding and the test-side oracle binding describe the same
plain-C structs.
"""
import ctypes as C

import numpy as np

YART_OK = 0
YART_ERR_INVALID, YART_ERR_CUDA, YART_ERR_NOMEM, YART_ERR_IO, YART_ERR_UNSUPPORTED = -1, -2, -3, -4, -5

(OBJ_SPHERE, OBJ_MOVING_SPHERE, OBJ_XY_RECT, OBJ_XZ_RECT, OBJ_YZ_RECT, OBJ_BOX, OBJ_TRIANGLE, OBJ_MESH,
 OBJ_GROUP) = range(9)
WRAP_ROTATE_Y, WRAP_TRANSLATE, WRAP_FLIP_FACE, WRAP_MEDIUM = 1, 2, 4, 8
MAT_NONE, MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_DIFFUSE_LIGHT, MAT_ISOTROPIC = range(6)
TEX_SOLID, TEX_CHECKER, TEX_NOISE, TEX_IMAGE = range(4)
NOISE_SQUARE, NOISE_TRILINEAR, NOISE_SMOOTH, NOISE_MARBLE, NOISE_NET = range(5)
ORDER_REFERENCE, ORDER_NEAR = 0, 1
FLAG_DEVICE_PTRS, FLAG_COUNT_VISITS = 1, 2
FLAG_UNBIASED_LIGHT_PICK, FLAG_RUSSIAN_ROULETTE, FLAG_DEPTH_ZERO_BLACK = 4, 8, 16
FLAG_NEXT_EVENT = 32
TARGET_WORLD = 0xFFFFFFFF
MISS = 0xFFFFFFFF


class Trimesh(C.Structure):
    _fields_ = [("n_tris", C.c_uint32), ("_pad", C.c_uint32), ("positions", C.POINTER(C.c_float)),
                ("normals", C.POINTER(C.c_double)), ("uvs", C.POINTER(C.c_float))]


class Object(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("wrap", C.c_uint32), ("material", C.c_uint32), ("index", C.c_uint32),
                ("p", C.c_double * 24), ("sin_theta", C.c_double), ("cos_theta", C.c_double),
                ("offset", C.c_double * 3), ("neg_inv_density", C.c_double)]


class Group(C.Structure):
    _fields_ = [("members", C.POINTER(Object)), ("n_members", C.c_uint32), ("_pad", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("texture", C.c_uint32), ("fuzz", C.c_double),
                ("sellmeier_b", C.c_double * 3), ("sellmeier_c", C.c_double * 3)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("noise_type", C.c_uint32), ("perlin", C.c_uint32), ("image", C.c_uint32),
                ("rgb_a", C.c_double * 3), ("rgb_b", C.c_double * 3), ("scale", C.c_double)]


class Perlin(C.Structure):
    _fields_ = [("ranfloat", C.c_double * 256), ("ranvec", (C.c_double * 3) * 256), ("perm_x", C.c_int32 * 256),
                ("perm_y", C.c_int32 * 256), ("perm_z", C.c_int32 * 256)]


class Image(C.Structure):
    _fields_ = [("rgb8", C.POINTER(C.c_uint8)), ("width", C.c_uint32), ("height", C.c_uint32)]


class SceneDesc(C.Structure):
    _fields_ = [("objects", C.POINTER(Object)), ("n_objects", C.c_uint32), ("_p0", C.c_uint32),
                ("lights", C.POINTER(Object)), ("n_lights", C.c_uint32), ("_p1", C.c_uint32),
                ("meshes", C.POINTER(Trimesh)), ("n_meshes", C.c_uint32), ("_p2", C.c_uint32),
                ("groups", C.POINTER(Group)), ("n_groups", C.c_uint32), ("_p3", C.c_uint32),
                ("materials", C.POINTER(Material)), ("n_materials", C.c_uint32), ("_p4", C.c_uint32),
                ("textures", C.POINTER(Texture)), ("n_textures", C.c_uint32), ("_p5", C.c_uint32),
                ("perlins", C.POINTER(Perlin)), ("n_perlins", C.c_uint32), ("_p6", C.c_uint32),
                ("images", C.POINTER(Image)), ("n_images", C.c_uint32), ("_p7", C.c_uint32),
                ("background_rgb", C.c_double * 3)]


class Camera(C.Structure):
    _fields_ = [("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3), ("vup", C.c_double * 3),
                ("vfov_degrees", C.c_double), ("aspect_ratio", C.c_double), ("aperture", C.c_double),
                ("focus_dist", C.c_double), ("time0", C.c_double), ("time1", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("paths", C.c_uint64), ("node_visits", C.c_uint64), ("tri_tests", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("gpu_ms", C.c_double), ("trace_ms", C.c_double),
                ("max_bounce", C.c_uint32), ("trace_launches", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if not k.startswith("_")}


class RenderOpts(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("sample_begin", C.c_uint32),
                ("sample_end", C.c_uint32), ("max_depth", C.c_uint32), ("order", C.c_uint32),
                ("batch_spp", C.c_uint32), ("flags", C.c_uint32), ("seed", C.c_uint64)]


class AovPlanes(C.Structure):
    _fields_ = [("albedo", C.c_void_p), ("normal", C.c_void_p), ("depth", C.c_void_p)]


class DenoiseOpts(C.Structure):
    _fields_ = [("levels", C.c_uint32), ("flags", C.c_uint32), ("sigma_color", C.c_double), ("sigma_normal", C.c_double),
                ("sigma_depth", C.c_double)]


class QbvhInfo(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("n_leaves", C.c_uint32), ("n_tris", C.c_uint32), ("height", C.c_uint32),
                ("root", C.c_uint32), ("max_stack", C.c_uint32), ("_pad0", C.c_uint32), ("_pad1", C.c_uint32),
                ("bbox_min", C.c_double * 3), ("bbox_max", C.c_double * 3)]


class PresetInfo(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples_per_pixel", C.c_uint32),
                ("max_depth", C.c_uint32), ("workers", C.c_uint32), ("_pad", C.c_uint32), ("vfov", C.c_double),
                ("aperture", C.c_double), ("lookfrom", C.c_double * 3), ("lookat", C.c_double * 3),
                ("output_filename", C.c_char * 64)]


# numpy views of the array-of-struct types that cross the ABI in bulk
RAY_DTYPE = np.dtype([("origin", "<f8", 3), ("direction", "<f8", 3)])
HIT_DTYPE = np.dtype([("t", "<f8"), ("u", "<f8"), ("v", "<f8"), ("prim_id", "<u4"), ("obj_id", "<u4"),
                      ("front_face", "<u4"), ("_pad", "<u4")])
assert RAY_DTYPE.itemsize == 48 and HIT_DTYPE.itemsize == 40
RECORD_DTYPE = np.dtype([("t", "<f8"), ("p", "<f8", 3), ("normal", "<f8", 3), ("u", "<f8"), ("v", "<f8"),
                         ("material", "<u4"), ("front_face", "<u4"), ("obj_id", "<u4"), ("prim_id", "<u4")])
assert RECORD_DTYPE.itemsize == 88
RAY_F32_DTYPE = np.dtype([("origin", "<f4", 3), ("direction", "<f4", 3)])
HIT_F32_DTYPE = np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim_id", "<u4")])
assert RAY_F32_DTYPE.itemsize == 24 and HIT_F32_DTYPE.itemsize == 16

# the flat QBVH layout (csrc/host_common.h)
NODE_DTYPE = np.dtype([("min_x", "<f4", 4), ("max_x", "<f4", 4), ("min_y", "<f4", 4), ("max_y", "<f4", 4),
                       ("min_z", "<f4", 4), ("max_z", "<f4", 4), ("child", "<u4", 4), ("axes", "<u4"),
                       ("pad", "<u4", 3)])
TRI_DTYPE = np.dtype([("v0", "<f4", 3), ("orig", "<u4"), ("v1", "<f4", 3), ("pad1", "<u4"), ("v2", "<f4", 3),
                      ("pad2", "<u4")])
assert NODE_DTYPE.itemsize == 128 and TRI_DTYPE.itemsize == 48


def make_rays(origins, directions):
    """Pack (n,3) origins and directions into the yart_ray array layout."""
    o = np.ascontiguousarray(origins, dtype=np.float64).reshape(-1, 3)
    d = np.ascontiguousarray(directions, dtype=np.float64).reshape(-1, 3)
    rays = np.empty(o.shape[0], dtype=RAY_DTYPE)
    rays["origin"] = o
    rays["direction"] = d
    return rays
