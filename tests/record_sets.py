"""Shared pieces of the hit-record tests (tests/test_record_oracle.py, tests/test_gpu_hit_records.py): a small
hand-built world whose answers are known in closed form, the kinds of primitive each record came from, and the
comparison under the exactness contract of yart_closest_hit_records."""
import ctypes as C
import math

import numpy as np

# the fields of a record that come from a libm call on one side and glibc on the other
SPHERE_UV_ATOL = 1e-15   # get_sphere_uv: acos / atan2 within 2 ulp, then / pi and / 2 pi
MEDIUM_REL = 1e-12       # a constant-medium hit's t (log of the draw) and the p computed from it


class SmallWorld:
    """A BVH group of three spheres with materials 0, 1, 2 (the group object itself carries material 3), a moving
    sphere of radius 0.5 whose centre goes from (0, 0, 0) at time 0 to (2, 0, 0) at time 1 (material 4), and a
    rotated, translated box (material 1).  `.desc` is what Context.set_scene and the references take."""

    GROUP_CENTRES = [(-3.0, 5.0, 0.0), (0.0, 5.0, 0.0), (3.0, 5.0, 0.0)]
    MOVING = ((0.0, 0.0, 0.0), (2.0, 0.0, 0.0), 0.5)

    def __init__(self, abi):
        self.abi = abi
        tex = abi.Texture()
        tex.kind = abi.TEX_SOLID
        tex.rgb_a[:] = [0.5, 0.5, 0.5]
        self.textures = (abi.Texture * 1)(tex)
        self.materials = (abi.Material * 5)()
        for m in self.materials:
            m.kind, m.texture = abi.MAT_LAMBERTIAN, 0
        self.members = (abi.Object * 3)()
        for i, c in enumerate(self.GROUP_CENTRES):
            m = self.members[i]
            m.kind, m.material, m.cos_theta = abi.OBJ_SPHERE, i, 1.0
            m.p[0], m.p[1], m.p[2], m.p[3] = c[0], c[1], c[2], 1.0
        self.groups = (abi.Group * 1)()
        self.groups[0].members, self.groups[0].n_members = C.cast(self.members, C.POINTER(abi.Object)), 3
        self.objects = (abi.Object * 3)()
        g, mv, bx = self.objects
        g.kind, g.index, g.material, g.cos_theta = abi.OBJ_GROUP, 0, 3, 1.0
        (c0, c1, r) = self.MOVING
        mv.kind, mv.material, mv.cos_theta = abi.OBJ_MOVING_SPHERE, 4, 1.0
        for k in range(3):
            mv.p[k], mv.p[3 + k] = c0[k], c1[k]
        mv.p[6], mv.p[7], mv.p[8] = 0.0, 1.0, r
        bx.kind, bx.material, bx.wrap = abi.OBJ_BOX, 1, abi.WRAP_ROTATE_Y | abi.WRAP_TRANSLATE
        bx.p[0:6] = [0.0, 0.0, 0.0, 1.0, 1.0, 1.0]
        bx.sin_theta, bx.cos_theta = math.sin(math.radians(15.0)), math.cos(math.radians(15.0))
        bx.offset[:] = [-1.0, -5.0, 0.0]
        self.sd = abi.SceneDesc()
        self.sd.objects, self.sd.n_objects = C.cast(self.objects, C.POINTER(abi.Object)), 3
        self.sd.groups, self.sd.n_groups = C.cast(self.groups, C.POINTER(abi.Group)), 1
        self.sd.materials, self.sd.n_materials = C.cast(self.materials, C.POINTER(abi.Material)), 5
        self.sd.textures, self.sd.n_textures = C.cast(self.textures, C.POINTER(abi.Texture)), 1
        self.desc = C.pointer(self.sd)

    def group_rays(self, n=300, seed=3):
        """Rays from below the group aimed at points near its members' centres."""
        r = np.random.default_rng(seed)
        tgt = np.asarray(self.GROUP_CENTRES)[r.integers(0, 3, n)] + r.uniform(-0.7, 0.7, (n, 3))
        o = np.column_stack([r.uniform(-4, 4, n), np.full(n, 0.0), np.full(n, -8.0)])
        return self.abi.make_rays(o, tgt - o)

    def moving_rays(self, n=200):
        """Rays along +z across the moving sphere's sweep, x from -0.8 to 2.8."""
        x = np.linspace(-0.8, 2.8, n)
        o = np.column_stack([x, np.full(n, 0.1), np.full(n, -10.0)])
        return self.abi.make_rays(o, np.tile([0.0, 0.0, 2.0], (n, 1)))


def ray_at(rays, t):
    """ray.at(t) (ray.rs:33-35) in the reference's operation order."""
    return rays["origin"] + t[:, None] * rays["direction"]


def leaf_kinds(abi, desc, rec, target):
    """(kind of the primitive each record's hit is on -- a group member's own kind --, medium flag, wrapper bits).
    Misses get kind -1."""
    n = len(rec)
    kind = np.full(n, -1, dtype=np.int64)
    medium = np.zeros(n, dtype=bool)
    wrap = np.zeros(n, dtype=np.int64)
    hit = rec["obj_id"] != abi.MISS
    if target != abi.TARGET_WORLD:
        kind[hit] = abi.OBJ_MESH
        return kind, medium, wrap
    sd = desc.contents
    for i in np.flatnonzero(hit):
        o = sd.objects[int(rec["obj_id"][i])]
        wrap[i] = o.wrap
        medium[i] = bool(o.wrap & abi.WRAP_MEDIUM)
        kind[i] = sd.groups[o.index].members[int(rec["prim_id"][i])].kind if o.kind == abi.OBJ_GROUP else o.kind
    return kind, medium, wrap


def _same(a, b):
    return (a == b) | ((a != a) & (b != b))


def assert_records_match(abi, desc, rays, got, want, target, what=""):
    """Every field bit-identical (NaN matches NaN), except the libm-derived ones: a sphere's or moving sphere's u, v
    within SPHERE_UV_ATOL, a constant-medium hit's t within MEDIUM_REL relative and its p within MEDIUM_REL of the
    magnitudes it is the sum of (|o| + |t d|)."""
    assert got.dtype == want.dtype and got.shape == want.shape
    kind, medium, _ = leaf_kinds(abi, desc, want, target)
    sphere = (kind == abi.OBJ_SPHERE) | (kind == abi.OBJ_MOVING_SPHERE)
    sphere &= ~medium

    def check(field, ok):
        bad = np.flatnonzero(~ok)
        assert bad.size == 0, "%s: field %s differs on %d of %d rays, first %d (kind %d, medium %s): gpu %r reference %r" % (
            what, field, bad.size, len(want), bad[0], kind[bad[0]], medium[bad[0]], got[bad[0]], want[bad[0]])

    for f in ("material", "front_face", "obj_id", "prim_id"):
        check(f, got[f] == want[f])
    with np.errstate(invalid="ignore"):
        t_ok = _same(got["t"], want["t"])
        t_ok |= medium & (np.abs(got["t"] - want["t"]) <= MEDIUM_REL * np.abs(want["t"]))
        check("t", t_ok)
        check("normal", _same(got["normal"], want["normal"]).all(axis=1))
        scale = np.abs(rays["origin"]) + np.abs(want["t"])[:, None] * np.abs(rays["direction"])
        p_ok = _same(got["p"], want["p"]).all(axis=1)
        p_ok |= medium & (np.abs(got["p"] - want["p"]) <= MEDIUM_REL * scale).all(axis=1)
        check("p", p_ok)
        for f in ("u", "v"):
            ok = _same(got[f], want[f]) | (sphere & (np.abs(got[f] - want[f]) <= SPHERE_UV_ATOL))
            check(f, ok)
