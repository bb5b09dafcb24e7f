// device_common.cuh -- device-side vocabulary: f64 vector math in the reference's operation
// order, Philox4x32-10, spectral tables, and the scene structures as they sit in HBM.
//
// Everything here is compiled with -fmad=false: the reference is plain f64 Rust without FMA
// contraction, and bit-exact closest-hit parity depends on evaluating (a*b + c*d) the same way.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

#include "../../include/yart.h"
#include "../../include/yart_rng.h"

namespace yart {

#define YART_DEV __device__ __forceinline__

constexpr double kPi = 3.14159265358979323846264338327950288;
constexpr double kF64Eps = 2.220446049250313e-16; // f64::EPSILON
constexpr double kF64Max = 1.7976931348623157e308;

__device__ __forceinline__ double d_inf() { return __longlong_as_double(0x7ff0000000000000LL); }

// ---------------------------------------------------------------------------------------------
// Vec3 (reference vec3.rs) -- same association order as the Rust operators
// ---------------------------------------------------------------------------------------------
struct D3 {
  double x, y, z;
};
YART_DEV D3 d3(double x, double y, double z) { return D3{x, y, z}; }
YART_DEV D3 operator+(D3 a, D3 b) { return d3(a.x + b.x, a.y + b.y, a.z + b.z); }
YART_DEV D3 operator-(D3 a, D3 b) { return d3(a.x - b.x, a.y - b.y, a.z - b.z); }
YART_DEV D3 operator-(D3 a) { return d3(-a.x, -a.y, -a.z); }
YART_DEV D3 operator*(D3 a, double s) { return d3(a.x * s, a.y * s, a.z * s); }
YART_DEV D3 operator*(double s, D3 a) { return d3(s * a.x, s * a.y, s * a.z); }
YART_DEV D3 vdiv(D3 a, double s) { // Div<f64> (vec3.rs:113-123)
  if (s == 0.0) return d3(kF64Max, kF64Max, kF64Max);
  return d3(a.x / s, a.y / s, a.z / s);
}
YART_DEV double dot(D3 a, D3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
YART_DEV D3 cross(D3 a, D3 b) {
  return d3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
YART_DEV double length_squared(D3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
// The largest double strictly below x (x = -inf and NaN stay).  NEAR-order traversal starts from just_below(t_max): its
// tests are non-strict (`t <= t_best`, `t_best >= t_near`: the mirrored tie rule needs that among THIS mesh's equal-t
// hits), and starting one step below makes them strict against what the caller / the earlier objects left -- which
// is what the reference's `t_max > t` (qbvh.rs:478) and `tfar > tnear` with tfar <= t_max (qbvh.rs:495-532) are.
YART_DEV double just_below(double x) {
  if (!(x > -d_inf())) return x;
  if (x == 0.0) return __longlong_as_double((long long)0x8000000000000001ull);
  const long long b = __double_as_longlong(x);
  return __longlong_as_double(b + (b < 0 ? 1 : -1));
}

YART_DEV double length(D3 a) { return sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
YART_DEV D3 unit_vector(D3 a) {
  double l = length(a);
  return d3(a.x / l, a.y / l, a.z / l);
}
YART_DEV double comp(D3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 and the draw contract (include/yart_rng.h)
// ---------------------------------------------------------------------------------------------
struct Rng {
  uint32_t k0, k1, pixel, sample;
};
YART_DEV Rng make_rng(uint64_t seed, uint32_t pixel, uint32_t sample) {
  Rng r;
  r.k0 = (uint32_t)(seed & 0xffffffffu);
  r.k1 = (uint32_t)(seed >> 32);
  r.pixel = pixel;
  r.sample = sample;
  return r;
}
YART_DEV void rng_draw(const Rng& r, uint32_t bounce, uint32_t slot, double& u0, double& u1) {
  uint32_t c0 = r.pixel, c1 = r.sample, c2 = bounce, c3 = slot, k0 = r.k0, k1 = r.k1;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t h0 = __umulhi(YART_PHILOX_M0, c0), l0 = YART_PHILOX_M0 * c0;
    const uint32_t h1 = __umulhi(YART_PHILOX_M1, c2), l1 = YART_PHILOX_M1 * c2;
    const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += YART_PHILOX_W0;
    k1 += YART_PHILOX_W1;
  }
  const uint64_t a = (uint64_t)c0 | ((uint64_t)c1 << 32);
  const uint64_t b = (uint64_t)c2 | ((uint64_t)c3 << 32);
  u0 = (double)(a >> 11) * (1.0 / 9007199254740992.0);
  u1 = (double)(b >> 11) * (1.0 / 9007199254740992.0);
}

// random_in_unit_sphere (material.rs:308-324) on the contract's slots
YART_DEV D3 random_in_unit_sphere(const Rng& rng, uint32_t bounce) {
  for (uint32_t i = 0; i < YART_MAX_REJECT; ++i) {
    double a, b, c, unused;
    rng_draw(rng, bounce, YART_SLOT_SPHERE + 2 * i, a, b);
    rng_draw(rng, bounce, YART_SLOT_SPHERE + 2 * i + 1, c, unused);
    D3 p = d3(-1.0 + 2.0 * a, -1.0 + 2.0 * b, -1.0 + 2.0 * c);
    if (length_squared(p) >= 1.0) continue;
    return p;
  }
  return d3(0.0, 0.0, 0.0);
}

// 256-bit read-only global load (LDG.E.256 on sm_100): one instruction and one L1 wavefront per
// 32-byte sector instead of two 128-bit loads
struct F8 {
  float4 lo, hi;
};
YART_DEV F8 ldg256(const float4* p) {
  F8 r;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z),
                 "=f"(r.hi.w)
               : "l"(p));
  return r;
}

YART_DEV void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---------------------------------------------------------------------------------------------
// Scene in HBM
// ---------------------------------------------------------------------------------------------
// Bounds-checked build (python -m build --bounds-check, tools/bounds_check.sh): every index a kernel forms
// into the tree, the triangle records, the traversal stack and the ray / hit arrays is checked and a
// violation traps (the next CUDA call of the context fails).  compute-sanitizer is not available on the
// GPU pool this was developed on; this build takes its place.  Compiled out of the product library.
#ifdef YART_BOUNDS_CHECK
#define YART_CHECK(cond)                                                              \
  do {                                                                                \
    if (!(cond)) {                                                                    \
      printf("YART_CHECK failed %s:%d: %s\n", __FILE__, __LINE__, #cond);             \
      __trap();                                                                       \
    }                                                                                 \
  } while (0)
#else
#define YART_CHECK(cond) ((void)0)
#endif

struct DevMesh {
  const float4* nodes;  // 8 float4 per node (host_common.h FlatNode: x, y, z slab pairs, children)
  const float4* tris;   // 3 float4 per triangle, tree order (FlatTri)
  const double* shade;  // 12 doubles per triangle (FlatTriShade: 9 normals + 6 float uvs)
  const float4* leafgeo; // per leaf, at 64 B x (its first triangle's position): the 9 vertex floats of each of
                         // its triangles back to back (36 B per triangle) -- a 3-triangle leaf is 4 sectors
  uint32_t root;
  uint32_t max_stack;
  uint32_t n_nodes, n_tris;
  double bound[3];      // max |coordinate| per axis
};

// The mesh instance one pass of a traversal kernel (k_traverse, k_traverse_lean, k_occlude) walks: the tree of its
// DevMesh, the instance's wrappers, and the scheduling of the persistent kernels.
struct MeshPass {
  const float4* nodes;
  const float4* tris;
  const float4* leafgeo;      // packed per-leaf vertex blocks (DevMesh::leafgeo)
  uint32_t root;
  uint32_t n_nodes, n_tris;   // array lengths (bounds-checked build)
  uint32_t wrap;              // YART_WRAP_ROTATE_Y / TRANSLATE of this instance
  double sin_theta, cos_theta, offset[3];
  double bound[3];            // max |coordinate| of the mesh per axis (for the f32 slab error bound)
  uint32_t refill_threshold;  // run the retire/fetch phase once this many lanes wait for it
  uint32_t node_threshold;    // leave the inner-node loop once fewer lanes than this are in it
  uint32_t* work_counter;     // zero before launch
};

// A flat 4-wide tree over the members of a BVHNode group (spheres / boxes).  Same 128-byte node
// as the triangle QBVH; leaves hold up to 4 member indices.
struct DevGroup {
  const float4* nodes;
  const yart_object* members;  // in tree order
  const uint32_t* member_orig; // tree position -> index in yart_group.members
  uint32_t root;      // 0xFFFFFFFF when the group is tiny and scanned linearly
  uint32_t n_members;
  double bound[3];    // max |coordinate| of the node boxes per axis (error bound of the f32 slab test)
};

struct DevImage {
  const uint8_t* rgb8;
  uint32_t width, height;
};

struct DevScene {
  const yart_object* objects;
  const yart_object* lights;
  const DevMesh* meshes;
  const DevGroup* groups;
  const yart_material* materials;
  const yart_texture* textures;
  const yart_perlin* perlins;
  const DevImage* images;
  const double* cie;   // [3][471]
  const double* smits; // [7][36]
  uint32_t n_objects, n_lights;
  double background[3];
};

// A 48-byte ray record as three 128-bit accesses instead of six 64-bit ones (half the L1 wavefronts).  Every
// ray array of the library is 16-byte aligned (cudaMalloc; yart_closest_hit checks device pointers it is given).
YART_DEV void load_ray(const yart_ray* p, D3& o, D3& d) {
  const double2* q = reinterpret_cast<const double2*>(p);
  const double2 a = q[0], b = q[1], c = q[2];
  o = d3(a.x, a.y, b.x);
  d = d3(b.y, c.x, c.y);
}
YART_DEV void store_ray(yart_ray* p, D3 o, D3 d) {
  double2* q = reinterpret_cast<double2*>(p);
  q[0] = make_double2(o.x, o.y);
  q[1] = make_double2(o.z, d.x);
  q[2] = make_double2(d.y, d.z);
}

// f32 ray records (yart_ray_f32, 24 bytes, 8-byte aligned): widened exactly; three 64-bit accesses
YART_DEV void load_ray_f32(const yart_ray_f32* p, D3& o, D3& d) {
  const float2* q = reinterpret_cast<const float2*>(p);
  const float2 a = q[0], b = q[1], c = q[2];
  o = d3((double)a.x, (double)a.y, (double)b.x);
  d = d3((double)b.y, (double)c.x, (double)c.y);
}

// A finished path's sample value (XYZ before sanitising) lives in the first 24 bytes of its ray record.
YART_DEV void store_sample(yart_ray* p, double x, double y, double z) {
  double2* q = reinterpret_cast<double2*>(p);
  q[0] = make_double2(x, y);
  reinterpret_cast<double*>(p)[2] = z;
}
YART_DEV void load_sample(const yart_ray* p, double& x, double& y, double& z) {
  const double2 a = reinterpret_cast<const double2*>(p)[0];
  x = a.x;
  y = a.y;
  z = reinterpret_cast<const double*>(p)[2];
}

// What a closest-hit query leaves behind for the shade stage (32 bytes).
struct alignas(16) DevHit {
  double t;      // +inf on a miss
  double bu, bv; // barycentric weights of v1, v2 (mesh / loose triangle hits)
  uint32_t obj;  // world object index, YART_MISS on a miss
  uint32_t prim; // mesh: triangle position in tree order; box: side; group: member
};

struct DevCamera { // Camera (camera.rs:11-23), derived on the host by Camera::new
  double llc[3], horizontal[3], vertical[3], origin[3], u[3], v[3];
  double lens_radius, time0, time1;
};

} // namespace yart
