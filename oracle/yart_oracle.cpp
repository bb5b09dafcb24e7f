// yart_oracle.cpp -- CPU ORACLE: a restatement of the reference's hot path in plain C++ (f64,
// compiled with -ffp-contract=off so no FMA contraction, like rustc's default).
//
// TEST INFRASTRUCTURE ONLY (see yart_oracle.h).  PARITY: the Rust reference cannot be built here and
// holds no golden vectors for this path, so single hits / samples are UNPINNED by the reference; this
// file is pinned at image level by digests of the reference's own shipped renders and by its scene
// constants parsed from its source (tests/test_reference_pins.py, tests/test_presets_golden.py), and
// below that by brute force, SURVEY.md Appendix D and the reference's unit tests restated in tests/.
//
// Every function cites the reference lines it follows (paths relative to the reference's
// raytracer/src/).  Arithmetic is written in the reference's operation order on purpose.
#include "yart_oracle.h"
#include "../include/yart_rng.h"
#include "../include/yart_spectral_tables.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

namespace {

const double kInf = std::numeric_limits<double>::infinity();
const double kPi = 3.14159265358979323846264338327950288; // std::f64::consts::PI
const double kEps = 2.220446049250313e-16;                // f64::EPSILON
const double kF64Max = std::numeric_limits<double>::max();

thread_local std::string g_err;

// ---------------------------------------------------------------------------------------
// The transcendentals on the film path (sphere uv, ConstantMedium, noise textures, cone and cosine sampling).  CUDA's
// sin/cos/acos/atan2 (2 ulp) and log (1 ulp) may differ from glibc's in the last bits, so the tests build variants
// of this file that move each result by a few ulp, to tell a sample that flips on such a difference from a real
// divergence (tests/perturbed_oracle.py).  YART_ORACLE_LIBM_PERTURB undefined: plain libm.  Defined as k: every
// result moves k ulp (0: the hook is compiled in and moves nothing); with YART_ORACLE_LIBM_SEED also defined, a hash
// of (seed, function, input bits) picks a move in [-|k|, |k|] per call.  Zero and non-finite results stay.
// ---------------------------------------------------------------------------------------
enum LibmFn : uint64_t { LM_SIN = 1, LM_COS, LM_ACOS, LM_ATAN2, LM_LOG };
#ifndef YART_ORACLE_LIBM_PERTURB
inline double libm_result(LibmFn, double, double, double r) { return r; }
#else
inline uint64_t libm_bits(double x) {
  uint64_t b;
  memcpy(&b, &x, sizeof b);
  return b;
}
inline double libm_result(LibmFn fn, double a, double b, double r) {
  if (r == 0.0 || !std::isfinite(r)) return r;
#ifdef YART_ORACLE_LIBM_SEED
  uint64_t h = (uint64_t)(YART_ORACLE_LIBM_SEED) * 0x9e3779b97f4a7c15ull ^ fn;
  for (uint64_t w : {libm_bits(a), libm_bits(b)}) { // splitmix64 steps
    h += w + 0x9e3779b97f4a7c15ull;
    h = (h ^ (h >> 30)) * 0xbf58476d1ce4e5b9ull;
    h = (h ^ (h >> 27)) * 0x94d049bb133111ebull;
    h ^= h >> 31;
  }
  const int span = (YART_ORACLE_LIBM_PERTURB) < 0 ? -(YART_ORACLE_LIBM_PERTURB) : (YART_ORACLE_LIBM_PERTURB);
  const int k = (int)(h % (uint64_t)(2 * span + 1)) - span;
#else
  (void)fn; (void)a; (void)b;
  const int k = YART_ORACLE_LIBM_PERTURB;
#endif
  for (int i = 0; i < (k < 0 ? -k : k); ++i) r = std::nextafter(r, k < 0 ? -INFINITY : INFINITY);
  if (fn == LM_SIN || fn == LM_COS) r = r > 1.0 ? 1.0 : (r < -1.0 ? -1.0 : r); // (as both libraries bound them)
  return r;
}
#endif
inline double lm_sin(double x) { return libm_result(LM_SIN, x, 0.0, std::sin(x)); }
inline double lm_cos(double x) { return libm_result(LM_COS, x, 0.0, std::cos(x)); }
inline double lm_acos(double x) { return libm_result(LM_ACOS, x, 0.0, std::acos(x)); }
inline double lm_atan2(double y, double x) { return libm_result(LM_ATAN2, y, x, std::atan2(y, x)); }
inline double lm_log(double x) { return libm_result(LM_LOG, x, 0.0, std::log(x)); }

// ---------------------------------------------------------------------------------------
// Vec3 (vec3.rs:8-247)
// ---------------------------------------------------------------------------------------
struct V3 {
  double x, y, z;
  double operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
  double& at(int i) { return i == 0 ? x : (i == 1 ? y : z); }
};
inline V3 v3(double x, double y, double z) { return V3{x, y, z}; }
inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
inline V3 operator*(V3 a, double s) { return v3(a.x * s, a.y * s, a.z * s); }
inline V3 operator*(double s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
// Div<f64> (vec3.rs:113-123): division by zero yields f64::MAX components
inline V3 vdiv(V3 a, double s) {
  if (s == 0.0) return v3(kF64Max, kF64Max, kF64Max);
  return v3(a.x / s, a.y / s, a.z / s);
}
inline double dot(V3 a, V3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); } // vec3.rs:222
inline V3 cross(V3 a, V3 b) {                                                     // vec3.rs:226
  return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
inline double length_squared(V3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; } // vec3.rs:200
inline double length(V3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
inline V3 unit_vector(V3 a) { // vec3.rs:204-212 (plain division, NaN for the zero vector)
  double l = length(a);
  return v3(a.x / l, a.y / l, a.z / l);
}

struct Ray { // ray.rs:4-9
  V3 o, d;
  double time, wl;
};
inline V3 ray_at(const Ray& r, double t) { return r.o + t * r.d; } // ray.rs:33-35

// ---------------------------------------------------------------------------------------
// Philox4x32-10 and the draw contract (include/yart_rng.h)
// ---------------------------------------------------------------------------------------
inline void philox(const uint32_t c_in[4], const uint32_t k_in[2], uint32_t out[4]) {
  uint32_t c0 = c_in[0], c1 = c_in[1], c2 = c_in[2], c3 = c_in[3];
  uint32_t k0 = k_in[0], k1 = k_in[1];
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)YART_PHILOX_M0 * c0;
    uint64_t p1 = (uint64_t)YART_PHILOX_M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += YART_PHILOX_W0;
    k1 += YART_PHILOX_W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct Rng {
  uint32_t key[2];
  uint32_t pixel, sample;
  void draw(uint32_t bounce, uint32_t slot, double& u0, double& u1) const {
    uint32_t c[4] = {pixel, sample, bounce, slot}, o[4];
    philox(c, key, o);
    uint64_t a = (uint64_t)o[0] | ((uint64_t)o[1] << 32);
    uint64_t b = (uint64_t)o[2] | ((uint64_t)o[3] << 32);
    u0 = (double)(a >> 11) * (1.0 / 9007199254740992.0);
    u1 = (double)(b >> 11) * (1.0 / 9007199254740992.0);
  }
};
inline Rng make_rng(uint64_t seed, uint32_t pixel, uint32_t sample) {
  Rng r;
  r.key[0] = (uint32_t)(seed & 0xffffffffu);
  r.key[1] = (uint32_t)(seed >> 32);
  r.pixel = pixel;
  r.sample = sample;
  return r;
}

// random_in_unit_sphere (material.rs:308-324)
inline V3 random_in_unit_sphere(const Rng& rng, uint32_t bounce) {
  for (uint32_t i = 0; i < YART_MAX_REJECT; ++i) {
    double a, b, c, unused;
    rng.draw(bounce, YART_SLOT_SPHERE + 2 * i, a, b);
    rng.draw(bounce, YART_SLOT_SPHERE + 2 * i + 1, c, unused);
    V3 p = v3(-1.0 + 2.0 * a, -1.0 + 2.0 * b, -1.0 + 2.0 * c);
    if (length_squared(p) >= 1.0) continue;
    return p;
  }
  return v3(0, 0, 0);
}

// ---------------------------------------------------------------------------------------
// Spectral colour (color.rs)
// ---------------------------------------------------------------------------------------
const double MIN_LAMBDA = 360.0, MAX_LAMBDA = 720.0, BIN_WIDTH = 10.0; // color.rs:7-9
const double CIE_Y_INTEGRAL = 106.856895;                               // color.rs:12
enum { B_WHITE = 0, B_CYAN, B_MAGENTA, B_YELLOW, B_RED, B_GREEN, B_BLUE };

// Spectrum::reflect's bin (color.rs:279-283): `as usize` truncates and saturates at 0
inline int spectrum_bin(double wl) {
  double q = (wl - MIN_LAMBDA) / BIN_WIDTH;
  long idx = (q != q || q <= 0.0) ? 0 : (q >= 1e18 ? (long)1e18 : (long)q);
  if (idx > YART_N_BINS - 1) idx = YART_N_BINS - 1;
  return (int)idx;
}
// RGB::reflect (color.rs:160-164) = into_spectrum (color.rs:54-90) then one bin.  Only the
// requested bin is evaluated; each bin is independent so the value is identical.
inline double rgb_reflect(const double rgb[3], double wl) {
  const int i = spectrum_bin(wl);
  const double red = rgb[0], green = rgb[1], blue = rgb[2];
  auto B = [&](int basis) { return YART_SMITS_BASIS[basis * YART_N_BINS + i]; };
  double s = 0.0;
  // `spectrum += c * BASIS` is `*b = *a + *b` with a = c*BASIS (color.rs:252-276)
  if (red <= green && red <= blue) {
    s = red * B(B_WHITE) + s;
    if (green <= blue) {
      s = (green - red) * B(B_CYAN) + s;
      s = (blue - green) * B(B_BLUE) + s;
    } else {
      s = (blue - red) * B(B_CYAN) + s;
      s = (green - blue) * B(B_GREEN) + s;
    }
  } else if (green <= red && green <= blue) {
    s = green * B(B_WHITE) + s;
    if (red <= blue) {
      s = (red - green) * B(B_MAGENTA) + s;
      s = (blue - red) * B(B_BLUE) + s;
    } else {
      s = (blue - green) * B(B_MAGENTA) + s;
      s = (red - blue) * B(B_RED) + s;
    }
  } else {
    s = blue * B(B_WHITE) + s;
    if (red <= green) {
      s = (red - blue) * B(B_YELLOW) + s;
      s = (green - red) * B(B_GREEN) + s;
    } else {
      s = (green - blue) * B(B_YELLOW) + s;
      s = (red - green) * B(B_RED) + s;
    }
  }
  return s;
}
// XYZ::from_wavelength (color.rs:216-227)
inline void xyz_from_wavelength(double wl, double out[3]) {
  double q = wl - MIN_LAMBDA;
  long idx = (q != q) ? 0 : (q <= -9e18 ? (long)-9e18 : (q >= 9e18 ? (long)9e18 : (long)q));
  if (idx < 0 || idx >= YART_N_CIE) {
    out[0] = out[1] = out[2] = 0.0;
  } else {
    out[0] = YART_CIE_X[idx];
    out[1] = YART_CIE_Y[idx];
    out[2] = YART_CIE_Z[idx];
  }
}
inline void xyz_into_rgb(const double c[3], double out[3]) { // color.rs:209-213
  out[0] = 2.6896552 * c[0] - 1.2758621 * c[1] - 0.4137931 * c[2];
  out[1] = -1.0221082 * c[0] + 1.9782866 * c[1] + 0.0438216 * c[2];
  out[2] = 0.0612245 * c[0] - 0.2244898 * c[1] + 1.1632653 * c[2];
}
inline double gamma_channel(double linear) { // color.rs:93-100
  linear = std::fmax(linear, 0.0);           // f64::max: NaN -> 0
  if (linear <= 0.0031308) return 12.92 * linear;
  return 1.055 * std::pow(linear, 1.0 / 2.4) - 0.055;
}
inline uint8_t clamp_display_channel(double c) { // main.rs:461-463
  double x = c;                                   // f64::clamp keeps NaN; `as u8` maps NaN -> 0
  if (x < 0.0) x = 0.0;
  if (x > 0.999) x = 0.999;
  double v = 256.0 * x;
  if (v != v) return 0;
  return (uint8_t)v;
}
inline void sanitize_sample_xyz(const double in[3], double out[3]) { // main.rs:448-459
  if (!std::isfinite(in[0]) || !std::isfinite(in[1]) || !std::isfinite(in[2])) {
    out[0] = out[1] = out[2] = 0.0;
    return;
  }
  double lum = in[1];
  if (lum <= 0.0 || lum <= 20.0) {
    out[0] = in[0]; out[1] = in[1]; out[2] = in[2];
    return;
  }
  double k = 20.0 / lum;
  out[0] = in[0] * k; out[1] = in[1] * k; out[2] = in[2] * k;
}

// ---------------------------------------------------------------------------------------
// L4QBVH (qbvh.rs)
// ---------------------------------------------------------------------------------------
struct Tri {
  V3 v[3], n[3];
  double uv[3][2];
  uint32_t orig;
  V3 bmin, bmax, centroid;
};
struct Box {
  V3 mn, mx;
  bool some;
};
struct Node { // QBVHNode (qbvh.rs:546-600)
  double bmin[3][4], bmax[3][4];
  uint32_t child[4];
  uint32_t axis[3]; // top, left, right
};
struct Mesh {
  std::vector<Tri> tris; // sorted in place by the build, like `triangles` (qbvh.rs:349)
  std::vector<Node> nodes;
  uint32_t n_leaves = 0, empty_children = 0, leaves_by_count[5] = {0, 0, 0, 0, 0};
};

inline Box surrounding(const Box& a, const Box& b) { // aabb.rs:172-185 (f64::min / f64::max)
  Box r;
  r.some = true;
  r.mn = v3(std::fmin(a.mn.x, b.mn.x), std::fmin(a.mn.y, b.mn.y), std::fmin(a.mn.z, b.mn.z));
  r.mx = v3(std::fmax(a.mx.x, b.mx.x), std::fmax(a.mx.y, b.mx.y), std::fmax(a.mx.z, b.mx.z));
  return r;
}
inline Box merge_opt(const Box& a, const Box& b) { // the match at qbvh.rs:322-337
  if (a.some && b.some) return surrounding(a, b);
  if (a.some) return a;
  return b;
}

// split (qbvh.rs:636-693).  sort_unstable_by's tie order is unspecified in Rust; ties are
// broken by original triangle index here AND in the product so both build the same tree.
uint32_t split_range(std::vector<Tri>& t, size_t lo, size_t hi) {
  double mnx = kInf, mxx = -kInf, mny = kInf, mxy = -kInf, mnz = kInf, mxz = -kInf;
  for (size_t i = lo; i < hi; ++i) {
    const V3& c = t[i].centroid;
    mnx = std::fmin(mnx, c.x); mxx = std::fmax(mxx, c.x);
    mny = std::fmin(mny, c.y); mxy = std::fmax(mxy, c.y);
    mnz = std::fmin(mnz, c.z); mxz = std::fmax(mxz, c.z);
  }
  uint32_t axis = 0;
  if (mxy - mny > mxx - mnx) axis = 1;
  if (mxz - mnz > std::fmax(mxy - mny, mxx - mnx)) axis = 2;
  std::sort(t.begin() + lo, t.begin() + hi, [axis](const Tri& a, const Tri& b) {
    double ca = a.centroid[axis], cb = b.centroid[axis];
    if (ca < cb) return true;
    if (ca > cb) return false;
    return a.orig < b.orig;
  });
  return axis;
}

Box construct(Mesh& m, size_t lo, size_t hi, uint32_t& id_out) { // qbvh.rs:253-347
  size_t n = hi - lo;
  Box none;
  none.some = false;
  none.mn = none.mx = v3(0, 0, 0);
  if (n == 0) {
    id_out = 0xFFFFFFFFu;
    return none;
  }
  if (n <= 4) {
    Box b;
    b.some = true;
    b.mn = m.tris[lo].bmin;
    b.mx = m.tris[lo].bmax;
    for (size_t i = lo + 1; i < hi; ++i) {
      Box tb;
      tb.some = true;
      tb.mn = m.tris[i].bmin;
      tb.mx = m.tris[i].bmax;
      b = surrounding(b, tb);
    }
    id_out = (uint32_t)lo | (1u << 31) | ((uint32_t)n << 27); // qbvh.rs:270
    m.n_leaves++;
    m.leaves_by_count[n]++;
    return b;
  }
  uint32_t top = split_range(m.tris, lo, hi);
  size_t mid = lo + n / 2;
  uint32_t la = split_range(m.tris, lo, mid);
  size_t lmid = lo + (mid - lo) / 2;
  uint32_t ll_id, lr_id, rl_id, rr_id;
  Box ll = construct(m, lo, lmid, ll_id);
  Box lr = construct(m, lmid, mid, lr_id);
  uint32_t ra = split_range(m.tris, mid, hi);
  size_t rmid = mid + (hi - mid) / 2;
  Box rl = construct(m, mid, rmid, rl_id);
  Box rr = construct(m, rmid, hi, rr_id);

  Node nd; // QBVHNode::new (qbvh.rs:557-599): absent children keep f64::MAX boxes, id u32::MAX
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 4; ++k) nd.bmin[a][k] = nd.bmax[a][k] = kF64Max;
  const Box* bs[4] = {&ll, &lr, &rl, &rr};
  const uint32_t ids[4] = {ll_id, lr_id, rl_id, rr_id};
  for (int k = 0; k < 4; ++k) {
    if (bs[k]->some) {
      for (int a = 0; a < 3; ++a) {
        nd.bmin[a][k] = bs[k]->mn[a];
        nd.bmax[a][k] = bs[k]->mx[a];
      }
    } else {
      m.empty_children++;
    }
    nd.child[k] = ids[k];
  }
  nd.axis[0] = top; nd.axis[1] = la; nd.axis[2] = ra;
  m.nodes.push_back(nd);
  id_out = (uint32_t)(m.nodes.size() - 1);
  return surrounding(merge_opt(ll, lr), merge_opt(rl, rr));
}

void build_mesh(const yart_trimesh& src, Mesh& m) {
  m.tris.resize(src.n_tris);
  for (uint32_t i = 0; i < src.n_tris; ++i) {
    Tri& t = m.tris[i];
    for (int k = 0; k < 3; ++k) {
      t.v[k] = v3((double)src.positions[i * 9 + k * 3 + 0], (double)src.positions[i * 9 + k * 3 + 1],
                  (double)src.positions[i * 9 + k * 3 + 2]);
      t.n[k] = v3(src.normals[i * 9 + k * 3 + 0], src.normals[i * 9 + k * 3 + 1],
                  src.normals[i * 9 + k * 3 + 2]);
      t.uv[k][0] = (double)src.uvs[i * 6 + k * 2 + 0];
      t.uv[k][1] = (double)src.uvs[i * 6 + k * 2 + 1];
    }
    t.orig = i;
    // Triangle::bounding_box (triangle.rs:20-45) and Hittable::centroid (hittable.rs:12-22)
    t.bmin = v3(std::fmin(std::fmin(std::fmin(kInf, t.v[0].x), t.v[1].x), t.v[2].x),
                std::fmin(std::fmin(std::fmin(kInf, t.v[0].y), t.v[1].y), t.v[2].y),
                std::fmin(std::fmin(std::fmin(kInf, t.v[0].z), t.v[1].z), t.v[2].z));
    t.bmax = v3(std::fmax(std::fmax(std::fmax(-kInf, t.v[0].x), t.v[1].x), t.v[2].x),
                std::fmax(std::fmax(std::fmax(-kInf, t.v[0].y), t.v[1].y), t.v[2].y),
                std::fmax(std::fmax(std::fmax(-kInf, t.v[0].z), t.v[1].z), t.v[2].z));
    t.centroid = v3((t.bmax.x + t.bmin.x) / 2.0, (t.bmax.y + t.bmin.y) / 2.0,
                    (t.bmax.z + t.bmin.z) / 2.0);
  }
  uint32_t root;
  construct(m, 0, m.tris.size(), root);
}

const uint32_t ORDER_TABLE[8] = {0x0123, 0x0132, 0x1023, 0x1032, 0x2301, 0x3201, 0x2310, 0x3210};

struct MeshHit {
  double t, bu, bv; // t and the barycentric weights of v1, v2
  uint32_t pos;     // position in the sorted triangle array
  bool some;
};

struct Counters {
  uint64_t rays = 0, node_visits = 0, leaf_visits = 0, tri_tests = 0, max_stack = 0;
};

// L4QBVH::hit (qbvh.rs:381-543).  NEAR=false is the reference verbatim.  NEAR=true is the
// mirrored order with mirrored tie rules (yart.h YART_ORDER_NEAR) and must return the same hit.
// The mirrored rules are non-strict (`t_max >= t`: the LAST equal-t hit found wins, which is the
// reference's first), so NEAR starts one step below the t_max it is given: against the caller's bound
// and the hits of earlier objects the reference is strict (`t_max > t`, `tfar > tnear` with
// tfar <= t_max), and a hit or box entry AT that bound must stay out.
template <bool NEAR>
MeshHit qbvh_hit(const Mesh& m, const Ray& ray, double t_min, double t_max_in, Counters* cnt) {
  MeshHit best;
  best.some = false;
  best.t = kInf; best.bu = best.bv = 0; best.pos = 0;
  if (m.nodes.empty()) return best; // the reference underflows here (SURVEY A-17); host guards
  uint32_t stack[64];
  size_t cursor = 0;
  stack[0] = (uint32_t)m.nodes.size() - 1;
  const bool pos[3] = {ray.d.x >= 0.0, ray.d.y >= 0.0, ray.d.z >= 0.0};
  const double ro[3] = {ray.o.x, ray.o.y, ray.o.z};
  const double rd[3] = {ray.d.x, ray.d.y, ray.d.z};
  const double inv[3] = {1.0 / rd[0], 1.0 / rd[1], 1.0 / rd[2]};
  double t_max = NEAR ? std::nextafter(t_max_in, -kInf) : t_max_in;
  size_t max_cursor = 0;

  for (;;) {
    uint32_t id = stack[cursor];
    if ((id >> 31) == 1) {
      const uint32_t count = (id >> 27) & 0xF;
      const uint32_t index = id & ((1u << 27) - 1);
      if (cnt) {
        cnt->leaf_visits++;
        cnt->tri_tests += count;
      }
      double tt[4], uu[4], vv[4];
      bool hit[4];
      const double t_max_entry = t_max;
      for (uint32_t i = 0; i < count; ++i) { // the f64x4 lanes of qbvh.rs:420-450
        const Tri& tr = m.tris[index + i];
        const double v0[3] = {tr.v[0].x, tr.v[0].y, tr.v[0].z};
        const double e1[3] = {tr.v[1].x - tr.v[0].x, tr.v[1].y - tr.v[0].y, tr.v[1].z - tr.v[0].z};
        const double e2[3] = {tr.v[2].x - tr.v[0].x, tr.v[2].y - tr.v[0].y, tr.v[2].z - tr.v[0].z};
        const double h[3] = {rd[1] * e2[2] - rd[2] * e2[1], rd[2] * e2[0] - rd[0] * e2[2],
                             rd[0] * e2[1] - rd[1] * e2[0]};
        const double a = e1[0] * h[0] + e1[1] * h[1] + e1[2] * h[2];
        bool ok = !((a > -kEps) && (a < kEps));
        const double f = 1.0 / a;
        const double s[3] = {ro[0] - v0[0], ro[1] - v0[1], ro[2] - v0[2]};
        const double u = f * (s[0] * h[0] + s[1] * h[1] + s[2] * h[2]);
        ok = ok && (u >= 0.0) && (u <= 1.0);
        const double q[3] = {s[1] * e1[2] - s[2] * e1[1], s[2] * e1[0] - s[0] * e1[2],
                             s[0] * e1[1] - s[1] * e1[0]};
        const double v = f * (rd[0] * q[0] + rd[1] * q[1] + rd[2] * q[2]);
        ok = ok && (v >= 0.0) && ((u + v) <= 1.0);
        const double t = f * (e2[0] * q[0] + e2[1] * q[1] + e2[2] * q[2]);
        ok = ok && (t >= t_min) && (t <= t_max_entry);
        tt[i] = t; uu[i] = u; vv[i] = v; hit[i] = ok;
      }
      if (!NEAR) {
        for (uint32_t i = 0; i < count; ++i) { // qbvh.rs:470-490
          if (hit[i] && t_max > tt[i]) {
            t_max = tt[i];
            best.some = true; best.t = tt[i]; best.bu = uu[i]; best.bv = vv[i]; best.pos = index + i;
          }
        }
      } else {
        for (uint32_t k = count; k-- > 0;) {
          if (hit[k] && t_max >= tt[k]) {
            t_max = tt[k];
            best.some = true; best.t = tt[k]; best.bu = uu[k]; best.bv = vv[k]; best.pos = index + k;
          }
        }
      }
    } else {
      const Node& nd = m.nodes[id];
      if (cnt) cnt->node_visits++;
      bool hits[4];
      for (int k = 0; k < 4; ++k) { // qbvh.rs:495-519, one f64x4 lane at a time
        double tn = t_min;
        double tf = NEAR ? kInf : t_max;
        for (int a = 0; a < 3; ++a) {
          const double t0 = (nd.bmin[a][k] - ro[a]) * inv[a];
          const double t1 = (nd.bmax[a][k] - ro[a]) * inv[a];
          tn = std::fmax(tn, std::fmin(t0, t1)); // simd_min / simd_max = IEEE minNum / maxNum
          tf = std::fmin(tf, std::fmax(t0, t1));
        }
        hits[k] = NEAR ? ((tf > tn) && (t_max >= tn)) : (tf > tn); // qbvh.rs:532
      }
      const bool p0 = NEAR ? !pos[nd.axis[0]] : pos[nd.axis[0]];
      const bool p1 = NEAR ? !pos[nd.axis[1]] : pos[nd.axis[1]];
      const bool p2 = NEAR ? !pos[nd.axis[2]] : pos[nd.axis[2]];
      const uint32_t enc = ORDER_TABLE[4 * (int)p0 + 2 * (int)p1 + (int)p2]; // qbvh.rs:521-524
      for (int j = 0; j < 4; ++j) { // push_hit_children (qbvh.rs:18-31)
        const uint32_t i = (enc >> (4 * j)) & 0xF;
        if (hits[i]) {
          stack[cursor] = nd.child[i];
          cursor++;
        }
      }
      if (cursor > max_cursor) max_cursor = cursor;
    }
    if (cursor == 0) break;
    cursor--;
  }
  if (cnt && max_cursor > cnt->max_stack) cnt->max_stack = max_cursor;
  return best;
}

// ---------------------------------------------------------------------------------------
// Scene: objects, wrappers, materials, textures (hittable.rs, sphere.rs, aarect.rs, ...)
// ---------------------------------------------------------------------------------------
struct HitRec { // HitRecord (hittable.rs:37-45) + ids for the parity harness
  double u, v, t;
  V3 p, normal;
  bool front_face;
  uint32_t material;
  uint32_t prim, obj;
  double bu, bv;
};

struct Scene {
  std::vector<yart_object> objects, lights;
  std::vector<Mesh> meshes;
  std::vector<std::vector<yart_object>> groups;
  std::vector<yart_material> materials;
  std::vector<yart_texture> textures;
  std::vector<yart_perlin> perlins;
  struct Image {
    std::vector<uint8_t> data;
    uint32_t w, h;
  };
  std::vector<Image> images;
  double background[3];
};

inline void get_sphere_uv(V3 p, double& u, double& v) { // sphere.rs:213-220
  double theta = lm_acos(-p.y);
  double phi = lm_atan2(-p.z, p.x) + kPi;
  u = phi / (2.0 * kPi);
  v = theta / kPi;
}

bool hit_sphere(const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  // StillSphere::hit (sphere.rs:48-86)
  const V3 center = v3(o.p[0], o.p[1], o.p[2]);
  const double radius = o.p[3];
  V3 oc = r.o - center;
  double a = length_squared(r.d);
  double half_b = dot(oc, r.d);
  double c = length_squared(oc) - radius * radius;
  double disc = half_b * half_b - a * c;
  if (disc < 0.0) return false;
  double t = (0.0 - half_b - std::sqrt(disc)) / a;
  if (t < t_min || t_max < t) {
    t = (0.0 - half_b + std::sqrt(disc)) / a;
    if (t < t_min || t_max < t) return false;
  }
  V3 p = ray_at(r, t);
  V3 outward = vdiv(p - center, std::fabs(radius));
  if (radius < 0.0) {
    rec.normal = -outward;
    rec.front_face = dot(r.d, outward) > 0.0;
  } else {
    rec.normal = outward;
    rec.front_face = dot(r.d, outward) < 0.0;
  }
  get_sphere_uv(outward, rec.u, rec.v);
  rec.t = t; rec.p = p; rec.material = o.material; rec.prim = 0; rec.bu = rec.bv = 0;
  return true;
}

bool hit_moving_sphere(const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  // MovingSphere::hit (sphere.rs:156-198), center(time) (sphere.rs:149-152)
  const V3 c0 = v3(o.p[0], o.p[1], o.p[2]), c1 = v3(o.p[3], o.p[4], o.p[5]);
  const double time0 = o.p[6], time1 = o.p[7], radius = o.p[8];
  V3 center = c0 + ((r.time - time0) / (time1 - time0)) * (c1 - c0);
  V3 oc = r.o - center;
  double a = length_squared(r.d);
  double half_b = dot(oc, r.d);
  double c = length_squared(oc) - radius * radius;
  double disc = half_b * half_b - a * c;
  if (disc < 0.0) return false;
  double t = (0.0 - half_b - std::sqrt(disc)) / a;
  if (t < t_min || t_max < t) {
    t = (0.0 - half_b + std::sqrt(disc)) / a;
    if (t < t_min || t_max < t) return false;
  }
  V3 p = ray_at(r, t);
  V3 outward = vdiv(p - center, radius);
  if (dot(r.d, outward) < 0.0) {
    rec.normal = outward; rec.front_face = true;
  } else {
    rec.normal = -outward; rec.front_face = false;
  }
  get_sphere_uv(outward, rec.u, rec.v);
  rec.t = t; rec.p = p; rec.material = o.material; rec.prim = 0; rec.bu = rec.bv = 0;
  return true;
}

// XYRect / XZRect / YZRect ::hit (aarect.rs:41-80, 111-146, 206-241).
// axis = the constant axis (2: XY, 1: XZ, 0: YZ); a/b = the two varying axes in struct order.
bool hit_rect_params(int kaxis, double a0, double a1, double b0, double b1, double k, uint32_t mat,
                     const Ray& r, double t_min, double t_max, HitRec& rec) {
  const int aa = (kaxis == 0) ? 1 : 0;
  const int ba = (kaxis == 2) ? 1 : 2;
  double t = (k - r.o[kaxis]) / r.d[kaxis];
  if (t < t_min || t > t_max) return false;
  double a = r.o[aa] + t * r.d[aa];
  double b = r.o[ba] + t * r.d[ba];
  if (a < a0 || a > a1 || b < b0 || b > b1) return false;
  rec.u = (a - a0) / (a1 - a0);
  rec.v = (b - b0) / (b1 - b0);
  rec.t = t;
  rec.p = ray_at(r, t);
  V3 outward = v3(kaxis == 0 ? 1.0 : 0.0, kaxis == 1 ? 1.0 : 0.0, kaxis == 2 ? 1.0 : 0.0);
  if (dot(r.d, outward) < 0.0) {
    rec.normal = outward; rec.front_face = true;
  } else {
    rec.normal = -outward; rec.front_face = false;
  }
  rec.material = mat; rec.prim = 0; rec.bu = rec.bv = 0;
  return true;
}
inline int rect_axis(uint32_t kind) {
  return kind == YART_OBJ_XY_RECT ? 2 : (kind == YART_OBJ_XZ_RECT ? 1 : 0);
}
bool hit_rect(const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  return hit_rect_params(rect_axis(o.kind), o.p[0], o.p[1], o.p[2], o.p[3], o.p[4], o.material, r,
                         t_min, t_max, rec);
}

bool hit_box(const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  // BoxEntity::new sides (box_entity.rs:23-46) and ::hit (box_entity.rs:51-70)
  const double x0 = o.p[0], y0 = o.p[1], z0 = o.p[2], x1 = o.p[3], y1 = o.p[4], z1 = o.p[5];
  bool any = false;
  double closest = t_max;
  HitRec tmp;
  struct S { int axis; double a0, a1, b0, b1, k; };
  const S sides[6] = {{2, x0, x1, y0, y1, z0}, {2, x0, x1, y0, y1, z1}, {1, x0, x1, z0, z1, y0},
                      {1, x0, x1, z0, z1, y1}, {0, y0, y1, z0, z1, x0}, {0, y0, y1, z0, z1, x1}};
  for (int i = 0; i < 6; ++i) {
    if (hit_rect_params(sides[i].axis, sides[i].a0, sides[i].a1, sides[i].b0, sides[i].b1,
                        sides[i].k, o.material, r, t_min, closest, tmp)) {
      closest = tmp.t;
      rec = tmp;
      rec.prim = (uint32_t)i;
      any = true;
    }
  }
  return any;
}

bool hit_triangle(const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  // Triangle::hit (triangle.rs:48-101)
  const V3 v0 = v3(o.p[0], o.p[1], o.p[2]), v1 = v3(o.p[3], o.p[4], o.p[5]), v2 = v3(o.p[6], o.p[7], o.p[8]);
  const V3 n0 = v3(o.p[9], o.p[10], o.p[11]), n1 = v3(o.p[12], o.p[13], o.p[14]),
           n2 = v3(o.p[15], o.p[16], o.p[17]);
  V3 e1 = v1 - v0, e2 = v2 - v0;
  V3 h = cross(r.d, e2);
  double a = dot(e1, h);
  if (a > -kEps && a < kEps) return false;
  double f = 1.0 / a;
  V3 s = r.o - v0;
  double u = f * dot(s, h);
  if (u < 0.0 || u > 1.0) return false;
  V3 q = cross(s, e1);
  double v = f * dot(r.d, q);
  if (v < 0.0 || u + v > 1.0) return false;
  double t = f * dot(e2, q);
  if (t < t_min || t > t_max) return false;
  double w = 1.0 - u - v;
  V3 outward = n0 * w + n1 * u + n2 * v;
  if (dot(r.d, outward) < 0.0) {
    rec.normal = outward; rec.front_face = true;
  } else {
    rec.normal = -outward; rec.front_face = false;
  }
  rec.u = o.p[18] * w + o.p[20] * u + o.p[22] * v;
  rec.v = o.p[19] * w + o.p[21] * u + o.p[23] * v;
  rec.t = t; rec.p = ray_at(r, t); rec.material = o.material; rec.prim = 0; rec.bu = u; rec.bv = v;
  return true;
}

// the HitRecord an L4QBVH leaf builds for its winning lane (qbvh.rs:452-489)
void mesh_hit_record(const Mesh& m, const MeshHit& mh, const Ray& r, uint32_t mat, HitRec& rec) {
  const Tri& tr = m.tris[mh.pos];
  const double u = mh.bu, v = mh.bv, t = mh.t;
  rec.p = v3(r.o.x + t * r.d.x, r.o.y + t * r.d.y, r.o.z + t * r.d.z);
  const double w = 1.0 - u - v;
  V3 outward = v3(tr.n[0].x * w + tr.n[1].x * u + tr.n[2].x * v,
                  tr.n[0].y * w + tr.n[1].y * u + tr.n[2].y * v,
                  tr.n[0].z * w + tr.n[1].z * u + tr.n[2].z * v);
  const bool ff = (r.d.x * outward.x + r.d.y * outward.y + r.d.z * outward.z) <= 0.0;
  const double sign = ff ? 1.0 : -1.0;
  rec.normal = v3(sign * outward.x, sign * outward.y, sign * outward.z);
  rec.front_face = ff;
  rec.u = tr.uv[0][0] * w + tr.uv[1][0] * u + tr.uv[2][0] * v;
  rec.v = tr.uv[0][1] * w + tr.uv[1][1] * u + tr.uv[2][1] * v;
  rec.t = t; rec.material = mat; rec.prim = tr.orig; rec.bu = u; rec.bv = v;
}

struct HitCtx {
  const Scene* s;
  uint32_t order;
  Counters* cnt;
};

bool hit_prim(const HitCtx& c, const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec);

// BVHNode::hit over a member list (bvh.rs:151-215).  The closest hit does not depend on the
// tree; members are scanned in list order with the shrinking interval of HittableList::hit.
bool hit_group(const HitCtx& c, const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  const std::vector<yart_object>& mem = c.s->groups[o.index];
  bool any = false;
  double closest = t_max;
  HitRec tmp;
  for (size_t i = 0; i < mem.size(); ++i) {
    if (hit_prim(c, mem[i], r, t_min, closest, tmp)) {
      closest = tmp.t;
      rec = tmp;
      rec.prim = (uint32_t)i;
      any = true;
    }
  }
  return any;
}

bool hit_prim(const HitCtx& c, const yart_object& o, const Ray& r, double t_min, double t_max, HitRec& rec) {
  switch (o.kind) {
    case YART_OBJ_SPHERE: return hit_sphere(o, r, t_min, t_max, rec);
    case YART_OBJ_MOVING_SPHERE: return hit_moving_sphere(o, r, t_min, t_max, rec);
    case YART_OBJ_XY_RECT:
    case YART_OBJ_XZ_RECT:
    case YART_OBJ_YZ_RECT: return hit_rect(o, r, t_min, t_max, rec);
    case YART_OBJ_BOX: return hit_box(o, r, t_min, t_max, rec);
    case YART_OBJ_TRIANGLE: return hit_triangle(o, r, t_min, t_max, rec);
    case YART_OBJ_MESH: {
      const Mesh& m = c.s->meshes[o.index];
      if (c.cnt) c.cnt->rays += 0;
      MeshHit mh = (c.order == YART_ORDER_NEAR) ? qbvh_hit<true>(m, r, t_min, t_max, c.cnt)
                                                : qbvh_hit<false>(m, r, t_min, t_max, c.cnt);
      if (!mh.some) return false;
      mesh_hit_record(m, mh, r, o.material, rec);
      return true;
    }
    case YART_OBJ_GROUP: return hit_group(c, o, r, t_min, t_max, rec);
    default: return false;
  }
}

// FlipFace / RotateY / Translate (hittable.rs:338-349, 217-251, 136-152) around a primitive
bool hit_inner(const HitCtx& c, const yart_object& o, const Ray& ray, double t_min, double t_max, HitRec& rec) {
  Ray r = ray;
  if (o.wrap & YART_WRAP_TRANSLATE) r.o = ray.o - v3(o.offset[0], o.offset[1], o.offset[2]);
  if (o.wrap & YART_WRAP_ROTATE_Y) {
    const double ct = o.cos_theta, st = o.sin_theta;
    V3 org = r.o, dir = r.d;
    org.x = ct * r.o.x - st * r.o.z;
    org.z = st * r.o.x + ct * r.o.z;
    dir.x = ct * r.d.x - st * r.d.z;
    dir.z = st * r.d.x + ct * r.d.z;
    r.o = org;
    r.d = dir;
  }
  if (!hit_prim(c, o, r, t_min, t_max, rec)) return false;
  if (o.wrap & YART_WRAP_FLIP_FACE) rec.front_face = !rec.front_face;
  if (o.wrap & YART_WRAP_ROTATE_Y) {
    const double ct = o.cos_theta, st = o.sin_theta;
    V3 p = rec.p, n = rec.normal;
    p.x = ct * rec.p.x + st * rec.p.z;
    p.z = -st * rec.p.x + ct * rec.p.z;
    n.x = ct * rec.normal.x + st * rec.normal.z;
    n.z = -st * rec.normal.x + ct * rec.normal.z;
    rec.p = p;
    rec.normal = n;
  }
  if (o.wrap & YART_WRAP_TRANSLATE) rec.p = rec.p + v3(o.offset[0], o.offset[1], o.offset[2]);
  return true;
}

// one top-level object, including ConstantMedium::hit (hittable.rs:274-321)
bool hit_object(const HitCtx& c, const yart_object& o, uint32_t obj_index, const Ray& ray, double t_min,
                double t_max, const Rng* rng, uint32_t bounce, HitRec& rec) {
  if (!(o.wrap & YART_WRAP_MEDIUM)) {
    if (!hit_inner(c, o, ray, t_min, t_max, rec)) return false;
    rec.obj = obj_index;
    return true;
  }
  HitRec rec1, rec2;
  if (!hit_inner(c, o, ray, -kInf, kInf, rec1)) return false;
  if (!hit_inner(c, o, ray, rec1.t + 0.0001, kInf, rec2)) return false;
  if (rec1.t < t_min) rec1.t = t_min;
  if (rec2.t > t_max) rec2.t = t_max;
  if (!(rec1.t < rec2.t)) return false;
  if (rec1.t < 0.0) rec1.t = 0.0;
  const double ray_length = length(ray.d);
  const double distance_inside = (rec2.t - rec1.t) * ray_length;
  double u0 = 0.5, u1;
  if (rng) rng->draw(bounce, YART_SLOT_MEDIUM + obj_index, u0, u1);
  const double hit_distance = o.neg_inv_density * lm_log(u0);
  if (!(hit_distance < distance_inside)) return false;
  rec.t = rec1.t + hit_distance / ray_length;
  rec.p = ray_at(ray, rec.t);
  rec.u = rec.v = 0.0;
  rec.normal = v3(1.0, 0.0, 0.0);
  rec.front_face = true;
  rec.material = o.material;
  rec.prim = 0; rec.bu = rec.bv = 0; rec.obj = obj_index;
  return true;
}

// HittableList::hit (hittable.rs:66-79)
bool world_hit(const HitCtx& c, const Ray& ray, double t_min, double t_max, const Rng* rng, uint32_t bounce,
               HitRec& rec) {
  bool any = false;
  double closest = t_max;
  HitRec tmp;
  const std::vector<yart_object>& objs = c.s->objects;
  for (size_t i = 0; i < objs.size(); ++i) {
    if (hit_object(c, objs[i], (uint32_t)i, ray, t_min, closest, rng, bounce, tmp)) {
      closest = tmp.t;
      rec = tmp;
      any = true;
    }
  }
  if (c.cnt) c.cnt->rays++;
  return any;
}

// ---------------------------------------------------------------------------------------
// Textures (texture.rs)
// ---------------------------------------------------------------------------------------
inline int32_t f64_as_i32(double x) { // Rust `as i32`: truncate, saturate, NaN -> 0
  if (x != x) return 0;
  if (x >= 2147483647.0) return 2147483647;
  if (x <= -2147483648.0) return (-2147483647 - 1);
  return (int32_t)x;
}
inline uint32_t f64_as_u32(double x) {
  if (x != x || x <= 0.0) return 0;
  if (x >= 4294967295.0) return 4294967295u;
  return (uint32_t)x;
}

double perlin_noise(const yart_perlin& pn, uint32_t type, V3 p) { // Perlin::noise (texture.rs:113-175)
  if (type == YART_NOISE_SQUARE) {
    int i = f64_as_i32(4.0 * p.x) & 255, j = f64_as_i32(4.0 * p.y) & 255, k = f64_as_i32(4.0 * p.z) & 255;
    return pn.ranfloat[pn.perm_x[i] ^ pn.perm_y[j] ^ pn.perm_z[k]];
  }
  if (type == YART_NOISE_TRILINEAR) {
    double u = p.x - std::floor(p.x), v = p.y - std::floor(p.y), w = p.z - std::floor(p.z);
    u = u * u * (3.0 - 2.0 * u);
    v = v * v * (3.0 - 2.0 * v);
    w = w * w * (3.0 - 2.0 * w);
    int i = f64_as_i32(std::floor(p.x)), j = f64_as_i32(std::floor(p.y)), k = f64_as_i32(std::floor(p.z));
    double accum = 0.0; // trilinear_interp (texture.rs:194-208)
    for (int di = 0; di < 2; ++di)
      for (int dj = 0; dj < 2; ++dj)
        for (int dk = 0; dk < 2; ++dk) {
          double c = pn.ranfloat[pn.perm_x[(i + di) & 255] ^ pn.perm_y[(j + dj) & 255] ^ pn.perm_z[(k + dk) & 255]];
          accum += ((double)di * u + (double)(1 - di) * (1.0 - u)) *
                   ((double)dj * v + (double)(1 - dj) * (1.0 - v)) *
                   ((double)dk * w + (double)(1 - dk) * (1.0 - w)) * c;
        }
    return accum;
  }
  double u = p.x - std::floor(p.x), v = p.y - std::floor(p.y), w = p.z - std::floor(p.z);
  int i = f64_as_i32(std::floor(p.x)), j = f64_as_i32(std::floor(p.y)), k = f64_as_i32(std::floor(p.z));
  double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
  double accum = 0.0; // perlin_interp (texture.rs:210-229)
  for (int di = 0; di < 2; ++di)
    for (int dj = 0; dj < 2; ++dj)
      for (int dk = 0; dk < 2; ++dk) {
        const double* c = pn.ranvec[pn.perm_x[(i + di) & 255] ^ pn.perm_y[(j + dj) & 255] ^ pn.perm_z[(k + dk) & 255]];
        V3 wv = v3(u - (double)di, v - (double)dj, w - (double)dk);
        accum += ((double)di * uu + (1.0 - (double)di) * (1.0 - uu)) *
                 ((double)dj * vv + (1.0 - (double)dj) * (1.0 - vv)) *
                 ((double)dk * ww + (1.0 - (double)dk) * (1.0 - ww)) * dot(wv, v3(c[0], c[1], c[2]));
      }
  return accum;
}
double perlin_turb(const yart_perlin& pn, uint32_t type, V3 p, int depth) { // texture.rs:231-243
  double accum = 0.0, weight = 1.0;
  V3 tp = p;
  for (int i = 0; i < depth; ++i) {
    accum += weight * perlin_noise(pn, type, tp);
    weight *= 0.5;
    tp = tp * 2.0;
  }
  return std::fabs(accum);
}

double texture_value(const Scene& s, uint32_t tex, const Ray& ray_in, const HitRec& rec) {
  const yart_texture& t = s.textures[tex];
  const double white[3] = {1.0, 1.0, 1.0};
  switch (t.kind) {
    case YART_TEX_SOLID: return rgb_reflect(t.rgb_a, ray_in.wl); // texture.rs:36-40
    case YART_TEX_CHECKER: {                                     // texture.rs:57-68
      double sines = lm_sin(10.0 * rec.p.x) * lm_sin(10.0 * rec.p.y) * lm_sin(10.0 * rec.p.z);
      return sines < 0.0 ? rgb_reflect(t.rgb_a, ray_in.wl) : rgb_reflect(t.rgb_b, ray_in.wl);
    }
    case YART_TEX_NOISE: { // texture.rs:260-284
      const yart_perlin& pn = s.perlins[t.perlin];
      if (t.noise_type == YART_NOISE_NET)
        return rgb_reflect(white, ray_in.wl) * perlin_turb(pn, t.noise_type, rec.p * t.scale, 7);
      if (t.noise_type == YART_NOISE_MARBLE)
        return rgb_reflect(white, ray_in.wl) * 0.5 *
               (1.0 + lm_sin(t.scale * rec.p.z + 10.0 * perlin_turb(pn, t.noise_type, rec.p, 7)));
      return rgb_reflect(white, ray_in.wl) * 0.5 * (1.0 + perlin_noise(pn, t.noise_type, rec.p * t.scale));
    }
    case YART_TEX_IMAGE: { // texture.rs:313-345
      const Scene::Image& im = s.images[t.image];
      if (im.data.empty()) return 1.0;
      double uu = rec.u < 0.0 ? 0.0 : (rec.u > 1.0 ? 1.0 : rec.u); // f64::clamp (NaN stays NaN)
      double vc = rec.v < 0.0 ? 0.0 : (rec.v > 1.0 ? 1.0 : rec.v);
      double vv = 1.0 - vc;
      uint32_t i = f64_as_u32(uu * (double)im.w);
      uint32_t j = f64_as_u32(vv * (double)im.h);
      if (i >= im.w) i = im.w - 1;
      if (j >= im.h) j = im.h - 1;
      const double cs = 1.0 / 255.0;
      size_t px = (size_t)j * 3 * im.w + (size_t)i * 3;
      const double rgb[3] = {cs * (double)im.data[px], cs * (double)im.data[px + 1], cs * (double)im.data[px + 2]};
      return rgb_reflect(rgb, ray_in.wl);
    }
    default: return 0.0;
  }
}

// ---------------------------------------------------------------------------------------
// ONB, PDFs, light sampling (onb.rs, pdf.rs, sphere.rs:95-118, aarect.rs:148-171)
// ---------------------------------------------------------------------------------------
struct Onb {
  V3 u, v, w;
};
inline Onb onb_from_w(V3 n) { // onb.rs:10-21
  Onb b;
  b.w = unit_vector(n);
  V3 a = std::fabs(b.w.x) > 0.9 ? v3(0.0, 1.0, 0.0) : v3(1.0, 0.0, 0.0);
  b.v = unit_vector(cross(b.w, a));
  b.u = cross(b.w, b.v);
  return b;
}
inline V3 onb_local(const Onb& b, V3 a) { return a.x * b.u + a.y * b.v + a.z * b.w; } // onb.rs:23-25

double light_pdf_value(const yart_object& l, V3 origin, V3 direction) {
  HitRec rec;
  Ray r{origin, direction, 0.0, 0.0};
  if (l.wrap != 0) return 0.0; // wrappers do not forward pdf_value (trait default hittable.rs:28-30)
  if (l.kind == YART_OBJ_SPHERE) { // sphere.rs:95-110
    if (!hit_sphere(l, r, 0.001, kInf, rec)) return 0.0;
    const V3 center = v3(l.p[0], l.p[1], l.p[2]);
    const double radius = l.p[3];
    double cos_theta_max = std::sqrt(1.0 - radius * radius / length_squared(center - origin));
    double solid_angle = 2.0 * kPi * (1.0 - cos_theta_max);
    return 1.0 / solid_angle;
  }
  if (l.kind == YART_OBJ_XZ_RECT) { // aarect.rs:148-162
    if (!hit_rect(l, r, 0.001, kInf, rec)) return 0.0;
    double area = (l.p[1] - l.p[0]) * (l.p[3] - l.p[2]);
    double distance_squared = rec.t * rec.t * length_squared(direction);
    double cosine = std::fabs(dot(direction, rec.normal)) / length(direction);
    return distance_squared / (cosine * area);
  }
  return 0.0;
}
V3 light_random(const yart_object& l, V3 origin, double r1, double r2) {
  if (l.wrap == 0 && l.kind == YART_OBJ_SPHERE) { // sphere.rs:112-118 + random_to_sphere :11-21
    const V3 center = v3(l.p[0], l.p[1], l.p[2]);
    const double radius = l.p[3];
    V3 direction = center - origin;
    double distance_squared = length_squared(direction);
    Onb uvw = onb_from_w(direction);
    double z = 1.0 + r2 * (std::sqrt(1.0 - radius * radius / distance_squared) - 1.0);
    double phi = 2.0 * kPi * r1;
    double x = lm_cos(phi) * std::sqrt(1.0 - z * z);
    double y = lm_sin(phi) * std::sqrt(1.0 - z * z);
    return onb_local(uvw, v3(x, y, z));
  }
  if (l.wrap == 0 && l.kind == YART_OBJ_XZ_RECT) { // aarect.rs:164-171
    V3 pt = v3(l.p[0] + (l.p[1] - l.p[0]) * r1, l.p[4], l.p[2] + (l.p[3] - l.p[2]) * r2);
    return pt - origin;
  }
  return v3(1.0, 0.0, 0.0); // trait default (hittable.rs:32-34)
}
double lights_pdf_value(const Scene& s, V3 origin, V3 direction) { // hittable.rs:103-111
  double weight = 1.0 / (double)s.lights.size();
  double sum = 0.0;
  for (size_t i = 0; i < s.lights.size(); ++i) sum += weight * light_pdf_value(s.lights[i], origin, direction);
  return sum;
}
// hittable.rs:113-122.  unbiased = YART_FLAG_UNBIASED_LIGHT_PICK (not the reference): uniform over all lights.
V3 lights_random(const Scene& s, V3 origin, double u_pick, double r1, double r2, bool unbiased) {
  size_t n = s.lights.size();
  if (n == 0) return v3(1.0, 0.0, 0.0);
  if (n == 1) return light_random(s.lights[0], origin, r1, r2);
  size_t m = unbiased ? n : n - 1;               // gen_range(0..len-1): never the last light
  size_t k = (size_t)(u_pick * (double)m);
  if (k > m - 1) k = m - 1;
  return light_random(s.lights[k], origin, r1, r2);
}

// ---------------------------------------------------------------------------------------
// Materials (material.rs) and the integrator (main.rs:526-588)
// ---------------------------------------------------------------------------------------
inline V3 reflect(V3 v, V3 n) { return v - 2.0 * dot(v, n) * n; } // material.rs:75-77
inline bool refract(V3 v, V3 n, double ni_over_nt, V3& out) {      // material.rs:195-205
  V3 uv = unit_vector(v);
  double dt = dot(uv, n);
  double disc = 1.0 - ni_over_nt * ni_over_nt * (1.0 - dt * dt);
  if (disc > 0.0) {
    out = (uv - n * dt) * ni_over_nt - n * std::sqrt(disc);
    return true;
  }
  return false;
}
inline double powi5(double x) { // f64::powi(x, 5) = llvm.powi: x * (x^2)^2 by squaring
  double x2 = x * x;
  double x4 = x2 * x2;
  return x4 * x;
}
inline double schlick(double cosine, double ref_idx) { // material.rs:207-211
  double r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
  r0 = r0 * r0;
  return r0 + (1.0 - r0) * powi5(1.0 - cosine);
}
inline double sellmeier_index(const yart_material& m, double wl) { // material.rs:247-253
  double wl2 = wl * wl;
  double n2 = 1.0 + m.sellmeier_b[0] * wl2 / (wl2 - m.sellmeier_c[0]) +
              m.sellmeier_b[1] * wl2 / (wl2 - m.sellmeier_c[1]) +
              m.sellmeier_b[2] * wl2 / (wl2 - m.sellmeier_c[2]);
  return std::sqrt(n2);
}

struct Factor {
  double atten, spdf, pdf;
  bool diffuse;
  bool roulette = false; // (flag only) atten holds the survival probability q: L = L / q
};

// ray_reflectance (main.rs:537-588), unrolled into a loop that records the per-bounce factors
// and then folds them innermost-first so the multiplication order equals the recursion's.
// `flags`: the better-sampling switches of yart_render_opts (YART_FLAG_UNBIASED_LIGHT_PICK / RUSSIAN_ROULETTE /
// DEPTH_ZERO_BLACK); 0 = the reference's estimator.
double ray_reflectance(const HitCtx& c, Ray ray, const Rng& rng, uint32_t max_depth, uint32_t* n_rays,
                       std::vector<Factor>& factors, std::vector<yart_ray>* dump, uint32_t flags = 0) {
  const Scene& s = *c.s;
  factors.clear();
  double terminal = (flags & YART_FLAG_DEPTH_ZERO_BLACK) ? 0.0 : 1.0; // depth == 0 returns 1.0 (main.rs:544-546)
  double run = 1.0; // running throughput, front to back like the device's: only the roulette looks at it
  bool cut = false;
  auto roulette = [&](uint32_t bounce) { // after a scattering bounce; true = the path was cut
    if (!(flags & YART_FLAG_RUSSIAN_ROULETTE) || bounce < YART_RR_FIRST_BOUNCE) return false;
    const double q = run < YART_RR_MIN_SURVIVAL ? YART_RR_MIN_SURVIVAL : (run > 1.0 ? 1.0 : run);
    double u_rr, unused;
    rng.draw(bounce, YART_SLOT_RR, u_rr, unused);
    if (u_rr >= q) return true;
    run = run / q;
    Factor f{q, 0, 0, false};
    f.roulette = true;
    factors.push_back(f);
    return false;
  };
  for (uint32_t bounce = 1; bounce <= max_depth; ++bounce) {
    HitRec rec;
    if (n_rays) (*n_rays)++;
    if (dump) {
      yart_ray yr = {{ray.o.x, ray.o.y, ray.o.z}, {ray.d.x, ray.d.y, ray.d.z}};
      dump->push_back(yr);
    }
    if (!world_hit(c, ray, 0.001, kInf, &rng, bounce, rec)) {
      terminal = rgb_reflect(s.background, ray.wl); // main.rs:587
      break;
    }
    const yart_material& mat = s.materials[rec.material];
    double emitted = 0.0;
    if (mat.kind == YART_MAT_DIFFUSE_LIGHT) // material.rs:347-355
      emitted = rec.front_face ? texture_value(s, mat.texture, ray, rec) : 0.0;
    if (mat.kind == YART_MAT_NONE || mat.kind == YART_MAT_DIFFUSE_LIGHT) { // scatter -> None
      terminal = emitted;
      break;
    }
    if (mat.kind == YART_MAT_METAL) { // material.rs:79-95
      V3 reflected = reflect(unit_vector(ray.d), rec.normal);
      V3 dir = reflected + mat.fuzz * random_in_unit_sphere(rng, bounce);
      factors.push_back(Factor{texture_value(s, mat.texture, ray, rec), 0, 0, false});
      run = run * factors.back().atten;
      ray = Ray{rec.p, dir, ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    if (mat.kind == YART_MAT_ISOTROPIC) { // material.rs:368-381
      factors.push_back(Factor{texture_value(s, mat.texture, ray, rec), 0, 0, false});
      run = run * factors.back().atten;
      ray = Ray{rec.p, random_in_unit_sphere(rng, bounce), ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    if (mat.kind == YART_MAT_DIELECTRIC) { // material.rs:213-301
      double n = sellmeier_index(mat, ray.wl);
      V3 outward;
      double ni_over_nt, cosine;
      double ddn = dot(ray.d, rec.normal);
      if (ddn > 0.0) {
        outward = -rec.normal;
        ni_over_nt = n;
        cosine = n * dot(ray.d, rec.normal) / length(ray.d);
      } else {
        outward = rec.normal;
        ni_over_nt = 1.0 / n;
        cosine = -dot(ray.d, rec.normal) / length(ray.d);
      }
      V3 refracted, dir;
      if (refract(ray.d, outward, ni_over_nt, refracted)) {
        double u0, u1;
        rng.draw(bounce, YART_SLOT_DIELECTRIC, u0, u1);
        dir = (u0 < schlick(cosine, n)) ? reflect(ray.d, rec.normal) : refracted;
      } else {
        dir = reflect(ray.d, rec.normal);
      }
      factors.push_back(Factor{1.0, 0, 0, false});
      run = run * 1.0;
      ray = Ray{rec.p, dir, ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    // Lambertian (material.rs:44-61) through the mixture pdf (main.rs:560-581)
    double atten = texture_value(s, mat.texture, ray, rec);
    Onb uvw = onb_from_w(rec.normal); // CosinePDF::new
    double u_mix, u_pick, r1, r2;
    rng.draw(bounce, YART_SLOT_MIX, u_mix, u_pick);
    rng.draw(bounce, YART_SLOT_DIR, r1, r2);
    auto cosine_dir = [&]() { // random_cosine_direction (pdf.rs:15-25)
      double z = std::sqrt(1.0 - r2);
      double phi = 2.0 * kPi * r1;
      double x = lm_cos(phi) * std::sqrt(r2);
      double y = lm_sin(phi) * std::sqrt(r2);
      return onb_local(uvw, v3(x, y, z));
    };
    V3 dir;
    const bool have_lights = !s.lights.empty();
    if (u_mix < 0.5) dir = have_lights ? lights_random(s, rec.p, u_pick, r1, r2, (flags & YART_FLAG_UNBIASED_LIGHT_PICK) != 0) : cosine_dir();
    else dir = cosine_dir();
    Ray sc{rec.p, dir, ray.time, ray.wl};
    double cosv = dot(unit_vector(dir), uvw.w); // CosinePDF::value (pdf.rs:39-47)
    double cos_pdf = cosv <= 0.0 ? 0.0 : cosv / kPi;
    double p0 = have_lights ? lights_pdf_value(s, rec.p, dir) : cos_pdf;
    double pdf_val = 0.5 * p0 + 0.5 * cos_pdf; // MixurePDF::value (pdf.rs:87-89)
    if (!std::isfinite(pdf_val) || pdf_val <= 0.0) { // main.rs:574-576
      terminal = emitted;
      break;
    }
    double cs = dot(rec.normal, unit_vector(sc.d)); // Lambertian::scatter_pdf (material.rs:53-60)
    double spdf = cs < 0.0 ? 0.0 : cs / kPi;
    factors.push_back(Factor{atten, spdf, pdf_val, true});
    run = run * atten * spdf / pdf_val;
    ray = sc;
    if (roulette(bounce)) { cut = true; break; }
  }
  double L = cut ? 0.0 : terminal;
  for (size_t i = factors.size(); i-- > 0;) {
    const Factor& f = factors[i];
    if (f.roulette) L = L / f.atten;
    else if (f.diffuse) L = f.atten * L * f.spdf / f.pdf; // main.rs:578-581
    else L = f.atten * L;                             // main.rs:553-554
  }
  return L;
}

// Camera (camera.rs:41-94)
struct Camera {
  V3 llc, horizontal, vertical, origin, u, v, w;
  double lens_radius, time0, time1;
};
Camera make_camera(const yart_camera& c) {
  Camera k;
  V3 lookfrom = v3(c.lookfrom[0], c.lookfrom[1], c.lookfrom[2]);
  V3 lookat = v3(c.lookat[0], c.lookat[1], c.lookat[2]);
  V3 vup = v3(c.vup[0], c.vup[1], c.vup[2]);
  double theta = c.vfov_degrees * kPi / 180.0;
  double h = std::tan(theta / 2.0);
  double vh = 2.0 * h;
  double vw = c.aspect_ratio * vh;
  k.w = unit_vector(lookfrom - lookat);
  k.u = unit_vector(cross(vup, k.w));
  k.v = cross(k.w, k.u);
  k.origin = lookfrom;
  k.horizontal = c.focus_dist * vw * k.u;
  k.vertical = c.focus_dist * vh * k.v;
  k.llc = k.origin - vdiv(k.horizontal, 2.0) - vdiv(k.vertical, 2.0) - c.focus_dist * k.w;
  k.lens_radius = c.aperture / 2.0;
  k.time0 = c.time0;
  k.time1 = c.time1;
  return k;
}
Ray camera_ray(const Camera& k, const Rng& rng, uint32_t px, uint32_t py, uint32_t W, uint32_t H) {
  double jx, jy, uwl, ut;
  rng.draw(0, YART_SLOT_CAM_JITTER, jx, jy);
  rng.draw(0, YART_SLOT_CAM_WL_TIME, uwl, ut);
  double target_x = (double)px + jx; // main.rs:693-696
  double u = target_x / (double)(W - 1);
  double target_y = (double)py + jy;
  double v = 1.0 - target_y / (double)(H - 1);
  double wl = MIN_LAMBDA + (MAX_LAMBDA - MIN_LAMBDA) * uwl; // gen_wavelength (color.rs:20-23)
  V3 disk = v3(0, 0, 0);                                     // random_in_unit_disk (camera.rs:25-33)
  for (uint32_t i = 0; i < YART_MAX_REJECT; ++i) {
    double a, b;
    rng.draw(0, YART_SLOT_CAM_LENS + i, a, b);
    V3 p = v3(-1.0 + 2.0 * a, -1.0 + 2.0 * b, 0.0);
    if (length_squared(p) >= 1.0) continue;
    disk = p;
    break;
  }
  V3 rd = k.lens_radius * disk;
  V3 offset = k.u * rd.x + k.v * rd.y;
  Ray r;
  r.o = k.origin + offset;
  r.d = k.llc + u * k.horizontal + v * k.vertical - k.origin - offset;
  r.time = k.time0 + (k.time1 - k.time0) * ut;
  r.wl = wl;
  return r;
}

// one sample of the loop at main.rs:690-707, before sanitising
void render_sample(const HitCtx& c, const Camera& cam, const yart_render_opts& o, uint32_t px, uint32_t py,
                   uint32_t sample, double xyz[3], uint32_t* n_rays, std::vector<Factor>& scratch,
                   std::vector<yart_ray>* dump) {
  Rng rng = make_rng(o.seed, py * o.width + px, sample);
  Ray r = camera_ray(cam, rng, px, py, o.width, o.height);
  double refl = ray_reflectance(c, r, rng, o.max_depth, n_rays, scratch, dump, o.flags);
  double cie[3];
  xyz_from_wavelength(r.wl, cie); // ray_color (main.rs:526-535)
  xyz[0] = cie[0] * refl; xyz[1] = cie[1] * refl; xyz[2] = cie[2] * refl;
}

// the reference only renders W/8 x H/8 tiles at (W*col/8, H*row/8) (main.rs:636-646)
inline bool pixel_is_rendered(uint32_t x, uint32_t W) {
  uint32_t cw = W / 8;
  for (uint32_t col = 0; col < 8; ++col) {
    uint32_t x0 = (uint32_t)((uint64_t)W * col / 8);
    if (x >= x0 && x < x0 + cw) return true;
  }
  return false;
}

} // namespace

struct orc_scene {
  Scene s;
};

// =========================================================================================
// C entry points
// =========================================================================================
extern "C" {

const char* orc_last_error(void) { return g_err.c_str(); }

int orc_scene_create(const yart_scene_desc* d, orc_scene** out) {
  if (!d || !out) { g_err = "null argument"; return YART_ERR_INVALID; }
  orc_scene* h = new orc_scene();
  Scene& s = h->s;
  s.objects.assign(d->objects, d->objects + d->n_objects);
  s.lights.assign(d->lights, d->lights + d->n_lights);
  s.materials.assign(d->materials, d->materials + d->n_materials);
  s.textures.assign(d->textures, d->textures + d->n_textures);
  s.perlins.assign(d->perlins, d->perlins + d->n_perlins);
  for (uint32_t i = 0; i < d->n_images; ++i) {
    Scene::Image im;
    im.w = d->images[i].width;
    im.h = d->images[i].height;
    im.data.assign(d->images[i].rgb8, d->images[i].rgb8 + (size_t)im.w * im.h * 3);
    s.images.push_back(std::move(im));
  }
  for (uint32_t i = 0; i < d->n_groups; ++i)
    s.groups.emplace_back(d->groups[i].members, d->groups[i].members + d->groups[i].n_members);
  s.meshes.resize(d->n_meshes);
  for (uint32_t i = 0; i < d->n_meshes; ++i) build_mesh(d->meshes[i], s.meshes[i]);
  for (int k = 0; k < 3; ++k) s.background[k] = d->background_rgb[k];
  for (const yart_object& o : s.objects) {
    bool bad = (o.kind == YART_OBJ_MESH && o.index >= s.meshes.size()) ||
               (o.kind == YART_OBJ_GROUP && o.index >= s.groups.size()) || o.material >= s.materials.size();
    if (bad) { delete h; g_err = "object refers to a missing mesh/group/material"; return YART_ERR_INVALID; }
  }
  *out = h;
  return YART_OK;
}
void orc_scene_free(orc_scene* s) { delete s; }

int orc_qbvh_info_get(const orc_scene* s, uint32_t mesh, orc_qbvh_info* out) {
  if (!s || mesh >= s->s.meshes.size()) { g_err = "bad mesh"; return YART_ERR_INVALID; }
  const Mesh& m = s->s.meshes[mesh];
  memset(out, 0, sizeof(*out));
  out->n_nodes = (uint32_t)m.nodes.size();
  out->n_leaves = m.n_leaves;
  out->n_tris = (uint32_t)m.tris.size();
  for (int i = 0; i < 5; ++i) out->leaves_by_count[i] = m.leaves_by_count[i];
  out->empty_children = m.empty_children;
  if (!m.nodes.empty()) { // L4QBVH::bounding_box (qbvh.rs:365-379)
    const Node& r = m.nodes.back();
    for (int a = 0; a < 3; ++a) {
      double mn = r.bmin[a][0], mx = r.bmax[a][0];
      for (int k = 1; k < 4; ++k) { mn = std::fmin(mn, r.bmin[a][k]); mx = std::fmax(mx, r.bmax[a][k]); }
      out->bbox_min[a] = mn;
      out->bbox_max[a] = mx;
    }
  }
  return YART_OK;
}
int orc_qbvh_node(const orc_scene* s, uint32_t mesh, uint32_t i, double* boxes24, uint32_t* children4, uint32_t* axes3) {
  if (!s || mesh >= s->s.meshes.size() || i >= s->s.meshes[mesh].nodes.size()) { g_err = "bad node"; return YART_ERR_INVALID; }
  const Node& n = s->s.meshes[mesh].nodes[i];
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 4; ++k) { boxes24[a * 4 + k] = n.bmin[a][k]; boxes24[12 + a * 4 + k] = n.bmax[a][k]; }
  for (int k = 0; k < 4; ++k) children4[k] = n.child[k];
  for (int k = 0; k < 3; ++k) axes3[k] = n.axis[k];
  return YART_OK;
}
int orc_qbvh_tri_order(const orc_scene* s, uint32_t mesh, uint32_t* out) {
  if (!s || mesh >= s->s.meshes.size()) { g_err = "bad mesh"; return YART_ERR_INVALID; }
  const Mesh& m = s->s.meshes[mesh];
  for (size_t i = 0; i < m.tris.size(); ++i) out[i] = m.tris[i].orig;
  return YART_OK;
}

static void fill_hit(yart_hit& h, bool some, const HitRec& rec) {
  if (!some) {
    h.t = kInf; h.u = h.v = 0.0; h.prim_id = YART_MISS; h.obj_id = YART_MISS; h.front_face = 0; h._pad = 0;
    return;
  }
  h.t = rec.t; h.prim_id = rec.prim; h.obj_id = rec.obj; h.front_face = rec.front_face ? 1u : 0u; h._pad = 0;
  h.u = rec.bu; h.v = rec.bv;
}

int orc_closest_hit(const orc_scene* s, uint32_t target, const yart_ray* rays, uint64_t n, double t_min,
                    double t_max, uint32_t order, yart_hit* hits, orc_counters* counters, int n_threads) {
  if (!s || (!rays && n) || (!hits && n)) { g_err = "null argument"; return YART_ERR_INVALID; }
  if (target != YART_TARGET_WORLD && target >= s->s.meshes.size()) { g_err = "bad target"; return YART_ERR_INVALID; }
  if (n_threads < 1) n_threads = 1;
  std::vector<Counters> cs((size_t)n_threads);
  auto work = [&](int tid) {
    Counters* cnt = &cs[(size_t)tid];
    HitCtx c{&s->s, order, cnt};
    uint64_t lo = n * (uint64_t)tid / (uint64_t)n_threads, hi = n * (uint64_t)(tid + 1) / (uint64_t)n_threads;
    for (uint64_t i = lo; i < hi; ++i) {
      Ray r{v3(rays[i].origin[0], rays[i].origin[1], rays[i].origin[2]),
            v3(rays[i].direction[0], rays[i].direction[1], rays[i].direction[2]), 0.0, 550.0};
      HitRec rec;
      bool some;
      if (target == YART_TARGET_WORLD) {
        Rng rng = make_rng(0, (uint32_t)i, 0);
        some = world_hit(c, r, t_min, t_max, &rng, 1, rec);
      } else {
        const Mesh& m = s->s.meshes[target];
        MeshHit mh = (order == YART_ORDER_NEAR) ? qbvh_hit<true>(m, r, t_min, t_max, cnt)
                                                : qbvh_hit<false>(m, r, t_min, t_max, cnt);
        cnt->rays++;
        some = mh.some;
        if (some) { mesh_hit_record(m, mh, r, 0, rec); rec.obj = 0; }
      }
      fill_hit(hits[i], some, rec);
    }
  };
  if (n_threads == 1) {
    work(0);
  } else {
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
  }
  if (counters) {
    memset(counters, 0, sizeof(*counters));
    for (const Counters& c : cs) {
      counters->rays += c.rays; counters->node_visits += c.node_visits; counters->leaf_visits += c.leaf_visits;
      counters->tri_tests += c.tri_tests;
      if (c.max_stack > counters->max_stack) counters->max_stack = c.max_stack;
    }
  }
  return YART_OK;
}

// Triangle::hit arithmetic (triangle.rs:48-79) on every triangle
static bool tri_test(const Tri& tr, const Ray& r, double t_min, double t_max, double& t, double& u, double& v) {
  V3 e1 = tr.v[1] - tr.v[0], e2 = tr.v[2] - tr.v[0];
  V3 h = cross(r.d, e2);
  double a = dot(e1, h);
  if (a > -kEps && a < kEps) return false;
  double f = 1.0 / a;
  V3 s = r.o - tr.v[0];
  u = f * dot(s, h);
  if (u < 0.0 || u > 1.0) return false;
  V3 q = cross(s, e1);
  v = f * dot(r.d, q);
  if (v < 0.0 || u + v > 1.0) return false;
  t = f * dot(e2, q);
  if (t < t_min || t > t_max) return false;
  return true;
}

int orc_brute_force_hit(const orc_scene* s, uint32_t mesh, const yart_ray* rays, uint64_t n, double t_min,
                        double t_max, yart_hit* hits, uint32_t* n_ties) {
  if (!s || mesh >= s->s.meshes.size()) { g_err = "bad mesh"; return YART_ERR_INVALID; }
  const Mesh& m = s->s.meshes[mesh];
  for (uint64_t i = 0; i < n; ++i) {
    Ray r{v3(rays[i].origin[0], rays[i].origin[1], rays[i].origin[2]),
          v3(rays[i].direction[0], rays[i].direction[1], rays[i].direction[2]), 0.0, 550.0};
    double bt = kInf, bu = 0, bv = 0;
    uint32_t bid = YART_MISS, ties = 0;
    for (const Tri& tr : m.tris) {
      double t, u, v;
      if (!tri_test(tr, r, t_min, t_max, t, u, v)) continue;
      if (t < bt) { bt = t; bu = u; bv = v; bid = tr.orig; ties = 1; }
      else if (t == bt) { ties++; if (tr.orig < bid) { bid = tr.orig; bu = u; bv = v; } }
    }
    hits[i].t = bt; hits[i].u = bu; hits[i].v = bv; hits[i].prim_id = bid;
    hits[i].obj_id = bid == YART_MISS ? YART_MISS : 0; hits[i].front_face = 0; hits[i]._pad = 0;
    if (n_ties) n_ties[i] = ties;
  }
  return YART_OK;
}

int orc_tie_set(const orc_scene* s, uint32_t mesh, const yart_ray* ray, double t_min, double t_max,
                uint32_t* ids, uint32_t cap, uint32_t* n_out) {
  if (!s || mesh >= s->s.meshes.size()) { g_err = "bad mesh"; return YART_ERR_INVALID; }
  const Mesh& m = s->s.meshes[mesh];
  Ray r{v3(ray->origin[0], ray->origin[1], ray->origin[2]), v3(ray->direction[0], ray->direction[1], ray->direction[2]), 0.0, 550.0};
  double bt = kInf;
  for (const Tri& tr : m.tris) {
    double t, u, v;
    if (tri_test(tr, r, t_min, t_max, t, u, v) && t < bt) bt = t;
  }
  uint32_t k = 0;
  for (const Tri& tr : m.tris) {
    double t, u, v;
    if (tri_test(tr, r, t_min, t_max, t, u, v) && t == bt) {
      if (k < cap) ids[k] = tr.orig;
      k++;
    }
  }
  *n_out = k;
  return YART_OK;
}

int orc_render_tiles(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, double* film,
                     yart_stats* stats, int n_threads, uint32_t tile_begin, uint32_t tile_end);

int orc_render(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, double* film,
               yart_stats* stats, int n_threads) {
  return orc_render_tiles(s, cam, o, film, stats, n_threads, 0, 64);
}

// the same loop restricted to jobs [tile_begin, tile_end) of the 64 tile jobs (main.rs:636-646),
// so a bounded SAMPLE of a big frame can be timed as the CPU baseline
int orc_render_tiles(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, double* film,
                     yart_stats* stats, int n_threads, uint32_t tile_begin, uint32_t tile_end) {
  if (!s || !cam || !o || !film) { g_err = "null argument"; return YART_ERR_INVALID; }
  if (o->width < 2 || o->height < 2) { g_err = "width/height must be >= 2"; return YART_ERR_INVALID; }
  if (n_threads < 1) n_threads = 1;
  const Camera k = make_camera(*cam);
  const uint32_t W = o->width, H = o->height;
  if (tile_end > 64) tile_end = 64;
  // jobs are handed out in row-bands of each tile so a small tile range still feeds all workers
  std::atomic<uint32_t> next_job(0);
  std::atomic<uint64_t> total_rays(0), total_paths(0);
  const uint32_t bands = 8;
  const uint32_t n_jobs = (tile_end > tile_begin ? tile_end - tile_begin : 0) * bands;
  auto worker = [&]() {
    std::vector<Factor> scratch;
    HitCtx c{&s->s, o->order, nullptr};
    uint64_t rays = 0, paths = 0;
    for (;;) {
      uint32_t jb = next_job.fetch_add(1);
      if (jb >= n_jobs) break;
      uint32_t job = tile_begin + jb / bands, band = jb % bands;
      uint32_t col = job / 8, row = job % 8; // main.rs:636-646
      uint32_t crop_x = (uint32_t)((uint64_t)W * col / 8), crop_y = (uint32_t)((uint64_t)H * row / 8);
      uint32_t cw = W / 8, ch = H / 8;
      for (uint32_t y = ch * band / bands; y < ch * (band + 1) / bands; ++y)
        for (uint32_t x = 0; x < cw; ++x) {
          uint32_t px = x + crop_x, py = y + crop_y;
          double* pix = film + ((size_t)py * W + px) * 3;
          for (uint32_t sm = o->sample_begin; sm < o->sample_end; ++sm) {
            double xyz[3], clean[3];
            uint32_t nr = 0;
            render_sample(c, k, *o, px, py, sm, xyz, &nr, scratch, nullptr);
            sanitize_sample_xyz(xyz, clean);
            pix[0] += clean[0]; pix[1] += clean[1]; pix[2] += clean[2]; // main.rs:707
            rays += nr;
            paths++;
          }
        }
    }
    total_rays += rays;
    total_paths += paths;
  };
  std::vector<std::thread> th;
  for (int t = 0; t < n_threads; ++t) th.emplace_back(worker);
  for (auto& t : th) t.join();
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->rays = total_rays.load();
    stats->paths = total_paths.load();
  }
  return YART_OK;
}

int orc_film_finalize(const double* film, uint32_t W, uint32_t H, uint32_t spp, uint8_t* rgba) {
  for (uint32_t y = 0; y < H; ++y)
    for (uint32_t x = 0; x < W; ++x) {
      uint8_t* px = rgba + ((size_t)y * W + x) * 4;
      if (!pixel_is_rendered(x, W) || !pixel_is_rendered(y, H)) { px[0] = px[1] = px[2] = px[3] = 0; continue; }
      const double* f = film + ((size_t)y * W + x) * 3;
      // pixel_color_xyz * (MAX_LAMBDA - MIN_LAMBDA) / (CIE_Y_INTERGAL * spp) (main.rs:710-711)
      const double mul = MAX_LAMBDA - MIN_LAMBDA, den = CIE_Y_INTEGRAL * (double)spp;
      V3 c = vdiv(v3(f[0] * mul, f[1] * mul, f[2] * mul), den);
      double xyz[3] = {c.x, c.y, c.z}, rgb[3];
      xyz_into_rgb(xyz, rgb);
      px[0] = clamp_display_channel(gamma_channel(rgb[0]));
      px[1] = clamp_display_channel(gamma_channel(rgb[1]));
      px[2] = clamp_display_channel(gamma_channel(rgb[2]));
      px[3] = 255;
    }
  return YART_OK;
}

int orc_camera_rays(const yart_camera* cam, const yart_render_opts* o, yart_ray* rays, double* wl, double* time) {
  if (!cam || !o || !rays) { g_err = "null argument"; return YART_ERR_INVALID; }
  const Camera k = make_camera(*cam);
  const uint32_t ns = o->sample_end - o->sample_begin;
  for (uint32_t py = 0; py < o->height; ++py)
    for (uint32_t px = 0; px < o->width; ++px)
      for (uint32_t sm = o->sample_begin; sm < o->sample_end; ++sm) {
        Rng rng = make_rng(o->seed, py * o->width + px, sm);
        Ray r = camera_ray(k, rng, px, py, o->width, o->height);
        size_t i = ((size_t)py * o->width + px) * ns + (sm - o->sample_begin);
        rays[i].origin[0] = r.o.x; rays[i].origin[1] = r.o.y; rays[i].origin[2] = r.o.z;
        rays[i].direction[0] = r.d.x; rays[i].direction[1] = r.d.y; rays[i].direction[2] = r.d.z;
        if (wl) wl[i] = r.wl;
        if (time) time[i] = r.time;
      }
  return YART_OK;
}

int orc_dump_path_rays(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, yart_ray* rays,
                       uint64_t cap, uint64_t* n_out) {
  if (!s || !cam || !o || !rays || !n_out) { g_err = "null argument"; return YART_ERR_INVALID; }
  const Camera k = make_camera(*cam);
  std::vector<Factor> scratch;
  std::vector<yart_ray> dump;
  HitCtx c{&s->s, o->order, nullptr};
  uint64_t n = 0;
  for (uint32_t sm = o->sample_begin; sm < o->sample_end && n < cap; ++sm)
    for (uint32_t py = 0; py < o->height && n < cap; ++py)
      for (uint32_t px = 0; px < o->width && n < cap; ++px) {
        double xyz[3];
        dump.clear();
        render_sample(c, k, *o, px, py, sm, xyz, nullptr, scratch, &dump);
        for (const yart_ray& r : dump) {
          if (n >= cap) break;
          rays[n++] = r;
        }
      }
  *n_out = n;
  return YART_OK;
}

int orc_sample_path(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, uint32_t pixel,
                    uint32_t sample, yart_ray* rays, uint64_t cap, uint64_t* n_out) {
  if (!s || !cam || !o || !rays || !n_out) { g_err = "null argument"; return YART_ERR_INVALID; }
  const Camera k = make_camera(*cam);
  std::vector<Factor> scratch;
  std::vector<yart_ray> dump;
  HitCtx c{&s->s, o->order, nullptr};
  double xyz[3];
  render_sample(c, k, *o, pixel % o->width, pixel / o->width, sample, xyz, nullptr, scratch, &dump);
  uint64_t n = std::min<uint64_t>(cap, dump.size());
  for (uint64_t i = 0; i < n; ++i) rays[i] = dump[i];
  *n_out = n;
  return YART_OK;
}

int orc_sample(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, uint32_t pixel,
               uint32_t sample, double* xyz3, uint32_t* n_rays) {
  if (!s || !cam || !o || !xyz3) { g_err = "null argument"; return YART_ERR_INVALID; }
  const Camera k = make_camera(*cam);
  std::vector<Factor> scratch;
  HitCtx c{&s->s, o->order, nullptr};
  uint32_t nr = 0;
  render_sample(c, k, *o, pixel % o->width, pixel / o->width, sample, xyz3, &nr, scratch, nullptr);
  if (n_rays) *n_rays = nr;
  return YART_OK;
}

void orc_sanitize_sample_xyz(const double* in3, double* out3) { sanitize_sample_xyz(in3, out3); }
uint8_t orc_clamp_display_channel(double c) { return clamp_display_channel(c); }
void orc_gamma_corrected(const double* rgb3, double* out3) {
  for (int i = 0; i < 3; ++i) out3[i] = gamma_channel(rgb3[i]);
}
double orc_rgb_reflect(const double* rgb3, double wavelength) { return rgb_reflect(rgb3, wavelength); }
void orc_xyz_from_wavelength(double wavelength, double* xyz3) { xyz_from_wavelength(wavelength, xyz3); }
void orc_xyz_into_rgb(const double* xyz3, double* rgb3) { xyz_into_rgb(xyz3, rgb3); }
double orc_sellmeier_index(const yart_material* m, double wavelength) { return sellmeier_index(*m, wavelength); }
int orc_push_hit_children(uint32_t* stack, uint32_t* cursor, const uint32_t* children4, const uint32_t* order4,
                          const uint8_t* hits4) {
  for (int j = 0; j < 4; ++j) { // qbvh.rs:25-30
    uint32_t i = order4[j];
    if (hits4[i]) {
      stack[*cursor] = children4[i];
      *cursor += 1;
    }
  }
  return YART_OK;
}
void orc_philox4x32_10(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4) { philox(ctr4, key2, out4); }
void orc_uniform2(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t slot, double* u2) {
  Rng r = make_rng(seed, pixel, sample);
  r.draw(bounce, slot, u2[0], u2[1]);
}

} // extern "C"
