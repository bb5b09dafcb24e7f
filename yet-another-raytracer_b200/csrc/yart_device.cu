// yart_device.cu -- the device half of the C ABI (include/yart.h): context, scene upload,
// yart_closest_hit, yart_occluded, yart_render, yart_film_finalize, yart_generate_camera_rays.
//
// There is no CPU fallback anywhere in this file: every entry point launches the sm_100a
// kernels of device_trace.cuh / device_shade.cuh or fails with YART_ERR_CUDA.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/yart_spectral_tables.h"
#include "device_build.h"
#include "device_occlude.h"
#include "device_shade.cuh"
#include "host_common.h"

namespace yart {

// ---------------------------------------------------------------------------------------------
// k_export: DevHit -> yart_hit for yart_closest_hit: original triangle id and front_face as the
// reference's HitRecord would carry them (qbvh.rs:452-489, triangle.rs:80-91 etc.)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_export(const DevScene S, const yart_ray* rays, const DevHit* hits, yart_hit* out_hits,
                                                 uint64_t n) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const DevHit h = hits[i];
    yart_hit out;
    if (h.obj == YART_MISS) {
      out.t = d_inf(); out.u = 0.0; out.v = 0.0; out.prim_id = YART_MISS; out.obj_id = YART_MISS; out.front_face = 0;
      out._pad = 0;
      out_hits[i] = out;
      continue;
    }
    const yart_ray wr = rays[i];
    const D3 wo = d3(wr.origin[0], wr.origin[1], wr.origin[2]);
    const D3 wd = d3(wr.direction[0], wr.direction[1], wr.direction[2]);
    const yart_object& o = S.objects[h.obj];
    HitRec rec; // rebuild the HitRecord of this object to get front_face exactly as the reference computes it
    world_record(S, h, wo, wd, 0.0, rec);
    out.t = h.t; out.u = h.bu; out.v = h.bv; out.obj_id = h.obj; out.front_face = rec.front_face ? 1u : 0u; out._pad = 0;
    if (o.wrap & YART_WRAP_MEDIUM) {
      out.prim_id = 0;
    } else if (o.kind == YART_OBJ_MESH) {
      const DevMesh m = S.meshes[o.index];
      out.prim_id = __float_as_uint(__ldg(m.tris + (size_t)h.prim * 3).w); // FlatTri.orig
    } else if (o.kind == YART_OBJ_GROUP) {
      out.prim_id = S.groups[o.index].member_orig[h.prim >> 3];
    } else {
      out.prim_id = h.prim;
    }
    out_hits[i] = out;
  }
}

// yart_closest_hit_f32: DevHit -> yart_hit_f32 (values rounded to nearest f32; original triangle id as k_export)
__global__ void __launch_bounds__(256) k_export_f32(const DevScene S, const yart_object* objects, const DevHit* hits, yart_hit_f32* out_hits,
                                                     uint64_t n) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const DevHit h = hits[i];
    yart_hit_f32 out;
    if (h.obj == YART_MISS) {
      out.t = __int_as_float(0x7f800000); out.u = 0.f; out.v = 0.f; out.prim_id = YART_MISS;
    } else {
      const yart_object& o = objects[h.obj];
      out.t = (float)h.t; out.u = (float)h.bu; out.v = (float)h.bv;
      if (o.wrap & YART_WRAP_MEDIUM) out.prim_id = 0;
      else if (o.kind == YART_OBJ_MESH) out.prim_id = __float_as_uint(__ldg(S.meshes[o.index].tris + (size_t)h.prim * 3).w);
      else if (o.kind == YART_OBJ_GROUP) out.prim_id = S.groups[o.index].member_orig[h.prim >> 3];
      else out.prim_id = h.prim;
    }
    out_hits[i] = out;
  }
}

// yart_dump_path_rays: the rays of bounce b (queue order) appended to `out` behind those of the earlier bounces of the
// batch (their counts are counts[1 .. b-1]) and of the earlier batches (`base`)
__global__ void __launch_bounds__(256) k_dump_rays(const yart_ray* __restrict__ rays, const uint32_t* __restrict__ queue,
                                                    const uint32_t* __restrict__ counts, uint32_t b, uint64_t base,
                                                    yart_ray* __restrict__ out, uint64_t cap) {
  uint64_t off = base;
  for (uint32_t j = 1; j < b; ++j) off += counts[j];
  const uint32_t n = counts[b];
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    if (off + i >= cap) break;
    D3 o, d;
    load_ray(rays + queue[i], o, d);
    store_ray(out + off + i, o, d);
  }
}

// DevMesh::leafgeo from the flattened tree: one thread per (node, child); a leaf child's triangles are copied
// vertex by vertex (9 floats each) to 64 B x (position of its first triangle)
__global__ void __launch_bounds__(256) k_pack_leaves(const FlatNode* __restrict__ nodes, uint32_t n_nodes, const FlatTri* __restrict__ tris,
                                                      float* __restrict__ leafgeo) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_nodes * 4u) return;
  const uint32_t id = nodes[w >> 2].child[w & 3u];
  if (id == 0xFFFFFFFFu || !(id >> 31)) return;
  const uint32_t count = (id >> 27) & 0xFu, first = id & 0x7FFFFFFu;
  float* out = leafgeo + (size_t)first * 16;
  for (uint32_t i = 0; i < count; ++i) {
    const FlatTri& t = tris[first + i];
    for (int j = 0; j < 3; ++j) {
      out[i * 9 + j] = t.v0[j];
      out[i * 9 + 3 + j] = t.v1[j];
      out[i * 9 + 6 + j] = t.v2[j];
    }
  }
}

// DevMesh::cnodes from the flattened tree, one thread per node.  Word layout of a 64-byte compact node (two 32-byte
// sectors; every 32-bit word holds the 16-bit values of two children, child 2j in the low half, 2j+1 in the high half):
//   sector 0: x lower planes (children 01, 23), x upper planes (01, 23), y lower (01, 23), y upper (01, 23)
//   sector 1: z lower (01, 23), z upper (01, 23), then the four child words exactly as in FlatNode::child, with the node's
//             three split axes stowed in the otherwise unused bits 29-30 of the first three words (child ids use bits
//             0-26 + the leaf flag 31 + the leaf count 27-28 as count-1).  0xFFFFFFFF = absent child, as in FlatNode.
// Quantisation, exact in f64: lower plane -> floor((b - origin) / scale), upper plane -> ceil(...): the quantised box
// contains the exact box, and shrinking it by one unit on every side gives a box contained in the exact one.
__global__ void __launch_bounds__(256) k_pack_nodes(const FlatNode* __restrict__ nodes, uint32_t n_nodes, float ox, float oy, float oz,
                                                     float scale, uint4* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_nodes) return;
  const FlatNode nd = nodes[i];
  const double o[3] = {(double)ox, (double)oy, (double)oz}, inv = 1.0 / (double)scale; // (scale is a power of two)
  const float* lo[3] = {nd.min_x, nd.min_y, nd.min_z};
  const float* hi[3] = {nd.max_x, nd.max_y, nd.max_z};
  uint32_t w[16];
  for (int a = 0; a < 3; ++a)
    for (int pair = 0; pair < 2; ++pair) {
      uint32_t ql[2], qh[2];
      for (int h = 0; h < 2; ++h) {
        const int k = pair * 2 + h;
        const bool present = nd.child[k] != 0xFFFFFFFFu;
        const double l = floor(((double)lo[a][k] - o[a]) * inv), u = ceil(((double)hi[a][k] - o[a]) * inv);
        ql[h] = present ? (uint32_t)fmin(fmax(l, 0.0), 65535.0) : 65535u; // (an absent child: an inverted box)
        qh[h] = present ? (uint32_t)fmin(fmax(u, 0.0), 65535.0) : 0u;
      }
      w[a * 4 + pair] = ql[0] | (ql[1] << 16);
      w[a * 4 + 2 + pair] = qh[0] | (qh[1] << 16);
    }
  for (int k = 0; k < 4; ++k) {
    uint32_t c = nd.child[k];
    if (c != 0xFFFFFFFFu) {
      if (c >> 31) c = 0x80000000u | ((((c >> 27) & 0xFu) - 1u) << 27) | (c & 0x7FFFFFFu); // leaf count 1..4 -> 2 bits
      if (k < 3) c |= ((nd.axes >> (2 * k)) & 3u) << 29;                                    // top, left, right axis
    }
    w[12 + k] = c;
  }
  for (int j = 0; j < 4; ++j) out[(size_t)i * 4 + j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
}

// yart_measure_fetch_peak: independent random 128-byte line fetches (one QBVH node visit = four LDG.E.256)
template <int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) k_fetch_peak(const float4* __restrict__ table, uint32_t n_lines, uint32_t iters,
                                                                     float* sink) {
  uint32_t s = (blockIdx.x * THREADS + threadIdx.x) * 2654435761u + 12345u;
  float acc = 0.f;
#pragma unroll 4
  for (uint32_t i = 0; i < iters; ++i) {
    s = s * 1664525u + 1013904223u;
    const uint32_t line = (uint32_t)(((uint64_t)s * n_lines) >> 32);
    const float4* p = table + (size_t)line * 8;
    const F8 a = ldg256(p), b = ldg256(p + 2), c = ldg256(p + 4), d = ldg256(p + 6);
    acc += a.lo.x + b.hi.y + c.lo.z + d.hi.w;
  }
  if (acc == 1234.5678f) sink[0] = acc; // keeps the loads alive
}

// The same with FOUR lanes per line: the lanes of a quad fetch the four 32-byte sectors of ONE random line with a single
// 256-bit load each (what a 4-lanes-per-ray traversal over child-major nodes would issue per visit).
template <int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) k_fetch_peak_quad(const float4* __restrict__ table, uint32_t n_lines, uint32_t iters,
                                                                          float* sink) {
  const uint32_t t = blockIdx.x * THREADS + threadIdx.x;
  uint32_t s = (t >> 2) * 2654435761u + 12345u; // (one sequence per quad)
  float acc = 0.f;
#pragma unroll 4
  for (uint32_t i = 0; i < iters; ++i) {
    s = s * 1664525u + 1013904223u;
    const uint32_t line = (uint32_t)(((uint64_t)s * n_lines) >> 32);
    const F8 a = ldg256(table + (size_t)line * 8 + 2 * (t & 3u));
    acc += a.lo.x + a.hi.w;
  }
  if (acc == 1234.5678f) sink[0] = acc;
}

namespace {

#define CUDA_TRY(ctx, expr)                                                                  \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess) {                                                                \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                      \
      if (e__ == cudaErrorMemoryAllocation) {                                                \
        cudaGetLastError(); /* not sticky: clear it so that the context stays usable */      \
        return YART_ERR_NOMEM;                                                               \
      }                                                                                      \
      return YART_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

// extern "C" bodies must not let C++ exceptions cross the ABI (std::bad_alloc from a vector, ...)
#define YART_ABI_GUARD_BEGIN try {
#define YART_ABI_GUARD_END(ctx, fn_name)                                                       \
  }                                                                                          \
  catch (const std::bad_alloc&) {                                                            \
    if (ctx) (ctx)->err = std::string(fn_name) + ": out of host memory";                        \
    return YART_ERR_NOMEM;                                                                   \
  }                                                                                          \
  catch (const std::exception& e) {                                                          \
    if (ctx) (ctx)->err = std::string(fn_name) + ": " + e.what();                               \
    return YART_ERR_INVALID;                                                                 \
  }                                                                                          \
  catch (...) {                                                                              \
    if (ctx) (ctx)->err = std::string(fn_name) + ": unknown C++ exception";                     \
    return YART_ERR_INVALID;                                                                 \
  }

int tune_env(const char* name, int dflt) { // tuning / debugging knobs from the environment
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p); // (cudaFree synchronises the device: work still using the old buffer has finished)
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

// flat 4-wide tree over the members of a BVHNode group (median split on the longest centroid
// axis; the shape is free -- closest-hit results do not depend on it)
struct GroupBuilder {
  std::vector<FlatNode> nodes;
  std::vector<uint32_t> order;
  std::vector<float> lo, hi; // [n][3], rounded outward
  std::vector<double> cen;

  struct Box {
    float mn[3], mx[3];
    bool some;
  };
  static void member_box(const yart_object& m, double mn[3], double mx[3]) {
    if (m.kind == YART_OBJ_SPHERE) {
      const double r = std::fabs(m.p[3]);
      for (int a = 0; a < 3; ++a) { mn[a] = m.p[a] - r; mx[a] = m.p[a] + r; }
    } else { // BOX
      for (int a = 0; a < 3; ++a) { mn[a] = std::fmin(m.p[a], m.p[3 + a]); mx[a] = std::fmax(m.p[a], m.p[3 + a]); }
    }
  }
  void prepare(const yart_object* mem, uint32_t n) {
    order.resize(n);
    std::iota(order.begin(), order.end(), 0u);
    lo.resize((size_t)n * 3);
    hi.resize((size_t)n * 3);
    cen.resize((size_t)n * 3);
    for (uint32_t i = 0; i < n; ++i) {
      double mn[3], mx[3];
      member_box(mem[i], mn, mx);
      for (int a = 0; a < 3; ++a) {
        float l = (float)mn[a], h = (float)mx[a];
        // pad outward: the rects of a box have zero thickness and f32 rounding may shrink
        l = nextafterf(nextafterf(l, -INFINITY), -INFINITY);
        h = nextafterf(nextafterf(h, INFINITY), INFINITY);
        lo[(size_t)i * 3 + a] = l;
        hi[(size_t)i * 3 + a] = h;
        cen[(size_t)i * 3 + a] = 0.5 * (mn[a] + mx[a]);
      }
    }
  }
  uint32_t split(size_t a, size_t b) {
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (size_t i = a; i < b; ++i)
      for (int k = 0; k < 3; ++k) {
        mn[k] = std::fmin(mn[k], cen[(size_t)order[i] * 3 + k]);
        mx[k] = std::fmax(mx[k], cen[(size_t)order[i] * 3 + k]);
      }
    uint32_t axis = 0;
    if (mx[1] - mn[1] > mx[0] - mn[0]) axis = 1;
    if (mx[2] - mn[2] > std::fmax(mx[1] - mn[1], mx[0] - mn[0])) axis = 2;
    const double* c = cen.data();
    std::sort(order.begin() + a, order.begin() + b, [c, axis](uint32_t x, uint32_t y) {
      const double cx = c[(size_t)x * 3 + axis], cy = c[(size_t)y * 3 + axis];
      return cx < cy || (cx == cy && x < y);
    });
    return axis;
  }
  static Box merge(const Box& a, const Box& b) {
    if (!a.some) return b;
    if (!b.some) return a;
    Box r;
    r.some = true;
    for (int k = 0; k < 3; ++k) { r.mn[k] = fminf(a.mn[k], b.mn[k]); r.mx[k] = fmaxf(a.mx[k], b.mx[k]); }
    return r;
  }
  Box construct(size_t a, size_t b, uint32_t& id) {
    const size_t n = b - a;
    Box none;
    none.some = false;
    if (n == 0) { id = 0xFFFFFFFFu; return none; }
    if (n <= 4) {
      Box bx;
      bx.some = true;
      for (int k = 0; k < 3; ++k) { bx.mn[k] = lo[(size_t)order[a] * 3 + k]; bx.mx[k] = hi[(size_t)order[a] * 3 + k]; }
      for (size_t i = a + 1; i < b; ++i)
        for (int k = 0; k < 3; ++k) {
          bx.mn[k] = fminf(bx.mn[k], lo[(size_t)order[i] * 3 + k]);
          bx.mx[k] = fmaxf(bx.mx[k], hi[(size_t)order[i] * 3 + k]);
        }
      id = (uint32_t)a | (1u << 31) | ((uint32_t)n << 27);
      return bx;
    }
    split(a, b);
    const size_t mid = a + n / 2;
    split(a, mid);
    const size_t lmid = a + (mid - a) / 2;
    uint32_t ids[4];
    Box bx[4];
    bx[0] = construct(a, lmid, ids[0]);
    bx[1] = construct(lmid, mid, ids[1]);
    split(mid, b);
    const size_t rmid = mid + (b - mid) / 2;
    bx[2] = construct(mid, rmid, ids[2]);
    bx[3] = construct(rmid, b, ids[3]);
    FlatNode nd;
    for (int k = 0; k < 4; ++k) {
      const bool s = bx[k].some;
      nd.min_x[k] = s ? bx[k].mn[0] : FLT_MAX; nd.min_y[k] = s ? bx[k].mn[1] : FLT_MAX; nd.min_z[k] = s ? bx[k].mn[2] : FLT_MAX;
      nd.max_x[k] = s ? bx[k].mx[0] : FLT_MAX; nd.max_y[k] = s ? bx[k].mx[1] : FLT_MAX; nd.max_z[k] = s ? bx[k].mx[2] : FLT_MAX;
      nd.child[k] = ids[k];
    }
    nd.axes = 0;
    nd.pad[0] = nd.pad[1] = nd.pad[2] = 0;
    nodes.push_back(nd);
    id = (uint32_t)nodes.size() - 1;
    return merge(merge(bx[0], bx[1]), merge(bx[2], bx[3]));
  }
};

} // namespace
} // namespace yart

using namespace yart;

struct yart_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string err;

  // scene
  bool have_scene = false;
  std::vector<void*> scene_allocs;
  DevScene scene;
  yart_object* d_solo = nullptr; // one un-wrapped MESH object per mesh, for mesh-only queries
  std::map<const void*, int> traverse_blocks; // resident CTAs per SM of each k_traverse variant
  std::vector<yart_object> h_objects; // host copy of the world list: the pass plan is made on the host
  std::vector<DevMesh> h_meshes;
  uint32_t n_meshes = 0;
  uint32_t max_stack = 0;
  bool has_media = false;
  uint32_t builder = YART_BUILDER_DEVICE;
  double* d_cie = nullptr;
  double* d_smits = nullptr;

  // work buffers
  DevBuf rays, hits_export, time, wavelength, throughput, hits, queue_a, queue_b, counts, work, counters, film, rgba;
  DevBuf nee_rays, nee_pending, nee_sum, nee_w, queue_s; // YART_FLAG_NEXT_EVENT's per-path state (NeeState)
  DevBuf occluded; // staging of yart_occluded's flags for host arrays
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> ev_pool;
  // host-buffer closest-hit queries: copy streams + events of the chunk pipeline (made on first use)
  cudaStream_t copy_in = nullptr, copy_out = nullptr;
  std::vector<cudaEvent_t> chunk_events;

  void free_scene() {
    for (void* p : scene_allocs) cudaFree(p);
    scene_allocs.clear();
    have_scene = false;
    d_solo = nullptr;
  }
};

namespace yart { // accessors for the other translation units of the library (device_comm.cu)
cudaStream_t ctx_stream(yart_ctx* ctx) { return ctx->stream; }
int ctx_device(const yart_ctx* ctx) { return ctx->device; }
void ctx_set_error(yart_ctx* ctx, const std::string& msg) { ctx->err = msg; }
} // namespace yart

namespace {

template <class T>
int upload(yart_ctx* ctx, const T* host, size_t n, T** out) {
  *out = nullptr;
  if (n == 0) return YART_OK;
  void* p = nullptr;
  CUDA_TRY(ctx, cudaMalloc(&p, n * sizeof(T)));
  ctx->scene_allocs.push_back(p);
  CUDA_TRY(ctx, cudaMemcpyAsync(p, host, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  *out = reinterpret_cast<T*>(p);
  return YART_OK;
}

DevCamera make_camera(const yart_camera& c) { // Camera::new (camera.rs:41-80), f64 on the host
  auto sub = [](const double* a, const double* b, double* o) { for (int i = 0; i < 3; ++i) o[i] = a[i] - b[i]; };
  auto unit = [](double* a) {
    double l = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    double x = a[0] / l, y = a[1] / l, z = a[2] / l;
    a[0] = x; a[1] = y; a[2] = z;
  };
  auto cross3 = [](const double* a, const double* b, double* o) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
  };
  DevCamera k;
  const double theta = c.vfov_degrees * 3.14159265358979323846264338327950288 / 180.0;
  const double h = std::tan(theta / 2.0);
  const double vh = 2.0 * h;
  const double vw = c.aspect_ratio * vh;
  double w[3], u[3], v[3];
  sub(c.lookfrom, c.lookat, w);
  unit(w);
  cross3(c.vup, w, u);
  unit(u);
  cross3(w, u, v);
  const double fh = c.focus_dist * vw, fv = c.focus_dist * vh;
  for (int i = 0; i < 3; ++i) {
    k.origin[i] = c.lookfrom[i];
    k.u[i] = u[i];
    k.v[i] = v[i];
    k.horizontal[i] = fh * u[i];
    k.vertical[i] = fv * v[i];
  }
  for (int i = 0; i < 3; ++i) // origin - horizontal/2 - vertical/2 - focus_dist*w
    k.llc[i] = k.origin[i] - k.horizontal[i] / 2.0 - k.vertical[i] / 2.0 - c.focus_dist * w[i];
  k.lens_radius = c.aperture / 2.0;
  k.time0 = c.time0;
  k.time1 = c.time1;
  return k;
}

typedef void (*TraverseKernel)(const TraverseParams);
} // namespace
namespace yart {
TraverseKernel lean_traverse_kernel(bool near, uint32_t max_stack, int ctas_per_sm, bool compact); // device_trace_lean.cu
}
namespace {
template <bool MIXED>
TraverseKernel pick_traverse_kernel_m(bool near, bool count, uint32_t max_stack) {
  if (max_stack <= 32) {
    if (near) return count ? k_traverse<true, true, 32, MIXED> : k_traverse<true, false, 32, MIXED>;
    return count ? k_traverse<false, true, 32, MIXED> : k_traverse<false, false, 32, MIXED>;
  }
  if (near) return count ? k_traverse<true, true, 64, MIXED> : k_traverse<true, false, 64, MIXED>;
  return count ? k_traverse<false, true, 64, MIXED> : k_traverse<false, false, 64, MIXED>;
}
TraverseKernel pick_traverse_kernel(bool near, bool count, uint32_t max_stack, bool mixed) {
  return mixed ? pick_traverse_kernel_m<true>(near, count, max_stack) : pick_traverse_kernel_m<false>(near, count, max_stack);
}

// What is the same for every pass of one closest-hit query.
struct QueryArgs {
  PassCommon c;
  const yart_object* d_objects; // device copy of the list the host plan walks
  const yart_object* h_objects;
  uint32_t n_objects;
  const double* ray_time;
  uint64_t seed;
  uint32_t bounce, spp_batch, sample_base, pixel_base;
  uint32_t* work_counters;      // one zeroed u32 per traverse pass (at least n_objects)
  unsigned long long* counters;
  bool near, count;
};

// HittableList::hit (hittable.rs:66-79) as passes over the ray queue, in list order: one k_traverse per
// mesh instance, one k_analytic per run of consecutive analytic objects.
int run_passes(yart_ctx* ctx, const QueryArgs& q, uint64_t* launches) {
  static const int rt = tune_env("YART_TUNE_RT", 8), nt = tune_env("YART_TUNE_NT", 12);
  static const int carve = tune_env("YART_TUNE_CARVEOUT", 35);
  static const int carve_lean = tune_env("YART_TUNE_CARVEOUT_LEAN", 50);
  static const int mixed = tune_env("YART_TUNE_MIXED", 1); // 0: all-f64 slab tests (same results, slower)
  bool first = true;
  uint32_t i = 0, n_trav = 0;
  auto is_mesh = [&](uint32_t k) {
    return q.h_objects[k].kind == YART_OBJ_MESH && !(q.h_objects[k].wrap & YART_WRAP_MEDIUM);
  };
  if (q.n_objects == 0) { // an empty world: every ray misses
    AnalyticParams A;
    memset(&A, 0, sizeof(A));
    A.c = q.c;
    A.c.first_pass = 1;
    A.scene = ctx->scene;
    A.objects = q.d_objects;
    A.spp_batch = 1;
    k_analytic<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(A);
    if (launches) (*launches)++;
  }
  while (i < q.n_objects) {
    if (is_mesh(i)) {
      const yart_object& o = q.h_objects[i];
      const DevMesh& m = ctx->h_meshes[o.index];
      TraverseParams T;
      memset(&T, 0, sizeof(T));
      T.c = q.c;
      T.c.first_pass = first ? 1u : 0u;
      T.nodes = m.nodes;
      T.tris = m.tris;
      T.leafgeo = m.leafgeo;
      T.cnodes = m.cnodes;
      T.cscale = m.cscale;
      for (int k = 0; k < 3; ++k) T.corigin[k] = m.corigin[k];
      T.root = m.root;
      T.n_nodes = m.n_nodes;
      T.n_tris = m.n_tris;
      T.obj_index = i;
      T.wrap = o.wrap & (YART_WRAP_ROTATE_Y | YART_WRAP_TRANSLATE);
      T.refill_threshold = (uint32_t)std::max(1, std::min(32, rt));
      T.node_threshold = (uint32_t)std::max(1, std::min(32, nt));
      T.sin_theta = o.sin_theta;
      T.cos_theta = o.cos_theta;
      for (int k = 0; k < 3; ++k) T.offset[k] = o.offset[k];
      T.work_counter = q.work_counters + n_trav++;
      T.counters = q.counters;
      for (int k = 0; k < 3; ++k) T.bound[k] = m.bound[k];
      // k_traverse_lean (device_trace_lean.cu): the same traversal with the f64-only state in shared memory -- 96
      // registers, FIVE 128-thread CTAs per SM (20 warps) instead of four: +7 % on the david render, +6 % on the sweep.
      // YART_TUNE_LEAN=0 selects k_traverse (which also serves visit counting and the all-f64 slab variant).
      static const int lean = tune_env("YART_TUNE_LEAN", 5);
      static const int lean_stack24 = tune_env("YART_TUNE_LEAN_STACK24", 1);
      // (the reference-order instantiation of the lean kernel spills 150 B at 96 registers and is 5 % SLOWER than
      // k_traverse on the sweep -- 2,074 vs 2,188 Mrays/s -- so only the near-first order, the default everywhere, uses it;
      // YART_TUNE_LEAN_REF=1 forces it for both)
      static const int lean_ref = tune_env("YART_TUNE_LEAN_REF", 0);
      const bool use_lean = lean && mixed && !q.count && (q.near || lean_ref);
      TraverseKernel k = use_lean ? yart::lean_traverse_kernel(q.near, (lean_stack24 || ctx->max_stack > 24) ? ctx->max_stack : 25u, lean,
                                                                 m.cnodes != nullptr && q.near)
                                  : pick_traverse_kernel(q.near, q.count, ctx->max_stack, mixed != 0);
      // occupancy query + carveout once per kernel variant (they cost tens of microseconds of host time,
      // which is the whole budget of a deep bounce)
      int& per_sm = ctx->traverse_blocks[(const void*)k];
      if (per_sm == 0) {
        // leave everything the stacks do not need to L1: the tree's upper levels live there
        // (the lean kernel keeps 22-42 KB of shared memory per CTA: five CTAs need the 132 KB configuration)
        cudaFuncSetAttribute(reinterpret_cast<const void*>(k), cudaFuncAttributePreferredSharedMemoryCarveout, use_lean ? carve_lean : carve);
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(k), kTraceThreads, 0));
        per_sm = std::max(per_sm, 1);
      }
      k<<<per_sm * ctx->sm_count, kTraceThreads, 0, ctx->stream>>>(T); // persistent: one resident wave
      i++;
    } else {
      uint32_t j = i;
      while (j < q.n_objects && !is_mesh(j)) ++j;
      AnalyticParams A;
      memset(&A, 0, sizeof(A));
      A.c = q.c;
      A.c.first_pass = first ? 1u : 0u;
      A.scene = ctx->scene;
      A.objects = q.d_objects;
      A.obj_begin = i;
      A.obj_end = j;
      A.ray_time = q.ray_time;
      A.seed = q.seed;
      A.bounce = q.bounce;
      A.spp_batch = q.spp_batch ? q.spp_batch : 1;
      A.sample_base = q.sample_base;
      A.pixel_base = q.pixel_base;
      A.media_mask = ctx->has_media ? 1u : 0u;
      k_analytic<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(A);
      i = j;
    }
    first = false;
    if (launches) (*launches)++;
  }
  CUDA_TRY(ctx, cudaGetLastError());
  return YART_OK;
}

// What is the same for every pass of one occlusion query.
struct OcclusionArgs {
  OccludeCommon c;
  const yart_object* d_objects;
  const yart_object* h_objects;
  uint32_t n_objects;
  uint32_t pixel_base;
  uint32_t* work_counters; // one zeroed u32 per mesh pass (at least n_objects)
};

// yart_occluded as passes over the rays in list order, like run_passes: one k_occlude per mesh instance, one
// k_analytic_occluded per run of consecutive analytic objects.  c.occluded must be zeroed: a pass only ever writes 1,
// and the passes after the first skip the rays already marked.  An empty world launches nothing.
int run_occlusion_passes(yart_ctx* ctx, const OcclusionArgs& q, uint64_t* launches) {
  static const int rt = tune_env("YART_TUNE_RT", 8), nt = tune_env("YART_TUNE_NT", 12);
  static const int carve = tune_env("YART_TUNE_CARVEOUT_LEAN", 50);
  // A closest-hit pass starts a ray that nothing has hit yet from t_max if it is the first mesh pass, and from
  // fmin(+inf, t_max) otherwise (the recorded miss is +inf).  The two differ only for a NaN t_max.
  const double t_max_later = std::fmin(INFINITY, q.c.t_max);
  bool first = true;
  uint32_t i = 0, n_trav = 0;
  auto is_mesh = [&](uint32_t k) {
    return q.h_objects[k].kind == YART_OBJ_MESH && !(q.h_objects[k].wrap & YART_WRAP_MEDIUM);
  };
  while (i < q.n_objects) {
    if (is_mesh(i)) {
      const yart_object& o = q.h_objects[i];
      const DevMesh& m = ctx->h_meshes[o.index];
      OccludeParams T;
      memset(&T, 0, sizeof(T));
      T.c = q.c;
      T.c.first_pass = first ? 1u : 0u;
      T.c.t_max = first ? q.c.t_max : t_max_later;
      T.nodes = m.nodes;
      T.tris = m.tris;
      T.leafgeo = m.leafgeo;
      T.root = m.root;
      T.n_nodes = m.n_nodes;
      T.n_tris = m.n_tris;
      T.wrap = o.wrap & (YART_WRAP_ROTATE_Y | YART_WRAP_TRANSLATE);
      T.refill_threshold = (uint32_t)std::max(1, std::min(32, rt));
      T.node_threshold = (uint32_t)std::max(1, std::min(32, nt));
      T.sin_theta = o.sin_theta;
      T.cos_theta = o.cos_theta;
      for (int k = 0; k < 3; ++k) T.offset[k] = o.offset[k];
      for (int k = 0; k < 3; ++k) T.bound[k] = m.bound[k];
      T.work_counter = q.work_counters + n_trav++;
      const OccludeKernel k = yart::occlude_kernel(ctx->max_stack);
      int& per_sm = ctx->traverse_blocks[(const void*)k]; // (occupancy query + carveout once per variant, as above)
      if (per_sm == 0) {
        cudaFuncSetAttribute(reinterpret_cast<const void*>(k), cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(k), kTraceThreads, 0));
        per_sm = std::max(per_sm, 1);
      }
      k<<<per_sm * ctx->sm_count, kTraceThreads, 0, ctx->stream>>>(T); // persistent: one resident wave
      i++;
    } else {
      uint32_t j = i;
      while (j < q.n_objects && !is_mesh(j)) ++j;
      AnalyticOccludedParams A;
      memset(&A, 0, sizeof(A));
      A.c = q.c;
      A.c.first_pass = first ? 1u : 0u;
      A.c.t_max = t_max_later;
      A.scene = ctx->scene;
      A.objects = q.d_objects;
      A.obj_begin = i;
      A.obj_end = j;
      A.pixel_base = q.pixel_base;
      A.media = ctx->has_media ? 1u : 0u;
      yart::analytic_occluded_kernel()<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(A);
      i = j;
    }
    first = false;
    if (launches) (*launches)++;
  }
  CUDA_TRY(ctx, cudaGetLastError());
  return YART_OK;
}

// One batched query over n rays.  Device arrays: run(0, n) once, between ctx->ev0 and ctx->ev1.  Host arrays: the
// rays are uploaded into d_in and the results downloaded from d_out (staging buffers of at least n records) in chunks,
// the upload of chunk i+1 and the download of chunk i-1 overlapping the kernels of chunk i on two copy streams (PCIe is
// full duplex; the transfers, not the traversal, bound such a call: 88 B per closest hit against ~1.5 ns of kernel
// time).  With pageable host memory the copies block the calling thread, so the kernels of a chunk are queued BEFORE
// the next upload is issued; with pinned memory everything is asynchronous.
// run(off, len) enqueues on ctx->stream the kernels that read the ray records at d_in + off * in_bytes and leave
// out_bytes per ray at d_out + off * out_bytes.  Everything is enqueued on return; after a synchronisation of
// ctx->stream, chunked_kernel_ms gives the kernels' time.
template <class Run>
int run_chunked(yart_ctx* ctx, bool dev, const void* in, size_t in_bytes, void* out, size_t out_bytes, uint64_t n,
                const char* d_in, char* d_out, Run&& run, uint64_t* n_chunks_out) {
  const int chunk_env = tune_env("YART_TUNE_HOST_CHUNK", 1 << 19); // (rays per chunk, read per call; 2^19 measured best: tools/host_chunk_probe.py)
  const uint64_t chunk = dev ? n : (uint64_t)std::max(chunk_env, 1024);
  const uint64_t n_chunks = (n + chunk - 1) / chunk;
  *n_chunks_out = n_chunks;
  char* stage_in = const_cast<char*>(d_in); // (host arrays: d_in is the context's staging buffer)
  if (dev || n_chunks == 1) {
    if (!dev) CUDA_TRY(ctx, cudaMemcpyAsync(stage_in, in, n * in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream)); // (stats->gpu_ms: the kernels, not the copies)
    const int rc = run(0, n);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (!dev) CUDA_TRY(ctx, cudaMemcpyAsync(out, d_out, n * out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  } else {
    if (!ctx->copy_in) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
    if (!ctx->copy_out) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
    while (ctx->chunk_events.size() < 3 * n_chunks + 1) {
      cudaEvent_t e;
      CUDA_TRY(ctx, cudaEventCreate(&e));
      ctx->chunk_events.push_back(e);
    }
    cudaEvent_t* up = ctx->chunk_events.data();                   // up[i]: chunk i is on the device
    cudaEvent_t* done = ctx->chunk_events.data() + n_chunks;      // done[i]: chunk i's results are in d_out
    cudaEvent_t* begun = ctx->chunk_events.data() + 2 * n_chunks; // begun[i]: chunk i's kernels start (its upload is in)
    cudaEvent_t start = ctx->chunk_events[3 * n_chunks];
    // (the device buffers may still be read by earlier work on the context's stream)
    CUDA_TRY(ctx, cudaEventRecord(start, ctx->stream));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_in, start, 0));
    auto upload_chunk = [&](uint64_t i) -> int {
      const uint64_t off = i * chunk, len = std::min(chunk, n - off);
      CUDA_TRY(ctx, cudaMemcpyAsync(stage_in + off * in_bytes, static_cast<const char*>(in) + off * in_bytes,
                                    len * in_bytes, cudaMemcpyHostToDevice, ctx->copy_in));
      CUDA_TRY(ctx, cudaEventRecord(up[i], ctx->copy_in));
      return YART_OK;
    };
    int rc = upload_chunk(0);
    if (rc) return rc;
    for (uint64_t i = 0; i < n_chunks; ++i) {
      const uint64_t off = i * chunk, len = std::min(chunk, n - off);
      CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, up[i], 0));
      CUDA_TRY(ctx, cudaEventRecord(begun[i], ctx->stream));
      if ((rc = run(off, len)) != YART_OK) break;
      CUDA_TRY(ctx, cudaEventRecord(done[i], ctx->stream));
      if (i + 1 < n_chunks && (rc = upload_chunk(i + 1)) != YART_OK) break;
      CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_out, done[i], 0));
      CUDA_TRY(ctx, cudaMemcpyAsync(static_cast<char*>(out) + off * out_bytes, d_out + off * out_bytes, len * out_bytes,
                                    cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    // nothing of this call may outlive it, error or not
    cudaStreamSynchronize(ctx->copy_in);
    cudaError_t ce = cudaStreamSynchronize(ctx->copy_out);
    if (rc) {
      cudaStreamSynchronize(ctx->stream);
      return rc;
    }
    CUDA_TRY(ctx, ce);
  }
  return YART_OK;
}

// the kernels of a finished run_chunked call: ev0 -> ev1, or the chunks without the waits for their uploads in between
int chunked_kernel_ms(yart_ctx* ctx, uint64_t n_chunks, bool dev, float* ms) {
  *ms = 0.f;
  if (dev || n_chunks == 1) {
    CUDA_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  } else {
    for (uint64_t i = 0; i < n_chunks; ++i) {
      float part = 0.f;
      CUDA_TRY(ctx, cudaEventElapsedTime(&part, ctx->chunk_events[2 * n_chunks + i], ctx->chunk_events[n_chunks + i]));
      *ms += part;
    }
  }
  return YART_OK;
}

} // namespace

extern "C" {

int yart_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int yart_ctx_create(int device, yart_ctx** out) {
  if (!out) {
    set_global_error("yart_ctx_create: null argument");
    return YART_ERR_INVALID;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    set_global_error(std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                     " (this library has no CPU fallback)");
    return YART_ERR_CUDA;
  }
  if (device < 0 || device >= n) {
    set_global_error("yart_ctx_create: device index out of range");
    return YART_ERR_INVALID;
  }
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    set_global_error(std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return YART_ERR_CUDA;
  }
  if (prop.major != 10) {
    set_global_error("this library is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor));
    return YART_ERR_CUDA;
  }
  yart_ctx* ctx = new yart_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
      (e = cudaMalloc((void**)&ctx->d_cie, sizeof(double) * 3 * YART_N_CIE)) != cudaSuccess ||
      (e = cudaMalloc((void**)&ctx->d_smits, sizeof(double) * 7 * YART_N_BINS)) != cudaSuccess) {
    set_global_error(std::string("context setup: ") + cudaGetErrorString(e));
    delete ctx;
    return YART_ERR_CUDA;
  }
  if ((e = cudaMemcpy(ctx->d_cie, YART_CIE_X, sizeof(double) * YART_N_CIE, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(ctx->d_cie + YART_N_CIE, YART_CIE_Y, sizeof(double) * YART_N_CIE, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(ctx->d_cie + 2 * YART_N_CIE, YART_CIE_Z, sizeof(double) * YART_N_CIE, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(ctx->d_smits, YART_SMITS_BASIS, sizeof(double) * 7 * YART_N_BINS, cudaMemcpyHostToDevice)) != cudaSuccess) {
    set_global_error(std::string("context setup (spectral tables): ") + cudaGetErrorString(e));
    yart_ctx_destroy(ctx);
    return YART_ERR_CUDA;
  }
  *out = ctx;
  return YART_OK;
}

void yart_ctx_destroy(yart_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  ctx->free_scene();
  DevBuf* bufs[] = {&ctx->rays, &ctx->hits_export, &ctx->time, &ctx->wavelength, &ctx->throughput, &ctx->hits,
                    &ctx->queue_a, &ctx->queue_b, &ctx->counts, &ctx->work, &ctx->counters, &ctx->film, &ctx->rgba,
                    &ctx->occluded};
  for (DevBuf* b : bufs) b->release();
  for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->chunk_events) cudaEventDestroy(e);
  if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
  if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->d_cie) cudaFree(ctx->d_cie);
  if (ctx->d_smits) cudaFree(ctx->d_smits);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* yart_last_error(const yart_ctx* ctx) { return ctx ? ctx->err.c_str() : yart_last_error_global(); }

int yart_ctx_set_stream(yart_ctx* ctx, void* cuda_stream) {
  if (!ctx) return YART_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (ctx->stream || !ctx->own_stream) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); // work queued on the old stream
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  ctx->own_stream = false;
  return YART_OK;
}

int yart_host_register(yart_ctx* ctx, void* ptr, uint64_t bytes) {
  if (!ctx) return YART_ERR_INVALID;
  if (!ptr || !bytes) {
    ctx->err = "yart_host_register: null pointer or zero size";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);
  if (e != cudaSuccess) {
    cudaGetLastError(); // not sticky
    ctx->err = std::string("yart_host_register: ") + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? YART_ERR_NOMEM : YART_ERR_INVALID; // (already registered, not host memory, ...)
  }
  return YART_OK;
}

int yart_host_unregister(yart_ctx* ctx, void* ptr) {
  if (!ctx) return YART_ERR_INVALID;
  if (!ptr) {
    ctx->err = "yart_host_unregister: null pointer";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); // copies from / to the array may still be queued
  const cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) {
    cudaGetLastError();
    ctx->err = std::string("yart_host_unregister: ") + cudaGetErrorString(e);
    return YART_ERR_INVALID;
  }
  return YART_OK;
}

int yart_ctx_set_builder(yart_ctx* ctx, uint32_t builder) {
  if (!ctx) return YART_ERR_INVALID;
  if (builder > YART_BUILDER_DEVICE) {
    ctx->err = "yart_ctx_set_builder: unknown builder";
    return YART_ERR_INVALID;
  }
  ctx->builder = builder;
  return YART_OK;
}

static int qbvh_build_device_impl(yart_ctx* ctx, const yart_trimesh* mesh, yart_qbvh** out);

int yart_qbvh_build_device(yart_ctx* ctx, const yart_trimesh* mesh, yart_qbvh** out) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  return qbvh_build_device_impl(ctx, mesh, out);
  YART_ABI_GUARD_END(ctx, "yart_qbvh_build_device")
}

static int qbvh_build_device_impl(yart_ctx* ctx, const yart_trimesh* mesh, yart_qbvh** out) {
  if (!mesh || !out) {
    ctx->err = "yart_qbvh_build_device: null argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  DeviceQbvh dq;
  std::string err;
  if (!build_qbvh_device(ctx->stream, *mesh, dq, err)) {
    ctx->err = "yart_qbvh_build_device: " + err;
    return err.find("cuda") != std::string::npos ? YART_ERR_CUDA : YART_ERR_INVALID;
  }
  yart_qbvh* q = new (std::nothrow) yart_qbvh();
  if (!q) {
    free_qbvh_device(dq);
    return YART_ERR_NOMEM;
  }
  q->q.nodes.resize(dq.n_nodes);
  q->q.tris.resize(dq.n_tris);
  q->q.shade.resize(dq.n_tris);
  cudaError_t e = cudaMemcpyAsync(q->q.nodes.data(), dq.nodes, (size_t)dq.n_nodes * sizeof(FlatNode), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(q->q.tris.data(), dq.tris, (size_t)dq.n_tris * sizeof(FlatTri), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(q->q.shade.data(), dq.shade, (size_t)dq.n_tris * sizeof(FlatTriShade), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  q->q.root = dq.root; q->q.n_leaves = dq.n_leaves; q->q.height = dq.height; q->q.max_stack = dq.max_stack;
  for (int a = 0; a < 3; ++a) { q->q.bbox_min[a] = dq.bbox_min[a]; q->q.bbox_max[a] = dq.bbox_max[a]; }
  q->n_tris = dq.n_tris;
  free_qbvh_device(dq);
  if (e != cudaSuccess) {
    delete q;
    ctx->err = std::string("yart_qbvh_build_device: copy back: ") + cudaGetErrorString(e);
    return YART_ERR_CUDA;
  }
  *out = q;
  return YART_OK;
}

int yart_ctx_synchronize(yart_ctx* ctx) {
  if (!ctx) return YART_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return YART_OK;
}

static int set_scene_impl(yart_ctx* ctx, const yart_scene_desc* d) {
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->free_scene();
  // ---- validation (the reference would panic on these; here a bad descriptor must never become a wild load) ----
  ctx->has_media = false;
  if ((d->n_objects && !d->objects) || (d->n_lights && !d->lights) || (d->n_meshes && !d->meshes) ||
      (d->n_groups && !d->groups) || (d->n_materials && !d->materials) || (d->n_textures && !d->textures) ||
      (d->n_perlins && !d->perlins) || (d->n_images && !d->images)) {
    ctx->err = "yart_ctx_set_scene: a table pointer is null although its count is not 0";
    return YART_ERR_INVALID;
  }
  auto check_obj = [&](const yart_object& o, bool member) -> const char* {
    if (o.kind > YART_OBJ_GROUP) return "unknown object kind";
    if (member && (o.wrap != 0 || (o.kind != YART_OBJ_SPHERE && o.kind != YART_OBJ_BOX)))
      return "group members must be plain spheres or boxes";
    // (a GROUP object carries no material of its own: every hit is shaded with its member's)
    if (o.kind != YART_OBJ_GROUP && o.material >= d->n_materials) return "object refers to a missing material";
    if (o.kind == YART_OBJ_MESH && o.index >= d->n_meshes) return "object refers to a missing mesh";
    if (o.kind == YART_OBJ_GROUP && o.index >= d->n_groups) return "object refers to a missing group";
    if ((o.wrap & YART_WRAP_MEDIUM) && (o.kind == YART_OBJ_MESH || o.kind == YART_OBJ_GROUP))
      return "ConstantMedium around a mesh or group is not supported";
    return nullptr;
  };
  for (uint32_t i = 0; i < d->n_objects; ++i) {
    if (const char* m = check_obj(d->objects[i], false)) {
      ctx->err = std::string("yart_ctx_set_scene: object ") + std::to_string(i) + ": " + m;
      return YART_ERR_INVALID;
    }
    if (d->objects[i].wrap & YART_WRAP_MEDIUM) ctx->has_media = true;
  }
  for (uint32_t i = 0; i < d->n_materials; ++i) {
    const yart_material& m = d->materials[i];
    const bool textured = m.kind == YART_MAT_LAMBERTIAN || m.kind == YART_MAT_METAL || m.kind == YART_MAT_DIFFUSE_LIGHT ||
                          m.kind == YART_MAT_ISOTROPIC;
    if (m.kind > YART_MAT_ISOTROPIC || (textured && m.texture >= d->n_textures)) {
      ctx->err = "yart_ctx_set_scene: bad material " + std::to_string(i);
      return YART_ERR_INVALID;
    }
  }
  for (uint32_t i = 0; i < d->n_textures; ++i) {
    const yart_texture& t = d->textures[i];
    if (t.kind > YART_TEX_IMAGE || (t.kind == YART_TEX_NOISE && (t.perlin >= d->n_perlins || t.noise_type > YART_NOISE_NET)) ||
        (t.kind == YART_TEX_IMAGE && t.image >= d->n_images)) {
      ctx->err = "yart_ctx_set_scene: bad texture " + std::to_string(i);
      return YART_ERR_INVALID;
    }
    if (t.kind == YART_TEX_IMAGE) { // ImageTexture::value indexes width-1 / height-1 (texture.rs:313-345)
      const yart_image& im = d->images[t.image];
      if (!im.rgb8 || im.width == 0 || im.height == 0) {
        ctx->err = "yart_ctx_set_scene: texture " + std::to_string(i) + " refers to an empty image";
        return YART_ERR_INVALID;
      }
    }
  }
  for (uint32_t i = 0; i < d->n_lights; ++i)
    if (d->lights[i].kind > YART_OBJ_GROUP) {
      ctx->err = "yart_ctx_set_scene: light " + std::to_string(i) + ": unknown object kind";
      return YART_ERR_INVALID;
    }
  for (uint32_t i = 0; i < d->n_meshes; ++i)
    if (d->meshes[i].n_tris && (!d->meshes[i].positions || !d->meshes[i].normals || !d->meshes[i].uvs)) {
      ctx->err = "yart_ctx_set_scene: mesh " + std::to_string(i) + " has null attribute arrays";
      return YART_ERR_INVALID;
    }
  // ---- meshes: QBVH build on the host, flat upload ----
  std::vector<DevMesh> meshes(d->n_meshes);
  std::vector<yart_object> solo(d->n_meshes);
  ctx->max_stack = 0;
  for (uint32_t i = 0; i < d->n_meshes; ++i) {
    struct { uint32_t root, max_stack, n_nodes, n_tris; double bbox_min[3], bbox_max[3]; } q;
    FlatNode* dn;
    FlatTri* dt;
    FlatTriShade* ds;
    std::string err;
    if (ctx->builder == YART_BUILDER_DEVICE) {
      DeviceQbvh dq;
      if (!build_qbvh_device(ctx->stream, d->meshes[i], dq, err)) {
        ctx->err = "yart_ctx_set_scene: mesh " + std::to_string(i) + " (device build): " + err;
        ctx->free_scene();
        return err.find("cuda") != std::string::npos ? YART_ERR_CUDA : YART_ERR_INVALID;
      }
      dn = dq.nodes; dt = dq.tris; ds = dq.shade;
      ctx->scene_allocs.push_back(dn);
      ctx->scene_allocs.push_back(dt);
      ctx->scene_allocs.push_back(ds);
      q.root = dq.root; q.max_stack = dq.max_stack; q.n_nodes = dq.n_nodes; q.n_tris = dq.n_tris;
      for (int a = 0; a < 3; ++a) { q.bbox_min[a] = dq.bbox_min[a]; q.bbox_max[a] = dq.bbox_max[a]; }
    } else {
      FlatQbvh hq;
      if (!build_qbvh(d->meshes[i], hq, err)) {
        ctx->err = "yart_ctx_set_scene: mesh " + std::to_string(i) + ": " + err;
        ctx->free_scene();
        return YART_ERR_INVALID;
      }
      int rc;
      if ((rc = upload(ctx, hq.nodes.data(), hq.nodes.size(), &dn)) || (rc = upload(ctx, hq.tris.data(), hq.tris.size(), &dt)) ||
          (rc = upload(ctx, hq.shade.data(), hq.shade.size(), &ds))) {
        ctx->free_scene();
        return rc;
      }
      CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); // hq goes out of scope
      q.root = hq.root; q.max_stack = hq.max_stack; q.n_nodes = (uint32_t)hq.nodes.size(); q.n_tris = (uint32_t)hq.tris.size();
      for (int a = 0; a < 3; ++a) { q.bbox_min[a] = hq.bbox_min[a]; q.bbox_max[a] = hq.bbox_max[a]; }
    }
    meshes[i].nodes = reinterpret_cast<const float4*>(dn);
    meshes[i].tris = reinterpret_cast<const float4*>(dt);
    meshes[i].shade = reinterpret_cast<const double*>(ds);
    {
      float* dl = nullptr; // 64 B per triangle position; only the first 36 B x count of a leaf's block are used
      CUDA_TRY(ctx, cudaMalloc((void**)&dl, (size_t)q.n_tris * 64));
      ctx->scene_allocs.push_back(dl);
      CUDA_TRY(ctx, cudaMemsetAsync(dl, 0, (size_t)q.n_tris * 64, ctx->stream));
      k_pack_leaves<<<(q.n_nodes * 4u + 255u) / 256u, 256, 0, ctx->stream>>>(dn, q.n_nodes, dt, dl);
      CUDA_TRY(ctx, cudaGetLastError());
      meshes[i].leafgeo = reinterpret_cast<const float4*>(dl);
    }
    {
      // Compact 64-byte nodes: an EXPERIMENT, off unless YART_TUNE_COMPACT=1 (2 = also for fine meshes).  It is
      // bit-identical (tests/test_gpu_flags_and_abi.py runs the parity cases with it on) and cuts L1 wavefronts by 40 %,
      // but costs ~55 % more instructions and loses ~20 % on the B200 (DESIGN.md section 7).  Eligible when inner node
      // ids fit 27 bits, the bounding box is finite, and the 16-bit grid is fine against the mesh: the grid step is
      // (largest extent) / 65534, and a mesh whose AVERAGE triangle is smaller than ~32 steps would send too many box
      // tests to the exact fallback.  (Read per scene, not cached, so that one process can compare both.)
      meshes[i].cnodes = nullptr;
      meshes[i].cscale = 0.f;
      for (int a = 0; a < 3; ++a) meshes[i].corigin[a] = 0.f;
      const int compact = tune_env("YART_TUNE_COMPACT", 0);
      double ext = 0.0;
      bool finite = true;
      for (int a = 0; a < 3; ++a) {
        ext = std::fmax(ext, q.bbox_max[a] - q.bbox_min[a]);
        finite = finite && std::isfinite(q.bbox_min[a]) && std::isfinite(q.bbox_max[a]) && std::fabs(q.bbox_min[a]) < 1e30 && std::fabs(q.bbox_max[a]) < 1e30;
      }
      if (compact && finite && ext > 0.0 && q.n_nodes < (1u << 27) && q.n_nodes > 0) {
        int e = 0;
        std::frexp(ext / 65534.0, &e); // ext / 65534 = m * 2^e with m in [0.5, 1): 2^e >= ext / 65534
        const double step = std::ldexp(1.0, e);
        const double avg_tri = ext / std::cbrt((double)std::max<uint32_t>(q.n_tris, 1u)); // a crude length scale of one triangle
        if (e > -100 && e < 100 && (avg_tri / step >= 32.0 || compact > 1)) {
          uint4* dc = nullptr;
          CUDA_TRY(ctx, cudaMalloc((void**)&dc, (size_t)q.n_nodes * 64));
          ctx->scene_allocs.push_back(dc);
          // (the corner is the f32 image of the f64 bounding box's minimum, rounded DOWN so that every plane lies above it)
          float org[3];
          for (int a = 0; a < 3; ++a) {
            float f = (float)q.bbox_min[a];
            if ((double)f > q.bbox_min[a]) f = nextafterf(f, -INFINITY);
            org[a] = f;
          }
          k_pack_nodes<<<(q.n_nodes + 255u) / 256u, 256, 0, ctx->stream>>>(dn, q.n_nodes, org[0], org[1], org[2], (float)step, dc);
          CUDA_TRY(ctx, cudaGetLastError());
          meshes[i].cnodes = dc;
          meshes[i].cscale = (float)step;
          for (int a = 0; a < 3; ++a) meshes[i].corigin[a] = org[a];
        }
      }
    }
    meshes[i].root = q.root;
    meshes[i].max_stack = q.max_stack;
    meshes[i].n_nodes = q.n_nodes;
    meshes[i].n_tris = q.n_tris;
    for (int a = 0; a < 3; ++a) meshes[i].bound[a] = std::fmax(std::fabs(q.bbox_min[a]), std::fabs(q.bbox_max[a]));
    ctx->max_stack = std::max(ctx->max_stack, q.max_stack);
    memset(&solo[i], 0, sizeof(yart_object));
    solo[i].kind = YART_OBJ_MESH;
    solo[i].index = i;
    solo[i].cos_theta = 1.0;
  }
  if (ctx->max_stack > 64) {
    ctx->err = "yart_ctx_set_scene: QBVH deeper than the 64-entry traversal stack (qbvh.rs:382)";
    ctx->free_scene();
    return YART_ERR_UNSUPPORTED;
  }
  // ---- groups ----
  std::vector<DevGroup> groups(d->n_groups);
  for (uint32_t i = 0; i < d->n_groups; ++i) {
    const yart_group& g = d->groups[i];
    if (g.n_members && !g.members) {
      ctx->err = "yart_ctx_set_scene: group " + std::to_string(i) + " has a null member array";
      return YART_ERR_INVALID;
    }
    for (uint32_t k = 0; k < g.n_members; ++k)
      if (const char* m = check_obj(g.members[k], true)) {
        ctx->err = std::string("yart_ctx_set_scene: group member: ") + m;
        ctx->free_scene();
        return YART_ERR_INVALID;
      }
    if (g.n_members > 65536u) { // tree height <= 7 keeps the traversal within its 24-entry stack (3 * height + 1)
      ctx->err = "yart_ctx_set_scene: a group holds more than 65536 members";
      ctx->free_scene();
      return YART_ERR_UNSUPPORTED;
    }
    std::vector<yart_object> members(g.members, g.members + g.n_members);
    std::vector<uint32_t> orig(g.n_members);
    std::iota(orig.begin(), orig.end(), 0u);
    GroupBuilder gb;
    uint32_t root = 0xFFFFFFFFu;
    if (g.n_members > 8) {
      gb.prepare(g.members, g.n_members);
      gb.construct(0, g.n_members, root);
      for (uint32_t k = 0; k < g.n_members; ++k) {
        members[k] = g.members[gb.order[k]];
        orig[k] = gb.order[k];
      }
    }
    FlatNode* dn;
    yart_object* dm;
    uint32_t* dorig;
    int rc;
    if ((rc = upload(ctx, gb.nodes.data(), gb.nodes.size(), &dn)) || (rc = upload(ctx, members.data(), members.size(), &dm)) ||
        (rc = upload(ctx, orig.data(), orig.size(), &dorig))) {
      ctx->free_scene();
      return rc;
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    groups[i].nodes = reinterpret_cast<const float4*>(dn);
    groups[i].members = dm;
    groups[i].member_orig = dorig;
    groups[i].root = root;
    groups[i].n_members = g.n_members;
    for (int a = 0; a < 3; ++a) groups[i].bound[a] = 0.0;
    for (const FlatNode& nd : gb.nodes)
      for (int k = 0; k < 4; ++k) {
        if (nd.child[k] == 0xFFFFFFFFu) continue;
        groups[i].bound[0] = std::fmax(groups[i].bound[0], std::fmax(std::fabs((double)nd.min_x[k]), std::fabs((double)nd.max_x[k])));
        groups[i].bound[1] = std::fmax(groups[i].bound[1], std::fmax(std::fabs((double)nd.min_y[k]), std::fabs((double)nd.max_y[k])));
        groups[i].bound[2] = std::fmax(groups[i].bound[2], std::fmax(std::fabs((double)nd.min_z[k]), std::fabs((double)nd.max_z[k])));
      }
  }
  // ---- images ----
  std::vector<DevImage> images(d->n_images);
  for (uint32_t i = 0; i < d->n_images; ++i) {
    uint8_t* dp;
    const size_t img_bytes = d->images[i].rgb8 ? (size_t)d->images[i].width * d->images[i].height * 3 : 0;
    int rc = upload(ctx, d->images[i].rgb8, img_bytes, &dp);
    if (rc) {
      ctx->free_scene();
      return rc;
    }
    images[i].rgb8 = dp;
    images[i].width = d->images[i].width;
    images[i].height = d->images[i].height;
  }
  // ---- tables ----
  DevScene& S = ctx->scene;
  memset(&S, 0, sizeof(S));
  yart_object *dobj, *dlights;
  DevMesh* dmeshes;
  DevGroup* dgroups;
  yart_material* dmat;
  yart_texture* dtex;
  yart_perlin* dper;
  DevImage* dimg;
  int rc;
  if ((rc = upload(ctx, d->objects, d->n_objects, &dobj)) || (rc = upload(ctx, d->lights, d->n_lights, &dlights)) ||
      (rc = upload(ctx, meshes.data(), meshes.size(), &dmeshes)) || (rc = upload(ctx, groups.data(), groups.size(), &dgroups)) ||
      (rc = upload(ctx, d->materials, d->n_materials, &dmat)) || (rc = upload(ctx, d->textures, d->n_textures, &dtex)) ||
      (rc = upload(ctx, d->perlins, d->n_perlins, &dper)) || (rc = upload(ctx, images.data(), images.size(), &dimg)) ||
      (rc = upload(ctx, solo.data(), solo.size(), &ctx->d_solo))) {
    ctx->free_scene();
    return rc;
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  S.objects = dobj;
  S.lights = dlights;
  S.meshes = dmeshes;
  S.groups = dgroups;
  S.materials = dmat;
  S.textures = dtex;
  S.perlins = dper;
  S.images = dimg;
  S.cie = ctx->d_cie;
  S.smits = ctx->d_smits;
  S.n_objects = d->n_objects;
  S.n_lights = d->n_lights;
  for (int k = 0; k < 3; ++k) S.background[k] = d->background_rgb[k];
  ctx->n_meshes = d->n_meshes;
  ctx->h_objects.assign(d->objects, d->objects + d->n_objects);
  ctx->h_meshes = meshes;
  ctx->have_scene = true;
  return YART_OK;
}

int yart_ctx_set_scene(yart_ctx* ctx, const yart_scene_desc* d) {
  if (!ctx) return YART_ERR_INVALID;
  if (!d) {
    ctx->err = "yart_ctx_set_scene: null scene";
    return YART_ERR_INVALID;
  }
  struct Cleanup { // every failing path, exceptions included: nothing half-built stays behind
    yart_ctx* c;
    bool armed;
    ~Cleanup() {
      if (armed) c->free_scene();
    }
  } cleanup{ctx, true};
  YART_ABI_GUARD_BEGIN
  const int rc = set_scene_impl(ctx, d);
  cleanup.armed = rc != YART_OK;
  return rc;
  YART_ABI_GUARD_END(ctx, "yart_ctx_set_scene")
}

static int closest_hit_impl(yart_ctx* ctx, uint32_t target, const void* rays, bool f32, uint64_t n, double t_min, double t_max,
                            uint32_t order, uint32_t flags, void* hits, yart_stats* stats) {
  const char* fn = f32 ? "yart_closest_hit_f32" : "yart_closest_hit";
  if (!ctx->have_scene) {
    ctx->err = std::string(fn) + ": no scene (call yart_ctx_set_scene first)";
    return YART_ERR_INVALID;
  }
  if ((n && (!rays || !hits)) || n > 0xFFFFFFF0ull || order > YART_ORDER_NEAR) {
    ctx->err = std::string(fn) + ": bad argument";
    return YART_ERR_INVALID;
  }
  const uintptr_t ray_align = f32 ? 7u : 15u, hit_align = f32 ? 3u : 7u;
  if ((flags & YART_FLAG_DEVICE_PTRS) && ((reinterpret_cast<uintptr_t>(rays) & ray_align) || (reinterpret_cast<uintptr_t>(hits) & hit_align))) {
    ctx->err = std::string(fn) + (f32 ? ": device ray arrays must be 8-byte aligned (hits: 4)" : ": device ray arrays must be 16-byte aligned (hits: 8)");
    return YART_ERR_INVALID;
  }
  if (target != YART_TARGET_WORLD && target >= ctx->n_meshes) {
    ctx->err = std::string(fn) + ": target is neither a mesh index nor YART_TARGET_WORLD";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n == 0) return YART_OK;
  const size_t ray_bytes = f32 ? sizeof(yart_ray_f32) : sizeof(yart_ray), hit_bytes = f32 ? sizeof(yart_hit_f32) : sizeof(yart_hit);
  const bool dev = (flags & YART_FLAG_DEVICE_PTRS) != 0;
  const bool count = (flags & YART_FLAG_COUNT_VISITS) != 0;
  const char* d_rays = static_cast<const char*>(rays);
  char* d_hits = static_cast<char*>(hits);
  if (!dev) {
    CUDA_TRY(ctx, ctx->rays.reserve(n * ray_bytes));
    CUDA_TRY(ctx, ctx->hits_export.reserve(n * hit_bytes));
    d_rays = ctx->rays.as<char>();
    d_hits = ctx->hits_export.as<char>();
  }
  const uint32_t n_list = (target == YART_TARGET_WORLD) ? ctx->scene.n_objects : 1u;
  const size_t work_bytes = ((size_t)n_list + 2) * sizeof(uint32_t);
  CUDA_TRY(ctx, ctx->work.reserve(work_bytes));
  CUDA_TRY(ctx, ctx->counters.reserve(64));
  CUDA_TRY(ctx, ctx->hits.reserve(n * sizeof(DevHit)));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counters.p, 0, 64, ctx->stream));

  yart_object solo;
  memset(&solo, 0, sizeof(solo));
  solo.kind = YART_OBJ_MESH;
  solo.cos_theta = 1.0;
  QueryArgs q;
  memset(&q, 0, sizeof(q));
  q.c.t_min = t_min;
  q.c.t_max = t_max;
  DevScene export_scene = ctx->scene;
  if (target == YART_TARGET_WORLD) {
    q.d_objects = ctx->scene.objects;
    q.h_objects = ctx->h_objects.data();
    q.n_objects = ctx->scene.n_objects;
  } else {
    solo.index = target;
    q.d_objects = ctx->d_solo + target;
    q.h_objects = &solo;
    q.n_objects = 1;
    export_scene.objects = ctx->d_solo + target;
  }
  q.seed = 0;
  q.bounce = 1;
  q.spp_batch = 1; // media inside world.hit: Philox stream of pixel = ray index, sample 0, bounce 1
  q.work_counters = ctx->work.as<uint32_t>();
  q.counters = ctx->counters.as<unsigned long long>();
  q.near = order == YART_ORDER_NEAR;
  q.count = count;
  uint64_t launches = 0;
  // The passes + the export over rays [off, off + len), on the context's stream.
  auto run_range = [&](uint64_t off, uint64_t len) -> int {
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->work.p, 0, work_bytes, ctx->stream));
    const char* r = d_rays + off * ray_bytes;
    q.c.rays = f32 ? nullptr : reinterpret_cast<const yart_ray*>(r);
    q.c.rays32 = f32 ? reinterpret_cast<const yart_ray_f32*>(r) : nullptr;
    q.c.n_items = len;
    q.c.n_rays = (uint32_t)len;
    q.c.hits = ctx->hits.as<DevHit>() + off;
    q.pixel_base = (uint32_t)off; // (keeps a ray's Philox stream = its index in the caller's array)
    const int rc = run_passes(ctx, q, &launches);
    if (rc) return rc;
    if (f32)
      k_export_f32<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(export_scene, export_scene.objects, q.c.hits,
                                                               reinterpret_cast<yart_hit_f32*>(d_hits + off * hit_bytes), len);
    else
      k_export<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(export_scene, q.c.rays, q.c.hits,
                                                           reinterpret_cast<yart_hit*>(d_hits + off * hit_bytes), len);
    launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return YART_OK;
  };
  uint64_t n_chunks = 0;
  const int rc = run_chunked(ctx, dev, rays, ray_bytes, hits, hit_bytes, n, d_rays, d_hits, run_range, &n_chunks);
  if (rc) return rc;
  unsigned long long c[2] = {0, 0};
  if (count) CUDA_TRY(ctx, cudaMemcpyAsync(c, ctx->counters.p, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (stats) {
    float ms = 0.f;
    const int erc = chunked_kernel_ms(ctx, n_chunks, dev, &ms);
    if (erc) return erc;
    stats->rays = n;
    stats->node_visits = c[0];
    stats->tri_tests = c[1];
    stats->kernel_launches = launches;
    stats->trace_launches = (uint32_t)(launches - (dev ? 1 : n_chunks)); // (one export kernel per chunk)
    stats->gpu_ms = ms;
    stats->trace_ms = ms;
  }
  return YART_OK;
}

int yart_closest_hit(yart_ctx* ctx, uint32_t target, const yart_ray* rays, uint64_t n, double t_min, double t_max,
                     uint32_t order, uint32_t flags, yart_hit* hits, yart_stats* stats) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  return closest_hit_impl(ctx, target, rays, false, n, t_min, t_max, order, flags, hits, stats);
  YART_ABI_GUARD_END(ctx, "yart_closest_hit")
}

int yart_closest_hit_f32(yart_ctx* ctx, uint32_t target, const yart_ray_f32* rays, uint64_t n, float t_min, float t_max,
                         uint32_t order, uint32_t flags, yart_hit_f32* hits, yart_stats* stats) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  return closest_hit_impl(ctx, target, rays, true, n, (double)t_min, (double)t_max, order, flags, hits, stats);
  YART_ABI_GUARD_END(ctx, "yart_closest_hit_f32")
}

static int occluded_impl(yart_ctx* ctx, uint32_t target, const void* rays, bool f32, uint64_t n, double t_min, double t_max,
                         uint32_t flags, uint8_t* occluded, yart_stats* stats) {
  const char* fn = f32 ? "yart_occluded_f32" : "yart_occluded";
  if (!ctx->have_scene) {
    ctx->err = std::string(fn) + ": no scene (call yart_ctx_set_scene first)";
    return YART_ERR_INVALID;
  }
  if ((n && (!rays || !occluded)) || n > 0xFFFFFFF0ull) {
    ctx->err = std::string(fn) + ": bad argument";
    return YART_ERR_INVALID;
  }
  if (flags & ~(uint32_t)YART_FLAG_DEVICE_PTRS) {
    ctx->err = std::string(fn) + ": the only flag it takes is YART_FLAG_DEVICE_PTRS";
    return YART_ERR_INVALID;
  }
  const bool dev = (flags & YART_FLAG_DEVICE_PTRS) != 0;
  if (dev && (reinterpret_cast<uintptr_t>(rays) & (f32 ? 7u : 15u))) {
    ctx->err = std::string(fn) + (f32 ? ": device ray arrays must be 8-byte aligned" : ": device ray arrays must be 16-byte aligned");
    return YART_ERR_INVALID;
  }
  if (target != YART_TARGET_WORLD && target >= ctx->n_meshes) {
    ctx->err = std::string(fn) + ": target is neither a mesh index nor YART_TARGET_WORLD";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n == 0) return YART_OK;
  const size_t ray_bytes = f32 ? sizeof(yart_ray_f32) : sizeof(yart_ray);
  const char* d_rays = static_cast<const char*>(rays);
  char* d_out = reinterpret_cast<char*>(occluded);
  if (!dev) { // (no export pass: the kernels write the flags straight into the staging buffer that is downloaded)
    CUDA_TRY(ctx, ctx->rays.reserve(n * ray_bytes));
    CUDA_TRY(ctx, ctx->occluded.reserve(n));
    d_rays = ctx->rays.as<char>();
    d_out = ctx->occluded.as<char>();
  }
  const uint32_t n_list = (target == YART_TARGET_WORLD) ? ctx->scene.n_objects : 1u;
  const size_t work_bytes = ((size_t)n_list + 2) * sizeof(uint32_t);
  CUDA_TRY(ctx, ctx->work.reserve(work_bytes));

  yart_object solo;
  memset(&solo, 0, sizeof(solo));
  solo.kind = YART_OBJ_MESH;
  solo.cos_theta = 1.0;
  OcclusionArgs q;
  memset(&q, 0, sizeof(q));
  q.c.t_min = t_min;
  q.c.t_max = t_max;
  if (target == YART_TARGET_WORLD) {
    q.d_objects = ctx->scene.objects;
    q.h_objects = ctx->h_objects.data();
    q.n_objects = ctx->scene.n_objects;
  } else {
    solo.index = target;
    q.d_objects = ctx->d_solo + target;
    q.h_objects = &solo;
    q.n_objects = 1;
  }
  q.work_counters = ctx->work.as<uint32_t>();
  uint64_t launches = 0;
  // the passes over rays [off, off + len), on the context's stream
  auto run_range = [&](uint64_t off, uint64_t len) -> int {
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->work.p, 0, work_bytes, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(d_out + off, 0, len, ctx->stream));
    const char* r = d_rays + off * ray_bytes;
    q.c.rays = f32 ? nullptr : reinterpret_cast<const yart_ray*>(r);
    q.c.rays32 = f32 ? reinterpret_cast<const yart_ray_f32*>(r) : nullptr;
    q.c.occluded = reinterpret_cast<uint8_t*>(d_out + off);
    q.c.n_rays = (uint32_t)len;
    q.pixel_base = (uint32_t)off; // (keeps a ray's Philox stream = its index in the caller's array)
    return run_occlusion_passes(ctx, q, &launches);
  };
  uint64_t n_chunks = 0;
  const int rc = run_chunked(ctx, dev, rays, ray_bytes, occluded, 1, n, d_rays, d_out, run_range, &n_chunks);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (stats) {
    float ms = 0.f;
    const int erc = chunked_kernel_ms(ctx, n_chunks, dev, &ms);
    if (erc) return erc;
    stats->rays = n;
    stats->kernel_launches = launches;
    stats->trace_launches = (uint32_t)launches;
    stats->gpu_ms = ms;
    stats->trace_ms = ms;
  }
  return YART_OK;
}

int yart_occluded(yart_ctx* ctx, uint32_t target, const yart_ray* rays, uint64_t n, double t_min, double t_max,
                  uint32_t flags, uint8_t* occluded, yart_stats* stats) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  return occluded_impl(ctx, target, rays, false, n, t_min, t_max, flags, occluded, stats);
  YART_ABI_GUARD_END(ctx, "yart_occluded")
}

int yart_occluded_f32(yart_ctx* ctx, uint32_t target, const yart_ray_f32* rays, uint64_t n, float t_min, float t_max,
                      uint32_t flags, uint8_t* occluded, yart_stats* stats) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  return occluded_impl(ctx, target, rays, true, n, (double)t_min, (double)t_max, flags, occluded, stats);
  YART_ABI_GUARD_END(ctx, "yart_occluded_f32")
}

static int fill_render_params(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, RenderParams& R) {
  if (o->width < 2 || o->height < 2 || o->sample_end < o->sample_begin || o->max_depth == 0 || o->order > YART_ORDER_NEAR ||
      (uint64_t)o->width * o->height > 0x7FFFFFFFull) {
    ctx->err = "render options: need width,height >= 2, sample_begin <= sample_end, max_depth >= 1";
    return YART_ERR_INVALID;
  }
  memset(&R, 0, sizeof(R));
  R.scene = ctx->scene;
  R.cam = make_camera(*cam);
  R.width = o->width;
  R.height = o->height;
  R.max_depth = o->max_depth;
  R.seed = o->seed;
  R.flags = o->flags & (YART_FLAG_UNBIASED_LIGHT_PICK | YART_FLAG_RUSSIAN_ROULETTE | YART_FLAG_DEPTH_ZERO_BLACK | YART_FLAG_NEXT_EVENT);
  if (R.flags & YART_FLAG_NEXT_EVENT) R.flags |= YART_FLAG_UNBIASED_LIGHT_PICK; // MIS needs the mixture's true density
  {
    // A trailing run of plain spheres that directly follows a mesh pass is intersected inside k_shade (which
    // reads the ray and the hit anyway) -- saves one read-modify-write pass over the queue per bounce.
    static const int fold = tune_env("YART_TUNE_FOLD_TAIL", 1);
    const uint32_t n_obj = ctx->scene.n_objects;
    uint32_t tb = n_obj;
    while (tb > 0 && ctx->h_objects[tb - 1].kind == YART_OBJ_SPHERE && ctx->h_objects[tb - 1].wrap == 0) tb--;
    const bool after_mesh = tb > 0 && ctx->h_objects[tb - 1].kind == YART_OBJ_MESH && !(ctx->h_objects[tb - 1].wrap & YART_WRAP_MEDIUM);
    if (!fold || !after_mesh || n_obj - tb > 16) tb = n_obj;
    R.tail_begin = tb;
    R.tail_end = n_obj;
  }
  return YART_OK;
}

static int render_impl(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, double* film_xyz, yart_stats* stats,
                       yart_ray* dump_out, uint64_t dump_cap);

int yart_render(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, double* film_xyz, yart_stats* stats) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  if (!film_xyz) {
    ctx->err = "yart_render: null film";
    return YART_ERR_INVALID;
  }
  return render_impl(ctx, cam, o, film_xyz, stats, nullptr, 0);
  YART_ABI_GUARD_END(ctx, "yart_render")
}

int yart_dump_path_rays(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, yart_ray* rays, uint64_t cap,
                        uint64_t* n_out) {
  if (!ctx) return YART_ERR_INVALID;
  YART_ABI_GUARD_BEGIN
  if (!o || (cap && !rays) || !n_out) {
    ctx->err = "yart_dump_path_rays: null argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const bool dev = (o->flags & YART_FLAG_DEVICE_PTRS) != 0;
  if (dev && (reinterpret_cast<uintptr_t>(rays) & 15u)) {
    ctx->err = "yart_dump_path_rays: device ray arrays must be 16-byte aligned";
    return YART_ERR_INVALID;
  }
  yart_ray* d_out = rays;
  if (!dev && cap) {
    CUDA_TRY(ctx, ctx->hits_export.reserve(cap * sizeof(yart_ray))); // (a scratch buffer no render kernel touches)
    d_out = ctx->hits_export.as<yart_ray>();
  }
  yart_stats st;
  const int rc = render_impl(ctx, cam, o, nullptr, &st, d_out, cap);
  if (rc) return rc;
  *n_out = st.rays;
  const uint64_t n_copy = std::min<uint64_t>(st.rays, cap);
  if (!dev && n_copy) {
    CUDA_TRY(ctx, cudaMemcpyAsync(rays, d_out, n_copy * sizeof(yart_ray), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return YART_OK;
  YART_ABI_GUARD_END(ctx, "yart_dump_path_rays")
}

// film_xyz == nullptr (yart_dump_path_rays): the samples are traced exactly as for a render, the film is a scratch
// buffer that is thrown away, and every bounce's rays are copied to dump_out.
static int render_impl(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, double* film_xyz, yart_stats* stats,
                       yart_ray* dump_out, uint64_t dump_cap) {
  if (!ctx->have_scene || !cam || !o) {
    ctx->err = "yart_render: missing scene or null argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  RenderParams R;
  int rc = fill_render_params(ctx, cam, o, R);
  if (rc) return rc;
  if (stats) memset(stats, 0, sizeof(*stats));
  const uint32_t n_pixels_total = o->width * o->height;
  const uint32_t n_samples = o->sample_end - o->sample_begin;
  const bool dumping = film_xyz == nullptr;
  const bool dev = !dumping && (o->flags & YART_FLAG_DEVICE_PTRS) != 0;
  const size_t film_bytes = (size_t)n_pixels_total * 3 * sizeof(double);
  double* d_film = film_xyz;
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  if (!dev) {
    CUDA_TRY(ctx, ctx->film.reserve(film_bytes));
    d_film = ctx->film.as<double>();
    if (dumping) CUDA_TRY(ctx, cudaMemsetAsync(d_film, 0, film_bytes, ctx->stream));
    else CUDA_TRY(ctx, cudaMemcpyAsync(d_film, film_xyz, film_bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  uint64_t total_rays = 0, total_paths = 0, launches = 0, trace_launches = 0;
  double trace_ms = 0.0;
  uint32_t deepest = 0;
  if (n_samples > 0) {
    // Batch shape: whole frame x spp_batch, or pixel chunks when the frame alone is too large.
    // Big batches: every batch pays ~12 ms of fixed cost (the nearly empty tail bounces run at the latency of
    // their longest ray), so put up to 256 Mi paths in flight -- 112 B of state each (48 ray + 8 time + 8 wavelength
    // + 8 throughput + 32 hit + 2 x 4 queue) = 30 GB of the 180 GB: david 1080p at 32 / 64 / 128 spp per batch
    // = 1121 / 1146 / 1158 Mrays/s.  The cap is also bounded by what is actually FREE on the device right now
    // (minus a margin), so that a busy GPU gets smaller batches instead of a failed cudaMalloc.
    static const int max_paths_log2 = std::max(10, std::min(30, tune_env("YART_TUNE_MAX_PATHS_LOG2", 28)));
    uint64_t kMaxPaths = 1ull << max_paths_log2;
    const bool nee = (R.flags & YART_FLAG_NEXT_EVENT) != 0;
    {
      // YART_FLAG_NEXT_EVENT adds 76 B: 48 shadow ray + 8 pending + 8 light-sample sum + 8 emission weight + 4 shadow queue
      // (the shadow passes write their hits into the path hits, which are dead from k_shade to the next bounce's passes)
      const uint64_t kNeeBytesPerPath = sizeof(yart_ray) + 3 * sizeof(double) + sizeof(uint32_t);
      const uint64_t kStateBytesPerPath = sizeof(yart_ray) + 3 * sizeof(double) + sizeof(DevHit) + 2 * sizeof(uint32_t) +
                                          (nee ? kNeeBytesPerPath : 0);
      if (!nee) // a flag-off render does not keep an earlier NEE render's state alive (no-op when there is none)
        for (DevBuf* b : {&ctx->nee_rays, &ctx->nee_pending, &ctx->nee_sum, &ctx->nee_w, &ctx->queue_s}) b->release();
      size_t free_b = 0, total_b = 0;
      CUDA_TRY(ctx, cudaMemGetInfo(&free_b, &total_b));
      const DevBuf* held[] = {&ctx->rays, &ctx->time, &ctx->wavelength, &ctx->throughput, &ctx->hits, &ctx->queue_a, &ctx->queue_b,
                              &ctx->nee_rays, &ctx->nee_pending, &ctx->nee_sum, &ctx->nee_w, &ctx->queue_s};
      uint64_t avail = free_b; // what the state buffers may grow into: free memory + what they already hold
      for (const DevBuf* b : held) avail += b->cap;
      const uint64_t margin = (256ull << 20) + (dev ? 0 : film_bytes);
      const uint64_t fit = avail > margin ? (avail - margin) / kStateBytesPerPath : 0;
      kMaxPaths = std::min<uint64_t>(kMaxPaths, fit);
      static const int mem_cap_mb = tune_env("YART_TUNE_STATE_MB", 0); // testing: pretend only this much is free
      if (mem_cap_mb > 0) kMaxPaths = std::min<uint64_t>(kMaxPaths, ((uint64_t)mem_cap_mb << 20) / kStateBytesPerPath);
      if (kMaxPaths < 1024) {
        ctx->err = "yart_render: not enough free device memory for the path state (" + std::to_string(free_b >> 20) +
                   " MiB free of " + std::to_string(total_b >> 20) + " MiB; " + std::to_string(kStateBytesPerPath) +
                   " bytes per path in flight)";
        return YART_ERR_NOMEM;
      }
    }
    uint32_t spp_batch = o->batch_spp ? o->batch_spp : (uint32_t)std::max<uint64_t>(1, kMaxPaths / n_pixels_total);
    spp_batch = std::min(spp_batch, n_samples);
    uint32_t pix_chunk = n_pixels_total;
    if ((uint64_t)pix_chunk * spp_batch > kMaxPaths) pix_chunk = (uint32_t)std::max<uint64_t>(1, kMaxPaths / spp_batch);
    const uint64_t cap = (uint64_t)pix_chunk * spp_batch;
    CUDA_TRY(ctx, ctx->rays.reserve(cap * sizeof(yart_ray)));
    CUDA_TRY(ctx, ctx->time.reserve(cap * sizeof(double)));
    CUDA_TRY(ctx, ctx->wavelength.reserve(cap * sizeof(double)));
    CUDA_TRY(ctx, ctx->throughput.reserve(cap * sizeof(double)));
    CUDA_TRY(ctx, ctx->hits.reserve(cap * sizeof(DevHit)));
    CUDA_TRY(ctx, ctx->queue_a.reserve(cap * sizeof(uint32_t)));
    CUDA_TRY(ctx, ctx->queue_b.reserve(cap * sizeof(uint32_t)));
    const uint32_t D = o->max_depth;
    // with NEE: path counts [0, D+2), then the shadow queue's count of bounce b at D+2+b; path work counters, then the
    // shadow passes' ones
    const size_t n_counts = (size_t)D + 2 + (nee ? (size_t)D + 1 : 0);
    const size_t n_obj_slots = (size_t)ctx->scene.n_objects + 1;
    const size_t n_work = n_obj_slots * D * (nee ? 2 : 1);
    CUDA_TRY(ctx, ctx->counts.reserve(n_counts * sizeof(uint32_t)));
    CUDA_TRY(ctx, ctx->work.reserve(n_work * sizeof(uint32_t)));
    NeeState N;
    memset(&N, 0, sizeof(N));
    if (nee) {
      CUDA_TRY(ctx, ctx->nee_rays.reserve(cap * sizeof(yart_ray)));
      CUDA_TRY(ctx, ctx->nee_pending.reserve(cap * sizeof(double)));
      CUDA_TRY(ctx, ctx->nee_sum.reserve(cap * sizeof(double)));
      CUDA_TRY(ctx, ctx->nee_w.reserve(cap * sizeof(double)));
      CUDA_TRY(ctx, ctx->queue_s.reserve(cap * sizeof(uint32_t)));
      N.rays = ctx->nee_rays.as<yart_ray>();
      N.pending = ctx->nee_pending.as<double>();
      N.sum = ctx->nee_sum.as<double>();
      N.w_emit = ctx->nee_w.as<double>();
      N.queue = ctx->queue_s.as<uint32_t>();
      N.counts = ctx->counts.as<uint32_t>() + D + 2;
    }
    // events: [0, 2D) closest-hit passes per bounce, [2D, 4D) YART_DEBUG_BOUNCES's shade timing, [4D, 6D) shadow passes
    while (ctx->ev_pool.size() < (nee ? 6 : 2) * (size_t)D) {
      cudaEvent_t e;
      CUDA_TRY(ctx, cudaEventCreate(&e));
      ctx->ev_pool.push_back(e);
    }
    R.st.rays = ctx->rays.as<yart_ray>();
    R.st.time = ctx->time.as<double>();
    R.st.wavelength = ctx->wavelength.as<double>();
    R.st.throughput = ctx->throughput.as<double>();
    R.st.hits = ctx->hits.as<DevHit>();
    uint32_t* counts = ctx->counts.as<uint32_t>();
    uint32_t* work = ctx->work.as<uint32_t>();
    std::vector<uint32_t> h_counts(n_counts);
    const bool near = o->order == YART_ORDER_NEAR;
    const bool count = (o->flags & YART_FLAG_COUNT_VISITS) != 0;
    const int stream_grid = ctx->sm_count * 8;
    CUDA_TRY(ctx, ctx->counters.reserve(64));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->counters.p, 0, 64, ctx->stream));

    for (uint32_t s0 = o->sample_begin; s0 < o->sample_end; s0 += spp_batch) {
      const uint32_t spp = std::min(spp_batch, o->sample_end - s0);
      for (uint32_t p0 = 0; p0 < n_pixels_total; p0 += pix_chunk) {
        R.pixel_base = p0;
        R.n_pixels = std::min(pix_chunk, n_pixels_total - p0);
        R.sample_base = s0;
        R.spp_batch = spp;
        CUDA_TRY(ctx, cudaMemsetAsync(counts, 0, n_counts * sizeof(uint32_t), ctx->stream));
        CUDA_TRY(ctx, cudaMemsetAsync(work, 0, n_work * sizeof(uint32_t), ctx->stream));
        uint32_t* qa = ctx->queue_a.as<uint32_t>();
        uint32_t* qb = ctx->queue_b.as<uint32_t>();
        if (nee) k_raygen<true><<<stream_grid, 256, 0, ctx->stream>>>(R, qa, counts + 1, N);
        else k_raygen<false><<<stream_grid, 256, 0, ctx->stream>>>(R, qa, counts + 1, N);
        launches++;
        uint32_t b_done = 0;
        for (uint32_t b = 1; b <= D; ++b) {
          QueryArgs q;
          memset(&q, 0, sizeof(q));
          q.c.rays = R.st.rays;
          q.c.queue = qa;
          q.c.n_items_dev = counts + b;
          q.c.n_rays = R.n_pixels * spp;
          q.c.hits = R.st.hits;
          q.c.t_min = 0.001; // world.hit(ray_in, 0.001, f64::INFINITY) (main.rs:548)
          q.c.t_max = INFINITY;
          q.d_objects = ctx->scene.objects;
          q.h_objects = ctx->h_objects.data();
          q.n_objects = R.tail_begin; // (== n_objects unless k_shade takes a trailing run of spheres)
          q.ray_time = R.st.time;
          q.seed = o->seed;
          q.bounce = b;
          q.spp_batch = spp;
          q.sample_base = s0;
          q.pixel_base = p0;
          q.work_counters = work + (size_t)(b - 1) * n_obj_slots;
          q.counters = ctx->counters.as<unsigned long long>();
          q.near = near;
          q.count = count;
          if (dump_out) {
            k_dump_rays<<<stream_grid, 256, 0, ctx->stream>>>(R.st.rays, qa, counts, b, total_rays, dump_out, dump_cap);
            launches++;
          }
          CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[2 * (b - 1)], ctx->stream));
          rc = run_passes(ctx, q, &trace_launches);
          if (rc) return rc;
          CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[2 * (b - 1) + 1], ctx->stream));
          static const int dbg_shade_ev = tune_env("YART_DEBUG_BOUNCES", 0);
          if (dbg_shade_ev) {
            while (ctx->ev_pool.size() < 4 * (size_t)D) {
              cudaEvent_t e;
              CUDA_TRY(ctx, cudaEventCreate(&e));
              ctx->ev_pool.push_back(e);
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[2 * D + 2 * (b - 1)], ctx->stream));
          }
          const int shade_grid = std::max(1, stream_grid * 256 / kShadeThreads);
          if (nee) k_shade<true><<<shade_grid, kShadeThreads, 0, ctx->stream>>>(R, qa, counts + b, qb, counts + b + 1, b, N);
          else k_shade<false><<<shade_grid, kShadeThreads, 0, ctx->stream>>>(R, qa, counts + b, qb, counts + b + 1, b, N);
          launches += 1;
          if (dbg_shade_ev) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[2 * D + 2 * (b - 1) + 1], ctx->stream));
          if (nee && b < D) { // the shadow rays k_shade queued: the same world query, on their own queue and Philox stream
            QueryArgs sq = q;
            sq.c.rays = N.rays;
            sq.c.queue = N.queue;
            sq.c.n_items_dev = N.counts + b;
            sq.bounce = YART_NEE_BOUNCE_BASE + b;
            sq.work_counters = work + (size_t)(D + b - 1) * n_obj_slots;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[4 * D + 2 * (b - 1)], ctx->stream));
            rc = run_passes(ctx, sq, &trace_launches);
            if (rc) return rc;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[4 * D + 2 * (b - 1) + 1], ctx->stream));
            k_nee_resolve<<<stream_grid, 256, 0, ctx->stream>>>(R, b, N);
            launches += 1;
          }
          std::swap(qa, qb);
          b_done = b;
          // the tail of the bounce loop is nearly empty: look at the live count now and then
          if (b >= 4 && (b % 4) == 0 && b < D) {
            uint32_t live = 0;
            CUDA_TRY(ctx, cudaMemcpyAsync(&live, counts + b + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            if (live == 0) break;
          }
        }
        if (nee) k_film_accumulate<true><<<stream_grid, 256, 0, ctx->stream>>>(R, d_film, N);
        else k_film_accumulate<false><<<stream_grid, 256, 0, ctx->stream>>>(R, d_film, N);
        launches++;
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaMemcpyAsync(h_counts.data(), counts, n_counts * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        total_paths += h_counts[1];
        static const int debug_bounces = tune_env("YART_DEBUG_BOUNCES", 0);
        for (uint32_t b = 1; b <= b_done; ++b) {
          total_rays += h_counts[b];
          if (h_counts[b]) deepest = std::max(deepest, b);
          float ms = 0.f;
          CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev_pool[2 * (b - 1)], ctx->ev_pool[2 * (b - 1) + 1]));
          trace_ms += ms;
          if (nee && b < D) {
            float shadow_ms = 0.f;
            CUDA_TRY(ctx, cudaEventElapsedTime(&shadow_ms, ctx->ev_pool[4 * D + 2 * (b - 1)], ctx->ev_pool[4 * D + 2 * (b - 1) + 1]));
            trace_ms += shadow_ms;
          }
          if (debug_bounces) {
            float gap = 0.f; // from the end of this bounce's closest-hit stage to the start of the next one
            if (b < b_done) cudaEventElapsedTime(&gap, ctx->ev_pool[2 * (b - 1) + 1], ctx->ev_pool[2 * b]);
            float shade = 0.f;
            cudaEventElapsedTime(&shade, ctx->ev_pool[2 * D + 2 * (b - 1)], ctx->ev_pool[2 * D + 2 * (b - 1) + 1]);
            fprintf(stderr, "bounce %2u: rays %9u  closest-hit %8.3f ms  shade %8.3f ms  shade+gap %8.3f ms", b, h_counts[b], ms, shade, gap);
            if (nee) fprintf(stderr, "  shadow rays %9u", b < D ? h_counts[D + 2 + b] : 0u);
            fprintf(stderr, "\n");
          }
        }
      }
    }
  }
  if (!dev && !dumping) CUDA_TRY(ctx, cudaMemcpyAsync(film_xyz, d_film, film_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  unsigned long long visit[2] = {0, 0};
  if ((o->flags & YART_FLAG_COUNT_VISITS) && n_samples > 0)
    CUDA_TRY(ctx, cudaMemcpyAsync(visit, ctx->counters.p, sizeof(visit), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (stats) {
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    stats->node_visits = visit[0];
    stats->tri_tests = visit[1];
    stats->rays = total_rays;
    stats->paths = total_paths;
    stats->kernel_launches = launches + trace_launches;
    stats->trace_launches = (uint32_t)trace_launches;
    stats->gpu_ms = ms;
    stats->trace_ms = trace_ms;
    stats->max_bounce = deepest;
  }
  return YART_OK;
}

int yart_film_finalize(yart_ctx* ctx, const double* film_xyz, uint32_t width, uint32_t height, uint32_t spp, uint32_t flags,
                       uint8_t* rgba8) {
  if (!ctx) return YART_ERR_INVALID;
  if (!film_xyz || !rgba8 || !width || !height || !spp) {
    ctx->err = "yart_film_finalize: bad argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)width * height;
  const bool dev = (flags & YART_FLAG_DEVICE_PTRS) != 0;
  const double* d_film = film_xyz;
  uint8_t* d_rgba = rgba8;
  if (!dev) {
    CUDA_TRY(ctx, ctx->film.reserve(n * 3 * sizeof(double)));
    CUDA_TRY(ctx, ctx->rgba.reserve(n * 4));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->film.p, film_xyz, n * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    d_film = ctx->film.as<double>();
    d_rgba = ctx->rgba.as<uint8_t>();
  }
  k_film_finalize<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_film, width, height, spp, d_rgba);
  CUDA_TRY(ctx, cudaGetLastError());
  if (!dev) CUDA_TRY(ctx, cudaMemcpyAsync(rgba8, d_rgba, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return YART_OK;
}

int yart_generate_camera_rays(yart_ctx* ctx, const yart_camera* cam, const yart_render_opts* o, yart_ray* rays_host,
                              double* wavelength_host, double* time_host) {
  if (!ctx) return YART_ERR_INVALID;
  if (!cam || !o || !rays_host) {
    ctx->err = "yart_generate_camera_rays: null argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  RenderParams R;
  int rc = fill_render_params(ctx, cam, o, R);
  if (rc) return rc;
  const uint32_t ns = o->sample_end - o->sample_begin;
  const uint64_t n = (uint64_t)o->width * o->height * ns;
  if (n == 0) return YART_OK;
  CUDA_TRY(ctx, ctx->rays.reserve(n * sizeof(yart_ray)));
  CUDA_TRY(ctx, ctx->wavelength.reserve(n * sizeof(double)));
  CUDA_TRY(ctx, ctx->time.reserve(n * sizeof(double)));
  R.pixel_base = 0;
  R.n_pixels = o->width * o->height;
  R.sample_base = o->sample_begin;
  R.spp_batch = ns;
  k_camera_rays<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(R, ctx->rays.as<yart_ray>(), ctx->wavelength.as<double>(),
                                                            ctx->time.as<double>());
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(rays_host, ctx->rays.p, n * sizeof(yart_ray), cudaMemcpyDeviceToHost, ctx->stream));
  if (wavelength_host)
    CUDA_TRY(ctx, cudaMemcpyAsync(wavelength_host, ctx->wavelength.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (time_host) CUDA_TRY(ctx, cudaMemcpyAsync(time_host, ctx->time.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return YART_OK;
}

int yart_measure_fetch_peak(yart_ctx* ctx, uint64_t table_bytes, uint32_t fetches_per_thread, uint32_t mode,
                            double* gbytes_per_s) {
  if (!ctx) return YART_ERR_INVALID;
  if (!gbytes_per_s || table_bytes < 128 || table_bytes > (1ull << 36) || fetches_per_thread == 0 || mode > 3) {
    ctx->err = "yart_measure_fetch_peak: bad argument";
    return YART_ERR_INVALID;
  }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const uint32_t n_lines = (uint32_t)std::min<uint64_t>(table_bytes / 128, 0x7FFFFFFFull);
  DevBuf table, sink;
  cudaError_t e = table.reserve((size_t)n_lines * 128);
  if (e == cudaSuccess) e = sink.reserve(64);
  if (e == cudaSuccess) e = cudaMemsetAsync(table.p, 0, (size_t)n_lines * 128, ctx->stream);
  float ms = 0.f;
  size_t threads = 0;
  if (e == cudaSuccess) {
    static const int carve = tune_env("YART_TUNE_CARVEOUT_LEAN", 50);
    auto run = [&](auto kernel, int block, bool set_carve) {
      if (set_carve) cudaFuncSetAttribute(reinterpret_cast<const void*>(kernel), cudaFuncAttributePreferredSharedMemoryCarveout, carve);
      int per_sm = 1;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(kernel), block, 0);
      const int grid = std::max(per_sm, 1) * ctx->sm_count;
      threads = (size_t)grid * block;
      kernel<<<grid, block, 0, ctx->stream>>>(table.as<float4>(), n_lines, fetches_per_thread / 8 + 1, sink.as<float>()); // warm L2
      cudaEventRecord(ctx->ev0, ctx->stream);
      kernel<<<grid, block, 0, ctx->stream>>>(table.as<float4>(), n_lines, fetches_per_thread, sink.as<float>());
      cudaEventRecord(ctx->ev1, ctx->stream);
    };
    // mode 0: 128-thread CTAs, 5 per SM -- 20 warps per SM like k_traverse_lean (its register budget, not this
    // kernel's, is what limits it), same carveout; mode 1: whatever fits
    // modes 2 / 3: the same two occupancies with four lanes per line (k_fetch_peak_quad)
    if (mode == 0) run(k_fetch_peak<128, 5>, 128, true);
    else if (mode == 1) run(k_fetch_peak<256, 8>, 256, false);
    else if (mode == 2) run(k_fetch_peak_quad<128, 5>, 128, true);
    else run(k_fetch_peak_quad<256, 8>, 256, false);
    e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  }
  table.release();
  sink.release();
  if (e != cudaSuccess) {
    ctx->err = std::string("yart_measure_fetch_peak: ") + cudaGetErrorString(e);
    return YART_ERR_CUDA;
  }
  *gbytes_per_s = (double)threads * fetches_per_thread * (mode >= 2 ? 32.0 : 128.0) / (ms * 1e-3) / 1e9;
  return YART_OK;
}

} // extern "C"
