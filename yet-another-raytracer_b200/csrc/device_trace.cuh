// device_trace.cuh -- closest-hit: the persistent-thread QBVH traversal kernel and the analytic
// primitives around it.
//
// HittableList::hit (reference hittable.rs:66-79) walks the world's object list in order with a
// shrinking [t_min, closest] interval.  Here the list is cut into PASSES, run in list order over
// the whole ray queue, each pass reading and updating the per-ray closest hit in HBM:
//   * a TriangleMesh object = one launch of k_traverse: L4QBVH::hit (qbvh.rs:381-543) with the
//     rays moved into the instance's space (Translate / RotateY, hittable.rs:136-152, 217-251);
//   * a run of consecutive analytic objects = one launch of k_analytic (one thread per ray).
// k_traverse is persistent: one lane = one ray; lanes that finish fetch the next ray from a global
// counter (warp-aggregated), so a warp stays full while rays of very different cost retire.
// The traversal stack lives in shared memory, one column per lane (no bank conflicts).
#pragma once
#include "device_common.cuh"

namespace yart {

#ifndef YART_TRACE_THREADS
#define YART_TRACE_THREADS 128
#endif
constexpr int kTraceThreads = YART_TRACE_THREADS;
constexpr uint32_t kSentinel = 0x7FFFFFFFu; // "no traversal in progress" (never a valid node id)


// ---------------------------------------------------------------------------------------------
// analytic primitives, t-only (the shade stage rebuilds the full HitRecord from t)
// ---------------------------------------------------------------------------------------------
// StillSphere::hit / MovingSphere::hit root selection (sphere.rs:48-66, 156-173)
YART_DEV bool sphere_t(D3 center, double radius, D3 ro, D3 rd, double t_min, double t_max, double& t) {
  D3 oc = ro - center;
  double a = length_squared(rd);
  double half_b = dot(oc, rd);
  double c = length_squared(oc) - radius * radius;
  double disc = half_b * half_b - a * c;
  if (disc < 0.0) return false;
  t = (0.0 - half_b - sqrt(disc)) / a;
  if (t < t_min || t_max < t) {
    t = (0.0 - half_b + sqrt(disc)) / a;
    if (t < t_min || t_max < t) return false;
  }
  return true;
}
YART_DEV D3 moving_center(const yart_object& o, double time) { // sphere.rs:149-152
  D3 c0 = d3(o.p[0], o.p[1], o.p[2]), c1 = d3(o.p[3], o.p[4], o.p[5]);
  return c0 + ((time - o.p[6]) / (o.p[7] - o.p[6])) * (c1 - c0);
}
// XYRect/XZRect/YZRect::hit (aarect.rs:41-57, 111-127, 206-222); kaxis = constant axis
YART_DEV bool rect_t(int kaxis, double a0, double a1, double b0, double b1, double k, D3 ro, D3 rd, double t_min,
                     double t_max, double& t) {
  const int aa = (kaxis == 0) ? 1 : 0;
  const int ba = (kaxis == 2) ? 1 : 2;
  t = (k - comp(ro, kaxis)) / comp(rd, kaxis);
  if (t < t_min || t > t_max) return false;
  double a = comp(ro, aa) + t * comp(rd, aa);
  double b = comp(ro, ba) + t * comp(rd, ba);
  if (a < a0 || a > a1 || b < b0 || b > b1) return false;
  return true;
}
YART_DEV int rect_axis(uint32_t kind) { return kind == YART_OBJ_XY_RECT ? 2 : (kind == YART_OBJ_XZ_RECT ? 1 : 0); }
// the six sides of BoxEntity::new in order (box_entity.rs:28-45)
YART_DEV void box_side(const double* p, int i, int& axis, double& a0, double& a1, double& b0, double& b1, double& k) {
  const double x0 = p[0], y0 = p[1], z0 = p[2], x1 = p[3], y1 = p[4], z1 = p[5];
  if (i < 2) { axis = 2; a0 = x0; a1 = x1; b0 = y0; b1 = y1; k = (i == 0) ? z0 : z1; }
  else if (i < 4) { axis = 1; a0 = x0; a1 = x1; b0 = z0; b1 = z1; k = (i == 2) ? y0 : y1; }
  else { axis = 0; a0 = y0; a1 = y1; b0 = z0; b1 = z1; k = (i == 4) ? x0 : x1; }
}
YART_DEV bool box_t(const double* p, D3 ro, D3 rd, double t_min, double t_max, double& t, uint32_t& side) {
  bool any = false; // BoxEntity::hit (box_entity.rs:51-70)
  double closest = t_max;
#pragma unroll 1
  for (int i = 0; i < 6; ++i) {
    int axis;
    double a0, a1, b0, b1, k, ti;
    box_side(p, i, axis, a0, a1, b0, b1, k);
    if (rect_t(axis, a0, a1, b0, b1, k, ro, rd, t_min, closest, ti)) {
      closest = ti;
      t = ti;
      side = (uint32_t)i;
      any = true;
    }
  }
  return any;
}
// Triangle::hit (triangle.rs:48-79)
YART_DEV bool triangle_t(const double* p, D3 ro, D3 rd, double t_min, double t_max, double& t, double& bu, double& bv) {
  D3 v0 = d3(p[0], p[1], p[2]), v1 = d3(p[3], p[4], p[5]), v2 = d3(p[6], p[7], p[8]);
  D3 e1 = v1 - v0, e2 = v2 - v0;
  D3 h = cross(rd, e2);
  double a = dot(e1, h);
  if (a > -kF64Eps && a < kF64Eps) return false;
  double f = 1.0 / a;
  D3 s = ro - v0;
  double u = f * dot(s, h);
  if (u < 0.0 || u > 1.0) return false;
  D3 q = cross(s, e1);
  double v = f * dot(rd, q);
  if (v < 0.0 || u + v > 1.0) return false;
  t = f * dot(e2, q);
  if (t < t_min || t > t_max) return false;
  bu = u;
  bv = v;
  return true;
}

// ray into the space of Translate(RotateY(.)) (hittable.rs:137-143, 218-227)
YART_DEV void instance_to_object(uint32_t wrap, const double* offset, double sin_theta, double cos_theta, D3& ro, D3& rd) {
  if (wrap & YART_WRAP_TRANSLATE) ro = ro - d3(offset[0], offset[1], offset[2]);
  if (wrap & YART_WRAP_ROTATE_Y) {
    const double ct = cos_theta, st = sin_theta;
    D3 org = ro, dir = rd;
    org.x = ct * ro.x - st * ro.z;
    org.z = st * ro.x + ct * ro.z;
    dir.x = ct * rd.x - st * rd.z;
    dir.z = st * rd.x + ct * rd.z;
    ro = org;
    rd = dir;
  }
}
YART_DEV void to_object_space(const yart_object& o, D3& ro, D3& rd) {
  instance_to_object(o.wrap, o.offset, o.sin_theta, o.cos_theta, ro, rd);
}

// one primitive record without wrappers; `prim` encodes what the shade stage needs
YART_DEV bool prim_hit_t(const yart_object& o, D3 ro, D3 rd, double time, double t_min, double t_max, double& t,
                         uint32_t& prim, double& bu, double& bv) {
  prim = 0;
  bu = bv = 0.0;
  switch (o.kind) {
    case YART_OBJ_SPHERE: return sphere_t(d3(o.p[0], o.p[1], o.p[2]), o.p[3], ro, rd, t_min, t_max, t);
    case YART_OBJ_MOVING_SPHERE: return sphere_t(moving_center(o, time), o.p[8], ro, rd, t_min, t_max, t);
    case YART_OBJ_XY_RECT:
    case YART_OBJ_XZ_RECT:
    case YART_OBJ_YZ_RECT: return rect_t(rect_axis(o.kind), o.p[0], o.p[1], o.p[2], o.p[3], o.p[4], ro, rd, t_min, t_max, t);
    case YART_OBJ_BOX: return box_t(o.p, ro, rd, t_min, t_max, t, prim);
    case YART_OBJ_TRIANGLE: return triangle_t(o.p, ro, rd, t_min, t_max, t, bu, bv);
    default: return false;
  }
}

// BVHNode group (bvh.rs:151-215): the closest member; prim = member*8 + box side
YART_DEV bool group_hit_t(const DevScene& S, const yart_object& o, D3 ro, D3 rd, double time, double t_min,
                          double t_max, double& t, uint32_t& prim) {
  const DevGroup g = S.groups[o.index];
  bool any = false;
  double closest = t_max;
  if (g.root == 0xFFFFFFFFu) {
    for (uint32_t i = 0; i < g.n_members; ++i) {
      double ti, bu, bv;
      uint32_t pr;
      if (prim_hit_t(g.members[i], ro, rd, time, t_min, closest, ti, pr, bu, bv)) {
        closest = ti; t = ti; prim = i * 8 + pr; any = true;
      }
    }
    return any;
  }
  // flat 4-wide tree over member boxes; visiting order does not change the closest member
  uint32_t stack[24];
  int sp = 0;
  stack[sp++] = g.root;
  const double ix = 1.0 / rd.x, iy = 1.0 / rd.y, iz = 1.0 / rd.z;
  // The boxes only cull, so the test may err on the side of visiting: a conservative f32 slab test (the
  // error bound of k_traverse's MIXED path: |t32 - t64| <= 2^-22 |t32| + A) that skips a child only when it is
  // PROVABLY missed needs no exact fallback.  Rays whose f32 image is unusable take the f64 test.
  const float ixf = (float)ix, iyf = (float)iy, izf = (float)iz;
  const float cxf = (float)(-(ro.x * ix)), cyf = (float)(-(ro.y * iy)), czf = (float)(-(ro.z * iz));
  const double am = fmax(fmax((g.bound[0] + fabs(ro.x)) * fabs(ix), (g.bound[1] + fabs(ro.y)) * fabs(iy)),
                         (g.bound[2] + fabs(ro.z)) * fabs(iz));
  const float amax2 = __double2float_ru(am * (1.0 / 4194304.0));
  const float lo_ok = 1e-30f, hi_ok = 1e30f;
  const bool f32_ok = fabsf(ixf) > lo_ok && fabsf(ixf) < hi_ok && fabsf(iyf) > lo_ok && fabsf(iyf) < hi_ok &&
                      fabsf(izf) > lo_ok && fabsf(izf) < hi_ok && fabsf(cxf) < hi_ok && fabsf(cyf) < hi_ok &&
                      fabsf(czf) < hi_ok && amax2 < hi_ok && isfinite(ro.x) && isfinite(ro.y) && isfinite(ro.z);
  const float t_min_f = (float)t_min;
  const bool px = rd.x >= 0.0, py = rd.y >= 0.0, pz = rd.z >= 0.0;
  while (sp > 0) {
    const uint32_t id = stack[--sp];
    if (id >> 31) {
      const uint32_t count = (id >> 27) & 0xF, first = id & 0x7FFFFFFu;
      YART_CHECK(first + count <= g.n_members);
      for (uint32_t i = first; i < first + count; ++i) {
        double ti, bu, bv;
        uint32_t pr;
        if (prim_hit_t(g.members[i], ro, rd, time, t_min, closest, ti, pr, bu, bv)) {
          // Equal-t ties between members (adjacent boxes share faces; spheres and rects accept t == t_max).
          // DOCUMENTED DEVIATION (DESIGN.md section 4 (iv)): the reference's BVHNode::hit (bvh.rs:176-213) lets the
          // child visited second win, and its visiting order depends on the ray and on a tree built with an
          // unstable sort -- not reproducible.  Here the member that comes LAST IN LIST ORDER wins, whatever
          // order this flat tree visits them in; only u, v / prim_id of such rays can differ from the reference.
          if (any && ti == closest && g.member_orig[i] < g.member_orig[prim >> 3]) continue;
          closest = ti; t = ti; prim = i * 8 + pr; any = true;
        }
      }
    } else {
      const float4* nd = g.nodes + (size_t)id * 8;
      const float4 mnx = __ldg(nd + 0), mny = __ldg(nd + 2), mnz = __ldg(nd + 4);
      const float4 mxx = __ldg(nd + 1), mxy = __ldg(nd + 3), mxz = __ldg(nd + 5);
      const uint4 ch = __ldg(reinterpret_cast<const uint4*>(nd + 6));
      const float lo[4][3] = {{mnx.x, mny.x, mnz.x}, {mnx.y, mny.y, mnz.y}, {mnx.z, mny.z, mnz.z}, {mnx.w, mny.w, mnz.w}};
      const float hi[4][3] = {{mxx.x, mxy.x, mxz.x}, {mxx.y, mxy.y, mxz.y}, {mxx.z, mxy.z, mxz.z}, {mxx.w, mxy.w, mxz.w}};
      const uint32_t cid[4] = {ch.x, ch.y, ch.z, ch.w};
      const float closest_f = (float)closest;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (cid[k] == 0xFFFFFFFFu) continue;
        bool visit;
        if (f32_ok) {
          const float tn = fmaxf(fmaxf(t_min_f, fmaf(px ? lo[k][0] : hi[k][0], ixf, cxf)),
                                 fmaxf(fmaf(py ? lo[k][1] : hi[k][1], iyf, cyf), fmaf(pz ? lo[k][2] : hi[k][2], izf, czf)));
          const float tf = fminf(fminf(closest_f, fmaf(px ? hi[k][0] : lo[k][0], ixf, cxf)),
                                 fminf(fmaf(py ? hi[k][1] : lo[k][1], iyf, cyf), fmaf(pz ? hi[k][2] : lo[k][2], izf, czf)));
          const float gap = tf - tn;
          const float e = fmaf(fabsf(tf) + fabsf(tn), 2.384185791015625e-7f, amax2);
          visit = !(gap < -e); // not provably missed (NaN compares false: visit)
        } else {
          // group boxes are padded outward by the builder, so a conservative >= test is safe
          double t0 = ((double)lo[k][0] - ro.x) * ix, t1 = ((double)hi[k][0] - ro.x) * ix;
          double tn = fmax(t_min, fmin(t0, t1)), tf = fmin(closest, fmax(t0, t1));
          t0 = ((double)lo[k][1] - ro.y) * iy; t1 = ((double)hi[k][1] - ro.y) * iy;
          tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));
          t0 = ((double)lo[k][2] - ro.z) * iz; t1 = ((double)hi[k][2] - ro.z) * iz;
          tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));
          visit = tf >= tn;
        }
        YART_CHECK(sp < 24 || !visit);
        if (visit && sp < 24) stack[sp++] = cid[k];
      }
    }
  }
  return any;
}

// Translate(RotateY(FlipFace(prim))) -- t only
YART_DEV bool inner_hit_t(const DevScene& S, const yart_object& o, D3 ro, D3 rd, double time, double t_min,
                          double t_max, double& t, uint32_t& prim, double& bu, double& bv) {
  to_object_space(o, ro, rd);
  if (o.kind == YART_OBJ_GROUP) {
    bu = bv = 0.0;
    return group_hit_t(S, o, ro, rd, time, t_min, t_max, t, prim);
  }
  return prim_hit_t(o, ro, rd, time, t_min, t_max, t, prim, bu, bv);
}

// one non-mesh world object incl. ConstantMedium::hit (hittable.rs:274-321)
YART_DEV bool object_hit_t(const DevScene& S, const yart_object& o, uint32_t obj_index, D3 ro, D3 rd, double time,
                           double t_min, double t_max, const Rng& rng, uint32_t bounce, double& t, uint32_t& prim,
                           double& bu, double& bv) {
  if (!(o.wrap & YART_WRAP_MEDIUM)) return inner_hit_t(S, o, ro, rd, time, t_min, t_max, t, prim, bu, bv);
  double t1, t2, b0, b1;
  uint32_t pr;
  if (!inner_hit_t(S, o, ro, rd, time, -d_inf(), d_inf(), t1, pr, b0, b1)) return false;
  if (!inner_hit_t(S, o, ro, rd, time, t1 + 0.0001, d_inf(), t2, pr, b0, b1)) return false;
  if (t1 < t_min) t1 = t_min;
  if (t2 > t_max) t2 = t_max;
  if (!(t1 < t2)) return false;
  if (t1 < 0.0) t1 = 0.0;
  const double ray_length = length(rd);
  const double distance_inside = (t2 - t1) * ray_length;
  double u0, u1;
  rng_draw(rng, bounce, YART_SLOT_MEDIUM + obj_index, u0, u1);
  const double hit_distance = o.neg_inv_density * log(u0);
  if (!(hit_distance < distance_inside)) return false;
  t = t1 + hit_distance / ray_length;
  prim = 0;
  bu = bv = 0.0;
  return true;
}

// ---------------------------------------------------------------------------------------------
// pass parameters
// ---------------------------------------------------------------------------------------------
struct PassCommon {
  const yart_ray* rays;        // indexed by ray id
  const yart_ray_f32* rays32;  // non-null: the rays are f32 records instead (yart_closest_hit_f32), `rays` is unused
  const uint32_t* queue;       // work item -> ray id, null = identity
  const uint32_t* n_items_dev; // number of work items in device memory, null = use n_items
  uint64_t n_items;
  DevHit* hits;                // indexed by ray id: the closest hit so far
  uint32_t first_pass;         // 1: nothing recorded yet, start from t_max and always write
  uint32_t n_rays;             // length of rays[] and hits[] (bounds-checked build)
  double t_min, t_max;
};

struct TraverseParams {
  PassCommon c;
  MeshPass m;
  uint32_t obj_index;         // world object index recorded with a hit
  unsigned long long* counters; // [0] node visits, [1] triangle tests, [2] exact-fallback nodes (COUNT only)
};

struct AnalyticParams {
  PassCommon c;
  DevScene scene;
  const yart_object* objects; // the world list
  uint32_t obj_begin, obj_end;
  const double* ray_time;     // indexed by ray id, may be null (time 0)
  uint64_t seed;              // Philox key for media inside world.hit
  uint32_t bounce;
  uint32_t spp_batch;         // ray id -> (pixel, sample) = (pixel_base + id / spp_batch, sample_base + id % spp_batch)
  uint32_t sample_base;
  uint32_t pixel_base;
  uint32_t media_mask;
  uint32_t _pad;
};

// The four slab tests of one node exactly as qbvh.rs:495-519 with IEEE minNum/maxNum folds -- the
// path for rays with a zero or non-finite component, whose slabs can be NaN (0 * inf).  Out of line:
// it is rare and its temporaries must not cost the common path registers.
template <bool NEAR>
__device__ __noinline__ uint32_t box4_ieee(const float4* nd, double ox, double oy, double oz, double ix, double iy,
                                           double iz, double t_min, double t_best) {
  const float4 mnx = __ldg(nd + 0), mny = __ldg(nd + 2), mnz = __ldg(nd + 4);
  const float4 mxx = __ldg(nd + 1), mxy = __ldg(nd + 3), mxz = __ldg(nd + 5);
  uint32_t hitmask = 0;
#define YART_BOX(K, LX, LY, LZ, HX, HY, HZ)                                        \
  {                                                                                \
    double t0 = ((double)(LX) - ox) * ix, t1 = ((double)(HX) - ox) * ix;           \
    double tn = fmax(t_min, fmin(t0, t1));                                         \
    double tf = fmin(NEAR ? d_inf() : t_best, fmax(t0, t1));                       \
    t0 = ((double)(LY) - oy) * iy; t1 = ((double)(HY) - oy) * iy;                  \
    tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));                      \
    t0 = ((double)(LZ) - oz) * iz; t1 = ((double)(HZ) - oz) * iz;                  \
    tn = fmax(tn, fmin(t0, t1)); tf = fmin(tf, fmax(t0, t1));                      \
    const bool h = NEAR ? ((tf > tn) && (t_best >= tn)) : (tf > tn);               \
    hitmask |= h ? (1u << (K)) : 0u;                                               \
  }
  YART_BOX(0, mnx.x, mny.x, mnz.x, mxx.x, mxy.x, mxz.x)
  YART_BOX(1, mnx.y, mny.y, mnz.y, mxx.y, mxy.y, mxz.y)
  YART_BOX(2, mnx.z, mny.z, mnz.z, mxx.z, mxy.z, mxz.z)
  YART_BOX(3, mnx.w, mny.w, mnz.w, mxx.w, mxy.w, mxz.w)
#undef YART_BOX
  return hitmask;
}

// ---------------------------------------------------------------------------------------------
// the steps of the QBVH walk (qbvh.rs:381-543) that k_traverse, k_traverse_lean and k_occlude share
// ---------------------------------------------------------------------------------------------
// Phase A's hand-out of work items to the lanes of a persistent warp.
// Work distribution: warp w starts with items [32w, 32w+32) without touching the counter and only then
// fetches dynamically from total_warps*32 + atomicAdd(counter).  Warps whose first slice is already past
// the end leave at once -- a nearly empty queue (the deep bounces) costs no same-address atomics.
// A short queue is spread thinly (rpw < 32 rays per warp): a warp's run time is the serialised work of
// its most divergent rays, so a deep bounce with a few hundred rays finishes sooner on many warps.
// Work items reach the lanes through a two-deep pipeline of 32-item chunks, so that neither the claim
// (an atomic), nor the queue read, nor the DRAM miss of the ray record sits on the warp's critical path:
//   chunk "cur": ids held one per lane (id_cur), handed to fetching lanes by shuffle;
//   chunk "nxt": claimed when cur was started (stage 1: atomic in flight), ids loaded one retire/fetch phase
//   later (stage 2), ray / hit records prefetched into L2 the phase after (stage 3).
// The first chunk of a warp is its static slice; all later ones come from the global counter.  Item counts are
// 32-bit: yart_closest_hit and yart_occluded cap n below 2^32, the renderer's queues hold at most 2^28 paths.
// `queue` maps items to ray ids (null = identity); `counter` is zero at launch.
struct ChunkQueue {
  uint32_t n_items, dyn_base;
  // the warp-uniform counters of the pipeline share ONE register (bit fields of a 32-bit word)
  struct {
    uint32_t cur_cnt : 6, cur_used : 6, nxt_cnt : 6, nxt_stage : 2, dyn_done : 1;
  } w;
  uint32_t id_cur, id_nxt, claim_raw;

  // false: the warp's static slice lies past the end of the queue, it has nothing to do
  YART_DEV bool start(uint32_t n, const uint32_t* queue, uint32_t* counter, uint32_t lane) {
    n_items = n;
    const uint32_t warp_global = (blockIdx.x * kTraceThreads + threadIdx.x) >> 5;
    const uint32_t total_warps = gridDim.x * (kTraceThreads / 32);
    const uint32_t rpw = max(1u, min(32u, (uint32_t)(((uint64_t)n_items + total_warps - 1) / total_warps)));
    dyn_base = total_warps * rpw; // (<= 2^17: at most a few thousand resident warps)
    if ((uint64_t)warp_global * rpw >= n_items) return false;
    const uint32_t cur_base = warp_global * rpw;
    w.cur_cnt = min(rpw, n_items - cur_base);
    w.cur_used = 0;
    id_cur = YART_MISS;
    id_nxt = YART_MISS;
    claim_raw = 0;
    if (lane < w.cur_cnt) id_cur = queue ? queue[cur_base + lane] : (uint32_t)(cur_base + lane);
    w.dyn_done = dyn_base >= n_items; // nothing beyond the static slices: never touch the counter
    w.nxt_cnt = 0;
    w.nxt_stage = 0;
    if (!w.dyn_done) {
      if (lane == 0) claim_raw = atomicAdd(counter, 32u);
      w.nxt_stage = 1;
    }
    return true;
  }

  // stage 1 -> 2: the claim has come back, read the chunk's ids
  YART_DEV void load_next(uint32_t lane, const uint32_t* queue) {
    const uint64_t nb = (uint64_t)dyn_base + __shfl_sync(0xffffffffu, claim_raw, 0);
    w.nxt_cnt = nb < n_items ? min(32u, n_items - (uint32_t)nb) : 0u;
    id_nxt = YART_MISS;
    if (lane < w.nxt_cnt) id_nxt = queue ? queue[nb + lane] : (uint32_t)(nb + lane);
    if (w.nxt_cnt < 32u) w.dyn_done = 1; // the counter has passed the end of the queue
    w.nxt_stage = 2;
  }

  // One retire/fetch phase (warp-uniform; all lanes take part in the shuffles): advance the pipeline by one stage
  // and hand an item to each fetching lane that can get one.  True with `id` for those lanes; `exhausted` is set for
  // a fetching lane that got nothing, which happens only once the queue is used up.  `second` is the other per-ray
  // record the kernel reads on fetch, prefetched with the ray (null = none).
  template <class Second>
  YART_DEV bool next(bool fetching, uint32_t lane, const uint32_t* queue, uint32_t* counter, const yart_ray* rays,
                     const yart_ray_f32* rays32, const Second* second, uint32_t n_rays, uint32_t& id, bool& exhausted) {
    if (w.nxt_stage == 2) {
      if (id_nxt != YART_MISS) {
        YART_CHECK(id_nxt < n_rays);
        if (rays32) {
          const char* rp = reinterpret_cast<const char*>(rays32 + id_nxt);
          prefetch_l2(rp);
          prefetch_l2(rp + 23); // a 24-byte record may straddle two 32-byte sectors
        } else {
          const char* rp = reinterpret_cast<const char*>(rays + id_nxt);
          prefetch_l2(rp);
          prefetch_l2(rp + 32); // a 48-byte record always spans two 32-byte sectors
        }
        if (second) prefetch_l2(second + id_nxt);
      }
      w.nxt_stage = 3;
    }
    const uint32_t fmask = __ballot_sync(0xffffffffu, fetching);
    const uint32_t need = (uint32_t)__popc(fmask);
    const uint32_t rank = (uint32_t)__popc(fmask & ((1u << lane) - 1u));
    const uint32_t take1 = min(need, (uint32_t)w.cur_cnt - (uint32_t)w.cur_used);
    uint32_t new_id = __shfl_sync(0xffffffffu, id_cur, ((uint32_t)w.cur_used + rank) & 31u);
    bool got = fetching && rank < take1;
    w.cur_used = w.cur_used + take1;
    if (need > take1) { // the current chunk ran out: the next one becomes current, and another is claimed
      if (w.nxt_stage == 1) load_next(lane, queue);
      if (w.nxt_stage >= 2) {
        id_cur = id_nxt;
        w.cur_cnt = w.nxt_cnt;
      } else {
        w.cur_cnt = 0;
      }
      w.cur_used = 0;
      w.nxt_stage = 0;
      w.nxt_cnt = 0;
      if (!w.dyn_done) {
        if (lane == 0) claim_raw = atomicAdd(counter, 32u);
        w.nxt_stage = 1;
      }
      const uint32_t rank2 = rank - take1; // (meaningful for the lanes that are still waiting)
      const uint32_t take2 = min(need - take1, (uint32_t)w.cur_cnt);
      const uint32_t id2 = __shfl_sync(0xffffffffu, id_cur, rank2 & 31u);
      if (fetching && !got && rank2 < take2) {
        new_id = id2;
        got = true;
      }
      w.cur_used = take2;
      if (fetching && !got) exhausted = true;
    } else if (w.nxt_stage == 1) { // no swap this time: use the phase to resolve the claim and load the ids
      load_next(lane, queue);
    }
    id = new_id;
    return got;
  }
};

// The ray in the mesh's space as the conservative f32 slab test below sees it.
struct SlabRay {
  float ixf, iyf, izf, cxf, cyf, czf; // per axis t = fma(b, inv, c)
  float amax2;                        // the absolute part of the error bound
  uint32_t pos; // bit a set: direction component a is >= 0 (qbvh.rs:388-392); bit 3: `weird`, exact tests throughout
  uint32_t sgn; // ORDER_TABLE sign bits, mirrored for near-first
};
YART_DEV SlabRay slab_ray(D3 o, D3 d, const double* bound, bool near) {
  SlabRay r;
  const double ix = 1.0 / d.x, iy = 1.0 / d.y, iz = 1.0 / d.z; // qbvh.rs:403-407
  r.pos = (d.x >= 0.0 ? 1u : 0u) | (d.y >= 0.0 ? 2u : 0u) | (d.z >= 0.0 ? 4u : 0u); // qbvh.rs:388-392
  r.sgn = near ? (r.pos ^ 7u) : r.pos;
  // (b - o) * (1/d) can only be NaN when 1/d is infinite or the ray itself is not finite
  if (!(isfinite(ix) && isfinite(iy) && isfinite(iz) && isfinite(o.x) && isfinite(o.y) && isfinite(o.z))) r.pos |= 8u;
  r.ixf = (float)ix; r.iyf = (float)iy; r.izf = (float)iz;
  r.cxf = (float)(-(o.x * ix)); r.cyf = (float)(-(o.y * iy)); r.czf = (float)(-(o.z * iz));
  // |t32 - t64| <= 2^-24 (|b| + |o|) |inv| + 2^-24 |t32| (+ f64 roundings); doubled for margin:
  // absolute part A = 2^-23 (B + |o|) |inv| maximised over the axes, kept as 2A (rounded up)
  const double a = fmax(fmax((bound[0] + fabs(o.x)) * fabs(ix), (bound[1] + fabs(o.y)) * fabs(iy)),
                        (bound[2] + fabs(o.z)) * fabs(iz));
  r.amax2 = __double2float_ru(a * (1.0 / 4194304.0)); // 2A = 2^-22 * a
  // rays whose f32 image is not well inside the normal range take the exact path throughout
  const float lo = 1e-30f, hi = 1e30f;
  const bool ok = fabsf(r.ixf) > lo && fabsf(r.ixf) < hi && fabsf(r.iyf) > lo && fabsf(r.iyf) < hi && fabsf(r.izf) > lo &&
                  fabsf(r.izf) < hi && fabsf(r.cxf) < hi && fabsf(r.cyf) < hi && fabsf(r.czf) < hi && r.amax2 < hi;
  if (!ok) r.pos |= 8u;
  return r;
}

// node `cur` of the pass's tree
YART_DEV const float4* node_at(const MeshPass& P, uint32_t cur) {
  YART_CHECK(cur < P.n_nodes);
  return P.nodes + (size_t)cur * 8;
}

// one 128-byte node (FlatNode) in four 256-bit loads, all in flight together
struct QNode {
  F8 x, y, z;     // per axis: the four children's lower planes, then their upper planes
  uint4 child;
  uint32_t axes;  // split axes of the top, left and right pair (2 bits each)
};
YART_DEV QNode load_node(const float4* nd) {
  QNode n;
  n.x = ldg256(nd + 0);
  n.y = ldg256(nd + 2);
  n.z = ldg256(nd + 4);
  const F8 cm8 = ldg256(nd + 6);
  n.child = make_uint4(__float_as_uint(cm8.lo.x), __float_as_uint(cm8.lo.y), __float_as_uint(cm8.lo.z), __float_as_uint(cm8.lo.w));
  n.axes = __float_as_uint(cm8.hi.x);
  return n;
}

// Which children of node `nd` the walk enters: the same hit mask as qbvh.rs:495-532.
// Conservative f32 test.  Per slab t32 = fma(b, inv32, c32); near32 / far32 are the max / min over
// the entry / exit planes with t_min / t_best folded in.  With R = 2^-22 and A as in slab_ray,
// |near32 - near64| <= R|near32| + A and the same for far, so
//   far32 - near32 >  R(|far32| + |near32|) + 2A  =>  far64 > near64   (the reference pushes)
//   far32 - near32 < -R(|far32| + |near32|) - 2A  =>  far64 < near64   (the reference does not)
// and everything in between (also any inf / NaN) is settled by the exact f64 test, which `weird` rays take for
// every box.  The f64 ray (o, d) is read from ray[0], ray[stride], .., ray[5 stride] only for that exact test.
// `undecided`: the children the exact test settled.
template <bool NEAR>
YART_DEV uint32_t node_hits(const float4* nd, const QNode& n, const SlabRay& r, float t_min_f, float t_best_f,
                            const double* ray, int stride, double t_min, double t_best, uint32_t& undecided) {
  undecided = 0;
  if (!(r.pos & 8u)) {
    const bool px = (r.pos & 1u) != 0, py = (r.pos & 2u) != 0, pz = (r.pos & 4u) != 0;
#define YART_SEL4(P_, A, B) make_float4((P_) ? A.x : B.x, (P_) ? A.y : B.y, (P_) ? A.z : B.z, (P_) ? A.w : B.w)
    const float4 nx = YART_SEL4(px, n.x.lo, n.x.hi), fx = YART_SEL4(px, n.x.hi, n.x.lo);
    const float4 ny = YART_SEL4(py, n.y.lo, n.y.hi), fy = YART_SEL4(py, n.y.hi, n.y.lo);
    const float4 nz = YART_SEL4(pz, n.z.lo, n.z.hi), fz = YART_SEL4(pz, n.z.hi, n.z.lo);
#undef YART_SEL4
    const float nxs[4] = {nx.x, nx.y, nx.z, nx.w}, nys[4] = {ny.x, ny.y, ny.z, ny.w}, nzs[4] = {nz.x, nz.y, nz.z, nz.w};
    const float fxs[4] = {fx.x, fx.y, fx.z, fx.w}, fys[4] = {fy.x, fy.y, fy.z, fy.w}, fzs[4] = {fz.x, fz.y, fz.z, fz.w};
    uint32_t hitmask = 0, amb = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float tn = fmaxf(fmaxf(t_min_f, fmaf(nxs[k], r.ixf, r.cxf)), fmaxf(fmaf(nys[k], r.iyf, r.cyf), fmaf(nzs[k], r.izf, r.czf)));
      const float tf = fminf(fminf(t_best_f, fmaf(fxs[k], r.ixf, r.cxf)), fminf(fmaf(fys[k], r.iyf, r.cyf), fmaf(fzs[k], r.izf, r.czf)));
      const float g = tf - tn;
      const float e = fmaf(fabsf(tf) + fabsf(tn), 2.384185791015625e-7f, r.amax2);
      hitmask |= (g > e) ? (1u << k) : 0u;
      amb |= ((g > e) || (g < -e)) ? 0u : (1u << k);
    }
    if (amb) {
      undecided = amb;
      const uint32_t exact = box4_ieee<NEAR>(nd, ray[0], ray[stride], ray[2 * stride], 1.0 / ray[3 * stride],
                                             1.0 / ray[4 * stride], 1.0 / ray[5 * stride], t_min, t_best);
      hitmask = (hitmask & ~amb) | (exact & amb);
    }
    return hitmask;
  }
  return box4_ieee<NEAR>(nd, ray[0], ray[stride], ray[2 * stride], 1.0 / ray[3 * stride], 1.0 / ray[4 * stride],
                         1.0 / ray[5 * stride], t_min, t_best);
}

// push_hit_children (qbvh.rs:18-31) in the order ORDER_TABLE[4*pos[top] + 2*pos[left] + pos[right]]
// (qbvh.rs:14-16, 521-524) gives; near-first walks pass mirrored sign bits, so the nearest child ends up on top.
// The table has structure: bit `top` says whether the left pair {0,1} is pushed before the right pair {2,3};
// `left` whether 0 goes before 1, `right` whether 2 goes before 3.  So every hit child's stack slot is a closed
// form of the hit bits -- four predicated stores, no table, no serial loop.  One stack column per lane.
template <int STACK>
YART_DEV void push_children(uint32_t (*s_stack)[kTraceThreads], int tid, int& sp, uint32_t hitmask, uint32_t sgn,
                            const QNode& n) {
  const uint32_t T = (sgn >> (n.axes & 3u)) & 1u, L = (sgn >> ((n.axes >> 2) & 3u)) & 1u,
                 Rr = (sgn >> ((n.axes >> 4) & 3u)) & 1u;
  const uint32_t h0 = hitmask & 1u, h1 = (hitmask >> 1) & 1u, h2 = (hitmask >> 2) & 1u, h3 = (hitmask >> 3) & 1u;
  const uint32_t nl = h0 + h1, nr = h2 + h3;
  const uint32_t bl = T ? 0u : nr, br = T ? nl : 0u; // slots taken by the pair pushed first
  if (h0) s_stack[sp + bl + (L ? 0u : h1)][tid] = n.child.x;
  if (h1) s_stack[sp + bl + (L ? h0 : 0u)][tid] = n.child.y;
  if (h2) s_stack[sp + br + (Rr ? 0u : h3)][tid] = n.child.z;
  if (h3) s_stack[sp + br + (Rr ? h2 : 0u)][tid] = n.child.w;
  sp += (int)(nl + nr);
  YART_CHECK(sp <= STACK + 1);
}
// the lane's next node or leaf, kSentinel once its stack is empty
YART_DEV uint32_t pop(uint32_t (*s_stack)[kTraceThreads], int tid, int& sp) {
  if (sp == 0) return kSentinel;
  sp--;
  return s_stack[sp][tid];
}

// one triangle as 9 floats: v0, v1, v2
struct Tri9 {
  float x0, y0, z0, x1, y1, z1, x2, y2, z2;
};
// Moeller-Trumbore exactly as qbvh.rs:419-489: true when the ray passes the edge tests and t >= t_min, with the
// hit's t and barycentrics u, v.  The test against t_max / the best hit so far is the caller's.
YART_DEV bool mt_hit(const Tri9& p, D3 o, D3 d, double t_min, double& t, double& u, double& v) {
  const double v0x = (double)p.x0, v0y = (double)p.y0, v0z = (double)p.z0;
  const double e1x = (double)p.x1 - v0x, e1y = (double)p.y1 - v0y, e1z = (double)p.z1 - v0z;
  const double e2x = (double)p.x2 - v0x, e2y = (double)p.y2 - v0y, e2z = (double)p.z2 - v0z;
  const double hx = d.y * e2z - d.z * e2y, hy = d.z * e2x - d.x * e2z, hz = d.x * e2y - d.y * e2x;
  const double a = e1x * hx + e1y * hy + e1z * hz;
  bool ok = !((a > -kF64Eps) && (a < kF64Eps));
  const double f = 1.0 / a;
  const double sx = o.x - v0x, sy = o.y - v0y, sz = o.z - v0z;
  u = f * (sx * hx + sy * hy + sz * hz);
  ok = ok && (u >= 0.0) && (u <= 1.0);
  const double qx = sy * e1z - sz * e1y, qy = sz * e1x - sx * e1z, qz = sx * e1y - sy * e1x;
  v = f * (d.x * qx + d.y * qy + d.z * qz);
  ok = ok && (v >= 0.0) && ((u + v) <= 1.0);
  t = f * (e2x * qx + e2y * qy + e2z * qz);
  return ok && (t >= t_min);
}

// One leaf (qbvh.rs:413-490): test(i, tri) for its triangles first + i, from the last one backwards when REVERSE;
// a test that returns true ends the leaf.  A leaf of up to three triangles is one packed block (36 B each, 32-byte
// aligned): 2 / 3 / 4 sector loads for 1 / 2 / 3 triangles instead of 3 loads per triangle, at most three sectors in
// registers at a time, the next one requested one test ahead.  4-triangle leaves are read one 48-byte record at a
// time, the next one requested before the current is tested.
template <bool REVERSE, class Test>
YART_DEV void visit_leaf(const float4* leafgeo, const float4* tris, uint32_t first, uint32_t count, Test&& test) {
  if (count <= 3u) {
    const float4* lp = leafgeo + (size_t)first * 4;
#define YART_TRI0 Tri9{s0.lo.x, s0.lo.y, s0.lo.z, s0.lo.w, s0.hi.x, s0.hi.y, s0.hi.z, s0.hi.w, s1.lo.x}
#define YART_TRI1 Tri9{s1.lo.y, s1.lo.z, s1.lo.w, s1.hi.x, s1.hi.y, s1.hi.z, s1.hi.w, s2.lo.x, s2.lo.y}
#define YART_TRI2 Tri9{s2.lo.z, s2.lo.w, s2.hi.x, s2.hi.y, s2.hi.z, s2.hi.w, s3.lo.x, s3.lo.y, s3.lo.z}
    if (REVERSE) { // from the last sector backwards
      F8 s1 = ldg256(lp + 2), s2, s3;
      s2.lo = s2.hi = s3.lo = s3.hi = make_float4(0.f, 0.f, 0.f, 0.f);
      if (count >= 2u) s2 = ldg256(lp + 4);
      if (count >= 3u) {
        s3 = ldg256(lp + 6);
        if (test(2u, YART_TRI2)) return;
      }
      const F8 s0 = ldg256(lp);
      if (count >= 2u && test(1u, YART_TRI1)) return;
      test(0u, YART_TRI0);
    } else {
      const F8 s0 = ldg256(lp), s1 = ldg256(lp + 2);
      F8 s2, s3;
      s2.lo = s2.hi = s3.lo = s3.hi = make_float4(0.f, 0.f, 0.f, 0.f);
      if (count >= 2u) s2 = ldg256(lp + 4);
      if (test(0u, YART_TRI0)) return;
      if (count >= 3u) s3 = ldg256(lp + 6);
      if (count >= 2u && test(1u, YART_TRI1)) return;
      if (count >= 3u) test(2u, YART_TRI2);
    }
#undef YART_TRI0
#undef YART_TRI1
#undef YART_TRI2
  } else {
    float4 n0, n1, n2;
    {
      const float4* tp = tris + (size_t)(first + (REVERSE ? (count - 1u) : 0u)) * 3;
      n0 = __ldg(tp); n1 = __ldg(tp + 1); n2 = __ldg(tp + 2);
    }
    for (uint32_t j = 0; j < count; ++j) {
      const uint32_t i = REVERSE ? (count - 1u - j) : j;
      const float4 a0 = n0, a1 = n1, a2 = n2;
      if (j + 1u < count) {
        const float4* tp = tris + (size_t)(first + (REVERSE ? (i - 1u) : (i + 1u))) * 3;
        n0 = __ldg(tp); n1 = __ldg(tp + 1); n2 = __ldg(tp + 2);
      }
      if (test(i, Tri9{a0.x, a0.y, a0.z, a1.x, a1.y, a1.z, a2.x, a2.y, a2.z})) return;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_traverse: one TriangleMesh instance against the whole ray queue
// ---------------------------------------------------------------------------------------------
#ifndef YART_TRAVERSE_MIN_BLOCKS
#define YART_TRAVERSE_MIN_BLOCKS 4
#endif

// The reference order, and visit counting in either order.  (Near-first without counting is k_traverse_lean,
// device_trace_lean.cu: the same walk with the f64 ray in shared memory.)  Here the f64 ray and the best hit's
// barycentrics stay in registers.
template <bool NEAR, bool COUNT, int STACK>
__global__ void __launch_bounds__(kTraceThreads, YART_TRAVERSE_MIN_BLOCKS) k_traverse(const TraverseParams P) {
  __shared__ uint32_t s_stack[STACK + 1][kTraceThreads];
  const int tid = threadIdx.x;
  const uint32_t lane = tid & 31;
  ChunkQueue q;
  if (!q.start(P.c.n_items_dev ? *P.c.n_items_dev : (uint32_t)P.c.n_items, P.c.queue, P.m.work_counter, lane)) return;
  const uint32_t RT = P.m.refill_threshold, NT = P.m.node_threshold;
  const double t_min = P.c.t_min;
  const float t_min_f = (float)t_min;

  // ---- lane state ----
  uint32_t ray_id = YART_MISS; // YART_MISS = idle
  uint32_t cur = kSentinel;    // current stack top (node or leaf id), kSentinel = not traversing
  int sp = 0;
  double ray[6] = {0, 0, 0, 0, 0, 0}; // the ray (o, d) in the mesh's space
  SlabRay r = {};
  double t_best = 0, best_bu = 0, best_bv = 0;
  float t_best_f = 0;
  uint32_t best_prim = YART_MISS; // YART_MISS = this mesh has not produced a hit
  bool exhausted = false;         // the global queue is empty
  unsigned long long n_nodes = 0, n_tris = 0, n_exact = 0;

  for (;;) {
    // =============== phase A: retire finished rays, fetch new ones ================================
    // Batched: lanes that finished wait until RT of them can run this together, unless nobody else has work.
    const bool want_a = (cur == kSentinel) && !(exhausted && ray_id == YART_MISS);
    const uint32_t a_mask = __ballot_sync(0xffffffffu, want_a);
    const uint32_t busy_mask = __ballot_sync(0xffffffffu, cur != kSentinel);
    if (a_mask != 0 && ((uint32_t)__popc(a_mask) >= RT || busy_mask == 0)) { // (warp-uniform)
      if (want_a && ray_id != YART_MISS) { // retire: record the hit if this mesh improved on the earlier objects
        if (best_prim != YART_MISS) {
          DevHit h;
          h.t = t_best; h.bu = best_bu; h.bv = best_bv; h.obj = P.obj_index; h.prim = best_prim;
          P.c.hits[ray_id] = h;
        } else if (P.c.first_pass) {
          DevHit h;
          h.t = d_inf(); h.bu = 0.0; h.bv = 0.0; h.obj = YART_MISS; h.prim = 0;
          P.c.hits[ray_id] = h;
        }
        ray_id = YART_MISS;
      }
      uint32_t id;
      if (q.next(want_a && !exhausted, lane, P.c.queue, P.m.work_counter, P.c.rays, P.c.rays32,
                 P.c.first_pass ? nullptr : P.c.hits, P.c.n_rays, id, exhausted)) {
        ray_id = id;
        YART_CHECK(ray_id < P.c.n_rays);
        D3 ro, rd;
        if (P.c.rays32) load_ray_f32(P.c.rays32 + ray_id, ro, rd);
        else load_ray(P.c.rays + ray_id, ro, rd);
        t_best = P.c.first_pass ? P.c.t_max : fmin(P.c.hits[ray_id].t, P.c.t_max);
        if (NEAR) t_best = just_below(t_best); // strict against earlier objects / the caller's t_max (device_common.cuh)
        instance_to_object(P.m.wrap, P.m.offset, P.m.sin_theta, P.m.cos_theta, ro, rd); // uniform across the launch
        ray[0] = ro.x; ray[1] = ro.y; ray[2] = ro.z;
        ray[3] = rd.x; ray[4] = rd.y; ray[5] = rd.z;
        r = slab_ray(ro, rd, P.m.bound, NEAR);
        t_best_f = (float)t_best;
        cur = P.m.root;
        sp = 0;
        best_prim = YART_MISS;
        best_bu = best_bv = 0.0;
      }
    }
    if (!__any_sync(0xffffffffu, ray_id != YART_MISS)) break;

    // =============== phase B: inner nodes (qbvh.rs:491-534) =====================================
    // Warp-uniform loop: keep stepping while at least NT lanes are on inner nodes; with fewer, yield to
    // the leaf / refill phases if they have something to do.
    for (;;) {
      const bool has_node = cur < 0x7FFFFFFFu; // bit31 clear and not the sentinel
      const uint32_t nm = __ballot_sync(0xffffffffu, has_node);
      if (nm == 0) break;
      if ((uint32_t)__popc(nm) < NT) {
        const uint32_t lm = __ballot_sync(0xffffffffu, cur >= 0x80000000u);
        const uint32_t wm = __ballot_sync(0xffffffffu, (cur == kSentinel) && !(exhausted && ray_id == YART_MISS));
        if (lm != 0 || (uint32_t)__popc(wm) >= RT) break;
      }
      if (has_node) {
        const float4* nd = node_at(P.m, cur);
        const QNode n = load_node(nd);
        if (COUNT) n_nodes++;
        uint32_t undecided;
        const uint32_t hitmask = node_hits<NEAR>(nd, n, r, t_min_f, t_best_f, ray, 1, t_min, t_best, undecided);
        if (COUNT && undecided) n_exact++;
        push_children<STACK>(s_stack, tid, sp, hitmask, r.sgn, n);
        cur = pop(s_stack, tid, sp);
      }
    }

    // =============== phase C: one leaf (qbvh.rs:413-490) ========================================
    if (cur >= 0x80000000u) {
      const uint32_t count = (cur >> 27) & 0xFu;
      const uint32_t first = cur & 0x7FFFFFFu;
      if (COUNT) n_tris += count;
      YART_CHECK(count >= 1 && count <= 4 && first + count <= P.m.n_tris);
      const D3 o = d3(ray[0], ray[1], ray[2]), d = d3(ray[3], ray[4], ray[5]);
      // NEAR tests the leaf's triangles in reverse order (the mirrored tie rule)
      visit_leaf<NEAR>(P.m.leafgeo, P.m.tris, first, count, [&](uint32_t i, const Tri9& tri) {
        double t, u, v;
        // REFERENCE: first found wins (`t_max > t`, qbvh.rs:478).  NEAR: mirrored -- last found wins among this
        // mesh's equal-t hits; strictness against earlier objects comes from the start value just_below(t_max).
        if (mt_hit(tri, o, d, t_min, t, u, v) && (NEAR ? (t <= t_best) : (t_best > t))) {
          t_best = t; best_prim = first + i; best_bu = u; best_bv = v;
          t_best_f = (float)t;
        }
        return false;
      });
      cur = pop(s_stack, tid, sp);
    }
  }
  if (COUNT) {
    atomicAdd(&P.counters[0], n_nodes);
    atomicAdd(&P.counters[1], n_tris);
    atomicAdd(&P.counters[2], n_exact);
  }
}

typedef void (*TraverseKernel)(const TraverseParams);
TraverseKernel lean_traverse_kernel(uint32_t max_stack); // device_trace_lean.cu

// ---------------------------------------------------------------------------------------------
// k_analytic: a run of consecutive non-mesh objects of the list, one thread per queued ray
// ---------------------------------------------------------------------------------------------
#ifndef YART_TRACE_NO_ANALYTIC_KERNEL // (the other translation unit that includes this header defines it)
__global__ void __launch_bounds__(256) k_analytic(const AnalyticParams P) {
  const uint64_t n = P.c.n_items_dev ? (uint64_t)*P.c.n_items_dev : P.c.n_items;
  for (uint64_t item = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; item < n; item += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t ray_id = P.c.queue ? P.c.queue[item] : (uint32_t)item;
    YART_CHECK(ray_id < P.c.n_rays);
    D3 wo, wd;
    if (P.c.rays32) load_ray_f32(P.c.rays32 + ray_id, wo, wd);
    else load_ray(P.c.rays + ray_id, wo, wd);
    DevHit h;
    if (P.c.first_pass) {
      h.t = d_inf(); h.bu = 0.0; h.bv = 0.0; h.obj = YART_MISS; h.prim = 0;
    } else {
      h = P.c.hits[ray_id];
    }
    double t_best = fmin(h.t, P.c.t_max);
    bool changed = P.c.first_pass != 0;
    Rng rng;
    if (P.media_mask) rng = make_rng(P.seed, P.pixel_base + ray_id / P.spp_batch, P.sample_base + ray_id % P.spp_batch);
    else rng = make_rng(0, 0, 0);
    const double time = P.ray_time ? P.ray_time[ray_id] : 0.0;
    for (uint32_t oi = P.obj_begin; oi < P.obj_end; ++oi) {
      const yart_object& o = P.objects[oi];
      double t, bu = 0.0, bv = 0.0;
      uint32_t prim = 0;
      bool hit;
      if (o.kind == YART_OBJ_SPHERE && o.wrap == 0)
        hit = sphere_t(d3(o.p[0], o.p[1], o.p[2]), o.p[3], wo, wd, P.c.t_min, t_best, t);
      else
        hit = object_hit_t(P.scene, o, oi, wo, wd, time, P.c.t_min, t_best, rng, P.bounce, t, prim, bu, bv);
      if (hit) {
        t_best = t; h.t = t; h.obj = oi; h.prim = prim; h.bu = bu; h.bv = bv;
        changed = true;
      }
    }
    if (changed) P.c.hits[ray_id] = h;
  }
}
#endif

} // namespace yart
