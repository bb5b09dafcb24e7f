// device_occlude.cu -- yart_occluded: "does ray i hit anything in (t_min, t_max)?" as an early-exit any-hit traversal.
//
// k_occlude is k_traverse_lean (device_trace_lean.cu) with the closest-hit state taken out: the same persistent grid,
// retire/fetch phase A, inner-node loop B and leaf phase C, built from the same steps of device_trace.cuh (chunk
// queue, conservative f32 slab test with the exact f64 fallback, packed leaf blocks).  What differs:
//   * t_best is the fixed t_max of the pass: no barycentrics, no best primitive, no shrinking interval;
//   * the first accepted triangle ends the ray: the lane writes occluded[ray] = 1, drops its stack and fetches anew;
//   * boxes and triangles are tested by the REFERENCE's rules (tfar > tnear with tfar <= t_max, qbvh.rs:532;
//     t >= t_min && t_max > t, qbvh.rs:478), while children are pushed nearest-first so that a hit comes early.
// Why the answer is then exactly yart_closest_hit(..., YART_ORDER_REFERENCE, ...)'s hit flag: the box test
// min(t_max, far) > max(t_min, near) is monotone in t_max, so the leaves a closest-hit traversal reaches while its
// t_best shrinks are a subset of those reachable with t_best = t_max; with no hit it never shrinks and visits all of
// them, in whatever order.  So "some reachable triangle is accepted against t_max" holds for any child order, and it
// holds iff closest-hit reports a hit.  The near-first tests of the lean kernel (just_below, t_best >= tnear) are a
// different test and are not used here.
#define YART_TRACE_NO_ANALYTIC_KERNEL
#include "device_trace.cuh"
#include "device_occlude.h"

namespace yart {

// Five 128-thread CTAs per SM (96 registers, no spills).  The 80-register build for six spills 70 B and measured
// 3-7 % slower on the david sweeps (DESIGN.md section 6).
template <int STACK>
__global__ void __launch_bounds__(kTraceThreads, 5) k_occlude(const OccludeParams P) {
  __shared__ uint32_t s_stack[STACK + 1][kTraceThreads];
  // the ray in the mesh's space (o, d), one column per lane: only the exact f64 code reads it
  __shared__ double s_ray[6][kTraceThreads];
  const int tid = threadIdx.x;
  const uint32_t lane = tid & 31;
  ChunkQueue q;
  if (!q.start(P.c.n_rays, nullptr, P.m.work_counter, lane)) return;
  const uint32_t RT = P.m.refill_threshold, NT = P.m.node_threshold;
  const double t_min = P.c.t_min, t_best = P.c.t_max;
  const float t_min_f = (float)t_min, t_best_f = (float)t_best;

  // ---- lane state ----
  uint32_t ray_id = YART_MISS; // YART_MISS = idle
  uint32_t cur = kSentinel;    // current stack top (node or leaf id), kSentinel = not traversing
  int sp = 0;
  SlabRay r = {};              // (sign bits mirrored: nearest child on top of the stack)
  bool exhausted = false;

  for (;;) {
    // =============== phase A: retire finished rays, fetch new ones ================================
    const bool want_a = (cur == kSentinel) && !(exhausted && ray_id == YART_MISS);
    const uint32_t a_mask = __ballot_sync(0xffffffffu, want_a);
    const uint32_t busy_mask = __ballot_sync(0xffffffffu, cur != kSentinel);
    if (a_mask != 0 && ((uint32_t)__popc(a_mask) >= RT || busy_mask == 0)) { // (warp-uniform)
      if (want_a) ray_id = YART_MISS; // (an occluded ray was marked when its hit was found)
      uint32_t id;
      if (q.next(want_a && !exhausted, lane, nullptr, P.m.work_counter, P.c.rays, P.c.rays32,
                 P.c.first_pass ? nullptr : P.c.occluded, P.c.n_rays, id, exhausted)) {
        ray_id = id;
        YART_CHECK(ray_id < P.c.n_rays);
        // a ray an earlier object of the world already occludes is retired at the next phase A without traversing
        if (P.c.first_pass || !P.c.occluded[ray_id]) {
          D3 ro, rd;
          if (P.c.rays32) load_ray_f32(P.c.rays32 + ray_id, ro, rd);
          else load_ray(P.c.rays + ray_id, ro, rd);
          instance_to_object(P.m.wrap, P.m.offset, P.m.sin_theta, P.m.cos_theta, ro, rd); // uniform across the launch
          s_ray[0][tid] = ro.x; s_ray[1][tid] = ro.y; s_ray[2][tid] = ro.z;
          s_ray[3][tid] = rd.x; s_ray[4][tid] = rd.y; s_ray[5][tid] = rd.z;
          r = slab_ray(ro, rd, P.m.bound, true);
          cur = P.m.root;
          sp = 0;
        }
      }
    }
    if (!__any_sync(0xffffffffu, ray_id != YART_MISS)) break;

    // =============== phase B: inner nodes (qbvh.rs:491-534) =====================================
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
        uint32_t undecided;
        // the reference's box test against the fixed t_max; children pushed nearest-first
        const uint32_t hitmask = node_hits<false>(nd, n, r, t_min_f, t_best_f, &s_ray[0][tid], kTraceThreads, t_min, t_best, undecided);
        push_children<STACK>(s_stack, tid, sp, hitmask, r.sgn, n);
        cur = pop(s_stack, tid, sp);
      }
    }

    // =============== phase C: one leaf (qbvh.rs:413-490) ========================================
    if (cur >= 0x80000000u) {
      const uint32_t count = (cur >> 27) & 0xFu;
      const uint32_t first = cur & 0x7FFFFFFu;
      YART_CHECK(count >= 1 && count <= 4 && first + count <= P.m.n_tris);
      const D3 o = d3(s_ray[0][tid], s_ray[1][tid], s_ray[2][tid]), d = d3(s_ray[3][tid], s_ray[4][tid], s_ray[5][tid]);
      // accepted as the reference accepts against a fixed t_max; the first accepted triangle ends the leaf (the order
      // within a leaf does not change whether one of its triangles is accepted)
      bool hit = false;
      visit_leaf<true>(P.m.leafgeo, P.m.tris, first, count, [&](uint32_t, const Tri9& tri) {
        double t, u, v;
        hit = mt_hit(tri, o, d, t_min, t, u, v) && t_best > t;
        return hit;
      });
      if (hit) { // the ray is occluded: nothing else of it is needed
        P.c.occluded[ray_id] = 1;
        sp = 0;
      }
      cur = pop(s_stack, tid, sp);
    }
  }
}

// A run of consecutive analytic (or media-wrapped) objects, one thread per ray: HittableList::hit (hittable.rs:66-79)
// reports a hit iff some object hits in (t_min, t_max), and the first object in list order that hits is called with
// the full t_max -- nothing before it hit -- so the OR over the objects, stopped at the first hit, is exactly the
// closest-hit query's answer.  Media draw from per-object Philox slots: the draw does not depend on what ran before.
__global__ void __launch_bounds__(256) k_analytic_occluded(const AnalyticOccludedParams P) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < P.c.n_rays; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t ray_id = (uint32_t)i;
    if (!P.c.first_pass && P.c.occluded[ray_id]) continue;
    D3 wo, wd;
    if (P.c.rays32) load_ray_f32(P.c.rays32 + ray_id, wo, wd);
    else load_ray(P.c.rays + ray_id, wo, wd);
    const Rng rng = P.media ? make_rng(0, P.pixel_base + ray_id, 0) : make_rng(0, 0, 0);
    for (uint32_t oi = P.obj_begin; oi < P.obj_end; ++oi) {
      const yart_object& o = P.objects[oi];
      double t, bu, bv;
      uint32_t prim;
      bool hit;
      if (o.kind == YART_OBJ_SPHERE && o.wrap == 0)
        hit = sphere_t(d3(o.p[0], o.p[1], o.p[2]), o.p[3], wo, wd, P.c.t_min, P.c.t_max, t);
      else
        hit = object_hit_t(P.scene, o, oi, wo, wd, 0.0, P.c.t_min, P.c.t_max, rng, 1u, t, prim, bu, bv);
      if (hit) {
        P.c.occluded[ray_id] = 1;
        break;
      }
    }
  }
}

// The stack is sized to the tree like k_traverse_lean's: 24 entries cover 7 node levels, 32 cover 10, 64 the
// reference's own limit.
OccludeKernel occlude_kernel(uint32_t max_stack) {
  if (max_stack <= 24) return k_occlude<24>;
  if (max_stack <= 32) return k_occlude<32>;
  return k_occlude<64>;
}
AnalyticOccludedKernel analytic_occluded_kernel() { return k_analytic_occluded; }

} // namespace yart
