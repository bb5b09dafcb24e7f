// device_trace_lean.cu -- k_traverse_lean: the near-first closest-hit traversal of device_trace.cuh (same phases, same
// arithmetic, same results bit for bit) on a register diet, so that five instead of four 128-thread CTAs fit an SM (20 warps).
//
// k_traverse is bound by the latency of its node / leaf fetches at 16 warps per SM (DESIGN.md section 7); its 128
// registers are the price of keeping the f64 ray next to the f32 slab coefficients.  Here everything only the exact
// f64 code touches -- the ray (o, d) and the best hit's barycentrics -- lives in shared memory (one column per
// lane, conflict-free) and is loaded when a leaf test or a (rare) exact box test needs it.  Measured: +7 % on the
// render step, +6 % on the sweep; at 20 warps the L1 data pipe (82-94 % busy) is the limiter.  The reference order
// stays with k_traverse: this kernel spills there and was 5 % slower on the sweep (2,074 vs 2,188 Mrays/s).
#define YART_TRACE_NO_ANALYTIC_KERNEL
#include "device_trace.cuh"

namespace yart {

template <int STACK>
__global__ void __launch_bounds__(kTraceThreads, 5) k_traverse_lean(const TraverseParams P) {
  __shared__ uint32_t s_stack[STACK + 1][kTraceThreads];
  // what only the exact f64 code needs lives in shared memory, one column per lane: the ray in the mesh's space
  // (o, d) and the barycentrics of the best hit
  __shared__ double s_ray[6][kTraceThreads];
  __shared__ double s_buv[2][kTraceThreads];
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
  SlabRay r = {};
  double t_best = 0;
  float t_best_f = 0;
  uint32_t best_prim = YART_MISS; // YART_MISS = this mesh has not produced a hit
  bool exhausted = false;         // the global queue is empty

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
          h.t = t_best; h.bu = s_buv[0][tid]; h.bv = s_buv[1][tid]; h.obj = P.obj_index; h.prim = best_prim;
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
        t_best = just_below(t_best); // strict against earlier objects / the caller's t_max (device_common.cuh)
        instance_to_object(P.m.wrap, P.m.offset, P.m.sin_theta, P.m.cos_theta, ro, rd); // uniform across the launch
        s_ray[0][tid] = ro.x; s_ray[1][tid] = ro.y; s_ray[2][tid] = ro.z;
        s_ray[3][tid] = rd.x; s_ray[4][tid] = rd.y; s_ray[5][tid] = rd.z;
        r = slab_ray(ro, rd, P.m.bound, true);
        t_best_f = (float)t_best;
        cur = P.m.root;
        sp = 0;
        best_prim = YART_MISS;
        s_buv[0][tid] = 0.0;
        s_buv[1][tid] = 0.0;
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
        uint32_t undecided;
        const uint32_t hitmask = node_hits<true>(nd, n, r, t_min_f, t_best_f, &s_ray[0][tid], kTraceThreads, t_min, t_best, undecided);
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
      // triangles in reverse order: the last found wins among this mesh's equal-t hits (the mirrored tie rule), still
      // strictly closer than what earlier objects left
      visit_leaf<true>(P.m.leafgeo, P.m.tris, first, count, [&](uint32_t i, const Tri9& tri) {
        double t, u, v;
        if (mt_hit(tri, o, d, t_min, t, u, v) && t <= t_best) {
          t_best = t; best_prim = first + i; s_buv[0][tid] = u; s_buv[1][tid] = v;
          t_best_f = (float)t;
        }
        return false;
      });
      cur = pop(s_stack, tid, sp);
    }
  }
}

// The stack is sized to the tree: 24 entries cover 7 node levels (3 * height + 1 = 22: david, sycee), 32 cover 10,
// 64 the reference's own limit.
TraverseKernel lean_traverse_kernel(uint32_t max_stack) {
  if (max_stack <= 24) return k_traverse_lean<24>;
  if (max_stack <= 32) return k_traverse_lean<32>;
  return k_traverse_lean<64>;
}

} // namespace yart
