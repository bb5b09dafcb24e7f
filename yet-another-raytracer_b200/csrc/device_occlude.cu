// device_occlude.cu -- yart_occluded: "does ray i hit anything in (t_min, t_max)?" as an early-exit any-hit traversal.
//
// k_occlude is k_traverse_lean (device_trace_lean.cu) with the closest-hit state taken out: the same persistent grid,
// chunk pipeline, retire/fetch phase A, inner-node loop B and leaf phase C, the same conservative f32 slab test with
// the exact f64 fallback, the same packed leaf blocks.  What differs:
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
  const uint32_t n_items = P.c.n_rays;
  // Work distribution and the two-deep pipeline of 32-item chunks exactly as in k_traverse_lean: warp w starts with
  // its static slice, later chunks are claimed from the counter one phase ahead, their ray records prefetched into L2
  // the phase after.
  const uint32_t warp_global = (blockIdx.x * kTraceThreads + tid) >> 5;
  const uint32_t total_warps = gridDim.x * (kTraceThreads / 32);
  const uint32_t rpw = max(1u, min(32u, (uint32_t)(((uint64_t)n_items + total_warps - 1) / total_warps)));
  const uint32_t dyn_base = total_warps * rpw;
  if ((uint64_t)warp_global * rpw >= n_items) return;
  const uint32_t cur_base = warp_global * rpw;
  struct {
    uint32_t cur_cnt : 6, cur_used : 6, nxt_cnt : 6, nxt_stage : 2, dyn_done : 1;
  } w;
  w.cur_cnt = min(rpw, n_items - cur_base);
  w.cur_used = 0;
  uint32_t id_cur = YART_MISS, id_nxt = YART_MISS, claim_raw = 0;
  if (lane < w.cur_cnt) id_cur = cur_base + lane;
  w.dyn_done = dyn_base >= n_items;
  w.nxt_cnt = 0;
  w.nxt_stage = 0;
  if (!w.dyn_done) {
    if (lane == 0) claim_raw = atomicAdd(P.work_counter, 32u);
    w.nxt_stage = 1;
  }
  const uint32_t RT = P.refill_threshold, NT = P.node_threshold;
  const float4* __restrict__ nodes = P.nodes;
  const float4* __restrict__ tris = P.tris;
  const double t_min = P.c.t_min, t_best = P.c.t_max;
  const float t_min_f = (float)t_min, t_best_f = (float)t_best;

  // ---- lane state ----
  uint32_t ray_id = YART_MISS; // YART_MISS = idle
  uint32_t cur = kSentinel;    // current stack top (node or leaf id), kSentinel = not traversing
  int sp = 0;
  uint32_t sgn = 0;  // ORDER_TABLE sign bits, mirrored: nearest child on top of the stack
  uint32_t pos = 0;  // bit a set: direction component a is >= 0 (qbvh.rs:388-392); bit 3: `weird`
  bool exhausted = false;
  float ixf = 0, iyf = 0, izf = 0, cxf = 0, cyf = 0, czf = 0, amax2 = 0; // t = fma(b, ixf, cxf) per slab

  for (;;) {
    // =============== phase A: retire finished rays, fetch new ones ================================
    const bool want_a = (cur == kSentinel) && !(exhausted && ray_id == YART_MISS);
    const uint32_t a_mask = __ballot_sync(0xffffffffu, want_a);
    const uint32_t busy_mask = __ballot_sync(0xffffffffu, cur != kSentinel);
    if (a_mask != 0 && ((uint32_t)__popc(a_mask) >= RT || busy_mask == 0)) { // (warp-uniform)
      if (want_a) ray_id = YART_MISS; // (an occluded ray was marked when its hit was found)
      // ---- advance the chunk pipeline by one stage (warp-uniform) ----
      if (w.nxt_stage == 2) {
        if (id_nxt != YART_MISS) {
          YART_CHECK(id_nxt < P.c.n_rays);
          if (P.c.rays32) {
            const char* rp = reinterpret_cast<const char*>(P.c.rays32 + id_nxt);
            prefetch_l2(rp);
            prefetch_l2(rp + 23); // a 24-byte record may straddle two 32-byte sectors
          } else {
            const char* rp = reinterpret_cast<const char*>(P.c.rays + id_nxt);
            prefetch_l2(rp);
            prefetch_l2(rp + 32); // a 48-byte record always spans two 32-byte sectors
          }
          if (!P.c.first_pass) prefetch_l2(P.c.occluded + id_nxt);
        }
        w.nxt_stage = 3;
      }
      // ---- hand out items (all lanes take part in the shuffles) ----
      const bool fetching = want_a && !exhausted;
      const uint32_t fmask = __ballot_sync(0xffffffffu, fetching);
      const uint32_t need = (uint32_t)__popc(fmask);
      const uint32_t rank = (uint32_t)__popc(fmask & ((1u << lane) - 1u));
      const uint32_t take1 = min(need, (uint32_t)w.cur_cnt - (uint32_t)w.cur_used);
      uint32_t new_id = __shfl_sync(0xffffffffu, id_cur, ((uint32_t)w.cur_used + rank) & 31u);
      bool got = fetching && rank < take1;
      w.cur_used = w.cur_used + take1;
      if (need > take1) { // the current chunk ran out: the next one becomes current, and another is claimed
        if (w.nxt_stage == 1) {
          const uint64_t nb = (uint64_t)dyn_base + __shfl_sync(0xffffffffu, claim_raw, 0);
          w.nxt_cnt = nb < n_items ? min(32u, n_items - (uint32_t)nb) : 0u;
          id_nxt = YART_MISS;
          if (lane < w.nxt_cnt) id_nxt = (uint32_t)(nb + lane);
          if (w.nxt_cnt < 32u) w.dyn_done = 1;
          w.nxt_stage = 2;
        }
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
          if (lane == 0) claim_raw = atomicAdd(P.work_counter, 32u);
          w.nxt_stage = 1;
        }
        const uint32_t rank2 = rank - take1;
        const uint32_t take2 = min(need - take1, (uint32_t)w.cur_cnt);
        const uint32_t id2 = __shfl_sync(0xffffffffu, id_cur, rank2 & 31u);
        if (fetching && !got && rank2 < take2) {
          new_id = id2;
          got = true;
        }
        w.cur_used = take2;
        if (fetching && !got) exhausted = true;
      } else if (w.nxt_stage == 1) {
        const uint64_t nb = (uint64_t)dyn_base + __shfl_sync(0xffffffffu, claim_raw, 0);
        w.nxt_cnt = nb < n_items ? min(32u, n_items - (uint32_t)nb) : 0u;
        id_nxt = YART_MISS;
        if (lane < w.nxt_cnt) id_nxt = (uint32_t)(nb + lane);
        if (w.nxt_cnt < 32u) w.dyn_done = 1;
        w.nxt_stage = 2;
      }
      if (got) {
        ray_id = new_id;
        YART_CHECK(ray_id < P.c.n_rays);
        // a ray an earlier object of the world already occludes is retired at the next phase A without traversing
        if (P.c.first_pass || !P.c.occluded[ray_id]) {
          D3 ro, rd;
          if (P.c.rays32) load_ray_f32(P.c.rays32 + ray_id, ro, rd);
          else load_ray(P.c.rays + ray_id, ro, rd);
          // ray into the instance's space (hittable.rs:137-143, 218-227); uniform across the launch
          if (P.wrap & YART_WRAP_TRANSLATE) ro = ro - d3(P.offset[0], P.offset[1], P.offset[2]);
          if (P.wrap & YART_WRAP_ROTATE_Y) {
            const double ct = P.cos_theta, st = P.sin_theta;
            D3 org = ro, dir = rd;
            org.x = ct * ro.x - st * ro.z;
            org.z = st * ro.x + ct * ro.z;
            dir.x = ct * rd.x - st * rd.z;
            dir.z = st * rd.x + ct * rd.z;
            ro = org;
            rd = dir;
          }
          const double ox = ro.x, oy = ro.y, oz = ro.z, dx = rd.x, dy = rd.y, dz = rd.z;
          const double ix = 1.0 / dx, iy = 1.0 / dy, iz = 1.0 / dz; // qbvh.rs:403-407
          s_ray[0][tid] = ox; s_ray[1][tid] = oy; s_ray[2][tid] = oz;
          s_ray[3][tid] = dx; s_ray[4][tid] = dy; s_ray[5][tid] = dz;
          pos = (dx >= 0.0 ? 1u : 0u) | (dy >= 0.0 ? 2u : 0u) | (dz >= 0.0 ? 4u : 0u); // qbvh.rs:388-392
          sgn = pos ^ 7u;
          if (!(isfinite(ix) && isfinite(iy) && isfinite(iz) && isfinite(ox) && isfinite(oy) && isfinite(oz))) pos |= 8u;
          ixf = (float)ix; iyf = (float)iy; izf = (float)iz;
          cxf = (float)(-(ox * ix)); cyf = (float)(-(oy * iy)); czf = (float)(-(oz * iz));
          // the error bound of k_traverse's MIXED path: 2A = 2^-22 max_a (B_a + |o_a|) |inv_a|, rounded up
          const double a = fmax(fmax((P.bound[0] + fabs(ox)) * fabs(ix), (P.bound[1] + fabs(oy)) * fabs(iy)),
                                (P.bound[2] + fabs(oz)) * fabs(iz));
          amax2 = __double2float_ru(a * (1.0 / 4194304.0));
          const float lo = 1e-30f, hi = 1e30f;
          const bool ok = fabsf(ixf) > lo && fabsf(ixf) < hi && fabsf(iyf) > lo && fabsf(iyf) < hi && fabsf(izf) > lo &&
                          fabsf(izf) < hi && fabsf(cxf) < hi && fabsf(cyf) < hi && fabsf(czf) < hi && amax2 < hi;
          if (!ok) pos |= 8u;
          cur = P.root;
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
        YART_CHECK(cur < P.n_nodes);
        const float4* nd = nodes + (size_t)cur * 8;
        const F8 sx8 = ldg256(nd + 0), sy8 = ldg256(nd + 2), sz8 = ldg256(nd + 4), cm8 = ldg256(nd + 6);
        const uint4 ch = make_uint4(__float_as_uint(cm8.lo.x), __float_as_uint(cm8.lo.y), __float_as_uint(cm8.lo.z),
                                    __float_as_uint(cm8.lo.w));
        const uint32_t axes = __float_as_uint(cm8.hi.x);
        uint32_t hitmask = 0;
        if (!(pos & 8u)) {
          // Conservative f32 test (k_traverse): decides every box that is clearly hit or clearly missed by the
          // reference's test; the undecided ones (also any inf / NaN) go to the exact f64 test.
          const bool px = (pos & 1u) != 0, py = (pos & 2u) != 0, pz = (pos & 4u) != 0;
#define YART_SEL4(P_, A, B) make_float4((P_) ? A.x : B.x, (P_) ? A.y : B.y, (P_) ? A.z : B.z, (P_) ? A.w : B.w)
          const float4 nx = YART_SEL4(px, sx8.lo, sx8.hi), fx = YART_SEL4(px, sx8.hi, sx8.lo);
          const float4 ny = YART_SEL4(py, sy8.lo, sy8.hi), fy = YART_SEL4(py, sy8.hi, sy8.lo);
          const float4 nz = YART_SEL4(pz, sz8.lo, sz8.hi), fz = YART_SEL4(pz, sz8.hi, sz8.lo);
#undef YART_SEL4
          uint32_t amb = 0;
#define YART_BOX_F32(K, C)                                                                                        \
  {                                                                                                               \
    const float tn = fmaxf(fmaxf(t_min_f, fmaf(nx.C, ixf, cxf)), fmaxf(fmaf(ny.C, iyf, cyf), fmaf(nz.C, izf, czf))); \
    const float tf = fminf(fminf(t_best_f, fmaf(fx.C, ixf, cxf)), fminf(fmaf(fy.C, iyf, cyf), fmaf(fz.C, izf, czf))); \
    const float g = tf - tn;                                                                                      \
    const float e = fmaf(fabsf(tf) + fabsf(tn), 2.384185791015625e-7f, amax2);                                    \
    hitmask |= (g > e) ? (1u << (K)) : 0u;                                                                        \
    amb |= ((g > e) || (g < -e)) ? 0u : (1u << (K));                                                              \
  }
          YART_BOX_F32(0, x)
          YART_BOX_F32(1, y)
          YART_BOX_F32(2, z)
          YART_BOX_F32(3, w)
#undef YART_BOX_F32
          if (amb) {
            const uint32_t exact = box4_ieee<false>(nd, s_ray[0][tid], s_ray[1][tid], s_ray[2][tid], 1.0 / s_ray[3][tid],
                                                    1.0 / s_ray[4][tid], 1.0 / s_ray[5][tid], t_min, t_best);
            hitmask = (hitmask & ~amb) | (exact & amb);
          }
        } else {
          hitmask = box4_ieee<false>(nd, s_ray[0][tid], s_ray[1][tid], s_ray[2][tid], 1.0 / s_ray[3][tid], 1.0 / s_ray[4][tid],
                                     1.0 / s_ray[5][tid], t_min, t_best);
        }
        // push_hit_children (qbvh.rs:18-31) in the mirrored ORDER_TABLE order: the nearest child ends up on top
        {
          const uint32_t T = (sgn >> (axes & 3u)) & 1u, L = (sgn >> ((axes >> 2) & 3u)) & 1u,
                         Rr = (sgn >> ((axes >> 4) & 3u)) & 1u;
          const uint32_t h0 = hitmask & 1u, h1 = (hitmask >> 1) & 1u, h2 = (hitmask >> 2) & 1u, h3 = (hitmask >> 3) & 1u;
          const uint32_t nl = h0 + h1, nr = h2 + h3;
          const uint32_t bl = T ? 0u : nr, br = T ? nl : 0u;
          if (h0) s_stack[sp + bl + (L ? 0u : h1)][tid] = ch.x;
          if (h1) s_stack[sp + bl + (L ? h0 : 0u)][tid] = ch.y;
          if (h2) s_stack[sp + br + (Rr ? 0u : h3)][tid] = ch.z;
          if (h3) s_stack[sp + br + (Rr ? h2 : 0u)][tid] = ch.w;
          sp += (int)(nl + nr);
          YART_CHECK(sp <= STACK + 1);
        }
        if (sp == 0) {
          cur = kSentinel;
        } else {
          sp--;
          cur = s_stack[sp][tid];
        }
      }
    }

    // =============== phase C: one leaf (qbvh.rs:413-490) ========================================
    if (cur >= 0x80000000u) {
      const uint32_t count = (cur >> 27) & 0xFu;
      const uint32_t first = cur & 0x7FFFFFFu;
      YART_CHECK(count >= 1 && count <= 4 && first + count <= P.n_tris);
      const double ox = s_ray[0][tid], oy = s_ray[1][tid], oz = s_ray[2][tid];
      const double dx = s_ray[3][tid], dy = s_ray[4][tid], dz = s_ray[5][tid];
      bool hit = false;
      // Moeller-Trumbore exactly as qbvh.rs:419-489; accepted as the reference accepts against a fixed t_max
#define YART_TRI_TEST(F0, F1, F2, F3, F4, F5, F6, F7, F8)                                                           \
  {                                                                                                                 \
    const double v0x = (double)(F0), v0y = (double)(F1), v0z = (double)(F2);                                        \
    const double e1x = (double)(F3) - v0x, e1y = (double)(F4) - v0y, e1z = (double)(F5) - v0z;                      \
    const double e2x = (double)(F6) - v0x, e2y = (double)(F7) - v0y, e2z = (double)(F8) - v0z;                      \
    const double hx = dy * e2z - dz * e2y, hy = dz * e2x - dx * e2z, hz = dx * e2y - dy * e2x;                      \
    const double a = e1x * hx + e1y * hy + e1z * hz;                                                                \
    bool ok = !((a > -kF64Eps) && (a < kF64Eps));                                                                   \
    const double f = 1.0 / a;                                                                                       \
    const double sx = ox - v0x, sy = oy - v0y, sz = oz - v0z;                                                       \
    const double u = f * (sx * hx + sy * hy + sz * hz);                                                             \
    ok = ok && (u >= 0.0) && (u <= 1.0);                                                                            \
    const double qx = sy * e1z - sz * e1y, qy = sz * e1x - sx * e1z, qz = sx * e1y - sy * e1x;                      \
    const double v = f * (dx * qx + dy * qy + dz * qz);                                                             \
    ok = ok && (v >= 0.0) && ((u + v) <= 1.0);                                                                      \
    const double t = f * (e2x * qx + e2y * qy + e2z * qz);                                                          \
    ok = ok && (t >= t_min) && (t_best > t);                                                                        \
    hit = hit || ok;                                                                                                \
  }
      if (count <= 3u) {
        // the leaf's packed block (2 / 3 / 4 sectors for 1 / 2 / 3 triangles), tested from the last triangle backwards
        // like k_traverse_lean's near-first leaves: at most three sectors in registers at a time (the order within a
        // leaf does not change whether one of its triangles is accepted)
        const float4* lp = P.leafgeo + (size_t)first * 4;
        F8 s1 = ldg256(lp + 2), s2, s3;
        s2.lo = s2.hi = s3.lo = s3.hi = make_float4(0.f, 0.f, 0.f, 0.f);
        if (count >= 2u) s2 = ldg256(lp + 4);
        if (count >= 3u) {
          s3 = ldg256(lp + 6);
          YART_TRI_TEST(s2.lo.z, s2.lo.w, s2.hi.x, s2.hi.y, s2.hi.z, s2.hi.w, s3.lo.x, s3.lo.y, s3.lo.z)
        }
        if (!hit) {
          const F8 s0 = ldg256(lp);
          if (count >= 2u) YART_TRI_TEST(s1.lo.y, s1.lo.z, s1.lo.w, s1.hi.x, s1.hi.y, s1.hi.z, s1.hi.w, s2.lo.x, s2.lo.y)
          if (!hit) YART_TRI_TEST(s0.lo.x, s0.lo.y, s0.lo.z, s0.lo.w, s0.hi.x, s0.hi.y, s0.hi.z, s0.hi.w, s1.lo.x)
        }
      } else {
        // 4-triangle leaves: one 48-byte FlatTri record at a time, the next one requested before the current is tested
        const float4* tp = tris + (size_t)first * 3;
        float4 n0 = __ldg(tp), n1 = __ldg(tp + 1), n2 = __ldg(tp + 2);
        for (uint32_t j = 0; j < count && !hit; ++j) {
          const float4 a0 = n0, a1 = n1, a2 = n2;
          if (j + 1u < count) {
            tp += 3;
            n0 = __ldg(tp); n1 = __ldg(tp + 1); n2 = __ldg(tp + 2);
          }
          YART_TRI_TEST(a0.x, a0.y, a0.z, a1.x, a1.y, a1.z, a2.x, a2.y, a2.z)
        }
      }
#undef YART_TRI_TEST
      if (hit) { // the ray is occluded: nothing else of it is needed
        P.c.occluded[ray_id] = 1;
        sp = 0;
      }
      if (sp == 0) {
        cur = kSentinel;
      } else {
        sp--;
        cur = s_stack[sp][tid];
      }
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
