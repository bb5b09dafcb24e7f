// occlusion_ref.cpp -- the CPU reference the occlusion tests compare yart_occluded against (test infrastructure only).
//
// An independent restatement of "does the ray hit anything in (t_min, t_max)?": an early-exit QBVH walk with t_max
// held fixed for a mesh target, and for the world the first object in list order that hits.  It is built on the CPU
// oracle's own scene, tree and object code: this file compiles oracle/yart_oracle.cpp into its own translation unit
// (the oracle itself is not changed), and tests/test_occlusion_oracle.py checks that the answer equals the hit flag of
// the oracle's orc_closest_hit in the reference's order.  Only the occref_* entry points are exported, so the library
// can be loaded next to liboracle.so.
#include "../oracle/yart_oracle.cpp"

#define YART_OCC_EXPORT extern "C" __attribute__((visibility("default")))

YART_OCC_EXPORT int occref_scene_create(const yart_scene_desc* desc, orc_scene** out) { return orc_scene_create(desc, out); }
YART_OCC_EXPORT void occref_scene_free(orc_scene* s) { orc_scene_free(s); }
YART_OCC_EXPORT const char* occref_last_error(void) { return orc_last_error(); }


// Whether L4QBVH::hit (qbvh.rs:381-543) finds anything, restated as an early-exit walk: t_max stays fixed, the box test
// is the reference's (qbvh.rs:495-532) and the first triangle the reference's rule accepts (t >= t_min, t_max > t,
// qbvh.rs:470-490) ends it.  Children in the reference's order.
static bool qbvh_occluded(const Mesh& m, const Ray& ray, double t_min, double t_max) {
  if (m.nodes.empty()) return false;
  uint32_t stack[64];
  size_t cursor = 0;
  stack[0] = (uint32_t)m.nodes.size() - 1;
  const bool pos[3] = {ray.d.x >= 0.0, ray.d.y >= 0.0, ray.d.z >= 0.0};
  const double ro[3] = {ray.o.x, ray.o.y, ray.o.z};
  const double rd[3] = {ray.d.x, ray.d.y, ray.d.z};
  const double inv[3] = {1.0 / rd[0], 1.0 / rd[1], 1.0 / rd[2]};
  for (;;) {
    const uint32_t id = stack[cursor];
    if ((id >> 31) == 1) {
      const uint32_t count = (id >> 27) & 0xF, index = id & ((1u << 27) - 1);
      for (uint32_t i = 0; i < count; ++i) { // the arithmetic of one f64x4 lane of qbvh.rs:420-450
        const Tri& tr = m.tris[index + i];
        const double v0[3] = {tr.v[0].x, tr.v[0].y, tr.v[0].z};
        const double e1[3] = {tr.v[1].x - tr.v[0].x, tr.v[1].y - tr.v[0].y, tr.v[1].z - tr.v[0].z};
        const double e2[3] = {tr.v[2].x - tr.v[0].x, tr.v[2].y - tr.v[0].y, tr.v[2].z - tr.v[0].z};
        const double h[3] = {rd[1] * e2[2] - rd[2] * e2[1], rd[2] * e2[0] - rd[0] * e2[2], rd[0] * e2[1] - rd[1] * e2[0]};
        const double a = e1[0] * h[0] + e1[1] * h[1] + e1[2] * h[2];
        if ((a > -kEps) && (a < kEps)) continue;
        const double f = 1.0 / a;
        const double sv[3] = {ro[0] - v0[0], ro[1] - v0[1], ro[2] - v0[2]};
        const double u = f * (sv[0] * h[0] + sv[1] * h[1] + sv[2] * h[2]);
        if (!((u >= 0.0) && (u <= 1.0))) continue;
        const double q[3] = {sv[1] * e1[2] - sv[2] * e1[1], sv[2] * e1[0] - sv[0] * e1[2], sv[0] * e1[1] - sv[1] * e1[0]};
        const double v = f * (rd[0] * q[0] + rd[1] * q[1] + rd[2] * q[2]);
        if (!((v >= 0.0) && ((u + v) <= 1.0))) continue;
        const double t = f * (e2[0] * q[0] + e2[1] * q[1] + e2[2] * q[2]);
        if ((t >= t_min) && (t_max > t)) return true;
      }
    } else {
      const Node& nd = m.nodes[id];
      bool hits[4];
      for (int k = 0; k < 4; ++k) {
        double tn = t_min, tf = t_max;
        for (int a = 0; a < 3; ++a) {
          const double t0 = (nd.bmin[a][k] - ro[a]) * inv[a];
          const double t1 = (nd.bmax[a][k] - ro[a]) * inv[a];
          tn = std::fmax(tn, std::fmin(t0, t1));
          tf = std::fmin(tf, std::fmax(t0, t1));
        }
        hits[k] = tf > tn;
      }
      const uint32_t enc = ORDER_TABLE[4 * (int)pos[nd.axis[0]] + 2 * (int)pos[nd.axis[1]] + (int)pos[nd.axis[2]]];
      for (int j = 0; j < 4; ++j) {
        const uint32_t i = (enc >> (4 * j)) & 0xF;
        if (hits[i]) stack[cursor++] = nd.child[i];
      }
    }
    if (cursor == 0) return false;
    cursor--;
  }
}

YART_OCC_EXPORT int occref_occluded(const orc_scene* s, uint32_t target, const yart_ray* rays, uint64_t n, double t_min, double t_max,
                 uint8_t* out, int n_threads) {
  if (!s || (!rays && n) || (!out && n)) { g_err = "null argument"; return YART_ERR_INVALID; }
  if (target != YART_TARGET_WORLD && target >= s->s.meshes.size()) { g_err = "bad target"; return YART_ERR_INVALID; }
  if (n_threads < 1) n_threads = 1;
  auto work = [&](int tid) {
    HitCtx c{&s->s, YART_ORDER_REFERENCE, nullptr};
    uint64_t lo = n * (uint64_t)tid / (uint64_t)n_threads, hi = n * (uint64_t)(tid + 1) / (uint64_t)n_threads;
    for (uint64_t i = lo; i < hi; ++i) {
      Ray r{v3(rays[i].origin[0], rays[i].origin[1], rays[i].origin[2]),
            v3(rays[i].direction[0], rays[i].direction[1], rays[i].direction[2]), 0.0, 550.0};
      bool hit = false;
      if (target == YART_TARGET_WORLD) { // HittableList::hit: the first object that hits sees the full t_max
        Rng rng = make_rng(0, (uint32_t)i, 0);
        HitRec rec;
        for (size_t k = 0; k < s->s.objects.size() && !hit; ++k)
          hit = hit_object(c, s->s.objects[k], (uint32_t)k, r, t_min, t_max, &rng, 1, rec);
      } else {
        hit = qbvh_occluded(s->s.meshes[target], r, t_min, t_max);
      }
      out[i] = hit ? 1 : 0;
    }
  };
  if (n_threads == 1) {
    work(0);
  } else {
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
  }
  return YART_OK;
}
