// record_ref.cpp -- the CPU reference the hit-record tests compare yart_closest_hit_records against (test infrastructure
// only).
//
// The whole HitRecord (hittable.rs:37-45) the CPU oracle's world.hit builds, for rays that carry their own Ray.time.
// This file compiles oracle/yart_oracle.cpp into its own translation unit (the oracle itself is not changed) and only
// writes out what the oracle computes: world_hit for the whole world, qbvh_hit + mesh_hit_record for a mesh target.
// tests/test_record_oracle.py checks that its t / ids / front_face equal orc_closest_hit's.  Only the recref_* entry
// points are exported, so the library can be loaded next to liboracle.so.
#include "../oracle/yart_oracle.cpp"

#define YART_REC_EXPORT extern "C" __attribute__((visibility("default")))

YART_REC_EXPORT int recref_scene_create(const yart_scene_desc* desc, orc_scene** out) { return orc_scene_create(desc, out); }
YART_REC_EXPORT void recref_scene_free(orc_scene* s) { orc_scene_free(s); }
YART_REC_EXPORT const char* recref_last_error(void) { return orc_last_error(); }

static void fill_record(yart_hit_record& o, bool some, const HitRec& rec, bool mesh_target) {
  if (!some) {
    o.t = kInf;
    for (int k = 0; k < 3; ++k) o.p[k] = o.normal[k] = 0.0;
    o.u = o.v = 0.0;
    o.material = YART_MISS; o.front_face = 0; o.obj_id = YART_MISS; o.prim_id = YART_MISS;
    return;
  }
  o.t = rec.t;
  o.p[0] = rec.p.x; o.p[1] = rec.p.y; o.p[2] = rec.p.z;
  o.normal[0] = rec.normal.x; o.normal[1] = rec.normal.y; o.normal[2] = rec.normal.z;
  o.u = rec.u; o.v = rec.v;
  o.material = mesh_target ? YART_MISS : rec.material;
  o.front_face = rec.front_face ? 1u : 0u;
  o.obj_id = rec.obj;
  o.prim_id = rec.prim;
}

// ray i is Ray{o, d, times ? times[i] : 0, 550}; constant media draw from make_rng(0, i, 0) at bounce 1, as
// orc_closest_hit does
YART_REC_EXPORT int recref_records(const orc_scene* s, uint32_t target, const yart_ray* rays, const double* times, uint64_t n,
                                   double t_min, double t_max, uint32_t order, yart_hit_record* out, int n_threads) {
  if (!s || (!rays && n) || (!out && n)) { g_err = "null argument"; return YART_ERR_INVALID; }
  if (target != YART_TARGET_WORLD && target >= s->s.meshes.size()) { g_err = "bad target"; return YART_ERR_INVALID; }
  if (order > YART_ORDER_NEAR) { g_err = "bad order"; return YART_ERR_INVALID; }
  if (n_threads < 1) n_threads = 1;
  auto work = [&](int tid) {
    HitCtx c{&s->s, order, nullptr};
    uint64_t lo = n * (uint64_t)tid / (uint64_t)n_threads, hi = n * (uint64_t)(tid + 1) / (uint64_t)n_threads;
    for (uint64_t i = lo; i < hi; ++i) {
      Ray r{v3(rays[i].origin[0], rays[i].origin[1], rays[i].origin[2]),
            v3(rays[i].direction[0], rays[i].direction[1], rays[i].direction[2]), times ? times[i] : 0.0, 550.0};
      HitRec rec;
      bool some;
      if (target == YART_TARGET_WORLD) {
        Rng rng = make_rng(0, (uint32_t)i, 0);
        some = world_hit(c, r, t_min, t_max, &rng, 1, rec);
      } else {
        const Mesh& m = s->s.meshes[target];
        MeshHit mh = (order == YART_ORDER_NEAR) ? qbvh_hit<true>(m, r, t_min, t_max, nullptr)
                                                : qbvh_hit<false>(m, r, t_min, t_max, nullptr);
        some = mh.some;
        if (some) { mesh_hit_record(m, mh, r, 0, rec); rec.obj = 0; }
      }
      fill_record(out[i], some, rec, target != YART_TARGET_WORLD);
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
