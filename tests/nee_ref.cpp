// nee_ref.cpp -- the CPU reference of YART_FLAG_NEXT_EVENT (next-event estimation with MIS) that the renderer is
// compared against (test infrastructure only).
//
// It is built on the CPU oracle's own scene, object, material and camera code: this file compiles
// oracle/yart_oracle.cpp into its own translation unit (the oracle itself is not changed) and adds the estimator as a
// second integrator next to the oracle's ray_reflectance.  tests/test_next_event.py checks it against the oracle where
// the two must agree (no lights, max_depth 1, the same path rays, the same expectation).  Only the neeref_* entry
// points are exported, so the library can be loaded next to liboracle.so.
#include "../oracle/yart_oracle.cpp"

#define YART_NEE_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

// One light sample at a Lambertian hit, relative to the throughput carried into the bounce: a uniform light pick, the
// light's own random() direction, and a closest-hit shadow ray (world.hit at t_min 0.001, like main.rs:548, drawing its
// media at bounce YART_NEE_BOUNCE_BASE + bounce).  A front-facing DiffuseLight it hits contributes
// atten * scatter_pdf / p_l * Le with the power-heuristic weight p_l^2 / (p_l^2 + p_mix^2).
double next_event_sample(const HitCtx& c, const Ray& ray, const Rng& rng, uint32_t bounce, const HitRec& rec,
                         const Onb& uvw, double atten) {
  const Scene& s = *c.s;
  double u_pick, unused, s1, s2;
  rng.draw(bounce, YART_SLOT_NEE_PICK, u_pick, unused);
  rng.draw(bounce, YART_SLOT_NEE_DIR, s1, s2);
  const size_t n = s.lights.size();
  size_t k = (size_t)(u_pick * (double)n);
  if (k > n - 1) k = n - 1;
  const V3 dl = light_random(s.lights[k], rec.p, s1, s2);
  const double p_l = lights_pdf_value(s, rec.p, dl);
  const double cosv = dot(unit_vector(dl), uvw.w);
  const double cos_pdf = cosv <= 0.0 ? 0.0 : cosv / kPi;
  const double p_m = 0.5 * p_l + 0.5 * cos_pdf;
  const double cs = dot(rec.normal, unit_vector(dl));
  const double spdf = cs < 0.0 ? 0.0 : cs / kPi;
  if (!std::isfinite(p_l) || !(p_l > 0.0) || !(spdf > 0.0)) return 0.0;
  const Ray sr{rec.p, dl, ray.time, ray.wl};
  HitRec srec;
  if (!world_hit(c, sr, 0.001, kInf, &rng, YART_NEE_BOUNCE_BASE + bounce, srec)) return 0.0;
  const yart_material& sm = s.materials[srec.material];
  if (sm.kind != YART_MAT_DIFFUSE_LIGHT || !srec.front_face) return 0.0;
  const double w = p_l * p_l / (p_l * p_l + p_m * p_m);
  return atten * spdf / p_l * w * texture_value(s, sm.texture, sr, srec);
}

// The oracle's ray_reflectance (main.rs:537-588) with next-event estimation: the same loop, draws and factors, plus
// per Lambertian bounce b a light sample nee_b folded in as L_b = nee_b + f_b * L_{b+1}, and emission reached from a
// Lambertian bounce weighted by pdf^2 / (pdf^2 + p_light^2).  The light pick is always the unbiased one.
double ray_reflectance_nee(const HitCtx& c, Ray ray, const Rng& rng, uint32_t max_depth, uint32_t* n_rays, uint32_t flags) {
  struct F {
    double atten, spdf, pdf, nee;
    int kind; // 0 plain factor, 1 Lambertian, 2 roulette (atten = q)
  };
  const Scene& s = *c.s;
  std::vector<F> factors;
  double terminal = (flags & YART_FLAG_DEPTH_ZERO_BLACK) ? 0.0 : 1.0; // depth == 0 returns 1.0 (main.rs:544-546)
  double run = 1.0;
  double w_emit = 1.0; // MIS weight of emission reached by the previous bounce's direction
  bool cut = false;
  auto roulette = [&](uint32_t bounce) {
    if (!(flags & YART_FLAG_RUSSIAN_ROULETTE) || bounce < YART_RR_FIRST_BOUNCE) return false;
    const double q = run < YART_RR_MIN_SURVIVAL ? YART_RR_MIN_SURVIVAL : (run > 1.0 ? 1.0 : run);
    double u_rr, unused;
    rng.draw(bounce, YART_SLOT_RR, u_rr, unused);
    if (u_rr >= q) return true;
    run = run / q;
    factors.push_back(F{q, 0, 0, 0, 2});
    return false;
  };
  for (uint32_t bounce = 1; bounce <= max_depth; ++bounce) {
    HitRec rec;
    if (n_rays) (*n_rays)++;
    if (!world_hit(c, ray, 0.001, kInf, &rng, bounce, rec)) {
      terminal = rgb_reflect(s.background, ray.wl);
      break;
    }
    const yart_material& mat = s.materials[rec.material];
    double emitted = 0.0;
    if (mat.kind == YART_MAT_DIFFUSE_LIGHT) emitted = rec.front_face ? texture_value(s, mat.texture, ray, rec) : 0.0;
    if (mat.kind == YART_MAT_NONE || mat.kind == YART_MAT_DIFFUSE_LIGHT) {
      terminal = emitted * w_emit;
      break;
    }
    w_emit = 1.0;
    if (mat.kind == YART_MAT_METAL) {
      V3 reflected = reflect(unit_vector(ray.d), rec.normal);
      V3 dir = reflected + mat.fuzz * random_in_unit_sphere(rng, bounce);
      factors.push_back(F{texture_value(s, mat.texture, ray, rec), 0, 0, 0, 0});
      run = run * factors.back().atten;
      ray = Ray{rec.p, dir, ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    if (mat.kind == YART_MAT_ISOTROPIC) {
      factors.push_back(F{texture_value(s, mat.texture, ray, rec), 0, 0, 0, 0});
      run = run * factors.back().atten;
      ray = Ray{rec.p, random_in_unit_sphere(rng, bounce), ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    if (mat.kind == YART_MAT_DIELECTRIC) {
      double n = sellmeier_index(mat, ray.wl);
      V3 outward;
      double ni_over_nt, cosine;
      if (dot(ray.d, rec.normal) > 0.0) {
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
      factors.push_back(F{1.0, 0, 0, 0, 0});
      ray = Ray{rec.p, dir, ray.time, ray.wl};
      if (roulette(bounce)) { cut = true; break; }
      continue;
    }
    // Lambertian through the mixture pdf, unbiased light pick
    const double atten = texture_value(s, mat.texture, ray, rec);
    const Onb uvw = onb_from_w(rec.normal);
    double u_mix, u_pick, r1, r2;
    rng.draw(bounce, YART_SLOT_MIX, u_mix, u_pick);
    rng.draw(bounce, YART_SLOT_DIR, r1, r2);
    auto cosine_dir = [&]() {
      double z = std::sqrt(1.0 - r2);
      double phi = 2.0 * kPi * r1;
      double x = lm_cos(phi) * std::sqrt(r2);
      double y = lm_sin(phi) * std::sqrt(r2);
      return onb_local(uvw, v3(x, y, z));
    };
    const bool have_lights = !s.lights.empty();
    const V3 dir = (u_mix < 0.5 && have_lights) ? lights_random(s, rec.p, u_pick, r1, r2, true) : cosine_dir();
    const double cosv = dot(unit_vector(dir), uvw.w);
    const double cos_pdf = cosv <= 0.0 ? 0.0 : cosv / kPi;
    const double p0 = have_lights ? lights_pdf_value(s, rec.p, dir) : cos_pdf;
    const double pdf_val = 0.5 * p0 + 0.5 * cos_pdf;
    // the light sample pairs with the emission bounce+1 would collect: none at max_depth, whose next hit is never traced
    const double nee = (have_lights && bounce < max_depth) ? next_event_sample(c, ray, rng, bounce, rec, uvw, atten) : 0.0;
    if (!std::isfinite(pdf_val) || pdf_val <= 0.0) {
      terminal = emitted + nee;
      break;
    }
    if (have_lights) w_emit = pdf_val * pdf_val / (pdf_val * pdf_val + p0 * p0);
    const double cs = dot(rec.normal, unit_vector(dir));
    const double spdf = cs < 0.0 ? 0.0 : cs / kPi;
    factors.push_back(F{atten, spdf, pdf_val, nee, 1});
    run = run * atten * spdf / pdf_val;
    ray = Ray{rec.p, dir, ray.time, ray.wl};
    if (roulette(bounce)) { cut = true; break; }
  }
  double L = cut ? 0.0 : terminal;
  for (size_t i = factors.size(); i-- > 0;) {
    const F& f = factors[i];
    if (f.kind == 2) L = L / f.atten;
    else if (f.kind == 1) L = f.nee + f.atten * L * f.spdf / f.pdf;
    else L = f.atten * L;
  }
  return L;
}

} // namespace

YART_NEE_EXPORT int neeref_scene_create(const yart_scene_desc* desc, orc_scene** out) { return orc_scene_create(desc, out); }
YART_NEE_EXPORT void neeref_scene_free(orc_scene* s) { orc_scene_free(s); }
YART_NEE_EXPORT const char* neeref_last_error(void) { return orc_last_error(); }

// The sample loop of orc_render (main.rs:690-707, the rendered 8x8 tiles only) with the NEE integrator: film += the
// sanitised XYZ of every sample.  stats->rays counts path rays only.
YART_NEE_EXPORT int neeref_render(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, double* film,
                                  yart_stats* stats, int n_threads) {
  if (!s || !cam || !o || !film) { g_err = "null argument"; return YART_ERR_INVALID; }
  if (o->width < 2 || o->height < 2) { g_err = "width/height must be >= 2"; return YART_ERR_INVALID; }
  if (n_threads < 1) n_threads = 1;
  const Camera k = make_camera(*cam);
  const uint32_t W = o->width, H = o->height;
  std::atomic<uint32_t> next_row(0);
  std::atomic<uint64_t> total_rays(0), total_paths(0);
  auto worker = [&]() {
    HitCtx c{&s->s, o->order, nullptr};
    uint64_t rays = 0, paths = 0;
    for (uint32_t py; (py = next_row.fetch_add(1)) < H;) {
      if (!pixel_is_rendered(py, H)) continue;
      for (uint32_t px = 0; px < W; ++px) {
        if (!pixel_is_rendered(px, W)) continue;
        double* pix = film + ((size_t)py * W + px) * 3;
        for (uint32_t sm = o->sample_begin; sm < o->sample_end; ++sm) {
          const Rng rng = make_rng(o->seed, py * W + px, sm);
          const Ray r = camera_ray(k, rng, px, py, W, H);
          uint32_t nr = 0;
          const double refl = ray_reflectance_nee(c, r, rng, o->max_depth, &nr, o->flags);
          double cie[3], xyz[3], clean[3];
          xyz_from_wavelength(r.wl, cie);
          xyz[0] = cie[0] * refl; xyz[1] = cie[1] * refl; xyz[2] = cie[2] * refl;
          sanitize_sample_xyz(xyz, clean);
          pix[0] += clean[0]; pix[1] += clean[1]; pix[2] += clean[2];
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
