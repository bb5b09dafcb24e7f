// aov_ref.cpp -- the CPU reference the AOV tests compare yart_render_aovs against (test infrastructure only).
//
// The unchanged oracle (oracle/yart_oracle.cpp, compiled into this translation unit) supplies the camera, the Philox
// streams and world.hit; this file adds the denoiser planes of include/yart.h's yart_render_aovs contract, restated
// from the contract, not from the CUDA code: the camera ray of (pixel, sample) as orc_camera_rays makes it, its
// world.hit(ray, 0.001, inf) with the render's rng at bounce 1, and the albedo / normal / depth rules.  Every
// transcendental goes through the oracle's libm_result hook, so a YART_ORACLE_LIBM_PERTURB build of this file moves
// them like tests/perturbed_oracle.py's variants.  Only the aovref_* entry points are exported.
#include "../oracle/yart_oracle.cpp"

#define YART_AOV_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

// one (pixel, sample): the HitRecord (as record_ref writes it) and the three plane contributions
struct AovSample {
  yart_hit_record rec;
  double albedo[3], normal[3], depth[3];
};

// the RGB texture_value hands to rgb_reflect (texture.rs): checker a / b, the texel, the solid colour, noise scalar
// times white; an image without texels is white
void texture_rgb(const Scene& s, uint32_t tex, const HitRec& rec, double out[3]) {
  const yart_texture& t = s.textures[tex];
  double k = 0.0;
  switch (t.kind) {
    case YART_TEX_SOLID:
      for (int i = 0; i < 3; ++i) out[i] = t.rgb_a[i];
      return;
    case YART_TEX_CHECKER: {
      const double sines = lm_sin(10.0 * rec.p.x) * lm_sin(10.0 * rec.p.y) * lm_sin(10.0 * rec.p.z);
      for (int i = 0; i < 3; ++i) out[i] = sines < 0.0 ? t.rgb_a[i] : t.rgb_b[i];
      return;
    }
    case YART_TEX_NOISE: {
      const yart_perlin& pn = s.perlins[t.perlin];
      if (t.noise_type == YART_NOISE_NET) k = perlin_turb(pn, t.noise_type, rec.p * t.scale, 7);
      else if (t.noise_type == YART_NOISE_MARBLE) k = 0.5 * (1.0 + lm_sin(t.scale * rec.p.z + 10.0 * perlin_turb(pn, t.noise_type, rec.p, 7)));
      else k = 0.5 * (1.0 + perlin_noise(pn, t.noise_type, rec.p * t.scale));
      break;
    }
    case YART_TEX_IMAGE: {
      const Scene::Image& im = s.images[t.image];
      if (im.data.empty()) { k = 1.0; break; }
      const double uu = rec.u < 0.0 ? 0.0 : (rec.u > 1.0 ? 1.0 : rec.u);
      const double vc = rec.v < 0.0 ? 0.0 : (rec.v > 1.0 ? 1.0 : rec.v);
      uint32_t i = f64_as_u32(uu * (double)im.w), j = f64_as_u32((1.0 - vc) * (double)im.h);
      if (i >= im.w) i = im.w - 1;
      if (j >= im.h) j = im.h - 1;
      for (int c = 0; c < 3; ++c) out[c] = (1.0 / 255.0) * (double)im.data[(size_t)j * 3 * im.w + (size_t)i * 3 + c];
      return;
    }
    default: break;
  }
  for (int i = 0; i < 3; ++i) out[i] = k;
}

double clamp01(double x) { return x > 0.0 ? (x < 1.0 ? x : 1.0) : 0.0; }

void aov_sample(const Scene& s, const Camera& cam, const yart_render_opts& o, uint32_t px, uint32_t py, uint32_t sample,
                AovSample& out) {
  const Rng rng = make_rng(o.seed, py * o.width + px, sample);
  const Ray ray = camera_ray(cam, rng, px, py, o.width, o.height);
  HitCtx c{&s, o.order, nullptr};
  HitRec rec;
  const bool some = world_hit(c, ray, 0.001, kInf, &rng, 1, rec);
  yart_hit_record& r = out.rec;
  for (int i = 0; i < 3; ++i) out.albedo[i] = out.normal[i] = out.depth[i] = 0.0;
  out.depth[2] = 1.0;
  if (!some) {
    r.t = kInf;
    for (int i = 0; i < 3; ++i) r.p[i] = r.normal[i] = 0.0;
    r.u = r.v = 0.0;
    r.material = r.obj_id = r.prim_id = YART_MISS;
    r.front_face = 0;
    for (int i = 0; i < 3; ++i) out.albedo[i] = clamp01(s.background[i]);
    return;
  }
  r.t = rec.t;
  r.p[0] = rec.p.x; r.p[1] = rec.p.y; r.p[2] = rec.p.z;
  r.normal[0] = rec.normal.x; r.normal[1] = rec.normal.y; r.normal[2] = rec.normal.z;
  r.u = rec.u; r.v = rec.v;
  r.material = rec.material; r.front_face = rec.front_face ? 1u : 0u; r.obj_id = rec.obj; r.prim_id = rec.prim;
  double alb[3] = {0.0, 0.0, 0.0};
  const yart_material& m = s.materials[rec.material];
  switch (m.kind) {
    case YART_MAT_LAMBERTIAN:
    case YART_MAT_METAL:
    case YART_MAT_ISOTROPIC: texture_rgb(s, m.texture, rec, alb); break;
    case YART_MAT_DIELECTRIC: alb[0] = alb[1] = alb[2] = 1.0; break;
    case YART_MAT_DIFFUSE_LIGHT:
      if (rec.front_face) texture_rgb(s, m.texture, rec, alb);
      break;
    default: break;
  }
  for (int i = 0; i < 3; ++i) out.albedo[i] = clamp01(alb[i]);
  const bool medium = (s.objects[rec.obj].wrap & YART_WRAP_MEDIUM) != 0;
  const double n2 = rec.normal.x * rec.normal.x + rec.normal.y * rec.normal.y + rec.normal.z * rec.normal.z;
  const double len = std::sqrt(n2);
  if (!medium && len > 0.0 && std::isfinite(len)) {
    out.normal[0] = rec.normal.x / len; out.normal[1] = rec.normal.y / len; out.normal[2] = rec.normal.z / len;
  }
  out.depth[0] = rec.t * std::sqrt(ray.d.x * ray.d.x + ray.d.y * ray.d.y + ray.d.z * ray.d.z);
  out.depth[1] = 1.0;
}

bool check_opts(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o) {
  if (!s || !cam || !o) { g_err = "null argument"; return false; }
  if (o->width < 2 || o->height < 2 || o->sample_end < o->sample_begin) { g_err = "bad options"; return false; }
  return true;
}

template <class F>
void parallel_rows(uint32_t H, int n_threads, F&& f) {
  if (n_threads < 1) n_threads = 1;
  std::vector<std::thread> th;
  for (int t = 0; t < n_threads; ++t)
    th.emplace_back([&, t]() {
      for (uint32_t y = (uint32_t)t; y < H; y += (uint32_t)n_threads) f(y);
    });
  for (auto& x : th) x.join();
}

} // namespace

YART_AOV_EXPORT int aovref_scene_create(const yart_scene_desc* desc, orc_scene** out) { return orc_scene_create(desc, out); }
YART_AOV_EXPORT void aovref_scene_free(orc_scene* s) { orc_scene_free(s); }
YART_AOV_EXPORT const char* aovref_last_error(void) { return orc_last_error(); }
YART_AOV_EXPORT uint32_t aovref_sample_bytes(void) { return (uint32_t)sizeof(AovSample); }

// every (pixel, sample) of samples [sample_begin, sample_end), tiles or not, pixel-major: out[pixel * ns + s - begin]
YART_AOV_EXPORT int aovref_samples(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, AovSample* out,
                                   int n_threads) {
  if (!check_opts(s, cam, o) || !out) return YART_ERR_INVALID;
  const Camera k = make_camera(*cam);
  const uint32_t ns = o->sample_end - o->sample_begin;
  parallel_rows(o->height, n_threads, [&](uint32_t y) {
    for (uint32_t x = 0; x < o->width; ++x)
      for (uint32_t sm = o->sample_begin; sm < o->sample_end; ++sm)
        aov_sample(s->s, k, *o, x, y, sm, out[((size_t)y * o->width + x) * ns + (sm - o->sample_begin)]);
  });
  return YART_OK;
}

// the planes of yart_render_aovs: added to per rendered pixel in sample order; null planes are skipped
YART_AOV_EXPORT int aovref_planes(const orc_scene* s, const yart_camera* cam, const yart_render_opts* o, double* albedo,
                                  double* normal, double* depth, int n_threads) {
  if (!check_opts(s, cam, o)) return YART_ERR_INVALID;
  const Camera k = make_camera(*cam);
  parallel_rows(o->height, n_threads, [&](uint32_t y) {
    if (!pixel_is_rendered(y, o->height)) return;
    for (uint32_t x = 0; x < o->width; ++x) {
      if (!pixel_is_rendered(x, o->width)) continue;
      const size_t px = ((size_t)y * o->width + x) * 3;
      for (uint32_t sm = o->sample_begin; sm < o->sample_end; ++sm) {
        AovSample a;
        aov_sample(s->s, k, *o, x, y, sm, a);
        for (int i = 0; i < 3; ++i) {
          if (albedo) albedo[px + i] += a.albedo[i];
          if (normal) normal[px + i] += a.normal[i];
          if (depth) depth[px + i] += a.depth[i];
        }
      }
    }
  });
  return YART_OK;
}

// texture tests: the RGB above, and the oracle's texture_value / rgb_reflect at a hit point p with texture u, v
YART_AOV_EXPORT void aovref_texture_rgb(const orc_scene* s, uint32_t tex, const double* p3, double u, double v, double* rgb3) {
  HitRec rec{};
  rec.p = v3(p3[0], p3[1], p3[2]);
  rec.u = u;
  rec.v = v;
  texture_rgb(s->s, tex, rec, rgb3);
}
YART_AOV_EXPORT double aovref_texture_value(const orc_scene* s, uint32_t tex, double wl, const double* p3, double u, double v) {
  HitRec rec{};
  rec.p = v3(p3[0], p3[1], p3[2]);
  rec.u = u;
  rec.v = v;
  Ray r{v3(0, 0, 0), v3(0, 0, 1), 0.0, wl};
  return texture_value(s->s, tex, r, rec);
}
YART_AOV_EXPORT double aovref_rgb_reflect(const double* rgb3, double wl) { return rgb_reflect(rgb3, wl); }
