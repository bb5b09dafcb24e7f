// device_shade.cuh -- everything after the closest hit: HitRecord reconstruction, textures,
// materials, light sampling, the camera, and the wavefront stage kernels (ray-gen, shade/scatter
// with queue compaction, film accumulation, display finalisation).
//
// All arithmetic is f64 in the reference's operation order (compiled with -fmad=false); the only
// values that can differ from the CPU oracle are the last bits of libm-style functions
// (sin, cos, log, acos, atan2, pow), whose CUDA implementations are not glibc's.
#pragma once
#include <type_traits>

#include "device_trace.cuh"

namespace yart {

// ---------------------------------------------------------------------------------------------
// spectral colour (reference color.rs)
// ---------------------------------------------------------------------------------------------
YART_DEV int spectrum_bin(double wl) { // Spectrum::reflect (color.rs:279-283): `as usize` saturates
  double q = (wl - 360.0) / 10.0;
  long long idx = (q != q || q <= 0.0) ? 0 : (q >= 1e18 ? (long long)1e18 : (long long)q);
  if (idx > 35) idx = 35;
  return (int)idx;
}
// RGB::reflect (color.rs:160-164) via into_spectrum (color.rs:54-90), evaluated for one bin
YART_DEV double rgb_reflect(const DevScene& S, const double* rgb, double wl) {
  const int i = spectrum_bin(wl);
  const double red = rgb[0], green = rgb[1], blue = rgb[2];
  const double* T = S.smits;
#define YART_B(b) __ldg(T + (b) * 36 + i)
  double s = 0.0;
  if (red <= green && red <= blue) {
    s = red * YART_B(0) + s;
    if (green <= blue) {
      s = (green - red) * YART_B(1) + s;
      s = (blue - green) * YART_B(6) + s;
    } else {
      s = (blue - red) * YART_B(1) + s;
      s = (green - blue) * YART_B(5) + s;
    }
  } else if (green <= red && green <= blue) {
    s = green * YART_B(0) + s;
    if (red <= blue) {
      s = (red - green) * YART_B(2) + s;
      s = (blue - red) * YART_B(6) + s;
    } else {
      s = (blue - green) * YART_B(2) + s;
      s = (red - blue) * YART_B(4) + s;
    }
  } else {
    s = blue * YART_B(0) + s;
    if (red <= green) {
      s = (red - blue) * YART_B(3) + s;
      s = (green - red) * YART_B(5) + s;
    } else {
      s = (green - blue) * YART_B(3) + s;
      s = (red - green) * YART_B(4) + s;
    }
  }
#undef YART_B
  return s;
}
YART_DEV void xyz_from_wavelength(const DevScene& S, double wl, double out[3]) { // color.rs:216-227
  double q = wl - 360.0;
  long long idx = (q != q) ? 0 : (q <= -9e18 ? (long long)-9e18 : (q >= 9e18 ? (long long)9e18 : (long long)q));
  if (idx < 0 || idx >= 471) {
    out[0] = out[1] = out[2] = 0.0;
  } else {
    out[0] = __ldg(S.cie + idx);
    out[1] = __ldg(S.cie + 471 + idx);
    out[2] = __ldg(S.cie + 942 + idx);
  }
}

// ---------------------------------------------------------------------------------------------
// HitRecord (hittable.rs:37-45) rebuilt from the compact DevHit
// ---------------------------------------------------------------------------------------------
struct HitRec {
  double u, v, t;
  D3 p, normal;
  bool front_face;
  uint32_t material;
};

YART_DEV void get_sphere_uv(D3 p, double& u, double& v) { // sphere.rs:213-220
  double theta = acos(-p.y);
  double phi = atan2(-p.z, p.x) + kPi;
  u = phi / (2.0 * kPi);
  v = theta / kPi;
}
YART_DEV void rect_record(int kaxis, double a0, double a1, double b0, double b1, D3 ro, D3 rd, double t, HitRec& rec) {
  const int aa = (kaxis == 0) ? 1 : 0;
  const int ba = (kaxis == 2) ? 1 : 2;
  double a = comp(ro, aa) + t * comp(rd, aa);
  double b = comp(ro, ba) + t * comp(rd, ba);
  rec.u = (a - a0) / (a1 - a0);
  rec.v = (b - b0) / (b1 - b0);
  rec.p = ro + t * rd;
  D3 outward = d3(kaxis == 0 ? 1.0 : 0.0, kaxis == 1 ? 1.0 : 0.0, kaxis == 2 ? 1.0 : 0.0);
  if (dot(rd, outward) < 0.0) {
    rec.normal = outward; rec.front_face = true;
  } else {
    rec.normal = -outward; rec.front_face = false;
  }
}
// record of an un-wrapped primitive in its own space.  ALL_UV = false: the renderer's record, which leaves a sphere's u, v
// at 0 where its material cannot read them; true: every field as the reference computes it (yart_closest_hit_records).
template <bool ALL_UV = false>
YART_DEV void prim_record(const DevScene& S, const yart_object& o, D3 ro, D3 rd, double time, double t, uint32_t prim,
                          double bu, double bv, HitRec& rec) {
  rec.t = t;
  rec.material = o.material;
  // get_sphere_uv (acos + atan2) only feeds ImageTexture::value; skip it when this material cannot read u, v
  bool need_uv = true;
  if (!ALL_UV) {
    const yart_material& pm = S.materials[o.material];
    need_uv = pm.kind != YART_MAT_NONE && pm.kind != YART_MAT_DIELECTRIC && S.textures[pm.texture].kind == YART_TEX_IMAGE;
  }
  switch (o.kind) {
    case YART_OBJ_SPHERE: // sphere.rs:68-85
    case YART_OBJ_MOVING_SPHERE: { // sphere.rs:175-197 (one copy of the shared steps: each `/` inlines a slow path)
      const bool moving = o.kind == YART_OBJ_MOVING_SPHERE;
      const D3 center = moving ? moving_center(o, time) : d3(o.p[0], o.p[1], o.p[2]);
      const double radius = moving ? o.p[8] : o.p[3];
      rec.p = ro + t * rd;
      D3 outward = vdiv(rec.p - center, moving ? radius : fabs(radius));
      if (moving) {
        if (dot(rd, outward) < 0.0) {
          rec.normal = outward; rec.front_face = true;
        } else {
          rec.normal = -outward; rec.front_face = false;
        }
      } else if (radius < 0.0) {
        rec.normal = -outward; rec.front_face = dot(rd, outward) > 0.0;
      } else {
        rec.normal = outward; rec.front_face = dot(rd, outward) < 0.0;
      }
      rec.u = rec.v = 0.0;
      if (need_uv) get_sphere_uv(outward, rec.u, rec.v);
      break;
    }
    case YART_OBJ_XY_RECT:
    case YART_OBJ_XZ_RECT:
    case YART_OBJ_YZ_RECT:
    case YART_OBJ_BOX: {
      int axis;
      double a0, a1, b0, b1, k;
      if (o.kind == YART_OBJ_BOX) {
        box_side(o.p, (int)(prim & 7u), axis, a0, a1, b0, b1, k);
      } else {
        axis = rect_axis(o.kind); a0 = o.p[0]; a1 = o.p[1]; b0 = o.p[2]; b1 = o.p[3];
      }
      rect_record(axis, a0, a1, b0, b1, ro, rd, t, rec);
      break;
    }
    case YART_OBJ_TRIANGLE: { // triangle.rs:80-100
      const double w = 1.0 - bu - bv;
      D3 n0 = d3(o.p[9], o.p[10], o.p[11]), n1 = d3(o.p[12], o.p[13], o.p[14]), n2 = d3(o.p[15], o.p[16], o.p[17]);
      D3 outward = n0 * w + n1 * bu + n2 * bv;
      if (dot(rd, outward) < 0.0) {
        rec.normal = outward; rec.front_face = true;
      } else {
        rec.normal = -outward; rec.front_face = false;
      }
      rec.u = o.p[18] * w + o.p[20] * bu + o.p[22] * bv;
      rec.v = o.p[19] * w + o.p[21] * bu + o.p[23] * bv;
      rec.p = ro + t * rd;
      break;
    }
    case YART_OBJ_MESH: { // the winning lane of an L4QBVH leaf (qbvh.rs:452-489)
      const DevMesh m = S.meshes[o.index];
      YART_CHECK(prim < m.n_tris);
      const double* sh = m.shade + (size_t)prim * 12;
      const float* uvf = reinterpret_cast<const float*>(sh + 9);
      rec.p = d3(ro.x + t * rd.x, ro.y + t * rd.y, ro.z + t * rd.z);
      const double w = 1.0 - bu - bv;
      D3 outward = d3(sh[0] * w + sh[3] * bu + sh[6] * bv, sh[1] * w + sh[4] * bu + sh[7] * bv,
                      sh[2] * w + sh[5] * bu + sh[8] * bv);
      const bool ff = (rd.x * outward.x + rd.y * outward.y + rd.z * outward.z) <= 0.0;
      const double sign = ff ? 1.0 : -1.0;
      rec.normal = d3(sign * outward.x, sign * outward.y, sign * outward.z);
      rec.front_face = ff;
      rec.u = (double)uvf[0] * w + (double)uvf[2] * bu + (double)uvf[4] * bv;
      rec.v = (double)uvf[1] * w + (double)uvf[3] * bu + (double)uvf[5] * bv;
      break;
    }
    default:
      rec.p = ro + t * rd;
      rec.normal = d3(1.0, 0.0, 0.0);
      rec.front_face = true;
      rec.u = rec.v = 0.0;
      break;
  }
}

// the HitRecord world.hit returns for (object, t): wrappers applied outside-in (ALL_UV: as for prim_record)
template <bool ALL_UV = false>
YART_DEV void world_record(const DevScene& S, const DevHit& h, D3 wo, D3 wd, double time, HitRec& rec) {
  const yart_object& o = S.objects[h.obj];
  if (o.wrap & YART_WRAP_MEDIUM) { // hittable.rs:296-308
    rec.t = h.t;
    rec.p = wo + h.t * wd;
    rec.u = rec.v = 0.0;
    rec.normal = d3(1.0, 0.0, 0.0);
    rec.front_face = true;
    rec.material = o.material;
    return;
  }
  D3 ro = wo, rd = wd;
  to_object_space(o, ro, rd);
  const bool group = o.kind == YART_OBJ_GROUP; // one inlined prim_record for a group member and a plain object
  const yart_object& po = group ? S.groups[o.index].members[h.prim >> 3] : o;
  prim_record<ALL_UV>(S, po, ro, rd, time, h.t, group ? (h.prim & 7u) : h.prim, h.bu, h.bv, rec);
  if (o.wrap & YART_WRAP_FLIP_FACE) rec.front_face = !rec.front_face;
  if (o.wrap & YART_WRAP_ROTATE_Y) { // hittable.rs:232-246
    const double ct = o.cos_theta, st = o.sin_theta;
    D3 p = rec.p, n = rec.normal;
    p.x = ct * rec.p.x + st * rec.p.z;
    p.z = -st * rec.p.x + ct * rec.p.z;
    n.x = ct * rec.normal.x + st * rec.normal.z;
    n.z = -st * rec.normal.x + ct * rec.normal.z;
    rec.p = p;
    rec.normal = n;
  }
  if (o.wrap & YART_WRAP_TRANSLATE) rec.p = rec.p + d3(o.offset[0], o.offset[1], o.offset[2]);
}

// ---------------------------------------------------------------------------------------------
// textures (texture.rs)
// ---------------------------------------------------------------------------------------------
YART_DEV int32_t f64_as_i32(double x) {
  if (x != x) return 0;
  if (x >= 2147483647.0) return 2147483647;
  if (x <= -2147483648.0) return (-2147483647 - 1);
  return (int32_t)x;
}
YART_DEV uint32_t f64_as_u32(double x) {
  if (x != x || x <= 0.0) return 0;
  if (x >= 4294967295.0) return 4294967295u;
  return (uint32_t)x;
}
__device__ __noinline__ double perlin_noise(const yart_perlin& pn, uint32_t type, D3 p) { // texture.rs:113-175
  if (type == YART_NOISE_SQUARE) {
    int i = f64_as_i32(4.0 * p.x) & 255, j = f64_as_i32(4.0 * p.y) & 255, k = f64_as_i32(4.0 * p.z) & 255;
    return pn.ranfloat[pn.perm_x[i] ^ pn.perm_y[j] ^ pn.perm_z[k]];
  }
  if (type == YART_NOISE_TRILINEAR) {
    double u = p.x - floor(p.x), v = p.y - floor(p.y), w = p.z - floor(p.z);
    u = u * u * (3.0 - 2.0 * u);
    v = v * v * (3.0 - 2.0 * v);
    w = w * w * (3.0 - 2.0 * w);
    int i = f64_as_i32(floor(p.x)), j = f64_as_i32(floor(p.y)), k = f64_as_i32(floor(p.z));
    double accum = 0.0;
    for (int di = 0; di < 2; ++di)
      for (int dj = 0; dj < 2; ++dj)
        for (int dk = 0; dk < 2; ++dk) {
          double c = pn.ranfloat[pn.perm_x[(i + di) & 255] ^ pn.perm_y[(j + dj) & 255] ^ pn.perm_z[(k + dk) & 255]];
          accum += ((double)di * u + (double)(1 - di) * (1.0 - u)) * ((double)dj * v + (double)(1 - dj) * (1.0 - v)) *
                   ((double)dk * w + (double)(1 - dk) * (1.0 - w)) * c;
        }
    return accum;
  }
  double u = p.x - floor(p.x), v = p.y - floor(p.y), w = p.z - floor(p.z);
  int i = f64_as_i32(floor(p.x)), j = f64_as_i32(floor(p.y)), k = f64_as_i32(floor(p.z));
  double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
  double accum = 0.0;
  for (int di = 0; di < 2; ++di)
    for (int dj = 0; dj < 2; ++dj)
      for (int dk = 0; dk < 2; ++dk) {
        const double* c = pn.ranvec[pn.perm_x[(i + di) & 255] ^ pn.perm_y[(j + dj) & 255] ^ pn.perm_z[(k + dk) & 255]];
        D3 wv = d3(u - (double)di, v - (double)dj, w - (double)dk);
        accum += ((double)di * uu + (1.0 - (double)di) * (1.0 - uu)) * ((double)dj * vv + (1.0 - (double)dj) * (1.0 - vv)) *
                 ((double)dk * ww + (1.0 - (double)dk) * (1.0 - ww)) * dot(wv, d3(c[0], c[1], c[2]));
      }
  return accum;
}
__device__ __noinline__ double perlin_turb(const yart_perlin& pn, uint32_t type, D3 p, int depth) { // texture.rs:231-243
  double accum = 0.0, weight = 1.0;
  D3 tp = p;
  for (int i = 0; i < depth; ++i) {
    accum += weight * perlin_noise(pn, type, tp);
    weight *= 0.5;
    tp = tp * 2.0;
  }
  return fabs(accum);
}
// Noise and image textures, out of line: they take the hit point / uv by value, so that no HitRec goes through
// local memory on the way here.
__device__ __noinline__ double texture_value_slow(const DevScene& S, const yart_texture& t, double wl, D3 p, double u,
                                                  double v) {
  const double white[3] = {1.0, 1.0, 1.0};
  switch (t.kind) {
    case YART_TEX_NOISE: {
      const yart_perlin& pn = S.perlins[t.perlin];
      if (t.noise_type == YART_NOISE_NET) return rgb_reflect(S, white, wl) * perlin_turb(pn, t.noise_type, p * t.scale, 7);
      if (t.noise_type == YART_NOISE_MARBLE)
        return rgb_reflect(S, white, wl) * 0.5 * (1.0 + sin(t.scale * p.z + 10.0 * perlin_turb(pn, t.noise_type, p, 7)));
      return rgb_reflect(S, white, wl) * 0.5 * (1.0 + perlin_noise(pn, t.noise_type, p * t.scale));
    }
    case YART_TEX_IMAGE: {
      const DevImage im = S.images[t.image];
      if (im.rgb8 == nullptr) return 1.0;
      double uu = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
      double vc = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
      double vv = 1.0 - vc;
      uint32_t i = f64_as_u32(uu * (double)im.width);
      uint32_t j = f64_as_u32(vv * (double)im.height);
      if (i >= im.width) i = im.width - 1;
      if (j >= im.height) j = im.height - 1;
      const double cs = 1.0 / 255.0;
      const size_t px = (size_t)j * 3 * im.width + (size_t)i * 3;
      const double rgb[3] = {cs * (double)im.rgb8[px], cs * (double)im.rgb8[px + 1], cs * (double)im.rgb8[px + 2]};
      return rgb_reflect(S, rgb, wl);
    }
    default: return 0.0;
  }
}
// Texture::value at hit point p, (u, v): solid and checker in line, the rest through texture_value_slow
YART_DEV double texture_value(const DevScene& S, uint32_t tex, double wl, D3 p, double u, double v) {
  const yart_texture& t = S.textures[tex];
  if (t.kind == YART_TEX_SOLID) return rgb_reflect(S, t.rgb_a, wl);
  if (t.kind == YART_TEX_CHECKER) {
    double sines = sin(10.0 * p.x) * sin(10.0 * p.y) * sin(10.0 * p.z);
    return sines < 0.0 ? rgb_reflect(S, t.rgb_a, wl) : rgb_reflect(S, t.rgb_b, wl);
  }
  return texture_value_slow(S, t, wl, p, u, v);
}

// The RGB a texture hands to rgb_reflect in texture_value (noise: its scalar times white; an image without texels:
// white).  A function of its own, not the first half of texture_value: for noise, rgb_reflect(white) * s and
// rgb_reflect(s * white) are different doubles, and the renderer keeps texture_value's.
YART_DEV void texture_rgb(const DevScene& S, uint32_t tex, const HitRec& rec, double rgb[3]) {
  const yart_texture& t = S.textures[tex];
  const double* c = nullptr;
  double s = 0.0;
  switch (t.kind) {
    case YART_TEX_SOLID: c = t.rgb_a; break;
    case YART_TEX_CHECKER: {
      double sines = sin(10.0 * rec.p.x) * sin(10.0 * rec.p.y) * sin(10.0 * rec.p.z);
      c = sines < 0.0 ? t.rgb_a : t.rgb_b;
      break;
    }
    case YART_TEX_NOISE: {
      const yart_perlin& pn = S.perlins[t.perlin];
      if (t.noise_type == YART_NOISE_NET) s = perlin_turb(pn, t.noise_type, rec.p * t.scale, 7);
      else if (t.noise_type == YART_NOISE_MARBLE) s = 0.5 * (1.0 + sin(t.scale * rec.p.z + 10.0 * perlin_turb(pn, t.noise_type, rec.p, 7)));
      else s = 0.5 * (1.0 + perlin_noise(pn, t.noise_type, rec.p * t.scale));
      break;
    }
    case YART_TEX_IMAGE: {
      const DevImage im = S.images[t.image];
      if (im.rgb8 == nullptr) { s = 1.0; break; }
      double uu = rec.u < 0.0 ? 0.0 : (rec.u > 1.0 ? 1.0 : rec.u);
      double vc = rec.v < 0.0 ? 0.0 : (rec.v > 1.0 ? 1.0 : rec.v);
      double vv = 1.0 - vc;
      uint32_t i = f64_as_u32(uu * (double)im.width);
      uint32_t j = f64_as_u32(vv * (double)im.height);
      if (i >= im.width) i = im.width - 1;
      if (j >= im.height) j = im.height - 1;
      const double cs = 1.0 / 255.0;
      const size_t px = (size_t)j * 3 * im.width + (size_t)i * 3;
      for (int k = 0; k < 3; ++k) rgb[k] = cs * (double)im.rgb8[px + k];
      return;
    }
    default: break;
  }
  for (int k = 0; k < 3; ++k) rgb[k] = c ? c[k] : s;
}

// ---------------------------------------------------------------------------------------------
// ONB, PDFs, light sampling (onb.rs, pdf.rs, sphere.rs:95-118, aarect.rs:148-171)
// ---------------------------------------------------------------------------------------------
struct Onb {
  D3 u, v, w;
};
YART_DEV Onb onb_from_w(D3 n) {
  Onb b;
  b.w = unit_vector(n);
  D3 a = fabs(b.w.x) > 0.9 ? d3(0.0, 1.0, 0.0) : d3(1.0, 0.0, 0.0);
  b.v = unit_vector(cross(b.w, a));
  b.u = cross(b.w, b.v);
  return b;
}
YART_DEV D3 onb_local(const Onb& b, D3 a) { return a.x * b.u + a.y * b.v + a.z * b.w; }

YART_DEV double light_pdf_value(const yart_object& l, D3 origin, D3 direction) {
  if (l.wrap != 0) return 0.0;
  if (l.kind == YART_OBJ_SPHERE) {
    double t;
    const D3 center = d3(l.p[0], l.p[1], l.p[2]);
    const double radius = l.p[3];
    if (!sphere_t(center, radius, origin, direction, 0.001, d_inf(), t)) return 0.0;
    double cos_theta_max = sqrt(1.0 - radius * radius / length_squared(center - origin));
    double solid_angle = 2.0 * kPi * (1.0 - cos_theta_max);
    return 1.0 / solid_angle;
  }
  if (l.kind == YART_OBJ_XZ_RECT) {
    double t;
    if (!rect_t(1, l.p[0], l.p[1], l.p[2], l.p[3], l.p[4], origin, direction, 0.001, d_inf(), t)) return 0.0;
    D3 outward = d3(0.0, 1.0, 0.0);
    D3 normal = dot(direction, outward) < 0.0 ? outward : -outward;
    double area = (l.p[1] - l.p[0]) * (l.p[3] - l.p[2]);
    double distance_squared = t * t * length_squared(direction);
    double cosine = fabs(dot(direction, normal)) / length(direction);
    return distance_squared / (cosine * area);
  }
  return 0.0;
}
// HAVE_CS: the caller gives cos / sin of the sphere case's phi = 2 pi r1 (shade_path forms them once for both halves of
// the mixture pdf, whose lanes would otherwise run the two f64 sin / cos evaluations one after the other).
template <bool HAVE_CS = false>
YART_DEV D3 light_random(const yart_object& l, D3 origin, double r1, double r2, double cos_phi = 0.0, double sin_phi = 0.0) {
  if (l.wrap == 0 && l.kind == YART_OBJ_SPHERE) {
    const D3 center = d3(l.p[0], l.p[1], l.p[2]);
    const double radius = l.p[3];
    D3 direction = center - origin;
    double distance_squared = length_squared(direction);
    Onb uvw = onb_from_w(direction);
    double z = 1.0 + r2 * (sqrt(1.0 - radius * radius / distance_squared) - 1.0);
    if (!HAVE_CS) {
      const double phi = 2.0 * kPi * r1;
      cos_phi = cos(phi);
      sin_phi = sin(phi);
    }
    double x = cos_phi * sqrt(1.0 - z * z);
    double y = sin_phi * sqrt(1.0 - z * z);
    return onb_local(uvw, d3(x, y, z));
  }
  if (l.wrap == 0 && l.kind == YART_OBJ_XZ_RECT) {
    D3 pt = d3(l.p[0] + (l.p[1] - l.p[0]) * r1, l.p[4], l.p[2] + (l.p[3] - l.p[2]) * r2);
    return pt - origin;
  }
  return d3(1.0, 0.0, 0.0);
}
YART_DEV double lights_pdf_value(const DevScene& S, D3 origin, D3 direction) { // hittable.rs:103-111
  double weight = 1.0 / (double)S.n_lights;
  double sum = 0.0;
  for (uint32_t i = 0; i < S.n_lights; ++i) sum += weight * light_pdf_value(S.lights[i], origin, direction);
  return sum;
}
// hittable.rs:113-122: `gen_range(0..len-1)` never picks the last light although pdf_value averages over all of
// them (SURVEY Appendix A-2).  unbiased (YART_FLAG_UNBIASED_LIGHT_PICK): uniform over all n lights.
YART_DEV D3 lights_random(const DevScene& S, D3 origin, double u_pick, double r1, double r2, bool unbiased, double cos_phi,
                          double sin_phi) {
  const uint32_t n = S.n_lights;
  if (n == 0) return d3(1.0, 0.0, 0.0);
  uint32_t k = 0;
  if (n > 1) {
    const uint32_t m = unbiased ? n : n - 1;
    k = (uint32_t)(u_pick * (double)m);
    if (k > m - 1) k = m - 1;
  }
  return light_random<true>(S.lights[k], origin, r1, r2, cos_phi, sin_phi); // (one inlined call site)
}

// ---------------------------------------------------------------------------------------------
// materials (material.rs)
// ---------------------------------------------------------------------------------------------
YART_DEV D3 reflect(D3 v, D3 n) { return v - 2.0 * dot(v, n) * n; }
YART_DEV bool refract(D3 v, D3 n, double ni_over_nt, D3& out) {
  D3 uv = unit_vector(v);
  double dt = dot(uv, n);
  double disc = 1.0 - ni_over_nt * ni_over_nt * (1.0 - dt * dt);
  if (disc > 0.0) {
    out = (uv - n * dt) * ni_over_nt - n * sqrt(disc);
    return true;
  }
  return false;
}
YART_DEV double schlick(double cosine, double ref_idx) {
  double r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
  r0 = r0 * r0;
  const double x = 1.0 - cosine;
  const double x2 = x * x;
  const double x4 = x2 * x2;
  return r0 + (1.0 - r0) * (x4 * x);
}
YART_DEV double sellmeier_index(const yart_material& m, double wl) {
  double wl2 = wl * wl;
  double n2 = 1.0 + m.sellmeier_b[0] * wl2 / (wl2 - m.sellmeier_c[0]) + m.sellmeier_b[1] * wl2 / (wl2 - m.sellmeier_c[1]) +
              m.sellmeier_b[2] * wl2 / (wl2 - m.sellmeier_c[2]);
  return sqrt(n2);
}

// ---------------------------------------------------------------------------------------------
// wavefront state and stage kernels
// ---------------------------------------------------------------------------------------------
struct PathState { // SoA over the paths of one batch, indexed by path id = pixel_local*spp_batch + s
  yart_ray* rays;
  double* time;
  double* wavelength;
  double* throughput;
  DevHit* hits;
  // The sample's XYZ (before sanitising) is written once, when the path ends, into the first 24 bytes of the
  // path's own -- by then dead -- ray record: k_film_accumulate reads it from there.
};

// YART_FLAG_NEXT_EVENT only, indexed by path id like PathState.  The stage kernels take it as their LAST parameter
// (null in the flag-off instances), so that the parameters before it keep their offsets there.
struct NeeState {
  yart_ray* rays;       // the shadow ray a Lambertian bounce aims at a light
  double* pending;      // what that ray adds per unit of emission it finds: thr_in * atten * spdf / p_l * MIS weight
  double* sum;          // light-sample contributions collected so far (added to the sample by k_film_accumulate)
  double* w_emit;       // MIS weight of emission the path's current ray reaches (1 unless it left a Lambertian hit)
  uint32_t* queue;      // the paths with a shadow ray this bounce
  uint32_t* counts;     // counts[bounce]: length of that queue
};

struct RenderParams {
  DevScene scene;
  DevCamera cam;
  PathState st;
  uint32_t width, height;
  uint32_t pixel_base, n_pixels; // this batch covers pixels [pixel_base, pixel_base + n_pixels)
  uint32_t sample_base, spp_batch;
  uint32_t max_depth;
  // objects [tail_begin, tail_end) of the world list -- a trailing run of plain spheres -- are intersected by
  // k_shade itself (it has the ray and the hit in hand) instead of costing a pass over the queue
  uint32_t tail_begin, tail_end;
  uint32_t flags; // YART_FLAG_UNBIASED_LIGHT_PICK | RUSSIAN_ROULETTE | DEPTH_ZERO_BLACK | NEXT_EVENT (all off = the reference)
  uint64_t seed;
};

YART_DEV bool pixel_is_rendered(uint32_t x, uint32_t W) { // 8 tiles of W/8 at W*col/8 (main.rs:636-646)
  const uint32_t cw = W / 8;
  for (uint32_t col = 0; col < 8; ++col) {
    const uint32_t x0 = (uint32_t)((uint64_t)W * col / 8);
    if (x >= x0 && x < x0 + cw) return true;
  }
  return false;
}
// Camera::get_ray for one (pixel, sample) (main.rs:690-698, camera.rs:82-94)
YART_DEV void camera_sample(const DevCamera& c, const Rng& rng, uint32_t px, uint32_t py, uint32_t W, uint32_t H, D3& ro,
                            D3& rd, double& time, double& wl) {
  double jx, jy, uwl, ut;
  rng_draw(rng, 0, YART_SLOT_CAM_JITTER, jx, jy);
  rng_draw(rng, 0, YART_SLOT_CAM_WL_TIME, uwl, ut);
  const double target_x = (double)px + jx;
  const double u = target_x / (double)(W - 1);
  const double target_y = (double)py + jy;
  const double v = 1.0 - target_y / (double)(H - 1);
  wl = 360.0 + (720.0 - 360.0) * uwl;
  D3 disk = d3(0.0, 0.0, 0.0);
  for (uint32_t i = 0; i < YART_MAX_REJECT; ++i) {
    double a, b;
    rng_draw(rng, 0, YART_SLOT_CAM_LENS + i, a, b);
    D3 p = d3(-1.0 + 2.0 * a, -1.0 + 2.0 * b, 0.0);
    if (length_squared(p) >= 1.0) continue;
    disk = p;
    break;
  }
  const D3 cu = d3(c.u[0], c.u[1], c.u[2]), cv = d3(c.v[0], c.v[1], c.v[2]);
  const D3 org = d3(c.origin[0], c.origin[1], c.origin[2]);
  const D3 llc = d3(c.llc[0], c.llc[1], c.llc[2]);
  const D3 hor = d3(c.horizontal[0], c.horizontal[1], c.horizontal[2]);
  const D3 ver = d3(c.vertical[0], c.vertical[1], c.vertical[2]);
  D3 lens = c.lens_radius * disk;
  D3 offset = cu * lens.x + cv * lens.y;
  ro = org + offset;
  rd = llc + u * hor + v * ver - org - offset;
  time = c.time0 + (c.time1 - c.time0) * ut;
}

template <bool NEE>
__global__ void __launch_bounds__(256) k_raygen(const RenderParams R, uint32_t* queue, uint32_t* queue_count, const NeeState N) {
  const uint64_t n = (uint64_t)R.n_pixels * R.spp_batch;
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t base = blockIdx.x * (uint64_t)blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t id = base + threadIdx.x;
    bool alive = false;
    if (id < n) {
      const uint32_t pixel = R.pixel_base + (uint32_t)(id / R.spp_batch);
      const uint32_t sample = R.sample_base + (uint32_t)(id % R.spp_batch);
      const uint32_t px = pixel % R.width, py = pixel / R.width;
      if (pixel_is_rendered(px, R.width) && pixel_is_rendered(py, R.height)) {
        const Rng rng = make_rng(R.seed, pixel, sample);
        D3 ro, rd;
        double time, wl;
        camera_sample(R.cam, rng, px, py, R.width, R.height, ro, rd, time, wl);
        store_ray(R.st.rays + id, ro, rd);
        R.st.time[id] = time;
        R.st.wavelength[id] = wl;
        R.st.throughput[id] = 1.0;
        if constexpr (NEE) N.w_emit[id] = 1.0;
        alive = true;
      } else { // outside the reference's 8x8 tiles (main.rs:643-646): never sampled
        store_sample(R.st.rays + id, 0.0, 0.0, 0.0);
        if constexpr (NEE) R.st.wavelength[id] = 0.0; // (k_film_accumulate<true> reads it: outside the CIE table, weight 0)
      }
      if constexpr (NEE) N.sum[id] = 0.0;
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, alive);
    if (ballot) {
      uint32_t pos = 0;
      const int leader = __ffs(ballot) - 1;
      if ((int)lane == leader) pos = atomicAdd(queue_count, (uint32_t)__popc(ballot));
      pos = __shfl_sync(0xffffffffu, pos, leader);
      YART_CHECK(pos + __popc(ballot) <= R.n_pixels * R.spp_batch);
      if (alive) queue[pos + __popc(ballot & ((1u << lane) - 1u))] = (uint32_t)id;
    }
  }
}

// camera rays only (yart_generate_camera_rays)
__global__ void __launch_bounds__(256) k_camera_rays(const RenderParams R, yart_ray* rays, double* wl_out, double* time_out) {
  const uint64_t n = (uint64_t)R.n_pixels * R.spp_batch;
  for (uint64_t id = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; id < n; id += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t pixel = R.pixel_base + (uint32_t)(id / R.spp_batch);
    const uint32_t sample = R.sample_base + (uint32_t)(id % R.spp_batch);
    const Rng rng = make_rng(R.seed, pixel, sample);
    D3 ro, rd;
    double time, wl;
    camera_sample(R.cam, rng, pixel % R.width, pixel / R.width, R.width, R.height, ro, rd, time, wl);
    yart_ray r;
    r.origin[0] = ro.x; r.origin[1] = ro.y; r.origin[2] = ro.z;
    r.direction[0] = rd.x; r.direction[1] = rd.y; r.direction[2] = rd.z;
    rays[id] = r;
    if (wl_out) wl_out[id] = wl;
    if (time_out) time_out[id] = time;
  }
}

// One bounce of ray_reflectance (main.rs:537-588) for every queued path.  Surviving paths are
// appended to the next queue (warp-aggregated atomics = stream compaction); finished paths write
// their sample value.  `bounce` is 1-based: the bounce-th world.hit of the path.
// One bounce of one path: everything k_shade does for path `id` except the compaction of the survivors.
// Returns true when the path goes on (its next ray and throughput are stored), false when it ended (its sample
// value is stored).
// NEE (YART_FLAG_NEXT_EVENT): a Lambertian bounce before max_depth may also store a shadow ray and its pending weight;
// the emission the path reaches is MIS-weighted, and an ended path stores the scalar thr * terminal instead of its
// XYZ (k_film_accumulate<true> adds the light samples and applies the CIE weights).  Returns bit 0 = goes on,
// bit 1 = has a shadow ray.  (No out-parameter: that perturbs the register allocation of the flag-off instance.)
template <bool NEE>
YART_DEV std::conditional_t<NEE, uint32_t, bool> shade_path(const RenderParams& R, const NeeState& N, uint32_t id, uint32_t bounce) {
  bool shadow = false;
  const DevScene& S = R.scene;
  bool alive = false;
  const uint32_t pixel = R.pixel_base + id / R.spp_batch;
  const uint32_t sample = R.sample_base + id % R.spp_batch;
  const Rng rng = make_rng(R.seed, pixel, sample);
  D3 wo, wd;
  load_ray(R.st.rays + id, wo, wd);
  const double time = R.st.time[id];
  const double wl = R.st.wavelength[id];
  double thr = R.st.throughput[id];
  const DevHit h = R.st.hits[id];
  double terminal = 0.0;
  bool done = true;
  D3 next_d = d3(0, 0, 0), next_o = d3(0, 0, 0);
  double w_next = 1.0; // (NEE) the MIS weight of emission next_d reaches: 1 unless this is a Lambertian bounce
  if (h.obj == YART_MISS) {
    terminal = rgb_reflect(S, S.background, wl); // main.rs:587
  } else {
    HitRec rec;
    world_record(S, h, wo, wd, time, rec);
    const yart_material& mat = S.materials[rec.material];
    // the texture of every material that reads one (a DiffuseLight only where it emits), from one inlined call site
    double tex = 0.0;
    if (mat.kind != YART_MAT_NONE && mat.kind != YART_MAT_DIELECTRIC && (mat.kind != YART_MAT_DIFFUSE_LIGHT || rec.front_face))
      tex = texture_value(S, mat.texture, wl, rec.p, rec.u, rec.v);
    const double emitted = mat.kind == YART_MAT_DIFFUSE_LIGHT ? tex : 0.0;
    if (mat.kind == YART_MAT_NONE || mat.kind == YART_MAT_DIFFUSE_LIGHT) {
      terminal = emitted;
      if constexpr (NEE) {
        if (emitted != 0.0) terminal = emitted * N.w_emit[id];
      }
    } else if (mat.kind == YART_MAT_METAL) {
      D3 reflected = reflect(unit_vector(wd), rec.normal);
      next_d = reflected + mat.fuzz * random_in_unit_sphere(rng, bounce);
      next_o = rec.p;
      thr = thr * tex;
      done = false;
    } else if (mat.kind == YART_MAT_ISOTROPIC) {
      next_d = random_in_unit_sphere(rng, bounce);
      next_o = rec.p;
      thr = thr * tex;
      done = false;
    } else if (mat.kind == YART_MAT_DIELECTRIC) { // material.rs:213-301
      const double nidx = sellmeier_index(mat, wl);
      D3 outward;
      double ni_over_nt, cosine;
      const double ddn = dot(wd, rec.normal);
      if (ddn > 0.0) {
        outward = -rec.normal;
        ni_over_nt = nidx;
      } else {
        outward = rec.normal;
        ni_over_nt = 1.0 / nidx;
      }
      cosine = (ddn > 0.0 ? nidx * ddn : -ddn) / length(wd);
      D3 refracted;
      if (refract(wd, outward, ni_over_nt, refracted)) {
        double u0, u1;
        rng_draw(rng, bounce, YART_SLOT_DIELECTRIC, u0, u1);
        next_d = (u0 < schlick(cosine, nidx)) ? reflect(wd, rec.normal) : refracted;
      } else {
        next_d = reflect(wd, rec.normal);
      }
      next_o = rec.p;
      thr = thr * 1.0;
      done = false;
    } else { // Lambertian through the mixture pdf (material.rs:44-61, main.rs:560-581)
      const double atten = tex;
      const Onb uvw = onb_from_w(rec.normal);
      double u_mix, u_pick, r1, r2;
      rng_draw(rng, bounce, YART_SLOT_MIX, u_mix, u_pick);
      rng_draw(rng, bounce, YART_SLOT_DIR, r1, r2);
      const bool have_lights = S.n_lights != 0;
      const double phi = 2.0 * kPi * r1; // both halves of the mixture turn r1 into this angle
      const double cos_phi = cos(phi), sin_phi = sin(phi);
      D3 dir;
      if (u_mix < 0.5 && have_lights) {
        dir = lights_random(S, rec.p, u_pick, r1, r2, (R.flags & YART_FLAG_UNBIASED_LIGHT_PICK) != 0, cos_phi, sin_phi);
      } else { // random_cosine_direction (pdf.rs:15-25)
        const double z = sqrt(1.0 - r2);
        const double x = cos_phi * sqrt(r2);
        const double y = sin_phi * sqrt(r2);
        dir = onb_local(uvw, d3(x, y, z));
      }
      const D3 udir = unit_vector(dir);
      const double cosv = dot(udir, uvw.w);
      const double cos_pdf = cosv <= 0.0 ? 0.0 : cosv / kPi;
      const double p0 = have_lights ? lights_pdf_value(S, rec.p, dir) : cos_pdf;
      const double pdf_val = 0.5 * p0 + 0.5 * cos_pdf;
      // the light sample pairs with the emission bounce+1 would collect: none at max_depth, whose next hit is never traced.
      // (thr is still the throughput carried into this bounce here)
      if constexpr (NEE) {
        if (have_lights && bounce < R.max_depth) {
          double u_light, unused, s1, s2;
          rng_draw(rng, bounce, YART_SLOT_NEE_PICK, u_light, unused);
          rng_draw(rng, bounce, YART_SLOT_NEE_DIR, s1, s2);
          uint32_t k = (uint32_t)(u_light * (double)S.n_lights);
          if (k > S.n_lights - 1) k = S.n_lights - 1;
          const D3 dl = light_random(S.lights[k], rec.p, s1, s2);
          const double p_l = lights_pdf_value(S, rec.p, dl);
          const D3 udl = unit_vector(dl);
          const double cl = dot(udl, uvw.w);
          const double p_m = 0.5 * p_l + 0.5 * (cl <= 0.0 ? 0.0 : cl / kPi);
          const double csl = dot(rec.normal, udl);
          const double spdf_l = csl < 0.0 ? 0.0 : csl / kPi;
          if (isfinite(p_l) && p_l > 0.0 && spdf_l > 0.0) {
            store_ray(N.rays + id, rec.p, dl);
            N.pending[id] = thr * atten * spdf_l / p_l * (p_l * p_l / (p_l * p_l + p_m * p_m));
            shadow = true;
          }
        }
      }
      if (!isfinite(pdf_val) || pdf_val <= 0.0) {
        terminal = emitted;
      } else {
        const double cs = dot(rec.normal, udir);
        const double spdf = cs < 0.0 ? 0.0 : cs / kPi;
        if constexpr (NEE) w_next = have_lights ? pdf_val * pdf_val / (pdf_val * pdf_val + p0 * p0) : 1.0;
        thr = thr * atten * spdf / pdf_val;
        next_o = rec.p;
        next_d = dir;
        done = false;
      }
    }
  }
  if (!done && (R.flags & YART_FLAG_RUSSIAN_ROULETTE) && bounce >= YART_RR_FIRST_BOUNCE) {
    // Russian roulette (off in the reference): survive with probability q = clamp(throughput, 0.05, 1), unbiased
    const double q = thr < YART_RR_MIN_SURVIVAL ? YART_RR_MIN_SURVIVAL : (thr > 1.0 ? 1.0 : thr);
    double u_rr, unused;
    rng_draw(rng, bounce, YART_SLOT_RR, u_rr, unused);
    if (u_rr >= q) {
      done = true;
      terminal = 0.0;
    } else {
      thr = thr / q;
    }
  }
  if (!done && bounce >= R.max_depth) { // depth exhausted: ray_reflectance(depth 0) = 1.0 (main.rs:544-546)
    done = true;
    terminal = (R.flags & YART_FLAG_DEPTH_ZERO_BLACK) ? 0.0 : 1.0;
  }
  if (done) {
    const double refl = thr * terminal;
    if constexpr (NEE) {
      store_sample(R.st.rays + id, refl, 0.0, 0.0);
    } else {
      double cie[3];
      xyz_from_wavelength(S, wl, cie);
      store_sample(R.st.rays + id, cie[0] * refl, cie[1] * refl, cie[2] * refl);
    }
  } else {
    store_ray(R.st.rays + id, next_o, next_d);
    R.st.throughput[id] = thr;
    if constexpr (NEE) N.w_emit[id] = w_next;
    alive = true;
  }
  if constexpr (NEE) return (alive ? 1u : 0u) | (shadow ? 2u : 0u);
  else return alive;
}

#ifndef YART_SHADE_THREADS
#define YART_SHADE_THREADS 256
#endif
#ifndef YART_SHADE_MIN_BLOCKS
#define YART_SHADE_MIN_BLOCKS (1024 / YART_SHADE_THREADS)
#endif
constexpr int kShadeThreads = YART_SHADE_THREADS;

// append `id` to a queue when `take`: one atomic per warp
YART_DEV void warp_append(bool take, uint32_t id, uint32_t* queue, uint32_t* count, uint32_t cap) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t ballot = __ballot_sync(0xffffffffu, take);
  if (ballot) {
    uint32_t pos = 0;
    const int leader = __ffs(ballot) - 1;
    if ((int)lane == leader) pos = atomicAdd(count, (uint32_t)__popc(ballot));
    pos = __shfl_sync(0xffffffffu, pos, leader);
    YART_CHECK(pos + __popc(ballot) <= cap);
    if (take) queue[pos + __popc(ballot & ((1u << lane) - 1u))] = id;
  }
}

template <bool NEE>
__global__ void __launch_bounds__(kShadeThreads, YART_SHADE_MIN_BLOCKS) k_shade(const RenderParams R, const uint32_t* queue, const uint32_t* queue_count,
                                                uint32_t* next_queue, uint32_t* next_count, uint32_t bounce, const NeeState N) {
  const DevScene& S = R.scene;
  const uint32_t n = *queue_count;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // Paths of one block are regrouped by what their hit needs (miss / emitter, Lambertian, dielectric,
  // other) before shading, so the warps run mostly one branch of the material switch.  Which thread
  // shades which path does not matter: every result is addressed by the path id.
  __shared__ uint32_t s_ids[kShadeThreads];
  __shared__ uint32_t s_cnt[kShadeThreads / 32][4];
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    {
      const uint32_t it = base + threadIdx.x;
      uint32_t my_id = YART_MISS, cls = 4;
      if (it < n) {
        my_id = queue[it];
        YART_CHECK(my_id < R.n_pixels * R.spp_batch);
        uint32_t obj = R.st.hits[my_id].obj;
        if (R.tail_end > R.tail_begin) {
          // the last objects of HittableList::hit's scan (hittable.rs:66-79), same calls as k_analytic makes
          D3 wo, wd;
          load_ray(R.st.rays + my_id, wo, wd);
          double t_best = R.st.hits[my_id].t; // (+inf on a miss; t_max of the scan is +inf, main.rs:548)
          bool changed = false;
          for (uint32_t oi = R.tail_begin; oi < R.tail_end; ++oi) {
            const yart_object& so = S.objects[oi];
            double t;
            if (sphere_t(d3(so.p[0], so.p[1], so.p[2]), so.p[3], wo, wd, 0.001, t_best, t)) {
              t_best = t; obj = oi; changed = true;
            }
          }
          if (changed) {
            DevHit h;
            h.t = t_best; h.bu = 0.0; h.bv = 0.0; h.obj = obj; h.prim = 0;
            R.st.hits[my_id] = h; // read back by whichever thread shades this path (after the barrier below)
          }
        }
        YART_CHECK(obj == YART_MISS || obj < S.n_objects);
        cls = 0;
        if (obj != YART_MISS) {
          const yart_object& ob = S.objects[obj];
          uint32_t mi = ob.material;
          if (ob.kind == YART_OBJ_GROUP && !(ob.wrap & YART_WRAP_MEDIUM)) // a group is shaded with its member's material
            mi = S.groups[ob.index].members[R.st.hits[my_id].prim >> 3].material;
          const uint32_t kind = S.materials[mi].kind;
          cls = (kind == YART_MAT_LAMBERTIAN) ? 1u : ((kind == YART_MAT_DIELECTRIC) ? 2u
                : ((kind == YART_MAT_NONE || kind == YART_MAT_DIFFUSE_LIGHT) ? 0u : 3u));
        }
      }
      uint32_t rank = 0;
#pragma unroll
      for (uint32_t c = 0; c < 4; ++c) {
        const uint32_t b = __ballot_sync(0xffffffffu, cls == c);
        if (cls == c) rank = __popc(b & ((1u << lane) - 1u));
        if (lane == 0) s_cnt[warp][c] = __popc(b);
      }
      __syncthreads();
      if (cls < 4) {
        uint32_t off = 0;
        for (uint32_t c = 0; c < cls; ++c)
          for (uint32_t w = 0; w < kShadeThreads / 32; ++w) off += s_cnt[w][c];
        for (uint32_t w = 0; w < warp; ++w) off += s_cnt[w][cls];
        s_ids[off + rank] = my_id;
      }
      __syncthreads();
    }
    const uint32_t item = base + threadIdx.x;
    bool alive = false, shadow = false;
    uint32_t id = 0;
    if (item < n) {
      id = s_ids[threadIdx.x];
      if constexpr (NEE) {
        const uint32_t r = shade_path<true>(R, N, id, bounce);
        alive = (r & 1u) != 0;
        shadow = (r & 2u) != 0;
      } else {
        alive = shade_path<false>(R, N, id, bounce);
      }
    }
    if constexpr (NEE) warp_append(shadow, id, N.queue, N.counts + bounce, R.n_pixels * R.spp_batch);
    // stream compaction: one atomic per warp
    const uint32_t ballot = __ballot_sync(0xffffffffu, alive);
    if (ballot) {
      uint32_t pos = 0;
      const int leader = __ffs(ballot) - 1;
      if ((int)lane == leader) pos = atomicAdd(next_count, (uint32_t)__popc(ballot));
      pos = __shfl_sync(0xffffffffu, pos, leader);
      YART_CHECK(pos + __popc(ballot) <= R.n_pixels * R.spp_batch);
      if (alive) next_queue[pos + __popc(ballot & ((1u << lane) - 1u))] = id;
    }
    __syncthreads(); // s_ids / s_cnt are rewritten by the next round
  }
}

// YART_FLAG_NEXT_EVENT: the shadow rays of one bounce have been traced (closest hit in R.st.hits, as far as the passes
// go); finish their world.hit with the trailing spheres k_shade folds in, and collect the emission of a front-facing
// DiffuseLight.  A path may have ended in the same bounce: its light sample still counts.
__global__ void __launch_bounds__(256) k_nee_resolve(const RenderParams R, uint32_t bounce, const NeeState N) {
  const DevScene& S = R.scene;
  const uint32_t n = N.counts[bounce];
  for (uint32_t item = blockIdx.x * blockDim.x + threadIdx.x; item < n; item += gridDim.x * blockDim.x) {
    const uint32_t id = N.queue[item];
    YART_CHECK(id < R.n_pixels * R.spp_batch);
    D3 wo, wd;
    load_ray(N.rays + id, wo, wd);
    DevHit h = R.st.hits[id];
    for (uint32_t oi = R.tail_begin; oi < R.tail_end; ++oi) { // the same calls as k_shade's tail
      const yart_object& so = S.objects[oi];
      double t;
      if (sphere_t(d3(so.p[0], so.p[1], so.p[2]), so.p[3], wo, wd, 0.001, h.t, t)) {
        h.t = t; h.bu = 0.0; h.bv = 0.0; h.obj = oi; h.prim = 0;
      }
    }
    if (h.obj == YART_MISS) continue;
    YART_CHECK(h.obj < S.n_objects);
    HitRec rec;
    world_record(S, h, wo, wd, R.st.time[id], rec);
    const yart_material& mat = S.materials[rec.material];
    if (mat.kind != YART_MAT_DIFFUSE_LIGHT || !rec.front_face) continue;
    N.sum[id] += N.pending[id] * texture_value(S, mat.texture, R.st.wavelength[id], rec.p, rec.u, rec.v);
  }
}

// sanitize_sample_xyz (main.rs:448-459) + `pixel_color_xyz += sample` in sample order (main.rs:707)
// NEE: the stored value is the scalar thr * terminal; the sample is cie(wl) * (that + the light samples' sum).
template <bool NEE>
__global__ void __launch_bounds__(256) k_film_accumulate(const RenderParams R, double* film, const NeeState N) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < R.n_pixels; p += gridDim.x * blockDim.x) {
    double* px = film + (size_t)(R.pixel_base + p) * 3;
    double ax = px[0], ay = px[1], az = px[2];
    const yart_ray* c = R.st.rays + (size_t)p * R.spp_batch;
    for (uint32_t s = 0; s < R.spp_batch; ++s) {
      double x, y, z;
      load_sample(c + s, x, y, z);
      if constexpr (NEE) {
        const size_t id = (size_t)p * R.spp_batch + s;
        const double refl = x + N.sum[id];
        double cie[3];
        xyz_from_wavelength(R.scene, R.st.wavelength[id], cie);
        x = cie[0] * refl; y = cie[1] * refl; z = cie[2] * refl;
      }
      if (!isfinite(x) || !isfinite(y) || !isfinite(z)) {
        x = y = z = 0.0;
      } else if (!(y <= 0.0 || y <= 20.0)) {
        const double k = 20.0 / y;
        x = x * k; y = y * k; z = z * k;
      }
      ax += x; ay += y; az += z;
    }
    px[0] = ax; px[1] = ay; px[2] = az;
  }
}

YART_DEV double gamma_channel(double linear) { // color.rs:93-100
  linear = fmax(linear, 0.0);
  if (linear <= 0.0031308) return 12.92 * linear;
  return 1.055 * pow(linear, 1.0 / 2.4) - 0.055;
}
YART_DEV uint8_t clamp_display_channel(double c) { // main.rs:461-463
  double x = c;
  if (x < 0.0) x = 0.0;
  if (x > 0.999) x = 0.999;
  const double v = 256.0 * x;
  if (v != v) return 0;
  return (uint8_t)v;
}
// main.rs:710-712: one pixel's XYZ sum * (720-360) / (106.856895*spp), then into_rgb -- linear RGB
YART_DEV void film_linear_rgb(const double* f, uint32_t spp, double& r, double& g, double& b) {
  const double mul = 720.0 - 360.0, den = 106.856895 * (double)spp;
  const D3 c = vdiv(d3(f[0] * mul, f[1] * mul, f[2] * mul), den);
  r = 2.6896552 * c.x - 1.2758621 * c.y - 0.4137931 * c.z;
  g = -1.0221082 * c.x + 1.9782866 * c.y + 0.0438216 * c.z;
  b = 0.0612245 * c.x - 0.2244898 * c.y + 1.1632653 * c.z;
}
// main.rs:710-718
__global__ void __launch_bounds__(256) k_film_finalize(const double* film, uint32_t W, uint32_t H, uint32_t spp, uint8_t* rgba) {
  const uint32_t n = W * H;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const uint32_t x = p % W, y = p / W;
    uint8_t* o = rgba + (size_t)p * 4;
    if (!pixel_is_rendered(x, W) || !pixel_is_rendered(y, H)) {
      o[0] = o[1] = o[2] = o[3] = 0;
      continue;
    }
    double r, g, b;
    film_linear_rgb(film + (size_t)p * 3, spp, r, g, b);
    o[0] = clamp_display_channel(gamma_channel(r));
    o[1] = clamp_display_channel(gamma_channel(g));
    o[2] = clamp_display_channel(gamma_channel(b));
    o[3] = 255;
  }
}

// yart_film_finalize_linear: the (r, g, b) k_film_finalize gamma-encodes, rounded to f32; 0 outside the tiles
__global__ void __launch_bounds__(256) k_film_finalize_linear(const double* film, uint32_t W, uint32_t H, uint32_t spp, float* rgb) {
  const uint32_t n = W * H;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    float* o = rgb + (size_t)p * 3;
    if (!pixel_is_rendered(p % W, W) || !pixel_is_rendered(p / W, H)) {
      o[0] = o[1] = o[2] = 0.f;
      continue;
    }
    double r, g, b;
    film_linear_rgb(film + (size_t)p * 3, spp, r, g, b);
    o[0] = (float)r; o[1] = (float)g; o[2] = (float)b;
  }
}

// ---------------------------------------------------------------------------------------------
// yart_render_aovs: the first hit of every camera sample as denoiser inputs
// ---------------------------------------------------------------------------------------------
YART_DEV double clamp01(double x) { return x > 0.0 ? (x < 1.0 ? x : 1.0) : 0.0; } // (NaN -> 0)

// One batch of k_raygen<false> samples after the bounce-1 passes over ALL objects (no k_shade, so no tail fold): adds,
// per rendered pixel and in sample order, each sample's albedo, unit normal and {distance, hit, 1} to the planes
// (null planes are skipped).  Pixels outside the tiles get nothing.
__global__ void __launch_bounds__(256) k_aov_accumulate(const RenderParams R, double* albedo, double* normal, double* depth) {
  const DevScene& S = R.scene;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < R.n_pixels; p += gridDim.x * blockDim.x) {
    const uint32_t pixel = R.pixel_base + p;
    if (!pixel_is_rendered(pixel % R.width, R.width) || !pixel_is_rendered(pixel / R.width, R.height)) continue;
    double a[3] = {0.0, 0.0, 0.0}, nm[3] = {0.0, 0.0, 0.0}, dp[3] = {0.0, 0.0, 0.0};
    for (int k = 0; k < 3; ++k) {
      if (albedo) a[k] = albedo[(size_t)pixel * 3 + k];
      if (normal) nm[k] = normal[(size_t)pixel * 3 + k];
      if (depth) dp[k] = depth[(size_t)pixel * 3 + k];
    }
    for (uint32_t s = 0; s < R.spp_batch; ++s) {
      const size_t id = (size_t)p * R.spp_batch + s;
      const DevHit h = R.st.hits[id];
      double alb[3] = {0.0, 0.0, 0.0}, n[3] = {0.0, 0.0, 0.0}, dist = 0.0;
      if (h.obj == YART_MISS) {
        for (int k = 0; k < 3; ++k) alb[k] = S.background[k];
      } else {
        YART_CHECK(h.obj < S.n_objects);
        D3 wo, wd;
        load_ray(R.st.rays + id, wo, wd);
        HitRec rec;
        world_record<true>(S, h, wo, wd, R.st.time[id], rec);
        const yart_material& mat = S.materials[rec.material];
        if (mat.kind == YART_MAT_LAMBERTIAN || mat.kind == YART_MAT_METAL || mat.kind == YART_MAT_ISOTROPIC ||
            (mat.kind == YART_MAT_DIFFUSE_LIGHT && rec.front_face)) {
          texture_rgb(S, mat.texture, rec, alb);
        } else if (mat.kind == YART_MAT_DIELECTRIC) {
          alb[0] = alb[1] = alb[2] = 1.0;
        }
        if (!(S.objects[h.obj].wrap & YART_WRAP_MEDIUM)) {
          const double len = sqrt(rec.normal.x * rec.normal.x + rec.normal.y * rec.normal.y + rec.normal.z * rec.normal.z);
          if (len > 0.0 && isfinite(len)) { n[0] = rec.normal.x / len; n[1] = rec.normal.y / len; n[2] = rec.normal.z / len; }
        }
        dist = rec.t * sqrt(wd.x * wd.x + wd.y * wd.y + wd.z * wd.z);
      }
      for (int k = 0; k < 3; ++k) { a[k] += clamp01(alb[k]); nm[k] += n[k]; }
      dp[0] += dist; dp[1] += h.obj == YART_MISS ? 0.0 : 1.0; dp[2] += 1.0;
    }
    for (int k = 0; k < 3; ++k) {
      if (albedo) albedo[(size_t)pixel * 3 + k] = a[k];
      if (normal) normal[(size_t)pixel * 3 + k] = nm[k];
      if (depth) depth[(size_t)pixel * 3 + k] = dp[k];
    }
  }
}

} // namespace yart
