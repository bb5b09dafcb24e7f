// device_denoise.cuh -- yart_denoise: the edge-avoiding a-trous wavelet filter of Dammertz, Sewtz, Hanika and Lensch
// (HPG 2010) over the film, guided by the planes of yart_render_aovs.  The contract (include/yart.h) is exact: f64
// throughout, a fixed tap order, no libm and no FMA contraction (-fmad=false), so tests/denoise_ref.py reproduces
// every bit of the f32 output.
//
// Scratch, per pixel: demodulated colour [2][4] f64 (ping-pong; the 4th slot keeps each pixel on one 32-byte sector),
// guide {normal, z} [4] f64, remodulation factor albedo + 1/128 [3] f64 and valid / hit flags u8: 121 bytes.
#pragma once
#include "device_shade.cuh"

namespace yart {

constexpr uint8_t kDenoiseValid = 1, kDenoiseHit = 2;
constexpr int kDenoiseTileX = 32, kDenoiseTileY = 8; // the 2-D block of k_denoise_atrous

// The per-pixel inputs of the filter: flags, demodulated colour c, guide {n, z} and remodulation factor m = a + 1/128.
__global__ void __launch_bounds__(256) k_denoise_prepare(const double* film, uint32_t spp, const double* albedo,
                                                         const double* normal, const double* depth, uint32_t n,
                                                         uint8_t* flags, double* color, double* guide, double* mod) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const size_t i3 = (size_t)p * 3, i4 = (size_t)p * 4;
    const double samples = depth[i3 + 2], hits = depth[i3 + 1];
    if (!(samples > 0.0)) {
      flags[p] = 0;
      continue;
    }
    double lin[3];
    film_linear_rgb(film + i3, spp, lin[0], lin[1], lin[2]);
    const bool hit = hits > 0.0;
    flags[p] = kDenoiseValid | (hit ? kDenoiseHit : 0);
    for (int k = 0; k < 3; ++k) {
      const double m = albedo[i3 + k] / samples + 1.0 / 128.0;
      mod[i3 + k] = m;
      color[i4 + k] = lin[k] / m;
      guide[i4 + k] = normal[i3 + k] / samples;
    }
    guide[i4 + 3] = hit ? depth[i3] / hits : 0.0;
  }
}

// The B3-spline taps H = {1/16, 1/4, 3/8, 1/4, 1/16} at d = -2..2 (a branch, not an array: no local memory)
YART_DEV double atrous_h(int d) { return d == 0 ? 3.0 / 8.0 : (d == 1 || d == -1 ? 1.0 / 4.0 : 1.0 / 16.0); }

// One level of the filter: step 2^level, kc = 4^level / sigma_c^2, kn = 1 / sigma_n^2, sz2 = sigma_z^2.  Taps in
// row-major (dy, dx) order; invalid pixels are never read as neighbours and are not written.
__global__ void __launch_bounds__(kDenoiseTileX * kDenoiseTileY)
    k_denoise_atrous(const uint8_t* __restrict__ flags, const double* __restrict__ guide, const double* __restrict__ in,
                     double* __restrict__ out, uint32_t W, uint32_t H, uint32_t step, double kc, double kn, double sz2) {
  const uint32_t x = blockIdx.x * kDenoiseTileX + threadIdx.x;
  if (x >= W) return;
  for (uint32_t y = blockIdx.y * kDenoiseTileY + threadIdx.y; y < H; y += gridDim.y * kDenoiseTileY) {
    const size_t p = (size_t)y * W + x;
    const uint8_t fp = __ldg(flags + p);
    if (!(fp & kDenoiseValid)) continue;
    const bool hit_p = (fp & kDenoiseHit) != 0;
    const double2 c01 = __ldg(reinterpret_cast<const double2*>(in + p * 4));
    const double cp[3] = {c01.x, c01.y, __ldg(in + p * 4 + 2)};
    const double2 g01 = __ldg(reinterpret_cast<const double2*>(guide + p * 4));
    const double2 g23 = __ldg(reinterpret_cast<const double2*>(guide + p * 4 + 2));
    const double np_[3] = {g01.x, g01.y, g23.x}, zp = g23.y;
    const double izp = hit_p ? 1.0 / ((sz2 * zp) * zp) : 0.0;
    double Wsum = 0.0, S[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
    for (int dy = -2; dy <= 2; ++dy) {
      const int64_t qy = (int64_t)y + (int64_t)dy * step;
      const bool row_in = qy >= 0 && qy < (int64_t)H;
#pragma unroll
      for (int dx = -2; dx <= 2; ++dx) {
        const int64_t qx = (int64_t)x + (int64_t)dx * step;
        if (!row_in || qx < 0 || qx >= (int64_t)W) continue;
        const double h = atrous_h(dy) * atrous_h(dx);
        if (dy == 0 && dx == 0) { // the centre: weight h, no edge terms
          Wsum += h;
          for (int k = 0; k < 3; ++k) S[k] += h * cp[k];
          continue;
        }
        const size_t q = (size_t)qy * W + (size_t)qx;
        YART_CHECK(q < (size_t)W * H);
        const uint8_t fq = __ldg(flags + q);
        if (!(fq & kDenoiseValid) || ((fq & kDenoiseHit) != 0) != hit_p) continue;
        const double2 q01 = __ldg(reinterpret_cast<const double2*>(in + q * 4));
        const double cq[3] = {q01.x, q01.y, __ldg(in + q * 4 + 2)};
        const double2 h01 = __ldg(reinterpret_cast<const double2*>(guide + q * 4));
        const double2 h23 = __ldg(reinterpret_cast<const double2*>(guide + q * 4 + 2));
        const double d0 = cq[0] - cp[0], d1 = cq[1] - cp[1], d2 = cq[2] - cp[2];
        const double e0 = h01.x - np_[0], e1 = h01.y - np_[1], e2 = h23.x - np_[2];
        double xw = ((d0 * d0 + d1 * d1) + d2 * d2) * kc + ((e0 * e0 + e1 * e1) + e2 * e2) * kn;
        if (hit_p) {
          const double dz = h23.y - zp;
          xw = xw + (dz * dz) * izp;
        }
        double t = 1.0 / (1.0 + xw * 0.125); // (1 + x/8)^-8, the libm-free stand-in for exp(-x)
        t = t * t;
        t = t * t;
        t = t * t;
        const double w = h * t;
        Wsum += w;
        for (int k = 0; k < 3; ++k) S[k] += w * cq[k];
      }
    }
    double* o = out + p * 4;
    for (int k = 0; k < 3; ++k) o[k] = S[k] / Wsum;
  }
}

// Remodulation and output: out = c * m as f32 linear RGB and/or through k_film_finalize's display rule as RGBA8;
// invalid pixels are all zero (alpha too).  Either output may be null.
__global__ void __launch_bounds__(256) k_denoise_finish(const uint8_t* flags, const double* color, const double* mod,
                                                        uint32_t n, float* rgb, uint8_t* rgba) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const bool valid = (flags[p] & kDenoiseValid) != 0;
    double v[3] = {0.0, 0.0, 0.0};
    if (valid)
      for (int k = 0; k < 3; ++k) v[k] = color[(size_t)p * 4 + k] * mod[(size_t)p * 3 + k];
    if (rgb)
      for (int k = 0; k < 3; ++k) rgb[(size_t)p * 3 + k] = (float)v[k];
    if (rgba) {
      uint8_t* o = rgba + (size_t)p * 4;
      for (int k = 0; k < 3; ++k) o[k] = valid ? clamp_display_channel(gamma_channel(v[k])) : 0;
      o[3] = valid ? 255 : 0;
    }
  }
}

} // namespace yart
