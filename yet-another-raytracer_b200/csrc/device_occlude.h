// device_occlude.h -- parameters of the occlusion-query kernels (device_occlude.cu) as yart_device.cu fills them.
#pragma once
#include "device_common.cuh"

namespace yart {

// What every pass of one occlusion query shares.
struct OccludeCommon {
  const yart_ray* rays;        // indexed by ray id
  const yart_ray_f32* rays32;  // non-null: the rays are f32 records instead (yart_occluded_f32), `rays` is unused
  uint8_t* occluded;           // indexed by ray id: 1 once some object hits; zeroed before the first pass
  uint32_t n_rays;
  uint32_t first_pass;         // 0: skip the rays an earlier pass has already marked
  double t_min, t_max;         // t_max: what yart_closest_hit's pass would start from on a ray nothing has hit yet
};

// one mesh instance (k_occlude)
struct OccludeParams {
  OccludeCommon c;
  MeshPass m;
};

// a run of consecutive analytic / media-wrapped objects of the world list (k_analytic_occluded)
struct AnalyticOccludedParams {
  OccludeCommon c;
  DevScene scene;
  const yart_object* objects; // the world list
  uint32_t obj_begin, obj_end;
  uint32_t pixel_base;        // a ray's Philox stream is pixel = pixel_base + ray id, sample 0, bounce 1
  uint32_t media;             // the scene has constant media
};

typedef void (*OccludeKernel)(const OccludeParams);
typedef void (*AnalyticOccludedKernel)(const AnalyticOccludedParams);
OccludeKernel occlude_kernel(uint32_t max_stack);
AnalyticOccludedKernel analytic_occluded_kernel();

} // namespace yart
