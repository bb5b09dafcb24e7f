/* yart.h -- C ABI of the B200-native path-tracing core.
 *
 * This is the drop-in boundary for the ONE hot path of themayflyman/yet-another-raytracer
 * (SURVEY.md section 8): closest-hit traversal of the 4-wide QBVH and the spectral bounce
 * loop.  The reference has no FFI today; the seams this ABI replaces are the Rust items
 * cited on each entry point (paths relative to the reference's raytracer/src/).  A Rust
 * `-sys` crate binds these symbols with a hand-written `extern "C"` block (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 (YART_OK) or a negative yart_status; nothing throws or aborts
 *     across the ABI; yart_last_error() gives the message of the last failure of a context
 *     (or of the calling thread for context-free calls).
 *   - plain pointers and sizes only.  The caller owns every pointer it passes; the library
 *     copies during the call and retains nothing, unless the function says otherwise.
 *   - a yart_ctx is bound to one GPU and is NOT thread-safe (one host thread per context,
 *     N GPUs = N contexts / N processes), matching `Hittable: Send + Sync` objects that are
 *     immutable after construction (hittable.rs:11).
 *   - there is NO CPU fallback: every compute entry point fails with YART_ERR_CUDA when no
 *     sm_100 device is usable.
 */
#ifndef YART_H
#define YART_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YART_ABI_VERSION 2

typedef enum yart_status {
  YART_OK = 0,
  YART_ERR_INVALID = -1,     /* bad argument / malformed scene (the reference panics)  */
  YART_ERR_CUDA = -2,        /* CUDA runtime error or no usable device                 */
  YART_ERR_NOMEM = -3,
  YART_ERR_IO = -4,          /* OBJ / asset could not be read (triangle.rs:113 expect) */
  YART_ERR_UNSUPPORTED = -5
} yart_status;

/* ------------------------------------------------------------------------------------ */
/* Geometry inputs                                                                      */
/* ------------------------------------------------------------------------------------ */

/* A triangle soup in tobj emission order: what TriangleMesh::from_obj hands to L4QBVH::new
 * (triangle.rs:110-175).  Positions and uvs are f32-exact because tobj parses f32
 * (triangle.rs:118-134); normals are f64 because the face-normal fallback for OBJs without
 * `vn` is computed in f64 (triangle.rs:146-153). */
typedef struct yart_trimesh {
  uint32_t n_tris;
  uint32_t _pad;
  const float* positions;  /* [n_tris][3 vertices][xyz]          */
  const double* normals;   /* [n_tris][3 vertices][xyz]          */
  const float* uvs;        /* [n_tris][3 vertices][u,v]          */
} yart_trimesh;

/* Object kinds: one per `impl Hittable` that scenes.rs instantiates. */
enum {
  YART_OBJ_SPHERE = 0,        /* StillSphere   sphere.rs:23-119   p = cx cy cz r                        */
  YART_OBJ_MOVING_SPHERE = 1, /* MovingSphere  sphere.rs:121-211  p = c0xyz c1xyz time0 time1 r         */
  YART_OBJ_XY_RECT = 2,       /* XYRect        aarect.rs:9-81     p = x0 x1 y0 y1 k                     */
  YART_OBJ_XZ_RECT = 3,       /* XZRect        aarect.rs:83-172   p = x0 x1 z0 z1 k                     */
  YART_OBJ_YZ_RECT = 4,       /* YZRect        aarect.rs:174-242  p = y0 y1 z0 z1 k                     */
  YART_OBJ_BOX = 5,           /* BoxEntity     box_entity.rs      p = p0xyz p1xyz                       */
  YART_OBJ_TRIANGLE = 6,      /* Triangle      triangle.rs:11-102 p = v0 v1 v2 n0 n1 n2 (uv0 uv1 uv2)   */
  YART_OBJ_MESH = 7,          /* TriangleMesh  triangle.rs:104-185 index = mesh index in the scene      */
  YART_OBJ_GROUP = 8          /* BVHNode over spheres/boxes bvh.rs:9-220: index = group index           */
};

/* Wrapper flags, applied outermost-first in this order: ConstantMedium(Translate(RotateY(
 * FlipFace(primitive)))) -- the only nestings scenes.rs uses. */
enum {
  YART_WRAP_ROTATE_Y = 1u,   /* RotateY        hittable.rs:158-256: sin_theta/cos_theta          */
  YART_WRAP_TRANSLATE = 2u,  /* Translate      hittable.rs:125-156: offset                       */
  YART_WRAP_FLIP_FACE = 4u,  /* FlipFace       hittable.rs:327-354                               */
  YART_WRAP_MEDIUM = 8u      /* ConstantMedium hittable.rs:258-325: neg_inv_density, `material`
                                is the Isotropic phase function                                  */
};

typedef struct yart_object {
  uint32_t kind;
  uint32_t wrap;          /* YART_WRAP_* bits                                      */
  uint32_t material;      /* index into yart_scene_desc.materials                  */
  uint32_t index;         /* mesh index (MESH) or group index (GROUP)              */
  double p[24];           /* kind-specific parameters, see the kind enum           */
  double sin_theta;       /* RotateY::new computes these from degrees on the host  */
  double cos_theta;
  double offset[3];
  double neg_inv_density; /* ConstantMedium::new: -1/density (hittable.rs:269)     */
} yart_object;

/* A BVHNode-accelerated set of spheres or boxes (scenes.rs:333-352, 411-424).  Closest-hit
 * results do not depend on the tree shape, so only the members are part of the ABI; the
 * library builds its own flat 4-wide tree over them. */
typedef struct yart_group {
  const yart_object* members; /* SPHERE or BOX records, no wrappers */
  uint32_t n_members;
  uint32_t _pad;
} yart_group;

/* ------------------------------------------------------------------------------------ */
/* Shading inputs                                                                       */
/* ------------------------------------------------------------------------------------ */
enum {
  YART_MAT_NONE = 0,          /* NoMaterial    material.rs:383-386 */
  YART_MAT_LAMBERTIAN = 1,    /* material.rs:33-61                 */
  YART_MAT_METAL = 2,         /* material.rs:63-95  (fuzz)         */
  YART_MAT_DIELECTRIC = 3,    /* material.rs:111-301 (Sellmeier b1..b3, c1..c3; wavelength in nm) */
  YART_MAT_DIFFUSE_LIGHT = 4, /* material.rs:336-355               */
  YART_MAT_ISOTROPIC = 5      /* material.rs:357-381               */
};

typedef struct yart_material {
  uint32_t kind;
  uint32_t texture; /* index into textures (albedo / emit); ignored by NONE and DIELECTRIC */
  double fuzz;
  double sellmeier_b[3];
  double sellmeier_c[3];
} yart_material;

enum {
  YART_TEX_SOLID = 0,   /* SolidColor<RGB>   texture.rs:18-40   rgb_a                         */
  YART_TEX_CHECKER = 1, /* CheckerTexture    texture.rs:42-68   odd = rgb_a, even = rgb_b     */
  YART_TEX_NOISE = 2,   /* NoiseTexture      texture.rs:245-285 noise_type, scale, perlin     */
  YART_TEX_IMAGE = 3    /* ImageTexture      texture.rs:287-345 image                         */
};
enum { /* NoiseType texture.rs:70-82 */
  YART_NOISE_SQUARE = 0, YART_NOISE_TRILINEAR = 1, YART_NOISE_SMOOTH = 2,
  YART_NOISE_MARBLE = 3, YART_NOISE_NET = 4
};

typedef struct yart_texture {
  uint32_t kind;
  uint32_t noise_type;
  uint32_t perlin; /* index into perlins */
  uint32_t image;  /* index into images  */
  double rgb_a[3];
  double rgb_b[3];
  double scale;
} yart_texture;

/* Perlin::new tables (texture.rs:84-111).  The reference fills them from an unseeded
 * thread_rng; presets here fill them from the scene seed. */
typedef struct yart_perlin {
  double ranfloat[256];
  double ranvec[256][3];
  int32_t perm_x[256];
  int32_t perm_y[256];
  int32_t perm_z[256];
} yart_perlin;

typedef struct yart_image { /* ImageTexture::new -> to_rgb8 (texture.rs:296-311) */
  const uint8_t* rgb8;      /* [height][width][3] */
  uint32_t width;
  uint32_t height;
} yart_image;

/* The whole scene: `world: HittableList` in list order (hittable.rs:47-79) plus the separate
 * sampling-lights list in preset order (main.rs:211-432; only SPHERE and XZ_RECT entries are
 * sampleable, every other kind has pdf 0 / direction (1,0,0) like the trait defaults
 * hittable.rs:28-34). */
typedef struct yart_scene_desc {
  const yart_object* objects;     uint32_t n_objects;   uint32_t _p0;
  const yart_object* lights;      uint32_t n_lights;    uint32_t _p1;
  const yart_trimesh* meshes;     uint32_t n_meshes;    uint32_t _p2;
  const yart_group* groups;       uint32_t n_groups;    uint32_t _p3;
  const yart_material* materials; uint32_t n_materials; uint32_t _p4;
  const yart_texture* textures;   uint32_t n_textures;  uint32_t _p5;
  const yart_perlin* perlins;     uint32_t n_perlins;   uint32_t _p6;
  const yart_image* images;       uint32_t n_images;    uint32_t _p7;
  double background_rgb[3];
} yart_scene_desc;

/* Camera::new arguments (camera.rs:41-80); render() passes vup=(0,1,0), focus_dist=10,
 * time0=0, time1=1 (main.rs:612-625). */
typedef struct yart_camera {
  double lookfrom[3];
  double lookat[3];
  double vup[3];
  double vfov_degrees;
  double aspect_ratio;
  double aperture;
  double focus_dist;
  double time0;
  double time1;
} yart_camera;

/* ------------------------------------------------------------------------------------ */
/* Rays and hits                                                                        */
/* ------------------------------------------------------------------------------------ */
typedef struct yart_ray { /* Ray (ray.rs:4-9); direction is NOT normalised */
  double origin[3];
  double direction[3];
} yart_ray;

#define YART_MISS 0xFFFFFFFFu

typedef struct yart_hit {
  double t;          /* HitRecord.t; +inf on a miss                                          */
  double u;          /* barycentric weight of vertex 1 (mesh / triangle hits), else tex u    */
  double v;          /* barycentric weight of vertex 2 (mesh / triangle hits), else tex v    */
  uint32_t prim_id;  /* mesh: ORIGINAL triangle index in tobj emission order; YART_MISS=miss */
  uint32_t obj_id;   /* index in yart_scene_desc.objects (0 for mesh-only queries)           */
  uint32_t front_face;
  uint32_t _pad;
} yart_hit;

/* The whole HitRecord (hittable.rs:37-45) as world.hit returns it, plus the ids of yart_hit: for
 * yart_closest_hit_records.  88 bytes. */
typedef struct yart_hit_record {
  double t;          /* HitRecord.t; +inf on a miss                                                    */
  double p[3];       /* HitRecord.p: ray.at(t) in the primitive's space, then the wrappers' transforms   */
                     /* (RotateY rotates it, Translate adds the offset); 0 on a miss                     */
  double normal[3];  /* HitRecord.normal exactly as the reference stores it: face-oriented, NOT          */
                     /* normalised (mesh / triangle: the interpolated vertex normals); 0 on a miss       */
  double u, v;       /* TEXTURE coordinates: mesh / triangle: the interpolated uvs; sphere and moving    */
                     /* sphere: get_sphere_uv; rect / box: the rect coordinates; medium: 0; 0 on a miss  */
  uint32_t material; /* index into yart_scene_desc.materials (a group hit: the member's material);
                        YART_MISS on a miss and for a mesh target (a bare mesh has no material)          */
  uint32_t front_face;
  uint32_t obj_id;   /* as yart_hit.obj_id; YART_MISS on a miss                                          */
  uint32_t prim_id;  /* as yart_hit.prim_id; YART_MISS on a miss                                         */
} yart_hit_record;

/* Single-precision ray / hit records for yart_closest_hit_f32: 24 + 16 bytes per ray instead of 48 + 40. */
typedef struct yart_ray_f32 {
  float origin[3];
  float direction[3];
} yart_ray_f32;

typedef struct yart_hit_f32 {
  float t;          /* +inf on a miss                                   */
  float u, v;       /* as yart_hit.u / .v                               */
  uint32_t prim_id; /* as yart_hit.prim_id; YART_MISS = miss            */
} yart_hit_f32;

/* Traversal order of the 4 children of a QBVH node.
 *  REFERENCE: exactly qbvh.rs:14-31,521-533 -- the ORDER_TABLE lookup, which visits the FAR
 *    child first; first-found wins among equal-t hits (qbvh.rs:478).
 *  NEAR: the mirrored table (near child first, ~30% fewer node visits) with mirrored tie
 *    rules (last-found wins, lanes reversed; strict against the t_max it is given).  It yields the
 *    same hit as REFERENCE on every ray of the parity sets (16 Mi random / axis / path rays per
 *    mesh, all presets).  The one known exception is a measure-zero set: a ray that passes within
 *    rounding of a vertex or edge lying ON a node's box face, where the slab value and the
 *    Moller-Trumbore t disagree in the last bit -- each order then culls the box the other enters
 *    and returns another member of the same near-tie set (|dt| <= a few ulp; tests/test_gpu_fuzz.py
 *    aims rays at such points and bounds it).  REFERENCE is exact always.                */
enum { YART_ORDER_REFERENCE = 0, YART_ORDER_NEAR = 1 };

/* flags of yart_closest_hit / yart_render */
enum {
  YART_FLAG_DEVICE_PTRS = 1u,   /* rays/hits (or the film) are device pointers on the ctx's GPU */
  YART_FLAG_COUNT_VISITS = 2u,  /* fill node/leaf visit counters in the stats (slower)          */
  /* Better sampling, yart_render only, OFF by default: with none of them set the renderer is the reference's
   * estimator bit for bit (SURVEY.md 8(f) row 4, Appendix A-1 / A-2). */
  YART_FLAG_UNBIASED_LIGHT_PICK = 4u, /* pick among ALL lights; the reference's HittableList::random draws from
                                         gen_range(0..len-1) and never samples the last one although pdf_value
                                         averages over all of them (hittable.rs:113-122 vs :103-111)            */
  YART_FLAG_RUSSIAN_ROULETTE = 8u,    /* from bounce 4 on a path survives with probability clamp(throughput, 0.05, 1)
                                         and is reweighted by 1/q (unbiased; the reference has no roulette)      */
  YART_FLAG_DEPTH_ZERO_BLACK = 16u,   /* a path cut at max_depth contributes 0; the reference's ray_reflectance
                                         returns 1.0 at depth 0 (main.rs:544-546)                                */
  YART_FLAG_NEXT_EVENT = 32u          /* next-event estimation with MIS (yart_render / yart_dump_path_rays only):
                                         at every Lambertian hit before max_depth one extra direction is drawn
                                         from the lights (uniform pick, YART_SLOT_NEE_*) and traced as a
                                         closest-hit shadow ray; a front-facing DiffuseLight it hits adds its
                                         emission with the power-heuristic weight p_l^2 / (p_l^2 + p_mix^2).
                                         Emission that the mixture-sampled continuation reaches is weighted
                                         p_mix^2 / (p_mix^2 + p_l^2) to match.  The path rays, and so
                                         yart_dump_path_rays and stats.rays, are those of the flag-off render.
                                         Implies YART_FLAG_UNBIASED_LIGHT_PICK (MIS needs the mixture's true
                                         density).  Costs 76 more bytes of device state per path in flight. */
};

#define YART_TARGET_WORLD 0xFFFFFFFFu

typedef struct yart_stats {
  uint64_t rays;            /* closest-hit queries executed (1 ray = 1 world.hit, main.rs:548); yart_render counts
                               path rays only, not the shadow rays of YART_FLAG_NEXT_EVENT, whose passes are
                               included in trace_ms, kernel_launches and trace_launches */
  uint64_t paths;           /* camera samples started                                           */
  uint64_t node_visits;     /* only with YART_FLAG_COUNT_VISITS                                 */
  uint64_t tri_tests;       /* only with YART_FLAG_COUNT_VISITS                                 */
  uint64_t kernel_launches; /* kernels of this library launched by the call                     */
  double gpu_ms;            /* CUDA-event time of the call's device work                        */
  double trace_ms;          /* ... of which closest-hit kernels                                 */
  uint32_t max_bounce;      /* deepest bounce that still had live paths                         */
  uint32_t trace_launches;  /* ... of kernel_launches: closest-hit kernels (k_traverse / k_analytic) */
} yart_stats;

typedef struct yart_render_opts {
  uint32_t width;
  uint32_t height;
  uint32_t sample_begin;  /* this call renders samples [sample_begin, sample_end) of every pixel; */
  uint32_t sample_end;    /* multi-GPU sharding is a host concern (SURVEY.md 8(e))                */
  uint32_t max_depth;     /* --max-depth (main.rs:95-96)                                          */
  uint32_t order;         /* YART_ORDER_*                                                         */
  uint32_t batch_spp;     /* samples per pixel per wavefront batch, 0 = library default           */
  uint32_t flags;         /* YART_FLAG_*                                                          */
  uint64_t seed;          /* Philox key; the reference is OS-seeded (thread_rng)                  */
} yart_render_opts;

/* ------------------------------------------------------------------------------------ */
/* Host-side front end (no GPU needed): OBJ loading, QBVH build + flattening, presets   */
/* ------------------------------------------------------------------------------------ */
typedef struct yart_objfile yart_objfile; /* owns a triangle soup */
typedef struct yart_qbvh yart_qbvh;       /* a built + flattened L4QBVH */
typedef struct yart_preset yart_preset;   /* an instantiated scene preset */

const char* yart_version(void);
/* message of the last failure on this thread for calls that take no context */
const char* yart_last_error_global(void);

/* TriangleMesh::from_obj up to the triangle list (triangle.rs:110-168): tobj load with
 * GPU_LOAD_OPTIONS semantics -- fan triangulation from the first vertex, per-corner v/vt/vn. */
int yart_obj_load(const char* path, yart_objfile** out);
void yart_obj_free(yart_objfile* obj);
int yart_obj_trimesh(const yart_objfile* obj, yart_trimesh* out); /* borrowed view, valid until free */

/* L4QBVH::new (qbvh.rs:251-361, split :636-693): median split on the longest centroid axis,
 * <=4-triangle leaves, post-order node emission (root = last node).  Ties of the unstable
 * sort are resolved by original triangle index (documented deviation: the Rust sort's tie
 * order is unspecified; closest-hit results do not depend on it). */
int yart_qbvh_build(const yart_trimesh* mesh, yart_qbvh** out);
void yart_qbvh_free(yart_qbvh* q);

typedef struct yart_qbvh_info {
  uint32_t n_nodes, n_leaves, n_tris, height, root, max_stack, _pad0, _pad1;
  double bbox_min[3], bbox_max[3];   /* L4QBVH::bounding_box (qbvh.rs:365-379) */
} yart_qbvh_info;
int yart_qbvh_get_info(const yart_qbvh* q, yart_qbvh_info* out);
/* The flattened device layout (DESIGN.md "data layout"): nodes = n_nodes x 32 x 4 bytes,
 * tris = n_tris x 12 x 4 bytes in tree order.  Borrowed, valid until free. */
const void* yart_qbvh_nodes(const yart_qbvh* q);
const void* yart_qbvh_tris(const yart_qbvh* q);
const void* yart_qbvh_shade(const yart_qbvh* q); /* n_tris x 96 bytes: vertex normals (f64) + uvs (f32), tree order */

/* build_scene_preset (main.rs:211-432) + scenes.rs.  `name` is the reference's kebab-case
 * --scene value (main.rs:61-76).  `assets_dir` holds cube.obj / david.obj / sycee.obj /
 * earthmap_1024x512.rgb8.  `seed` replaces thread_rng for random-scene, next-week-final and
 * the Perlin tables.  bunny.obj / teapot.obj are not shipped with the reference: they are used when assets_dir has
 * them; otherwise sycee.obj stands in and yart_preset_note() says so (with YART_STRICT_ASSETS=1 in the environment the
 * call fails with YART_ERR_IO instead, like the reference's "Failed to load OBJ file", triangle.rs:112-113). */
int yart_preset_build(const char* name, const char* assets_dir, uint64_t seed, yart_preset** out);
void yart_preset_free(yart_preset* p);
/* "" or a sentence the front end must show the user (a stand-in mesh was loaded).  Borrowed, valid until free. */
const char* yart_preset_note(const yart_preset* p);
const yart_scene_desc* yart_preset_scene(const yart_preset* p);

typedef struct yart_preset_info { /* RenderDefaults + ScenePreset fields (main.rs:109-146) */
  uint32_t width, height, samples_per_pixel, max_depth, workers, _pad;
  double vfov, aperture;
  double lookfrom[3], lookat[3];
  char output_filename[64];
} yart_preset_info;
int yart_preset_get_info(const yart_preset* p, yart_preset_info* out);
int yart_preset_count(void);
const char* yart_preset_name(int i);

/* resolve_dimensions (main.rs:166-186); 0 = "not given". */
void yart_resolve_dimensions(uint32_t default_w, uint32_t default_h, uint32_t w_override,
                             uint32_t h_override, uint32_t* w, uint32_t* h);
/* render()'s camera (main.rs:605-625) for a preset at a given size; vfov/aperture < 0 = default */
int yart_preset_camera(const yart_preset* p, uint32_t width, uint32_t height, double vfov,
                       double aperture, yart_camera* out);

/* ------------------------------------------------------------------------------------ */
/* Device side                                                                          */
/* ------------------------------------------------------------------------------------ */
typedef struct yart_ctx yart_ctx;

int yart_device_count(void);
int yart_ctx_create(int device, yart_ctx** out);
void yart_ctx_destroy(yart_ctx* ctx);
const char* yart_last_error(const yart_ctx* ctx);
/* Optional: run on an existing CUDA stream (cudaStream_t) instead of the context's own. */
int yart_ctx_set_stream(yart_ctx* ctx, void* cuda_stream);
int yart_ctx_synchronize(yart_ctx* ctx);

/* Which L4QBVH builder yart_ctx_set_scene uses for the meshes.  Both give the same tree byte for byte
 * (qbvh.rs:251-361); with YART_BUILDER_DEVICE (the default) the sorts run on the GPU and the tree never visits
 * the host. */
#define YART_BUILDER_HOST 0u
#define YART_BUILDER_DEVICE 1u
int yart_ctx_set_builder(yart_ctx* ctx, uint32_t builder);

/* L4QBVH::new on the GPU of `ctx`, copied back into a yart_qbvh so that yart_qbvh_get_info / _nodes / _tris
 * (and a comparison with yart_qbvh_build) work on it. */
int yart_qbvh_build_device(yart_ctx* ctx, const yart_trimesh* mesh, yart_qbvh** out);

/* Builds the QBVH of every mesh (see yart_ctx_set_builder), flattens and uploads everything.  Replaces the
 * construction of `world: Arc<HittableList>` + `lights` (main.rs:434-446). */
int yart_ctx_set_scene(yart_ctx* ctx, const yart_scene_desc* scene);

/* Batched `Hittable::hit(&self, &Ray, t_min, t_max) -> Option<HitRecord>` (hittable.rs:24).
 * target = mesh index: L4QBVH::hit (qbvh.rs:381-543) on that mesh alone;
 * target = YART_TARGET_WORLD: HittableList::hit (hittable.rs:66-79) over the whole world
 *   (constant media use the Philox stream of pixel=ray index, sample 0, bounce 1).
 * rays/hits: n elements, host pointers unless YART_FLAG_DEVICE_PTRS (device ray arrays must be 16-byte
 * aligned, which every cudaMalloc'ed array is).
 * Rays with zero, infinite or NaN components are legal input: a mesh target reproduces the reference's
 * NaN-ignoring min / max and its all-false NaN comparisons exactly, and so do the analytic objects.  The one
 * unspecified case is a ray with NaN components against a GROUP: the reference's BVHNode culls with NaN
 * comparisons (bvh.rs:151-215), so its own answer depends on the shape of its tree.
 * Host arrays go through in chunks of 2^19 rays, the upload of one chunk and the download of another overlapping the
 * kernels of a third on separate copy streams; page-locked (cudaHostAlloc / cudaHostRegister) arrays make that fully
 * asynchronous -- 0.92 Grays/s (f64 records) / 2.0 Grays/s (f32 records) end to end on a B200 behind PCIe 5, against
 * 0.52 / 0.99 unpipelined.  The call returns when `hits` is complete either way; stats->gpu_ms is the time of
 * the kernels alone (summed over the chunks), as with device arrays. */
int yart_closest_hit(yart_ctx* ctx, uint32_t target, const yart_ray* rays, uint64_t n,
                     double t_min, double t_max, uint32_t order, uint32_t flags,
                     yart_hit* hits, yart_stats* stats /* may be NULL */);

/* The same query on single-precision records (SURVEY.md 8(b) "f32 variant too"; halves the ray / hit streams of the
 * incoherent-ray sweep).  Each f32 ray is widened to f64 -- exactly -- and traced with the very same f64 arithmetic,
 * so the hit is the one yart_closest_hit returns for the widened ray, with t, u, v rounded to nearest f32 and obj_id /
 * front_face not reported.  Device ray arrays must be 8-byte aligned. */
int yart_closest_hit_f32(yart_ctx* ctx, uint32_t target, const yart_ray_f32* rays, uint64_t n,
                         float t_min, float t_max, uint32_t order, uint32_t flags,
                         yart_hit_f32* hits, yart_stats* stats /* may be NULL */);

/* The same query returning the whole HitRecord (hittable.rs:37-45) -- p, the stored normal, the texture u, v and the
 * material -- for hosts that shade on the CPU, and tracing each ray at its own Ray.time (ray.rs:4-9).
 *   t, obj_id, prim_id and front_face equal yart_closest_hit's for the same rays, target, order, t_min and t_max when
 *   `times` is NULL, bit for bit, in both orders and with all its documented quirks (constant media draw from the same
 *   Philox stream: pixel = ray index, sample 0, bounce 1).
 *   times: NULL (every ray at time 0, as yart_closest_hit traces) or n doubles, times[i] = ray i's Ray.time; it reaches
 *   MovingSphere::hit / center(time) (sphere.rs:149-198) both in the traversal and in the record.
 *   Every other field is what the reference's world.hit stores: wrappers applied (RotateY, Translate, FlipFace), the
 *   mesh's interpolated normals and uvs, a group member's own material, the constant-medium record (p = ray.at(t),
 *   normal (1,0,0), front_face 1, u = v = 0, the medium's phase-function material).  Sphere u, v are always computed.
 *   Fields from a libm call differ from the reference's glibc by its last bits: sphere u, v (acos / atan2) and the t
 *   and p of a constant-medium hit (log).
 * flags: YART_FLAG_DEVICE_PTRS (rays, times and records are device arrays; rays 16-byte aligned, times and records
 * 8-byte aligned) and YART_FLAG_COUNT_VISITS; any other bit is YART_ERR_INVALID.  Host arrays go through the chunk
 * pipeline of yart_closest_hit, the times uploaded with the rays.  stats as in yart_closest_hit: the one record export
 * launch per chunk counts in kernel_launches, not in trace_launches.  There is no f32 variant. */
int yart_closest_hit_records(yart_ctx* ctx, uint32_t target, const yart_ray* rays, const double* times /* may be NULL */,
                             uint64_t n, double t_min, double t_max, uint32_t order, uint32_t flags,
                             yart_hit_record* records, yart_stats* stats /* may be NULL */);

/* Batched occlusion query (Embree's rtcOccluded, an OptiX any-hit that terminates on the first hit): occluded[i] = 1
 * if ray i hits anything of `target` (a mesh index or YART_TARGET_WORLD) that yart_closest_hit(..., YART_ORDER_REFERENCE,
 * ...) would report with the same t_min / t_max, else 0 -- exactly, for every ray, with all the reference's quirks
 * (flat leaves never entered, NaN slabs, the strict `t_max > t`, constant media drawing the same Philox numbers).
 * The traversal stops at the first hit it finds; nothing but the flag is computed.  There is no order argument: the
 * answer does not depend on the order the tree is walked in.  For shadow rays toward a point q from p, use the
 * direction q - p and a t_max just below 1.
 * flags: YART_FLAG_DEVICE_PTRS only (rays and occluded are then device arrays; rays aligned as for
 * yart_closest_hit); any other bit is YART_ERR_INVALID.  Host arrays go through the same chunk pipeline as
 * yart_closest_hit.  stats (may be NULL): rays, gpu_ms = trace_ms, kernel_launches = trace_launches; the visit
 * counters stay 0. */
int yart_occluded(yart_ctx* ctx, uint32_t target, const yart_ray* rays, uint64_t n, double t_min, double t_max,
                  uint32_t flags, uint8_t* occluded, yart_stats* stats /* may be NULL */);
/* The same on single-precision ray records, widened exactly as in yart_closest_hit_f32. */
int yart_occluded_f32(yart_ctx* ctx, uint32_t target, const yart_ray_f32* rays, uint64_t n, float t_min,
                      float t_max, uint32_t flags, uint8_t* occluded, yart_stats* stats /* may be NULL */);

/* Batched `render(config)` sample loop (main.rs:650-708) for samples
 * [sample_begin, sample_end): adds, per pixel and in sample order, the sanitised XYZ of each
 * sample (sanitize_sample_xyz main.rs:448-459) into film_xyz[height][width][3] (f64; host
 * pointer unless YART_FLAG_DEVICE_PTRS).  The film is NOT cleared: call with a zeroed
 * buffer, or chain calls to continue a render. */
int yart_render(yart_ctx* ctx, const yart_camera* camera, const yart_render_opts* opts,
                double* film_xyz, yart_stats* stats /* may be NULL */);

/* Per-pixel finalisation (main.rs:710-718): XYZ * (720-360)/(106.856895*spp) -> into_rgb ->
 * sRGB OETF -> (256*clamp(c,0,0.999)) as u8, alpha 255.  Host buffers; runs on the GPU. */
int yart_film_finalize(yart_ctx* ctx, const double* film_xyz, uint32_t width, uint32_t height,
                       uint32_t spp, uint32_t flags, uint8_t* rgba8);

/* The film as LINEAR RGB, the HDR colour input of a denoiser: yart_film_finalize's (r, g, b) after into_rgb and
 * before the sRGB OETF and the clamp, i.e. XYZ * (720-360)/(106.856895*spp) -> into_rgb, computed in f64 and
 * rounded to f32.  Pixels outside the reference's 8x8 tiles are 0.  rgb: [height][width][3].  flags:
 * YART_FLAG_DEVICE_PTRS (film_xyz and rgb are device arrays). */
int yart_film_finalize_linear(yart_ctx* ctx, const double* film_xyz, uint32_t width, uint32_t height,
                              uint32_t spp, uint32_t flags, float* rgb);

/* Auxiliary images (AOVs) for a denoiser.  Each plane is a film: [height][width][3] f64, added to like film_xyz. */
typedef struct yart_aov_planes {
  double* albedo;  /* [height][width][3] or NULL */
  double* normal;  /* [height][width][3] or NULL */
  double* depth;   /* [height][width][3] or NULL: {sum of distance over the samples that hit, samples that hit, samples} */
} yart_aov_planes;

/* What each camera sample of yart_render first hits, summed per pixel: the albedo, normal and distance planes that
 * denoisers (Open Image Denoise, the OptiX denoiser) take beside the linear colour of yart_film_finalize_linear.
 *   Samples: [sample_begin, sample_end) of every pixel, with yart_render's camera rays: the same Philox (pixel, sample)
 *   draws for jitter, lens, wavelength and time, and the same 8x8 tiles.  Pixels the reference never samples get
 *   nothing, not even a sample count.
 *   First hit: the render's bounce-1 world.hit(ray, 0.001, inf), bit for bit: the same `order`, the ray's own time
 *   (MovingSphere), constant media drawing at (pixel, sample, bounce 1).  AOV sample s of pixel p describes exactly
 *   the surface beauty sample s reached first.
 *   Accumulation: per pixel and in sample order, like the film.  Chaining calls over consecutive sample ranges, and
 *   any batch_spp, give the same bits as one call.  yart_film_create / _read / _reduce work on the planes unchanged.
 *   Per sample, with h the first hit's HitRecord:
 *     albedo  an RGB from h's material, each channel clamped to [0, 1] (NaN to 0): Lambertian, Metal and Isotropic:
 *             the RGB their texture hands to RGB::reflect at (u, v, p) -- checker a / b, the image texel, the solid
 *             colour, or the noise scalar times white; Dielectric: (1, 1, 1); DiffuseLight: its emit texture's RGB
 *             when h.front_face, else 0; no material: 0; a miss: background_rgb.
 *     normal  h.normal / |h.normal| (world space, face-oriented as the reference stores it); 0 for a miss, a
 *             constant-medium hit, and a zero or non-finite length.  |n| = sqrt(x*x + y*y + z*z), in that order.
 *     depth   {t * |d|, 1, 1} for a hit, {0, 0, 1} for a miss: the Euclidean distance from the ray's origin on the
 *             lens (d is the camera ray's direction, not normalised; |d| as for the normal).
 *   Values from a libm call differ from the reference's glibc in the last bits where they feed the planes: sphere u, v
 *   read by an image texture (acos / atan2), a checker's sin, noise, and a constant medium's log.
 * opts: the struct of the beauty call may be passed as it is.  The sampling flags are accepted and change nothing
 * (none of them changes a camera ray or its first hit); max_depth is validated as in yart_render and otherwise unused.
 * Flags: YART_FLAG_DEVICE_PTRS (the planes are device arrays, 8-byte aligned), YART_FLAG_COUNT_VISITS as in yart_render.
 * All three planes NULL is YART_ERR_INVALID.
 * stats (may be NULL): rays = camera rays traced, paths = samples started, trace_ms / trace_launches = the closest-hit
 * passes; max_bounce is 1 when anything was traced. */
int yart_render_aovs(yart_ctx* ctx, const yart_camera* camera, const yart_render_opts* opts,
                     const yart_aov_planes* planes, yart_stats* stats /* may be NULL */);

typedef struct yart_denoise_opts {
  uint32_t levels;      /* a-trous levels L, 1..10; 0 = 5 */
  uint32_t flags;       /* YART_FLAG_DEVICE_PTRS only */
  double sigma_color;   /* <= 0: 8 */
  double sigma_normal;  /* <= 0: 0.3 */
  double sigma_depth;   /* <= 0: 0.05 */
} yart_denoise_opts;

/* A denoised image from a film and the planes of yart_render_aovs: the edge-avoiding a-trous wavelet filter of
 * Dammertz, Sewtz, Hanika and Lensch (HPG 2010), guided by albedo, normal and distance, on the GPU.  Everything is f64
 * in a fixed order without libm or FMA, so tests/denoise_ref.py (numpy) reproduces `rgb` bit for bit.  Per pixel p:
 *   Prepare:  p is valid iff depth[p][2] > 0 (it has AOV samples); invalid pixels are never neighbours and output 0.
 *     lin = the film as yart_film_finalize_linear computes it (f64, not rounded), a = albedo / depth[2],
 *     n = normal / depth[2], hit = depth[1] > 0, z = depth[0] / depth[1] if hit, m = a + 1/128, c = lin / m
 *     (demodulation, per channel).
 *   Level i = 0 .. L-1, step s = 2^i: taps (dy, dx) in {-2..2}^2, row-major, at (y + dy*s, x + dx*s); taps outside the
 *     image or at invalid pixels are skipped.  h = H[dy] * H[dx], H = {1/16, 1/4, 3/8, 1/4, 1/16}.  The centre tap has
 *     weight h.  Another tap q is skipped if exactly one of p, q hits; else its weight is h * r(x) with
 *       x = dc * kc + dn * kn (+ dz * dz * iz if both hit),
 *       dc = ((c_q0-c_p0)^2 + (c_q1-c_p1)^2) + (c_q2-c_p2)^2, dn likewise for n, dz = z_q - z_p,
 *       kc = 4^i / (sigma_color * sigma_color) (the colour term tightens by 4 per level), kn = 1 / (sigma_normal *
 *       sigma_normal), iz = 1 / ((sigma_depth * sigma_depth * z_p) * z_p),
 *       r(x) = (1 + x * 0.125)^-8 as t = 1 / (1 + x * 0.125); t = t * t; t = t * t; t = t * t (a stand-in for exp(-x)).
 *     In tap order W += w, S += w * c_q; then c_p = S / W.
 *   Finish: out = c * m (remodulation).  rgb: out rounded to f32; rgba8: yart_film_finalize's sRGB curve and clamp
 *     applied to out, alpha 255.  Invalid pixels are 0 in both, alpha included.
 * film_xyz: [height][width][3] f64 as yart_render fills it, with spp samples per pixel (>= 1).  planes: all three
 * required, as yart_render_aovs fills them (any sample count; films and planes combined by yart_film_reduce are valid
 * input, so a multi-GPU host denoises on the root).  The inputs are not modified.  opts: NULL = all defaults with host
 * arrays.  With YART_FLAG_DEVICE_PTRS every array is a device array on ctx's GPU (f64 ones 8-byte aligned, rgb 4-byte
 * aligned); any other flag bit is YART_ERR_INVALID, as are levels > 10, a non-finite sigma, width * height >= 2^32,
 * spp 0 and both outputs NULL.  Scratch of 121 bytes a pixel stays on the context for the next call.
 * stats (may be NULL): gpu_ms and kernel_launches (L + 2); the other fields are 0. */
int yart_denoise(yart_ctx* ctx, const double* film_xyz, uint32_t spp, const yart_aov_planes* planes, uint32_t width,
                 uint32_t height, const yart_denoise_opts* opts, float* rgb /* or NULL */, uint8_t* rgba8 /* or NULL */,
                 yart_stats* stats /* may be NULL */);

/* Camera rays exactly as the render loop generates them (main.rs:690-698, camera.rs:82-94):
 * one ray per (pixel, sample) in [sample_begin, sample_end), pixel-major.  For parity tests
 * and for dumping the ray distribution the renderer really sees. */
int yart_generate_camera_rays(yart_ctx* ctx, const yart_camera* camera,
                              const yart_render_opts* opts, yart_ray* rays_host,
                              double* wavelength_host /* may be NULL */,
                              double* time_host /* may be NULL */);

/* ------------------------------------------------------------------------------------ */
/* Multi-GPU: sample-range sharding + one NCCL reduce of the film                       */
/* ------------------------------------------------------------------------------------ */
/* The reference shards its frame into 64 tiles over a thread pool and gathers them through an mpsc channel
 * (main.rs:629-646, 746-760).  Here every GPU renders its own SAMPLE RANGE of every pixel (yart_render_opts
 * sample_begin / sample_end; exact because sanitize_sample_xyz acts per sample, main.rs:700-707) into its own
 * device-resident f64 film, and the films are summed onto the root with one ncclReduce over NVLink -- in place, on
 * the context's stream, in the very buffer the render kernels accumulate into.  NCCL is loaded at run time
 * (libnccl.so.2, or $YART_NCCL_LIB); without it these calls return YART_ERR_UNSUPPORTED.
 *
 *   one process per GPU (torchrun, MPI, N host processes of any kind):
 *       rank 0: yart_comm_unique_id(id); ship the 128 bytes to the other ranks by any means;
 *       every rank: yart_comm_init_rank(ctx, id, rank, n_ranks, &comm)
 *   one process driving N GPUs (one host thread per context while rendering):
 *       yart_comm_init(ctxs, n, &comm)
 *   then, per frame:  yart_film_create / yart_film_clear -> yart_render(..., YART_FLAG_DEVICE_PTRS) with this rank's
 *       sample range -> yart_film_reduce(comm, films, w, h, root) -> on the root: yart_film_finalize / yart_film_read. */
typedef struct yart_comm yart_comm;
#define YART_COMM_ID_BYTES 128

int yart_comm_unique_id(uint8_t id[YART_COMM_ID_BYTES]);
int yart_comm_init_rank(yart_ctx* ctx, const uint8_t id[YART_COMM_ID_BYTES], int rank, int n_ranks, yart_comm** out);
int yart_comm_init(yart_ctx* const* ctxs, int n, yart_comm** out); /* rank i = ctxs[i]; all GPUs distinct */
void yart_comm_destroy(yart_comm* comm);
int yart_comm_info(const yart_comm* comm, int* n_ranks, int* n_local, int* first_local_rank, int* nccl_version);
const char* yart_comm_last_error(const yart_comm* comm);

/* dev_films: one device pointer per LOCAL rank (1 with yart_comm_init_rank, n with yart_comm_init), each a
 * [height][width][3] f64 film on that rank's GPU.  root >= 0: the sum lands in root's film (the others keep their
 * partial sums); root < 0: all-reduce.  Asynchronous on each context's stream. */
int yart_film_reduce(yart_comm* comm, double* const* dev_films, uint32_t width, uint32_t height, int root);

/* Device-resident films for hosts without CUDA of their own: zeroed on creation; pass them to yart_render /
 * yart_film_finalize with YART_FLAG_DEVICE_PTRS. */
int yart_film_create(yart_ctx* ctx, uint32_t width, uint32_t height, double** dev_film);
int yart_film_clear(yart_ctx* ctx, double* dev_film, uint32_t width, uint32_t height);
int yart_film_read(yart_ctx* ctx, const double* dev_film, uint32_t width, uint32_t height, double* host_film);
void yart_film_destroy(yart_ctx* ctx, double* dev_film);

/* The rays the renderer itself traces -- every `world.hit` of every path of samples [sample_begin, sample_end)
 * (main.rs:548) -- in the order the closest-hit kernels see them: batch by batch, bounce by bounce, queue order within
 * a bounce.  No film is produced.  rays: room for `cap` records (host, or device with YART_FLAG_DEVICE_PTRS in
 * opts->flags); *n_out = the number of rays traced, which may exceed cap (only the first cap are stored).  For the
 * "path-ray set" of the closest-hit sweep (SURVEY.md 8(d)) and for parity tests on the renderer's own ray distribution. */
int yart_dump_path_rays(yart_ctx* ctx, const yart_camera* camera, const yart_render_opts* opts, yart_ray* rays,
                        uint64_t cap, uint64_t* n_out);

/* Roofline denominator for the closest-hit stage (SURVEY.md 8(d): "a measured L2 fetch peak"): every thread
 * fetches `fetches_per_thread` whole 128-byte lines (four 256-bit loads, like one QBVH node visit) at
 * independent random positions of a `table_bytes` table, with the occupancy (20 warps per SM) and cache carveout the
 * traversal kernel runs at (mode 0) or at full occupancy (mode 1).  Returns the sustained rate in GB/s.  A 7 MB table is the david
 * tree: L2-resident, partly L1-resident.  Modes 2 / 3: the same occupancies, but the four lanes of a quad fetch the four
 * sectors of ONE line with one 256-bit load each -- the roof of a four-lanes-per-ray traversal (DESIGN.md section 7). */
int yart_measure_fetch_peak(yart_ctx* ctx, uint64_t table_bytes, uint32_t fetches_per_thread, uint32_t mode,
                            double* gbytes_per_s);

/* Page-lock / unlock a host array the caller owns (cudaHostRegister / cudaHostUnregister), for hosts that hold their
 * rays, hits or film in ordinary heap memory (a Rust Vec) and do not link the CUDA runtime themselves.  With
 * registered arrays the chunk pipeline of yart_closest_hit* and the film copies of yart_render run at the PCIe rate
 * (0.8-0.9 Grays/s end to end for f64 ray records against 0.15 from pageable memory).  Registration costs time in
 * proportion to the size: do it once per buffer, not per call.  The array must stay allocated until it is unregistered. */
int yart_host_register(yart_ctx* ctx, void* ptr, uint64_t bytes);
int yart_host_unregister(yart_ctx* ctx, void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* YART_H */
