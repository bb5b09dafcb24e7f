//! Raw bindings to `include/yart.h` (ABI version 1), written by hand: every struct is `#[repr(C)]` and
//! field-for-field the C one, every entry point of the header is declared below (tests/test_host.py checks the
//! list against the header).  NOT compiled in the repository's build environment (no Rust toolchain there);
//! the same ABI is exercised from C (`examples/yart_main.c`) and Python (`yet-another-raytracer_b200/__init__.py`).
//!
//! Which reference item each call replaces is listed in INTEGRATION.md; in short
//! `world.hit(ray, 0.001, inf)` (main.rs:548) -> `yart_closest_hit`, `render(config)` (main.rs:590) -> `yart_render`.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const YART_ABI_VERSION: u32 = 2;
pub const YART_OK: c_int = 0;
pub const YART_ERR_INVALID: c_int = -1;
pub const YART_ERR_CUDA: c_int = -2;
pub const YART_ERR_NOMEM: c_int = -3;
pub const YART_ERR_IO: c_int = -4;
pub const YART_ERR_UNSUPPORTED: c_int = -5;

pub const YART_OBJ_SPHERE: u32 = 0;
pub const YART_OBJ_MOVING_SPHERE: u32 = 1;
pub const YART_OBJ_XY_RECT: u32 = 2;
pub const YART_OBJ_XZ_RECT: u32 = 3;
pub const YART_OBJ_YZ_RECT: u32 = 4;
pub const YART_OBJ_BOX: u32 = 5;
pub const YART_OBJ_TRIANGLE: u32 = 6;
pub const YART_OBJ_MESH: u32 = 7;
pub const YART_OBJ_GROUP: u32 = 8;
pub const YART_WRAP_ROTATE_Y: u32 = 1;
pub const YART_WRAP_TRANSLATE: u32 = 2;
pub const YART_WRAP_FLIP_FACE: u32 = 4;
pub const YART_WRAP_MEDIUM: u32 = 8;
pub const YART_MAT_NONE: u32 = 0;
pub const YART_MAT_LAMBERTIAN: u32 = 1;
pub const YART_MAT_METAL: u32 = 2;
pub const YART_MAT_DIELECTRIC: u32 = 3;
pub const YART_MAT_DIFFUSE_LIGHT: u32 = 4;
pub const YART_MAT_ISOTROPIC: u32 = 5;
pub const YART_TEX_SOLID: u32 = 0;
pub const YART_TEX_CHECKER: u32 = 1;
pub const YART_TEX_NOISE: u32 = 2;
pub const YART_TEX_IMAGE: u32 = 3;
pub const YART_MISS: u32 = 0xFFFF_FFFF;
pub const YART_TARGET_WORLD: u32 = 0xFFFF_FFFF;
pub const YART_ORDER_REFERENCE: u32 = 0;
pub const YART_ORDER_NEAR: u32 = 1;
pub const YART_FLAG_DEVICE_PTRS: u32 = 1;
pub const YART_FLAG_COUNT_VISITS: u32 = 2;
pub const YART_FLAG_UNBIASED_LIGHT_PICK: u32 = 4;
pub const YART_FLAG_RUSSIAN_ROULETTE: u32 = 8;
pub const YART_FLAG_DEPTH_ZERO_BLACK: u32 = 16;
pub const YART_FLAG_NEXT_EVENT: u32 = 32;
pub const YART_COMM_ID_BYTES: usize = 128;
pub const YART_BUILDER_HOST: u32 = 0;
pub const YART_BUILDER_DEVICE: u32 = 1;

#[repr(C)] pub struct yart_ctx { _private: [u8; 0] }
#[repr(C)] pub struct yart_comm { _private: [u8; 0] }
#[repr(C)] pub struct yart_preset { _private: [u8; 0] }
#[repr(C)] pub struct yart_objfile { _private: [u8; 0] }
#[repr(C)] pub struct yart_qbvh { _private: [u8; 0] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_trimesh { pub n_tris: u32, pub _pad: u32, pub positions: *const f32, pub normals: *const f64, pub uvs: *const f32 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_object {
    pub kind: u32, pub wrap: u32, pub material: u32, pub index: u32,
    pub p: [f64; 24], pub sin_theta: f64, pub cos_theta: f64, pub offset: [f64; 3], pub neg_inv_density: f64,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_group { pub members: *const yart_object, pub n_members: u32, pub _pad: u32 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_material { pub kind: u32, pub texture: u32, pub fuzz: f64, pub sellmeier_b: [f64; 3], pub sellmeier_c: [f64; 3] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_texture {
    pub kind: u32, pub noise_type: u32, pub perlin: u32, pub image: u32,
    pub rgb_a: [f64; 3], pub rgb_b: [f64; 3], pub scale: f64,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_perlin {
    pub ranfloat: [f64; 256], pub ranvec: [[f64; 3]; 256],
    pub perm_x: [i32; 256], pub perm_y: [i32; 256], pub perm_z: [i32; 256],
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_image { pub rgb8: *const u8, pub width: u32, pub height: u32 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_scene_desc {
    pub objects: *const yart_object, pub n_objects: u32, pub _p0: u32,
    pub lights: *const yart_object, pub n_lights: u32, pub _p1: u32,
    pub meshes: *const yart_trimesh, pub n_meshes: u32, pub _p2: u32,
    pub groups: *const yart_group, pub n_groups: u32, pub _p3: u32,
    pub materials: *const yart_material, pub n_materials: u32, pub _p4: u32,
    pub textures: *const yart_texture, pub n_textures: u32, pub _p5: u32,
    pub perlins: *const yart_perlin, pub n_perlins: u32, pub _p6: u32,
    pub images: *const yart_image, pub n_images: u32, pub _p7: u32,
    pub background_rgb: [f64; 3],
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_camera {
    pub lookfrom: [f64; 3], pub lookat: [f64; 3], pub vup: [f64; 3], pub vfov_degrees: f64,
    pub aspect_ratio: f64, pub aperture: f64, pub focus_dist: f64, pub time0: f64, pub time1: f64,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_ray { pub origin: [f64; 3], pub direction: [f64; 3] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_ray_f32 { pub origin: [f32; 3], pub direction: [f32; 3] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_hit_f32 { pub t: f32, pub u: f32, pub v: f32, pub prim_id: u32 }

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_hit { pub t: f64, pub u: f64, pub v: f64, pub prim_id: u32, pub obj_id: u32, pub front_face: u32, pub _pad: u32 }

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct yart_stats {
    pub rays: u64, pub paths: u64, pub node_visits: u64, pub tri_tests: u64, pub kernel_launches: u64,
    pub gpu_ms: f64, pub trace_ms: f64, pub max_bounce: u32, pub trace_launches: u32,
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct yart_render_opts {
    pub width: u32, pub height: u32, pub sample_begin: u32, pub sample_end: u32, pub max_depth: u32,
    pub order: u32, pub batch_spp: u32, pub flags: u32, pub seed: u64,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_qbvh_info {
    pub n_nodes: u32, pub n_leaves: u32, pub n_tris: u32, pub height: u32, pub root: u32, pub max_stack: u32,
    pub _pad0: u32, pub _pad1: u32, pub bbox_min: [f64; 3], pub bbox_max: [f64; 3],
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct yart_preset_info {
    pub width: u32, pub height: u32, pub samples_per_pixel: u32, pub max_depth: u32, pub workers: u32, pub _pad: u32,
    pub vfov: f64, pub aperture: f64, pub lookfrom: [f64; 3], pub lookat: [f64; 3], pub output_filename: [c_char; 64],
}

extern "C" {
    pub fn yart_version() -> *const c_char;
    pub fn yart_last_error_global() -> *const c_char;
    // host front end (no GPU needed)
    pub fn yart_obj_load(path: *const c_char, out: *mut *mut yart_objfile) -> c_int;
    pub fn yart_obj_free(obj: *mut yart_objfile);
    pub fn yart_obj_trimesh(obj: *const yart_objfile, out: *mut yart_trimesh) -> c_int;
    pub fn yart_qbvh_build(mesh: *const yart_trimesh, out: *mut *mut yart_qbvh) -> c_int;
    pub fn yart_qbvh_free(q: *mut yart_qbvh);
    pub fn yart_qbvh_get_info(q: *const yart_qbvh, out: *mut yart_qbvh_info) -> c_int;
    pub fn yart_qbvh_nodes(q: *const yart_qbvh) -> *const c_void;
    pub fn yart_qbvh_tris(q: *const yart_qbvh) -> *const c_void;
    pub fn yart_qbvh_shade(q: *const yart_qbvh) -> *const c_void;
    pub fn yart_preset_build(name: *const c_char, assets_dir: *const c_char, seed: u64, out: *mut *mut yart_preset) -> c_int;
    pub fn yart_preset_free(p: *mut yart_preset);
    pub fn yart_preset_note(p: *const yart_preset) -> *const c_char;
    pub fn yart_preset_scene(p: *const yart_preset) -> *const yart_scene_desc;
    pub fn yart_preset_get_info(p: *const yart_preset, out: *mut yart_preset_info) -> c_int;
    pub fn yart_preset_count() -> c_int;
    pub fn yart_preset_name(i: c_int) -> *const c_char;
    pub fn yart_resolve_dimensions(default_w: u32, default_h: u32, w_override: u32, h_override: u32, w: *mut u32, h: *mut u32);
    pub fn yart_preset_camera(p: *const yart_preset, width: u32, height: u32, vfov: f64, aperture: f64, out: *mut yart_camera) -> c_int;
    // device side
    pub fn yart_device_count() -> c_int;
    pub fn yart_ctx_create(device: c_int, out: *mut *mut yart_ctx) -> c_int;
    pub fn yart_ctx_destroy(ctx: *mut yart_ctx);
    pub fn yart_last_error(ctx: *const yart_ctx) -> *const c_char;
    pub fn yart_ctx_set_stream(ctx: *mut yart_ctx, cuda_stream: *mut c_void) -> c_int;
    pub fn yart_ctx_synchronize(ctx: *mut yart_ctx) -> c_int;
    pub fn yart_ctx_set_builder(ctx: *mut yart_ctx, builder: u32) -> c_int;
    pub fn yart_qbvh_build_device(ctx: *mut yart_ctx, mesh: *const yart_trimesh, out: *mut *mut yart_qbvh) -> c_int;
    pub fn yart_ctx_set_scene(ctx: *mut yart_ctx, scene: *const yart_scene_desc) -> c_int;
    pub fn yart_closest_hit(ctx: *mut yart_ctx, target: u32, rays: *const yart_ray, n: u64, t_min: f64, t_max: f64,
                            order: u32, flags: u32, hits: *mut yart_hit, stats: *mut yart_stats) -> c_int;
    pub fn yart_closest_hit_f32(ctx: *mut yart_ctx, target: u32, rays: *const yart_ray_f32, n: u64, t_min: f32, t_max: f32,
                                order: u32, flags: u32, hits: *mut yart_hit_f32, stats: *mut yart_stats) -> c_int;
    pub fn yart_occluded(ctx: *mut yart_ctx, target: u32, rays: *const yart_ray, n: u64, t_min: f64, t_max: f64,
                         flags: u32, occluded: *mut u8, stats: *mut yart_stats) -> c_int;
    pub fn yart_occluded_f32(ctx: *mut yart_ctx, target: u32, rays: *const yart_ray_f32, n: u64, t_min: f32, t_max: f32,
                             flags: u32, occluded: *mut u8, stats: *mut yart_stats) -> c_int;
    pub fn yart_render(ctx: *mut yart_ctx, camera: *const yart_camera, opts: *const yart_render_opts, film_xyz: *mut f64,
                       stats: *mut yart_stats) -> c_int;
    pub fn yart_film_finalize(ctx: *mut yart_ctx, film_xyz: *const f64, width: u32, height: u32, spp: u32, flags: u32,
                              rgba8: *mut u8) -> c_int;
    pub fn yart_generate_camera_rays(ctx: *mut yart_ctx, camera: *const yart_camera, opts: *const yart_render_opts,
                                     rays_host: *mut yart_ray, wavelength_host: *mut f64, time_host: *mut f64) -> c_int;
    pub fn yart_dump_path_rays(ctx: *mut yart_ctx, camera: *const yart_camera, opts: *const yart_render_opts,
                               rays: *mut yart_ray, cap: u64, n_out: *mut u64) -> c_int;
    pub fn yart_measure_fetch_peak(ctx: *mut yart_ctx, table_bytes: u64, fetches_per_thread: u32, mode: u32,
                                   gbytes_per_s: *mut f64) -> c_int;
    // page-lock a Vec the host owns, so that host-array queries and film copies run at the PCIe rate
    pub fn yart_host_register(ctx: *mut yart_ctx, ptr: *mut c_void, bytes: u64) -> c_int;
    pub fn yart_host_unregister(ctx: *mut yart_ctx, ptr: *mut c_void) -> c_int;
    // multi-GPU: sample-range sharding + one in-place NCCL reduce of the f64 film (replaces main.rs:746-760)
    pub fn yart_comm_unique_id(id: *mut u8) -> c_int; // YART_COMM_ID_BYTES bytes
    pub fn yart_comm_init_rank(ctx: *mut yart_ctx, id: *const u8, rank: c_int, n_ranks: c_int, out: *mut *mut yart_comm) -> c_int;
    pub fn yart_comm_init(ctxs: *const *mut yart_ctx, n: c_int, out: *mut *mut yart_comm) -> c_int;
    pub fn yart_comm_destroy(comm: *mut yart_comm);
    pub fn yart_comm_info(comm: *const yart_comm, n_ranks: *mut c_int, n_local: *mut c_int, first_local_rank: *mut c_int,
                          nccl_version: *mut c_int) -> c_int;
    pub fn yart_comm_last_error(comm: *const yart_comm) -> *const c_char;
    pub fn yart_film_reduce(comm: *mut yart_comm, dev_films: *const *mut f64, width: u32, height: u32, root: c_int) -> c_int;
    pub fn yart_film_create(ctx: *mut yart_ctx, width: u32, height: u32, dev_film: *mut *mut f64) -> c_int;
    pub fn yart_film_clear(ctx: *mut yart_ctx, dev_film: *mut f64, width: u32, height: u32) -> c_int;
    pub fn yart_film_read(ctx: *mut yart_ctx, dev_film: *const f64, width: u32, height: u32, host_film: *mut f64) -> c_int;
    pub fn yart_film_destroy(ctx: *mut yart_ctx, dev_film: *mut f64);
}
