//! Safe wrapper over `yart-sys` -- what the reference (raytracer/src/) would depend on.  NOT compiled in the
//! repository's build environment (no Rust toolchain there).
//!
//! `GpuScene` plays the part of `world: Arc<HittableList>` (main.rs:434-446): `hit` has the shape of
//! `Hittable::hit(&self, &Ray, t_min, t_max) -> Option<HitRecord>` (hittable.rs:24) for drop-in testing, `hit_many`
//! is the batched form the GPU is for, `hit_records` / `hit_record` return the whole `HitRecord`, `render` replaces the tile loop of `render()` (main.rs:629-760), `render_aovs` gives a denoiser its inputs, `denoise` renders and denoises on the GPU.
use std::ffi::{CStr, CString};
use std::ptr;
use yart_sys as sys;

#[derive(Debug)]
pub struct Error { pub code: i32, pub message: String }
pub type Result<T> = std::result::Result<T, Error>;

#[derive(Clone, Copy, Debug)]
pub struct Ray { pub origin: [f64; 3], pub direction: [f64; 3] }

/// The part of the reference's `HitRecord` the closest-hit query returns (the shade stage rebuilds the rest).
#[derive(Clone, Copy, Debug)]
pub struct Hit { pub t: f64, pub u: f64, pub v: f64, pub prim_id: u32, pub obj_id: u32, pub front_face: bool }

/// The reference's whole `HitRecord` (hittable.rs:37-45) as `world.hit` returns it, plus the ids of `Hit`:
/// `p`, the stored (face-oriented, unnormalised) normal, the texture `u, v`, and `material`, an index into the scene's
/// material table (a group hit: the member's; `YART_MISS` for a bare mesh).
#[derive(Clone, Copy, Debug)]
pub struct Record {
    pub t: f64, pub p: [f64; 3], pub normal: [f64; 3], pub u: f64, pub v: f64,
    pub material: u32, pub front_face: bool, pub obj_id: u32, pub prim_id: u32,
}

pub struct GpuScene { ctx: *mut sys::yart_ctx, preset: *mut sys::yart_preset }

// One context per host thread (yart.h); the scene itself is immutable after construction like the reference's
// `Hittable: Send + Sync` objects, but calls go through the context, so no `Sync`.
unsafe impl Send for GpuScene {}

impl GpuScene {
    fn ctx_err(&self, code: i32) -> Error {
        let message = unsafe { CStr::from_ptr(sys::yart_last_error(self.ctx)) }.to_string_lossy().into_owned();
        Error { code, message }
    }
    fn global_err(code: i32) -> Error {
        let message = unsafe { CStr::from_ptr(sys::yart_last_error_global()) }.to_string_lossy().into_owned();
        Error { code, message }
    }

    /// `build_scene_preset` (main.rs:211-432) on GPU `device`; `name` is the kebab-case `--scene` value.
    pub fn from_preset(name: &str, assets_dir: &str, seed: u64, device: i32) -> Result<GpuScene> {
        let (name, assets) = (CString::new(name).unwrap(), CString::new(assets_dir).unwrap());
        let mut s = GpuScene { ctx: ptr::null_mut(), preset: ptr::null_mut() };
        unsafe {
            let rc = sys::yart_preset_build(name.as_ptr(), assets.as_ptr(), seed, &mut s.preset);
            if rc != 0 { return Err(Self::global_err(rc)); }
            let rc = sys::yart_ctx_create(device, &mut s.ctx);
            if rc != 0 { return Err(Self::global_err(rc)); } // no CPU fallback: YART_ERR_CUDA without a B200
            let rc = sys::yart_ctx_set_scene(s.ctx, sys::yart_preset_scene(s.preset));
            if rc != 0 { return Err(s.ctx_err(rc)); }
        }
        Ok(s)
    }

    /// Batched `world.hit(ray, t_min, t_max)` (main.rs:548): one result per ray, `None` = miss.
    pub fn hit_many(&self, rays: &[Ray], t_min: f64, t_max: f64) -> Result<Vec<Option<Hit>>> {
        let raw: Vec<sys::yart_ray> = rays.iter().map(|r| sys::yart_ray { origin: r.origin, direction: r.direction }).collect();
        let mut hits = vec![sys::yart_hit { t: 0.0, u: 0.0, v: 0.0, prim_id: 0, obj_id: 0, front_face: 0, _pad: 0 }; rays.len()];
        let rc = unsafe {
            sys::yart_closest_hit(self.ctx, sys::YART_TARGET_WORLD, raw.as_ptr(), raw.len() as u64, t_min, t_max,
                                  sys::YART_ORDER_NEAR, 0, hits.as_mut_ptr(), ptr::null_mut())
        };
        if rc != 0 { return Err(self.ctx_err(rc)); }
        Ok(hits.iter().map(|h| if h.obj_id == sys::YART_MISS { None } else {
            Some(Hit { t: h.t, u: h.u, v: h.v, prim_id: h.prim_id, obj_id: h.obj_id, front_face: h.front_face != 0 })
        }).collect())
    }

    /// Batched `world.hit(ray, t_min, t_max)` returning whole records (`yart_closest_hit_records`), each ray traced at
    /// its own `Ray.time` (`times`: one per ray; `None` = every ray at time 0).  `None` in the result = miss.
    pub fn hit_records(&self, rays: &[Ray], times: Option<&[f64]>, t_min: f64, t_max: f64) -> Result<Vec<Option<Record>>> {
        if let Some(t) = times { assert_eq!(t.len(), rays.len()); }
        let raw: Vec<sys::yart_ray> = rays.iter().map(|r| sys::yart_ray { origin: r.origin, direction: r.direction }).collect();
        let mut recs = vec![sys::yart_hit_record { t: 0.0, p: [0.0; 3], normal: [0.0; 3], u: 0.0, v: 0.0, material: 0,
                                                   front_face: 0, obj_id: 0, prim_id: 0 }; rays.len()];
        let rc = unsafe {
            sys::yart_closest_hit_records(self.ctx, sys::YART_TARGET_WORLD, raw.as_ptr(), times.map_or(ptr::null(), |t| t.as_ptr()),
                                          raw.len() as u64, t_min, t_max, sys::YART_ORDER_NEAR, 0, recs.as_mut_ptr(),
                                          ptr::null_mut())
        };
        if rc != 0 { return Err(self.ctx_err(rc)); }
        Ok(recs.iter().map(|r| if r.obj_id == sys::YART_MISS { None } else {
            Some(Record { t: r.t, p: r.p, normal: r.normal, u: r.u, v: r.v, material: r.material, front_face: r.front_face != 0,
                          obj_id: r.obj_id, prim_id: r.prim_id })
        }).collect())
    }

    /// `Hittable::hit` for a single ray at time `time` with the whole record -- for drop-in tests; use `hit_records` for work.
    pub fn hit_record(&self, ray: &Ray, time: f64, t_min: f64, t_max: f64) -> Result<Option<Record>> {
        Ok(self.hit_records(std::slice::from_ref(ray), Some(std::slice::from_ref(&time)), t_min, t_max)?.pop().flatten())
    }

    /// Batched occlusion query (`yart_occluded`): `true` where the ray hits anything of the world in (t_min, t_max) --
    /// exactly where `hit_many` would return `Some` -- found with a traversal that stops at the first hit.  Shadow rays
    /// toward a point q from p: direction q - p and a t_max just below 1.
    pub fn occluded_many(&self, rays: &[Ray], t_min: f64, t_max: f64) -> Result<Vec<bool>> {
        let raw: Vec<sys::yart_ray> = rays.iter().map(|r| sys::yart_ray { origin: r.origin, direction: r.direction }).collect();
        let mut flags = vec![0u8; rays.len()];
        let rc = unsafe {
            sys::yart_occluded(self.ctx, sys::YART_TARGET_WORLD, raw.as_ptr(), raw.len() as u64, t_min, t_max, 0,
                               flags.as_mut_ptr(), ptr::null_mut())
        };
        if rc != 0 { return Err(self.ctx_err(rc)); }
        Ok(flags.iter().map(|&f| f != 0).collect())
    }

    /// `Hittable::hit` for a single ray (hittable.rs:24) -- for drop-in tests; use `hit_many` for work.
    pub fn hit(&self, ray: &Ray, t_min: f64, t_max: f64) -> Option<Hit> {
        self.hit_many(std::slice::from_ref(ray), t_min, t_max).ok().and_then(|mut v| v.pop().flatten())
    }

    /// The batched query on single-precision records (`yart_closest_hit_f32`): 24-byte rays in, 16-byte hits out;
    /// the traversal arithmetic is the same f64, `prim_id == YART_MISS` marks a miss.
    pub fn hit_many_f32(&self, rays: &[sys::yart_ray_f32], t_min: f32, t_max: f32) -> Result<Vec<sys::yart_hit_f32>> {
        let mut hits = vec![sys::yart_hit_f32 { t: 0.0, u: 0.0, v: 0.0, prim_id: 0 }; rays.len()];
        let rc = unsafe {
            sys::yart_closest_hit_f32(self.ctx, sys::YART_TARGET_WORLD, rays.as_ptr(), rays.len() as u64, t_min, t_max,
                                      sys::YART_ORDER_NEAR, 0, hits.as_mut_ptr(), ptr::null_mut())
        };
        if rc != 0 { return Err(self.ctx_err(rc)); }
        Ok(hits)
    }

    /// The batched query on buffers the caller keeps (no allocation, no conversion): page-lock them once with `pin`
    /// and every call moves them over PCIe at full rate, upload / kernels / download overlapped inside the library.
    pub fn hit_many_into(&self, rays: &[sys::yart_ray], t_min: f64, t_max: f64, hits: &mut [sys::yart_hit]) -> Result<()> {
        assert_eq!(rays.len(), hits.len());
        let rc = unsafe {
            sys::yart_closest_hit(self.ctx, sys::YART_TARGET_WORLD, rays.as_ptr(), rays.len() as u64, t_min, t_max,
                                  sys::YART_ORDER_NEAR, 0, hits.as_mut_ptr(), ptr::null_mut())
        };
        if rc != 0 { Err(self.ctx_err(rc)) } else { Ok(()) }
    }

    /// Page-lock a slice in place (`yart_host_register`); the guard unlocks it when dropped.  The slice must not be
    /// reallocated while the guard lives (it borrows it mutably for that reason).
    pub fn pin<'a, T>(&'a self, buf: &'a mut [T]) -> Result<Pinned<'a, T>> {
        let rc = unsafe { sys::yart_host_register(self.ctx, buf.as_mut_ptr() as *mut _, std::mem::size_of_val(buf) as u64) };
        if rc != 0 { return Err(self.ctx_err(rc)); }
        Ok(Pinned { scene: self, buf })
    }

    /// "" or the sentence a front end must show (a stand-in mesh was loaded for the unshipped bunny.obj / teapot.obj).
    pub fn note(&self) -> String {
        unsafe { CStr::from_ptr(sys::yart_preset_note(self.preset)) }.to_string_lossy().into_owned()
    }

    /// `render()` (main.rs:590-775) up to the RGBA8 image; samples `[0, spp)` of every pixel.
    pub fn render(&self, width: u32, height: u32, spp: u32, max_depth: u32, seed: u64) -> Result<Vec<u8>> {
        let mut cam: sys::yart_camera = unsafe { std::mem::zeroed() };
        let rc = unsafe { sys::yart_preset_camera(self.preset, width, height, -1.0, -1.0, &mut cam) };
        if rc != 0 { return Err(Self::global_err(rc)); }
        let opts = sys::yart_render_opts { width, height, sample_begin: 0, sample_end: spp, max_depth,
                                           order: sys::YART_ORDER_NEAR, seed, ..Default::default() };
        let mut film = vec![0f64; (width as usize) * (height as usize) * 3];
        let mut rgba = vec![0u8; (width as usize) * (height as usize) * 4];
        unsafe {
            let rc = sys::yart_render(self.ctx, &cam, &opts, film.as_mut_ptr(), ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
            let rc = sys::yart_film_finalize(self.ctx, film.as_ptr(), width, height, spp, 0, rgba.as_mut_ptr());
            if rc != 0 { return Err(self.ctx_err(rc)); }
        }
        Ok(rgba)
    }

    /// Denoiser inputs for the image `render(width, height, spp, ..)` makes: the film as linear RGB
    /// (`yart_film_finalize_linear`) from samples `[0, spp)`, and the first-hit means of samples `[0, aov_spp)`
    /// (`yart_render_aovs`) -- albedo and normal per pixel (`[h][w][3]`), and the mean distance of the samples that
    /// hit (`[h][w]`, 0 where none did).  The two calls draw the same camera samples, so the planes line up with the
    /// beauty image.
    pub fn render_aovs(&self, width: u32, height: u32, spp: u32, aov_spp: u32, max_depth: u32, seed: u64) -> Result<Aovs> {
        let mut cam: sys::yart_camera = unsafe { std::mem::zeroed() };
        let rc = unsafe { sys::yart_preset_camera(self.preset, width, height, -1.0, -1.0, &mut cam) };
        if rc != 0 { return Err(Self::global_err(rc)); }
        let n = (width as usize) * (height as usize);
        let mut opts = sys::yart_render_opts { width, height, sample_begin: 0, sample_end: spp, max_depth,
                                               order: sys::YART_ORDER_NEAR, seed, ..Default::default() };
        let mut film = vec![0f64; n * 3];
        let (mut albedo, mut normal, mut depth) = (vec![0f64; n * 3], vec![0f64; n * 3], vec![0f64; n * 3]);
        let mut color = vec![0f32; n * 3];
        unsafe {
            let rc = sys::yart_render(self.ctx, &cam, &opts, film.as_mut_ptr(), ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
            let rc = sys::yart_film_finalize_linear(self.ctx, film.as_ptr(), width, height, spp, 0, color.as_mut_ptr());
            if rc != 0 { return Err(self.ctx_err(rc)); }
            opts.sample_end = aov_spp;
            let planes = sys::yart_aov_planes { albedo: albedo.as_mut_ptr(), normal: normal.as_mut_ptr(), depth: depth.as_mut_ptr() };
            let rc = sys::yart_render_aovs(self.ctx, &cam, &opts, &planes, ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
        }
        let mut out = Aovs { color, albedo: vec![0f32; n * 3], normal: vec![0f32; n * 3], depth: vec![0f32; n] };
        for i in 0..n {
            let (hits, samples) = (depth[i * 3 + 1], depth[i * 3 + 2]);
            for k in 0..3 {
                if samples > 0.0 {
                    out.albedo[i * 3 + k] = (albedo[i * 3 + k] / samples) as f32;
                    out.normal[i * 3 + k] = (normal[i * 3 + k] / samples) as f32;
                }
            }
            if hits > 0.0 { out.depth[i] = (depth[i * 3] / hits) as f32; }
        }
        Ok(out)
    }

    /// `render(width, height, spp, ..)` denoised by the library's a-trous filter (`yart_denoise`, default options),
    /// guided by the first-hit planes of samples `[0, aov_spp)`: linear RGB (`[h][w][3]` f32) and the RGBA8 image
    /// through the same display rule as `render`.
    pub fn denoise(&self, width: u32, height: u32, spp: u32, aov_spp: u32, max_depth: u32, seed: u64) -> Result<(Vec<f32>, Vec<u8>)> {
        let mut cam: sys::yart_camera = unsafe { std::mem::zeroed() };
        let rc = unsafe { sys::yart_preset_camera(self.preset, width, height, -1.0, -1.0, &mut cam) };
        if rc != 0 { return Err(Self::global_err(rc)); }
        let n = (width as usize) * (height as usize);
        let mut opts = sys::yart_render_opts { width, height, sample_begin: 0, sample_end: spp, max_depth,
                                               order: sys::YART_ORDER_NEAR, seed, ..Default::default() };
        let mut film = vec![0f64; n * 3];
        let (mut albedo, mut normal, mut depth) = (vec![0f64; n * 3], vec![0f64; n * 3], vec![0f64; n * 3]);
        let (mut rgb, mut rgba) = (vec![0f32; n * 3], vec![0u8; n * 4]);
        unsafe {
            let rc = sys::yart_render(self.ctx, &cam, &opts, film.as_mut_ptr(), ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
            opts.sample_end = aov_spp;
            let planes = sys::yart_aov_planes { albedo: albedo.as_mut_ptr(), normal: normal.as_mut_ptr(), depth: depth.as_mut_ptr() };
            let rc = sys::yart_render_aovs(self.ctx, &cam, &opts, &planes, ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
            let dn = sys::yart_denoise_opts::default();
            let rc = sys::yart_denoise(self.ctx, film.as_ptr(), spp, &planes, width, height, &dn, rgb.as_mut_ptr(),
                                       rgba.as_mut_ptr(), ptr::null_mut());
            if rc != 0 { return Err(self.ctx_err(rc)); }
        }
        Ok((rgb, rgba))
    }
}

/// What `GpuScene::render_aovs` returns: row-major images, top row first.
pub struct Aovs { pub color: Vec<f32>, pub albedo: Vec<f32>, pub normal: Vec<f32>, pub depth: Vec<f32> }

/// A page-locked view of a caller's slice (see `GpuScene::pin`).
pub struct Pinned<'a, T> {
    scene: &'a GpuScene,
    pub buf: &'a mut [T],
}

impl<'a, T> Drop for Pinned<'a, T> {
    fn drop(&mut self) {
        unsafe { sys::yart_host_unregister(self.scene.ctx, self.buf.as_mut_ptr() as *mut _) };
    }
}

/// Better sampling switches of `yart_render_opts.flags` -- all off is the reference's estimator bit for bit
/// (hittable.rs:113-122 light pick over len-1, main.rs:544-546 depth exhaustion = 1.0, no roulette, no light sampling).
/// `next_event` (next-event estimation with MIS) implies `unbiased_light_pick`.
#[derive(Clone, Copy, Debug, Default)]
pub struct Sampling { pub unbiased_light_pick: bool, pub russian_roulette: bool, pub depth_zero_black: bool, pub next_event: bool }

impl Sampling {
    fn bits(self) -> u32 {
        (if self.unbiased_light_pick { sys::YART_FLAG_UNBIASED_LIGHT_PICK } else { 0 })
            | (if self.russian_roulette { sys::YART_FLAG_RUSSIAN_ROULETTE } else { 0 })
            | (if self.depth_zero_black { sys::YART_FLAG_DEPTH_ZERO_BLACK } else { 0 })
            | (if self.next_event { sys::YART_FLAG_NEXT_EVENT } else { 0 })
    }
}

/// `render()` on N GPUs of one box: the tile jobs + mpsc gather of main.rs:629-646, 746-760 become sample-range
/// shards (one host thread per context) + ONE in-place `ncclReduce` of the f64 film (`yart_film_reduce`).
pub struct MultiGpu { scenes: Vec<GpuScene>, comm: *mut sys::yart_comm }

impl MultiGpu {
    pub fn from_preset(name: &str, assets_dir: &str, seed: u64, devices: &[i32]) -> Result<MultiGpu> {
        let scenes = devices.iter().map(|&d| GpuScene::from_preset(name, assets_dir, seed, d)).collect::<Result<Vec<_>>>()?;
        let ctxs: Vec<*mut sys::yart_ctx> = scenes.iter().map(|s| s.ctx).collect();
        let mut comm = ptr::null_mut();
        if ctxs.len() > 1 {
            let rc = unsafe { sys::yart_comm_init(ctxs.as_ptr(), ctxs.len() as i32, &mut comm) };
            if rc != 0 { return Err(GpuScene::global_err(rc)); }
        }
        Ok(MultiGpu { scenes, comm })
    }

    /// The RGBA8 frame of samples `[0, spp)`: every GPU renders its contiguous share, the root finalises.
    pub fn render(&self, width: u32, height: u32, spp: u32, max_depth: u32, seed: u64, sampling: Sampling) -> Result<Vec<u8>> {
        let n = self.scenes.len() as u32;
        let mut cam: sys::yart_camera = unsafe { std::mem::zeroed() };
        let rc = unsafe { sys::yart_preset_camera(self.scenes[0].preset, width, height, -1.0, -1.0, &mut cam) };
        if rc != 0 { return Err(GpuScene::global_err(rc)); }
        let mut films = vec![ptr::null_mut::<f64>(); n as usize];
        for (s, f) in self.scenes.iter().zip(films.iter_mut()) {
            let rc = unsafe { sys::yart_film_create(s.ctx, width, height, f) };
            if rc != 0 { return Err(s.ctx_err(rc)); }
        }
        let results: Vec<i32> = std::thread::scope(|scope| {
            let handles: Vec<_> = self.scenes.iter().zip(films.iter()).enumerate().map(|(r, (s, &film))| {
                let (ctx, film, cam) = (s.ctx as usize, film as usize, cam);   // raw pointers cross the thread as integers
                scope.spawn(move || {
                    let (base, extra, r) = (spp / n, spp % n, r as u32);
                    let lo = r * base + r.min(extra);
                    let hi = lo + base + u32::from(r < extra);
                    let opts = sys::yart_render_opts { width, height, sample_begin: lo, sample_end: hi, max_depth,
                        order: sys::YART_ORDER_NEAR, flags: sys::YART_FLAG_DEVICE_PTRS | sampling.bits(), seed, ..Default::default() };
                    if hi == lo { return 0; }
                    unsafe { sys::yart_render(ctx as *mut sys::yart_ctx, &cam, &opts, film as *mut f64, ptr::null_mut()) }
                })
            }).collect();
            handles.into_iter().map(|h| h.join().unwrap()).collect()
        });
        if let Some((r, &rc)) = results.iter().enumerate().find(|(_, &rc)| rc != 0) { return Err(self.scenes[r].ctx_err(rc)); }
        if !self.comm.is_null() {
            let rc = unsafe { sys::yart_film_reduce(self.comm, films.as_ptr(), width, height, 0) };
            if rc != 0 { return Err(GpuScene::global_err(rc)); }
        }
        let root = &self.scenes[0];
        let mut film = vec![0f64; (width as usize) * (height as usize) * 3];
        let mut rgba = vec![0u8; (width as usize) * (height as usize) * 4];
        unsafe {
            let rc = sys::yart_film_read(root.ctx, films[0], width, height, film.as_mut_ptr());
            if rc != 0 { return Err(root.ctx_err(rc)); }
            let rc = sys::yart_film_finalize(root.ctx, film.as_ptr(), width, height, spp, 0, rgba.as_mut_ptr());
            if rc != 0 { return Err(root.ctx_err(rc)); }
            for (s, &f) in self.scenes.iter().zip(films.iter()) { sys::yart_film_destroy(s.ctx, f); }
        }
        Ok(rgba)
    }
}

impl Drop for MultiGpu {
    fn drop(&mut self) { if !self.comm.is_null() { unsafe { sys::yart_comm_destroy(self.comm) } } }
}

impl Drop for GpuScene {
    fn drop(&mut self) {
        unsafe {
            if !self.ctx.is_null() { sys::yart_ctx_destroy(self.ctx); }
            if !self.preset.is_null() { sys::yart_preset_free(self.preset); }
        }
    }
}
