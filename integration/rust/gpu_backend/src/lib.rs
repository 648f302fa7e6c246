//! GPU drop-in for `RendererImage::<SrgbRenderer{Pt,Nee,Mis}>::render::<S>()` (renderer/src/renderer.rs:101-149) over libtcpt.
//!
//! Usage in renderer/src/main.rs:142-237 (`render_with_sampler`): build the scene through `GpuScene` (same `load_obj` /
//! `create_primitive` / `build` calls as `scene::Scene`, which it wraps), then
//! ```ignore
//! let mut image = GpuRendererImage::new(&gpu_scene, &camera, width, height, spp, seed, Integrator::Mis, 1.0, max_depth);
//! image.render::<ZSobolSampler>();      // one tcpt_render call: the whole frame, all samples
//! image.save("output.png");             // byte-for-byte the reference's writer
//! ```
//! NOT COMPILED here (no Rust toolchain in the image this backend was built in); see ../README.md.
pub mod ffi;
pub mod flatten;

use std::ffi::CStr;
use std::path::Path;

use ffi::*;
use flatten::{Recorded, Uploader};

#[derive(Clone, Copy)]
pub enum Integrator {
    Pt = 0,
    Nee = 1,
    Mis = 2,
    Albedo = 3,
    Normal = 4,
}

/// Sampler marker: implemented for renderer::sampler::{RandomSampler, ZSobolSampler} so that `render::<S>()` keeps its shape.
pub trait GpuSampler {
    const ID: i32;
}
impl GpuSampler for renderer::sampler::RandomSampler {
    const ID: i32 = SAMPLER_RANDOM; // statistical parity only: ThreadRng is OS-seeded in the reference
}
impl GpuSampler for renderer::sampler::ZSobolSampler {
    const ID: i32 = SAMPLER_SOBOL; // bit-exact sample streams (tests/test_sobol.py)
}

/// Records the construction calls next to forwarding them to the wrapped `scene::Scene` (kept so that CPU and GPU renders of the
/// same scene object can be compared, as renderer/tests/renderer_consistency_test.rs does between integrators).
pub struct GpuScene<Id: scene::SceneId> {
    pub cpu: scene::Scene<Id>,
    obj_paths: Vec<String>,
    recorded: Vec<Recorded>,
    ctx: *mut TcptCtx,
}
impl<Id: scene::SceneId> GpuScene<Id> {
    pub fn new(cpu: scene::Scene<Id>, device: i32, std_tables: &[u8], rgb2spec: &[f32]) -> Self {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { tcpt_create(device, &mut ctx) };
        if rc != TCPT_OK {
            panic!("tcpt_create: {} (no CPU fallback: an sm_100 GPU is required)", last_error(ctx));
        }
        // std_tables: tools/extract_reference_tables.py output (Sobol matrices, CIE, D65, presets); rgb2spec: the table
        // rgb_to_spec/src/lib.rs embeds with include_bytes! (64 z-nodes + [3][64][64][64][3] f32)
        let rc = unsafe { tcpt_set_tables(ctx, std_tables.as_ptr() as *const _, std_tables.len(), rgb2spec.as_ptr(), rgb2spec.len()) };
        if rc != TCPT_OK {
            panic!("tcpt_set_tables: {}", last_error(ctx));
        }
        Self { cpu, obj_paths: Vec::new(), recorded: Vec::new(), ctx }
    }
    pub fn load_obj(&mut self, path: &str) -> scene::GeometryIndex<Id> {
        self.obj_paths.push(path.to_owned());
        self.cpu.load_obj(path)
    }
    pub fn create_primitive(&mut self, desc: scene::CreatePrimitiveDesc<Id>) -> scene::PrimitiveIndex<Id> {
        self.recorded.push(record(&desc)); // POD copy of the desc (Material is an Arc: cloned, not deep-copied)
        self.cpu.create_primitive(desc)
    }
    /// Scene::build(&camera) on both sides.  `meshes` hands over the loaded TriangleMesh of every geometry index (needs the accessor
    /// `Scene::geometry(&self, GeometryIndex) -> &TriangleMesh` listed in README.md); `describe` maps a Material to its parameters.
    pub fn build<F: renderer::filter::Filter>(&mut self, camera: &renderer::camera::Camera<F>) {
        self.cpu.build(camera);
        let mut up = Uploader::new(self.ctx);
        unsafe { tcpt_scene_clear(self.ctx) };
        let geometry_map: Vec<i32> = (0..self.obj_paths.len()).map(|g| up.mesh(self.cpu.geometry(scene::GeometryIndex::new(g)))).collect();
        let p = camera.position(); // accessor listed in README.md (Camera.position is private, camera.rs:15-16)
        up.primitives(&self.recorded, &|m| scene::gpu_describe(m), &geometry_map, [p.x(), p.y(), p.z()]);
    }
}
impl<Id: scene::SceneId> Drop for GpuScene<Id> {
    fn drop(&mut self) {
        unsafe { tcpt_destroy(self.ctx) };
    }
}

fn last_error(ctx: *const TcptCtx) -> String {
    if ctx.is_null() {
        return "no context".into();
    }
    unsafe { CStr::from_ptr(tcpt_last_error(ctx)) }.to_string_lossy().into_owned()
}

fn cols(t: &math::Transform<math::Local, math::World>) -> [f32; 16] {
    t.to_mat4().to_cols_array() // column major, what glam holds (accessor `to_mat4` listed in README.md)
}

fn record<Id: scene::SceneId>(desc: &scene::CreatePrimitiveDesc<Id>) -> Recorded {
    use scene::CreatePrimitiveDesc as D;
    match desc {
        D::GeometryPrimitive { geometry_index, surface_material, transform } => {
            Recorded::Geometry { geometry: geometry_index.0, material: surface_material.clone(), local_to_world: cols(transform) }
        }
        D::SingleTrianglePrimitive { positions, normals, uvs, surface_material, transform } => {
            let mut p = [0.0; 9];
            let mut n = [0.0; 9];
            let mut t = [0.0; 6];
            for k in 0..3 {
                p[3 * k..3 * k + 3].copy_from_slice(&[positions[k].x(), positions[k].y(), positions[k].z()]);
                n[3 * k..3 * k + 3].copy_from_slice(&[normals[k].x(), normals[k].y(), normals[k].z()]);
                t[2 * k..2 * k + 2].copy_from_slice(&[uvs[k].x, uvs[k].y]);
            }
            Recorded::SingleTriangle { positions: p, normals: n, uvs: t, material: surface_material.clone(), local_to_world: cols(transform) }
        }
        D::PointLightPrimitive { intensity, spectrum, transform } => Recorded::Delta {
            kind: LIGHT_POINT, intensity: *intensity, spectrum: spectrum::gpu_describe(spectrum), angle_inner: 0.0, angle_outer: 0.0, local_to_world: cols(transform),
        },
        D::SpotLightPrimitive { angle_inner, angle_outer, intensity, spectrum, transform } => Recorded::Delta {
            kind: LIGHT_SPOT, intensity: *intensity, spectrum: spectrum::gpu_describe(spectrum), angle_inner: *angle_inner, angle_outer: *angle_outer,
            local_to_world: cols(transform),
        },
        D::DirectionalLightPrimitive { intensity, spectrum, transform } => Recorded::Delta {
            kind: LIGHT_DIRECTIONAL, intensity: *intensity, spectrum: spectrum::gpu_describe(spectrum), angle_inner: 0.0, angle_outer: 0.0, local_to_world: cols(transform),
        },
        D::EnvironmentLightPrimitive { intensity, texture_path, transform } => {
            // same decode as EnvironmentLight::new (environment_light.rs:34-40): image::open(..).to_rgb32f()
            let img = image::open(texture_path).expect("environment texture").to_rgb32f();
            let (w, h) = (img.width(), img.height());
            Recorded::Environment { intensity: *intensity, rgb: img.into_raw(), width: w, height: h, local_to_world: cols(transform) }
        }
    }
}

/// Same surface as `RendererImage` (`new` / `render::<S>` / `save`, renderer.rs:101-149); `pixels` holds the same tone-mapped sRGB triples.
pub struct GpuRendererImage {
    ctx: *mut TcptCtx,
    params: TcptRenderParams,
    pub pixels: Vec<[f32; 3]>,
    pub accumulators: Vec<[f32; 3]>, // Sensor accumulators (linear sRGB sums, sensor.rs:76-77): what a multi-GPU host reduces
}
impl GpuRendererImage {
    #[allow(clippy::too_many_arguments)]
    pub fn new<Id: scene::SceneId, F: renderer::filter::Filter>(
        scene: &GpuScene<Id>, camera: &renderer::camera::Camera<F>, width: u32, height: u32, spp: u32, seed: u32,
        integrator: Integrator, exposure: f32, max_depth: usize,
    ) -> Self {
        let (p, d, u) = (camera.position(), camera.direction(), camera.up());
        let params = TcptRenderParams {
            width, height, spp, seed, max_depth: max_depth as u32, integrator: integrator as i32, sampler: SAMPLER_SOBOL, exposure,
            fov_deg: camera.fov(), cam_pos: [p.x(), p.y(), p.z()], cam_dir: [d.x(), d.y(), d.z()], cam_up: [u.x(), u.y(), u.z()],
            ..Default::default() // row_offset / row_stride / spp_begin / spp_end = 0: the whole frame on this GPU
        };
        let n = (width * height) as usize;
        Self { ctx: scene.ctx, params, pixels: vec![[0.0; 3]; n], accumulators: vec![[0.0; 3]; n] }
    }
    /// One GPU of `n`: image rows y % n == rank (bitwise equal to a single-GPU render after summing the accumulators) ...
    pub fn shard_rows(&mut self, rank: u32, n: u32) {
        self.params.row_offset = rank;
        self.params.row_stride = n;
    }
    /// ... or sample indices [begin, end) of every pixel (best balance; sum order changes in the last bits).
    pub fn shard_samples(&mut self, begin: u32, end: u32) {
        self.params.spp_begin = begin;
        self.params.spp_end = end;
    }
    pub fn render<S: GpuSampler>(&mut self) {
        self.params.sampler = S::ID;
        let rc = unsafe { tcpt_render(self.ctx, &self.params, self.accumulators.as_mut_ptr() as *mut f32, self.pixels.as_mut_ptr() as *mut f32) };
        if rc != TCPT_OK {
            panic!("tcpt_render: {}", last_error(self.ctx)); // the reference panics on errors too (main.rs:61,91,138,235)
        }
    }
    /// Adaptive sampling (`tcpt_render_adaptive`): every pixel renders samples [0, min_spp), then `step` more per round until the
    /// relative standard error of its mean luminance drops below `threshold` or it reaches the image's spp.  Each pixel's accumulator
    /// is bitwise the one `render` gives for the window [0, count) of the same job; `pixels` are divided by each pixel's own count.
    /// Returns the per-pixel sample counts (row major).
    pub fn render_adaptive<S: GpuSampler>(&mut self, threshold: f32, min_spp: u32, step: u32) -> Vec<u32> {
        self.params.sampler = S::ID;
        let ap = TcptAdaptiveParams { threshold, min_spp, step };
        let mut counts = vec![0u32; (self.params.width * self.params.height) as usize];
        let rc = unsafe {
            tcpt_render_adaptive(self.ctx, &self.params, &ap, self.accumulators.as_mut_ptr() as *mut f32, self.pixels.as_mut_ptr() as *mut f32,
                                 counts.as_mut_ptr())
        };
        if rc != TCPT_OK {
            panic!("tcpt_render_adaptive: {}", last_error(self.ctx));
        }
        counts
    }
    /// One complete frame from every GPU of the communicator this context belongs to (`tcpt_comm_init`, one process per GPU): every
    /// rank calls it with the same image; rank 0's `pixels` / `accumulators` receive the frame after ONE ncclReduce inside the library.
    /// `TCPT_SHARD_TILE` reproduces the one-GPU film bit for bit, `TCPT_SHARD_SPP` balances best.
    pub fn render_sharded<S: GpuSampler>(&mut self, shard_mode: i32) {
        self.params.sampler = S::ID;
        let rc = unsafe { tcpt_render_sharded(self.ctx, &self.params, shard_mode, self.accumulators.as_mut_ptr() as *mut f32, self.pixels.as_mut_ptr() as *mut f32) };
        if rc != TCPT_OK {
            panic!("tcpt_render_sharded: {}", last_error(self.ctx));
        }
    }
    /// The same from ONE host process that owns all GPUs of the box (`tcpt_group_create`; the scene was built with `tcpt_group_build`).
    pub fn render_group<S: GpuSampler>(&mut self, group: *mut TcptGroup, shard_mode: i32) {
        self.params.sampler = S::ID;
        let rc = unsafe { tcpt_group_render(group, &self.params, shard_mode, self.accumulators.as_mut_ptr() as *mut f32, self.pixels.as_mut_ptr() as *mut f32) };
        if rc != TCPT_OK {
            let msg = unsafe { std::ffi::CStr::from_ptr(tcpt_group_last_error(group)) }.to_string_lossy().into_owned();
            panic!("tcpt_group_render: {}", msg);
        }
    }
    /// `render_adaptive` from every GPU of the communicator (`tcpt_render_adaptive_sharded`): each rank runs the rounds over its image
    /// rows y % n == rank alone and ONE grouped reduce hands rank 0 the frame, bitwise the one-GPU `render_adaptive` frame. Every rank
    /// calls it with the same image; `pixels`, `accumulators` and the returned sample counts are filled on rank 0 only.
    pub fn render_adaptive_sharded<S: GpuSampler>(&mut self, threshold: f32, min_spp: u32, step: u32) -> Vec<u32> {
        self.params.sampler = S::ID;
        let ap = TcptAdaptiveParams { threshold, min_spp, step };
        let mut counts = vec![0u32; (self.params.width * self.params.height) as usize];
        let rc = unsafe {
            tcpt_render_adaptive_sharded(self.ctx, &self.params, &ap, self.accumulators.as_mut_ptr() as *mut f32,
                                         self.pixels.as_mut_ptr() as *mut f32, counts.as_mut_ptr())
        };
        if rc != TCPT_OK {
            panic!("tcpt_render_adaptive_sharded: {}", last_error(self.ctx));
        }
        counts
    }
    /// The same from ONE host process that owns all GPUs of the box (`tcpt_group_render_adaptive`); returns the sample counts.
    pub fn render_group_adaptive<S: GpuSampler>(&mut self, group: *mut TcptGroup, threshold: f32, min_spp: u32, step: u32) -> Vec<u32> {
        self.params.sampler = S::ID;
        let ap = TcptAdaptiveParams { threshold, min_spp, step };
        let mut counts = vec![0u32; (self.params.width * self.params.height) as usize];
        let rc = unsafe {
            tcpt_group_render_adaptive(group, &self.params, &ap, self.accumulators.as_mut_ptr() as *mut f32, self.pixels.as_mut_ptr() as *mut f32,
                                       counts.as_mut_ptr())
        };
        if rc != TCPT_OK {
            let msg = unsafe { std::ffi::CStr::from_ptr(tcpt_group_last_error(group)) }.to_string_lossy().into_owned();
            panic!("tcpt_group_render_adaptive: {}", msg);
        }
        counts
    }
    pub fn stats(&self) -> TcptStats {
        let mut s = TcptStats::default();
        unsafe { tcpt_get_stats(self.ctx, &mut s) };
        s
    }
    /// RendererImage::save (renderer.rs:137-148): `(v * 255.0) as u8`, truncating and saturating.
    pub fn save(&self, path: impl AsRef<Path>) {
        let w = self.params.width;
        image::RgbImage::from_fn(w, self.params.height, |x, y| {
            let p = self.pixels[(y * w + x) as usize];
            image::Rgb([(p[0] * 255.0) as u8, (p[1] * 255.0) as u8, (p[2] * 255.0) as u8])
        })
        .save_with_format(path, image::ImageFormat::Png)
        .unwrap();
    }
}
