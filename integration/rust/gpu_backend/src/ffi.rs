//! `extern "C"` mirror of include/tcpt.h, one to one (field order and widths are the header's; every struct is `#[repr(C)]`).
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct TcptCtx {
    _opaque: [u8; 0],
}
#[repr(C)]
pub struct TcptGroup {
    _opaque: [u8; 0],
}
#[repr(C)]
pub struct TcptObj {
    _opaque: [u8; 0],
}

pub const TCPT_OK: c_int = 0;
pub const TCPT_ERR_INVALID: c_int = -1;
pub const TCPT_ERR_CUDA: c_int = -2;
pub const TCPT_ERR_LIMIT: c_int = -3;
pub const TCPT_ERR_NOMEM: c_int = -4;

pub const INTEGRATOR_PT: i32 = 0;
pub const INTEGRATOR_NEE: i32 = 1;
pub const INTEGRATOR_MIS: i32 = 2;
pub const INTEGRATOR_ALBEDO: i32 = 3;
pub const INTEGRATOR_NORMAL: i32 = 4;
pub const SAMPLER_RANDOM: i32 = 0;
pub const SAMPLER_SOBOL: i32 = 1;

pub const MAT_LAMBERT: i32 = 0;
pub const MAT_EMISSIVE: i32 = 1;
pub const MAT_PLASTIC: i32 = 2;
pub const MAT_SIMPLE_PBR: i32 = 3;
pub const MAT_CLEARCOAT_PBR: i32 = 4;
pub const MAT_METAL: i32 = 5;
pub const MAT_GLASS: i32 = 6;

pub const SPEC_CONSTANT: i32 = 0;
pub const SPEC_RGB_ALBEDO_SRGB: i32 = 1;
pub const SPEC_RGB_ALBEDO_LINEAR: i32 = 2;
pub const SPEC_D65: i32 = 3;
pub const SPEC_TEXTURE_SRGB: i32 = 4;
pub const SPEC_PRESET: i32 = 5;

pub const LIGHT_POINT: c_int = 3;
pub const LIGHT_SPOT: c_int = 4;
pub const LIGHT_DIRECTIONAL: c_int = 5;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptSpectrumParam {
    pub kind: i32,
    pub value: [f32; 3],
    pub texture: i32, // texture index (SPEC_TEXTURE_SRGB) or TCPT_PRESET_* id (SPEC_PRESET)
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptFloatParam {
    pub kind: i32, // 0 constant, 1 gray8 FloatTexture
    pub value: f32,
    pub texture: i32,
    pub gamma_corrected: i32,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct TcptNormalParam {
    pub texture: i32, // -1 = NormalParameter::none()
    pub flip_y: i32,
}
impl Default for TcptNormalParam {
    fn default() -> Self {
        Self { texture: -1, flip_y: 0 }
    }
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptMaterialDesc {
    pub ty: i32,
    pub color: TcptSpectrumParam,
    pub intensity: TcptFloatParam,
    pub normal: TcptNormalParam,
    pub eta: f32,
    pub thin_surface: i32,
    pub roughness: TcptFloatParam,
    pub metallic: TcptFloatParam,
    pub ior: TcptFloatParam,
    pub coat_ior: TcptFloatParam,
    pub coat_roughness: TcptFloatParam,
    pub coat_thickness: TcptFloatParam,
    pub coat_tint: TcptSpectrumParam,
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptRenderParams {
    pub width: u32,
    pub height: u32,
    pub spp: u32,
    pub seed: u32,
    pub max_depth: u32,
    pub integrator: i32,
    pub sampler: i32,
    pub exposure: f32,
    pub fov_deg: f32,
    pub cam_pos: [f32; 3],
    pub cam_dir: [f32; 3],
    pub cam_up: [f32; 3],
    pub row_offset: u32,
    pub row_stride: u32,
    pub spp_begin: u32,
    pub spp_end: u32,
    pub max_slots: u32,
}
/// Adaptive sampling (tcpt_render_adaptive): stop a pixel once the relative standard error of its mean luminance is below `threshold`
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptAdaptiveParams {
    pub threshold: f32,
    pub min_spp: u32,
    pub step: u32,
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct TcptStats {
    pub paths: u64,
    pub closest_rays: u64,
    pub shadow_rays: u64,
    pub box_tests: u64,
    pub tri_tests: u64,
    pub kernel_launches: u64,
    pub render_ms: f64,
    pub trace_closest_ms: f64,
    pub trace_shadow_ms: f64,
    pub shade_ms: f64,
    pub generate_ms: f64,
    pub film_ms: f64,
    pub passes: u32,
    pub max_bvh_depth: u32,
    pub sobol_prefix_ms: f64,
    pub sobol_prefix_bytes: u64,
    pub reduce_ms: f64,
    pub trace_launches: u32,
    pub shade_launches: u32,
}

unsafe extern "C" {
    pub fn tcpt_create(device_id: c_int, out: *mut *mut TcptCtx) -> c_int;
    pub fn tcpt_destroy(ctx: *mut TcptCtx);
    pub fn tcpt_last_error(ctx: *const TcptCtx) -> *const c_char;
    pub fn tcpt_set_option(ctx: *mut TcptCtx, name: *const c_char, value: c_int) -> c_int;
    pub fn tcpt_set_tables(ctx: *mut TcptCtx, std_tables: *const c_void, std_len: usize, rgb2spec: *const f32, rgb2spec_floats: usize) -> c_int;

    pub fn tcpt_scene_clear(ctx: *mut TcptCtx) -> c_int;
    pub fn tcpt_scene_add_mesh(ctx: *mut TcptCtx, positions: *const f32, normals: *const f32, uvs: *const f32, n_vertices: c_int,
                               indices: *const u32, n_triangles: c_int) -> c_int;
    pub fn tcpt_scene_add_single_triangle(ctx: *mut TcptCtx, positions: *const f32, normals: *const f32, uvs: *const f32) -> c_int;
    pub fn tcpt_scene_add_texture(ctx: *mut TcptCtx, data: *const u8, width: u32, height: u32, channels: u32) -> c_int;
    pub fn tcpt_scene_add_material(ctx: *mut TcptCtx, desc: *const TcptMaterialDesc) -> c_int;
    pub fn tcpt_scene_add_primitive(ctx: *mut TcptCtx, geometry: c_int, material: c_int, local_to_world: *const f32) -> c_int;
    pub fn tcpt_scene_add_env_light(ctx: *mut TcptCtx, intensity: f32, rgb: *const f32, width: u32, height: u32, local_to_world: *const f32) -> c_int;
    pub fn tcpt_scene_add_delta_light(ctx: *mut TcptCtx, kind: c_int, intensity: f32, spectrum: *const TcptSpectrumParam, angle_inner: f32,
                                      angle_outer: f32, local_to_world: *const f32) -> c_int;
    pub fn tcpt_scene_build(ctx: *mut TcptCtx, cam_pos: *const f32) -> c_int;

    // asset ingestion: what Scene::load_obj / the texture loaders do with tobj and the image crate in the CPU build (include/tcpt.h)
    pub fn tcpt_obj_load(path: *const c_char, out: *mut *mut TcptObj, err: *mut c_char, err_len: usize) -> c_int;
    pub fn tcpt_obj_counts(obj: *const TcptObj, counts: *mut u32) -> c_int;
    pub fn tcpt_obj_copy(obj: *const TcptObj, positions: *mut f32, normals: *mut f32, texcoords: *mut f32, indices: *mut u32, tangent_tri: *mut u32) -> c_int;
    pub fn tcpt_obj_free(obj: *mut TcptObj);
    pub fn tcpt_scene_load_obj(ctx: *mut TcptCtx, path: *const c_char) -> c_int;
    pub fn tcpt_scene_set_tangent_source(ctx: *mut TcptCtx, geometry: c_int, tri: *const u32, n_triangles: c_int) -> c_int;
    pub fn tcpt_scene_build_soup(ctx: *mut TcptCtx, triangles: *const f32, n_triangles: u32) -> c_int;
    pub fn tcpt_soup_build_info(ctx: *const TcptCtx, build_ms: *mut f64, n_records: *mut u64, levels: *mut u32) -> c_int;
    pub fn tcpt_image_convert(src: *const c_void, width: u32, height: u32, channels: u32, sample_type: c_int, dst_kind: c_int, dst: *mut c_void) -> c_int;

    pub fn tcpt_render(ctx: *mut TcptCtx, params: *const TcptRenderParams, out_acc: *mut f32, out_srgb: *mut f32) -> c_int;
    pub fn tcpt_render_device(ctx: *mut TcptCtx, params: *const TcptRenderParams, dev_acc: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn tcpt_finalize_device(ctx: *mut TcptCtx, dev_acc: *const c_void, width: u32, height: u32, spp: u32, dev_srgb: *mut c_void,
                                stream: *mut c_void) -> c_int;
    pub fn tcpt_render_adaptive(ctx: *mut TcptCtx, params: *const TcptRenderParams, ap: *const TcptAdaptiveParams, out_acc: *mut f32,
                                out_srgb: *mut f32, out_spp: *mut u32) -> c_int;
    pub fn tcpt_render_adaptive_device(ctx: *mut TcptCtx, params: *const TcptRenderParams, ap: *const TcptAdaptiveParams, dev_acc: *mut c_void,
                                       dev_spp: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn tcpt_get_stats(ctx: *const TcptCtx, out: *mut TcptStats) -> c_int;

    // multi-GPU: one context per GPU; the library owns the NCCL communicator (include/tcpt.h "multi-GPU")
    pub fn tcpt_comm_get_unique_id(id128: *mut c_void) -> c_int;
    pub fn tcpt_comm_init(ctx: *mut TcptCtx, nranks: c_int, rank: c_int, id128: *const c_void) -> c_int;
    pub fn tcpt_comm_destroy(ctx: *mut TcptCtx) -> c_int;
    pub fn tcpt_shard_params(job: *const TcptRenderParams, shard_mode: c_int, rank: c_int, nranks: c_int, out: *mut TcptRenderParams) -> c_int;
    pub fn tcpt_render_sharded(ctx: *mut TcptCtx, job: *const TcptRenderParams, shard_mode: c_int, out_acc: *mut f32, out_srgb: *mut f32) -> c_int;
    pub fn tcpt_render_sharded_device(ctx: *mut TcptCtx, job: *const TcptRenderParams, shard_mode: c_int, dev_acc: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn tcpt_render_adaptive_sharded(ctx: *mut TcptCtx, job: *const TcptRenderParams, ap: *const TcptAdaptiveParams, out_acc: *mut f32,
                                        out_srgb: *mut f32, out_spp: *mut u32) -> c_int;
    // one host process, N GPUs: what GpuRendererImage::render_multi binds
    pub fn tcpt_group_create(device_ids: *const c_int, n: c_int, out: *mut *mut TcptGroup) -> c_int;
    pub fn tcpt_group_destroy(g: *mut TcptGroup);
    pub fn tcpt_group_size(g: *const TcptGroup) -> c_int;
    pub fn tcpt_group_context(g: *mut TcptGroup, i: c_int) -> *mut TcptCtx;
    pub fn tcpt_group_last_error(g: *const TcptGroup) -> *const c_char;
    pub fn tcpt_group_set_tables(g: *mut TcptGroup, std_tables: *const c_void, std_len: usize, rgb2spec: *const f32, rgb2spec_floats: usize) -> c_int;
    pub fn tcpt_group_build(g: *mut TcptGroup, cam_pos: *const f32) -> c_int;
    pub fn tcpt_group_render(g: *mut TcptGroup, job: *const TcptRenderParams, shard_mode: c_int, out_acc: *mut f32, out_srgb: *mut f32) -> c_int;
    pub fn tcpt_group_render_adaptive(g: *mut TcptGroup, job: *const TcptRenderParams, ap: *const TcptAdaptiveParams, out_acc: *mut f32,
                                      out_srgb: *mut f32, out_spp: *mut u32) -> c_int;
}
pub const TCPT_SHARD_TILE: c_int = 0;
pub const TCPT_SHARD_SPP: c_int = 1;
pub const TCPT_COMM_ID_BYTES: usize = 128;
