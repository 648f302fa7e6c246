/* tcpt.h — C ABI of the B200-native path-integration backend (libtcpt.so / libtcpt.a, nvcc sm_100a).
 *
 * Drop-in boundary for toy-cpu-pathtracing's per-pixel path-integration hot path.  The reference has NO FFI at this seam;
 * the seam is the generic Rust trait
 *     pub trait Renderer { fn render<S: Sampler>(&mut self, p: UVec2) -> Self::Color }      renderer/src/renderer.rs:93-98
 * driven one pixel at a time by RendererImage::render (renderer/src/renderer.rs:120-134).  A GPU backend replaces the
 * whole-frame loop, so the entry points below are what a `GpuRendererImage::render` would bind (see INTEGRATION.md for the
 * Rust `extern "C"` block and `flatten.rs`).  Everything is POD: plain pointers and sizes, caller-owned host buffers unless a
 * parameter says "device"; the context owns all device memory.  Every function returns 0 on success or a negative
 * TCPT_ERR_* code and never unwinds across the boundary (the reference panics instead: renderer/src/main.rs:61,91,138,235).
 * There is no CPU fallback: every entry point that computes anything fails with TCPT_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef TCPT_H
#define TCPT_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tcpt_ctx tcpt_ctx;

enum {
    TCPT_OK = 0,
    TCPT_ERR_INVALID = -1, /* bad argument / call order */
    TCPT_ERR_CUDA = -2,    /* CUDA runtime error or no device */
    TCPT_ERR_LIMIT = -3,   /* scene exceeds a compiled limit (BVH depth, lights) */
    TCPT_ERR_NOMEM = -4
};

/* ---- enumerations mirrored from the reference CLI (renderer/src/main.rs:20-53) */
enum { TCPT_INTEGRATOR_PT = 0, TCPT_INTEGRATOR_NEE = 1, TCPT_INTEGRATOR_MIS = 2, /* SrgbRendererPt / Nee / Mis */
       TCPT_INTEGRATOR_ALBEDO = 3, TCPT_INTEGRATOR_NORMAL = 4 }; /* AOV renderers: AlbedoRenderer / NormalRenderer (renderer/src/renderer/{albedo,normal}_renderer.rs); max_depth, sharding by samples and exposure do not apply */
enum { TCPT_SAMPLER_RANDOM = 0, TCPT_SAMPLER_SOBOL = 1 };                          /* RandomSampler / ZSobolSampler */

/* ---- material description (scene/src/material/impls/ constructors; SURVEY.md Appendix C.1) */
enum {
    TCPT_MAT_LAMBERT = 0,       /* LambertMaterial::new(albedo, normal)                         lambert_material.rs:15-31 */
    TCPT_MAT_EMISSIVE = 1,      /* EmissiveMaterial::new(radiance, intensity)                   emissive_material.rs:15-37 */
    TCPT_MAT_PLASTIC = 2,       /* PlasticMaterial::new(eta, color, normal, thin, roughness)    plastic_material.rs:17-52 */
    TCPT_MAT_SIMPLE_PBR = 3,    /* SimplePbrMaterial::new(base, metallic, roughness, normal, ior) simple_pbr_material.rs:38-53 */
    TCPT_MAT_CLEARCOAT_PBR = 4, /* SimpleClearcoatPbrMaterial::new(...)                          simple_pbr_clearcoat_material.rs:17-73 */
    TCPT_MAT_METAL = 5,         /* MetalMaterial::new(metal_type, normal, roughness): color = eta preset, coat_tint = k preset   metal_material.rs:39-110 */
    TCPT_MAT_GLASS = 6          /* GlassMaterial::new(glass_type, normal, thin_surface, roughness): color = eta preset          glass_material.rs:49-86 */
};
/* SpectrumParameter (material/parameter.rs:13-21) over the Spectrum kinds that reach the hot path */
enum {
    TCPT_SPEC_CONSTANT = 0,        /* ConstantSpectrum::new(value[0]) */
    TCPT_SPEC_RGB_ALBEDO_SRGB = 1, /* RgbAlbedoSpectrum::<ColorSrgb>::new(value)        (gamma-encoded sRGB colour) */
    TCPT_SPEC_RGB_ALBEDO_LINEAR = 2, /* RgbAlbedoSpectrum::<ColorSrgbLinear>::new(value) */
    TCPT_SPEC_D65 = 3,             /* presets::cie_illum_d6500() */
    TCPT_SPEC_TEXTURE_SRGB = 4,    /* SpectrumParameter::texture(RgbTexture::load_srgb, SpectrumType::Albedo) */
    TCPT_SPEC_PRESET = 5           /* a DenselySampledSpectrum preset of spectrum/src/presets.rs; `texture` holds the TCPT_PRESET_* id */
};
/* presets::au_eta() ... presets::glass_sf11_eta() (spectrum/src/presets.rs:336-462), in the order the std_tables blob stores them */
enum {
    TCPT_PRESET_AU_ETA = 0, TCPT_PRESET_AU_K, TCPT_PRESET_AG_ETA, TCPT_PRESET_AG_K, TCPT_PRESET_CU_ETA, TCPT_PRESET_CU_K,
    TCPT_PRESET_AL_ETA, TCPT_PRESET_AL_K, TCPT_PRESET_CU_ZN_ETA, TCPT_PRESET_CU_ZN_K,
    TCPT_PRESET_GLASS_BK7, TCPT_PRESET_GLASS_BAF10, TCPT_PRESET_GLASS_FK51A, TCPT_PRESET_GLASS_LASF9, TCPT_PRESET_GLASS_SF5,
    TCPT_PRESET_GLASS_SF10, TCPT_PRESET_GLASS_SF11, TCPT_PRESET_COUNT
};
typedef struct { int32_t kind; float value[3]; int32_t texture; } tcpt_spectrum_param;
typedef struct { int32_t kind; /* 0 constant, 1 gray8 FloatTexture */ float value; int32_t texture; int32_t gamma_corrected; } tcpt_float_param;
typedef struct { int32_t texture; /* -1 = NormalParameter::none() */ int32_t flip_y; } tcpt_normal_param;
typedef struct {
    int32_t type;
    tcpt_spectrum_param color;   /* albedo | radiance | plastic colour | base colour */
    tcpt_float_param intensity;  /* emissive */
    tcpt_normal_param normal;
    float eta;                   /* plastic */
    int32_t thin_surface;        /* plastic */
    tcpt_float_param roughness, metallic, ior;
    tcpt_float_param coat_ior, coat_roughness, coat_thickness;
    tcpt_spectrum_param coat_tint;
} tcpt_material_desc;

/* ---- render parameters = RendererArgs + Camera + SrgbRenderer*::new arguments
 *      (renderer/src/renderer.rs:84-90, camera.rs:26-48, pt_renderer.rs:92-101) */
typedef struct {
    uint32_t width, height, spp, seed, max_depth;
    int32_t integrator, sampler;
    float exposure, fov_deg;
    float cam_pos[3], cam_dir[3], cam_up[3]; /* Camera::set_look_to arguments (normalised again inside, like the reference) */
    /* sharding: this call renders image rows y with y % row_stride == row_offset and sample indices [spp_begin, spp_end)
     * (0,0 = all rows / all samples).  Tile(row) sharding keeps the per-pixel sample order => bitwise equal to one GPU. */
    uint32_t row_offset, row_stride;
    uint32_t spp_begin, spp_end;
    uint32_t max_slots;                      /* wavefront size in paths (0 = default: up to 128 Mi, 304 B of device memory each, at most 45 % of free memory; halved and retried when the allocation fails) */
} tcpt_render_params;

typedef struct {
    uint64_t paths;          /* (pixel, sample) iterations of base_renderer.rs:160 */
    uint64_t closest_rays;   /* Scene::intersect calls   (scene.rs:80) */
    uint64_t shadow_rays;    /* Scene::intersect_p calls (scene.rs:93) */
    uint64_t box_tests, tri_tests; /* only counted when tcpt_set_option(ctx,"count_tests",1) */
    uint64_t kernel_launches;
    double render_ms;        /* device time of the last tcpt_render* (CUDA events) */
    double trace_closest_ms, trace_shadow_ms, shade_ms, generate_ms, film_ms; /* per stage, when option "stage_timing" = 1 */
    uint32_t passes, max_bvh_depth;
    double sobol_prefix_ms;  /* device time of the last build of the ZSobol pixel-prefix table (once per resolution / spp; 0 when reused) */
    uint64_t sobol_prefix_bytes; /* size of that table in device memory */
    double reduce_ms;        /* device time of the film reduce of the last tcpt_render_sharded* (0 on one GPU) */
    uint32_t trace_launches, shade_launches; /* launches of the traversal kernels / the shading kernels among kernel_launches */
} tcpt_stats;

/* ---- context.  tcpt_create returns TCPT_ERR_CUDA when no sm_100 device is usable; *out is then still a context on which only
 * the HOST-side functions work (scene construction, tcpt_get_bvh, tcpt_rgb_to_coeffs, tcpt_get_mesh_tangents, tcpt_last_error):
 * tcpt_set_tables and tcpt_scene_build do their host half and then report TCPT_ERR_CUDA.  Nothing is ever rendered on the CPU. */
int tcpt_create(int device_id, tcpt_ctx** out);
void tcpt_destroy(tcpt_ctx* ctx);
const char* tcpt_last_error(const tcpt_ctx* ctx);
/* options: "count_tests" (box/triangle test counters), "stage_timing" (per-kernel event timing), "blocks_per_sm",
 * "binned_builder" (fast non-reference BVH for synthetic soups), "sobol_prefix" (1: Z-Sobol pixel-digit table, default; 0: recompute
 * every digit per sampler call), "sobol_prefix_mb" (memory cap of that table, default 8192), "sobol_pass" (1: per-pass table of the permuted
 * sample digits shared by all samples of a pixel inside one pass, default; 0: off), "sobol_pass_dims" (dimensions it covers, default 11),
 * "sobol_hash" (1, default: the 64-bit Owen-scramble seeds of the sampler dimensions, a function of (dimension, seed) alone, are read from a
 * 4 KB table built when the seed changes; 0: hashed per sampler call), "illum_half" (1, default: the largest component of an illuminant colour is
 * exactly 0.5 after its normalisation, so its sRGB decoding and z-node interval are constants evaluated once on the device; 0: per lookup;
 * takes effect at the next scene upload), "generate_pixels" (1, default: camera rays of a Z-Sobol pass by one thread per pixel looping over the
 * pass's samples; 0: one thread per path), "sobol_pass_cache" (1, default: the per-pass table is built incrementally from the permutation rows
 * the previous pass left behind; 0: every row recomputed), "refill_b0" / "refill" (1..32: idle lanes at which a warp of the persistent
 * traversal kernel fetches new rays, for the camera-ray launch / the later ones; default 32 / 16: camera rays are coherent, a warp that
 * traces 32 of them to the end also files them into the shading buckets in pixel order),
 * "fused_launches" (bit 0: shadow rays of one bounce and extension rays of the next in one launch, bit 1: all shading buckets in one
 * launch from bounce "fused_shade_from" on; default 3 / 3; 0 = one launch per queue and per bucket), "light_shortcut" (1: a scene whose
 * only light has strictly positive power skips the per-vertex light-power table, its selection probability being exactly 1), "env_nee_table" (1, default: per-texel table of what environment-light sampling computes from the drawn texel alone -- direction, pdf, illuminant
 * coefficients; 32 B per texel, built on the device at scene upload by the code it replaces, bit-transparent; 0: compute per sample), "pin_host_buffers" (1: tcpt_render page-locks the caller's output
 * buffers on first use and keeps them registered while the same pointers are passed; 0: releases them — set 0 before freeing) */
int tcpt_set_option(tcpt_ctx* ctx, const char* name, int value);
/* std_tables = data/std_tables.bin (Sobol matrices 0-1: sampler/sobol_matrices.rs:7; CIE XYZ, D65 and the metal / glass presets:
 * spectrum/src/presets.rs; layout in tools/extract_reference_tables.py);
 * rgb2spec = rgb_to_spec table, 64 z-nodes + [3][64][64][64][3] f32 (spectrum/src/rgb_sigmoid_polynomial.rs:35-84) */
int tcpt_set_tables(tcpt_ctx* ctx, const void* std_tables, size_t std_len, const float* rgb2spec, size_t rgb2spec_floats);

/* ---- host scene construction: replaces scene::Scene::{load_obj, create_primitive, build} (scene/src/scene.rs:54-76).
 * Meshes are passed as the arrays TriangleMesh::load_obj holds after tobj (geometry/impls/triangle_mesh.rs:141-180). */
int tcpt_scene_clear(tcpt_ctx* ctx);
int tcpt_scene_add_mesh(tcpt_ctx* ctx, const float* positions, const float* normals, const float* uvs /*nullable*/, int n_vertices,
                        const uint32_t* indices, int n_triangles);               /* returns geometry index */
/* geometry of CreatePrimitiveDesc::SingleTrianglePrimitive (primitive/impls/single_triangle.rs:24-41): one triangle given inline; it is
 * intersected without any box test, its TLAS box is the box of the transformed vertices and its tangent is not re-orthogonalised.
 * Returns a geometry index for tcpt_scene_add_primitive. */
int tcpt_scene_add_single_triangle(tcpt_ctx* ctx, const float positions[9], const float normals[9], const float uvs[6]);
int tcpt_scene_add_texture(tcpt_ctx* ctx, const uint8_t* data, uint32_t width, uint32_t height, uint32_t channels /*1|3*/);
int tcpt_scene_add_material(tcpt_ctx* ctx, const tcpt_material_desc* desc);
int tcpt_scene_add_primitive(tcpt_ctx* ctx, int geometry, int material, const float local_to_world[16] /*column major*/);
int tcpt_scene_add_env_light(tcpt_ctx* ctx, float intensity, const float* rgb /*h*w*3*/, uint32_t width, uint32_t height,
                             const float local_to_world[16]);                    /* EnvironmentLight::new environment_light.rs:34-84 */
/* CreatePrimitiveDesc::{PointLight,SpotLight,DirectionalLight}Primitive (primitive/repository.rs:108-134; point_light.rs:22-35,
 * spot_light.rs:28-44, directional_light.rs:23-38).  The light sits at the local origin / shines along local +z; angles in radians. */
enum { TCPT_LIGHT_POINT = 3, TCPT_LIGHT_SPOT = 4, TCPT_LIGHT_DIRECTIONAL = 5 };   /* = tcpt_flat_primitive.kind */
int tcpt_scene_add_delta_light(tcpt_ctx* ctx, int kind, float intensity, const tcpt_spectrum_param* spectrum, float angle_inner, float angle_outer,
                               const float local_to_world[16]);
/* ---- asset ingestion.  Scene::load_obj (scene.rs:54-57) = TriangleMesh::load_obj (geometry/impls/triangle_mesh.rs:141-243): tobj 4.0.3
 * load_obj with { single_index, triangulate, ignore_points, ignore_lines } and the reference's concatenation of the returned models
 * (no vertex offset between models; see csrc/host_obj.h for the rules and the two quirks).  tcpt_obj_* hand the arrays to the caller
 * (counts = {position vertices, normal vertices, texcoord vertices, triangles, models}; copy: any pointer may be NULL; tangent_tri[j] =
 * the triangle whose load-time tangent triangle j receives, identity for one-model files).  tcpt_scene_load_obj adds the mesh to the
 * scene and returns its geometry index; TCPT_ERR_INVALID when the file does not parse, lacks vn normals (the reference panics:
 * triangle_mesh.rs:57-61) or carries texcoords for only some vertices. */
typedef struct tcpt_obj tcpt_obj;
int tcpt_obj_load(const char* path, tcpt_obj** out, char* err /*nullable*/, size_t err_len);
int tcpt_obj_counts(const tcpt_obj* obj, uint32_t counts[5]);
int tcpt_obj_copy(const tcpt_obj* obj, float* positions, float* normals, float* texcoords, uint32_t* indices, uint32_t* tangent_tri);
void tcpt_obj_free(tcpt_obj* obj);
int tcpt_scene_load_obj(tcpt_ctx* ctx, const char* path);
/* triangle j of `geometry` takes the load-time tangent of triangle tri[j] (multi-model OBJ files, see above) */
int tcpt_scene_set_tangent_source(tcpt_ctx* ctx, int geometry, const uint32_t* tri, int n_triangles);
/* The `image` crate's (0.25.6) buffer conversions behind the texture loaders (texture/loader.rs:43-87: anything that is not Rgb8 / Rgb32F resp.
 * Luma8 / LumaA8 goes through DynamicImage::to_rgb8 / to_luma8; environment_light.rs:36-37: to_rgb32f), for an already DECODED image
 * (rules in csrc/host_image.h).  src = height*width*channels samples, channels 1 L | 2 LA | 3 RGB | 4 RGBA; sample_type 0 u8 | 1 u16 | 2 f32;
 * dst_kind 0 = rgb8 (u8 x 3 per pixel), 1 = luma8 (u8), 2 = rgb32f (f32 x 3). */
int tcpt_image_convert(const void* src, uint32_t width, uint32_t height, uint32_t channels, int sample_type, int dst_kind, void* dst);
/* Scene::build(&camera): bakes world_to_render = translate(-cam_pos), builds BLAS/TLAS with the reference's exact SAH topology,
 * flattens to the device layout and uploads (scene.rs:64-76, bvh.rs:92-295). */
int tcpt_scene_build(tcpt_ctx* ctx, const float cam_pos[3]);

/* ---- the hot path: replaces RendererImage::<SrgbRenderer{Pt,Nee,Mis}>::render::<S>() (renderer/src/renderer.rs:120-134).
 * out_acc  : host, width*height*3 f32, the Sensor accumulators (sum over samples of exposed linear-sRGB; sensor.rs:76-77)
 * out_srgb : host, optional, width*height*3 f32 after /spp, clip, Reinhard, sRGB OETF (sensor.rs:81-88) — what `pixels` holds */
int tcpt_render(tcpt_ctx* ctx, const tcpt_render_params* params, float* out_acc, float* out_srgb);
/* same, accumulating into a DEVICE buffer (width*height*3 f32) for multi-GPU film reduction; stream = cudaStream_t or NULL */
int tcpt_render_device(tcpt_ctx* ctx, const tcpt_render_params* params, void* dev_acc, void* stream);
/* Sensor::to_rgb on a device accumulator (after the NCCL reduce): dev_srgb = OETF(Reinhard(max(acc/spp,0))) */
int tcpt_finalize_device(tcpt_ctx* ctx, const void* dev_acc, uint32_t width, uint32_t height, uint32_t spp, void* dev_srgb, void* stream);
/* ---- adaptive sampling: the job `params` (spp = N) runs in rounds.  Round 0 renders samples [0, min_spp) of every pixel, every later
 * round the next `step` samples (clipped at N) of the pixels still active.  After a round that ends at k < N an active pixel stops with
 * count k when S1 and S2 are finite and e < threshold * (|m| + 1e-3), where, in f32 without contraction, y = (0.2126 r + 0.7152 g) +
 * 0.0722 b of each sample's sensor RGB, S1 = sum y, S2 = sum y*y in sample order, m = S1/k, v = max(S2/k - m*m, 0), e = sqrt(v/(k - 1)).
 * A pixel that never stops has count N.  A pixel with count k holds BITWISE the accumulator tcpt_render gives for the window [0, k) of the
 * same job.  Outputs (host, any may be NULL, not all three): out_acc W*H*3 f32 sums, out_srgb W*H*3 f32 (tcpt_render's output transform
 * with each pixel divided by its own count), out_spp W*H u32 counts.  Stats: paths = sum of the counts, render_ms = the whole call,
 * passes / kernel_launches over all rounds.  Integrators pt / nee / mis, both samplers; max_slots is honoured; row_offset / row_stride
 * and spp_begin / spp_end must be 0.  TCPT_ERR_INVALID: threshold negative or not finite, min_spp < 2 or > spp, step 0.  A communicator on
 * the context (tcpt_comm_init, a tcpt_group context) is not used: the whole frame is rendered and returned by this GPU alone, on any rank
 * (tcpt_render_adaptive_sharded is the multi-GPU form). */
typedef struct { float threshold; uint32_t min_spp; uint32_t step; } tcpt_adaptive_params;
int tcpt_render_adaptive(tcpt_ctx* ctx, const tcpt_render_params* params, const tcpt_adaptive_params* ap,
                         float* out_acc, float* out_srgb, uint32_t* out_spp);
/* One row shard of an adaptive job into caller-owned DEVICE buffers on `stream` (cudaStream_t or NULL, as in tcpt_render_device); no
 * collective.  `params` may carry a row shard, any row_offset < row_stride as tcpt_shard_params(..., TCPT_SHARD_TILE, ...) makes it;
 * spp_begin / spp_end must be 0 (tcpt_shard_params writes the job's range [0, spp) there: reset both).  The rounds, the rule and the checks on `ap` and the integrator are those of tcpt_render_adaptive, over
 * the owned pixels only: each owned pixel stops exactly where it stops in tcpt_render_adaptive of the whole job.  dev_acc (W*H*3 f32) and
 * dev_spp (W*H u32) are both required: each owned pixel's sum is ADDED into dev_acc (the caller zeroes it) and its count WRITTEN into
 * dev_spp; no other pixel of either buffer is touched.  Stats: paths = sum of the owned counts, render_ms = the whole call.
 * TCPT_ERR_INVALID: as tcpt_render_adaptive, a null buffer, row_offset >= row_stride (row_stride 0 = the whole frame). */
int tcpt_render_adaptive_device(tcpt_ctx* ctx, const tcpt_render_params* params, const tcpt_adaptive_params* ap,
                                void* dev_acc, void* dev_spp, void* stream);
int tcpt_get_stats(const tcpt_ctx* ctx, tcpt_stats* out);

/* ---- multi-GPU (SURVEY.md 8b / 8e).  The reference has no distributed path; every (pixel, sample) is independent and the only shared
 * output is the per-pixel Sensor accumulator (sensor.rs:76-77), so a frame is split across GPUs and summed once.  The library owns
 * the NCCL communicator (libnccl.so.2 is opened when the first one is made; a single-GPU host never loads it).
 *   one process per GPU : tcpt_create -> tcpt_comm_init(nranks, rank, id) on every rank (id from tcpt_comm_get_unique_id on one rank,
 *                         handed over by any transport) -> tcpt_render_sharded on every rank, same job
 *   one process, N GPUs : tcpt_group_* below (one context per GPU, one host thread per GPU inside tcpt_group_render)
 * shard modes: TILE = rank r renders rows y % nranks == r with every sample: the reduced film is BITWISE the one-GPU film;
 *              SPP  = rank r renders an equal slice of the job's sample indices of every pixel: best balance, sums re-associated.
 * Exactly one collective per frame: ncclReduce(sum) of width*height*3 f32 onto rank 0, then Sensor::to_rgb and ONE device -> host
 * copy per requested buffer on rank 0. */
#define TCPT_COMM_ID_BYTES 128
enum { TCPT_SHARD_TILE = 0, TCPT_SHARD_SPP = 1 };
int tcpt_comm_get_unique_id(void* id128);
int tcpt_comm_init(tcpt_ctx* ctx, int nranks, int rank, const void* id128);   /* collective: every rank calls it */
int tcpt_comm_destroy(tcpt_ctx* ctx);
/* the slice of `job` rank `rank` of `nranks` renders (pure function; job->row_offset / row_stride must be 0, [spp_begin, spp_end) = the
 * job's sample range, 0,0 = all `spp`) */
int tcpt_shard_params(const tcpt_render_params* job, int shard_mode, int rank, int nranks, tcpt_render_params* out);
/* One complete frame from all ranks.  Every rank passes the SAME job; out_acc / out_srgb (host, width*height*3 f32, either may be NULL)
 * are written on rank 0 only and may be NULL elsewhere.  out_srgb = Sensor::to_rgb over the job's sample count.  Without a
 * communicator (one GPU) it is tcpt_render. */
int tcpt_render_sharded(tcpt_ctx* ctx, const tcpt_render_params* job, int shard_mode, float* out_acc, float* out_srgb);
/* same, accumulating into a caller-owned DEVICE buffer (zeroed by the caller) on `stream`; after the call rank 0's buffer holds the sum */
int tcpt_render_sharded_device(tcpt_ctx* ctx, const tcpt_render_params* job, int shard_mode, void* dev_acc, void* stream);
/* One complete ADAPTIVE frame (tcpt_render_adaptive) from all ranks.  Every rank passes the SAME whole-frame job (row_offset / row_stride,
 * spp_begin / spp_end 0) and `ap`; rank r runs the rounds over its TILE shard alone (a rank without rows renders nothing but still joins
 * the collective) with no collective per round: the rule reads only a pixel's own moments, so the frame -- accumulators, counts, sRGB --
 * is BITWISE tcpt_render_adaptive's.  Then ONE grouped collective on the rendering stream: ncclReduce(sum) of the W*H*3 f32 accumulators
 * and of the W*H u32 counts onto rank 0 (exact: every pixel not owned by a rank is +0 / 0 there).  Rank 0 applies the per-count output
 * transform and makes one device -> host copy per requested buffer (out_acc, out_srgb, out_spp as in tcpt_render_adaptive; not all NULL);
 * on the other ranks they may be NULL and are never written.  Stats as tcpt_render_adaptive over this rank's shard, reduce_ms as
 * tcpt_render_sharded_device.  Without a communicator it is tcpt_render_adaptive.  No shard mode: the rule needs every sample of a pixel on
 * one rank. */
int tcpt_render_adaptive_sharded(tcpt_ctx* ctx, const tcpt_render_params* job, const tcpt_adaptive_params* ap,
                                 float* out_acc, float* out_srgb, uint32_t* out_spp);

typedef struct tcpt_group tcpt_group;
int tcpt_group_create(const int* device_ids, int n, tcpt_group** out);     /* n contexts + one communicator clique */
void tcpt_group_destroy(tcpt_group* g);
int tcpt_group_size(const tcpt_group* g);
tcpt_ctx* tcpt_group_context(tcpt_group* g, int i);                        /* describe the scene on context 0 (tcpt_scene_add_*) */
const char* tcpt_group_last_error(const tcpt_group* g);
int tcpt_group_set_tables(tcpt_group* g, const void* std_tables, size_t std_len, const float* rgb2spec, size_t rgb2spec_floats);
int tcpt_group_build(tcpt_group* g, const float cam_pos[3]);               /* Scene::build on context 0, replica on every other GPU */
int tcpt_group_render(tcpt_group* g, const tcpt_render_params* job, int shard_mode, float* out_acc, float* out_srgb);
/* tcpt_render_adaptive_sharded on every GPU of the group, one host thread per GPU; out_* filled from device 0 */
int tcpt_group_render_adaptive(tcpt_group* g, const tcpt_render_params* job, const tcpt_adaptive_params* ap,
                               float* out_acc, float* out_srgb, uint32_t* out_spp);

/* ---- synthetic triangle soups (BASELINE.json configs[4], 1 M - 100 M triangles): a TRAVERSAL-ONLY scene whose BVH is built on the device
 * (Morton order + radix tree, collapsed to the 4-wide records the traversal kernels read: csrc/lbvh.cuh; the reference's O(N^2) builder is
 * a parity requirement for the config scenes only).  triangles = n_triangles x 9 floats on the host (world space = Render space, one
 * primitive with the identity transform, primitive index 0, triangle index = position in the array).  Afterwards tcpt_trace /
 * tcpt_trace_device work; tcpt_render* refuse.  Refused before any device work: n_triangles = 0 or option "soup_leaf" outside [1, 16]
 * (TCPT_ERR_INVALID), n_triangles >= 2^27 - 16 (TCPT_ERR_LIMIT).  tcpt_soup_build_info: device time of the build, 128-byte records, wide levels. */
int tcpt_scene_build_soup(tcpt_ctx* ctx, const float* triangles, uint32_t n_triangles);
int tcpt_soup_build_info(const tcpt_ctx* ctx, double* build_ms, uint64_t* n_records, uint32_t* levels);

/* ---- single stages, exposed for parity tests and the traversal micro-benchmark */
/* rays: n x {o[3], d[3], tmax}; out: n x {prim, tri, t bits, b0 bits, b1 bits, b2 bits} (prim -1 = miss; any_hit: out[0] = 0|1) */
int tcpt_trace(tcpt_ctx* ctx, const float* rays, int n, int any_hit, int32_t* out_hit);
/* device-resident variant used by the micro-benchmark (SoA, fully coalesced):
 * dev_rays = n x float4 {o.xyz, tmax} followed by n x float4 {d.xyz, -}; dev_hits = n x float4 {t,b0,b1,b2} followed by n x uint2 {prim,tri} */
int tcpt_trace_device(tcpt_ctx* ctx, const void* dev_rays, int n, int any_hit, void* dev_hits, void* stream);
int tcpt_sampler_stream(tcpt_ctx* ctx, int sampler, uint32_t spp, uint32_t width, uint32_t height, uint32_t seed, uint32_t px,
                        uint32_t py, uint32_t sample_index, const int32_t* kinds /*1 = get_1d, 2 = get_2d*/, int n, float* out);
/* the CDF search of EnvironmentLight::sample_infinite_light (environment_light.rs:218-223: slice::binary_search_by + clamp) as the device runs it:
 * cdf = n non-decreasing values, guide_cells = a power of two (the device's guide table is built for it), u = m numbers, out = m indices */
int tcpt_cdf_search(tcpt_ctx* ctx, const float* cdf, uint32_t n, uint32_t guide_cells, const float* u, int m, uint32_t* out);
/* RGB contribution of individual (pixel, sample) paths = what Sensor::add_sample adds for that sample */
int tcpt_path_samples(tcpt_ctx* ctx, const tcpt_render_params* params, const uint32_t* pixels_xy, const uint32_t* sample_indices,
                      int n, float* out_rgb);

/* ---- host-side introspection for bit-exactness tests (BVH topology, table indexing, load-time tangents) */
/* which = -1: TLAS, else geometry index.  Records of 8 x u32 in the REFERENCE's flattened order (bvh.rs:234-295):
 * {kind 0 inner|1 leaf|2 item, value = second_offset|item_count|item, min.xyz bits, max.xyz bits}.  Returns the node count. */
int tcpt_get_bvh(tcpt_ctx* ctx, int which, uint32_t* out, int max_nodes);
/* the DEVICE layout of the same BVH (include/tcpt_flat.h): 4-wide records of 32 x u32 (rows lo.x hi.x lo.y hi.y lo.z hi.z entries counts).
 * Entries are absolute: *first_record = index of record 0 of this BVH in the flat node array, *slot_base = its first item slot.
 * Returns the record count.  The tests check that every reference leaf survives the collapse with its box bits and item order. */
int tcpt_get_wide_bvh(tcpt_ctx* ctx, int which, uint32_t* out, int max_records, uint32_t* first_record, uint32_t* slot_base);
int tcpt_build_bvh_boxes(const float* boxes /*n x {min[3],max[3]}*/, int n, uint32_t* out, int max_nodes); /* builder alone, no device */
int tcpt_rgb_to_coeffs(tcpt_ctx* ctx, const float rgb[3], int gamma_encoded, float coeffs[3], int32_t index[4] /*m,zi,yi,xi*/);
int tcpt_get_mesh_tangents(tcpt_ctx* ctx, int geometry, float* out, int max_triangles);

#ifdef __cplusplus
}
#endif
#endif /* TCPT_H */
