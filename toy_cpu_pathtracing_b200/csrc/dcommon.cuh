// Device-side common definitions: math helpers, device scene view, wavefront buffers, samplers, spectra, textures.
// Compiled with --fmad=false: the parity-critical arithmetic (slab test, watertight triangle test, instance transforms,
// Sobol float conversion, table indexing) must round exactly like the reference's unfused f32 operations
// (SURVEY.md Appendix D, last bullet).  Shading arithmetic shares the flag (measured cost: see DESIGN.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tcpt_flat.h"

namespace tcpt {

#define TCPT_PI 3.14159265358979323846f
#define TCPT_FLT_MAX 3.402823466e+38f
#define TCPT_INF __int_as_float(0x7f800000)

// ---------------------------------------------------------------- float3 helpers (component order as in glam's scalar Vec3)
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float3 operator/(float3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
__device__ __forceinline__ float dot(float3 a, float3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
__device__ __forceinline__ float3 cross(float3 a, float3 b) { return f3(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y); }
__device__ __forceinline__ float length_squared(float3 a) { return dot(a, a); }
__device__ __forceinline__ float length(float3 a) { return sqrtf(dot(a, a)); }
__device__ __forceinline__ float3 normalize(float3 a) { return a * (1.0f / length(a)); }
__device__ __forceinline__ float comp(float3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
// Rust f32::max/min ignore a NaN operand; CUDA fmaxf/fminf have the same rule
__device__ __forceinline__ float rmax(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ float rmin(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float signum(float x) { return isnan(x) ? x : (signbit(x) ? -1.0f : 1.0f); }
__device__ __forceinline__ float clampf(float x, float lo, float hi) { return x < lo ? lo : (x > hi ? hi : x); }
__device__ __forceinline__ uint32_t f2u_sat(float x) { return __float2uint_rz(x); }  // saturating, NaN -> 0, like Rust `as u32`

// 3x4 affine stored as four columns of xyz (tcpt_flat_primitive::l2r / r2l)
__device__ __forceinline__ float3 xf_point(const float* __restrict__ m, float3 p) {
    return f3(((m[0] * p.x + m[3] * p.y) + m[6] * p.z) + m[9], ((m[1] * p.x + m[4] * p.y) + m[7] * p.z) + m[10],
              ((m[2] * p.x + m[5] * p.y) + m[8] * p.z) + m[11]);
}
__device__ __forceinline__ float3 xf_vector(const float* __restrict__ m, float3 v) {
    return f3((m[0] * v.x + m[3] * v.y) + m[6] * v.z, (m[1] * v.x + m[4] * v.y) + m[7] * v.z, (m[2] * v.x + m[5] * v.y) + m[8] * v.z);
}
// Transform * Normal = transpose(inverse(M)) * n, re-normalised: pass the INVERSE matrix (math/src/transform.rs:44-51)
__device__ __forceinline__ float3 xf_normal_by_inverse(const float* __restrict__ inv, float3 n) {
    float3 r = f3((inv[0] * n.x + inv[1] * n.y) + inv[2] * n.z, (inv[3] * n.x + inv[4] * n.y) + inv[5] * n.z, (inv[6] * n.x + inv[7] * n.y) + inv[8] * n.z);
    return normalize(r);
}

// 3x3 linear part of the tangent-frame transforms (column major: c0, c1, c2).  The reference builds a glam Mat4 from three
// columns and calls Mat4::inverse (math/src/transform.rs:186-203, 216-244); with last row/column (0,0,0,1) the cofactor scheme
// reduces to the expressions below term by term (the vanished terms are exact zeros), so the values match the 4x4 inverse.
struct M3 { float3 c0, c1, c2; };
__device__ __forceinline__ M3 m3_inverse(const M3& s) {
    const float m00 = s.c0.x, m01 = s.c0.y, m02 = s.c0.z, m10 = s.c1.x, m11 = s.c1.y, m12 = s.c1.z, m20 = s.c2.x, m21 = s.c2.y, m22 = s.c2.z;
    M3 r;
    r.c0 = f3(m11 * m22 - m12 * m21, -(m01 * m22 - m02 * m21), m01 * m12 - m02 * m11);
    r.c1 = f3(-(m10 * m22 - m12 * m20), m00 * m22 - m02 * m20, -(m00 * m12 - m02 * m10));
    r.c2 = f3(m10 * m21 - m11 * m20, -(m00 * m21 - m01 * m20), m00 * m11 - m01 * m10);
    const float det = (m00 * r.c0.x + m01 * r.c1.x) + m02 * r.c2.x;
    const float rcp = 1.0f / det;
    r.c0 = r.c0 * rcp; r.c1 = r.c1 * rcp; r.c2 = r.c2 * rcp;
    return r;
}
__device__ __forceinline__ float3 m3_vector(const M3& m, float3 v) { return (m.c0 * v.x + m.c1 * v.y) + m.c2 * v.z; }
// Transform * Normal with the per-call inverse().transpose() (math/src/transform.rs:44-51): pass inverse(M)
__device__ __forceinline__ float3 m3_normal_by_inverse(const M3& inv, float3 n) {
    return normalize(f3((inv.c0.x * n.x + inv.c0.y * n.y) + inv.c0.z * n.z, (inv.c1.x * n.x + inv.c1.y * n.y) + inv.c1.z * n.z,
                        (inv.c2.x * n.x + inv.c2.y * n.y) + inv.c2.z * n.z));
}

// ---------------------------------------------------------------- 4-lane spectra (spectrum/src/sampled_spectrum.rs)
struct S4 { float v[4]; };
__device__ __forceinline__ S4 s4(float c) { S4 r; r.v[0] = r.v[1] = r.v[2] = r.v[3] = c; return r; }
__device__ __forceinline__ S4 s4(float4 a) { S4 r; r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; return r; }
__device__ __forceinline__ float4 to_f4(const S4& a) { return make_float4(a.v[0], a.v[1], a.v[2], a.v[3]); }
#define S4_BINOP(op)                                                                                                   \
    __device__ __forceinline__ S4 operator op(const S4& a, const S4& b) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = a.v[i] op b.v[i]; return r; }
S4_BINOP(+) S4_BINOP(-) S4_BINOP(*)
__device__ __forceinline__ S4 operator*(const S4& a, float s) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = a.v[i] * s; return r; }
__device__ __forceinline__ S4 operator*(float s, const S4& a) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = s * a.v[i]; return r; }
// division by zero yields zero (sampled_spectrum.rs:59-83)
__device__ __forceinline__ S4 operator/(const S4& a, float s) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = s == 0.0f ? 0.0f : a.v[i] / s; return r; }
__device__ __forceinline__ S4 operator/(const S4& a, const S4& b) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = b.v[i] == 0.0f ? 0.0f : a.v[i] / b.v[i]; return r; }
__device__ __forceinline__ float s4_max(const S4& a) { return rmax(rmax(rmax(rmax(-TCPT_INF, a.v[0]), a.v[1]), a.v[2]), a.v[3]); }
__device__ __forceinline__ float s4_avg(const S4& a) { return ((((0.0f + a.v[0]) + a.v[1]) + a.v[2]) + a.v[3]) / 4.0f; }
__device__ __forceinline__ bool s4_is_constant(const S4& a) { return a.v[1] == a.v[0] && a.v[2] == a.v[0] && a.v[3] == a.v[0]; }
__device__ __forceinline__ S4 s4_sqrt(const S4& a) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = sqrtf(a.v[i]); return r; }
__device__ __forceinline__ S4 s4_clamp(const S4& a, float lo, float hi) { S4 r; _Pragma("unroll") for (int i = 0; i < 4; ++i) r.v[i] = clampf(a.v[i], lo, hi); return r; }

// ---------------------------------------------------------------- device scene view
struct DTexture { const uint8_t* data; uint32_t w, h, channels, pad; };
struct DEnv {
    const float* data; const float* marginal; const float* conditional;
    const uint32_t* marginal_guide; const uint32_t* conditional_guide; uint32_t guide_h, guide_w;
    float intensity, total_weight; uint32_t w, h; tcpt_flat_spectrum integrated; int32_t primitive;
    // per texel {wi_render.xyz, pdf_dir}, {sigmoid coefficients, scale}: everything light sampling computes that only depends on WHICH texel
    // was drawn (see env_nee_texel, kernels.cuh k_env_nee_table); null = compute per sample (option "env_nee_table" 0)
    const float4* nee_table;
};
struct DScene {
    const float4* nodes;            // 8 x float4 per 4-wide record (include/tcpt_flat.h)
    const int2* tlas_items;         // {primitive, leaf_first_slot}
    const float4* tri_verts;        // 3 x float4 per slot
    const float* positions; const float* normals; const float* uvs; const uint32_t* indices; const float* tangents;
    const tcpt_flat_geometry* geometries;
    const tcpt_flat_primitive* primitives; uint32_t n_primitives;
    const tcpt_flat_material* materials;
    const uint8_t* prim_mat_type;   // material type of every primitive (0xff: none), so that filing a hit into its shading bucket is one load
    const DTexture* textures;
    const float* area_list; const float* area_table;
    int32_t light_list[TCPT_MAX_LIGHTS]; uint32_t n_lights;
    uint32_t one_light_always_on;   // one light, power finite and > 0 at every wavelength: it is chosen with probability exactly 1 (see tcpt_upload_flat_scene)
    const DEnv* envs; uint32_t n_envs;
    const float4* cmf;              // 470 x {x_bar, y_bar, z_bar, d65}  (spectrum/src/presets.rs tables, densely resampled)
    const float* z_nodes; const float* rgb2spec;
    // srgb_to_linear(0.5f) as THIS build's device code evaluates it, and its z-node interval (k_illum_half, once per table upload): the largest
    // component of an RgbIlluminantSpectrum's colour is exactly 0.5 after the division by 2 * max (rgb_illuminant_spectrum.rs:27-40), so one of
    // the three decodings and the node search of every environment lookup are constants.  half_zi < 0: not available, compute per call.
    float half_lin; int32_t half_zi;
    const float* presets;           // dense metal / glass tables (spectrum/src/presets.rs), n x 470
    float xyz_to_rgb[9];            // column major (color/src/gamut.rs:43-69)
};

struct DCamera { float3 s, u, nf; float scale, aspect; };

struct DRender {
    uint32_t width, height, spp, seed, max_depth;
    int32_t integrator, sampler;
    float exposure;
    uint32_t log2_spp, n_base4_digits;  // ZSobolSampler::new (z_sobol_sampler.rs:179-196)
    // pass geometry: slot = s_local * n_pix + p_local ; owned pixel index = pix_begin + p_local ;
    // owned pixel k -> x = k % width, y = row_offset + (k / width) * row_stride ; sample_index = s_begin + s_local
    // (with pix_list != nullptr the owned pixel index is pix_list[pix_begin + p_local] instead: a subset of the owned pixels, see owned_pixel)
    uint32_t n_pix, pix_begin, s_begin, s_count, row_offset, row_stride;
    const uint32_t* pix_list;
    // exact division of a 32-bit number by n_pix / by width as one 64 x 64 -> high multiply: magic = floor(2^64 / d) + 1 (0 = divisor 1);
    // floor(n * magic / 2^64) == n / d for every n < 2^32 because n * (magic * d - 2^64) <= n * d < 2^64 (set by set_div_magics on the host)
    uint64_t n_pix_magic, width_magic;
    // ZSobol pixel-prefix table (see DSampler::sample_index): prefix[dim * prefix_stride + y * width + x], dims < prefix_dims
    const uint32_t* sobol_prefix; uint32_t prefix_dims, prefix_stride;
    // ZSobol pass table (see DSampler::sample_index): rows prefix_dims .. prefix_dims + pass_dims of the same allocation, rebuilt for
    // every pass by k_sobol_pass.  pass_info = pass_dims | n_varying_digits << 8 (0 = no pass table)
    uint32_t pass_info;
    // hash(k, seed) of DSampler::hash for k < TCPT_SOBOL_HASH_N (the Owen-scramble seeds of sampler dimension k - 1 / k - 2): frame constants,
    // built by k_sobol_hash when the seed changes (nullptr: computed per call)
    const unsigned long long* sobol_hash;
};
#define TCPT_SOBOL_HASH_N 512

// An entry of the bucketed shading order: {queue position, path slot}.  The slot rides along so that the head of the path state is
// asked for together with the ray and the hit record instead of after the ray has arrived (one round trip less in front of every vertex).
typedef uint2 OrderEntry;

// Wavefront buffers.  Path state is a structure of arrays of 16-byte records indexed by path slot; ray queues, hit records
// and shadow queues are indexed by QUEUE POSITION so every stage reads and writes them fully coalesced.
struct DState {
    float4* thr; float4* con; float4* fprev; float4* misc;  // misc = {pdf_prev, lambda0, bits(dim), bits(flags | depth << 8)}
    float4* ppos;                                           // previous path vertex (MIS light pdf needs it)
    float4* rgb;                                            // per-path sensor contribution, reduced per pixel by k_film
    float4* ext_o[2]; float4* ext_d[2];                     // {o.xyz, tmax} | {d.xyz, bits(slot)}   (ping-pong)
    float4* hit0; uint2* hit1;                              // {t, b0, b1, b2} | {prim, tri}
    float4* sh_o; float4* sh_d; float4* sh_c;               // shadow ray + pending NEE contribution (sh_d.w = slot | finalize << 31)
    OrderEntry* order; uint32_t capacity;                   // TCPT_N_BUCKETS x capacity order entries, bucketed by shading work
    uint32_t* counters;                                     // [0],[1] extension queue sizes (ping-pong), [2] shadow queue size,
                                                            // [4..10), [12..18) bucket sizes of even / odd bounces
    unsigned long long* stats;                              // [0] closest rays [1] shadow rays [2] box tests [3] tri tests [4] paths
};

enum : uint32_t { FLAG_SPEC_PREV = 1u, FLAG_LAMBDA_TERMINATED = 2u, FLAG_SAMPLED_PREV = 4u };

// ---------------------------------------------------------------- samplers
__constant__ uint32_t c_sobol_dim1[52];  // SOBOL_MATRICES_32[52..104) (dimension 1); dimension 0 is the bit reversal
// the same matrix folded per index byte: tab[pos * 256 + b] = XOR of c_sobol_dim1[8 * pos + i] over the set bits i of b
// (7 x 256 words in global memory, L1 resident); XOR is associative, so 5-7 gathers replace up to 52 bit-serial steps
__constant__ const uint32_t* c_sobol_dim1_bytes;

// Z-Sobol / counter-hash sampler.  The per-path part is four registers (Morton index, dimension counter, counter-hash key, pixel
// index); everything the frame fixes (seed, log2 spp, digit count, tables) is read from the kernel parameters at the call.  The heavy
// work sits in two __noinline__ functions that take every input BY VALUE: as member functions they took `this`, which forced the
// sampler into the caller's stack frame and turned every field read of every call into a local-memory load.
__device__ __forceinline__ uint32_t div_magic(uint32_t n, uint64_t magic) { return magic ? (uint32_t)__umul64hi((uint64_t)n, magic) : n; }
struct SobolFrame {  // the frame-constant inputs of a Sobol call, packed for the by-value call
    const uint32_t* prefix;   // DRender::sobol_prefix (nullptr: no tables)
    uint32_t prefix_stride, tables;  // tables = prefix_dims | pass_dims << 16 | n_varying_digits << 24
    uint32_t cfg;             // log2_spp | n_base4_digits << 8
    uint32_t seed;
    const unsigned long long* hash_table;   // DRender::sobol_hash
};
struct DSampler {
    uint32_t morton, dim, key, pix;

    __device__ __forceinline__ static uint32_t part1by1(uint32_t x) {  // left_shift2 of a 32-bit value truncated to u32 (z_sobol_sampler.rs:54-65)
        x &= 0x0000ffffu;
        x = (x ^ (x << 8)) & 0x00ff00ffu;
        x = (x ^ (x << 4)) & 0x0f0f0f0fu;
        x = (x ^ (x << 2)) & 0x33333333u;
        x = (x ^ (x << 1)) & 0x55555555u;
        return x;
    }
    __device__ __forceinline__ static uint64_t mix_bits(uint64_t v) {
        v ^= v >> 31; v *= 0x7fb5d329728ea185ull; v ^= v >> 27; v *= 0x81dadef4bc2dd44dull; v ^= v >> 33;
        return v;
    }
    __device__ __forceinline__ static uint64_t hash(uint32_t dimension, uint32_t seed) {  // MurmurHash64A (z_sobol_sampler.rs:76-99)
        const uint64_t M = 0xc6a4a7935bd1e995ull;
        uint64_t h = 8ull * M;
        uint64_t k = (uint64_t)dimension | ((uint64_t)seed << 32);
        k *= M; k ^= k >> 47; k *= M;
        h ^= k; h *= M;
        h ^= h >> 47; h *= M; h ^= h >> 47;
        return h;
    }
    // hash(k, f.seed) from the frame's table (three 64-bit multiplies of dependent latency less per sampler call)
    __device__ __forceinline__ static uint64_t hash_of(uint32_t k, const SobolFrame& f) {
        if (f.hash_table != nullptr && k < (uint32_t)TCPT_SOBOL_HASH_N) return __ldg(f.hash_table + k);
        return hash(k, f.seed);
    }
    __device__ __forceinline__ static uint32_t owen(uint32_t v, uint32_t seed) {  // FastOwenScrambler (z_sobol_sampler.rs:3-29)
        v = __brev(v);
        v ^= v * 0x3d20adeau; v += seed; v *= (seed >> 16) | 1u; v ^= v * 0x05526c56u; v ^= v * 0x53a22864u;
        return __brev(v);
    }
    __device__ __forceinline__ static uint32_t pcg_hash2(uint32_t key, uint32_t ctr) {
        uint32_t x = key * 747796405u + ctr * 2891336453u + 0x9e3779b9u;
        x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
        uint32_t w = ((x >> ((x >> 28u) + 4u)) ^ x) * 277803737u;
        return (w >> 22u) ^ w;
    }
    __device__ __forceinline__ static float unit_float(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }
    __device__ __forceinline__ static float to_unit(uint32_t v) { return fminf((float)v * 2.3283064365386963e-10f, 0.99999994f); }

    __device__ __forceinline__ static uint32_t morton_of(uint32_t px, uint32_t py, uint32_t sample_index, uint32_t log2_spp) {
        // encode_morton2 computes in u64 then truncates to u32: only the low 16 bits of x and y survive (z_sobol_sampler.rs:54-66)
        return (((part1by1(py) << 1) | part1by1(px)) << log2_spp) | sample_index;
    }
    __device__ __forceinline__ void start(const DRender& R, uint32_t px, uint32_t py, uint32_t sample_index) {
        dim = 0;
        morton = morton_of(px, py, sample_index, R.log2_spp);
        key = (px * 0x9e3779b9u) ^ (py * 0x85ebca6bu) ^ (sample_index * 0xc2b2ae35u) ^ R.seed;
        pix = py * R.width + px;
    }
    __device__ __forceinline__ static SobolFrame frame_of(const DRender& R) {
        SobolFrame f;
        f.prefix = R.sobol_prefix; f.prefix_stride = R.prefix_stride;
        f.tables = R.sobol_prefix ? (R.prefix_dims | (R.pass_info << 16)) : 0u;
        f.cfg = R.log2_spp | (R.n_base4_digits << 8); f.seed = R.seed; f.hash_table = R.sobol_hash;
        return f;
    }

    __device__ __forceinline__ static uint32_t perm_digit(uint32_t p, uint32_t digit) {
        // rows of PERMUTATIONS (z_sobol_sampler.rs:102-127): one byte per row, digit d stored at bits [2d, 2d+2).  The 24 bytes
        // live in six immediates; the row is picked with three byte-permutes and mask arithmetic, so there is no table in
        // memory and no branch (a ?: chain compiled to six divergent paths: 7 of 32 lanes active in the first profile).
        const uint32_t k = p & 7u, g = p >> 3;
        const uint32_t r0 = __byte_perm(0x78D8B4E4u, 0xB1E19C6Cu, k), r1 = __byte_perm(0x8D2D39C9u, 0x72D236C6u, k), r2 = __byte_perm(0x87271E4Eu, 0x93634B1Bu, k);
        const uint32_t m0 = 0u - (uint32_t)(g == 0u), m1 = 0u - (uint32_t)(g == 1u), m2 = 0u - (uint32_t)(g == 2u);
        const uint32_t row = (r0 & m0) | (r1 & m1) | (r2 & m2);
        return (row >> (2u * digit)) & 3u;
    }
    // (v >> 24) % 24 of a 64-bit hash with 32-bit arithmetic: v' = hi * 2^32 + lo with hi < 2^8 and 2^32 mod 24 = 16
    __device__ __forceinline__ static uint32_t perm_index(uint64_t mixed) {
        const uint64_t v = mixed >> 24;
        const uint32_t hi = (uint32_t)(v >> 32), lo = (uint32_t)v;
        const uint32_t t = hi * 16u + lo % 24u;          // <= 255 * 16 + 23 = 4103
        return t - 24u * ((t * 2731u) >> 16);             // exact t % 24 for t < 4104 (2731 = ceil(2^16 / 24))
    }
    // ZSobolSampler::get_sample_index (z_sobol_sampler.rs:101-156).
    // Every base-4 digit is permuted independently, keyed by the digits ABOVE it and the dimension.  The digits that hold the
    // pixel's Morton code (shift >= log2_spp) therefore depend on (pixel, dimension) only -- not on the sample index, the seed
    // or the path -- and are read from a table built once per (resolution, spp) by k_sobol_prefix; only the log2_spp / 2 sample
    // digits are permuted here (6 of 18 digits for a 4096-spp 4K frame: HBM capacity traded for ~700 integer instructions per
    // sampler call).  Dimensions past the table fall back to the full loop.
    __device__ __forceinline__ static uint64_t permuted_digits(uint32_t morton, uint32_t dim, uint32_t log2_spp, int i_from, int i_to) {  // digits i_from down to i_to
        uint64_t sidx = 0;
        const int odd = (int)(log2_spp & 1u);
        const uint64_t dk = 0x55555555ull * (uint64_t)dim;
#pragma unroll 1
        for (int i = i_from; i >= i_to; --i) {
            const int digit_shift = 2 * i - odd;
            const uint32_t digit = (uint32_t)(((uint64_t)morton >> digit_shift) & 3ull);
            const uint64_t higher = (uint64_t)morton >> (digit_shift + 2);
            const uint32_t p = perm_index(mix_bits(higher ^ dk));
            sidx |= (uint64_t)perm_digit(p, digit) << digit_shift;
        }
        return sidx;
    }
    __device__ __forceinline__ static int first_pixel_digit(uint32_t log2_spp) { return (int)((log2_spp + 1u) >> 1); }
    // the table entries a sampler call at `dim` reads (prefix row, pass row), split from the arithmetic so that a vertex can ask for the
    // entries of several calls at once (sobol_draws3)
    struct SobolLoads { uint32_t hi, e; };
    __device__ __forceinline__ static SobolLoads sample_index_loads(uint32_t dim, uint32_t pix, const SobolFrame f) {
        SobolLoads l; l.hi = 0u; l.e = 0u;
        const uint32_t n_prefix = f.tables & 0xffffu, n_pass = (f.tables >> 16) & 0xffu;
        const uint32_t* __restrict__ col = f.prefix + pix;   // this pixel's column of the tables
        if (dim < n_prefix || dim < n_pass) l.hi = __ldg(col + (size_t)dim * f.prefix_stride);
        if (dim < n_pass) l.e = __ldg(col + (size_t)(n_prefix + dim) * f.prefix_stride);
        return l;
    }
    __device__ __forceinline__ static uint64_t sample_index_from(uint32_t morton, uint32_t dim, const SobolFrame f, const SobolLoads l) {
        const uint32_t log2_spp = f.cfg & 0xffu, nb4 = f.cfg >> 8;
        const bool pow2 = (log2_spp & 1u) == 1u;
        const int last_digit = pow2 ? 1 : 0;
        uint64_t sidx;
        const uint32_t n_prefix = f.tables & 0xffffu, n_pass = (f.tables >> 16) & 0xffu;
        if (dim < n_pass) {
            // Pass table: the samples of one pass differ in their lowest `iv` base-4 digits only, so the permuted digits above those
            // (they are keyed by the digits above them: pixel and pass, not sample) and the permutation of digit iv - 1 (keyed by
            // everything above it) are the same for every sample of the pixel in this pass: computed once per (dimension, pixel,
            // pass) by k_sobol_pass instead of once per path vertex.  Left here: one table-driven digit and iv - 1 hashed ones.
            const uint32_t iv = f.tables >> 24;
            const uint32_t hi = l.hi;
            const uint32_t e = l.e;
            sidx = ((uint64_t)hi << log2_spp) | ((uint64_t)(e & 0xffffu) << (2u * iv));
            if (iv >= 1u) {
                const uint32_t sh = 2u * iv - 2u;
                sidx |= (uint64_t)perm_digit(e >> 16, (morton >> sh) & 3u) << sh;
                if (iv >= 2u) sidx |= permuted_digits(morton, dim, log2_spp, (int)iv - 2, 0);
            }
            return sidx;   // (the pass table is only built for even log2_spp: no trailing binary digit)
        }
        if (dim < n_prefix) {
            const uint32_t hi = l.hi;
            sidx = ((uint64_t)hi << log2_spp) | permuted_digits(morton, dim, log2_spp, first_pixel_digit(log2_spp) - 1, last_digit);
        } else {
            sidx = permuted_digits(morton, dim, log2_spp, (int)nb4 - 1, last_digit);
        }
        if (pow2) {
            // quirk: the reference ANDs with the loop variable, which is last_digit - 1 = 0 after the loop; pbrt-v4 has `& 1`
            const uint64_t digit = (uint64_t)morton & 0ull;
            const uint64_t dk = 0x55555555ull * (uint64_t)dim;
            sidx |= digit ^ (mix_bits(((uint64_t)morton >> 1) ^ dk) & 1ull);
        }
        return sidx;
    }
    __device__ __forceinline__ static uint64_t sample_index(uint32_t morton, uint32_t dim, uint32_t pix, const SobolFrame f) {
        return sample_index_from(morton, dim, f, sample_index_loads(dim, pix, f));
    }
    // table entry of (pixel, dimension): the permuted pixel digits, shifted down by log2_spp
    __device__ __forceinline__ static uint32_t pixel_prefix(uint32_t morton, uint32_t dim, uint32_t log2_spp, uint32_t nb4) {
        return (uint32_t)(permuted_digits(morton, dim, log2_spp, (int)nb4 - 1, first_pixel_digit(log2_spp)) >> log2_spp);
    }
    // pass-table entry of (pixel, dimension) for a pass whose samples differ in their lowest iv digits (log2_spp even):
    // bits 0-15 = permuted sample digits iv .. log2_spp/2 - 1, shifted down; bits 16-20 = permutation row of digit iv - 1
    __device__ __forceinline__ static uint32_t pass_entry(uint32_t morton, uint32_t dim, uint32_t log2_spp, uint32_t iv) {
        const int top = (int)(log2_spp >> 1) - 1;
        uint32_t c = 0u, p = 0u;
        if (top >= (int)iv) c = (uint32_t)(permuted_digits(morton, dim, log2_spp, top, (int)iv) >> (2u * iv));
        if (iv >= 1u) p = perm_index(mix_bits(((uint64_t)morton >> (2u * iv)) ^ (0x55555555ull * (uint64_t)dim)));
        return c | (p << 16);
    }
    __device__ __forceinline__ static uint32_t sobol_dim1(uint64_t a) {
        const uint32_t* __restrict__ tab = c_sobol_dim1_bytes;
        uint32_t lo = (uint32_t)a, hi = (uint32_t)(a >> 32);
        uint32_t v = __ldg(tab + (lo & 255u)) ^ __ldg(tab + 256 + ((lo >> 8) & 255u)) ^ __ldg(tab + 512 + ((lo >> 16) & 255u)) ^ __ldg(tab + 768 + (lo >> 24));
        if (hi != 0u) v ^= __ldg(tab + 1024 + (hi & 255u)) ^ __ldg(tab + 1280 + ((hi >> 8) & 255u)) ^ __ldg(tab + 1536 + ((hi >> 16) & 15u));  // matrix has 52 rows
        return v;
    }
    // ZSobolSampler::get_1d / get_2d (z_sobol_sampler.rs:198-235); `dim` = the dimension counter BEFORE the call (the reference
    // increments it before hashing, :204-207,215-218)
    __device__ __noinline__ static float sobol_1d(uint32_t morton, uint32_t dim, uint32_t pix, const SobolFrame f) {
        const uint64_t a = sample_index(morton, dim, pix, f);
        const uint64_t h = hash_of(dim + 1u, f);
        return to_unit(owen(__brev((uint32_t)a), (uint32_t)h));  // Sobol matrix 0 = identity on reversed bits; rows >= 32 are zero
    }
    __device__ __noinline__ static float2 sobol_2d(uint32_t morton, uint32_t dim, uint32_t pix, const SobolFrame f) {
        const uint64_t a = sample_index(morton, dim, pix, f);
        const uint64_t h = hash_of(dim + 2u, f);
        float2 r;
        r.x = to_unit(owen(__brev((uint32_t)a), (uint32_t)h));
        r.y = to_unit(owen(sobol_dim1(a), (uint32_t)(h >> 32)));
        return r;
    }
    // Three sampler calls of one vertex at once (a 2-D call at dimension da, a 2-D call at db, a 1-D call at dc): the values are pure
    // functions of (pixel, sample, dimension), so drawing them before they are needed changes nothing but WHEN their six table entries are
    // asked for: together, one round trip instead of three in a row in front of the BSDF sample, the light sample and Russian roulette.
    struct Draws3 { float2 a, b; float c; };
    __device__ __noinline__ static Draws3 sobol_draws3(uint32_t morton, uint32_t da, uint32_t db, uint32_t dc, uint32_t pix, const SobolFrame f) {
        const SobolLoads la = sample_index_loads(da, pix, f), lb = sample_index_loads(db, pix, f), lc = sample_index_loads(dc, pix, f);
        Draws3 r;
        {
            const uint64_t a = sample_index_from(morton, da, f, la);
            const uint64_t h = hash_of(da + 2u, f);
            r.a.x = to_unit(owen(__brev((uint32_t)a), (uint32_t)h));
            r.a.y = to_unit(owen(sobol_dim1(a), (uint32_t)(h >> 32)));
        }
        {
            const uint64_t a = sample_index_from(morton, db, f, lb);
            const uint64_t h = hash_of(db + 2u, f);
            r.b.x = to_unit(owen(__brev((uint32_t)a), (uint32_t)h));
            r.b.y = to_unit(owen(sobol_dim1(a), (uint32_t)(h >> 32)));
        }
        {
            const uint64_t a = sample_index_from(morton, dc, f, lc);
            const uint64_t h = hash_of(dc + 1u, f);
            r.c = to_unit(owen(__brev((uint32_t)a), (uint32_t)h));
        }
        return r;
    }
    // get_1d whose value the caller provably does not use: both samplers are pure functions of the dimension counter, so
    // advancing the counter is all that has to happen (the reference computes and discards the value)
    __device__ __forceinline__ void skip_1d() { dim += 1; }
    __device__ __forceinline__ float get_1d(const DRender& R) {
        if (R.sampler == TCPT_SAMPLER_SOBOL) {
            const float r = sobol_1d(morton, dim, pix, frame_of(R));
            dim += 1;
            return r;
        }
        return unit_float(pcg_hash2(key, dim++));
    }
    __device__ __forceinline__ float2 get_2d(const DRender& R) {
        if (R.sampler == TCPT_SAMPLER_SOBOL) {
            const float2 r = sobol_2d(morton, dim, pix, frame_of(R));
            dim += 2;
            return r;
        }
        float2 r;
        r.x = unit_float(pcg_hash2(key, dim++));
        r.y = unit_float(pcg_hash2(key, dim++));
        return r;
    }
};

// Independent stream standing in for rand::rng() inside shading (generalized_schlick.rs:901, an OS-seeded ThreadRng in the
// reference, so only its distribution can be reproduced): keyed by (path, bounce, call site), shared by definition with the oracle.
struct DAuxRng {
    uint32_t key, ctr;
    __device__ __forceinline__ float next() { return DSampler::unit_float(DSampler::pcg_hash2(key, ctr++)); }
};
__device__ __forceinline__ DAuxRng aux_rng(uint32_t path_key, uint32_t depth, uint32_t site) {
    DAuxRng r; r.key = path_key ^ 0x5bd1e995u ^ ((depth * 4u + site) * 0x27d4eb2fu); r.ctr = 0; return r;
}

// ---------------------------------------------------------------- wavelengths and spectra
struct DWavelengths { float lambda[4]; float pdf[4]; bool terminated; };
__device__ __forceinline__ DWavelengths wavelengths_uniform(float lambda0, bool terminated) {  // sampled_spectrum.rs:318-336 with lambda[0] given
    DWavelengths w;
    w.lambda[0] = lambda0;
    const float delta = (830.0f - 360.0f) / 4.0f;
#pragma unroll
    for (int i = 1; i < 4; ++i) {
        float l = w.lambda[i - 1] + delta;
        if (l >= 830.0f) l = 360.0f + (l - 830.0f);
        w.lambda[i] = l;
    }
    const float p = 1.0f / (830.0f - 360.0f);
    w.pdf[0] = terminated ? p / 4.0f : p;
    w.pdf[1] = w.pdf[2] = w.pdf[3] = terminated ? 0.0f : p;
    w.terminated = terminated;
    return w;
}
__device__ __forceinline__ float srgb_to_linear(float c) { return c <= 0.04045f ? c / 12.92f : powf((c + 0.055f) / 1.055f, 2.4f); }
__device__ __forceinline__ float linear_to_srgb(float c) { return c <= 0.0031308f ? 12.92f * c : 1.055f * powf(c, 1.0f / 2.4f) - 0.055f; }
__device__ __forceinline__ float sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float4 cmf_at(const DScene& sc, float lambda) {  // DenselySampledSpectrum::value for x,y,z,D65 at once
    if (!(lambda >= 360.0f && lambda <= 830.0f)) return make_float4(0, 0, 0, 0);
    uint32_t i = f2u_sat(floorf(lambda - 360.0f));
    return i < 470u ? __ldg(&sc.cmf[i]) : make_float4(0, 0, 0, 0);
}

// RgbToSpectrumTable::get (rgb_sigmoid_polynomial.rs:87-155), sRGB-gamma typed colour
// (returns by value: an out-array lived in local memory and cost a store -> load -> store -> load chain through L1 before the first
// wavelength could be evaluated)
// HALF: the caller guarantees nothing, but expects the largest component to be exactly 0.5 (illuminant_from_rgb): that component is not
// decoded again and the node search is skipped when the largest linear value is the precomputed one.  Same values either way: the shortcut
// replaces a pure function of a constant by its result (computed by the same device code) and a search by its (unique) answer.
template <bool HALF>
__device__ __noinline__ float3 rgb_to_coeffs_t(const DScene& sc, float3 rgb_in) {
    float cs[3];
    float rgb[3];
    const int h = !HALF || sc.half_zi < 0 ? -1 : (rgb_in.x == 0.5f ? 0 : (rgb_in.y == 0.5f ? 1 : (rgb_in.z == 0.5f ? 2 : -1)));
    if (HALF && h >= 0) {
        const float la = srgb_to_linear(h == 0 ? rgb_in.y : rgb_in.x), lb = srgb_to_linear(h == 2 ? rgb_in.y : rgb_in.z);   // the two other components, in order
        rgb[0] = h == 0 ? sc.half_lin : la; rgb[1] = h == 1 ? sc.half_lin : (h == 0 ? la : lb); rgb[2] = h == 2 ? sc.half_lin : lb;
    } else {
        rgb[0] = srgb_to_linear(rgb_in.x); rgb[1] = srgb_to_linear(rgb_in.y); rgb[2] = srgb_to_linear(rgb_in.z);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) rgb[k] = rgb[k] > 0.0f ? rgb[k] : 0.0f;
    // (component > 1 panics in the reference; u8/255 texels and half-scaled illuminant colours never exceed 1)
    if (rgb[0] == rgb[1] && rgb[1] == rgb[2]) return f3(0.0f, 0.0f, logf(rgb[0] / (1.0f - rgb[0])));
    int m = 0;
    { float best = rgb[0]; if (rgb[1] > best) { best = rgb[1]; m = 1; } if (rgb[2] > best) m = 2; }
    const float z = m == 0 ? rgb[0] : (m == 1 ? rgb[1] : rgb[2]);
    const float xr = m == 0 ? rgb[1] : (m == 1 ? rgb[2] : rgb[0]);
    const float yr = m == 0 ? rgb[2] : (m == 1 ? rgb[0] : rgb[1]);
    const float x = xr * (64.0f - 1.0f) / z;
    const float y = yr * (64.0f - 1.0f) / z;
    const uint32_t xi = min(f2u_sat(x), 62u), yi = min(f2u_sat(y), 62u);
    // zi = first i with z_nodes[i+1] > z, else 62 (rgb_sigmoid_polynomial.rs:124-126); the nodes are increasing, so a
    // binary search over the same predicate returns the same index
    uint32_t zi;
    if (HALF && h >= 0 && z == sc.half_lin) zi = (uint32_t)sc.half_zi;
    else {
        uint32_t lo = 0, hi = 62;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(&sc.z_nodes[mid + 1]) > z) hi = mid; else lo = mid + 1; }
        zi = lo;
    }
    const float z0 = __ldg(&sc.z_nodes[zi]), z1 = __ldg(&sc.z_nodes[zi + 1]);
    const float dx = x - (float)xi, dy = y - (float)yi, dz = (z - z0) / (z1 - z0);
    const float* base = sc.rgb2spec + ((((size_t)m * 64 + zi) * 64 + yi) * 64 + xi) * 3;
    const size_t sx = 3, sy = 64 * 3, sz = 64 * 64 * 3;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float c000 = __ldg(base + i), c100 = __ldg(base + sx + i), c010 = __ldg(base + sy + i), c110 = __ldg(base + sy + sx + i);
        const float c001 = __ldg(base + sz + i), c101 = __ldg(base + sz + sx + i), c011 = __ldg(base + sz + sy + i), c111 = __ldg(base + sz + sy + sx + i);
        const float a0 = c000 + (c100 - c000) * dx, a1 = c010 + (c110 - c010) * dx;
        const float b0 = c001 + (c101 - c001) * dx, b1 = c011 + (c111 - c011) * dx;
        const float a = a0 + (a1 - a0) * dy, b = b0 + (b1 - b0) * dy;
        cs[i] = a + (b - a) * dz;
    }
    return f3(cs[0], cs[1], cs[2]);
}
__device__ __forceinline__ float3 rgb_to_coeffs(const DScene& sc, float3 rgb_in) { return rgb_to_coeffs_t<false>(sc, rgb_in); }

// a resolved Spectrum (SpectrumTrait object) on the device
struct DSpectrum { int kind; float c[3]; float scale; int table; };  // 0 const 1 sigmoid 2 sigmoid*scale*D65 3 D65 5 dense preset table
__device__ __forceinline__ float spectrum_value(const DScene& sc, const DSpectrum& s, float lambda) {
    if (s.kind == 0) return s.c[0];
    if (s.kind == 3) return cmf_at(sc, lambda).w;
    if (s.kind == 5) {  // DenselySampledSpectrum::value (densely_sampled_spectrum.rs:57-67)
        if (!(lambda >= 360.0f && lambda <= 830.0f)) return 0.0f;
        const uint32_t i = f2u_sat(floorf(lambda - 360.0f));
        return i < 470u ? __ldg(sc.presets + (size_t)s.table * 470u + i) : 0.0f;
    }
    const float t = (lambda - 360.0f) / (830.0f - 360.0f);
    const float sg = sigmoidf(t * t * s.c[0] + t * s.c[1] + s.c[2]);
    if (s.kind == 1) return sg;
    return s.scale * sg * cmf_at(sc, lambda).w;
}
// (everything by value: by reference the spectrum and the wavelength record sat in the caller's stack frame and each of the 4 x 3
// coefficient reads and 5 wavelength reads was a separate local-memory load.  A wavelength record is always
// wavelengths_uniform(lambda[0], terminated) -- that is also what terminate_secondary leaves -- so two scalars carry it.)
__device__ __noinline__ S4 spectrum_sample_v(const DScene& sc, const DSpectrum s, float lambda0, bool terminated) {
    S4 r = s4(0.0f);
    r.v[0] = spectrum_value(sc, s, lambda0);
    if (terminated) return r;
    const float delta = (830.0f - 360.0f) / 4.0f;
    float l = lambda0;
#pragma unroll
    for (int i = 1; i < 4; ++i) {   // the same arithmetic as wavelengths_uniform
        l = l + delta;
        if (l >= 830.0f) l = 360.0f + (l - 830.0f);
        r.v[i] = spectrum_value(sc, s, l);
    }
    return r;
}
__device__ __forceinline__ S4 spectrum_sample(const DScene& sc, const DSpectrum& s, const DWavelengths& wl) { return spectrum_sample_v(sc, s, wl.lambda[0], wl.terminated); }
__device__ __forceinline__ DSpectrum spectrum_from_flat(const tcpt_flat_spectrum& p) {
    DSpectrum s; s.kind = p.kind; s.c[0] = p.c[0]; s.c[1] = p.c[1]; s.c[2] = p.c[2]; s.scale = p.scale; s.table = p.texture; return s;
}
// RgbIlluminantSpectrum::<ColorSrgb>::new (rgb_illuminant_spectrum.rs:27-40)
__device__ __forceinline__ DSpectrum illuminant_from_rgb(const DScene& sc, float3 rgb) {
    DSpectrum s; s.kind = 2; s.table = 0;
    const float mx = rmax(rgb.x, rmax(rgb.y, rgb.z));
    s.scale = 2.0f * mx;
    const float3 c = rgb_to_coeffs_t<true>(sc, rgb / s.scale);
    s.c[0] = c.x; s.c[1] = c.y; s.c[2] = c.z;
    return s;
}

// ---------------------------------------------------------------- textures (scene/src/texture/sampler.rs)
__device__ __forceinline__ float fract_rs(float x) { return x - truncf(x); }
struct Taps { uint32_t x0, y0, x1, y1; float fx, fy; };
__device__ __forceinline__ Taps bilinear_taps(uint32_t w, uint32_t h, float2 uv) {
    const float u = fabsf(fract_rs(uv.x)), v = 1.0f - fabsf(fract_rs(uv.y));
    const float x = u * ((float)w - 1.0f), y = v * ((float)h - 1.0f);
    Taps t;
    t.x0 = f2u_sat(floorf(x)); t.y0 = f2u_sat(floorf(y));
    t.x1 = min(t.x0 + 1u, w - 1u); t.y1 = min(t.y0 + 1u, h - 1u);
    t.fx = x - (float)t.x0; t.fy = y - (float)t.y0;
    return t;
}
__device__ __forceinline__ float lerp2d(float p00, float p10, float p01, float p11, float fx, float fy) {
    const float top = p00 * (1.0f - fx) + p10 * fx, bottom = p01 * (1.0f - fx) + p11 * fx;
    return top * (1.0f - fy) + bottom * fy;
}
__device__ __noinline__ float3 tex_rgb(const DTexture& t, float2 uv) {
    const Taps k = bilinear_taps(t.w, t.h, uv);
    const uint8_t* a = t.data + ((size_t)k.y0 * t.w + k.x0) * 3; const uint8_t* b = t.data + ((size_t)k.y0 * t.w + k.x1) * 3;
    const uint8_t* c = t.data + ((size_t)k.y1 * t.w + k.x0) * 3; const uint8_t* d = t.data + ((size_t)k.y1 * t.w + k.x1) * 3;
    float o[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
        o[ch] = lerp2d((float)__ldg(a + ch) / 255.0f, (float)__ldg(b + ch) / 255.0f, (float)__ldg(c + ch) / 255.0f, (float)__ldg(d + ch) / 255.0f, k.fx, k.fy);
    return f3(o[0], o[1], o[2]);
}
__device__ __noinline__ float tex_gray(const DTexture& t, float2 uv) {
    const Taps k = bilinear_taps(t.w, t.h, uv);
    return lerp2d((float)__ldg(t.data + (size_t)k.y0 * t.w + k.x0) / 255.0f, (float)__ldg(t.data + (size_t)k.y0 * t.w + k.x1) / 255.0f,
                  (float)__ldg(t.data + (size_t)k.y1 * t.w + k.x0) / 255.0f, (float)__ldg(t.data + (size_t)k.y1 * t.w + k.x1) / 255.0f, k.fx, k.fy);
}

__device__ __forceinline__ DSpectrum param_spectrum(const DScene& sc, const tcpt_flat_spectrum& p, float2 uv) {
    DSpectrum s;
    if (p.kind == 4) {  // rgb_texture.rs:48-66
        s.kind = 1; s.scale = 1.0f; s.table = 0;
        const float3 c = rgb_to_coeffs(sc, tex_rgb(sc.textures[p.texture], uv));
        s.c[0] = c.x; s.c[1] = c.y; s.c[2] = c.z;
        return s;
    }
    return spectrum_from_flat(p);
}
__device__ __forceinline__ float param_float(const DScene& sc, const tcpt_flat_float& p, float2 uv) {
    if (!p.is_texture) return p.value;
    const float v = tex_gray(sc.textures[p.texture], uv);
    return p.gamma_corrected ? srgb_to_linear(v) : v;  // float_texture.rs:45-52
}

// two appends at once (extension ray and shadow ray of one vertex): lanes 0 and 1 issue the two atomics back to back, so the warp
// pays ONE round trip to L2 instead of two dependent ones.  Every lane of the warp must call it.
__device__ __forceinline__ void warp_push2(uint32_t* ca, bool pa, uint32_t* cb, bool pb, uint32_t* ia, uint32_t* ib) {
    const uint32_t ma = __ballot_sync(0xffffffffu, pa), mb = __ballot_sync(0xffffffffu, pb);
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t base = 0;
    if (lane == 0u) { if (ma) base = atomicAdd(ca, (uint32_t)__popc(ma)); }
    else if (lane == 1u) { if (mb) base = atomicAdd(cb, (uint32_t)__popc(mb)); }
    const uint32_t ba = __shfl_sync(0xffffffffu, base, 0), bb = __shfl_sync(0xffffffffu, base, 1);
    const uint32_t below = (1u << lane) - 1u;
    *ia = ba + (uint32_t)__popc(ma & below); *ib = bb + (uint32_t)__popc(mb & below);
}
// warp-aggregated queue append: every lane of the warp must call it (pred = false for lanes with nothing to push)
__device__ __forceinline__ uint32_t warp_push(uint32_t* counter, bool pred) {
    const uint32_t mask = __ballot_sync(0xffffffffu, pred);
    if (mask == 0) return 0;
    const uint32_t lane = threadIdx.x & 31u;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

}  // namespace tcpt
