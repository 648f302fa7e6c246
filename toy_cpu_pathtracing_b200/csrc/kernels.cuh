// The wavefront kernels of the path-integration hot path (sm_100a).  One frame =
//   for each pass (a block of pixels x a block of sample indices that fits the path-slot budget):
//     k_generate                      camera rays + sampler dimensions 0..2          base_renderer.rs:160-177
//     for bounce = 0 .. max_depth:
//       k_trace_closest               Scene::intersect over the extension-ray queue  scene.rs:80-90
//       k_shade                       everything between two intersect calls          base_renderer.rs:178-272
//       k_trace_shadow                Scene::intersect_p + visible-branch add         scene.rs:93-103, common.rs:134-170
//     k_film                          per-pixel in-order sum of the pass's samples    sensor.rs:76-77
//   k_finalize                        /spp, clip, Reinhard, sRGB OETF                 sensor.rs:81-88
// Queues are sized on the device (no host round trip inside a frame); every kernel is a grid-stride loop over a queue
// whose length it reads from `counters`.
#pragma once
#include "dshade.cuh"
#include "dtraverse.cuh"

// shading buckets (see bucket_of): counters[4 + TCPT_BUCKET_STRIDE * parity + bucket] holds their sizes
#define TCPT_N_BUCKETS 9
#ifndef TCPT_SHADE_MIN_BLOCKS_LAMBERT
#define TCPT_SHADE_MIN_BLOCKS_LAMBERT 4
#endif
#ifndef TCPT_TRACE_MIN_BLOCKS
#define TCPT_TRACE_MIN_BLOCKS 8   // 64 registers + 13 KB of shared memory per block: 32 warps per SM (measured 6 / 7 / 8 blocks: 35.7 / 33.5 / 32.1 ms per step)
#endif
#define TCPT_BUCKET_STRIDE 10

namespace tcpt {

struct PathList { const uint32_t* xy; const uint32_t* sample; };  // explicit (pixel, sample) lists for tcpt_path_samples

// owned pixel index of pass pixel p_local: consecutive from pix_begin, or the pix_begin + p_local-th entry of the pass's pixel list
// (adaptive rounds: the owned indices of the pixels still active, in ascending order; the frame index for a whole-frame job)
__device__ __forceinline__ uint32_t owned_pixel(const DRender& R, uint32_t p_local) {
    return R.pix_list ? __ldg(R.pix_list + R.pix_begin + p_local) : R.pix_begin + p_local;
}

__device__ __forceinline__ void path_coords(const DRender& R, const PathList& L, uint32_t slot, uint32_t* px, uint32_t* py, uint32_t* si) {
    if (L.xy) { *px = __ldg(L.xy + 2 * (size_t)slot); *py = __ldg(L.xy + 2 * (size_t)slot + 1); *si = __ldg(L.sample + slot); return; }
    const uint32_t s_local = div_magic(slot, R.n_pix_magic), p_local = slot - s_local * R.n_pix;
    const uint32_t k = owned_pixel(R, p_local);
    const uint32_t row = div_magic(k, R.width_magic);
    *px = k - row * R.width;
    *py = R.row_offset + row * R.row_stride;
    *si = R.s_begin + s_local;
}

__device__ __forceinline__ DSampler make_sampler(const DRender& R, uint32_t px, uint32_t py, uint32_t si) {
    DSampler s;
    s.start(R, px, py, si);
    return s;
}

// builds DRender::sobol_prefix: entry (dim, pixel) = permuted pixel digits of ZSobolSampler::get_sample_index (see DSampler)
__global__ void __launch_bounds__(256) k_sobol_prefix(uint32_t* __restrict__ table, uint32_t width, uint32_t height, uint32_t log2_spp, uint32_t nb4, uint32_t dims) {
    const size_t n_pix = (size_t)width * height, total = n_pix * dims;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t dim = (uint32_t)(i / n_pix), k = (uint32_t)(i - (size_t)dim * n_pix);
        const uint32_t py = k / width, px = k - py * width;
        table[i] = DSampler::pixel_prefix(DSampler::morton_of(px, py, 0u, log2_spp), dim, log2_spp, nb4);
    }
}

// DScene::half_lin / half_zi: srgb_to_linear(0.5f) and its z-node interval, evaluated by the code the lookups run (out = {bits of the value, index})
__global__ void k_illum_half(const float* __restrict__ z_nodes, uint32_t* __restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const volatile float half_in = 0.5f;   // (volatile: evaluated at run time by the device's powf, not folded by the compiler's)
    const float z = srgb_to_linear(half_in);
    uint32_t lo = 0, hi = 62;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (z_nodes[mid + 1] > z) hi = mid; else lo = mid + 1; }
    out[0] = __float_as_uint(z); out[1] = lo;
}

// builds DRender::sobol_hash
__global__ void k_sobol_hash(unsigned long long* __restrict__ table, uint32_t seed) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < (uint32_t)TCPT_SOBOL_HASH_N) table[k] = DSampler::hash(k, seed);
}

// builds the pass rows of DRender::sobol_prefix for the pixels and the sample block of ONE pass (see DSampler::sample_index):
// row prefix_dims + dim, column = the pixel's frame index
__global__ void __launch_bounds__(256) k_sobol_pass(uint32_t* __restrict__ table, const __grid_constant__ DRender R, uint32_t dims, uint32_t iv) {
    const size_t total = (size_t)R.n_pix * dims;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t dim = (uint32_t)(i / R.n_pix), p_local = (uint32_t)(i - (size_t)dim * R.n_pix);
        const uint32_t k = owned_pixel(R, p_local), row = k / R.width;
        const uint32_t px = k - row * R.width, py = R.row_offset + row * R.row_stride;
        table[(size_t)(R.prefix_dims + dim) * R.prefix_stride + (size_t)py * R.width + px] =
            DSampler::pass_entry(DSampler::morton_of(px, py, R.s_begin, R.log2_spp), dim, R.log2_spp, iv);
    }
}

// The same rows, built INCREMENTALLY.  The permutation row of digit i is keyed by the digits above i and the dimension; from one pass to the
// next only the low sample digits of the table change, so most rows are the ones the previous pass computed.  Per (dimension, pixel) a cache
// word keeps the rows of the digits iv .. top (5 bits each, at most four), the sample digits they were computed for (the tag) and iv; an
// entry recomputes the rows below the highest digit that changed (all of them when the word is invalid) and always the row of digit iv - 1.
// On consecutive 16-sample passes of a 4096-spp frame that is 1.33 hashes per entry instead of 5.  Same values: rows are pure functions of
// their keys.  cache word: bit 31 valid | iv << 28 | tag << 20 | rows.
__global__ void __launch_bounds__(256) k_sobol_pass_cached(uint32_t* __restrict__ table, const __grid_constant__ DRender R, uint32_t dims, uint32_t iv, uint32_t cache_row0) {
    const uint32_t top = (R.log2_spp >> 1) - 1u, levels = top - iv + 1u;
    const uint32_t tag_new = (R.s_begin >> (2u * iv)) & ((1u << (2u * levels)) - 1u);
    // one thread per PIXEL, looping over the dimensions: coordinates and Morton code once per pixel; a warp's accesses to a row stay contiguous
    for (uint32_t p_local = blockIdx.x * blockDim.x + threadIdx.x; p_local < R.n_pix; p_local += gridDim.x * blockDim.x) {
        const uint32_t k = owned_pixel(R, p_local), row = div_magic(k, R.width_magic);
        const uint32_t px = k - row * R.width, py = R.row_offset + row * R.row_stride;
        const size_t col = (size_t)py * R.width + px;
        const uint32_t morton = DSampler::morton_of(px, py, R.s_begin, R.log2_spp);
        for (uint32_t dim = 0; dim < dims; ++dim) {
            uint32_t* cache = table + (size_t)(cache_row0 + dim) * R.prefix_stride + col;
            const uint32_t cw = *cache;
            uint32_t stale = levels;   // rows of the digits iv .. iv + stale - 1 have to be recomputed
            if ((cw >> 31) != 0u && ((cw >> 28) & 7u) == iv) { const uint32_t diff = ((cw >> 20) & 0xffu) ^ tag_new; stale = diff ? (31u - (uint32_t)__clz(diff)) >> 1 : 0u; }
            uint32_t rows = cw & 0xfffffu;
            const uint64_t dk = 0x55555555ull * (uint64_t)dim;
            uint32_t c = 0u;
            for (uint32_t j = 0; j < levels; ++j) {
                const uint32_t sh = 2u * (iv + j);
                if (j < stale) rows = (rows & ~(31u << (5u * j))) | (DSampler::perm_index(DSampler::mix_bits(((uint64_t)morton >> (sh + 2u)) ^ dk)) << (5u * j));
                c |= DSampler::perm_digit((rows >> (5u * j)) & 31u, (morton >> sh) & 3u) << (2u * j);
            }
            const uint32_t p = DSampler::perm_index(DSampler::mix_bits(((uint64_t)morton >> (2u * iv)) ^ dk));
            table[(size_t)(R.prefix_dims + dim) * R.prefix_stride + col] = c | (p << 16);
            *cache = 0x80000000u | (iv << 28) | (tag_new << 20) | rows;
        }
    }
}

// builds DEnv::nee_table (once per scene upload): one thread per texel runs env_nee_texel, the code the shading kernels would run per sample
__global__ void __launch_bounds__(256) k_env_nee_table(const __grid_constant__ DScene sc, uint32_t env_index, float4* __restrict__ table) {
    const DEnv& e = sc.envs[env_index];
    const tcpt_flat_primitive& LP = sc.primitives[e.primitive];
    const uint32_t n = e.w * e.h;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t yy = i / e.w, xx = i - yy * e.w;
        const EnvNee r = env_nee_texel(sc, LP, e, xx, yy);
        table[2 * (size_t)i] = make_float4(r.wi_r.x, r.wi_r.y, r.wi_r.z, r.pdf_dir);
        table[2 * (size_t)i + 1] = make_float4(r.spec.c[0], r.spec.c[1], r.spec.c[2], r.spec.scale);
    }
}

// ---------------------------------------------------------------- K0 generate
// camera ray of one path from its two sampler values (BoxFilter::sample + Camera::sample_ray / generate_ray, filter.rs:24-30, camera.rs:51-81)
__device__ __forceinline__ void generate_store(const DRender& R, const DCamera& cam, const DState& st, uint32_t slot, uint32_t px, uint32_t py, float u, float2 uv, uint32_t dim_after) {
    // NormalRenderer draws the pixel sample first and no wavelength (normal_renderer.rs:33-40); the AOV renderers do not push the ray forward
    const bool aov = R.integrator >= TCPT_INTEGRATOR_ALBEDO;
    const float lambda0 = 360.0f + u * (830.0f - 360.0f);  // SampledWavelengths::new_uniform (sampled_spectrum.rs:318-336)
    const float fx = uv.x * 1.0f - 1.0f * 0.5f, fy = uv.y * 1.0f - 1.0f * 0.5f;
    const float x = (float)px + fx + 0.5f, y = (float)py + fy + 0.5f;
    const float dir_x = (2.0f * x / (float)R.width - 1.0f) * cam.aspect * cam.scale;
    const float dir_y = (1.0f - 2.0f * y / (float)R.height) * cam.scale;
    const float3 rd = normalize(f3(dir_x, dir_y, -1.0f));
    const float3 d = normalize((cam.s * rd.x + cam.u * rd.y) + cam.nf * rd.z);
    const float3 o = aov ? f3(0.0f, 0.0f, 0.0f) : f3(0.0f, 0.0f, 0.0f) + d * 1e-5f;  // move_forward(1e-5) (base_renderer.rs:177)
    st.ext_o[0][slot] = make_float4(o.x, o.y, o.z, TCPT_FLT_MAX);
    st.ext_d[0][slot] = make_float4(d.x, d.y, d.z, __uint_as_float(slot));
    // throughput = 1 and contribution = 0 are implied at bounce 0 (shade_vertex does not load them there): 32 B per path less each way
    st.misc[slot] = make_float4(0.0f, lambda0, __uint_as_float(dim_after), __uint_as_float(0u));
}
__device__ __forceinline__ void generate_reset(const DState& st, uint32_t n_slots) {
    st.counters[0] = n_slots; st.counters[1] = 0; st.counters[2] = 0; st.counters[3] = 0;
    for (int b = 0; b < 2 * TCPT_BUCKET_STRIDE; ++b) st.counters[4 + b] = 0;  // both sets of bucket sizes
    st.counters[24] = 0; st.counters[25] = 0;             // work counters of the persistent trace kernels
    atomicAdd(&st.stats[4], (unsigned long long)n_slots);
}
__global__ void __launch_bounds__(256) k_generate(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DCamera cam,
                                                   const __grid_constant__ DState st, const __grid_constant__ PathList L, uint32_t n_slots) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < n_slots; slot += stride) {
        uint32_t px, py, si;
        path_coords(R, L, slot, &px, &py, &si);
        DSampler smp = make_sampler(R, px, py, si);
        float u = 0.0f;
        if (R.integrator != TCPT_INTEGRATOR_NORMAL) u = smp.get_1d(R);
        const float2 uv = smp.get_2d(R);
        generate_store(R, cam, st, slot, px, py, u, uv, smp.dim);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) generate_reset(st, n_slots);
}
// The same for a pass of the Z-Sobol sampler, one thread per PIXEL looping over the pass's sample indices (slot = sample * n_pix + pixel:
// the stores of a warp stay contiguous): what a sampler call derives from the pixel alone -- its coordinates, the Morton prefix, the four
// table entries, the two Owen-scramble seeds -- is fetched once per pixel instead of once per path.  Same functions, same values.
__global__ void __launch_bounds__(256) k_generate_pixels(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DCamera cam,
                                                          const __grid_constant__ DState st, uint32_t n_slots) {
    const uint32_t stride = gridDim.x * blockDim.x;
    const SobolFrame f = DSampler::frame_of(R);
    const bool with_lambda = R.integrator != TCPT_INTEGRATOR_NORMAL;
    const uint32_t d_uv = with_lambda ? 1u : 0u;
    const uint64_t h_u = DSampler::hash_of(1u, f), h_uv = DSampler::hash_of(d_uv + 2u, f);
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < R.n_pix; p += stride) {
        const uint32_t k = owned_pixel(R, p);
        const uint32_t row = div_magic(k, R.width_magic);
        const uint32_t px = k - row * R.width, py = R.row_offset + row * R.row_stride;
        const uint32_t pix = py * R.width + px;
        const uint32_t pixel_morton = DSampler::morton_of(px, py, 0u, R.log2_spp);
        const DSampler::SobolLoads l_u = DSampler::sample_index_loads(0u, pix, f), l_uv = DSampler::sample_index_loads(d_uv, pix, f);
        for (uint32_t s = 0; s < R.s_count; ++s) {
            const uint32_t morton = pixel_morton | (R.s_begin + s);
            float u = 0.0f;
            if (with_lambda) u = DSampler::to_unit(DSampler::owen(__brev((uint32_t)DSampler::sample_index_from(morton, 0u, f, l_u)), (uint32_t)h_u));
            const uint64_t a = DSampler::sample_index_from(morton, d_uv, f, l_uv);
            float2 uv;
            uv.x = DSampler::to_unit(DSampler::owen(__brev((uint32_t)a), (uint32_t)h_uv));
            uv.y = DSampler::to_unit(DSampler::owen(DSampler::sobol_dim1(a), (uint32_t)(h_uv >> 32)));
            generate_store(R, cam, st, s * R.n_pix + p, px, py, u, uv, d_uv + 2u);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) generate_reset(st, n_slots);
}

// ---------------------------------------------------------------- K1 closest hit
// Besides the hit record, every ray is filed into a BUCKET by what k_shade will have to do with it (miss / material type of
// the hit), so that k_shade's warps run one material's code instead of serialising up to six branches (ncu on the first
// version: 8.6 of 32 lanes active in the bounce-1 shade launch).  Filing = one warp-aggregated atomic per distinct bucket.
#ifndef TCPT_SHADE_MIN_BLOCKS
#define TCPT_SHADE_MIN_BLOCKS 4
#endif
// shading order: heaviest code first so the tail of the launch is made of cheap vertices
// `killed`: Russian roulette already ended the path behind this ray (decided when the ray was spawned, see shade_vertex); its hit
// only matters if it is a light, so non-emissive hits go to a terminal bucket that just hands the path to the sensor.
__device__ __forceinline__ uint32_t bucket_of(const DScene& sc, int prim, bool killed) {
    if (prim < 0) return 7u;                                     // miss: environment lookup only
    const int t = (int)__ldg(sc.prim_mat_type + prim);
    if (killed && t != TCPT_MAT_EMISSIVE) return 8u;
    return t == TCPT_MAT_CLEARCOAT_PBR ? 0u : t == TCPT_MAT_SIMPLE_PBR ? 1u : t == TCPT_MAT_PLASTIC ? 2u : t == TCPT_MAT_GLASS ? 3u : t == TCPT_MAT_METAL ? 4u
         : t == TCPT_MAT_LAMBERT ? 5u : 6u;
}

// work counters of the persistent trace kernels: counters[24] closest, counters[25] shadow.  Each is zeroed by an earlier kernel
// of the same bounce (stream order): k_generate / k_shade zero [24] for the next k_trace_closest, k_trace_closest zeroes [25].
// what a finished extension ray leaves behind: its hit record and its place in a shading bucket
struct CommitClosest {
    const DScene& sc; const DState& st; const float4* __restrict__ q_d; float4* __restrict__ hit0; uint2* __restrict__ hit1; uint32_t* bcount;
    // the hit record, the bucket, and the warp-aggregated atomic that reserves the bucket's next positions (its result is not waited for)
    __device__ __forceinline__ CommitToken begin(uint32_t i, const DHit& h) const {
        hit0[i] = make_float4(h.t, h.b0, h.b1, h.b2);
        hit1[i] = make_uint2((uint32_t)h.prim, h.tri);
        const float dw = q_d[i].w;
        const bool killed = (__float_as_uint(dw) & 0x80000000u) != 0u;  // ext_d.w = slot | killed << 31
        const uint32_t b = bucket_of(sc, h.prim, killed);
        const uint32_t peers = __match_any_sync(__activemask(), b);
        const uint32_t lane = threadIdx.x & 31u;
        const int leader = __ffs(peers) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&bcount[b], (uint32_t)__popc(peers));
        return CommitToken{base, peers, b, i, __float_as_uint(dw) & 0x7fffffffu};
    }
    __device__ __forceinline__ void end(const CommitToken& t) const {
        const uint32_t lane = threadIdx.x & 31u, peers = t.b, b = t.c, i = t.d;
        const uint32_t base = __shfl_sync(peers, t.a, __ffs(peers) - 1);
        st.order[(size_t)b * st.capacity + base + (uint32_t)__popc(peers & ((1u << lane) - 1u))] = make_uint2(i, t.e);
    }
};
// what a finished shadow ray does: add the pending NEE contribution if the light is visible (common.rs:134-170); hand a path that
// ended at this vertex (failed BSDF sample) to the sensor
struct CommitShadow {
    const DScene& sc; const DRender& R; const DState& st;
    __device__ __forceinline__ CommitToken begin(uint32_t i, const DHit& h) const {
        const uint32_t tag = __float_as_uint(st.sh_d[i].w);
        return CommitToken{tag, i, h.prim < 0 ? 1u : 0u, 0u, 0u};
    }
    __device__ __forceinline__ void end(const CommitToken& t) const {
        const uint32_t tag = t.a, i = t.b;
        const uint32_t slot = tag & 0x7fffffffu;
        const bool visible = t.c != 0u, last = (tag & 0x80000000u) != 0;
        if (!visible && !last) return;
        S4 con = s4(st.con[slot]);
        if (visible) {
            con = con + s4(st.sh_c[i]);
            st.con[slot] = to_f4(con);
        }
        if (last) {
            const float4 misc = st.misc[slot];
            const DWavelengths wl = wavelengths_uniform(misc.y, (__float_as_uint(misc.w) & FLAG_LAMBDA_TERMINATED) != 0);
            const float3 rgb = sensor_rgb(sc, wl.lambda[0], wl.terminated, con, R.exposure);
            st.rgb[slot] = make_float4(rgb.x, rgb.y, rgb.z, 0.0f);
        }
    }
};

template <bool COUNT>
__global__ void __launch_bounds__(128, 6) k_trace_closest(const __grid_constant__ DScene sc, const float4* __restrict__ q_o, const float4* __restrict__ q_d,
                                                        float4* __restrict__ hit0, uint2* __restrict__ hit1, const __grid_constant__ DState st, int cur) {
    const uint32_t n = st.counters[cur];
    uint32_t* bcount = st.counters + 4 + TCPT_BUCKET_STRIDE * cur;  // this bounce's bucket sizes (zeroed one bounce ago)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        // the queues this bounce's k_shade appends to were last read one bounce ago (stream order): reset them here
        st.counters[cur ^ 1] = 0; st.counters[2] = 0; st.counters[25] = 0;
        for (int b = 0; b < TCPT_N_BUCKETS; ++b) st.counters[4 + TCPT_BUCKET_STRIDE * (cur ^ 1) + b] = 0;
        atomicAdd(&st.stats[0], (unsigned long long)n);
    }
    uint32_t nb = 0, nt = 0;
    __shared__ TraceShared ts;
    trace_queue<false, COUNT>(sc, ts, q_o, q_d, n, &st.counters[24], &nb, &nt, CommitClosest{sc, st, q_d, hit0, hit1, bcount});
    if (COUNT) { atomicAdd(&st.stats[2], (unsigned long long)nb); atomicAdd(&st.stats[3], (unsigned long long)nt); }
}

// ---------------------------------------------------------------- K3/K4 shadow rays + visible-branch accumulation
template <bool COUNT>
__global__ void __launch_bounds__(128, 6) k_trace_shadow(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DState st) {
    const uint32_t n = st.counters[2];
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&st.stats[1], (unsigned long long)n);
    uint32_t nb = 0, nt = 0;
    __shared__ TraceShared ts;
    trace_queue<true, COUNT>(sc, ts, st.sh_o, st.sh_d, n, &st.counters[25], &nb, &nt, CommitShadow{sc, R, st});
    if (COUNT) { atomicAdd(&st.stats[2], (unsigned long long)nb); atomicAdd(&st.stats[3], (unsigned long long)nt); }
}

// ---------------------------------------------------------------- fused trace: the shadow rays of bounce s and the extension rays of bounce s + 1
// Both queues are written by k_shade of bounce s and are independent of each other, so one persistent launch drains them back
// to back (shadow first: it is the shorter one) instead of two launches each paying its own ramp-up and tail.  Deep bounces
// hold few rays and are pure launch latency: measured 7.8 ms of fixed cost per pass at about 170 launches (36 ms step).
// `cur` = parity of the extension queue to trace, `sh` = index (2 or 3) of the shadow-queue size to read; the sizes the next
// k_shade appends to (counters[cur ^ 1], counters[sh ^ 1]) were last read one launch ago and are reset here.
template <bool COUNT>
__global__ void __launch_bounds__(128, TCPT_TRACE_MIN_BLOCKS) k_trace_fused(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DState st, int cur, int sh, uint32_t refill_lanes, uint32_t max_chunk) {
    const uint32_t n_sh = st.counters[sh], n = st.counters[cur];
    uint32_t* bcount = st.counters + 4 + TCPT_BUCKET_STRIDE * cur;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st.counters[cur ^ 1] = 0; st.counters[sh ^ 1] = 0;
        for (int b = 0; b < TCPT_N_BUCKETS; ++b) st.counters[4 + TCPT_BUCKET_STRIDE * (cur ^ 1) + b] = 0;
        atomicAdd(&st.stats[0], (unsigned long long)n);
        atomicAdd(&st.stats[1], (unsigned long long)n_sh);
    }
    uint32_t nb = 0, nt = 0;
    __shared__ TraceShared ts;
    // (shadow first: it is the shorter queue.  Letting half of the blocks start on the extension queue so that short queues are
    // walked side by side was measured slower: 16.6 vs 15.3 ms per 33 M paths.)
    if (n_sh) trace_queue<true, COUNT>(sc, ts, st.sh_o, st.sh_d, n_sh, &st.counters[25], &nb, &nt, CommitShadow{sc, R, st}, refill_lanes, max_chunk);
    float4* __restrict__ hit0 = st.hit0; uint2* __restrict__ hit1 = st.hit1;
    if (n) trace_queue<false, COUNT>(sc, ts, st.ext_o[cur], st.ext_d[cur], n, &st.counters[24], &nb, &nt, CommitClosest{sc, st, st.ext_d[cur], hit0, hit1, bcount}, refill_lanes, max_chunk);
    if (COUNT) { atomicAdd(&st.stats[2], (unsigned long long)nb); atomicAdd(&st.stats[3], (unsigned long long)nt); }
}

// ---------------------------------------------------------------- K2 shade
struct ShadeOut {
    bool push_ext, push_sh;
    float4 eo, ed, so, sd, sc;
};

// bucket -> compile-time material type (see bucket_of)
template <int B> struct BucketInfo {
    static constexpr bool miss = B == 7;
    static constexpr bool terminal = B == 8;   // Russian roulette ended the path and the hit is not a light: nothing left to shade
    static constexpr int mat = B == 0 ? TCPT_MAT_CLEARCOAT_PBR : B == 1 ? TCPT_MAT_SIMPLE_PBR : B == 2 ? TCPT_MAT_PLASTIC : B == 3 ? TCPT_MAT_GLASS : B == 4 ? TCPT_MAT_METAL
                              : B == 5 ? TCPT_MAT_LAMBERT : TCPT_MAT_EMISSIVE;
};

// FIRST = compiled for bounce 0 only (k_shade<B, true>): no previous-bounce half, no state loads beyond the wavelength record
template <int B, bool FIRST = false>
__device__ __forceinline__ void shade_vertex(const DScene& sc, const DRender& R, const DState& st, const PathList& L, uint32_t stage_in,
                                             float3 ray_d, uint32_t slot, const float4 h0, const uint2 h1, const float4 misc, ShadeOut& out) {
    constexpr int MT = BucketInfo<B>::mat;
    const uint32_t stage = FIRST ? 0u : stage_in;
    out.push_ext = false; out.push_sh = false;
    float pdf_prev = misc.x;
    const float lambda0 = misc.y;
    uint32_t flags = __float_as_uint(misc.w);
    DWavelengths wl = wavelengths_uniform(lambda0, (flags & FLAG_LAMBDA_TERMINATED) != 0);
    uint32_t px, py, si;
    path_coords(R, L, slot, &px, &py, &si);
    DSampler smp = make_sampler(R, px, py, si);
    smp.dim = __float_as_uint(misc.z);
    // sampler calls of one bounce sit at dimension offsets 0 (lobe choice; Lambert and metal skip it), 1 (direction), 3 (light choice, skipped
    // with one light), 4 (triangle of an area light), 5 (point on the light) and 7 (Russian roulette; 3 under pt, which draws nothing for lights)
    // Lambert under nee / mis with the Sobol sampler: the direction, the point on the light and Russian roulette sit at dimension offsets 1, 5
    // and 7 on the usual way through the vertex; all three are drawn here in one call (DSampler::sobol_draws3) and handed out below if the
    // dimension counter is where it was expected to be (otherwise the ordinary call runs: same values either way)
    constexpr bool NO_LOBE = MT == TCPT_MAT_LAMBERT || MT == TCPT_MAT_METAL;   // these never read the lobe-choice number
    constexpr bool PRE = MT == TCPT_MAT_LAMBERT;
    DSampler::Draws3 pre; bool have_pre = false; const uint32_t pre_d0 = smp.dim;
    if (PRE && R.sampler == TCPT_SAMPLER_SOBOL && R.integrator != TCPT_INTEGRATOR_PT && (FIRST || stage < R.max_depth)) {
        pre = DSampler::sobol_draws3(smp.morton, pre_d0 + 1u, pre_d0 + 5u, pre_d0 + 7u, smp.pix, DSampler::frame_of(R));
        have_pre = true;
    }
    S4 thr = s4(1.0f), con = s4(0.0f);
    if (!FIRST && stage != 0u) { thr = s4(st.thr[slot]); con = s4(st.con[slot]); }
    const int integrator = R.integrator;
    constexpr bool miss = BucketInfo<B>::miss;

    auto finish = [&]() {
        const float3 rgb = sensor_rgb(sc, wl.lambda[0], wl.terminated, con, R.exposure);
        st.rgb[slot] = make_float4(rgb.x, rgb.y, rgb.z, 0.0f);
    };
    // LightSamplerFactory::create is re-run by the reference at every use (light_sampler.rs:190-220); its result only depends
    // on the wavelengths, so one evaluation per vertex serves the BSDF-side MIS weight and the NEE draw
    LightTable lt; bool lt_ready = false;
    auto lights = [&]() -> const LightTable& {
        if (!lt_ready) {
            if (sc.one_light_always_on) { lt.w[0] = 1.0f; lt.sum = 1.0f; }  // w / w = 1 / 1: every probability derived from the table is exactly 1
            else light_table(sc, wl, lt);
            lt_ready = true;
        }
        return lt;
    };

    if constexpr (BucketInfo<B>::terminal) {
        // calculate_bsdf_contribution of a NON-emissive hit: the reference still adds throughput * next_emissive(= 0) [* w], and with an
        // infinite BSDF pdf the MIS weight inf / (inf + 0) is NaN, which poisons the contribution (scene 11's NaN pixels): same arithmetic here
        const S4 zero = s4(0.0f);
        const bool spec_prev = (flags & FLAG_SPEC_PREV) != 0;
        if (integrator == TCPT_INTEGRATOR_PT) con = con + thr * zero;
        else if (integrator == TCPT_INTEGRATOR_NEE || spec_prev) { if (spec_prev) con = con + thr * zero; }
        else {
            const float a = pdf_prev, b = 0.0f;  // Scene::pdf_light_sample of a non-emissive primitive
            const float w = (a == 0.0f && b == 0.0f) ? 0.0f : a / (a + b);
            con = con + thr * zero * w;
        }
        finish();
        return;
    }
    if constexpr (miss) {
        if (sc.n_envs != 0) {
            if (FIRST || stage == 0) {
                S4 radiance;
                scene_env_radiance_pdf(sc, nullptr, ray_d, wl, &radiance, nullptr);
                con = con + thr * radiance;  // base_renderer.rs:180-186
            } else if (integrator != TCPT_INTEGRATOR_NEE) {
                const S4 fprev = s4(st.fprev[slot]);
                if (integrator == TCPT_INTEGRATOR_PT) {
                    S4 radiance;
                    scene_env_radiance_pdf(sc, nullptr, ray_d, wl, &radiance, nullptr);
                    con = con + thr * fprev * radiance / pdf_prev;  // pt_renderer.rs:80-81
                } else {
                    S4 radiance; float light_pdf;
                    scene_env_radiance_pdf(sc, &lights(), ray_d, wl, &radiance, &light_pdf);
                    const float a = pdf_prev, b = light_pdf;
                    const float w = (a == 0.0f && b == 0.0f) ? 0.0f : a / (a + b);
                    const float tf = 1.0f / pdf_prev;
                    con = con + thr * fprev * radiance * tf * w;  // mis_renderer.rs:228-229
                }
            }
        }
        finish();
        return;
    } else {

    DSurface hit;
    reconstruct_hit(sc, (int)h1.x, h1.y, h0.y, h0.z, h0.w, ray_d, hit);
    const tcpt_flat_material& mat = sc.materials[hit.material];
    constexpr bool emissive = MT == TCPT_MAT_EMISSIVE;

    if (FIRST || stage == 0) {
        if (emissive) con = con + thr * emissive_radiance(sc, mat, hit.uv, wl);  // base_renderer.rs:190-194
    } else {
        // second half of the previous bounce: calculate_bsdf_contribution, throughput update, Russian roulette
        const S4 fprev = s4(st.fprev[slot]);
        const float tf = 1.0f / pdf_prev;
        S4 next_emissive = s4(0.0f);
        if (emissive) next_emissive = fprev * emissive_radiance(sc, mat, hit.uv, wl) * tf;  // base_renderer.rs:125-131
        const S4 modifier = fprev * tf;
        const bool spec_prev = (flags & FLAG_SPEC_PREV) != 0;
        if (integrator == TCPT_INTEGRATOR_PT) {
            con = con + thr * next_emissive;                                  // pt_renderer.rs:41-43
        } else if (integrator == TCPT_INTEGRATOR_NEE) {
            if (spec_prev) con = con + thr * next_emissive;                   // nee_renderer.rs:139-147
        } else {
            if (spec_prev) con = con + thr * next_emissive;                   // mis_renderer.rs:160-163
            else {
                const float4 pp = st.ppos[slot];
                const float pdf_light = scene_pdf_light_sample(sc, lights(), f3(pp.x, pp.y, pp.z), hit.prim, hit.tri, hit.position, hit.normal);
                const float a = pdf_prev, b = pdf_light;
                const float w = (a == 0.0f && b == 0.0f) ? 0.0f : a / (a + b);
                con = con + thr * next_emissive * w;                          // mis_renderer.rs:164-179
            }
        }
        // Russian roulette (base_renderer.rs:76-92) was DECIDED one launch ago, when this ray was spawned (see the end of this
        // function): the throughput after the bounce does not depend on what the ray hits.  A ray that reaches a material bucket
        // survived; its random number is already drawn, only the rescaling is left.
        thr = thr * modifier;
        const float p_rr = s4_max(thr);
        if (!emissive && !(p_rr >= 1.0f) && p_rr != 0.0f) { thr.v[0] /= p_rr; thr.v[1] /= p_rr; thr.v[2] /= p_rr; thr.v[3] /= p_rr; }
    }
    if (stage >= R.max_depth || emissive) { finish(); return; }  // depth loop bound (:197) / emitters have no BSDF (:199-202)
    if constexpr (!emissive) {

    // ---- one bounce (base_renderer.rs:199-237)
    M3 r2t, t2r;
    shading_frame(hit, r2t, t2r);
    const float3 wo = m3_vector(r2t, hit.wo);
    const float3 ng_t = m3_normal_by_inverse(t2r, hit.normal);  // Transform * Normal = inverse(r2t)^T n, normalised
    MatCtx mc; mc.sc = &sc; mc.path_key = smp.key; mc.depth = stage + 1;
    // `uc` only selects between lobes; LambertMaterial::sample and MetalMaterial::sample never read it (lambert_material.rs:42-97, metal_material.rs:124)
    float uc = 0.0f;
    if (NO_LOBE) smp.skip_1d();
    else uc = smp.get_1d(R);
    float2 uv;
    if (PRE && have_pre && smp.dim == pre_d0 + 1u) { uv = pre.a; smp.dim += 2; } else uv = smp.get_2d(R);
    const bool was_terminated = wl.terminated;
    NmFrame nmf;
    material_frame(sc, mat, hit.uv, nmf);
    MatParams mp;
    load_mat_params<MT>(sc, mat, hit.uv, wl, mp);
    mc.mp = &mp;
    const MatSample ms = material_sample<MT>(mc, mat, nmf, uc, uv, wl, wo, ng_t, hit.uv);
    if (wl.terminated != was_terminated) lt_ready = false;  // a dispersive material collapsed the wavelengths: light powers change

    if (!ms.is_specular() && integrator != TCPT_INTEGRATOR_PT) {
        // next event estimation (nee_renderer.rs:18-102, mis_renderer.rs:21-123)
        const bool with_mis = integrator == TCPT_INTEGRATOR_MIS;
        float p_light = 0.0f;
        int li;
        if (sc.n_lights == 1) {
            // one light: sample_light returns it for every u (light_sampler.rs:31-43), with probability w/w
            smp.skip_1d();
            const LightTable& t1 = lights();
            li = t1.sum == 0.0f ? -1 : 0;
            p_light = t1.w[0] / t1.sum;
        } else {
            const float u = smp.get_1d(R);
            li = sample_light(sc, lights(), u, &p_light);
        }
        if (li >= 0) {
            const int lprim = sc.light_list[li];
            const tcpt_flat_primitive& LP = sc.primitives[lprim];
            // `s` picks the triangle of an area light; the environment light ignores it (scene.rs:127-153)
            // (delta lights read neither: the reference draws s and uv before it looks at the kind of light, nee_renderer.rs:41-43)
            float s = 0.0f;
            if (LP.kind == 1) s = smp.get_1d(R); else smp.skip_1d();
            float2 luv = make_float2(0.0f, 0.0f);
            if (LP.kind <= 2) { if (PRE && have_pre && smp.dim == pre_d0 + 5u) { luv = pre.b; smp.dim += 2; } else luv = smp.get_2d(R); }
            else { smp.skip_1d(); smp.skip_1d(); }
            float3 sh_dir; float sh_tmax; S4 pending; float sh_eps = 1e-4f;
            if (LP.kind == 3 || LP.kind == 4) {
                // PointLight / SpotLight::calculate_intensity (point_light.rs:75-88, spot_light.rs:98-122) + evaluate_delta_point_light
                // (common.rs:23-55); delta lights carry no MIS weight (nee_renderer.rs:52-77, mis_renderer.rs:65-100)
                const float3 lpos = xf_point(LP.l2r, f3(0.0f, 0.0f, 0.0f));
                S4 inten = spectrum_sample(sc, spectrum_from_flat(LP.light_spectrum), wl) * LP.light_intensity;
                const float3 dv = lpos - hit.position;
                const float3 wi_r = normalize(dv);
                if (LP.kind == 4) {
                    // quirk: the cosine to the cone axis is compared with the cone ANGLES, smoothstep(angle_outer, angle_inner, cos)
                    const float cos_theta = xf_vector(LP.r2l, wi_r).z;
                    const float t = clampf((cos_theta - LP.angle_outer) / (LP.angle_inner - LP.angle_outer), 0.0f, 1.0f);
                    inten = inten * (t * t * (3.0f - 2.0f * t));
                }
                const float3 wi = m3_vector(r2t, wi_r);
                S4 f; float bpdf;
                material_eval_pdf<MT>(mc, mat, nmf, wl, wo, wi, ng_t, hit.uv, false, &f, &bpdf);
                pending = thr * (f * inten / (length_squared(dv) * p_light));
                sh_dir = wi_r; sh_tmax = length(dv) - 2.0f * 1e-4f;
            } else if (LP.kind == 5) {
                // DirectionalLight::calculate_intensity (directional_light.rs:92-107) + evaluate_delta_directional_light (common.rs:58-79):
                // the shadow ray starts ON the surface (no forward offset) and is unbounded
                const float3 dir = normalize(xf_vector(LP.l2r, f3(0.0f, 0.0f, 1.0f)));
                const S4 inten = spectrum_sample(sc, spectrum_from_flat(LP.light_spectrum), wl) * LP.light_intensity;
                const float3 wi = m3_vector(r2t, normalize(dir));
                S4 f; float bpdf;
                material_eval_pdf<MT>(mc, mat, nmf, wl, wo, wi, ng_t, hit.uv, false, &f, &bpdf);
                pending = thr * (f * inten / p_light);
                sh_dir = dir; sh_tmax = TCPT_FLT_MAX; sh_eps = 0.0f;
            } else if (LP.kind == 2) {
                // EnvironmentLight::sample_infinite_light (environment_light.rs:326-350) + evaluate_infinite_light{,_with_mis} (common.rs:174-241)
                const DEnv& e = sc.envs[LP.env];
                const uint32_t yy = sample_from_cdf(e.marginal, e.h, e.marginal_guide, e.guide_h, luv.x);
                const uint32_t xx = sample_from_cdf(e.conditional + (size_t)yy * e.w, e.w, e.conditional_guide + (size_t)yy * (e.guide_w + 1u), e.guide_w, luv.y);
                const EnvNee en = env_nee_lookup(sc, LP, e, xx, yy);
                const float3 wi_r = en.wi_r;
                const float pdf_dir = en.pdf_dir;
                const S4 radiance = spectrum_sample(sc, en.spec, wl) * e.intensity;
                const float3 wi = m3_vector(r2t, wi_r);
                S4 f; float bpdf;
                material_eval_pdf<MT>(mc, mat, nmf, wl, wo, wi, ng_t, hit.uv, with_mis, &f, &bpdf);
                const float w = with_mis ? ((pdf_dir == 0.0f && bpdf == 0.0f) ? 0.0f : pdf_dir / (pdf_dir + bpdf)) : 1.0f;
                const S4 c = f * radiance / (pdf_dir * p_light);
                pending = with_mis ? thr * c * w : thr * c;
                sh_dir = wi_r; sh_tmax = TCPT_FLT_MAX;
            } else {
                // EmissiveTriangleMesh::sample_radiance (emissive_triangle_mesh.rs:176-309) + evaluate_area_light{,_with_mis} (common.rs:82-171)
                const tcpt_flat_geometry& G = sc.geometries[LP.geometry];
                const float* table = sc.area_table + LP.area_base;
                uint32_t index = 0;
                for (uint32_t i = 0; i < G.tri_count; ++i) if (s < __ldg(table + i)) { index = i; break; }
                float b0, b1;
                if (luv.x < luv.y) { b0 = luv.x / 2.0f; b1 = luv.y - b0; } else { b1 = luv.y / 2.0f; b0 = luv.x - b1; }
                const float b2 = 1.0f - b0 - b1;
                const uint32_t* idx = sc.indices + 3 * ((size_t)G.index_base + index);
                const uint32_t i0 = __ldg(idx) + G.vertex_base, i1 = __ldg(idx + 1) + G.vertex_base, i2 = __ldg(idx + 2) + G.vertex_base;
                const float* pp = sc.positions;
                const float3 p0 = xf_point(LP.l2r, f3(__ldg(pp + 3 * (size_t)i0), __ldg(pp + 3 * (size_t)i0 + 1), __ldg(pp + 3 * (size_t)i0 + 2)));
                const float3 p1 = xf_point(LP.l2r, f3(__ldg(pp + 3 * (size_t)i1), __ldg(pp + 3 * (size_t)i1 + 1), __ldg(pp + 3 * (size_t)i1 + 2)));
                const float3 p2 = xf_point(LP.l2r, f3(__ldg(pp + 3 * (size_t)i2), __ldg(pp + 3 * (size_t)i2 + 1), __ldg(pp + 3 * (size_t)i2 + 2)));
                const float3 lpos = (p0 * b0 + p1 * b1) + p2 * b2;
                const float3 lnormal = normalize(normalize(cross(p1 - p0, p2 - p0)));
                float2 tuv = make_float2(0.0f, 0.0f);
                if (G.has_uv) {
                    const float* uu = sc.uvs;
                    tuv.x = (__ldg(uu + 2 * (size_t)i0) * b0 + __ldg(uu + 2 * (size_t)i1) * b1) + __ldg(uu + 2 * (size_t)i2) * b2;
                    tuv.y = (__ldg(uu + 2 * (size_t)i0 + 1) * b0 + __ldg(uu + 2 * (size_t)i1 + 1) * b1) + __ldg(uu + 2 * (size_t)i2 + 1) * b2;
                }
                // EmissiveSingleTriangle::sample_radiance passes the sample's random numbers on as the light point's uv
                // (emissive_single_triangle.rs:190-252); the rest of it coincides with a one-triangle EmissiveTriangleMesh
                if (G.single) tuv = luv;
                const float3 dv = lpos - hit.position;
                const float3 wi_r = normalize(dv);
                const S4 radiance = emissive_radiance(sc, sc.materials[LP.material], tuv, wl);
                const float pdf_area = 1.0f / LP.area_sum;
                const float distance = length(dv);
                const float pdf_dir = pdf_area * (distance * distance) / rmax(fabsf(dot(lnormal, -wi_r)), 1e-8f);
                const float3 wi = m3_vector(r2t, wi_r);
                S4 f; float bpdf;
                material_eval_pdf<MT>(mc, mat, nmf, wl, wo, wi, ng_t, hit.uv, with_mis, &f, &bpdf);
                const float distance2 = length_squared(dv);
                const float3 ln_t = m3_normal_by_inverse(t2r, lnormal);
                const float cos_light = fabsf(dot(ln_t, -wi));
                const float g = cos_light / distance2;
                const float w = with_mis ? ((pdf_dir == 0.0f && bpdf == 0.0f) ? 0.0f : pdf_dir / (pdf_dir + bpdf)) : 1.0f;
                const S4 c = f * radiance * g / (pdf_area * p_light);
                pending = with_mis ? thr * c * w : thr * c;
                sh_dir = wi_r; sh_tmax = distance - 2.0f * 1e-4f;
            }
            const float3 so = sh_eps != 0.0f ? hit.position + sh_dir * sh_eps : hit.position;  // move_forward(1e-4), no normal offset (common.rs:12,134-140)
            out.push_sh = true;
            out.so = make_float4(so.x, so.y, so.z, sh_tmax);
            out.sd = make_float4(sh_dir.x, sh_dir.y, sh_dir.z, __uint_as_float(slot));
            out.sc = to_f4(pending);
        }
    }

    if (!ms.sampled) {
        // process_bsdf_sampling returned None: the path ends here (base_renderer.rs:240-253 adds nothing for a failed sample)
        st.con[slot] = to_f4(con);
        if (out.push_sh) {
            out.sd.w = __uint_as_float(slot | 0x80000000u);
            st.misc[slot] = make_float4(0.0f, lambda0, __uint_as_float(smp.dim), __uint_as_float(wl.terminated ? FLAG_LAMBDA_TERMINATED : 0u));
        } else finish();
        return;
    }
    // spawn the extension ray (base_renderer.rs:111-121)
    const float3 wi_render = m3_vector(t2r, ms.wi);
    const float sign = dot(hit.normal, wi_render) < 0.0f ? -1.0f : 1.0f;
    const float3 origin = hit.position + (sign * hit.normal) * 1e-5f;
    const float3 o2 = origin + wi_render * 1e-5f;
    // Russian roulette of this bounce, decided now (base_renderer.rs:76-92 runs it after the next intersection, but neither the
    // throughput nor the sampler dimension depends on that hit, and an emissive or missed hit ends the path whatever the outcome).
    // A killed path still needs its ray traced -- the hit may be a light -- but then goes to the terminal bucket instead of
    // riding through a material's shading code with its lane switched off (bounce-1 shading ran at 16-22 of 32 lanes).
    bool killed = false;
    if (stage + 1 <= R.max_depth) {
        const S4 thr2 = thr * (ms.f * (1.0f / ms.pdf));
        const float p_rr = s4_max(thr2);
        if (!(p_rr >= 1.0f)) {
            float u_rr;
            if (PRE && have_pre && smp.dim == pre_d0 + 7u) { u_rr = pre.c; smp.dim += 1; } else u_rr = smp.get_1d(R);
            killed = !(u_rr < p_rr);
        }
    }
    out.push_ext = true;
    out.eo = make_float4(o2.x, o2.y, o2.z, TCPT_FLT_MAX);
    out.ed = make_float4(wi_render.x, wi_render.y, wi_render.z, __uint_as_float(slot | (killed ? 0x80000000u : 0u)));
    st.thr[slot] = to_f4(thr);
    st.con[slot] = to_f4(con);
    st.fprev[slot] = to_f4(ms.f);
    st.ppos[slot] = make_float4(hit.position.x, hit.position.y, hit.position.z, 0.0f);
    flags = (ms.is_specular() ? FLAG_SPEC_PREV : 0u) | (wl.terminated ? FLAG_LAMBDA_TERMINATED : 0u);
    st.misc[slot] = make_float4(ms.pdf, lambda0, __uint_as_float(smp.dim), __uint_as_float(flags));
    }  // !emissive
    }  // !miss
}

// What a vertex reads before it can start: its queue position (through the bucketed order), the ray it arrived on, the hit record and
// the head of its path state: a chain of DEPENDENT loads (order -> ray -> slot -> state), each a DRAM round trip at the benchmarked pass
// size.  The order entry of the NEXT vertex is asked for before this one is shaded (two registers across the vertex).
struct VertexIn { float4 d, h0, misc; uint2 h1; };
template <int B>
__device__ __forceinline__ OrderEntry load_order(const DState& st, uint32_t p, uint32_t n) {
    OrderEntry o = make_uint2(0u, 0u);
    if (p < n) o = st.order[(size_t)B * st.capacity + p];
    return o;
}
template <int B>
__device__ __forceinline__ VertexIn load_vertex(const DState& st, int cur, OrderEntry o, bool valid) {
    VertexIn v;
    v.d = make_float4(0.0f, 0.0f, 0.0f, 0.0f); v.h0 = v.d; v.misc = v.d; v.h1 = make_uint2(0u, 0u);
    if (valid) {
        const uint32_t i = o.x;
        v.misc = st.misc[o.y];
        v.d = st.ext_d[cur][i];
        if (B < 7) { v.h0 = st.hit0[i]; v.h1 = st.hit1[i]; }   // an escaped ray and a path Russian roulette ended read nothing of the hit record: 24 B per vertex less
    }
    return v;
}
// Appends the extension and shadow rays a vertex of bucket b spawned to their queues.  Every lane of the warp must call it with the same b.
__device__ __forceinline__ void push_rays(const DState& st, int cur, int sh, int b, const ShadeOut& out) {
    if (b < 6) {   // emissive hits and misses end the path: nothing to push
        uint32_t pe, ps;
        warp_push2(&st.counters[cur ^ 1], out.push_ext, &st.counters[sh], out.push_sh, &pe, &ps);
        if (out.push_ext) { st.ext_o[cur ^ 1][pe] = out.eo; st.ext_d[cur ^ 1][pe] = out.ed; }
        if (out.push_sh) { st.sh_o[ps] = out.so; st.sh_d[ps] = out.sd; st.sh_c[ps] = out.sc; }
    }
}

// One instantiation per shading bucket; each walks only its own range of the bucketed order.
#ifndef TCPT_SHADE_THREADS
#define TCPT_SHADE_THREADS 512
#endif
#ifndef TCPT_SHADE_THREADS_LAMBERT
#define TCPT_SHADE_THREADS_LAMBERT TCPT_SHADE_THREADS
#endif
#ifndef TCPT_SHADE_THREADS_MISS
#define TCPT_SHADE_THREADS_MISS TCPT_SHADE_THREADS   // block size of the buckets that end the path (emissive, miss, terminal)
#endif
#ifndef TCPT_SHADE_MIN_BLOCKS_MISS
#define TCPT_SHADE_MIN_BLOCKS_MISS 8                 // their resident 128-thread units per SM (8: 64 registers).  256-thread blocks x 3 (85 registers, no spills) / x 4, 128-thread blocks x 5: 31.5 / 31.4 / 32.4 ms of shading per step against 31.4 (profiles/r02l_ab_miss_bucket_configs.log)
#endif
// block shape of k_shade<B>: the material buckets run ONE big block per SM whose warps start every vertex together (see the kernel);
// the register budget follows from the block size (512 threads: 128 registers, 640: 96, 768: 80)
template <int B> struct ShadeCfg {
    static constexpr int threads = B >= 6 ? TCPT_SHADE_THREADS_MISS : B == 5 ? TCPT_SHADE_THREADS_LAMBERT : TCPT_SHADE_THREADS;
    static constexpr int per_sm_128 = B >= 6 ? TCPT_SHADE_MIN_BLOCKS_MISS : B == 5 ? TCPT_SHADE_MIN_BLOCKS_LAMBERT : TCPT_SHADE_MIN_BLOCKS;   // resident blocks if blocks were 128 threads
    static constexpr int min_blocks = per_sm_128 * 128 / threads > 0 ? per_sm_128 * 128 / threads : 1;
};
template <int B, bool FIRST = false>
__global__ void __launch_bounds__(ShadeCfg<B>::threads, ShadeCfg<B>::min_blocks) k_shade(const __grid_constant__ DScene sc, const __grid_constant__ DRender R,
                                                                                     const __grid_constant__ DState st, const __grid_constant__ PathList L, int cur, int sh, uint32_t stage) {
    if (B == 0 && blockIdx.x == 0 && threadIdx.x == 0) { st.counters[24] = 0; st.counters[25] = 0; }  // work counters of the next trace launch
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t n = st.counters[4 + TCPT_BUCKET_STRIDE * cur + B];
    // whole warps iterate together (push_rays is warp-collective); in the material buckets whole blocks do, and start every vertex together
    const uint32_t unit = B < 6 ? (uint32_t)ShadeCfg<B>::threads : 32u;
    const uint32_t n_round = (n + unit - 1u) / unit * unit;
    // the order entry of the NEXT vertex is loaded before this one is shaded: of the dependent round trips in front of a vertex only one
    // is left exposed (ncu: 15 % of the Lambert kernel's stall samples sat on these loads).  Loading the whole next vertex ahead holds
    // 15 registers across the shading and was slower (DESIGN.md section 3).
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    VertexIn v = load_vertex<B>(st, cur, load_order<B>(st, p, n), p < n);
    for (; p < n_round; p += stride) {
        const uint32_t pn = p + stride;
        const bool more = pn < n && pn > p;
        const OrderEntry o_next = load_order<B>(st, pn, more ? n : 0u);
        if (B < 6) __syncthreads();
        ShadeOut out; out.push_ext = false; out.push_sh = false;   // (p >= n: the lane only takes part in the warp-collective push)
        if (p < n) shade_vertex<B, FIRST>(sc, R, st, L, stage, f3(v.d.x, v.d.y, v.d.z), __float_as_uint(v.d.w) & 0x7fffffffu, v.h0, v.h1, v.misc, out);
        push_rays(st, cur, sh, B, out);
        v = load_vertex<B>(st, cur, o_next, more);
    }
}

// shade_vertex<B> behind a call, so that the eight instantiations keep their own register allocation inside k_shade_all
template <int B>
__device__ __noinline__ void shade_vertex_call(const DScene& sc, const DRender& R, const DState& st, const PathList& L, int cur, uint32_t stage, uint32_t i, ShadeOut& out) {
    const float4 d = st.ext_d[cur][i];
    const uint32_t slot = __float_as_uint(d.w) & 0x7fffffffu;
    shade_vertex<B>(sc, R, st, L, stage, f3(d.x, d.y, d.z), slot, st.hit0[i], st.hit1[i], st.misc[slot], out);
}

// All buckets in one launch: the launch is cut into chunks of 128 consecutive positions of ONE bucket, numbered bucket by bucket
// (heaviest code first), and blocks take chunks round-robin.  A block only ever runs one material's code at a time and
// neighbouring blocks mostly run the same one, so the instruction cache behaves as with eight launches, without seven
// launch boundaries per bounce (each bounded below by the latency of one warp running a 5000-instruction program from a cold
// instruction cache: about 0.3 ms per bounce whatever the queue length).
__global__ void __launch_bounds__(128, TCPT_SHADE_MIN_BLOCKS) k_shade_all(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DState st,
                                                                           const __grid_constant__ PathList L, int cur, int sh, uint32_t stage) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { st.counters[24] = 0; st.counters[25] = 0; }  // work counters of the next trace launch
    uint32_t cnt[TCPT_N_BUCKETS], total = 0;
#pragma unroll
    for (int b = 0; b < TCPT_N_BUCKETS; ++b) { cnt[b] = st.counters[4 + TCPT_BUCKET_STRIDE * cur + b]; total += (cnt[b] + 127u) >> 7; }
    for (uint32_t v = blockIdx.x; v < total; v += gridDim.x) {
        uint32_t c = v, n = cnt[0]; int b = 0;
#pragma unroll
        for (int k = 0; k < TCPT_N_BUCKETS - 1; ++k) { const uint32_t ch = (cnt[k] + 127u) >> 7; if (b == k && c >= ch) { c -= ch; b = k + 1; n = cnt[k + 1]; } }
        const uint32_t p = c * 128u + threadIdx.x;
        ShadeOut out; out.push_ext = false; out.push_sh = false;
        if (p < n) {
            const uint32_t i = st.order[(size_t)b * st.capacity + p].x;
            switch (b) {
                case 0: shade_vertex_call<0>(sc, R, st, L, cur, stage, i, out); break;
                case 1: shade_vertex_call<1>(sc, R, st, L, cur, stage, i, out); break;
                case 2: shade_vertex_call<2>(sc, R, st, L, cur, stage, i, out); break;
                case 3: shade_vertex_call<3>(sc, R, st, L, cur, stage, i, out); break;
                case 4: shade_vertex_call<4>(sc, R, st, L, cur, stage, i, out); break;
                case 5: shade_vertex_call<5>(sc, R, st, L, cur, stage, i, out); break;
                case 6: shade_vertex_call<6>(sc, R, st, L, cur, stage, i, out); break;
                case 7: shade_vertex_call<7>(sc, R, st, L, cur, stage, i, out); break;
                default: shade_vertex_call<8>(sc, R, st, L, cur, stage, i, out); break;
            }
        }
        push_rays(st, cur, sh, b, out);   // (b is uniform over the block)
    }
}

// ---------------------------------------------------------------- AOV renderers (renderer/src/renderer/{albedo,normal}_renderer.rs): one camera ray per sample
__device__ __noinline__ S4 material_albedo(const DScene& sc, const tcpt_flat_material& m, float2 uv, const DWavelengths& wl) {  // BsdfSurfaceMaterial::sample_albedo_spectrum
    switch (m.type) {
        case TCPT_MAT_LAMBERT: case TCPT_MAT_SIMPLE_PBR: case TCPT_MAT_CLEARCOAT_PBR: return spectrum_sample(sc, param_spectrum(sc, m.color, uv), wl);
        case TCPT_MAT_METAL: return fresnel_complex(1.0f, spectrum_sample(sc, spectrum_from_flat(m.color), wl), spectrum_sample(sc, spectrum_from_flat(m.coat_tint), wl));  // metal_material.rs:267-278
        case TCPT_MAT_PLASTIC: case TCPT_MAT_GLASS: return s4(1.0f);
        default: return s4(0.0f);
    }
}
__global__ void __launch_bounds__(128) k_aov(const __grid_constant__ DScene sc, const __grid_constant__ DRender R, const __grid_constant__ DState st) {
    const uint32_t n = st.counters[0], stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float4 d = st.ext_d[0][i];
        const uint32_t slot = __float_as_uint(d.w) & 0x7fffffffu;
        const float4 h0 = st.hit0[i]; const uint2 h1 = st.hit1[i];
        float3 rgb = f3(0.0f, 0.0f, 0.0f);
        if ((int)h1.x >= 0) {
            DSurface hit;
            reconstruct_hit(sc, (int)h1.x, h1.y, h0.y, h0.z, h0.w, f3(d.x, d.y, d.z), hit);
            const tcpt_flat_material& mat = sc.materials[hit.material];
            if (R.integrator == TCPT_INTEGRATOR_NORMAL) {  // normal_renderer.rs:44-66
                float3 nrm = hit.shading_normal;
                if (mat.type != TCPT_MAT_EMISSIVE) { M3 r2t, t2r; shading_frame(hit, r2t, t2r); nrm = m3_normal_by_inverse(t2r, hit.shading_normal); }
                rgb = f3(nrm.x * 0.5f + 0.5f, nrm.y * 0.5f + 0.5f, nrm.z * 0.5f + 0.5f) * 1.0f;
            } else if (mat.type != TCPT_MAT_EMISSIVE) {    // albedo_renderer.rs:52-62
                const DWavelengths wl = wavelengths_uniform(st.misc[slot].y, false);
                const S4 a = material_albedo(sc, mat, hit.uv, wl) * 1.0f;
                S4 s;
#pragma unroll
                for (int k = 0; k < 4; ++k) s.v[k] = a.v[k] * cmf_at(sc, wl.lambda[k]).w;  // multiply_spectrum with D65 (sampled_spectrum.rs:270-281)
                rgb = sensor_rgb(sc, wl.lambda[0], wl.terminated, s, 1.0f);
            }
        }
        st.rgb[slot] = make_float4(rgb.x, rgb.y, rgb.z, 0.0f);
    }
}

// ---------------------------------------------------------------- K5 film: acc[pixel] += rgb of samples s_begin .. s_begin + s_count, in order
__global__ void __launch_bounds__(256) k_film(const __grid_constant__ DRender R, const float4* __restrict__ rgb, float* __restrict__ acc) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < R.n_pix; p += stride) {
        const uint32_t k = R.pix_begin + p;   // passes over a pixel list (R.pix_list) use k_film_moments
        const uint32_t row = k / R.width;
        const uint32_t px = k - row * R.width, py = R.row_offset + row * R.row_stride;
        float* a = acc + 3 * ((size_t)py * R.width + px);
        float r = a[0], g = a[1], b = a[2];
        for (uint32_t s = 0; s < R.s_count; ++s) {
            const float4 v = rgb[(size_t)s * R.n_pix + p];
            r += v.x; g += v.y; b += v.z;
        }
        a[0] = r; a[1] = g; a[2] = b;
    }
}

// Sensor::to_rgb (sensor.rs:81-88) + ReinhardToneMap (tone_map.rs:20-28) + sRGB OETF (color/src/eotf.rs:53-61)
// mode: 0 = the integrators (Reinhard), 1 = AlbedoRenderer (NoneToneMap sensor: no tone map), 2 = NormalRenderer (mean only, normal_renderer.rs:72-74)
__global__ void __launch_bounds__(256) k_finalize(const float* __restrict__ acc, float* __restrict__ out, uint32_t n_values, float spp, int mode) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_values; i += stride) {
        float c = acc[i] / spp;
        if (mode == 2) { out[i] = c; continue; }
        c = c > 0.0f ? c : 0.0f;  // Vec3::max(ZERO)
        if (mode == 0) c = c / (1.0f + c);
        out[i] = linear_to_srgb(c);
    }
}

// ---------------------------------------------------------------- adaptive sampling (tcpt_render_adaptive)
// k_film plus the per-pixel luminance moments of the stopping rule: mom[pixel] = {S1, S2} += {y, y*y} with y = (0.2126 r + 0.7152 g) + 0.0722 b
// of every sample the film adds, in the same loop and the same order (f32, no contraction: the library builds with --fmad=false)
__global__ void __launch_bounds__(256) k_film_moments(const __grid_constant__ DRender R, const float4* __restrict__ rgb, float* __restrict__ acc, float2* __restrict__ mom) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < R.n_pix; p += stride) {
        const uint32_t k = owned_pixel(R, p);
        const uint32_t row = k / R.width;
        const uint32_t px = k - row * R.width, py = R.row_offset + row * R.row_stride;
        const size_t pix = (size_t)py * R.width + px;
        float* a = acc + 3 * pix;
        float r = a[0], g = a[1], b = a[2];
        float2 m = mom[pix];
        for (uint32_t s = 0; s < R.s_count; ++s) {
            const float4 v = rgb[(size_t)s * R.n_pix + p];
            r += v.x; g += v.y; b += v.z;
            const float y = (0.2126f * v.x + 0.7152f * v.y) + 0.0722f * v.z;
            m.x += y; m.y += y * y;
        }
        a[0] = r; a[1] = g; a[2] = b;
        mom[pix] = m;
    }
}

// the stopping rule after k samples: relative standard error of the mean luminance below `threshold`, with an absolute floor of 1e-3
// (IEEE division and square root; a pixel whose sums are not finite never stops)
__device__ __forceinline__ bool adaptive_converged(float2 m2, uint32_t k, float threshold) {
    const float kf = (float)k;
    const float m = m2.x / kf;
    float v = m2.y / kf - m * m;
    v = v > 0.0f ? v : 0.0f;
    const float e = sqrtf(v / (kf - 1.0f));
    return isfinite(m2.x) && isfinite(m2.y) && e < threshold * (fabsf(m) + 1e-3f);
}

// Stream compaction of the active pixel list, count / scan / scatter: tiles of TCPT_SELECT_THREADS x TCPT_SELECT_ITEMS consecutive entries,
// each thread owning TCPT_SELECT_ITEMS consecutive ones, so the survivors keep their (ascending) order.  Deterministic: no atomics.
#define TCPT_SELECT_THREADS 256
#define TCPT_SELECT_ITEMS 4
#define TCPT_SELECT_TILE (TCPT_SELECT_THREADS * TCPT_SELECT_ITEMS)

// exclusive prefix sum of v over the block (blockDim.x a multiple of 32, at most 1024); *total = the block's sum.  Every thread must call it.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (uint32_t o = 1; o < 32u; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31u) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < n_warps ? warp_sums[lane] : 0u;
#pragma unroll
        for (uint32_t o = 1; o < 32u; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
        if (lane < n_warps) warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t excl = x - v + (warp ? warp_sums[warp - 1] : 0u);
    *total = warp_sums[n_warps - 1];
    __syncthreads();   // warp_sums is reused by the next call
    return excl;
}

// The rows of a job (DRender::row_offset / row_stride) and the exact division by the width (DRender::width_magic): owned pixel index ->
// frame pixel index, the index of the per-pixel tables (moments, counts)
struct RowMap {
    uint32_t width, row_offset, row_stride; uint64_t width_magic;
    __device__ __forceinline__ uint32_t frame_pixel(uint32_t k) const {
        const uint32_t row = div_magic(k, width_magic);
        return (row_offset + row * row_stride) * width + (k - row * width);
    }
};

// this thread's entries of the active list (nullptr = the identity list 0 .. n - 1): owned indices, their frame indices and the mask of
// the ones that stay active
__device__ __forceinline__ uint32_t adaptive_items(const uint32_t* __restrict__ list, uint32_t n, const float2* __restrict__ mom, uint32_t k, float threshold,
                                                   const RowMap& rm, uint32_t own[TCPT_SELECT_ITEMS], uint32_t pix[TCPT_SELECT_ITEMS], uint32_t* valid) {
    const uint32_t first = (blockIdx.x * TCPT_SELECT_THREADS + threadIdx.x) * TCPT_SELECT_ITEMS;
    uint32_t keep = 0u, ok = 0u;
#pragma unroll
    for (uint32_t j = 0; j < TCPT_SELECT_ITEMS; ++j) {
        const uint32_t i = first + j;
        own[j] = pix[j] = 0u;
        if (i >= n) continue;
        own[j] = list ? list[i] : i;
        pix[j] = rm.frame_pixel(own[j]);
        ok |= 1u << j;
        if (!adaptive_converged(mom[pix[j]], k, threshold)) keep |= 1u << j;
    }
    *valid = ok;
    return keep;
}

// count: every pixel that stops gets its sample count k (at its frame index); tile_counts[tile] = survivors of the tile
__global__ void __launch_bounds__(TCPT_SELECT_THREADS) k_adaptive_count(const uint32_t* __restrict__ list, uint32_t n, const float2* __restrict__ mom,
                                                                        uint32_t k, float threshold, const RowMap rm, uint32_t* __restrict__ counts,
                                                                        uint32_t* __restrict__ tile_counts) {
    uint32_t own[TCPT_SELECT_ITEMS], pix[TCPT_SELECT_ITEMS], valid;
    const uint32_t keep = adaptive_items(list, n, mom, k, threshold, rm, own, pix, &valid);
#pragma unroll
    for (uint32_t j = 0; j < TCPT_SELECT_ITEMS; ++j)
        if (((valid & ~keep) >> j) & 1u) counts[pix[j]] = k;
    uint32_t total;
    block_exclusive_scan((uint32_t)__popc(keep), &total);
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

// scan: tile_counts -> exclusive offsets in place, *n_out = number of survivors (one block of 1024 threads walks the tiles in order)
__global__ void __launch_bounds__(1024) k_adaptive_scan(uint32_t* __restrict__ tile_counts, uint32_t n_tiles, uint32_t* __restrict__ n_out) {
    uint32_t carry = 0u;
    for (uint32_t base = 0; base < n_tiles; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < n_tiles ? tile_counts[i] : 0u;
        uint32_t sum;
        const uint32_t e = block_exclusive_scan(v, &sum);
        if (i < n_tiles) tile_counts[i] = carry + e;
        carry += sum;
    }
    if (threadIdx.x == 0) *n_out = carry;
}

// scatter: the owned indices of every tile's survivors to list_out from the tile's offset, in list (ascending) order (the rule is evaluated
// again: same inputs, same answer)
__global__ void __launch_bounds__(TCPT_SELECT_THREADS) k_adaptive_scatter(const uint32_t* __restrict__ list, uint32_t n, const float2* __restrict__ mom,
                                                                          uint32_t k, float threshold, const RowMap rm, const uint32_t* __restrict__ tile_offsets,
                                                                          uint32_t* __restrict__ list_out) {
    uint32_t own[TCPT_SELECT_ITEMS], pix[TCPT_SELECT_ITEMS], valid;
    const uint32_t keep = adaptive_items(list, n, mom, k, threshold, rm, own, pix, &valid);
    uint32_t total;
    uint32_t o = tile_offsets[blockIdx.x] + block_exclusive_scan((uint32_t)__popc(keep), &total);
#pragma unroll
    for (uint32_t j = 0; j < TCPT_SELECT_ITEMS; ++j)
        if ((keep >> j) & 1u) list_out[o++] = own[j];
}

// k_finalize mode 0 with a per-pixel divisor: the value of a pixel with count k is bitwise what k_finalize gives with spp = k
__global__ void __launch_bounds__(256) k_finalize_counts(const float* __restrict__ acc, const uint32_t* __restrict__ counts, float* __restrict__ out, uint32_t n_values) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_values; i += stride) {
        float c = acc[i] / (float)counts[i / 3u];
        c = c > 0.0f ? c : 0.0f;
        c = c / (1.0f + c);
        out[i] = linear_to_srgb(c);
    }
}

// p[frame pixel of owned index i] = value for the n owned pixels of a job; no other entry of p is written
__global__ void __launch_bounds__(256) k_fill_owned_u32(uint32_t* __restrict__ p, uint32_t n, const RowMap rm, uint32_t value) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[rm.frame_pixel(i)] = value;
}

// ---------------------------------------------------------------- single-stage probes for parity tests and the traversal micro-benchmark
template <bool COUNT>
__global__ void __launch_bounds__(128) k_trace_rays(const __grid_constant__ DScene sc, const float4* __restrict__ q_o, const float4* __restrict__ q_d, uint32_t n,
                                                     int any_hit, float4* __restrict__ hit0, uint2* __restrict__ hit1, unsigned long long* stats, uint32_t* work) {
    uint32_t nb = 0, nt = 0;
    __shared__ TraceShared ts;
    auto store = [&](uint32_t i, const DHit& h) {
        hit0[i] = make_float4(h.t, h.b0, h.b1, h.b2);
        hit1[i] = make_uint2((uint32_t)h.prim, h.tri);
    };
    if (any_hit) trace_queue<true, COUNT>(sc, ts, q_o, q_d, n, work, &nb, &nt, commit_now(store));
    else trace_queue<false, COUNT>(sc, ts, q_o, q_d, n, work, &nb, &nt, commit_now(store));
    if (COUNT && stats) { atomicAdd(&stats[2], (unsigned long long)nb); atomicAdd(&stats[3], (unsigned long long)nt); }
}

// tcpt_trace's host-facing layouts <-> the SoA queues: rays n x {o[3], d[3], tmax} -> n x {o, tmax} then n x {d, 0};
// hit records n x {t, b0, b1, b2} then n x {prim, tri} -> n x {prim, tri, t bits, b0 bits, b1 bits, b2 bits} (any hit: {0|1, 0, 0, 0, 0, 0})
__global__ void __launch_bounds__(256) k_pack_rays(const float* __restrict__ in, int n, float4* __restrict__ q) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* r = in + 7 * (size_t)i;
        q[i] = make_float4(r[0], r[1], r[2], r[6]);
        q[(size_t)n + i] = make_float4(r[3], r[4], r[5], 0.0f);
    }
}
__global__ void __launch_bounds__(256) k_unpack_hits(const float4* __restrict__ h0, int n, int any_hit, int32_t* __restrict__ out) {
    const uint2* h1 = (const uint2*)(h0 + n);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 a = h0[i]; const uint2 b = h1[i];
        int32_t* o = out + 6 * (size_t)i;
        const int32_t prim = (int32_t)b.x;
        if (any_hit) { o[0] = prim >= 0 ? 1 : 0; o[1] = o[2] = o[3] = o[4] = o[5] = 0; }
        else if (prim < 0) { o[0] = -1; o[1] = o[2] = o[3] = o[4] = o[5] = 0; }
        else { o[0] = prim; o[1] = (int32_t)b.y; o[2] = __float_as_int(a.x); o[3] = __float_as_int(a.y); o[4] = __float_as_int(a.z); o[5] = __float_as_int(a.w); }
    }
}

__global__ void k_cdf_search(const float* __restrict__ cdf, uint32_t n, const uint32_t* __restrict__ guide, uint32_t G, const float* __restrict__ u, int m, uint32_t* __restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) out[i] = sample_from_cdf(cdf, n, guide, G, u[i]);
}

__global__ void k_sampler_stream(const __grid_constant__ DRender R, uint32_t px, uint32_t py, uint32_t si, const int32_t* kinds, int n, float* out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    DSampler smp = make_sampler(R, px, py, si);
    int k = 0;
    for (int i = 0; i < n; ++i) {
        if (kinds[i] == 1) out[k++] = smp.get_1d(R);
        else { const float2 v = smp.get_2d(R); out[k++] = v.x; out[k++] = v.y; }
    }
}

}  // namespace tcpt
