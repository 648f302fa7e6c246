// libtcpt: context, device memory, frame orchestration and the C ABI of include/tcpt.h / include/tcpt_flat.h.
// Product code.  There is no CPU fallback: without a usable sm_100 device every computing entry point fails with TCPT_ERR_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include "host_image.h"
#include "host_obj.h"
#include <nccl.h>   // types only: the library is opened at run time by tcpt_comm_init (see NcclApi)

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/tcpt.h"
#include "../../include/tcpt_flat.h"
#include "host_scene.h"
#include "kernels.cuh"
#include "lbvh.cuh"

using namespace tcpt;

namespace {

struct DeviceBuffers {  // one flattened scene on the device
    std::vector<void*> allocs;
    DScene view{};
    uint32_t max_bvh_depth = 0;
    bool valid = false;
    bool traversal_only = false;   // built by tcpt_scene_build_soup: BVH and triangles only, nothing to shade with
};

struct Options { int count_tests = 0, stage_timing = 0, blocks_per_sm = 8, pin_host_buffers = 0, debug_path_log = 0, sobol_prefix = 1, sobol_prefix_mb = 8192, sobol_pass = 1, sobol_pass_dims = 11, sobol_hash = 1, illum_half = 1, generate_pixels = 1, sobol_pass_cache = 1, refill_b0 = 32, refill = TCPT_REFILL_IDLE_LANES, chunk_b0 = 512, chunk = 512, fused_launches = 3, fused_shade_from = 3, light_shortcut = 1, env_nee_table = 1, soup_leaf = 1; };
struct HostPin { void* ptr = nullptr; size_t bytes = 0; };

}  // namespace

// NCCL entry points, resolved from libnccl.so.2 when the first communicator is made.  libtcpt carries no link-time dependency on NCCL:
// a single-GPU host never loads it, and inside a process that already holds an NCCL (PyTorch's) the same copy is reused by soname.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
    bool load() {
        static std::mutex m;
        std::lock_guard<std::mutex> lock(m);
        if (handle) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) { handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (handle) break; }
        if (!handle) { error = std::string("cannot open libnccl.so.2: ") + dlerror(); return false; }
        bool ok = true;
        auto sym = [&](const char* name) { void* p = dlsym(handle, name); if (!p) { ok = false; error = std::string("libnccl lacks ") + name; } return p; };
        GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
        Reduce = (decltype(Reduce))sym("ncclReduce");
        GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
        if (!ok) { dlclose(handle); handle = nullptr; }
        return ok;
    }
};
static NcclApi g_nccl;

struct tcpt_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string error;
    HostScene host;
    FlatStorage flat;
    DeviceBuffers dev;
    // tables on the device
    float4* d_cmf = nullptr; float* d_rgb2spec = nullptr;  // d_rgb2spec = 64 z nodes + table
    uint32_t* d_sobol_bytes = nullptr;                      // Sobol matrix 1 folded per index byte (7 x 256)
    float* d_presets = nullptr;                             // dense metal / glass tables, n x 470
    float xyz_to_rgb[9];
    // wavefront buffers
    DState st{};
    uint32_t st_capacity = 0;
    std::vector<void*> st_allocs;
    unsigned long long* d_stats = nullptr;
    uint32_t* d_counters = nullptr;
    Options opt;
    tcpt_stats stats{};
    int sm_count = 148;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0; std::vector<int> ev_stage;  // stage timing (see StageTimer)
    // tcpt_render's own film buffers (grow-only) and the caller's output buffers currently page-locked for direct DMA
    float* film_acc = nullptr; float* film_srgb = nullptr; size_t film_cap = 0;
    HostPin pins[3];   // out_acc, out_srgb, out_spp
    // tcpt_render_adaptive's buffers (grow-only, in pixels): luminance moments (float2), sample counts, two active lists, compaction scratch
    void* adapt_buf = nullptr; size_t adapt_cap = 0;
    // ZSobol pixel-prefix table (DSampler::sample_index), cached per (width, height, log2_spp); grows when more dimensions are asked for
    float half_lin = 0.0f; int32_t half_zi = -1;   // DScene::half_lin / half_zi (tcpt_set_tables)
    void* trace_scratch = nullptr; size_t trace_scratch_cap = 0;   // device staging of tcpt_trace (rays in, hit records out), kept between calls
    unsigned long long* d_sobol_hash = nullptr; uint32_t sobol_hash_seed = 0; bool sobol_hash_valid = false;
    uint32_t* d_prefix = nullptr; uint32_t prefix_w = 0, prefix_h = 0, prefix_log2spp = 0, prefix_dims = 0, pass_rows = 0; size_t prefix_cap = 0;
    double prefix_build_ms = 0.0;
    uint64_t default_slots = 0;  // path-slot budget of a pass when the caller gives none (see render_into)
    // multi-GPU: this context's rank in an NCCL communicator (tcpt_comm_init); the ctx owns the communicator
    ncclComm_t comm = nullptr; int comm_rank = 0, comm_size = 1;
    double soup_build_ms = 0.0; uint64_t soup_records = 0; uint32_t soup_levels = 0;   // last tcpt_scene_build_soup
    cudaEvent_t ev_r0 = nullptr, ev_r1 = nullptr;
};

namespace {

int fail(tcpt_ctx* c, int code, const std::string& msg) { if (c) c->error = msg; return code; }
#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(ctx, TCPT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

template <class T>
int upload(tcpt_ctx* ctx, DeviceBuffers& db, const T* src, size_t n, const T** dst) {
    *dst = nullptr;
    void* p = nullptr;
    const size_t bytes = (n ? n : 1) * sizeof(T);
    CU(cudaMalloc(&p, bytes));
    db.allocs.push_back(p);
    if (n) CU(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
    *dst = (const T*)p;
    return TCPT_OK;
}

void free_scene(DeviceBuffers& db) {
    for (void* p : db.allocs) cudaFree(p);
    db.allocs.clear();
    db.valid = false;
    db.traversal_only = false;
}

// color/src/gamut.rs:29-69 with glam's Mat3 arithmetic (column major), evaluated on the host like the reference does
void srgb_xyz_to_rgb(float out[9]) {
    struct V { float x, y, z; };
    auto xy = [](float x, float y) { return y == 0.0f ? V{0, 0, 0} : V{x * 1.0f / y, 1.0f, (1.0f - x - y) * 1.0f / y}; };
    auto cross = [](V a, V b) { return V{a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y}; };
    auto dot = [](V a, V b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); };
    auto scale = [](V a, float s) { return V{a.x * s, a.y * s, a.z * s}; };
    auto add = [](V a, V b) { return V{a.x + b.x, a.y + b.y, a.z + b.z}; };
    struct M { V c0, c1, c2; };
    auto mulv = [&](const M& m, V v) { return add(add(scale(m.c0, v.x), scale(m.c1, v.y)), scale(m.c2, v.z)); };
    auto inv = [&](const M& m) {
        V t0 = cross(m.c1, m.c2), t1 = cross(m.c2, m.c0), t2 = cross(m.c0, m.c1);
        float id = 1.0f / dot(m.c2, t2);
        V a = scale(t0, id), b = scale(t1, id), c = scale(t2, id);
        return M{V{a.x, b.x, c.x}, V{a.y, b.y, c.y}, V{a.z, b.z, c.z}};
    };
    const M rgb{xy(0.6400f, 0.3300f), xy(0.3000f, 0.6000f), xy(0.1500f, 0.0600f)};
    const V w = xy(0.3127f, 0.3290f);
    const V c = mulv(inv(rgb), w);
    const M diag{V{c.x, 0, 0}, V{0, c.y, 0}, V{0, 0, c.z}};
    const M m{mulv(rgb, diag.c0), mulv(rgb, diag.c1), mulv(rgb, diag.c2)};
    const M r = inv(m);
    const float v[9] = {r.c0.x, r.c0.y, r.c0.z, r.c1.x, r.c1.y, r.c1.z, r.c2.x, r.c2.y, r.c2.z};
    std::memcpy(out, v, sizeof v);
}

// device memory of one path slot: 14 float4 records (path state, both extension queues, hit record, shadow queue), the uint2 half of the
// hit record and one order entry per shading bucket (ensure_state below allocates exactly this list)
constexpr uint64_t kBytesPerSlot = 14 * sizeof(float4) + sizeof(uint2) + sizeof(tcpt::OrderEntry) * TCPT_N_BUCKETS;
static_assert(kBytesPerSlot == 304,"update the figure quoted in include/tcpt.h and DESIGN.md");

int ensure_state(tcpt_ctx* ctx, uint32_t capacity) {
    if (ctx->st_capacity >= capacity) return TCPT_OK;
    for (void* p : ctx->st_allocs) cudaFree(p);
    ctx->st_allocs.clear();
    ctx->st_capacity = 0;
    auto alloc = [&](size_t bytes, void** out) -> int {
        const cudaError_t e = cudaMalloc(out, bytes);
        if (e != cudaSuccess) {   // give back what this attempt took: the caller may retry with a smaller pass
            cudaGetLastError();
            for (void* q : ctx->st_allocs) cudaFree(q);
            ctx->st_allocs.clear();
            ctx->error = std::string("cudaMalloc of the wavefront state: ") + cudaGetErrorString(e);
            return TCPT_ERR_NOMEM;
        }
        ctx->st_allocs.push_back(*out);
        return TCPT_OK;
    };
    DState& s = ctx->st;
    const size_t n = capacity;
    float4** f4s[] = {&s.thr, &s.con, &s.fprev, &s.misc, &s.ppos, &s.rgb, &s.ext_o[0], &s.ext_o[1], &s.ext_d[0], &s.ext_d[1], &s.hit0, &s.sh_o, &s.sh_d, &s.sh_c};
    for (float4** p : f4s) { int r = alloc(n * sizeof(float4), (void**)p); if (r) return r; }
    { int r = alloc(n * sizeof(uint2), (void**)&s.hit1); if (r) return r; }
    { int r = alloc(n * sizeof(tcpt::OrderEntry) * TCPT_N_BUCKETS, (void**)&s.order); if (r) return r; }
    s.capacity = capacity;
    s.counters = ctx->d_counters;
    s.stats = ctx->d_stats;
    ctx->st_capacity = capacity;
    return TCPT_OK;
}

int grid_for(const tcpt_ctx* ctx, uint64_t n, int block) {
    const uint64_t want = (n + block - 1) / block;
    const uint64_t cap = (uint64_t)ctx->sm_count * (uint64_t)ctx->opt.blocks_per_sm;
    return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

uint32_t log2_int(uint32_t v) { return v == 0 ? 0 : 31 - (uint32_t)__builtin_clz(v); }
uint32_t round_up_pow2(uint32_t v) { return v <= 1 ? 1u : 1u << (32 - __builtin_clz(v - 1)); }

// the multiplier of div_magic for the divisor d
uint64_t div_magic_of(uint32_t d) { return d <= 1u ? 0ull : (~0ull) / d + 1ull; }   // floor((2^64 - 1) / d) + 1 == floor(2^64 / d) + 1 unless d divides 2^64: then one more than that, still exact (n / 2^64 < 1 / d)

// DRender::n_pix_magic / width_magic (see div_magic): call after n_pix and width are set
void set_div_magics(DRender& R) {
    R.n_pix_magic = div_magic_of(R.n_pix); R.width_magic = div_magic_of(R.width);
}

int make_render(tcpt_ctx* ctx, const tcpt_render_params* p, DRender& R, DCamera& cam) {
    if (!p || p->width == 0 || p->height == 0 || p->spp == 0) return fail(ctx, TCPT_ERR_INVALID, "render: width, height and spp must be positive");
    if (p->integrator < 0 || p->integrator > TCPT_INTEGRATOR_NORMAL || p->sampler < 0 || p->sampler > 1) return fail(ctx, TCPT_ERR_INVALID, "render: unknown integrator or sampler");
    if (!ctx->dev.valid) return fail(ctx, TCPT_ERR_INVALID, "render: no scene uploaded (call tcpt_scene_build or tcpt_upload_flat_scene)");
    if (ctx->dev.traversal_only) return fail(ctx, TCPT_ERR_INVALID, "render: the scene of tcpt_scene_build_soup holds traversal data only (tcpt_trace / tcpt_trace_device)");
    std::memset(&R, 0, sizeof R);
    R.width = p->width; R.height = p->height; R.spp = p->spp; R.seed = p->seed; R.max_depth = p->max_depth;
    R.integrator = p->integrator; R.sampler = p->sampler; R.exposure = p->exposure;
    // ZSobolSampler::new (z_sobol_sampler.rs:179-196)
    R.log2_spp = log2_int(p->spp);
    const uint32_t res = round_up_pow2(p->width > p->height ? p->width : p->height);
    R.n_base4_digits = log2_int(res) + (R.log2_spp + 1) / 2;
    R.row_offset = p->row_stride ? p->row_offset : 0;
    R.row_stride = p->row_stride ? p->row_stride : 1;
    // Camera::set_look_to + generate_ray constants (camera.rs:39-65); glam Mat3::look_to_rh columns s, u, -f after the transpose
    auto nrm = [](const float v[3], float o[3]) { float l = std::sqrt((v[0] * v[0]) + (v[1] * v[1]) + (v[2] * v[2])); float r = 1.0f / l; o[0] = v[0] * r; o[1] = v[1] * r; o[2] = v[2] * r; };
    float f[3], up[3], s[3], u[3];
    nrm(p->cam_dir, f); nrm(p->cam_up, up);
    float sx[3] = {f[1] * up[2] - up[1] * f[2], f[2] * up[0] - up[2] * f[0], f[0] * up[1] - up[0] * f[1]};
    nrm(sx, s);
    u[0] = s[1] * f[2] - f[1] * s[2]; u[1] = s[2] * f[0] - f[2] * s[0]; u[2] = s[0] * f[1] - f[0] * s[1];
    cam.s = make_float3(s[0], s[1], s[2]); cam.u = make_float3(u[0], u[1], u[2]); cam.nf = make_float3(-f[0], -f[1], -f[2]);
    const float fov_rad = p->fov_deg * (3.14159265358979323846f / 180.0f);  // f32::to_radians
    cam.scale = std::tan(fov_rad / 2.0f);
    cam.aspect = (float)p->width / (float)p->height;
    return TCPT_OK;
}

// ZSobol pixel-prefix table: one u32 per (dimension, pixel) holding the permuted Morton digits of the pixel (everything of
// ZSobolSampler::get_sample_index that does not depend on the sample index), built on `stream` ahead of the frame's first pass and
// kept until the resolution or spp changes.  Dimensions covered: what a max_depth path can draw (3 + 8 per bounce), capped by
// option "sobol_prefix_mb"; deeper dimensions are computed in full by the sampler.
int ensure_sobol_prefix(tcpt_ctx* ctx, DRender& R, cudaStream_t stream) {
    R.sobol_prefix = nullptr; R.prefix_dims = 0; R.prefix_stride = 0; R.pass_info = 0; R.sobol_hash = nullptr;
    if (R.sampler == TCPT_SAMPLER_SOBOL && ctx->opt.sobol_hash) {
        // the 64-bit seeds of the per-dimension Owen scrambles only depend on (dimension, seed): one 4 KB table per context, rebuilt in
        // stream order when the seed changes (a failed allocation just leaves the per-call hash in place)
        if (!ctx->d_sobol_hash && cudaMalloc((void**)&ctx->d_sobol_hash, TCPT_SOBOL_HASH_N * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); ctx->d_sobol_hash = nullptr; }
        if (ctx->d_sobol_hash) {
            if (!ctx->sobol_hash_valid || ctx->sobol_hash_seed != R.seed) {
                k_sobol_hash<<<(TCPT_SOBOL_HASH_N + 255) / 256, 256, 0, stream>>>(ctx->d_sobol_hash, R.seed);
                ctx->sobol_hash_seed = R.seed; ctx->sobol_hash_valid = true;
            }
            R.sobol_hash = ctx->d_sobol_hash;
        }
    }
    if (R.sampler != TCPT_SAMPLER_SOBOL || !ctx->opt.sobol_prefix) return TCPT_OK;
    // Both tables assume that the bits of the Morton index at and above log2_spp belong to the pixel alone.  The reference takes any
    // spp (main.rs only warns) with log2_spp = floor(log2(spp)) and ORs the sample index in (z_sobol_sampler.rs:200), so for a spp that
    // is not a power of two the samples >= 2^log2_spp spill into the pixel digits: no tables then, every digit is computed per call.
    if ((R.spp & (R.spp - 1u)) != 0u) return TCPT_OK;
    const size_t n_pix = (size_t)R.width * R.height;
    size_t dims = 3 + 8 * ((size_t)R.max_depth + 1);
    const size_t cap_dims = ((size_t)ctx->opt.sobol_prefix_mb << 20) / (n_pix * 4);
    if (dims > cap_dims) dims = cap_dims;
    if (dims == 0) return TCPT_OK;
    // rows behind the prefix rows for the per-pass table (k_sobol_pass).  Default 11 = the camera's 3 dimensions + the 8 of bounce 0, where
    // every path still is (measured on the 4K frame, 16 samples per pass: 0.115 ms per row to build; 0 / 3 / 11 / 16 / 40 rows give
    // 105.5 / 103.8 / 102.7 / 103.4 / 106.6 ms per step: deeper bounces hold too few vertices to pay for their rows)
    size_t pass_rows = ctx->opt.sobol_pass ? (size_t)(ctx->opt.sobol_pass_dims < 0 ? 0 : ctx->opt.sobol_pass_dims) : 0;
    if (pass_rows > dims) pass_rows = dims;
    if (pass_rows > 255) pass_rows = 255;
    const bool same = ctx->d_prefix && ctx->prefix_w == R.width && ctx->prefix_h == R.height && ctx->prefix_log2spp == R.log2_spp && ctx->pass_rows == pass_rows;
    if (!same || ctx->prefix_dims < dims) {
        const size_t need = n_pix * (dims + 2 * pass_rows);   // prefix rows, pass rows, cache rows of the incremental pass build
        if (need > ctx->prefix_cap) {
            if (ctx->d_prefix) { cudaStreamSynchronize(stream); cudaFree(ctx->d_prefix); ctx->d_prefix = nullptr; ctx->prefix_cap = 0; }
            if (cudaMalloc((void**)&ctx->d_prefix, need * 4) != cudaSuccess) { cudaGetLastError(); ctx->prefix_dims = 0; return TCPT_OK; }  // no table: full loop
            ctx->prefix_cap = need;
        }
        cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, stream);
        const size_t total = n_pix * dims;
        const int grid = (int)((total + 255) / 256 < (size_t)ctx->sm_count * 64 ? (total + 255) / 256 : (size_t)ctx->sm_count * 64);
        k_sobol_prefix<<<grid, 256, 0, stream>>>(ctx->d_prefix, R.width, R.height, R.log2_spp, R.n_base4_digits, (uint32_t)dims);
        cudaEventRecord(b, stream);
        CU(cudaEventSynchronize(b));
        float ms = 0.0f; cudaEventElapsedTime(&ms, a, b); ctx->prefix_build_ms = ms; ctx->stats.sobol_prefix_ms = ms;
        cudaEventDestroy(a); cudaEventDestroy(b);
        CU(cudaGetLastError());
        if (pass_rows) CU(cudaMemsetAsync(ctx->d_prefix + n_pix * (dims + pass_rows), 0, n_pix * pass_rows * 4, stream));   // cache words: invalid
        ctx->prefix_w = R.width; ctx->prefix_h = R.height; ctx->prefix_log2spp = R.log2_spp; ctx->prefix_dims = (uint32_t)dims; ctx->pass_rows = (uint32_t)pass_rows;
    }
    R.sobol_prefix = ctx->d_prefix; R.prefix_dims = ctx->prefix_dims; R.prefix_stride = (uint32_t)n_pix;
    ctx->stats.sobol_prefix_bytes = (uint64_t)n_pix * ctx->prefix_dims * 4;
    return TCPT_OK;
}

// Per-stage device timing without host round trips: an event pair is recorded around every launch on the launching stream
// and the pairs are read back once, after the frame's final synchronisation (option "stage_timing").
struct StageTimer {
    tcpt_ctx* ctx; bool on; int stage; size_t slot;
    StageTimer(tcpt_ctx* c, int stage_id, cudaStream_t s) : ctx(c), on(c->opt.stage_timing != 0), stage(stage_id), slot(0) {
        if (!on) return;
        slot = ctx->ev_used;
        while (ctx->ev_pool.size() < slot + 2) { cudaEvent_t e; cudaEventCreate(&e); ctx->ev_pool.push_back(e); }
        ctx->ev_used += 2;
        ctx->ev_stage.push_back(stage);
        cudaEventRecord(ctx->ev_pool[slot], s);
        stream = s;
    }
    ~StageTimer() { if (on) cudaEventRecord(ctx->ev_pool[slot + 1], stream); }
    cudaStream_t stream = nullptr;
};
enum { STAGE_GENERATE = 0, STAGE_CLOSEST = 1, STAGE_SHADE = 2, STAGE_SHADOW = 3, STAGE_FILM = 4 };

// ZSobol pass table: the rows behind the prefix rows, rebuilt on `stream` at the start of every pass for the pass's pixels and sample
// block (see DSampler::sample_index).  Worth it when a pass holds several samples per pixel (each entry costs about what it saves one
// sampler call); needs the prefix table, an even log2(spp) (no trailing binary digit) and sample digits that fit 16 bits.
void build_sobol_pass(tcpt_ctx* ctx, DRender& Rp, cudaStream_t stream) {
    Rp.pass_info = 0;
    if (!Rp.sobol_prefix || ctx->pass_rows == 0 || (Rp.log2_spp & 1u) || Rp.log2_spp > 16u || Rp.s_count < 4u) return;
    uint32_t v = 0;   // number of low sample-index bits that differ inside [s_begin, s_begin + s_count)
    while ((Rp.s_begin >> v) != ((Rp.s_begin + Rp.s_count - 1u) >> v)) ++v;
    const uint32_t iv = (v + 1u) >> 1;
    const size_t total = (size_t)Rp.n_pix * ctx->pass_rows;
    const int grid = (int)((total + 255) / 256 < (size_t)ctx->sm_count * 64 ? (total + 255) / 256 : (size_t)ctx->sm_count * 64);
    StageTimer t(ctx, STAGE_GENERATE, stream);
    // digits iv .. log2_spp / 2 - 1 of the sample index sit in the table: with one to four of them the rows are built incrementally
    const uint32_t half = Rp.log2_spp >> 1;
    if (ctx->opt.sobol_pass_cache && iv >= 1u && iv <= 7u && half >= iv + 1u && half - iv <= 4u)
        k_sobol_pass_cached<<<grid_for(ctx, Rp.n_pix, 256), 256, 0, stream>>>(ctx->d_prefix, Rp, ctx->pass_rows, iv, ctx->prefix_dims + ctx->pass_rows);
    else
        k_sobol_pass<<<grid, 256, 0, stream>>>(ctx->d_prefix, Rp, ctx->pass_rows, iv);
    ctx->stats.kernel_launches++;
    Rp.pass_info = ctx->pass_rows | (iv << 8);
}

void collect_stage_times(tcpt_ctx* ctx) {  // call after the stream has been synchronised
    double* acc[5] = {&ctx->stats.generate_ms, &ctx->stats.trace_closest_ms, &ctx->stats.shade_ms, &ctx->stats.trace_shadow_ms, &ctx->stats.film_ms};
    for (size_t i = 0; i < ctx->ev_stage.size(); ++i) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, ctx->ev_pool[2 * i], ctx->ev_pool[2 * i + 1]) == cudaSuccess) *acc[ctx->ev_stage[i]] += ms;
    }
    ctx->ev_used = 0;
    ctx->ev_stage.clear();
}

// developer option "debug_path_log": with a single path in flight, print its queue entries and state after every stage (stderr)
static void debug_dump(tcpt_ctx* ctx, const char* what, uint32_t stage, int cur, cudaStream_t stream) {
    const DState& st = ctx->st;
    cudaStreamSynchronize(stream);
    uint32_t cnt[4]; float4 o, d, h0, thr, con, misc, so, sd, sc_; uint2 h1;
    cudaMemcpy(cnt, st.counters, sizeof cnt, cudaMemcpyDeviceToHost);
    cudaMemcpy(&o, st.ext_o[cur], 16, cudaMemcpyDeviceToHost); cudaMemcpy(&d, st.ext_d[cur], 16, cudaMemcpyDeviceToHost);
    cudaMemcpy(&h0, st.hit0, 16, cudaMemcpyDeviceToHost); cudaMemcpy(&h1, st.hit1, 8, cudaMemcpyDeviceToHost);
    cudaMemcpy(&thr, st.thr, 16, cudaMemcpyDeviceToHost); cudaMemcpy(&con, st.con, 16, cudaMemcpyDeviceToHost); cudaMemcpy(&misc, st.misc, 16, cudaMemcpyDeviceToHost);
    cudaMemcpy(&so, st.sh_o, 16, cudaMemcpyDeviceToHost); cudaMemcpy(&sd, st.sh_d, 16, cudaMemcpyDeviceToHost); cudaMemcpy(&sc_, st.sh_c, 16, cudaMemcpyDeviceToHost);
    uint32_t dim, fl; std::memcpy(&dim, &misc.z, 4); std::memcpy(&fl, &misc.w, 4);
    std::fprintf(stderr, "[tcpt %s stage %u] q=%u/%u sh=%u ray o(%.9g %.9g %.9g) d(%.9g %.9g %.9g) tmax %.9g | hit t %.9g prim %d tri %d | thr %.9g %.9g %.9g %.9g con %.9g %.9g %.9g %.9g pdf_prev %.9g dim %u flags %u | shadow o(%.9g %.9g %.9g) d(%.9g %.9g %.9g) tmax %.9g c %.9g %.9g %.9g %.9g\n",
                 what, stage, cnt[0], cnt[1], cnt[2], o.x, o.y, o.z, d.x, d.y, d.z, o.w, h0.x, (int)h1.x, (int)h1.y, thr.x, thr.y, thr.z, thr.w, con.x, con.y, con.z, con.w, misc.x, dim, fl,
                 so.x, so.y, so.z, sd.x, sd.y, sd.z, so.w, sc_.x, sc_.y, sc_.z, sc_.w);
}

// one pass = generate + (max_depth + 1) x {closest, shade, shadow} (+ film when acc != nullptr; with the luminance moments when dev_mom != nullptr)
int run_pass(tcpt_ctx* ctx, const DRender& R, const DCamera& cam, const PathList& L, uint32_t n_slots, float* dev_acc, cudaStream_t stream, float2* dev_mom = nullptr) {
    const DScene& sc = ctx->dev.view;
    const DState& st = ctx->st;
    const bool count = ctx->opt.count_tests != 0;
    {
        StageTimer t(ctx, STAGE_GENERATE, stream);
        // a Z-Sobol pass over whole pixels: one thread per pixel (what the sampler derives from the pixel is fetched once); else one thread per path
        if (ctx->opt.generate_pixels && L.xy == nullptr && R.sampler == TCPT_SAMPLER_SOBOL && R.s_count >= 2u && (uint64_t)R.n_pix * R.s_count == n_slots)
            k_generate_pixels<<<grid_for(ctx, R.n_pix, 256), 256, 0, stream>>>(sc, R, cam, st, n_slots);
        else
            k_generate<<<grid_for(ctx, n_slots, 256), 256, 0, stream>>>(sc, R, cam, st, L, n_slots);
        ctx->stats.kernel_launches++;
    }
    const int g128 = grid_for(ctx, n_slots, 128);
    // the shading kernels' own block sizes (ShadeCfg<B>): as many blocks as the trace grid has threads for
    auto shade_grid = [&](int threads) { return (int)std::max<uint64_t>(1, std::min<uint64_t>(((uint64_t)n_slots + threads - 1) / threads, (uint64_t)ctx->sm_count * ctx->opt.blocks_per_sm * 128 / threads)); };
#define TCPT_SHADE_LAUNCH(...) k_shade<__VA_ARGS__><<<shade_grid(ShadeCfg<TCPT_FIRST_ARG(__VA_ARGS__)>::threads), ShadeCfg<TCPT_FIRST_ARG(__VA_ARGS__)>::threads, 0, stream>>>(sc, R, st, L, cur, sh, stage)
#define TCPT_FIRST_ARG(a, ...) a
    if (R.integrator >= TCPT_INTEGRATOR_ALBEDO) {  // AOV renderers: one camera ray per sample, no bounces
        if (count) k_trace_fused<true><<<g128, 128, 0, stream>>>(sc, R, st, 0, 3, (uint32_t)ctx->opt.refill_b0, (uint32_t)ctx->opt.chunk_b0);
        else k_trace_fused<false><<<g128, 128, 0, stream>>>(sc, R, st, 0, 3, (uint32_t)ctx->opt.refill_b0, (uint32_t)ctx->opt.chunk_b0);
        k_aov<<<g128, 128, 0, stream>>>(sc, R, st);
        ctx->stats.kernel_launches += 2; ctx->stats.trace_launches++; ctx->stats.shade_launches++;
    } else {
    // option "fused_launches": bit 0 = k_trace_fused (shadow rays of the previous bounce + this bounce's extension rays in one
    // launch), bit 1 = k_shade_all (all shading buckets in one launch); 0 = one launch per queue and per bucket
    const bool fuse_trace = (ctx->opt.fused_launches & 1) != 0;
    for (uint32_t stage = 0; stage <= R.max_depth; ++stage) {
        const int cur = (int)(stage & 1u);
        // the first bounces hold most of the vertices and run faster as one launch per bucket (17.6 vs 22.1 ms of shading per 33 M
        // paths); from bounce "fused_shade_from" on the queues are short and launch latency dominates
        const bool fuse_shade = (ctx->opt.fused_launches & 2) != 0 && stage >= (uint32_t)ctx->opt.fused_shade_from;
        // size of the shadow queue this bounce's shading appends to: ping-pong 2 / 3 with the fused trace (it resets the one it is
        // not reading), always 2 otherwise (k_trace_closest resets it)
        const int sh = fuse_trace ? 2 + cur : 2, sh_prev = 2 + (int)((stage + 1u) & 1u);
        {
            StageTimer t(ctx, STAGE_CLOSEST, stream);
            if (fuse_trace) {
                if (count) k_trace_fused<true><<<g128, 128, 0, stream>>>(sc, R, st, cur, sh_prev, (uint32_t)(stage == 0 ? ctx->opt.refill_b0 : ctx->opt.refill), (uint32_t)(stage == 0 ? ctx->opt.chunk_b0 : ctx->opt.chunk));
                else k_trace_fused<false><<<g128, 128, 0, stream>>>(sc, R, st, cur, sh_prev, (uint32_t)(stage == 0 ? ctx->opt.refill_b0 : ctx->opt.refill), (uint32_t)(stage == 0 ? ctx->opt.chunk_b0 : ctx->opt.chunk));
            } else {
                if (count) k_trace_closest<true><<<g128, 128, 0, stream>>>(sc, st.ext_o[cur], st.ext_d[cur], st.hit0, st.hit1, st, cur);
                else k_trace_closest<false><<<g128, 128, 0, stream>>>(sc, st.ext_o[cur], st.ext_d[cur], st.hit0, st.hit1, st, cur);
            }
            ctx->stats.kernel_launches++; ctx->stats.trace_launches++;
        }
        {
            StageTimer t(ctx, STAGE_SHADE, stream);
            if (fuse_shade) {
                k_shade_all<<<g128, 128, 0, stream>>>(sc, R, st, L, cur, sh, stage);
                ctx->stats.kernel_launches++; ctx->stats.shade_launches++;
            } else {
                if (stage == 0) {  // bounce 0 has its own instantiations (no previous-bounce half; the terminal bucket is empty)
                    TCPT_SHADE_LAUNCH(0, true);
                    TCPT_SHADE_LAUNCH(1, true);
                    TCPT_SHADE_LAUNCH(2, true);
                    TCPT_SHADE_LAUNCH(3, true);
                    TCPT_SHADE_LAUNCH(4, true);
                    TCPT_SHADE_LAUNCH(5, true);
                    TCPT_SHADE_LAUNCH(6, true);
                    TCPT_SHADE_LAUNCH(7, true);
                    TCPT_SHADE_LAUNCH(8, true);
                } else {
                    TCPT_SHADE_LAUNCH(0);
                    TCPT_SHADE_LAUNCH(1);
                    TCPT_SHADE_LAUNCH(2);
                    TCPT_SHADE_LAUNCH(3);
                    TCPT_SHADE_LAUNCH(4);
                    TCPT_SHADE_LAUNCH(5);
                    TCPT_SHADE_LAUNCH(6);
                    TCPT_SHADE_LAUNCH(7);
                    TCPT_SHADE_LAUNCH(8);
                }
                ctx->stats.kernel_launches += 9; ctx->stats.shade_launches += 9;
            }
        }
        if (ctx->opt.debug_path_log && n_slots == 1) debug_dump(ctx, "after shade", stage, cur ^ 1, stream);
        // k_shade of bounce max_depth ends every remaining path before it samples a light or a direction: nothing left to trace
        if (!fuse_trace && R.integrator != TCPT_INTEGRATOR_PT && stage < R.max_depth) {
            StageTimer t(ctx, STAGE_SHADOW, stream);
            if (count) k_trace_shadow<true><<<g128, 128, 0, stream>>>(sc, R, st);
            else k_trace_shadow<false><<<g128, 128, 0, stream>>>(sc, R, st);
            ctx->stats.kernel_launches++; ctx->stats.trace_launches++;
        }
    }
    }
    if (dev_acc) {
        StageTimer t(ctx, STAGE_FILM, stream);
        if (dev_mom) k_film_moments<<<grid_for(ctx, R.n_pix, 256), 256, 0, stream>>>(R, st.rgb, dev_acc, dev_mom);
        else k_film<<<grid_for(ctx, R.n_pix, 256), 256, 0, stream>>>(R, st.rgb, dev_acc);
        ctx->stats.kernel_launches++;
    }
    ctx->stats.passes++;
    CU(cudaGetLastError());
    return TCPT_OK;
}

int fetch_stats(tcpt_ctx* ctx) {
    unsigned long long h[8];
    CU(cudaMemcpy(h, ctx->d_stats, sizeof h, cudaMemcpyDeviceToHost));
    ctx->stats.closest_rays = h[0]; ctx->stats.shadow_rays = h[1]; ctx->stats.box_tests = h[2]; ctx->stats.tri_tests = h[3]; ctx->stats.paths = h[4];
    return TCPT_OK;
}

void reset_stats(tcpt_ctx* ctx) {
    cudaMemsetAsync(ctx->d_stats, 0, 8 * sizeof(unsigned long long), ctx->stream);
    ctx->stats = tcpt_stats{};
    ctx->stats.max_bvh_depth = ctx->dev.max_bvh_depth;
    ctx->ev_used = 0; ctx->ev_stage.clear();
}

// The pass loop of a job: `owned` pixels -- owned indices 0 .. owned - 1, or the entries of the device list `pix_list` (owned indices,
// ascending; see owned_pixel) -- times the sample window [s0, s1), cut into (pixel block x sample window) passes that fit the
// path-slot budget.  R comes from make_render + ensure_sobol_prefix.  dev_mom != nullptr: the film also adds the luminance moments.
int render_passes(tcpt_ctx* ctx, const DRender& R, const DCamera& cam, uint64_t owned, const uint32_t* pix_list, uint32_t s0, uint32_t s1,
                  uint32_t max_slots, float* dev_acc, float2* dev_mom, cudaStream_t stream) {
    if (pix_list && dev_acc && !dev_mom) return fail(ctx, TCPT_ERR_INVALID, "render: a pass over a pixel list films through k_film_moments");
    int rc = TCPT_OK;
    // Path-slot budget of one pass.  Every pass pays a fixed latency (about 35 launches whose deep-bounce queues are nearly
    // empty: 4 to 8 ms on the 4K frame), so passes are made as large as memory comfortably allows: up to 128 Mi slots
    // (304 B each: 40 GB of the 180 GB), never more than 45 % of the memory that is free.
    uint64_t budget = max_slots;
    if (budget == 0) {
        if (ctx->default_slots == 0) {  // asked once per context: cudaMemGetInfo was measured to stall a render by up to 80 ms
            size_t free_b = 0, total_b = 0;
            if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = (size_t)16 << 30; }
            const uint64_t avail = (uint64_t)free_b + (uint64_t)ctx->st_capacity * kBytesPerSlot;
            uint64_t b = (uint64_t)(0.45 * (double)avail) / kBytesPerSlot;
            if (b > (128ull << 20)) b = 128ull << 20;
            if (b < (1ull << 20)) b = 1ull << 20;
            ctx->default_slots = b;
        }
        budget = ctx->default_slots;
    }
    if (budget > 0xffffffffull) budget = 0xffffffffull;   // slots are indexed with 32 bits
    uint32_t np, sc_per_pass;
    for (;;) {
        np = (uint32_t)(owned < budget ? owned : budget);
        sc_per_pass = (uint32_t)(budget / np);
        if (sc_per_pass < 1) sc_per_pass = 1;
        if (sc_per_pass > s1 - s0) sc_per_pass = s1 - s0;
        rc = ensure_state(ctx, (uint32_t)((uint64_t)np * sc_per_pass));
        // the budget is a guess made once per context (other tenants, a Z-Sobol table that has grown since): shrink the pass instead of failing
        if (rc == TCPT_ERR_NOMEM && max_slots == 0 && budget > (1ull << 20)) { budget >>= 1; ctx->default_slots = budget; continue; }
        break;
    }
    if (rc) return rc;
    PathList none{nullptr, nullptr};
    for (uint64_t pb = 0; pb < owned; pb += np) {
        const uint32_t n_pix = (uint32_t)((owned - pb) < np ? (owned - pb) : np);
        for (uint32_t sb = s0; sb < s1; sb += sc_per_pass) {
            DRender Rp = R;
            Rp.n_pix = n_pix; Rp.pix_begin = (uint32_t)pb; Rp.pix_list = pix_list; Rp.s_begin = sb; Rp.s_count = (s1 - sb) < sc_per_pass ? (s1 - sb) : sc_per_pass;
            set_div_magics(Rp);
            build_sobol_pass(ctx, Rp, stream);
            rc = run_pass(ctx, Rp, cam, none, n_pix * Rp.s_count, dev_acc, stream, dev_mom);
            if (rc) return rc;
        }
    }
    return TCPT_OK;
}

int render_into(tcpt_ctx* ctx, const tcpt_render_params* p, float* dev_acc, cudaStream_t stream) {
    DRender R; DCamera cam;
    int rc = make_render(ctx, p, R, cam);
    if (rc) return rc;
    if (R.row_offset >= R.row_stride) return fail(ctx, TCPT_ERR_INVALID, "render: row_offset must be < row_stride");
    rc = ensure_sobol_prefix(ctx, R, stream);
    if (rc) return rc;
    const uint32_t s0 = (p->spp_begin == 0 && p->spp_end == 0) ? 0 : p->spp_begin;
    const uint32_t s1 = (p->spp_begin == 0 && p->spp_end == 0) ? p->spp : p->spp_end;
    if (s1 > p->spp || s0 > s1) return fail(ctx, TCPT_ERR_INVALID, "render: bad sample range");
    const uint32_t rows = R.row_offset < p->height ? (p->height - R.row_offset + R.row_stride - 1) / R.row_stride : 0;
    const uint64_t owned = (uint64_t)rows * p->width;
    if (owned == 0 || s0 == s1) return TCPT_OK;
    return render_passes(ctx, R, cam, owned, nullptr, s0, s1, p->max_slots, dev_acc, nullptr, stream);
}

void unpin_all(tcpt_ctx* ctx) {
    for (HostPin& h : ctx->pins) { if (h.ptr) cudaHostUnregister(h.ptr); h = HostPin(); }
}

// Device -> caller's host buffer.  With option "pin_host_buffers" the buffer is page-locked once (and stays so while the same
// pointer is passed again) so the copy is a direct DMA at PCIe rate instead of a staged pageable copy.
int copy_out(tcpt_ctx* ctx, int slot, void* host, const void* dev, size_t bytes) {
    if (ctx->opt.pin_host_buffers) {
        HostPin& h = ctx->pins[slot];
        if (h.ptr != host || h.bytes != bytes) {
            if (h.ptr) cudaHostUnregister(h.ptr);
            h = HostPin();
            if (cudaHostRegister(host, bytes, cudaHostRegisterDefault) == cudaSuccess) { h.ptr = host; h.bytes = bytes; }
            else cudaGetLastError();  // not registrable (e.g. already pinned by the caller): plain copy below
        }
    }
    CU(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TCPT_OK;
}

// the context's film buffers (tcpt_render and tcpt_render_adaptive), grown to n floats each
int ensure_film(tcpt_ctx* ctx, size_t n) {
    if (ctx->film_cap >= n) return TCPT_OK;
    if (ctx->film_acc) cudaFree(ctx->film_acc);
    if (ctx->film_srgb) cudaFree(ctx->film_srgb);
    ctx->film_acc = ctx->film_srgb = nullptr; ctx->film_cap = 0;
    CU(cudaMalloc((void**)&ctx->film_acc, n * sizeof(float)));
    CU(cudaMalloc((void**)&ctx->film_srgb, n * sizeof(float)));
    ctx->film_cap = n;
    return TCPT_OK;
}

// the adaptive entry points' per-pixel buffers, carved from one grow-only allocation
struct AdaptiveBuffers { float2* mom; uint32_t* counts; uint32_t* list[2]; uint32_t* tiles; uint32_t* n_active; };
size_t adaptive_bytes(size_t n_pix) { return n_pix * (sizeof(float2) + 3 * sizeof(uint32_t)) + ((n_pix + TCPT_SELECT_TILE - 1) / TCPT_SELECT_TILE + 1) * sizeof(uint32_t); }
int ensure_adaptive(tcpt_ctx* ctx, size_t n_pix, AdaptiveBuffers& b) {
    if (ctx->adapt_cap < n_pix) {
        if (ctx->adapt_buf) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->adapt_buf); }
        ctx->adapt_buf = nullptr; ctx->adapt_cap = 0;
        CU(cudaMalloc(&ctx->adapt_buf, adaptive_bytes(n_pix)));
        ctx->adapt_cap = n_pix;
    }
    const size_t cap = ctx->adapt_cap;
    b.mom = (float2*)ctx->adapt_buf;
    b.counts = (uint32_t*)(b.mom + cap);
    b.list[0] = b.counts + cap; b.list[1] = b.list[0] + cap;
    b.n_active = b.list[1] + cap;
    b.tiles = b.n_active + 1;
    return TCPT_OK;
}

// The checks every adaptive entry point makes on `ap` and the job before it looks at the device (include/tcpt.h).  The row shard is the
// caller's to check: each entry point has its own rule.
int check_adaptive(tcpt_ctx* ctx, const tcpt_render_params* p, const tcpt_adaptive_params* ap, const char* who) {
    auto bad = [&](const char* why) { return fail(ctx, TCPT_ERR_INVALID, std::string(who) + ": " + why); };
    if (!std::isfinite(ap->threshold) || ap->threshold < 0.0f) return bad("threshold must be finite and >= 0");
    if (ap->min_spp < 2 || ap->min_spp > p->spp) return bad("min_spp must lie in [2, spp]");
    if (ap->step == 0) return bad("step must be positive");
    if (p->integrator < TCPT_INTEGRATOR_PT || p->integrator > TCPT_INTEGRATOR_MIS) return bad("integrators pt, nee and mis only");
    if (p->spp_begin || p->spp_end) return bad("spp_begin / spp_end must be 0 (all samples)");
    if ((uint64_t)p->width * p->height * 3 > 0xffffffffull) return bad("frame too large");
    return TCPT_OK;
}

// The adaptive rounds of one job on `s`: the whole frame, or the rows row_offset + i * row_stride.  R / cam come from make_render of `p`,
// which the caller runs before it records anything on the device; the caller also checks the row shard (row_offset < row_stride).  Round 0 takes
// every owned pixel (no list); after each round that ends below spp, k_adaptive_count / _scan / _scatter write the counts of the pixels that
// stop and compact the others, in ascending owned order, into the next list.  One 4-byte device -> host copy per round (the active count)
// sizes the next round.  Each owned pixel's sum is ADDED into dev_acc and its count WRITTEN into dev_counts (both frame-indexed, W*H*3 f32
// and W*H u32); no other pixel of either buffer is touched.
int render_adaptive_into(tcpt_ctx* ctx, const tcpt_render_params* p, DRender R, const DCamera& cam, const tcpt_adaptive_params* ap, float* dev_acc,
                         uint32_t* dev_counts, cudaStream_t s) {
    int rc;
    const uint32_t n_pix = p->width * p->height, N = p->spp;
    const uint32_t rows = R.row_offset < p->height ? (p->height - R.row_offset + R.row_stride - 1) / R.row_stride : 0;
    const uint32_t owned = rows * p->width;
    AdaptiveBuffers B;
    if ((rc = ensure_adaptive(ctx, n_pix, B)) != TCPT_OK) return rc;
    if (owned == 0) return TCPT_OK;
    if ((rc = ensure_sobol_prefix(ctx, R, s)) != TCPT_OK) return rc;
    const RowMap rm{R.width, R.row_offset, R.row_stride, div_magic_of(R.width)};
    CU(cudaMemsetAsync(B.mom, 0, (size_t)n_pix * sizeof(float2), s));
    k_fill_owned_u32<<<grid_for(ctx, owned, 256), 256, 0, s>>>(dev_counts, owned, rm, N);   // a pixel that never stops has count N
    ctx->stats.kernel_launches++;
    uint32_t k = 0, active = owned, cur = 0;
    const uint32_t* list = nullptr;   // round 0: every owned pixel, in order
    while (active > 0) {
        const uint64_t want = k == 0 ? ap->min_spp : (uint64_t)k + ap->step;
        const uint32_t k_next = want < N ? (uint32_t)want : N;
        if ((rc = render_passes(ctx, R, cam, active, list, k, k_next, p->max_slots, dev_acc, B.mom, s)) != TCPT_OK) return rc;
        k = k_next;
        if (k >= N) break;
        const uint32_t n_tiles = (active + TCPT_SELECT_TILE - 1) / TCPT_SELECT_TILE;
        k_adaptive_count<<<n_tiles, TCPT_SELECT_THREADS, 0, s>>>(list, active, B.mom, k, ap->threshold, rm, dev_counts, B.tiles);
        k_adaptive_scan<<<1, 1024, 0, s>>>(B.tiles, n_tiles, B.n_active);
        k_adaptive_scatter<<<n_tiles, TCPT_SELECT_THREADS, 0, s>>>(list, active, B.mom, k, ap->threshold, rm, B.tiles, B.list[cur]);
        ctx->stats.kernel_launches += 3;
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&active, B.n_active, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        list = B.list[cur]; cur ^= 1u;
    }
    return TCPT_OK;
}

// One adaptive frame on the context's stream: `mine` (the whole job, or this rank's tile shard of it) through render_adaptive_into into the
// context's film and count buffers.  collective = false: the frame is this context's alone (any communicator it has is not used) and it
// finalizes and copies out.  collective = true (tcpt_render_adaptive_sharded): with a communicator of more than one rank, ONE grouped
// collective then sums both buffers onto rank 0 (exact: every pixel is owned by one rank, the others hold +0 and 0); rank 0 finalizes and
// copies out, the other ranks write no host buffer.
int adaptive_frame(tcpt_ctx* ctx, const tcpt_render_params* mine, const tcpt_adaptive_params* ap, bool collective, float* out_acc, float* out_srgb,
                   uint32_t* out_spp) {
    const uint32_t n_pix = mine->width * mine->height;
    const size_t n = (size_t)n_pix * 3;
    const bool reduce = collective && ctx->comm_size > 1, root = !collective || ctx->comm_rank == 0;
    cudaStream_t s = ctx->stream;
    DRender R; DCamera cam;
    int rc = make_render(ctx, mine, R, cam);
    if (rc) return rc;
    AdaptiveBuffers B;
    if ((rc = ensure_film(ctx, n)) != TCPT_OK || (rc = ensure_adaptive(ctx, n_pix, B)) != TCPT_OK) return rc;
    reset_stats(ctx);
    CU(cudaEventRecord(ctx->ev0, s));
    CU(cudaMemsetAsync(ctx->film_acc, 0, n * sizeof(float), s));
    if (reduce) CU(cudaMemsetAsync(B.counts, 0, (size_t)n_pix * sizeof(uint32_t), s));   // the pixels of the other ranks
    if ((rc = render_adaptive_into(ctx, mine, R, cam, ap, ctx->film_acc, B.counts, s)) != TCPT_OK) return rc;
    if (reduce) {
        if (!ctx->ev_r0) { cudaEventCreate(&ctx->ev_r0); cudaEventCreate(&ctx->ev_r1); }
        CU(cudaEventRecord(ctx->ev_r0, s));
        g_nccl.GroupStart();
        const ncclResult_t ra = g_nccl.Reduce(ctx->film_acc, ctx->film_acc, n, ncclFloat32, ncclSum, 0, ctx->comm, s);
        const ncclResult_t rb = g_nccl.Reduce(B.counts, B.counts, n_pix, ncclUint32, ncclSum, 0, ctx->comm, s);
        const ncclResult_t re = g_nccl.GroupEnd();
        const ncclResult_t r = ra != ncclSuccess ? ra : rb != ncclSuccess ? rb : re;
        if (r != ncclSuccess) return fail(ctx, TCPT_ERR_CUDA, std::string("ncclReduce: ") + g_nccl.GetErrorString(r));
        CU(cudaEventRecord(ctx->ev_r1, s));
    }
    if (root && out_srgb) {
        k_finalize_counts<<<grid_for(ctx, n, 256), 256, 0, s>>>(ctx->film_acc, B.counts, ctx->film_srgb, (uint32_t)n);
        ctx->stats.kernel_launches++;
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(ctx->ev1, s));
    CU(cudaEventSynchronize(ctx->ev1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->stats.render_ms = ms;
    if (reduce) { float rms = 0; if (cudaEventElapsedTime(&rms, ctx->ev_r0, ctx->ev_r1) == cudaSuccess) ctx->stats.reduce_ms = rms; }
    collect_stage_times(ctx);
    if ((rc = fetch_stats(ctx)) != TCPT_OK || !root) return rc;
    if (out_acc && (rc = copy_out(ctx, 0, out_acc, ctx->film_acc, n * sizeof(float))) != TCPT_OK) return rc;
    if (out_srgb && (rc = copy_out(ctx, 1, out_srgb, ctx->film_srgb, n * sizeof(float))) != TCPT_OK) return rc;
    if (out_spp && (rc = copy_out(ctx, 2, out_spp, B.counts, (size_t)n_pix * sizeof(uint32_t))) != TCPT_OK) return rc;
    return TCPT_OK;
}

}  // namespace

extern "C" {

int tcpt_create(int device_id, tcpt_ctx** out) {
    if (!out) return TCPT_ERR_INVALID;
    *out = nullptr;
    tcpt_ctx* ctx = new tcpt_ctx();
    ctx->device = device_id;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    auto bail = [&](const std::string& m) { ctx->error = m; *out = ctx; return TCPT_ERR_CUDA; };  // ctx is returned so the message can be read; destroy it
    if (e != cudaSuccess || n <= 0) return bail(std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device_id < 0 || device_id >= n) return bail("device index out of range");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return bail(cudaGetErrorString(e));
    if (prop.major != 10) return bail("libtcpt is built for sm_100a only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    if ((e = cudaSetDevice(device_id)) != cudaSuccess) return bail(cudaGetErrorString(e));
    ctx->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(cudaGetErrorString(e));
    if ((e = cudaMalloc((void**)&ctx->d_stats, 8 * sizeof(unsigned long long))) != cudaSuccess) return bail(cudaGetErrorString(e));
    if ((e = cudaMalloc((void**)&ctx->d_counters, 32 * sizeof(uint32_t))) != cudaSuccess) return bail(cudaGetErrorString(e));
    cudaMemset(ctx->d_stats, 0, 8 * sizeof(unsigned long long));
    cudaMemset(ctx->d_counters, 0, 32 * sizeof(uint32_t));
    cudaEventCreate(&ctx->ev0); cudaEventCreate(&ctx->ev1);
    srgb_xyz_to_rgb(ctx->xyz_to_rgb);
    *out = ctx;
    return TCPT_OK;
}

void tcpt_destroy(tcpt_ctx* ctx) {
    if (!ctx) return;
    if (ctx->stream) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
    if (ctx->comm && g_nccl.CommDestroy) { g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    if (ctx->ev_r0) cudaEventDestroy(ctx->ev_r0);
    if (ctx->ev_r1) cudaEventDestroy(ctx->ev_r1);
    free_scene(ctx->dev);
    for (void* p : ctx->st_allocs) cudaFree(p);
    unpin_all(ctx);
    if (ctx->film_acc) cudaFree(ctx->film_acc);
    if (ctx->film_srgb) cudaFree(ctx->film_srgb);
    if (ctx->adapt_buf) cudaFree(ctx->adapt_buf);
    if (ctx->d_cmf) cudaFree(ctx->d_cmf);
    if (ctx->d_sobol_bytes) cudaFree(ctx->d_sobol_bytes);
    if (ctx->d_presets) cudaFree(ctx->d_presets);
    if (ctx->d_prefix) cudaFree(ctx->d_prefix);
    if (ctx->d_sobol_hash) cudaFree(ctx->d_sobol_hash);
    if (ctx->trace_scratch) cudaFree(ctx->trace_scratch);
    if (ctx->d_rgb2spec) cudaFree(ctx->d_rgb2spec);
    if (ctx->d_stats) cudaFree(ctx->d_stats);
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* tcpt_last_error(const tcpt_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int tcpt_set_option(tcpt_ctx* ctx, const char* name, int value) {
    if (!ctx || !name) return TCPT_ERR_INVALID;
    const std::string n(name);
    if (n == "count_tests") ctx->opt.count_tests = value;
    else if (n == "stage_timing") ctx->opt.stage_timing = value;
    else if (n == "debug_path_log") ctx->opt.debug_path_log = value;
    else if (n == "sobol_prefix") ctx->opt.sobol_prefix = value;
    else if (n == "sobol_hash") ctx->opt.sobol_hash = value;
    else if (n == "illum_half") ctx->opt.illum_half = value;
    else if (n == "generate_pixels") ctx->opt.generate_pixels = value;
    else if (n == "sobol_pass_cache") ctx->opt.sobol_pass_cache = value;
    else if (n == "refill_b0") ctx->opt.refill_b0 = value < 1 ? 1 : (value > 32 ? 32 : value);
    else if (n == "refill") ctx->opt.refill = value < 1 ? 1 : (value > 32 ? 32 : value);
    else if (n == "chunk_b0") ctx->opt.chunk_b0 = value < 32 ? 32 : value;
    else if (n == "chunk") ctx->opt.chunk = value < 32 ? 32 : value;
    else if (n == "fused_launches") ctx->opt.fused_launches = value;
    else if (n == "fused_shade_from") ctx->opt.fused_shade_from = value;
    else if (n == "light_shortcut") ctx->opt.light_shortcut = value;   // takes effect at the next scene upload
    else if (n == "soup_leaf") ctx->opt.soup_leaf = value;               // triangles per leaf of tcpt_scene_build_soup
    else if (n == "env_nee_table") ctx->opt.env_nee_table = value;       // takes effect at the next scene upload
    else if (n == "sobol_prefix_mb") ctx->opt.sobol_prefix_mb = value;
    else if (n == "sobol_pass") ctx->opt.sobol_pass = value;
    else if (n == "sobol_pass_dims") ctx->opt.sobol_pass_dims = value;
    else if (n == "blocks_per_sm") ctx->opt.blocks_per_sm = value > 0 ? value : 8;
    else if (n == "binned_builder") ctx->host.use_binned_builder = value != 0;
    else if (n == "pin_host_buffers") { ctx->opt.pin_host_buffers = value != 0; if (!value) unpin_all(ctx); }
    else return fail(ctx, TCPT_ERR_INVALID, "unknown option " + n);
    return TCPT_OK;
}

int tcpt_set_tables(tcpt_ctx* ctx, const void* std_tables, size_t std_len, const float* rgb2spec, size_t rgb2spec_floats) {
    if (!ctx) return TCPT_ERR_INVALID;
    const size_t base_len = 8 + 104 * 4 + 4 * 470 * 4;
    const bool v1 = std_tables && std_len == base_len && std::memcmp(std_tables, "TCPTSTD1", 8) == 0;
    const bool v2 = std_tables && std_len >= base_len + 4 && std::memcmp(std_tables, "TCPTSTD2", 8) == 0;
    if (!v1 && !v2) return fail(ctx, TCPT_ERR_INVALID, "set_tables: bad std_tables blob");
    if (!rgb2spec || rgb2spec_floats != 64 + (size_t)3 * 64 * 64 * 64 * 3) return fail(ctx, TCPT_ERR_INVALID, "set_tables: bad rgb2spec table size");
    HostTables& T = ctx->host.tables;
    const uint8_t* p = (const uint8_t*)std_tables + 8;
    std::memcpy(T.sobol, p, 104 * 4); p += 104 * 4;
    const float* f = (const float*)p;
    T.cie_x.assign(f, f + 470); T.cie_y.assign(f + 470, f + 940); T.cie_z.assign(f + 940, f + 1410); T.d65.assign(f + 1410, f + 1880);
    T.rgb2spec.assign(rgb2spec, rgb2spec + rgb2spec_floats);
    T.presets.clear();
    if (v2) {
        uint32_t n_presets; std::memcpy(&n_presets, (const uint8_t*)std_tables + base_len, 4);
        if (std_len != base_len + 4 + (size_t)n_presets * 470 * 4) return fail(ctx, TCPT_ERR_INVALID, "set_tables: bad preset table size");
        const float* pf = (const float*)((const uint8_t*)std_tables + base_len + 4);
        T.presets.assign(pf, pf + (size_t)n_presets * 470);
    }
    T.set = true;
    // Sobol matrix 0 must be the bit-reversal identity (the device uses __brev for dimension 0) and its rows >= 32 zero
    for (int i = 0; i < 52; ++i) if (T.sobol[i] != (i < 32 ? (0x80000000u >> i) : 0u)) return fail(ctx, TCPT_ERR_INVALID, "set_tables: Sobol matrix 0 is not the identity");
    // host tables are usable from here on (material resolution, tcpt_rgb_to_coeffs); the device copies need the GPU
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyToSymbol(c_sobol_dim1, T.sobol + 52, 52 * 4));
    {
        std::vector<uint32_t> tab(7 * 256, 0u);
        for (int pos = 0; pos < 7; ++pos)
            for (int b = 0; b < 256; ++b) {
                uint32_t v = 0;
                for (int i = 0; i < 8; ++i) if ((b >> i) & 1) { const int row = 8 * pos + i; if (row < 52) v ^= T.sobol[52 + row]; }
                tab[pos * 256 + b] = v;
            }
        if (!ctx->d_sobol_bytes) CU(cudaMalloc((void**)&ctx->d_sobol_bytes, tab.size() * 4));
        CU(cudaMemcpy(ctx->d_sobol_bytes, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
        const uint32_t* p = ctx->d_sobol_bytes;
        CU(cudaMemcpyToSymbol(c_sobol_dim1_bytes, &p, sizeof p));
    }
    std::vector<float> cmf(470 * 4);
    for (int i = 0; i < 470; ++i) { cmf[4 * i] = T.cie_x[i]; cmf[4 * i + 1] = T.cie_y[i]; cmf[4 * i + 2] = T.cie_z[i]; cmf[4 * i + 3] = T.d65[i]; }
    if (!ctx->d_cmf) CU(cudaMalloc((void**)&ctx->d_cmf, 470 * sizeof(float4)));
    CU(cudaMemcpy(ctx->d_cmf, cmf.data(), 470 * sizeof(float4), cudaMemcpyHostToDevice));
    if (ctx->d_presets) { cudaFree(ctx->d_presets); ctx->d_presets = nullptr; }
    CU(cudaMalloc((void**)&ctx->d_presets, (T.presets.size() + 1) * sizeof(float)));
    if (!T.presets.empty()) CU(cudaMemcpy(ctx->d_presets, T.presets.data(), T.presets.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (!ctx->d_rgb2spec) CU(cudaMalloc((void**)&ctx->d_rgb2spec, rgb2spec_floats * sizeof(float)));
    CU(cudaMemcpy(ctx->d_rgb2spec, rgb2spec, rgb2spec_floats * sizeof(float), cudaMemcpyHostToDevice));
    {   // srgb_to_linear(0.5f) and its z-node interval as the device evaluates them (DScene::half_lin / half_zi)
        uint32_t* d_out = ctx->d_counters + 28;   // two scratch words of the counter block
        k_illum_half<<<1, 32, 0, ctx->stream>>>(ctx->d_rgb2spec, d_out);
        uint32_t h[2] = {0u, 0u};
        CU(cudaMemcpyAsync(h, d_out, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        std::memcpy(&ctx->half_lin, &h[0], 4); ctx->half_zi = (int32_t)h[1];
        // a scene uploaded before the tables were replaced keeps reading the table allocations in place: its constants follow
        if (ctx->dev.valid) { ctx->dev.view.half_lin = ctx->half_lin; ctx->dev.view.half_zi = ctx->opt.illum_half ? ctx->half_zi : -1; }
    }
    return TCPT_OK;
}

int tcpt_scene_clear(tcpt_ctx* ctx) { if (!ctx) return TCPT_ERR_INVALID; ctx->host.clear(); return TCPT_OK; }
int tcpt_scene_add_mesh(tcpt_ctx* ctx, const float* positions, const float* normals, const float* uvs, int n_vertices, const uint32_t* indices, int n_triangles) {
    if (!ctx) return TCPT_ERR_INVALID;
    int r = ctx->host.add_mesh(positions, normals, uvs, n_vertices, indices, n_triangles);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}
// ---- asset ingestion (csrc/host_obj.h)
struct tcpt_obj { tcpt::ObjData d; };
int tcpt_obj_load(const char* path, tcpt_obj** out, char* err, size_t err_len) {
    if (!path || !out) return TCPT_ERR_INVALID;
    *out = nullptr;
    tcpt_obj* o = new tcpt_obj();
    std::string e;
    if (!tcpt::load_obj_file(path, o->d, e)) {
        if (err && err_len) { std::strncpy(err, e.c_str(), err_len - 1); err[err_len - 1] = 0; }
        delete o;
        return TCPT_ERR_INVALID;
    }
    *out = o;
    return TCPT_OK;
}
int tcpt_obj_counts(const tcpt_obj* o, uint32_t counts[5]) {
    if (!o || !counts) return TCPT_ERR_INVALID;
    counts[0] = (uint32_t)(o->d.positions.size() / 3); counts[1] = (uint32_t)(o->d.normals.size() / 3); counts[2] = (uint32_t)(o->d.texcoords.size() / 2);
    counts[3] = (uint32_t)(o->d.indices.size() / 3); counts[4] = o->d.n_models;
    return TCPT_OK;
}
int tcpt_obj_copy(const tcpt_obj* o, float* positions, float* normals, float* texcoords, uint32_t* indices, uint32_t* tangent_tri) {
    if (!o) return TCPT_ERR_INVALID;
    const tcpt::ObjData& d = o->d;
    if (positions) std::memcpy(positions, d.positions.data(), d.positions.size() * sizeof(float));
    if (normals) std::memcpy(normals, d.normals.data(), d.normals.size() * sizeof(float));
    if (texcoords) std::memcpy(texcoords, d.texcoords.data(), d.texcoords.size() * sizeof(float));
    if (indices) std::memcpy(indices, d.indices.data(), d.indices.size() * sizeof(uint32_t));
    if (tangent_tri) for (size_t t = 0; t < d.indices.size() / 3; ++t) tangent_tri[t] = d.tangent_tri.empty() ? (uint32_t)t : d.tangent_tri[t];
    return TCPT_OK;
}
void tcpt_obj_free(tcpt_obj* o) { delete o; }
int tcpt_scene_load_obj(tcpt_ctx* ctx, const char* path) {
    if (!ctx || !path) return TCPT_ERR_INVALID;
    tcpt::ObjData d;
    std::string e;
    if (!tcpt::load_obj_file(path, d, e)) return fail(ctx, TCPT_ERR_INVALID, "load_obj: " + e);
    const size_t nv = d.positions.size() / 3;
    if (d.normals.size() != d.positions.size()) return fail(ctx, TCPT_ERR_INVALID, "load_obj: every face vertex must carry a vn normal (the reference panics without them)");
    if (!d.texcoords.empty() && d.texcoords.size() / 2 != nv) return fail(ctx, TCPT_ERR_INVALID, "load_obj: texcoords on only some of the vertices (the reference would misindex them)");
    const int g = ctx->host.add_mesh(d.positions.data(), d.normals.data(), d.texcoords.empty() ? nullptr : d.texcoords.data(), (int)nv, d.indices.data(), (int)(d.indices.size() / 3));
    if (g < 0) { ctx->error = ctx->host.error; return g; }
    if (!d.tangent_tri.empty()) {
        const int rc = ctx->host.set_tangent_source(g, d.tangent_tri.data(), (int)d.tangent_tri.size());
        if (rc < 0) { ctx->error = ctx->host.error; return rc; }
    }
    return g;
}
int tcpt_image_convert(const void* src, uint32_t width, uint32_t height, uint32_t channels, int sample_type, int dst_kind, void* dst) {
    return tcpt::image_convert(src, width, height, channels, sample_type, dst_kind, dst) ? TCPT_OK : TCPT_ERR_INVALID;
}
int tcpt_scene_set_tangent_source(tcpt_ctx* ctx, int geometry, const uint32_t* tri, int n_triangles) {
    if (!ctx) return TCPT_ERR_INVALID;
    const int rc = ctx->host.set_tangent_source(geometry, tri, n_triangles);
    if (rc < 0) ctx->error = ctx->host.error;
    return rc;
}
int tcpt_scene_add_texture(tcpt_ctx* ctx, const uint8_t* data, uint32_t width, uint32_t height, uint32_t channels) {
    if (!ctx) return TCPT_ERR_INVALID;
    int r = ctx->host.add_texture(data, width, height, channels);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}
int tcpt_scene_add_material(tcpt_ctx* ctx, const tcpt_material_desc* desc) {
    if (!ctx || !desc) return TCPT_ERR_INVALID;
    int r = ctx->host.add_material(*desc);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}
int tcpt_scene_add_primitive(tcpt_ctx* ctx, int geometry, int material, const float local_to_world[16]) {
    if (!ctx || !local_to_world) return TCPT_ERR_INVALID;
    int r = ctx->host.add_primitive(geometry, material, local_to_world);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}
int tcpt_scene_add_env_light(tcpt_ctx* ctx, float intensity, const float* rgb, uint32_t width, uint32_t height, const float local_to_world[16]) {
    if (!ctx || !local_to_world) return TCPT_ERR_INVALID;
    int r = ctx->host.add_env_light(intensity, rgb, width, height, local_to_world);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}

int tcpt_scene_add_single_triangle(tcpt_ctx* ctx, const float positions[9], const float normals[9], const float uvs[6]) {
    if (!ctx) return TCPT_ERR_INVALID;
    int r = ctx->host.add_single_triangle(positions, normals, uvs);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}

int tcpt_scene_add_delta_light(tcpt_ctx* ctx, int kind, float intensity, const tcpt_spectrum_param* spectrum, float angle_inner, float angle_outer, const float local_to_world[16]) {
    if (!ctx || !spectrum || !local_to_world) return TCPT_ERR_INVALID;
    int r = ctx->host.add_delta_light(kind, intensity, *spectrum, angle_inner, angle_outer, local_to_world);
    if (r < 0) ctx->error = ctx->host.error;
    return r;
}

// A scene with ONE light whose power phi(lambda).average() is finite and strictly positive for every wavelength set: the light
// sampler then returns that light with probability w / w = 1 whatever the wavelengths (light_sampler.rs:26-44, 190-220), so the
// device skips evaluating phi at every vertex (DScene::one_light_always_on).  Checked on the 1 nm grid of the dense tables.
static bool spectrum_strictly_positive(const tcpt_flat_spectrum& sp, const HostTables& T) {
    for (int i = 0; i < 470; ++i) {
        const float lambda = 360.0f + (float)i;
        float v;
        if (sp.kind == 0) v = sp.c[0];
        else if (sp.kind == 3) v = T.d65[i];
        else if (sp.kind == 5) { if ((size_t)sp.texture * 470 + i >= T.presets.size()) return false; v = T.presets[(size_t)sp.texture * 470 + i]; }
        else if (sp.kind == 1 || sp.kind == 2) {
            const float t = (lambda - 360.0f) / (830.0f - 360.0f);
            const float sg = 1.0f / (1.0f + std::exp(-(t * t * sp.c[0] + t * sp.c[1] + sp.c[2])));
            v = sp.kind == 1 ? sg : sp.scale * sg * T.d65[i];
        } else return false;  // textures: not decided here
        if (!(v > 1e-20f) || !(v < 1e20f)) return false;
    }
    return true;
}
static bool one_light_always_on(const tcpt_flat_scene* s, const HostTables& T) {
    if (s->n_lights != 1) return false;
    const tcpt_flat_primitive& P = s->primitives[s->light_list[0]];
    auto ok = [](float x) { return x > 1e-20f && x < 1e20f; };
    if (P.kind == 1) {
        const tcpt_flat_material& m = s->materials[P.material];
        return !m.intensity.is_texture && ok(m.intensity.value) && ok(P.area_sum) && spectrum_strictly_positive(m.color, T);
    }
    if (P.kind == 2) { const tcpt_flat_env& e = s->envs[P.env]; return ok(e.intensity) && spectrum_strictly_positive(e.integrated, T); }
    if (P.kind == 3) return ok(P.light_intensity) && spectrum_strictly_positive(P.light_spectrum, T);
    if (P.kind == 5) return ok(P.light_intensity) && ok(P.dir_area) && spectrum_strictly_positive(P.light_spectrum, T);
    return false;  // spot lights: the cone factor can vanish
}

// Every cross-reference of a flattened scene, checked before anything is uploaded: this is the ABI a foreign flatten.rs calls, and an
// index out of range would otherwise surface as a device fault instead of TCPT_ERR_INVALID.
static bool validate_flat(const tcpt_flat_scene* s, std::string& why) {
    auto bad = [&](const std::string& w) { why = "upload: " + w; return false; };
    if (s->n_bvh_nodes == 0 || !s->bvh_nodes || s->tlas_node_count == 0 || s->tlas_node_count > s->n_bvh_nodes) return bad("no BVH nodes / bad tlas_node_count");
    if (s->n_primitives == 0 || !s->primitives) return bad("no primitives");
    if ((s->n_tlas_items && !s->tlas_items) || (s->n_tri_slots && !s->tri_verts) || (s->n_geometries && !s->geometries) || (s->n_materials && !s->materials) ||
        (s->n_textures && !s->textures) || (s->n_lights && !s->light_list) || (s->n_envs && !s->envs)) return bad("a non-empty table has a null pointer");
    for (uint32_t i = 0; i < s->n_tlas_items; ++i) {
        const int32_t prim = s->tlas_items[2 * (size_t)i];
        if (prim < 0 || (uint32_t)prim >= s->n_primitives) return bad("tlas_items names a primitive out of range");
        if (s->primitives[prim].geometry < 0) return bad("tlas_items names a primitive without geometry");
    }
    for (uint32_t i = 0; i < s->n_geometries; ++i) {
        const tcpt_flat_geometry& g = s->geometries[i];
        if (!g.single && g.node_base >= s->n_bvh_nodes) return bad("geometry node_base out of range");
        if ((uint64_t)g.slot_base + g.tri_count > s->n_tri_slots && s->n_tri_slots != 0) return bad("geometry triangle slots out of range");
        if (s->n_triangles != 0 && (uint64_t)g.index_base + g.tri_count > s->n_triangles) return bad("geometry index range out of range");
        if (s->n_vertices != 0 && g.vertex_base >= s->n_vertices) return bad("geometry vertex_base out of range");
    }
    for (uint32_t i = 0; i < s->n_materials; ++i) {
        const tcpt_flat_material& m = s->materials[i];
        auto tex_ok = [&](int32_t t) { return t < 0 || (uint32_t)t < s->n_textures; };
        if (m.type < TCPT_MAT_LAMBERT || m.type > TCPT_MAT_GLASS) return bad("unknown material type");
        if ((m.color.kind == 4 && (m.color.texture < 0 || !tex_ok(m.color.texture))) || (m.coat_tint.kind == 4 && (m.coat_tint.texture < 0 || !tex_ok(m.coat_tint.texture))) || !tex_ok(m.normal_texture))
            return bad("material texture index out of range");
        const tcpt_flat_float* fl[] = {&m.intensity, &m.roughness, &m.metallic, &m.ior, &m.coat_ior, &m.coat_roughness, &m.coat_thickness};
        for (const tcpt_flat_float* f : fl) if (f->is_texture && (f->texture < 0 || (uint32_t)f->texture >= s->n_textures)) return bad("material float texture index out of range");
    }
    for (uint32_t i = 0; i < s->n_textures; ++i) {
        const tcpt_flat_texture& t = s->textures[i];
        if (t.channels != 1 && t.channels != 3) return bad("texture channels must be 1 or 3");
        if (t.width == 0 || t.height == 0 || t.offset + (uint64_t)t.width * t.height * t.channels > s->n_texture_bytes) return bad("texture outside texture_bytes");
    }
    for (uint32_t i = 0; i < s->n_primitives; ++i) {
        const tcpt_flat_primitive& P = s->primitives[i];
        if (P.kind < 0 || P.kind > 5) return bad("unknown primitive kind");
        if (P.kind <= 1) {
            if (P.geometry < 0 || (uint32_t)P.geometry >= s->n_geometries) return bad("primitive geometry out of range");
            if (P.material < 0 || (uint32_t)P.material >= s->n_materials) return bad("primitive material out of range");
            if (P.kind == 1 && (uint64_t)P.area_base + s->geometries[P.geometry].tri_count > s->n_area) return bad("emissive primitive area table out of range");
        }
        if (P.kind == 2 && (P.env < 0 || (uint32_t)P.env >= s->n_envs)) return bad("environment primitive env index out of range");
        if (P.light_index >= (int32_t)s->n_lights) return bad("primitive light_index out of range");
    }
    for (uint32_t i = 0; i < s->n_lights; ++i) {
        const int32_t prim = s->light_list[i];
        if (prim < 0 || (uint32_t)prim >= s->n_primitives || s->primitives[prim].kind == 0) return bad("light_list names a primitive that is not a light");
    }
    for (uint32_t i = 0; i < s->n_envs; ++i) {
        const tcpt_flat_env& e = s->envs[i];
        const uint64_t px = (uint64_t)e.width * e.height;
        if (px == 0 || e.data_offset + 3 * px > s->n_env_floats || e.marginal_offset + e.height > s->n_env_floats || e.conditional_offset + px > s->n_env_floats) return bad("environment map outside env_floats");
        if (e.guide_h == 0 || e.guide_w == 0 || (e.guide_h & (e.guide_h - 1)) || (e.guide_w & (e.guide_w - 1))) return bad("environment guide sizes must be powers of two");
        if (e.marginal_guide_offset + e.guide_h + 1 > s->n_env_guides || e.conditional_guide_offset + (uint64_t)e.height * (e.guide_w + 1) > s->n_env_guides) return bad("environment guides outside env_guides");
        if (e.primitive < 0 || (uint32_t)e.primitive >= s->n_primitives) return bad("environment map names a primitive out of range");
    }
    return true;
}

int tcpt_upload_flat_scene(tcpt_ctx* ctx, const tcpt_flat_scene* s) {
    if (!ctx || !s) return TCPT_ERR_INVALID;
    { std::string why; if (!validate_flat(s, why)) return fail(ctx, TCPT_ERR_INVALID, why); }
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (!ctx->d_cmf) return fail(ctx, TCPT_ERR_INVALID, "upload: call tcpt_set_tables first");
    if (s->n_lights > TCPT_MAX_LIGHTS) return fail(ctx, TCPT_ERR_LIMIT, "upload: too many lights");
    if (s->max_bvh_depth >= TCPT_TRAVERSAL_STACK) return fail(ctx, TCPT_ERR_LIMIT, "upload: BVH deeper than the traversal stack");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    free_scene(ctx->dev);
    DeviceBuffers& db = ctx->dev;
    DScene& v = db.view;
    std::memset(&v, 0, sizeof v);
    int rc;
#define UP(expr) if ((rc = (expr)) != TCPT_OK) return rc
    const tcpt_bvh_node* nodes; UP(upload(ctx, db, s->bvh_nodes, s->n_bvh_nodes, &nodes)); v.nodes = (const float4*)nodes;
    const int32_t* items; UP(upload(ctx, db, s->tlas_items, (size_t)s->n_tlas_items * 2, &items)); v.tlas_items = (const int2*)items;
    const float* tv; UP(upload(ctx, db, s->tri_verts, s->n_tri_slots * 12, &tv)); v.tri_verts = (const float4*)tv;
    UP(upload(ctx, db, s->positions, s->n_vertices * 3, &v.positions));
    UP(upload(ctx, db, s->normals, s->n_vertices * 3, &v.normals));
    UP(upload(ctx, db, s->uvs, s->n_vertices * 2, &v.uvs));
    UP(upload(ctx, db, s->indices, s->n_triangles * 3, &v.indices));
    UP(upload(ctx, db, s->tangents, s->n_triangles * 3, &v.tangents));
    UP(upload(ctx, db, s->geometries, s->n_geometries, &v.geometries));
    UP(upload(ctx, db, s->primitives, s->n_primitives, &v.primitives)); v.n_primitives = s->n_primitives;
    UP(upload(ctx, db, s->materials, s->n_materials, &v.materials));
    {
        std::vector<uint8_t> pt(s->n_primitives, 0xff);
        for (uint32_t i = 0; i < s->n_primitives; ++i) { const int m = s->primitives[i].material; if (m >= 0 && (uint32_t)m < s->n_materials) pt[i] = (uint8_t)s->materials[m].type; }
        UP(upload(ctx, db, pt.data(), pt.size(), &v.prim_mat_type));
    }
    const uint8_t* tex_bytes; UP(upload(ctx, db, s->texture_bytes, s->n_texture_bytes, &tex_bytes));
    std::vector<DTexture> dt(s->n_textures);
    for (uint32_t i = 0; i < s->n_textures; ++i) dt[i] = DTexture{tex_bytes + s->textures[i].offset, s->textures[i].width, s->textures[i].height, s->textures[i].channels, 0};
    UP(upload(ctx, db, dt.data(), dt.size(), &v.textures));
    UP(upload(ctx, db, s->area_list, s->n_area, &v.area_list));
    UP(upload(ctx, db, s->area_table, s->n_area, &v.area_table));
    for (uint32_t i = 0; i < s->n_lights; ++i) v.light_list[i] = s->light_list[i];
    v.n_lights = s->n_lights;
    v.one_light_always_on = (ctx->opt.light_shortcut && one_light_always_on(s, ctx->host.tables)) ? 1u : 0u;
    const float* envf; UP(upload(ctx, db, s->env_floats, s->n_env_floats, &envf));
    const uint32_t* envg; UP(upload(ctx, db, s->env_guides, s->n_env_guides, &envg));
    std::vector<DEnv> de(s->n_envs);
    for (uint32_t i = 0; i < s->n_envs; ++i) {
        const tcpt_flat_env& e = s->envs[i];
        de[i] = DEnv{envf + e.data_offset, envf + e.marginal_offset, envf + e.conditional_offset,
                     envg + e.marginal_guide_offset, envg + e.conditional_guide_offset, e.guide_h, e.guide_w, e.intensity, e.total_weight, e.width, e.height, e.integrated, e.primitive, nullptr};
    }
    UP(upload(ctx, db, de.data(), de.size(), &v.envs)); v.n_envs = s->n_envs;
#undef UP
    v.cmf = ctx->d_cmf; v.z_nodes = ctx->d_rgb2spec; v.rgb2spec = ctx->d_rgb2spec + 64; v.presets = ctx->d_presets;
    v.half_lin = ctx->half_lin; v.half_zi = ctx->opt.illum_half ? ctx->half_zi : -1;
    std::memcpy(v.xyz_to_rgb, ctx->xyz_to_rgb, sizeof v.xyz_to_rgb);
    // per-texel light-sampling table of every environment map (32 B per texel), filled on the device by the code it replaces
    if (ctx->opt.env_nee_table) {
        bool any = false;
        for (uint32_t i = 0; i < s->n_envs; ++i) {
            const size_t texels = (size_t)de[i].w * de[i].h;
            if (texels == 0 || de[i].primitive < 0 || texels * 32 > ((size_t)1 << 31)) continue;
            void* t = nullptr;
            CU(cudaMalloc(&t, texels * 2 * sizeof(float4)));
            db.allocs.push_back(t);
            k_env_nee_table<<<grid_for(ctx, texels, 256), 256, 0, ctx->stream>>>(v, i, (float4*)t);
            CU(cudaGetLastError());
            de[i].nee_table = (const float4*)t; any = true;
        }
        if (any) {
            CU(cudaStreamSynchronize(ctx->stream));
            CU(cudaMemcpy((void*)v.envs, de.data(), de.size() * sizeof(DEnv), cudaMemcpyHostToDevice));
        }
    }
    db.max_bvh_depth = s->max_bvh_depth;
    ctx->stats.max_bvh_depth = s->max_bvh_depth;
    db.valid = true;
    return TCPT_OK;
}

// BASELINE.json configs[4]: a triangle soup as a traversal-only scene, BVH built on the device (csrc/lbvh.cuh)
int tcpt_scene_build_soup(tcpt_ctx* ctx, const float* triangles, uint32_t n_triangles) {
    if (!ctx || !triangles || n_triangles == 0) return TCPT_ERR_INVALID;
    // refused before the device is touched: the scene built before stays in place
    if (ctx->opt.soup_leaf < 1 || ctx->opt.soup_leaf > 16) return fail(ctx, TCPT_ERR_INVALID, "build_soup: option soup_leaf must be in [1, 16]");
    if (n_triangles >= (1u << 27) - 16u) return fail(ctx, TCPT_ERR_LIMIT, "build_soup: 2^27 - 16 triangles or more (a stack entry addresses 2^27 item slots)");
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    // the small tables of a one-primitive scene (identity transform, Render space = world space) go through the ordinary upload ...
    tcpt_flat_scene f{};
    tcpt_bvh_node dummy[2] = {};      // placeholders for the TLAS record and the BLAS root: the real records are built on the device below
    const int32_t items[2] = {0, 0};
    tcpt_flat_geometry g{}; g.node_base = 1; g.node_count = 1; g.slot_base = 0; g.tri_count = n_triangles;
    tcpt_flat_primitive P{};
    const float ident[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
    std::memcpy(P.l2r, ident, sizeof ident); std::memcpy(P.r2l, ident, sizeof ident);
    P.geometry = 0; P.material = 0; P.kind = 0; P.light_index = -1; P.identity = 1; P.env = -1;
    tcpt_flat_material m{}; m.type = TCPT_MAT_LAMBERT; m.color.kind = 0; m.color.c[0] = 0.5f; m.color.texture = -1; m.coat_tint.texture = -1; m.normal_texture = -1; m.eta = 1.5f;
    f.bvh_nodes = dummy; f.n_bvh_nodes = 2; f.tlas_node_count = 1; f.tlas_items = items; f.n_tlas_items = 1;
    f.geometries = &g; f.n_geometries = 1; f.primitives = &P; f.n_primitives = 1; f.materials = &m; f.n_materials = 1;
    f.max_bvh_depth = 1;
    int rc = tcpt_upload_flat_scene(ctx, &f);
    if (rc != TCPT_OK) return rc;
    ctx->dev.valid = false;
    // ... the triangles and the BVH never exist on the host
    float* d_tri = nullptr;
    CU(cudaMalloc((void**)&d_tri, (size_t)n_triangles * 9 * sizeof(float)));
    cudaError_t e = cudaMemcpy(d_tri, triangles, (size_t)n_triangles * 9 * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(d_tri); return fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e)); }
    tcpt::lbvh::Built b;
    std::string err;
    const bool ok = tcpt::lbvh::build(d_tri, n_triangles, (uint32_t)ctx->opt.soup_leaf, ctx->sm_count, ctx->stream, b, err);
    cudaFree(d_tri);
    if (!ok) return fail(ctx, b.too_deep ? TCPT_ERR_LIMIT : TCPT_ERR_CUDA, "build_soup: " + err);
    ctx->dev.allocs.push_back(b.nodes); ctx->dev.allocs.push_back(b.tri_verts);
    if (b.max_stack >= TCPT_TRAVERSAL_STACK) return fail(ctx, TCPT_ERR_LIMIT, "build_soup: BVH deeper than the traversal stack");
    ctx->dev.view.nodes = b.nodes; ctx->dev.view.tri_verts = b.tri_verts;
    ctx->dev.max_bvh_depth = b.max_stack; ctx->stats.max_bvh_depth = b.max_stack;
    ctx->soup_build_ms = b.build_ms; ctx->soup_records = b.n_nodes; ctx->soup_levels = b.levels;
    ctx->dev.traversal_only = true;
    ctx->dev.valid = true;
    return TCPT_OK;
}
int tcpt_soup_build_info(const tcpt_ctx* ctx, double* build_ms, uint64_t* n_records, uint32_t* levels) {
    if (!ctx) return TCPT_ERR_INVALID;
    if (build_ms) *build_ms = ctx->soup_build_ms;
    if (n_records) *n_records = ctx->soup_records;
    if (levels) *levels = ctx->soup_levels;
    return TCPT_OK;
}

int tcpt_scene_build(tcpt_ctx* ctx, const float cam_pos[3]) {
    if (!ctx || !cam_pos) return TCPT_ERR_INVALID;
    int r = ctx->host.build(cam_pos, ctx->flat);
    if (r != TCPT_OK) { ctx->error = ctx->host.error; return r; }
    ctx->stats.max_bvh_depth = ctx->flat.view.max_bvh_depth;   // readable on a host-only context too
    return tcpt_upload_flat_scene(ctx, &ctx->flat.view);
}

int tcpt_render_device(tcpt_ctx* ctx, const tcpt_render_params* params, void* dev_acc, void* stream) {
    if (!ctx || !dev_acc) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    reset_stats(ctx);
    if (s != ctx->stream) CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaEventRecord(ctx->ev0, s));
    int rc = render_into(ctx, params, (float*)dev_acc, s);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev1, s));
    CU(cudaEventSynchronize(ctx->ev1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->stats.render_ms = ms;
    collect_stage_times(ctx);
    return fetch_stats(ctx);
}

int tcpt_finalize_device(tcpt_ctx* ctx, const void* dev_acc, uint32_t width, uint32_t height, uint32_t spp, void* dev_srgb, void* stream) {
    if (!ctx || !dev_acc || !dev_srgb || spp == 0) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    const uint32_t n = width * height * 3;
    k_finalize<<<grid_for(ctx, n, 256), 256, 0, s>>>((const float*)dev_acc, (float*)dev_srgb, n, (float)spp, 0);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));
    return TCPT_OK;
}

int tcpt_render(tcpt_ctx* ctx, const tcpt_render_params* params, float* out_acc, float* out_srgb) {
    if (!ctx || !params || (!out_acc && !out_srgb)) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)params->width * params->height * 3;
    int rc = ensure_film(ctx, n);
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->film_acc, 0, n * sizeof(float), ctx->stream));
    rc = tcpt_render_device(ctx, params, ctx->film_acc, nullptr);
    if (rc) return rc;
    if (out_acc && (rc = copy_out(ctx, 0, out_acc, ctx->film_acc, n * sizeof(float))) != TCPT_OK) return rc;
    if (out_srgb) {
        k_finalize<<<grid_for(ctx, n, 256), 256, 0, ctx->stream>>>(ctx->film_acc, ctx->film_srgb, (uint32_t)n, (float)params->spp,
                                                                    params->integrator == TCPT_INTEGRATOR_NORMAL ? 2 : params->integrator == TCPT_INTEGRATOR_ALBEDO ? 1 : 0);
        CU(cudaGetLastError());
        if ((rc = copy_out(ctx, 1, out_srgb, ctx->film_srgb, n * sizeof(float))) != TCPT_OK) return rc;
    }
    return TCPT_OK;
}

// Adaptive sampling (include/tcpt.h): the whole frame through adaptive_frame / render_adaptive_into.
int tcpt_render_adaptive(tcpt_ctx* ctx, const tcpt_render_params* params, const tcpt_adaptive_params* ap, float* out_acc, float* out_srgb, uint32_t* out_spp) {
    if (!ctx || !params || !ap) return TCPT_ERR_INVALID;
    if (!out_acc && !out_srgb && !out_spp) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive: no output buffer");
    int rc = check_adaptive(ctx, params, ap, "render_adaptive");
    if (rc) return rc;
    if (params->row_offset || params->row_stride) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive: row_offset / row_stride must be 0 (whole frame)");
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    return adaptive_frame(ctx, params, ap, false, out_acc, out_srgb, out_spp);
}

// One row shard of an adaptive job into the caller's device buffers, on the caller's stream; no collective.
int tcpt_render_adaptive_device(tcpt_ctx* ctx, const tcpt_render_params* params, const tcpt_adaptive_params* ap, void* dev_acc, void* dev_spp, void* stream) {
    if (!ctx || !params || !ap) return TCPT_ERR_INVALID;
    if (!dev_acc || !dev_spp) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_device: dev_acc and dev_spp are required");
    int rc = check_adaptive(ctx, params, ap, "render_adaptive_device");
    if (rc) return rc;
    if (params->row_offset && params->row_offset >= params->row_stride) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_device: row_offset must be < row_stride");
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    DRender R; DCamera cam;
    if ((rc = make_render(ctx, params, R, cam)) != TCPT_OK) return rc;
    reset_stats(ctx);
    if (s != ctx->stream) CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaEventRecord(ctx->ev0, s));
    if ((rc = render_adaptive_into(ctx, params, R, cam, ap, (float*)dev_acc, (uint32_t*)dev_spp, s)) != TCPT_OK) return rc;
    CU(cudaEventRecord(ctx->ev1, s));
    CU(cudaEventSynchronize(ctx->ev1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->stats.render_ms = ms;
    collect_stage_times(ctx);
    return fetch_stats(ctx);
}

// ---------------------------------------------------------------- multi-GPU: NCCL inside the library (SURVEY.md 8b / 8e)
int tcpt_comm_get_unique_id(void* id128) {
    if (!id128) return TCPT_ERR_INVALID;
    if (!g_nccl.load()) return TCPT_ERR_CUDA;
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return TCPT_ERR_CUDA;
    static_assert(sizeof id == TCPT_COMM_ID_BYTES, "ncclUniqueId size");
    std::memcpy(id128, &id, sizeof id);
    return TCPT_OK;
}

int tcpt_comm_init(tcpt_ctx* ctx, int nranks, int rank, const void* id128) {
    if (!ctx || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (!g_nccl.load()) return fail(ctx, TCPT_ERR_CUDA, g_nccl.error);
    CU(cudaSetDevice(ctx->device));
    if (ctx->comm) { g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    ncclUniqueId id; std::memcpy(&id, id128, sizeof id);
    const ncclResult_t r = g_nccl.CommInitRank(&ctx->comm, nranks, id, rank);
    if (r != ncclSuccess) { ctx->comm = nullptr; return fail(ctx, TCPT_ERR_CUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r)); }
    ctx->comm_rank = rank; ctx->comm_size = nranks;
    if (!ctx->ev_r0) { cudaEventCreate(&ctx->ev_r0); cudaEventCreate(&ctx->ev_r1); }
    return TCPT_OK;
}

int tcpt_comm_destroy(tcpt_ctx* ctx) {
    if (!ctx) return TCPT_ERR_INVALID;
    if (ctx->comm) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    ctx->comm_rank = 0; ctx->comm_size = 1;
    return TCPT_OK;
}

int tcpt_shard_params(const tcpt_render_params* job, int shard_mode, int rank, int nranks, tcpt_render_params* out) {
    if (!job || !out || nranks < 1 || rank < 0 || rank >= nranks) return TCPT_ERR_INVALID;
    if (job->row_stride != 0 || job->row_offset != 0) return TCPT_ERR_INVALID;   // the job describes the whole frame
    *out = *job;
    const uint32_t s0 = (job->spp_begin == 0 && job->spp_end == 0) ? 0 : job->spp_begin;
    const uint32_t s1 = (job->spp_begin == 0 && job->spp_end == 0) ? job->spp : job->spp_end;
    if (s1 > job->spp || s0 > s1) return TCPT_ERR_INVALID;
    if (shard_mode == TCPT_SHARD_TILE) {
        // rows y with y % nranks == rank, every sample of the job: each pixel is summed on ONE rank in the reference's sample order
        // (sensor.rs:76-77), the other ranks add exact zeros, so the reduced film is bitwise the one-GPU film
        out->row_offset = (uint32_t)rank; out->row_stride = (uint32_t)nranks; out->spp_begin = s0; out->spp_end = s1;
    } else if (shard_mode == TCPT_SHARD_SPP) {
        // an equal slice of the job's sample indices for every pixel: best balance; per-pixel sums are re-associated across ranks
        const uint64_t n = s1 - s0;
        out->spp_begin = s0 + (uint32_t)(n * (uint64_t)rank / (uint64_t)nranks);
        out->spp_end = s0 + (uint32_t)(n * (uint64_t)(rank + 1) / (uint64_t)nranks);
    } else return TCPT_ERR_INVALID;
    return TCPT_OK;
}

int tcpt_render_sharded_device(tcpt_ctx* ctx, const tcpt_render_params* job, int shard_mode, void* dev_acc, void* stream) {
    if (!ctx || !job || !dev_acc) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (ctx->comm_size > 1 && !ctx->comm) return fail(ctx, TCPT_ERR_INVALID, "render_sharded: call tcpt_comm_init first");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    tcpt_render_params mine;
    if (tcpt_shard_params(job, shard_mode, ctx->comm_rank, ctx->comm_size, &mine) != TCPT_OK) return fail(ctx, TCPT_ERR_INVALID, "render_sharded: bad job (row shard or sample range) or shard mode");
    reset_stats(ctx);
    if (s != ctx->stream) CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaEventRecord(ctx->ev0, s));
    // a rank without samples (more ranks than sample indices) renders nothing and contributes zeros
    if (mine.spp_begin != mine.spp_end) { int rc = render_into(ctx, &mine, (float*)dev_acc, s); if (rc) return rc; }
    if (ctx->comm_size > 1) {
        // the ONE collective of a frame: sum of the Sensor accumulators onto rank 0, in place, on the rendering stream
        if (!ctx->ev_r0) { cudaEventCreate(&ctx->ev_r0); cudaEventCreate(&ctx->ev_r1); }
        CU(cudaEventRecord(ctx->ev_r0, s));
        const ncclResult_t r = g_nccl.Reduce(dev_acc, dev_acc, (size_t)job->width * job->height * 3, ncclFloat32, ncclSum, 0, ctx->comm, s);
        if (r != ncclSuccess) return fail(ctx, TCPT_ERR_CUDA, std::string("ncclReduce: ") + g_nccl.GetErrorString(r));
        CU(cudaEventRecord(ctx->ev_r1, s));
    }
    CU(cudaEventRecord(ctx->ev1, s));
    CU(cudaEventSynchronize(ctx->ev1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->stats.render_ms = ms;
    if (ctx->comm_size > 1) { float rms = 0; if (cudaEventElapsedTime(&rms, ctx->ev_r0, ctx->ev_r1) == cudaSuccess) ctx->stats.reduce_ms = rms; }
    collect_stage_times(ctx);
    return fetch_stats(ctx);
}

int tcpt_render_sharded(tcpt_ctx* ctx, const tcpt_render_params* job, int shard_mode, float* out_acc, float* out_srgb) {
    if (!ctx || !job) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    const bool root = ctx->comm_rank == 0;
    if (root && !out_acc && !out_srgb) return TCPT_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)job->width * job->height * 3;
    if (ctx->film_cap < n) {
        if (ctx->film_acc) cudaFree(ctx->film_acc);
        if (ctx->film_srgb) cudaFree(ctx->film_srgb);
        ctx->film_acc = ctx->film_srgb = nullptr; ctx->film_cap = 0;
        CU(cudaMalloc((void**)&ctx->film_acc, n * sizeof(float)));
        CU(cudaMalloc((void**)&ctx->film_srgb, n * sizeof(float)));
        ctx->film_cap = n;
    }
    CU(cudaMemsetAsync(ctx->film_acc, 0, n * sizeof(float), ctx->stream));
    int rc = tcpt_render_sharded_device(ctx, job, shard_mode, ctx->film_acc, nullptr);
    if (rc || !root) return rc;
    // rank 0 holds the whole film: Sensor::to_rgb over the job's sample count, one device -> host copy per requested buffer
    const uint32_t s0 = (job->spp_begin == 0 && job->spp_end == 0) ? 0 : job->spp_begin, s1 = (job->spp_begin == 0 && job->spp_end == 0) ? job->spp : job->spp_end;
    if (out_acc && (rc = copy_out(ctx, 0, out_acc, ctx->film_acc, n * sizeof(float))) != TCPT_OK) return rc;
    if (out_srgb) {
        k_finalize<<<grid_for(ctx, n, 256), 256, 0, ctx->stream>>>(ctx->film_acc, ctx->film_srgb, (uint32_t)n, (float)(s1 - s0),
                                                                    job->integrator == TCPT_INTEGRATOR_NORMAL ? 2 : job->integrator == TCPT_INTEGRATOR_ALBEDO ? 1 : 0);
        CU(cudaGetLastError());
        if ((rc = copy_out(ctx, 1, out_srgb, ctx->film_srgb, n * sizeof(float))) != TCPT_OK) return rc;
    }
    return TCPT_OK;
}

// One complete adaptive frame from all ranks: rank r runs the rounds over its tile shard alone (the stopping rule reads only a pixel's own
// moments, so every pixel stops where it stops on one GPU) and the ranks meet once, in adaptive_frame's grouped reduce.
int tcpt_render_adaptive_sharded(tcpt_ctx* ctx, const tcpt_render_params* job, const tcpt_adaptive_params* ap, float* out_acc, float* out_srgb, uint32_t* out_spp) {
    if (!ctx || !job || !ap) return TCPT_ERR_INVALID;
    const bool root = ctx->comm_rank == 0;
    if (root && !out_acc && !out_srgb && !out_spp) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_sharded: no output buffer on rank 0");
    int rc = check_adaptive(ctx, job, ap, "render_adaptive_sharded");
    if (rc) return rc;
    if (job->row_offset || job->row_stride) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_sharded: the job describes the whole frame (row_offset / row_stride 0)");
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (ctx->comm_size > 1 && !ctx->comm) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_sharded: call tcpt_comm_init first");
    CU(cudaSetDevice(ctx->device));
    tcpt_render_params mine;
    if (tcpt_shard_params(job, TCPT_SHARD_TILE, ctx->comm_rank, ctx->comm_size, &mine) != TCPT_OK) return fail(ctx, TCPT_ERR_INVALID, "render_adaptive_sharded: bad job");
    mine.spp_begin = mine.spp_end = 0;   // every sample of the owned rows
    return adaptive_frame(ctx, &mine, ap, true, root ? out_acc : nullptr, root ? out_srgb : nullptr, root ? out_spp : nullptr);
}


// ---------------------------------------------------------------- one host process, several GPUs (the shape a Rust `GpuRendererImage` would use)
struct tcpt_group {
    std::vector<tcpt_ctx*> ctx;
    std::string error;
};

int tcpt_group_create(const int* device_ids, int n, tcpt_group** out) {
    if (!out || !device_ids || n < 1) return TCPT_ERR_INVALID;
    *out = nullptr;
    tcpt_group* g = new tcpt_group();
    *out = g;   // returned even on failure so the message can be read; destroy it
    for (int i = 0; i < n; ++i) {
        tcpt_ctx* c = nullptr;
        const int rc = tcpt_create(device_ids[i], &c);
        if (c) g->ctx.push_back(c);
        if (rc != TCPT_OK) { g->error = c ? c->error : "tcpt_create failed"; return rc; }
    }
    if (n > 1) {
        // one communicator clique over the group's devices: a unique id, then every rank's ncclCommInitRank inside one NCCL group call
        // (a single thread may only initialise several ranks that way)
        if (!g_nccl.load()) { g->error = g_nccl.error; return TCPT_ERR_CUDA; }
        ncclUniqueId id;
        if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g->error = "ncclGetUniqueId failed"; return TCPT_ERR_CUDA; }
        g_nccl.GroupStart();
        ncclResult_t bad = ncclSuccess;
        for (int i = 0; i < n; ++i) {
            cudaSetDevice(g->ctx[i]->device);
            const ncclResult_t r = g_nccl.CommInitRank(&g->ctx[i]->comm, n, id, i);
            if (r != ncclSuccess) bad = r;
            g->ctx[i]->comm_rank = i; g->ctx[i]->comm_size = n;
        }
        const ncclResult_t e = g_nccl.GroupEnd();
        if (bad != ncclSuccess || e != ncclSuccess) {
            for (tcpt_ctx* c : g->ctx) c->comm = nullptr;
            g->error = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(bad != ncclSuccess ? bad : e);
            return TCPT_ERR_CUDA;
        }
    }
    return TCPT_OK;
}

void tcpt_group_destroy(tcpt_group* g) {
    if (!g) return;
    for (tcpt_ctx* c : g->ctx) tcpt_destroy(c);
    delete g;
}

int tcpt_group_size(const tcpt_group* g) { return g ? (int)g->ctx.size() : 0; }
tcpt_ctx* tcpt_group_context(tcpt_group* g, int i) { return (g && i >= 0 && i < (int)g->ctx.size()) ? g->ctx[i] : nullptr; }
const char* tcpt_group_last_error(const tcpt_group* g) { return g ? g->error.c_str() : "null group"; }

int tcpt_group_set_tables(tcpt_group* g, const void* std_tables, size_t std_len, const float* rgb2spec, size_t rgb2spec_floats) {
    if (!g) return TCPT_ERR_INVALID;
    for (tcpt_ctx* c : g->ctx) { const int rc = tcpt_set_tables(c, std_tables, std_len, rgb2spec, rgb2spec_floats); if (rc) { g->error = c->error; return rc; } }
    return TCPT_OK;
}

// Scene::build on context 0 (the scene is described through tcpt_scene_add_* on tcpt_group_context(g, 0)), then the same flattened
// scene is uploaded to every other device: the scene is small and read-only, every GPU keeps a replica (SURVEY.md 8e)
int tcpt_group_build(tcpt_group* g, const float cam_pos[3]) {
    if (!g || g->ctx.empty()) return TCPT_ERR_INVALID;
    int rc = tcpt_scene_build(g->ctx[0], cam_pos);
    if (rc) { g->error = g->ctx[0]->error; return rc; }
    for (size_t i = 1; i < g->ctx.size(); ++i) {
        g->ctx[i]->host.tables = g->ctx[0]->host.tables;   // one_light_always_on reads the dense tables
        rc = tcpt_upload_flat_scene(g->ctx[i], &g->ctx[0]->flat.view);
        if (rc) { g->error = g->ctx[i]->error; return rc; }
    }
    return TCPT_OK;
}

// render(ctx, root) on every context of the group, one host thread per GPU; root = whether ctx is device 0, the one whose out_* are filled
extern "C++" {
template <class F>
static int group_each(tcpt_group* g, F render) {
    const size_t n = g->ctx.size();
    std::vector<int> rcs(n, TCPT_OK);
    std::vector<std::thread> th;
    for (size_t i = 1; i < n; ++i) th.emplace_back([&, i] { rcs[i] = render(g->ctx[i], false); });
    rcs[0] = render(g->ctx[0], true);
    for (auto& t : th) t.join();
    for (size_t i = 0; i < n; ++i) if (rcs[i]) { g->error = g->ctx[i]->error; return rcs[i]; }
    return TCPT_OK;
}
}

// One complete frame from all GPUs of the group: one host thread per GPU (tcpt_render_sharded), out_* filled from device 0.
int tcpt_group_render(tcpt_group* g, const tcpt_render_params* job, int shard_mode, float* out_acc, float* out_srgb) {
    if (!g || g->ctx.empty() || !job || (!out_acc && !out_srgb)) return TCPT_ERR_INVALID;
    return group_each(g, [&](tcpt_ctx* c, bool root) { return tcpt_render_sharded(c, job, shard_mode, root ? out_acc : nullptr, root ? out_srgb : nullptr); });
}

// The same for an adaptive frame (tcpt_render_adaptive_sharded on every GPU).
int tcpt_group_render_adaptive(tcpt_group* g, const tcpt_render_params* job, const tcpt_adaptive_params* ap, float* out_acc, float* out_srgb, uint32_t* out_spp) {
    if (!g || g->ctx.empty() || !job || !ap || (!out_acc && !out_srgb && !out_spp)) return TCPT_ERR_INVALID;
    return group_each(g, [&](tcpt_ctx* c, bool root) {
        return tcpt_render_adaptive_sharded(c, job, ap, root ? out_acc : nullptr, root ? out_srgb : nullptr, root ? out_spp : nullptr);
    });
}

int tcpt_get_stats(const tcpt_ctx* ctx, tcpt_stats* out) {
    if (!ctx || !out) return TCPT_ERR_INVALID;
    *out = ctx->stats;
    return TCPT_OK;
}

int tcpt_trace_device(tcpt_ctx* ctx, const void* dev_rays, int n, int any_hit, void* dev_hits, void* stream) {
    if (!ctx || !dev_rays || !dev_hits || n < 0) return TCPT_ERR_INVALID;
    if (!ctx->dev.valid) return fail(ctx, TCPT_ERR_INVALID, "trace: no scene uploaded");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    if (n == 0) return TCPT_OK;
    // dev_rays: n x {o.xyz, tmax} followed by n x {d.xyz, -}; dev_hits: n x float4 {t,b0,b1,b2} followed by n x uint2 {prim, tri}
    const float4* q_o = (const float4*)dev_rays; const float4* q_d = q_o + n;
    float4* h0 = (float4*)dev_hits; uint2* h1 = (uint2*)(h0 + n);
    const int grid = grid_for(ctx, (uint64_t)n, 128);
    uint32_t* work = ctx->d_counters + 26;  // work counter of the persistent trace loop
    CU(cudaMemsetAsync(work, 0, sizeof(uint32_t), s));
    if (ctx->opt.count_tests) {
        // counting mode is synchronous: the box / triangle test totals of this call are readable through tcpt_get_stats afterwards
        CU(cudaMemsetAsync(ctx->d_stats, 0, 8 * sizeof(unsigned long long), s));
        k_trace_rays<true><<<grid, 128, 0, s>>>(ctx->dev.view, q_o, q_d, (uint32_t)n, any_hit, h0, h1, ctx->d_stats, work);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(s));
        return fetch_stats(ctx);
    }
    k_trace_rays<false><<<grid, 128, 0, s>>>(ctx->dev.view, q_o, q_d, (uint32_t)n, any_hit, h0, h1, nullptr, work);
    CU(cudaGetLastError());
    return TCPT_OK;
}

int tcpt_trace(tcpt_ctx* ctx, const float* rays, int n, int any_hit, int32_t* out_hit) {
    if (!ctx || !rays || !out_hit || n < 0) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (!ctx->dev.valid) return fail(ctx, TCPT_ERR_INVALID, "trace: no scene uploaded");
    if (n == 0) return TCPT_OK;
    CU(cudaSetDevice(ctx->device));
    // the caller's AoS rays go up as they are and come back as AoS hit records: the SoA queues the kernels read are (un)packed on the
    // device (a host loop over 16 M rays cost more than the traversal)
    // One staging allocation per context, grown when a call needs more and kept between calls: a cudaMalloc / cudaFree pair per call cost
    // more than the traversal (and a cudaFree lets the driver trim the kernels' local-memory pool, which the next launch rebuilds).
    const size_t b_in = ((size_t)n * 7 * sizeof(float) + 255) & ~(size_t)255, b_rays = (size_t)n * 32, b_hits = ((size_t)n * 24 + 255) & ~(size_t)255, b_out = (size_t)n * 6 * sizeof(int32_t);
    const size_t need = b_in + b_rays + b_hits + b_out;
    if (need > ctx->trace_scratch_cap) {
        if (ctx->trace_scratch) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->trace_scratch); ctx->trace_scratch = nullptr; ctx->trace_scratch_cap = 0; }
        const cudaError_t e0 = cudaMalloc(&ctx->trace_scratch, need);
        if (e0 != cudaSuccess) { cudaGetLastError(); ctx->trace_scratch = nullptr; return fail(ctx, TCPT_ERR_NOMEM, cudaGetErrorString(e0)); }
        ctx->trace_scratch_cap = need;
    }
    char* base = (char*)ctx->trace_scratch;
    float* d_in = (float*)base; void* d_rays = base + b_in; void* d_hits = base + b_in + b_rays; int32_t* d_out = (int32_t*)(base + b_in + b_rays + b_hits);
    cudaError_t e = cudaSuccess;
    reset_stats(ctx);
    cudaMemcpyAsync(d_in, rays, (size_t)n * 7 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    k_pack_rays<<<grid_for(ctx, (uint64_t)n, 256), 256, 0, ctx->stream>>>(d_in, n, (float4*)d_rays);
    int rc = tcpt_trace_device(ctx, d_rays, n, any_hit, d_hits, nullptr);
    if (rc == TCPT_OK) {
        k_unpack_hits<<<grid_for(ctx, (uint64_t)n, 256), 256, 0, ctx->stream>>>((const float4*)d_hits, n, any_hit, d_out);
        e = cudaMemcpyAsync(out_hit, d_out, (size_t)n * 6 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e));
    }
    if (rc) return rc;
    return fetch_stats(ctx);
}

// the CDF search of EnvironmentLight::sample_infinite_light (environment_light.rs:218-223) alone, as the device runs it (guide table + bisection)
int tcpt_cdf_search(tcpt_ctx* ctx, const float* cdf, uint32_t n, uint32_t guide_cells, const float* u, int m, uint32_t* out) {
    if (!ctx || !cdf || !u || !out || n == 0 || m <= 0 || guide_cells == 0 || (guide_cells & (guide_cells - 1)) != 0) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    std::vector<uint32_t> guide(guide_cells + 1);
    build_cdf_guide(cdf, n, guide_cells, guide.data());
    float *d_cdf = nullptr, *d_u = nullptr; uint32_t *d_g = nullptr, *d_o = nullptr;
    CU(cudaMalloc((void**)&d_cdf, n * sizeof(float))); CU(cudaMalloc((void**)&d_u, (size_t)m * sizeof(float)));
    CU(cudaMalloc((void**)&d_g, guide.size() * sizeof(uint32_t))); CU(cudaMalloc((void**)&d_o, (size_t)m * sizeof(uint32_t)));
    CU(cudaMemcpy(d_cdf, cdf, n * sizeof(float), cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_u, u, (size_t)m * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_g, guide.data(), guide.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    k_cdf_search<<<grid_for(ctx, (uint64_t)m, 128), 128, 0, ctx->stream>>>(d_cdf, n, d_g, guide_cells, d_u, m, d_o);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaMemcpy(out, d_o, (size_t)m * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    cudaFree(d_cdf); cudaFree(d_u); cudaFree(d_g); cudaFree(d_o);
    return TCPT_OK;
}

int tcpt_sampler_stream(tcpt_ctx* ctx, int sampler, uint32_t spp, uint32_t width, uint32_t height, uint32_t seed, uint32_t px, uint32_t py,
                        uint32_t sample_index, const int32_t* kinds, int n, float* out) {
    if (!ctx || !kinds || !out || n <= 0) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    if (!ctx->d_cmf) return fail(ctx, TCPT_ERR_INVALID, "sampler_stream: call tcpt_set_tables first");
    CU(cudaSetDevice(ctx->device));
    DRender R; std::memset(&R, 0, sizeof R);
    R.width = width; R.height = height; R.spp = spp; R.seed = seed; R.sampler = sampler;
    R.log2_spp = log2_int(spp);
    R.n_base4_digits = log2_int(round_up_pow2(width > height ? width : height)) + (R.log2_spp + 1) / 2;
    int total = 0;
    for (int i = 0; i < n; ++i) total += kinds[i] == 1 ? 1 : 2;
    int32_t* d_k = nullptr; float* d_o = nullptr;
    CU(cudaMalloc((void**)&d_k, n * 4));
    cudaError_t e = cudaMalloc((void**)&d_o, total * 4);
    if (e != cudaSuccess) { cudaFree(d_k); return fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e)); }
    cudaMemcpyAsync(d_k, kinds, n * 4, cudaMemcpyHostToDevice, ctx->stream);
    k_sampler_stream<<<1, 32, 0, ctx->stream>>>(R, px, py, sample_index, d_k, n, d_o);
    e = cudaMemcpyAsync(out, d_o, total * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_k); cudaFree(d_o);
    if (e != cudaSuccess) return fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e));
    return total;
}

int tcpt_path_samples(tcpt_ctx* ctx, const tcpt_render_params* params, const uint32_t* pixels_xy, const uint32_t* sample_indices, int n, float* out_rgb) {
    if (!ctx || !params || !pixels_xy || !sample_indices || !out_rgb || n <= 0) return TCPT_ERR_INVALID;
    if (!ctx->stream) return fail(ctx, TCPT_ERR_CUDA, "no CUDA device");
    CU(cudaSetDevice(ctx->device));
    DRender R; DCamera cam;
    int rc = make_render(ctx, params, R, cam);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        if (pixels_xy[2 * (size_t)i] >= params->width || pixels_xy[2 * (size_t)i + 1] >= params->height) return fail(ctx, TCPT_ERR_INVALID, "path_samples: pixel outside the frame");
        if (sample_indices[i] >= params->spp) return fail(ctx, TCPT_ERR_INVALID, "path_samples: sample index >= spp");
    }
    rc = ensure_state(ctx, (uint32_t)n);
    if (rc) return rc;
    uint32_t* d_xy = nullptr; uint32_t* d_s = nullptr;
    CU(cudaMalloc((void**)&d_xy, (size_t)n * 8));
    cudaError_t e = cudaMalloc((void**)&d_s, (size_t)n * 4);
    if (e != cudaSuccess) { cudaFree(d_xy); return fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e)); }
    cudaMemcpyAsync(d_xy, pixels_xy, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(d_s, sample_indices, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
    reset_stats(ctx);
    rc = ensure_sobol_prefix(ctx, R, ctx->stream);
    if (rc) { cudaFree(d_xy); cudaFree(d_s); return rc; }
    R.n_pix = (uint32_t)n; R.s_count = 1;
    set_div_magics(R);
    PathList L{d_xy, d_s};
    rc = run_pass(ctx, R, cam, L, (uint32_t)n, nullptr, ctx->stream);
    std::vector<float> rgb((size_t)n * 4);
    if (rc == TCPT_OK) {
        e = cudaMemcpyAsync(rgb.data(), ctx->st.rgb, rgb.size() * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, TCPT_ERR_CUDA, cudaGetErrorString(e));
    }
    cudaFree(d_xy); cudaFree(d_s);
    if (rc) return rc;
    collect_stage_times(ctx);
    for (int i = 0; i < n; ++i) { out_rgb[3 * (size_t)i] = rgb[4 * (size_t)i]; out_rgb[3 * (size_t)i + 1] = rgb[4 * (size_t)i + 1]; out_rgb[3 * (size_t)i + 2] = rgb[4 * (size_t)i + 2]; }
    return fetch_stats(ctx);
}

int tcpt_get_bvh(tcpt_ctx* ctx, int which, uint32_t* out, int max_nodes) {
    if (!ctx || (!out && max_nodes > 0)) return TCPT_ERR_INVALID;
    return ctx->host.dump_bvh(which, out, max_nodes);
}

int tcpt_get_wide_bvh(tcpt_ctx* ctx, int which, uint32_t* out, int max_records, uint32_t* first_record, uint32_t* slot_base) {
    if (!ctx || (!out && max_records > 0)) return TCPT_ERR_INVALID;
    const tcpt_flat_scene& v = ctx->flat.view;
    if (!v.bvh_nodes) return fail(ctx, TCPT_ERR_INVALID, "get_wide_bvh: no scene built");
    uint32_t first = 0, count = v.tlas_node_count, sbase = 0;
    if (which >= 0) {
        if (which >= (int)ctx->host.geom_flat.size() || ctx->host.geom_flat[which] < 0) return fail(ctx, TCPT_ERR_INVALID, "get_wide_bvh: geometry not in the scene");
        const tcpt_flat_geometry& g = v.geometries[ctx->host.geom_flat[which]];
        first = g.node_base; count = g.node_count; sbase = g.slot_base;
    }
    if (first_record) *first_record = first;
    if (slot_base) *slot_base = sbase;
    for (uint32_t i = 0; i < count && (int)i < max_records; ++i) std::memcpy(out + 32 * (size_t)i, v.bvh_nodes[first + i].q, 128);
    return (int)count;
}

int tcpt_build_bvh_boxes(const float* boxes, int n, uint32_t* out, int max_nodes) {
    if (!boxes || n <= 0) return TCPT_ERR_INVALID;
    std::vector<Box> ib(n);
    for (int i = 0; i < n; ++i) ib[i] = Box{{boxes[6 * i], boxes[6 * i + 1], boxes[6 * i + 2]}, {boxes[6 * i + 3], boxes[6 * i + 4], boxes[6 * i + 5]}};
    BuiltBvh b = SahBuilder(ib).build();
    return HostScene::dump_built(b, out, max_nodes);
}

int tcpt_rgb_to_coeffs(tcpt_ctx* ctx, const float rgb[3], int gamma_encoded, float coeffs[3], int32_t index[4]) {
    if (!ctx || !rgb || !coeffs) return TCPT_ERR_INVALID;
    return ctx->host.rgb_to_coeffs(rgb, gamma_encoded != 0, coeffs, index) ? TCPT_OK : fail(ctx, TCPT_ERR_INVALID, "rgb_to_coeffs: tables not set or component > 1");
}

int tcpt_get_mesh_tangents(tcpt_ctx* ctx, int geometry, float* out, int max_triangles) {
    if (!ctx || geometry < 0 || geometry >= (int)ctx->host.meshes.size()) return TCPT_ERR_INVALID;
    const HostMesh& m = ctx->host.meshes[geometry];
    const int n = (int)m.tangents.size();
    for (int i = 0; i < n && i < max_triangles; ++i) { out[3 * i] = m.tangents[i].x; out[3 * i + 1] = m.tangents[i].y; out[3 * i + 2] = m.tangents[i].z; }
    return n;
}

}  // extern "C"
