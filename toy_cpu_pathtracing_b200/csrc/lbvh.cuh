// Device-side BVH builder for TRAVERSAL-ONLY scenes: the synthetic triangle soups of BASELINE.json configs[4] (1 M - 100 M triangles).
//
// The reference's builder (scene/src/bvh.rs:92-295) is O(N^2) per level and its topology is only a parity requirement for the config
// scenes; SURVEY.md 8(d) allows any builder for the soups.  The host binned-SAH builder needs 168 s for 100 M triangles, so the soup
// BVH is built where the triangles already are:
//   1. Morton order: 63-bit codes of the triangle centroids, cub::DeviceRadixSort (a library sort: set-up work, not the hot path);
//   2. leaves = clusters of `leaf` consecutive triangles in Morton order (option "soup_leaf"; measured on the 1 M soup, see DESIGN.md);
//   3. binary radix tree over the cluster codes (Karras 2012: every inner node finds its own key range, no global synchronisation);
//   4. boxes bottom-up (the second child to arrive at a node merges);
//   5. collapse into the 4-wide 128-byte records of include/tcpt_flat.h, level by level from the root: a record starts from a binary
//      node's two children and replaces its largest inner child by that child's children until it holds four (the rule of
//      host_scene.cpp put_nodes); triangles are pre-gathered into the 48-byte slots the traversal reads (w0 = triangle index,
//      w1 = degenerate flag, w2 = first slot of the leaf: the closest-hit tie-break keys of dtraverse.cuh).
// The traversal kernels run unchanged on the result: same record layout, same slab / watertight tests, same (t, leaf, slot) order.
#pragma once
#include <cub/cub.cuh>

#include <string>

#include "dtraverse.cuh"

namespace tcpt {
namespace lbvh {

__device__ __forceinline__ uint32_t f2ord(float f) { const uint32_t u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(uint32_t u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

// bounds of the centroids (Morton normalisation): mm[0..2] = min, mm[3..5] = max, as order-preserving integers
__global__ void __launch_bounds__(256) k_centroid_bounds(const float* __restrict__ tri9, uint32_t n, uint32_t* mm) {
    float lo[3] = {TCPT_INF, TCPT_INF, TCPT_INF}, hi[3] = {-TCPT_INF, -TCPT_INF, -TCPT_INF};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* p = tri9 + 9 * (size_t)i;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float c = (p[a] + p[3 + a] + p[6 + a]) * (1.0f / 3.0f);
            lo[a] = fminf(lo[a], c); hi[a] = fmaxf(hi[a], c);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) { lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o)); hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o)); }
        if ((threadIdx.x & 31u) == 0u) { atomicMin(&mm[a], f2ord(lo[a])); atomicMax(&mm[3 + a], f2ord(hi[a])); }
    }
}
__device__ __forceinline__ uint64_t spread21(uint32_t v) {   // bit i of v -> bit 3 i
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
__global__ void __launch_bounds__(256) k_keys(const float* __restrict__ tri9, uint32_t n, const uint32_t* __restrict__ mm, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    float lo[3], inv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = ord2f(mm[a]); const float e = ord2f(mm[3 + a]) - lo[a]; inv[a] = e > 0.0f ? 2097151.0f / e : 0.0f; }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* p = tri9 + 9 * (size_t)i;
        uint32_t q[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float c = (p[a] + p[3 + a] + p[6 + a]) * (1.0f / 3.0f);
            q[a] = min((uint32_t)fmaxf((c - lo[a]) * inv[a], 0.0f), 2097151u);
        }
        keys[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
        vals[i] = i;
    }
}
// pre-gathered triangle slots in Morton order (include/tcpt_flat.h): slot s holds triangle order[s]; leaf = the cluster of `leaf` slots around it
__global__ void __launch_bounds__(256) k_gather(const float* __restrict__ tri9, const uint32_t* __restrict__ order, uint32_t n, uint32_t leaf, float4* __restrict__ tri_verts) {
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        const uint32_t tri = order[s];
        const float* p = tri9 + 9 * (size_t)tri;
        const float3 p0 = f3(p[0], p[1], p[2]), p1 = f3(p[3], p[4], p[5]), p2 = f3(p[6], p[7], p[8]);
        const float3 nrm = cross(p1 - p0, p2 - p0);
        const uint32_t degenerate = dot(nrm, nrm) == 0.0f ? 1u : 0u;   // math/src/ray.rs:50-57, the arithmetic of host_scene.cpp
        tri_verts[3 * (size_t)s] = make_float4(p0.x, p0.y, p0.z, __uint_as_float(tri));
        tri_verts[3 * (size_t)s + 1] = make_float4(p1.x, p1.y, p1.z, __uint_as_float(degenerate));
        tri_verts[3 * (size_t)s + 2] = make_float4(p2.x, p2.y, p2.z, __uint_as_float(s - s % leaf));
    }
}
// cluster c = slots [leaf c, leaf c + leaf): its box (exact min / max of the vertices) goes to binary-tree node (M - 1) + c, its key is the first triangle's code
__global__ void __launch_bounds__(256) k_clusters(const float4* __restrict__ tri_verts, const uint64_t* __restrict__ keys_sorted, uint32_t n, uint32_t leaf, uint32_t M, float4* __restrict__ blo,
                                                    float4* __restrict__ bhi, uint64_t* __restrict__ ckeys) {
    for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < M; c += gridDim.x * blockDim.x) {
        float3 lo = f3(TCPT_INF, TCPT_INF, TCPT_INF), hi = f3(-TCPT_INF, -TCPT_INF, -TCPT_INF);
        const uint32_t first = leaf * c, last = min(first + leaf, n);
        for (uint32_t s = first; s < last; ++s)
            for (int k = 0; k < 3; ++k) {
                const float4 v = tri_verts[3 * (size_t)s + k];
                lo = f3(fminf(lo.x, v.x), fminf(lo.y, v.y), fminf(lo.z, v.z)); hi = f3(fmaxf(hi.x, v.x), fmaxf(hi.y, v.y), fmaxf(hi.z, v.z));
            }
        blo[(size_t)(M - 1u) + c] = make_float4(lo.x, lo.y, lo.z, 0.0f); bhi[(size_t)(M - 1u) + c] = make_float4(hi.x, hi.y, hi.z, 0.0f);
        ckeys[c] = keys_sorted[first];
    }
}
// length of the common prefix of keys i and j (equal keys: continue with the indices); -1 outside the array
__device__ __forceinline__ int delta(const uint64_t* __restrict__ k, int M, int i, int j) {
    if (j < 0 || j >= M) return -1;
    const uint64_t a = k[i], b = k[j];
    return a == b ? 64 + __clz((uint32_t)(i ^ j)) : __clzll((long long)(a ^ b));
}
// Karras 2012, "Maximizing parallelism in the construction of BVHs, octrees and k-d trees": inner node i covers a key range that starts or
// ends at i.  Node ids: inner i -> i, leaf (cluster) c -> (M - 1) + c.
__global__ void __launch_bounds__(256) k_radix_tree(const uint64_t* __restrict__ keys, int M, int* __restrict__ left, int* __restrict__ right, int* __restrict__ parent) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M - 1; i += gridDim.x * blockDim.x) {
        const int d = delta(keys, M, i, i + 1) - delta(keys, M, i, i - 1) >= 0 ? 1 : -1;
        const int dmin = delta(keys, M, i, i - d);
        long long lmax = 2;
        while (delta(keys, M, i, (int)min((long long)M, max(-1ll, i + lmax * d))) > dmin) lmax *= 2;
        long long l = 0;
        for (long long t = lmax / 2; t >= 1; t /= 2) {
            const long long j = i + (l + t) * d;
            if (j >= 0 && j < M && delta(keys, M, i, (int)j) > dmin) l += t;
        }
        const int j = (int)(i + l * d);
        const int dnode = delta(keys, M, i, j);
        long long s = 0, t = l;
        do {
            t = (t + 1) >> 1;
            const long long q = i + (s + t) * d;
            if (q >= 0 && q < M && delta(keys, M, i, (int)q) > dnode) s += t;
        } while (t > 1);
        const int gamma = (int)(i + s * d + (d < 0 ? -1 : 0));
        const int lc = min(i, j) == gamma ? (M - 1) + gamma : gamma;
        const int rc = max(i, j) == gamma + 1 ? (M - 1) + gamma + 1 : gamma + 1;
        left[i] = lc; right[i] = rc;
        parent[lc] = i; parent[rc] = i;
        if (i == 0) parent[0] = -1;
    }
}
// boxes of the inner nodes, bottom-up: every leaf walks towards the root, the SECOND arrival at a node merges its children (the first one stops)
__global__ void __launch_bounds__(256) k_fit(int M, const int* __restrict__ parent, const int* __restrict__ left, const int* __restrict__ right, float4* blo, float4* bhi, uint32_t* flags) {
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < M; c += gridDim.x * blockDim.x) {
        int node = parent[(M - 1) + c];
        while (node >= 0) {
            if (atomicAdd(&flags[node], 1u) == 0u) break;
            const int l = left[node], r = right[node];
            const float4 a = __ldcg(&blo[l]), b = __ldcg(&blo[r]), e = __ldcg(&bhi[l]), f = __ldcg(&bhi[r]);
            __stcg(&blo[node], make_float4(fminf(a.x, b.x), fminf(a.y, b.y), fminf(a.z, b.z), 0.0f));
            __stcg(&bhi[node], make_float4(fmaxf(e.x, f.x), fmaxf(e.y, f.y), fmaxf(e.z, f.z), 0.0f));
            __threadfence();
            node = parent[node];
        }
    }
}

struct QItem { int node; uint32_t rec; };
__device__ __forceinline__ float box_area(const float4 lo, const float4 hi) { const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z; return dx * dy + dx * dz + dy * dz; }
__device__ __forceinline__ void write_record(float4* __restrict__ rec, const float4* lo, const float4* hi, const uint32_t* entry, const uint32_t* count, int cnt) {
    float q[32];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool on = k < cnt;
        q[0 + k] = on ? lo[k].x : TCPT_INF; q[4 + k] = on ? hi[k].x : -TCPT_INF; q[8 + k] = on ? lo[k].y : TCPT_INF; q[12 + k] = on ? hi[k].y : -TCPT_INF;
        q[16 + k] = on ? lo[k].z : TCPT_INF; q[20 + k] = on ? hi[k].z : -TCPT_INF;
        q[24 + k] = __uint_as_float(on ? entry[k] : TCPT_ENTRY_NONE); q[28 + k] = __uint_as_float(on ? count[k] : 0u);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) rec[r] = make_float4(q[4 * r], q[4 * r + 1], q[4 * r + 2], q[4 * r + 3]);
}
// one level of the 4-wide collapse: every queue item (binary inner node, its record) emits its record and queues its inner children
__global__ void __launch_bounds__(128) k_collapse(const QItem* __restrict__ in, uint32_t n_in, QItem* __restrict__ out, uint32_t* n_out, uint32_t* n_rec, int M, uint32_t n_tris, uint32_t leaf,
                                                   const int* __restrict__ left, const int* __restrict__ right, const float4* __restrict__ blo, const float4* __restrict__ bhi,
                                                   float4* __restrict__ nodes, uint32_t rec_base) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_in; q += gridDim.x * blockDim.x) {
        const QItem it = in[q];
        int ch[4]; int cnt = 2;
        ch[0] = left[it.node]; ch[1] = right[it.node];
        while (cnt < 4) {
            int best = -1; float best_a = -1.0f;
            for (int k = 0; k < cnt; ++k) if (ch[k] < M - 1) { const float a = box_area(blo[ch[k]], bhi[ch[k]]); if (a > best_a) { best_a = a; best = k; } }
            if (best < 0) break;
            const int c = ch[best];
            for (int k = cnt; k > best + 1; --k) ch[k] = ch[k - 1];
            ch[best] = left[c]; ch[best + 1] = right[c];
            ++cnt;
        }
        float4 lo[4], hi[4]; uint32_t entry[4], count[4];
        for (int k = 0; k < cnt; ++k) {
            const int c = ch[k];
            lo[k] = blo[c]; hi[k] = bhi[c];
            if (c >= M - 1) {
                const uint32_t first = leaf * (uint32_t)(c - (M - 1)), items = min(leaf, n_tris - first);
                entry[k] = TCPT_ENTRY_LEAF | ((items - 1u) << 27) | first; count[k] = items;
            } else {
                const uint32_t idx = atomicAdd(n_rec, 1u);
                entry[k] = rec_base + idx; count[k] = 0u;
                out[atomicAdd(n_out, 1u)] = QItem{c, idx};
            }
        }
        write_record(nodes + 8 * (size_t)(rec_base + it.rec), lo, hi, entry, count, cnt);
    }
}
// record 0 = the TLAS (one leaf with one item: the soup primitive, identity transform), and the BLAS root when the soup is a single cluster
__global__ void k_roots(float4* nodes, const float4* blo, const float4* bhi, int M, uint32_t n_tris) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int root = M > 1 ? 0 : (M - 1);
    float4 lo[4], hi[4]; uint32_t entry[4], count[4];
    lo[0] = blo[root]; hi[0] = bhi[root]; entry[0] = TCPT_ENTRY_LEAF | 0u; count[0] = 1u;
    write_record(nodes, lo, hi, entry, count, 1);
    if (M == 1) { entry[0] = TCPT_ENTRY_LEAF | ((n_tris - 1u) << 27) | 0u; count[0] = n_tris; write_record(nodes + 8, lo, hi, entry, count, 1); }
}

struct Built {
    float4* nodes = nullptr; uint64_t n_nodes = 0;      // record 0 = TLAS, records 1.. = the BLAS (root = 1)
    float4* tri_verts = nullptr; uint64_t n_slots = 0;
    uint32_t levels = 0, max_stack = 0;
    float build_ms = 0.0f;
    bool too_deep = false;                              // (on failure) the tree is deeper than the wide levels the build allows
};

#define LB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); cleanup(); return false; } } while (0)

// d_tri9: n x 9 floats on the device (vertices of triangle i).  On success `out` owns nodes and tri_verts (cudaFree).
inline bool build(const float* d_tri9, uint32_t n, uint32_t leaf, int sm_count, cudaStream_t s, Built& out, std::string& err) {
    if (n == 0 || n >= (1u << 27) - 16u) { err = "soup: triangle count must be in [1, 2^27 - 16)"; return false; }
    if (leaf < 1u || leaf > 16u) { err = "soup: leaf size must be in [1, 16]"; return false; }
    const uint32_t M = (n + leaf - 1u) / leaf;
    const int grid = sm_count * 8;
    uint32_t* d_mm = nullptr; uint64_t *d_keys = nullptr, *d_keys2 = nullptr, *d_ckeys = nullptr; uint32_t *d_vals = nullptr, *d_vals2 = nullptr;
    void* d_tmp = nullptr; float4 *d_blo = nullptr, *d_bhi = nullptr; int *d_left = nullptr, *d_right = nullptr, *d_parent = nullptr; uint32_t* d_flags = nullptr;
    QItem *d_q0 = nullptr, *d_q1 = nullptr; uint32_t* d_cnt = nullptr;
    float4 *d_nodes = nullptr, *d_tv = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto cleanup = [&]() {
        cudaFree(d_mm); cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_ckeys); cudaFree(d_vals); cudaFree(d_vals2); cudaFree(d_tmp); cudaFree(d_blo); cudaFree(d_bhi);
        cudaFree(d_left); cudaFree(d_right); cudaFree(d_parent); cudaFree(d_flags); cudaFree(d_q0); cudaFree(d_q1); cudaFree(d_cnt);
        if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1);
        if (!out.nodes) { cudaFree(d_nodes); cudaFree(d_tv); }
    };
    LB_CU(cudaEventCreate(&e0)); LB_CU(cudaEventCreate(&e1));
    LB_CU(cudaMalloc((void**)&d_mm, 6 * sizeof(uint32_t)));
    LB_CU(cudaMalloc((void**)&d_keys, (size_t)n * 8)); LB_CU(cudaMalloc((void**)&d_keys2, (size_t)n * 8));
    LB_CU(cudaMalloc((void**)&d_vals, (size_t)n * 4)); LB_CU(cudaMalloc((void**)&d_vals2, (size_t)n * 4));
    LB_CU(cudaMalloc((void**)&d_tv, (size_t)n * 3 * sizeof(float4)));
    LB_CU(cudaEventRecord(e0, s));
    { const uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u}; LB_CU(cudaMemcpyAsync(d_mm, init, sizeof init, cudaMemcpyHostToDevice, s)); }
    k_centroid_bounds<<<grid, 256, 0, s>>>(d_tri9, n, d_mm);
    k_keys<<<grid, 256, 0, s>>>(d_tri9, n, d_mm, d_keys, d_vals);
    size_t tmp_bytes = 0;
    LB_CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys2, d_vals, d_vals2, (int)n, 0, 63, s));
    LB_CU(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 1));
    LB_CU(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, d_vals2, (int)n, 0, 63, s));
    k_gather<<<grid, 256, 0, s>>>(d_tri9, d_vals2, n, leaf, d_tv);
    LB_CU(cudaMalloc((void**)&d_blo, (size_t)(2 * (size_t)M) * sizeof(float4))); LB_CU(cudaMalloc((void**)&d_bhi, (size_t)(2 * (size_t)M) * sizeof(float4)));
    LB_CU(cudaMalloc((void**)&d_ckeys, (size_t)M * 8));
    k_clusters<<<grid, 256, 0, s>>>(d_tv, d_keys2, n, leaf, M, d_blo, d_bhi, d_ckeys);
    LB_CU(cudaMalloc((void**)&d_left, (size_t)M * 4)); LB_CU(cudaMalloc((void**)&d_right, (size_t)M * 4)); LB_CU(cudaMalloc((void**)&d_parent, (size_t)2 * M * 4));
    LB_CU(cudaMalloc((void**)&d_flags, (size_t)M * 4));
    LB_CU(cudaMemsetAsync(d_flags, 0, (size_t)M * 4, s));
    const size_t max_rec = (size_t)M + 1;     // one record per binary inner node at most, + the TLAS record
    LB_CU(cudaMalloc((void**)&d_nodes, max_rec * 8 * sizeof(float4)));
    uint32_t n_rec = 1, levels = 1;
    if (M > 1) {
        k_radix_tree<<<grid, 256, 0, s>>>(d_ckeys, (int)M, d_left, d_right, d_parent);
        k_fit<<<grid, 256, 0, s>>>((int)M, d_parent, d_left, d_right, d_blo, d_bhi, d_flags);
        LB_CU(cudaMalloc((void**)&d_q0, (size_t)M * sizeof(QItem))); LB_CU(cudaMalloc((void**)&d_q1, (size_t)M * sizeof(QItem)));
        LB_CU(cudaMalloc((void**)&d_cnt, 2 * sizeof(uint32_t)));
        const QItem root{0, 0u};
        LB_CU(cudaMemcpyAsync(d_q0, &root, sizeof root, cudaMemcpyHostToDevice, s));
        const uint32_t init[2] = {0u, 1u};   // {next queue length, records allocated}
        LB_CU(cudaMemcpyAsync(d_cnt, init, sizeof init, cudaMemcpyHostToDevice, s));
        uint32_t n_in = 1;
        levels = 0;
        while (n_in) {
            ++levels;
            k_collapse<<<(int)std::min<uint64_t>((n_in + 127u) / 128u, (uint64_t)grid), 128, 0, s>>>(d_q0, n_in, d_q1, d_cnt, d_cnt + 1, (int)M, n, leaf, d_left, d_right, d_blo, d_bhi, d_nodes, 1u);
            uint32_t h[2];
            LB_CU(cudaMemcpyAsync(h, d_cnt, sizeof h, cudaMemcpyDeviceToHost, s));
            LB_CU(cudaStreamSynchronize(s));
            n_in = h[0]; n_rec = h[1];
            const uint32_t zero = 0u;
            LB_CU(cudaMemcpyAsync(d_cnt, &zero, sizeof zero, cudaMemcpyHostToDevice, s));
            std::swap(d_q0, d_q1);
            if (levels > 64) { out.too_deep = true; err = "soup: radix tree deeper than 64 wide levels"; cleanup(); return false; }
        }
    }
    k_roots<<<1, 32, 0, s>>>(d_nodes, d_blo, d_bhi, (int)M, n);
    LB_CU(cudaGetLastError());
    LB_CU(cudaEventRecord(e1, s));
    LB_CU(cudaStreamSynchronize(s));
    float ms = 0.0f; cudaEventElapsedTime(&ms, e0, e1);
    out.nodes = d_nodes; out.n_nodes = 1 + (uint64_t)n_rec; out.tri_verts = d_tv; out.n_slots = n;
    out.levels = levels; out.max_stack = 3u * levels + 4u; out.build_ms = ms;
    cleanup();
    return true;
}
#undef LB_CU

}  // namespace lbvh
}  // namespace tcpt
