// Two-level BVH traversal on the device (software; B200 has no RT cores).
//
// Reproduces the RESULT of the reference's exhaustive recursive traversal (/root/reference/scene/src/bvh.rs:344-520) with an
// ordered, t-shrinking, stack-based walk over a 4-WIDE COLLAPSE of the reference's binary tree (include/tcpt_flat.h):
//   * slab test = math/src/bounds.rs:27-55.  Rays whose origin and reciprocal direction are finite take a NaN-free form of it
//     (near / far plane picked by the direction's sign, 3-input min / max) that is the same function on those inputs (see
//     node_step); axis-parallel rays (an infinite reciprocal: 0 * inf = NaN is then possible and the reference's
//     compare-selects ignore NaNs in a particular way) run the reference's own sequence of operations (slab_exact);
//   * triangle test = math/src/ray.rs:44-158 (watertight shear, f64 fallback when an edge function is 0, conservative t > delta_t);
//   * instance transform = primitive/impls/triangle_mesh.rs:97 (ray parameter t preserved, direction not re-normalised);
//   * the reference never shrinks t_max and keeps candidates by  Node: ties -> second child,  Leaf: ties -> earlier item
//     (bvh.rs:384-388, 413-420).  That is the total order  (t, later leaf first, earlier item first)  applied per level
//     (TLAS, then BLAS), so any visiting order that sees every candidate the winner competes with gives the same hit.
//
// Why a wide tree sees the same candidates (DESIGN.md section 3, "containment").  A candidate of the reference is an item of a
// LEAF whose own box and all of whose ancestors' boxes pass Bounds::intersect.  Every inner box is the exact component-wise
// min / max of the boxes below it (bvh.rs:83-89: a fold of `merge`, and min / max do not round), and the slab test is monotone in
// the box: (b - o) * inv_d is a composition of correctly rounded, hence monotone, operations, so enlarging the box can only lower
// t0 and raise t1, axis by axis (a NaN on an axis drops that axis' constraint, which is weaker still).  A ray that passes a leaf
// box therefore passes every ancestor box: testing the LEAF boxes alone, with the reference's arithmetic, yields exactly the
// reference's candidate set, whatever inner boxes are tested (or skipped) on the way down.  The wide tree keeps every reference
// leaf, its box bits and its item order; inner boxes of the reference that became interior to a wide node are simply not tested.
// Boxes are additionally culled against  t_best * (1 + 2^-10) + 2^-10  instead of t_best: the slab interval of a box and the
// watertight t of a triangle inside it are rounded independently, so the margin (empirical, not derived: the bit-exact hit tests
// are its gate) keeps every box that could still hold an equal-or-smaller t; the triangle test always runs with the caller's t_max.
#pragma once
#include "dcommon.cuh"

#ifndef TCPT_MIN_CHUNK
#define TCPT_MIN_CHUNK 32         // smallest block of ray indices a warp reserves at a time
#endif
static_assert(TCPT_MIN_CHUNK >= 32, "a refill hands the idle lanes of a warp consecutive indices of ONE chunk: it must cover a whole warp");
#ifndef TCPT_SMEM_STACK
#define TCPT_SMEM_STACK 8         // the SHORT stack: the first 8 traversal-stack entries live in shared memory (one word per thread and row), deeper ones spill to local memory (measured 0 / 8 / 16 entries: 29.87 / 29.76 / 30.2 ms of traversal per step)
#endif
static_assert(TCPT_SMEM_STACK > 0, "the traversal stack keeps its first entries in shared memory");

namespace tcpt {

struct DHit {
    float t, b0, b1, b2;
    int prim;      // primitive index, -1 = miss
    uint32_t tri;  // triangle index within the geometry
};

struct RayXform {  // per-space ray constants for the slab and watertight tests (math/src/ray.rs:63-78)
    float3 o, inv_d;
    int kz;        // bits 0-1: the shear axis; bits 4-6: byte offsets (0 | 16) of the NEAR plane vector inside an axis pair of a wide node, x y z;
                   // bit 8: the ray takes the NaN-free slab test
    float sx, sy, sz;
};

#define TCPT_RAY_FAST 0x100

__device__ __forceinline__ void ray_setup(RayXform& r, float3 o, float3 d) {
    r.o = o;
    r.inv_d = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);  // bvh.rs:433
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int kz = 0; float m = ax;
    if (ay > m) { m = ay; kz = 1; }
    if (az > m) { kz = 2; }
    const float dx = kz == 0 ? d.y : (kz == 1 ? d.z : d.x), dy = kz == 0 ? d.z : (kz == 1 ? d.x : d.y), dz = kz == 0 ? d.x : (kz == 1 ? d.y : d.z);
    r.sx = -dx / dz; r.sy = -dy / dz; r.sz = 1.0f / dz;
    // finite origin and finite reciprocal direction: no product of the slab test can be NaN (0 * inf needs an infinity)
    const bool fast = fabsf(r.inv_d.x) < TCPT_INF && fabsf(r.inv_d.y) < TCPT_INF && fabsf(r.inv_d.z) < TCPT_INF &&
                      fabsf(o.x) < TCPT_INF && fabsf(o.y) < TCPT_INF && fabsf(o.z) < TCPT_INF;
    r.kz = kz | (r.inv_d.x < 0.0f ? 0x10 : 0) | (r.inv_d.y < 0.0f ? 0x20 : 0) | (r.inv_d.z < 0.0f ? 0x40 : 0) | (fast ? TCPT_RAY_FAST : 0);
}
// the origin moved into another space with the direction bits unchanged: everything but `o` and the fast flag carries over
__device__ __forceinline__ void ray_move_origin(RayXform& r, float3 o) {
    r.o = o;
    const bool fin = fabsf(o.x) < TCPT_INF && fabsf(o.y) < TCPT_INF && fabsf(o.z) < TCPT_INF &&
                     fabsf(r.inv_d.x) < TCPT_INF && fabsf(r.inv_d.y) < TCPT_INF && fabsf(r.inv_d.z) < TCPT_INF;
    r.kz = (r.kz & ~TCPT_RAY_FAST) | (fin ? TCPT_RAY_FAST : 0);
}

// Bounds::intersect as written (bounds.rs:35-52); NaNs (0 * inf) are ignored by the ordered compare-selects exactly as in the reference
__device__ __forceinline__ bool slab_exact(float lox, float loy, float loz, float hix, float hiy, float hiz, const RayXform& r, float t_max, float* t_entry) {
    float t0 = 0.0f, t1 = t_max;
    {
        float tn = (lox - r.o.x) * r.inv_d.x, tf = (hix - r.o.x) * r.inv_d.x;
        if (tn > tf) { const float s = tn; tn = tf; tf = s; }
        t0 = tn > t0 ? tn : t0; t1 = tf < t1 ? tf : t1;
    }
    {
        float tn = (loy - r.o.y) * r.inv_d.y, tf = (hiy - r.o.y) * r.inv_d.y;
        if (tn > tf) { const float s = tn; tn = tf; tf = s; }
        t0 = tn > t0 ? tn : t0; t1 = tf < t1 ? tf : t1;
    }
    {
        float tn = (loz - r.o.z) * r.inv_d.z, tf = (hiz - r.o.z) * r.inv_d.z;
        if (tn > tf) { const float s = tn; tn = tf; tf = s; }
        t0 = tn > t0 ? tn : t0; t1 = tf < t1 ? tf : t1;
    }
    *t_entry = t0;
    return !(t0 > t1);
}

// math::intersect_triangle up to the accept decision; returns true and t/barycentrics on a hit
__device__ __forceinline__ bool tri_test(const float4 v0, const float4 v1, const float4 v2, const RayXform& r, float t_max, float* t_out, float* b0, float* b1, float* b2) {
    if (__float_as_uint(v1.w) != 0u) return false;  // degenerate (|e1 x e2|^2 == 0), decided on the host
    const float ax = v0.x - r.o.x, ay = v0.y - r.o.y, az = v0.z - r.o.z;
    const float bx = v1.x - r.o.x, by = v1.y - r.o.y, bz = v1.z - r.o.z;
    const float cx = v2.x - r.o.x, cy = v2.y - r.o.y, cz = v2.z - r.o.z;
    float p0x, p0y, p0z, p1x, p1y, p1z, p2x, p2y, p2z;
    const int kz = r.kz & 3;
    if (kz == 0) { p0x = ay; p0y = az; p0z = ax; p1x = by; p1y = bz; p1z = bx; p2x = cy; p2y = cz; p2z = cx; }
    else if (kz == 1) { p0x = az; p0y = ax; p0z = ay; p1x = bz; p1y = bx; p1z = by; p2x = cz; p2y = cx; p2z = cy; }
    else { p0x = ax; p0y = ay; p0z = az; p1x = bx; p1y = by; p1z = bz; p2x = cx; p2y = cy; p2z = cz; }
    p0x += r.sx * p0z; p0y += r.sy * p0z;
    p1x += r.sx * p1z; p1y += r.sy * p1z;
    p2x += r.sx * p2z; p2y += r.sy * p2z;
    float e0 = p2x * p1y - p2y * p1x;
    float e1 = p0x * p2y - p0y * p2x;
    float e2 = p1x * p0y - p1y * p0x;
    if (e0 == 0.0f || e1 == 0.0f || e2 == 0.0f) {
        e0 = (float)__dsub_rn(__dmul_rn((double)p2x, (double)p1y), __dmul_rn((double)p2y, (double)p1x));
        e1 = (float)__dsub_rn(__dmul_rn((double)p0x, (double)p2y), __dmul_rn((double)p0y, (double)p2x));
        e2 = (float)__dsub_rn(__dmul_rn((double)p1x, (double)p0y), __dmul_rn((double)p1y, (double)p0x));
    }
    if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
    const float det = e0 + e1 + e2;
    if (det == 0.0f) return false;
    p0z *= r.sz; p1z *= r.sz; p2z *= r.sz;
    const float t_scaled = e0 * p0z + e1 * p1z + e2 * p2z;
    if (det < 0.0f && (t_scaled >= 0.0f || t_scaled < t_max * det)) return false;
    else if (det > 0.0f && (t_scaled <= 0.0f || t_scaled > t_max * det)) return false;
    const float inv_det = 1.0f / det;
    const float t_hit = t_scaled * inv_det;
    // conservative t > delta_t (ray.rs:137-158); gamma(n) = n*eps/(1-n*eps) evaluated in f32 like the reference's const fn
    const float EPS = 5.9604644775390625e-8f;
    const float g2 = (2.0f * EPS) / (1.0f - 2.0f * EPS), g3 = (3.0f * EPS) / (1.0f - 3.0f * EPS), g5 = (5.0f * EPS) / (1.0f - 5.0f * EPS);
    const float max_zt = rmax(fabsf(p0z), rmax(fabsf(p1z), fabsf(p2z)));
    const float delta_z = g3 * max_zt;
    const float max_xt = rmax(fabsf(p0x), rmax(fabsf(p1x), fabsf(p2x)));
    const float max_yt = rmax(fabsf(p0y), rmax(fabsf(p1y), fabsf(p2y)));
    const float delta_x = g5 * max_xt, delta_y = g5 * max_yt;
    const float delta_e = 2.0f * (g2 * max_xt * max_yt + delta_y * max_xt + delta_x * max_yt);
    const float max_e = rmax(fabsf(e0), rmax(fabsf(e1), fabsf(e2)));
    const float delta_t = 3.0f * (g3 * max_e * max_zt + delta_e * max_zt + delta_z * max_e) * fabsf(inv_det);
    if (t_hit < delta_t) return false;
    *t_out = t_hit; *b0 = e0 * inv_det; *b1 = e1 * inv_det; *b2 = e2 * inv_det;
    return true;
}

__device__ __forceinline__ float cull_limit(float t_best) { return t_best * 1.0009765625f + 0.0009765625f; }

// ---- stack / child entries (include/tcpt_flat.h): bit 31 = leaf range {bits 27-30: count - 1, bits 0-26: first item slot}, else a wide-node index
// (a reference leaf of more than 16 items is cut into ranges by the host, all under the leaf's own box: same box test, same candidates)
#define TCPT_ENTRY_LEAF 0x80000000u
#define TCPT_ENTRY_NONE 0xffffffffu
#define TCPT_ENTRY_SLOT_MASK 0x07ffffffu
#define TCPT_ENTRY_ONE_ITEM (1u - (1u << 27))   // entry + this = the same range without its first item
__device__ __forceinline__ uint32_t entry_slot(uint32_t e) { return e & TCPT_ENTRY_SLOT_MASK; }
__device__ __forceinline__ uint32_t entry_more(uint32_t e) { return (e >> 27) & 15u; }   // items behind the first one

// Per-thread state that is touched a few times per ray lives in shared memory, one word per thread and row (bank = lane: no conflicts),
// so that the registers hold only what every step reads.
enum {
    TS_OX = 0, TS_OY, TS_OZ, TS_DX, TS_DY, TS_DZ,             // the ray in Render space (read when an instance is entered)
    TS_WIX, TS_WIY, TS_WIZ, TS_WKZ, TS_WSX, TS_WSY, TS_WSZ,   // Render-space ray constants (restored when a BLAS is left)
    TS_BT, TS_B0, TS_B1, TS_B2, TS_BPRIM, TS_BTRI,            // best hit
    TS_BTLEAF, TS_BTSLOT, TS_BBLEAF, TS_BBSLOT,               // its tie-break keys: TLAS (leaf first slot, slot), BLAS (same)
    TS_CPRIM, TS_CTLEAF, TS_CTSLOT,                           // the instance being traversed
    TS_WORDS
};
struct TraceShared {
    uint32_t w[TS_WORDS][128];
    uint32_t stack[TCPT_SMEM_STACK][128];
    float stack_t[TCPT_SMEM_STACK][128];
};
#define TS_F(row) __uint_as_float(S.w[row][tid])
#define TS_U(row) S.w[row][tid]

// One ray in flight.  The walk is an explicit state machine so that a warp can keep its lanes busy:
//   * a lane whose ray is finished picks up the next ray of the queue instead of idling until the slowest ray of the warp is
//     done (persistent threads with dynamic fetch; first profile, one ray per thread: 4.2 of 32 lanes active on bounce rays);
//   * reaching a leaf only RECORDS its triangle range; the warp switches to a triangle phase (one triangle per lane per
//     iteration) once enough lanes hold pending triangles (second profile: the inline leaf loops ran with 1.9 lanes active and
//     were 60 % of the kernel's warp instructions).
struct Traversal {
    RayXform r;                  // ray constants of the space being traversed (Render space in the TLAS, instance space inside a BLAS)
    float t_max, limit;          // caller's t_max; box-culling bound (t_max until the first hit)
    uint32_t cur;                // what this lane looks at next: a wide node, a leaf range, or NONE (= take the next entry off the stack)
    int sp, blas_sp;             // stack height; stack height at BLAS entry (-1 = traversing the TLAS)

    __device__ __forceinline__ void init(TraceShared& S, uint32_t tid, float3 o, float3 d, float t_max_) {
        t_max = t_max_; limit = t_max_;
        ray_setup(r, o, d);
        TS_U(TS_OX) = __float_as_uint(o.x); TS_U(TS_OY) = __float_as_uint(o.y); TS_U(TS_OZ) = __float_as_uint(o.z);
        TS_U(TS_DX) = __float_as_uint(d.x); TS_U(TS_DY) = __float_as_uint(d.y); TS_U(TS_DZ) = __float_as_uint(d.z);
        TS_U(TS_WIX) = __float_as_uint(r.inv_d.x); TS_U(TS_WIY) = __float_as_uint(r.inv_d.y); TS_U(TS_WIZ) = __float_as_uint(r.inv_d.z);
        TS_U(TS_WKZ) = (uint32_t)r.kz; TS_U(TS_WSX) = __float_as_uint(r.sx); TS_U(TS_WSY) = __float_as_uint(r.sy); TS_U(TS_WSZ) = __float_as_uint(r.sz);
        TS_U(TS_BT) = __float_as_uint(t_max_); TS_U(TS_BPRIM) = 0xffffffffu; TS_U(TS_BTRI) = 0u;
        TS_U(TS_B0) = 0u; TS_U(TS_B1) = 0u; TS_U(TS_B2) = 0u;
        sp = 0; blas_sp = -1; cur = 0u;   // wide node 0 = the TLAS root
    }
    __device__ __forceinline__ void result(const TraceShared& S, uint32_t tid, DHit& h) const {
        h.t = TS_F(TS_BT); h.b0 = TS_F(TS_B0); h.b1 = TS_F(TS_B1); h.b2 = TS_F(TS_B2); h.prim = (int)TS_U(TS_BPRIM); h.tri = TS_U(TS_BTRI);
    }
    __device__ __forceinline__ bool holds_triangles() const { return (cur & TCPT_ENTRY_LEAF) != 0u && blas_sp >= 0; }   // (cur is never NONE between steps)

    // A stack entry of a closest-hit walk carries the entry distance `te` of its box: see advance().
    template <bool ANY>
    __device__ __forceinline__ void push(TraceShared& S, uint32_t tid, uint32_t* stack, float* stack_t, uint32_t v, float te) {
        if (sp < TCPT_SMEM_STACK) {
            S.stack[sp][tid] = v;
            if (!ANY) S.stack_t[sp][tid] = te;
        } else {
            stack[sp - TCPT_SMEM_STACK] = v;
            if (!ANY) stack_t[sp - TCPT_SMEM_STACK] = te;
        }
        ++sp;
    }
    template <bool ANY>
    __device__ __forceinline__ uint32_t pop(TraceShared& S, uint32_t tid, uint32_t* stack, float* stack_t, float* te) {
        --sp;
        if (!ANY) *te = sp < TCPT_SMEM_STACK ? S.stack_t[sp][tid] : stack_t[sp - TCPT_SMEM_STACK];
        return sp < TCPT_SMEM_STACK ? S.stack[sp][tid] : stack[sp - TCPT_SMEM_STACK];
    }

    // Tests the first triangle of the pending leaf range.  ANY = Scene::intersect_p (scene.rs:93-103): returns true (ray finished) at the first accepted triangle.
    template <bool ANY, bool COUNT>
    __device__ __forceinline__ bool tri_step(const DScene& sc, TraceShared& S, uint32_t tid, uint32_t* stack, float* stack_t, uint32_t* n_tri) {
        const uint32_t bslot = entry_slot(cur);
        cur = entry_more(cur) != 0u ? cur + TCPT_ENTRY_ONE_ITEM : TCPT_ENTRY_NONE;
        const size_t s = 3 * (size_t)bslot;
        const float4 v0 = __ldg(&sc.tri_verts[s]), v1 = __ldg(&sc.tri_verts[s + 1]), v2 = __ldg(&sc.tri_verts[s + 2]);
        float t, b0, b1, b2;
        if (COUNT) (*n_tri)++;
        if (tri_test(v0, v1, v2, r, t_max, &t, &b0, &b1, &b2)) {
            if (ANY) { TS_U(TS_BPRIM) = 0u; TS_U(TS_BT) = __float_as_uint(t); return true; }
            // total order: smaller t; then (TLAS) later leaf, earlier slot; then (BLAS) later leaf, earlier slot
            const uint32_t bleaf = __float_as_uint(v2.w);
            const float best_t = TS_F(TS_BT);
            bool take;
            if ((int)TS_U(TS_BPRIM) < 0) take = true;
            else if (t != best_t) take = t < best_t;
            else {
                const uint32_t ctleaf = TS_U(TS_CTLEAF), ctslot = TS_U(TS_CTSLOT);
                if (ctleaf != TS_U(TS_BTLEAF)) take = ctleaf > TS_U(TS_BTLEAF);
                else if (ctslot != TS_U(TS_BTSLOT)) take = ctslot < TS_U(TS_BTSLOT);
                else if (bleaf != TS_U(TS_BBLEAF)) take = bleaf > TS_U(TS_BBLEAF);
                else take = bslot < TS_U(TS_BBSLOT);
            }
            if (take) {
                TS_U(TS_BT) = __float_as_uint(t); TS_U(TS_B0) = __float_as_uint(b0); TS_U(TS_B1) = __float_as_uint(b1); TS_U(TS_B2) = __float_as_uint(b2);
                TS_U(TS_BPRIM) = TS_U(TS_CPRIM); TS_U(TS_BTRI) = __float_as_uint(v0.w);
                TS_U(TS_BTLEAF) = TS_U(TS_CTLEAF); TS_U(TS_BTSLOT) = TS_U(TS_CTSLOT); TS_U(TS_BBLEAF) = bleaf; TS_U(TS_BBSLOT) = bslot;
                limit = fminf(t_max, cull_limit(t));
            }
        }
        return advance<ANY>(S, tid, stack, stack_t);
    }

    // One walking step: open the instance of a TLAS item if that is what the lane holds, then visit a wide node (four slab tests; the
    // nearest hit child is looked at next, the others are pushed).  Returns true when the ray is finished.
    template <bool ANY, bool COUNT>
    __device__ __forceinline__ bool node_step(const DScene& sc, TraceShared& S, uint32_t tid, uint32_t* stack, float* stack_t, uint32_t* n_box) {
        if (cur & TCPT_ENTRY_LEAF) {
            // TLAS leaf (a leaf inside a BLAS belongs to the triangle phase): open its first primitive, leave the others on the stack
            const uint32_t tslot = entry_slot(cur);
            if (entry_more(cur) != 0u) push<ANY>(S, tid, stack, stack_t, cur + TCPT_ENTRY_ONE_ITEM, 0.0f);   // (entry distance 0: the other items of the leaf are never dropped)
            const int2 item = __ldg(&sc.tlas_items[tslot]);
            TS_U(TS_CPRIM) = (uint32_t)item.x; TS_U(TS_CTLEAF) = (uint32_t)item.y; TS_U(TS_CTSLOT) = tslot;
            const tcpt_flat_primitive& P = sc.primitives[item.x];
            const tcpt_flat_geometry& G = sc.geometries[P.geometry];
            // local_to_render.inverse() * ray (primitive/impls/triangle_mesh.rs:97).  An instance without rotation or scale maps the
            // direction onto the same bits, and everything ray_setup derives (1/d, the shear constants) depends on the direction
            // alone: keep the Render-space values instead of six IEEE divisions
            const float3 o = f3(TS_F(TS_OX), TS_F(TS_OY), TS_F(TS_OZ)), d = f3(TS_F(TS_DX), TS_F(TS_DY), TS_F(TS_DZ));
            const float3 ol = xf_point(P.r2l, o), dl = xf_vector(P.r2l, d);
            if (__float_as_uint(dl.x) == __float_as_uint(d.x) && __float_as_uint(dl.y) == __float_as_uint(d.y) && __float_as_uint(dl.z) == __float_as_uint(d.z)) ray_move_origin(r, ol);
            else ray_setup(r, ol, dl);
            blas_sp = sp;
            if (G.single) { cur = TCPT_ENTRY_LEAF | G.slot_base; return false; }   // SingleTriangle: straight to the triangle test, no boxes (cur != NONE: nothing to advance)
            cur = G.node_base;   // the root wide node of the BLAS
        }
        // ---- wide-node visit: rows {lo.x, hi.x, lo.y, hi.y, lo.z, hi.z} x 4 children, then the children's entries and item counts
        const float4* rec = sc.nodes + 8 * (size_t)cur;
        const uint4 ent = __ldg((const uint4*)(rec + 6));
        float te0, te1, te2, te3; bool h0, h1, h2, h3;
        if (r.kz & TCPT_RAY_FAST) {
            // NaN-free slab test.  With finite o and inv_d every product is a number, (lo - o) <= (hi - o) survives the rounding, so the
            // reference's `if tn > tf swap` picks near = lo for inv_d > 0 and near = hi for inv_d < 0 (equal products: same values
            // either way), and its compare-selects are max / min.  The near / far rows are picked by ADDRESS (16 bytes apart).
            const char* base = (const char*)rec;
            const uint32_t nx = (uint32_t)r.kz & 0x10u, ny = ((uint32_t)r.kz >> 1) & 0x10u, nz = ((uint32_t)r.kz >> 2) & 0x10u;
            const float4 ax = __ldg((const float4*)(base + nx)), bx = __ldg((const float4*)(base + (nx ^ 16u)));
            const float4 ay = __ldg((const float4*)(base + 32 + ny)), by = __ldg((const float4*)(base + 32 + (ny ^ 16u)));
            const float4 az = __ldg((const float4*)(base + 64 + nz)), bz = __ldg((const float4*)(base + 64 + (nz ^ 16u)));
#define TCPT_SLAB(c, TE, H)                                                                                                          \
            {                                                                                                                        \
                const float tnx = (ax.c - r.o.x) * r.inv_d.x, tny = (ay.c - r.o.y) * r.inv_d.y, tnz = (az.c - r.o.z) * r.inv_d.z;     \
                const float tfx = (bx.c - r.o.x) * r.inv_d.x, tfy = (by.c - r.o.y) * r.inv_d.y, tfz = (bz.c - r.o.z) * r.inv_d.z;     \
                const float t0 = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f)), t1 = fminf(fminf(tfx, tfy), fminf(tfz, limit));             \
                TE = t0; H = !(t0 > t1);                                                                                             \
            }
            TCPT_SLAB(x, te0, h0) TCPT_SLAB(y, te1, h1) TCPT_SLAB(z, te2, h2) TCPT_SLAB(w, te3, h3)
#undef TCPT_SLAB
            // (an absent child has the box (+inf, -inf): near = +-inf gives t0 = +inf > t1 = -inf, no separate check)
        } else {
            const float4 lx = __ldg(rec), hx = __ldg(rec + 1), ly = __ldg(rec + 2), hy = __ldg(rec + 3), lz = __ldg(rec + 4), hz = __ldg(rec + 5);
            h0 = ent.x != TCPT_ENTRY_NONE && slab_exact(lx.x, ly.x, lz.x, hx.x, hy.x, hz.x, r, limit, &te0);
            h1 = ent.y != TCPT_ENTRY_NONE && slab_exact(lx.y, ly.y, lz.y, hx.y, hy.y, hz.y, r, limit, &te1);
            h2 = ent.z != TCPT_ENTRY_NONE && slab_exact(lx.z, ly.z, lz.z, hx.z, hy.z, hz.z, r, limit, &te2);
            h3 = ent.w != TCPT_ENTRY_NONE && slab_exact(lx.w, ly.w, lz.w, hx.w, hy.w, hz.w, r, limit, &te3);
        }
        if (COUNT) (*n_box) += (ent.x != TCPT_ENTRY_NONE) + (ent.y != TCPT_ENTRY_NONE) + (ent.z != TCPT_ENTRY_NONE) + (ent.w != TCPT_ENTRY_NONE);
        // order the hit children by entry distance (misses sort last): the nearest is visited next, the others are pushed far to near
        float k0 = h0 ? te0 : TCPT_INF, k1 = h1 ? te1 : TCPT_INF, k2 = h2 ? te2 : TCPT_INF, k3 = h3 ? te3 : TCPT_INF;
        uint32_t e0 = h0 ? ent.x : TCPT_ENTRY_NONE, e1 = h1 ? ent.y : TCPT_ENTRY_NONE, e2 = h2 ? ent.z : TCPT_ENTRY_NONE, e3 = h3 ? ent.w : TCPT_ENTRY_NONE;
#define TCPT_CE(ka, ea, kb, eb) { const bool sw = kb < ka; const float kt = sw ? kb : ka; kb = sw ? ka : kb; ka = kt; const uint32_t et = sw ? eb : ea; eb = sw ? ea : eb; ea = et; }
        // (any hit: the answer does not depend on the order of the walk, and a ray that reaches its light -- most do -- visits every box it
        // passes whatever the order: no ordering network)
        if (!ANY) {
            TCPT_CE(k0, e0, k1, e1) TCPT_CE(k2, e2, k3, e3) TCPT_CE(k0, e0, k2, e2)
            TCPT_CE(k1, e1, k3, e3) TCPT_CE(k1, e1, k2, e2)
        }
#undef TCPT_CE
        if (e3 != TCPT_ENTRY_NONE) push<ANY>(S, tid, stack, stack_t, e3, k3);
        if (e2 != TCPT_ENTRY_NONE) push<ANY>(S, tid, stack, stack_t, e2, k2);
        if (e1 != TCPT_ENTRY_NONE) push<ANY>(S, tid, stack, stack_t, e1, k1);
        cur = e0;   // NONE when nothing was hit
        return advance<ANY>(S, tid, stack, stack_t);
    }

    // The cheap transitions, taken eagerly at the end of a step so that a lane enters the next iteration with a wide node, an instance
    // or a triangle at hand -- or is finished NOW: with nothing at hand, the ray is done when the stack is empty; a stack back at
    // its height of BLAS entry means this instance is exhausted (back to the Render-space ray); otherwise the next entry comes off.
    // (As separate walking steps these cost every ray one or two of its five or so iterations: rays here are short.)
    // Closest hit: an entry whose box is entered behind the culling bound is dropped as it comes off the stack.  The bound has
    // shrunk since the entry was pushed; every box below it is entered at or behind its own entry distance (the slab test is monotone
    // in the box, see the header), so the visit would have failed all of its slab tests: same candidates, one wide-node visit (or one
    // instance transform plus the visit of the BLAS root) less.
    template <bool ANY>
    __device__ __forceinline__ bool advance(TraceShared& S, uint32_t tid, uint32_t* stack, float* stack_t) {
        if (cur != TCPT_ENTRY_NONE) return false;
        for (;;) {
            if (sp == 0) return true;
            if (sp == blas_sp) {
                blas_sp = -1;
                r.o = f3(TS_F(TS_OX), TS_F(TS_OY), TS_F(TS_OZ));
                r.inv_d = f3(TS_F(TS_WIX), TS_F(TS_WIY), TS_F(TS_WIZ));
                r.kz = (int)TS_U(TS_WKZ); r.sx = TS_F(TS_WSX); r.sy = TS_F(TS_WSY); r.sz = TS_F(TS_WSZ);
            }
            float te = 0.0f;
            cur = pop<ANY>(S, tid, stack, stack_t, &te);
            if (ANY || !(te > limit)) return false;
        }
    }
};

#ifndef TCPT_REFILL_IDLE_LANES
#define TCPT_REFILL_IDLE_LANES 16  // a warp fetches new rays once this many of its lanes are idle (4-wide tree, eager advance: 8 / 12 / 16 / 20 give 31.8 / 30.4 / 29.9 / 30.0 ms of tracing per step).
                                   // The threshold is a kernel argument (options "refill_b0", "refill"): the camera-ray launch runs with 32, i.e. a warp traces 32 consecutive rays to the end
                                   // (12 / 16 / 20 / 24 / 32 there: 29.80 / 29.68 / 29.48 / 29.32 / 29.39 ms of tracing, and with 32 the bounce-0 shading reads its vertices in pixel order: 31.0 -> 30.65 ms)
#endif
#ifndef TCPT_TRI_PHASE_LANES
#define TCPT_TRI_PHASE_LANES 8    // a warp runs a triangle iteration once this many lanes hold pending triangles (4 / 8 / 12: 31.4 / 30.4 / 30.9 ms; no vote at all, both phases every iteration: 31.2)
#endif
#define TCPT_LOCAL_STACK (TCPT_TRAVERSAL_STACK - TCPT_SMEM_STACK)

// What a finished ray leaves behind, in two halves around the refill's ray loads: begin() issues the loads / the atomic whose results
// end() needs (ncu: the shuffle waiting for the bucket counter's atomic and the first use of the freshly loaded ray were the two top stall
// sites of the camera-ray launch, one after the other).
struct CommitToken { uint32_t a, b, c, d, e; };
template <class F> struct CommitNow {   // a commit without a second half
    F f;
    __device__ __forceinline__ CommitToken begin(uint32_t i, const DHit& h) const { f(i, h); return CommitToken{0u, 0u, 0u, 0u, 0u}; }
    __device__ __forceinline__ void end(const CommitToken&) const {}
};
template <class F> __device__ __forceinline__ CommitNow<F> commit_now(F f) { return CommitNow<F>{f}; }

// Traces the rays of a queue with persistent warps.  `work` is a global counter zeroed before the launch.  A finished ray's
// result stays in the lane's shared-memory rows until the warp's next refill point, where `commit(i, hit)` is called for all finished
// lanes together (converged): result stores, bucket filing and shadow accumulation then cost one memory round trip per refill
// instead of one per finishing lane in a divergent branch (third profile: the filing atomic at 4 lanes was the top stall).
// Every warp of the grid must call this with all 32 lanes; blocks are 128 threads (TraceShared).
template <bool ANY, bool COUNT, class Commit>
__device__ __forceinline__ void trace_queue(const DScene& sc, TraceShared& S, const float4* __restrict__ q_o, const float4* __restrict__ q_d, uint32_t n,
                                            uint32_t* work, uint32_t* n_box, uint32_t* n_tri, Commit&& commit, uint32_t refill_lanes = (uint32_t)TCPT_REFILL_IDLE_LANES, uint32_t max_chunk = 512u) {
    const uint32_t FULL = 0xffffffffu, NONE = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31u, tid = threadIdx.x;
    uint32_t stack[TCPT_LOCAL_STACK];
    float stack_t[ANY ? 1 : TCPT_LOCAL_STACK];
    Traversal T;
    T.cur = TCPT_ENTRY_NONE; T.blas_sp = -1;
    uint32_t ray = NONE, fin = NONE;
    // Ray indices are reserved from the global counter a CHUNK at a time and handed out from a warp-local pool, so most refills
    // cost no global atomic (fourth profile: the warp waiting on the counter's round trip at every refill was the top stall).
    // The chunk shrinks with the queue so that short queues (deep bounces) still spread over the whole grid.
    const uint32_t n_warps = gridDim.x * (blockDim.x >> 5);
    uint32_t chunk = n / (n_warps * 8u);
    chunk = chunk < (uint32_t)TCPT_MIN_CHUNK ? (uint32_t)TCPT_MIN_CHUNK : (chunk > max_chunk ? max_chunk : chunk);
    uint32_t pool = 0, pool_end = 0;  // warp-uniform: indices [pool, pool_end) belong to this warp
    bool drained = false;             // the global counter has passed n
    for (;;) {
        const uint32_t idle = __ballot_sync(FULL, ray == NONE);
        const uint32_t n_idle = (uint32_t)__popc(idle);
        const uint32_t left = pool_end - pool;
        const bool fetch = n_idle > left && !drained;
        uint32_t fetched = 0;
        if (fetch && lane == 0) fetched = atomicAdd(work, chunk);  // in flight while the finished rays are committed
        CommitToken tok{0u, 0u, 0u, 0u, 0u};
        const bool committing = fin != NONE;
        if (committing) {
            DHit h; T.result(S, tid, h); tok = commit.begin(fin, h); fin = NONE;
        }
        float4 new_o = make_float4(0.0f, 0.0f, 0.0f, 0.0f), new_d = new_o;
        uint32_t mine = NONE;
        if (n_idle != 0u) {
            uint32_t base_b = 0;
            if (fetch) {
                base_b = __shfl_sync(FULL, fetched, 0);
                drained = base_b + chunk >= n;
            }
            if (ray == NONE) {
                // the first `left` idle lanes take what remains of the old chunk, the others start the new one
                const uint32_t rk = (uint32_t)__popc(idle & ((1u << lane) - 1u));
                if (rk < left) mine = pool + rk;
                else if (fetch) mine = base_b + (rk - left);
                if (mine < n) { new_o = q_o[mine]; new_d = q_d[mine]; }
            }
            if (fetch) { pool = base_b + (n_idle - left); pool_end = base_b + chunk; if (pool_end > n) pool_end = n; if (pool > pool_end) pool = pool_end; }
            else { pool += n_idle; if (pool > pool_end) pool = pool_end; }
        }
        if (committing) commit.end(tok);
        if (mine < n) {   // (mine == NONE for a lane that did not refill)
            T.init(S, tid, f3(new_o.x, new_o.y, new_o.z), f3(new_d.x, new_d.y, new_d.z), new_o.w);
            ray = mine;
        }
        const bool exhausted = drained && pool >= pool_end;
        if (__ballot_sync(FULL, ray != NONE) == 0u) break;  // nothing in flight and nothing left to fetch
        const uint32_t stop_at = exhausted ? 32u : refill_lanes;
        uint32_t n_idle_now;
        do {
            const bool has_tri = ray != NONE && T.holds_triangles();
            const bool walks = ray != NONE && !has_tri;
            const uint32_t tri_mask = __ballot_sync(FULL, has_tri);
            const uint32_t node_mask = __ballot_sync(FULL, walks);
            bool finished = false;
            if (tri_mask != 0u && ((uint32_t)__popc(tri_mask) >= (uint32_t)TCPT_TRI_PHASE_LANES || node_mask == 0u)) {
                if (has_tri) finished = T.template tri_step<ANY, COUNT>(sc, S, tid, stack, stack_t, n_tri);
            } else {
                if (walks) finished = T.template node_step<ANY, COUNT>(sc, S, tid, stack, stack_t, n_box);
            }
            if (finished) { fin = ray; ray = NONE; T.cur = TCPT_ENTRY_NONE; }
            n_idle_now = (uint32_t)__popc(__ballot_sync(FULL, ray == NONE));
        } while (n_idle_now < stop_at);
    }
}

#undef TS_F
#undef TS_U

}  // namespace tcpt
