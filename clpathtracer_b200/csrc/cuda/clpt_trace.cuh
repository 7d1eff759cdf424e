// clpt_trace.cuh -- device functions shared by the render kernels (internal).
//
// fp32 helpers that are never contracted into FMAs, the per-ray traversal of
// the packed kd-tree (src/kernel.cl:311-389), hit shading inputs, Philox, and
// camera ray generation (src/kernel.cl:443-456).  See render_kernel.cu for the
// numerics contract; every kernel that traces rays includes this file so that
// there is exactly one statement of the arithmetic.
#pragma once

#include "clpt_device.cuh"

#ifndef CLPT_EXPERIMENT_FMA
#define CLPT_EXPERIMENT_FMA 0
#endif
#ifndef CLPT_START_LUT
#define CLPT_START_LUT 1
#endif
#ifndef CLPT_MIN_BLOCKS
#define CLPT_MIN_BLOCKS 8 // resident 256-thread blocks per SM the register allocation aims for (measured: 3 -> 2029, 4 -> 2488, 6 -> 2921, 8 -> 3054 Mrays/s)
#endif

#ifndef CLPT_FAT_MIN_BLOCKS
// Engine 2, for trees with fat leaves (the reference builder's DEPTH-15 trees: ~56 triangles per
// leaf at 1M triangles): the same code compiled for fewer resident blocks.  Such a frame is one long
// triangle loop, which spills at 32 registers and does not at 64; the 32 warps then resident still
// keep the issue slots 62% busy (measured: 3 blocks 3.01 ms, 4 2.86, 5 4.13, 8 3.76;
// profiles/r02_experiments.json).
#define CLPT_FAT_MIN_BLOCKS 4
#endif

namespace {

struct V3 {
    float x, y, z;
};

__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
// 1/x: the correctly rounded reciprocal is the same number as the IEEE quotient 1.0f/x
__device__ __forceinline__ float frcp(float a) { return __frcp_rn(a); }
__device__ __forceinline__ V3 mk(float x, float y, float z) { V3 r = { x, y, z }; return r; }
__device__ __forceinline__ V3 vadd(V3 a, V3 b) { return mk(fadd(a.x, b.x), fadd(a.y, b.y), fadd(a.z, b.z)); }
__device__ __forceinline__ V3 vsub(V3 a, V3 b) { return mk(fsub(a.x, b.x), fsub(a.y, b.y), fsub(a.z, b.z)); }
__device__ __forceinline__ V3 vscale(V3 a, float k) { return mk(fmul(a.x, k), fmul(a.y, k), fmul(a.z, k)); }
#if CLPT_EXPERIMENT_FMA
// EXPERIMENT ONLY (never the shipped build): contracted dot/cross, to measure what
// bit-parity with the un-contracted oracle costs.  Parity tests fail in this build.
__device__ __forceinline__ float vdot(V3 a, V3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)); }
__device__ __forceinline__ V3 vcross(V3 a, V3 b) {
    return mk(fmaf(a.y, b.z, -(a.z * b.y)), fmaf(a.z, b.x, -(a.x * b.z)), fmaf(a.x, b.y, -(a.y * b.x)));
}
#else
__device__ __forceinline__ float vdot(V3 a, V3 b) {
    return fadd(fadd(fmul(a.x, b.x), fmul(a.y, b.y)), fmul(a.z, b.z));
}
__device__ __forceinline__ V3 vcross(V3 a, V3 b) {
    return mk(fsub(fmul(a.y, b.z), fmul(a.z, b.y)), fsub(fmul(a.z, b.x), fmul(a.x, b.z)),
              fsub(fmul(a.x, b.y), fmul(a.y, b.x)));
}
#endif
__device__ __forceinline__ V3 vnormalize(V3 a) {
    float len = __fsqrt_rn(vdot(a, a));
    return mk(fdiv(a.x, len), fdiv(a.y, len), fdiv(a.z, len));
}
__device__ __forceinline__ V3 xyz(float4 a) { return mk(a.x, a.y, a.z); }

// What survives the traversal loop is only the winning triangle SLOT and its t:
// primitive id, u and v are re-derived afterwards (hit_details) by the same
// arithmetic on the same operands, which keeps the loop's register footprint low.
struct Hit {
    int ref; // triangle slot of the accepted hit, -1 = none
    float t;
    int inst; // instanced kernel only: the instance hit (ref is a slot of its mesh), -1 = the base scene
};

struct HitDetails {
    int prim;
    float u, v;
};

struct Counters {
    unsigned int rays, splits, leaves, tris, shade_vn, capped;
};

// ---- the four steps of the traversal, src/kernel.cl:311-389 ----------------
// They are separate functions because two kernels compose them differently: the
// render kernel runs one ray to completion per call (closest_hit below).

// Root clip, kernel.cl:101-144.  False when the ray misses the scene box.
__device__ __forceinline__ bool root_clip(const ClptScene &S, V3 o, V3 inv, float &tmin, float &tmax) {
    const bool sx = inv.x < 0.0f, sy = inv.y < 0.0f, sz = inv.z < 0.0f;
    const float nx = sx ? S.root_max[0] : S.root_min[0], fx = sx ? S.root_min[0] : S.root_max[0];
    const float ny = sy ? S.root_max[1] : S.root_min[1], fy = sy ? S.root_min[1] : S.root_max[1];
    const float nz = sz ? S.root_max[2] : S.root_min[2], fz = sz ? S.root_min[2] : S.root_max[2];
    tmin = fmul(fsub(nx, o.x), inv.x);
    tmax = fmul(fsub(fx, o.x), inv.x);
    const float tymin = fmul(fsub(ny, o.y), inv.y), tymax = fmul(fsub(fy, o.y), inv.y);
    if ((tmin > tymax) || (tymin > tmax)) return false;
    if (tymin > tmin) tmin = tymin;
    if (tymax < tmax) tmax = tymax;
    const float tzmin = fmul(fsub(nz, o.z), inv.z), tzmax = fmul(fsub(fz, o.z), inv.z);
    if ((tmin > tzmax) || (tzmin > tmax)) return false;
    if (tzmin > tmin) tmin = tzmin;
    if (tzmax < tmax) tmax = tzmax;
    return tmax > 0.0f;
}

// Node to start the first descent of a ray from: the start-node table entry of
// the grid cell holding p1 (clpt_device.cuh).  Equivalent to starting at the root.
__device__ __forceinline__ int start_node(const ClptScene &S, V3 p1) {
#if CLPT_START_LUT
    // float -> int conversion saturates and maps NaN to 0, like "always left"
    int cx = __float2int_rd(fmul(fsub(p1.x, S.root_min[0]), S.lut_scale[0]));
    int cy = __float2int_rd(fmul(fsub(p1.y, S.root_min[1]), S.lut_scale[1]));
    int cz = __float2int_rd(fmul(fsub(p1.z, S.root_min[2]), S.lut_scale[2]));
    cx = min(max(cx, 0), S.lut_dim[0] - 1);
    cy = min(max(cy, 0), S.lut_dim[1] - 1);
    cz = min(max(cz, 0), S.lut_dim[2] - 1);
    return __ldg(S.lut + ((size_t)cz * S.lut_dim[1] + cy) * S.lut_dim[0] + cx);
#else
    return 0;
#endif
}

// Descend from node word n to the leaf containing p1, kernel.cl:325-330
// (selects, no branches).  Returns the leaf's node word.
template <bool COUNT>
__device__ __forceinline__ uint2 descend(const uint2 *__restrict__ nodes, uint2 n, V3 p1, Counters &cn) {
    while ((int)n.y >= 0) { // bit 31 marks a leaf: one sign test
        // Bits 0-1 of n.y: the axis, tested bit by bit; the rest: the low child's index.  The selects and
        // the child increment are spelled in PTX because of what ptxas makes of the C form: a bit test
        // as LOP3 + ISETP where LOP3 with a predicate result does it in one, and both child indices
        // computed and one moved where a predicated +1 does it.  12 instructions a step instead of 14
        // -- the step is a fifth of all the instructions of a frame (c3: +2.5%, profiles/r02_experiments.json).
        float p;
        unsigned index = n.y >> 2;
        asm("{\n\t.reg .pred q0, q1, f;\n\t.reg .b32 t;\n\tsetp.eq.u32 f, 1, 0;\n\t"
            "lop3.or.b32 t|q0, %4, 1, 0, 0xC0, f;\n\tlop3.or.b32 t|q1, %4, 2, 0, 0xC0, f;\n\t"
            "selp.f32 %0, %2, %1, q0;\n\tselp.f32 %0, %3, %0, q1;\n\t}"
            : "=&f"(p)
            : "f"(p1.x), "f"(p1.y), "f"(p1.z), "r"(n.y));
        asm("{\n\t.reg .pred q;\n\tsetp.gt.f32 q, %1, %2;\n\t@q add.u32 %0, %0, 1;\n\t}"
            : "+r"(index)
            : "f"(p), "f"(__uint_as_float(n.x)));
        n = __ldg(nodes + index);
        if (COUNT) cn.splits++;
    }
    return n;
}

// Leaf slab interval, kernel.cl:146-174, in two halves.  The exit half (tmax and
// the face the ray leaves by) is needed at every leaf; the entry half (tmin) only
// feeds the early-out test, which can only fire once a hit exists, so it is
// evaluated lazily.  Same expressions, same order, as the single function.
__device__ __forceinline__ void leaf_exit(float4 lmin, float4 lmax, V3 o, V3 inv, float &tmax, int &far) {
    const bool sx = inv.x < 0.0f, sy = inv.y < 0.0f, sz = inv.z < 0.0f;
    far = sx ? 0 : 1;
    tmax = fmul(fsub(sx ? lmin.x : lmax.x, o.x), inv.x);
    const float tymax = fmul(fsub(sy ? lmin.y : lmax.y, o.y), inv.y);
    if (tymax < tmax) {
        tmax = tymax;
        far = sy ? 2 : 3;
    }
    const float tzmax = fmul(fsub(sz ? lmin.z : lmax.z, o.z), inv.z);
    if (tzmax < tmax) {
        tmax = tzmax;
        far = sz ? 4 : 5;
    }
}

__device__ __forceinline__ float leaf_entry(float4 lmin, float4 lmax, V3 o, V3 inv) {
    const bool sx = inv.x < 0.0f, sy = inv.y < 0.0f, sz = inv.z < 0.0f;
    float tmin = fmul(fsub(sx ? lmax.x : lmin.x, o.x), inv.x);
    const float tymin = fmul(fsub(sy ? lmax.y : lmin.y, o.y), inv.y);
    if (tymin > tmin) tmin = tymin;
    const float tzmin = fmul(fsub(sz ? lmax.z : lmin.z, o.z), inv.z);
    if (tzmin > tmin) tmin = tzmin;
    return tmin;
}

// Triangle run of a leaf, kernel.cl:333-368 / 227-255.  Early exits are kept as
// branches: a fully predicated test measured 8% slower (profiles/).
template <bool COUNT>
__device__ __forceinline__ void triangle_run(const float4 *__restrict__ tri, int first, int count, V3 o, V3 d,
                                             int &ref, float &min_hit, Counters &cn) {
    for (int i = first; i < first + count; i++) {
        const float4 b = __ldg(tri + 3 * (size_t)i + 1);
        const float4 c = __ldg(tri + 3 * (size_t)i + 2);
        if (COUNT) cn.tris++;
        const V3 e1 = xyz(b), e2 = xyz(c);
        const V3 pvec = vcross(d, e2);
        const float det = vdot(e1, pvec);
        if (det < 0.0f) continue;
        const float4 a = __ldg(tri + 3 * (size_t)i);
        const float idet = frcp(det);
        const V3 tvec = vsub(o, xyz(a));
        const float u = fmul(vdot(tvec, pvec), idet);
        if (u < 0.0f || u > 1.0f) continue;
        // e1 and e2 are NOT kept live from the determinant to where they are next needed:
        // the few candidates that get this far fetch them again (L1 hits).  At 32 registers
        // the test otherwise fills the file and the ray constants spill around it -- spill
        // traffic was half of the L1 data pipe's load, the busiest unit (profiles/).  The
        // laundered pointers stop the compiler from merging the loads back together.
        const float4 *again1 = tri + 3 * (size_t)i + 1;
        asm volatile("" : "+l"(again1));
        const V3 qvec = vcross(tvec, xyz(__ldg(again1)));
        const float v = fmul(vdot(d, qvec), idet);
        if (v < 0.0f || fadd(u, v) > 1.0f) continue;
        const float4 *again2 = tri + 3 * (size_t)i + 2;
        asm volatile("" : "+l"(again2));
        const float t = fmul(vdot(xyz(__ldg(again2)), qvec), idet);
        if (!(t > 0.0f)) continue;
        if (ref < 0 || t <= min_hit) { // the later triangle wins ties (:344)
            min_hit = t;
            ref = i;
        }
    }
}

// ---- several lanes per ray (engine 2, one sample per pixel) -------------------------------
// On a reference-built tree a leaf holds ~56 triangles and a grazing ray tests thousands.  Here K
// neighbouring lanes walk the SAME ray -- the descent and the leaf steps are done redundantly
// (identical control flow, broadcast loads) -- and share a leaf's triangle run: lane j tests
// triangles j, j+K, j+2K, ...  A warp tile is then 32/K pixels: fewer distinct leaves per warp (the
// run's trip count is the longest among the lanes), K times as many claims, each 1/K as long.
// Measured on the 1M-triangle reference tree (as shipped, 1080p): K = 1 3.00 ms, K = 2 2.63 ms,
// K = 4 2.87, 8 3.39, 16 4.77, 32 7.59 (the redundant walk costs more than the shorter runs save),
// so K = 2 is used.  (Not a tail effect: the claims fill 96% of the resident warps' time.)
// Combining the K partial results reproduces the serial loop exactly: the smallest t wins; among
// equal t a triangle accepted in THIS leaf beats the hit carried in from earlier leaves
// (`t <= minHit`, src/kernel.cl:344) and the later triangle beats the earlier.
template <bool COUNT>
__device__ __forceinline__ void triangle_run_shared(const float4 *__restrict__ tri, int first, int count, int sub,
                                                    int log2_k, V3 o, V3 d, int &ref, float &min_hit, Counters &cn) {
    bool changed = false;
    for (int i = first + sub; i < first + count; i += 1 << log2_k) {
        const float4 b = __ldg(tri + 3 * (size_t)i + 1);
        const float4 c = __ldg(tri + 3 * (size_t)i + 2);
        if (COUNT) cn.tris++;
        const V3 e1 = xyz(b), e2 = xyz(c);
        const V3 pvec = vcross(d, e2);
        const float det = vdot(e1, pvec);
        if (det < 0.0f) continue;
        const float4 a = __ldg(tri + 3 * (size_t)i);
        const float idet = frcp(det);
        const V3 tvec = vsub(o, xyz(a));
        const float u = fmul(vdot(tvec, pvec), idet);
        if (u < 0.0f || u > 1.0f) continue;
        const V3 qvec = vcross(tvec, e1);
        const float v = fmul(vdot(d, qvec), idet);
        if (v < 0.0f || fadd(u, v) > 1.0f) continue;
        const float t = fmul(vdot(e2, qvec), idet);
        if (!(t > 0.0f)) continue;
        if (ref < 0 || t <= min_hit) {
            min_hit = t;
            ref = i;
            changed = true;
        }
    }
    // combine over the K lanes of the ray (they are converged: same ray, same control flow)
    const int lane = threadIdx.x & 31;
    const unsigned mask = ((1u << (1 << log2_k)) - 1u) << (lane & ~((1 << log2_k) - 1));
    float t = ref >= 0 ? min_hit : __int_as_float(0x7f800000);
    int pri = changed ? ref : -1, r = ref;
    for (int off = 1; off < (1 << log2_k); off <<= 1) {
        const float ot = __shfl_xor_sync(mask, t, off);
        const int opri = __shfl_xor_sync(mask, pri, off), orf = __shfl_xor_sync(mask, r, off);
        if (ot < t || (ot == t && opri > pri)) {
            t = ot;
            pri = opri;
            r = orf;
        }
    }
    ref = r;
    if (r >= 0) min_hit = t;
}

// Early-out after a leaf: 0.001 is a double literal in the reference (:381).
__device__ __forceinline__ bool hit_is_final(int ref, float tmin, float min_hit) {
    return ref >= 0 && (double)tmin + 0.001 > (double)min_hit;
}

// Step across the exit face of a leaf: p1 = orig + tmax*dir (:385), follow the rope
// (:384); true when the ray leaves the scene or exhausts its rope-hop budget.
template <bool COUNT>
__device__ __forceinline__ bool leave_leaf(const uint2 *__restrict__ nodes, const float4 *L, int far, V3 o, V3 d,
                                           float tmax, V3 &p1, uint2 &n, int &visits_left, Counters &cn) {
    p1 = vadd(o, vscale(d, tmax));
    const int next = __ldg(reinterpret_cast<const int *>(L + 2) + far);
    if (next == -1) return true;
    // the rope-hop budget counts DOWN: one live value and one add + test per leaf, where counting up
    // against max_visits had the bound re-derived from constant memory at every leaf
    if (--visits_left <= 0) {
        if (COUNT) cn.capped++;
        return true;
    }
    // ropes <= -2 name a leaf record directly: its node word is implied, nothing to fetch
    n = next >= 0 ? __ldg(nodes + next) : make_uint2((unsigned)(-2 - next), CLPT_LEAF_WORD);
    return false;
}

// The walk of one ray through one tree, from its root-clip entry tmin to completion.  SHARE:
// 1 << log2_k neighbouring lanes walk this same ray and split the triangle runs (lane `sub` of
// them; only sub 0 counts the per-ray work).
template <bool COUNT, bool SHARE>
__device__ __forceinline__ Hit walk(const ClptScene &S, V3 o, V3 d, V3 inv, float tmin, int max_visits,
                                    Counters &cn_in, int sub, int log2_k) {
    Hit h;
    h.ref = -1;
    h.t = 0.0f;
    Counters scratch = { 0, 0, 0, 0, 0, 0 };
    Counters &cn = (SHARE && sub != 0) ? scratch : cn_in; // (the helpers' visits are not the algorithm's)
    float tmax;
    V3 p1 = o;
    if (tmin > 0.0f) p1 = vadd(p1, vscale(d, tmin));

    int visits_left = max_visits > 1 ? max_visits : 1; // (the budget ends the walk at hop max(max_visits, 1))
    float min_hit = 0.0f;
    const uint2 *__restrict__ nodes = S.nodes;
    // the instrumented twin walks from the root so that its counters are the
    // reference algorithm's visit counts (the roofline's algorithmic work)
    uint2 n = __ldg(nodes + (COUNT ? 0 : start_node(S, p1)));
    for (;;) {
        n = descend<COUNT>(nodes, n, p1, cn);
        if (COUNT) cn.leaves++;
        const float4 *L = S.leaves + 4 * (size_t)n.x;
        const float4 lmin = __ldg(L), lmax = __ldg(L + 1);
        // The exit depends only on the leaf box and the ray, so it is evaluated BEFORE the
        // triangle run: two values stay live across the run instead of the box.  (Also
        // requesting the rope and the neighbour's node word here, to overlap them with the
        // run, was measured: three more live values spill at 32 registers and the L1 data
        // pipe is the busiest unit, so it costs 4%.  A separate inner loop for empty leaves
        // was measured too: -8%.  profiles/r01_experiments.json)
        int far;
        leaf_exit(lmin, lmax, o, inv, tmax, far);
        if (SHARE) {
            triangle_run_shared<COUNT>(S.tri, __float_as_int(lmin.w), __float_as_int(lmax.w), sub, log2_k, o, d, h.ref,
                                       min_hit, cn_in);
        } else {
            triangle_run<COUNT>(S.tri, __float_as_int(lmin.w), __float_as_int(lmax.w), o, d, h.ref, min_hit, cn);
        }
        // (the box is re-read from L1 rather than kept live across the run)
        if (h.ref >= 0 && hit_is_final(h.ref, leaf_entry(__ldg(L), __ldg(L + 1), o, inv), min_hit)) break;
        if (leave_leaf<COUNT>(nodes, L, far, o, d, tmax, p1, n, visits_left, cn)) break;
    }
    h.t = min_hit;
    return h;
}

// Closest hit of one ray in one tree (one "ray" of the counters).
template <bool COUNT, bool SHARE = false>
__device__ __forceinline__ Hit closest_hit(const ClptScene &S, V3 o, V3 d, int max_visits, Counters &cn_in,
                                           int sub = 0, int log2_k = 0) {
    Hit h;
    h.ref = -1;
    h.t = 0.0f;
    Counters scratch = { 0, 0, 0, 0, 0, 0 };
    Counters &cn = (SHARE && sub != 0) ? scratch : cn_in;
    if (COUNT) cn.rays++;
    const V3 inv = mk(frcp(d.x), frcp(d.y), frcp(d.z));
    float tmin, tmax;
    if (!root_clip(S, o, inv, tmin, tmax)) return h;
    return walk<COUNT, SHARE>(S, o, d, inv, tmin, max_visits, cn_in, sub, log2_k);
}

// ---- rigid instances (DESIGN.md "Rigid instances") ---------------------------------------------
// The world ray in an instance's object space: row r of [A | b] applied left to right, un-contracted
// (the form of unproject).  d' is not normalised, so t along (o', d') is the world ray's t.
__device__ __forceinline__ void object_ray(const float *m, V3 o, V3 d, V3 &lo, V3 &ld) {
    lo = mk(fadd(fadd(fadd(fmul(m[0], o.x), fmul(m[1], o.y)), fmul(m[2], o.z)), m[3]),
            fadd(fadd(fadd(fmul(m[4], o.x), fmul(m[5], o.y)), fmul(m[6], o.z)), m[7]),
            fadd(fadd(fadd(fmul(m[8], o.x), fmul(m[9], o.y)), fmul(m[10], o.z)), m[11]));
    ld = mk(fadd(fadd(fmul(m[0], d.x), fmul(m[1], d.y)), fmul(m[2], d.z)),
            fadd(fadd(fmul(m[4], d.x), fmul(m[5], d.y)), fmul(m[6], d.z)),
            fadd(fadd(fmul(m[8], d.x), fmul(m[9], d.y)), fmul(m[10], d.z)));
}

// Closest hit in the base scene and then in every instance, in array order.  An instance is
// skipped when a hit exists and the ray enters the instance's root box beyond it; a later tree's
// hit replaces the current one at t <= best (the later tree wins ties, like the later triangle at
// kernel.cl:344).  INST = false is closest_hit itself.
template <bool COUNT, bool SHARE, bool INST>
__device__ __forceinline__ Hit scene_hit(const ClptScene &S, const ClptInstances &I, V3 o, V3 d, int max_visits,
                                         Counters &cn, int sub, int log2_k) {
    Hit h = closest_hit<COUNT, SHARE>(S, o, d, max_visits, cn, sub, log2_k);
    if (INST) {
        h.inst = -1;
        for (int k = 0; k < I.count; k++) {
            const ClptInstanceRec &R = I.rec[k];
            V3 lo, ld;
            object_ray(R.w2o, o, d, lo, ld);
            const V3 inv = mk(frcp(ld.x), frcp(ld.y), frcp(ld.z));
            float tmin, tmax;
            if (!root_clip(R.mesh, lo, inv, tmin, tmax)) continue;
            if (h.ref >= 0 && tmin > h.t) continue;
            const Hit hi = walk<COUNT, SHARE>(R.mesh, lo, ld, inv, tmin, max_visits, cn, sub, log2_k);
            if (hi.ref >= 0 && (h.ref < 0 || hi.t <= h.t)) {
                h.ref = hi.ref;
                h.t = hi.t;
                h.inst = k;
            }
        }
    }
    return h;
}

// Primitive id and barycentrics of the accepted hit: hit_triangle's u and v
// (kernel.cl:243-249) evaluated again for the winning slot.
__device__ __forceinline__ HitDetails hit_details(const ClptScene &S, const Hit &h, V3 o, V3 d) {
    HitDetails r;
    const float4 a = __ldg(S.tri + 3 * (size_t)h.ref);
    const V3 e1 = xyz(__ldg(S.tri + 3 * (size_t)h.ref + 1));
    const V3 e2 = xyz(__ldg(S.tri + 3 * (size_t)h.ref + 2));
    const V3 pvec = vcross(d, e2);
    const float idet = frcp(vdot(e1, pvec));
    const V3 tvec = vsub(o, xyz(a));
    r.prim = __float_as_int(a.w);
    r.u = fmul(vdot(tvec, pvec), idet);
    r.v = fmul(vdot(d, vcross(tvec, e1)), idet);
    return r;
}

// Shading normal of an accepted hit, kernel.cl:349-365.  The flat normal is a property of the
// primitive and comes from ClptScene::flat_n (one 16-byte load instead of two, a cross product, a
// square root and three IEEE divisions at every hit); its w says whether the primitive is shaded
// with interpolated vertex normals instead.
// The vertex normals of primitive `prim` interpolated at the hit, before normalisation.
template <bool COUNT>
__device__ __forceinline__ V3 vertex_normal_sum(const ClptScene &S, const Hit &h, int prim, V3 o, V3 d, Counters &cn) {
    const int4 c1 = __ldg(S.corners + 3 * (size_t)prim);
    const HitDetails hd = hit_details(S, h, o, d);
    const int4 c2 = __ldg(S.corners + 3 * (size_t)prim + 1);
    const int4 c3 = __ldg(S.corners + 3 * (size_t)prim + 2);
    const V3 n1 = xyz(__ldg(S.norms + c1.y)), n2 = xyz(__ldg(S.norms + c2.y)), n3 = xyz(__ldg(S.norms + c3.y));
    const float w = fsub(fsub(1.0f, hd.u), hd.v);
    if (COUNT) cn.shade_vn++;
    return vadd(vadd(vscale(n1, w), vscale(n2, hd.u)), vscale(n3, hd.v));
}

template <bool COUNT>
__device__ __forceinline__ V3 hit_normal(const ClptScene &S, const Hit &h, V3 o, V3 d, Counters &cn) {
    const int prim = __float_as_int(__ldg(&S.tri[3 * (size_t)h.ref].w));
    const float4 fn = __ldg(S.flat_n + prim);
    if (fn.w != 0.0f) return vnormalize(vertex_normal_sum<COUNT>(S, h, prim, o, d, cn));
    return xyz(fn);
}

// Shading normal of an instance hit, (o', d') the object-space ray: the object-space normal BEFORE
// normalisation -- the flat normal's cross product (e1 x e2 of the triangle slot, the operands of
// ClptScene::flat_n) or the interpolated vertex normals -- mapped to world space by A^T, then
// normalised once.  (Normalising in object space too would make an identity instance shade
// differently from its own mesh: normalize is not idempotent in fp32, about a third of unit
// vectors move by an ulp when normalised again.)
template <bool COUNT>
__device__ __forceinline__ V3 instance_normal(const ClptInstanceRec &R, const Hit &h, V3 lo, V3 ld, Counters &cn) {
    const ClptScene &S = R.mesh;
    const int prim = __float_as_int(__ldg(&S.tri[3 * (size_t)h.ref].w));
    V3 m;
    if (__ldg(&S.flat_n[prim].w) != 0.0f) {
        m = vertex_normal_sum<COUNT>(S, h, prim, lo, ld, cn);
    } else {
        m = vcross(xyz(__ldg(S.tri + 3 * (size_t)h.ref + 1)), xyz(__ldg(S.tri + 3 * (size_t)h.ref + 2)));
    }
    const float *a = R.w2o;
    return vnormalize(mk(fadd(fadd(fmul(a[0], m.x), fmul(a[4], m.y)), fmul(a[8], m.z)),
                         fadd(fadd(fmul(a[1], m.x), fmul(a[5], m.y)), fmul(a[9], m.z)),
                         fadd(fadd(fmul(a[2], m.x), fmul(a[6], m.y)), fmul(a[10], m.z))));
}

template <bool COUNT, bool INST>
__device__ __forceinline__ V3 shading_normal(const ClptScene &S, const ClptInstances &I, const Hit &h, V3 o, V3 d,
                                             Counters &cn) {
    if (INST && h.inst >= 0) {
        const ClptInstanceRec &R = I.rec[h.inst];
        V3 lo, ld;
        object_ray(R.w2o, o, d, lo, ld);
        return instance_normal<COUNT>(R, h, lo, ld, cn);
    }
    return hit_normal<COUNT>(S, h, o, d, cn);
}

template <bool COUNT>
__device__ __forceinline__ void write_aov(const ClptScene &S, const ClptFrame &F, const Hit &h, V3 o, V3 d,
                                          int x, int y, int prim_offset = 0) {
    const size_t px = (size_t)y * F.width + x;
    if (h.ref >= 0) {
        const HitDetails hd = hit_details(S, h, o, d);
        F.aov_prim[px] = hd.prim + prim_offset;
        F.aov_t[px] = h.t;
        F.aov_uv[px] = make_float2(hd.u, hd.v);
    } else {
        F.aov_prim[px] = -1;
        F.aov_t[px] = 0.0f;
        F.aov_uv[px] = make_float2(0.0f, 0.0f);
    }
}

// AOVs of a first hit: an instance hit reports its primitive shifted by the instance's offset and
// u, v in its own triangle (the object-space ray); t is the world t either way.
template <bool COUNT, bool INST>
__device__ __forceinline__ void write_hit_aov(const ClptScene &S, const ClptInstances &I, const ClptFrame &F,
                                              const Hit &h, V3 o, V3 d, int x, int y) {
    if (INST && h.ref >= 0 && h.inst >= 0) {
        const ClptInstanceRec &R = I.rec[h.inst];
        V3 lo, ld;
        object_ray(R.w2o, o, d, lo, ld);
        write_aov<COUNT>(R.mesh, F, h, lo, ld, x, y, R.prim_offset);
        return;
    }
    write_aov<COUNT>(S, F, h, o, d, x, y);
}

// Philox4x32-10, counter (pixel, sample, dimension block, lane), key (seed, 'clpt').
__device__ __forceinline__ void philox(unsigned c[4], unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const unsigned n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0;
        c[1] = lo1;
        c[2] = n2;
        c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ float u01(unsigned x) { return fmul((float)(x >> 8), 0x1p-24f); }
#define CLPT_KEY1 0x636c7074u

// Cosine-weighted direction about n (extension; oracle_kernel.c cosine_dir).
__device__ __forceinline__ V3 cosine_dir(V3 n, unsigned pixel, unsigned sample, unsigned bounce,
                                         unsigned seed) {
    float a = 0.0f, b = 0.0f;
    bool found = false;
#pragma unroll 1
    for (unsigned blk = 0; blk < 2 && !found; blk++) {
        unsigned c[4] = { pixel, sample, 1u + bounce, blk };
        philox(c, seed, CLPT_KEY1);
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const float x = fsub(fmul(2.0f, u01(c[2 * k])), 1.0f);
            const float y = fsub(fmul(2.0f, u01(c[2 * k + 1])), 1.0f);
            if (!found && fadd(fmul(x, x), fmul(y, y)) <= 1.0f) {
                a = x;
                b = y;
                found = true;
            }
        }
    }
    const float zz = fsub(fsub(1.0f, fmul(a, a)), fmul(b, b));
    const float z = __fsqrt_rn(zz > 0.0f ? zz : 0.0f);
    const float sg = n.z >= 0.0f ? 1.0f : -1.0f;
    const float p = fdiv(-1.0f, fadd(sg, n.z));
    const float q = fmul(fmul(n.x, n.y), p);
    const V3 t1 = mk(fadd(1.0f, fmul(fmul(fmul(sg, n.x), n.x), p)), fmul(sg, q), fmul(-sg, n.x));
    const V3 t2 = mk(q, fadd(sg, fmul(fmul(n.y, n.y), p)), -n.y);
    return vnormalize(vadd(vadd(vscale(t1, a), vscale(t2, b)), vscale(n, z)));
}

__device__ __forceinline__ V3 unproject(const float *M, V3 X) { // kernel.cl:89-94
    const float w = fadd(fadd(fadd(fmul(M[12], X.x), fmul(M[13], X.y)), fmul(M[14], X.z)), M[15]);
    const float a = fadd(fadd(fadd(fmul(M[0], X.x), fmul(M[1], X.y)), fmul(M[2], X.z)), M[3]);
    const float b = fadd(fadd(fadd(fmul(M[4], X.x), fmul(M[5], X.y)), fmul(M[6], X.z)), M[7]);
    const float c = fadd(fadd(fadd(fmul(M[8], X.x), fmul(M[9], X.y)), fmul(M[10], X.z)), M[11]);
    return mk(fdiv(a, w), fdiv(b, w), fdiv(c, w));
}


// Camera ray of one pixel sample, kernel.cl:443-456 (+ optional Philox jitter,
// dimension block 0).  Without jitter this is exactly the reference's ray.
__device__ __forceinline__ void primary_ray(const ClptFrame &F, int x, int y, unsigned pixel, unsigned sample,
                                            V3 &o, V3 &d) {
    const float *M = F.cam;
    o = mk(F.eye[0], F.eye[1], F.eye[2]); // :443-445, divided once per frame on the host (ClptFrame::eye)
    float fx = fsub((float)(unsigned)x, F.half_width);
    float fy = fsub((float)(unsigned)y, F.half_height);
    if (F.flags & CLPT_F_JITTER) {
        unsigned c[4] = { pixel, sample, 0u, 0u };
        philox(c, F.seed, CLPT_KEY1);
        fx = fadd(fx, fsub(u01(c[0]), 0.5f));
        fy = fadd(fy, fsub(u01(c[1]), 0.5f));
    }
    const V3 ncp = unproject(M, mk(fx, fy, -1.0f));
    const V3 fcp = unproject(M, mk(fx, fy, 1.0f));
    d = vnormalize(vsub(fcp, ncp));
}

// Row of this rank's slab -> image row: tiles of tile_rows rows dealt round-robin.
__device__ __forceinline__ int slab_row_to_image_row(const ClptFrame &F, int ly) {
    const int lt = ly / F.tile_rows;
    return (lt * F.nranks + F.rank) * F.tile_rows + (ly - lt * F.tile_rows);
}

// Final store of a pixel's ordered sample sum.
__device__ __forceinline__ void store_pixel(const ClptFrame &F, int x, int ly, V3 acc, int spp) {
    float4 *dst = F.target + (size_t)ly * F.width + x;
    float4 out;
    if (spp == 1) {
        out = make_float4(acc.x, acc.y, acc.z, 1.0f);
    } else {
        const float k = fdiv(1.0f, (float)spp);
        out = make_float4(fmul(acc.x, k), fmul(acc.y, k), fmul(acc.z, k), 1.0f);
    }
    *dst = out;
    if (F.n_peer_images > 0) { // multi-GPU direct placement: 16-byte stores into every rank's frame
        const size_t at = (size_t)slab_row_to_image_row(F, ly) * F.width + x;
        for (int r = 0; r < F.n_peer_images; r++) F.peer_image[r][at] = out;
    }
}

// Progressive frames: add this frame's samples of a pixel to the fixed-point sums.
__device__ __forceinline__ void accumulate_pixel(const ClptFrame &F, int x, int y, unsigned long long r,
                                                 unsigned long long g, unsigned long long b, int spp) {
    ulonglong2 *p = reinterpret_cast<ulonglong2 *>(F.accum + 4 * ((size_t)y * F.width + x));
    ulonglong2 rg = p[0], bn = p[1];
    rg.x += r;
    rg.y += g;
    bn.x += b;
    bn.y += (unsigned long long)spp;
    p[0] = rg;
    p[1] = bn;
}

} // namespace
