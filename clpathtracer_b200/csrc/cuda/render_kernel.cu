// render_kernel.cu -- the render hot path for sm_100a.
//
// One launch = one frame (or one rank's row tiles of it): per pixel sample,
// camera ray generation -> stackless kd-tree traversal with ropes ->
// Moller-Trumbore over the leaf's contiguous triangle run -> shading ->
// ordered accumulation over the samples -> one float4 store.
//
// What it computes is what the reference kernel computes (src/kernel.cl:296-473,
// see oracle/oracle_kernel.c for the restatement it is checked against); how
// it computes it is not: the camera matrix comes from the constant bank
// instead of global memory, split nodes are 8 bytes and siblings adjacent,
// leaves are one aligned 64-byte record, triangles are pre-gathered per leaf
// with the edge vectors precomputed, the hit normal is evaluated once per ray
// instead of once per accepted candidate, the tail recursion is a loop, and the
// lanes of a warp trace samples of the SAME pixel (see "Lane mapping" below).
//
// Numerics: every fp32 operation that decides a hit is written with the
// round-to-nearest intrinsics (__fmul_rn, __fadd_rn, ...), which the compiler
// never contracts into FMAs, and in the reference's operand order, so hit
// ids, t, u, v and colours are bit-identical to the restatement compiled with
// -ffp-contract=off.  Division and square root are the IEEE-rounded ones.
#include <math_constants.h>

#include "clpt_trace.cuh"

namespace {

// Lane mapping.  A warp works on 32 / S pixels at a time, S lanes per pixel, where
// S = sample_lanes = the largest power of two <= min(spp, 32): the S lanes of a
// pixel trace S jittered samples of that pixel side by side, so the rays of a
// warp share origin, leaves and triangles (warp-coherent by construction), node
// and triangle loads collapse into broadcasts, and lanes finish together.  At
// 1 spp this degenerates to one lane per pixel over an 8x4 pixel tile.
//   pixels per warp   1     2     4     8     16    32
//   warp tile (w x h) 1x1   2x1   2x2   4x2   4x4   8x4
// A block is 8 warps laid out 4 x 2, i.e. (4*tw) x (2*th) pixels.
// The samples of a pixel are summed in ascending sample order (shuffles in a
// fixed order), which keeps the result independent of the mapping.
__host__ __device__ inline void warp_tile_dims(int log2_ppw, int &tw, int &th) {
    tw = 1 << ((log2_ppw + 1) >> 1);
    th = 1 << (log2_ppw >> 1);
}

// INST: 0 no instances, 1 the instance list, 2 the instance tree (clpt_trace.cuh: scene_hit); the
// instanced variants are launched only while instances exist.
// ---- mode 3 (DESIGN.md "Light sampling (mode 3)"; oracle/oracle_nee.c states every operation) ----
// MIS weight of a BSDF-sampled hit at t along d on emitter k, pb the density of the bounce.
__device__ __forceinline__ float bsdf_weight(const ClptEmitters &E, int k, V3 d, float t, float pb) {
    const float pa = __ldg(&E.rec[4 * (size_t)k + 1].w);
    const float cl = -vdot(d, xyz(__ldg(E.rec + 4 * (size_t)k + 3)));
    if (!(pa > 0.0f) || !(cl > 0.0f)) return 1.0f;
    const float q = fdiv(fdiv(fmul(pa, fmul(t, t)), cl), pb);
    return fdiv(1.0f, fadd(1.0f, fmul(q, q)));
}

// The light sample of a diffuse vertex at x (shading normal nrm, throughput T after the albedo):
// an emitter chosen by its integer weight, a point on it, a shadow ray, and the MIS-weighted
// estimate times (1 - p).
template <bool COUNT, bool SHARE, int INST>
__device__ __noinline__ V3 light_sample(const ClptScene &S, const ClptInstances &I, const ClptEmitters &E,
                                        const ClptFrame &F, V3 x, V3 nrm, V3 T, unsigned pixel, unsigned sample,
                                        unsigned seg, Counters &cn, int sub, int log2_k) {
    unsigned c[4] = { pixel, sample, 1u + seg, 2u };
    philox(c, F.seed, CLPT_KEY1);
    const unsigned long long Q = __ldg(E.header + 1);
    const unsigned long long target = __umul64hi((unsigned long long)c[0] << 32, Q); // (r0 * Q) >> 32
    unsigned long long lo = 0, hi = __ldg(E.header);
    while (hi - lo > 1ull) { // the largest i with cdf[i] <= target
        const unsigned long long mid = (lo + hi) >> 1;
        if (__ldg(E.cdf + mid) <= target) lo = mid;
        else hi = mid;
    }
    const float4 *R = E.rec + 4 * (size_t)lo;
    const float4 r0 = __ldg(R), r1 = __ldg(R + 1), r2 = __ldg(R + 2), r3 = __ldg(R + 3);
    const V3 e1 = xyz(r1), e2 = xyz(r2);
    const float su = __fsqrt_rn(u01(c[1])), u2 = u01(c[2]);
    const V3 y = vadd(vadd(xyz(r0), vscale(e1, fmul(su, fsub(1.0f, u2)))), vscale(e2, fmul(su, u2)));
    const V3 L = vsub(y, x);
    const float d2 = vdot(L, L), dist = __fsqrt_rn(d2);
    const V3 l = mk(fdiv(L.x, dist), fdiv(L.y, dist), fdiv(L.z, dist));
    const float cx = vdot(l, nrm);
    const float det = vdot(e1, vcross(l, e2));
    const float cl = -vdot(l, xyz(r3));
    const V3 none = mk(0.0f, 0.0f, 0.0f);
    if (!(cx > 0.0f) || !(det > 0.0f) || !(cl > 0.0f)) return none;
    if (occluded<COUNT, SHARE, INST>(S, I, vadd(x, vscale(l, 0.0001f)), l, fmul(fsub(dist, 0.0001f), CLPT_NEE_TMAX_SCALE),
                                     F.max_leaf_visits, cn, sub, log2_k))
        return none;
    const int prim = __float_as_int(r0.w);
    int m = S.tri_material ? __ldg(S.tri_material + prim) : 0;
    if (m < 0 || m >= S.n_materials) m = 0;
    const float *em = S.materials[m].emission;
    const float r = fdiv(fmul(cx, CLPT_NEE_PB), fdiv(fmul(r1.w, d2), cl));
    const float k = fdiv(r, fadd(1.0f, fmul(r, r)));
    return mk(fmul(fmul(T.x, em[0]), k), fmul(fmul(T.y, em[1]), k), fmul(fmul(T.z, em[2]), k));
}

// ---- environment (DESIGN.md "Environment light"; oracle/oracle_env.c states every operation) ----
__device__ __forceinline__ int env_index(float x, int n) {
    const int i = __float2int_rz(fmul(fmul(fadd(x, 1.0f), 0.5f), (float)n));
    return min(max(i, 0), n - 1);
}

// The texel env(d) looks up (OpenGL cube-map faces, nearest texel) and its face coordinates a, b.
__device__ __forceinline__ int env_texel(int n, V3 d, float &a, float &b) {
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int face;
    float sc, tc, ma;
    if (ax >= ay && ax >= az) {
        ma = ax, tc = -d.y;
        if (d.x > 0.0f) face = 0, sc = -d.z;
        else face = 1, sc = d.z;
    } else if (ay >= az) {
        ma = ay, sc = d.x;
        if (d.y > 0.0f) face = 2, tc = d.z;
        else face = 3, tc = -d.z;
    } else {
        ma = az, tc = -d.y;
        if (d.z > 0.0f) face = 4, sc = d.x;
        else face = 5, sc = -d.x;
    }
    a = fdiv(sc, ma);
    b = fdiv(tc, ma);
    return (face * n + env_index(b, n)) * n + env_index(a, n);
}

// The solid-angle density of face coordinates (a, b) in a texel of pdf `pdf`: pdf * s2^(3/2).
__device__ __forceinline__ float env_pe(float pdf, float a, float b) {
    const float s2 = fadd(fadd(1.0f, fmul(a, a)), fmul(b, b));
    return fmul(pdf, fmul(s2, __fsqrt_rn(s2)));
}

// What a path that leaves the scene along d adds: T * env(d); with MIS (mode 3), after a diffuse
// bounce that did not fall back (mis) of density pb, weighted against the environment's light sample.
template <bool MIS>
__device__ __forceinline__ V3 env_miss(const ClptEnvironment &V, V3 d, V3 T, bool mis, float pb) {
    float a, b;
    const float4 tx = __ldg(V.tex + env_texel(V.n, d, a, b));
    const V3 e = mk(fmul(T.x, tx.x), fmul(T.y, tx.y), fmul(T.z, tx.z));
    if (!MIS || !mis || !(tx.w > 0.0f)) return e;
    const float q = fdiv(env_pe(tx.w, a, b), pb);
    return vscale(e, fdiv(1.0f, fadd(1.0f, fmul(q, q))));
}

// The environment's light sample of a diffuse vertex at x: a texel chosen by its integer weight, a
// uniform point in it, a shadow ray without end, and the MIS-weighted estimate times (1 - p).
template <bool COUNT, bool SHARE, int INST>
__device__ __noinline__ V3 env_sample(const ClptScene &S, const ClptInstances &I, const ClptEnvironment &V,
                                      const ClptFrame &F, V3 x, V3 nrm, V3 T, unsigned pixel, unsigned sample,
                                      unsigned seg, Counters &cn, int sub, int log2_k) {
    unsigned c[4] = { pixel, sample, 1u + seg, 3u };
    philox(c, F.seed, CLPT_KEY1);
    const int n = V.n;
    const unsigned long long Q = __ldg(V.header + 1);
    const unsigned long long target = __umul64hi((unsigned long long)c[0] << 32, Q); // (r0 * Q) >> 32
    unsigned long long lo = 0, hi = 6ull * (unsigned long long)n * (unsigned long long)n;
    while (hi - lo > 1ull) { // the largest i with cdf[i] <= target
        const unsigned long long mid = (lo + hi) >> 1;
        if (__ldg(V.cdf + mid) <= target) lo = mid;
        else hi = mid;
    }
    const int texel = (int)lo, face = texel / (n * n), rem = texel - face * (n * n), row = rem / n, col = rem - row * n;
    const float fn = (float)n;
    const float a = fsub(fmul(fdiv(fadd((float)col, u01(c[1])), fn), 2.0f), 1.0f);
    const float b = fsub(fmul(fdiv(fadd((float)row, u01(c[2])), fn), 2.0f), 1.0f);
    V3 v;
    switch (face) { // the face point whose (sc, tc, ma) is (a, b, +-1)
    case 0: v = mk(1.0f, -b, -a); break;
    case 1: v = mk(-1.0f, -b, a); break;
    case 2: v = mk(a, 1.0f, b); break;
    case 3: v = mk(a, -1.0f, -b); break;
    case 4: v = mk(a, -b, 1.0f); break;
    default: v = mk(-a, -b, -1.0f); break;
    }
    const V3 l = vnormalize(v);
    const float cx = vdot(l, nrm);
    const V3 none = mk(0.0f, 0.0f, 0.0f);
    if (!(cx > 0.0f)) return none;
    if (occluded<COUNT, SHARE, INST>(S, I, vadd(x, vscale(l, 0.0001f)), l, CUDART_MAX_NORMAL_F, F.max_leaf_visits, cn, sub,
                                     log2_k))
        return none;
    const float4 tx = __ldg(V.tex + texel);
    const float r = fdiv(fmul(cx, CLPT_NEE_PB), env_pe(tx.w, a, b));
    const float k = fdiv(r, fadd(1.0f, fmul(r, r)));
    return mk(fmul(fmul(T.x, tx.x), k), fmul(fmul(T.y, tx.y), k), fmul(fmul(T.z, tx.z), k));
}

// MODE 3 traces mode 2's paths and adds light samples combined by MIS (DESIGN.md "Light sampling
// (mode 3)"; oracle/oracle_nee.c is the definition).  ENV (modes 2 and 3 only): escaping paths add
// T * env(d) instead of T, and mode 3 also samples the environment (oracle/oracle_env.c).
template <int MODE, bool COUNT, bool SHARE, int INST, bool ENV>
__device__ __forceinline__ V3 trace_sample(const ClptScene &S, const ClptInstances &I, const ClptEmitters &E,
                                           const ClptEnvironment &V, const ClptFrame &F, int x, int y, unsigned pixel, unsigned sample, bool aov,
                                           Counters &cn_in, int sub, int log2_k) {
    Counters scratch = { 0, 0, 0, 0, 0, 0 };
    Counters &cn = (SHARE && sub != 0) ? scratch : cn_in; // shading is counted once per ray
    V3 o, d;
    primary_ray(F, x, y, pixel, sample, o, d);
    if (MODE == 3) { // mode 2's loop with the light samples and MIS weights
        V3 Lsum = mk(0.0f, 0.0f, 0.0f), T = mk(1.0f, 1.0f, 1.0f);
        bool mis = false; // the last bounce was a diffuse one that did not fall back to the normal
        float pb = 0.0f;  // ... and its density (1 - p) cos / pi
        for (int seg = 0; seg < F.depth; seg++) {
            const Hit h = scene_hit<COUNT, SHARE, INST>(S, I, o, d, F.max_leaf_visits, cn_in, sub, log2_k);
            if (seg == 0 && aov) write_hit_aov<COUNT, INST>(S, I, F, h, o, d, x, y);
            if (h.ref < 0) {
                if (ENV) Lsum = vadd(Lsum, env_miss<true>(V, d, T, mis, pb));
                else Lsum = vadd(Lsum, T);
                break;
            }
            const V3 nrm = shading_normal<COUNT, INST>(S, I, h, o, d, cn);
            float al[3] = { 0.5f, 0.5f, 0.5f }, em[3] = { 0.0f, 0.0f, 0.0f };
            int kind = 0;
            if (S.n_materials > 0) {
                int m;
                if (INST == 1 && h.inst >= 0) m = I.rec[h.inst].material;
                else if (INST == 2 && h.inst >= 0) m = I.crec[h.inst].material;
                else m = S.tri_material ? __ldg(S.tri_material + __float_as_int(__ldg(&S.tri[3 * (size_t)h.ref].w))) : 0;
                if (m < 0 || m >= S.n_materials) m = 0;
                const ClptMaterial *mp = S.materials + m;
                al[0] = mp->albedo[0]; al[1] = mp->albedo[1]; al[2] = mp->albedo[2];
                em[0] = mp->emission[0]; em[1] = mp->emission[1]; em[2] = mp->emission[2];
                kind = mp->kind;
            }
            V3 e = mk(fmul(T.x, em[0]), fmul(T.y, em[1]), fmul(T.z, em[2]));
            if (mis && !(INST != 0 && h.inst >= 0)) {
                const int k = __ldg(E.map + __float_as_int(__ldg(&S.tri[3 * (size_t)h.ref].w)));
                if (k >= 0) e = vscale(e, bsdf_weight(E, k, d, h.t, pb));
            }
            Lsum = vadd(Lsum, e);
            T = mk(fmul(T.x, al[0]), fmul(T.y, al[1]), fmul(T.z, al[2]));
            const V3 hp = vadd(o, vscale(d, h.t));
            V3 nd;
            if (kind == 1) {
                nd = vnormalize(vsub(d, vscale(nrm, fmul(2.0f, vdot(d, nrm)))));
                mis = false;
            } else {
                if (seg + 1 < F.depth && __ldg(E.header + 1) > 0ull)
                    Lsum = vadd(Lsum, light_sample<COUNT, SHARE, INST>(S, I, E, F, hp, nrm, T, pixel, sample, (unsigned)seg,
                                                                       cn_in, sub, log2_k));
                if (ENV && seg + 1 < F.depth && __ldg(V.header + 1) > 0ull)
                    Lsum = vadd(Lsum, env_sample<COUNT, SHARE, INST>(S, I, V, F, hp, nrm, T, pixel, sample, (unsigned)seg,
                                                                     cn_in, sub, log2_k));
                bool fell_back;
                nd = cosine_dir(nrm, pixel, sample, (unsigned)seg, F.seed, fell_back);
                mis = !fell_back;
                pb = fmul(vdot(nd, nrm), CLPT_NEE_PB);
            }
            o = vadd(hp, vscale(nd, 0.0001f));
            d = nd;
        }
        return Lsum;
    }
    if (MODE == 2) {
        V3 Lsum = mk(0.0f, 0.0f, 0.0f), T = mk(1.0f, 1.0f, 1.0f);
        for (int seg = 0; seg < F.depth; seg++) {
            const Hit h = scene_hit<COUNT, SHARE, INST>(S, I, o, d, F.max_leaf_visits, cn_in, sub, log2_k);
            if (seg == 0 && aov) write_hit_aov<COUNT, INST>(S, I, F, h, o, d, x, y);
            if (h.ref < 0) {
                if (ENV) Lsum = vadd(Lsum, env_miss<false>(V, d, T, false, 0.0f));
                else Lsum = vadd(Lsum, T);
                break;
            }
            const V3 nrm = shading_normal<COUNT, INST>(S, I, h, o, d, cn);
            float al[3] = { 0.5f, 0.5f, 0.5f }, em[3] = { 0.0f, 0.0f, 0.0f };
            int kind = 0;
            if (S.n_materials > 0) {
                int m;
                if (INST == 1 && h.inst >= 0) m = I.rec[h.inst].material;
                else if (INST == 2 && h.inst >= 0) m = I.crec[h.inst].material;
                else m = S.tri_material ? __ldg(S.tri_material + __float_as_int(__ldg(&S.tri[3 * (size_t)h.ref].w))) : 0;
                if (m < 0 || m >= S.n_materials) m = 0;
                const ClptMaterial *mp = S.materials + m;
                al[0] = mp->albedo[0]; al[1] = mp->albedo[1]; al[2] = mp->albedo[2];
                em[0] = mp->emission[0]; em[1] = mp->emission[1]; em[2] = mp->emission[2];
                kind = mp->kind;
            }
            Lsum = vadd(Lsum, mk(fmul(T.x, em[0]), fmul(T.y, em[1]), fmul(T.z, em[2])));
            T = mk(fmul(T.x, al[0]), fmul(T.y, al[1]), fmul(T.z, al[2]));
            const V3 hp = vadd(o, vscale(d, h.t));
            V3 nd;
            if (kind == 1) {
                nd = vnormalize(vsub(d, vscale(nrm, fmul(2.0f, vdot(d, nrm)))));
            } else {
                nd = cosine_dir(nrm, pixel, sample, (unsigned)seg, F.seed);
            }
            o = vadd(hp, vscale(nd, 0.0001f));
            d = nd;
        }
        return Lsum;
    }
    // modes A/B: kernel.cl:296-422 with the tail recursion as a loop
    V3 col = mk(0.0f, 0.0f, 0.0f);
    float str = 1.0f;
    int depth = F.depth;
    if (MODE == 0) depth = depth > 0 ? 1 : 0;
    const int first_depth = depth;
    for (; depth > 0; depth--) {
        const Hit h = scene_hit<COUNT, SHARE, INST>(S, I, o, d, F.max_leaf_visits, cn_in, sub, log2_k);
        if (depth == first_depth && aov) write_hit_aov<COUNT, INST>(S, I, F, h, o, d, x, y);
        if (h.ref < 0) break;
        const V3 nrm = shading_normal<COUNT, INST>(S, I, h, o, d, cn);
        // (n + 1) / 2 (:395): halving is exact in binary floating point, so the product by 0.5 is the
        // quotient by 2 bit for bit -- and one instruction instead of an IEEE division
        const V3 nc = mk(fmul(fadd(nrm.x, 1.0f), 0.5f), fmul(fadd(nrm.y, 1.0f), 0.5f),
                         fmul(fadd(nrm.z, 1.0f), 0.5f));
        if (MODE == 0) return nc; // the `return` at :396
        V3 no = vadd(o, vscale(d, h.t));
        const V3 nd = vnormalize(vsub(d, vscale(nrm, fmul(2.0f, vdot(d, nrm)))));
        no = vadd(no, vscale(nd, 0.0001f));
        col = vadd(vscale(col, fsub(1.0f, str)), vscale(nc, str));
        str = fmul(str, 0.2f);
        o = no;
        d = nd;
    }
    const float k = fsub(1.0f, str); // :421
    return mk(fadd(fmul(k, col.x), str), fadd(fmul(k, col.y), str), fadd(fmul(k, col.z), str));
}

// Barrier among the G warps that share a pixel (__syncwarp for G = 1).  Named barriers 1-4,
// one per group, with IMMEDIATE ids: a barrier id held in a register makes ptxas reserve all
// 16 barriers for the block, and barriers are an occupancy limit like registers
// (launch__occupancy_limit_barriers) -- 16 per block allowed 4 resident blocks instead of 8
// and cost 40% of the frame rate (profiles/r02_experiments.json).
__device__ __forceinline__ void group_sync(int log2_g, int group) {
    if (log2_g == 0) {
        __syncwarp();
        return;
    }
    const int threads = 32 << log2_g;
    switch (group) {
    case 0: asm volatile("bar.sync 1, %0;" ::"r"(threads) : "memory"); break;
    case 1: asm volatile("bar.sync 2, %0;" ::"r"(threads) : "memory"); break;
    case 2: asm volatile("bar.sync 3, %0;" ::"r"(threads) : "memory"); break;
    default: asm volatile("bar.sync 4, %0;" ::"r"(threads) : "memory"); break;
    }
}

// VARIANT 0: compiled for 8 resident blocks per SM (engine 1).  1: the same code for
// CLPT_FAT_MIN_BLOCKS (engine 2, trees with fat leaves).  INST 1 (list) or 2 (tree): walks the
// instances of I after the base scene; INST 0 ignores I and is the kernel of a frame without instances.
// ENV (modes 2 and 3, launched only while an environment is set): reads the environment V.
template <int MODE, bool COUNT, int VARIANT, int INST, bool ENV = false>
__global__ void __launch_bounds__(256, VARIANT == 1 ? CLPT_FAT_MIN_BLOCKS : CLPT_MIN_BLOCKS)
render_kernel(const __grid_constant__ ClptScene S, const __grid_constant__ ClptFrame F,
              const __grid_constant__ ClptInstances I, const __grid_constant__ ClptEmitters E,
              const __grid_constant__ ClptEnvironment V) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int log2_s = F.log2_sample_lanes, s_lanes = 1 << log2_s;
    // Warps per pixel.  At >= 64 spp a pixel's samples are spread over G = 2, 4 or 8 warps of
    // the block (32 samples each, side by side) instead of being walked by one warp in
    // several rounds: a claim is then 1/G as long, which is what the END of a frame is made
    // of (the last claims run while the rest of the GPU idles; on 8 GPUs a frame is only
    // ~27 claims per warp long).  The warps of a group share the claim and the staging
    // rows; the group's first warp does the ordered sum.  G = 1 is the plain scheme.
    const int log2_g = F.log2_warps_per_pixel, g_warps = 1 << log2_g;
    const int group = warp >> log2_g, member = warp & (g_warps - 1);
    // Lanes per ray (engine 2 at one sample per pixel only, clpt_trace.cuh: triangle_run_shared):
    // 1 << log2_r neighbouring lanes walk the same ray, a warp tile is 32 >> log2_r pixels.
    const int log2_r = VARIANT == 1 ? F.log2_lanes_per_ray : 0;
    const int sub = lane & ((1 << log2_r) - 1);
    int tw, th;
    warp_tile_dims(5 - log2_s - log2_r, tw, th);
    const int pslot = lane >> (log2_s + log2_r), sslot = (lane >> log2_r) & (s_lanes - 1);
    const int spp = F.spp < 1 ? 1 : F.spp;
    const int group_base = lane & ~(s_lanes - 1);
    Counters cn = { 0, 0, 0, 0, 0, 0 };
    // Ordered per-pixel sum.  The colours of a round are staged in shared memory and
    // summed in ascending sample order by one lane per channel (lane c of the pixel's
    // group sums channel c; with fewer than 4 lanes per pixel, lane 0 sums all three).
    // Same additions in the same order as a serial loop over the samples.
    // Rows: [warp group][channel][32 * G samples + 1], padded against bank conflicts.
    __shared__ float stage[8 * 3 * 33];
    const int row_len = 32 * g_warps + 1;
    float *const my_stage = stage + group * 3 * row_len; // this group's three channel rows
    const int my_col = member * 32 + lane;               // this lane's column in them
    const bool per_channel = s_lanes >= 4;
    const bool accumulate = (F.flags & CLPT_F_ACCUMULATE) != 0;
    // Persistent warps: the grid only fills the machine; every warp (group) claims warp tiles
    // from a global counter until none are left.  Blocks cost anything from nothing
    // (sky) to hundreds of microseconds (grazing ground), and with one tile per warp
    // fixed at launch the last heavy blocks left most SMs idle at the end of a frame
    // (40% idle on a 4 ms frame).  Tile t = ((by * tiles_x + bx) * 8 + w): the same
    // 4 x 2 arrangement of warp tiles as a block of the static mapping, so
    // consecutive claims are neighbours on screen.
    // Claim direction.  A warp tile is a whole pixel's samples and bounces (up to ~1 ms of
    // one warp), so a frame whose most expensive tiles are claimed LATE ends with a few
    // warps busy for ~0.9 ms while the rest of the GPU idles: 2% of a 37 ms frame, 13% of
    // one GPU's share of it on 8 GPUs.  CLExecute therefore measures where the cost of a
    // frame sits (row_cost) and has the next one start from the end nearer to its costliest
    // rows.  Screen order is kept either way: neighbouring claims stay neighbours in the
    // tree (sorting rows by cost outright was measured and loses more in locality than it
    // wins, profiles/r01_experiments.json).
    __shared__ unsigned tile_t0[8], tile_row[8], tile_claim[8]; // kept out of registers across the trace
    const unsigned bx_count = (unsigned)F.blocks_x, n_tiles = (unsigned)F.n_warp_tiles;
    for (;;) {
        unsigned t = 0;
        if (lane == 0 && member == 0) {
            t = atomicAdd(F.work_counter, 1u);
            tile_t0[warp] = (unsigned)clock();
            tile_claim[group] = t;
        }
        if (log2_g == 0) {
            t = __shfl_sync(0xffffffffu, t, 0);
        } else {
            group_sync(log2_g, group);
            t = tile_claim[group];
        }
        if (t >= n_tiles) break;
        if (F.flags & CLPT_F_REVERSE) t = n_tiles - 1u - t;
        const unsigned w = t & 7u, b = t >> 3;
        const int bx = (int)(b % bx_count), by = (int)(b / bx_count);
        if (lane == 0 && member == 0) tile_row[warp] = (unsigned)by;
        const int x = (bx * 4 + (int)(w & 3u)) * tw + (pslot & (tw - 1));
        const int ly = (by * 2 + (int)(w >> 2)) * th + pslot / tw; // row within this rank's slab
        const int y = slab_row_to_image_row(F, ly);
        const bool valid = x < F.width && y < F.height && ly < F.local_rows;
        const unsigned pixel = (unsigned)(y * F.width + x);
        V3 acc = mk(0.0f, 0.0f, 0.0f); // per_channel: only .x is used, for channel `sslot`
        // progressive frames sum the samples in 2^-32 fixed point (order-free, see ClptFrame::accum)
        unsigned long long fx = 0ull, fy = 0ull, fz = 0ull; // per_channel: only fx is used
        const int round_samples = s_lanes << log2_g;
        for (int base = 0; base < spp; base += round_samples) {
            const int s = base + (member << log2_s) + sslot; // (member > 0 only when s_lanes == 32)
            V3 colour = mk(0.0f, 0.0f, 0.0f);
            if (valid && s == 0 && sub == 0 && F.aov_prim != nullptr && F.depth <= 0) {
                // nothing is traced: the AOVs say "miss" instead of keeping the previous frame's
                Hit none;
                none.ref = -1;
                none.t = 0.0f;
                write_aov<COUNT>(S, F, none, mk(0.0f, 0.0f, 0.0f), mk(0.0f, 0.0f, 0.0f), x, y);
            }
            const int in_round = min(round_samples, spp - base);
            if (valid && s < spp) {
                colour = trace_sample<MODE, COUNT, VARIANT == 1, INST, ENV>(S, I, E, V, F, x, y, pixel, F.sample_base + (unsigned)s,
                                                                 s == 0 && sub == 0 && F.aov_prim != nullptr, cn, sub,
                                                                 log2_r);
            }
            my_stage[0 * row_len + my_col] = colour.x;
            my_stage[1 * row_len + my_col] = colour.y;
            my_stage[2 * row_len + my_col] = colour.z;
            group_sync(log2_g, group);
            if (member == 0) {
                if (per_channel) {
                    if (sslot < 3) {
                        const float *src = my_stage + sslot * row_len + group_base;
                        if (accumulate) {
                            for (int j = 0; j < in_round; j++) fx += clpt_fix32(src[j]);
                        } else {
                            for (int j = 0; j < in_round; j++) acc.x = fadd(acc.x, src[j]);
                        }
                    }
                } else if (sslot == 0) {
                    for (int j = 0; j < in_round; j++) {
                        const V3 c = mk(my_stage[0 * row_len + group_base + j], my_stage[1 * row_len + group_base + j],
                                        my_stage[2 * row_len + group_base + j]);
                        if (accumulate) {
                            fx += clpt_fix32(c.x);
                            fy += clpt_fix32(c.y);
                            fz += clpt_fix32(c.z);
                        } else {
                            acc = vadd(acc, c);
                        }
                    }
                }
            }
            group_sync(log2_g, group);
        }
        if (member == 0) {
            if (per_channel) { // bring the three channel sums to the group's first lane
                if (accumulate) {
                    fy = __shfl_sync(0xffffffffu, fx, group_base + 1);
                    fz = __shfl_sync(0xffffffffu, fx, group_base + 2);
                    fx = __shfl_sync(0xffffffffu, fx, group_base);
                } else {
                    const float r = __shfl_sync(0xffffffffu, acc.x, group_base);
                    const float g = __shfl_sync(0xffffffffu, acc.x, group_base + 1);
                    const float bl = __shfl_sync(0xffffffffu, acc.x, group_base + 2);
                    acc = mk(r, g, bl);
                }
            }
            if (valid && sslot == 0 && sub == 0) {
                if (accumulate) accumulate_pixel(F, x, y, fx, fy, fz, spp);
                else store_pixel(F, x, ly, acc, spp);
            }
            if (lane == 0 && F.row_cost) {
                const unsigned long long took = (unsigned long long)((unsigned)clock() - tile_t0[warp]);
                atomicAdd(F.row_cost + tile_row[warp], took);
                atomicMax(F.row_cost + F.row_count + tile_row[warp], took);
            }
        }
    }
    if (COUNT) {
        unsigned v[6] = { cn.rays, cn.splits, cn.leaves, cn.tris, cn.shade_vn, cn.capped };
#pragma unroll
        for (int k = 0; k < 6; k++) {
            unsigned sum = v[k];
            for (int off = 16; off > 0; off >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, off);
            if (lane == 0 && sum) atomicAdd(F.counters + k, (unsigned long long)sum);
        }
    }
}

// Gathered slabs [rank][slab_rows][width] -> image rows.
template <typename PX>
__global__ void deinterleave_kernel(const PX *__restrict__ gathered, PX *__restrict__ image,
                                    int width, int height, int nranks, int tile_rows,
                                    int slab_rows) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)width * height) return;
    const int y = (int)(i / width), x = (int)(i - (size_t)y * width);
    const int t = y / tile_rows, r = t % nranks, lt = t / nranks;
    const int ly = lt * tile_rows + (y - t * tile_rows);
    image[i] = gathered[((size_t)r * slab_rows + ly) * width + x];
}

__global__ void fill_kernel(float4 *dst, size_t n, float value) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = make_float4(value, value, value, value);
}

// Progressive target (fixed-point sums + sample count) -> displayable average.
__global__ void normalise_kernel(const unsigned long long *__restrict__ accum, float4 *__restrict__ dst, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ulonglong2 rg = reinterpret_cast<const ulonglong2 *>(accum)[2 * i], bn = reinterpret_cast<const ulonglong2 *>(accum)[2 * i + 1];
    if (bn.y > 0ull) {
        const double k = (double)bn.y * 4294967296.0; // (one IEEE division per channel, as the oracle's mean)
        dst[i] = make_float4((float)((double)rg.x / k), (float)((double)rg.y / k), (float)((double)bn.x / k), 1.0f);
    } else {
        dst[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
}

__global__ void fill_u64_kernel(unsigned long long *dst, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = 0ull;
}

// Displayable float4 frame -> RGBA8 UNORM texels, the format of the reference's render
// target (src/GLHandler.c:177-185): what write_imagef does to a CL_UNORM_INT8 image,
// clamp to [0,1], scale by 255, round to nearest even.
__global__ void pack_rgba8_kernel(const float4 *__restrict__ src, uchar4 *__restrict__ dst, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 c = src[i];
    dst[i] = make_uchar4((unsigned char)clpt_to_unorm8(c.x), (unsigned char)clpt_to_unorm8(c.y),
                         (unsigned char)clpt_to_unorm8(c.z), (unsigned char)clpt_to_unorm8(c.w));
}

// One block, one thread per rank.  The stores of the kernels before this one on the stream
// (pixels placed into the peers' frames) are ordered before the signal by the system-scope
// fence + release store; the acquire load orders the peers' pixels before whatever follows.
__global__ void flag_barrier_kernel(const __grid_constant__ ClptFlagPeers peers, int rank, int nranks,
                                    unsigned int epoch) {
    const int r = threadIdx.x;
    if (r >= nranks) return;
    __threadfence_system();
    unsigned int *signal = peers.flags[r] + rank * 8;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(signal), "r"(epoch) : "memory");
    const unsigned int *wait = peers.flags[rank] + r * 8;
    unsigned int seen;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(wait) : "memory");
    } while ((int)(seen - epoch) < 0);
}

template <int MODE, int INST, bool ENV>
void launch_variant(const ClptScene &scene, const ClptFrame &frame, const ClptInstances &inst, const ClptEmitters &emit,
                    const ClptEnvironment &env, unsigned grid, cudaStream_t stream) {
    const bool fat = (frame.flags & CLPT_F_FAT) != 0;
    if (frame.flags & CLPT_F_COUNTERS) {
        if (fat) render_kernel<MODE, true, 1, INST, ENV><<<grid, 256, 0, stream>>>(scene, frame, inst, emit, env);
        else render_kernel<MODE, true, 0, INST, ENV><<<grid, 256, 0, stream>>>(scene, frame, inst, emit, env);
    } else {
        if (fat) render_kernel<MODE, false, 1, INST, ENV><<<grid, 256, 0, stream>>>(scene, frame, inst, emit, env);
        else render_kernel<MODE, false, 0, INST, ENV><<<grid, 256, 0, stream>>>(scene, frame, inst, emit, env);
    }
}

template <int MODE, bool ENV = false>
void launch_mode(const ClptScene &scene, const ClptFrame &frame, const ClptInstances &inst, const ClptEmitters &emit,
                 const ClptEnvironment &env, unsigned grid, cudaStream_t stream) {
    if (inst.count > 0 && inst.tree) launch_variant<MODE, 2, ENV>(scene, frame, inst, emit, env, grid, stream);
    else if (inst.count > 0) launch_variant<MODE, 1, ENV>(scene, frame, inst, emit, env, grid, stream);
    else launch_variant<MODE, 0, ENV>(scene, frame, inst, emit, env, grid, stream);
}

} // namespace

int clpt_render_block_rows(const ClptFrame &frame) {
    int tw, th;
    warp_tile_dims(5 - frame.log2_sample_lanes - ((frame.flags & CLPT_F_FAT) ? frame.log2_lanes_per_ray : 0), tw, th);
    const int block_h = 2 * th;
    return (frame.local_rows + block_h - 1) / block_h;
}

int clpt_render_blocks_per_sm(int engine) { return engine == 2 ? CLPT_FAT_MIN_BLOCKS : CLPT_MIN_BLOCKS; }

void clpt_launch_render(const ClptScene &scene, const ClptFrame &frame_in, const ClptInstances &inst,
                        const ClptEmitters &emit, const ClptEnvironment &env, int sm_count, cudaStream_t stream) {
    ClptFrame frame = frame_in;
    if (!(frame.flags & CLPT_F_FAT)) frame.log2_lanes_per_ray = 0;
    int tw, th;
    warp_tile_dims(5 - frame.log2_sample_lanes - frame.log2_lanes_per_ray, tw, th);
    const int block_w = 4 * tw, block_h = 2 * th;
    const unsigned bx = (unsigned)((frame.width + block_w - 1) / block_w);
    const unsigned by = (unsigned)((frame.local_rows + block_h - 1) / block_h);
    if (bx == 0 || by == 0) return;
    frame.blocks_x = (int)bx;
    frame.n_warp_tiles = (int)(bx * by * 8u);
    // persistent grid: enough blocks to fill every SM, never more than there are tiles
    unsigned grid = (unsigned)sm_count * ((frame.flags & CLPT_F_FAT) ? CLPT_FAT_MIN_BLOCKS : CLPT_MIN_BLOCKS);
    if (grid > bx * by) grid = bx * by;
    cudaMemsetAsync(frame.work_counter, 0, sizeof(unsigned), stream);
    switch (frame.mode) {
    case 0: launch_mode<0>(scene, frame, inst, emit, env, grid, stream); break;
    case 1: launch_mode<1>(scene, frame, inst, emit, env, grid, stream); break;
    case 2:
        if (env.n > 0) launch_mode<2, true>(scene, frame, inst, emit, env, grid, stream);
        else launch_mode<2>(scene, frame, inst, emit, env, grid, stream);
        break;
    default:
        if (env.n > 0) launch_mode<3, true>(scene, frame, inst, emit, env, grid, stream);
        else launch_mode<3>(scene, frame, inst, emit, env, grid, stream);
        break;
    }
}

void clpt_launch_deinterleave(const float4 *gathered, float4 *image, int width, int height,
                              int nranks, int tile_rows, int slab_rows, cudaStream_t stream) {
    const size_t n = (size_t)width * height;
    if (n == 0) return;
    deinterleave_kernel<float4><<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(gathered, image, width, height,
                                                                                 nranks, tile_rows, slab_rows);
}

void clpt_launch_fill(float4 *dst, size_t n, float value, cudaStream_t stream) {
    if (n == 0) return;
    fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(dst, n, value);
}

void clpt_launch_normalise(const unsigned long long *accum, float4 *dst, size_t n, cudaStream_t stream) {
    if (n == 0) return;
    normalise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(accum, dst, n);
}

void clpt_launch_fill_u64(unsigned long long *dst, size_t n, cudaStream_t stream) {
    if (n == 0) return;
    fill_u64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(dst, n);
}

void clpt_launch_flag_barrier(const ClptFlagPeers &peers, int rank, int nranks, unsigned int epoch,
                              cudaStream_t stream) {
    flag_barrier_kernel<<<1, 32, 0, stream>>>(peers, rank, nranks, epoch);
}

void clpt_launch_pack_rgba8(const float4 *src, uchar4 *dst, size_t n, cudaStream_t stream) {
    if (n == 0) return;
    pack_rgba8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(src, dst, n);
}

const void *clpt_render_kernel_symbol(void) {
    return reinterpret_cast<const void *>(&render_kernel<0, false, 0, 0>);
}
