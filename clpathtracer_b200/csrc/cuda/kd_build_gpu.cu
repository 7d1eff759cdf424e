// kd_build_gpu.cu -- kd-tree construction on the device (SURVEY.md section 8f row 1).
//
// The reference builds its tree on one host core (src/kd_tree.c:95-200, ~20 s for a
// million triangles) and this library's host builders (csrc/host/kd_build.c) on all of
// them (~1 s).  For scenes that change every frame (BASELINE config 5) even that is the
// frame: this file builds the tree where the triangles already are.
//
// Level-synchronous binned SAH, one pass over the references per level:
//   bin      every reference adds its bounds to its node's 3 x 2 x 32 histograms
//            (where a bound starts, where it ends; shared-memory copy for the node a
//            block starts in, so the few huge nodes of the top levels do not serialise)
//   choose   one warp per node: prefix sums over the bins, the surface-area heuristic
//            cost(plane) = Ct + Ci (SA(L) NL + SA(R) NR) / SA(cell), x empty_bonus when a
//            side is empty (the same cost as build_kd_sah, kd_build.c), leaf when no plane
//            beats Ci N
//   scan     three running counts over the references (goes left, goes right, stays in a
//            finished leaf) -- the references of a node are contiguous and keep their
//            order, so the counts place every reference of the next level without
//            atomics: the tree and the order of the triangles inside each leaf (which
//            decides ties, src/kernel.cl:344) are DETERMINISTIC, and every GPU of a node
//            builds the same bytes from the same mesh
//   emit     split and leaf records in the reference's 68-byte wire format
//            (include/kd_tree.h:31-50), children two by two, ropes inherited from the
//            parent (src/kd_tree.c:64-83)
// and after the last level one thread per leaf face pushes its rope down to the deepest
// node that still covers the face (kd_build.c: push_down_link, full).
//
// A level is seven launches (bin, choose, three for the two scans, split = emit + scatter,
// commit); every kernel reads the level's counts from a LevelState in device memory.  Two
// drivers share them (clpt_gpu_build): small meshes replay ONE recorded CUDA graph of all
// levels with capacity-sized launches and synchronise once per build; big meshes go level
// by level with two totals read back per level to size the next one exactly.
//
// The output is the wire format ON THE DEVICE; the second half of this file turns it into
// the traversal layout without leaving the device, and CLDownloadKd hands it to a host that
// wants to look at it (the parity tests walk it with the oracle).
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "CLHandler.h"
#include "clpt_device.cuh"
#include "kd_build_gpu.h"

#define CU(call) handle_err((int)(call), __FILE__, __LINE__)

namespace {

constexpr int NBINS = 32;
// Nodes with at most this many references do not use the binned planes: every bound of
// every reference is a candidate plane, evaluated exactly by the node's warp (two
// references per lane).  Planes on triangle bounds separate neighbours without cutting
// them; uniform bins in a small cell almost never do (measured on the heightfields: 6.4x
// triangle references with bins only, 1.5x with exact candidates, like build_kd_sah).
constexpr int EXACT_MAX = 64;
constexpr int SCAN_BLOCK = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_BLOCK * SCAN_ITEMS;

// A node of the level being split.
struct ANode {
    float mn[3], mx[3];
    int begin, count; // its references: [begin, begin + count) of the level's reference array
    int out;          // index of its record in the wire array
    int links[6];     // neighbour across each face (wire node index, -1 = outside), not yet pushed down
    int depth_left;
    int hist_slot;    // its histograms (nodes with more than EXACT_MAX references only), else -1
};

struct Decision { // what `choose` decided for a node
    float plane;
    int axis;      // -1: the node becomes a leaf
    int rank;      // exclusive rank among this level's splits (filled by the scan over nodes)
};

struct Triple {
    unsigned l, r, f;
};

// The counts of the level being split, ON THE DEVICE: every kernel of a level reads them from here,
// so a whole build can be enqueued (or replayed as a CUDA graph) without the host knowing them.
struct LevelState {
    int n_nodes, n_refs;       // this level
    int n_out, n_leaf_refs;    // wire nodes allocated / leaf references written so far
    int overflow;              // a capacity was exceeded: the build stopped, the host falls back
    int levels;                // levels that had nodes
    int pad[10];
};
__host__ __device__ inline Triple operator+(Triple a, Triple b) { return Triple{ a.l + b.l, a.r + b.r, a.f + b.f }; }

// ---- bounds of every triangle (SoA) ---------------------------------------------------
__global__ void tri_bounds_kernel(const float4 *__restrict__ verts, const int4 *__restrict__ corners, int n_tris,
                                  int n_verts, float *__restrict__ lo, float *__restrict__ hi, int *__restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tris) return;
    const int a = corners[3 * (size_t)i].x, b = corners[3 * (size_t)i + 1].x, c = corners[3 * (size_t)i + 2].x;
    if (a < 0 || b < 0 || c < 0 || a >= n_verts || b >= n_verts || c >= n_verts) {
        atomicExch(bad, 1);
        return;
    }
    const float4 A = verts[a], B = verts[b], C = verts[c];
    lo[i] = fminf(fminf(A.x, B.x), C.x);
    hi[i] = fmaxf(fmaxf(A.x, B.x), C.x);
    lo[n_tris + i] = fminf(fminf(A.y, B.y), C.y);
    hi[n_tris + i] = fmaxf(fmaxf(A.y, B.y), C.y);
    lo[2 * (size_t)n_tris + i] = fminf(fminf(A.z, B.z), C.z);
    hi[2 * (size_t)n_tris + i] = fmaxf(fmaxf(A.z, B.z), C.z);
}

// Scene box: min/max over the triangle bounds.  Floats compare like their sign-adjusted
// integer images, so the reduction is integer atomics (exact, order-independent).
__device__ __forceinline__ int float_key(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__global__ void scene_box_kernel(const float *__restrict__ lo, const float *__restrict__ hi, int n_tris,
                                 int *__restrict__ box_keys /* [6]: min xyz, max xyz */) {
    int mn[3] = { INT_MAX, INT_MAX, INT_MAX }, mx[3] = { INT_MIN, INT_MIN, INT_MIN };
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tris; i += gridDim.x * blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; a++) {
            mn[a] = min(mn[a], float_key(lo[(size_t)a * n_tris + i]));
            mx[a] = max(mx[a], float_key(hi[(size_t)a * n_tris + i]));
        }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
        for (int off = 16; off > 0; off >>= 1) {
            mn[a] = min(mn[a], __shfl_down_sync(0xffffffffu, mn[a], off));
            mx[a] = max(mx[a], __shfl_down_sync(0xffffffffu, mx[a], off));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(box_keys + a, mn[a]);
            atomicMax(box_keys + 3 + a, mx[a]);
        }
    }
}

__global__ void root_kernel(const int *__restrict__ box_keys, int n_tris, int max_depth, ANode *__restrict__ nodes,
                            int *__restrict__ ref_tri, int *__restrict__ ref_node, LevelState *__restrict__ ls,
                            int *__restrict__ big_counter) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        *big_counter = 0; // (was the bad-mesh flag of tri_bounds, already on its way to the host)
        LevelState st = {};
        st.n_nodes = 1;
        st.n_refs = n_tris;
        st.n_out = 1;
        *ls = st;
        ANode r;
        for (int a = 0; a < 3; a++) {
            r.mn[a] = key_float(box_keys[a]);
            r.mx[a] = key_float(box_keys[3 + a]);
        }
        r.begin = 0;
        r.count = n_tris;
        r.out = 0;
        for (int f = 0; f < 6; f++) r.links[f] = -1;
        r.depth_left = max_depth;
        r.hist_slot = n_tris > EXACT_MAX ? 0 : -1;
        nodes[0] = r;
    }
    if (i < n_tris) {
        ref_tri[i] = i;
        ref_node[i] = 0;
    }
}

// ---- bin -------------------------------------------------------------------------------
__device__ __forceinline__ int bin_of(float x, float mn, float scale) {
    const int b = __float2int_rd((x - mn) * scale); // NaN -> 0, saturates
    return min(max(b, 0), NBINS - 1);
}

__global__ void __launch_bounds__(256)
bin_kernel(const LevelState *__restrict__ ls, const ANode *__restrict__ nodes, const int *__restrict__ ref_tri,
           const int *__restrict__ ref_node, const float *__restrict__ lo, const float *__restrict__ hi, int n_tris,
           int min_split, unsigned *__restrict__ hist /* [node][axis][start|end][bin] */) {
    __shared__ unsigned local[3 * 2 * NBINS];
    __shared__ int home; // histogram slot of the node this block's first reference belongs to (-1: a small node)
    const int n_refs = ls->n_refs;
    const int first = blockIdx.x * blockDim.x;
    if (first >= n_refs) return; // (uniform per block)
    if (threadIdx.x == 0) home = nodes[ref_node[min(first, n_refs - 1)]].hist_slot;
    for (int k = threadIdx.x; k < 3 * 2 * NBINS; k += blockDim.x) local[k] = 0;
    __syncthreads();
    const int i = first + threadIdx.x;
    if (i < n_refs) {
        const int a = ref_node[i];
        const ANode &nd = nodes[a];
        if (nd.hist_slot >= 0 && nd.count >= min_split && nd.depth_left > 0) {
            const int t = ref_tri[i];
            unsigned *dst = nd.hist_slot == home ? local : hist + (size_t)nd.hist_slot * (3 * 2 * NBINS);
#pragma unroll
            for (int ax = 0; ax < 3; ax++) {
                const float ext = nd.mx[ax] - nd.mn[ax];
                const float scale = ext > 0.0f ? (float)NBINS / ext : 0.0f;
                const int bs = bin_of(lo[(size_t)ax * n_tris + t], nd.mn[ax], scale);
                const int be = bin_of(hi[(size_t)ax * n_tris + t], nd.mn[ax], scale);
                atomicAdd(dst + (ax * 2 + 0) * NBINS + bs, 1u);
                atomicAdd(dst + (ax * 2 + 1) * NBINS + be, 1u);
            }
        }
    }
    __syncthreads();
    if (home < 0) return;
    unsigned *dst = hist + (size_t)home * (3 * 2 * NBINS);
    for (int k = threadIdx.x; k < 3 * 2 * NBINS; k += blockDim.x) {
        if (local[k]) atomicAdd(dst + k, local[k]);
    }
}

// ---- choose ----------------------------------------------------------------------------
__device__ __forceinline__ float box_area(float ex, float ey, float ez) { return 2.0f * (ex * ey + ey * ez + ez * ex); }

// Lower cost first; among equal costs the lower axis, then the lower plane: a total order, so the
// choice does not depend on which lane or bin proposed it.
__device__ __forceinline__ bool better(float c, int ax, float p, float bc, int bax, float bp) {
    return c < bc || (c == bc && (ax < bax || (ax == bax && p < bp)));
}

__device__ __forceinline__ float sah_cost(const float *ext, int ax, float left_extent, int nl, int nr, int n, float ct,
                                          float ci, float empty_bonus, float inv_area) {
    if (nl == n && nr == n) return 3.0e38f; // a plane that leaves everything on both sides separates nothing
    float el[3] = { ext[0], ext[1], ext[2] }, er[3] = { ext[0], ext[1], ext[2] };
    el[ax] = left_extent;
    er[ax] = ext[ax] - left_extent;
    float cost = ct + ci * (box_area(el[0], el[1], el[2]) * (float)nl + box_area(er[0], er[1], er[2]) * (float)nr) * inv_area;
    if (nl == 0 || nr == 0) cost *= empty_bonus;
    return cost;
}

// W lanes per node.  W = 8 serves the nodes of at most SMALL_MAX references (four nodes per warp:
// near the leaves almost every node is that small, and a whole warp per node left most lanes
// idle -- the kernel was half of the build); W = 32 serves the rest, two references per lane above 32.
constexpr int SMALL_MAX = 8;

template <int W>
__device__ __forceinline__ void choose_nodes(int block, int n_blocks, const LevelState *__restrict__ ls,
                                             const ANode *__restrict__ nodes, unsigned *__restrict__ hist,
                                             const int *__restrict__ ref_tri, const float *__restrict__ lo,
                                             const float *__restrict__ hi, int n_tris, int min_split, float ct, float ci,
                                             float empty_bonus, Decision *__restrict__ decisions) {
    const int lane = threadIdx.x & 31, sub = lane & (W - 1);
    const unsigned mask = W == 32 ? 0xffffffffu : (((1u << W) - 1u) << (lane & ~(W - 1)));
    const int n_nodes = ls->n_nodes;
    const int groups = (int)(((size_t)n_blocks * blockDim.x) / W);
    // grid-stride over the nodes (whole groups move together: `a` is uniform in a group)
    for (int a = (int)(((size_t)block * blockDim.x + threadIdx.x) / W); a < n_nodes; a += groups) {
    const ANode nd = nodes[a];
    if ((W == 8) != (nd.count <= SMALL_MAX)) continue; // the other launch's node
    Decision d;
    d.axis = -1;
    d.plane = 0.0f;
    d.rank = 0;
    if (nd.count >= min_split && nd.depth_left > 0) {
        const float ext[3] = { nd.mx[0] - nd.mn[0], nd.mx[1] - nd.mn[1], nd.mx[2] - nd.mn[2] };
        const float area = box_area(ext[0], ext[1], ext[2]);
        const float inv_area = area > 0.0f ? 1.0f / area : 0.0f;
        float best = ci * (float)nd.count; // the cost of leaving the node a leaf
        int best_ax = -1;
        float best_plane = 0.0f;
        const bool exact = nd.hist_slot < 0;
        const bool two = W == 32 && nd.count > 32; // a second reference per lane
        const int t0 = exact && sub < nd.count ? ref_tri[nd.begin + sub] : -1;
        const int t1 = exact && two && sub + 32 < nd.count ? ref_tri[nd.begin + sub + 32] : -1;
        for (int ax = 0; ax < 3; ax++) {
            if (!(ext[ax] > 0.0f) || !(inv_area > 0.0f)) continue;
            float c = 3.0e38f, p = 0.0f; // this lane's best candidate on this axis
            if (exact) {
                // every bound of every reference is a candidate; a lane evaluates its own references' bounds
                const float l0 = t0 >= 0 ? lo[(size_t)ax * n_tris + t0] : 0.0f, h0 = t0 >= 0 ? hi[(size_t)ax * n_tris + t0] : 0.0f;
                float l1 = 0.0f, h1 = 0.0f;
                if (two && t1 >= 0) {
                    l1 = lo[(size_t)ax * n_tris + t1];
                    h1 = hi[(size_t)ax * n_tris + t1];
                }
                int nl0 = 0, nr0 = 0, nl1 = 0, nr1 = 0, nl2 = 0, nr2 = 0, nl3 = 0, nr3 = 0;
                const int first_n = nd.count < W ? nd.count : W;
                for (int j = 0; j < first_n; j++) {
                    const float lj = __shfl_sync(mask, l0, j, W), hj = __shfl_sync(mask, h0, j, W);
                    nr0 += hj > l0 ? 1 : 0;
                    nl0 += (lj < l0 || !(hj > l0)) ? 1 : 0;
                    nr1 += hj > h0 ? 1 : 0;
                    nl1 += (lj < h0 || !(hj > h0)) ? 1 : 0;
                    if (two) {
                        nr2 += hj > l1 ? 1 : 0;
                        nl2 += (lj < l1 || !(hj > l1)) ? 1 : 0;
                        nr3 += hj > h1 ? 1 : 0;
                        nl3 += (lj < h1 || !(hj > h1)) ? 1 : 0;
                    }
                }
                if (two) {
                    for (int j = 32; j < nd.count; j++) {
                        const float lj = __shfl_sync(mask, l1, j - 32, W), hj = __shfl_sync(mask, h1, j - 32, W);
                        nr0 += hj > l0 ? 1 : 0;
                        nl0 += (lj < l0 || !(hj > l0)) ? 1 : 0;
                        nr1 += hj > h0 ? 1 : 0;
                        nl1 += (lj < h0 || !(hj > h0)) ? 1 : 0;
                        nr2 += hj > l1 ? 1 : 0;
                        nl2 += (lj < l1 || !(hj > l1)) ? 1 : 0;
                        nr3 += hj > h1 ? 1 : 0;
                        nl3 += (lj < h1 || !(hj > h1)) ? 1 : 0;
                    }
                }
                const float cand[4] = { l0, h0, l1, h1 };
                const int nl[4] = { nl0, nl1, nl2, nl3 }, nr[4] = { nr0, nr1, nr2, nr3 };
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const bool present = k < 2 ? t0 >= 0 : t1 >= 0;
                    if (!present || !(cand[k] > nd.mn[ax] && cand[k] < nd.mx[ax])) continue;
                    const float ck = sah_cost(ext, ax, cand[k] - nd.mn[ax], nl[k], nr[k], nd.count, ct, ci, empty_bonus, inv_area);
                    if (ck < 3.0e38f && better(ck, ax, cand[k], c, ax, p)) {
                        c = ck;
                        p = cand[k];
                    }
                }
            } else if (W == 32) {
                unsigned *h = hist + (size_t)nd.hist_slot * (3 * 2 * NBINS);
                const unsigned s = h[(ax * 2 + 0) * NBINS + lane], e = h[(ax * 2 + 1) * NBINS + lane];
                // exclusive prefix sums: plane k (k = lane, 1..31) sits at the low edge of bin k
                unsigned ps = s, pe = e;
                for (int off = 1; off < 32; off <<= 1) {
                    const unsigned us = __shfl_up_sync(mask, ps, off), ue = __shfl_up_sync(mask, pe, off);
                    if (lane >= off) {
                        ps += us;
                        pe += ue;
                    }
                }
                const int nl = (int)(ps - s), nr = nd.count - (int)(pe - e);
                if (lane >= 1) {
                    const float left = ext[ax] * ((float)lane / (float)NBINS);
                    const float plane = nd.mn[ax] + left;
                    // the plane has to cut the cell strictly inside, or a child would be the cell again
                    if (plane > nd.mn[ax] && plane < nd.mx[ax]) {
                        c = sah_cost(ext, ax, left, nl, nr, nd.count, ct, ci, empty_bonus, inv_area);
                        p = plane;
                    }
                }
            }
            // argmin over the node's lanes under the total order
            for (int off = W / 2; off > 0; off >>= 1) {
                const float oc = __shfl_xor_sync(mask, c, off, W), op = __shfl_xor_sync(mask, p, off, W);
                if (better(oc, ax, op, c, ax, p)) {
                    c = oc;
                    p = op;
                }
            }
            if (c < best) { // strictly: among equal costs the lower axis keeps the choice
                best = c;
                best_ax = ax;
                best_plane = p;
            }
        }
        if (best_ax >= 0) {
            d.axis = best_ax;
            d.plane = best_plane;
        }
    }
    if (sub == 0) decisions[a] = d;
    // the histograms are left zeroed for the next level (they are cleared once per build, not per level)
    if (W == 32 && nd.hist_slot >= 0) {
        unsigned *h = hist + (size_t)nd.hist_slot * (3 * 2 * NBINS);
#pragma unroll
        for (int k = 0; k < 3 * 2; k++) h[k * NBINS + lane] = 0u;
    }
    }
}

// One launch for both widths: the first `blocks32` blocks serve the nodes of more than SMALL_MAX
// references, the rest the small ones.
__global__ void __launch_bounds__(256)
choose_kernel(int blocks32, const LevelState *__restrict__ ls, const ANode *__restrict__ nodes,
              unsigned *__restrict__ hist, const int *__restrict__ ref_tri, const float *__restrict__ lo,
              const float *__restrict__ hi, int n_tris, int min_split, float ct, float ci, float empty_bonus,
              Decision *__restrict__ decisions) {
    if ((int)blockIdx.x < blocks32) {
        choose_nodes<32>((int)blockIdx.x, blocks32, ls, nodes, hist, ref_tri, lo, hi, n_tris, min_split, ct, ci,
                         empty_bonus, decisions);
    } else {
        choose_nodes<8>((int)blockIdx.x - blocks32, (int)gridDim.x - blocks32, ls, nodes, hist, ref_tri, lo, hi, n_tris,
                        min_split, ct, ci, empty_bonus, decisions);
    }
}

// ---- scans -----------------------------------------------------------------------------
// Where a reference goes.  Left: its bound starts below the plane (or it lies in the
// plane); right: it ends above the plane.  Triangles that only touch the plane from one
// side stay on that side (kd_build.c, partition).
__device__ __forceinline__ Triple ref_flags(const ANode *__restrict__ nodes, const Decision *__restrict__ dec,
                                            const int *__restrict__ ref_tri, const int *__restrict__ ref_node,
                                            const float *__restrict__ lo, const float *__restrict__ hi, int n_tris,
                                            int i) {
    const int a = ref_node[i];
    const Decision d = dec[a];
    if (d.axis < 0) return Triple{ 0u, 0u, 1u };
    const int t = ref_tri[i];
    const float l = lo[(size_t)d.axis * n_tris + t], h = hi[(size_t)d.axis * n_tris + t];
    const bool right = h > d.plane;
    const bool left = l < d.plane || !right; // (lying in the plane, or wholly below it)
    return Triple{ left ? 1u : 0u, right ? 1u : 0u, 0u };
}

// Two sequences are scanned by every launch (the references and the nodes of a level: both
// depend on the decisions only): blocks [0, tiles_a) serve sequence A, the rest sequence B.
template <typename F>
__device__ __forceinline__ void scan_tile_sums(int tile, int n, const F &f, Triple *__restrict__ tile_sums) {
    __shared__ Triple warp_sums[SCAN_BLOCK / 32];
    const int base = tile * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    Triple s = { 0u, 0u, 0u };
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) s = s + f(base + k);
    }
    for (int off = 16; off > 0; off >>= 1) {
        s.l += __shfl_down_sync(0xffffffffu, s.l, off);
        s.r += __shfl_down_sync(0xffffffffu, s.r, off);
        s.f += __shfl_down_sync(0xffffffffu, s.f, off);
    }
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        Triple t = { 0u, 0u, 0u };
        for (int w = 0; w < SCAN_BLOCK / 32; w++) t = t + warp_sums[w];
        tile_sums[tile] = t;
    }
}

template <typename FA, typename FB>
__global__ void __launch_bounds__(SCAN_BLOCK)
scan_tile_sums_kernel(int tiles_a, const int *__restrict__ na, FA fa, Triple *__restrict__ sums_a,
                      const int *__restrict__ nb, FB fb, Triple *__restrict__ sums_b) {
    if ((int)blockIdx.x < tiles_a) scan_tile_sums((int)blockIdx.x, *na, fa, sums_a);
    else scan_tile_sums((int)blockIdx.x - tiles_a, *nb, fb, sums_b);
}

// Exclusive scan of the tile sums in place, one block per sequence; the grand totals land in total[0] (A), total[1] (B).
__global__ void __launch_bounds__(1024) scan_tile_offsets_kernel(Triple *__restrict__ sums_a, int tiles_a,
                                                                 Triple *__restrict__ sums_b, int tiles_b,
                                                                 Triple *__restrict__ total) {
    __shared__ Triple warp_sums[32];
    __shared__ Triple carry;
    Triple *tile_sums = blockIdx.x == 0 ? sums_a : sums_b;
    const int n_tiles = blockIdx.x == 0 ? tiles_a : tiles_b;
    if (threadIdx.x == 0) carry = Triple{ 0u, 0u, 0u };
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + threadIdx.x;
        const Triple v = i < n_tiles ? tile_sums[i] : Triple{ 0u, 0u, 0u };
        Triple s = v;
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned l = __shfl_up_sync(0xffffffffu, s.l, off), r = __shfl_up_sync(0xffffffffu, s.r, off),
                           f = __shfl_up_sync(0xffffffffu, s.f, off);
            if ((threadIdx.x & 31) >= off) s = s + Triple{ l, r, f };
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = s;
        __syncthreads();
        Triple before = carry;
        for (int w = 0; w < (int)(threadIdx.x >> 5); w++) before = before + warp_sums[w];
        if (i < n_tiles) tile_sums[i] = Triple{ before.l + s.l - v.l, before.r + s.r - v.r, before.f + s.f - v.f };
        __syncthreads();
        if (threadIdx.x == 1023) carry = Triple{ before.l + s.l, before.r + s.r, before.f + s.f };
        __syncthreads();
    }
    if (threadIdx.x == 0) total[blockIdx.x] = carry;
}

// Exclusive scan values for every item (plus one past the end = totals).
template <typename F>
__device__ __forceinline__ void scan_write(int tile, int n, const F &f, const Triple *__restrict__ tile_offsets,
                                           const Triple *__restrict__ total, Triple *__restrict__ out /* n + 1 */) {
    __shared__ Triple warp_sums[SCAN_BLOCK / 32];
    const int base = tile * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    Triple v[SCAN_ITEMS];
    Triple s = { 0u, 0u, 0u };
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = base + k < n ? f(base + k) : Triple{ 0u, 0u, 0u };
        s = s + v[k];
    }
    Triple inc = s;
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned l = __shfl_up_sync(0xffffffffu, inc.l, off), r = __shfl_up_sync(0xffffffffu, inc.r, off),
                       ff = __shfl_up_sync(0xffffffffu, inc.f, off);
        if ((threadIdx.x & 31) >= off) inc = inc + Triple{ l, r, ff };
    }
    if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = inc;
    __syncthreads();
    Triple before = tile_offsets[tile];
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) before = before + warp_sums[w];
    Triple run = Triple{ before.l + inc.l - s.l, before.r + inc.r - s.r, before.f + inc.f - s.f };
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) out[base + k] = run;
        run = run + v[k];
    }
    if (tile == 0 && threadIdx.x == 0) out[n] = total[0];
}

template <typename FA, typename FB>
__global__ void __launch_bounds__(SCAN_BLOCK)
scan_write_kernel(int tiles_a, const int *__restrict__ na, FA fa, const Triple *__restrict__ offsets_a,
                  Triple *__restrict__ out_a, const int *__restrict__ nb, FB fb, const Triple *__restrict__ offsets_b,
                  Triple *__restrict__ out_b, const Triple *__restrict__ total) {
    if ((int)blockIdx.x < tiles_a) scan_write((int)blockIdx.x, *na, fa, offsets_a, total, out_a);
    else scan_write((int)blockIdx.x - tiles_a, *nb, fb, offsets_b, total + 1, out_b);
}

struct NoItemsFn { // the empty second sequence of a single scan
    __device__ Triple operator()(int) const { return Triple{ 0u, 0u, 0u }; }
};

struct RefFlagFn {
    const ANode *nodes;
    const Decision *dec;
    const int *ref_tri, *ref_node;
    const float *lo, *hi;
    int n_tris;
    __device__ Triple operator()(int i) const { return ref_flags(nodes, dec, ref_tri, ref_node, lo, hi, n_tris, i); }
};
struct SplitFlagFn { // over the nodes of a level: .l counts splits, .f counts leaves
    const Decision *dec;
    __device__ Triple operator()(int i) const { return dec[i].axis >= 0 ? Triple{ 1u, 0u, 0u } : Triple{ 0u, 0u, 1u }; }
};

// ---- emit ------------------------------------------------------------------------------
// Wire record of node `out`: 17 words (include/kd_tree.h:31-50; the struct is packed, so it
// is written word by word).
__device__ __forceinline__ void write_box(int *__restrict__ wire, int out, const float *mn, const float *mx) {
    int *w = wire + 17 * (size_t)out;
    w[0] = __float_as_int(mn[0]);
    w[1] = __float_as_int(mn[1]);
    w[2] = __float_as_int(mn[2]);
    w[3] = 0;
    w[4] = __float_as_int(mx[0]);
    w[5] = __float_as_int(mx[1]);
    w[6] = __float_as_int(mx[2]);
    w[7] = 0;
}

// Room in the buffers a level's split writes.  Every thread of the split checks the level's
// totals against it (a few broadcast loads) and leaves the level alone when it does not fit;
// `commit` then stops the build and tells the host, which starts over level by level with
// every buffer sized exactly.
struct Room {
    int nodes_next, refs, out, leaf;
};

__device__ __forceinline__ bool level_fits(const LevelState *__restrict__ ls, const Triple *__restrict__ totals,
                                           const Room &room) {
    const long long nx_nodes = 2ll * totals[1].l, nx_refs = (long long)totals[0].l + totals[0].r, nx_leaf = totals[0].f;
    return ls->n_out + nx_nodes <= room.out && ls->n_leaf_refs + nx_leaf <= room.leaf && nx_refs <= room.refs &&
           nx_nodes <= room.nodes_next;
}

__device__ __forceinline__ void emit_node(int a, const LevelState *__restrict__ ls, const ANode *__restrict__ nodes,
                                          const Decision *__restrict__ dec,
                                          const Triple *__restrict__ node_scan /* n_nodes + 1 */,
                                          const Triple *__restrict__ ref_scan /* n_refs + 1 */, int *__restrict__ wire,
                                          ANode *__restrict__ next_nodes, int *__restrict__ big_counter) {
    if (a >= ls->n_nodes) return;
    const int next_out_base = ls->n_out, leaf_ref_base = ls->n_leaf_refs;
    const ANode nd = nodes[a];
    const Decision d = dec[a];
    write_box(wire, nd.out, nd.mn, nd.mx);
    int *w = wire + 17 * (size_t)nd.out;
    if (d.axis < 0) {
        w[8] = 1; // KD_LEAF
        w[9] = nd.count > 0 ? leaf_ref_base + (int)ref_scan[nd.begin].f : -1;
        w[10] = nd.count;
        for (int f = 0; f < 6; f++) w[11 + f] = nd.links[f];
        return;
    }
    const int rank = (int)node_scan[a].l;
    const int lo_out = next_out_base + 2 * rank, hi_out = lo_out + 1;
    w[8] = 0; // KD_SPLIT
    w[9] = __float_as_int(d.plane);
    w[10] = d.axis;
    w[11] = lo_out;
    w[12] = hi_out;
    w[13] = w[14] = w[15] = w[16] = 0;
    const Triple at_begin = ref_scan[nd.begin], at_end = ref_scan[nd.begin + nd.count];
    const int nl = (int)(at_end.l - at_begin.l), nr = (int)(at_end.r - at_begin.r);
    ANode L = nd, R = nd;
    L.mx[d.axis] = d.plane;
    R.mn[d.axis] = d.plane;
    L.begin = (int)(at_begin.l + at_begin.r);
    L.count = nl;
    R.begin = L.begin + nl;
    R.count = nr;
    L.out = lo_out;
    R.out = hi_out;
    L.links[2 * d.axis + 1] = hi_out; // max face of the low child
    R.links[2 * d.axis] = lo_out;     // min face of the high child
    L.depth_left = R.depth_left = nd.depth_left - 1;
    // (which slot a node gets depends on the order of the atomics; the histograms' content does not)
    L.hist_slot = nl > EXACT_MAX ? atomicAdd(big_counter, 1) : -1;
    R.hist_slot = nr > EXACT_MAX ? atomicAdd(big_counter, 1) : -1;
    next_nodes[2 * rank] = L;
    next_nodes[2 * rank + 1] = R;
}

__device__ __forceinline__ void scatter_ref(int i, const ANode *__restrict__ nodes, const Decision *__restrict__ dec,
                                            const Triple *__restrict__ node_scan, const Triple *__restrict__ ref_scan,
                                            const int *__restrict__ ref_tri, const int *__restrict__ ref_node,
                                            const LevelState *__restrict__ ls, const float *__restrict__ lo,
                                            const float *__restrict__ hi, int n_tris, int *__restrict__ next_tri,
                                            int *__restrict__ next_node, int *__restrict__ tri_indices) {
    if (i >= ls->n_refs) return;
    const int leaf_ref_base = ls->n_leaf_refs;
    const int a = ref_node[i], t = ref_tri[i];
    const Triple here = ref_scan[i];
    const Triple fl = ref_flags(nodes, dec, ref_tri, ref_node, lo, hi, n_tris, i);
    if (fl.f) {
        tri_indices[leaf_ref_base + here.f] = t;
        return;
    }
    const ANode &nd = nodes[a];
    const Triple at_begin = ref_scan[nd.begin], at_end = ref_scan[nd.begin + nd.count];
    const int child_base = (int)(at_begin.l + at_begin.r), nl = (int)(at_end.l - at_begin.l);
    const int rank = (int)node_scan[a].l;
    if (fl.l) {
        const int p = child_base + (int)(here.l - at_begin.l);
        next_tri[p] = t;
        next_node[p] = 2 * rank;
    }
    if (fl.r) {
        const int p = child_base + nl + (int)(here.r - at_begin.r);
        next_tri[p] = t;
        next_node[p] = 2 * rank + 1;
    }
}

// The split of a level in one launch: blocks [0, emit_blocks) write the wire nodes and the
// next level's nodes (one thread per node), the rest move the references (one thread each).
struct SplitArgs {
    const ANode *nodes;
    const Decision *dec;
    const Triple *node_scan, *ref_scan, *totals;
    const int *ref_tri, *ref_node;
    const float *lo, *hi;
    int n_tris;
    int *wire;
    ANode *next_nodes;
    int *big_counter, *next_tri, *next_node, *tri_indices;
    Room room;
};

__global__ void split_kernel(int emit_blocks, const LevelState *__restrict__ ls, const SplitArgs A) {
    if (!level_fits(ls, A.totals, A.room)) return;
    if ((int)blockIdx.x < emit_blocks) {
        emit_node((int)(blockIdx.x * blockDim.x + threadIdx.x), ls, A.nodes, A.dec, A.node_scan, A.ref_scan, A.wire,
                  A.next_nodes, A.big_counter);
    } else {
        scatter_ref((int)((blockIdx.x - emit_blocks) * blockDim.x + threadIdx.x), A.nodes, A.dec, A.node_scan, A.ref_scan,
                    A.ref_tri, A.ref_node, ls, A.lo, A.hi, A.n_tris, A.next_tri, A.next_node, A.tri_indices);
    }
}

// ---- level bookkeeping on the device ------------------------------------------------------
// After the split: the level state moves on to the next level (or the build stops, see Room).
__global__ void commit_kernel(LevelState *__restrict__ ls, const Triple *__restrict__ totals, const Room room,
                              int *__restrict__ big_counter) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    *big_counter = 0; // the histogram slots of the next level are handed out from 0 again
    if (ls->n_nodes > 0) ls->levels++;
    if (!level_fits(ls, totals, room)) {
        ls->overflow = 1;
        ls->n_nodes = ls->n_refs = 0;
        return;
    }
    const int nx_nodes = 2 * (int)totals[1].l;
    ls->n_out += nx_nodes;
    ls->n_leaf_refs += (int)totals[0].f;
    ls->n_nodes = nx_nodes;
    ls->n_refs = (int)(totals[0].l + totals[0].r);
}

// ---- ropes -----------------------------------------------------------------------------
// One thread per (node, face): a leaf's link is pushed down to the deepest node that the
// whole face still looks into (kd_build.c: push_down_link with full = 1).
__global__ void push_ropes_kernel(int *__restrict__ wire, const LevelState *__restrict__ ls) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int node = i / 6, face = i - node * 6;
    if (node >= ls->n_out) return;
    int *w = wire + 17 * (size_t)node;
    if (w[8] != 1) return;
    int link = w[11 + face];
    while (link != -1) {
        const int *nb = wire + 17 * (size_t)link;
        if (nb[8] == 1) break;
        const int ax = nb[10];
        if (face / 2 == ax) {
            link = nb[(face & 1) ? 11 : 12];
            continue;
        }
        const float plane = __int_as_float(nb[9]);
        if (plane >= __int_as_float(w[4 + ax])) {
            link = nb[11];
        } else if (plane <= __int_as_float(w[ax])) {
            link = nb[12];
        } else {
            break;
        }
    }
    w[11 + face] = link;
}

bool g_last_build_recorded = false;

// Working storage, kept between builds (an animated scene rebuilds every frame).
struct Workspace {
    DevBuf<float> lo, hi;
    DevBuf<int> ref_tri[2], ref_node[2];
    DevBuf<ANode> nodes[2];
    DevBuf<Decision> dec;
    DevBuf<unsigned> hist;
    DevBuf<Triple> ref_scan, node_scan, tiles, totals;
    DevBuf<int> box_keys, bad, box_init;
    DevBuf<LevelState> level; // [0] the build's, [1] scratch (`n` of a stand-alone scan)
    // the re-layout's (clpt_gpu_pack)
    DevBuf<int> new_of;
    DevBuf<Triple> wire_scan;
    struct Pinned { // what comes back to the host
        Triple totals[2]; // [0] references, [1] nodes
        int bad;
        int n;
        LevelState level;
    } *host = nullptr;
    // the whole build of a small mesh, recorded once and replayed (see clpt_gpu_build)
    cudaGraphExec_t graph = nullptr;
    struct GraphKey {
        const void *verts, *corners, *wire, *tri_indices;
        size_t reallocations, room;
        int n_verts, n_tris, max_depth, min_split;
        float ct, ci, empty_bonus;
        bool operator==(const GraphKey &o) const {
            return verts == o.verts && corners == o.corners && wire == o.wire && tri_indices == o.tri_indices &&
                   reallocations == o.reallocations && room == o.room && n_verts == o.n_verts && n_tris == o.n_tris && max_depth == o.max_depth && min_split == o.min_split &&
                   ct == o.ct && ci == o.ci && empty_bonus == o.empty_bonus;
        }
    } graph_key = {};
    int graph_refused_tris = -1, graph_refused_room = 0; // the recorded capacities were too small for a mesh of this size: do not try again
} W;

void ensure_host() {
    if (!W.host) CU(cudaMallocHost((void **)&W.host, sizeof(Workspace::Pinned)));
    W.level.reserve(2);
    W.totals.reserve(2);
}

void drop_graph() {
    if (W.graph) (void)cudaGraphExecDestroy(W.graph);
    W.graph = nullptr;
}

int scan_tiles(size_t n_cap) { return (int)std::max<size_t>(1, (n_cap + SCAN_TILE - 1) / SCAN_TILE); }

// Two scans in three launches (see scan_tile_sums_kernel): f(0..na-1) and g(0..nb-1), the counts read
// from device memory; `cap_a`, `cap_b` (>= the counts) size the launches.  Totals land in total_dev[0], [1].
template <typename FA, typename FB>
void scan2(const int *na, size_t cap_a, FA fa, Triple *out_a, const int *nb, size_t cap_b, FB fb, Triple *out_b,
           Triple *total_dev, cudaStream_t s) {
    const int ta = scan_tiles(cap_a), tb = scan_tiles(cap_b);
    Triple *sums_a = W.tiles.ptr, *sums_b = W.tiles.ptr + ta;
    scan_tile_sums_kernel<<<ta + tb, SCAN_BLOCK, 0, s>>>(ta, na, fa, sums_a, nb, fb, sums_b);
    scan_tile_offsets_kernel<<<2, 1024, 0, s>>>(sums_a, ta, sums_b, tb, total_dev);
    scan_write_kernel<<<ta + tb, SCAN_BLOCK, 0, s>>>(ta, na, fa, sums_a, out_a, nb, fb, sums_b, out_b, total_dev);
}

constexpr int T = 256;
constexpr int CHOOSE_MAX_BLOCKS = 148 * 16;

struct BuildArgs {
    const float4 *verts;
    const int4 *corners;
    int n_verts, n_tris, max_depth, min_split;
    float ct, ci, empty_bonus;
};

// Triangle bounds, scene box, the root node and its reference list, the level state.
void enqueue_prologue(const BuildArgs &A, cudaStream_t s) {
    CU(cudaMemsetAsync(W.bad.ptr, 0, sizeof(int), s));
    tri_bounds_kernel<<<(A.n_tris + T - 1) / T, T, 0, s>>>(A.verts, A.corners, A.n_tris, A.n_verts, W.lo.ptr, W.hi.ptr,
                                                           W.bad.ptr);
    CU(cudaMemcpyAsync(W.box_keys.ptr, W.box_init.ptr, 6 * sizeof(int), cudaMemcpyDeviceToDevice, s));
    scene_box_kernel<<<std::min(1024, (A.n_tris + T - 1) / T), T, 0, s>>>(W.lo.ptr, W.hi.ptr, A.n_tris, W.box_keys.ptr);
    CU(cudaMemcpyAsync(&W.host->bad, W.bad.ptr, sizeof(int), cudaMemcpyDeviceToHost, s));
    root_kernel<<<(A.n_tris + T - 1) / T, T, 0, s>>>(W.box_keys.ptr, A.n_tris, A.max_depth, W.nodes[0].ptr,
                                                     W.ref_tri[0].ptr, W.ref_node[0].ptr, W.level.ptr, W.bad.ptr);
}

size_t hist_words(size_t refs) { // nodes with histograms hold more than EXACT_MAX references
    return (refs / (EXACT_MAX + 1) + 1) * 3 * 2 * NBINS;
}

// The first half of a level: histograms, the split decisions, the two scans.  `refs` and
// `nodes` size the launches (the true counts, or upper bounds -- the kernels read the true
// counts from the level state).  The histograms must be zero on entry and are zero on exit.
void enqueue_decide(const BuildArgs &A, int cur, size_t refs, size_t nodes, cudaStream_t s) {
    const LevelState *ls = W.level.ptr;
    const ANode *nodes_cur = W.nodes[cur].ptr;
    const int *ref_tri = W.ref_tri[cur].ptr, *ref_node = W.ref_node[cur].ptr;
    if (refs > 0) {
        bin_kernel<<<(unsigned)((refs + 255) / 256), 256, 0, s>>>(ls, nodes_cur, ref_tri, ref_node, W.lo.ptr, W.hi.ptr,
                                                                  A.n_tris, A.min_split, W.hist.ptr);
    }
    // nodes of more than SMALL_MAX references: there are at most refs / SMALL_MAX of them
    const size_t big = std::min(nodes, refs / SMALL_MAX + 1);
    const int g32 = (int)std::max<size_t>(1, std::min<size_t>(CHOOSE_MAX_BLOCKS, (big * 32 + 255) / 256));
    const int g8 = (int)std::max<size_t>(1, std::min<size_t>(CHOOSE_MAX_BLOCKS, (nodes * 8 + 255) / 256));
    choose_kernel<<<g32 + g8, 256, 0, s>>>(g32, ls, nodes_cur, W.hist.ptr, ref_tri, W.lo.ptr, W.hi.ptr, A.n_tris,
                                           A.min_split, A.ct, A.ci, A.empty_bonus, W.dec.ptr);
    RefFlagFn rf{ nodes_cur, W.dec.ptr, ref_tri, ref_node, W.lo.ptr, W.hi.ptr, A.n_tris };
    SplitFlagFn sf{ W.dec.ptr };
    scan2(&ls->n_refs, refs, rf, W.ref_scan.ptr, &ls->n_nodes, nodes, sf, W.node_scan.ptr, W.totals.ptr, s);
}

// The second half: wire nodes and the next level's nodes written, references moved to their
// children or to the leaf lists (all of it only if the level fits `room`), the level state advanced.
void enqueue_split(const BuildArgs &A, int cur, size_t refs, size_t nodes, const Room &room, ClptGpuTree &out,
                   cudaStream_t s) {
    const int nxt = cur ^ 1;
    SplitArgs sa = { W.nodes[cur].ptr,    W.dec.ptr,          W.node_scan.ptr,     W.ref_scan.ptr,
                     W.totals.ptr,        W.ref_tri[cur].ptr, W.ref_node[cur].ptr, W.lo.ptr,
                     W.hi.ptr,            A.n_tris,           out.wire.ptr,        W.nodes[nxt].ptr,
                     W.bad.ptr,           W.ref_tri[nxt].ptr, W.ref_node[nxt].ptr, out.tri_indices.ptr,
                     room };
    const int emit_blocks = (int)std::max<size_t>(1, (nodes + T - 1) / T);
    const int scatter_blocks = (int)((refs + T - 1) / T);
    split_kernel<<<emit_blocks + scatter_blocks, T, 0, s>>>(emit_blocks, W.level.ptr, sa);
    commit_kernel<<<1, 32, 0, s>>>(W.level.ptr, W.totals.ptr, room, W.bad.ptr);
}

// Meshes up to this size are built without the host in the loop (below).
constexpr int GRAPH_MAX_TRIS = 1 << 18;

// One recording of the WHOLE build for small meshes: every level's launches sized by fixed
// capacities, the counts living in the level state, max_depth + 1 levels whatever the tree
// turns out to need (levels past the last are empty launches).  The recording is replayed
// while mesh size, buffers and parameters stay the same -- an animated scene.  Returns
// false if the capacities were too small (the caller then takes the level-by-level path).
bool build_recorded(const BuildArgs &A, int room_pc, ClptGpuTree &out, cudaStream_t s, char *err, size_t errlen,
                    bool *bad_mesh) {
    const size_t n = (size_t)A.n_tris;
    size_t cap_refs = 6 * n + 4096, cap_nodes = 4 * n + 1024, cap_out = 8 * n + 4096, cap_leaf = 8 * n + 4096;
    if (room_pc != 100) {
        const size_t pc = (size_t)room_pc;
        cap_refs = std::max(n, cap_refs * pc / 100), cap_nodes = std::max<size_t>(2, cap_nodes * pc / 100);
        cap_out = std::max<size_t>(2, cap_out * pc / 100), cap_leaf = std::max<size_t>(2, cap_leaf * pc / 100);
    }
    for (int k = 0; k < 2; k++) {
        W.ref_tri[k].reserve(cap_refs);
        W.ref_node[k].reserve(cap_refs);
        W.nodes[k].reserve(cap_nodes);
    }
    W.dec.reserve(cap_nodes);
    W.hist.reserve(hist_words(cap_refs));
    W.ref_scan.reserve(cap_refs + 1);
    W.node_scan.reserve(cap_nodes + 1);
    // (the second term: what the re-layout of this tree will ask for)
    W.tiles.reserve((size_t)std::max(scan_tiles(cap_refs) + scan_tiles(cap_nodes), scan_tiles(cap_out) + 1));
    out.wire.reserve(cap_out * 17);
    out.tri_indices.reserve(cap_leaf);
    const Workspace::GraphKey key = { A.verts, A.corners, out.wire.ptr, out.tri_indices.ptr, clpt_devbuf_reallocations,
                                      cap_refs, A.n_verts, A.n_tris, A.max_depth, A.min_split, A.ct, A.ci, A.empty_bonus };
    if (!W.graph || !(key == W.graph_key)) {
        drop_graph();
        cudaGraph_t g = nullptr;
        CU(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        CU(cudaMemsetAsync(W.hist.ptr, 0, hist_words(cap_refs) * sizeof(unsigned), s)); // (each level leaves it zeroed)
        enqueue_prologue(A, s);
        int cur = 0;
        for (int level = 0; level <= A.max_depth; level++) {
            // a level has at most 2^level nodes, and its references all come from the level above
            const size_t nodes = level < 30 ? std::min<size_t>(cap_nodes, (size_t)1 << level) : cap_nodes;
            const size_t nodes_next = level + 1 < 30 ? std::min<size_t>(cap_nodes, (size_t)2 << level) : cap_nodes;
            const size_t refs = level == 0 ? n : cap_refs;
            enqueue_decide(A, cur, refs, nodes, s);
            enqueue_split(A, cur, refs, nodes, Room{ (int)nodes_next, (int)cap_refs, (int)cap_out, (int)cap_leaf }, out, s);
            cur ^= 1;
        }
        push_ropes_kernel<<<(unsigned)((cap_out * 6 + T - 1) / T), T, 0, s>>>(out.wire.ptr, W.level.ptr);
        CU(cudaMemcpyAsync(&W.host->level, W.level.ptr, sizeof(LevelState), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamEndCapture(s, &g));
        CU(cudaGraphInstantiate(&W.graph, g, 0));
        CU(cudaGraphDestroy(g));
        W.graph_key = key;
    }
    CU(cudaGraphLaunch(W.graph, s));
    CU(cudaStreamSynchronize(s));
    if (W.host->bad) {
        *bad_mesh = true;
        snprintf(err, errlen, "triangle corner references a missing vertex");
        return false;
    }
    const LevelState &L = W.host->level;
    if (L.overflow || L.n_nodes != 0) return false; // (n_nodes != 0: deeper than max_depth cannot happen; belt and braces)
    out.n_nodes = L.n_out;
    out.n_refs = L.n_leaf_refs;
    out.levels = L.levels;
    return true;
}

} // namespace

bool clpt_gpu_build(const float4 *verts, int n_verts, const int4 *corners, int n_tris, const ClptGpuBuildParams &P,
                    ClptGpuTree &out, cudaStream_t s, char *err, size_t errlen) {
    if (n_tris <= 0 || n_verts <= 0) {
        snprintf(err, errlen, "empty mesh");
        return false;
    }
    BuildArgs A = { verts, corners, n_verts, n_tris, P.max_depth, P.min_split > 1 ? P.min_split : 2, P.ct, P.ci,
                    P.empty_bonus };
    if (A.max_depth <= 0) { // 8 + 1.3 log2(N), the usual bound for SAH kd-trees
        int lg = 0;
        while ((1 << lg) < n_tris) lg++;
        A.max_depth = 8 + (13 * lg) / 10;
    }
    ensure_host();
    W.lo.reserve((size_t)n_tris * 3);
    W.hi.reserve((size_t)n_tris * 3);
    W.box_keys.reserve(8);
    W.bad.reserve(1);
    if (!W.box_init.ptr) {
        W.box_init.reserve(8);
        const int init_keys[6] = { INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN };
        CU(cudaMemcpy(W.box_init.ptr, init_keys, sizeof(init_keys), cudaMemcpyHostToDevice));
    }

    const char *no_graph = getenv("CLPT_BUILD_NO_GRAPH"); // measurement and tests: always level by level
    const char *room = getenv("CLPT_BUILD_RECORD_ROOM"); // tests: per cent of the usual room, to meet the fallback
    const int room_pc = room ? std::max(1, atoi(room)) : 100;
    const bool refused = W.graph_refused_tris == n_tris && W.graph_refused_room == room_pc;
    if (n_tris <= GRAPH_MAX_TRIS && !refused && !(no_graph && atoi(no_graph) != 0)) {
        bool bad_mesh = false;
        if (build_recorded(A, room_pc, out, s, err, errlen, &bad_mesh)) {
            g_last_build_recorded = true;
            return true;
        }
        if (bad_mesh) return false;
        W.graph_refused_room = room_pc;
        W.graph_refused_tris = n_tris; // this mesh needs more room than the recording gives: size every level exactly
        drop_graph();
    }
    g_last_build_recorded = false;

    // Level by level with the host in the loop: two counters come back per level to size the
    // next level's buffers and launches exactly (any mesh size).
    int cur = 0;
    W.ref_tri[0].reserve((size_t)n_tris);
    W.ref_node[0].reserve((size_t)n_tris);
    W.nodes[0].reserve(1);
    enqueue_prologue(A, s);
    size_t n_out = 1;       // wire nodes allocated so far (the root)
    size_t n_leaf_refs = 0; // tri_indices written so far
    size_t n_nodes = 1, n_refs = (size_t)n_tris;
    out.wire.reserve((size_t)17 * 1024);
    int levels = 0;
    while (n_nodes > 0) {
        levels++;
        W.dec.reserve(n_nodes);
        W.hist.reserve(hist_words(n_refs));
        W.ref_scan.reserve(n_refs + 1);
        W.node_scan.reserve(n_nodes + 1);
        W.tiles.reserve((size_t)(scan_tiles(n_refs) + scan_tiles(n_nodes)));
        // (the buffer may just have moved; otherwise the previous level left it zeroed and this is redundant)
        CU(cudaMemsetAsync(W.hist.ptr, 0, hist_words(n_refs) * sizeof(unsigned), s));
        enqueue_decide(A, cur, n_refs, n_nodes, s);
        CU(cudaMemcpyAsync(W.host->totals, W.totals.ptr, 2 * sizeof(Triple), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (levels == 1 && W.host->bad) {
            snprintf(err, errlen, "triangle corner references a missing vertex");
            return false;
        }
        const Triple rt = W.host->totals[0], nt = W.host->totals[1];
        const size_t next_refs = (size_t)rt.l + rt.r, next_nodes = (size_t)2 * nt.l;
        if (next_refs > 0x7fff0000u || n_out + next_nodes > 0x1fff0000u) {
            snprintf(err, errlen, "tree too large (%zu references, %zu nodes)", next_refs, n_out + next_nodes);
            return false;
        }
        out.wire.grow_keep((n_out + next_nodes) * 17, n_out * 17, s);
        out.tri_indices.grow_keep(n_leaf_refs + rt.f, n_leaf_refs, s);
        const int nxt = cur ^ 1;
        W.ref_tri[nxt].reserve(next_refs);
        W.ref_node[nxt].reserve(next_refs);
        W.nodes[nxt].reserve(next_nodes);
        enqueue_split(A, cur, n_refs, n_nodes, Room{ INT_MAX, INT_MAX, INT_MAX, INT_MAX }, out, s);
        n_out += next_nodes;
        n_leaf_refs += rt.f;
        n_nodes = next_nodes;
        n_refs = next_refs;
        cur = nxt;
    }
    push_ropes_kernel<<<(unsigned)((n_out * 6 + T - 1) / T), T, 0, s>>>(out.wire.ptr, W.level.ptr);
    CU(cudaGetLastError());
    out.n_nodes = (int)n_out;
    out.n_refs = (int)n_leaf_refs;
    out.levels = levels;
    return true;
}

// ======================================================================================
// Re-layout on the device: the twin of clpt_pack_scene (scene_pack.cpp).  Same numbering
// (the children of the k-th split node in input order become nodes 1+2k and 2+2k; leaves
// keep their input order), same records, same start-node table -- the two packers produce
// the same bytes from the same wire arrays (tests/test_gpu_build.py).
// ======================================================================================
namespace {

struct WireTypeFn { // .l counts split nodes, .f counts leaves, .r counts fat-leaf triangle slots
    const int *wire;
    __device__ Triple operator()(int i) const {
        const int *w = wire + 17 * (size_t)i;
        if (w[8] == 0) return Triple{ 1u, 0u, 0u };
        return Triple{ 0u, w[10] >= CLPT_COOP_LEAF_MIN ? (unsigned)w[10] : 0u, 1u };
    }
};

__global__ void renumber_kernel(const int *__restrict__ wire, int n_nodes, const Triple *__restrict__ scan,
                                int *__restrict__ new_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    if (i == 0) new_of[0] = 0;
    const int *w = wire + 17 * (size_t)i;
    if (w[8] == 0) {
        const int ks = (int)scan[i].l;
        new_of[w[11]] = 1 + 2 * ks; // each child has one parent: no two threads write one slot
        new_of[w[12]] = 2 + 2 * ks;
    }
}

__global__ void pack_nodes_kernel(const int *__restrict__ wire, int n_nodes, const Triple *__restrict__ scan,
                                  const int *__restrict__ new_of, uint2 *__restrict__ nodes, float4 *__restrict__ leaves) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const int *w = wire + 17 * (size_t)i;
    const int ni = new_of[i];
    if (w[8] == 0) {
        nodes[ni] = make_uint2((unsigned)w[9], ((unsigned)new_of[w[11]] << 2) | (unsigned)w[10]);
        return;
    }
    const int li = (int)scan[i].f;
    nodes[ni] = make_uint2((unsigned)li, 0x80000003u);
    const int count = w[10], first = count > 0 ? w[9] : 0;
    float4 *L = leaves + 4 * (size_t)li;
    L[0] = make_float4(__int_as_float(w[0]), __int_as_float(w[1]), __int_as_float(w[2]), __int_as_float(first));
    L[1] = make_float4(__int_as_float(w[4]), __int_as_float(w[5]), __int_as_float(w[6]), __int_as_float(count));
    int ropes[6];
    for (int f = 0; f < 6; f++) {
        const int r = w[11 + f];
        if (r < 0 || r >= n_nodes) {
            ropes[f] = -1;
        } else if (wire[17 * (size_t)r + 8] == 1) {
            ropes[f] = -2 - (int)scan[r].f; // straight to the leaf record
        } else {
            ropes[f] = new_of[r];
        }
    }
    L[2] = make_float4(__int_as_float(ropes[0]), __int_as_float(ropes[1]), __int_as_float(ropes[2]),
                       __int_as_float(ropes[3]));
    L[3] = make_float4(__int_as_float(ropes[4]), __int_as_float(ropes[5]), 0.0f, 0.0f);
}

__global__ void pack_tris_kernel(const int *__restrict__ tri_indices, int n_refs, const int4 *__restrict__ corners,
                                 const float4 *__restrict__ verts, float4 *__restrict__ tri) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_refs) return;
    const int b = tri_indices[s];
    const float4 v0 = verts[corners[3 * (size_t)b].x], v1 = verts[corners[3 * (size_t)b + 1].x],
                 v2 = verts[corners[3 * (size_t)b + 2].x];
    float4 *T = tri + 3 * (size_t)s;
    T[0] = make_float4(v0.x, v0.y, v0.z, __int_as_float(b));
    // one fp32 subtraction each, the same rounding as `v1 - v0` in the kernel
    T[1] = make_float4(__fsub_rn(v1.x, v0.x), __fsub_rn(v1.y, v0.y), __fsub_rn(v1.z, v0.z), 0.0f);
    T[2] = make_float4(__fsub_rn(v2.x, v0.x), __fsub_rn(v2.y, v0.y), __fsub_rn(v2.z, v0.z), 0.0f);
}

// Flat shading normal per primitive (ClptScene::flat_n; the host twin is in scene_pack.cpp).
__global__ void pack_flat_normals_kernel(const int4 *__restrict__ corners, const float4 *__restrict__ verts, int n_prims,
                                         float4 *__restrict__ flat_n) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_prims) return;
    const int4 c0 = corners[3 * (size_t)p];
    const float4 v0 = verts[c0.x], v1 = verts[corners[3 * (size_t)p + 1].x], v2 = verts[corners[3 * (size_t)p + 2].x];
    const float ax = __fsub_rn(v1.x, v0.x), ay = __fsub_rn(v1.y, v0.y), az = __fsub_rn(v1.z, v0.z);
    const float bx = __fsub_rn(v2.x, v0.x), by = __fsub_rn(v2.y, v0.y), bz = __fsub_rn(v2.z, v0.z);
    const float cx = __fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by));
    const float cy = __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz));
    const float cz = __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
    const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz)));
    flat_n[p] = make_float4(__fdiv_rn(cx, len), __fdiv_rn(cy, len), __fdiv_rn(cz, len), c0.y >= 0 ? 1.0f : 0.0f);
}

struct LutGrid {
    double root_min[3], ext[3], scale[3]; // scale = (double)(float)(dim / ext), as the host packer reads it back
    int dim[3];
};

// Start-node table: per cell, follow the branches the whole (slightly enlarged) cell is
// forced to take from the root (scene_pack.cpp, "start-node table").
__global__ void pack_lut_kernel(const int *__restrict__ wire, const int *__restrict__ new_of, const LutGrid G,
                                int *__restrict__ lut) {
    const size_t total = (size_t)G.dim[0] * G.dim[1] * G.dim[2];
    const size_t cell = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= total) return;
    const int c[3] = { (int)(cell % G.dim[0]), (int)((cell / G.dim[0]) % G.dim[1]),
                       (int)(cell / ((size_t)G.dim[0] * G.dim[1])) };
    double lo[3], hi[3];
    for (int a = 0; a < 3; a++) {
        const double sc = G.scale[a];
        const double margin = 1e-5 * (1.0 + G.ext[a] + fabs(G.root_min[a]));
        if (sc > 0) {
            lo[a] = G.root_min[a] + c[a] / sc - margin;
            hi[a] = G.root_min[a] + (c[a] + 1) / sc + margin;
        } else {
            lo[a] = -1e300;
            hi[a] = 1e300;
        }
        if (c[a] == 0) lo[a] = -1e300;
        if (c[a] == G.dim[a] - 1) hi[a] = 1e300;
    }
    int o = 0;
    for (;;) {
        const int *w = wire + 17 * (size_t)o;
        if (w[8] != 0) break;
        const int ax = w[10];
        const double plane = (double)__int_as_float(w[9]);
        if (hi[ax] <= plane) {
            o = w[11];
        } else if (lo[ax] > plane) {
            o = w[12];
        } else {
            break;
        }
    }
    lut[cell] = new_of[o];
}

} // namespace

bool clpt_gpu_pack(const ClptGpuTree &tree, const float4 *verts, const int4 *corners, int n_prims, ClptSceneLayout &out,
                   cudaStream_t s, char *err, size_t errlen) {
    const int n = tree.n_nodes;
    if (n <= 0) {
        snprintf(err, errlen, "empty node array");
        return false;
    }
    ensure_host();
    W.new_of.reserve((size_t)n);
    W.wire_scan.reserve((size_t)n + 2);
    W.tiles.reserve((size_t)scan_tiles((size_t)n) + 1);
    W.host->n = n;
    int *n_dev = &W.level.ptr[1].n_nodes;
    CU(cudaMemcpyAsync(n_dev, &W.host->n, sizeof(int), cudaMemcpyHostToDevice, s));
    WireTypeFn tf{ tree.wire.ptr };
    int *zero_dev = &W.level.ptr[1].n_refs; // (an empty second sequence)
    CU(cudaMemsetAsync(zero_dev, 0, sizeof(int), s));
    Triple *scan = W.wire_scan.ptr;
    scan2(n_dev, (size_t)n, tf, scan, zero_dev, 0, NoItemsFn{}, scan /* one word past the first */ + n + 1, W.totals.ptr, s);
    CU(cudaMemcpyAsync(W.host->totals, W.totals.ptr, sizeof(Triple), cudaMemcpyDeviceToHost, s));
    float box[8];
    CU(cudaMemcpyAsync(box, tree.wire.ptr, sizeof(box), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const int n_splits = (int)W.host->totals[0].l, n_leaves = (int)W.host->totals[0].f;
    out.fat_refs = W.host->totals[0].r;
    out.n_nodes = 1 + 2 * n_splits;
    out.n_leaves = n_leaves;
    out.n_refs = tree.n_refs;
    out.nodes.reserve((size_t)out.n_nodes);
    out.leaves.reserve((size_t)n_leaves * 4);
    out.tri.reserve((size_t)std::max(tree.n_refs, 1) * 3);
    const int *wire = tree.wire.ptr;
    int *new_of = W.new_of.ptr;
    renumber_kernel<<<(n + T - 1) / T, T, 0, s>>>(wire, n, scan, new_of);
    pack_nodes_kernel<<<(n + T - 1) / T, T, 0, s>>>(wire, n, scan, new_of, out.nodes.ptr, out.leaves.ptr);
    if (tree.n_refs > 0) {
        pack_tris_kernel<<<(tree.n_refs + T - 1) / T, T, 0, s>>>(tree.tri_indices.ptr, tree.n_refs, corners, verts,
                                                                 out.tri.ptr);
    }
    out.flat_n.reserve((size_t)std::max(n_prims, 1));
    if (n_prims > 0) {
        // (the builder has checked every corner's vertex index, tri_bounds_kernel)
        pack_flat_normals_kernel<<<(n_prims + T - 1) / T, T, 0, s>>>(corners, verts, n_prims, out.flat_n.ptr);
    }
    // start-node table geometry: the host packer's arithmetic (scene_pack.cpp), so that both give the same table
    LutGrid G;
    double vol = 1.0;
    for (int a = 0; a < 3; a++) {
        out.root_min[a] = box[a];
        out.root_max[a] = box[4 + a];
        G.root_min[a] = (double)box[a];
        G.ext[a] = (double)box[4 + a] - (double)box[a];
        if (!(G.ext[a] > 0)) G.ext[a] = 0;
        vol *= G.ext[a] > 0 ? G.ext[a] : 1.0;
    }
    double target_cells = (double)n / 2;
    target_cells = n < 64 ? 1.0 : (target_cells < 4096.0 ? 4096.0 : (target_cells > 2097152.0 ? 2097152.0 : target_cells));
    const double cell = cbrt(vol / target_cells);
    size_t total = 1;
    for (int a = 0; a < 3; a++) {
        int d = G.ext[a] > 0 && cell > 0 ? (int)ceil(G.ext[a] / cell) : 1;
        d = d < 1 ? 1 : (d > 1024 ? 1024 : d);
        out.lut_dim[a] = G.dim[a] = d;
        out.lut_scale[a] = G.ext[a] > 0 ? (float)(d / G.ext[a]) : 0.0f;
        G.scale[a] = (double)out.lut_scale[a];
        total *= (size_t)d;
    }
    out.lut.reserve(total);
    pack_lut_kernel<<<(unsigned)((total + T - 1) / T), T, 0, s>>>(wire, new_of, G, out.lut.ptr);
    CU(cudaGetLastError());
    return true;
}

bool clpt_gpu_build_was_recorded(void) { return g_last_build_recorded; }

void clpt_gpu_build_release(void) {
    W.lo.release(), W.hi.release(), W.dec.release(), W.hist.release();
    for (int k = 0; k < 2; k++) W.ref_tri[k].release(), W.ref_node[k].release(), W.nodes[k].release();
    W.ref_scan.release(), W.node_scan.release(), W.tiles.release(), W.totals.release();
    W.box_keys.release(), W.bad.release(), W.box_init.release(), W.level.release();
    W.new_of.release(), W.wire_scan.release();
    if (W.host) (void)cudaFreeHost(W.host);
    drop_graph();
    W = Workspace();
    g_last_build_recorded = false;
}

