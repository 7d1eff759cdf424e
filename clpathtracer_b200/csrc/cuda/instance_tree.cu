// instance_tree.cu -- the top-level tree over the instances' world boxes (CLPT_INSTANCES_TREE).
//
// A linear BVH in the manner of Karras, "Maximizing Parallelism in the Construction of BVHs,
// Octrees, and k-d Trees" (HPG 2012), built in stream order with no host round trip:
//   1. world box of every instance (float64, padded, rounded outward to fp32) and the bounds of
//      the boxes' centroids;
//   2. key = morton30(centroid quantised to 10 bits per axis) << 20 | k -- 50 bits, unique;
//   3. keys sorted (CUB radix sort over the 50 bits);
//   4. the n - 1 internal nodes from the sorted keys (parent links only);
//   5. child boxes filled bottom-up, the second of two arrivals at a node going on.
// Every step is a function of the records alone (unique keys; min and max do not depend on the
// order they are taken in), so the node bytes are the same on every GPU and equal those of the
// CPU twin (oracle/oracle_instance_tree.c).  DESIGN.md "Instance tree" is the definition.
#include <cub/device/device_radix_sort.cuh>

#include <cfloat>

#include "CLHandler.h"
#include "clpt_device.cuh"

namespace {

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dadd_rn(a, -b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double dmin(double a, double b) { return b < a ? b : a; }
__device__ __forceinline__ double dmax(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ float fmin_(float a, float b) { return b < a ? b : a; }
__device__ __forceinline__ float fmax_(float a, float b) { return b > a ? b : a; }

// fp32 -> an unsigned key with the same order (for atomicMin / atomicMax)
__device__ __forceinline__ unsigned order_key(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float order_value(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct Box {
    float lo[3], hi[3];
};

// World box of instance R over the object-space box [mn, mx] of its mesh.
__device__ Box world_box(const ClptInstRec &R, const float *mn, const float *mx) {
    double a[9], b[3];
    for (int r = 0; r < 3; r++) {
        a[3 * r] = R.w2o[4 * r];
        a[3 * r + 1] = R.w2o[4 * r + 1];
        a[3 * r + 2] = R.w2o[4 * r + 2];
        b[r] = R.w2o[4 * r + 3];
    }
    // A^-1 = adj(A) / det(A), entry by entry
    const double c00 = dsub(dmul(a[4], a[8]), dmul(a[5], a[7]));
    const double c01 = dsub(dmul(a[5], a[6]), dmul(a[3], a[8]));
    const double c02 = dsub(dmul(a[3], a[7]), dmul(a[4], a[6]));
    const double det = dadd(dadd(dmul(a[0], c00), dmul(a[1], c01)), dmul(a[2], c02));
    double m[9];
    m[0] = ddiv(c00, det);
    m[1] = ddiv(dsub(dmul(a[2], a[7]), dmul(a[1], a[8])), det);
    m[2] = ddiv(dsub(dmul(a[1], a[5]), dmul(a[2], a[4])), det);
    m[3] = ddiv(c01, det);
    m[4] = ddiv(dsub(dmul(a[0], a[8]), dmul(a[2], a[6])), det);
    m[5] = ddiv(dsub(dmul(a[2], a[3]), dmul(a[0], a[5])), det);
    m[6] = ddiv(c02, det);
    m[7] = ddiv(dsub(dmul(a[1], a[6]), dmul(a[0], a[7])), det);
    m[8] = ddiv(dsub(dmul(a[0], a[4]), dmul(a[1], a[3])), det);
    double t[3], lo[3], hi[3];
    for (int r = 0; r < 3; r++) t[r] = -dadd(dadd(dmul(m[3 * r], b[0]), dmul(m[3 * r + 1], b[1])), dmul(m[3 * r + 2], b[2]));
    for (int c = 0; c < 8; c++) {
        const double x = (c & 1) ? mx[0] : mn[0], y = (c & 2) ? mx[1] : mn[1], z = (c & 4) ? mx[2] : mn[2];
        for (int r = 0; r < 3; r++) {
            const double w = dadd(dadd(dadd(dmul(m[3 * r], x), dmul(m[3 * r + 1], y)), dmul(m[3 * r + 2], z)), t[r]);
            lo[r] = c == 0 ? w : dmin(lo[r], w);
            hi[r] = c == 0 ? w : dmax(hi[r], w);
        }
    }
    double ext = 0.0, mag = 0.0;
    bool finite = det != 0.0;
    for (int r = 0; r < 3; r++) {
        finite = finite && isfinite(lo[r]) && isfinite(hi[r]);
        ext = dmax(ext, dsub(hi[r], lo[r]));
        mag = dmax(mag, dmax(fabs(lo[r]), fabs(hi[r])));
    }
    const double pad = dadd(dmul(ext, 0x1p-12), dmul(mag, 0x1p-20));
    Box B;
    for (int r = 0; r < 3; r++) {
        if (finite && isfinite(pad)) {
            B.lo[r] = fmax_(__double2float_rd(dsub(lo[r], pad)), -FLT_MAX);
            B.hi[r] = fmin_(__double2float_ru(dadd(hi[r], pad)), FLT_MAX);
        } else {
            B.lo[r] = -FLT_MAX;
            B.hi[r] = FLT_MAX;
        }
    }
    return B;
}

__device__ __forceinline__ float centroid(const Box &B, int r) {
    return __fadd_rn(__fmul_rn(B.lo[r], 0.5f), __fmul_rn(B.hi[r], 0.5f));
}

// World boxes (lo, hi as two float4 per instance) and the centroids' bounds (order keys:
// cb[0..2] min, cb[3..5] max).
__global__ void world_boxes_kernel(const ClptInstRec *__restrict__ recs, const ClptScene *__restrict__ meshes, int n,
                                   float4 *__restrict__ boxes, unsigned *__restrict__ cb) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned kmin[3] = { 0xffffffffu, 0xffffffffu, 0xffffffffu }, kmax[3] = { 0u, 0u, 0u };
    if (k < n) {
        const ClptInstRec R = recs[k];
        const ClptScene &M = meshes[R.mesh];
        const Box B = world_box(R, M.root_min, M.root_max);
        boxes[2 * k] = make_float4(B.lo[0], B.lo[1], B.lo[2], 0.0f);
        boxes[2 * k + 1] = make_float4(B.hi[0], B.hi[1], B.hi[2], 0.0f);
        for (int r = 0; r < 3; r++) kmin[r] = kmax[r] = order_key(centroid(B, r));
    }
    for (int r = 0; r < 3; r++) {
        const unsigned lo = __reduce_min_sync(0xffffffffu, kmin[r]), hi = __reduce_max_sync(0xffffffffu, kmax[r]);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(cb + r, lo);
            atomicMax(cb + 3 + r, hi);
        }
    }
}

__device__ __forceinline__ unsigned expand10(unsigned v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

// Centroid axis r -> 10 bits: floor((c - min) * (1024 / (max - min))) clamped to [0, 1023]; NaN
// (a zero extent) -> 0.
__device__ __forceinline__ unsigned quantise(float c, float lo, float hi) {
    const float s = __fdiv_rn(1024.0f, __fsub_rn(hi, lo));
    const float f = floorf(__fmul_rn(__fsub_rn(c, lo), s));
    return f >= 0.0f ? (f < 1023.0f ? (unsigned)f : 1023u) : 0u;
}

__global__ void keys_kernel(const float4 *__restrict__ boxes, const unsigned *__restrict__ cb, int n,
                            unsigned long long *__restrict__ keys) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const float4 lo = boxes[2 * k], hi = boxes[2 * k + 1];
    Box B = { { lo.x, lo.y, lo.z }, { hi.x, hi.y, hi.z } };
    unsigned q[3];
    for (int r = 0; r < 3; r++) q[r] = quantise(centroid(B, r), order_value(cb[r]), order_value(cb[3 + r]));
    const unsigned morton = expand10(q[0]) * 4u + expand10(q[1]) * 2u + expand10(q[2]);
    keys[k] = ((unsigned long long)morton << 20) | (unsigned long long)k;
}

// length of the common prefix of sorted keys i and j; -1 outside [0, n)
__device__ __forceinline__ int delta(const unsigned long long *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    return __clzll(keys[i] ^ keys[j]);
}

// Internal node i: its key range, its split, and the parent links of its two children
// (up = parent << 1 | slot; leaves by sorted position, internal nodes by index).
__global__ void hierarchy_kernel(const unsigned long long *__restrict__ keys, int n, int *__restrict__ up_leaf,
                                 int *__restrict__ up_node, float4 *__restrict__ nodes) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (n == 1) { // one instance: the root's slot 1 is an empty box
        if (i == 0) {
            up_leaf[0] = 0;
            nodes[2] = make_float4(FLT_MAX, FLT_MAX, FLT_MAX, __int_as_float(-1));
            nodes[3] = make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, 0.0f);
        }
        return;
    }
    if (i >= n - 1) return;
    const int d = delta(keys, n, i, i + 1) > delta(keys, n, i, i - 1) ? 1 : -1;
    const int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1) {
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    }
    const int j = i + l * d;
    const int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int div = 2;; div <<= 1) {
        const int t = (l + div - 1) / div;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    if (min(i, j) == gamma) up_leaf[gamma] = i << 1;
    else up_node[gamma] = i << 1;
    if (max(i, j) == gamma + 1) up_leaf[gamma + 1] = (i << 1) | 1;
    else up_node[gamma + 1] = (i << 1) | 1;
}

// One thread per leaf: write its box into its parent's slot; the second arrival at a node writes
// the union of the node's two slots into the node's own parent, and so on up to the root.
__global__ void boxes_kernel(const unsigned long long *__restrict__ keys, const float4 *__restrict__ boxes, int n,
                             const int *__restrict__ up_leaf, const int *__restrict__ up_node,
                             unsigned *__restrict__ arrivals, float4 *nodes) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int k = (int)(keys[p] & 0xFFFFFull);
    float4 lo = boxes[2 * k], hi = boxes[2 * k + 1];
    int ref = -1 - k, up = up_leaf[p];
    for (;;) {
        const int node = up >> 1, slot = up & 1;
        nodes[4 * node + 2 * slot] = make_float4(lo.x, lo.y, lo.z, __int_as_float(ref));
        nodes[4 * node + 2 * slot + 1] = make_float4(hi.x, hi.y, hi.z, 0.0f);
        if (node == 0) return;
        __threadfence();
        if (atomicAdd(arrivals + node, 1u) == 0u) return;
        __threadfence();
        const float4 l0 = __ldcg(nodes + 4 * node), h0 = __ldcg(nodes + 4 * node + 1);
        const float4 l1 = __ldcg(nodes + 4 * node + 2), h1 = __ldcg(nodes + 4 * node + 3);
        lo = make_float4(fmin_(l0.x, l1.x), fmin_(l0.y, l1.y), fmin_(l0.z, l1.z), 0.0f);
        hi = make_float4(fmax_(h0.x, h1.x), fmax_(h0.y, h1.y), fmax_(h0.z, h1.z), 0.0f);
        ref = node;
        up = up_node[node];
    }
}

// Scratch layout: boxes (2n float4), keys in and out (2n u64), up_leaf, up_node, arrivals (n int
// each), centroid bounds (8 u32), then the sort's workspace.
struct Layout {
    size_t boxes, keys_in, keys_out, up_leaf, up_node, arrivals, cb, sort, sort_bytes, total;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

Layout layout_for(int n) {
    Layout L;
    size_t at = 0;
    L.boxes = at, at = align256(at + 2 * (size_t)n * sizeof(float4));
    L.keys_in = at, at = align256(at + (size_t)n * 8);
    L.keys_out = at, at = align256(at + (size_t)n * 8);
    L.up_leaf = at, at = align256(at + (size_t)n * 4);
    L.up_node = at, at = align256(at + (size_t)n * 4);
    L.arrivals = at, at = align256(at + (size_t)n * 4);
    L.cb = at, at = align256(at + 8 * 4);
    L.sort_bytes = 0;
    HANDLE_ERR(cub::DeviceRadixSort::SortKeys(nullptr, L.sort_bytes, (const unsigned long long *)nullptr,
                                              (unsigned long long *)nullptr, n, 0, 50));
    L.sort = at, at = align256(at + L.sort_bytes);
    L.total = at;
    return L;
}

} // namespace

size_t clpt_instance_tree_scratch_bytes(int n) { return layout_for(n).total; }

void clpt_build_instance_tree(const ClptInstRec *recs, const ClptScene *meshes, int n, float4 *nodes, void *scratch,
                              cudaStream_t stream) {
    if (n < 1) return;
    const Layout L = layout_for(n);
    char *base = (char *)scratch;
    float4 *boxes = (float4 *)(base + L.boxes);
    unsigned long long *keys_in = (unsigned long long *)(base + L.keys_in);
    unsigned long long *keys_out = (unsigned long long *)(base + L.keys_out);
    int *up_leaf = (int *)(base + L.up_leaf), *up_node = (int *)(base + L.up_node);
    unsigned *arrivals = (unsigned *)(base + L.arrivals), *cb = (unsigned *)(base + L.cb);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    HANDLE_ERR(cudaMemsetAsync(cb, 0xff, 3 * sizeof(unsigned), stream));
    HANDLE_ERR(cudaMemsetAsync(cb + 3, 0, 3 * sizeof(unsigned), stream));
    HANDLE_ERR(cudaMemsetAsync(arrivals, 0, (size_t)n * sizeof(unsigned), stream));
    world_boxes_kernel<<<blocks, 256, 0, stream>>>(recs, meshes, n, boxes, cb);
    keys_kernel<<<blocks, 256, 0, stream>>>(boxes, cb, n, keys_in);
    size_t sort_bytes = L.sort_bytes;
    HANDLE_ERR(cub::DeviceRadixSort::SortKeys(base + L.sort, sort_bytes, keys_in, keys_out, n, 0, 50, stream));
    hierarchy_kernel<<<blocks, 256, 0, stream>>>(keys_out, n, up_leaf, up_node, nodes);
    boxes_kernel<<<blocks, 256, 0, stream>>>(keys_out, boxes, n, up_leaf, up_node, arrivals, nodes);
    HANDLE_ERR(cudaGetLastError());
}
