// emitters.cu -- the emitter table of the base scene (mode 3, CLPT_MODE_PATH_NEE).
//
// Built in stream order from the resident traversal layout, with no host round trip, so it reads
// the same after CLSetMeshes, CLSetMeshesRaw, CLBuildMeshes and CLRebuildMeshes:
//   1. slot_of[prim] = a triangle slot of a leaf's run that holds the primitive (leaf records give
//      the runs; a slot no leaf covers is never tested and lists nothing; every slot of a primitive
//      holds the same v0, e1, e2, so which one wins the race does not matter);
//   2. flags: listed primitives whose material (tri_material clamped as mode 2 clamps it) has a
//      nonzero emission component;
//   3. their ids compacted in ascending order (CUB select);
//   4. records, float64 areas and weights, the largest weight (an atomic max on the weights'
//      bits, which order like the non-negative doubles they are), the primitive -> emitter map;
//   5. integer weights q = (uint64)(w / wmax * 2^32);
//   6. cdf = exclusive uint64 scan of q (integer sums: the same in any order) -- steps 5 and 6 are
//      clpt_quantise_scan, which the environment table (environment.cu) shares;
//   7. each record's area pdf (q / Q) / area, and the header {n, Q}.
// The bytes equal those of the CPU twin (oracle/oracle_nee.c: oracle_build_emitters), whose header
// is the definition.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <math_constants.h>

#include "CLHandler.h"
#include "clpt_device.cuh"

namespace {

// one thread per leaf record: its triangle run [first, first + count)
__global__ void slots_kernel(const float4 *__restrict__ leaves, int n_leaves, const float4 *__restrict__ tri,
                             int *__restrict__ slot_of) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_leaves) return;
    const int first = __float_as_int(leaves[4 * (size_t)l].w), count = __float_as_int(leaves[4 * (size_t)l + 1].w);
    for (int s = first; s < first + count; s++) slot_of[__float_as_int(tri[3 * (size_t)s].w)] = s;
}

__device__ __forceinline__ int material_of(const ClptScene &S, int prim) {
    int m = S.tri_material ? S.tri_material[prim] : 0;
    if (m < 0 || m >= S.n_materials) m = 0;
    return m;
}

__global__ void flags_kernel(const __grid_constant__ ClptScene S, const int *__restrict__ slot_of,
                             unsigned char *__restrict__ flags) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= S.n_prims) return;
    bool emits = false;
    if (slot_of[p] >= 0 && S.n_materials > 0) {
        const float *e = S.materials[material_of(S, p)].emission;
        emits = e[0] != 0.0f || e[1] != 0.0f || e[2] != 0.0f;
    }
    flags[p] = emits ? 1 : 0;
}

__global__ void weights_kernel(const __grid_constant__ ClptScene S, const int *__restrict__ slot_of,
                               const int *__restrict__ ids, const int *__restrict__ count, float4 *__restrict__ rec,
                               int *__restrict__ map, double *__restrict__ area, double *__restrict__ weight,
                               unsigned long long *__restrict__ wmax) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *count) return;
    const int p = ids[i], s = slot_of[p];
    const float4 a = S.tri[3 * (size_t)s], b = S.tri[3 * (size_t)s + 1], c = S.tri[3 * (size_t)s + 2];
    const float4 nl = S.flat_n[p];
    const double ax = b.x, ay = b.y, az = b.z, bx = c.x, by = c.y, bz = c.z;
    const double cx = __dadd_rn(__dmul_rn(ay, bz), -__dmul_rn(az, by));
    const double cy = __dadd_rn(__dmul_rn(az, bx), -__dmul_rn(ax, bz));
    const double cz = __dadd_rn(__dmul_rn(ax, by), -__dmul_rn(ay, bx));
    const double A = __dmul_rn(0.5, __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(cx, cx), __dmul_rn(cy, cy)), __dmul_rn(cz, cz))));
    const float *e = S.materials[material_of(S, p)].emission;
    const double ww = __dmul_rn(A, __dadd_rn(__dadd_rn((double)e[0], (double)e[1]), (double)e[2]));
    const double w = (ww > 0.0 && ww < CUDART_INF) ? ww : 0.0;
    area[i] = A;
    weight[i] = w;
    atomicMax(wmax, (unsigned long long)__double_as_longlong(w));
    rec[4 * (size_t)i] = a; // v0 and the primitive id's bits
    rec[4 * (size_t)i + 1] = make_float4(b.x, b.y, b.z, 0.0f);
    rec[4 * (size_t)i + 2] = make_float4(c.x, c.y, c.z, 0.0f);
    rec[4 * (size_t)i + 3] = make_float4(nl.x, nl.y, nl.z, 0.0f);
    map[p] = i;
}

// q for i < count, 0 for the padding up to n (the scan runs over a fixed n + 1 items)
__global__ void quantise_kernel(const double *__restrict__ weight, const unsigned long long *__restrict__ wmax,
                                const int *__restrict__ count, int n, unsigned long long *__restrict__ q) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    const double m = __longlong_as_double((long long)*wmax);
    q[i] = (i < *count && m > 0.0) ? __double2ull_rz(__dmul_rn(__ddiv_rn(weight[i], m), 4294967296.0)) : 0ull;
}

__global__ void finish_kernel(const unsigned long long *__restrict__ q, const unsigned long long *__restrict__ cdf,
                              const double *__restrict__ area, const int *__restrict__ count, float4 *__restrict__ rec,
                              unsigned long long *__restrict__ header) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = *count;
    const unsigned long long Q = cdf[n];
    if (i == 0) {
        header[0] = (unsigned long long)n;
        header[1] = Q;
    }
    if (i >= n) return;
    rec[4 * (size_t)i + 1].w =
        q[i] > 0ull ? __double2float_rn(__ddiv_rn(__ddiv_rn((double)q[i], __ull2double_rn(Q)), area[i])) : 0.0f;
}

struct Layout {
    size_t slot_of, flags, ids, count, area, weight, wmax, q, temp, temp_bytes, total;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

Layout layout_for(int n) {
    Layout L;
    size_t at = 0;
    L.slot_of = at, at = align256(at + (size_t)n * 4);
    L.flags = at, at = align256(at + (size_t)n);
    L.ids = at, at = align256(at + (size_t)n * 4);
    L.count = at, at = align256(at + 4);
    L.area = at, at = align256(at + (size_t)n * 8);
    L.weight = at, at = align256(at + (size_t)n * 8);
    L.wmax = at, at = align256(at + 8);
    L.q = at, at = align256(at + ((size_t)n + 1) * 8);
    size_t select_bytes = 0;
    HANDLE_ERR(cub::DeviceSelect::Flagged(nullptr, select_bytes, cub::CountingInputIterator<int>(0),
                                          (const unsigned char *)nullptr, (int *)nullptr, (int *)nullptr, n));
    const size_t scan_bytes = clpt_quantise_scan_temp_bytes(n);
    L.temp_bytes = select_bytes > scan_bytes ? select_bytes : scan_bytes;
    L.temp = at, at = align256(at + L.temp_bytes);
    L.total = at;
    return L;
}

} // namespace

size_t clpt_quantise_scan_temp_bytes(int n) {
    size_t scan_bytes = 0;
    HANDLE_ERR(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const unsigned long long *)nullptr,
                                             (unsigned long long *)nullptr, n + 1));
    return scan_bytes;
}

void clpt_quantise_scan(const double *weight, const unsigned long long *wmax, const int *count, int n,
                        unsigned long long *q, unsigned long long *cdf, void *temp, cudaStream_t stream) {
    quantise_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, stream>>>(weight, wmax, count, n, q);
    size_t temp_bytes = clpt_quantise_scan_temp_bytes(n);
    HANDLE_ERR(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, q, cdf, n + 1, stream));
}

size_t clpt_emitter_scratch_bytes(int n_prims) { return layout_for(n_prims).total; }

void clpt_build_emitters(const ClptScene &S, float4 *rec, unsigned long long *cdf, int *map,
                         unsigned long long *header, void *scratch, cudaStream_t stream) {
    const int n = S.n_prims;
    HANDLE_ERR(cudaMemsetAsync(header, 0, 2 * sizeof(unsigned long long), stream));
    if (n < 1) return;
    const Layout L = layout_for(n);
    char *base = (char *)scratch;
    int *slot_of = (int *)(base + L.slot_of), *ids = (int *)(base + L.ids), *count = (int *)(base + L.count);
    unsigned char *flags = (unsigned char *)(base + L.flags);
    double *area = (double *)(base + L.area), *weight = (double *)(base + L.weight);
    unsigned long long *wmax = (unsigned long long *)(base + L.wmax), *q = (unsigned long long *)(base + L.q);
    const unsigned prim_blocks = (unsigned)((n + 255) / 256);
    HANDLE_ERR(cudaMemsetAsync(slot_of, 0xff, (size_t)n * sizeof(int), stream));
    HANDLE_ERR(cudaMemsetAsync(map, 0xff, (size_t)n * sizeof(int), stream));
    HANDLE_ERR(cudaMemsetAsync(wmax, 0, sizeof(unsigned long long), stream));
    if (S.n_leaves > 0)
        slots_kernel<<<(unsigned)((S.n_leaves + 255) / 256), 256, 0, stream>>>(S.leaves, S.n_leaves, S.tri, slot_of);
    flags_kernel<<<prim_blocks, 256, 0, stream>>>(S, slot_of, flags);
    size_t temp_bytes = L.temp_bytes;
    HANDLE_ERR(cub::DeviceSelect::Flagged(base + L.temp, temp_bytes, cub::CountingInputIterator<int>(0), flags, ids,
                                          count, n, stream));
    weights_kernel<<<prim_blocks, 256, 0, stream>>>(S, slot_of, ids, count, rec, map, area, weight, wmax);
    clpt_quantise_scan(weight, wmax, count, n, q, cdf, base + L.temp, stream);
    finish_kernel<<<prim_blocks, 256, 0, stream>>>(q, cdf, area, count, rec, header);
    HANDLE_ERR(cudaGetLastError());
}
