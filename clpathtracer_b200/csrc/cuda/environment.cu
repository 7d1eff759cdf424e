// environment.cu -- the environment table (modes 2 and 3, DESIGN.md "Environment light").
//
// Built in stream order from the uploaded float32 cube, with no host round trip:
//   1. per texel, the float64 weight w = ((r + g) + b) / (s2c * sqrt(s2c)) at the texel's centre
//      (radiance x solid angle up to a constant), and the largest weight (a warp's maximum, then
//      an atomic max on the weights' bits, which order like the non-negative doubles they are);
//   2. integer weights q = (uint64)(w / wmax * 2^32) and cdf = their exclusive uint64 scan
//      (emitters.cu: clpt_quantise_scan, the emitter table's own steps);
//   3. each texel's record {r, g, b, pdf}, pdf = ((q / Q) * n^2) * 0.25, and the header {n, Q}.
// The bytes equal those of the CPU twin (oracle/oracle_env.c: oracle_build_env), whose header is
// the definition.
#include <math_constants.h>

#include "CLHandler.h"
#include "clpt_device.cuh"

namespace {

__global__ void env_weights_kernel(const float *__restrict__ rgb, int n, int texels, double *__restrict__ weight,
                                   unsigned long long *__restrict__ wmax, int *__restrict__ count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *count = texels;
    double w = 0.0;
    if (i < texels) {
        const int nn = n * n, rem = i % nn, row = rem / n, col = rem - row * n;
        const double N = (double)n;
        const double ac = __dadd_rn(__dmul_rn(__ddiv_rn(__dadd_rn((double)col, 0.5), N), 2.0), -1.0);
        const double bc = __dadd_rn(__dmul_rn(__ddiv_rn(__dadd_rn((double)row, 0.5), N), 2.0), -1.0);
        const double s2 = __dadd_rn(__dadd_rn(1.0, __dmul_rn(ac, ac)), __dmul_rn(bc, bc));
        const float *c = rgb + 3 * (size_t)i;
        const double e = __dadd_rn(__dadd_rn((double)c[0], (double)c[1]), (double)c[2]);
        const double ww = __ddiv_rn(e, __dmul_rn(s2, __dsqrt_rn(s2)));
        w = (ww > 0.0 && ww < CUDART_INF) ? ww : 0.0;
        weight[i] = w;
    }
    unsigned long long bits = (unsigned long long)__double_as_longlong(w);
    for (int off = 16; off > 0; off >>= 1) {
        const unsigned long long o = __shfl_down_sync(0xffffffffu, bits, off);
        bits = o > bits ? o : bits;
    }
    if ((threadIdx.x & 31) == 0 && bits) atomicMax(wmax, bits);
}

__global__ void env_finish_kernel(const float *__restrict__ rgb, const unsigned long long *__restrict__ q,
                                  const unsigned long long *__restrict__ cdf, int n, int texels, float4 *__restrict__ tex,
                                  unsigned long long *__restrict__ header) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long Q = cdf[texels];
    if (i == 0) {
        header[0] = (unsigned long long)n;
        header[1] = Q;
    }
    if (i >= texels) return;
    const float *c = rgb + 3 * (size_t)i;
    const double nn = __dmul_rn((double)n, (double)n);
    const float pdf =
        q[i] > 0ull ? __double2float_rn(__dmul_rn(__dmul_rn(__ddiv_rn((double)q[i], __ull2double_rn(Q)), nn), 0.25)) : 0.0f;
    tex[i] = make_float4(c[0], c[1], c[2], pdf);
}

struct Layout {
    size_t weight, wmax, count, q, temp, total;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

Layout layout_for(int texels) {
    Layout L;
    size_t at = 0;
    L.weight = at, at = align256(at + (size_t)texels * 8);
    L.wmax = at, at = align256(at + 8);
    L.count = at, at = align256(at + 4);
    L.q = at, at = align256(at + ((size_t)texels + 1) * 8);
    L.temp = at, at = align256(at + clpt_quantise_scan_temp_bytes(texels));
    L.total = at;
    return L;
}

} // namespace

size_t clpt_environment_scratch_bytes(int n) { return layout_for(6 * n * n).total; }

void clpt_build_environment(const float *rgb, int n, float4 *tex, unsigned long long *cdf, unsigned long long *header,
                            void *scratch, cudaStream_t stream) {
    const int texels = 6 * n * n;
    const Layout L = layout_for(texels);
    char *base = (char *)scratch;
    double *weight = (double *)(base + L.weight);
    unsigned long long *wmax = (unsigned long long *)(base + L.wmax), *q = (unsigned long long *)(base + L.q);
    int *count = (int *)(base + L.count);
    const unsigned blocks = (unsigned)((texels + 255) / 256);
    HANDLE_ERR(cudaMemsetAsync(wmax, 0, sizeof(unsigned long long), stream));
    env_weights_kernel<<<blocks, 256, 0, stream>>>(rgb, n, texels, weight, wmax, count);
    clpt_quantise_scan(weight, wmax, count, texels, q, cdf, base + L.temp, stream);
    env_finish_kernel<<<blocks, 256, 0, stream>>>(rgb, q, cdf, n, texels, tex, header);
    HANDLE_ERR(cudaGetLastError());
}
