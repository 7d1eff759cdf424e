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

// INST: the instanced variant (clpt_trace.cuh: scene_hit), launched only while instances exist.
template <int MODE, bool COUNT, bool SHARE, bool INST>
__device__ __forceinline__ V3 trace_sample(const ClptScene &S, const ClptInstances &I, const ClptFrame &F, int x, int y, unsigned pixel,
                                           unsigned sample, bool aov, Counters &cn_in, int sub, int log2_k) {
    Counters scratch = { 0, 0, 0, 0, 0, 0 };
    Counters &cn = (SHARE && sub != 0) ? scratch : cn_in; // shading is counted once per ray
    V3 o, d;
    primary_ray(F, x, y, pixel, sample, o, d);
    if (MODE == 2) {
        V3 Lsum = mk(0.0f, 0.0f, 0.0f), T = mk(1.0f, 1.0f, 1.0f);
        for (int seg = 0; seg < F.depth; seg++) {
            const Hit h = scene_hit<COUNT, SHARE, INST>(S, I, o, d, F.max_leaf_visits, cn_in, sub, log2_k);
            if (seg == 0 && aov) write_hit_aov<COUNT, INST>(S, I, F, h, o, d, x, y);
            if (h.ref < 0) {
                Lsum = vadd(Lsum, T);
                break;
            }
            const V3 nrm = shading_normal<COUNT, INST>(S, I, h, o, d, cn);
            float al[3] = { 0.5f, 0.5f, 0.5f }, em[3] = { 0.0f, 0.0f, 0.0f };
            int kind = 0;
            if (S.n_materials > 0) {
                int m;
                if (INST && h.inst >= 0) m = I.rec[h.inst].material;
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
// CLPT_FAT_MIN_BLOCKS (engine 2, trees with fat leaves).  INST: walks the instances of I after the
// base scene; the variants without it ignore I and are the kernels of a frame without instances.
template <int MODE, bool COUNT, int VARIANT, bool INST>
__global__ void __launch_bounds__(256, VARIANT == 1 ? CLPT_FAT_MIN_BLOCKS : CLPT_MIN_BLOCKS)
render_kernel(const __grid_constant__ ClptScene S, const __grid_constant__ ClptFrame F,
              const __grid_constant__ ClptInstances I) {
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
                colour = trace_sample<MODE, COUNT, VARIANT == 1, INST>(S, I, F, x, y, pixel, F.sample_base + (unsigned)s,
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

template <int MODE, bool INST>
void launch_variant(const ClptScene &scene, const ClptFrame &frame, const ClptInstances &inst, unsigned grid,
                    cudaStream_t stream) {
    const bool fat = (frame.flags & CLPT_F_FAT) != 0;
    if (frame.flags & CLPT_F_COUNTERS) {
        if (fat) render_kernel<MODE, true, 1, INST><<<grid, 256, 0, stream>>>(scene, frame, inst);
        else render_kernel<MODE, true, 0, INST><<<grid, 256, 0, stream>>>(scene, frame, inst);
    } else {
        if (fat) render_kernel<MODE, false, 1, INST><<<grid, 256, 0, stream>>>(scene, frame, inst);
        else render_kernel<MODE, false, 0, INST><<<grid, 256, 0, stream>>>(scene, frame, inst);
    }
}

template <int MODE>
void launch_mode(const ClptScene &scene, const ClptFrame &frame, const ClptInstances &inst, unsigned grid,
                 cudaStream_t stream) {
    if (inst.count > 0) launch_variant<MODE, true>(scene, frame, inst, grid, stream);
    else launch_variant<MODE, false>(scene, frame, inst, grid, stream);
}

} // namespace

int clpt_render_block_rows(const ClptFrame &frame) {
    int tw, th;
    warp_tile_dims(5 - frame.log2_sample_lanes - ((frame.flags & CLPT_F_FAT) ? frame.log2_lanes_per_ray : 0), tw, th);
    const int block_h = 2 * th;
    return (frame.local_rows + block_h - 1) / block_h;
}

int clpt_render_blocks_per_sm(int engine) { return engine == 2 ? CLPT_FAT_MIN_BLOCKS : CLPT_MIN_BLOCKS; }

void clpt_launch_render(const ClptScene &scene, const ClptFrame &frame_in, const ClptInstances &inst, int sm_count,
                        cudaStream_t stream) {
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
    case 0: launch_mode<0>(scene, frame, inst, grid, stream); break;
    case 1: launch_mode<1>(scene, frame, inst, grid, stream); break;
    default: launch_mode<2>(scene, frame, inst, grid, stream); break;
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
    return reinterpret_cast<const void *>(&render_kernel<0, false, 0, false>);
}
