// clpt_device.cuh -- device-side data layout and launch interface (internal).
//
// HBM layout produced by CLSetMeshes (scene_pack.cpp) from the reference's wire
// format (68-byte packed nodes + tri_indices -> tris -> verts indirection,
// include/kd_tree.h:31-50, src/kernel.cl:333-340):
//
//   nodes   uint2[n_nodes]   8 B per node, siblings adjacent
//             split: x = float bits of the plane, y = (first_child << 2) | axis
//                    children are first_child (p <= plane) and first_child+1
//             leaf : x = leaf record index,        y = 0x80000003 (bit 31 set)
//   leaves  float4[4*n_leaves]  64 B per leaf, 64-byte aligned
//             [0] = min.xyz, int bits of the first triangle slot
//             [1] = max.xyz, int bits of the triangle count
//             [2] = ropes 0..3 (int bits; >= 0: node index in `nodes`; -1: outside;
//                   <= -2: the neighbour is itself a leaf, record -2 - value)
//             [3] = ropes 4..5, 0, 0
//   tri     float4[3*n_refs]    48 B per leaf triangle slot, in leaf order, so a
//                               leaf's triangles are one contiguous run
//             [0] = v0.xyz, int bits of the primitive id
//             [1] = v1 - v0 (fp32, same rounding as kernel.cl:235)
//             [2] = v2 - v0
//   corners int4[3*n_prims], norms float4[]: as uploaded, only read when
//             shading a hit with vertex normals (once per ray)
//   lut     int[gx*gy*gz]       start-node table: a uniform grid over the root box
//             (<= ~2M cells); entry = the deepest node that every point of the
//             cell reaches by the root descent, so a descent may start there
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define CLPT_LEAF_WORD 0x80000003u

struct ClptMaterial {
    float albedo[3];
    int kind;
    float emission[3];
    float pad;
};

struct ClptScene {
    const uint2 *nodes;
    const float4 *leaves;
    const float4 *tri;
    const int4 *corners;
    // Per primitive: xyz = the flat shading normal normalize((v2-v1) x (v3-v1)) (src/kernel.cl:362),
    // evaluated once at scene preparation with the operations the kernel would repeat at every hit;
    // w = 0 when the primitive is flat-shaded, 1 when its first corner carries a vertex normal
    // (the interpolated path, kernel.cl:349-360, then reads `corners` and `norms`).
    const float4 *flat_n;
    const float4 *norms;
    const int *tri_material;
    const ClptMaterial *materials;
    int n_materials;
    int n_nodes, n_leaves, n_refs, n_prims, n_norms;
    float root_min[3], root_max[3];
    // Start-node table: a uniform grid over the root box; cell -> the deepest node
    // the whole (slightly enlarged) cell descends to.  Skips the top of the tree.
    const int *lut;
    int lut_dim[3];
    float lut_scale[3]; // cells per unit length
};

// Rigid instances (CLSetInstances): a mesh with its own tree, walked with the world ray
// mapped into object space.  One record per instance, rewritten by clstate.cu whenever the
// instances or the base scene change.
struct ClptInstanceRec {
    float w2o[12];   // world to object, row-major 3x4 [A | b]
    int material;    // mode 2: the material of every triangle of the instance
    int prim_offset; // base scene's primitives + those of the instances before this one
    int pad[2];
    ClptScene mesh;  // the instance mesh's traversal layout (materials unused)
};

// Instance tree (CLPT_INSTANCES_TREE): one 64-byte record per instance, the CLInstance layout with
// the primitive offset in its first pad word; the mesh is an index into a table of ClptScenes.
struct ClptInstRec {
    float w2o[12];   // world to object, row-major 3x4 [A | b]
    int mesh;        // index into ClptInstances::meshes
    int material;
    int prim_offset;
    int pad;
};

// Instance tree node, four float4s (64 bytes): slot s in [0, 1] is f[2s] = (min.xyz, ref as int
// bits), f[2s + 1] = (max.xyz, 0).  ref >= 0 names an internal node, ref < 0 instance -1 - ref.
// Node 0 is the root.  With one instance, slot 1 of the root is an empty box (min > max).
#define CLPT_TREE_STACK 64 // the tree's depth is at most 50: each split consumes a bit of a 50-bit key

struct ClptInstances {
    const ClptInstanceRec *rec; // list: device table of `count` records
    int count;
    // tree: `count` compact records, the mesh table and the node array (count >= 1)
    const ClptInstRec *crec;
    const ClptScene *meshes;
    const float4 *tree;
};

// instance_tree.cu: builds the tree over the world boxes of n >= 1 instances into `nodes`
// (max(n - 1, 1) records) in stream order, without a host round trip.  `scratch` holds
// clpt_instance_tree_scratch_bytes(n) bytes: world boxes, keys, parent links, arrival flags and
// the sort's workspace.
size_t clpt_instance_tree_scratch_bytes(int n);
void clpt_build_instance_tree(const ClptInstRec *recs, const ClptScene *meshes, int n, float4 *nodes,
                              void *scratch, cudaStream_t stream);

// Emitter table of the base scene (mode 3, DESIGN.md "Light sampling (mode 3)"): the primitives
// listed by a leaf whose material emits, in ascending primitive id.  Record i is four float4s,
// {v0, prim bits}, {e1, area pdf}, {e2, 0}, {flat normal, 0}; cdf[i] is the exclusive uint64 prefix
// sum of the integer weights; map[prim] = i or -1; header = {emitter count, total weight Q}.  The
// counts stay on the device: the table is built without a host round trip.
struct ClptEmitters {
    const float4 *rec;
    const unsigned long long *cdf;
    const int *map;
    const unsigned long long *header;
};

// emitters.cu: builds the table of the scene S (materials and tri_material included) in stream
// order.  Capacities: rec 4 * max(n_prims, 1) float4s, cdf n_prims + 1, map max(n_prims, 1),
// header 2; `scratch` holds clpt_emitter_scratch_bytes(n_prims) bytes.
size_t clpt_emitter_scratch_bytes(int n_prims);
void clpt_build_emitters(const ClptScene &S, float4 *rec, unsigned long long *cdf, int *map,
                         unsigned long long *header, void *scratch, cudaStream_t stream);

// emitters.cu, shared with the environment table: q[i] = (uint64)(weight[i] / wmax * 2^32) for
// i < *count (0 when wmax = 0) and 0 up to n, then cdf = the exclusive uint64 scan of q over n + 1
// items.  `temp` holds clpt_quantise_scan_temp_bytes(n) bytes.
size_t clpt_quantise_scan_temp_bytes(int n);
void clpt_quantise_scan(const double *weight, const unsigned long long *wmax, const int *count, int n,
                        unsigned long long *q, unsigned long long *cdf, void *temp, cudaStream_t stream);

// Environment (modes 2 and 3, DESIGN.md "Environment light"): a cube map of n x n texels per face,
// faces +X, -X, +Y, -Y, +Z, -Z, texel (face * n + row) * n + col.  tex[i] = {r, g, b, pdf}, pdf the
// texel's density per unit area of face coordinates; cdf[i] the exclusive uint64 prefix sum of the
// integer weights; header = {n, total weight Q}.  n = 0: no environment (the kernels without one run).
struct ClptEnvironment {
    const float4 *tex;
    const unsigned long long *cdf;
    const unsigned long long *header;
    int n;
};

// environment.cu: builds the table of rgb float[6 n^2][3] (on the device) in stream order.
// Capacities: tex 6 n^2, cdf 6 n^2 + 1, header 2; `scratch` holds clpt_environment_scratch_bytes(n).
size_t clpt_environment_scratch_bytes(int n);
void clpt_build_environment(const float *rgb, int n, float4 *tex, unsigned long long *cdf, unsigned long long *header,
                            void *scratch, cudaStream_t stream);

#define CLPT_MAX_PEERS 8

struct ClptFrame {
    float cam[16]; // row-major inverse camera matrix
    // Per-frame constants of the camera ray (src/kernel.cl:443-449), evaluated once on the host with
    // the same IEEE single-precision operations the kernel would repeat for every sample: the eye
    // (column 2 of the matrix over its w) and half the image size.
    float eye[3], half_width, half_height;
    int width, height;
    int mode, depth, spp, flags;
    int log2_sample_lanes;       // lanes per pixel = 1 << this (largest power of two <= min(spp, 32))
    int log2_warps_per_pixel;    // warps of a block sharing one pixel's samples (> 0 only at >= 64 spp)
    int log2_lanes_per_ray;      // engine 2 at 1 spp: neighbouring lanes that walk the same ray and share its
                                 // leaves' triangle runs (0 or 1); a warp tile is then 32 >> this pixels
    unsigned int seed, sample_base;
    int max_leaf_visits;
    int rank, nranks, tile_rows; // row-tile sharding; nranks == 1 -> whole image
    int local_rows;              // rows this rank renders (slab height)
    float4 *target;              // slab (nranks > 1) or the image itself
    // Progressive frames (CLPT_F_ACCUMULATE): four 64-bit words per pixel of the WHOLE image -- the
    // sums of the samples' r, g, b in 2^-32 fixed point and the sample count.  Integer sums do not
    // depend on the order of the additions, so the accumulated frame is the same bits whether one
    // GPU adds the samples one after the other or N GPUs each add every N-th sample and the
    // read-back adds the N buffers (which is how progressive frames are spread over GPUs: by
    // sample, every rank renders the whole frame).
    unsigned long long *accum;
    // Direct placement across GPUs: when n_peer_images > 0, every finished pixel is also
    // stored at its image position in each of these full-size frames -- this rank's own
    // and, through peer mappings over NVLink, every other rank's -- so the frame is
    // assembled by the render kernel itself and no gather pass follows it.
    float4 *peer_image[CLPT_MAX_PEERS];
    int n_peer_images;
    int *aov_prim;               // full-image indexed, may be null
    float *aov_t;
    float2 *aov_uv;
    unsigned long long *counters; // 6 counters, may be null
    unsigned int *work_counter;   // warp-tile claim counter of the persistent render kernel
    // Claim direction: warp tiles are handed out in screen order, top to bottom, or with
    // CLPT_F_REVERSE bottom to top.  Every warp tile adds its duration to
    // row_cost[its block row] (null = not recorded); CLExecute looks at where one frame's
    // cost sits and points the next frame's claims so that they END at the cheap side.
    // row_cost[row_count + block row] keeps the row's LONGEST warp tile (what a frame's tail is made of).
    unsigned long long *row_cost;
    int row_count;
    int blocks_x, n_warp_tiles;   // filled in by clpt_launch_render
};

#ifdef __CUDACC__
// Sample colour -> 2^-32 fixed point, round to nearest even; negative and NaN -> 0, saturates at
// 2^20 (oracle_kernel.c: fix32).  The product with 2^32 is exact.
__device__ __forceinline__ unsigned long long clpt_fix32(float x) {
    if (!(x > 0.0f)) return 0ull;
    if (x >= 1048576.0f) return 1ull << 52;
    return __float2ull_rn(x * 4294967296.0f);
}
// float in [0,1] -> UNORM8, round to nearest even, NaN -> 0: a UNORM8 image write.
__device__ __forceinline__ unsigned clpt_to_unorm8(float v) {
    return (unsigned)__float2int_rn(__saturatef(v) * 255.0f);
}
#endif

enum { CLPT_F_JITTER = 1, CLPT_F_ACCUMULATE = 2, CLPT_F_COUNTERS = 4, CLPT_F_REVERSE = 0x100 /* internal */,
       CLPT_F_FAT = 0x200 /* internal: engine 2, the kernel compiled for fewer resident blocks (fat leaves) */ };

// render_kernel.cu
// inst.count > 0 launches the instanced variant of the render kernel; `emit` is read in mode 3 only;
// env.n > 0 launches the variant with the environment in modes 2 and 3 (modes 0 and 1 ignore it)
void clpt_launch_render(const ClptScene &scene, const ClptFrame &frame, const ClptInstances &inst,
                        const ClptEmitters &emit, const ClptEnvironment &env, int sm_count, cudaStream_t stream);
int clpt_render_blocks_per_sm(int engine);          // resident 256-thread blocks per SM the render kernel is compiled for
int clpt_render_block_rows(const ClptFrame &frame); // rows of blocks the launch will walk (size of row_cost)
void clpt_launch_deinterleave(const float4 *gathered, float4 *image, int width, int height,
                              int nranks, int tile_rows, int slab_rows, cudaStream_t stream);
void clpt_launch_fill(float4 *dst, size_t n, float value, cudaStream_t stream);
void clpt_launch_fill_u64(unsigned long long *dst, size_t n, cudaStream_t stream);
void clpt_launch_normalise(const unsigned long long *accum, float4 *dst, size_t n, cudaStream_t stream);
struct ClptFlagPeers {
    unsigned int *flags[CLPT_MAX_PEERS]; // rank r's barrier words (peer mappings; this rank's own at [rank])
};
// Barrier across the ranks of a node through peer-mapped words: word [src * 8] of rank dst's
// array is written by src only.  Epochs only grow.
void clpt_launch_flag_barrier(const ClptFlagPeers &peers, int rank, int nranks, unsigned int epoch,
                              cudaStream_t stream);
void clpt_launch_pack_rgba8(const float4 *src, uchar4 *dst, size_t n, cudaStream_t stream);
const void *clpt_render_kernel_symbol(void);
