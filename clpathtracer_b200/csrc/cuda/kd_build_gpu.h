// kd_build_gpu.h -- device-side kd-tree construction and re-layout (internal).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>

#include "dev_buf.h"
#include "scene_pack.h"

struct ClptGpuBuildParams {
    int max_depth = 0;  // <= 0: 8 + 1.3 log2(triangles)
    int min_split = 2;  // nodes with fewer references become leaves without looking for a plane
    float ct = 1.0f, ci = 1.0f, empty_bonus = 0.9f; // the surface-area heuristic's constants (as build_kd_sah)
};

// The tree in the reference's wire format, in device memory (owned by the caller's
// ClptGpuTree, reused and grown across builds).
struct ClptGpuTree {
    DevBuf<int> wire;        // 17 words per node (include/kd_tree.h:31-50)
    DevBuf<int> tri_indices; // leaf triangle lists
    int n_nodes = 0, n_refs = 0, levels = 0;
    void release() {
        wire.release();
        tri_indices.release();
        *this = ClptGpuTree();
    }
};

// Builds the tree of `n_tris` triangles (corners: three int4 {v, vn, vt, 0} per triangle,
// verts: float4) on stream `s`.  Meshes of up to 2^18 triangles: the whole build is one recorded
// CUDA graph (level counts stay on the device, launches sized by fixed capacities), replayed
// while mesh size and buffers stay the same, one synchronisation at the end.  Larger meshes,
// or a mesh that outgrows the recorded capacities: level by level, one synchronisation per
// level (two counters come back to size the next level exactly).  Both give the same tree.
// False + message on malformed input.
bool clpt_gpu_build(const float4 *verts, int n_verts, const int4 *corners, int n_tris, const ClptGpuBuildParams &P,
                    ClptGpuTree &out, cudaStream_t s, char *err, size_t errlen);
bool clpt_gpu_build_was_recorded(void); // the last build ran as the recorded graph
void clpt_gpu_build_release(void);

// The traversal layout (clpt_device.cuh) in device memory.  Two producers write it: the host
// path uploads what clpt_pack_scene made, the device path re-lays the wire format out in place
// (clpt_gpu_pack).  Both grow the buffers with DevBuf::reserve and never shrink them.
struct ClptSceneLayout : ClptLayoutInfo {
    DevBuf<uint2> nodes;
    DevBuf<float4> leaves, tri, flat_n;
    DevBuf<int> lut;
    void release() {
        nodes.release();
        leaves.release();
        tri.release();
        flat_n.release();
        lut.release();
    }
};

// Device twin of clpt_pack_scene (scene_pack.cpp): wire format -> traversal layout, same
// numbering, same bytes.
bool clpt_gpu_pack(const ClptGpuTree &tree, const float4 *verts, const int4 *corners, int n_prims, ClptSceneLayout &out,
                   cudaStream_t s, char *err, size_t errlen);
