// scene_pack.h -- host-side re-layout of an uploaded scene (internal).
#pragma once

#include <stdint.h>

#include <stddef.h>

#include <string>
#include <vector>

#include "clpt_types.h"

struct ClptNode8 {
    uint32_t x, y;
};
struct ClptFloat4 {
    float x, y, z, w;
};

// A grow-only array in host memory obtained from caller-supplied functions: the
// library hands in cudaMallocHost / cudaFreeHost, so the packed scene is written
// straight into page-locked memory and uploads run at full PCIe speed instead of
// being staged by the driver (measured at 1M triangles: 48 ms -> see DESIGN.md).
typedef void *(*clpt_host_alloc_fn)(size_t bytes);
typedef void (*clpt_host_free_fn)(void *ptr);
extern clpt_host_alloc_fn clpt_pack_alloc; // default malloc
extern clpt_host_free_fn clpt_pack_free;   // default free

template <typename T>
class ClptStaging {
  public:
    ClptStaging() = default;
    ClptStaging(const ClptStaging &) = delete;
    ClptStaging &operator=(const ClptStaging &) = delete;
    ~ClptStaging() { release(); }
    void resize(size_t n) {
        if (n > cap_) {
            release();
            ptr_ = static_cast<T *>(clpt_pack_alloc((n ? n : 1) * sizeof(T)));
            cap_ = n;
        }
        size_ = n;
    }
    void release() {
        if (ptr_) clpt_pack_free(ptr_);
        ptr_ = nullptr;
        cap_ = size_ = 0;
    }
    T *data() { return ptr_; }
    const T *data() const { return ptr_; }
    size_t size() const { return size_; }
    T &operator[](size_t i) { return ptr_[i]; }
    const T &operator[](size_t i) const { return ptr_[i]; }

  private:
    T *ptr_ = nullptr;
    size_t size_ = 0, cap_ = 0;
};

// A "fat" leaf for the automatic engine choice: trees whose triangle slots mostly live in
// leaves of at least this many triangles are rendered by engine 2.
#define CLPT_COOP_LEAF_MIN 8
#define CLPT_FAT_ENGINE_MIN_REFS 500000

// What a re-layout computes besides its arrays.  Both re-layouts fill it: clpt_pack_scene
// here and its device twin clpt_gpu_pack (kd_build_gpu.h).
struct ClptLayoutInfo {
    int n_nodes = 0, n_leaves = 0, n_refs = 0;
    float root_min[3] = {}, root_max[3] = {};
    int lut_dim[3] = { 1, 1, 1 };
    float lut_scale[3] = { 0, 0, 0 };
    size_t fat_refs = 0; // triangle slots living in leaves of >= CLPT_COOP_LEAF_MIN triangles
};

struct ClptPackedScene : ClptLayoutInfo {
    ClptStaging<ClptNode8> nodes;
    ClptStaging<ClptFloat4> leaves; // 4 per leaf
    ClptStaging<ClptFloat4> tri;    // 3 per leaf triangle slot
    ClptStaging<ClptFloat4> flat_n; // 1 per primitive: flat normal, w = 1 if the primitive uses vertex normals
    ClptStaging<int> lut;           // start-node table, lut_dim[0] fastest
    int n_prims = 0;
};

// Returns false and fills `err` when the input is inconsistent (index out of
// range, malformed node); the caller treats that as a fatal error.
bool clpt_pack_scene(const kdnode *nodes, size_t n_nodes, const int *tri_indices, size_t n_refs,
                     const cl_int3 *corners, size_t n_corners, const Vector4 *verts, size_t n_verts,
                     size_t n_norms, ClptPackedScene &out, std::string &err);
