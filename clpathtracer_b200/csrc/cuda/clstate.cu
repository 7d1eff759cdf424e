// clstate.cu -- the CLState.h boundary on top of the CUDA runtime.
//
// Mirrors the reference's render-state layer (src/CLState.c): a file-static
// singleton that owns the device buffers, takes the scene and camera from the
// host, and launches one frame per CLExecute.  Every call is synchronous and
// any failure is fatal, as in the reference (src/error.c:147-154).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "CLHandler.h"
#include "CLState.h"
#include "clpt_device.cuh"
#include "clpt_host.h"
#include "../host/frame_sched.h"
#include "kd_build_gpu.h"
#include "scene_pack.h"

#define CU(call) handle_err((int)(call), __FILE__, __LINE__)

// gl_interop.cu
void clpt_gl_register(unsigned int texture);
void clpt_gl_unregister(void);
bool clpt_gl_registered(void);
void clpt_gl_size(int *width, int *height, cudaStream_t stream);
void clpt_gl_present(const float4 *frame, int width, int height, cudaStream_t stream);

namespace {

[[noreturn]] void fatal(const char *file, int line, const char *what) {
    fprintf(stderr, "%s:%d: CLState Error: %s\n", file, line, what);
    exit(EXIT_FAILURE);
}
#define FATAL(msg) fatal(__FILE__, __LINE__, (msg))

// ---- NCCL, resolved at run time so the library loads on a box without it ----
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                              cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;

void nccl_load() {
    if (g_nccl.lib) return;
    const char *names[] = { "libnccl.so.2", "libnccl.so" };
    for (const char *n : names) {
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) FATAL("NCCL is required for multi-GPU rendering but libnccl.so.2 could not be loaded");
    auto sym = [](const char *name) {
        void *p = dlsym(g_nccl.lib, name);
        if (!p) {
            fprintf(stderr, "missing NCCL symbol %s\n", name);
            exit(EXIT_FAILURE);
        }
        return p;
    };
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))sym("ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))sym("ncclCommInitRank");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))sym("ncclAllGather");
    g_nccl.AllReduce = (decltype(g_nccl.AllReduce))sym("ncclAllReduce");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))sym("ncclCommDestroy");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))sym("ncclGetErrorString");
}

void nccl_check(ncclResult_t r, const char *file, int line) {
    if (r == ncclSuccess) return;
    fprintf(stderr, "%s:%d: NCCL Error: %s\n", file, line,
            g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "unknown");
    exit(EXIT_FAILURE);
}
#define NC(call) nccl_check((call), __FILE__, __LINE__)

ClptPackedScene g_packed; // host staging of the re-laid-out scene (page-locked once CLInit ran)

struct {
    bool inited = false;
    int device = -1; // -1: take $CLPT_DEVICE or 0
    cudaStream_t stream = nullptr;
    cudaDeviceProp prop;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    cudaEvent_t ev_user[8] = {};
    cudaEvent_t ev_build[3] = {};

    kd host_kd = { nullptr, nullptr, nullptr, nullptr, nullptr };
    bool owns_kd = false;

    ClptSceneLayout layout; // the traversal layout of the current scene, whichever path made it
    DevBuf<float4> norms;
    DevBuf<int4> corners;
    // device-side build (CLBuildMeshes): the mesh and the wire-format tree live on the device
    DevBuf<float4> verts;
    ClptGpuBuildParams build_params;
    ClptGpuTree gpu_tree;
    bool scene_on_gpu = false; // gpu_tree is the tree of the current scene
    bool mesh_on_gpu = false;  // verts/corners hold a mesh uploaded by CLBuildMeshes
    float last_build_ms = 0, last_pack_ms = 0;
    DevBuf<unsigned char> objects;
    int objcount = 0;
    DevBuf<ClptMaterial> materials;
    DevBuf<int> tri_material;
    ClptScene scene = {};
    bool have_scene = false;

    // rigid instances: every instance mesh owns its mesh, its wire tree (CLDownloadInstanceKd) and
    // its traversal layout; the device table (ClptInstanceRec) is rewritten before the next frame
    // whenever the instances or the base scene's primitive count may have changed
    struct InstanceMesh {
        DevBuf<float4> verts, norms;
        DevBuf<int4> corners;
        ClptGpuTree tree;
        ClptSceneLayout layout;
        ClptScene scene = {};
    };
    std::vector<std::unique_ptr<InstanceMesh>> inst_meshes;
    std::vector<CLInstance> instances;
    DevBuf<ClptInstanceRec> inst_table;
    bool inst_table_stale = true;

    float cam[16] = { 0 };

    int mode = CLPT_MODE_NORMAL, depth = 2, spp = 1, flags = 0; // depth 2: src/kernel.cl:468
    unsigned seed = 0, sample_base = 0;
    int max_leaf_visits = 4096;

    int width = 0, height = 0;
    bool headless = false, have_image = false;
    DevBuf<float4> image, slab, gathered, scratch;
    // progressive frames: 2^-32 fixed-point sums + sample count, four words per pixel of the whole
    // image (ClptFrame::accum); accum_sum = the ranks' buffers added up for a read-back
    DevBuf<unsigned long long> accum, accum_sum;
    bool aov = false;
    DevBuf<int> aov_prim;
    DevBuf<float> aov_t;
    DevBuf<float2> aov_uv;
    DevBuf<unsigned long long> counters;
    DevBuf<unsigned int> work_counter;
    // claim direction (ClptFrame::row_cost): where this frame's cost sits points the next frame
    DevBuf<unsigned long long> row_cost;
    unsigned long long *host_row_cost = nullptr; // pinned
    int row_capacity = 0;
    int row_count = 0;         // rows the current direction was measured on
    long long row_key[8] = {}; // ... and under which image / sharding / parameters
    bool claim_reverse = false;

    unsigned long long frames_rendered = 0;
    unsigned long long host_counters[6] = { 0 };
    float last_kernel_ms = 0;
    int last_launches = 0;
    DevBuf<unsigned char> l2_flush;
    // Read-back pipeline (CLReadImageAsync): two device staging buffers; the frame is copied or
    // packed into one on the library's stream, and travels to the host on a second stream while
    // the next frame renders.
    cudaStream_t copy_stream = nullptr;
    struct ReadSlot {
        DevBuf<unsigned char> staging;
        cudaEvent_t ready = nullptr, done = nullptr;
        bool in_flight = false;
        unsigned long long ticket = 0;
    } rd[2];
    unsigned long long rd_issued = 0;
    int engine = 0;      // 0 auto, 1 full occupancy, 2 fat-leaf variant (fewer resident blocks)
    int auto_engine = 1; // what "auto" means for the current tree (decided in adopt_layout)
    int last_engine = 1;

    int rank = 0, nranks = 1, tile_rows = 8;
    ncclComm_t comm = nullptr;
    int comm_ranks = 0;
    // direct placement (peer-mapped frames), see p2p_setup
    bool p2p = false;
    int p2p_self = -1; // this rank's slot in peer_image (its own frame, not a mapping)
    float4 *peer_image[CLPT_MAX_PEERS] = {};
    // flag-word barrier: every rank owns one word per peer (32 B apart) in `flags`, mapped by all
    DevBuf<unsigned int> bar_flags;
    unsigned int *peer_flags[CLPT_MAX_PEERS] = {};
    unsigned int flag_epoch = 0;
    DevBuf<int> dist_word;           // operand of the barrier all-reduce
    DevBuf<unsigned char> dist_xchg; // handle exchange staging
} St;

void require_init(const char *who) {
    if (!St.inited) {
        fprintf(stderr, "%s: CLInit has not been called\n", who);
        exit(EXIT_FAILURE);
    }
}

int slab_rows_for(int height) {
    const int tiles = (height + St.tile_rows - 1) / St.tile_rows;
    const int per_rank = (tiles + St.nranks - 1) / St.nranks;
    return per_rank * St.tile_rows;
}

int local_rows_for(int height) {
    // rows of the slab that map to real image rows for this rank
    const int tiles = (height + St.tile_rows - 1) / St.tile_rows;
    int mine = 0;
    for (int t = St.rank; t < tiles; t += St.nranks) mine++;
    return mine * St.tile_rows;
}

// The traversal fields of a scene record: layout L of a mesh with these corners and normals.
void set_scene_mesh(ClptScene &S, const ClptSceneLayout &L, const DevBuf<int4> &corners, const DevBuf<float4> &norms) {
    S.nodes = L.nodes.ptr;
    S.leaves = L.leaves.ptr;
    S.tri = L.tri.ptr;
    S.corners = corners.ptr;
    S.flat_n = L.flat_n.ptr;
    S.lut = L.lut.ptr;
    S.norms = norms.ptr;
    S.n_norms = (int)norms.count;
    S.n_nodes = L.n_nodes;
    S.n_leaves = L.n_leaves;
    S.n_refs = L.n_refs;
    for (int a = 0; a < 3; a++) {
        S.root_min[a] = L.root_min[a];
        S.root_max[a] = L.root_max[a];
        S.lut_dim[a] = L.lut_dim[a];
        S.lut_scale[a] = L.lut_scale[a];
    }
}

void rebuild_scene_struct() {
    ClptScene &S = St.scene;
    set_scene_mesh(S, St.layout, St.corners, St.norms);
    S.tri_material = St.tri_material.ptr;
    S.materials = St.materials.ptr;
    S.n_materials = (int)St.materials.count;
}

// St.layout holds a new scene of `n_prims` primitives: point the launch at it and choose the engine.
void adopt_layout(int n_prims) {
    const ClptSceneLayout &L = St.layout;
    St.scene.n_prims = n_prims;
    rebuild_scene_struct();
    St.have_scene = true;
    St.inst_table_stale = true; // the instances' primitive ids follow the base scene's
    // "automatic" engine for this tree: the fat-leaf variant when most triangle slots live in
    // fat leaves AND the tree is big (the reference builder's DEPTH-15 trees from a few hundred
    // thousand triangles up; measured at 100k triangles engine 1 is still 10% faster)
    St.auto_engine = (L.n_refs >= CLPT_FAT_ENGINE_MIN_REFS && L.fat_refs * 2 > (size_t)L.n_refs) ? 2 : 1;
    if (const char *e = getenv("CLPT_ENGINE")) {
        if (atoi(e) == 1 || atoi(e) == 2) St.auto_engine = atoi(e);
    }
}

// Host staging -> St.layout, one copy per array on the library's stream.
template <typename T, typename S>
void upload_layout_array(DevBuf<T> &dst, const ClptStaging<S> &src) {
    static_assert(sizeof(T) == sizeof(S), "staging and device element sizes differ");
    dst.reserve(src.size());
    if (src.size()) CU(cudaMemcpyAsync(dst.ptr, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, St.stream));
}

void upload_scene(const kdnode *nodes, size_t node_bytes, const int *tri_indices, size_t tri_index_bytes,
                  const cl_int3 *tris, size_t tri_bytes, const Vector4 *verts, size_t vert_bytes,
                  const Vector4 *norms, size_t norm_bytes) {
    ClptPackedScene &packed = g_packed; // keeps its staging capacity between uploads
    const char *verbose = getenv("CLPT_VERBOSE");
    const bool timing = verbose && atoi(verbose) >= 2;
    const auto t0 = std::chrono::steady_clock::now();

    std::string err;
    const size_t n_norms = norms ? norm_bytes / sizeof(Vector4) : 0;
    if (!clpt_pack_scene(nodes, node_bytes / sizeof(kdnode), tri_indices, tri_index_bytes / sizeof(int), tris,
                         tri_bytes / sizeof(cl_int3), verts, vert_bytes / sizeof(Vector4), n_norms, packed,
                         err)) {
        fprintf(stderr, "CLSetMeshes: invalid scene: %s\n", err.c_str());
        exit(EXIT_FAILURE);
    }
    const auto t1 = std::chrono::steady_clock::now();
    upload_layout_array(St.layout.nodes, packed.nodes);
    upload_layout_array(St.layout.leaves, packed.leaves);
    upload_layout_array(St.layout.tri, packed.tri);
    upload_layout_array(St.layout.flat_n, packed.flat_n);
    upload_layout_array(St.layout.lut, packed.lut);
    static_cast<ClptLayoutInfo &>(St.layout) = packed;
    CU(cudaStreamSynchronize(St.stream)); // (the staging is rewritten by the next upload)
    St.corners.upload(reinterpret_cast<const int4 *>(tris), tri_bytes / sizeof(cl_int3), St.stream);
    if (n_norms) {
        St.norms.upload(reinterpret_cast<const float4 *>(norms), n_norms, St.stream);
    } else {
        St.norms.release(); // the reference keeps a stale buffer here (src/CLState.c:146); unused either way
    }
    // per-triangle materials belong to the previous mesh
    St.tri_material.release();
    St.scene_on_gpu = St.mesh_on_gpu = false; // (the corner buffer now belongs to this scene)
    adopt_layout(packed.n_prims);
    if (timing) {
        const auto t2 = std::chrono::steady_clock::now();
        fprintf(stderr, "CLSetMeshes: pack %.3f ms, upload %.3f ms (%d nodes, %d leaves, %d triangle slots, %zu table cells)\n",
                std::chrono::duration<double, std::milli>(t1 - t0).count(),
                std::chrono::duration<double, std::milli>(t2 - t1).count(), packed.n_nodes, packed.n_leaves,
                packed.n_refs, packed.lut.size());
    }
}

void *pinned_alloc(size_t bytes) {
    void *p = nullptr;
    CU(cudaMallocHost(&p, bytes));
    return p;
}
void pinned_free(void *p) { (void)cudaFreeHost(p); } // may run during process teardown: never fatal

void release_host_kd() {
    if (St.owns_kd) delete_kd(St.host_kd);
    St.host_kd = kd{ nullptr, nullptr, nullptr, nullptr, nullptr };
    St.owns_kd = false;
}

// ---- multi-GPU direct placement -----------------------------------------------
// With a communicator the render kernel assembles the frame itself: every rank maps
// every other rank's frame (CUDA IPC; the mapping enables peer access over NVLink) and
// store_pixel writes each finished pixel into all of them.  What is left of the
// collective is ordering: one barrier before a frame (every rank is done reading the
// previous one) and one after it (every rank's pixels have landed).  The barrier is a
// one-word all-reduce on the library's stream.  If the mapping cannot be made on some
// rank ($CLPT_P2P=0 on all ranks, no IPC, more than CLPT_MAX_PEERS ranks) every rank
// falls back to slab + ncclAllGather + de-interleave.

void dist_word_ready() {
    if (!St.dist_word.ptr) {
        St.dist_word.resize(2);
        CU(cudaMemsetAsync(St.dist_word.ptr, 0, 2 * sizeof(int), St.stream));
    }
}

void dist_barrier() {
    dist_word_ready();
    NC(g_nccl.AllReduce(St.dist_word.ptr, St.dist_word.ptr + 1, 1, ncclInt, ncclSum, St.comm, St.stream));
}

// Barrier over the peer-mapped flag words (direct placement only): a one-block kernel on the
// library's stream stores this frame's epoch into its word on every rank and spins until every
// rank's epoch has arrived in its own words -- a few microseconds over NVLink, against ~20 for a
// one-word ncclAllReduce, twice per frame.
void flag_barrier() {
    ClptFlagPeers peers;
    for (int r = 0; r < CLPT_MAX_PEERS; r++) peers.flags[r] = St.peer_flags[r];
    clpt_launch_flag_barrier(peers, St.rank, St.nranks, ++St.flag_epoch, St.stream);
    CU(cudaGetLastError());
}

int dist_min(int v) {
    dist_word_ready();
    int out = 0;
    CU(cudaMemcpyAsync(St.dist_word.ptr, &v, sizeof(int), cudaMemcpyHostToDevice, St.stream));
    NC(g_nccl.AllReduce(St.dist_word.ptr, St.dist_word.ptr + 1, 1, ncclInt, ncclMin, St.comm, St.stream));
    CU(cudaMemcpyAsync(&out, St.dist_word.ptr + 1, sizeof(int), cudaMemcpyDeviceToHost, St.stream));
    CU(cudaStreamSynchronize(St.stream));
    CU(cudaMemsetAsync(St.dist_word.ptr, 0, 2 * sizeof(int), St.stream));
    return out;
}

void p2p_close_mappings() {
    for (int r = 0; r < CLPT_MAX_PEERS; r++) {
        if (St.peer_image[r] && r != St.p2p_self) {
            const cudaError_t e = cudaIpcCloseMemHandle(St.peer_image[r]);
            if (e != cudaSuccess) {
                fprintf(stderr, "rank %d: unmapping rank %d's frame: %s\n", St.rank, r, cudaGetErrorName(e));
                (void)cudaGetLastError(); // not fatal, and must not surface at the next launch check
            }
        }
        St.peer_image[r] = nullptr;
        if (St.peer_flags[r] && r != St.p2p_self) {
            if (cudaIpcCloseMemHandle(St.peer_flags[r]) != cudaSuccess) (void)cudaGetLastError();
        }
        St.peer_flags[r] = nullptr;
    }
    St.p2p_self = -1;
}

// Collective over the communicator.  Must run before a mapped frame is freed or resized
// and before the communicator goes away: an exporter may not free what a peer still maps.
void p2p_teardown() {
    if (!St.p2p) return;
    CU(cudaStreamSynchronize(St.stream));
    p2p_close_mappings();
    St.p2p = false;
    if (St.comm) {
        dist_barrier();
        CU(cudaStreamSynchronize(St.stream));
    }
}

// Collective over the communicator: exchange the frames' IPC handles and map the peers'.
void p2p_setup() {
    St.p2p = false;
    if (!St.comm || St.nranks < 2 || St.nranks > CLPT_MAX_PEERS || St.nranks != St.comm_ranks || !St.image.ptr) return;
    if (const char *e = getenv("CLPT_P2P")) {
        if (atoi(e) == 0) return; // has to be set on every rank alike
    }
    struct Slot {
        cudaIpcMemHandle_t handle, flags_handle;
        int ok;
        int pad[31];
    };
    static_assert(sizeof(Slot) == 256, "exchange slot is 256 bytes");
    Slot mine;
    memset(&mine, 0, sizeof(mine));
    // the barrier words: zeroed here, before the exchange below orders every rank's zeroing
    // ahead of any rank's first signal
    // (a whole 2 MiB block of its own: IPC handles cover the driver's underlying allocation)
    St.bar_flags.resize((2u << 20) / sizeof(unsigned int));
    CU(cudaMemsetAsync(St.bar_flags.ptr, 0, CLPT_MAX_PEERS * 8 * sizeof(unsigned int), St.stream));
    St.flag_epoch = 0;
    mine.ok = cudaIpcGetMemHandle(&mine.handle, St.image.ptr) == cudaSuccess &&
                      cudaIpcGetMemHandle(&mine.flags_handle, St.bar_flags.ptr) == cudaSuccess
                  ? 1
                  : 0;
    if (!mine.ok) (void)cudaGetLastError();
    const size_t n = (size_t)St.nranks;
    St.dist_xchg.resize(sizeof(Slot) * (n + 1));
    std::vector<Slot> all(n);
    CU(cudaMemcpyAsync(St.dist_xchg.ptr, &mine, sizeof(Slot), cudaMemcpyHostToDevice, St.stream));
    NC(g_nccl.AllGather(St.dist_xchg.ptr, St.dist_xchg.ptr + sizeof(Slot), sizeof(Slot), ncclChar, St.comm,
                        St.stream));
    CU(cudaMemcpyAsync(all.data(), St.dist_xchg.ptr + sizeof(Slot), sizeof(Slot) * n, cudaMemcpyDeviceToHost,
                       St.stream));
    CU(cudaStreamSynchronize(St.stream));
    int ok = 1;
    for (size_t r = 0; r < n; r++) ok &= all[r].ok;
    St.p2p_self = St.rank;
    for (size_t r = 0; ok && r < n; r++) {
        if ((int)r == St.rank) {
            St.peer_image[r] = St.image.ptr;
            St.peer_flags[r] = St.bar_flags.ptr;
            continue;
        }
        void *mapped = nullptr, *mapped_flags = nullptr;
        if (cudaIpcOpenMemHandle(&mapped, all[r].handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            (void)cudaGetLastError();
            ok = 0;
        } else {
            St.peer_image[r] = (float4 *)mapped;
            if (cudaIpcOpenMemHandle(&mapped_flags, all[r].flags_handle, cudaIpcMemLazyEnablePeerAccess) !=
                cudaSuccess) {
                (void)cudaGetLastError();
                ok = 0;
            } else {
                St.peer_flags[r] = (unsigned int *)mapped_flags;
            }
        }
    }
    ok = dist_min(ok);
    if (!ok) {
        p2p_close_mappings();
        dist_barrier();
        CU(cudaStreamSynchronize(St.stream));
        if (St.rank == 0) fprintf(stderr, "CLDistInit: peer frames could not be mapped; using ncclAllGather\n");
        return;
    }
    St.p2p = true;
    St.gathered.release(); // only the all-gather path needs it
    if (getenv("CLPT_VERBOSE") && St.rank == 0) {
        fprintf(stderr, "CLDistInit: %d ranks, frames peer-mapped, direct placement\n", St.nranks);
    }
}

void release_read_pipeline();

// The instances of the next frame: the device table, written again if anything it holds changed.
ClptInstances current_instances() {
    ClptInstances I = { nullptr, 0 };
    if (St.instances.empty()) return I;
    if (St.inst_table_stale) {
        std::vector<ClptInstanceRec> recs(St.instances.size());
        int offset = St.scene.n_prims;
        for (size_t k = 0; k < recs.size(); k++) {
            const CLInstance &in = St.instances[k];
            ClptInstanceRec &r = recs[k];
            memset(&r, 0, sizeof(r));
            memcpy(r.w2o, in.world_to_object, sizeof(r.w2o));
            r.material = in.material;
            r.prim_offset = offset;
            r.mesh = St.inst_meshes[in.mesh]->scene;
            offset += r.mesh.n_prims;
        }
        St.inst_table.upload(recs.data(), recs.size(), St.stream);
        St.inst_table_stale = false;
    }
    I.rec = St.inst_table.ptr;
    I.count = (int)St.instances.size();
    return I;
}

void release_instance_meshes() {
    for (auto &m : St.inst_meshes) {
        m->verts.release();
        m->norms.release();
        m->corners.release();
        m->tree.release();
        m->layout.release();
    }
    St.inst_meshes.clear();
    St.instances.clear();
    St.inst_table.release();
    St.inst_table_stale = true;
}

// A device-built tree and its mesh as fresh host lists (CLDownloadKd, CLDownloadInstanceKd).
void download_tree(const ClptGpuTree &tree, const DevBuf<float4> &verts, const DevBuf<int4> &corners,
                   const DevBuf<float4> &norms, kd *out) {
    CU(cudaStreamSynchronize(St.stream));
    const size_t n = (size_t)tree.n_nodes, r = (size_t)tree.n_refs;
    out->node_vec = (kdnode *)init_list(n, sizeof(kdnode));
    out->tri_indices = (int *)init_list(r, sizeof(int));
    out->vert_vec = (Vector4 *)init_list(verts.count, sizeof(Vector4));
    out->tri_vec = (cl_int3 *)init_list(corners.count, sizeof(cl_int3));
    out->norm_vec = (Vector4 *)init_list(norms.count, sizeof(Vector4));
    CU(cudaMemcpy(out->node_vec, tree.wire.ptr, n * sizeof(kdnode), cudaMemcpyDeviceToHost));
    if (r) CU(cudaMemcpy(out->tri_indices, tree.tri_indices.ptr, r * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out->vert_vec, verts.ptr, verts.count * sizeof(Vector4), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out->tri_vec, corners.ptr, corners.count * sizeof(cl_int3), cudaMemcpyDeviceToHost));
    if (norms.count) CU(cudaMemcpy(out->norm_vec, norms.ptr, norms.count * sizeof(Vector4), cudaMemcpyDeviceToHost));
}

// The AOV buffers at the size of the render target, cleared (prim_id -1: no hit).
void alloc_aovs() {
    const size_t px = (size_t)St.width * St.height;
    St.aov_prim.resize(px);
    St.aov_t.resize(px);
    St.aov_uv.resize(px);
    CU(cudaMemsetAsync(St.aov_prim.ptr, 0xff, px * sizeof(int), St.stream));
    CU(cudaMemsetAsync(St.aov_t.ptr, 0, px * sizeof(float), St.stream));
    CU(cudaMemsetAsync(St.aov_uv.ptr, 0, px * sizeof(float2), St.stream));
    CU(cudaStreamSynchronize(St.stream));
}

// Frees the render target and the buffers frames made for it (the caller has torn down the peer
// mappings and the read-back pipeline first).
void release_targets() {
    St.image.release();
    St.slab.release();
    St.gathered.release();
    St.scratch.release();
    St.accum.release();
    St.accum_sum.release();
    St.aov_prim.release();
    St.aov_t.release();
    St.aov_uv.release();
}

void alloc_targets() {
    p2p_teardown();
    release_read_pipeline();
    const size_t px = (size_t)St.width * St.height;
    St.image.resize(px);
    clpt_launch_fill(St.image.ptr, px, 0.0f, St.stream);
    if (St.nranks > 1) {
        const size_t slab_px = (size_t)slab_rows_for(St.height) * St.width;
        St.slab.resize(slab_px);
        clpt_launch_fill(St.slab.ptr, slab_px, 0.0f, St.stream);
        if (St.comm) St.gathered.resize(slab_px * St.nranks);
    } else {
        St.slab.release();
        St.gathered.release();
    }
    if (St.aov) alloc_aovs();
    St.scratch.release();
    St.accum.release();
    St.accum_sum.release();
    St.sample_base = 0;
    CU(cudaStreamSynchronize(St.stream));
    p2p_setup();
}

// Progressive frames are spread over GPUs by SAMPLE: every rank renders the whole frame with its own
// sample indices into its own fixed-point buffer, nothing crosses GPUs per frame, and a read-back
// adds the buffers up (SURVEY.md section 8e, "accumulate locally per rank; gather only on
// display/readback").  Integer sums are order-free, so the result is the single-GPU frame bit for bit.
bool sample_parallel() { return (St.flags & CLPT_FLAG_ACCUMULATE) && St.nranks > 1; }

void ensure_accum() {
    const size_t words = (size_t)St.width * St.height * 4;
    if (St.accum.count != words) {
        St.accum.resize(words);
        clpt_launch_fill_u64(St.accum.ptr, words, St.stream);
        St.sample_base = 0;
    }
}

// The current frame as displayable float4 (rgb, 1) on the library's stream.  Replace mode: the
// frame itself.  Progressive mode: sums / count into `scratch`; across GPUs the ranks' buffers are
// added first (ncclAllReduce, 64-bit integer sum), which makes the call COLLECTIVE in that case.
const float4 *displayable_frame() {
    const size_t px = (size_t)St.width * St.height;
    if (!(St.flags & CLPT_FLAG_ACCUMULATE)) return St.image.ptr;
    ensure_accum();
    if (St.scratch.count != px) St.scratch.resize(px);
    const unsigned long long *sums = St.accum.ptr;
    if (St.nranks > 1 && St.comm) {
        if (St.accum_sum.count != px * 4) St.accum_sum.resize(px * 4);
        NC(g_nccl.AllReduce(St.accum.ptr, St.accum_sum.ptr, px * 4, ncclUint64, ncclSum, St.comm, St.stream));
        sums = St.accum_sum.ptr;
    } // (sharded without a communicator: this rank's samples only)
    clpt_launch_normalise(sums, St.scratch.ptr, px, St.stream);
    CU(cudaGetLastError());
    return St.scratch.ptr;
}

size_t frame_bytes(int format) {
    return (size_t)St.width * St.height * (format == CLPT_READ_RGBA8 ? sizeof(uchar4) : sizeof(float4));
}

void check_read(const char *who, size_t bytes, int format) {
    require_init(who);
    if (!St.have_image) {
        fprintf(stderr, "%s: no render target\n", who);
        exit(EXIT_FAILURE);
    }
    if (format != CLPT_READ_FLOAT4 && format != CLPT_READ_RGBA8) {
        fprintf(stderr, "%s: format must be CLPT_READ_FLOAT4 or CLPT_READ_RGBA8\n", who);
        exit(EXIT_FAILURE);
    }
    if (bytes != frame_bytes(format)) {
        fprintf(stderr, "%s: %zu bytes given, the %dx%d %s frame is %zu\n", who, bytes, St.width, St.height,
                format == CLPT_READ_RGBA8 ? "RGBA8" : "float4", frame_bytes(format));
        exit(EXIT_FAILURE);
    }
}

// Frame -> slot staging on the library's stream; staging -> host on the copy stream.
void enqueue_read(void *dst, size_t bytes, int format) {
    auto &slot = St.rd[St.rd_issued & 1];
    if (!slot.ready) {
        CU(cudaEventCreateWithFlags(&slot.ready, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&slot.done, cudaEventDisableTiming));
    }
    if (!St.copy_stream) CU(cudaStreamCreateWithFlags(&St.copy_stream, cudaStreamNonBlocking));
    // the copy that last used this staging buffer must have drained before it is rewritten
    if (slot.in_flight) CU(cudaStreamWaitEvent(St.stream, slot.done, 0));
    if (slot.staging.count < bytes) slot.staging.resize(bytes);
    if (format == CLPT_READ_RGBA8) {
        const float4 *src = displayable_frame();
        clpt_launch_pack_rgba8(src, reinterpret_cast<uchar4 *>(slot.staging.ptr), (size_t)St.width * St.height,
                               St.stream);
        CU(cudaGetLastError());
    } else {
        const float4 *src = displayable_frame();
        CU(cudaMemcpyAsync(slot.staging.ptr, src, bytes, cudaMemcpyDeviceToDevice, St.stream));
    }
    CU(cudaEventRecord(slot.ready, St.stream));
    CU(cudaStreamWaitEvent(St.copy_stream, slot.ready, 0));
    CU(cudaMemcpyAsync(dst, slot.staging.ptr, bytes, cudaMemcpyDeviceToHost, St.copy_stream));
    CU(cudaEventRecord(slot.done, St.copy_stream));
    slot.in_flight = true;
    slot.ticket = ++St.rd_issued;
}

void wait_reads(unsigned long long leave_pending) {
    // oldest first
    for (int k = 0; k < 2; k++) {
        auto &slot = St.rd[(St.rd_issued + k) & 1];
        if (slot.in_flight && slot.ticket + leave_pending <= St.rd_issued) {
            CU(cudaEventSynchronize(slot.done));
            slot.in_flight = false;
        }
    }
}

void release_read_pipeline() {
    wait_reads(0);
    for (auto &slot : St.rd) {
        slot.staging.release();
        if (slot.ready) CU(cudaEventDestroy(slot.ready));
        if (slot.done) CU(cudaEventDestroy(slot.done));
        slot.ready = slot.done = nullptr;
        slot.in_flight = false;
    }
}

} // namespace

// Internal: the frame launch, shared by CLExecute and CLEnqueueKernel.
void clpt_state_launch_frame(int width, int height) {
    require_init("CLExecute");
    if (!St.have_image) FATAL("no render target: call CLCreateImage or CLCreateImageHeadless first");
    if (width != St.width || height != St.height) {
        fprintf(stderr, "CLExecute: launch size %dx%d does not match the %dx%d render target\n", width, height,
                St.width, St.height);
        exit(EXIT_FAILURE);
    }
    if (!St.have_scene) FATAL("no scene: call CLSetMeshes first");
    St.last_launches = 0;

    ClptFrame F;
    memcpy(F.cam, St.cam, sizeof(F.cam));
    {   // (volatile: one rounded single-precision division each, never folded into something wider)
        volatile float w = St.cam[14], ex = St.cam[2] / w, ey = St.cam[6] / w, ez = St.cam[10] / w;
        F.eye[0] = ex, F.eye[1] = ey, F.eye[2] = ez;
        F.half_width = (float)(unsigned)width * 0.5f;   // == width / 2.0f exactly
        F.half_height = (float)(unsigned)height * 0.5f;
    }
    F.width = width;
    F.height = height;
    F.mode = St.mode;
    F.depth = St.depth;
    F.spp = St.spp;
    F.flags = St.flags;
    F.log2_sample_lanes = 0;
    while (F.log2_sample_lanes < 5 && (2 << F.log2_sample_lanes) <= St.spp) F.log2_sample_lanes++;
    // At >= 64 spp the samples of a pixel can be spread over 2, 4 or 8 warps (render_kernel.cu): a
    // claim is then 1/G as long.  That only pays when a warp gets few claims per frame and the end
    // of the frame is a visible part of it -- one GPU's share of a frame sharded over several
    // (measured: +3..4% on an eighth of the bench frame, -1% on the whole of it).
    F.log2_warps_per_pixel = 0;
    {
        const int rows = F.local_rows;
        const double claims_per_warp = (double)rows * width / ((double)St.prop.multiProcessorCount * 64.0);
        if (claims_per_warp < 150.0) {
            while (F.log2_warps_per_pixel < 3 && (64 << F.log2_warps_per_pixel) <= St.spp) F.log2_warps_per_pixel++;
        }
    }
    if (const char *e = getenv("CLPT_WARPS_PER_PIXEL")) { // measurement only
        int lg = 0;
        while ((2 << lg) <= atoi(e) && lg < 3 && (64 << lg) <= St.spp) lg++;
        F.log2_warps_per_pixel = lg;
    }
    F.seed = St.seed;
    F.sample_base = St.sample_base;
    F.accum = nullptr;
    F.max_leaf_visits = St.max_leaf_visits;
    F.rank = St.rank;
    F.nranks = St.nranks;
    F.tile_rows = St.tile_rows;
    F.local_rows = St.nranks > 1 ? local_rows_for(height) : height;
    F.target = St.nranks > 1 ? St.slab.ptr : St.image.ptr;
    const int spp_frame = St.spp < 1 ? 1 : St.spp;
    if (St.flags & CLPT_FLAG_ACCUMULATE) {
        // progressive: the whole frame on every rank, rank r takes samples base + r*spp .. + spp - 1
        ensure_accum();
        F.accum = St.accum.ptr;
        F.rank = 0;
        F.nranks = 1;
        F.local_rows = height;
        F.target = St.image.ptr; // (not written)
        F.sample_base = St.sample_base + (unsigned)(St.rank * spp_frame);
    }
    F.aov_prim = St.aov ? St.aov_prim.ptr : nullptr;
    F.aov_t = St.aov ? St.aov_t.ptr : nullptr;
    F.aov_uv = St.aov ? St.aov_uv.ptr : nullptr;
    F.counters = nullptr;
    if (!St.work_counter.ptr) St.work_counter.resize(1);
    F.work_counter = St.work_counter.ptr;
    F.blocks_x = F.n_warp_tiles = 0;
    F.row_cost = nullptr;
    F.row_count = 0;
    const bool local_only = sample_parallel(); // progressive across GPUs: nothing crosses GPUs per frame
    const bool p2p = St.p2p && St.comm && St.nranks > 1 && !local_only;
    F.n_peer_images = p2p ? St.nranks : 0;
    for (int r = 0; r < CLPT_MAX_PEERS; r++) F.peer_image[r] = p2p ? St.peer_image[r] : nullptr;
    if (St.flags & CLPT_FLAG_COUNTERS) {
        if (!St.counters.ptr) St.counters.resize(6);
        CU(cudaMemsetAsync(St.counters.ptr, 0, 6 * sizeof(unsigned long long), St.stream));
        F.counters = St.counters.ptr;
    }

    // Engine: 1 = the kernel compiled for 8 resident blocks per SM; 2 = for 4 (trees with fat
    // leaves, render_kernel.cu); 0 = chosen from the tree at CLSetMeshes.
    St.last_engine = St.engine != 0 ? St.engine : St.auto_engine;
    if (St.last_engine == 2) F.flags |= CLPT_F_FAT;
    // engine 2, one sample per pixel: two lanes per ray (clpt_trace.cuh: triangle_run_shared)
    F.log2_lanes_per_ray = (St.last_engine == 2 && F.log2_sample_lanes == 0) ? 1 : 0;
    if (const char *e = getenv("CLPT_LANES_PER_RAY")) { // measurement only: 1, 2 or 4
        if (St.last_engine == 2 && F.log2_sample_lanes == 0) {
            int k = atoi(e), lg = 0;
            while ((2 << lg) <= k && lg < 5) lg++;
            F.log2_lanes_per_ray = lg;
        }
    }

    // Claim direction (megakernel): decided from the previous frame's per-row cost under
    // the same image, sharding and parameters.  $CLPT_ROW_ORDER=0 turns it off.
    int order_rows = 0;
    {
        const char *e = getenv("CLPT_ROW_ORDER");
        if (!(e && atoi(e) == 0)) order_rows = clpt_render_block_rows(F);
        // the bookkeeping (a memset and a small copy, ~15 us) is only worth it on frames long
        // enough to have a tail: skipped while the previous frame took under half a millisecond
        if (St.frames_rendered > 0 && St.last_kernel_ms < 0.5f) order_rows = 0;
    }
    if (order_rows > 0) {
        const long long key[8] = { width, height, St.spp, St.mode, St.depth, St.rank, St.nranks, St.tile_rows };
        if (order_rows != St.row_count || memcmp(key, St.row_key, sizeof(key)) != 0) {
            St.claim_reverse = false;
            St.row_count = order_rows;
            memcpy(St.row_key, key, sizeof(key));
        }
        if (order_rows > St.row_capacity) {
            if (St.host_row_cost) CU(cudaFreeHost(St.host_row_cost));
            CU(cudaMallocHost((void **)&St.host_row_cost, (size_t)2 * order_rows * sizeof(unsigned long long)));
            St.row_cost.resize((size_t)2 * order_rows); // [rows] summed claim clocks, [rows] the longest claim
            St.row_capacity = order_rows;
        }
        CU(cudaMemsetAsync(St.row_cost.ptr, 0, (size_t)2 * order_rows * sizeof(unsigned long long), St.stream));
        F.row_cost = St.row_cost.ptr;
        F.row_count = order_rows;
        if (St.claim_reverse) F.flags |= CLPT_F_REVERSE;
    }
    const ClptInstances inst = current_instances();
    if (p2p) {
        flag_barrier(); // every rank has finished with (reading) the previous frame
        St.last_launches++;
    }
    CU(cudaEventRecord(St.ev_start, St.stream));
    clpt_launch_render(St.scene, F, inst, St.prop.multiProcessorCount, St.stream);
    St.last_launches++;
    CU(cudaGetLastError());
    CU(cudaEventRecord(St.ev_stop, St.stream));
    if (order_rows > 0) {
        CU(cudaMemcpyAsync(St.host_row_cost, St.row_cost.ptr, (size_t)2 * order_rows * sizeof(unsigned long long),
                           cudaMemcpyDeviceToHost, St.stream));
    }

    if (p2p) {
        flag_barrier(); // every rank's pixels have landed in this rank's frame
        St.last_launches++;
    } else if (local_only) {
        // this rank's samples went into its own sums; CLReadImage* adds the ranks' buffers (displayable_frame)
    } else if (St.nranks > 1 && St.comm) {
        const size_t slab_px = (size_t)slab_rows_for(height) * width;
        if (St.gathered.count != slab_px * St.nranks) St.gathered.resize(slab_px * St.nranks);
        NC(g_nccl.AllGather(St.slab.ptr, St.gathered.ptr, slab_px * 4, ncclFloat, St.comm, St.stream));
        clpt_launch_deinterleave(St.gathered.ptr, St.image.ptr, width, height, St.nranks, St.tile_rows,
                                 slab_rows_for(height), St.stream);
        CU(cudaGetLastError());
        St.last_launches++;
    } else if (St.nranks > 1) {
        // sharded without a communicator: place this rank's rows only
        const size_t slab_px = (size_t)slab_rows_for(height) * width;
        if (St.gathered.count != slab_px * St.nranks) {
            St.gathered.resize(slab_px * St.nranks);
            CU(cudaMemsetAsync(St.gathered.ptr, 0, slab_px * St.nranks * sizeof(float4), St.stream));
        }
        CU(cudaMemcpyAsync(St.gathered.ptr + slab_px * St.rank, St.slab.ptr, slab_px * sizeof(float4),
                           cudaMemcpyDeviceToDevice, St.stream));
        clpt_launch_deinterleave(St.gathered.ptr, St.image.ptr, width, height, St.nranks, St.tile_rows,
                                 slab_rows_for(height), St.stream);
        CU(cudaGetLastError());
        St.last_launches++;
    }
    if (!St.headless && clpt_gl_registered()) {
        clpt_gl_present(displayable_frame(), width, height, St.stream); // acquire/write/release, :207-218
        St.last_launches++;
    }
    CU(cudaStreamSynchronize(St.stream)); // clFinish, src/CLState.c:212
    CU(cudaEventElapsedTime(&St.last_kernel_ms, St.ev_start, St.ev_stop));
    St.frames_rendered++;
    if (order_rows > 0) { // next frame starts from the end nearer to this frame's costliest rows
        double where = 0.0;
        St.claim_reverse = clpt_claim_direction(St.host_row_cost, order_rows, St.claim_reverse ? 1 : 0, &where) != 0;
        if (getenv("CLPT_VERBOSE") && atoi(getenv("CLPT_VERBOSE")) >= 3) {
            fprintf(stderr, "CLExecute: costliest rows at %.2f of %d, next frame claims %s\n", where, order_rows,
                    St.claim_reverse ? "bottom-up" : "top-down");
            {   // how much of the resident warps' time was spent inside claims (the rest: the frame's tail)
                unsigned long long in_claims = 0, longest = 0;
                for (int r = 0; r < order_rows; r++) {
                    in_claims += St.host_row_cost[r];
                    if (St.host_row_cost[order_rows + r] > longest) longest = St.host_row_cost[order_rows + r];
                }
                const int per_sm = clpt_render_blocks_per_sm(St.last_engine);
                const double groups = (double)St.prop.multiProcessorCount * per_sm * (8 >> F.log2_warps_per_pixel);
                const double clocks = (double)St.last_kernel_ms * 1e-3 * (double)St.prop.clockRate * 1e3;
                fprintf(stderr, "CLExecute: %.3f ms; claims fill %.1f%% of the resident warp groups' time (at %d MHz); "
                                "longest claim %.3f ms\n", St.last_kernel_ms, 100.0 * (double)in_claims / (groups * clocks),
                        St.prop.clockRate / 1000, (double)longest / ((double)St.prop.clockRate * 1e3) * 1e3);
            }
            if (atoi(getenv("CLPT_VERBOSE")) >= 4) {
                for (int r = 0; r < order_rows; r++) {
                    fprintf(stderr, "  row %d: claims %llu kclk in all, longest %llu kclk\n", r,
                            St.host_row_cost[r] / 1000ull, St.host_row_cost[order_rows + r] / 1000ull);
                }
            }
        }
    }
    if (St.flags & CLPT_FLAG_COUNTERS) {
        CU(cudaMemcpy(St.host_counters, St.counters.ptr, sizeof(St.host_counters), cudaMemcpyDeviceToHost));
    }
    if (St.flags & CLPT_FLAG_ACCUMULATE) St.sample_base += (unsigned)(spp_frame * St.nranks);
}

cudaStream_t clpt_state_stream() { return St.stream; }
int clpt_state_device() { return St.device; }

extern "C" {

void CLSelectDevice(int ordinal) {
    if (St.inited) FATAL("CLSelectDevice must be called before CLInit");
    St.device = ordinal;
}

void CLInit(const char *kernel_filename, const char *kernel_name) {
    (void)kernel_filename;
    (void)kernel_name;
    if (St.inited) return;
    // same bring-up order as src/CLState.c:228-234, through the CLHandler layer
    CLPlatform platform = CLGetPlatform();
    CLDevice device = CLGetDevice(platform);
    CLContext context = CLCreateContext(platform, device);
    CLBuildProgram(kernel_filename, context, device);
    St.device = (int)(intptr_t)device - 1;
    St.stream = (cudaStream_t)CLCreateQueue(context, device);
    CLCreateKernel(kernel_name ? kernel_name : "render", nullptr);
    CU(cudaGetDeviceProperties(&St.prop, St.device));
    CU(cudaEventCreate(&St.ev_start));
    CU(cudaEventCreate(&St.ev_stop));
    for (auto &e : St.ev_user) CU(cudaEventCreate(&e));
    for (auto &e : St.ev_build) CU(cudaEventCreate(&e));
    memset(St.cam, 0, sizeof(St.cam));
    clpt_pack_alloc = pinned_alloc; // the packed scene is staged in page-locked memory
    clpt_pack_free = pinned_free;
    St.inited = true;
}

void CLTerminate(void) {
    if (!St.inited) return;
    release_host_kd(); // delete_kd(State.kd), src/CLState.c:223
    CU(cudaStreamSynchronize(St.stream));
    release_read_pipeline();
    if (St.copy_stream) CU(cudaStreamDestroy(St.copy_stream));
    St.copy_stream = nullptr;
    p2p_teardown();
    if (St.comm) {
        NC(g_nccl.CommDestroy(St.comm));
        St.comm = nullptr;
        St.comm_ranks = 0;
    }
    if (clpt_gl_registered()) clpt_gl_unregister();
    St.layout.release();
    St.norms.release();
    St.corners.release();
    St.verts.release();
    St.gpu_tree.release();
    St.scene_on_gpu = St.mesh_on_gpu = false;
    release_instance_meshes();
    clpt_gpu_build_release();
    St.objects.release();
    St.materials.release();
    St.tri_material.release();
    release_targets();
    St.counters.release();
    St.work_counter.release();
    St.row_cost.release();
    if (St.host_row_cost) CU(cudaFreeHost(St.host_row_cost));
    St.host_row_cost = nullptr;
    St.row_capacity = St.row_count = 0;
    St.claim_reverse = false;
    St.dist_word.release();
    St.dist_xchg.release();
    St.bar_flags.release();
    St.l2_flush.release();
    g_packed.nodes.release();
    g_packed.leaves.release();
    g_packed.tri.release();
    g_packed.lut.release();
    CU(cudaEventDestroy(St.ev_start));
    CU(cudaEventDestroy(St.ev_stop));
    for (auto &e : St.ev_user) CU(cudaEventDestroy(e));
    for (auto &e : St.ev_build) CU(cudaEventDestroy(e));
    CU(cudaStreamDestroy(St.stream));
    St.stream = nullptr;
    St.have_scene = St.have_image = St.headless = false;
    St.objcount = 0;
    St.rank = 0;
    St.nranks = 1;
    St.inited = false;
    St.device = -1;
}

void CLSetCameraMatrixPtr(const Matrix *matrix) {
    require_init("CLSetCameraMatrix");
    // The reference writes 64 bytes into a device buffer the kernel re-reads per
    // thread (src/CLState.c:67-79, src/kernel.cl:443-454); here the matrix rides
    // in the launch parameters (constant bank), so "upload" is a host copy.
    memcpy(St.cam, matrix, sizeof(St.cam));
}

void CLSetCameraMatrix(Matrix matrix) { CLSetCameraMatrixPtr(&matrix); }

void CLSetObjects(Object *vec_objects, size_t size) {
    require_init("CLSetObjects");
    if (size / sizeof(Object) != (size_t)St.objcount) {
        St.objects.resize(size);
        St.objcount = (int)(size / sizeof(Object));
    }
    if (size == 0) return;
    CU(cudaMemcpyAsync(St.objects.ptr, vec_objects, size, cudaMemcpyHostToDevice, St.stream));
    CU(cudaStreamSynchronize(St.stream));
}

void CLSetMeshes(kd *models) {
    require_init("CLSetMeshes");
    if (models == nullptr || list_size(models) / sizeof(kd) == 0) return; // src/CLState.c:126-129
    kd m = models[0];                                                     // models[0] only, :130
    // The reference never frees on a re-set (src/CLState.c:124-131 overwrites State.kd), so calling
    // CLSetMeshes again with the SAME kd -- an in-place updated scene, or simply a repeat -- is legal
    // there.  A previously adopted list is released only if the new kd does not carry it again.
    if (St.owns_kd) {
        const void *incoming[5] = { m.node_vec, m.tri_indices, m.vert_vec, m.norm_vec, m.tri_vec };
        void *held[5] = { St.host_kd.node_vec, St.host_kd.tri_indices, St.host_kd.vert_vec, St.host_kd.norm_vec,
                          St.host_kd.tri_vec };
        for (void *old : held) {
            bool again = false;
            for (const void *in : incoming) again |= (old == in);
            if (old && !again) delete_list(old);
        }
        St.owns_kd = false;
    }
    St.host_kd = m;
    St.owns_kd = true;
    upload_scene(m.node_vec, list_size(m.node_vec), m.tri_indices, list_size(m.tri_indices), m.tri_vec,
                 list_size(m.tri_vec), m.vert_vec, list_size(m.vert_vec), m.norm_vec,
                 m.norm_vec ? list_size(m.norm_vec) : 0);
}

void CLSetMeshesRaw(const void *nodes, size_t node_bytes, const int *tri_indices, size_t tri_index_bytes,
                    const void *tris, size_t tri_bytes, const void *verts, size_t vert_bytes,
                    const void *norms, size_t norm_bytes) {
    require_init("CLSetMeshesRaw");
    release_host_kd();
    upload_scene((const kdnode *)nodes, node_bytes, tri_indices, tri_index_bytes, (const cl_int3 *)tris,
                 tri_bytes, (const Vector4 *)verts, vert_bytes, (const Vector4 *)norms, norm_bytes);
}

void CLSetBuildParams(int max_depth, int min_split, float traversal_cost, float intersect_cost, float empty_bonus) {
    St.build_params.max_depth = max_depth;
    St.build_params.min_split = min_split < 2 ? 2 : min_split;
    St.build_params.ct = traversal_cost;
    St.build_params.ci = intersect_cost;
    St.build_params.empty_bonus = empty_bonus;
}

namespace {
// Build the tree of the device-resident mesh and re-lay it out, all on the device.
void rebuild_on_device(const char *who) {
    const size_t n_verts = St.verts.count, n_corners = St.corners.count;
    char err[256] = "";
    CU(cudaEventRecord(St.ev_build[0], St.stream));
    if (!clpt_gpu_build(St.verts.ptr, (int)n_verts, St.corners.ptr, (int)(n_corners / 3), St.build_params, St.gpu_tree,
                        St.stream, err, sizeof err)) {
        fprintf(stderr, "%s: invalid scene: %s\n", who, err);
        exit(EXIT_FAILURE);
    }
    CU(cudaEventRecord(St.ev_build[1], St.stream));
    if (!clpt_gpu_pack(St.gpu_tree, St.verts.ptr, St.corners.ptr, (int)(n_corners / 3), St.layout, St.stream, err,
                       sizeof err)) {
        fprintf(stderr, "%s: invalid scene: %s\n", who, err);
        exit(EXIT_FAILURE);
    }
    CU(cudaEventRecord(St.ev_build[2], St.stream));
    CU(cudaStreamSynchronize(St.stream));
    CU(cudaEventElapsedTime(&St.last_build_ms, St.ev_build[0], St.ev_build[1]));
    CU(cudaEventElapsedTime(&St.last_pack_ms, St.ev_build[1], St.ev_build[2]));
    St.scene_on_gpu = true;
    adopt_layout((int)(n_corners / 3));
}
} // namespace

void CLBuildMeshes(const void *verts, size_t vert_bytes, const void *tris, size_t tri_bytes, const void *norms,
                   size_t norm_bytes) {
    require_init("CLBuildMeshes");
    release_host_kd();
    const size_t n_verts = vert_bytes / sizeof(Vector4), n_corners = tri_bytes / sizeof(cl_int3);
    const size_t n_norms = norms ? norm_bytes / sizeof(Vector4) : 0;
    if (n_verts == 0 || n_corners < 3) FATAL("CLBuildMeshes: empty mesh");
    // the mesh crosses PCIe once; everything after it happens on the device
    St.verts.resize(n_verts);
    CU(cudaMemcpyAsync(St.verts.ptr, verts, n_verts * sizeof(float4), cudaMemcpyHostToDevice, St.stream));
    St.corners.resize(n_corners);
    CU(cudaMemcpyAsync(St.corners.ptr, tris, n_corners * sizeof(int4), cudaMemcpyHostToDevice, St.stream));
    if (n_norms) {
        St.norms.resize(n_norms);
        CU(cudaMemcpyAsync(St.norms.ptr, norms, n_norms * sizeof(float4), cudaMemcpyHostToDevice, St.stream));
    } else {
        St.norms.release();
    }
    St.tri_material.release();
    St.mesh_on_gpu = true;
    rebuild_on_device("CLBuildMeshes");
}

void CLUpdateVertices(size_t first_vertex, const void *verts, size_t vert_bytes) {
    require_init("CLUpdateVertices");
    if (!St.mesh_on_gpu) FATAL("CLUpdateVertices: no mesh was uploaded with CLBuildMeshes");
    const size_t n = vert_bytes / sizeof(Vector4);
    if (first_vertex + n > St.verts.count) FATAL("CLUpdateVertices: range past the end of the vertex array");
    if (n) {
        CU(cudaMemcpyAsync(St.verts.ptr + first_vertex, verts, n * sizeof(float4), cudaMemcpyHostToDevice, St.stream));
    }
}

void CLRebuildMeshes(void) {
    require_init("CLRebuildMeshes");
    if (!St.mesh_on_gpu) FATAL("CLRebuildMeshes: no mesh was uploaded with CLBuildMeshes");
    rebuild_on_device("CLRebuildMeshes");
}

void CLLastBuildMs(float *build_ms, float *pack_ms) {
    if (build_ms) *build_ms = St.last_build_ms;
    if (pack_ms) *pack_ms = St.last_pack_ms;
}

void CLBuildStats(int *nodes, int *tri_refs, int *levels) {
    if (nodes) *nodes = St.gpu_tree.n_nodes;
    if (tri_refs) *tri_refs = St.gpu_tree.n_refs;
    if (levels) *levels = St.gpu_tree.levels;
}

int CLLastBuildWasRecorded(void) { return clpt_gpu_build_was_recorded() ? 1 : 0; }

void CLDownloadKd(kd *out) {
    require_init("CLDownloadKd");
    if (!St.scene_on_gpu) FATAL("CLDownloadKd: the current scene was not built by CLBuildMeshes");
    download_tree(St.gpu_tree, St.verts, St.corners, St.norms, out);
}

int CLAddInstanceMesh(const void *verts, size_t vert_bytes, const void *tris, size_t tri_bytes, const void *norms,
                      size_t norm_bytes) {
    require_init("CLAddInstanceMesh");
    const size_t n_verts = vert_bytes / sizeof(Vector4), n_corners = tri_bytes / sizeof(cl_int3);
    const size_t n_norms = norms ? norm_bytes / sizeof(Vector4) : 0;
    if (!verts || !tris || n_verts == 0 || n_corners < 3) FATAL("CLAddInstanceMesh: empty mesh");
    auto M = std::make_unique<decltype(St)::InstanceMesh>();
    M->verts.resize(n_verts);
    CU(cudaMemcpyAsync(M->verts.ptr, verts, n_verts * sizeof(float4), cudaMemcpyHostToDevice, St.stream));
    M->corners.resize(n_corners);
    CU(cudaMemcpyAsync(M->corners.ptr, tris, n_corners * sizeof(int4), cudaMemcpyHostToDevice, St.stream));
    if (n_norms) {
        M->norms.resize(n_norms);
        CU(cudaMemcpyAsync(M->norms.ptr, norms, n_norms * sizeof(float4), cudaMemcpyHostToDevice, St.stream));
    }
    // The builder's recorded graph is keyed by the buffers it writes, so a build into this mesh's
    // tree after one of the base scene (or the other way round) records the graph again: correct,
    // and only the steady replay of one and the same build is what the recording is for.
    const int n_prims = (int)(n_corners / 3);
    char err[256] = "";
    if (!clpt_gpu_build(M->verts.ptr, (int)n_verts, M->corners.ptr, n_prims, St.build_params, M->tree, St.stream, err,
                        sizeof err) ||
        !clpt_gpu_pack(M->tree, M->verts.ptr, M->corners.ptr, n_prims, M->layout, St.stream, err, sizeof err)) {
        fprintf(stderr, "CLAddInstanceMesh: invalid scene: %s\n", err);
        exit(EXIT_FAILURE);
    }
    CU(cudaStreamSynchronize(St.stream));
    set_scene_mesh(M->scene, M->layout, M->corners, M->norms);
    M->scene.n_prims = n_prims;
    St.inst_meshes.push_back(std::move(M));
    return (int)St.inst_meshes.size() - 1;
}

void CLSetInstances(const CLInstance *instances, size_t bytes) {
    require_init("CLSetInstances");
    static_assert(sizeof(CLInstance) == 64, "CLInstance is 64 bytes");
    if (bytes % sizeof(CLInstance) != 0) {
        fprintf(stderr, "CLSetInstances: %zu bytes is not a whole number of 64-byte CLInstance records\n", bytes);
        exit(EXIT_FAILURE);
    }
    const size_t n = bytes / sizeof(CLInstance);
    if (n > CLPT_MAX_INSTANCES) {
        fprintf(stderr, "CLSetInstances: %zu instances, at most %d\n", n, CLPT_MAX_INSTANCES);
        exit(EXIT_FAILURE);
    }
    if (n && !instances) FATAL("CLSetInstances: NULL instances");
    for (size_t k = 0; k < n; k++) {
        const CLInstance &in = instances[k];
        if (in.mesh < 0 || (size_t)in.mesh >= St.inst_meshes.size()) {
            fprintf(stderr, "CLSetInstances: instance %zu names mesh %d; %zu instance meshes exist\n", k, in.mesh,
                    St.inst_meshes.size());
            exit(EXIT_FAILURE);
        }
        for (int e = 0; e < 12; e++) {
            if (!std::isfinite(in.world_to_object[e])) {
                fprintf(stderr, "CLSetInstances: instance %zu: world_to_object[%d] is not finite\n", k, e);
                exit(EXIT_FAILURE);
            }
        }
    }
    St.instances.assign(instances, instances + n);
    St.inst_table_stale = true;
}

void CLClearInstanceMeshes(void) {
    require_init("CLClearInstanceMeshes");
    CU(cudaStreamSynchronize(St.stream));
    release_instance_meshes();
}

void CLDownloadInstanceKd(int mesh, kd *out) {
    require_init("CLDownloadInstanceKd");
    if (mesh < 0 || (size_t)mesh >= St.inst_meshes.size()) {
        fprintf(stderr, "CLDownloadInstanceKd: no instance mesh %d (%zu exist)\n", mesh, St.inst_meshes.size());
        exit(EXIT_FAILURE);
    }
    const auto &M = *St.inst_meshes[mesh];
    download_tree(M.tree, M.verts, M.corners, M.norms, out);
}

size_t CLDebugReadPacked(int which, void *dst, size_t bytes) {
    require_init("CLDebugReadPacked");
    if (!St.have_scene) FATAL("CLDebugReadPacked: no scene");
    const ClptScene &S = St.scene;
    const void *src = nullptr;
    size_t have = 0;
    switch (which) {
    case 0: src = S.nodes, have = (size_t)S.n_nodes * sizeof(uint2); break;
    case 1: src = S.leaves, have = (size_t)S.n_leaves * 4 * sizeof(float4); break;
    case 2: src = S.tri, have = (size_t)S.n_refs * 3 * sizeof(float4); break;
    case 3: src = S.lut, have = (size_t)S.lut_dim[0] * S.lut_dim[1] * S.lut_dim[2] * sizeof(int); break;
    case 4: src = S.flat_n, have = (size_t)S.n_prims * sizeof(float4); break;
    default: FATAL("CLDebugReadPacked: which must be 0 (nodes), 1 (leaves), 2 (triangles), 3 (start table) or 4 (flat normals)");
    }
    if (dst && bytes >= have && have) CU(cudaMemcpy(dst, src, have, cudaMemcpyDeviceToHost));
    return have;
}

void CLSetMaterials(const CLMaterial *materials, size_t material_bytes, const int *tri_material,
                    size_t tri_material_bytes) {
    require_init("CLSetMaterials");
    static_assert(sizeof(CLMaterial) == sizeof(ClptMaterial), "material layout");
    St.materials.upload(reinterpret_cast<const ClptMaterial *>(materials), material_bytes / sizeof(CLMaterial),
                        St.stream);
    const size_t n = tri_material ? tri_material_bytes / sizeof(int) : 0;
    if (n && St.have_scene && n != (size_t)St.scene.n_prims) {
        fprintf(stderr, "CLSetMaterials: %zu per-triangle ids for %d triangles\n", n, St.scene.n_prims);
        exit(EXIT_FAILURE);
    }
    if (n) {
        St.tri_material.upload(tri_material, n, St.stream);
    } else {
        St.tri_material.release();
    }
    rebuild_scene_struct();
}

void CLSetRenderParams(int mode, int depth, int spp, unsigned int seed, int flags) {
    require_init("CLSetRenderParams");
    if (mode < 0 || mode > 2) FATAL("CLSetRenderParams: mode must be 0, 1 or 2");
    if (spp < 1) FATAL("CLSetRenderParams: spp must be >= 1");
    St.mode = mode;
    St.depth = depth;
    St.spp = spp;
    St.seed = seed;
    St.flags = flags & (CLPT_FLAG_JITTER | CLPT_FLAG_ACCUMULATE | CLPT_FLAG_COUNTERS); // other bits are internal
}

void CLSetEngine(int engine) {
    if (engine < 0 || engine > 2) FATAL("CLSetEngine: 0 auto, 1 full occupancy, 2 fat-leaf variant");
    St.engine = engine;
}

int CLLastEngine(void) { return St.last_engine; }

void CLSetMaxLeafVisits(int cap) {
    if (cap < 1) FATAL("CLSetMaxLeafVisits: cap must be >= 1");
    St.max_leaf_visits = cap;
}

void CLDeleteImage(void) {
    require_init("CLDeleteImage");
    if (!St.have_image) FATAL("CLDeleteImage: no render target"); // clReleaseMemObject(0) errors too
    p2p_teardown(); // collective: no rank frees a frame its peers still map
    release_read_pipeline();
    if (clpt_gl_registered()) clpt_gl_unregister();
    release_targets();
    St.have_image = St.headless = false;
    St.width = St.height = 0;
}

void CLCreateImageHeadless(int width, int height) {
    require_init("CLCreateImageHeadless");
    if (width < 1 || height < 1) FATAL("CLCreateImageHeadless: bad size");
    St.width = width;
    St.height = height;
    St.headless = true;
    St.have_image = true;
    alloc_targets();
}

void CLCreateImage(unsigned int texture) {
    require_init("CLCreateImage");
    // needs a GL context current on this thread; fails loudly otherwise (gl_interop.cu)
    clpt_gl_register(texture);
    clpt_gl_size(&St.width, &St.height, St.stream);
    St.headless = false;
    St.have_image = true;
    alloc_targets(); // the float4 frame the kernels render into; presented to the texture per frame
}

void CLResetAccumulation(void) {
    require_init("CLResetAccumulation");
    if (!St.have_image) return;
    if (St.accum.ptr) clpt_launch_fill_u64(St.accum.ptr, St.accum.count, St.stream);
    CU(cudaStreamSynchronize(St.stream));
    St.sample_base = 0;
}

void CLExecute(int width, int height) { clpt_state_launch_frame(width, height); }

void CLReadImage(float *dst_rgba, size_t bytes) {
    check_read("CLReadImage", bytes, CLPT_READ_FLOAT4);
    wait_reads(0);
    const float4 *src = displayable_frame();
    CU(cudaMemcpyAsync(dst_rgba, src, bytes, cudaMemcpyDeviceToHost, St.stream));
    CU(cudaStreamSynchronize(St.stream));
}

void CLReadImageRGBA8(unsigned char *dst_rgba8, size_t bytes) {
    check_read("CLReadImageRGBA8", bytes, CLPT_READ_RGBA8);
    enqueue_read(dst_rgba8, bytes, CLPT_READ_RGBA8);
    wait_reads(0);
}

void CLReadImageAsync(void *dst, size_t bytes, int format) {
    check_read("CLReadImageAsync", bytes, format);
    enqueue_read(dst, bytes, format);
}

void CLReadImageWait(int leave_pending) {
    require_init("CLReadImageWait");
    wait_reads(leave_pending < 0 ? 0 : (unsigned long long)leave_pending);
}

void CLEnableAOV(int enable) {
    require_init("CLEnableAOV");
    St.aov = enable != 0;
    if (St.have_image && St.aov && St.aov_prim.count != (size_t)St.width * St.height) alloc_aovs();
}

void CLReadAOV(int *prim_id, float *t_hit, float *uv) {
    require_init("CLReadAOV");
    if (!St.aov || !St.aov_prim.ptr) FATAL("CLReadAOV: AOVs are not enabled (CLEnableAOV before the frame)");
    const size_t px = (size_t)St.width * St.height;
    if (prim_id) CU(cudaMemcpy(prim_id, St.aov_prim.ptr, px * sizeof(int), cudaMemcpyDeviceToHost));
    if (t_hit) CU(cudaMemcpy(t_hit, St.aov_t.ptr, px * sizeof(float), cudaMemcpyDeviceToHost));
    if (uv) CU(cudaMemcpy(uv, St.aov_uv.ptr, px * sizeof(float2), cudaMemcpyDeviceToHost));
}

void CLGetCounters(unsigned long long out[6]) { memcpy(out, St.host_counters, sizeof(St.host_counters)); }
float CLLastKernelMs(void) { return St.last_kernel_ms; }
int CLLastLaunchCount(void) { return St.last_launches; }

void CLEventRecord(int slot) {
    require_init("CLEventRecord");
    if (slot < 0 || slot >= 8) FATAL("CLEventRecord: slot out of range");
    CU(cudaEventRecord(St.ev_user[slot], St.stream));
}

float CLEventElapsedMs(int start_slot, int stop_slot) {
    require_init("CLEventElapsedMs");
    if (start_slot < 0 || start_slot >= 8 || stop_slot < 0 || stop_slot >= 8)
        FATAL("CLEventElapsedMs: slot out of range");
    float ms = 0;
    CU(cudaEventSynchronize(St.ev_user[stop_slot]));
    CU(cudaEventElapsedTime(&ms, St.ev_user[start_slot], St.ev_user[stop_slot]));
    return ms;
}

void CLFlushL2(void) {
    require_init("CLFlushL2");
    const size_t bytes = (size_t)St.prop.l2CacheSize * 2 > (256u << 20) ? (size_t)St.prop.l2CacheSize * 2
                                                                         : (size_t)(256u << 20);
    if (St.l2_flush.count != bytes) St.l2_flush.resize(bytes);
    CU(cudaMemsetAsync(St.l2_flush.ptr, 0, bytes, St.stream));
    CU(cudaStreamSynchronize(St.stream));
}

void CLSetTileShard(int rank, int nranks, int tile_rows) {
    require_init("CLSetTileShard");
    if (nranks < 1 || rank < 0 || rank >= nranks || tile_rows < 4 || (tile_rows % 4) != 0)
        FATAL("CLSetTileShard: need 0 <= rank < nranks and tile_rows a positive multiple of 4");
    // "sharding without a communicator": with a live communicator the gather buffers and the
    // peer mappings are sized for ITS rank count, so the shard has to agree with it
    if (St.comm && nranks != St.comm_ranks)
        FATAL("CLSetTileShard: nranks differs from the live communicator's (CLDistShutdown first, or use CLDistInit)");
    p2p_teardown(); // under the sharding the mappings were made for
    St.rank = rank;
    St.nranks = nranks;
    St.tile_rows = tile_rows;
    if (St.have_image) alloc_targets();
}

void CLDistGetUniqueId(void *id128) {
    nccl_load();
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NC(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
}

void CLDistInit(int rank, int nranks, const void *id128, int tile_rows) {
    require_init("CLDistInit");
    nccl_load();
    if (nranks < 1 || rank < 0 || rank >= nranks || tile_rows < 4 || (tile_rows % 4) != 0)
        FATAL("CLDistInit: need 0 <= rank < nranks and tile_rows a positive multiple of 4");
    p2p_teardown(); // collective over the OLD communicator, before it goes away
    if (St.comm) {
        CU(cudaStreamSynchronize(St.stream));
        NC(g_nccl.CommDestroy(St.comm));
        St.comm = nullptr;
        St.comm_ranks = 0;
    }
    St.rank = rank;
    St.nranks = nranks;
    St.tile_rows = tile_rows;
    if (nranks > 1) {
        ncclUniqueId id;
        memcpy(&id, id128, sizeof(id));
        CU(cudaSetDevice(St.device));
        NC(g_nccl.CommInitRank(&St.comm, nranks, id, rank));
        St.comm_ranks = nranks;
    }
    if (St.have_image) alloc_targets(); // collective: exchanges the frames' handles
}

void CLDistShutdown(void) {
    p2p_teardown();
    if (St.comm) {
        CU(cudaStreamSynchronize(St.stream));
        NC(g_nccl.CommDestroy(St.comm));
        St.comm = nullptr;
        St.comm_ranks = 0;
    }
    St.rank = 0;
    St.nranks = 1;
    if (St.inited && St.have_image) alloc_targets();
}

int CLDistDirectPlacement(void) { return St.p2p ? 1 : 0; }

const char *CLDeviceName(void) {
    require_init("CLDeviceName");
    return St.prop.name;
}

int CLDeviceSMCount(void) {
    require_init("CLDeviceSMCount");
    return St.prop.multiProcessorCount;
}

} // extern "C"
