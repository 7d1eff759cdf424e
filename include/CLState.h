/* CLState.h -- the render boundary, B200 edition.
 *
 * Drop-in for the reference's include/CLState.h:13-28: the same eight entry
 * points with the same names, argument meaning, ownership and error
 * behaviour, implemented with hand-written CUDA for sm_100a instead of an
 * OpenCL kernel.  A caller written against the reference header (GLState.c is
 * the only one, src/GLState.c:28-30,76-89,109,115,139-140) links against
 * libclpt.so unchanged.
 *
 * Conventions kept from the reference:
 *   - every function returns void; any device/runtime failure prints
 *     "file:line: CUDA Error: NAME" to stderr and exit(EXIT_FAILURE)s
 *     (include/error.h:3, src/error.c:147-154)
 *   - single host thread, every call is synchronous; CLExecute returns when
 *     the frame (and, multi-GPU, its gather) is complete (src/CLState.c:212)
 *   - file-static singleton state (src/CLState.c:21-40)
 *   - CLSetMeshes takes models[0]'s five host lists; CLTerminate frees them
 *     (src/CLState.c:130,221-225)
 *
 * The "headless" block below has no counterpart in the reference, where the
 * frame only ever lives in a GL texture: it adds a float4 framebuffer that can
 * be read back, the render parameters the reference hard-codes, raw-pointer
 * twins of the by-value/fat-pointer calls for FFI callers, timing, and the
 * row-tile sharding used across GPUs.
 */
#ifndef CLSTATE_H
#define CLSTATE_H

#include <stddef.h>

#include "clpt_types.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- the reference's eight (include/CLState.h:13-28) ---- */

/* Bring the device up: pick the CUDA device (ordinal from CLSelectDevice or
 * $CLPT_DEVICE, default 0 -- never a stdin prompt, unlike src/CLHandler.c:42-53),
 * create the stream, the 64-byte camera buffer and default render parameters.
 * Both arguments are accepted for source compatibility and ignored: the
 * kernels are compiled into the library.  Replaces src/CLState.c:227-265. */
void CLInit(const char *kernel_filename, const char *kernel_name);

/* Free the host lists taken by CLSetMeshes and every device resource.
 * Replaces src/CLState.c:221-225. */
void CLTerminate(void);

/* Blocking upload of the inverse camera matrix (row-major, rows[r].s[c]).
 * Replaces src/CLState.c:67-79. */
void CLSetCameraMatrix(Matrix matrix);

/* Upload `size` BYTES of 24-byte packed Objects; no-op at size 0.  The
 * reference uploads spheres but never intersects them (src/kernel.cl:199-225
 * is unreferenced), and neither does this library: the slot exists for ABI
 * compatibility.  Replaces src/CLState.c:104-122. */
void CLSetObjects(Object *vec_objects, size_t size);

/* Take models[0] (models is a list.c vector of kd; an empty vector is a
 * no-op), re-pack its node array / tri_indices / tris / verts / norms into the
 * device layout (DESIGN.md "data layout in HBM") and upload it.  Ownership of
 * models[0]'s five lists passes to the library.  A later CLSetMeshes frees the
 * lists adopted before EXCEPT those the new kd carries again (same pointer), so
 * calling it again with the same kd after an in-place update is legal, as it is
 * in the reference (which never frees on a re-set).  Replaces src/CLState.c:124-202. */
void CLSetMeshes(kd *models);

/* Release the current render target.  Replaces src/CLState.c:42-45. */
void CLDeleteImage(void);

/* Bind a GL_TEXTURE_2D (RGBA8) as the render target through
 * cudaGraphicsGLRegisterImage; each CLExecute then maps it, writes the frame as
 * UNORM8 texels through a surface and unmaps it (the acquire/release of
 * src/CLState.c:207-218).  Needs an OpenGL context current on the calling
 * thread; without one the registration fails and the call aborts with the CUDA
 * error.  Replaces src/CLState.c:47-58. */
void CLCreateImage(unsigned int texture);

/* Render one frame of width x height pixels with the current camera, scene
 * and parameters into the render target, then synchronise.
 * Replaces src/CLState.c:204-219. */
void CLExecute(int width, int height);

/* ---- headless additions ---- */

enum {
    CLPT_MODE_NORMAL = 0, /* as shipped: first-hit normal colour (src/kernel.cl:395-397) */
    CLPT_MODE_MIRROR = 1, /* the dead code enabled: mirror bounces (src/kernel.cl:399-417) */
    CLPT_MODE_PATH = 2    /* extension: diffuse/mirror materials, stochastic */
};
enum {
    CLPT_FLAG_JITTER = 1,     /* sub-pixel jitter (implied by spp > 1 is NOT automatic: set it) */
    CLPT_FLAG_ACCUMULATE = 2, /* progressive: every frame adds its samples to per-pixel running sums
                               * (2^-32 fixed point, so the sums do not depend on the order of the
                               * additions); with N ranks a frame is N x spp samples per pixel --
                               * rank r renders the WHOLE frame with samples base + r*spp .. */
    CLPT_FLAG_COUNTERS = 4    /* instrumented launch: fill the work counters */
};

typedef struct CLMaterial { /* 32 bytes */
    float albedo[3];
    int kind; /* 0 diffuse, 1 mirror */
    float emission[3];
    float pad;
} CLMaterial;

void CLSelectDevice(int ordinal);          /* before CLInit; default $CLPT_DEVICE or 0 */
void CLSetCameraMatrixPtr(const Matrix *matrix);
/* Like CLSetMeshes but from plain pointers + byte sizes; the data is copied,
 * nothing is owned.  norms may be NULL / 0. */
void CLSetMeshesRaw(const void *nodes, size_t node_bytes,
                    const int *tri_indices, size_t tri_index_bytes,
                    const void *tris, size_t tri_bytes,
                    const void *verts, size_t vert_bytes,
                    const void *norms, size_t norm_bytes);
/* Device-side scene preparation (SURVEY.md section 8f row 1; no counterpart in the
 * reference, whose tree is built on the host by src/kd_tree.c:202-276 before
 * CLSetMeshes): the mesh -- verts 16 B each, three 16-byte corners {v, vn, vt, 0} per
 * triangle, optional normals; the lists LoadModel produces (src/model.c:74-145) -- is
 * uploaded once, a binned-SAH kd-tree with ropes is built ON THE DEVICE in the
 * reference's wire format and re-laid-out there for traversal.  Nothing is owned; the
 * data is copied.  The build is deterministic: the same mesh gives the same tree,
 * byte for byte, on every GPU.  CLSetBuildParams: max_depth <= 0 means
 * 8 + 1.3 log2(triangles); the cost constants are build_kd_sah's. */
void CLBuildMeshes(const void *verts, size_t vert_bytes, const void *tris, size_t tri_bytes,
                   const void *norms, size_t norm_bytes);
void CLSetBuildParams(int max_depth, int min_split, float traversal_cost, float intersect_cost,
                      float empty_bonus);
/* Animated scenes (BASELINE config 5: per-frame object transform + kd-tree re-upload):
 * overwrite a range of the uploaded vertex array in place -- only the vertices that
 * moved cross PCIe -- and rebuild tree and layout on the device from the resident
 * mesh.  CLBuildMeshes == upload + CLRebuildMeshes. */
void CLUpdateVertices(size_t first_vertex, const void *verts, size_t vert_bytes);
void CLRebuildMeshes(void);
void CLLastBuildMs(float *build_ms, float *pack_ms); /* device time of the last CLBuildMeshes */
void CLBuildStats(int *nodes, int *tri_refs, int *levels);
/* Meshes of up to 2^18 triangles are built without the host in the loop: the launches of
 * every level are recorded once (a CUDA graph, level counts in device memory, launch sizes
 * from fixed capacities) and replayed by every later CLRebuildMeshes of the same mesh size.
 * Larger meshes, and any mesh that outgrows the recorded capacities, are built level by
 * level with one synchronisation per level; the tree is the same either way.  1 if the
 * last build was the recorded one.  $CLPT_BUILD_NO_GRAPH=1 forces level by level. */
int CLLastBuildWasRecorded(void);
/* The tree CLBuildMeshes built, as a regular `kd` (fresh host lists the caller owns and
 * frees with delete_kd): what the oracle walks in the parity tests, and what write_kd
 * can cache. */
void CLDownloadKd(kd *out);
/* Test hook: the traversal layout in device memory, which = 0 nodes, 1 leaf records,
 * 2 triangle slots, 3 start-node table, 4 flat normals (one float4 per primitive).
 * Returns the size in bytes; copies when dst is large enough. */
size_t CLDebugReadPacked(int which, void *dst, size_t bytes);
void CLSetMaterials(const CLMaterial *materials, size_t material_bytes,
                    const int *tri_material, size_t tri_material_bytes);

/* Rigid instances: a mesh uploaded and built once, drawn any number of times under a rigid
 * (or any affine) transform by mapping each ray into the mesh's object space -- moving an
 * object costs one small upload per frame and no tree rebuild.
 *   - Object-space ray: o' = A o + b and d' = A d, each row left to right without FMA
 *     contraction; d' is NOT normalised, so the object-space t is the world ray's t.
 *   - A frame walks the base scene first, then the instances in array order, each with its own
 *     root clip, start table, ropes and rope-hop budget.  A later hit replaces the current one
 *     when t <= best (the later tree wins ties).  An instance is skipped when a hit exists and
 *     the ray enters the instance's root box beyond it.
 *   - Shading: the object-space normal before normalisation (the flat normal's cross product
 *     or the interpolated vertex normals) is mapped by A^T and normalised; the hit point and
 *     the bounce use the world ray.
 *   - Primitive ids: the base scene keeps [0, P); instance k's primitives follow at
 *     P + the primitives of the instances before it, P being the base scene current at
 *     CLExecute.  AOVs report that id, the world t and u, v in the instance's triangle.
 *   - Mode 2: every triangle of an instance has the instance's material (clamped like
 *     tri_material ids); work counters count one ray per world query and sum every walk.
 * A frame still needs a base scene.  Bad input (a handle out of range, a non-finite matrix
 * entry, a byte count that is not a multiple of 64, more than CLPT_MAX_INSTANCES) prints a
 * message and exit(EXIT_FAILURE)s. */
#define CLPT_MAX_INSTANCES 64
typedef struct CLInstance {      /* 64 bytes */
    float world_to_object[12];   /* row-major 3x4 [A | b]: object point = A * world point + b;
                                  * from an object-to-world matrix with mat_inverse (clpt_host.h) */
    int mesh;                    /* handle from CLAddInstanceMesh */
    int material;                /* mode 2: material of all its triangles */
    int pad[2];
} CLInstance;
/* Upload a mesh (the formats of CLBuildMeshes) and build its kd-tree and traversal layout on
 * the device, once.  Returns a handle >= 0.  The base scene (CLSetMeshes / CLBuildMeshes) is
 * untouched, and instance meshes survive base-scene changes until CLClearInstanceMeshes or
 * CLTerminate. */
int CLAddInstanceMesh(const void *verts, size_t vert_bytes, const void *tris, size_t tri_bytes,
                      const void *norms, size_t norm_bytes);
/* The instances of the next frames (replaces the previous set; NULL / 0 = none).  Per frame
 * this is the only upload a rigid motion needs.  At most CLPT_MAX_INSTANCES. */
void CLSetInstances(const CLInstance *instances, size_t bytes);
void CLClearInstanceMeshes(void);              /* frees every instance mesh and clears the instances */
void CLDownloadInstanceKd(int mesh, kd *out);  /* an instance mesh's tree, like CLDownloadKd */
/* mode, depth (= bounces + 1; the reference passes 2, src/kernel.cl:468),
 * samples per pixel per frame, RNG seed, CLPT_FLAG_* */
void CLSetRenderParams(int mode, int depth, int spp, unsigned int seed, int flags);
void CLSetMaxLeafVisits(int cap);          /* rope-hop cap per ray; default 4096 */
/* Execution engine: 1 = the render kernel compiled for 8 resident blocks per SM (32
 * registers), the fastest on deep trees where latency hiding decides; 2 = the same
 * code compiled for 4 (64 registers, no spills) -- made for trees from the
 * reference's own builder, whose DEPTH 15 cap (src/kd_tree.c:8-9) leaves ~56
 * triangles per leaf at 1M triangles: their frames are one long triangle loop,
 * which spills at 32 registers and does not at 64 (at one sample per pixel two
 * neighbouring lanes also walk each ray together and split its leaves' triangle
 * runs);
 * 0 = automatic: chosen per tree at CLSetMeshes (2 when most triangle slots sit in
 * leaves of >= 8 triangles).  Both produce the same bits. */
void CLSetEngine(int engine);
int CLLastEngine(void);                    /* engine the last CLExecute used: 1 or 2 */
void CLCreateImageHeadless(int width, int height); /* float4 target, zeroed */
void CLResetAccumulation(void);            /* zero the running sums and the sample counter */
/* Blocking device->host copy of the whole float4 frame (bytes must be
 * width*height*16).  With CLPT_FLAG_ACCUMULATE the running sums are divided by
 * the sample count on the way out.  Across GPUs progressive frames are spread by
 * sample, every rank keeps its own sums, and the read-back adds them
 * (ncclAllReduce of 64-bit integers: the same bits as one GPU adding all the
 * samples), which makes the CLReadImage* calls COLLECTIVE while
 * CLPT_FLAG_ACCUMULATE is set and a communicator is live; in every other case
 * only the calling rank pays. */
void CLReadImage(float *dst_rgba, size_t bytes);
/* The same frame as RGBA8 UNORM texels -- the format of the reference's render
 * target (src/GLHandler.c:177-185; what write_imagef stores: clamp, x255, round to
 * nearest even), 4 bytes per pixel (bytes must be width*height*4).  Blocking. */
void CLReadImageRGBA8(unsigned char *dst_rgba8, size_t bytes);
/* Pipelined read-back: the frame is snapshotted on the device in stream order and
 * travels to `dst` on a second stream, so the next CLExecute overlaps the copy.
 * `dst` (ideally page-locked) must stay valid until CLReadImageWait says the read
 * has landed.  Two reads may be in flight.  CLReadImageWait(n) returns once at most
 * n reads are still pending (0 = all landed). */
enum { CLPT_READ_FLOAT4 = 0, CLPT_READ_RGBA8 = 1 };
void CLReadImageAsync(void *dst, size_t bytes, int format);
void CLReadImageWait(int leave_pending);
/* First-hit outputs of sample 0 of the last frame: primitive id (-1 miss),
 * t, (u,v).  Any pointer may be NULL.  Only this rank's rows are valid when
 * sharded. */
void CLEnableAOV(int enable);
void CLReadAOV(int *prim_id, float *t_hit, float *uv);
/* rays, split visits, leaf visits, triangle tests, vn-shaded hits, capped
 * rays of the last frame rendered with CLPT_FLAG_COUNTERS */
void CLGetCounters(unsigned long long out[6]);
float CLLastKernelMs(void);                /* device time of the last frame's render kernel */
int CLLastLaunchCount(void);               /* kernels launched by the last CLExecute */
/* CUDA events on the library's own stream, for callers that time many frames */
void CLEventRecord(int slot);              /* slot 0..7 */
float CLEventElapsedMs(int start_slot, int stop_slot); /* synchronises stop */
void CLFlushL2(void);                      /* overwrite a buffer larger than L2 */

/* ---- multi-GPU: one process per GPU, row tiles interleaved round-robin ----
 * Rank r renders tiles t with t % nranks == r (tile = tile_rows image rows).
 * Direct placement (default, up to 8 ranks on one node): every rank maps the
 * other ranks' frames (CUDA IPC, peer access over NVLink) and the render kernel
 * stores each finished pixel into all of them; CLExecute brackets the frame
 * with two one-word barriers on the communicator and there is no gather pass.
 * Fallback ($CLPT_P2P=0 on every rank, or the mapping fails on any rank): the
 * rank renders into a compact slab, CLExecute all-gathers the slabs with NCCL
 * and de-interleaves them into every rank's target.
 * The id is created on rank 0 with CLDistGetUniqueId and carried to the others
 * by the caller.  With a communicator, CLDistInit, CLDistShutdown,
 * CLCreateImageHeadless, CLCreateImage, CLDeleteImage, CLSetTileShard, CLExecute
 * and CLTerminate are collective: every rank calls them in the same order. */
void CLDistGetUniqueId(void *id128);       /* 128 bytes out; one id per CLDistInit (NCCL ids are single-use) */
void CLDistInit(int rank, int nranks, const void *id128, int tile_rows);
void CLDistShutdown(void);
int CLDistDirectPlacement(void);           /* 1 while frames are peer-mapped (no gather pass), else 0 */
/* Sharding without a communicator (each rank keeps only its own rows). */
void CLSetTileShard(int rank, int nranks, int tile_rows);

const char *CLDeviceName(void);
int CLDeviceSMCount(void);

#ifdef __cplusplus
}
#endif

#endif /* CLSTATE_H */
