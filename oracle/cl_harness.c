/* cl_harness.c -- run the reference's OWN kernel.cl through an OpenCL ICD.
 *
 * TEST INFRASTRUCTURE.  Harness C of SURVEY.md section 7/8c.  The reference's
 * device code (src/kernel.cl) is OpenCL C that is JIT-compiled at run time by
 * clBuildProgram (src/CLHandler.c:233-240); there is no OpenCL in the build
 * container, but the GPU box's driver ships libnvidia-opencl.so.1.  This file
 * drives the reference's kernel source through it (unmodified where the
 * compiler accepts it; see the build attempts in refcl_render), headless: the GL texture of
 * the reference (src/CLState.c:47-58) is replaced by a plain RGBA/float
 * image2d_t, everything else -- the nine kernel arguments, their order, the
 * raw 68-byte node array and index buffers, NDRange {w,h} with a NULL local
 * size, no build options -- is what src/CLState.c:204-265 does.
 *
 * The kernel source is not in this repository.  `make -C oracle ref` links
 * it into oracle/_ref/libref_kernel.so as an opaque data blob taken from
 * $CLPT_REFERENCE/src/kernel.cl where it lies (ld -r -b binary); oracle/_ref is
 * git-ignored and only travels to the GPU box next to the other built
 * checkers.
 *
 * No OpenCL headers exist in this image, so the handful of entry points and
 * constants used are declared here by hand (values from the Khronos
 * OpenCL 1.2 headers) and resolved with dlopen("libOpenCL.so.1").
 */
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

extern const char _binary_kernel_cl_start[];
extern const char _binary_kernel_cl_end[];

typedef int32_t cl_int;
typedef uint32_t cl_uint;
typedef uint64_t cl_ulong;
typedef cl_ulong cl_bitfield;
typedef struct _cl_platform_id *cl_platform_id;
typedef struct _cl_device_id *cl_device_id;
typedef struct _cl_context *cl_context;
typedef struct _cl_command_queue *cl_command_queue;
typedef struct _cl_mem *cl_mem;
typedef struct _cl_program *cl_program;
typedef struct _cl_kernel *cl_kernel;
typedef struct _cl_event *cl_event;
typedef struct { cl_uint image_channel_order, image_channel_data_type; } cl_image_format;

#define CL_DEVICE_TYPE_GPU (1 << 2)
#define CL_DEVICE_TYPE_ALL 0xFFFFFFFF
#define CL_MEM_WRITE_ONLY (1 << 1)
#define CL_MEM_READ_ONLY (1 << 2)
#define CL_MEM_COPY_HOST_PTR (1 << 5)
#define CL_RGBA 0x10B5
#define CL_FLOAT 0x10DE
#define CL_PROGRAM_BUILD_LOG 0x1183
#define CL_DEVICE_NAME 0x102B
#define CL_PLATFORM_NAME 0x0902
#define CL_QUEUE_PROFILING_ENABLE (1 << 1)
#define CL_PROFILING_COMMAND_START 0x1282
#define CL_PROFILING_COMMAND_END 0x1283

static struct {
    void *lib;
    cl_int (*GetPlatformIDs)(cl_uint, cl_platform_id *, cl_uint *);
    cl_int (*GetPlatformInfo)(cl_platform_id, cl_uint, size_t, void *, size_t *);
    cl_int (*GetDeviceIDs)(cl_platform_id, cl_bitfield, cl_uint, cl_device_id *, cl_uint *);
    cl_int (*GetDeviceInfo)(cl_device_id, cl_uint, size_t, void *, size_t *);
    cl_context (*CreateContext)(const intptr_t *, cl_uint, const cl_device_id *, void *, void *, cl_int *);
    cl_command_queue (*CreateCommandQueue)(cl_context, cl_device_id, cl_bitfield, cl_int *);
    cl_program (*CreateProgramWithSource)(cl_context, cl_uint, const char **, const size_t *, cl_int *);
    cl_int (*BuildProgram)(cl_program, cl_uint, const cl_device_id *, const char *, void *, void *);
    cl_int (*GetProgramBuildInfo)(cl_program, cl_device_id, cl_uint, size_t, void *, size_t *);
    cl_kernel (*CreateKernel)(cl_program, const char *, cl_int *);
    cl_mem (*CreateBuffer)(cl_context, cl_bitfield, size_t, void *, cl_int *);
    cl_mem (*CreateImage2D)(cl_context, cl_bitfield, const cl_image_format *, size_t, size_t, size_t, void *, cl_int *);
    cl_int (*SetKernelArg)(cl_kernel, cl_uint, size_t, const void *);
    cl_int (*EnqueueNDRangeKernel)(cl_command_queue, cl_kernel, cl_uint, const size_t *, const size_t *,
                                   const size_t *, cl_uint, const cl_event *, cl_event *);
    cl_int (*EnqueueReadImage)(cl_command_queue, cl_mem, cl_uint, const size_t *, const size_t *, size_t, size_t,
                               void *, cl_uint, const cl_event *, cl_event *);
    cl_int (*Finish)(cl_command_queue);
    cl_int (*GetEventProfilingInfo)(cl_event, cl_uint, size_t, void *, size_t *);
    cl_int (*ReleaseMemObject)(cl_mem);
    cl_int (*ReleaseKernel)(cl_kernel);
    cl_int (*ReleaseProgram)(cl_program);
    cl_int (*ReleaseCommandQueue)(cl_command_queue);
    cl_int (*ReleaseContext)(cl_context);
    cl_int (*ReleaseEvent)(cl_event);
} cl;

static int load_cl(char *msg, int len) {
    if (cl.lib) return 0;
    const char *names[] = { "libOpenCL.so.1", "libOpenCL.so", "/usr/local/cuda/targets/x86_64-linux/lib/libOpenCL.so.1" };
    for (int i = 0; i < 3 && !cl.lib; i++) cl.lib = dlopen(names[i], RTLD_NOW | RTLD_LOCAL);
    if (!cl.lib) {
        snprintf(msg, len, "no libOpenCL.so.1: %s", dlerror());
        return 1;
    }
#define SYM(field, name)                                                   \
    *(void **)(&cl.field) = dlsym(cl.lib, name);                           \
    if (!cl.field) { snprintf(msg, len, "missing symbol %s", name); return 1; }
    SYM(GetPlatformIDs, "clGetPlatformIDs") SYM(GetPlatformInfo, "clGetPlatformInfo")
    SYM(GetDeviceIDs, "clGetDeviceIDs") SYM(GetDeviceInfo, "clGetDeviceInfo")
    SYM(CreateContext, "clCreateContext") SYM(CreateCommandQueue, "clCreateCommandQueue")
    SYM(CreateProgramWithSource, "clCreateProgramWithSource") SYM(BuildProgram, "clBuildProgram")
    SYM(GetProgramBuildInfo, "clGetProgramBuildInfo") SYM(CreateKernel, "clCreateKernel")
    SYM(CreateBuffer, "clCreateBuffer") SYM(CreateImage2D, "clCreateImage2D")
    SYM(SetKernelArg, "clSetKernelArg") SYM(EnqueueNDRangeKernel, "clEnqueueNDRangeKernel")
    SYM(EnqueueReadImage, "clEnqueueReadImage") SYM(Finish, "clFinish")
    SYM(GetEventProfilingInfo, "clGetEventProfilingInfo") SYM(ReleaseMemObject, "clReleaseMemObject")
    SYM(ReleaseKernel, "clReleaseKernel") SYM(ReleaseProgram, "clReleaseProgram")
    SYM(ReleaseCommandQueue, "clReleaseCommandQueue") SYM(ReleaseContext, "clReleaseContext")
    SYM(ReleaseEvent, "clReleaseEvent")
#undef SYM
    return 0;
}

static int pick_device(cl_platform_id *plat, cl_device_id *dev, char *msg, int len) {
    cl_platform_id plats[8];
    cl_uint np = 0;
    cl_int e = cl.GetPlatformIDs(8, plats, &np);
    if (e != 0 || np == 0) {
        snprintf(msg, len, "clGetPlatformIDs: error %d, %u platforms (set OCL_ICD_FILENAMES to the vendor library)", e, np);
        return 1;
    }
    for (cl_uint p = 0; p < np; p++) {
        cl_uint nd = 0;
        if (cl.GetDeviceIDs(plats[p], CL_DEVICE_TYPE_ALL, 1, dev, &nd) == 0 && nd > 0) {
            *plat = plats[p];
            return 0;
        }
    }
    snprintf(msg, len, "no OpenCL device on %u platform(s)", np);
    return 1;
}

/* 0 when an OpenCL device is usable; msg receives "platform / device" or the reason. */
int refcl_available(char *msg, int len) {
    cl_platform_id plat;
    cl_device_id dev;
    if (load_cl(msg, len) || pick_device(&plat, &dev, msg, len)) return 1;
    char pn[128] = "", dn[128] = "";
    cl.GetPlatformInfo(plat, CL_PLATFORM_NAME, sizeof pn, pn, NULL);
    cl.GetDeviceInfo(dev, CL_DEVICE_NAME, sizeof dn, dn, NULL);
    snprintf(msg, len, "%s / %s", pn, dn);
    return 0;
}

static const char *g_build_options = "";
/* The clBuildProgram options the last successful refcl_render needed ("" = none, like the reference). */
const char *refcl_build_options(void) { return g_build_options; }

size_t refcl_kernel_source_bytes(void) { return (size_t)(_binary_kernel_cl_end - _binary_kernel_cl_start); }

#define CHECK(e, what)                                             \
    if ((e) != 0) {                                                \
        snprintf(log, loglen, "%s: OpenCL error %d", what, (int)(e)); \
        return 2;                                                  \
    }

/* ---- the bounce code of the reference, made runnable (mode B pin) ----------
 *
 * As shipped, trace_ray returns at src/kernel.cl:396-397 and the mirror bounce
 * after that `return` (:399-417) is dead; it is also a self-recursion (:406),
 * which OpenCL C forbids and the device stack does not survive.  To let the
 * VENDOR compiler execute exactly that code, the source is rewritten as TEXT:
 * trace_ray (:296-422) is cloned `depth` times, each clone is the reference's
 * function character for character except that
 *   - it has its own name,
 *   - the early `return convert_color((normal + 1) / 2) ... ;` statement is
 *     removed (so :399-417 runs), and
 *   - the recursive call names the next clone instead of itself.
 * The last clone is the function AS SHIPPED (early return kept; it is entered
 * with depth 0 and falls through to `return (1-str)*col + str;`, :421).  The
 * depth literal `2` in render (:468) becomes `depth`.  No arithmetic, no
 * operand order and no constant is touched.  Returns a malloc'd string, or
 * NULL (what is set) when the expected text is not found. */
static char *find_in(char *hay, const char *needle) { return hay ? strstr(hay, needle) : NULL; }

static void replace_once(char **text, const char *needle, const char *with, const char **what) {
    char *at = find_in(*text, needle);
    if (!at) {
        if (*text) *what = needle;
        free(*text);
        *text = NULL;
        return;
    }
    size_t head = (size_t)(at - *text), nl = strlen(needle), wl = strlen(with), tl = strlen(*text);
    char *out = malloc(tl - nl + wl + 1);
    memcpy(out, *text, head);
    memcpy(out + head, with, wl);
    memcpy(out + head + wl, at + nl, tl - head - nl + 1);
    free(*text);
    *text = out;
}

static char *dup_range(const char *a, const char *b) {
    char *r = malloc((size_t)(b - a) + 1);
    memcpy(r, a, (size_t)(b - a));
    r[b - a] = '\0';
    return r;
}

static char *bounce_source(const char *src, size_t srclen, int depth, const char **what) {
    static const char fn_head[] = "color\ntrace_ray(Ray r,";
    static const char fn_next[] = "kernel void";
    static const char early_a[] = "return convert_color((normal + 1) / 2)/*";
    static const char early_b[] = "*/;";
    static const char call[] = "return trace_ray(newRay,";
    static const char literal[] = "kd_tree,\n                    2,\n";
    char *all = dup_range(src, src + srclen);
    char *fs = strstr(all, fn_head), *fe = fs ? strstr(fs, fn_next) : NULL;
    if (!fs || !fe) {
        *what = "trace_ray definition";
        free(all);
        return NULL;
    }
    char *fn = dup_range(fs, fe);
    size_t cap = srclen + (size_t)(depth + 2) * (strlen(fn) + 64) + 64, len = 0;
    char *out = malloc(cap);
    memcpy(out, all, (size_t)(fs - all));
    len = (size_t)(fs - all);
    /* clones, deepest first so that every callee is defined before its caller */
    for (int level = depth; level >= 0; level--) {
        char name[32], callee[64], defn[64];
        char *c = dup_range(fn, fn + strlen(fn));
        if (level == 0) snprintf(name, sizeof name, "trace_ray");
        else snprintf(name, sizeof name, "trace_ray_%d", level);
        snprintf(defn, sizeof defn, "color\n%s(Ray r,", name);
        replace_once(&c, fn_head, defn, what);
        if (level == depth) { /* as shipped; its dead self-call keeps naming itself */
            snprintf(callee, sizeof callee, "return %s(newRay,", name);
            replace_once(&c, call, callee, what);
        } else {
            char *a = find_in(c, early_a), *b = a ? strstr(a, early_b) : NULL;
            if (!a || !b) {
                *what = "early return statement";
                free(c);
                c = NULL;
            } else {
                memmove(a, b + sizeof early_b - 1, strlen(b + sizeof early_b - 1) + 1);
                snprintf(callee, sizeof callee, "return trace_ray_%d(newRay,", level + 1);
                replace_once(&c, call, callee, what);
            }
        }
        if (!c) {
            free(out);
            free(fn);
            free(all);
            return NULL;
        }
        memcpy(out + len, c, strlen(c));
        len += strlen(c);
        free(c);
    }
    size_t tail = strlen(fe);
    memcpy(out + len, fe, tail + 1);
    free(fn);
    free(all);
    char lit[64];
    snprintf(lit, sizeof lit, "kd_tree,\n                    %d,\n", depth);
    /* the literal sits in render, after every clone */
    char *render_at = strstr(out + len, literal);
    if (!render_at) {
        *what = "depth literal in render";
        free(out);
        return NULL;
    }
    char *headpart = dup_range(out, render_at), *rest = dup_range(render_at, out + len + tail);
    free(out);
    replace_once(&rest, literal, lit, what);
    if (!rest) {
        free(headpart);
        return NULL;
    }
    out = malloc(strlen(headpart) + strlen(rest) + 1);
    strcpy(out, headpart);
    strcat(out, rest);
    free(headpart);
    free(rest);
    return out;
}

/* The rewritten source the last bounce render compiled (for inspection/tests); caller frees. */
char *refcl_bounce_source(int depth) {
    const char *what = NULL;
    return bounce_source(_binary_kernel_cl_start, refcl_kernel_source_bytes(), depth, &what);
}
void refcl_free(void *p) { free(p); }

/* Render one frame with the reference kernel, exactly the launch of
 * src/CLState.c:204-219.  rgba_out: w*h*4 floats.  kernel_ms: device time of the
 * NDRange from event profiling, best of `repeats`. */
int refcl_render_depth(const void *nodes, size_t node_bytes, const int *tri_indices, size_t tri_index_bytes,
                       const void *tris, size_t tri_bytes, const void *verts, size_t vert_bytes, const void *norms,
                       size_t norm_bytes, const float cam[16], int w, int h, int repeats, int bounce_depth,
                       float *rgba_out, double *kernel_ms, char *log, int loglen) {
    cl_platform_id plat;
    cl_device_id dev;
    cl_int e;
    if (load_cl(log, loglen) || pick_device(&plat, &dev, log, loglen)) return 1;
    cl_context ctx = cl.CreateContext(NULL, 1, &dev, NULL, NULL, &e);
    CHECK(e, "clCreateContext");
    cl_command_queue q = cl.CreateCommandQueue(ctx, dev, CL_QUEUE_PROFILING_ENABLE, &e);
    CHECK(e, "clCreateCommandQueue");
    /* The reference builds its source with no options (src/CLHandler.c:240).
     * Its helper `mul(const matrix M, vec3 X)` (kernel.cl:90) takes a pointer
     * with no address space and is called with the __global camera buffer
     * (kernel.cl:447,451).  Compilers that enforce OpenCL C 1.x address spaces
     * (NVIDIA's) reject that; the reference evidently ran on a lenient one.
     * Attempts, in order, until one builds -- the one used is reported by
     * refcl_build_options():
     *   1. the unmodified source, no options              (the reference's own build)
     *   2. the unmodified source, -cl-std=CL2.0 / CL3.0   (generic address space)
     *   3. the source with that ONE parameter declaration qualified __global,
     *      patched in memory -- no arithmetic is touched. */
    static const char *labels[] = { "", "-cl-std=CL2.0", "-cl-std=CL3.0",
                                    "source patched in memory: mul() parameter `const matrix M` -> `global const vec4 *M`" };
    static const char *options[] = { NULL, "-cl-std=CL2.0", "-cl-std=CL3.0", NULL };
    /* bounce_depth <= 0: the source as shipped.  Otherwise the text rewrite above. */
    const char *refsrc = _binary_kernel_cl_start;
    size_t reflen = refcl_kernel_source_bytes();
    char *bounce = NULL;
    if (bounce_depth > 0) {
        const char *what = NULL;
        bounce = bounce_source(refsrc, reflen, bounce_depth, &what);
        if (!bounce) {
            snprintf(log, loglen, "bounce rewrite: `%s` not found in kernel.cl", what ? what : "?");
            return 3;
        }
        refsrc = bounce;
        reflen = strlen(bounce);
    }
    static const char needle[] = "mul(const matrix M, vec3 X)";
    static const char patch[] = "mul(global const vec4 *M, vec3 X)";
    char *patched = NULL;
    cl_program prog = NULL;
    int used = -1;
    char first_log[4096] = "";
    for (int i = 0; i < 4 && used < 0; i++) {
        const char *src = refsrc;
        size_t srclen = reflen;
        if (i == 3) {
            const char *at = NULL;
            for (size_t p = 0; p + sizeof needle - 1 <= reflen; p++) {
                if (memcmp(refsrc + p, needle, sizeof needle - 1) == 0) {
                    at = refsrc + p;
                    break;
                }
            }
            if (!at) break;
            size_t head = (size_t)(at - refsrc);
            patched = malloc(reflen + sizeof patch);
            memcpy(patched, refsrc, head);
            memcpy(patched + head, patch, sizeof patch - 1);
            memcpy(patched + head + sizeof patch - 1, at + sizeof needle - 1, reflen - head - (sizeof needle - 1));
            src = patched;
            srclen = reflen - (sizeof needle - 1) + (sizeof patch - 1);
        }
        if (prog) cl.ReleaseProgram(prog);
        prog = cl.CreateProgramWithSource(ctx, 1, &src, &srclen, &e);
        CHECK(e, "clCreateProgramWithSource");
        e = cl.BuildProgram(prog, 0, NULL, options[i], NULL, NULL);
        if (e == 0) {
            used = i;
        } else if (i == 0) {
            cl.GetProgramBuildInfo(prog, dev, CL_PROGRAM_BUILD_LOG, sizeof first_log - 1, first_log, NULL);
        }
    }
    if (used < 0) {
        size_t n = 0;
        int off = snprintf(log, loglen, "clBuildProgram: error %d on every attempt; log of the unmodified build:\n%s\nlast log:\n",
                           e, first_log);
        if (off < loglen - 1) cl.GetProgramBuildInfo(prog, dev, CL_PROGRAM_BUILD_LOG, (size_t)(loglen - off - 1), log + off, &n);
        free(patched);
        free(bounce);
        return 2;
    }
    free(patched);
    free(bounce);
    g_build_options = labels[used];
    cl_kernel k = cl.CreateKernel(prog, "render", &e); /* KERNEL_NAME, src/main.c:7 */
    CHECK(e, "clCreateKernel");

    cl_image_format fmt = { CL_RGBA, CL_FLOAT };
    cl_mem image = cl.CreateImage2D(ctx, CL_MEM_WRITE_ONLY, &fmt, (size_t)w, (size_t)h, 0, NULL, &e);
    CHECK(e, "clCreateImage2D");
    char dummy[64] = { 0 };
#define BUF(name, ptr, bytes)                                                                          \
    cl_mem name = cl.CreateBuffer(ctx, CL_MEM_READ_ONLY | CL_MEM_COPY_HOST_PTR, (bytes) ? (bytes) : sizeof dummy, \
                                  (bytes) ? (void *)(ptr) : (void *)dummy, &e);                         \
    CHECK(e, "clCreateBuffer " #name);
    BUF(b_cam, cam, (size_t)64)
    BUF(b_obj, NULL, (size_t)0)
    BUF(b_verts, verts, vert_bytes)
    BUF(b_norms, norms, norm_bytes)
    BUF(b_tris, tris, tri_bytes)
    BUF(b_idx, tri_indices, tri_index_bytes)
    BUF(b_kd, nodes, node_bytes)
#undef BUF
    cl_int objcount = 0;
    /* argument table of src/CLState.c:235-264 */
    CHECK(cl.SetKernelArg(k, 0, sizeof(cl_mem), &image), "arg0");
    CHECK(cl.SetKernelArg(k, 1, sizeof(cl_mem), &b_cam), "arg1");
    CHECK(cl.SetKernelArg(k, 2, sizeof(cl_mem), &b_obj), "arg2");
    CHECK(cl.SetKernelArg(k, 3, sizeof(cl_int), &objcount), "arg3");
    CHECK(cl.SetKernelArg(k, 4, sizeof(cl_mem), &b_verts), "arg4");
    CHECK(cl.SetKernelArg(k, 5, sizeof(cl_mem), &b_norms), "arg5");
    CHECK(cl.SetKernelArg(k, 6, sizeof(cl_mem), &b_tris), "arg6");
    CHECK(cl.SetKernelArg(k, 7, sizeof(cl_mem), &b_idx), "arg7");
    CHECK(cl.SetKernelArg(k, 8, sizeof(cl_mem), &b_kd), "arg8");

    size_t global[2] = { (size_t)w, (size_t)h };
    double best = -1;
    for (int r = 0; r < (repeats < 1 ? 1 : repeats); r++) {
        cl_event ev;
        CHECK(cl.EnqueueNDRangeKernel(q, k, 2, NULL, global, NULL, 0, NULL, &ev), "clEnqueueNDRangeKernel");
        CHECK(cl.Finish(q), "clFinish");
        cl_ulong t0 = 0, t1 = 0;
        cl.GetEventProfilingInfo(ev, CL_PROFILING_COMMAND_START, sizeof t0, &t0, NULL);
        cl.GetEventProfilingInfo(ev, CL_PROFILING_COMMAND_END, sizeof t1, &t1, NULL);
        cl.ReleaseEvent(ev);
        double ms = (double)(t1 - t0) * 1e-6;
        if (best < 0 || ms < best) best = ms;
    }
    if (kernel_ms) *kernel_ms = best;
    size_t origin[3] = { 0, 0, 0 }, region[3] = { (size_t)w, (size_t)h, 1 };
    CHECK(cl.EnqueueReadImage(q, image, 1, origin, region, 0, 0, rgba_out, 0, NULL, NULL), "clEnqueueReadImage");
    cl.ReleaseMemObject(image);
    cl.ReleaseMemObject(b_cam);
    cl.ReleaseMemObject(b_obj);
    cl.ReleaseMemObject(b_verts);
    cl.ReleaseMemObject(b_norms);
    cl.ReleaseMemObject(b_tris);
    cl.ReleaseMemObject(b_idx);
    cl.ReleaseMemObject(b_kd);
    cl.ReleaseKernel(k);
    cl.ReleaseProgram(prog);
    cl.ReleaseCommandQueue(q);
    cl.ReleaseContext(ctx);
    if (log && loglen) log[0] = '\0';
    return 0;
}

/* The kernel as shipped (first-hit normal colour). */
int refcl_render(const void *nodes, size_t node_bytes, const int *tri_indices, size_t tri_index_bytes,
                 const void *tris, size_t tri_bytes, const void *verts, size_t vert_bytes, const void *norms,
                 size_t norm_bytes, const float cam[16], int w, int h, int repeats, float *rgba_out,
                 double *kernel_ms, char *log, int loglen) {
    return refcl_render_depth(nodes, node_bytes, tri_indices, tri_index_bytes, tris, tri_bytes, verts, vert_bytes,
                              norms, norm_bytes, cam, w, h, repeats, 0, rgba_out, kernel_ms, log, loglen);
}
