// scene_pack.cpp -- wire format -> device layout (host side of CLSetMeshes).
//
// Input is exactly what the reference uploads verbatim (src/CLState.c:124-202):
// the 68-byte preorder node array, tri_indices, three cl_int3 corners per
// triangle, float4 verts.  Output is the layout documented in clpt_device.cuh.
// The tree TOPOLOGY, the order of triangles inside each leaf and every float
// are preserved, so a traversal of the packed scene visits the same leaves and
// triangles in the same order as the reference kernel walking the input.
#include "scene_pack.h"

#ifdef _OPENMP
#include <omp.h>
#endif

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

clpt_host_alloc_fn clpt_pack_alloc = malloc;
clpt_host_free_fn clpt_pack_free = free;

namespace {

struct PackTimer {
    bool on = getenv("CLPT_PACK_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char *what) {
        if (!on) return;
        auto n = std::chrono::steady_clock::now();
        fprintf(stderr, "  pack %-12s %.2f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};

inline int as_int(float f) {
    int i;
    std::memcpy(&i, &f, 4);
    return i;
}
inline float as_float(int i) {
    float f;
    std::memcpy(&f, &i, 4);
    return f;
}
inline uint32_t float_bits(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}

} // namespace

bool clpt_pack_scene(const kdnode *nodes, size_t n_nodes, const int *tri_indices, size_t n_refs,
                     const cl_int3 *corners, size_t n_corners, const Vector4 *verts, size_t n_verts,
                     size_t n_norms, ClptPackedScene &out, std::string &err) {
    char msg[256];
    PackTimer timer;
    if (n_nodes == 0) {
        err = "empty node array";
        return false;
    }
    if (n_nodes >= (1u << 29)) {
        err = "too many nodes for the 29-bit child field";
        return false;
    }
    const size_t n_prims = n_corners / 3;

    // ---- renumber nodes: siblings adjacent, pairs in the order of their parents ----
    // The children of the k-th split node (in input order) become nodes 1+2k and
    // 2+2k.  For the preorder arrays the builders emit this is the depth-first pair
    // order (a subtree's pairs are contiguous); for any other input it is still a
    // valid numbering.  Ranks come from parallel prefix sums over the node types.
    std::vector<int> new_of(n_nodes, -1), leaf_of(n_nodes, -1);
    int n_leaves = 0, n_splits = 0;
    {
        int nthreads = 1;
#ifdef _OPENMP
        nthreads = omp_get_max_threads();
#endif
        std::vector<long long> split_base((size_t)nthreads + 1, 0), leaf_base((size_t)nthreads + 1, 0);
        long long bad_type = -1;
#pragma omp parallel num_threads(nthreads)
        {
            int t = 0, nt = 1;
#ifdef _OPENMP
            t = omp_get_thread_num();
            nt = omp_get_num_threads();
#endif
            const size_t lo = n_nodes * (size_t)t / nt, hi = n_nodes * (size_t)(t + 1) / nt;
            long long ns = 0, nl = 0;
            for (size_t i = lo; i < hi; i++) {
                if (nodes[i].type == KD_SPLIT) ns++;
                else if (nodes[i].type == KD_LEAF) nl++;
                else {
#pragma omp critical(clpt_pack_err)
                    if (bad_type < 0 || (long long)i < bad_type) bad_type = (long long)i;
                }
            }
            split_base[t + 1] = ns;
            leaf_base[t + 1] = nl;
#pragma omp barrier
#pragma omp single
            for (int k = 0; k < nt; k++) {
                split_base[k + 1] += split_base[k];
                leaf_base[k + 1] += leaf_base[k];
            }
            long long ks = split_base[t], kl = leaf_base[t];
            for (size_t i = lo; i < hi; i++) {
                if (nodes[i].type == KD_SPLIT) {
                    const int c0 = nodes[i].split.children[0], c1 = nodes[i].split.children[1];
                    if (c0 > 0 && c1 > 0 && (size_t)c0 < n_nodes && (size_t)c1 < n_nodes && c0 != c1) {
                        new_of[c0] = (int)(1 + 2 * ks); // each child has one parent: no two threads write one slot
                        new_of[c1] = (int)(2 + 2 * ks);
                    }
                    ks++;
                } else if (nodes[i].type == KD_LEAF) {
                    leaf_of[i] = (int)kl++; // input order: neighbours in space stay neighbours in memory
                }
            }
            if (t == nt - 1) {
                n_splits = (int)split_base[nt];
                n_leaves = (int)leaf_base[nt];
            }
        }
        if (bad_type >= 0) {
            snprintf(msg, sizeof msg, "node %lld has type %d", bad_type, nodes[bad_type].type);
            err = msg;
            return false;
        }
    }
    new_of[0] = 0;
    // every split must own exactly the pair its rank says (catches malformed or shared children)
    {
        long long bad_split = -1;
        long long ks_check = 0;
        (void)ks_check;
#pragma omp parallel for schedule(static)
        for (long long i = 0; i < (long long)n_nodes; i++) {
            if (nodes[i].type != KD_SPLIT) continue;
            const int c0 = nodes[i].split.children[0], c1 = nodes[i].split.children[1];
            const int ax = nodes[i].split.axis;
            bool ok = c0 > 0 && c1 > 0 && (size_t)c0 < n_nodes && (size_t)c1 < n_nodes && c0 != c1 && ax >= 0 && ax <= 2;
            if (ok) ok = new_of[c1] == new_of[c0] + 1 && (new_of[c0] & 1) == 1;
            if (!ok) {
#pragma omp critical(clpt_pack_err)
                if (bad_split < 0 || i < bad_split) bad_split = i;
            }
        }
        if (bad_split >= 0) {
            const kdnode &k = nodes[bad_split];
            snprintf(msg, sizeof msg, "split node %lld is malformed (children %d,%d axis %d)", bad_split,
                     k.split.children[0], k.split.children[1], k.split.axis);
            err = msg;
            return false;
        }
    }
    const int next = 1 + 2 * n_splits;
    const int n_packed = next;
    timer.lap("renumber");

    out.nodes.resize((size_t)n_packed);
    out.leaves.resize((size_t)n_leaves * 4);
    long long bad_node = -1;
    int bad_kind = 0;
    size_t fat_refs = 0;
#pragma omp parallel for schedule(static) reduction(+ : fat_refs)
    for (long long i = 0; i < (long long)n_nodes; i++) {
        const int ni = new_of[i];
        if (ni < 0) continue; // unreachable from the root
        const kdnode &k = nodes[i];
        if (k.type == KD_SPLIT) {
            out.nodes[ni].x = float_bits(k.split.value);
            out.nodes[ni].y = ((uint32_t)new_of[k.split.children[0]] << 2) | (uint32_t)k.split.axis;
            continue;
        }
        const int li = leaf_of[i];
        out.nodes[ni].x = (uint32_t)li;
        out.nodes[ni].y = 0x80000003u; // CLPT_LEAF_WORD
        const int first = k.leaf.tris, count = k.leaf.tri_count;
        bool bad = count < 0 || (count > 0 && (first < 0 || (size_t)first + (size_t)count > n_refs));
        if (count >= CLPT_COOP_LEAF_MIN) fat_refs += (size_t)count;
        ClptFloat4 *L = &out.leaves[(size_t)li * 4];
        L[0] = ClptFloat4{ k.min.s[0], k.min.s[1], k.min.s[2], as_float(count > 0 ? first : 0) };
        L[1] = ClptFloat4{ k.max.s[0], k.max.s[1], k.max.s[2], as_float(count) };
        int ropes[6];
        int kind = bad ? 1 : 0;
        for (int f = 0; f < 6; f++) {
            const int r = k.leaf.ropes[f];
            if (r == -1) {
                ropes[f] = -1;
            } else if (r < 0 || (size_t)r >= n_nodes || new_of[r] < 0) {
                ropes[f] = -1;
                kind = 2;
            } else if (nodes[r].type == KD_LEAF) {
                ropes[f] = -2 - leaf_of[r]; // straight to the leaf record: no node word to fetch
            } else {
                ropes[f] = new_of[r];
            }
        }
        L[2] = ClptFloat4{ as_float(ropes[0]), as_float(ropes[1]), as_float(ropes[2]), as_float(ropes[3]) };
        L[3] = ClptFloat4{ as_float(ropes[4]), as_float(ropes[5]), 0, 0 };
        if (kind) {
#pragma omp critical(clpt_pack_err)
            if (bad_node < 0 || i < bad_node) {
                bad_node = i;
                bad_kind = kind;
            }
        }
    }
    if (bad_node >= 0) {
        const kdnode &k = nodes[bad_node];
        if (bad_kind == 1)
            snprintf(msg, sizeof msg, "leaf node %lld references triangles [%d,+%d) of %zu", bad_node, k.leaf.tris,
                     k.leaf.tri_count, n_refs);
        else
            snprintf(msg, sizeof msg, "leaf node %lld has a rope that is out of range", bad_node);
        err = msg;
        return false;
    }

    timer.lap("nodes+leaves");
    // ---- pre-gather triangles in leaf order, edges precomputed ----
    out.tri.resize(n_refs * 3);
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long s = 0; s < (long long)n_refs; s++) {
        const int b = tri_indices[s];
        if (b < 0 || (size_t)b >= n_prims) {
            bad |= 1;
            continue;
        }
        const int i0 = corners[3 * (size_t)b].s[0], i1 = corners[3 * (size_t)b + 1].s[0],
                  i2 = corners[3 * (size_t)b + 2].s[0];
        if (i0 < 0 || i1 < 0 || i2 < 0 || (size_t)i0 >= n_verts || (size_t)i1 >= n_verts ||
            (size_t)i2 >= n_verts) {
            bad |= 2;
            continue;
        }
        const Vector4 &v0 = verts[i0], &v1 = verts[i1], &v2 = verts[i2];
        ClptFloat4 *T = &out.tri[(size_t)s * 3];
        T[0] = ClptFloat4{ v0.s[0], v0.s[1], v0.s[2], as_float(b) };
        // one fp32 subtraction each, the same rounding as `v1 - v0` in the kernel
        T[1] = ClptFloat4{ v1.s[0] - v0.s[0], v1.s[1] - v0.s[1], v1.s[2] - v0.s[2], 0 };
        T[2] = ClptFloat4{ v2.s[0] - v0.s[0], v2.s[1] - v0.s[1], v2.s[2] - v0.s[2], 0 };
    }
    if (bad) {
        err = (bad & 1) ? "tri_indices entry out of range" : "triangle corner references a missing vertex";
        return false;
    }
    timer.lap("triangles");
    // ---- flat shading normals, one per primitive ----
    // normalize(e1 x e2) with e1 = v1 - v0, e2 = v2 - v0: the expressions of the kernel's V3 helpers
    // (clpt_trace.cuh: vcross, vdot, vnormalize), one rounding per operation (-ffp-contract=off), so
    // the stored normal is bit for bit what the kernel used to compute at every hit.
    out.flat_n.resize(n_prims);
#pragma omp parallel for schedule(static)
    for (long long p = 0; p < (long long)n_prims; p++) {
        ClptFloat4 &N = out.flat_n[(size_t)p];
        N = ClptFloat4{ 0, 0, 0, corners[3 * (size_t)p].s[1] >= 0 ? 1.0f : 0.0f };
        const int i0 = corners[3 * (size_t)p].s[0], i1 = corners[3 * (size_t)p + 1].s[0],
                  i2 = corners[3 * (size_t)p + 2].s[0];
        if (i0 < 0 || i1 < 0 || i2 < 0 || (size_t)i0 >= n_verts || (size_t)i1 >= n_verts || (size_t)i2 >= n_verts) {
            continue; // (a primitive no leaf lists; the ones that are listed were checked above)
        }
        const Vector4 &v0 = verts[i0], &v1 = verts[i1], &v2 = verts[i2];
        const float ax = v1.s[0] - v0.s[0], ay = v1.s[1] - v0.s[1], az = v1.s[2] - v0.s[2];
        const float bx = v2.s[0] - v0.s[0], by = v2.s[1] - v0.s[1], bz = v2.s[2] - v0.s[2];
        const float m0 = ay * bz, m1 = az * by, m2 = az * bx, m3 = ax * bz, m4 = ax * by, m5 = ay * bx;
        const float cx = m0 - m1, cy = m2 - m3, cz = m4 - m5;
        const float q0 = cx * cx, q1 = cy * cy, q2 = cz * cz;
        const float s01 = q0 + q1, s012 = s01 + q2;
        const float len = sqrtf(s012);
        N.x = cx / len;
        N.y = cy / len;
        N.z = cz / len;
    }
    timer.lap("flat normals");
    // vertex-normal indices are dereferenced when shading.  Like the reference
    // (kernel.cl:349) only the FIRST corner decides whether normals are used, so
    // when it has one the other two must be valid as well.
    for (size_t p = 0; p < n_prims; p++) {
        if (corners[3 * p].s[1] < 0) continue;
        for (int c = 0; c < 3; c++) {
            const int vn = corners[3 * p + c].s[1];
            if (vn < 0 || (size_t)vn >= n_norms) {
                snprintf(msg, sizeof msg, "triangle %zu corner %d references normal %d of %zu", p, c, vn,
                         n_norms);
                err = msg;
                return false;
            }
        }
    }
    for (int a = 0; a < 3; a++) {
        out.root_min[a] = nodes[0].min.s[a];
        out.root_max[a] = nodes[0].max.s[a];
    }
    timer.lap("normals check");
    // ---- start-node table ----
    // For a point p the kernel's descent takes child[1] iff p[axis] > plane.  Every
    // point of a cell [lo, hi] takes the same branch at a split when hi <= plane
    // (all left) or lo > plane (all right); the walk below follows those forced
    // branches from the root and stops at the first split the cell straddles.  The
    // cell is enlarged by a margin that covers the fp32 rounding of the cell index
    // computed on the device, so starting a descent at the table entry reaches
    // exactly the leaf a descent from the root would.
    {
        double ext[3], vol = 1.0;
        for (int a = 0; a < 3; a++) {
            ext[a] = (double)out.root_max[a] - (double)out.root_min[a];
            if (!(ext[a] > 0)) ext[a] = 0;
            vol *= ext[a] > 0 ? ext[a] : 1.0;
        }
        // about one cell per two nodes, between 4K and 2M cells
        double target_cells = (double)n_nodes / 2;
        target_cells = n_nodes < 64 ? 1.0 : (target_cells < 4096.0 ? 4096.0 : (target_cells > 2097152.0 ? 2097152.0 : target_cells));
        const double cell = std::cbrt(vol / target_cells);
        size_t total = 1;
        for (int a = 0; a < 3; a++) {
            int d = ext[a] > 0 && cell > 0 ? (int)std::ceil(ext[a] / cell) : 1;
            d = d < 1 ? 1 : (d > 1024 ? 1024 : d);
            out.lut_dim[a] = d;
            out.lut_scale[a] = ext[a] > 0 ? (float)(d / ext[a]) : 0.0f;
            total *= (size_t)d;
        }
        out.lut.resize(total);
        const int gx = out.lut_dim[0], gy = out.lut_dim[1], gz = out.lut_dim[2];
#pragma omp parallel for schedule(static) collapse(2)
        for (int cz = 0; cz < gz; cz++) {
            for (int cy = 0; cy < gy; cy++) {
                for (int cx = 0; cx < gx; cx++) {
                    const int c[3] = { cx, cy, cz };
                    double lo[3], hi[3];
                    for (int a = 0; a < 3; a++) {
                        const double sc = out.lut_scale[a];
                        const double margin = 1e-5 * (1.0 + ext[a] + std::fabs((double)out.root_min[a]));
                        if (sc > 0) {
                            lo[a] = (double)out.root_min[a] + c[a] / sc - margin;
                            hi[a] = (double)out.root_min[a] + (c[a] + 1) / sc + margin;
                        } else {
                            lo[a] = -1e300;
                            hi[a] = 1e300;
                        }
                        // the first and last cells also receive everything beyond the box
                        if (c[a] == 0) lo[a] = -1e300;
                        if (c[a] == out.lut_dim[a] - 1) hi[a] = 1e300;
                    }
                    int o = 0;
                    while (nodes[o].type == KD_SPLIT) {
                        const int ax = nodes[o].split.axis;
                        const double plane = nodes[o].split.value;
                        if (hi[ax] <= plane) {
                            o = nodes[o].split.children[0];
                        } else if (lo[ax] > plane) {
                            o = nodes[o].split.children[1];
                        } else {
                            break;
                        }
                    }
                    out.lut[((size_t)cz * gy + cy) * gx + cx] = new_of[o];
                }
            }
        }
    }
    timer.lap("start table");
    out.n_nodes = n_packed;
    out.n_leaves = n_leaves;
    out.n_refs = (int)n_refs;
    out.n_prims = (int)n_prims;
    out.fat_refs = fat_refs;
    (void)as_int;
    return true;
}
