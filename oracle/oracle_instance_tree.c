/* oracle_instance_tree.c -- the instance tree in the CPU restatement.  TEST INFRASTRUCTURE, like
 * oracle_instances.c, which it includes unchanged: this file adds the CPU twin of the device's
 * tree builder (clpathtracer_b200/csrc/cuda/instance_tree.cu), the world query that walks a given
 * tree, and a copy of oracle_render_instanced's loop that calls it.
 *
 * Instance tree (EXTENSION; this is the definition the CUDA path equals bit for bit, and the
 * builder below produces the device's node bytes).  Everything the list does per instance stays
 * (oracle_instances.c header): object ray, root clip, skip rule, walk, shading, ids, material,
 * counters (one ray per world query, every walk summed; tree nodes are not counted).  New:
 *   world box   of instance k, in float64 (every operation rounded once, no contraction):
 *               A^-1 = adj(A) / det(A) entry by entry and t = -(A^-1 b); the 8 corners of the
 *               mesh's root box mapped by x -> A^-1 x + t, each row ((m0*x + m1*y) + m2*z) + t;
 *               their min and max; each side padded outward by
 *               pad = 2^-12 * largest extent + 2^-20 * largest |coordinate| and rounded outward to
 *               fp32 (clamped to +-FLT_MAX).  det == 0 or a non-finite corner or pad: +-FLT_MAX.
 *               The pad is far above fp32 rounding, so a ray whose object-space walk hits the
 *               mesh enters the world box, and enters it before the hit.
 *   keys        centroid_r = lo_r*0.5f + hi_r*0.5f (fp32); over the centroids' bounds [cl, ch],
 *               q_r = floor((c_r - cl_r) * (1024.0f / (ch_r - cl_r))) clamped to [0, 1023], NaN
 *               -> 0; morton30 = spread(q_x)*4 + spread(q_y)*2 + spread(q_z);
 *               key = morton30 << 20 | k, 50 bits and unique; sorted ascending.
 *   hierarchy   Karras (HPG 2012) over the sorted keys: n - 1 internal nodes, root 0, the split
 *               of a node at its range's highest differing key bit.  Each split consumes a bit,
 *               so the depth is at most 50.
 *   node        64 bytes: slot s = {min.xyz, ref}, {max.xyz, 0} at floats 8s..8s+7; ref >= 0 an
 *               internal node, ref < 0 instance -1 - ref.  A slot's box is its leaf's world box
 *               or the union of the child node's two slots.  n = 1: one node, slot 1 the empty
 *               box (+FLT_MAX, -FLT_MAX) with ref -1.
 *   walk        the world ray's box test is clip_root (acceptance tmax > 0, entry tmin).  At a
 *               node both slots are tested; a slot whose entry is beyond the current hit (a hit
 *               exists and entry > best) is not taken; the nearer entry goes first (slot 0 on
 *               equal entries), the other is pushed with its entry; a popped entry beyond the
 *               current hit is dropped.  At a leaf, the list's step for instance k, whose hit
 *               replaces the current one when t < best, or t == best and k > the current
 *               instance (the base scene is -1).
 *   consequence when no instance's hit lies within rounding of the entry of an instance's world
 *               box, the tree renders the list's frame bit for bit (a pruned subtree's entry is
 *               beyond the current hit, hence beyond the final hit, and every hit inside it lies
 *               beyond its padded entry); the counters differ, the tree walks fewer instances.
 * With tree == NULL, oracle_render_instance_tree is oracle_render_instanced.
 */
#include <float.h>

#include "oracle_instances.c"

/* ---------------------------------------------------------------- the builder's twin */
static double dmin_(double a, double b) { return b < a ? b : a; }
static double dmax_(double a, double b) { return b > a ? b : a; }
static float fmin_(float a, float b) { return b < a ? b : a; }
static float fmax_(float a, float b) { return b > a ? b : a; }
static float f_down(double x) { /* x rounded toward -inf */
    float f = (float)x;
    if ((double)f > x) f = nextafterf(f, -INFINITY);
    return f;
}
static float f_up(double x) {
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}

/* world box of the instance with world-to-object w over the object-space box [mn, mx] */
static void world_box(const float *w, const float *mn, const float *mx, float *blo, float *bhi) {
    double a[9], b[3], m[9], t[3], lo[3], hi[3];
    for (int r = 0; r < 3; r++) {
        a[3 * r] = w[4 * r];
        a[3 * r + 1] = w[4 * r + 1];
        a[3 * r + 2] = w[4 * r + 2];
        b[r] = w[4 * r + 3];
    }
    const double c00 = a[4] * a[8] - a[5] * a[7];
    const double c01 = a[5] * a[6] - a[3] * a[8];
    const double c02 = a[3] * a[7] - a[4] * a[6];
    const double det = (a[0] * c00 + a[1] * c01) + a[2] * c02;
    m[0] = c00 / det;
    m[1] = (a[2] * a[7] - a[1] * a[8]) / det;
    m[2] = (a[1] * a[5] - a[2] * a[4]) / det;
    m[3] = c01 / det;
    m[4] = (a[0] * a[8] - a[2] * a[6]) / det;
    m[5] = (a[2] * a[3] - a[0] * a[5]) / det;
    m[6] = c02 / det;
    m[7] = (a[1] * a[6] - a[0] * a[7]) / det;
    m[8] = (a[0] * a[4] - a[1] * a[3]) / det;
    for (int r = 0; r < 3; r++) t[r] = -((m[3 * r] * b[0] + m[3 * r + 1] * b[1]) + m[3 * r + 2] * b[2]);
    for (int c = 0; c < 8; c++) {
        const double x = (c & 1) ? mx[0] : mn[0], y = (c & 2) ? mx[1] : mn[1], z = (c & 4) ? mx[2] : mn[2];
        for (int r = 0; r < 3; r++) {
            const double v = ((m[3 * r] * x + m[3 * r + 1] * y) + m[3 * r + 2] * z) + t[r];
            lo[r] = c == 0 ? v : dmin_(lo[r], v);
            hi[r] = c == 0 ? v : dmax_(hi[r], v);
        }
    }
    double ext = 0.0, mag = 0.0;
    int finite = det != 0.0;
    for (int r = 0; r < 3; r++) {
        finite = finite && isfinite(lo[r]) && isfinite(hi[r]);
        ext = dmax_(ext, hi[r] - lo[r]);
        mag = dmax_(mag, dmax_(fabs(lo[r]), fabs(hi[r])));
    }
    const double pad = ext * 0x1p-12 + mag * 0x1p-20;
    for (int r = 0; r < 3; r++) {
        if (finite && isfinite(pad)) {
            blo[r] = fmax_(f_down(lo[r] - pad), -FLT_MAX);
            bhi[r] = fmin_(f_up(hi[r] + pad), FLT_MAX);
        } else {
            blo[r] = -FLT_MAX;
            bhi[r] = FLT_MAX;
        }
    }
}

static uint32_t order_key(float f) { /* fp32 -> unsigned of the same order (the device's atomics) */
    uint32_t u;
    memcpy(&u, &f, 4);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
static uint32_t expand10(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
static uint32_t quantise(float c, float lo, float hi) {
    const float s = 1024.0f / (hi - lo);
    const float f = floorf((c - lo) * s);
    return f >= 0.0f ? (f < 1023.0f ? (uint32_t)f : 1023u) : 0u;
}
static int cmp_u64(const void *a, const void *b) {
    const uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : (x > y ? 1 : 0);
}
static int delta(const uint64_t *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    return __builtin_clzll(keys[i] ^ keys[j]);
}
static void put_slot(float *nodes, int node, int slot, const float *lo, const float *hi, int32_t ref) {
    float *s = nodes + 16 * node + 8 * slot;
    s[0] = lo[0], s[1] = lo[1], s[2] = lo[2];
    memcpy(s + 3, &ref, 4);
    s[4] = hi[0], s[5] = hi[1], s[6] = hi[2], s[7] = 0.0f;
}

/* The tree over n >= 1 instances: w2o float[n][12], root boxes float[n][6] (min xyz, max xyz);
 * nodes receives max(n - 1, 1) * 16 floats.  0 on success. */
int oracle_build_instance_tree(const float *w2o, const float *root, int32_t n, float *nodes) {
    if (n < 1 || n > (1 << 20)) return 1;
    float *box = malloc((size_t)n * 6 * sizeof(float));
    uint64_t *keys = malloc((size_t)n * sizeof(uint64_t));
    int *up_leaf = malloc((size_t)n * sizeof(int)), *up_node = malloc((size_t)n * sizeof(int));
    int *arrivals = calloc((size_t)n, sizeof(int));
    uint32_t kmin[3] = { 0xffffffffu, 0xffffffffu, 0xffffffffu }, kmax[3] = { 0, 0, 0 };
    float cl[3], ch[3];
    for (int k = 0; k < n; k++) {
        world_box(w2o + 12 * (size_t)k, root + 6 * (size_t)k, root + 6 * (size_t)k + 3, box + 6 * (size_t)k,
                  box + 6 * (size_t)k + 3);
        for (int r = 0; r < 3; r++) {
            const float c = box[6 * (size_t)k + r] * 0.5f + box[6 * (size_t)k + 3 + r] * 0.5f;
            const uint32_t q = order_key(c);
            if (q < kmin[r]) kmin[r] = q, cl[r] = c;
            if (q > kmax[r]) kmax[r] = q, ch[r] = c;
        }
    }
    for (int k = 0; k < n; k++) {
        uint32_t q[3];
        for (int r = 0; r < 3; r++)
            q[r] = quantise(box[6 * (size_t)k + r] * 0.5f + box[6 * (size_t)k + 3 + r] * 0.5f, cl[r], ch[r]);
        const uint32_t morton = expand10(q[0]) * 4u + expand10(q[1]) * 2u + expand10(q[2]);
        keys[k] = ((uint64_t)morton << 20) | (uint64_t)k;
    }
    qsort(keys, (size_t)n, sizeof(uint64_t), cmp_u64);
    if (n == 1) {
        const float elo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, ehi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
        up_leaf[0] = 0;
        put_slot(nodes, 0, 1, elo, ehi, -1);
    }
    for (int i = 0; i < n - 1; i++) {
        const int d = delta(keys, n, i, i + 1) > delta(keys, n, i, i - 1) ? 1 : -1;
        const int dmin = delta(keys, n, i, i - d);
        int lmax = 2;
        while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
        int l = 0;
        for (int t = lmax >> 1; t >= 1; t >>= 1)
            if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
        const int j = i + l * d;
        const int dnode = delta(keys, n, i, j);
        int s = 0;
        for (int div = 2;; div <<= 1) {
            const int t = (l + div - 1) / div;
            if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
            if (t == 1) break;
        }
        const int gamma = i + s * d + (d < 0 ? d : 0);
        if ((i < j ? i : j) == gamma) up_leaf[gamma] = i << 1;
        else up_node[gamma] = i << 1;
        if ((i > j ? i : j) == gamma + 1) up_leaf[gamma + 1] = (i << 1) | 1;
        else up_node[gamma + 1] = (i << 1) | 1;
    }
    /* bottom-up: the second arrival at a node carries the union of its slots to the node's parent */
    for (int p = 0; p < n; p++) {
        const int k = (int)(keys[p] & 0xFFFFFu);
        float lo[3], hi[3];
        memcpy(lo, box + 6 * (size_t)k, sizeof lo);
        memcpy(hi, box + 6 * (size_t)k + 3, sizeof hi);
        int ref = -1 - k, up = up_leaf[p];
        for (;;) {
            const int node = up >> 1;
            put_slot(nodes, node, up & 1, lo, hi, ref);
            if (node == 0 || arrivals[node]++ == 0) break;
            const float *N = nodes + 16 * node;
            for (int r = 0; r < 3; r++) {
                lo[r] = fmin_(N[r], N[8 + r]);
                hi[r] = fmax_(N[4 + r], N[12 + r]);
            }
            ref = node;
            up = up_node[node];
        }
    }
    free(box), free(keys), free(up_leaf), free(up_node), free(arrivals);
    return 0;
}

/* ---------------------------------------------------------------- the walk */
static int32_t ref_of(float f) {
    int32_t r;
    memcpy(&r, &f, 4);
    return r;
}

/* One world query: the base scene, then the instances the tree leads to (header).  tree == NULL:
 * world_hit, the list. */
static hit_t world_hit_tree(const oracle_params *P, const oracle_instance *I, int n, const float *tree,
                            const ray_t *r, uint64_t *cnt, int *inst) {
    if (!tree) return world_hit(P, I, n, r, cnt, inst);
    cnt[0]++;
    hit_t h = walk(P, r, cnt);
    *inst = -1;
    const i4 *tris = P->tris;
    const f4 *norms = P->norms;
    int local = h.prim;
    int stack_ref[64];
    float stack_entry[64];
    int sp = 0, ref = 0;
    while (n > 0) {
        if (ref >= 0) {
            const float *N = tree + 16 * (size_t)ref;
            const f3 b0[2] = { v3(N[0], N[1], N[2]), v3(N[4], N[5], N[6]) };
            const f3 b1[2] = { v3(N[8], N[9], N[10]), v3(N[12], N[13], N[14]) };
            float e0, e1, tmax;
            const int in0 = clip_root(b0, r, &e0, &tmax) && !(h.did_hit && e0 > h.t);
            const int in1 = clip_root(b1, r, &e1, &tmax) && !(h.did_hit && e1 > h.t);
            if (in0 && in1) {
                const int first1 = e1 < e0;
                stack_ref[sp] = ref_of(first1 ? N[3] : N[11]);
                stack_entry[sp++] = first1 ? e0 : e1;
                ref = ref_of(first1 ? N[11] : N[3]);
                continue;
            }
            if (in0 || in1) {
                ref = ref_of(in0 ? N[3] : N[11]);
                continue;
            }
        } else {
            /* the list's step for instance k (world_hit's loop body), with the tree's replace rule */
            const int k = -1 - ref;
            const float *m = I[k].w2o;
            const f3 o = r->orig, d = r->dir;
            const f3 lo = v3(((m[0] * o.x + m[1] * o.y) + m[2] * o.z) + m[3],
                             ((m[4] * o.x + m[5] * o.y) + m[6] * o.z) + m[7],
                             ((m[8] * o.x + m[9] * o.y) + m[10] * o.z) + m[11]);
            const f3 ld = v3((m[0] * d.x + m[1] * d.y) + m[2] * d.z, (m[4] * d.x + m[5] * d.y) + m[6] * d.z,
                             (m[8] * d.x + m[9] * d.y) + m[10] * d.z);
            const ray_t lr = make_ray(lo, ld);
            const f3 rb[2] = { xyz(I[k].nodes[0].min), xyz(I[k].nodes[0].max) };
            float tmin, tmax;
            if (clip_root(rb, &lr, &tmin, &tmax) && !(h.did_hit && tmin > h.t)) {
                oracle_params Q = *P;
                Q.nodes = I[k].nodes;
                Q.tri_indices = I[k].tri_indices;
                Q.tris = I[k].tris;
                Q.verts = I[k].verts;
                Q.norms = I[k].norms;
                hit_t hi = walk(&Q, &lr, cnt);
                if (hi.did_hit && (!h.did_hit || hi.t < h.t || (hi.t == h.t && k > *inst))) {
                    const int b = hi.prim;
                    const i4 c1 = I[k].tris[3 * b + 0], c2 = I[k].tris[3 * b + 1], c3 = I[k].tris[3 * b + 2];
                    f3 mn;
                    if (c1.s[1] >= 0) {
                        const f3 n1 = xyz(I[k].norms[c1.s[1]]), n2 = xyz(I[k].norms[c2.s[1]]),
                                 n3 = xyz(I[k].norms[c3.s[1]]);
                        const float w = 1.0f - hi.u - hi.v;
                        mn = add3(add3(scale3(n1, w), scale3(n2, hi.u)), scale3(n3, hi.v));
                    } else {
                        const f3 v1 = xyz(I[k].verts[c1.s[0]]), v2 = xyz(I[k].verts[c2.s[0]]),
                                 v3_ = xyz(I[k].verts[c3.s[0]]);
                        mn = cross3(sub3(v2, v1), sub3(v3_, v1));
                    }
                    hi.normal = normalize3(v3((m[0] * mn.x + m[4] * mn.y) + m[8] * mn.z,
                                              (m[1] * mn.x + m[5] * mn.y) + m[9] * mn.z,
                                              (m[2] * mn.x + m[6] * mn.y) + m[10] * mn.z));
                    hi.prim = b + I[k].prim_offset;
                    h = hi;
                    *inst = k;
                    tris = I[k].tris;
                    norms = I[k].norms;
                    local = b;
                }
            }
        }
        int found = 0;
        while (sp > 0) {
            sp--;
            if (h.did_hit && stack_entry[sp] > h.t) continue;
            ref = stack_ref[sp];
            found = 1;
            break;
        }
        if (!found) break;
    }
    if (h.did_hit && norms != NULL && tris[3 * local].s[1] >= 0) cnt[4]++;
    return h;
}

/* shade_sample_instanced with world_hit_tree (its copy, the query replaced) */
static f3 shade_sample_tree(const oracle_params *P, const oracle_instance *I, int n, const float *tree, ray_t r,
                            uint32_t pixel, uint32_t sample, hit_t *first, float *edge, uint64_t *cnt) {
    int depth = P->depth;
    int inst;
    if (P->mode == 0) depth = depth > 0 ? 1 : 0;
    if (P->mode == 2) {
        f3 L = v3(0, 0, 0), T = v3(1, 1, 1);
        for (int seg = 0; seg < depth; seg++) {
            hit_t h = world_hit_tree(P, I, n, tree, &r, cnt, &inst);
            if (seg == 0 && first) *first = h;
            note_edge(edge, &h);
            if (!h.did_hit) { L = add3(L, T); return L; }
            int m = inst >= 0 ? I[inst].material : (P->tri_material ? P->tri_material[h.prim] : 0);
            if (m < 0 || m >= P->n_materials) m = 0;
            oracle_material mat;
            if (P->n_materials > 0) mat = P->materials[m];
            else { mat.albedo[0] = mat.albedo[1] = mat.albedo[2] = 0.5f; mat.kind = 0;
                   mat.emission[0] = mat.emission[1] = mat.emission[2] = 0; }
            L = add3(L, v3(T.x * mat.emission[0], T.y * mat.emission[1], T.z * mat.emission[2]));
            T = v3(T.x * mat.albedo[0], T.y * mat.albedo[1], T.z * mat.albedo[2]);
            f3 hitp = add3(r.orig, scale3(r.dir, h.t));
            f3 nd;
            if (mat.kind == 1) {
                nd = normalize3(sub3(r.dir, scale3(h.normal, 2 * dot3(r.dir, h.normal))));
            } else {
                nd = cosine_dir(h.normal, pixel, sample, (uint32_t)seg, P->seed);
            }
            hitp = add3(hitp, scale3(nd, 0.0001f));
            r = make_ray(hitp, nd);
        }
        return L;
    }
    f3 col = v3(0, 0, 0);
    float str = 1.0f;
    for (; depth > 0; depth--) {
        hit_t h = world_hit_tree(P, I, n, tree, &r, cnt, &inst);
        if (first) { *first = h; first = NULL; }
        note_edge(edge, &h);
        if (!h.did_hit) break;
        f3 nc = v3((h.normal.x + 1) / 2, (h.normal.y + 1) / 2, (h.normal.z + 1) / 2);
        if (P->mode == 0) return nc;
        f3 no = add3(r.orig, scale3(r.dir, h.t));
        f3 nd = normalize3(sub3(r.dir, scale3(h.normal, 2 * dot3(r.dir, h.normal))));
        no = add3(no, scale3(nd, 0.0001f));
        col = add3(scale3(col, 1 - str), scale3(nc, str));
        str *= 0.2f;
        r = make_ray(no, nd);
    }
    return v3((1 - str) * col.x + str, (1 - str) * col.y + str, (1 - str) * col.z + str);
}

/* oracle_render_instanced's loop (its copy), with shade_sample_tree */
int oracle_render_instance_tree(oracle_params *P, const oracle_instance *I, int32_t n_instances, const float *tree) {
    const int W = P->width, H = P->height;
    if ((P->flags & ORACLE_ACCUMULATE) && (!P->accum || !P->rgba)) return 1;
    const float *M = P->cam;
    int spp = P->spp < 1 ? 1 : P->spp;
    int jitter = (P->flags & ORACLE_JITTER) != 0;
    uint64_t total[6] = { 0, 0, 0, 0, 0, 0 };
#ifdef _OPENMP
    if (P->threads > 0) omp_set_num_threads(P->threads);
#endif
#pragma omp parallel
    {
        uint64_t cnt[6] = { 0, 0, 0, 0, 0, 0 };
#pragma omp for schedule(dynamic, 1) nowait
        for (int y = P->y0; y < P->y1; y++) {
            for (int x = 0; x < W; x++) {
                uint32_t pixel = (uint32_t)(y * W + x);
                f3 origin = v3(M[2] / M[14], M[6] / M[14], M[10] / M[14]);
                f3 acc = v3(0, 0, 0);
                uint64_t fsum[3] = { 0, 0, 0 };
                hit_t first;
                float edge = 2.0f;
                memset(&first, 0, sizeof(first));
                first.prim = -1;
                for (int s = 0; s < spp; s++) {
                    uint32_t sample = P->sample_base + (uint32_t)s;
                    float fx = (float)(uint32_t)x - (float)(uint32_t)W / 2;
                    float fy = (float)(uint32_t)y - (float)(uint32_t)H / 2;
                    if (jitter) {
                        uint32_t c[4] = { pixel, sample, 0, 0 };
                        philox4x32_10(c, P->seed, ORACLE_KEY1);
                        fx = fx + (u01(c[0]) - 0.5f);
                        fy = fy + (u01(c[1]) - 0.5f);
                    }
                    f3 ncp = unproject(M, v3(fx, fy, -1));
                    f3 fcp = unproject(M, v3(fx, fy, 1));
                    f3 dir = normalize3(sub3(fcp, ncp));
                    ray_t r = make_ray(origin, dir);
                    f3 c = shade_sample_tree(P, I, n_instances, tree, r, pixel, sample, s == 0 ? &first : NULL,
                                             s == 0 ? &edge : NULL, cnt);
                    acc = add3(acc, c);
                    fsum[0] += fix32(c.x);
                    fsum[1] += fix32(c.y);
                    fsum[2] += fix32(c.z);
                }
                size_t o = (size_t)y * (size_t)W + (size_t)x;
                if (P->rgba) {
                    float *px = P->rgba + 4 * o;
                    if (P->flags & ORACLE_ACCUMULATE) {
                        uint64_t *a = P->accum + 4 * o;
                        a[0] += fsum[0]; a[1] += fsum[1]; a[2] += fsum[2]; a[3] += (uint64_t)spp;
                        const double k = (double)a[3] * 4294967296.0;
                        px[0] = (float)((double)a[0] / k); px[1] = (float)((double)a[1] / k);
                        px[2] = (float)((double)a[2] / k); px[3] = 1.0f;
                    } else if (spp == 1) {
                        px[0] = acc.x; px[1] = acc.y; px[2] = acc.z; px[3] = 1.0f;
                    } else {
                        float inv = 1.0f / (float)spp;
                        px[0] = acc.x * inv; px[1] = acc.y * inv; px[2] = acc.z * inv; px[3] = 1.0f;
                    }
                }
                if (P->prim_id) P->prim_id[o] = first.did_hit ? first.prim : -1;
                if (P->t_hit) P->t_hit[o] = first.did_hit ? first.t : 0.0f;
                if (P->uv) { P->uv[2 * o] = first.u; P->uv[2 * o + 1] = first.v; }
                if (P->path_edge) P->path_edge[o] = edge;
                if (P->normal) {
                    P->normal[3 * o] = first.normal.x;
                    P->normal[3 * o + 1] = first.normal.y;
                    P->normal[3 * o + 2] = first.normal.z;
                }
            }
        }
#pragma omp critical
        for (int k = 0; k < 6; k++) total[k] += cnt[k];
    }
    for (int k = 0; k < 6; k++) P->counters[k] = total[k];
    return 0;
}

