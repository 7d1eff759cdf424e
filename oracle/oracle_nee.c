/* oracle_nee.c -- light sampling (mode 3) in the CPU restatement.  TEST INFRASTRUCTURE, like
 * oracle_instance_tree.c, which it includes unchanged: this file adds the CPU twin of the device's
 * emitter table (clpathtracer_b200/csrc/cuda/emitters.cu), the occlusion query over the base scene
 * and the instances, and the mode-3 render loop for no instances, the list and the tree.
 *
 * Mode 3, CLPT_MODE_PATH_NEE (EXTENSION; this is the definition the CUDA path equals bit for bit,
 * and the builder below produces the device's table bytes).  Everything mode 2 does stays: the
 * world query, shading normal, materials (tri_material clamped to [0, n_materials), instances take
 * their own), emission added as throughput * emission, throughput *= albedo, mirror reflection,
 * cosine_dir for diffuse vertices with Philox counter (pixel, sample, 1 + segment, 0/1), the 1e-4
 * start offset along the new direction, the miss colour (throughput * white) and `depth` segments.
 * New:
 *   emitters    the base-scene primitives listed by at least one leaf whose material has a
 *               nonzero emission component, in ascending primitive id.  Instance triangles are
 *               never light-sampled.  Geometry: v0, e1 = v1 - v0, e2 = v2 - v0 (fp32, the hit
 *               test's operands) and the flat normal nl = normalize(e1 x e2).
 *   weights     in float64, one rounding per operation: area = 0.5 * sqrt(c.c), c = e1 x e2;
 *               esum = (e_r + e_g) + e_b; w = area * esum, or 0 unless w > 0 and finite;
 *               q = (uint64)(w / wmax * 2^32) (0 when wmax = 0), wmax the largest w.
 *   table       record i, 64 bytes: {v0, prim bits}, {e1, pa}, {e2, 0}, {nl, 0} with
 *               pa = (float)(((double)q / Q) / area) (0 when q = 0), the emitter's area pdf;
 *               cdf[i] = q_0 + ... + q_{i-1} (uint64, exact in any order), Q = the sum of all q;
 *               map[prim] = i, -1 for a primitive that is not an emitter; header {n, Q}.
 *   selection   at a diffuse vertex of segment s with s + 1 < depth and Q > 0: Philox counter
 *               (pixel, sample, 1 + s, 2) -> words r0..r2; target = (r0 * Q) >> 32 (128-bit
 *               product); i = the largest index with cdf[i] <= target (q_i > 0 follows).
 *   point       su = sqrt(u01(r1)), u2 = u01(r2); y = (v0 + e1 * (su * (1 - u2))) + e2 * (su * u2).
 *   NEE         L = y - x (x the hit point o + t d), d2 = L.L, dist = sqrt(d2), l = L / dist
 *               (three divisions); cx = l.n (n the shading normal), det = e1.(l x e2),
 *               cl = -(l.nl); nothing unless cx > 0, det > 0 and cl > 0.  Shadow ray: origin
 *               x + l * 1e-4, direction l, t_max = (dist - 1e-4) * (1 - 2^-12).  Visible ->
 *               pb = cx * PB, pl = (pa * d2) / cl, r = pb / pl, k = r / (1 + r * r), and the
 *               vertex adds (T.c * emission_c) * k per channel, T the throughput after the
 *               albedo; emission is the emitter primitive's material's.
 *               PB = (1 - p) / pi in fp32 = 0x1.45420cp-2, p = 0.0021209640721610596 the chance
 *               that all four disk tries are rejected.  k = pb/pl * pl^2/(pl^2 + pb^2): the NEE
 *               estimate times (1 - p) times the power heuristic's weight.
 *   BSDF hits   an emitter hit at segment s + 1 whose bounce at s was diffuse and did not fall
 *               back to the normal (cosine_dir_flag), on a base-scene primitive with
 *               map[prim] >= 0, adds (T.c * emission_c) * w with pb = (d.n) * PB of that bounce,
 *               cl = -(d.nl), pl = (pa * (t * t)) / cl, q = pl / pb and w = 1 / (1 + q * q);
 *               w = 1 when pa or cl is not > 0.  Every other emitter hit (camera ray, after a
 *               mirror, after the fallback, an instance) keeps w = 1 -- so with no emitters
 *               (Q = 0 and no MIS) mode 3 is mode 2 bit for bit.
 *   occlusion   visible when no triangle is accepted with 0 < t < t_max: back-face culled hit
 *               test; the base scene, then the instances (list order, or the instance tree with
 *               child 0 first and child 1 deferred).  A tree is entered when its root clip
 *               passes with entry <= t_max; a walk ends without a hit at a leaf whose entry
 *               exceeds t_max or when it leaves the tree, ends occluded after the first leaf
 *               that accepted a triangle (its whole run is tested) and counts as occluded when
 *               it uses up the rope-hop budget.  Visibility is an OR over triangles, so neither
 *               the order of the walk nor the traversal (list or tree) changes it.
 *   counters    one ray per shadow ray; its splits, leaves, tests and capped walks are summed.
 */
#include "oracle_instance_tree.c"

#define NEE_PB 0x1.45420cp-2f
#define NEE_TMAX_SCALE 0x1.ffep-1f

typedef struct oracle_emitters {
    const float *rec;       /* 16 floats per emitter */
    const uint64_t *cdf;    /* n + 1 entries, cdf[n] = Q */
    const int32_t *map;     /* per base primitive */
    uint64_t n, Q;
} oracle_emitters;

/* ---------------------------------------------------------------- the table's twin */
static int material_of(const oracle_params *P, int prim) {
    int m = P->tri_material ? P->tri_material[prim] : 0;
    if (m < 0 || m >= P->n_materials) m = 0;
    return m;
}

/* The emitter table of the scene in P (n_nodes wire nodes, n_prims primitives): rec float[16 *
 * n_prims], cdf uint64[n_prims + 1], map int32[n_prims], hdr uint64[2] = {n, Q}.  0 on success. */
int oracle_build_emitters(const oracle_params *P, int32_t n_nodes, int32_t n_prims, float *rec, uint64_t *cdf,
                          int32_t *map, uint64_t *hdr) {
    char *listed = calloc((size_t)n_prims + 1, 1);
    double *area = malloc(((size_t)n_prims + 1) * sizeof(double)), *w = malloc(((size_t)n_prims + 1) * sizeof(double));
    int32_t *ids = malloc(((size_t)n_prims + 1) * sizeof(int32_t));
    for (int i = 0; i < n_nodes; i++) {
        const onode *nd = &P->nodes[i];
        if (nd->type != 1 || nd->leaf.tris == -1) continue;
        for (int k = 0; k < nd->leaf.tri_count; k++) listed[P->tri_indices[nd->leaf.tris + k]] = 1;
    }
    uint64_t n = 0;
    for (int p = 0; p < n_prims; p++) {
        map[p] = -1;
        if (!listed[p] || P->n_materials <= 0) continue;
        const oracle_material *M = &P->materials[material_of(P, p)];
        if (M->emission[0] != 0.0f || M->emission[1] != 0.0f || M->emission[2] != 0.0f) ids[n++] = p;
    }
    double wmax = 0.0;
    for (uint64_t i = 0; i < n; i++) {
        const int p = ids[i];
        const i4 c1 = P->tris[3 * p], c2 = P->tris[3 * p + 1], c3 = P->tris[3 * p + 2];
        const f3 v0 = xyz(P->verts[c1.s[0]]), e1 = sub3(xyz(P->verts[c2.s[0]]), v0), e2 = sub3(xyz(P->verts[c3.s[0]]), v0);
        const f3 nl = normalize3(cross3(e1, e2));
        const double ax = e1.x, ay = e1.y, az = e1.z, bx = e2.x, by = e2.y, bz = e2.z;
        const double cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
        area[i] = 0.5 * sqrt((cx * cx + cy * cy) + cz * cz);
        const float *em = P->materials[material_of(P, p)].emission;
        const double ww = area[i] * (((double)em[0] + (double)em[1]) + (double)em[2]);
        w[i] = (ww > 0.0 && ww < INFINITY) ? ww : 0.0;
        if (w[i] > wmax) wmax = w[i];
        float *R = rec + 16 * i;
        R[0] = v0.x, R[1] = v0.y, R[2] = v0.z, memcpy(R + 3, &p, 4);
        R[4] = e1.x, R[5] = e1.y, R[6] = e1.z;
        R[8] = e2.x, R[9] = e2.y, R[10] = e2.z, R[11] = 0.0f;
        R[12] = nl.x, R[13] = nl.y, R[14] = nl.z, R[15] = 0.0f;
        map[p] = (int32_t)i;
    }
    uint64_t Q = 0;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t q = wmax > 0.0 ? (uint64_t)(w[i] / wmax * 4294967296.0) : 0;
        cdf[i] = Q;
        Q += q;
        w[i] = (double)q; /* (w is not needed again) */
    }
    cdf[n] = Q;
    for (uint64_t i = 0; i < n; i++) rec[16 * i + 7] = w[i] > 0.0 ? (float)(w[i] / (double)Q / area[i]) : 0.0f;
    hdr[0] = n;
    hdr[1] = Q;
    free(listed), free(area), free(w), free(ids);
    return 0;
}

/* ---------------------------------------------------------------- occlusion */
/* Any-hit walk of one tree (the base scene's or an instance mesh's, in P) with ray r. */
static int any_hit(const oracle_params *P, const ray_t *r, float t_max, uint64_t *cnt) {
    const onode *kd = P->nodes;
    const f3 rb[2] = { xyz(kd[0].min), xyz(kd[0].max) };
    float tmin, tmax;
    if (!clip_root(rb, r, &tmin, &tmax) || tmin > t_max) return 0;
    f3 p1 = r->orig;
    if (tmin > 0) p1 = add3(p1, scale3(r->dir, tmin));
    int index = 0, visits = 0;
    for (;;) {
        while (kd[index].type == 0) {
            index = kd[index].split.children[comp(p1, kd[index].split.axis) > kd[index].split.value];
            cnt[1]++;
        }
        cnt[2]++;
        const onode *leaf = &kd[index];
        const f3 lb[2] = { xyz(leaf->min), xyz(leaf->max) };
        int far;
        leaf_exit(lb, r, &tmin, &tmax, &far);
        if (tmin > t_max) return 0;
        int hit = 0;
        if (leaf->leaf.tris != -1) {
            for (int i = 0; i < leaf->leaf.tri_count; i++) {
                const int b = P->tri_indices[leaf->leaf.tris + i];
                const i4 c1 = P->tris[3 * b + 0], c2 = P->tris[3 * b + 1], c3 = P->tris[3 * b + 2];
                float t = 0, u = 0, v = 0;
                cnt[3]++;
                if (hit_tri(xyz(P->verts[c1.s[0]]), xyz(P->verts[c2.s[0]]), xyz(P->verts[c3.s[0]]), r->orig, r->dir,
                            &t, &u, &v) && t < t_max)
                    hit = 1;
            }
        }
        if (hit) return 1;
        index = leaf->leaf.ropes[far];
        p1 = add3(r->orig, scale3(r->dir, tmax));
        if (index == -1) return 0;
        if (++visits >= P->max_leaf_visits) { cnt[5]++; return 1; }
    }
}

/* any_hit in instance k's mesh with the world ray mapped to object space */
static int any_hit_instance(const oracle_params *P, const oracle_instance *I, int k, const ray_t *r, float t_max,
                            uint64_t *cnt) {
    const float *m = I[k].w2o;
    const f3 o = r->orig, d = r->dir;
    const f3 lo = v3(((m[0] * o.x + m[1] * o.y) + m[2] * o.z) + m[3], ((m[4] * o.x + m[5] * o.y) + m[6] * o.z) + m[7],
                     ((m[8] * o.x + m[9] * o.y) + m[10] * o.z) + m[11]);
    const f3 ld = v3((m[0] * d.x + m[1] * d.y) + m[2] * d.z, (m[4] * d.x + m[5] * d.y) + m[6] * d.z,
                     (m[8] * d.x + m[9] * d.y) + m[10] * d.z);
    const ray_t lr = make_ray(lo, ld);
    oracle_params Q = *P;
    Q.nodes = I[k].nodes;
    Q.tri_indices = I[k].tri_indices;
    Q.tris = I[k].tris;
    Q.verts = I[k].verts;
    Q.norms = I[k].norms;
    return any_hit(&Q, &lr, t_max, cnt);
}

/* The shadow ray's query: 1 when occluded.  tree == NULL: the instance list. */
static int occluded(const oracle_params *P, const oracle_instance *I, int n, const float *tree, const ray_t *r,
                    float t_max, uint64_t *cnt) {
    cnt[0]++;
    if (any_hit(P, r, t_max, cnt)) return 1;
    if (!tree) {
        for (int k = 0; k < n; k++)
            if (any_hit_instance(P, I, k, r, t_max, cnt)) return 1;
        return 0;
    }
    int stack[64], sp = 0, ref = 0;
    while (n > 0) {
        if (ref >= 0) {
            const float *N = tree + 16 * (size_t)ref;
            const f3 b0[2] = { v3(N[0], N[1], N[2]), v3(N[4], N[5], N[6]) };
            const f3 b1[2] = { v3(N[8], N[9], N[10]), v3(N[12], N[13], N[14]) };
            float e0, e1, tmax;
            const int in0 = clip_root(b0, r, &e0, &tmax) && !(e0 > t_max);
            const int in1 = clip_root(b1, r, &e1, &tmax) && !(e1 > t_max);
            if (in0 && in1) {
                stack[sp++] = ref_of(N[11]);
                ref = ref_of(N[3]);
                continue;
            }
            if (in0 || in1) {
                ref = ref_of(in0 ? N[3] : N[11]);
                continue;
            }
        } else if (any_hit_instance(P, I, -1 - ref, r, t_max, cnt)) {
            return 1;
        }
        if (sp == 0) break;
        ref = stack[--sp];
    }
    return 0;
}

/* ---------------------------------------------------------------- mode 3 */
/* oracle_kernel.c's cosine_dir, also saying whether all four disk tries were rejected */
static f3 cosine_dir_flag(f3 n, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t seed, int *fell_back) {
    float a = 0, b = 0;
    *fell_back = 1;
    for (uint32_t blk = 0; blk < 2 && *fell_back; blk++) {
        uint32_t c[4] = { pixel, sample, 1u + bounce, blk };
        philox4x32_10(c, seed, ORACLE_KEY1);
        for (int k = 0; k < 2 && *fell_back; k++) {
            float x = 2 * u01(c[2 * k]) - 1, y = 2 * u01(c[2 * k + 1]) - 1;
            if (x * x + y * y <= 1) { a = x; b = y; *fell_back = 0; }
        }
    }
    float zz = 1 - a * a - b * b;
    float z = sqrtf(zz > 0 ? zz : 0);
    float sg = n.z >= 0 ? 1.0f : -1.0f;
    float p = -1 / (sg + n.z);
    float q = n.x * n.y * p;
    f3 t1 = v3(1 + sg * n.x * n.x * p, sg * q, -sg * n.x);
    f3 t2 = v3(q, sg + n.y * n.y * p, -n.y);
    f3 d = add3(add3(scale3(t1, a), scale3(t2, b)), scale3(n, z));
    return normalize3(d);
}

/* The emitter a 32-bit word selects: target = (word * Q) >> 32, the largest i with cdf[i] <= target
 * (n >= 1, Q > 0; q_i > 0 follows). */
uint64_t oracle_select_emitter(const uint64_t *cdf, uint64_t n, uint64_t Q, uint32_t word) {
    const uint64_t target = (uint64_t)(((unsigned __int128)word * Q) >> 32);
    uint64_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) / 2;
        if (cdf[mid] <= target) lo = mid;
        else hi = mid;
    }
    return lo;
}

/* the light sample of a diffuse vertex at x with shading normal nrm and throughput T */
static f3 nee(const oracle_params *P, const oracle_instance *I, int n, const float *tree, const oracle_emitters *E,
              f3 x, f3 nrm, f3 T, uint32_t pixel, uint32_t sample, uint32_t seg, uint64_t *cnt) {
    uint32_t c[4] = { pixel, sample, 1u + seg, 2 };
    philox4x32_10(c, P->seed, ORACLE_KEY1);
    const float *R = E->rec + 16 * oracle_select_emitter(E->cdf, E->n, E->Q, c[0]);
    const f3 v0 = v3(R[0], R[1], R[2]), e1 = v3(R[4], R[5], R[6]), e2 = v3(R[8], R[9], R[10]);
    const f3 nl = v3(R[12], R[13], R[14]);
    const float su = sqrtf(u01(c[1])), u2 = u01(c[2]);
    const f3 y = add3(add3(v0, scale3(e1, su * (1 - u2))), scale3(e2, su * u2));
    const f3 L = sub3(y, x);
    const float d2 = dot3(L, L), dist = sqrtf(d2);
    const f3 l = v3(L.x / dist, L.y / dist, L.z / dist);
    const float cx = dot3(l, nrm);
    const float det = dot3(e1, cross3(l, e2));
    const float cl = -dot3(l, nl);
    const f3 none = v3(0, 0, 0);
    if (!(cx > 0) || !(det > 0) || !(cl > 0)) return none;
    const ray_t sr = make_ray(add3(x, scale3(l, 0.0001f)), l);
    if (occluded(P, I, n, tree, &sr, (dist - 0.0001f) * NEE_TMAX_SCALE, cnt)) return none;
    int prim;
    memcpy(&prim, R + 3, 4);
    const float *em = P->materials[material_of(P, prim)].emission;
    const float pb = cx * NEE_PB, pl = R[7] * d2 / cl;
    const float r = pb / pl, k = r / (1 + r * r);
    return v3(T.x * em[0] * k, T.y * em[1] * k, T.z * em[2] * k);
}

/* the MIS weight of a BSDF-sampled hit on emitter record R along d at t, pb the bounce's pdf */
static float bsdf_weight(const float *R, f3 d, float t, float pb) {
    const float pa = R[7], cl = -dot3(d, v3(R[12], R[13], R[14]));
    if (!(pa > 0) || !(cl > 0)) return 1.0f;
    const float pl = pa * (t * t) / cl, q = pl / pb;
    return 1 / (1 + q * q);
}

/* shade_sample_tree's mode-2 loop with light sampling (header) */
static f3 shade_sample_nee(const oracle_params *P, const oracle_instance *I, int n, const float *tree,
                           const oracle_emitters *E, ray_t r, uint32_t pixel, uint32_t sample, hit_t *first,
                           float *edge, uint64_t *cnt) {
    f3 L = v3(0, 0, 0), T = v3(1, 1, 1);
    int inst, mis = 0;
    float pb = 0;
    for (int seg = 0; seg < P->depth; seg++) {
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
        float w = 1.0f;
        if (mis && inst < 0 && E->n > 0 && E->map[h.prim] >= 0) w = bsdf_weight(E->rec + 16 * (size_t)E->map[h.prim], r.dir, h.t, pb);
        L = add3(L, v3(T.x * mat.emission[0] * w, T.y * mat.emission[1] * w, T.z * mat.emission[2] * w));
        T = v3(T.x * mat.albedo[0], T.y * mat.albedo[1], T.z * mat.albedo[2]);
        f3 hitp = add3(r.orig, scale3(r.dir, h.t));
        f3 nd;
        if (mat.kind == 1) {
            nd = normalize3(sub3(r.dir, scale3(h.normal, 2 * dot3(r.dir, h.normal))));
            mis = 0;
        } else {
            if (seg + 1 < P->depth && E->Q > 0)
                L = add3(L, nee(P, I, n, tree, E, hitp, h.normal, T, pixel, sample, (uint32_t)seg, cnt));
            int fell;
            nd = cosine_dir_flag(h.normal, pixel, sample, (uint32_t)seg, P->seed, &fell);
            mis = !fell;
            pb = dot3(nd, h.normal) * NEE_PB;
        }
        hitp = add3(hitp, scale3(nd, 0.0001f));
        r = make_ray(hitp, nd);
    }
    return L;
}

/* oracle_render_instance_tree's loop (its copy) in mode 3, with shade_sample_nee.  The emitter
 * table is oracle_build_emitters'; tree == NULL walks the instance list. */
int oracle_render_nee(oracle_params *P, const oracle_instance *I, int32_t n_instances, const float *tree,
                      const float *rec, const uint64_t *cdf, const int32_t *map, const uint64_t *hdr) {
    const int W = P->width, H = P->height;
    if ((P->flags & ORACLE_ACCUMULATE) && (!P->accum || !P->rgba)) return 1;
    const oracle_emitters E = { rec, cdf, map, hdr[0], hdr[1] };
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
                    f3 c = shade_sample_nee(P, I, n_instances, tree, &E, r, pixel, sample, s == 0 ? &first : NULL,
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

/* occluded() for caller-supplied rays (the brute-force check in tests/test_oracle_nee.py):
 * rays float[n][7] = origin, direction, t_max; out[i] = 1 when occluded. */
int oracle_occluded_rays(const oracle_params *P, const oracle_instance *I, int32_t n_instances, const float *tree,
                         const float *rays, int32_t n, int32_t *out) {
    uint64_t cnt[6] = { 0, 0, 0, 0, 0, 0 };
    for (int i = 0; i < n; i++) {
        const float *q = rays + 7 * (size_t)i;
        const ray_t r = make_ray(v3(q[0], q[1], q[2]), v3(q[3], q[4], q[5]));
        out[i] = occluded(P, I, n_instances, tree, &r, q[6], cnt);
    }
    return 0;
}
