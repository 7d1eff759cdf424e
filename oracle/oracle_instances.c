/* oracle_instances.c -- rigid instances in the CPU restatement.  TEST INFRASTRUCTURE, like
 * oracle_kernel.c, which it includes: the traversal, intersection, sampling and accumulation
 * below are that file's, unchanged; this file adds the walk over instances and the render loop
 * that calls it (oracle_render's loop with world_hit in place of closest_hit).
 *
 * Rigid instances (EXTENSION, no reference behaviour; this is the definition the CUDA path
 * equals bit for bit).  Instance k = a mesh with its own wire tree, a world-to-object matrix
 * [A | b] (row-major 3x4), a material and a primitive offset.
 *   object-space ray  o'_r = ((A_r0*o.x + A_r1*o.y) + A_r2*o.z) + b_r,
 *                     d'_r = (A_r0*d.x + A_r1*d.y) + A_r2*d.z   (un-contracted fp32, the form
 *                     of unproject); d' is not normalised, so the object-space t is the world
 *                     ray's t.
 *   walk              closest_hit on the instance's own tree with (o', d'): its root clip,
 *                     ropes, tie rule (:344), 0.001 early-out and its own rope-hop budget.
 *   order, ties       the base scene first, then the instances in array order; a later hit
 *                     replaces the current one when t <= best (the later tree wins ties).  An
 *                     instance is skipped when a hit exists and its root-clip entry tmin > best.
 *   shading           m = the object-space normal before normalisation: the flat normal's
 *                     cross((v2-v1), (v3-v1)), or the vertex normals interpolated with u, v of
 *                     the object-space ray.  The world normal is normalize(A^T m),
 *                     n_x = (A00*m.x + A10*m.y) + A20*m.z and so on.  (Normalising m first would
 *                     make an identity instance shade unlike its own mesh: normalize is not
 *                     idempotent in fp32.)  Hit point and bounce use the world ray.
 *   ids, materials    prim = the instance's prim offset + the mesh's primitive; AOVs report
 *                     it, the world t and u, v in the instance's triangle.  Mode C gives every
 *                     triangle of the instance the instance's material.
 *   counters          one ray per world query; splits, leaves, tests, capped summed over every
 *                     walk; a vn-shaded hit counted for the hit that is shaded.
 * With no instances, oracle_render_instanced is oracle_render (tests/test_oracle_instances.py).
 */
#include "oracle_kernel.c"

typedef struct oracle_instance {
    /* the mesh, in the wire layout CLSetMeshes receives */
    const onode *nodes;
    const int32_t *tri_indices;
    const i4 *tris;
    const f4 *verts;
    const f4 *norms; /* may be NULL */
    float w2o[12];   /* world to object, row-major 3x4 [A | b] */
    int32_t material;
    int32_t prim_offset;
} oracle_instance;

/* closest_hit of one walk: every counter but the ray and the vn-shaded hit, which belong to
 * the world query (world_hit) */
static hit_t walk(const oracle_params *P, const ray_t *r, uint64_t *cnt) {
    uint64_t own[6] = { 0, 0, 0, 0, 0, 0 };
    hit_t h = closest_hit(P, r, own);
    cnt[1] += own[1];
    cnt[2] += own[2];
    cnt[3] += own[3];
    cnt[5] += own[5];
    return h;
}

/* One world query: the base scene, then the instances.  *inst = the instance hit, -1 = base. */
static hit_t world_hit(const oracle_params *P, const oracle_instance *I, int n, const ray_t *r, uint64_t *cnt,
                       int *inst) {
    cnt[0]++;
    hit_t h = walk(P, r, cnt);
    *inst = -1;
    const i4 *tris = P->tris;
    const f4 *norms = P->norms;
    int local = h.prim;
    for (int k = 0; k < n; k++) {
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
        if (!clip_root(rb, &lr, &tmin, &tmax)) continue;
        if (h.did_hit && tmin > h.t) continue;
        oracle_params Q = *P;
        Q.nodes = I[k].nodes;
        Q.tri_indices = I[k].tri_indices;
        Q.tris = I[k].tris;
        Q.verts = I[k].verts;
        Q.norms = I[k].norms;
        hit_t hi = walk(&Q, &lr, cnt);
        if (!hi.did_hit || (h.did_hit && hi.t > h.t)) continue;
        /* the object-space normal before normalisation: closest_hit's expressions for this hit */
        const int b = hi.prim;
        const i4 c1 = I[k].tris[3 * b + 0], c2 = I[k].tris[3 * b + 1], c3 = I[k].tris[3 * b + 2];
        f3 mn;
        if (c1.s[1] >= 0) {
            const f3 n1 = xyz(I[k].norms[c1.s[1]]), n2 = xyz(I[k].norms[c2.s[1]]), n3 = xyz(I[k].norms[c3.s[1]]);
            const float w = 1.0f - hi.u - hi.v;
            mn = add3(add3(scale3(n1, w), scale3(n2, hi.u)), scale3(n3, hi.v));
        } else {
            const f3 v1 = xyz(I[k].verts[c1.s[0]]), v2 = xyz(I[k].verts[c2.s[0]]), v3_ = xyz(I[k].verts[c3.s[0]]);
            mn = cross3(sub3(v2, v1), sub3(v3_, v1));
        }
        hi.normal = normalize3(v3((m[0] * mn.x + m[4] * mn.y) + m[8] * mn.z, (m[1] * mn.x + m[5] * mn.y) + m[9] * mn.z,
                                  (m[2] * mn.x + m[6] * mn.y) + m[10] * mn.z));
        hi.prim = b + I[k].prim_offset;
        h = hi;
        *inst = k;
        tris = I[k].tris;
        norms = I[k].norms;
        local = b;
    }
    if (h.did_hit && norms != NULL && tris[3 * local].s[1] >= 0) cnt[4]++;
    return h;
}

/* shade_sample with world_hit; an instance hit takes the instance's material */
static f3 shade_sample_instanced(const oracle_params *P, const oracle_instance *I, int n, ray_t r, uint32_t pixel,
                                 uint32_t sample, hit_t *first, float *edge, uint64_t *cnt) {
    int depth = P->depth;
    int inst;
    if (P->mode == 0) depth = depth > 0 ? 1 : 0;
    if (P->mode == 2) {
        f3 L = v3(0, 0, 0), T = v3(1, 1, 1);
        for (int seg = 0; seg < depth; seg++) {
            hit_t h = world_hit(P, I, n, &r, cnt, &inst);
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
        hit_t h = world_hit(P, I, n, &r, cnt, &inst);
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

/* oracle_render's loop over pixels and samples, with shade_sample_instanced */
int oracle_render_instanced(oracle_params *P, const oracle_instance *I, int32_t n_instances) {
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
                    f3 c = shade_sample_instanced(P, I, n_instances, r, pixel, sample, s == 0 ? &first : NULL,
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

size_t oracle_sizeof_instance(void) { return sizeof(oracle_instance); }
