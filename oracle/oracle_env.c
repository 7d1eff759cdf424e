/* oracle_env.c -- environment lighting (modes 2 and 3) in the CPU restatement.  TEST INFRASTRUCTURE,
 * like oracle_nee.c, which it includes unchanged: this file adds the CPU twin of the device's
 * environment table (clpathtracer_b200/csrc/cuda/environment.cu), the lookup, the light sample and
 * the mode-2/3 render loop with an environment, for no instances, the list and the tree.
 *
 * Environment (EXTENSION; this is the definition the CUDA path equals bit for bit, and the builder
 * below produces the device's table bytes).  Every fp32 operation is one correctly rounded + - * /
 * or sqrt, never contracted.
 *   cube        six square faces of n x n texels of linear RGB radiance, 1 <= n <= 2048, face order
 *               +X, -X, +Y, -Y, +Z, -Z, texel (face * n + row) * n + col; host input float32
 *               [6][n][n][3], every value finite and >= 0.  Faces follow the OpenGL cube map:
 *                 face  sc   tc   ma        face  sc   tc   ma
 *                 +X    -z   -y   x         -X    +z   -y   x
 *                 +Y    +x   +z   y         -Y    +x   -z   y
 *                 +Z    +x   -y   z         -Z    -x   -y   z
 *               row j covers t in [j/n, (j+1)/n), column i covers s in [i/n, (i+1)/n).
 *   lookup      env(d): ax = |d.x|, ay = |d.y|, az = |d.z|; face X if ax >= ay and ax >= az, else Y
 *               if ay >= az, else Z, positive when that component is > 0; a = sc / |ma|,
 *               b = tc / |ma|; col = min(n - 1, (int)(((a + 1) * 0.5) * n)), row likewise with b
 *               (both also clamped at 0, which no direction reaches); the nearest texel, unfiltered.
 *   table       per texel in float64: ac = ((col + 0.5) / n) * 2 - 1, bc likewise with row,
 *               s2c = (1 + ac * ac) + bc * bc, w = ((r + g) + b) / (s2c * sqrt(s2c)) (radiance x
 *               the texel's solid angle, up to a constant), 0 unless w > 0 and finite;
 *               q = (uint64)(w / wmax * 2^32) (0 when wmax = 0); cdf = exclusive uint64 scan of q,
 *               Q = sum of q.  Record per texel float4 {r, g, b, pdf},
 *               pdf = (float)((((double)q / Q) * ((double)n * n)) * 0.25), 0 when q = 0: the density
 *               per unit area of face coordinates (a, b).  Header {n, Q}.
 *   miss        modes 2 and 3: a path that leaves the scene adds T * env(d) per channel (instead of
 *               T), so an all-ones environment renders the frame without one bit for bit.
 *   sample      mode 3, at every diffuse vertex of segment s with s + 1 < depth and Q > 0, after the
 *               emitter sample (and added after it): Philox counter (pixel, sample, 1 + s, 3) ->
 *               r0..r2; target = (r0 * Q) >> 32, the texel = the largest i with cdf[i] <= target;
 *               a = ((col + u01(r1)) / n) * 2 - 1, b likewise with row and r2; v = the face point
 *               whose (sc, tc, ma) is (a, b, +-1); l = normalize(v); s2 = (1 + a * a) + b * b;
 *               pe = pdf * (s2 * sqrt(s2)).  Nothing unless cx = l.n > 0.  Shadow ray from
 *               x + l * 1e-4 along l, t_max = FLT_MAX (oracle_nee.c: occluded).  Visible -> pb =
 *               cx * PB, r = pb / pe, k = r / (1 + r * r), and the vertex adds (T.c * texel.c) * k.
 *   MIS         mode 3, a miss whose last bounce was diffuse and did not fall back to the normal:
 *               the lookup's texel, a and b give pe = pdf * (s2 * sqrt(s2)), q = pe / pb (pb of that
 *               bounce) and the miss adds (T.c * texel.c) * w, w = 1 / (1 + q * q); no weight when
 *               pdf is not > 0.  Camera-ray misses, misses after a mirror and after the fallback
 *               keep weight 1.  Triangle emitters and the environment are disjoint light sets, so
 *               each one's two-strategy power heuristic is exact: mode 3 keeps mode 2's expectation.
 *   counters    one ray per environment shadow ray; its walk counters are summed.
 * Modes 0 and 1 ignore the environment.
 */
#include "oracle_nee.c"

#include <float.h>

typedef struct oracle_env {
    const float *tex;    /* 4 floats per texel: r, g, b, pdf */
    const uint64_t *cdf; /* 6 n^2 entries */
    int32_t n;           /* face size, 0: no environment */
    uint64_t Q;
} oracle_env;

/* ---------------------------------------------------------------- the table's twin */
/* rgb float[6 n^2 * 3] -> tex float[6 n^2 * 4], cdf uint64[6 n^2 + 1], hdr uint64[2] = {n, Q}. */
int oracle_build_env(const float *rgb, int32_t n, float *tex, uint64_t *cdf, uint64_t *hdr) {
    if (n < 1) return 1;
    const size_t T = 6 * (size_t)n * (size_t)n, nn = (size_t)n * (size_t)n;
    double *w = malloc(T * sizeof(double)), wmax = 0.0;
    for (size_t i = 0; i < T; i++) {
        const size_t rem = i % nn, row = rem / (size_t)n, col = rem - row * (size_t)n;
        const double ac = (((double)col + 0.5) / (double)n) * 2.0 - 1.0;
        const double bc = (((double)row + 0.5) / (double)n) * 2.0 - 1.0;
        const double s2 = (1.0 + ac * ac) + bc * bc;
        const double ww = (((double)rgb[3 * i] + (double)rgb[3 * i + 1]) + (double)rgb[3 * i + 2]) / (s2 * sqrt(s2));
        w[i] = (ww > 0.0 && ww < INFINITY) ? ww : 0.0;
        if (w[i] > wmax) wmax = w[i];
    }
    uint64_t Q = 0;
    for (size_t i = 0; i < T; i++) {
        const uint64_t q = wmax > 0.0 ? (uint64_t)(w[i] / wmax * 4294967296.0) : 0;
        cdf[i] = Q;
        Q += q;
        w[i] = (double)q;
    }
    cdf[T] = Q;
    for (size_t i = 0; i < T; i++) {
        tex[4 * i] = rgb[3 * i], tex[4 * i + 1] = rgb[3 * i + 1], tex[4 * i + 2] = rgb[3 * i + 2];
        tex[4 * i + 3] = w[i] > 0.0 ? (float)(((w[i] / (double)Q) * ((double)n * (double)n)) * 0.25) : 0.0f;
    }
    hdr[0] = (uint64_t)n;
    hdr[1] = Q;
    free(w);
    return 0;
}

/* ---------------------------------------------------------------- lookup and sample */
static int env_index(float x, int n) {
    int i = (int)(((x + 1.0f) * 0.5f) * (float)n);
    if (i > n - 1) i = n - 1;
    if (i < 0) i = 0;
    return i;
}

/* The texel env(d) looks up, and its face coordinates a, b (header). */
static size_t env_texel(int n, f3 d, float *a, float *b) {
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int face;
    float sc, tc, ma;
    if (ax >= ay && ax >= az) {
        ma = ax, tc = -d.y;
        if (d.x > 0) face = 0, sc = -d.z;
        else face = 1, sc = d.z;
    } else if (ay >= az) {
        ma = ay, sc = d.x;
        if (d.y > 0) face = 2, tc = d.z;
        else face = 3, tc = -d.z;
    } else {
        ma = az, tc = -d.y;
        if (d.z > 0) face = 4, sc = d.x;
        else face = 5, sc = -d.x;
    }
    *a = sc / ma;
    *b = tc / ma;
    return ((size_t)face * (size_t)n + (size_t)env_index(*b, n)) * (size_t)n + (size_t)env_index(*a, n);
}

/* the face point whose (sc, tc, ma) is (a, b, +-1) */
static f3 env_face_point(int face, float a, float b) {
    switch (face) {
    case 0: return v3(1.0f, -b, -a);
    case 1: return v3(-1.0f, -b, a);
    case 2: return v3(a, 1.0f, b);
    case 3: return v3(a, -1.0f, -b);
    case 4: return v3(a, -b, 1.0f);
    default: return v3(-a, -b, -1.0f);
    }
}

/* pe = pdf * (s2 * sqrt(s2)), s2 = (1 + a * a) + b * b: the solid-angle density of direction (a, b) */
static float env_pe(float pdf, float a, float b) {
    const float s2 = (1.0f + a * a) + b * b;
    return pdf * (s2 * sqrtf(s2));
}

/* The texel that words r0, r1, r2 select, the point (a, b) in it and its direction l (header). */
static size_t env_draw(const oracle_env *V, uint32_t r0, uint32_t r1, uint32_t r2, float *a, float *b, f3 *l) {
    const int n = V->n;
    const size_t texel = oracle_select_emitter(V->cdf, 6 * (uint64_t)n * (uint64_t)n, V->Q, r0);
    const size_t nn = (size_t)n * (size_t)n, face = texel / nn, rem = texel - face * nn;
    const size_t row = rem / (size_t)n, col = rem - row * (size_t)n;
    *a = (((float)col + u01(r1)) / (float)n) * 2.0f - 1.0f;
    *b = (((float)row + u01(r2)) / (float)n) * 2.0f - 1.0f;
    *l = normalize3(env_face_point((int)face, *a, *b));
    return texel;
}

/* the environment's light sample of a diffuse vertex at x with shading normal nrm and throughput T */
static f3 env_sample(const oracle_params *P, const oracle_instance *I, int n, const float *tree, const oracle_env *V,
                     f3 x, f3 nrm, f3 T, uint32_t pixel, uint32_t sample, uint32_t seg, uint64_t *cnt) {
    uint32_t c[4] = { pixel, sample, 1u + seg, 3 };
    philox4x32_10(c, P->seed, ORACLE_KEY1);
    float a, b;
    f3 l;
    const float *tx = V->tex + 4 * env_draw(V, c[0], c[1], c[2], &a, &b, &l);
    const float cx = dot3(l, nrm);
    const f3 none = v3(0, 0, 0);
    if (!(cx > 0)) return none;
    const ray_t sr = make_ray(add3(x, scale3(l, 0.0001f)), l);
    if (occluded(P, I, n, tree, &sr, FLT_MAX, cnt)) return none;
    const float r = cx * NEE_PB / env_pe(tx[3], a, b), k = r / (1 + r * r);
    return v3(T.x * tx[0] * k, T.y * tx[1] * k, T.z * tx[2] * k);
}

/* shade_sample_nee's loop with the environment: mode 2 (no light samples, no MIS) or 3 (header) */
static f3 shade_sample_env(const oracle_params *P, const oracle_instance *I, int n, const float *tree,
                           const oracle_emitters *E, const oracle_env *V, ray_t r, uint32_t pixel, uint32_t sample,
                           hit_t *first, float *edge, uint64_t *cnt) {
    const int m3 = P->mode == 3;
    f3 L = v3(0, 0, 0), T = v3(1, 1, 1);
    int inst, mis = 0;
    float pb = 0;
    for (int seg = 0; seg < P->depth; seg++) {
        hit_t h = world_hit_tree(P, I, n, tree, &r, cnt, &inst);
        if (seg == 0 && first) *first = h;
        note_edge(edge, &h);
        if (!h.did_hit) {
            float a, b;
            const float *tx = V->tex + 4 * env_texel(V->n, r.dir, &a, &b);
            f3 e = v3(T.x * tx[0], T.y * tx[1], T.z * tx[2]);
            if (m3 && mis && tx[3] > 0) {
                const float q = env_pe(tx[3], a, b) / pb;
                e = scale3(e, 1 / (1 + q * q));
            }
            return add3(L, e);
        }
        int m = inst >= 0 ? I[inst].material : (P->tri_material ? P->tri_material[h.prim] : 0);
        if (m < 0 || m >= P->n_materials) m = 0;
        oracle_material mat;
        if (P->n_materials > 0) mat = P->materials[m];
        else { mat.albedo[0] = mat.albedo[1] = mat.albedo[2] = 0.5f; mat.kind = 0;
               mat.emission[0] = mat.emission[1] = mat.emission[2] = 0; }
        float w = 1.0f;
        if (m3 && mis && inst < 0 && E->n > 0 && E->map[h.prim] >= 0)
            w = bsdf_weight(E->rec + 16 * (size_t)E->map[h.prim], r.dir, h.t, pb);
        L = add3(L, v3(T.x * mat.emission[0] * w, T.y * mat.emission[1] * w, T.z * mat.emission[2] * w));
        T = v3(T.x * mat.albedo[0], T.y * mat.albedo[1], T.z * mat.albedo[2]);
        f3 hitp = add3(r.orig, scale3(r.dir, h.t));
        f3 nd;
        if (mat.kind == 1) {
            nd = normalize3(sub3(r.dir, scale3(h.normal, 2 * dot3(r.dir, h.normal))));
            mis = 0;
        } else {
            if (m3 && seg + 1 < P->depth && E->Q > 0)
                L = add3(L, nee(P, I, n, tree, E, hitp, h.normal, T, pixel, sample, (uint32_t)seg, cnt));
            if (m3 && seg + 1 < P->depth && V->Q > 0)
                L = add3(L, env_sample(P, I, n, tree, V, hitp, h.normal, T, pixel, sample, (uint32_t)seg, cnt));
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

/* oracle_render_nee's loop (its copy) in mode P->mode = 2 or 3 with the environment (tex, env_cdf,
 * env_hdr from oracle_build_env).  The emitter table is oracle_build_emitters' (read in mode 3
 * only); tree == NULL walks the instance list. */
int oracle_render_env(oracle_params *P, const oracle_instance *I, int32_t n_instances, const float *tree,
                      const float *rec, const uint64_t *cdf, const int32_t *map, const uint64_t *hdr, const float *tex,
                      const uint64_t *env_cdf, const uint64_t *env_hdr) {
    const int W = P->width, H = P->height;
    if ((P->flags & ORACLE_ACCUMULATE) && (!P->accum || !P->rgba)) return 1;
    if (P->mode != 2 && P->mode != 3) return 1;
    const oracle_emitters E = { rec, cdf, map, P->mode == 3 ? hdr[0] : 0, P->mode == 3 ? hdr[1] : 0 };
    const oracle_env V = { tex, env_cdf, (int32_t)env_hdr[0], env_hdr[1] };
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
                    f3 c = shade_sample_env(P, I, n_instances, tree, &E, &V, r, pixel, sample, s == 0 ? &first : NULL,
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

/* ---------------------------------------------------------------- test hooks */
/* env(d) for dirs float[count][3]: texel[i], ab[2i], ab[2i + 1] */
int oracle_env_lookup(int32_t n, const float *dirs, int32_t count, int64_t *texel, float *ab) {
    for (int i = 0; i < count; i++)
        texel[i] = (int64_t)env_texel(n, v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]), ab + 2 * i, ab + 2 * i + 1);
    return 0;
}

/* The light sample's draw for words uint32[count][3] (r0, r1, r2): texel[i], ab[2i..], l[3i..], and
 * pe[i] = the solid-angle density of l. */
int oracle_env_draw(const float *tex, const uint64_t *cdf, const uint64_t *hdr, const uint32_t *words, int32_t count,
                    int64_t *texel, float *ab, float *l, float *pe) {
    const oracle_env V = { tex, cdf, (int32_t)hdr[0], hdr[1] };
    if (V.Q == 0) return 1;
    for (int i = 0; i < count; i++) {
        f3 d;
        texel[i] = (int64_t)env_draw(&V, words[3 * i], words[3 * i + 1], words[3 * i + 2], ab + 2 * i, ab + 2 * i + 1, &d);
        l[3 * i] = d.x, l[3 * i + 1] = d.y, l[3 * i + 2] = d.z;
        pe[i] = env_pe(tex[4 * texel[i] + 3], ab[2 * i], ab[2 * i + 1]);
    }
    return 0;
}
