"""A float64 replay of what a frame means, checked against the CPU restatements and the CUDA frames.

Every other frame test holds CUDA to the CPU restatement (oracle/oracle_kernel.c, oracle_instances.c,
oracle_instance_tree.c) bit for bit, so a mistake made the same way in both passes them.  The replay
here restates the definition from its description alone -- no traversal, no tree, no fp32 after the
camera ray -- and is compared with both:

  scene     every world triangle in float64: the base scene's, and each instance mesh's mapped by its
            float64 object-to-world M.  Per triangle: material, vertex normals (mapped by M^-T, which
            commutes with the barycentric blend) and sign(det M).
  rays      camera rays in fp32 exactly as the oracle makes them (unproject, normalise, Philox jitter
            with counter (pixel, sample, 0, 0) and key (seed, 'clpt')), then lifted to float64.
  hits      brute force over all triangles: the closest hit with t > 0, u, v >= 0, u + v <= 1,
            front-facing when det_world * sign(det M) > 0 (object-space culling said in world space).
            det, u, v and t are Moller-Trumbore's quantities, evaluated as dot products of the ray with
            per-triangle vectors so that one matrix product serves a block of rays.
  shading   flat: sign(det M) * normalize(e1 x e2) = normalize(M^-T (e1' x e2')); vertex normals:
            normalize(w n1 + u n2 + v n3) of the mapped normals.
  mode 0    (n + 1) / 2, white on a miss.
  mode 1    mirror bounces, next origin hit + 1e-4 nd; col = col (1 - str) + nc str, str *= 0.2;
            finished with (1 - str) col + str.
  mode 2    emission times throughput, throughput times albedo, throughput added on a miss; diffuse
            bounces cosine-weighted (the same Philox disk tries, mapped through the Duff et al. basis in
            float64), mirror materials reflect.  Instances take their material; ids out of range are 0.

fp32 and float64 legitimately part ways where a ray passes within rounding of an edge, of a second
surface or of grazing, so the replay also records how well each segment is conditioned, and the frames
must agree on the pixels where every segment of every sample is well conditioned (see _conditioned).

test_mode_c_is_the_form_factor then checks that the mode C estimator is unbiased where the answer is
known in closed form: a diffuse floor under a rectangular emitter.
"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import oracle_instance_tree_py as ot
from oracle import oracle_instances_py as oi

f32 = np.float32
KEY1 = 0x636C7074

# Conditioning bars (segment by segment; _conditioned)
MARGIN = 1e-4        # smallest barycentric coordinate of the hit
GAP = 1e-3           # t gap to the next front-facing hit (also >= 1e-4 t); the traversal's 0.001 early-out
GAP_REL = 1e-4
COS = 1e-3           # |cos| between the ray and the geometric normal
NEXT_T = 1e-3        # t of every bounce segment's hit
NEAR_MISS = 1e-4     # a front-facing triangle missed by less than this barycentric margin
# Agreement bars on well-conditioned pixels: (mode 0 normal, mode 1/2 colour times max(1, |value|)).
# With instances: observed up to 6.6e-6 and 1.7e-5 -- the oracle maps rays and normals by the fp32
# world-to-object matrix and interpolates normals with fp32 u, v of the object-space ray, which the
# anisotropic and sheared matrices stretch.  Base scenes have no matrix in the chain: observed up to
# 1.8e-7 (one fp32 normalise), so their bars are tightened to 1e-6.
TOL_INSTANCES = (1e-5, 1e-4)
TOL_BASE = (1e-6, 1e-6)
CRACK_BUDGET = 5e-4  # share of well-conditioned pixels allowed to disagree; observed 0 in every case
MIN_WELL = 0.95      # share of hit pixels that must be well conditioned; observed >= 0.985


# ------------------------------------------------------------------------------------------ Philox
def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (oracle_kernel.c philox4x32_10) on uint32 arrays, vectorised."""
    c = [np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & m32
        k1 = (k1 + np.uint64(0xBB67AE85)) & m32
    return [x.astype(np.uint32) for x in c]


def u01(x):
    """(x >> 8) * 2^-24 in fp32: exact."""
    return (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(f32) * f32(2.0 ** -24)


def disk_point(pixel, sample, bounce, seed):
    """cosine_dir's point in the unit disk: four tries from two Philox blocks, accepted by the fp32
    test x*x + y*y <= 1 (each operation rounded), else the centre.  float32 arrays a, b."""
    a = np.zeros(np.shape(pixel), dtype=f32)
    b = np.zeros(np.shape(pixel), dtype=f32)
    found = np.zeros(np.shape(pixel), dtype=bool)
    for blk in range(2):
        c = philox(pixel, sample, 1 + np.asarray(bounce, dtype=np.uint64), blk, seed, KEY1)
        for k in range(2):
            x = f32(2) * u01(c[2 * k]) - f32(1)
            y = f32(2) * u01(c[2 * k + 1]) - f32(1)
            take = ~found & ((x * x + y * y) <= f32(1))
            a = np.where(take, x, a)
            b = np.where(take, y, b)
            found |= take
    return a, b


def cosine_dir64(n, a, b):
    """Malley's lift of the disk point (a, b) about the unit normal n, in the branch-free basis of
    Duff et al. 2017, in float64."""
    a, b = a.astype(np.float64), b.astype(np.float64)
    z = np.sqrt(np.maximum(1 - a * a - b * b, 0))
    nx, ny, nz = n[:, 0], n[:, 1], n[:, 2]
    sg = np.where(nz >= 0, 1.0, -1.0)
    p = -1 / (sg + nz)
    q = nx * ny * p
    t1 = np.stack([1 + sg * nx * nx * p, sg * q, -sg * nx], -1)
    t2 = np.stack([q, sg + ny * ny * p, -ny], -1)
    d = a[:, None] * t1 + b[:, None] * t2 + z[:, None] * n
    return d / np.linalg.norm(d, axis=1, keepdims=True)


# ------------------------------------------------------------------------------------- camera rays
def primary_rays(cam, w, h, spp, seed, jitter):
    """The oracle's camera rays (oracle_render) in fp32, lifted to float64.  Ray r = pixel * spp + s."""
    M = np.asarray(cam, dtype=f32).reshape(16)
    ys, xs = np.meshgrid(np.arange(h, dtype=np.uint32), np.arange(w, dtype=np.uint32), indexing="ij")
    pixel = np.repeat((ys * np.uint32(w) + xs).reshape(-1), spp)
    sample = np.tile(np.arange(spp, dtype=np.uint32), w * h)
    fx = np.repeat(xs.reshape(-1).astype(f32), spp) - f32(w) / f32(2)
    fy = np.repeat(ys.reshape(-1).astype(f32), spp) - f32(h) / f32(2)
    if jitter:
        c = philox(pixel, sample, 0, 0, seed, KEY1)
        fx = fx + (u01(c[0]) - f32(0.5))
        fy = fy + (u01(c[1]) - f32(0.5))

    def unproject(z):
        z = f32(z)
        wd = ((M[12] * fx + M[13] * fy) + M[14] * z) + M[15]
        return [(((M[4 * r] * fx + M[4 * r + 1] * fy) + M[4 * r + 2] * z) + M[4 * r + 3]) / wd for r in range(3)]

    ncp, fcp = unproject(-1), unproject(1)
    d = [fcp[k] - ncp[k] for k in range(3)]
    ln = np.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
    d = np.stack([d[k] / ln for k in range(3)], -1).astype(np.float64)
    o = np.array([M[2] / M[14], M[6] / M[14], M[10] / M[14]], dtype=f32).astype(np.float64)
    return np.broadcast_to(o, d.shape).copy(), d, pixel, sample


# ------------------------------------------------------------------------------------------- scene
class World:
    """Every triangle of base scene + instances in float64."""

    def __init__(self, base, instances=(), tri_material=None):
        """base = (verts, corners, norms); instances = [((verts, corners, norms), o2w 3x4, material)]."""
        parts = [(base, np.hstack([np.eye(3), np.zeros((3, 1))]), None, tri_material)]
        parts += [(mesh, np.asarray(m, dtype=np.float64), mat, None) for mesh, m, mat in instances]
        V, VN, HAS, SG, MAT, SRC = [], [], [], [], [], []
        for k, ((verts, corners, norms), m, inst_mat, tm) in enumerate(parts):
            A, b = m[:, :3], m[:, 3]
            c = np.asarray(corners).reshape(-1, 3, 4)
            v = np.asarray(verts, dtype=f32)[:, :3].astype(np.float64)
            V.append(v[c[:, :, 0]] @ A.T + b)
            has = c[:, 0, 1] >= 0
            vn = np.zeros((len(c), 3, 3))
            if has.any():
                nn = np.asarray(norms, dtype=f32)[:, :3].astype(np.float64)
                vn[has] = nn[c[has][:, :, 1]] @ np.linalg.inv(A)  # rows n^T A^-1 = (A^-T n)^T
            VN.append(vn)
            HAS.append(has)
            SG.append(np.full(len(c), np.sign(np.linalg.det(A))))
            if inst_mat is not None:
                MAT.append(np.full(len(c), inst_mat))
            else:
                MAT.append(np.zeros(len(c), dtype=np.int64) if tm is None else np.asarray(tm, dtype=np.int64))
            SRC.append(np.full(len(c), k - 1))
        tri = np.concatenate(V)
        self.v0, self.e1, self.e2 = tri[:, 0], tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]
        self.vn, self.has_vn = np.concatenate(VN), np.concatenate(HAS)
        self.sign, self.material, self.source = np.concatenate(SG), np.concatenate(MAT), np.concatenate(SRC)
        n = np.cross(self.e1, self.e2)
        nn = (n * n).sum(1)
        self.n, self.nlen = n, np.sqrt(nn)
        # u = au . p + bu and v = av . p + bv at a point p of the plane (exact in real arithmetic)
        au, av = np.cross(self.e2, n) / nn[:, None], np.cross(n, self.e1) / nn[:, None]
        self.lin = np.concatenate([n, au, av])              # [3T, 3]
        self.off = -np.concatenate([(n * self.v0).sum(1), (au * self.v0).sum(1), (av * self.v0).sum(1)])
        self.T = len(tri)

    def shading_normal(self, i, u, v):
        flat = self.sign[i, None] * self.n[i] / self.nlen[i, None]
        vn = self.vn[i]
        w = 1 - u - v
        sm = w[:, None] * vn[:, 0] + u[:, None] * vn[:, 1] + v[:, None] * vn[:, 2]
        with np.errstate(invalid="ignore", divide="ignore"):
            sm = sm / np.linalg.norm(sm, axis=1, keepdims=True)
        return np.where(self.has_vn[i, None], sm, flat)


def _intersect_block(world, o, d):
    T = world.T
    D = d @ world.lin.T                                  # [r, 3T]: n.d, au.d, av.d
    O = o @ world.lin.T + world.off                      # n.(o - v0), u and v of the origin's projection
    nd, no = D[:, :T], O[:, :T]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = -no / nd                                     # MT: t = (o - v0).n / det, det = -n.d
        u = O[:, T:2 * T] + t * D[:, T:2 * T]
        v = O[:, 2 * T:] + t * D[:, 2 * T:]
    margin = np.minimum(np.minimum(u, v), 1 - u - v)
    front = (-nd * world.sign) > 0
    hit = front & (margin >= 0) & (t > 0)
    tt = np.where(hit, t, np.inf)
    idx = T - 1 - np.argmin(tt[:, ::-1], axis=1)         # the later source wins exact ties
    rows = np.arange(len(d))
    best = tt[rows, idx]
    did = np.isfinite(best)
    tt[rows, idx] = np.inf
    second = tt.min(1)
    gap_bar = np.where(did, np.maximum(GAP, GAP_REL * best), np.inf)
    near = front & (margin < 0) & (margin >= -NEAR_MISS)
    near_miss = (near & (t > 0) & (t < (best + gap_bar)[:, None])).any(1)
    # a front-facing triangle through the origin: fp32 may put it on either side
    at_origin = (front & (margin >= -NEAR_MISS) & (np.abs(t) < 1e-5)).any(1)
    cos = np.abs(nd[rows, idx]) / world.nlen[idx]
    with np.errstate(invalid="ignore"):
        gap = second - best
    return (np.where(did, idx, -1), best, u[rows, idx], v[rows, idx], margin[rows, idx], gap, cos,
            near_miss, at_origin)


def intersect(world, o, d, block=256):
    """Brute-force closest hits of rays (o, d) in float64 plus the conditioning of each."""
    n = len(d)
    starts = list(range(0, n, block))
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        res = list(ex.map(lambda s: _intersect_block(world, o[s:s + block], d[s:s + block]), starts))
    return [np.concatenate([r[k] for r in res]) for k in range(9)]


def _conditioned(seg, t, margin, gap, cos, near_miss, at_origin, did):
    ok = ~near_miss & ~at_origin
    ok &= ~did | ((margin >= MARGIN) & (gap >= np.maximum(GAP, GAP_REL * t)) & (cos >= COS))
    if seg > 0:
        ok &= ~did | (t >= NEXT_T)
    return ok


# ------------------------------------------------------------------------------------------ replay
def replay(world, cam, w, h, mode, depth, spp, seed, jitter, materials=None):
    """The frame in float64.  Returns dict: value (h, w, 3) -- the mean normal in mode 0 (misses
    (1, 1, 1)), the mean colour otherwise; well (h, w) bool; hit (h, w) bool (the primary ray of some
    sample hits); hits (h*w*spp,) segments that hit per path."""
    o, d, pixel, sample = primary_rays(cam, w, h, spp, seed, jitter)
    R = len(d)
    ok = np.ones(R, dtype=bool)
    hits = np.zeros(R, dtype=np.int64)
    alive = np.arange(R)
    if mode == 0:
        depth = min(depth, 1)
    out = np.ones((R, 3))
    col, strength = np.zeros((R, 3)), np.ones(R)
    L, T = np.zeros((R, 3)), np.ones((R, 3))
    first_hit = np.zeros(R, dtype=bool)
    mats = None if materials is None else np.asarray(materials, dtype=f32).astype(np.float64)
    kinds = None if materials is None else np.asarray(materials, dtype=f32).view(np.int32)[:, 3]
    for seg in range(depth):
        if len(alive) == 0:
            break
        oo, dd = o[alive], d[alive]
        idx, t, u, v, margin, gap, cos, near_miss, at_origin = intersect(world, oo, dd)
        did = idx >= 0
        ok[alive] &= _conditioned(seg, t, margin, gap, cos, near_miss, at_origin, did)
        if seg == 0:
            first_hit[alive] = did
        hits[alive] += did
        miss = alive[~did]
        if mode == 2:
            L[miss] += T[miss]
        a, ih = alive[did], idx[did]
        n = world.shading_normal(ih, u[did], v[did])
        if mode == 0:
            out[a] = n
            break
        dda = dd[did]
        hp = oo[did] + t[did, None] * dda
        refl = dda - 2 * (dda * n).sum(1, keepdims=True) * n
        refl /= np.linalg.norm(refl, axis=1, keepdims=True)
        if mode == 1:
            nc = (n + 1) / 2
            col[a] = col[a] * (1 - strength[a, None]) + nc * strength[a, None]
            strength[a] *= 0.2
            nd = refl
        else:
            m = world.material[ih]
            m = np.where((m < 0) | (m >= len(mats)), 0, m)
            L[a] += T[a] * mats[m, 4:7]
            T[a] *= mats[m, 0:3]
            diffuse = kinds[m] != 1
            nd = refl.copy()
            if diffuse.any():
                pa, sa = disk_point(pixel[a][diffuse], sample[a][diffuse], seg, seed)
                nd[diffuse] = cosine_dir64(n[diffuse], pa, sa)
                # the basis flips with the sign of n.z: a normal within rounding of n.z = 0 is ill posed
                tiny = (np.abs(n[diffuse, 2]) < 1e-6) & (n[diffuse, 2] != 0)
                ok[a[diffuse][tiny]] = False
        o[a] = hp + 1e-4 * nd
        d[a] = nd
        alive = a
    if mode == 1:
        out = (1 - strength[:, None]) * col + strength[:, None]
    elif mode == 2:
        out = L
    value = out.reshape(h * w, spp, 3).mean(1).reshape(h, w, 3)
    return dict(value=value, well=ok.reshape(h * w, spp).all(1).reshape(h, w),
                hit=first_hit.reshape(h * w, spp).any(1).reshape(h, w), hits=hits)


# ------------------------------------------------------------------------------------------- cases
def _o2w(angles, scale, translate, shear=None):
    """3x4 object-to-world: translate . Rz . Ry . Rx . (shear) . diag(scale)."""
    ax, ay, az = angles
    rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    sh = np.eye(3) if shear is None else np.asarray(shear, dtype=np.float64)
    m = np.zeros((3, 4))
    m[:, :3] = rz @ ry @ rx @ sh @ np.diag(scale)
    m[:, 3] = translate
    return m


SHEAR = [[1, 0.6, -0.3], [0.2, 1, 0.5], [-0.4, 0.1, 1]]
# instance cases over hf22n: (mesh, angles, scale, translate, shear, material) per instance.  Material 3
# is the emitter of CORNELL_MATERIALS; 7 is out of range (mode C clamps it to 0).
INSTANCE_CASES = {
    "rotscale": [("icon", (1.1, -0.4, 0.3), (0.5, 0.12, 0.2), (0.0, 0.2, -0.45), None, 1),
                 ("ico", (0.3, 0.7, -0.2), (0.35, 0.2, 0.25), (-0.45, 0.25, 0.1), None, 2)],
    "shear": [("ico", (0.4, -0.3, 0.8), (0.3, 0.2, 0.25), (0.1, 0.3, -0.3), SHEAR, 2),
              ("icon", (-0.6, 0.5, 0.2), (0.25, 0.3, 0.2), (-0.4, 0.2, 0.2), SHEAR, 3)],
    "mirror": [("icon", (0.3, 0.7, -0.2), (-0.35, 0.2, 0.25), (-0.15, 0.25, -0.3), None, 1),
               ("ico", (-0.5, 0.2, 0.9), (0.3, -0.25, 0.3), (0.35, 0.25, 0.0), SHEAR, 7)],
    "overlap": [("icon", (0.2, 0.1, 0.4), (0.45, 0.3, 0.4), (0.0, -0.05, -0.2), None, 0),
                ("ico", (0.7, 0.0, -0.3), (0.3, 0.25, 0.35), (0.45, 0.0, 0.3), None, 3)],
}
# (case, mode, depth, spp); jitter at spp > 1
RUNS = [(c, 0, 1, 1) for c in ("hf22", "cornell", "sah")] + [("hf22", 1, 5, 4), ("cornell", 1, 5, 1), ("sah", 1, 4, 4),
                                                            ("hf22", 2, 5, 4), ("cornell", 2, 5, 4), ("sah", 2, 4, 1)]
RUNS += [(c, 0, 1, 4 if c in ("shear", "mirror") else 1) for c in INSTANCE_CASES]
RUNS += [(c, 1, 4, 4 if c in ("rotscale", "overlap") else 1) for c in INSTANCE_CASES]
RUNS += [(c, 2, 4, 4) for c in INSTANCE_CASES]
W, H = 96, 72
SEED = 21


def _ids(run):
    return "%s-m%d-d%d-spp%d" % run


def _mesh(name):
    import bench
    from clpathtracer_b200 import corners_from_faces, scenes

    if name in ("ico", "icon"):
        v, f = bench.icosphere(2)
        return v.astype(f32), corners_from_faces(f, name == "icon"), v.astype(f32) if name == "icon" else None
    if name == "cornell":
        return scenes.cornell(6)[:3]
    return scenes.heightfield(22, name == "hf22n")


def _case(name):
    """(base mesh arrays, tri_material, camera kwargs, how to build the base tree, instances)."""
    from clpathtracer_b200 import scenes

    if name == "cornell":
        return _mesh("cornell"), scenes.cornell(6)[3], scenes.CORNELL_CAMERA, "median", []
    if name in ("hf22", "sah"):
        return _mesh("hf22"), None, scenes.CANONICAL_CAMERA, "sah" if name == "sah" else "median", []
    inst = [(mesh, _o2w(a, s, t, sh), mat) for mesh, a, s, t, sh, mat in INSTANCE_CASES[name]]
    return _mesh("hf22n"), None, scenes.CANONICAL_CAMERA, "median", inst


_replays = {}


def _replay(clpt, run):
    """The replay of a run (computed once per session) and its camera."""
    from clpathtracer_b200 import scenes

    name, mode, depth, spp = run
    base, tm, camkw, _, inst = _case(name)
    cam = clpt.cam_matrix(clpt.make_camera(**camkw), H)
    if run not in _replays:
        world = World(base, [(_mesh(m), o2w, mat) for m, o2w, mat in inst], tm)
        _replays[run] = replay(world, cam, W, H, mode, depth, spp, SEED, spp > 1,
                               scenes.CORNELL_MATERIALS if mode == 2 else None)
    return _replays[run], cam


def _render_kw(run):
    from clpathtracer_b200 import scenes

    name, mode, depth, spp = run
    kw = dict(mode=mode, depth=depth, spp=spp, seed=SEED, flags=1 if spp > 1 else 0)
    if mode == 2:
        kw.update(materials=scenes.CORNELL_MATERIALS, tri_material=scenes.cornell(6)[3] if name == "cornell" else None)
    return kw


def _compare(rep, rgba, run, what, normal_aov=None):
    """Agreement of a frame with the replay on the well-conditioned pixels; returns the report line."""
    well, hit = rep["well"], rep["hit"]
    mode = run[1]
    NORMAL_TOL, COLOUR_TOL = TOL_INSTANCES if run[0] in INSTANCE_CASES else TOL_BASE
    if mode == 0:
        got = 2 * rgba[..., :3].astype(np.float64) - 1
        err = np.abs(got - rep["value"]).max(-1)
        bad = well & (err > NORMAL_TOL)
    else:
        got = rgba[..., :3].astype(np.float64)
        err = (np.abs(got - rep["value"]) / np.maximum(1, np.abs(rep["value"]))).max(-1)
        bad = well & (err > COLOUR_TOL)
    aov_err = 0.0
    if normal_aov is not None:  # sample 0's first-hit normal
        aov_err = np.abs(normal_aov - rep["value"]).max(-1)[well & hit].max()
        assert aov_err <= NORMAL_TOL, (what, aov_err)
    hits = rep["hits"]
    share = well[hit].mean()
    line = ("%s: well %.4f of %d hit pixels, %d disagree, max err %.2e (aov %.2e), paths with >=2 hits %.3f, "
            ">=3 %.3f" % (what, share, hit.sum(), bad.sum(), err[well].max(), aov_err, (hits >= 2).mean(),
                          (hits >= 3).mean()))
    print(line)
    assert share >= MIN_WELL, line
    assert bad.sum() <= CRACK_BUDGET * well.sum(), line
    return line


def _paths_bounce(run, rep):
    """The frame must check paths, not only first hits."""
    name, mode, depth, spp = run
    hits = rep["hits"]
    if mode != 0:  # observed: >= 3.3% of all paths (about half the frame is sky), 46% in the Cornell box
        assert (hits >= 2).mean() > 0.02, (run, (hits >= 2).mean())
        if name == "cornell":
            assert (hits >= 3).mean() > 0.3, (run, (hits >= 3).mean())


def _oracle_scenes(clpt, name):
    base, tm, _, how, inst = _case(name)
    tree = clpt.build_kd_sah(*base) if how == "sah" else clpt.build_kd(*base)
    meshes = {m: clpt.build_kd(*_mesh(m)) for m in {m for m, _, _ in inst}}
    return tree, [(meshes[m], clpt.world_to_object(o2w), mat) for m, o2w, mat in inst]


# --------------------------------------------------------------------------------------- CPU tests
def test_instance_cases_are_what_they_say():
    """rotscale and overlap keep orientation, shear has a sheared linear part, mirror mirrors both
    instances, and overlap's first instance reaches below and above the whole terrain."""
    for name, spec in INSTANCE_CASES.items():
        for mesh, a, s, t, sh, _ in spec:
            A = _o2w(a, s, t, sh)[:, :3]
            assert (np.linalg.det(A) < 0) == (name == "mirror"), name
            ata = A.T @ A  # diagonal for rotation times axis scale, not under shear
            assert (np.abs(ata - np.diag(np.diag(ata))).max() > 1e-3) == (sh is not None), name
    assert any(sh is not None for *_, sh, _ in INSTANCE_CASES["mirror"])
    v = _mesh("icon")[0].astype(np.float64) @ _o2w(*INSTANCE_CASES["overlap"][0][1:5])[:, :3].T
    y = v[:, 1] + INSTANCE_CASES["overlap"][0][3][1]
    terrain = _mesh("hf22n")[0][:, 1]
    assert y.min() < terrain.min() and y.max() > terrain.max()


def test_philox_matches_the_oracle(oracle):
    """The vectorised Philox gives the Random123 known answers and the oracle's words."""
    kat = [([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
           ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
           ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
            [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1])]
    for ctr, key, want in kat:
        assert [int(x) for x in philox(*ctr, *key)] == want
    rng = np.random.default_rng(0)
    ctr = rng.integers(0, 2 ** 32, (64, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, (64, 2), dtype=np.uint64).astype(np.uint32)
    got = np.stack(philox(*ctr.T, key[0, 0], key[0, 1]), -1)
    for i in range(64):
        assert np.array_equal(got[i], oracle.philox(ctr[i], key[0]))


def test_primary_rays_are_the_oracles(clpt, oracle):
    """Without and with jitter, the replay's fp32 camera rays hit the oracle's t bit for bit on the
    pixels whose first hit is a well-separated triangle, so they are the same rays."""
    from clpathtracer_b200 import scenes

    tree, _ = _oracle_scenes(clpt, "hf22")
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), H)
    for jitter in (False, True):
        o, d, _, sample = primary_rays(cam, W, H, 4, SEED, jitter)
        first = sample == 0
        ref = oracle.render(tree, cam, W, H, mode=0, depth=1, spp=4, seed=SEED, flags=int(jitter))
        world = World(_mesh("hf22"))
        idx, t, *_ = intersect(world, o[first], d[first])
        prim = ref["prim"].reshape(-1)
        same = (idx == prim) & (idx >= 0)
        assert (prim >= 0).mean() > 0.3 and same.sum() > 0.99 * (prim >= 0).sum(), jitter
        assert np.allclose(t[same], ref["t"].reshape(-1)[same], rtol=1e-5, atol=0)  # fp32 Moller-Trumbore t: ~2e-6


@pytest.mark.parametrize("run", RUNS, ids=_ids)
def test_oracle_matches_replay(clpt, oracle, run):
    name, mode, depth, spp = run
    rep, cam = _replay(clpt, run)
    tree, inst = _oracle_scenes(clpt, name)
    kw = _render_kw(run)
    if inst:
        ref = oi.render(tree, cam, W, H, instances=inst, **kw)
        by_tree = ot.render(tree, cam, W, H, instances=inst, tree=ot.tree_of(inst), **kw)
        for key in ("rgba", "prim", "t", "uv", "normal"):
            assert np.array_equal(np.ascontiguousarray(ref[key]).view(np.uint8),
                                  np.ascontiguousarray(by_tree[key]).view(np.uint8)), key
    else:
        ref = oracle.render(tree, cam, W, H, **kw)
    if inst and mode == 0:  # every instance is the first hit somewhere
        offset = tree.n_tris
        for mesh, _, _ in inst:
            assert ((ref["prim"] >= offset) & (ref["prim"] < offset + mesh.n_tris)).sum() > 20
            offset += mesh.n_tris
    aov = ref["normal"].astype(np.float64) if mode == 0 and spp == 1 else None
    _compare(rep, ref["rgba"], run, "oracle " + _ids(run), aov)
    _paths_bounce(run, rep)


# ----------------------------------------------------------------------------- mode C, analytically
# A diffuse floor (albedo A_FLOOR, flat normal +y) under a rectangular emitter facing down (albedo 0,
# emission E_LIGHT) at height H_LIGHT, seen from above through the emitter's culled back.  Mode 2 at
# depth 2 without jitter: every sample of a pixel starts at the same floor point x, and its bounce
# either reaches the emitter (colour a E) or escapes (colour a), so the sample colour is
#     a + a (E - 1) Bernoulli(P),   P = (1 - p) F(x) + p 1(x under the emitter),
# with F the form factor of the rectangle seen from x (cosine-weighted directions that hit it) and p
# the chance that all four disk tries are rejected and the bounce leaves along the normal.  The 1e-4
# start offset moves the bounce origin along the bounce direction itself, so the bounce ray is the same
# line and meets the emitter (0.5 away) or not exactly as without it: it changes nothing here.
# a = 0.5 and E = 3 make every sample colour (0.5 or 1.5) and every partial sum exact in fp32.
A_FLOOR, E_LIGHT, H_LIGHT = 0.5, 3.0, 0.5
LIGHT = (-0.6, 0.6, -0.45, 0.55)  # x0, x1, z0, z1
FLOOR_CAMERA = dict(near=0.1, far=1.0, fov=np.pi / 3, position=(0.0, 1.6, 0.0), forward=(0.0, -0.999, 0.045))


def _floor_scene():
    x0, x1, z0, z1 = LIGHT
    s = 3.0
    verts = np.array([[-s, 0, -s], [-s, 0, s], [s, 0, s], [s, 0, -s],
                      [x0, H_LIGHT, z0], [x0, H_LIGHT, z1], [x1, H_LIGHT, z1], [x1, H_LIGHT, z0]], dtype=f32)
    faces = np.array([[0, 1, 2], [0, 2, 3], [4, 6, 5], [4, 7, 6]])  # floor faces +y, the emitter -y
    from clpathtracer_b200 import corners_from_faces

    mats = np.zeros((2, 8), dtype=f32)
    mats[0, :3] = A_FLOOR
    mats[1, 4:7] = E_LIGHT
    return verts, corners_from_faces(faces, False), np.array([0, 0, 1, 1], dtype=np.int32), mats


def form_factor(px, pz):
    """Differential area at (px, 0, pz) facing +y to the parallel rectangle LIGHT at height H_LIGHT:
    the corner formula (a rectangle with one corner above the point), odd in each side, combined over
    the four corners."""
    def corner(a, b):
        A, B = a / H_LIGHT, b / H_LIGHT
        sa, sb = np.sqrt(1 + A * A), np.sqrt(1 + B * B)
        return (A / sa * np.arctan(B / sa) + B / sb * np.arctan(A / sb)) / (2 * np.pi)

    x0, x1, z0, z1 = LIGHT
    return corner(x1 - px, z1 - pz) - corner(x0 - px, z1 - pz) - corner(x1 - px, z0 - pz) + corner(x0 - px, z0 - pz)


def test_form_factor_formula():
    """The corner-formula form factor against midpoint quadrature of cos cos' / (pi r^2) over the
    rectangle."""
    x0, x1, z0, z1 = LIGHT
    n = 2000
    xs = x0 + (np.arange(n) + 0.5) * (x1 - x0) / n
    zs = z0 + (np.arange(n) + 0.5) * (z1 - z0) / n
    X, Z = np.meshgrid(xs, zs)
    for px, pz in [(0.0, 0.0), (0.55, -0.4), (1.2, 0.9), (-1.0, 0.2)]:
        r2 = (X - px) ** 2 + (Z - pz) ** 2 + H_LIGHT ** 2
        q = (H_LIGHT ** 2 / (np.pi * r2 * r2)).sum() * (x1 - x0) * (z1 - z0) / n ** 2
        assert abs(q - form_factor(px, pz)) < 1e-6, (px, pz)


def all_rejected():
    """p: the chance that four independent disk tries are all rejected, counted exactly on the grid
    the tries come from (x = 2 u01 - 1 = -1 + k 2^-23) with the fp32 test x*x + y*y <= 1."""
    j = np.arange(2 ** 23 + 1, dtype=np.int64)              # |x| = j 2^-23 (j = 2^23 is x = -1 only)
    x = j.astype(f32) * f32(2.0 ** -23)
    xx = x * x
    lo = np.zeros(len(j), dtype=np.int64)                    # passes: y = 0
    hi = np.full(len(j), 2 ** 23 + 1, dtype=np.int64)       # beyond the grid
    while (hi - lo > 1).any():                              # the fp32 test is monotone in |y|
        mid = (lo + hi) // 2
        y = mid.astype(f32) * f32(2.0 ** -23)
        ok = (xx + y * y) <= f32(1)
        lo, hi = np.where(ok, mid, lo), np.where(ok, hi, mid)
    best = lo                                               # the largest |y| / 2^-23 accepted
    count = best + 1 + np.minimum(best, 2 ** 23 - 1)        # y = -best..0 and 1..min(best, 2^23 - 1)
    accepted = count.sum() + count[1:2 ** 23].sum()         # x = -j 2^-23 (j = 0..2^23) and +j (j = 1..2^23-1)
    return (1 - accepted / 2.0 ** 48) ** 4


def _mode_c_statistic(clpt, rgba, w, h, spp):
    cam = clpt.cam_matrix(clpt.make_camera(**FLOOR_CAMERA), h)
    o, d, _, _ = primary_rays(cam, w, h, 1, 0, False)
    t = -o[:, 1] / d[:, 1]
    x = o + t[:, None] * d
    x0, x1, z0, z1 = LIGHT
    under = (x[:, 0] > x0) & (x[:, 0] < x1) & (x[:, 2] > z0) & (x[:, 2] < z1)
    p = all_rejected()
    P = (1 - p) * form_factor(x[:, 0], x[:, 2]) + p * under
    expected = A_FLOOR + A_FLOOR * (E_LIGHT - 1) * P
    sigma = A_FLOOR * abs(E_LIGHT - 1) * np.sqrt(P * (1 - P))
    assert (spp * P * (1 - P)).min() > 10  # every pixel's count is far from 0 and from spp
    mean = rgba[..., 0].reshape(-1).astype(np.float64)
    assert np.array_equal(rgba[..., 0], rgba[..., 1]) and np.array_equal(rgba[..., 0], rgba[..., 2])
    z = (mean - expected) / (sigma / np.sqrt(spp))
    n = len(z)
    line = "mode C %dx%d at %d spp: p = %.7f, mean z %+.4f (bar %.4f), mean z^2 %.4f (bar 1 +- %.4f), max |z| %.2f" % (
        w, h, spp, p, z.mean(), 5 / np.sqrt(n), (z * z).mean(), 5 * np.sqrt(2 / n), np.abs(z).max())
    print(line)
    assert abs(z.mean()) < 5 / np.sqrt(n), line
    assert abs((z * z).mean() - 1) < 5 * np.sqrt(2 / n), line
    assert np.abs(z).max() < 6, line


def test_mode_c_is_the_form_factor(clpt, oracle):
    """The oracle's mode C estimate is unbiased: per-pixel means against the form factor, at 1,024
    samples per pixel (seed fixed, so the statistic is a fixed number)."""
    verts, corners, tm, mats = _floor_scene()
    scene = clpt.build_kd(verts, corners)
    w, h, spp = 48, 36, 1024
    cam = clpt.cam_matrix(clpt.make_camera(**FLOOR_CAMERA), h)
    ref = oracle.render(scene, cam, w, h, mode=2, depth=2, spp=spp, seed=5, materials=mats, tri_material=tm)
    assert np.all(ref["prim"] <= 1)  # every primary ray ends on the floor
    _mode_c_statistic(clpt, ref["rgba"], w, h, spp)


# --------------------------------------------------------------------------------------- GPU tests
@pytest.fixture
def replay_renderer(renderer, clpt):
    renderer.clear_instance_meshes()
    yield renderer
    renderer.clear_instance_meshes()
    renderer.set_instance_traversal("list")
    renderer.set_materials(np.zeros((0, 8), dtype=f32))
    clpt.lib().CLSetEngine(0)
    renderer.set_params(mode=0, depth=2)


@pytest.mark.gpu
@pytest.mark.parametrize("run", RUNS, ids=_ids)
def test_cuda_matches_replay(clpt, replay_renderer, run):
    """CUDA frames on both engines, and under the instance list and the instance tree, against the
    replay; the sheared and mirrored cases also against the oracle bit for bit, so that a replay
    mismatch there tells a kernel bug from a definition bug."""
    from clpathtracer_b200 import scenes

    name, mode, depth, spp = run
    r = replay_renderer
    L = clpt.lib()
    rep, cam = _replay(clpt, run)
    base, tm, _, how, inst = _case(name)
    tree = clpt.build_kd_sah(*base) if how == "sah" else clpt.build_kd(*base)
    r.set_meshes(tree)
    handles = {m: r.add_instance_mesh(*_mesh(m)) for m in sorted({m for m, _, _ in inst})}
    if inst:
        r.set_instances([(handles[m], o2w, mat) for m, o2w, mat in inst])
    oracle_inst = [(r.download_instance_kd(handles[m]), clpt.world_to_object(o2w), mat) for m, o2w, mat in inst]
    kw = _render_kw(run)
    if mode == 2:
        r.set_materials(scenes.CORNELL_MATERIALS, kw["tri_material"])
    r.set_camera_matrix(cam)
    r.create_image(W, H)
    r.set_params(mode=mode, depth=depth, spp=spp, seed=SEED, flags=kw["flags"])
    for traversal in ("list", "tree") if inst else ("list",):
        r.set_instance_traversal(traversal)
        exact = None
        if name in ("shear", "mirror"):
            exact = ot.render(tree, cam, W, H, instances=oracle_inst,
                              tree=r.instance_tree() if traversal == "tree" else None, aov=False, **kw)["rgba"]
        for engine in (1, 2):
            L.CLSetEngine(engine)
            r.execute()
            assert L.CLLastEngine() == engine
            img = r.read_image()
            _compare(rep, img, run, "cuda %s %s engine %d" % (_ids(run), traversal, engine))
            if exact is not None:
                assert np.array_equal(img.view(np.uint32), exact.view(np.uint32)), (traversal, engine)


@pytest.mark.gpu
def test_cuda_mode_c_is_the_form_factor(clpt, replay_renderer):
    """The CUDA mode C estimate is unbiased, at 4,096 samples per pixel: the >= 64 spp launch that
    spreads one pixel's samples over several warps."""
    verts, corners, tm, mats = _floor_scene()
    r = replay_renderer
    w, h, spp = 128, 96, 4096
    r.set_meshes(clpt.build_kd(verts, corners))
    r.set_materials(mats, tm)
    r.set_camera_matrix(clpt.cam_matrix(clpt.make_camera(**FLOOR_CAMERA), h))
    r.create_image(w, h)
    r.set_params(mode=2, depth=2, spp=spp, seed=5)
    for engine in (1, 2):
        clpt.lib().CLSetEngine(engine)
        r.execute()
        _mode_c_statistic(clpt, r.read_image(), w, h, spp)
