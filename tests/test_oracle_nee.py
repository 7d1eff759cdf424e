"""Light sampling (mode 3) in the CPU restatement (oracle/oracle_nee.c).

The emitter table's twin is checked for order, integer weights, selection boundaries and the
degenerate cases; mode 3 against mode 2 where nothing is light-sampled (bit for bit) and where
lights are (in expectation); the shadow-ray query against a float64 brute force; and the
estimator against the analytic floor of tests/test_replay64.py, with and without an occluder.
"""
import numpy as np
import pytest

from oracle import oracle_instance_tree_py as ot
from oracle import oracle_instances_py as oi
from oracle import oracle_nee_py as on
from test_oracle_instance_tree import separated_grid, w2o_of
from test_oracle_instances import INSTANCES, _o2w, _world_tris
from test_replay64 import A_FLOOR, E_LIGHT, FLOOR_CAMERA, H_LIGHT, LIGHT, _floor_scene, all_rejected, form_factor

f32 = np.float32


def twin_reference(scene, materials, tri_material):
    """The table by its definition, in numpy: emitters, float64 weights, integer weights."""
    listed = np.zeros(scene.n_tris, dtype=bool)
    for nd in scene.nodes[scene.nodes["type"] == 1]:
        if nd["a"] != -1:
            listed[scene.tri_indices[nd["a"]:nd["a"] + nd["b"]]] = True
    m = np.zeros(scene.n_tris, dtype=np.int64) if tri_material is None else np.asarray(tri_material, dtype=np.int64)
    m = np.where((m < 0) | (m >= len(materials)), 0, m)
    em = materials[m, 4:7]
    ids = np.flatnonzero(listed & (em != 0).any(1))
    v = scene.verts[scene.tris[:, 0], :3].reshape(-1, 3, 3)[ids]
    e1, e2 = (v[:, 1] - v[:, 0]).astype(np.float64), (v[:, 2] - v[:, 0]).astype(np.float64)
    c = np.cross(e1, e2)
    area = 0.5 * np.sqrt((c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]) + c[:, 2] * c[:, 2])
    e = em[ids].astype(np.float64)
    w = area * ((e[:, 0] + e[:, 1]) + e[:, 2])
    w = np.where((w > 0) & np.isfinite(w), w, 0.0)
    q = (w / w.max() * 2.0 ** 32).astype(np.uint64) if len(w) and w.max() > 0 else np.zeros(len(w), np.uint64)
    return ids, area, q


def check_table(scene, materials, tri_material, tab):
    ids, area, q = twin_reference(scene, materials, tri_material)
    n, Q = int(tab["header"][0]), int(tab["header"][1])
    assert n == len(ids) and Q == int(q.sum())
    rec = tab["records"]
    assert np.array_equal(rec["prim"], ids)
    assert np.array_equal(tab["cdf"], np.concatenate([[0], np.cumsum(q)[:-1]]).astype(np.uint64) if n else tab["cdf"])
    expect_map = np.full(scene.n_tris, -1, dtype=np.int32)
    expect_map[ids] = np.arange(n)
    assert np.array_equal(tab["map"], expect_map)
    pa = np.where(q > 0, (q.astype(np.float64) / Q / area).astype(f32) if Q else 0, 0).astype(f32)
    assert np.array_equal(rec["pa"], pa)
    v = scene.verts[scene.tris[:, 0], :3].reshape(-1, 3, 3)[ids]
    assert np.array_equal(rec["v0"], v[:, 0]) and np.array_equal(rec["e1"], v[:, 1] - v[:, 0])
    assert (rec["pad0"] == 0).all() and (rec["pad1"] == 0).all()
    return q


def test_emitter_table_twin(clpt):
    """Cornell box: the ceiling's 200 triangles in ascending id, integer weights and sums, the map,
    the area pdf; every boundary of the integer search selects the emitter that owns it."""
    from clpathtracer_b200 import scenes

    v, c, nn, tm = scenes.cornell(10)
    scene = clpt.build_kd(v, c, nn)
    tab = on.build_emitters(scene, scenes.CORNELL_MATERIALS, tm)
    q = check_table(scene, scenes.CORNELL_MATERIALS, tm, tab)
    assert len(q) == 200 and (q > 0).all()
    check_selection(tab, q)
    # A table with Q = 2^32, where the target is the word itself and every boundary is hit exactly,
    # zero weights included (first, inside and last)
    q = np.array([0, 2 ** 30, 0, 2 ** 31, 0, 2 ** 30 - 1, 1, 0], dtype=np.uint64)
    cdf = np.concatenate([[0], np.cumsum(q)]).astype(np.uint64)
    check_selection({"cdf": cdf[:-1], "_cdf_full": cdf, "header": np.array([len(q), 2 ** 32], dtype=np.uint64)}, q)


def check_selection(tab, q):
    """The oracle's selection (oracle_select_emitter, the search the light sample runs) on every
    32-bit word at a boundary: the first word of each emitter's range and the word before it, against
    an integer search on the prefix sums.  Every emitter with q > 0 owns its range and nothing else."""
    cdf, Q = [int(x) for x in tab["cdf"]], int(tab["header"][1])
    first = [-(-(c << 32) // Q) for c in cdf]  # the smallest word r with (r * Q) >> 32 >= cdf[i]
    words = sorted({r for x in first for r in (x - 1, x) if 0 <= r < 2 ** 32} | {0, 2 ** 32 - 1})
    want = np.searchsorted(tab["cdf"], np.array([(r * Q) >> 32 for r in words], dtype=np.uint64), side="right") - 1
    got = on.select(tab, words)
    assert np.array_equal(got, want)
    assert (q[got] > 0).all()
    owner = dict(zip(words, got))
    for i, r in enumerate(first):
        if q[i] > 0:
            assert owner[r] == i and (r == 0 or owner[r - 1] < i), i


def test_emitter_table_zero_weight_and_all_emit(clpt):
    """A tiny emitter whose weight rounds to 0 stays in the table with pdf 0 (reached by bounces
    only); a scene where every triangle emits maps every primitive."""
    from clpathtracer_b200 import scenes

    verts, corners, tm, mats = _floor_scene()
    verts = np.concatenate([verts, np.array([[0, 1, 0], [1e-6, 1, 0], [0, 1, 1e-6]], dtype=f32)])
    corners = np.concatenate([corners, clpt.corners_from_faces(np.array([[8, 10, 9]]), False)])
    tm = np.concatenate([tm, [1]]).astype(np.int32)
    scene = clpt.build_kd(verts, corners)
    tab = on.build_emitters(scene, mats, tm)
    q = check_table(scene, mats, tm, tab)
    assert len(q) == 3 and q[2] == 0 and tab["records"]["pa"][2] == 0 and tab["map"][4] == 2
    check_selection(tab, q)  # the zero-weight emitter is never selected

    v, c, nn = scenes.heightfield(22, False)
    scene = clpt.build_kd(v, c, nn)
    mats = scenes.CORNELL_MATERIALS[3:]
    tab = on.build_emitters(scene, mats, None)
    check_table(scene, mats, None, tab)
    assert np.array_equal(tab["map"], np.arange(scene.n_tris))
    # no materials: nothing emits
    assert int(on.build_emitters(scene)["header"][0]) == 0


def unlisted_emitter_scene(clpt):
    """The analytic floor's scene plus an emissive triangle (primitive 4) that tri_indices holds past
    the leaves' runs: no leaf lists it, so no ray can hit it and it must not be light-sampled."""
    verts, corners, tm, mats = _floor_scene()
    scene = clpt.build_kd(verts, corners)
    verts = np.concatenate([verts, np.array([[0.2, 0.4, 0.2], [0.4, 0.4, 0.2], [0.2, 0.4, 0.4]], dtype=f32)])
    corners = np.concatenate([corners, clpt.corners_from_faces(np.array([[8, 9, 10]]), False)])
    v4 = np.zeros((len(verts), 4), dtype=f32)
    v4[:, :3] = verts
    out = clpt.Scene(scene.nodes, np.concatenate([scene.tri_indices, [4]]), corners, v4, scene.norms)
    return out, np.concatenate([tm, [1]]).astype(np.int32), mats


def test_emitter_table_lists_leaves_only(clpt):
    scene, tm, mats = unlisted_emitter_scene(clpt)
    tab = on.build_emitters(scene, mats, tm)
    check_table(scene, mats, tm, tab)
    assert list(tab["records"]["prim"]) == [2, 3] and tab["map"][4] == -1


def _same(a, b, keys=("rgba", "prim", "t", "uv", "normal")):
    for key in keys:
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"] == b["counters"]


@pytest.mark.parametrize("case", ["hf22", "cornell_dark", "instances"])
def test_without_emitters_mode3_is_mode2(clpt, case):
    """Nothing light-sampled: the mode-3 frame, AOVs and counters are mode 2's bit for bit (the
    instance case has an emissive instance, which is never light-sampled)."""
    from clpathtracer_b200 import scenes

    w, h = 64, 48
    kw = dict(depth=4, spp=2, seed=9, flags=1)
    inst = ()
    if case == "hf22":
        scene = clpt.build_kd(*scenes.heightfield(22, False))
        cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), h)
    else:
        v, c, nn, tm = scenes.cornell(6)
        scene = clpt.build_kd(v, c, nn)
        mats = scenes.CORNELL_MATERIALS.copy()
        mats[3, 4:7] = 0
        cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), h)
        kw.update(materials=mats, tri_material=tm)
        if case == "instances":
            sv, sf = __import__("bench").icosphere(2)
            sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, False), None)
            inst = [(sphere, clpt.world_to_object(_o2w((0.2, 0.1, 0), (0.3, 0.3, 0.3), (0.3, 0.0, 0.2))), 1),
                    (sphere, clpt.world_to_object(_o2w((0, 0, 0), (0.2, 0.2, 0.2), (-0.4, 0.5, 0.3))), 3)]
            kw["materials"] = scenes.CORNELL_MATERIALS.copy()
            kw["materials"][0, 4:7] = 0
            kw["tri_material"] = np.where(tm == 3, 0, tm).astype(np.int32)
    m2 = oi.render(scene, cam, w, h, mode=2, instances=inst, **kw)
    m3 = on.render(scene, cam, w, h, instances=inst, **kw)
    assert int(on.build_emitters(scene, kw.get("materials"), kw.get("tri_material"))["header"][1]) == 0
    _same(m2, m3)
    if case != "hf22":
        assert (m3["rgba"][..., 0] > 0).mean() > 0.3


def _shadow_rays(rng, n, lo, hi):
    o = rng.uniform(lo, hi, (n, 3))
    t = rng.uniform(lo, hi, (n, 3))
    d = t - o
    dist = np.linalg.norm(d, axis=1)
    rays = np.zeros((n, 7), dtype=f32)
    rays[:, :3] = o
    rays[:, 3:6] = d / dist[:, None]
    rays[:, 6] = dist
    return rays


def _any_hit64(rays, tris):
    """float64 any-hit with back faces culled, and whether every triangle is clearly on one side."""
    o, d, tmax = rays[:, :3].astype(np.float64), rays[:, 3:6].astype(np.float64), rays[:, 6].astype(np.float64)
    v0, e1, e2 = tris[:, 0], tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0]
    scale = np.linalg.norm(np.cross(e1, e2), axis=1)
    hit = np.zeros(len(rays), bool)
    clear = np.ones(len(rays), bool)
    for s in range(0, len(rays), 256):
        dd, oo, tm = d[s:s + 256, None], o[s:s + 256, None], tmax[s:s + 256, None]
        p = np.cross(dd, e2[None])
        det = (e1[None] * p).sum(-1)
        with np.errstate(divide="ignore", invalid="ignore"):
            tv = oo - v0[None]
            u = (tv * p).sum(-1) / det
            q = np.cross(tv, e1[None])
            v = (dd * q).sum(-1) / det
            t = (e2[None] * q).sum(-1) / det
        m = np.minimum(np.minimum(u, v), 1 - u - v)
        inside = (det > 0) & (m >= 0) & (t > 0) & (t < tm)
        hit[s:s + 256] = inside.any(1)
        grazing = np.abs(det) < 1e-3 * scale[None]
        near_edge = (np.abs(m) < 1e-4) & (t > -1e-3) & (t < tm * (1 + 1e-3))
        near_end = (m > -1e-4) & ((np.abs(t) < 1e-3) | (np.abs(t - tm) < 1e-3 * tm))
        clear[s:s + 256] = ~(((grazing & (m > -1e-3)) | near_edge | near_end).any(1))
    return hit, clear


def test_occlusion_matches_float64_any_hit(clpt):
    """The shadow-ray query over the terrain and three sphere instances against a float64 brute force
    over every world triangle, on the well-conditioned rays; the list and the tree agree everywhere."""
    from clpathtracer_b200 import scenes

    base = clpt.build_kd(*scenes.heightfield(22, False))
    sv, sf = __import__("bench").icosphere(2)
    sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, False), None)
    o2w = [_o2w(*p) for p in INSTANCES]
    inst = [(sphere, clpt.world_to_object(m), 0) for m in o2w]
    rays = _shadow_rays(np.random.default_rng(3), 6000, -0.8, 0.6)
    occ = on.occluded(base, rays, instances=inst)
    occ_tree = on.occluded(base, rays, instances=inst, tree=ot.tree_of(inst))
    assert np.array_equal(occ, occ_tree)
    tris = np.concatenate([_world_tris(base)] + [_world_tris(sphere, m) for m in o2w])
    hit, clear = _any_hit64(rays, tris)
    assert clear.mean() > 0.9 and 0.2 < hit[clear].mean() < 0.8
    assert np.array_equal(occ[clear], hit[clear])
    base_only = on.occluded(base, rays)
    assert (occ & ~base_only).sum() > 100  # the instances occlude rays the terrain does not


# ------------------------------------------------------------------ the analytic floor
OCCLUDER = (0.15, 0.75, -0.75, -0.15, 0.1)  # x0, x1, z0, z1, height: an instance quad facing -y, emission 1


def _floor_with_occluder(clpt):
    verts, corners, tm, mats = _floor_scene()
    scene = clpt.build_kd(verts, corners)
    x0, x1, z0, z1, hy = OCCLUDER
    qv = np.array([[x0, hy, z0], [x0, hy, z1], [x1, hy, z1], [x1, hy, z0]], dtype=f32)
    quad = clpt.build_kd(qv, clpt.corners_from_faces(np.array([[0, 2, 1], [0, 3, 2]]), False), None)
    ident = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]], dtype=f32)
    mats = np.concatenate([mats, np.zeros((1, 8), dtype=f32)])
    mats[2, 4:7] = 1.0  # a hit on it adds a * 1: the same as the miss it replaces
    return scene, tm, mats, [(quad, ident, 2)]


def floor_expectation(clpt, w, h):
    """Per pixel: the expected colour and whether the pixel is fully shadowed, fully clear of the
    occluder, or neither.  Shadowed pixels see the occluder cover the whole emitter."""
    from test_replay64 import primary_rays

    cam = clpt.cam_matrix(clpt.make_camera(**FLOOR_CAMERA), h)
    o, d, _, _ = primary_rays(cam, w, h, 1, 0, False)
    t = -o[:, 1] / d[:, 1]
    x = o + t[:, None] * d
    lx0, lx1, lz0, lz1 = LIGHT
    ox0, ox1, oz0, oz1, hy = OCCLUDER
    s = hy / H_LIGHT  # the emitter seen from x, projected onto the occluder's plane
    px0, px1 = x[:, 0] + (lx0 - x[:, 0]) * s, x[:, 0] + (lx1 - x[:, 0]) * s
    pz0, pz1 = x[:, 2] + (lz0 - x[:, 2]) * s, x[:, 2] + (lz1 - x[:, 2]) * s
    m = 1e-3
    shadowed = (px0 > ox0 + m) & (px1 < ox1 - m) & (pz0 > oz0 + m) & (pz1 < oz1 - m)
    clear = (px1 < ox0 - m) | (px0 > ox1 + m) | (pz1 < oz0 - m) | (pz0 > oz1 + m)
    under = (x[:, 0] > lx0) & (x[:, 0] < lx1) & (x[:, 2] > lz0) & (x[:, 2] < lz1)
    p = all_rejected()
    P = (1 - p) * form_factor(x[:, 0], x[:, 2]) + p * under
    expected = np.where(shadowed, A_FLOOR, A_FLOOR + A_FLOOR * (E_LIGHT - 1) * P)
    return cam, expected, shadowed, clear


def nee_floor_statistic(frames, expected, shadowed, clear, label):
    """frames float[K, pixels]: K independent frame means per pixel.  z of each pixel's mean against
    its expectation with the frames' own spread; t-distributed with K - 1 degrees of freedom."""
    K = len(frames)
    mean = frames.mean(0)
    sd = frames.std(0, ddof=1)
    assert np.all(frames[:, shadowed] == A_FLOOR)  # every sample of a shadowed pixel is exactly a
    use = clear & (sd > 0)
    z = (mean[use] - expected[use]) / (sd[use] / np.sqrt(K))
    n = len(z)
    var_t = (K - 1) / (K - 3)
    line = "%s: %d clear pixels, %d shadowed, K = %d: mean z %+.4f (bar %.4f), mean z^2 %.4f (bar %.3f +- %.4f), max |z| %.2f" % (
        label, n, shadowed.sum(), K, z.mean(), 5 / np.sqrt(n), (z * z).mean(), var_t, 8 * np.sqrt(2 / n), np.abs(z).max())
    print(line)
    assert n > 0.3 * len(expected) and shadowed.sum() > 20
    assert abs(z.mean()) < 5 / np.sqrt(n), line
    assert abs((z * z).mean() - var_t) < 8 * np.sqrt(2 / n), line
    assert np.abs(z).max() < 7, line


def test_mode3_is_the_form_factor(clpt):
    """The oracle's mode-3 estimate has mode 2's expectation on the analytic floor at depth 2 (the
    formula of test_replay64), and exactly a where the occluder hides the whole emitter; it is far
    less noisy than mode 2 with the same seeds."""
    scene, tm, mats, inst = _floor_with_occluder(clpt)
    w, h, spp, K = 48, 36, 32, 48
    cam, expected, shadowed, clear = floor_expectation(clpt, w, h)
    f3, f2 = [], []
    for k in range(K):
        kw = dict(depth=2, spp=spp, seed=100 + k, materials=mats, tri_material=tm, instances=inst, aov=False)
        f3.append(on.render(scene, cam, w, h, **kw)["rgba"][..., 0].reshape(-1).astype(np.float64))
        f2.append(oi.render(scene, cam, w, h, mode=2, **kw)["rgba"][..., 0].reshape(-1).astype(np.float64))
    f3, f2 = np.array(f3), np.array(f2)
    nee_floor_statistic(f3, expected, shadowed, clear, "mode 3 oracle %dx%d, %d x %d spp" % (w, h, K, spp))
    ratio = f2[:, clear].var(0, ddof=1).sum() / f3[:, clear].var(0, ddof=1).sum()
    print("variance ratio mode 2 / mode 3 on the clear pixels: %.3f" % ratio)
    assert ratio > 2.0  # observed 2.33: the miss (a) stays a coin flip, only the emitter term is smoothed


def test_mode3_matches_mode2_on_small_light(clpt):
    """cornell_small_light, both boxes occluding: per-region means of modes 2 and 3 agree within their
    statistical bars at matched samples (8 seeds each); mode 3's regions are less noisy."""
    from clpathtracer_b200 import scenes

    v, c, nn, tm = scenes.cornell_small_light(6)
    scene = clpt.build_kd(v, c, nn)
    w, h, spp, K = 48, 36, 64, 8
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), h)
    kw = dict(depth=4, spp=spp, flags=1, materials=scenes.CORNELL_SMALL_LIGHT_MATERIALS, tri_material=tm, aov=False)

    def regions(img):
        return img[..., :3].sum(-1).reshape(6, h // 6, 8, w // 8).mean((1, 3)).reshape(-1)

    r2 = np.array([regions(oi.render(scene, cam, w, h, mode=2, seed=k, **kw)["rgba"]) for k in range(K)])
    r3 = np.array([regions(on.render(scene, cam, w, h, seed=50 + k, **kw)["rgba"]) for k in range(K)])
    se = np.sqrt(r2.var(0, ddof=1) / K + r3.var(0, ddof=1) / K)
    z = (r3.mean(0) - r2.mean(0)) / se
    print("small light: region z max |z| %.2f, mean z^2 %.3f; noise ratio %.2f" % (
        np.abs(z).max(), (z * z).mean(), r2.std(0).mean() / r3.std(0).mean()))
    assert np.abs(z).max() < 5.5 and (z * z).mean() < 2.5
    assert r2.std(0).mean() > 2 * r3.std(0).mean()


@pytest.mark.parametrize("depth,spp", [(3, 1), (4, 4)])
def test_tree_equals_list_in_mode3(clpt, oracle, depth, spp):
    """Separated instances over a terrain with emissive base triangles: the list and the tree give
    the same mode-3 frame bit for bit (shadow rays are answered the same way under both)."""
    from clpathtracer_b200 import scenes

    v, c, n = scenes.heightfield(22, True)
    base = clpt.build_kd(v, c, n)
    sv, sf = __import__("bench").icosphere(2)
    sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, True), sv)
    inst = [(sphere, m, k % 3) for k, m in enumerate(w2o_of(clpt, separated_grid(clpt)))]
    tm = (np.arange(base.n_tris) % 37 == 0).astype(np.int32) * 3
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 72)
    kw = dict(depth=depth, spp=spp, seed=2, flags=oracle.FLAG_JITTER if spp > 1 else 0,
              materials=scenes.CORNELL_MATERIALS, tri_material=tm, instances=inst)
    a = on.render(base, cam, 96, 72, **kw)
    b = on.render(base, cam, 96, 72, tree=ot.tree_of(inst), **kw)
    for key in ("rgba", "prim", "t", "uv", "normal"):
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"]["rays"] == b["counters"]["rays"]
    m2 = oi.render(base, cam, 96, 72, mode=2, **kw)
    assert a["counters"]["rays"] > m2["counters"]["rays"]  # shadow rays were cast
