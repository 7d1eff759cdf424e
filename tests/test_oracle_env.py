"""Environment lighting (modes 2 and 3) in the CPU restatement (oracle/oracle_env.c).

The lookup is checked on texel centres, axes and exact ties and against a float64 face selection;
the table's twin against a numpy float64 restatement byte for byte; the pdf by quadrature and by
Monte Carlo; frames against the existing mode-2 restatements where nothing may change (bit for bit);
and both modes against the analytic expectation of a diffuse floor under a sun and sky, with an
occluder that hides the sun from part of the floor.
"""
import numpy as np
import pytest

from clpathtracer_b200 import envmap
from oracle import oracle_env_py as oe
from oracle import oracle_instance_tree_py as ot
from test_oracle_instance_tree import separated_grid, w2o_of
from test_replay64 import FLOOR_CAMERA, all_rejected

f32 = np.float32
A_FLOOR = 0.5
SUN_DIR = (0.3, 1.0, 0.2)               # on the +Y face: a = 0.3, b = 0.2
OCCLUDER = (-0.4, 0.2, -0.5, 0.1, 0.3)  # x0, x1, z0, z1, height: an instance quad facing -y


# ------------------------------------------------------------------ lookup
@pytest.mark.parametrize("n", [1, 3, 8])
def test_texel_centres_look_up_their_texel(n):
    d = envmap.texel_directions(n)[:, :, :, 0].reshape(-1, 3).astype(f32)
    texel, a, b = oe.lookup(n, d)
    assert np.array_equal(texel, np.arange(6 * n * n))
    assert np.array_equal(texel, envmap.lookup(d, n))


def test_axes_and_exact_ties():
    n = 4
    cases = {  # direction: (face, a, b)
        (1, 0, 0): (0, 0, 0), (-1, 0, 0): (1, 0, 0), (0, 1, 0): (2, 0, 0), (0, -1, 0): (3, 0, 0),
        (0, 0, 1): (4, 0, 0), (0, 0, -1): (5, 0, 0),
        (1, 1, 0): (0, 0, -1), (1, 0, 1): (0, -1, 0), (1, 1, 1): (0, -1, -1), (-1, -1, -1): (1, -1, 1),
        (0, 1, 1): (2, 0, 1), (0, -1, -1): (3, 0, 1), (0, 1, -1): (2, 0, -1), (-1, 1, 0): (1, 0, -1),
        (0.5, 0, 0.5): (0, -1, 0), (-0.0, 0, -1): (5, 0, 0), (0, -0.0, 1): (4, 0, 0),
    }
    d = np.array(list(cases), dtype=f32)
    texel, a, b = oe.lookup(n, d)
    for k, (face, wa, wb) in enumerate(cases.values()):
        col, row = min(n - 1, int((wa + 1) * 0.5 * n)), min(n - 1, int((wb + 1) * 0.5 * n))
        assert (a[k], b[k]) == (wa, wb), d[k]
        assert texel[k] == (face * n + row) * n + col, d[k]


def test_lookup_agrees_with_float64():
    """10^5 random directions: the fp32 lookup and a float64 face selection agree except within
    rounding of a texel edge (or of a face-selection tie)."""
    rng = np.random.default_rng(5)
    n = 16
    d = rng.normal(size=(100_000, 3)).astype(f32)
    texel, _, _ = oe.lookup(n, d)
    want = envmap.lookup(d, n)
    d64 = d.astype(np.float64)
    ab = np.sort(np.abs(d64), axis=1)
    ma = ab[:, 2]
    tie = (ab[:, 2] - ab[:, 1]) < 1e-6 * ma
    # distance of the float64 face coordinates to the nearest texel edge, in texels
    frac = ((d64 / ma[:, None] + 1) * 0.5 * n) % 1.0
    minor = np.ones(d.shape, dtype=bool)
    minor[np.arange(len(d)), np.abs(d64).argmax(1)] = False
    near = ((np.minimum(frac, 1 - frac) < 1e-4) & minor).any(1)
    ok = ~(tie | near)
    assert ok.mean() > 0.99
    assert np.array_equal(texel[ok], want[ok])


def _sun_sky(n=8, sun=400.0):
    from clpathtracer_b200 import scenes
    return scenes.sun_sky(n, SUN_DIR, 0.0, sun, 1.0, 0.3)


def test_samples_look_up_their_texel():
    rng = np.random.default_rng(2)
    cube = rng.uniform(0, 1, (6, 16, 16, 3)).astype(f32)
    cube[2, 3, 4] = 500
    tab = oe.build_env(cube)
    words = rng.integers(0, 2 ** 32, (100_000, 3), dtype=np.uint64).astype(np.uint32)
    texel, a, b, l, pe = oe.draw(tab, words)
    assert (tab["texels"][texel, 3] > 0).all()
    back, _, _ = oe.lookup(16, l)
    assert (back != texel).mean() < 1e-3
    # the bright texel is drawn in proportion to its weight
    q = np.diff(tab["_cdf_full"]).astype(np.float64)
    i = (2 * 16 + 3) * 16 + 4
    share = (texel == i).mean()
    assert abs(share - q[i] / q.sum()) < 5 * np.sqrt(share * (1 - share) / len(texel))


# ------------------------------------------------------------------ the table
def table_reference(cube):
    """The table by its definition, in numpy float64: texels, cdf, header."""
    cube = np.asarray(cube, dtype=f32)
    n = cube.shape[1]
    k = (np.arange(n, dtype=np.float64) + 0.5) / n * 2 - 1
    bc, ac = np.meshgrid(k, k, indexing="ij")
    s2 = (1 + ac * ac) + bc * bc
    c = cube.astype(np.float64)
    w = ((c[..., 0] + c[..., 1]) + c[..., 2]) / (s2 * np.sqrt(s2))[None]
    w = np.where((w > 0) & np.isfinite(w), w, 0.0).reshape(-1)
    q = (w / w.max() * 2.0 ** 32).astype(np.uint64) if w.max() > 0 else np.zeros(len(w), np.uint64)
    Q = int(q.sum())
    cdf = np.concatenate([[0], np.cumsum(q)[:-1]]).astype(np.uint64)
    tex = np.zeros((len(w), 4), dtype=f32)
    tex[:, :3] = cube.reshape(-1, 3)
    with np.errstate(invalid="ignore", divide="ignore"):
        pdf = ((q.astype(np.float64) / float(np.float64(Q))) * (float(n) * float(n))) * 0.25
    tex[:, 3] = np.where(q > 0, pdf, 0).astype(f32)
    return tex, cdf, np.array([n, Q], dtype=np.uint64), q


def _cubes():
    rng = np.random.default_rng(11)
    one_hot = np.zeros((6, 5, 5, 3), dtype=f32)
    one_hot[4, 1, 3, 1] = 7.0
    return {"uniform": np.ones((6, 4, 4, 3), dtype=f32), "one_hot": one_hot,
            "zero": np.zeros((6, 3, 3, 3), dtype=f32), "random": rng.exponential(1.0, (6, 9, 9, 3)).astype(f32),
            "sun_sky": _sun_sky(16), "n1": rng.uniform(0, 2, (6, 1, 1, 3)).astype(f32)}


@pytest.mark.parametrize("case", ["uniform", "one_hot", "zero", "random", "sun_sky", "n1"])
def test_table_twin_equals_float64_restatement(case):
    cube = _cubes()[case]
    tab = oe.build_env(cube)
    tex, cdf, hdr, q = table_reference(cube)
    assert np.array_equal(tab["header"], hdr)
    assert tab["texels"].tobytes() == tex.tobytes()
    assert tab["cdf"].tobytes() == cdf.tobytes()
    assert int(tab["_cdf_full"][-1]) == int(hdr[1])
    if case == "zero":
        assert int(hdr[1]) == 0 and (tab["texels"][:, 3] == 0).all()
    if case == "one_hot":
        assert (q > 0).sum() == 1 and int(hdr[1]) == 2 ** 32


def test_pdf_integrates_to_the_selection_probability():
    """Per texel, the float64 integral of pe x (d omega / dA) over the texel (Gauss-Legendre) is
    q / Q; the texels' exact solid angles add up to 4 pi; uniform directions give mean pe 4 pi = 1."""
    rng = np.random.default_rng(4)
    n = 6
    cube = rng.exponential(1.0, (6, n, n, 3)).astype(f32)
    cube[0, 2, 2] = 300
    tab = oe.build_env(cube)
    q = np.diff(tab["_cdf_full"]).astype(np.float64)
    Q = float(tab["header"][1])
    x, wq = np.polynomial.legendre.leggauss(8)
    h = 1.0 / n
    k = np.arange(n)
    a = (2 * k[:, None] + 1 + x[None]) * h - 1       # [col, node]
    A, B = np.meshgrid(a.reshape(-1), a.reshape(-1), indexing="ij")  # B rows, A cols
    s2 = 1 + A * A + B * B
    jac = (s2 ** -1.5).reshape(n, 8, n, 8).transpose(0, 2, 1, 3)      # [row, col, node_b, node_a]
    wts = (wq[:, None] * wq[None, :]) * h * h
    pdf = tab["texels"][:, 3].astype(np.float64).reshape(6, n, n)
    pe_jac = pdf[:, :, :, None, None] * (s2 ** 1.5).reshape(n, 8, n, 8).transpose(0, 2, 1, 3)[None] * jac[None]
    integral = (pe_jac * wts[None, None, None]).sum((3, 4)).reshape(-1)
    assert np.allclose(integral, q / Q, rtol=1e-6, atol=0)
    omega = (jac * wts[None, None]).sum((2, 3))
    corner = np.arange(n + 1) / n * 2 - 1
    ca, cb = np.meshgrid(corner, corner, indexing="xy")
    F = np.arctan(ca * cb / np.sqrt(1 + ca * ca + cb * cb))
    exact = F[1:, 1:] - F[1:, :-1] - F[:-1, 1:] + F[:-1, :-1]
    assert np.allclose(omega, exact, rtol=1e-9) and abs(6 * exact.sum() - 4 * np.pi) < 1e-12
    d = rng.normal(size=(400_000, 3)).astype(f32)
    texel, ta, tb = oe.lookup(n, d)
    s = (1 + ta.astype(np.float64) ** 2) + tb.astype(np.float64) ** 2
    pe = tab["texels"][texel, 3].astype(np.float64) * s ** 1.5 * 4 * np.pi
    assert abs(pe.mean() - 1) < 5 * pe.std() / np.sqrt(len(pe))


# ------------------------------------------------------------------ frames that must not change
def _same(a, b, keys=("rgba", "prim", "t", "uv", "normal")):
    for key in keys:
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"] == b["counters"]


@pytest.mark.parametrize("traversal", [None, "list", "tree"])
def test_all_ones_environment_is_the_white_sky(clpt, oracle, traversal):
    """Mode 2 with an all-ones environment is mode 2 without one bit for bit (x * 1 is exact); mode 3
    with an all-zero environment and no emitters is mode 2 with the same environment."""
    from clpathtracer_b200 import scenes

    v, c, n = scenes.heightfield(22, True)
    base = clpt.build_kd(v, c, n)
    inst, tree = (), None
    if traversal is not None:
        sv, sf = __import__("bench").icosphere(2)
        sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, True), sv)
        inst = [(sphere, m, k % 3) for k, m in enumerate(w2o_of(clpt, separated_grid(clpt)))]
        tree = ot.tree_of(inst) if traversal == "tree" else None
    mats = scenes.CORNELL_MATERIALS.copy()
    mats[3, 4:7] = 0
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 48)
    kw = dict(depth=4, spp=2, seed=3, flags=oracle.FLAG_JITTER, materials=mats,
              tri_material=(np.arange(base.n_tris) % 5 == 0).astype(np.int32), instances=inst, tree=tree)
    ones = np.ones((6, 3, 3, 3), dtype=f32)
    ref = ot.render(base, cam, 64, 48, mode=2, **kw)
    _same(oe.render(base, cam, 64, 48, ones, mode=2, **kw), ref)
    zero = np.zeros((6, 3, 3, 3), dtype=f32)
    _same(oe.render(base, cam, 64, 48, zero, mode=3, **kw), oe.render(base, cam, 64, 48, zero, mode=2, **kw))
    # an environment that is not all ones changes the misses only
    sky = oe.render(base, cam, 64, 48, _sun_sky(), mode=2, **kw)
    _same(sky, ref, keys=("prim", "t", "uv", "normal"))
    assert not np.array_equal(sky["rgba"], ref["rgba"])


def test_mode3_samples_the_environment(clpt, oracle):
    """Mode 3 casts one shadow ray per diffuse vertex to the environment (on top of the emitter
    sample's), and the list and the tree give the same frame."""
    from clpathtracer_b200 import scenes

    v, c, n = scenes.heightfield(22, True)
    base = clpt.build_kd(v, c, n)
    sv, sf = __import__("bench").icosphere(2)
    sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, True), sv)
    inst = [(sphere, m, k % 3) for k, m in enumerate(w2o_of(clpt, separated_grid(clpt)))]
    tm = (np.arange(base.n_tris) % 37 == 0).astype(np.int32) * 3
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 48)
    kw = dict(depth=3, spp=2, seed=2, flags=oracle.FLAG_JITTER, materials=scenes.CORNELL_MATERIALS,
              tri_material=tm, instances=inst)
    a = oe.render(base, cam, 64, 48, _sun_sky(), **kw)
    b = oe.render(base, cam, 64, 48, _sun_sky(), tree=ot.tree_of(inst), **kw)
    for key in ("rgba", "prim", "t", "uv", "normal"):
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"]["rays"] == b["counters"]["rays"]  # the walks differ, the answers do not
    nee = __import__("oracle.oracle_nee_py", fromlist=["render"]).render(base, cam, 64, 48, **kw)
    assert a["counters"]["rays"] > nee["counters"]["rays"]


# ------------------------------------------------------------------ the analytic floor


def env_floor_scene(clpt, sky):
    """A diffuse floor (albedo A_FLOOR) and an occluder quad instance of albedo 0 whose emission is
    the sky's radiance, so that it changes nothing but the sun it hides."""
    s = 3.0
    verts = np.array([[-s, 0, -s], [-s, 0, s], [s, 0, s], [s, 0, -s]], dtype=f32)
    scene = clpt.build_kd(verts, clpt.corners_from_faces(np.array([[0, 1, 2], [0, 2, 3]]), False))
    x0, x1, z0, z1, hy = OCCLUDER
    qv = np.array([[x0, hy, z0], [x0, hy, z1], [x1, hy, z1], [x1, hy, z0]], dtype=f32)
    quad = clpt.build_kd(qv, clpt.corners_from_faces(np.array([[0, 2, 1], [0, 3, 2]]), False), None)
    mats = np.zeros((2, 8), dtype=f32)
    mats[0, :3] = A_FLOOR
    mats[1, 4:7] = sky
    ident = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]], dtype=f32)
    return scene, np.zeros(2, dtype=np.int32), mats, [(quad, ident, 1)]


def projected_solid_angle(corners):
    """Lambert's edge formula in float64: the projected solid angle about +y of the spherical polygon
    through the directions `corners` (in order)."""
    v = np.asarray(corners, dtype=np.float64)
    v = v / np.linalg.norm(v, axis=1, keepdims=True)
    total = 0.0
    for i in range(len(v)):
        p, q = v[i], v[(i + 1) % len(v)]
        c = np.cross(p, q)
        total += np.arccos(np.clip(p @ q, -1, 1)) * c[1] / np.linalg.norm(c)
    return abs(total) / 2


def env_floor_expectation(clpt, n, sun, w, h):
    """Per pixel: the expected colour, and whether the sun texel is wholly hidden by the occluder
    (shadowed) or wholly visible (clear).  The sun is one texel of the +Y face, [a0, a1] x [b0, b1];
    from a floor point x its corner rays cross the occluder's plane at x + hy (a, 1, b), so the
    cones are rectangles there and the classification is exact."""
    from test_replay64 import primary_rays

    cam = clpt.cam_matrix(clpt.make_camera(**FLOOR_CAMERA), h)
    o, d, _, _ = primary_rays(cam, w, h, 1, 0, False)
    t = -o[:, 1] / d[:, 1]
    x = o + t[:, None] * d
    col, row = int((SUN_DIR[0] + 1) * 0.5 * n), int((SUN_DIR[2] + 1) * 0.5 * n)
    a0, a1, b0, b1 = 2 * col / n - 1, 2 * (col + 1) / n - 1, 2 * row / n - 1, 2 * (row + 1) / n - 1
    ox0, ox1, oz0, oz1, hy = OCCLUDER
    px0, px1, pz0, pz1 = x[:, 0] + hy * a0, x[:, 0] + hy * a1, x[:, 2] + hy * b0, x[:, 2] + hy * b1
    m = 1e-3
    shadowed = (px0 > ox0 + m) & (px1 < ox1 - m) & (pz0 > oz0 + m) & (pz1 < oz1 - m)
    clear = (px1 < ox0 - m) | (px0 > ox1 + m) | (pz1 < oz0 - m) | (pz0 > oz1 + m)
    # sum over the upper-hemisphere texels of L_t Phi_t / pi: sky everywhere plus the sun's excess
    # (the hemisphere's projected solid angle is pi; the horizon is a texel boundary)
    phi = projected_solid_angle([(a0, 1, b0), (a1, 1, b0), (a1, 1, b1), (a0, 1, b1)])
    p = all_rejected()
    clear_value = A_FLOOR * ((1 - p) * (1.0 + (sun - 1.0) * phi / np.pi) + p * 1.0)
    expected = np.where(shadowed, A_FLOOR * 1.0, clear_value)
    return cam, expected, shadowed, clear, phi


def test_lambert_formula_matches_quadrature():
    x, wq = np.polynomial.legendre.leggauss(32)
    a0, a1, b0, b1 = 0.25, 0.5, 0.0, 0.25
    A, B = np.meshgrid(a0 + (x + 1) / 2 * (a1 - a0), b0 + (x + 1) / 2 * (b1 - b0))
    quad = ((1 + A * A + B * B) ** -2 * np.outer(wq, wq)).sum() * (a1 - a0) * (b1 - b0) / 4
    assert abs(projected_solid_angle([(a0, 1, b0), (a1, 1, b0), (a1, 1, b1), (a0, 1, b1)]) - quad) < 1e-14


def env_floor_statistic(frames, expected, use, label):
    """frames float[K, pixels]: K independent frame means per pixel.  z of each used pixel's mean
    against its expectation with the frames' own spread (the statistic and bars of
    test_oracle_nee.nee_floor_statistic); t-distributed with K - 1 degrees of freedom."""
    K = len(frames)
    mean = frames.mean(0)
    sd = frames.std(0, ddof=1)
    use = use & (sd > 0)
    z = (mean[use] - expected[use]) / (sd[use] / np.sqrt(K))
    n = len(z)
    var_t = (K - 1) / (K - 3)
    line = "%s: %d pixels, K = %d: mean z %+.4f (bar %.4f), mean z^2 %.4f (bar %.3f +- %.4f), max |z| %.2f" % (
        label, n, K, z.mean(), 5 / np.sqrt(n), (z * z).mean(), var_t, 8 * np.sqrt(2 / n), np.abs(z).max())
    print(line)
    assert n > 0.3 * len(expected)
    assert abs(z.mean()) < 5 / np.sqrt(n), line
    assert abs((z * z).mean() - var_t) < 8 * np.sqrt(2 / n), line
    assert np.abs(z).max() < 7, line


ENV_N, SUN = 8, 400.0


def test_floor_under_sun_and_sky(clpt):
    """Both modes have the analytic expectation on the floor at depth 2, clear and shadowed pixels;
    mode 3 is far less noisy than mode 2 where the sun is visible."""
    sky = 1.0
    scene, tm, mats, inst = env_floor_scene(clpt, sky)
    w, h, K = 48, 36, 48
    cam, expected, shadowed, clear, phi = env_floor_expectation(clpt, ENV_N, SUN, w, h)
    assert shadowed.sum() > 100 and clear.sum() > 500
    env = oe.build_env(_sun_sky(ENV_N, SUN))
    frames = {2: [], 3: []}
    for k in range(K):
        for mode, spp in ((2, 256), (3, 32)):
            out = oe.render(scene, cam, w, h, env, mode=mode, depth=2, spp=spp, seed=100 + k, materials=mats,
                            tri_material=tm, instances=inst, aov=k == 0)
            if k == 0:
                assert np.all(out["prim"].reshape(-1) <= 1)  # every camera ray ends on the floor
            frames[mode].append(out["rgba"][..., 0].reshape(-1).astype(np.float64))
    f2, f3 = np.array(frames[2]), np.array(frames[3])
    use = clear | shadowed
    env_floor_statistic(f3, expected, use, "mode 3 oracle %dx%d, %d x 32 spp" % (w, h, K))
    env_floor_statistic(f2, expected, use, "mode 2 oracle %dx%d, %d x 256 spp" % (w, h, K))
    ratio = 8 * f2[:, clear].var(0, ddof=1).sum() / f3[:, clear].var(0, ddof=1).sum()
    print("variance ratio mode 2 / mode 3 per sample on the clear pixels: %.2f" % ratio)
    assert ratio > 100.0  # observed 166.5: the sun texel is found by every light sample, not by 1 bounce in 300


def test_latlong_to_cube_and_sun_sky():
    """An equirectangular image whose pixels hold their own direction resamples to a cube whose
    texels hold (close to) theirs; a constant image stays constant; sun_sky puts the sun where its
    direction looks and the horizon on a texel boundary."""
    from clpathtracer_b200 import scenes

    H, W = 256, 512
    theta = np.pi * (np.arange(H) + 0.5) / H
    phi = 2 * np.pi * (np.arange(W) + 0.5) / W
    T, P = np.meshgrid(theta, phi, indexing="ij")
    img = np.stack([np.sin(T) * np.sin(P), np.cos(T), -np.sin(T) * np.cos(P)], axis=-1)
    n = 8
    cube = envmap.latlong_to_cube(img + 2.0, n).astype(np.float64) - 2.0  # shift to keep it positive
    want = envmap.texel_directions(n, 4).mean(axis=3)
    assert cube.shape == (6, n, n, 3) and np.abs(cube - want).max() < 0.03
    assert np.array_equal(envmap.latlong_to_cube(np.full((16, 32, 3), 0.25), 4), np.full((6, 4, 4, 3), 0.25, f32))
    c = scenes.sun_sky(8, SUN_DIR, 0.0, 400.0, (0.1, 0.2, 0.3), 0.05)
    sun = np.argwhere((c == 400).all(-1))
    assert len(sun) == 1 and envmap.lookup(np.array(SUN_DIR), 8) == (sun[0][0] * 8 + sun[0][1]) * 8 + sun[0][2]
    up = envmap.texel_directions(8)[:, :, :, 0, 1] > 0
    assert np.array_equal((c == np.array([0.1, 0.2, 0.3], f32)).all(-1) | (c == 400).all(-1), up)
    assert np.all(c[0, :4] != 0.05) and np.all(c[0, 4:] == 0.05)  # rows above / below the horizon on +X
    with pytest.raises(ValueError):
        scenes.sun_sky(7)
