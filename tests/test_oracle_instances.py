"""Rigid instances in the CPU restatement (oracle/oracle_instances.c).

The oracle is the definition the CUDA path is held to, so it is checked here on its own:
its first hits against a float64 brute force over every transformed triangle, and an
identity instance of the base scene's own tree against the base scene alone.
"""
import numpy as np
import pytest

from oracle import oracle_instances_py as oi


def _o2w(angles, scale, translate):
    """3x4 object-to-world: translate . Rz . Ry . Rx . diag(scale)."""
    ax, ay, az = angles
    rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    m = np.zeros((3, 4))
    m[:, :3] = rz @ ry @ rx @ np.diag(scale)
    m[:, 3] = translate
    return m


# Three overlapping ellipsoids crossing the terrain (and the base scene's box) under the canonical camera.
INSTANCES = [((0.3, 0.7, -0.2), (0.35, 0.2, 0.25), (-0.15, 0.05, -0.3)),
             ((-0.5, 0.2, 0.9), (0.2, 0.3, 0.45), (0.1, 0.1, -0.2)),
             ((1.1, -0.4, 0.3), (0.5, 0.12, 0.2), (0.0, 0.2, -0.45))]


def _primary_rays(cam, w, h):
    """The oracle's camera rays (kernel.cl:443-456) in float32, without jitter."""
    M = cam.astype(np.float32).reshape(16)
    f32 = np.float32

    def unproject(x, y, z):
        w_ = ((M[12] * x + M[13] * y) + M[14] * z) + M[15]
        return np.stack([((M[4 * r] * x + M[4 * r + 1] * y) + M[4 * r + 2] * z) + M[4 * r + 3] for r in range(3)],
                        -1) / w_[..., None]

    ys, xs = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing="ij")
    fx, fy = xs - f32(w) / f32(2), ys - f32(h) / f32(2)
    d = unproject(fx, fy, np.full_like(fx, 1)) - unproject(fx, fy, np.full_like(fx, -1))
    d = d / np.sqrt((d * d).sum(-1, keepdims=True))
    o = np.array([M[2] / M[14], M[6] / M[14], M[10] / M[14]], dtype=np.float32)
    return o.astype(np.float64), d.reshape(-1, 3).astype(np.float64)


def _brute_force(o, dirs, tris):
    """float64 Moller-Trumbore, back faces culled: per ray the nearest t, its triangle, the
    triangle's smallest barycentric margin and the relative gap to the second-nearest hit."""
    v0, e1, e2 = tris[:, 0], tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0]
    n = len(dirs)
    best_t = np.full(n, np.inf)
    best_i = np.full(n, -1)
    margin = np.zeros(n)
    second = np.full(n, np.inf)
    for s in range(0, n, 512):
        d = dirs[s:s + 512, None, :]
        p = np.cross(d, e2[None])
        det = (e1[None] * p).sum(-1)
        with np.errstate(divide="ignore", invalid="ignore"):
            inv = 1.0 / det
            tv = o - v0
            u = (tv[None] * p).sum(-1) * inv
            q = np.cross(tv, e1)
            v = (d * q[None]).sum(-1) * inv
            t = (e2 * q).sum(-1)[None] * inv
        ok = (det > 0) & (u >= 0) & (v >= 0) & (u + v <= 1) & (t > 0)
        t = np.where(ok, t, np.inf)
        order = np.argsort(t, axis=1)[:, :2]
        rows = np.arange(len(t))
        best_i[s:s + 512] = np.where(np.isfinite(t[rows, order[:, 0]]), order[:, 0], -1)
        best_t[s:s + 512] = t[rows, order[:, 0]]
        second[s:s + 512] = t[rows, order[:, 1]]
        uu, vv = u[rows, order[:, 0]], v[rows, order[:, 0]]
        margin[s:s + 512] = np.minimum(np.minimum(uu, vv), 1 - uu - vv)
    return best_t, best_i, margin, second


def _world_tris(scene, o2w=None):
    tri = scene.verts[scene.tris[:, 0], :3].astype(np.float64).reshape(-1, 3, 3)
    if o2w is not None:
        tri = tri @ o2w[:, :3].T + o2w[:, 3]
    return tri


def test_instances_match_world_space_brute_force(clpt, oracle):
    import bench
    from clpathtracer_b200 import scenes

    base = clpt.build_kd(*scenes.heightfield(22, False))
    sv, sf = bench.icosphere(2)
    sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, False), None)
    o2w = [_o2w(*p) for p in INSTANCES]
    assert all(np.linalg.det(m[:, :3]) > 0 for m in o2w)  # (orientation kept: the same faces are culled)
    w, h = 96, 72
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), h)
    inst = [(sphere, clpt.world_to_object(m), 0) for m in o2w]
    ref = oi.render(base, cam, w, h, mode=0, depth=1, instances=inst)

    o, dirs = _primary_rays(cam, w, h)
    tris = np.concatenate([_world_tris(base)] + [_world_tris(sphere, m) for m in o2w])
    bt, bi, margin, second = _brute_force(o, dirs, tris)
    prim, t = ref["prim"].reshape(-1), ref["t"].reshape(-1).astype(np.float64)
    P, S = base.n_tris, sphere.n_tris
    assert (bi >= P).sum() > 0.05 * len(bi) and ((bi >= 0) & (bi < P)).sum() > 0.1 * len(bi)
    for k in range(3):  # every instance is seen, and in front of another or of the terrain somewhere
        assert ((bi >= P + k * S) & (bi < P + (k + 1) * S)).sum() > 20, k
    clear = (bi >= 0) & (margin > 1e-4) & (second > bt * (1 + 1e-4))
    assert clear.sum() > 0.8 * (bi >= 0).sum()
    assert np.array_equal(prim[clear], bi[clear])
    assert np.allclose(t[clear], bt[clear], rtol=1e-4, atol=0)
    # misses and hits agree everywhere but on a few grazing pixels
    assert ((prim >= 0) != (bi >= 0)).mean() < 0.005


def _identity_case(clpt, name):
    from clpathtracer_b200 import scenes

    if name == "hf22n":
        v, c, n = scenes.heightfield(22, True)
        return clpt.build_kd(v, c, n), clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 72)
    v, c, n, _ = scenes.cornell(6)
    return clpt.build_kd(v, c, n), clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), 72)


@pytest.mark.parametrize("name,mode,depth,spp", [("hf22n", 1, 3, 2), ("cornell", 1, 4, 1), ("hf22n", 2, 3, 2),
                                                 ("cornell", 0, 1, 3)])
def test_identity_instance_is_the_base_scene(clpt, oracle, name, mode, depth, spp):
    """An identity instance of the base scene's own tree finds every hit the base finds at the same
    t and wins the tie, so the frame is the base frame bit for bit and every first hit's primitive
    is the instance's (base id + P).  Jittered camera: no exactly-zero ray components."""
    base, cam = _identity_case(clpt, name)
    w, h = 96, 72
    kw = dict(mode=mode, depth=depth, spp=spp, seed=3, flags=oracle.FLAG_JITTER)
    if mode == 2:
        from clpathtracer_b200 import scenes

        kw["materials"] = scenes.CORNELL_MATERIALS[:1]
    alone = oracle.render(base, cam, w, h, **kw)
    ident = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0]], dtype=np.float32)
    both = oi.render(base, cam, w, h, instances=[(base, ident, 0)], **kw)
    assert np.array_equal(both["rgba"].view(np.uint32), alone["rgba"].view(np.uint32))
    hit = alone["prim"] >= 0
    assert hit.mean() > 0.3
    assert np.array_equal(both["prim"][hit], alone["prim"][hit] + base.n_tris)
    assert np.array_equal(both["prim"][~hit], alone["prim"][~hit])
    assert np.array_equal(both["t"].view(np.uint32), alone["t"].view(np.uint32))
    c, c2 = alone["counters"], both["counters"]
    assert c2["rays"] == c["rays"] and c2["shade_vn"] == c["shade_vn"] and c2["leaves"] > c["leaves"]


@pytest.mark.parametrize("name,mode,depth,spp,flags", [("hf22n", 0, 2, 1, 0), ("hf22n", 1, 3, 2, 1), ("cornell", 2, 4, 2, 1),
                                                       ("cornell", 1, 2, 3, 3)])
def test_without_instances_it_is_the_oracle(clpt, oracle, name, mode, depth, spp, flags):
    """With no instances the instanced render loop is oracle_render: the same frame, AOVs, work
    counters and (progressive) running sums."""
    from clpathtracer_b200 import scenes

    base, cam = _identity_case(clpt, name)
    kw = dict(mode=mode, depth=depth, spp=spp, seed=5, flags=flags)
    if mode == 2:
        kw.update(materials=scenes.CORNELL_MATERIALS, tri_material=scenes.cornell(6)[3])
    a = oracle.render(base, cam, 96, 72, **kw)
    b = oi.render(base, cam, 96, 72, **kw)
    for key in ("rgba", "prim", "t", "uv", "normal", "path_edge") + (("accum",) if flags & 2 else ()):
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"] == b["counters"]


def test_world_to_object_inverts_in_float64(clpt):
    m = _o2w((0.3, -1.2, 2.0), (0.5, 2.0, 0.25), (1.0, -2.0, 3.0))
    w2o = clpt.world_to_object(m)
    assert w2o.dtype == np.float32 and w2o.shape == (3, 4)
    full = np.eye(4)
    full[:3] = m
    assert np.allclose(np.vstack([w2o, [0, 0, 0, 1]]) @ full, np.eye(4), atol=1e-6)
    assert np.array_equal(clpt.world_to_object(full), w2o)
