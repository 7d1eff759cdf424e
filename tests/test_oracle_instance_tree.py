"""The instance tree in the CPU restatement (oracle/oracle_instance_tree.c).

The builder's CPU twin is checked for structure and conservative world boxes, the tree walk
against a float64 brute force and, on scenes whose instances float apart on a gapped grid, against
the list walk bit for bit.  Exact ties (duplicated instances, an identity instance of the base
mesh) resolve the same way in both traversals.
"""
import numpy as np
import pytest

from oracle import oracle_instance_tree_py as ot
from oracle import oracle_instances_py as oi
from test_oracle_instances import INSTANCES, _brute_force, _o2w, _primary_rays, _world_tris


def random_o2w(rng, n, scale=(0.05, 0.2), spread=1.0):
    """n object-to-world 3x4 matrices: random rotation, per-axis scale in `scale`, translation."""
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    R = np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
                  np.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
                  np.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], 1)
    s = np.exp(rng.uniform(np.log(scale[0]), np.log(scale[1]), (n, 3)))
    m = np.zeros((n, 3, 4))
    m[:, :, :3] = R * s[:, None, :]
    m[:, :, 3] = rng.uniform(-spread, spread, (n, 3))
    return m


def w2o_of(clpt, o2w):
    return clpt.world_to_object_batch(o2w)


def leaf_boxes(nodes, n):
    """Instance k -> (lo, hi) of the slot that holds it; checks every structural property on the way:
    each instance in exactly one leaf, every slot's box the union of the slots below it, depth <= 50."""
    lo = np.full((n, 3), np.nan, dtype=np.float32)
    hi = np.full((n, 3), np.nan, dtype=np.float32)
    seen = np.zeros(n, dtype=np.int64)
    visited = 0
    stack = [(0, 1)]
    while stack:
        node, depth = stack.pop()
        assert depth <= 50
        visited += 1
        rec = nodes[node]
        for s in (0, 1):
            ref, mn, mx = int(rec[f"ref{s}"]), rec[f"min{s}"], rec[f"max{s}"]
            assert rec[f"pad{s}"] == 0
            if n == 1 and s == 1:
                assert ref == -1 and (mn == np.float32(3.4028235e38)).all() and (mx == -mn).all()
                continue
            if ref >= 0:
                child = nodes[ref]
                assert np.array_equal(mn, np.minimum(child["min0"], child["min1"]))
                assert np.array_equal(mx, np.maximum(child["max0"], child["max1"]))
                stack.append((ref, depth + 1))
            else:
                k = -1 - ref
                seen[k] += 1
                lo[k], hi[k] = mn, mx
    assert visited == len(nodes) and (seen == 1).all()
    return lo, hi


def corners64(w2o, root):
    """The 8 corners of each root box mapped to world space in float64: float64[n, 8, 3]."""
    n = len(w2o)
    full = np.broadcast_to(np.eye(4), (n, 4, 4)).copy()
    full[:, :3, :] = np.asarray(w2o, dtype=np.float64).reshape(n, 3, 4)
    inv = np.linalg.inv(full)
    c = np.array([[(i >> a) & 1 for a in range(3)] for i in range(8)], dtype=np.float64)
    pts = root[:, None, :3].astype(np.float64) + c[None] * (root[:, None, 3:] - root[:, None, :3]).astype(np.float64)
    return np.einsum("nij,nkj->nki", inv[:, :3, :3], pts) + inv[:, None, :3, 3]


@pytest.mark.parametrize("n", [1, 2, 3, 64, 65536])
def test_twin_tree_structure(clpt, n):
    rng = np.random.default_rng(n)
    w2o = w2o_of(clpt, random_o2w(rng, n))
    root = np.concatenate([rng.uniform(-1, -0.2, (n, 3)), rng.uniform(0.2, 1, (n, 3))], 1).astype(np.float32)
    nodes = ot.build_tree(w2o, root)
    assert len(nodes) == max(n - 1, 1)
    lo, hi = leaf_boxes(nodes, n)
    c = corners64(w2o, root)
    assert (lo[:, None] <= c).all() and (hi[:, None] >= c).all()
    assert ot.build_tree(w2o, root).tobytes() == nodes.tobytes()


@pytest.mark.parametrize("case", ["identical", "singular", "huge", "scales"])
def test_twin_tree_degenerate(clpt, case):
    """Every Morton code equal, a zero determinant, an inverse beyond fp32, scales 1e-3 to 1e3."""
    rng = np.random.default_rng(7)
    n = 300
    root = np.tile(np.array([-1, -1, -1, 1, 1, 1], dtype=np.float32), (n, 1))
    if case == "identical":
        w2o = np.tile(w2o_of(clpt, random_o2w(rng, 1)), (n, 1, 1))
    elif case == "scales":
        w2o = w2o_of(clpt, random_o2w(rng, n, scale=(1e-3, 1e3), spread=1e3))
    else:
        w2o = w2o_of(clpt, random_o2w(rng, n))
        w2o[::3, :, :3] = 0 if case == "singular" else 1e-36 * np.eye(3)  # det 0 / inverse ~1e36 * box
        if case == "huge":
            w2o[1::3, :, :3] = 1e-39 * np.eye(3)  # boxes ~1e39 about the origin, beyond fp32: clamped at +-FLT_MAX
            w2o[1::3, :, 3] = 0
        if case == "singular":
            w2o[1::3, :, :3] = [[1, 2, 3], [2, 4, 6], [0, 0, 1]]  # rank 2, determinant exactly 0
    nodes = ot.build_tree(w2o, root)
    lo, hi = leaf_boxes(nodes, n)
    big = np.float32(3.4028235e38)
    if case == "singular":
        assert (lo[::3] == -big).all() and (hi[::3] == big).all()
        assert (lo[1::3] == -big).all() and (hi[1::3] == big).all()
    if case == "huge":
        assert (np.abs(lo[::3]) <= big).all() and (np.abs(hi[::3]) <= big).all()
        assert (lo[1::3] == -big).all() and (hi[1::3] == big).all()
    # (A finite fp32 matrix always has a finite float64 inverse unless det == 0, so the builder's
    # non-finite branch is defensive; det == 0 is the case that reaches it.)
    if case in ("identical", "scales"):
        c = corners64(w2o, root)
        assert (lo[:, None] <= c).all() and (hi[:, None] >= c).all()
    if case == "identical":
        assert (lo == lo[0]).all() and (hi == hi[0]).all()
    assert ot.build_tree(w2o, root).tobytes() == nodes.tobytes()


def _sphere(clpt, subdiv=2):
    import bench

    v, f = bench.icosphere(subdiv)
    return clpt.build_kd(v, clpt.corners_from_faces(f, False), None)


def test_world_boxes_hold_every_instance_hit(clpt, oracle):
    """About 10^5 camera rays at one instance from all around (grazing ones at its silhouette): the
    tree, whose only box is the instance's world box, finds every hit the list finds."""
    from clpathtracer_b200 import scenes

    base = clpt.build_kd(*scenes.heightfield(4, False))  # far below, out of the way
    base.verts[:, 1] -= 50.0
    base = clpt.build_kd(base.verts, base.tris, None)
    sphere = _sphere(clpt, 1)
    rng = np.random.default_rng(3)
    total = 0
    for f in range(10):
        o2w = random_o2w(rng, 1, scale=(0.02, 3.0), spread=2.0)[0]
        centre = o2w[:, 3]
        away = rng.standard_normal(3)
        away /= np.linalg.norm(away)
        pos = centre + away * rng.uniform(2.5, 4) * np.abs(o2w[:, :3]).max()
        cam = clpt.cam_matrix(clpt.make_camera(position=tuple(pos), forward=tuple(-away), fov=0.5), 100)
        inst = [(sphere, clpt.world_to_object(o2w), 0)]
        a = oi.render(base, cam, 100, 100, mode=0, depth=1, instances=inst)
        b = ot.render(base, cam, 100, 100, mode=0, depth=1, instances=inst, tree=ot.tree_of(inst))
        assert np.array_equal(a["prim"], b["prim"]), f
        assert np.array_equal(a["t"].view(np.uint32), b["t"].view(np.uint32)), f
        total += int((a["prim"] >= 0).sum())
    assert total > 20000


def test_tree_matches_world_space_brute_force(clpt, oracle):
    from clpathtracer_b200 import scenes

    base = clpt.build_kd(*scenes.heightfield(22, False))
    sphere = _sphere(clpt)
    o2w = [_o2w(*p) for p in INSTANCES]
    w, h = 96, 72
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), h)
    inst = [(sphere, clpt.world_to_object(m), 0) for m in o2w]
    ref = ot.render(base, cam, w, h, mode=0, depth=1, instances=inst, tree=ot.tree_of(inst))
    o, dirs = _primary_rays(cam, w, h)
    tris = np.concatenate([_world_tris(base)] + [_world_tris(sphere, m) for m in o2w])
    bt, bi, margin, second = _brute_force(o, dirs, tris)
    prim, t = ref["prim"].reshape(-1), ref["t"].reshape(-1).astype(np.float64)
    P, S = base.n_tris, sphere.n_tris
    for k in range(3):
        assert ((bi >= P + k * S) & (bi < P + (k + 1) * S)).sum() > 20, k
    clear = (bi >= 0) & (margin > 1e-4) & (second > bt * (1 + 1e-4))
    assert clear.sum() > 0.8 * (bi >= 0).sum()
    assert np.array_equal(prim[clear], bi[clear])
    assert np.allclose(t[clear], bt[clear], rtol=1e-4, atol=0)
    assert ((prim >= 0) != (bi >= 0)).mean() < 0.005


def separated_grid(clpt, count_x=4, count_z=4, height=0.45, seed=11):
    """Instances on a gapped grid floating clear of the terrain (and of each other's boxes)."""
    rng = np.random.default_rng(seed)
    xs, zs = np.linspace(-0.75, 0.75, count_x), np.linspace(-0.6, 0.6, count_z)
    o2w = random_o2w(rng, count_x * count_z, scale=(0.04, 0.09))
    o2w[:, :, 3] = [(x, height + 0.1 * rng.uniform(), z) for x in xs for z in zs]
    return o2w


@pytest.mark.parametrize("mode,depth,spp", [(0, 1, 1), (1, 3, 1), (1, 3, 4), (2, 3, 1), (2, 4, 4)])
def test_tree_equals_list_on_separated_scenes(clpt, oracle, mode, depth, spp):
    from clpathtracer_b200 import scenes

    v, c, n = scenes.heightfield(22, True)
    base = clpt.build_kd(v, c, n)
    sv, sf = __import__("bench").icosphere(2)
    sphere = clpt.build_kd(sv, clpt.corners_from_faces(sf, True), sv)
    o2w = separated_grid(clpt)
    inst = [(sphere, m, k % 3) for k, m in enumerate(w2o_of(clpt, o2w))]
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 72)
    kw = dict(mode=mode, depth=depth, spp=spp, seed=2, flags=oracle.FLAG_JITTER if spp > 1 else 0)
    if mode == 2:
        kw["materials"] = scenes.CORNELL_MATERIALS
    a = oi.render(base, cam, 96, 72, instances=inst, **kw)
    b = ot.render(base, cam, 96, 72, instances=inst, tree=ot.tree_of(inst), **kw)
    for key in ("rgba", "prim", "t", "uv", "normal"):
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert (a["prim"] >= base.n_tris).mean() > 0.03
    assert a["counters"]["rays"] == b["counters"]["rays"]


def test_without_a_tree_it_is_the_list(clpt, oracle):
    """tree=None is oracle_instances_py.render: the copied render loop is the list's."""
    from clpathtracer_b200 import scenes

    base = clpt.build_kd(*scenes.heightfield(22, True))
    inst = [(_sphere(clpt), clpt.world_to_object(_o2w(*p)), 1) for p in INSTANCES]
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 72)
    kw = dict(mode=1, depth=3, spp=2, seed=4, flags=oracle.FLAG_JITTER | oracle.FLAG_ACCUMULATE, instances=inst)
    a, b = oi.render(base, cam, 96, 72, **kw), ot.render(base, cam, 96, 72, **kw)
    for key in ("rgba", "prim", "t", "uv", "normal", "path_edge", "accum"):
        assert np.array_equal(np.ascontiguousarray(a[key]).view(np.uint8), np.ascontiguousarray(b[key]).view(np.uint8)), key
    assert a["counters"] == b["counters"]


def test_exact_ties(clpt, oracle):
    """Duplicated instances resolve to the higher index in both traversals; an identity instance of
    the base mesh renders the base frame's colours; with no instances the tree is oracle_render."""
    from clpathtracer_b200 import scenes

    v, c, n = scenes.heightfield(22, True)
    base = clpt.build_kd(v, c, n)
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 72)
    kw = dict(mode=1, depth=3, spp=2, seed=3, flags=oracle.FLAG_JITTER)
    sphere = _sphere(clpt)
    m = clpt.world_to_object(_o2w(*INSTANCES[0]))
    other = clpt.world_to_object(_o2w(*INSTANCES[1]))
    inst = [(sphere, m, 0), (sphere, other, 0), (sphere, m, 0), (sphere, m, 0)]
    P, S = base.n_tris, sphere.n_tris
    lst = oi.render(base, cam, 96, 72, instances=inst, **kw)
    tre = ot.render(base, cam, 96, 72, instances=inst, tree=ot.tree_of(inst), **kw)
    assert np.array_equal(lst["rgba"].view(np.uint32), tre["rgba"].view(np.uint32))
    assert np.array_equal(lst["prim"], tre["prim"])
    dup = lst["prim"][(lst["prim"] >= P) & ((lst["prim"] - P) // S != 1)]
    assert len(dup) > 50 and ((dup - P) // S == 3).all()
    # identity instance of the base mesh: the base frame's colours, every first hit the instance's
    alone = oracle.render(base, cam, 96, 72, **kw)
    ident = [(base, np.eye(3, 4, dtype=np.float32), 0)]
    both = ot.render(base, cam, 96, 72, instances=ident, tree=ot.tree_of(ident), **kw)
    assert np.array_equal(both["rgba"].view(np.uint32), alone["rgba"].view(np.uint32))
    hit = alone["prim"] >= 0
    assert np.array_equal(both["prim"][hit], alone["prim"][hit] + P)
    # no instances
    none = ot.render(base, cam, 96, 72, instances=[], tree=np.zeros(1, dtype=ot.NODE_DTYPE), **kw)
    for key in ("rgba", "prim", "t", "uv"):
        assert np.array_equal(np.ascontiguousarray(none[key]).view(np.uint8), np.ascontiguousarray(alone[key]).view(np.uint8))
    assert none["counters"] == alone["counters"]


def test_batched_inversion_matches_world_to_object(clpt):
    rng = np.random.default_rng(5)
    o2w = random_o2w(rng, 200, scale=(1e-3, 1e3), spread=100.0)
    batch = clpt.world_to_object_batch(o2w)
    assert batch.dtype == np.float32 and batch.shape == (200, 3, 4)
    for k in range(200):
        assert batch[k].tobytes() == clpt.world_to_object(o2w[k]).tobytes()
    full = np.broadcast_to(np.eye(4), (200, 4, 4)).copy()
    full[:, :3] = o2w
    assert clpt.world_to_object_batch(full).tobytes() == batch.tobytes()
