"""The instance tree on the device (CLSetInstanceTraversal(CLPT_INSTANCES_TREE)): the device-built
tree equals the CPU twin's byte for byte, and every frame equals the tree oracle
(oracle/oracle_instance_tree.c) walking the downloaded tree bit for bit -- colours, first-hit
primitive, t, u, v and the work counters -- on both engines, at one and several samples per pixel,
with instances moving every frame, progressive, row-tile sharded and under a replaced base scene."""
import numpy as np
import pytest

from oracle import oracle_instance_tree_py as ot
from test_gpu_instances import CASES, W, H, _bits, _cam, _mesh, _o2w, inst_renderer  # noqa: F401
from test_oracle_instance_tree import random_o2w, separated_grid

pytestmark = pytest.mark.gpu


@pytest.fixture
def tree_renderer(inst_renderer):
    inst_renderer.set_instance_traversal("tree")
    yield inst_renderer
    inst_renderer.clear_instance_meshes()
    inst_renderer.set_instance_traversal("list")


def _equal(a, b):
    return np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()


@pytest.mark.parametrize("case", ["n1", "n2", "n3", "n64", "n1000", "n65536", "duplicates", "singular", "huge",
                                  "scales"])
def test_device_tree_equals_twin(clpt, tree_renderer, case):
    import bench

    r = tree_renderer
    rng = np.random.default_rng(len(case))
    v, f = bench.icosphere(1)
    handles_avail = [r.add_instance_mesh(v, clpt.corners_from_faces(f, False)),
                     r.add_instance_mesh(v * [2.0, 0.5, 1.0], clpt.corners_from_faces(f, False))]
    n = int(case[1:]) if case.startswith("n") else 500
    o2w = random_o2w(rng, n, scale=(1e-3, 1e3) if case == "scales" else (0.05, 0.2),
                     spread=1e3 if case == "scales" else 1.0)
    if case == "duplicates":
        o2w[n // 2:] = o2w[: n - n // 2]
    if case == "huge":
        o2w[::4, :, :3] *= 1e39  # world boxes beyond fp32: clamped at +-FLT_MAX
    handles = np.array(handles_avail)[rng.integers(0, 2, n)]
    table = np.zeros(n, dtype=clpt.CLINSTANCE_DTYPE)
    table["world_to_object"] = clpt.world_to_object_batch(o2w).reshape(n, 12)
    if case == "singular":  # determinant 0: the box +-FLT_MAX
        table["world_to_object"][::4] = [1, 2, 3, 0, 2, 4, 6, 0, 0, 0, 1, 0]
    table["mesh"] = handles
    for _ in range(2):  # built twice: the same bytes
        r.L.CLSetInstances(table.ctypes.data, table.nbytes)
        dev = r.instance_tree()
        assert r.instance_build_ms() > 0
        roots = {h: ot.root_box(r.download_instance_kd(h)) for h in handles_avail}
        twin = ot.build_tree(table["world_to_object"].reshape(n, 3, 4), np.stack([roots[int(h)] for h in handles]))
        assert _equal(dev, twin)


def _setup_case(clpt, r, case):
    base_name, camera, mesh_name, spec = CASES[case]
    r.build_meshes(*_mesh(base_name))
    base = r.download_kd()
    handle = r.add_instance_mesh(*_mesh(mesh_name))
    mesh = r.download_instance_kd(handle)
    o2w = np.stack([_o2w(a, s, t) for a, s, t, _ in spec])
    mats = [m for *_, m in spec]
    r.set_instance_arrays([handle] * len(o2w), o2w, mats)
    inst = [(mesh, w, m) for w, m in zip(clpt.world_to_object_batch(o2w), mats)]
    return base, _cam(clpt, camera), inst


def _setup_crowd(clpt, r, n=4096):
    """n small icospheres scattered over a heightfield."""
    rng = np.random.default_rng(9)
    r.build_meshes(*_mesh("hf22n"))
    base = r.download_kd()
    handle = r.add_instance_mesh(*_mesh("icon"))
    mesh = r.download_instance_kd(handle)
    o2w = random_o2w(rng, n, scale=(0.01, 0.03))
    o2w[:, 0, 3] *= 0.9
    o2w[:, 1, 3] = rng.uniform(-0.1, 0.3, n)
    mats = rng.integers(0, 4, n)
    r.set_instance_arrays(np.full(n, handle), o2w, mats)
    inst = [(mesh, w, int(m)) for w, m in zip(clpt.world_to_object_batch(o2w), mats)]
    return base, _cam(clpt, "canonical"), inst


@pytest.mark.parametrize("engine", [1, 2])
@pytest.mark.parametrize("spp", [1, 4])
@pytest.mark.parametrize("mode,depth", [(0, 1), (1, 3), (2, 3)])
@pytest.mark.parametrize("case", list(CASES) + ["crowd4096"])
def test_tree_frames_equal_oracle(clpt, tree_renderer, case, mode, depth, spp, engine):
    from clpathtracer_b200 import scenes

    r = tree_renderer
    base, cam, inst = _setup_crowd(clpt, r) if case == "crowd4096" else _setup_case(clpt, r, case)
    kw = dict(mode=mode, depth=depth, spp=spp, seed=9, flags=clpt.FLAG_JITTER if spp > 1 else 0)
    if mode == 2:
        tm = scenes.cornell(6)[3] if case.startswith("cornell") else None
        r.set_materials(scenes.CORNELL_MATERIALS, tm)
        kw.update(materials=scenes.CORNELL_MATERIALS, tri_material=tm)
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(cam)
    r.create_image(W, H, aov=True)
    kw_dev = {k: v for k, v in kw.items() if k not in ("materials", "tri_material")}
    tree = r.instance_tree()
    ref = ot.render(base, cam, W, H, instances=inst, tree=tree, **kw)
    for flags in (kw["flags"], kw["flags"] | clpt.FLAG_COUNTERS):
        r.set_params(**{**kw_dev, "flags": flags})
        r.execute()
        assert clpt.lib().CLLastEngine() == engine
        prim, t, uv = r.read_aov()
        assert _equal(r.read_image(), ref["rgba"])
        assert np.array_equal(prim, ref["prim"])
        assert _equal(t, ref["t"]) and _equal(uv, ref["uv"])
        if flags & clpt.FLAG_COUNTERS:
            assert r.counters() == ref["counters"]
    assert (prim >= base.n_tris).mean() > 0.01


def test_moving_instances_rebuild_the_tree(clpt, tree_renderer):
    """Instances move every frame (a new tree each frame), the traversal switches between frames,
    and the base scene is replaced under the instances."""
    r = tree_renderer
    L = clpt.lib()
    base, cam, _ = _setup_case(clpt, r, "hf22n+ico")
    mesh = r.download_instance_kd(0)
    r.set_camera_matrix(cam)
    kw = dict(mode=1, depth=3, spp=2, seed=4, flags=clpt.FLAG_JITTER)
    r.set_params(**kw)
    r.create_image(W, H, aov=True)
    for f in range(4):
        o2w = np.stack([_o2w((0.2 * f, 0.5, 0.1 * f), (0.2, 0.25, 0.3), (-0.3 + 0.15 * f, 0.1, -0.3 + 0.05 * f)),
                        _o2w((0.0, -0.3 * f, 0.4), (0.3, 0.15, 0.2), (0.2, 0.15 - 0.04 * f, -0.5)),
                        _o2w((0.1, 0.2, 0.3), (0.1, 0.1, 0.1), (0.05 * f, 0.3, -0.6))])
        r.set_instance_arrays([0, 0, 0], o2w, 0)
        r.set_instance_traversal("tree" if f != 2 else "list")
        r.execute()
        inst = [(mesh, w, 0) for w in clpt.world_to_object_batch(o2w)]
        tree = r.instance_tree() if f != 2 else None
        ref = ot.render(base, cam, W, H, instances=inst, tree=tree, **kw)
        assert _equal(r.read_image(), ref["rgba"]), f
        assert np.array_equal(r.read_aov()[0], ref["prim"]), f
        assert (ref["prim"] >= base.n_tris).any()
    assert L.CLInstanceTraversal() == 1
    build = r.instance_build_ms()
    r.build_meshes(*_mesh("hf30"))  # a new base scene: ids move, the tree is not rebuilt
    base2 = r.download_kd()
    r.set_params(mode=0, depth=1)
    r.execute()
    assert r.instance_build_ms() == build
    ref = ot.render(base2, cam, W, H, mode=0, depth=1, instances=inst, tree=r.instance_tree())
    assert _equal(r.read_image(), ref["rgba"])
    assert np.array_equal(r.read_aov()[0], ref["prim"])


def test_progressive_and_sharded_with_the_tree(clpt, oracle, tree_renderer):
    r = tree_renderer
    L = clpt.lib()
    base, cam, inst = _setup_case(clpt, r, "cornell+soup")
    tree = r.instance_tree()
    r.set_camera_matrix(cam)
    flags = clpt.FLAG_JITTER | clpt.FLAG_ACCUMULATE
    r.set_params(mode=1, depth=3, spp=2, seed=3, flags=flags)
    r.create_image(W, H)
    acc = oracle.new_accumulator(W, H)
    for frame in range(3):
        r.execute()
        want = ot.render(base, cam, W, H, mode=1, depth=3, spp=2, seed=3, flags=flags, sample_base=2 * frame,
                         accumulate_into=acc, aov=False, instances=inst, tree=tree)["rgba"]
    assert _equal(r.read_image(), want)
    full = ot.render(base, cam, W, H, mode=1, depth=3, aov=False, instances=inst, tree=tree)["rgba"]
    r.set_params(mode=1, depth=3)
    for rank in range(2):
        r.create_image(W, H)
        L.CLSetTileShard(rank, 2, 8)
        r.execute()
        rows = np.array([y for y in range(H) if (y // 8) % 2 == rank])
        assert _equal(r.read_image()[rows], full[rows]), rank


@pytest.mark.parametrize("mode,depth,spp", [(0, 1, 1), (1, 3, 4), (2, 3, 1)])
def test_tree_equals_list_on_the_device(clpt, tree_renderer, mode, depth, spp):
    """Instances floating apart on a gapped grid: the tree's frame is the list's, bit for bit."""
    from clpathtracer_b200 import scenes

    r = tree_renderer
    r.build_meshes(*_mesh("hf22n"))
    handle = r.add_instance_mesh(*_mesh("icon"))
    o2w = separated_grid(clpt)
    r.set_instance_arrays(np.full(len(o2w), handle), o2w, np.arange(len(o2w)) % 3)
    r.set_materials(scenes.CORNELL_MATERIALS)
    r.set_camera_matrix(_cam(clpt, "canonical"))
    r.set_params(mode=mode, depth=depth, spp=spp, seed=2, flags=clpt.FLAG_JITTER if spp > 1 else 0)
    r.create_image(W, H, aov=True)
    out = {}
    for traversal in ("list", "tree"):
        r.set_instance_traversal(traversal)
        r.execute()
        out[traversal] = (r.read_image(), *r.read_aov())
    for a, b in zip(out["list"], out["tree"]):
        assert _equal(a, b)
    assert (out["tree"][1] >= 0).mean() > 0.3


@pytest.mark.parametrize("what,code,message", [
    ("bad traversal", "L.CLSetInstanceTraversal(2)", "CLSetInstanceTraversal: 2 is neither"),
    ("list over 64", "L.CLSetInstanceTraversal(1);r.set_instance_arrays([h]*65,np.tile(np.eye(4),(65,1,1)),0);"
     "L.CLSetInstanceTraversal(0)", "CLSetInstanceTraversal: 65 instances are set; the list takes at most 64"),
    ("65 under the list", "r.set_instance_arrays([h]*65,np.tile(np.eye(4),(65,1,1)),0)",
     "CLSetInstances: 65 instances, at most 64"),
    ("over 2^20", "L.CLSetInstanceTraversal(1);r.set_instance_arrays([h]*(2**20+1),np.tile(np.eye(4),(2**20+1,1,1)),0)",
     "CLSetInstances: 1048577 instances, at most 1048576"),
    ("ids past INT32_MAX", "L.CLSetInstanceTraversal(1);v4,f4=bench.icosphere(4);"
     "g=r.add_instance_mesh(v4,cl.corners_from_faces(f4,False));r.build_meshes(v,cl.corners_from_faces(f,False));"
     "r.set_instance_arrays([g]*2**19,np.tile(np.eye(4),(2**19,1,1)),0);r.create_image(8,8);r.execute()",
     "would pass INT32_MAX"),
])
def test_tree_rejects_bad_input(clpt, what, code, message):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    prog = ("import sys;sys.path.insert(0,%r);import ctypes as C;import numpy as np;import clpathtracer_b200 as cl;"
            "import bench;v,f=bench.icosphere(1);r=cl.Renderer(0);L=r.L;"
            "h=r.add_instance_mesh(v,cl.corners_from_faces(f,False));%s") % (str(root), code)
    p = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True)
    assert p.returncode == 1 and message in p.stderr, (what, p.stderr)
