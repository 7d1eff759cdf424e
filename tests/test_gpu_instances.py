"""Rigid instances on the device (CLAddInstanceMesh / CLSetInstances): every frame equals the
oracle's restatement (oracle/oracle_instances.c) bit for bit -- colours,
first-hit primitive, t, u, v and the work counters -- on both engines, at one and several
samples per pixel, progressive and row-tile sharded, while instances move without any
rebuild and while the base scene underneath them is replaced."""
import numpy as np
import pytest

from oracle import oracle_instances_py as oi

pytestmark = pytest.mark.gpu

W, H = 160, 120


def _o2w(angles, scale, translate):
    ax, ay, az = angles
    rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    m = np.zeros((3, 4))
    m[:, :3] = rz @ ry @ rx @ np.diag(scale)
    m[:, 3] = translate
    return m


def _mesh(name):
    import bench
    from clpathtracer_b200 import corners_from_faces, scenes

    if name == "ico":
        v, f = bench.icosphere(2)
        return v, corners_from_faces(f, False), None
    if name == "icon":  # with vertex normals: the interpolated shading path
        v, f = bench.icosphere(2)
        return v, corners_from_faces(f, True), v
    if name == "cornell":
        return scenes.cornell(6)[:3]
    if name.startswith("soup"):
        return scenes.soup(int(name[4:]), size=0.08)
    with_n = name.endswith("n")
    return scenes.heightfield(int(name[2:-1] if with_n else name[2:]), with_n)


# base, camera, instance mesh, instances (angles, scale, translate, material): overlapping each
# other and crossing the base scene's box; material 7 is out of range (clamped to 0 in mode 2)
CASES = {
    "hf22n+ico": ("hf22n", "canonical", "icon", [((0.3, 0.7, -0.2), (0.35, 0.2, 0.25), (-0.15, 0.05, -0.3), 1),
                                                 ((-0.5, 0.2, 0.9), (0.2, 0.3, 0.45), (0.1, 0.1, -0.2), 3),
                                                 ((1.1, -0.4, 0.3), (0.5, 0.12, 0.2), (0.0, 0.2, -0.45), 7)]),
    "cornell+soup": ("cornell", "cornell", "soup300", [((0.2, 0.4, 0.1), (0.9, 0.6, 0.8), (-0.2, -0.3, 0.2), 2),
                                                       ((0.0, 1.2, 0.0), (0.5, 1.4, 0.5), (0.4, 0.2, -0.1), 1)]),
}


def _cam(clpt, which):
    from clpathtracer_b200 import scenes

    kw = {"canonical": scenes.CANONICAL_CAMERA, "cornell": scenes.CORNELL_CAMERA}[which]
    return clpt.cam_matrix(clpt.make_camera(**kw), H)


@pytest.fixture
def inst_renderer(renderer, clpt):
    renderer.clear_instance_meshes()
    yield renderer
    L = clpt.lib()
    renderer.clear_instance_meshes()
    renderer.set_materials(np.zeros((0, 8), dtype=np.float32))
    L.CLSetEngine(0)
    L.CLSetTileShard(0, 1, 8)
    renderer.set_params(mode=0, depth=2)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _setup(clpt, renderer, case):
    base_name, camera, mesh_name, spec = CASES[case]
    renderer.build_meshes(*_mesh(base_name))
    base = renderer.download_kd()
    handle = renderer.add_instance_mesh(*_mesh(mesh_name))
    mesh = renderer.download_instance_kd(handle)
    o2w = [_o2w(a, s, t) for a, s, t, _ in spec]
    mats = [m for *_, m in spec]
    renderer.set_instances([(handle, m, mat) for m, mat in zip(o2w, mats)])
    oracle_inst = [(mesh, clpt.world_to_object(m), mat) for m, mat in zip(o2w, mats)]
    return base, _cam(clpt, camera), oracle_inst


@pytest.mark.parametrize("engine", [1, 2])
@pytest.mark.parametrize("spp", [1, 4])
@pytest.mark.parametrize("mode,depth", [(0, 1), (1, 3), (2, 3)])
@pytest.mark.parametrize("case", list(CASES))
def test_instances_equal_oracle(clpt, oracle, inst_renderer, case, mode, depth, spp, engine):
    from clpathtracer_b200 import scenes

    r = inst_renderer
    base, cam, inst = _setup(clpt, r, case)
    kw, materials = dict(mode=mode, depth=depth, spp=spp, seed=9), {}
    if mode == 2:
        tm = scenes.cornell(6)[3] if case.startswith("cornell") else None
        r.set_materials(scenes.CORNELL_MATERIALS, tm)
        materials = dict(materials=scenes.CORNELL_MATERIALS, tri_material=tm)
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(cam)
    r.create_image(W, H, aov=True)
    jitter = clpt.FLAG_JITTER if spp > 1 else 0
    ref = oi.render(base, cam, W, H, flags=jitter, instances=inst, **kw, **materials)
    for flags in (jitter, jitter | clpt.FLAG_COUNTERS):
        r.set_params(flags=flags, **kw)
        r.execute()
        assert clpt.lib().CLLastEngine() == engine
        prim, t, uv = r.read_aov()
        assert np.array_equal(_bits(r.read_image()), _bits(ref["rgba"]))
        assert np.array_equal(prim, ref["prim"])
        assert np.array_equal(_bits(t), _bits(ref["t"])) and np.array_equal(_bits(uv), _bits(ref["uv"]))
        if flags & clpt.FLAG_COUNTERS:
            assert r.counters() == ref["counters"]
    P = base.n_tris
    assert (prim >= P).mean() > 0.01 and ((prim >= 0) & (prim < P)).mean() > 0.1
    for k in range(len(inst)):  # every instance is the first hit somewhere
        lo = P + k * inst[0][0].n_tris
        assert ((prim >= lo) & (prim < lo + inst[0][0].n_tris)).any(), k


def test_moving_instances_need_no_rebuild(clpt, oracle, inst_renderer):
    r = inst_renderer
    base, cam, _ = _setup(clpt, r, "hf22n+ico")
    mesh = r.download_instance_kd(0)
    build = r.build_ms()
    r.set_camera_matrix(cam)
    r.set_params(mode=1, depth=3, spp=2, seed=4, flags=clpt.FLAG_JITTER)
    r.create_image(W, H, aov=True)
    for f in range(4):
        o2w = [_o2w((0.2 * f, 0.5, 0.1 * f), (0.2, 0.25, 0.3), (-0.3 + 0.15 * f, 0.1, -0.3 + 0.05 * f)),
               _o2w((0.0, -0.3 * f, 0.4), (0.3, 0.15, 0.2), (0.2, 0.15 - 0.04 * f, -0.5))]
        r.set_instances([(0, m, 0) for m in o2w])
        r.execute()
        ref = oi.render(base, cam, W, H, mode=1, depth=3, spp=2, seed=4, flags=oi.FLAG_JITTER,
                            instances=[(mesh, clpt.world_to_object(m), 0) for m in o2w])
        assert np.array_equal(_bits(r.read_image()), _bits(ref["rgba"])), f
        assert np.array_equal(r.read_aov()[0], ref["prim"]), f
        assert (ref["prim"] >= base.n_tris).any()
        assert r.build_ms() == build


def test_identity_instance_and_no_instances(clpt, inst_renderer):
    """An identity instance of the base mesh (the device builder gives the same mesh the same tree)
    renders the base frame bit for bit with every first hit moved to the instance's ids; removing
    the instances gives back the frame rendered before any existed."""
    r = inst_renderer
    v, c, n = _mesh("hf22n")
    r.build_meshes(v, c, n)
    r.set_camera_matrix(_cam(clpt, "canonical"))
    r.set_params(mode=1, depth=3, spp=2, seed=6, flags=clpt.FLAG_JITTER)
    r.create_image(W, H, aov=True)
    r.execute()
    alone, (prim0, t0, _) = r.read_image(), r.read_aov()
    handle = r.add_instance_mesh(v, c, n)
    assert r.download_instance_kd(handle).nodes.tobytes() == r.download_kd().nodes.tobytes()
    r.set_instances([(handle, np.eye(4), 0)])
    r.execute()
    prim1, t1, _ = r.read_aov()
    assert np.array_equal(_bits(r.read_image()), _bits(alone))
    hit = prim0 >= 0
    assert hit.mean() > 0.3
    assert np.array_equal(prim1[hit], prim0[hit] + len(c) // 3) and np.array_equal(prim1[~hit], prim0[~hit])
    assert np.array_equal(_bits(t1), _bits(t0))
    r.set_instances([])
    r.execute()
    assert np.array_equal(_bits(r.read_image()), _bits(alone))
    assert np.array_equal(r.read_aov()[0], prim0)


def test_progressive_and_sharded_with_instances(clpt, oracle, inst_renderer):
    r = inst_renderer
    L = clpt.lib()
    base, cam, inst = _setup(clpt, r, "cornell+soup")
    r.set_camera_matrix(cam)
    flags = clpt.FLAG_JITTER | clpt.FLAG_ACCUMULATE
    r.set_params(mode=1, depth=3, spp=2, seed=3, flags=flags)
    r.create_image(W, H)
    acc = oracle.new_accumulator(W, H)
    for frame in range(3):
        r.execute()
        want = oi.render(base, cam, W, H, mode=1, depth=3, spp=2, seed=3, flags=flags, sample_base=2 * frame,
                             accumulate_into=acc, aov=False, instances=inst)["rgba"]
    assert np.array_equal(_bits(r.read_image()), _bits(want))
    full = oi.render(base, cam, W, H, mode=1, depth=3, aov=False, instances=inst)["rgba"]
    r.set_params(mode=1, depth=3)
    for rank in range(2):
        r.create_image(W, H)
        L.CLSetTileShard(rank, 2, 8)
        r.execute()
        rows = np.array([y for y in range(H) if (y // 8) % 2 == rank])
        assert np.array_equal(_bits(r.read_image()[rows]), _bits(full[rows])), rank


def test_base_scene_replaced_under_instances(clpt, oracle, inst_renderer, scene_cache):
    """Instance meshes survive base-scene changes; the instances' primitive ids follow the base
    scene current at the frame, through CLBuildMeshes and through CLSetMeshes."""
    r = inst_renderer
    _, cam, inst = _setup(clpt, r, "hf22n+ico")
    r.set_camera_matrix(cam)
    r.set_params(mode=0, depth=1)
    r.create_image(W, H, aov=True)
    r.build_meshes(*_mesh("hf30"))
    device_tree = r.download_kd()
    host_tree = scene_cache("hf22")[0]
    for tree, upload in ((device_tree, None), (host_tree, r.set_meshes)):
        if upload:
            upload(tree)
        r.execute()
        ref = oi.render(tree, cam, W, H, mode=0, depth=1, instances=inst)
        assert np.array_equal(_bits(r.read_image()), _bits(ref["rgba"]))
        prim = r.read_aov()[0]
        assert np.array_equal(prim, ref["prim"])
        assert (prim >= tree.n_tris).any()


@pytest.mark.parametrize("what,code,message", [
    ("bad handle", "r.set_instances([(h + 1, np.eye(4), 0)])", "names mesh 1"),
    ("nan matrix", "t = (cl.CLInstance * 1)(); t[0].world_to_object[7] = float('nan'); L.CLSetInstances(t, 64)",
     "world_to_object[7] is not finite"),
    ("65 instances", "r.set_instances([(h, np.eye(4), 0)] * 65)", "at most 64"),
    ("partial record", "L.CLSetInstances((C.c_char * 96)(), 96)", "64-byte"),
])
def test_instances_reject_bad_input(clpt, what, code, message):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    prog = ("import sys;sys.path.insert(0,%r);import ctypes as C;import numpy as np;import clpathtracer_b200 as cl;"
            "import bench;v,f=bench.icosphere(1);r=cl.Renderer(0);L=r.L;"
            "h=r.add_instance_mesh(v,cl.corners_from_faces(f,False));%s") % (str(root), code)
    p = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True)
    assert p.returncode == 1 and "CLSetInstances" in p.stderr and message in p.stderr, (what, p.stderr)
