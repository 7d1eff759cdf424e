"""Light sampling (mode 3) on the device: the emitter table equals the CPU twin byte for byte
whichever path built the scene, and every mode-3 frame equals the mode-3 oracle
(oracle/oracle_nee.c) bit for bit -- colours, first-hit primitive, t, u, v and the work counters --
on both engines, at 1, 4 and 64 samples per pixel, with no instances, the instance list and the
instance tree, progressive and row-tile sharded.  The analytic floor checks the estimate itself."""
import numpy as np
import pytest

from oracle import oracle_instance_tree_py as ot
from oracle import oracle_nee_py as on
from test_gpu_instances import _mesh, _o2w, inst_renderer  # noqa: F401
from test_oracle_nee import _floor_with_occluder, floor_expectation, nee_floor_statistic, unlisted_emitter_scene

pytestmark = pytest.mark.gpu

W, H = 64, 48


@pytest.fixture
def nee_renderer(inst_renderer):
    yield inst_renderer
    inst_renderer.set_instance_traversal("list")


def _equal(a, b):
    return np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()


def _same_table(dev, twin):
    assert np.array_equal(dev["header"], twin["header"])
    for key in ("records", "cdf", "map"):
        assert _equal(dev[key], twin[key]), key


def test_device_table_equals_twin(clpt, nee_renderer):
    """The host path, the device path, moved vertices, changed materials, a smaller scene, and a
    scene where all of a million triangles emit."""
    from clpathtracer_b200 import scenes

    r = nee_renderer
    v, c, nn, tm = scenes.cornell_small_light(10)
    mats = scenes.CORNELL_SMALL_LIGHT_MATERIALS
    host = clpt.build_kd(v, c, nn)
    r.set_meshes(host)
    r.set_materials(mats, tm)
    _same_table(r.read_emitters(), on.build_emitters(host, mats, tm))
    assert int(r.read_emitters()["header"][0]) == 2

    r.build_meshes(v, c, nn)
    r.set_materials(scenes.CORNELL_MATERIALS, scenes.cornell(10)[3].tolist() + [3, 3])
    dev = r.download_kd()
    tm2 = np.array(scenes.cornell(10)[3].tolist() + [3, 3], dtype=np.int32)
    _same_table(r.read_emitters(), on.build_emitters(dev, scenes.CORNELL_MATERIALS, tm2))
    assert int(r.read_emitters()["header"][0]) == 202

    moved = v.copy()
    moved[-4:, 1] -= 0.05  # the lamp drops
    moved[-4:, 0] *= 1.5
    r.update_vertices(len(v) - 4, moved[-4:])
    r.rebuild_meshes()
    _same_table(r.read_emitters(), on.build_emitters(r.download_kd(), scenes.CORNELL_MATERIALS, tm2))

    m3 = scenes.CORNELL_MATERIALS.copy()
    m3[1, 4:7] = (0.5, 0.0, 0.25)  # the red wall now emits too, and the ceiling does not
    m3[3, 4:7] = 0
    r.set_materials(m3, tm2)
    _same_table(r.read_emitters(), on.build_emitters(r.download_kd(), m3, tm2))
    assert int(r.read_emitters()["header"][0]) == 200

    fv, fc, ftm, fmats = __import__("test_replay64")._floor_scene()
    small = clpt.build_kd(fv, fc)
    r.set_meshes(small)
    r.set_materials(fmats, ftm)
    dev = r.read_emitters()
    _same_table(dev, on.build_emitters(small, fmats, ftm))
    assert len(dev["map"]) == 4 and int(dev["header"][0]) == 2

    # tri_indices holds an emissive primitive past the leaves' runs: not listed, not light-sampled
    odd, otm, omats = unlisted_emitter_scene(clpt)
    r.set_meshes(odd)
    r.set_materials(omats, otm)
    dev = r.read_emitters()
    _same_table(dev, on.build_emitters(odd, omats, otm))
    assert int(dev["header"][0]) == 2 and dev["map"][4] == -1
    cam = clpt.cam_matrix(clpt.make_camera(**__import__("test_replay64").FLOOR_CAMERA), 24)
    r.set_camera_matrix(cam)
    r.create_image(32, 24)
    r.set_params(mode=3, depth=2, spp=4, seed=2, flags=clpt.FLAG_JITTER)
    r.execute()
    ref = on.render(odd, cam, 32, 24, depth=2, spp=4, seed=2, flags=clpt.FLAG_JITTER, materials=omats,
                    tri_material=otm, aov=False)
    assert _equal(r.read_image(), ref["rgba"])

    hv, hc, _ = scenes.heightfield(707, False)
    r.build_meshes(hv, hc)
    r.set_materials(scenes.CORNELL_MATERIALS[3:])
    dev = r.read_emitters()
    assert int(dev["header"][0]) == 999_698
    _same_table(dev, on.build_emitters(r.download_kd(), scenes.CORNELL_MATERIALS[3:]))


def _occluders(clpt, r, traversal):
    """Two spheres in the box, as instances (list or tree); [] for none."""
    if traversal is None:
        return []
    h = r.add_instance_mesh(*_mesh("icon"))
    mesh = r.download_instance_kd(h)
    o2w = np.stack([_o2w((0.3, 0.7, -0.2), (0.3, 0.3, 0.3), (0.3, 0.2, 0.1)),
                    _o2w((-0.5, 0.2, 0.9), (0.2, 0.2, 0.2), (-0.4, 0.5, -0.2))])
    r.set_instance_traversal(traversal)
    r.set_instance_arrays([h, h], o2w, [1, 2])
    return [(mesh, w, m) for w, m in zip(clpt.world_to_object_batch(o2w), [1, 2])]


@pytest.mark.parametrize("engine", [1, 2])
@pytest.mark.parametrize("spp", [1, 4, 64])
@pytest.mark.parametrize("traversal", [None, "list", "tree"])
def test_mode3_frames_equal_oracle(clpt, nee_renderer, traversal, spp, engine):
    from clpathtracer_b200 import scenes

    r = nee_renderer
    v, c, nn, tm = scenes.cornell_small_light(6)
    mats = scenes.CORNELL_SMALL_LIGHT_MATERIALS
    r.build_meshes(v, c, nn)
    base = r.download_kd()
    r.set_materials(mats, tm)
    inst = _occluders(clpt, r, traversal)
    tree = r.instance_tree() if traversal == "tree" else None
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H)
    kw = dict(depth=4, spp=spp, seed=7, flags=clpt.FLAG_JITTER if spp > 1 else 0)
    ref = on.render(base, cam, W, H, materials=mats, tri_material=tm, instances=inst, tree=tree, **kw)
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(cam)
    r.create_image(W, H, aov=True)
    for flags in (kw["flags"], kw["flags"] | clpt.FLAG_COUNTERS):
        r.set_params(mode=clpt.MODE_PATH_NEE, depth=4, spp=spp, seed=7, flags=flags)
        r.execute()
        assert clpt.lib().CLLastEngine() == engine
        prim, t, uv = r.read_aov()
        assert _equal(r.read_image(), ref["rgba"])
        assert np.array_equal(prim, ref["prim"])
        assert _equal(t, ref["t"]) and _equal(uv, ref["uv"])
        if flags & clpt.FLAG_COUNTERS:
            assert r.counters() == ref["counters"]
    m2 = ot.render(base, cam, W, H, mode=2, materials=mats, tri_material=tm, instances=inst, tree=tree, **kw)
    assert ref["counters"]["rays"] > m2["counters"]["rays"]  # the shadow rays


def test_mode3_progressive_and_sharded(clpt, oracle, nee_renderer):
    from clpathtracer_b200 import scenes

    r = nee_renderer
    L = clpt.lib()
    v, c, nn, tm = scenes.cornell_small_light(6)
    mats = scenes.CORNELL_SMALL_LIGHT_MATERIALS
    r.build_meshes(v, c, nn)
    base = r.download_kd()
    r.set_materials(mats, tm)
    inst = _occluders(clpt, r, "tree")
    tree = r.instance_tree()
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H)
    r.set_camera_matrix(cam)
    flags = clpt.FLAG_JITTER | clpt.FLAG_ACCUMULATE
    r.set_params(mode=3, depth=3, spp=2, seed=3, flags=flags)
    r.create_image(W, H)
    acc = oracle.new_accumulator(W, H)
    kw = dict(materials=mats, tri_material=tm, instances=inst, tree=tree, aov=False)
    for frame in range(3):
        r.execute()
        want = on.render(base, cam, W, H, depth=3, spp=2, seed=3, flags=flags, sample_base=2 * frame,
                         accumulate_into=acc, **kw)["rgba"]
    assert _equal(r.read_image(), want)
    full = on.render(base, cam, W, H, depth=3, **kw)["rgba"]
    r.set_params(mode=3, depth=3)
    for rank in range(2):
        r.create_image(W, H)
        L.CLSetTileShard(rank, 2, 8)
        r.execute()
        rows = np.array([y for y in range(H) if (y // 8) % 2 == rank])
        assert _equal(r.read_image()[rows], full[rows]), rank


@pytest.mark.parametrize("engine", [1, 2])
def test_without_emitters_mode3_is_mode2_on_the_device(clpt, nee_renderer, engine):
    from clpathtracer_b200 import scenes

    r = nee_renderer
    v, c, nn, tm = scenes.cornell(6)
    r.build_meshes(v, c, nn)
    mats = np.concatenate([scenes.CORNELL_MATERIALS, scenes.CORNELL_MATERIALS[3:]])
    mats[3, 4:7] = 0  # the ceiling goes dark; material 4 emits, on an instance only
    r.set_materials(mats, tm)
    _occluders(clpt, r, "list")
    r.set_instance_arrays([0, 0], [_o2w((0, 0, 0), (0.3, 0.3, 0.3), (0.3, 0.2, 0.1)),
                                   _o2w((0, 0, 0), (0.2, 0.2, 0.2), (-0.4, 0.5, -0.2))], [1, 4])
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H))
    r.create_image(W, H, aov=True)
    out = []
    for mode in (2, 3):
        r.set_params(mode=mode, depth=4, spp=4, seed=1, flags=clpt.FLAG_JITTER | clpt.FLAG_COUNTERS)
        r.execute()
        out.append((r.read_image(), *r.read_aov(), r.counters()))
    for a, b in zip(out[0][:4], out[1][:4]):
        assert _equal(a, b)
    assert out[0][4] == out[1][4]
    assert (out[1][0][..., 0] > 0).mean() > 0.3


def test_cuda_mode3_is_the_form_factor(clpt, nee_renderer):
    """The CUDA mode-3 estimate on the analytic floor with the occluder, 16 seeds x 256 samples per
    pixel (4,096 in all; the >= 64 spp launch that spreads a pixel over several warps), both engines."""
    r = nee_renderer
    scene, tm, mats, inst = _floor_with_occluder(clpt)
    quad = inst[0][0]
    w, h, spp, K = 128, 96, 256, 16
    cam, expected, shadowed, clear = floor_expectation(clpt, w, h)
    r.set_meshes(scene)
    r.set_materials(mats, tm)
    g = r.add_instance_mesh(quad.verts, quad.tris)
    r.set_instances([(g, np.eye(4), 2)])
    r.set_camera_matrix(cam)
    r.create_image(w, h)
    for engine in (1, 2):
        clpt.lib().CLSetEngine(engine)
        frames = []
        for k in range(K):
            r.set_params(mode=3, depth=2, spp=spp, seed=1000 + k)
            r.execute()
            frames.append(r.read_image()[..., 0].reshape(-1).astype(np.float64))
        nee_floor_statistic(np.array(frames), expected, shadowed, clear,
                            "cuda mode 3 engine %d %dx%d, %d x %d spp" % (engine, w, h, K, spp))


def test_mode4_is_rejected(clpt):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    prog = "import sys;sys.path.insert(0,%r);import clpathtracer_b200 as cl;r=cl.Renderer(0);r.set_params(mode=4)" % str(root)
    p = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True)
    assert p.returncode == 1 and "CLSetRenderParams: mode must be 0, 1, 2 or 3" in p.stderr, p.stderr
