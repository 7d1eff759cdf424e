"""Environment lighting (modes 2 and 3) on the device: the environment table equals the CPU twin byte
for byte, and every frame with an environment equals the environment oracle (oracle/oracle_env.c) bit
for bit -- colours, first-hit primitive, t, u, v and the work counters -- on both engines, at 1, 4
and 64 samples per pixel, with no instances, the instance list and the instance tree, with and
without triangle emitters, progressive and row-tile sharded.  The analytic floor checks the estimate
itself; bad input is rejected."""
import numpy as np
import pytest

from oracle import oracle_env_py as oe
from test_gpu_instances import inst_renderer  # noqa: F401
from test_gpu_nee import _occluders
from test_oracle_env import env_floor_expectation, env_floor_scene, env_floor_statistic, _sun_sky, ENV_N, SUN

pytestmark = pytest.mark.gpu

W, H = 64, 48


@pytest.fixture
def env_renderer(inst_renderer):
    yield inst_renderer
    inst_renderer.set_environment(None)
    inst_renderer.set_instance_traversal("list")


def _equal(a, b):
    return np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()


def _same_table(dev, twin):
    assert np.array_equal(dev["header"], twin["header"])
    assert _equal(dev["texels"], twin["texels"])
    assert _equal(dev["cdf"], twin["cdf"])


def test_device_table_equals_twin(env_renderer):
    r = env_renderer
    rng = np.random.default_rng(1)
    for n in (1, 7, 64, 2048):
        cube = rng.exponential(1.0, (6, n, n, 3)).astype(np.float32)
        cube[2, n // 2, n // 3] = 1e4  # a sun
        r.set_environment(cube)
        _same_table(r.read_environment(), oe.build_env(cube))
    small = _sun_sky(8, SUN)  # a smaller one after the largest
    r.set_environment(small)
    _same_table(r.read_environment(), oe.build_env(small))
    zero = np.zeros((6, 3, 3, 3), dtype=np.float32)
    r.set_environment(zero)
    _same_table(r.read_environment(), oe.build_env(zero))
    r.set_environment(None)
    cleared = r.read_environment()
    assert np.array_equal(cleared["header"], [0, 0]) and len(cleared["texels"]) == 0 and len(cleared["cdf"]) == 0


def _scene(clpt, r, emitters):
    from clpathtracer_b200 import scenes

    v, c, nn, tm = scenes.cornell_small_light(6)
    mats = scenes.CORNELL_SMALL_LIGHT_MATERIALS.copy()
    if not emitters:
        mats[3, 4:7] = 0
    r.build_meshes(v, c, nn)
    base = r.download_kd()
    r.set_materials(mats, tm)
    return base, mats, tm


@pytest.mark.parametrize("engine", [1, 2])
@pytest.mark.parametrize("spp", [1, 4, 64])
@pytest.mark.parametrize("traversal", [None, "list", "tree"])
@pytest.mark.parametrize("mode", [2, 3])
def test_env_frames_equal_oracle(clpt, env_renderer, mode, traversal, spp, engine):
    """The Cornell box with its open side (-z) towards the sky: the camera sees out of it and light
    comes in through it."""
    from clpathtracer_b200 import scenes

    r = env_renderer
    emitters = spp != 4  # with and without triangle emitters
    base, mats, tm = _scene(clpt, r, emitters)
    inst = _occluders(clpt, r, traversal)
    tree = r.instance_tree() if traversal == "tree" else None
    env = _sun_sky(16, SUN) if spp != 64 else oe_cube_sun_behind_camera()
    r.set_environment(env)
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H)
    kw = dict(depth=4, spp=spp, seed=7, flags=clpt.FLAG_JITTER if spp > 1 else 0)
    ref = oe.render(base, cam, W, H, env, mode=mode, materials=mats, tri_material=tm, instances=inst, tree=tree, **kw)
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(cam)
    r.create_image(W, H, aov=True)
    for flags in (kw["flags"], kw["flags"] | clpt.FLAG_COUNTERS):
        r.set_params(mode=mode, depth=4, spp=spp, seed=7, flags=flags)
        r.execute()
        assert clpt.lib().CLLastEngine() == engine
        prim, t, uv = r.read_aov()
        assert _equal(r.read_image(), ref["rgba"])
        assert np.array_equal(prim, ref["prim"])
        assert _equal(t, ref["t"]) and _equal(uv, ref["uv"])
        if flags & clpt.FLAG_COUNTERS:
            assert r.counters() == ref["counters"]
    assert (prim < 0).mean() > 0.02  # some camera rays leave through the open side


def oe_cube_sun_behind_camera():
    """A coloured sky whose sun lies behind the camera (-z), shining into the box."""
    from clpathtracer_b200 import scenes

    return scenes.sun_sky(16, (0.1, 0.3, -1.0), 0.05, (900.0, 800.0, 600.0), (0.4, 0.6, 1.0), (0.3, 0.25, 0.2))


def test_env_progressive_and_sharded(clpt, oracle, env_renderer):
    from clpathtracer_b200 import scenes

    r = env_renderer
    L = clpt.lib()
    base, mats, tm = _scene(clpt, r, True)
    inst = _occluders(clpt, r, "tree")
    tree = r.instance_tree()
    env = oe_cube_sun_behind_camera()
    r.set_environment(env)
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H)
    r.set_camera_matrix(cam)
    flags = clpt.FLAG_JITTER | clpt.FLAG_ACCUMULATE
    r.set_params(mode=3, depth=3, spp=2, seed=3, flags=flags)
    r.create_image(W, H)
    acc = oracle.new_accumulator(W, H)
    kw = dict(materials=mats, tri_material=tm, instances=inst, tree=tree, aov=False)
    for frame in range(3):
        r.execute()
        want = oe.render(base, cam, W, H, env, depth=3, spp=2, seed=3, flags=flags, sample_base=2 * frame,
                         accumulate_into=acc, **kw)["rgba"]
    assert _equal(r.read_image(), want)
    full = oe.render(base, cam, W, H, env, depth=3, **kw)["rgba"]
    r.set_params(mode=3, depth=3)
    for rank in range(2):
        r.create_image(W, H)
        L.CLSetTileShard(rank, 2, 8)
        r.execute()
        rows = np.array([y for y in range(H) if (y // 8) % 2 == rank])
        assert _equal(r.read_image()[rows], full[rows]), rank


@pytest.mark.parametrize("engine", [1, 2])
def test_clearing_and_all_ones_give_the_frame_without(clpt, env_renderer, engine):
    """Setting and clearing an environment gives the frame rendered before it was set (modes 2 and
    3); mode 2 with an all-ones environment is mode 2 without one, bit for bit."""
    from clpathtracer_b200 import scenes

    r = env_renderer
    _scene(clpt, r, True)
    _occluders(clpt, r, "list")
    clpt.lib().CLSetEngine(engine)
    r.set_camera_matrix(clpt.cam_matrix(clpt.make_camera(**scenes.CORNELL_CAMERA), H))
    r.create_image(W, H, aov=True)

    def frame(mode):
        r.set_params(mode=mode, depth=4, spp=4, seed=1, flags=clpt.FLAG_JITTER | clpt.FLAG_COUNTERS)
        r.execute()
        return (r.read_image(), *r.read_aov(), r.counters())

    def same(a, b):
        for x, y in zip(a[:4], b[:4]):
            assert _equal(x, y)
        assert a[4] == b[4]

    before = {m: frame(m) for m in (2, 3)}
    r.set_environment(oe_cube_sun_behind_camera())
    assert not _equal(frame(2)[0], before[2][0])
    r.set_environment(None)
    for m in (2, 3):
        same(frame(m), before[m])
    r.set_environment(np.ones((6, 5, 5, 3), dtype=np.float32))
    same(frame(2), before[2])


def test_cuda_floor_under_sun_and_sky(clpt, env_renderer):
    """Both modes on the analytic floor, 16 seeds x 256 samples per pixel (4,096 in all), both engines."""
    r = env_renderer
    scene, tm, mats, inst = env_floor_scene(clpt, 1.0)
    quad = inst[0][0]
    w, h, spp, K = 128, 96, 256, 16
    cam, expected, shadowed, clear, _ = env_floor_expectation(clpt, ENV_N, SUN, w, h)
    r.set_meshes(scene)
    r.set_materials(mats, tm)
    g = r.add_instance_mesh(quad.verts, quad.tris)
    r.set_instances([(g, np.eye(4), 1)])
    r.set_environment(_sun_sky(ENV_N, SUN))
    r.set_camera_matrix(cam)
    r.create_image(w, h)
    for engine in (1, 2):
        clpt.lib().CLSetEngine(engine)
        for mode, spp in ((2, 4 * spp), (3, spp)):  # mode 2 finds the sun by chance: more samples
            frames = []
            for k in range(K):
                r.set_params(mode=mode, depth=2, spp=spp, seed=1000 + k)
                r.execute()
                frames.append(r.read_image()[..., 0].reshape(-1).astype(np.float64))
            env_floor_statistic(np.array(frames), expected, clear | shadowed,
                                "cuda mode %d engine %d %dx%d, %d x %d spp" % (mode, engine, w, h, K, spp))


@pytest.mark.parametrize("case,message", [
    ("n=0", "face_size must be in"), ("n=2049", "face_size must be in"), ("bytes", "bytes must be"),
    ("nan", "finite and not negative"), ("inf", "finite and not negative"), ("negative", "finite and not negative")])
def test_bad_environment_is_rejected(clpt, case, message):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    body = {
        "n=0": "c=np.ones((6,2,2,3),np.float32);r.L.CLSetEnvironment(c.ctypes.data,c.nbytes,0)",
        "n=2049": "c=np.ones(18,np.float32);r.L.CLSetEnvironment(c.ctypes.data,6*2049*2049*12,2049)",
        "bytes": "c=np.ones((6,2,2,3),np.float32);r.L.CLSetEnvironment(c.ctypes.data,c.nbytes-4,2)",
        "nan": "c=np.ones((6,2,2,3),np.float32);c[3,1,0,2]=np.nan;r.set_environment(c)",
        "inf": "c=np.ones((6,2,2,3),np.float32);c[0,0,0,0]=np.inf;r.set_environment(c)",
        "negative": "c=np.ones((6,2,2,3),np.float32);c[5,1,1,1]=-1e-30;r.set_environment(c)",
    }[case]
    prog = "import sys;sys.path.insert(0,%r);import numpy as np;import clpathtracer_b200 as cl;r=cl.Renderer(0);%s" % (
        str(root), body)
    p = subprocess.run([sys.executable, "-c", prog], capture_output=True, text=True)
    assert p.returncode == 1 and "CLSetEnvironment: " in p.stderr and message in p.stderr, p.stderr

