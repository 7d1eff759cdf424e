"""The device-side kd builder and re-layout (CLBuildMeshes; SURVEY.md section 8f row 1).

The tree is built on the GPU in the reference's wire format (include/kd_tree.h:31-50),
downloaded, checked structurally on the host, walked by the oracle, and rendered by the
CUDA path from the device-side re-layout: the frames must be bit-identical.  The
device-side re-layout must produce the bytes of the host one (scene_pack.cpp) from the
same wire arrays, and two builds of the same mesh the same bytes.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _mesh(name):
    from clpathtracer_b200 import scenes

    if name == "cornell":
        return scenes.cornell(10)[:3]
    if name.startswith("soup"):
        return scenes.soup(int(name[4:]))
    with_n = name.endswith("n")
    return scenes.heightfield(int(name[2:-1] if with_n else name[2:]), with_n)


def _cam(clpt, which, height):
    from clpathtracer_b200 import scenes

    kw = {"canonical": scenes.CANONICAL_CAMERA, "cornell": scenes.CORNELL_CAMERA}[which]
    return clpt.cam_matrix(clpt.make_camera(**kw), height)


def _check_tree(s, exhaustive):
    """Any node order: reachability, boxes, leaf runs, coverage, ropes."""
    nodes = s.nodes
    n = len(nodes)
    split = nodes["type"] == 0
    leaf = nodes["type"] == 1
    assert np.all(split | leaf)
    kids = nodes["c"][split, :2]
    assert np.all((kids > 0) & (kids < n))
    seen = np.bincount(kids.reshape(-1), minlength=n)
    assert seen[0] == 0 and np.all(seen[1:] == 1)  # a tree: every node but the root has one parent
    assert leaf.sum() == split.sum() + 1
    ax = nodes["b"][split]
    plane = nodes["a"][split].view(np.float32)
    si = np.flatnonzero(split)
    assert np.all((ax >= 0) & (ax <= 2))
    lo_k, hi_k = kids[:, 0], kids[:, 1]
    r = np.arange(len(si))
    assert np.array_equal(nodes["max"][lo_k, ax], plane) and np.array_equal(nodes["min"][hi_k, ax], plane)
    assert np.all(nodes["min"][si, ax] < plane) and np.all(plane < nodes["max"][si, ax])
    for a2 in range(3):  # the other faces are inherited
        keep = ax != a2
        for k in (lo_k, hi_k):
            assert np.array_equal(nodes["min"][k[keep], a2], nodes["min"][si[keep], a2])
            assert np.array_equal(nodes["max"][k[keep], a2], nodes["max"][si[keep], a2])
    del r
    # leaf runs tile tri_indices without gaps or overlaps
    li = np.flatnonzero(leaf)
    first, cnt = nodes["a"][li], nodes["b"][li]
    assert np.all(cnt >= 0) and cnt.sum() == len(s.tri_indices)
    order = np.argsort(np.where(cnt > 0, first, np.iinfo(np.int32).max), kind="stable")
    f_sorted, c_sorted = first[order][cnt[order] > 0], cnt[order][cnt[order] > 0]
    assert np.array_equal(f_sorted, np.concatenate([[0], np.cumsum(c_sorted)[:-1]]))
    assert np.array_equal(np.unique(s.tri_indices), np.arange(s.n_tris))
    # coverage: a triangle whose bounds reach into the inside of a leaf is listed there
    tri_v = s.tris[:, 0].reshape(-1, 3)
    p = s.verts[tri_v][..., :3]
    tlo, thi = p.min(axis=1), p.max(axis=1)
    pick = li if exhaustive else li[:: max(1, len(li) // 400)]
    for i in pick:
        inside = np.all((tlo < nodes["max"][i, :3]) & (thi > nodes["min"][i, :3]), axis=1)
        listed = np.zeros(s.n_tris, dtype=bool)
        listed[s.tri_indices[nodes["a"][i]: nodes["a"][i] + nodes["b"][i]]] = True
        assert not np.any(inside & ~listed), f"leaf {i} misses {np.flatnonzero(inside & ~listed)[:5]}"
    # ropes: -1 or a node across the face that covers the leaf's extent there
    ropes = nodes["c"][li]
    assert np.all((ropes >= -1) & (ropes < n))
    for i in li[:: max(1, len(li) // 500)]:
        for f in range(6):
            rp = nodes["c"][i, f]
            a, hi = f // 2, f % 2
            if rp < 0:
                root_face = nodes["max"][0, a] if hi else nodes["min"][0, a]
                assert (nodes["max"][i, a] if hi else nodes["min"][i, a]) == root_face
                continue
            face = nodes["max"][i, a] if hi else nodes["min"][i, a]
            other = nodes["min"][rp, a] if hi else nodes["max"][rp, a]
            assert other == face
            for a2 in range(3):
                if a2 != a:
                    assert nodes["min"][rp, a2] <= nodes["min"][i, a2] and nodes["max"][rp, a2] >= nodes["max"][i, a2]


@pytest.mark.parametrize("name,camera,mode,depth,spp", [("hf22n", "canonical", 1, 3, 1), ("cornell", "cornell", 1, 5, 2),
                                                         ("soup3000", "cornell", 1, 4, 1), ("hf100", "canonical", 0, 2, 1),
                                                         ("hf224", "canonical", 1, 5, 4)])
def test_device_built_tree(clpt, oracle, renderer, name, camera, mode, depth, spp):
    v, c, n = _mesh(name)
    renderer.build_meshes(v, c, n)
    tree = renderer.download_kd()
    assert tree.n_tris == len(c) // 3
    _check_tree(tree, exhaustive=tree.n_tris <= 4000)
    st = tree.stats()
    assert st["leaf_tri_refs"] < 4 * tree.n_tris and st["max_leaf_tris"] <= 64
    # the frame rendered from the device-side re-layout equals the oracle's walk of the downloaded tree
    w, h = 320, 240
    cam = _cam(clpt, camera, h)
    flags = clpt.FLAG_JITTER if spp > 1 else 0
    renderer.set_camera_matrix(cam)
    renderer.set_params(mode=mode, depth=depth, spp=spp, seed=11, flags=flags)
    renderer.create_image(w, h, aov=True)
    renderer.execute()
    img = renderer.read_image()
    prim, t, uv = renderer.read_aov()
    ref = oracle.render(tree, cam, w, h, mode=mode, depth=depth, spp=spp, seed=11, flags=flags)
    assert np.array_equal(prim, ref["prim"])
    assert np.array_equal(img.view(np.uint32), ref["rgba"].view(np.uint32))
    assert (prim >= 0).mean() > 0.01
    # device re-layout == host re-layout of the same wire arrays, byte for byte
    dev = [renderer.read_packed(k) for k in range(5)]
    renderer.set_meshes(tree)  # CLSetMeshes: scene_pack.cpp
    host = [renderer.read_packed(k) for k in range(5)]
    for k, what in enumerate(("nodes", "leaves", "triangles", "start table", "flat normals")):
        assert dev[k].size == host[k].size and np.array_equal(dev[k], host[k]), what
    renderer.execute()
    assert np.array_equal(renderer.read_image().view(np.uint32), img.view(np.uint32))


def test_device_build_is_deterministic(clpt, renderer):
    v, c, n = _mesh("hf100")
    renderer.build_meshes(v, c, n)
    a = renderer.download_kd()
    v2, c2, n2 = _mesh("soup3000")
    renderer.build_meshes(v2, c2, n2)  # something else in between, workspace reused
    renderer.build_meshes(v, c, n)
    b = renderer.download_kd()
    assert a.nodes.tobytes() == b.nodes.tobytes() and a.tri_indices.tobytes() == b.tri_indices.tobytes()


@pytest.mark.parametrize("name", ["hf60", "soup3000", "hf224"])
def test_recorded_build_equals_level_by_level(clpt, renderer, monkeypatch, name):
    """Small meshes are built by replaying one recorded graph (level counts on the device, launches
    sized by capacities); the level-by-level path sizes every level exactly from counters read back.
    Same tree byte for byte -- also when the mesh outgrows the recorded capacities half way and the
    build starts over level by level, and on a replay."""
    v, c, n = _mesh(name)
    monkeypatch.delenv("CLPT_BUILD_NO_GRAPH", raising=False)
    monkeypatch.delenv("CLPT_BUILD_RECORD_ROOM", raising=False)
    renderer.build_meshes(v, c, n)
    assert renderer.build_was_recorded()
    a = renderer.download_kd()
    renderer.rebuild_meshes()  # the replay
    assert renderer.build_was_recorded()
    a2 = renderer.download_kd()
    monkeypatch.setenv("CLPT_BUILD_NO_GRAPH", "1")
    renderer.build_meshes(v, c, n)
    assert not renderer.build_was_recorded()
    b = renderer.download_kd()
    monkeypatch.delenv("CLPT_BUILD_NO_GRAPH")
    monkeypatch.setenv("CLPT_BUILD_RECORD_ROOM", "12")  # an eighth of the room: overflows some levels down
    renderer.build_meshes(v, c, n)
    assert not renderer.build_was_recorded()
    d = renderer.download_kd()
    for other in (a2, b, d):
        assert a.nodes.tobytes() == other.nodes.tobytes() and a.tri_indices.tobytes() == other.tri_indices.tobytes()
    _check_tree(a, exhaustive=False)


def test_update_vertices_and_rebuild(clpt, renderer):
    """Animated scenes: moving some vertices in place and rebuilding from the device-resident mesh
    gives the tree a fresh upload of the moved mesh gives."""
    v, c, n = _mesh("hf60")
    renderer.build_meshes(v, c, n)
    moved = v.copy()
    moved[100:400, 1] += np.float32(0.07)
    renderer.update_vertices(100, moved[100:400])
    renderer.rebuild_meshes()
    a = renderer.download_kd()
    renderer.build_meshes(moved, c, n)
    b = renderer.download_kd()
    assert a.nodes.tobytes() == b.nodes.tobytes() and a.tri_indices.tobytes() == b.tri_indices.tobytes()
    assert a.verts.tobytes() == b.verts.tobytes()
    _check_tree(a, exhaustive=False)


def test_device_build_quality_and_speed(clpt, renderer):
    """On a 100k-triangle mesh the device tree is in the class of the host SAH tree (within 2x
    of its triangle references) and is built in milliseconds, not the host's hundreds."""
    v, c, n = _mesh("hf224")
    renderer.build_meshes(v, c, n)
    renderer.build_meshes(v, c, n)  # second build: workspace is warm
    build_ms, pack_ms = renderer.build_ms()
    dev = renderer.download_kd().stats()
    host = clpt.build_kd_sah(v, c, n, intersect_cost=1.0, empty_bonus=0.9).stats()
    assert dev["leaf_tri_refs"] < 2 * host["leaf_tri_refs"], (dev, host)
    assert build_ms < 50.0 and pack_ms < 10.0, (build_ms, pack_ms)
    print("device build", build_ms, "ms, re-layout", pack_ms, "ms", dev, "host", host)


def test_host_and_device_layouts_take_turns(clpt, oracle, renderer, scene_cache, monkeypatch):
    """CLSetMeshes (host re-layout) and CLBuildMeshes / CLRebuildMeshes (device re-layout) write the
    same device buffers.  Taking turns in one renderer, a smaller scene after a bigger one, every
    frame is the oracle's walk of that step's tree and the layout has that tree's sizes; the
    automatic engine is the same whichever path laid out the same tree."""
    w, h = 160, 120
    renderer.set_params(mode=1, depth=2, spp=1, seed=5, flags=0)
    renderer.create_image(w, h, aov=True)

    def check(scene, camera):
        cam = _cam(clpt, camera, h)
        renderer.set_camera_matrix(cam)
        renderer.execute()
        img = renderer.read_image()
        prim, _, _ = renderer.read_aov()
        ref = oracle.render(scene, cam, w, h, mode=1, depth=2, seed=5)
        assert np.array_equal(prim, ref["prim"])
        assert np.array_equal(img.view(np.uint32), ref["rgba"].view(np.uint32))
        assert (prim >= 0).mean() > 0.01
        split = int((scene.nodes["type"] == 0).sum())
        n_nodes, n_leaves = 1 + 2 * split, len(scene.nodes) - split
        sizes = [renderer.read_packed(k).size for k in (0, 1, 2, 4)]
        assert sizes == [8 * n_nodes, 64 * n_leaves, 48 * len(scene.tri_indices), 16 * scene.n_tris]
        lut = renderer.read_packed(3).view(np.int32)
        assert lut.size > 0 and lut.min() >= 0 and lut.max() < n_nodes

    def device(name):
        renderer.build_meshes(*_mesh(name))
        return renderer.download_kd()

    host_big = scene_cache("hf224", sah=True)[0]
    renderer.set_meshes(host_big)
    check(host_big, "canonical")
    check(device("soup3000"), "cornell")
    host_small = scene_cache("hf22n")[0]
    assert len(host_small.nodes) < len(host_big.nodes)
    renderer.set_meshes(host_small)
    check(host_small, "canonical")
    check(device("hf60"), "canonical")
    renderer.rebuild_meshes()
    check(renderer.download_kd(), "canonical")

    # engine policy: a shallow device tree of more than CLPT_FAT_ENGINE_MIN_REFS (500,000) triangle
    # slots in fat leaves, then the same tree through the host path
    from clpathtracer_b200 import scenes

    monkeypatch.delenv("CLPT_ENGINE", raising=False)
    L = clpt.lib()
    L.CLSetEngine(0)
    renderer.set_camera_matrix(_cam(clpt, "canonical", h))
    L.CLSetBuildParams(12, 2, 1.0, 1.0, 0.9)
    try:
        renderer.build_meshes(*scenes.heightfield(520, False))  # 540,800 triangles
    finally:
        L.CLSetBuildParams(0, 2, 1.0, 1.0, 0.9)  # the defaults (kd_build_gpu.h)
    renderer.execute()
    assert L.CLLastEngine() == 2
    renderer.set_meshes(renderer.download_kd())
    renderer.execute()
    assert L.CLLastEngine() == 2


def test_device_build_rejects_bad_mesh(clpt):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    code = ("import sys;sys.path.insert(0,%r);import numpy as np;import clpathtracer_b200 as cl;"
            "from clpathtracer_b200 import scenes;v,c,n=scenes.heightfield(6,False);c=c.copy();c[5,0]=10**6;"
            "r=cl.Renderer(0);r.build_meshes(v,c,n)") % str(root)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert p.returncode == 1 and "invalid scene" in p.stderr and "missing vertex" in p.stderr, p.stderr
