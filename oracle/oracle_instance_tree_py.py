"""ctypes bindings for the instance-tree oracle (oracle_instance_tree.c) -- TEST INFRASTRUCTURE.

Only tests/ and profiles/experiments/ import this.  `build_tree` is the CPU twin of the device's
tree builder; `render` takes the arguments of oracle_instances_py.render plus `tree` (a node array,
the device's or the twin's) and walks it; with tree=None it is oracle_instances_py.render.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from clpathtracer_b200 import INSTANCE_TREE_DTYPE
from oracle import oracle_instances_py as oi
from oracle.oracle_py import COUNTER_NAMES, FLAG_ACCUMULATE, FLAG_JITTER, OracleParams, new_accumulator  # noqa: F401

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_instance_tree.so"
SOURCES = [HERE / "oracle_instance_tree.c", HERE / "oracle_instances.c", HERE / "oracle_kernel.c"]

# the node record of CLDebugReadInstanceTree
NODE_DTYPE = INSTANCE_TREE_DTYPE

_lib = None


def build(force: bool = False) -> None:
    """Compiled like liboracle.so (oracle/Makefile): one rounding per fp32 and fp64 operation."""
    if force or not LIB.exists() or any(s.stat().st_mtime > LIB.stat().st_mtime for s in SOURCES):
        subprocess.run(["gcc", "-std=c11", "-O2", "-fPIC", "-ffp-contract=off", "-fopenmp", "-w", "-shared",
                        "-o", str(LIB), str(SOURCES[0]), "-lm"], check=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB), mode=C.RTLD_LOCAL)
        L.oracle_render_instance_tree.restype = C.c_int
        L.oracle_render_instance_tree.argtypes = [C.POINTER(OracleParams), C.c_void_p, C.c_int32, C.c_void_p]
        L.oracle_build_instance_tree.restype = C.c_int
        L.oracle_build_instance_tree.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.oracle_sizeof_params.restype = C.c_size_t
        L.oracle_sizeof_instance.restype = C.c_size_t
        assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
        assert L.oracle_sizeof_instance() == C.sizeof(oi.OracleInstance)
        _lib = L
    return _lib


def root_box(mesh) -> np.ndarray:
    """float32[6]: the root box of a wire-format tree (min xyz, max xyz), what the walks clip against."""
    return np.concatenate([mesh.nodes[0]["min"][:3], mesh.nodes[0]["max"][:3]]).astype(np.float32)


def build_tree(w2o: np.ndarray, roots: np.ndarray) -> np.ndarray:
    """The twin's tree over n >= 1 instances: w2o float32[n,3,4], roots float32[n,6] (root_box of
    each instance's mesh).  NODE_DTYPE[max(n - 1, 1)]."""
    w = np.ascontiguousarray(w2o, dtype=np.float32).reshape(-1, 12)
    r = np.ascontiguousarray(roots, dtype=np.float32).reshape(-1, 6)
    assert len(w) == len(r) >= 1
    out = np.zeros(max(len(w) - 1, 1), dtype=NODE_DTYPE)
    assert lib().oracle_build_instance_tree(w.ctypes.data, r.ctypes.data, len(w), out.ctypes.data) == 0
    return out


def tree_of(instances) -> np.ndarray:
    """build_tree for [(Scene, world_to_object, material), ...], render's `instances`."""
    return build_tree(np.stack([np.asarray(w, dtype=np.float32) for _, w, _ in instances]),
                      np.stack([root_box(m) for m, _, _ in instances]))


def render(scene, cam: np.ndarray, width: int, height: int, mode: int = 0, depth: int = 2, spp: int = 1,
           seed: int = 0, flags: int = 0, rows=None, threads: int = 0, max_leaf_visits: int = 4096,
           materials: np.ndarray | None = None, tri_material: np.ndarray | None = None,
           sample_base: int = 0, aov: bool = True, accumulate_into: np.ndarray | None = None,
           instances=(), tree: np.ndarray | None = None) -> dict:
    """oracle_instances_py.render walking the instance tree `tree` (NODE_DTYPE; None = the list)."""
    L = lib()
    P = OracleParams()
    camf = np.ascontiguousarray(cam, dtype=np.float32).reshape(16)
    keep = [camf]
    P.nodes = scene.nodes.ctypes.data
    P.tri_indices = scene.tri_indices.ctypes.data
    P.tris = scene.tris.ctypes.data
    P.verts = scene.verts.ctypes.data
    P.norms = scene.norms.ctypes.data if len(scene.norms) else None
    P.cam = camf.ctypes.data
    P.width, P.height = width, height
    P.y0, P.y1 = (0, height) if rows is None else rows
    P.mode, P.depth, P.spp, P.flags = mode, depth, spp, flags
    P.seed, P.sample_base = seed, sample_base
    P.max_leaf_visits, P.threads = max_leaf_visits, threads
    if materials is not None:
        m = np.ascontiguousarray(materials, dtype=np.float32).reshape(-1, 8)
        keep.append(m)
        P.materials, P.n_materials = m.ctypes.data, len(m)
        if tri_material is not None:
            tm = np.ascontiguousarray(tri_material, dtype=np.int32)
            keep.append(tm)
            P.tri_material = tm.ctypes.data
    table = (oi.OracleInstance * max(1, len(instances)))()
    offset = scene.n_tris
    for k, (mesh, w2o, material) in enumerate(instances):
        I = table[k]
        I.nodes, I.tri_indices = mesh.nodes.ctypes.data, mesh.tri_indices.ctypes.data
        I.tris, I.verts = mesh.tris.ctypes.data, mesh.verts.ctypes.data
        I.norms = mesh.norms.ctypes.data if len(mesh.norms) else None
        C.memmove(I.w2o, np.ascontiguousarray(w2o, dtype=np.float32).reshape(12).ctypes.data, 48)
        I.material, I.prim_offset = int(material), offset
        offset += mesh.n_tris
    if tree is not None:
        tree = np.ascontiguousarray(tree)
        assert tree.dtype.itemsize == 64 and len(tree) == max(len(instances) - 1, 1)
    out = {}
    rgba = np.zeros((height, width, 4), dtype=np.float32)
    out["rgba"] = rgba
    P.rgba = rgba.ctypes.data
    if flags & FLAG_ACCUMULATE:
        if accumulate_into is None:
            accumulate_into = new_accumulator(width, height)
        assert accumulate_into.dtype == np.uint64 and accumulate_into.shape == (height, width, 4)
        out["accum"] = accumulate_into
        P.accum = accumulate_into.ctypes.data
    if aov:
        out["prim"] = np.full((height, width), -1, dtype=np.int32)
        out["t"] = np.zeros((height, width), dtype=np.float32)
        out["uv"] = np.zeros((height, width, 2), dtype=np.float32)
        out["normal"] = np.zeros((height, width, 3), dtype=np.float32)
        P.prim_id, P.t_hit = out["prim"].ctypes.data, out["t"].ctypes.data
        P.uv, P.normal = out["uv"].ctypes.data, out["normal"].ctypes.data
        out["path_edge"] = np.full((height, width), 2.0, dtype=np.float32)
        P.path_edge = out["path_edge"].ctypes.data
    rc = L.oracle_render_instance_tree(C.byref(P), C.addressof(table), len(instances),
                                       None if tree is None else tree.ctypes.data)
    assert rc == 0
    out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in P.counters]))
    return out
