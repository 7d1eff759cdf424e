"""ctypes bindings for the rigid-instance oracle (oracle_instances.c) -- TEST INFRASTRUCTURE.

Only tests/ and profiles/experiments/ import this.  `render` takes the arguments of
oracle_py.render plus `instances`, and with no instances returns what oracle_py.render returns.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from oracle.oracle_py import COUNTER_NAMES, FLAG_ACCUMULATE, FLAG_JITTER, OracleParams, new_accumulator  # noqa: F401

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_instances.so"
SOURCES = [HERE / "oracle_instances.c", HERE / "oracle_kernel.c"]


class OracleInstance(C.Structure):
    _fields_ = [("nodes", C.c_void_p), ("tri_indices", C.c_void_p), ("tris", C.c_void_p),
                ("verts", C.c_void_p), ("norms", C.c_void_p), ("w2o", C.c_float * 12),
                ("material", C.c_int32), ("prim_offset", C.c_int32)]


_lib = None


def build(force: bool = False) -> None:
    """Compiled like liboracle.so (oracle/Makefile): one rounding per fp32 operation."""
    if force or not LIB.exists() or any(s.stat().st_mtime > LIB.stat().st_mtime for s in SOURCES):
        subprocess.run(["gcc", "-std=c11", "-O2", "-fPIC", "-ffp-contract=off", "-fopenmp", "-w", "-shared",
                        "-o", str(LIB), str(SOURCES[0]), "-lm"], check=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB), mode=C.RTLD_LOCAL)
        L.oracle_render_instanced.restype = C.c_int
        L.oracle_render_instanced.argtypes = [C.POINTER(OracleParams), C.c_void_p, C.c_int32]
        L.oracle_sizeof_params.restype = C.c_size_t
        L.oracle_sizeof_instance.restype = C.c_size_t
        assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
        assert L.oracle_sizeof_instance() == C.sizeof(OracleInstance)
        _lib = L
    return _lib


def render(scene, cam: np.ndarray, width: int, height: int, mode: int = 0, depth: int = 2, spp: int = 1,
           seed: int = 0, flags: int = 0, rows=None, threads: int = 0, max_leaf_visits: int = 4096,
           materials: np.ndarray | None = None, tri_material: np.ndarray | None = None,
           sample_base: int = 0, aov: bool = True, accumulate_into: np.ndarray | None = None,
           instances=()) -> dict:
    """oracle_py.render with rigid instances: [(Scene, world_to_object float32[3,4], material), ...],
    walked after the base scene (oracle_instances.c header).  Instance k's primitive ids start at
    scene.n_tris + the triangles of the instances before it."""
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
    table = (OracleInstance * max(1, len(instances)))()
    offset = scene.n_tris
    for k, (mesh, w2o, material) in enumerate(instances):
        I = table[k]
        I.nodes, I.tri_indices = mesh.nodes.ctypes.data, mesh.tri_indices.ctypes.data
        I.tris, I.verts = mesh.tris.ctypes.data, mesh.verts.ctypes.data
        I.norms = mesh.norms.ctypes.data if len(mesh.norms) else None
        I.w2o[:] = [float(x) for x in np.asarray(w2o, dtype=np.float32).reshape(12)]
        I.material, I.prim_offset = int(material), offset
        offset += mesh.n_tris
        keep.append(mesh)
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
    rc = L.oracle_render_instanced(C.byref(P), C.addressof(table), len(instances))
    assert rc == 0
    out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in P.counters]))
    return out
