"""ctypes bindings for the light-sampling oracle (oracle_nee.c) -- TEST INFRASTRUCTURE.

Only tests/ and profiles/experiments/ import this.  `build_emitters` is the CPU twin of the device's
emitter table; `render` takes the arguments of oracle_instance_tree_py.render and renders mode 3
(CLPT_MODE_PATH_NEE) with the twin's table; `occluded` answers shadow-ray queries.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from clpathtracer_b200 import EMITTER_DTYPE
from oracle import oracle_instances_py as oi
from oracle.oracle_py import COUNTER_NAMES, FLAG_ACCUMULATE, OracleParams, new_accumulator

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_nee.so"
SOURCES = [HERE / "oracle_nee.c", HERE / "oracle_instance_tree.c", HERE / "oracle_instances.c",
           HERE / "oracle_kernel.c"]


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
        vp = C.c_void_p
        L.oracle_build_emitters.restype = C.c_int
        L.oracle_build_emitters.argtypes = [C.POINTER(OracleParams), C.c_int32, C.c_int32, vp, vp, vp, vp]
        L.oracle_render_nee.restype = C.c_int
        L.oracle_render_nee.argtypes = [C.POINTER(OracleParams), vp, C.c_int32, vp, vp, vp, vp, vp]
        L.oracle_occluded_rays.restype = C.c_int
        L.oracle_occluded_rays.argtypes = [C.POINTER(OracleParams), vp, C.c_int32, vp, vp, C.c_int32, vp]
        L.oracle_select_emitter.restype = C.c_uint64
        L.oracle_select_emitter.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint32]
        L.oracle_sizeof_params.restype = C.c_size_t
        L.oracle_sizeof_instance.restype = C.c_size_t
        assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
        assert L.oracle_sizeof_instance() == C.sizeof(oi.OracleInstance)
        _lib = L
    return _lib


def _params(scene, materials, tri_material, keep):
    P = OracleParams()
    P.nodes = scene.nodes.ctypes.data
    P.tri_indices = scene.tri_indices.ctypes.data
    P.tris = scene.tris.ctypes.data
    P.verts = scene.verts.ctypes.data
    P.norms = scene.norms.ctypes.data if len(scene.norms) else None
    if materials is not None:
        m = np.ascontiguousarray(materials, dtype=np.float32).reshape(-1, 8)
        keep.append(m)
        P.materials, P.n_materials = m.ctypes.data, len(m)
        if tri_material is not None:
            tm = np.ascontiguousarray(tri_material, dtype=np.int32)
            keep.append(tm)
            P.tri_material = tm.ctypes.data
    return P


def build_emitters(scene, materials=None, tri_material=None) -> dict:
    """The twin's emitter table of a wire-format scene: header uint64[2] = (n, Q), records
    EMITTER_DTYPE[n], cdf uint64[n] (exclusive prefix sums of the integer weights), map int32[prims]."""
    keep = []
    P = _params(scene, materials, tri_material, keep)
    n_prims = scene.n_tris
    rec = np.zeros(max(n_prims, 1), dtype=EMITTER_DTYPE)
    cdf = np.zeros(n_prims + 1, dtype=np.uint64)
    emap = np.zeros(max(n_prims, 1), dtype=np.int32)
    hdr = np.zeros(2, dtype=np.uint64)
    assert lib().oracle_build_emitters(C.byref(P), len(scene.nodes), n_prims, rec.ctypes.data, cdf.ctypes.data,
                                       emap.ctypes.data, hdr.ctypes.data) == 0
    n = int(hdr[0])
    return {"header": hdr, "records": rec[:n].copy(), "cdf": cdf[:n].copy(), "map": emap[:n_prims].copy(),
            "_cdf_full": cdf, "_rec_full": rec, "_map_full": emap}


def select(emitters: dict, words) -> np.ndarray:
    """The emitter index each 32-bit word selects in the light sample (oracle_select_emitter)."""
    cdf = emitters["_cdf_full"]
    n, Q = int(emitters["header"][0]), int(emitters["header"][1])
    assert n >= 1 and Q > 0
    return np.array([lib().oracle_select_emitter(cdf.ctypes.data, n, Q, int(w)) for w in words], dtype=np.int64)


def _instance_table(scene, instances):
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
    return table


def render(scene, cam: np.ndarray, width: int, height: int, depth: int = 2, spp: int = 1, seed: int = 0,
           flags: int = 0, rows=None, threads: int = 0, max_leaf_visits: int = 4096,
           materials: np.ndarray | None = None, tri_material: np.ndarray | None = None, sample_base: int = 0,
           aov: bool = True, accumulate_into: np.ndarray | None = None, instances=(),
           tree: np.ndarray | None = None, emitters: dict | None = None) -> dict:
    """A mode-3 frame (the arguments of oracle_instance_tree_py.render; `emitters` defaults to the
    twin's table of this scene and materials)."""
    L = lib()
    keep = []
    P = _params(scene, materials, tri_material, keep)
    camf = np.ascontiguousarray(cam, dtype=np.float32).reshape(16)
    P.cam = camf.ctypes.data
    P.width, P.height = width, height
    P.y0, P.y1 = (0, height) if rows is None else rows
    P.mode, P.depth, P.spp, P.flags = 3, depth, spp, flags
    P.seed, P.sample_base = seed, sample_base
    P.max_leaf_visits, P.threads = max_leaf_visits, threads
    E = emitters if emitters is not None else build_emitters(scene, materials, tri_material)
    table = _instance_table(scene, instances)
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
    rc = L.oracle_render_nee(C.byref(P), C.addressof(table), len(instances),
                             None if tree is None else tree.ctypes.data, E["_rec_full"].ctypes.data,
                             E["_cdf_full"].ctypes.data, E["_map_full"].ctypes.data, E["header"].ctypes.data)
    assert rc == 0
    out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in P.counters]))
    return out


def occluded(scene, rays: np.ndarray, instances=(), tree: np.ndarray | None = None,
             max_leaf_visits: int = 4096) -> np.ndarray:
    """The shadow-ray query for rays float32[n, 7] (origin, direction, t_max): bool[n], True when
    a triangle is accepted with 0 < t < t_max (or the rope-hop budget runs out)."""
    keep = []
    P = _params(scene, None, None, keep)
    P.max_leaf_visits = max_leaf_visits
    table = _instance_table(scene, instances)
    q = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 7)
    out = np.zeros(len(q), dtype=np.int32)
    assert lib().oracle_occluded_rays(C.byref(P), C.addressof(table), len(instances),
                                      None if tree is None else np.ascontiguousarray(tree).ctypes.data,
                                      q.ctypes.data, len(q), out.ctypes.data) == 0
    return out.astype(bool)
