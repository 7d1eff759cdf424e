"""ctypes bindings for the environment oracle (oracle_env.c) -- TEST INFRASTRUCTURE.

Only tests/ and profiles/experiments/ import this.  `build_env` is the CPU twin of the device's
environment table; `lookup` and `draw` expose env(d) and the light sample's draw; `render` takes the
arguments of oracle_nee_py.render plus `mode` (2 or 3) and `env` and renders with the environment.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from oracle import oracle_nee_py as on
from oracle.oracle_py import COUNTER_NAMES, FLAG_ACCUMULATE, OracleParams, new_accumulator

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_env.so"
SOURCES = [HERE / "oracle_env.c", HERE / "oracle_nee.c", HERE / "oracle_instance_tree.c", HERE / "oracle_instances.c",
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
        L.oracle_build_env.restype = C.c_int
        L.oracle_build_env.argtypes = [vp, C.c_int32, vp, vp, vp]
        L.oracle_render_env.restype = C.c_int
        L.oracle_render_env.argtypes = [C.POINTER(OracleParams), vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp]
        L.oracle_env_lookup.restype = C.c_int
        L.oracle_env_lookup.argtypes = [C.c_int32, vp, C.c_int32, vp, vp]
        L.oracle_env_draw.restype = C.c_int
        L.oracle_env_draw.argtypes = [vp, vp, vp, vp, C.c_int32, vp, vp, vp, vp]
        L.oracle_sizeof_params.restype = C.c_size_t
        assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
        _lib = L
    return _lib


def build_env(cube: np.ndarray) -> dict:
    """The twin's table of a cube float32 [6, n, n, 3]: header uint64[2] = (n, Q), texels
    float32[6 n^2, 4] (r, g, b, pdf), cdf uint64[6 n^2] (exclusive prefix sums of the weights)."""
    cube = np.ascontiguousarray(cube, dtype=np.float32)
    n = cube.shape[1]
    assert cube.shape == (6, n, n, 3)
    T = 6 * n * n
    tex = np.zeros((T, 4), dtype=np.float32)
    cdf = np.zeros(T + 1, dtype=np.uint64)
    hdr = np.zeros(2, dtype=np.uint64)
    assert lib().oracle_build_env(cube.ctypes.data, n, tex.ctypes.data, cdf.ctypes.data, hdr.ctypes.data) == 0
    return {"header": hdr, "texels": tex, "cdf": cdf[:T].copy(), "_cdf_full": cdf}


def lookup(n: int, dirs: np.ndarray):
    """env(d) for float32 directions [k, 3]: (texel int64[k], a float32[k], b float32[k])."""
    d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
    texel = np.zeros(len(d), dtype=np.int64)
    ab = np.zeros((len(d), 2), dtype=np.float32)
    assert lib().oracle_env_lookup(n, d.ctypes.data, len(d), texel.ctypes.data, ab.ctypes.data) == 0
    return texel, ab[:, 0], ab[:, 1]


def draw(table: dict, words: np.ndarray):
    """The light sample's draw for uint32 words [k, 3] (r0, r1, r2): (texel, a, b, l float32[k, 3],
    pe float32[k] the solid-angle density of l)."""
    w = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, 3)
    k = len(w)
    texel, ab, l, pe = (np.zeros(k, np.int64), np.zeros((k, 2), np.float32), np.zeros((k, 3), np.float32),
                        np.zeros(k, np.float32))
    assert lib().oracle_env_draw(table["texels"].ctypes.data, table["_cdf_full"].ctypes.data,
                                 table["header"].ctypes.data, w.ctypes.data, k, texel.ctypes.data, ab.ctypes.data,
                                 l.ctypes.data, pe.ctypes.data) == 0
    return texel, ab[:, 0], ab[:, 1], l, pe


def render(scene, cam: np.ndarray, width: int, height: int, env, mode: int = 3, depth: int = 2, spp: int = 1,
           seed: int = 0, flags: int = 0, rows=None, threads: int = 0, max_leaf_visits: int = 4096,
           materials: np.ndarray | None = None, tri_material: np.ndarray | None = None, sample_base: int = 0,
           aov: bool = True, accumulate_into: np.ndarray | None = None, instances=(),
           tree: np.ndarray | None = None, emitters: dict | None = None) -> dict:
    """A mode-2 or mode-3 frame with the environment `env` (a cube or build_env's table); the other
    arguments are oracle_nee_py.render's."""
    assert mode in (2, 3)
    V = env if isinstance(env, dict) else build_env(env)
    L = lib()
    keep = []
    P = on._params(scene, materials, tri_material, keep)
    camf = np.ascontiguousarray(cam, dtype=np.float32).reshape(16)
    P.cam = camf.ctypes.data
    P.width, P.height = width, height
    P.y0, P.y1 = (0, height) if rows is None else rows
    P.mode, P.depth, P.spp, P.flags = mode, depth, spp, flags
    P.seed, P.sample_base = seed, sample_base
    P.max_leaf_visits, P.threads = max_leaf_visits, threads
    E = emitters if emitters is not None else on.build_emitters(scene, materials, tri_material)
    table = on._instance_table(scene, instances)
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
    rc = L.oracle_render_env(C.byref(P), C.addressof(table), len(instances),
                             None if tree is None else tree.ctypes.data, E["_rec_full"].ctypes.data,
                             E["_cdf_full"].ctypes.data, E["_map_full"].ctypes.data, E["header"].ctypes.data,
                             V["texels"].ctypes.data, V["_cdf_full"].ctypes.data, V["header"].ctypes.data)
    assert rc == 0
    out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in P.counters]))
    return out

