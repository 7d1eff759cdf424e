"""ctypes bindings for the checker libraries -- TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs import this.  Nothing under clpathtracer_b200/ does.

  liboracle.so            CPU restatement of src/kernel.cl (oracle_kernel.c)
  _ref/libref_host.so     the reference's own host code, compiled unmodified
                          from the checkout $CLPT_REFERENCE names (Makefile
                          target `ref`); present only where it was built
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_LIB = HERE / "liboracle.so"
REF_LIB = HERE / "_ref" / "libref_host.so"

FLAG_JITTER, FLAG_ACCUMULATE = 1, 2


class OracleParams(C.Structure):
    _fields_ = [
        ("nodes", C.c_void_p), ("tri_indices", C.c_void_p), ("tris", C.c_void_p),
        ("verts", C.c_void_p), ("norms", C.c_void_p), ("cam", C.c_void_p),
        ("width", C.c_int32), ("height", C.c_int32), ("y0", C.c_int32), ("y1", C.c_int32),
        ("mode", C.c_int32), ("depth", C.c_int32), ("spp", C.c_int32), ("flags", C.c_int32),
        ("seed", C.c_uint32), ("sample_base", C.c_uint32),
        ("max_leaf_visits", C.c_int32), ("threads", C.c_int32),
        ("materials", C.c_void_p), ("tri_material", C.c_void_p),
        ("n_materials", C.c_int32), ("reserved", C.c_int32),
        ("rgba", C.c_void_p), ("prim_id", C.c_void_p), ("t_hit", C.c_void_p),
        ("uv", C.c_void_p), ("normal", C.c_void_p), ("path_edge", C.c_void_p), ("accum", C.c_void_p),
        ("counters", C.c_uint64 * 6),
    ]


_oracle = None
_ref = None


def build(force: bool = False) -> None:
    if force or not ORACLE_LIB.exists():
        subprocess.run(["make", "-s", "-C", str(HERE), "oracle"], check=True)


def oracle() -> C.CDLL:
    global _oracle
    if _oracle is None:
        build()
        L = C.CDLL(str(ORACLE_LIB), mode=C.RTLD_LOCAL)
        L.oracle_render.restype = C.c_int
        L.oracle_render.argtypes = [C.POINTER(OracleParams)]
        L.oracle_sizeof_params.restype = C.c_size_t
        L.oracle_num_threads.restype = C.c_int
        L.oracle_host_cores.restype = C.c_int
        L.oracle_philox.restype = None
        L.oracle_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        assert L.oracle_sizeof_params() == C.sizeof(OracleParams)
        _oracle = L
    return _oracle


def have_ref() -> bool:
    return REF_LIB.exists()


def ref() -> C.CDLL:
    """The reference's own host functions (list/vector/matrix/camera/kd_tree/model)."""
    global _ref
    if _ref is None:
        L = C.CDLL(str(REF_LIB), mode=C.RTLD_LOCAL)
        vp, sz = C.c_void_p, C.c_size_t
        L.new_list.restype, L.new_list.argtypes = vp, [sz]
        L.init_list.restype, L.init_list.argtypes = vp, [sz, sz]
        L.list_size.restype, L.list_size.argtypes = sz, [vp]
        L.delete_list.restype, L.delete_list.argtypes = None, [vp]
        L.ref_cam_matrix_ptr.restype, L.ref_cam_matrix_ptr.argtypes = None, [vp, C.c_int, vp]
        L.ref_sizeof_kdnode.restype = sz
        L.ref_sizeof_camera.restype = sz
        _ref = L
    return _ref


def philox(ctr, key) -> np.ndarray:
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    oracle().oracle_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return out


def new_accumulator(width: int, height: int) -> np.ndarray:
    """Zeroed progressive state for render(..., flags=FLAG_ACCUMULATE, accumulate_into=...)."""
    return np.zeros((height, width, 4), dtype=np.uint64)


COUNTER_NAMES = ["rays", "splits", "leaves", "tris", "shade_vn", "capped"]


def render(scene, cam: np.ndarray, width: int, height: int, mode: int = 0, depth: int = 2, spp: int = 1,
           seed: int = 0, flags: int = 0, rows=None, threads: int = 0, max_leaf_visits: int = 4096,
           materials: np.ndarray | None = None, tri_material: np.ndarray | None = None,
           sample_base: int = 0, aov: bool = True, accumulate_into: np.ndarray | None = None) -> dict:
    """Render with the CPU restatement.  `scene` has numpy members nodes (68-byte
    records), tri_indices, tris (3t,4) int32, verts (v,4), norms (k,4) -- the wire
    format.  Returns rgba (h,w,4), prim (h,w), t (h,w), uv (h,w,2), normal (h,w,3)
    and the work counters."""
    L = oracle()
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
    out = {}
    rgba = np.zeros((height, width, 4), dtype=np.float32)
    out["rgba"] = rgba
    P.rgba = rgba.ctypes.data
    if flags & FLAG_ACCUMULATE:
        # progressive: `accumulate_into` is the uint64[h, w, 4] running state (fixed-point sums of
        # r, g, b and the sample count); out["rgba"] is the mean after this call, rows rendered only
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
    rc = L.oracle_render(C.byref(P))
    assert rc == 0
    out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in P.counters]))
    return out


# ---------------------------------------------------------------- Harness C
# The reference's own kernel.cl through an OpenCL ICD (cl_harness.c).
REF_KERNEL_LIB = HERE / "_ref" / "libref_kernel.so"
_refk = None


def _ref_kernel():
    global _refk
    if _refk is None:
        import os

        if "OCL_ICD_FILENAMES" not in os.environ and "OCL_ICD_VENDORS" not in os.environ:
            for cand in ("/usr/lib/libnvidia-opencl.so.1", "/usr/local/nvidia/lib/libnvidia-opencl.so.1",
                         "/usr/lib/x86_64-linux-gnu/libnvidia-opencl.so.1"):
                if Path(cand).exists():
                    os.environ["OCL_ICD_FILENAMES"] = cand
                    break
        L = C.CDLL(str(REF_KERNEL_LIB), mode=C.RTLD_LOCAL)
        L.refcl_available.restype, L.refcl_available.argtypes = C.c_int, [C.c_char_p, C.c_int]
        L.refcl_render.restype = C.c_int
        L.refcl_render.argtypes = [C.c_void_p, C.c_size_t] * 5 + [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                                 C.POINTER(C.c_double), C.c_char_p, C.c_int]
        L.refcl_render_depth.restype = C.c_int
        L.refcl_render_depth.argtypes = [C.c_void_p, C.c_size_t] * 5 + [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                                       C.c_void_p, C.POINTER(C.c_double), C.c_char_p,
                                                                       C.c_int]
        L.refcl_bounce_source.restype, L.refcl_bounce_source.argtypes = C.c_void_p, [C.c_int]
        L.refcl_free.restype, L.refcl_free.argtypes = None, [C.c_void_p]
        L.refcl_build_options.restype = C.c_char_p
        _refk = L
    return _refk


def ref_kernel_available() -> tuple[bool, str]:
    """(usable, 'platform / device' or the reason it is not)."""
    if not REF_KERNEL_LIB.exists():
        return False, "oracle/_ref/libref_kernel.so not built (needs $CLPT_REFERENCE at build time)"
    msg = C.create_string_buffer(512)
    rc = _ref_kernel().refcl_available(msg, 512)
    return rc == 0, msg.value.decode(errors="replace")


def ref_kernel_bounce_source(depth: int) -> str:
    """The text the vendor compiler is given for a bounce render (cl_harness.c:
    trace_ray cloned `depth` times with the early return removed)."""
    L = _ref_kernel()
    p = L.refcl_bounce_source(depth)
    if not p:
        raise RuntimeError("bounce rewrite failed: kernel.cl does not have the expected text")
    try:
        return C.string_at(p).decode()
    finally:
        L.refcl_free(p)


def ref_kernel_render(scene, cam: np.ndarray, width: int, height: int, repeats: int = 1, bounce_depth: int = 0):
    """One frame of the reference kernel.  bounce_depth 0: UNMODIFIED, as shipped
    (first-hit normal colour).  bounce_depth D >= 1: the reference's dead mirror
    bounce (src/kernel.cl:399-417) made runnable by the textual clone in
    cl_harness.c, trace depth D (the literal at :468 is 2).
    Returns (rgba float32[h,w,4], kernel_ms)."""
    L = _ref_kernel()
    camf = np.ascontiguousarray(cam, dtype=np.float32).reshape(16)
    out = np.zeros((height, width, 4), dtype=np.float32)
    ms = C.c_double(0)
    log = C.create_string_buffer(16384)
    norms = scene.norms if len(scene.norms) else None
    rc = L.refcl_render_depth(scene.nodes.ctypes.data, scene.nodes.nbytes, scene.tri_indices.ctypes.data,
                              scene.tri_indices.nbytes, scene.tris.ctypes.data, scene.tris.nbytes,
                              scene.verts.ctypes.data, scene.verts.nbytes,
                              None if norms is None else norms.ctypes.data, 0 if norms is None else norms.nbytes,
                              camf.ctypes.data, width, height, repeats, bounce_depth, out.ctypes.data,
                              C.byref(ms), log, 16384)
    if rc != 0:
        raise RuntimeError("reference kernel run failed: " + log.value.decode(errors="replace"))
    return out, ms.value


def ref_kernel_build_options() -> str:
    return _ref_kernel().refcl_build_options().decode()
