"""clpathtracer_b200 -- Python host mirror of the CLState.h render boundary.

The product is ``libclpt.so`` (C host code + hand-written CUDA for sm_100a,
see ``include/*.h``).  This package is the thin host side used by the tests
and ``bench.py``: it loads the library through ctypes and exposes the
reference's own entry points under their own names (``CLInit``,
``CLSetMeshes`` ... ``CLExecute``, ``build_kd``, ``cam_matrix``, ``LoadModel``)
with numpy arrays standing in for the reference's fat-pointer lists.

There is no CPU fallback: if the library is missing, importing works but the
first call raises; if no CUDA device exists, ``CLInit`` aborts the process the
way the reference aborts on an OpenCL error.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
# $CLPT_LIB selects another build of the same library (kernel experiments)
LIB_PATH = Path(os.environ["CLPT_LIB"]) if os.environ.get("CLPT_LIB") else PKG / "libclpt.so"

# ---------------------------------------------------------------- wire types
KDNODE_DTYPE = np.dtype(
    {
        "names": ["min", "max", "type", "a", "b", "c"],
        "formats": [("<f4", 4), ("<f4", 4), "<i4", "<i4", "<i4", ("<i4", 6)],
        "offsets": [0, 16, 32, 36, 40, 44],
        "itemsize": 68,
    }
)
"""68-byte packed node (include/clpt_types.h).  For a split: a = float bits of
the plane, b = axis, c[0:2] = children.  For a leaf: a = first slot in
tri_indices, b = triangle count, c[0:6] = ropes."""

MODE_NORMAL, MODE_MIRROR, MODE_PATH, MODE_PATH_NEE = 0, 1, 2, 3
READ_FLOAT4, READ_RGBA8 = 0, 1
FLAG_JITTER, FLAG_ACCUMULATE, FLAG_COUNTERS = 1, 2, 4


class Vector4(C.Structure):
    _fields_ = [("s", C.c_float * 4)]


class Matrix(C.Structure):
    _fields_ = [("rows", Vector4 * 4)]


class Camera(C.Structure):
    # Near, Far, FOV, 4 bytes of padding (Position is 16-aligned), Position, Forward
    _fields_ = [("Near", C.c_float), ("Far", C.c_float), ("FOV", C.c_float), ("_pad", C.c_float),
                ("Position", Vector4), ("Forward", Vector4)]


class KD(C.Structure):
    _fields_ = [("node_vec", C.c_void_p), ("tri_indices", C.c_void_p), ("vert_vec", C.c_void_p),
                ("norm_vec", C.c_void_p), ("tri_vec", C.c_void_p)]


class KDStats(C.Structure):
    _fields_ = [("leaf_tri_refs", C.c_longlong), ("leaf_count", C.c_longlong),
                ("empty_leaves", C.c_longlong), ("node_count", C.c_longlong),
                ("max_leaf_tris", C.c_int), ("max_depth", C.c_int)]


class CLMaterial(C.Structure):
    _fields_ = [("albedo", C.c_float * 3), ("kind", C.c_int), ("emission", C.c_float * 3),
                ("pad", C.c_float)]


MAX_INSTANCES = 64
MAX_TREE_INSTANCES = 1 << 20
INSTANCES_LIST, INSTANCES_TREE = 0, 1

INSTANCE_TREE_DTYPE = np.dtype(
    {
        "names": ["min0", "ref0", "max0", "pad0", "min1", "ref1", "max1", "pad1"],
        "formats": [("<f4", 3), "<i4", ("<f4", 3), "<i4", ("<f4", 3), "<i4", ("<f4", 3), "<i4"],
        "offsets": [0, 12, 16, 28, 32, 44, 48, 60],
        "itemsize": 64,
    }
)
"""Instance-tree node (CLDebugReadInstanceTree): the boxes of child 0 and child 1 and their
references; ref >= 0 is an internal node, ref < 0 is instance -1 - ref.  Node 0 is the root."""


EMITTER_DTYPE = np.dtype({"names": ["v0", "prim", "e1", "pa", "e2", "pad0", "n", "pad1"],
                          "formats": [("<f4", 3), "<i4", ("<f4", 3), "<f4", ("<f4", 3), "<f4", ("<f4", 3), "<f4"],
                          "offsets": [0, 12, 16, 28, 32, 44, 48, 60], "itemsize": 64})
"""Emitter record (CLDebugReadEmitters): v0, primitive id, e1 = v1 - v0, the emitter's area pdf
(selection probability / area), e2 = v2 - v0, and its flat normal."""


class CLInstance(C.Structure):
    """One rigid instance (CLState.h): world_to_object is the row-major 3x4 [A | b]."""
    _fields_ = [("world_to_object", C.c_float * 12), ("mesh", C.c_int), ("material", C.c_int),
                ("pad", C.c_int * 2)]


def world_to_object(object_to_world) -> np.ndarray:
    """float32[3,4] [A | b] of the inverse of a 3x4 or 4x4 affine object-to-world matrix,
    inverted in float64."""
    m = np.asarray(object_to_world, dtype=np.float64)
    full = np.eye(4)
    full[:3, :] = m[:3, :4]
    return np.linalg.inv(full)[:3, :].astype(np.float32)


def world_to_object_batch(object_to_world) -> np.ndarray:
    """world_to_object of every matrix of float[n,3,4] or float[n,4,4], in one batched float64
    inversion; the same float32 bytes as world_to_object matrix by matrix."""
    m = np.asarray(object_to_world, dtype=np.float64)
    full = np.broadcast_to(np.eye(4), (len(m), 4, 4)).copy()
    full[:, :3, :] = m[:, :3, :4]
    return np.linalg.inv(full)[:, :3, :].astype(np.float32)


CLINSTANCE_DTYPE = np.dtype({"names": ["world_to_object", "mesh", "material", "pad"],
                             "formats": [("<f4", 12), "<i4", "<i4", ("<i4", 2)],
                             "offsets": [0, 48, 52, 56], "itemsize": 64})


_lib = None


def lib() -> C.CDLL:
    """The loaded libclpt.so.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m clpathtracer_b200.build` "
            "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for the render path.")
    L = C.CDLL(str(LIB_PATH), mode=C.RTLD_LOCAL)
    vp, sz, i, f, u = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_uint
    sig = {
        # lists
        "new_list": (vp, [sz]), "init_list": (vp, [sz, sz]), "delete_list": (None, [vp]),
        "list_size": (sz, [vp]), "copy_list": (vp, [vp]),
        # camera / kd / models
        "cam_matrix_ptr": (None, [C.POINTER(Camera), i, C.POINTER(Matrix)]),
        "build_kd_ex": (KD, [vp, vp, vp, C.c_char_p, i, i]),
        "build_kd": (KD, [vp, vp, vp, C.c_char_p]),
        "build_kd_sah": (KD, [vp, vp, vp, C.c_char_p, i, i, f, f, f]),
        "parse_kd": (i, [C.c_char_p, C.POINTER(KD)]),
        "write_kd": (i, [C.c_char_p, C.POINTER(KD)]),
        "delete_kd": (None, [KD]),
        "kd_get_stats": (None, [C.POINTER(KD), C.POINTER(KDStats)]),
        "LoadModel": (i, [C.c_char_p, C.POINTER(KD)]),
        "load_obj_lists": (i, [C.c_char_p, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
        "write_obj": (i, [C.c_char_p, vp, vp, vp]),
        "kd_set_build_params": (None, [i, i]), "kd_set_sah_clip": (None, [i]),
        "AddPhysObject": (None, [vp, vp]), "PhysStep": (None, [C.c_double]), "PhysTerminate": (None, []),
        # boundary
        "CLInit": (None, [C.c_char_p, C.c_char_p]), "CLTerminate": (None, []),
        "CLSetCameraMatrixPtr": (None, [C.POINTER(Matrix)]),
        "CLSetObjects": (None, [vp, sz]), "CLSetMeshes": (None, [vp]),
        "CLSetMeshesRaw": (None, [vp, sz, vp, sz, vp, sz, vp, sz, vp, sz]),
        "CLSetMaterials": (None, [vp, sz, vp, sz]),
        "CLBuildMeshes": (None, [vp, sz, vp, sz, vp, sz]), "CLSetBuildParams": (None, [i, i, f, f, f]),
        "CLLastBuildMs": (None, [C.POINTER(f), C.POINTER(f)]), "CLBuildStats": (None, [C.POINTER(i), C.POINTER(i), C.POINTER(i)]),
        "CLLastBuildWasRecorded": (i, []),
        "CLDownloadKd": (None, [C.POINTER(KD)]), "CLDebugReadPacked": (sz, [i, vp, sz]),
        "CLAddInstanceMesh": (i, [vp, sz, vp, sz, vp, sz]), "CLSetInstances": (None, [vp, sz]),
        "CLClearInstanceMeshes": (None, []), "CLDownloadInstanceKd": (None, [i, C.POINTER(KD)]),
        "CLSetInstanceTraversal": (None, [i]), "CLInstanceTraversal": (i, []),
        "CLDebugReadInstanceTree": (sz, [vp, sz]), "CLLastInstanceBuildMs": (None, [C.POINTER(f)]),
        "CLDebugReadEmitters": (sz, [i, vp, sz]),
        "CLSetEnvironment": (None, [vp, sz, i]), "CLDebugReadEnvironment": (sz, [i, vp, sz]),
        "CLUpdateVertices": (None, [sz, vp, sz]), "CLRebuildMeshes": (None, []),
        "CLDeleteImage": (None, []), "CLCreateImage": (None, [u]), "CLExecute": (None, [i, i]),
        "CLSelectDevice": (None, [i]), "CLSetRenderParams": (None, [i, i, i, u, i]),
        "CLSetMaxLeafVisits": (None, [i]), "CLSetEngine": (None, [i]), "CLLastEngine": (i, []), "CLCreateImageHeadless": (None, [i, i]),
        "CLResetAccumulation": (None, []), "CLReadImage": (None, [vp, sz]),
        "CLReadImageRGBA8": (None, [vp, sz]), "CLReadImageAsync": (None, [vp, sz, i]), "CLReadImageWait": (None, [i]),
        "CLEnableAOV": (None, [i]), "CLReadAOV": (None, [vp, vp, vp]),
        "CLGetCounters": (None, [vp]), "CLLastKernelMs": (f, []), "CLLastLaunchCount": (i, []),
        "CLEventRecord": (None, [i]), "CLEventElapsedMs": (f, [i, i]), "CLFlushL2": (None, []),
        "CLDistGetUniqueId": (None, [vp]), "CLDistInit": (None, [i, i, vp, i]),
        "CLDistShutdown": (None, []), "CLDistDirectPlacement": (i, []), "CLSetTileShard": (None, [i, i, i]),
        "CLDeviceName": (C.c_char_p, []), "CLDeviceSMCount": (i, []),
    }
    for name, (res, args) in sig.items():
        try:
            fn = getattr(L, name)
        except AttributeError:
            if os.environ.get("CLPT_LIB"):  # an experimental / older build selected on purpose: bind what it has
                continue
            raise
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


# ------------------------------------------------------------ list <-> numpy
def to_list(arr: np.ndarray | None) -> int:
    """Copy a numpy array into a freshly allocated fat-pointer list."""
    L = lib()
    if arr is None:
        return L.new_list(0)
    a = np.ascontiguousarray(arr)
    p = L.init_list(a.nbytes, 1)
    if a.nbytes:
        C.memmove(p, a.ctypes.data, a.nbytes)
    return p


def from_list(ptr: int, dtype, cols: int | None = None) -> np.ndarray:
    """Copy a fat-pointer list out into a numpy array."""
    L = lib()
    dt = np.dtype(dtype)
    if not ptr:
        out = np.zeros(0, dtype=dt)
    else:
        n = L.list_size(ptr)
        out = np.empty(n // dt.itemsize, dtype=dt)
        if n:
            C.memmove(out.ctypes.data, ptr, n)  # (string_at cannot take sizes past 2 GiB)
    return out.reshape(-1, cols) if cols else out


class Scene:
    """A model in the reference's wire format, as numpy arrays.

    nodes  : KDNODE_DTYPE[n]       (68-byte records, preorder)
    tri_indices : int32[r]
    tris   : int32[3*t, 4]         one {v, vn, vt, pad} per corner
    verts  : float32[v, 4]
    norms  : float32[k, 4]         may be empty
    """

    def __init__(self, nodes, tri_indices, tris, verts, norms):
        self.nodes = np.ascontiguousarray(nodes, dtype=KDNODE_DTYPE)
        self.tri_indices = np.ascontiguousarray(tri_indices, dtype=np.int32)
        self.tris = np.ascontiguousarray(tris, dtype=np.int32).reshape(-1, 4)
        self.verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 4)
        self.norms = np.ascontiguousarray(norms, dtype=np.float32).reshape(-1, 4)

    @property
    def n_tris(self) -> int:
        return len(self.tris) // 3

    @classmethod
    def from_kd(cls, k: KD, free: bool = True) -> "Scene":
        s = cls(from_list(k.node_vec, KDNODE_DTYPE), from_list(k.tri_indices, np.int32),
                from_list(k.tri_vec, np.int32, 4), from_list(k.vert_vec, np.float32, 4),
                from_list(k.norm_vec, np.float32, 4))
        if free:
            lib().delete_kd(k)
        return s

    def to_kd(self) -> KD:
        """Fresh C lists holding a copy of this scene (caller/CLSetMeshes owns them)."""
        return KD(to_list(self.nodes), to_list(self.tri_indices), to_list(self.verts),
                  to_list(self.norms), to_list(self.tris))

    def stats(self) -> dict:
        leaf = self.nodes["type"] == 1
        cnt = self.nodes["b"][leaf]
        return {"nodes": int(len(self.nodes)), "leaves": int(leaf.sum()),
                "empty_leaves": int((cnt == 0).sum()), "leaf_tri_refs": int(cnt.sum()),
                "max_leaf_tris": int(cnt.max()) if len(cnt) else 0, "tris": self.n_tris}


def corners_from_faces(faces: np.ndarray, with_normals: bool) -> np.ndarray:
    """(t,3) vertex ids -> (3t,4) corner records {v, vn, vt, 0}.  Without
    normals the vn/vt slots carry the loader's 'missing' value (negative)."""
    faces = np.asarray(faces, dtype=np.int64).reshape(-1)
    out = np.zeros((len(faces), 4), dtype=np.int32)
    out[:, 0] = faces
    out[:, 1] = faces if with_normals else np.int32(-2147483648)
    out[:, 2] = np.int32(-2147483648)
    return out


def build_kd(verts: np.ndarray, corners: np.ndarray, norms: np.ndarray | None = None,
             depth: int = 15, nbins: int = 25, path: str | None = None) -> Scene:
    """kd-tree build (clpt_host.h build_kd_ex; reference src/kd_tree.c:202-276).
    verts (v,3|4) float32, corners (3t,4) int32, norms (k,3|4) float32 or None."""
    L = lib()
    v4 = _as_vec4(verts)
    n4 = _as_vec4(norms) if norms is not None and len(norms) else None
    k = L.build_kd_ex(to_list(np.ascontiguousarray(corners, dtype=np.int32)), to_list(v4), to_list(n4),
                      path.encode() if path else None, depth, nbins)
    return Scene.from_kd(k)


def build_kd_sah(verts: np.ndarray, corners: np.ndarray, norms: np.ndarray | None = None,
                 max_depth: int | None = None, nbins: int = 32, traversal_cost: float = 1.0,
                 intersect_cost: float = 1.0, empty_bonus: float = 0.9, path: str | None = None,
                 clip: bool = True) -> Scene:
    """SAH kd-tree (extension, clpt_host.h build_kd_sah): same wire format and ropes.
    nbins <= 0: candidate planes on every triangle bound (exact sweep); clip: perfect splits."""
    L = lib()
    L.kd_set_sah_clip(1 if clip else 0)
    v4 = _as_vec4(verts)
    n4 = _as_vec4(norms) if norms is not None and len(norms) else None
    if max_depth is None:
        max_depth = int(8 + 1.3 * np.log2(max(len(corners) // 3, 2)))
    k = L.build_kd_sah(to_list(np.ascontiguousarray(corners, dtype=np.int32)), to_list(v4), to_list(n4),
                       path.encode() if path else None, max_depth, nbins, traversal_cost, intersect_cost,
                       empty_bonus)
    return Scene.from_kd(k)


def _as_vec4(a: np.ndarray) -> np.ndarray:
    a = np.asarray(a, dtype=np.float32)
    if a.ndim == 2 and a.shape[1] == 4:
        return np.ascontiguousarray(a)
    out = np.zeros((len(a), 4), dtype=np.float32)
    out[:, :3] = a.reshape(-1, 3)
    return out


def load_model(filename: str) -> Scene:
    """LoadModel (include/model.h:6-7): .obj (build + cache .kd) or .kd."""
    k = KD()
    if lib().LoadModel(filename.encode(), C.byref(k)):
        raise RuntimeError(f"LoadModel failed for {filename}")
    return Scene.from_kd(k)


def make_camera(near=0.1, far=1.0, fov=np.pi / 3, position=(0, 0.1, -0.2), forward=(0, 0, 1)) -> Camera:
    cam = Camera()
    cam.Near, cam.Far, cam.FOV = float(near), float(far), float(fov)
    for k in range(3):
        cam.Position.s[k] = float(np.float32(position[k]))
        cam.Forward.s[k] = float(np.float32(forward[k]))
    return cam


def cam_matrix(cam: Camera, height: int) -> np.ndarray:
    """inverse(device * projection * view) as float32[4,4] (src/camera.c:62-70)."""
    m = Matrix()
    lib().cam_matrix_ptr(C.byref(cam), int(height), C.byref(m))
    return np.frombuffer(bytes(m), dtype=np.float32).reshape(4, 4).copy()


# ------------------------------------------------------------ the boundary
class Renderer:
    """One process = one device = one renderer (the library state is a
    singleton, like the reference's).  Thin sugar over the C entry points; the
    call order is the reference's: init -> set meshes -> per frame
    {set camera, execute} (src/game.c:219-260)."""

    def __init__(self, device: int | None = None):
        self.L = lib()
        if device is not None:
            self.L.CLSelectDevice(int(device))
        self.L.CLInit(b"src/kernel.cl", b"render")
        self.width = self.height = 0
        self._keep = None

    def set_meshes(self, scene: Scene) -> None:
        s = scene
        self.L.CLSetMeshesRaw(s.nodes.ctypes.data, s.nodes.nbytes, s.tri_indices.ctypes.data,
                              s.tri_indices.nbytes, s.tris.ctypes.data, s.tris.nbytes,
                              s.verts.ctypes.data, s.verts.nbytes,
                              s.norms.ctypes.data if len(s.norms) else None, s.norms.nbytes)

    def set_meshes_owned(self, scene: Scene) -> None:
        """The reference's own CLSetMeshes(kd *models): a list.c vector of kd whose
        first element's lists become the library's."""
        k = scene.to_kd()
        models = self.L.init_list(1, C.sizeof(KD))
        C.memmove(models, C.byref(k), C.sizeof(KD))
        self.L.CLSetMeshes(models)
        self.L.delete_list(models)  # the caller frees only the outer list (src/game.c:177-178)

    def build_meshes(self, verts: np.ndarray, corners: np.ndarray, norms: np.ndarray | None = None) -> None:
        """Upload a mesh and build its kd-tree on the device (CLBuildMeshes)."""
        v4 = _as_vec4(verts)
        c4 = np.ascontiguousarray(corners, dtype=np.int32).reshape(-1, 4)
        n4 = _as_vec4(norms) if norms is not None and len(norms) else None
        self.L.CLBuildMeshes(v4.ctypes.data, v4.nbytes, c4.ctypes.data, c4.nbytes,
                             None if n4 is None else n4.ctypes.data, 0 if n4 is None else n4.nbytes)

    def update_vertices(self, first: int, verts: np.ndarray) -> None:
        """Overwrite vertices [first, first + len(verts)) of the mesh uploaded by build_meshes."""
        v4 = _as_vec4(verts)
        self.L.CLUpdateVertices(int(first), v4.ctypes.data, v4.nbytes)

    def rebuild_meshes(self) -> None:
        self.L.CLRebuildMeshes()

    def download_kd(self) -> "Scene":
        """The device-built tree as a Scene (wire format) for the oracle."""
        k = KD()
        self.L.CLDownloadKd(C.byref(k))
        return Scene.from_kd(k)

    def add_instance_mesh(self, verts: np.ndarray, corners: np.ndarray, norms: np.ndarray | None = None) -> int:
        """Upload a mesh and build its tree on the device once (CLAddInstanceMesh); returns its handle."""
        v4 = _as_vec4(verts)
        c4 = np.ascontiguousarray(corners, dtype=np.int32).reshape(-1, 4)
        n4 = _as_vec4(norms) if norms is not None and len(norms) else None
        return int(self.L.CLAddInstanceMesh(v4.ctypes.data, v4.nbytes, c4.ctypes.data, c4.nbytes,
                                            None if n4 is None else n4.ctypes.data, 0 if n4 is None else n4.nbytes))

    def set_instances(self, instances) -> None:
        """The instances of the next frames: [(mesh handle, object_to_world 3x4 or 4x4, material), ...]
        (material only matters in mode 2).  The matrices are inverted here, in float64; an empty
        list removes every instance."""
        table = (CLInstance * len(instances))()
        for k, (mesh, o2w, material) in enumerate(instances):
            table[k].world_to_object[:] = [float(x) for x in world_to_object(o2w).reshape(12)]
            table[k].mesh, table[k].material = int(mesh), int(material)
        self.L.CLSetInstances(C.addressof(table) if instances else None, C.sizeof(table))

    def set_instance_arrays(self, meshes, object_to_world, materials) -> None:
        """set_instances from arrays: mesh handles int[n], object_to_world float[n,3,4] or
        float[n,4,4], materials int[n] (or one int for all), inverted in one batched float64 call."""
        n = len(object_to_world)
        table = np.zeros(n, dtype=CLINSTANCE_DTYPE)
        if n:
            table["world_to_object"] = world_to_object_batch(object_to_world).reshape(n, 12)
        table["mesh"] = meshes
        table["material"] = materials
        self.L.CLSetInstances(table.ctypes.data if n else None, table.nbytes)

    def set_instance_traversal(self, traversal: str) -> None:
        """"list" (the default) or "tree" (CLSetInstanceTraversal), from the next frame on."""
        self.L.CLSetInstanceTraversal({"list": INSTANCES_LIST, "tree": INSTANCES_TREE}[traversal])

    def instance_traversal(self) -> str:
        return ["list", "tree"][self.L.CLInstanceTraversal()]

    def instance_tree(self) -> np.ndarray:
        """The instance tree's nodes (INSTANCE_TREE_DTYPE), built first if stale; empty without instances."""
        n = self.L.CLDebugReadInstanceTree(None, 0)
        out = np.zeros(n // 64, dtype=INSTANCE_TREE_DTYPE)
        if n:
            self.L.CLDebugReadInstanceTree(out.ctypes.data, n)
        return out

    def read_emitters(self) -> dict:
        """The emitter table of mode 3 (CLDebugReadEmitters), built first if stale: header uint64[2]
        (emitter count n, total weight Q), records EMITTER_DTYPE[n], cdf uint64[n] (exclusive prefix
        sums of the integer weights), map int32[primitives] (emitter of each base primitive or -1)."""
        out = {}
        for which, name, dtype in ((0, "header", np.uint64), (1, "records", EMITTER_DTYPE), (2, "cdf", np.uint64),
                                   (3, "map", np.int32)):
            n = self.L.CLDebugReadEmitters(which, None, 0)
            a = np.zeros(n // np.dtype(dtype).itemsize, dtype=dtype)
            if n:
                self.L.CLDebugReadEmitters(which, a.ctypes.data, n)
            out[name] = a
        return out

    def set_environment(self, cube: np.ndarray | None) -> None:
        """The environment of modes 2 and 3 (CLSetEnvironment): float32 [6][n][n][3] linear RGB
        radiance, faces +X, -X, +Y, -Y, +Z, -Z in the OpenGL cube-map convention (envmap.py), or
        None for the constant white sky.  Invalid input ends the process with a message."""
        if cube is None:
            self.L.CLSetEnvironment(None, 0, 0)
            return
        cube = np.ascontiguousarray(cube, dtype=np.float32)
        self.L.CLSetEnvironment(cube.ctypes.data, cube.nbytes, cube.shape[1] if cube.ndim == 4 else 0)

    def read_environment(self) -> dict:
        """The environment table (CLDebugReadEnvironment): header uint64[2] (face size n, total
        weight Q; zeros without an environment), texels float32[6 n^2, 4] (r, g, b and the pdf per
        unit area of face coordinates), cdf uint64[6 n^2] (exclusive prefix sums of the weights)."""
        out = {}
        for which, name, dtype in ((0, "header", np.uint64), (1, "texels", np.float32), (2, "cdf", np.uint64)):
            n = self.L.CLDebugReadEnvironment(which, None, 0)
            a = np.zeros(n // np.dtype(dtype).itemsize, dtype=dtype)
            if n:
                self.L.CLDebugReadEnvironment(which, a.ctypes.data, n)
            out[name] = a
        out["texels"] = out["texels"].reshape(-1, 4)
        return out

    def instance_build_ms(self) -> float:
        """Device time of the last instance-tree build."""
        ms = C.c_float(0)
        self.L.CLLastInstanceBuildMs(C.byref(ms))
        return ms.value

    def clear_instance_meshes(self) -> None:
        self.L.CLClearInstanceMeshes()

    def download_instance_kd(self, mesh: int) -> "Scene":
        """An instance mesh's device-built tree as a Scene (wire format) for the oracle."""
        k = KD()
        self.L.CLDownloadInstanceKd(int(mesh), C.byref(k))
        return Scene.from_kd(k)

    def build_ms(self) -> tuple[float, float]:
        b, p = C.c_float(0), C.c_float(0)
        self.L.CLLastBuildMs(C.byref(b), C.byref(p))
        return b.value, p.value

    def build_was_recorded(self) -> bool:
        """CLLastBuildWasRecorded: the last device build ran as the recorded graph."""
        return bool(self.L.CLLastBuildWasRecorded())

    def read_packed(self, which: int) -> np.ndarray:
        n = self.L.CLDebugReadPacked(which, None, 0)
        out = np.zeros(n, dtype=np.uint8)
        if n:
            self.L.CLDebugReadPacked(which, out.ctypes.data, n)
        return out

    def set_materials(self, materials: np.ndarray, tri_material: np.ndarray | None = None) -> None:
        m = np.ascontiguousarray(materials, dtype=np.float32).reshape(-1, 8)
        t = None if tri_material is None else np.ascontiguousarray(tri_material, dtype=np.int32)
        self.L.CLSetMaterials(m.ctypes.data, m.nbytes, None if t is None else t.ctypes.data,
                              0 if t is None else t.nbytes)

    def set_camera_matrix(self, m: np.ndarray) -> None:
        a = np.ascontiguousarray(m, dtype=np.float32).reshape(16)
        self.L.CLSetCameraMatrixPtr(C.cast(a.ctypes.data, C.POINTER(Matrix)))

    def set_params(self, mode=MODE_NORMAL, depth=2, spp=1, seed=0, flags=0) -> None:
        self.L.CLSetRenderParams(int(mode), int(depth), int(spp), int(seed), int(flags))

    def create_image(self, width: int, height: int, aov: bool = False) -> None:
        if self.width:
            self.L.CLDeleteImage()
        self.L.CLEnableAOV(1 if aov else 0)
        self.L.CLCreateImageHeadless(int(width), int(height))
        self.width, self.height = int(width), int(height)

    def execute(self) -> None:
        self.L.CLExecute(self.width, self.height)

    def read_image(self, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.height, self.width, 4), dtype=np.float32)
        self.L.CLReadImage(out.ctypes.data, out.nbytes)
        return out

    def read_image_rgba8(self, out: np.ndarray | None = None) -> np.ndarray:
        """The frame as RGBA8 UNORM texels, the reference's render-target format."""
        if out is None:
            out = np.empty((self.height, self.width, 4), dtype=np.uint8)
        self.L.CLReadImageRGBA8(out.ctypes.data, out.nbytes)
        return out

    def read_image_async(self, out: np.ndarray) -> None:
        """Pipelined read-back into `out` (float32 -> float4 frame, uint8 -> RGBA8); `out`
        must stay alive and untouched until read_wait() says the read has landed."""
        fmt = READ_RGBA8 if out.dtype == np.uint8 else READ_FLOAT4
        self.L.CLReadImageAsync(out.ctypes.data, out.nbytes, fmt)

    def read_wait(self, leave_pending: int = 0) -> None:
        self.L.CLReadImageWait(int(leave_pending))

    def read_aov(self):
        n = self.width * self.height
        prim = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float32)
        uv = np.empty((n, 2), dtype=np.float32)
        self.L.CLReadAOV(prim.ctypes.data, t.ctypes.data, uv.ctypes.data)
        shape = (self.height, self.width)
        return prim.reshape(shape), t.reshape(shape), uv.reshape(shape + (2,))

    def counters(self) -> dict:
        c = (C.c_ulonglong * 6)()
        self.L.CLGetCounters(c)
        return dict(zip(["rays", "splits", "leaves", "tris", "shade_vn", "capped"], [int(x) for x in c]))

    def kernel_ms(self) -> float:
        return float(self.L.CLLastKernelMs())

    def close(self) -> None:
        self.L.CLTerminate()
        self.width = self.height = 0


def default_device() -> int:
    return int(os.environ.get("LOCAL_RANK", os.environ.get("CLPT_DEVICE", "0")))
