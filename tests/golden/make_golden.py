"""Regenerate tests/golden/host_golden.json.

Run where $CLPT_REFERENCE names a checkout of the reference: the values are
produced by the REFERENCE's own host code (oracle/_ref/libref_host.so, built by
oracle/Makefile from $CLPT_REFERENCE/src/*.c unmodified), not by this repo's
code.  The file pins, for deterministic synthetic scenes, the sha256 of the
reference builder's node array and tri_indices, and camera matrices as raw
float bits.

    python tests/golden/make_golden.py
"""
import ctypes as C
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

import clpathtracer_b200 as cl  # noqa: E402  (only for scene generation + Camera struct)
from clpathtracer_b200 import scenes  # noqa: E402
from oracle import oracle_py as op  # noqa: E402


class KD(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ["node_vec", "tri_indices", "vert_vec", "norm_vec", "tri_vec"]]


def ref_list(R, a):
    if a is None:
        return R.new_list(0)
    a = np.ascontiguousarray(a)
    p = R.init_list(a.nbytes, 1)
    C.memmove(p, a.ctypes.data, a.nbytes)
    return p


def ref_build(verts, corners, norms):
    R = op.ref()
    R.build_kd.restype = KD
    R.build_kd.argtypes = [C.c_void_p] * 3 + [C.c_char_p]
    k = R.build_kd(ref_list(R, corners), ref_list(R, cl._as_vec4(verts)),
                   ref_list(R, cl._as_vec4(norms) if norms is not None else None), None)
    nodes = C.string_at(k.node_vec, R.list_size(k.node_vec))
    idx = C.string_at(k.tri_indices, R.list_size(k.tri_indices))
    return nodes, idx


def ref_cam(cam, height):
    R = op.ref()
    m = cl.Matrix()
    R.ref_cam_matrix_ptr(C.byref(cam), height, C.byref(m))
    return np.frombuffer(bytes(m), dtype=np.uint32).tolist()


SCENES = {
    "hf4n": lambda: scenes.heightfield(4, True),
    "hf22n": lambda: scenes.heightfield(22, True),
    "hf22": lambda: scenes.heightfield(22, False),
    "hf60": lambda: scenes.heightfield(60, False),
    "hf224": lambda: scenes.heightfield(224, False),
    "cornell": lambda: scenes.cornell(10)[:3],
    "soup500": lambda: scenes.soup(500),
}

CAMERAS = {
    "reference_default_480": (scenes.REFERENCE_CAMERA, 480),
    "canonical_480": (scenes.CANONICAL_CAMERA, 480),
    "canonical_1080": (scenes.CANONICAL_CAMERA, 1080),
    "cornell_480": (scenes.CORNELL_CAMERA, 480),
    "oblique_777": (dict(near=0.05, far=3.0, fov=1.2, position=(0.3, 0.7, -1.1), forward=(0.48, -0.6, 0.64)), 777),
}


def main():
    assert op.have_ref(), "oracle/_ref/libref_host.so missing: run `make -C oracle ref` with $CLPT_REFERENCE set"
    assert op.ref().ref_sizeof_kdnode() == 68 and op.ref().ref_sizeof_camera() == 48
    out = {"generated_by": "tests/golden/make_golden.py using oracle/_ref/libref_host.so (reference host code, unmodified)",
           "kd": {}, "cam": {}}
    for name, gen in SCENES.items():
        v, c, n = gen()
        nodes, idx = ref_build(v, c, n)
        out["kd"][name] = {
            "tris": len(c) // 3, "nodes": len(nodes) // 68, "tri_refs": len(idx) // 4,
            "nodes_sha256": hashlib.sha256(nodes).hexdigest(),
            "tri_indices_sha256": hashlib.sha256(idx).hexdigest(),
            "verts_sha256": hashlib.sha256(cl._as_vec4(v).tobytes()).hexdigest(),
        }
        print(name, out["kd"][name])
    for name, (kw, h) in CAMERAS.items():
        out["cam"][name] = {"camera": {k: (list(v) if isinstance(v, tuple) else float(v)) for k, v in kw.items()},
                            "height": h, "matrix_bits": ref_cam(cl.make_camera(**kw), h)}
    (Path(__file__).parent / "host_golden.json").write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
