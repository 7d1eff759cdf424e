"""The instance tree against the instance list, on one GPU (DESIGN.md section 5, "Instance tree").

Everything runs in one process; list and tree alternate in blocks.
1. The static config-2 frame of instance_timing.py (1920x1080, 16 spp, depth 5, mirror mode,
   heightfield 224): render-kernel time with 0, 1, 8 and 64 icosphere instances, in view (over the
   terrain) and out of view (behind and below the camera), list against tree.
2. Tree only, the same frame: 1,024, 16,384 and 65,536 small icospheres scattered over the terrain.
3. Tree build time (CLLastInstanceBuildMs) and CLSetInstances time at 1k, 64k and 1M instances; the
   device tree is compared with the CPU twin's byte for byte.
4. Config 5 with its one instance (bench.py's c5 motion, 1920x1080, 4 spp, depth 2, RGBA8
   read-back), list against tree.
Every arm's last frame is checked against the oracle on a band of rows.

    python profiles/experiments/instance_tree_timing.py --out instance_tree_timing.json
"""
import argparse
import ctypes as C
import gc
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles" / "experiments"))

import bench  # noqa: E402
import clpathtracer_b200 as cl  # noqa: E402
from clpathtracer_b200 import scenes  # noqa: E402
from instance_timing import gpu_info, pct, translate  # noqa: E402
from oracle import oracle_instance_tree_py as ot  # noqa: E402

BAND = 8  # rows of the oracle check


def band_check(r, base, cam, w, h, inst, traversal, kw):
    """Words of a band of rows in the middle of the frame that differ from the oracle."""
    y0 = h // 2 - BAND // 2
    tree = r.instance_tree() if traversal == "tree" and inst else None
    ref = ot.render(base, cam, w, h, rows=(y0, y0 + BAND), aov=False, threads=os.cpu_count(), instances=inst,
                    tree=tree, **kw)["rgba"]
    got = r.read_image()
    return int(np.count_nonzero(got[y0:y0 + BAND].view(np.uint32) != ref[y0:y0 + BAND].view(np.uint32)))


def kernel_ms(r, repeats):
    for _ in range(2):
        r.execute()
    ms = []
    for _ in range(repeats):
        r.execute()
        ms.append(r.kernel_ms())
    return ms


def static_frames(r, blocks, repeats):
    w, h = 1920, 1080
    kw = dict(mode=1, depth=5, spp=16, seed=0, flags=cl.FLAG_JITTER)
    v, c, n = scenes.heightfield(224, False)
    r.build_meshes(v, c, n)
    base = r.download_kd()
    r.clear_instance_meshes()
    sv, sf = bench.icosphere(3)
    sphere = r.add_instance_mesh(sv * np.float32(0.08), cl.corners_from_faces(sf, False))
    small = r.add_instance_mesh(sv * np.float32(0.01), cl.corners_from_faces(sf, False))
    mesh, small_mesh = r.download_instance_kd(sphere), r.download_instance_kd(small)
    cam = cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), h)
    r.create_image(w, h)
    r.set_camera_matrix(cam)
    r.set_params(**kw)
    grid = np.linspace(-0.7, 0.7, 8)
    spots = {"in_view": np.stack([translate((x, 0.25, z)) for z in grid for x in grid]),
             "out_of_view": np.stack([translate((x, -3.0, -4.0 + z)) for z in grid for x in grid])}
    rows = []
    for where in ("in_view", "out_of_view"):
        for k in (0, 1, 8, 64):
            pick = spots[where][np.linspace(0, 63, k).astype(int)] if k else np.zeros((0, 4, 4))
            times = {"list": [], "tree": []}
            for b in range(blocks):
                for traversal in ("list", "tree"):
                    r.set_instance_arrays(np.full(k, sphere), pick, 0)
                    r.set_instance_traversal(traversal)
                    times[traversal] += kernel_ms(r, repeats)
            row = {"where": where, "instances": k}
            for traversal in ("list", "tree"):
                r.set_instance_traversal(traversal)
                r.execute()
                inst = [(mesh, wo, 0) for wo in cl.world_to_object_batch(pick)] if k else []
                row[traversal] = {"kernel_ms_median": round(float(np.median(times[traversal])), 4),
                                  "kernel_ms_min": round(float(np.min(times[traversal])), 4),
                                  "frames": len(times[traversal]),
                                  "band_words_differ": band_check(r, base, cam, w, h, inst, traversal, kw)}
            rows.append(row)
            print(json.dumps(row), flush=True)
    r.set_instance_traversal("tree")
    rng = np.random.default_rng(1)
    crowd = []
    for k in (1024, 16384, 65536):
        o2w = np.zeros((k, 3, 4))
        o2w[:, :, :3] = np.eye(3)
        o2w[:, :, 3] = np.stack([rng.uniform(-0.95, 0.95, k), rng.uniform(0.0, 0.3, k), rng.uniform(-0.95, 0.95, k)], 1)
        r.set_instance_arrays(np.full(k, small), o2w, 0)
        ms = []
        for _ in range(blocks):
            ms += kernel_ms(r, repeats)
        inst = [(small_mesh, wo, 0) for wo in cl.world_to_object_batch(o2w)]
        row = {"instances": k, "kernel_ms_median": round(float(np.median(ms)), 4),
               "kernel_ms_min": round(float(np.min(ms)), 4), "frames": len(ms),
               "band_words_differ": band_check(r, base, cam, w, h, inst, "tree", kw)}
        crowd.append(row)
        print(json.dumps(row), flush=True)
    r.set_instance_arrays([], np.zeros((0, 4, 4)), 0)
    r.set_instance_traversal("list")
    return {"config": dict(width=w, height=h, spp=16, depth=5, mode="mirror", terrain_triangles=len(c) // 3,
                           sphere_triangles=len(sf), sphere_radius=0.08, crowd_sphere_radius=0.01,
                           blocks=blocks, repeats_per_block=repeats),
            "list_vs_tree": rows, "tree_only": crowd}


def build_times(r, repeats):
    r.clear_instance_meshes()
    sv, sf = bench.icosphere(1)
    sphere = r.add_instance_mesh(sv * np.float32(0.01), cl.corners_from_faces(sf, False))
    root = ot.root_box(r.download_instance_kd(sphere))
    r.set_instance_traversal("tree")
    rng = np.random.default_rng(2)
    out = []
    for k in (1024, 65536, 1 << 20):
        o2w = np.zeros((k, 3, 4))
        o2w[:, :, :3] = np.eye(3)
        o2w[:, :, 3] = rng.uniform(-1, 1, (k, 3))
        set_s, arrays_s, build = [], [], []
        table = np.zeros(k, dtype=cl.CLINSTANCE_DTYPE)
        table["world_to_object"] = cl.world_to_object_batch(o2w).reshape(k, 12)
        table["mesh"] = sphere
        for _ in range(repeats):
            t0 = time.perf_counter()
            r.set_instance_arrays(np.full(k, sphere), o2w, 0)
            arrays_s.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            r.L.CLSetInstances(table.ctypes.data, table.nbytes)
            set_s.append(time.perf_counter() - t0)
            nodes = r.instance_tree()  # uploads the records and builds the tree
            build.append(r.instance_build_ms())
        twin = ot.build_tree(table["world_to_object"].reshape(k, 3, 4), np.tile(root, (k, 1)))
        row = {"instances": k, "build_ms_median": round(float(np.median(build)), 4),
               "build_ms_min": round(float(np.min(build)), 4), "CLSetInstances_ms_median": pct(set_s, 50),
               "set_instance_arrays_ms_median": pct(arrays_s, 50), "repeats": repeats,
               "tree_equals_twin": nodes.tobytes() == twin.tobytes()}
        out.append(row)
        print(json.dumps(row), flush=True)
    r.clear_instance_meshes()
    r.set_instance_traversal("list")
    return out


def c5_list_vs_tree(r, L, blocks, frames, warmup):
    w, h, spp, depth, seed = 1920, 1080, 4, 2, 0
    kw = dict(mode=1, depth=depth, spp=spp, seed=seed, flags=cl.FLAG_JITTER)
    tv, tc, _ = scenes.heightfield(158, False)
    sv, sf = bench.icosphere(3)
    r.clear_instance_meshes()
    sphere = r.add_instance_mesh(sv * np.float32(0.12), cl.corners_from_faces(sf, False))
    mesh = r.download_instance_kd(sphere)
    r.build_meshes(tv, tc, None)
    base = r.download_kd()
    cam = cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), h)
    r.create_image(w, h)
    r.set_camera_matrix(cam)
    r.set_params(**kw)
    host = np.empty((h, w, 4), dtype=np.uint8)
    res = {}
    for traversal in ("list", "tree"):
        res[traversal] = []
    gc.disable()
    for b in range(blocks):
        for traversal in ("list", "tree"):
            r.set_instance_traversal(traversal)
            pos, vel = cl.Vector4(), cl.Vector4()
            pos.s[:] = [0.0, 0.6, -0.4, 0.0]
            vel.s[:] = [0.25, 0.0, 0.35, 0.0]
            L.AddPhysObject(C.byref(pos), C.byref(vel))
            for f in range(warmup + frames):
                t0 = time.perf_counter()
                vel.s[1] = vel.s[1] - 1.5 / 60.0
                L.PhysStep(1.0 / 60.0)
                if pos.s[1] < 0.3 and vel.s[1] < 0:
                    vel.s[1] = -vel.s[1]
                r.set_instance_arrays([sphere], translate(pos.s)[None], 0)
                r.execute()
                r.read_image_rgba8(host)
                if f >= warmup:
                    res[traversal].append(time.perf_counter() - t0)
            L.PhysTerminate()
            if b == blocks - 1:
                inst = [(mesh, cl.world_to_object(translate(pos.s)), 0)]
                res[traversal + "_band"] = band_check(r, base, cam, w, h, inst, traversal, kw)
    gc.enable()
    r.clear_instance_meshes()
    r.set_instance_traversal("list")
    return {"config": dict(width=w, height=h, spp=spp, depth=depth, mode="mirror", terrain_triangles=len(tc) // 3,
                           sphere_triangles=len(sf), blocks=blocks, frames_per_block=frames),
            **{t: {"p50_ms": pct(res[t], 50), "p99_ms": pct(res[t], 99), "frames": len(res[t]),
                   "band_words_differ": res[t + "_band"]} for t in ("list", "tree")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="instance_tree_timing.json")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    r = cl.Renderer(device=0)
    L = cl.lib()
    try:
        result = {"device": L.CLDeviceName().decode(), "nvidia_smi_name_power_limit_max_sm_clock": gpu_info()}
        result["static"] = static_frames(r, a.blocks, a.repeats)
        result["build"] = build_times(r, a.repeats)
        result["c5"] = c5_list_vs_tree(r, L, a.blocks, a.frames, a.warmup)
        print(json.dumps(result["c5"]), flush=True)
    finally:
        r.close()
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
