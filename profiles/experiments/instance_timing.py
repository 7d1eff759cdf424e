"""Rigid instances against per-frame rebuilds, on one GPU (DESIGN.md section 5, "Rigid instances").

1. BASELINE config 5 two ways, alternated in blocks in one process: bench.py's terrain (heightfield
   158) and icosphere, the same PhysStep motion, 1920x1080, 4 spp, depth 2 (bench's c5 values),
   RGBA8 read-back, blocking and pipelined one frame deep.
     rebuild   : terrain + sphere in one mesh, CLUpdateVertices + CLRebuildMeshes every frame (bench.py c5)
     instance  : the terrain built once, the sphere one instance mesh, CLSetInstances every frame
   The last frame of each arm is checked bit for bit against the oracle.
2. What instances cost on a static frame: render-kernel time (CLLastKernelMs) at the config 2 size
   (1920x1080, 16 spp, depth 5, heightfield 224, mirror mode) with 0, 1, 8 and 64 icosphere instances,
   in view (over the terrain) and out of view (behind and below the camera).

    python profiles/experiments/instance_timing.py --out instance_timing.json
"""
import argparse
import ctypes as C
import gc
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
import clpathtracer_b200 as cl  # noqa: E402
from clpathtracer_b200 import scenes  # noqa: E402
from oracle import oracle_instances_py as oi  # noqa: E402
from oracle import oracle_py as op  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def pct(x, q):
    return round(float(np.percentile(x, q)) * 1e3, 3)


def translate(p):
    m = np.eye(4)
    m[:3, 3] = p[:3]
    return m


def c5_both_ways(r, L, blocks, frames, warmup):
    w, h, spp, depth, seed = 1920, 1080, 4, 2, 0
    tv, tc, _ = scenes.heightfield(158, False)
    sv, sf = bench.icosphere(3)
    sv = sv * np.float32(0.12)
    sc = cl.corners_from_faces(sf + len(tv), False)
    corners = np.concatenate([tc, sc])
    verts = np.zeros((len(tv) + len(sv), 4), dtype=np.float32)
    verts[:len(tv), :3] = tv[:, :3]
    pos, vel = cl.Vector4(), cl.Vector4()
    pos.s[:] = [0.0, 0.6, -0.4, 0.0]
    vel.s[:] = [0.25, 0.0, 0.35, 0.0]
    L.AddPhysObject(C.byref(pos), C.byref(vel))
    r.clear_instance_meshes()
    sphere = r.add_instance_mesh(sv, cl.corners_from_faces(sf, False))
    cam = cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), h)
    r.create_image(w, h)
    r.set_params(mode=cl.MODE_MIRROR, depth=depth, spp=spp, seed=seed, flags=cl.FLAG_JITTER)
    hosts = [np.empty((h, w, 4), dtype=np.uint8) for _ in range(2)]
    dt, g = 1.0 / 60.0, -1.5

    def step():
        vel.s[1] = vel.s[1] + g * dt
        L.PhysStep(dt)
        if pos.s[1] < 0.3 and vel.s[1] < 0:
            vel.s[1] = -vel.s[1]

    def frame(arm, first, pipelined, f):
        t0 = time.perf_counter()
        step()
        if arm == "rebuild":
            verts[len(tv):, :3] = sv + np.array(pos.s[:3], dtype=np.float32)
            if first:
                r.set_instances([])
                r.build_meshes(verts, corners, None)
            else:
                r.update_vertices(len(tv), verts[len(tv):])
                r.rebuild_meshes()
        else:
            if first:
                r.build_meshes(tv, tc, None)
            r.set_instances([(sphere, translate(pos.s), 0)])
        r.set_camera_matrix(cam)
        r.execute()
        if pipelined:
            r.read_image_async(hosts[f % 2])
            r.read_wait(1)
        else:
            r.read_image_rgba8(hosts[0])
        return time.perf_counter() - t0

    res = {arm: {"blocking": [], "pipelined": [], "build_ms": []} for arm in ("rebuild", "instance")}
    gc.disable()
    for b in range(blocks):
        for arm in ("rebuild", "instance"):
            for pipelined in (False, True):
                key = "pipelined" if pipelined else "blocking"
                for f in range(warmup + frames):
                    t = frame(arm, f == 0, pipelined, f)
                    if f >= warmup:
                        res[arm][key].append(t)
                        if arm == "rebuild":
                            res[arm]["build_ms"].append(r.build_ms()[0])
                r.read_wait(0)
            # parity: the last frame of this block against the oracle walking the same trees
            if b == blocks - 1:
                frame_now = r.read_image()
                if arm == "rebuild":
                    ref = op.render(r.download_kd(), cam, w, h, mode=1, depth=depth, spp=spp, seed=seed,
                                    flags=op.FLAG_JITTER, aov=False, threads=os.cpu_count())
                else:
                    ref = oi.render(r.download_kd(), cam, w, h, mode=1, depth=depth, spp=spp, seed=seed,
                                    flags=op.FLAG_JITTER, aov=False, threads=os.cpu_count(),
                                    instances=[(r.download_instance_kd(sphere), cl.world_to_object(translate(pos.s)), 0)])
                res[arm]["parity_words_differ"] = int(np.count_nonzero(frame_now.view(np.uint32) !=
                                                                       ref["rgba"].view(np.uint32)))
    gc.enable()
    L.PhysTerminate()
    out = {"config": dict(width=w, height=h, spp=spp, depth=depth, mode="mirror", terrain_triangles=len(tc) // 3,
                          sphere_triangles=len(sf), blocks=blocks, frames_per_block=frames, warmup_per_block=warmup)}
    for arm, d in res.items():
        out[arm] = {"p50_ms": pct(d["blocking"], 50), "p99_ms": pct(d["blocking"], 99),
                    "pipelined_p50_ms": pct(d["pipelined"], 50), "pipelined_p99_ms": pct(d["pipelined"], 99),
                    "frames": len(d["blocking"]), "parity_words_differ": d.get("parity_words_differ")}
        if d["build_ms"]:
            out[arm]["device_build_p50_ms"] = round(float(np.median(d["build_ms"])), 3)
    r.set_instances([])
    return out


def static_cost(r, repeats):
    w, h = 1920, 1080
    v, c, n = scenes.heightfield(224, False)
    r.build_meshes(v, c, n)
    r.clear_instance_meshes()
    sv, sf = bench.icosphere(3)
    sphere = r.add_instance_mesh(sv * np.float32(0.08), cl.corners_from_faces(sf, False))
    r.create_image(w, h)
    r.set_camera_matrix(cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), h))
    r.set_params(mode=cl.MODE_MIRROR, depth=5, spp=16, seed=0, flags=cl.FLAG_JITTER)
    grid = np.linspace(-0.7, 0.7, 8)
    in_view = [translate((x, 0.25, z)) for z in grid for x in grid]                      # 64 over the terrain
    out_view = [translate((x, -3.0, -4.0 + z)) for z in grid for x in grid]            # below and behind the camera
    rows = []
    for where, spots in (("in_view", in_view), ("out_of_view", out_view)):
        for k in (0, 1, 8, 64):
            pick = [spots[i] for i in np.linspace(0, 63, k).astype(int)] if k else []
            r.set_instances([(sphere, m, 0) for m in pick])
            for _ in range(2):
                r.execute()
            ms = []
            for _ in range(repeats):
                r.execute()
                ms.append(r.kernel_ms())
            rows.append({"where": where, "instances": k, "kernel_ms_median": round(float(np.median(ms)), 4),
                         "kernel_ms_min": round(float(np.min(ms)), 4), "repeats": repeats})
            print(rows[-1], flush=True)
    r.set_instances([])
    return {"config": dict(width=w, height=h, spp=16, depth=5, mode="mirror", terrain_triangles=len(c) // 3,
                           sphere_triangles=len(sf), sphere_radius=0.08), "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="instance_timing.json")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=7)
    a = ap.parse_args()
    r = cl.Renderer(device=0)
    L = cl.lib()
    try:
        result = {"device": L.CLDeviceName().decode(), "nvidia_smi_name_power_limit_max_sm_clock": gpu_info()}
        result["c5"] = c5_both_ways(r, L, a.blocks, a.frames, a.warmup)
        print(json.dumps(result["c5"]), flush=True)
        result["static"] = static_cost(r, a.repeats)
    finally:
        r.close()
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
