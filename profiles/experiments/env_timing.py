"""Environment light: mode 2 against mode 3 under a sun and sky, on one GPU (DESIGN.md "Environment
light").

Everything runs in one process; modes 2 and 3 alternate in blocks.
1. The 999,698-triangle terrain (heightfield 707, no emitters) under scenes.sun_sky(64), and
   cornell_small_light() with a sun and sky seen through its open side, at 1920x1080, depth 5, 4 spp,
   jittered: render-kernel time (CUDA events, L2 flushed before every frame), modes 2 and 3.
2. The same scenes at 320x180: RMSE of 8 seeds per mode at 4 spp against a converged mode-3
   reference (16 progressive frames of 256 spp), and efficiency = 1 / (MSE x 1080p kernel ms).
3. Environment-table builds at N = 64, 512 and 2048: host wall time of set_environment (validating
   6 N^2 x 3 floats, the upload, the build and a synchronisation), each table checked against the twin.
Every arm's last 1080p frame is checked against the oracle on a band of rows.

    python profiles/experiments/env_timing.py --out profiles/r06_env_timing_b200.json
"""
import argparse
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "profiles" / "experiments"))

import clpathtracer_b200 as cl  # noqa: E402
from clpathtracer_b200 import scenes  # noqa: E402
from instance_timing import gpu_info  # noqa: E402
from oracle import oracle_env_py as oe  # noqa: E402

BAND = 8
TERRAIN_SKY = dict(n=64)  # scenes.sun_sky's defaults: a 50,000-radiance sun texel over a blue sky
BOX_SKY = dict(n=64, sun_dir=(0.1, 0.3, -1.0), sun_radiance=(9000.0, 8000.0, 6000.0))  # behind the camera


def scene_of(name):
    """verts, corners, norms, tri_material, materials, camera, environment"""
    if name == "terrain":
        v, c, n = scenes.heightfield(707, False)
        return v, c, n, None, None, scenes.CANONICAL_CAMERA, scenes.sun_sky(**TERRAIN_SKY)
    v, c, n, tm = scenes.cornell_small_light(10)
    return v, c, n, tm, scenes.CORNELL_SMALL_LIGHT_MATERIALS, scenes.CORNELL_CAMERA, scenes.sun_sky(**BOX_SKY)


def setup(r, name, h):
    v, c, n, tm, mats, camera, env = scene_of(name)
    r.build_meshes(v, c, n)
    if mats is not None:
        r.set_materials(mats, tm)
    else:
        r.set_materials(np.zeros((0, 8), dtype=np.float32))
    r.set_environment(env)
    cam = cl.cam_matrix(cl.make_camera(**camera), h)
    r.set_camera_matrix(cam)
    return cam, env, mats, tm


def timed(r, L, repeats):
    ms = []
    for k in range(repeats + 2):
        L.CLFlushL2()
        r.execute()
        if k >= 2:
            ms.append(r.kernel_ms())
    return ms


def frame_times(r, L, name, blocks, repeats):
    w, h, spp = 1920, 1080, 4
    cam, env, mats, tm = setup(r, name, h)
    base = r.download_kd()
    r.create_image(w, h)
    ms = {2: [], 3: []}
    for _ in range(blocks):
        for mode in (2, 3):
            r.set_params(mode=mode, depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER)
            ms[mode] += timed(r, L, repeats)
    out = {}
    table = oe.build_env(env)
    for mode in (2, 3):
        r.set_params(mode=mode, depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER)
        r.execute()
        y0 = h // 2 - BAND // 2
        ref = oe.render(base, cam, w, h, table, mode=mode, depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER,
                        materials=mats, tri_material=tm, rows=(y0, y0 + BAND), aov=False, threads=os.cpu_count())
        got = r.read_image()
        differ = int(np.count_nonzero(got[y0:y0 + BAND].view(np.uint32) != ref["rgba"][y0:y0 + BAND].view(np.uint32)))
        out[mode] = {"kernel_ms_median": round(float(np.median(ms[mode])), 4),
                     "kernel_ms_min": round(float(np.min(ms[mode])), 4), "frames": len(ms[mode]),
                     "band_words_differing_from_oracle": differ}
    return out


def errors(r, name, seeds, ref_frames, ref_spp):
    w, h = 320, 180
    setup(r, name, h)
    r.create_image(w, h)
    r.set_params(mode=3, depth=5, spp=ref_spp, seed=12345, flags=cl.FLAG_JITTER | cl.FLAG_ACCUMULATE)
    for _ in range(ref_frames):
        r.execute()
    ref = r.read_image()[..., :3].astype(np.float64)
    mse = {}
    for mode in (2, 3):
        e = []
        for s in range(seeds):
            r.set_params(mode=mode, depth=5, spp=4, seed=s, flags=cl.FLAG_JITTER)
            r.execute()
            e.append(((r.read_image()[..., :3] - ref) ** 2).mean())
        mse[mode] = float(np.mean(e))
    return mse, ref_frames * ref_spp


def build_times(r, repeats):
    rows = []
    rng = np.random.default_rng(0)
    for n in (64, 512, 2048):
        cube = rng.exponential(1.0, (6, n, n, 3)).astype(np.float32)
        cube[2, n // 3, n // 2] = 5e4
        ms = []
        for _ in range(repeats + 1):
            t0 = time.perf_counter()
            r.set_environment(cube)
            ms.append((time.perf_counter() - t0) * 1e3)
        tab, twin = r.read_environment(), oe.build_env(cube)
        same = all(np.ascontiguousarray(tab[k]).tobytes() == np.ascontiguousarray(twin[k]).tobytes()
                   for k in ("header", "texels", "cdf"))
        rows.append({"face_size": n, "texels": 6 * n * n, "set_environment_wall_ms_median": round(float(np.median(ms[1:])), 4),
                     "equals_twin": bool(same)})
        print(json.dumps(rows[-1]), flush=True)
    r.set_environment(None)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="env_timing.json")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=10)
    a = ap.parse_args()
    r = cl.Renderer(0)
    L = r.L
    result = {"device": L.CLDeviceName().decode(), "nvidia_smi_name_power_limit_max_sm_clock": gpu_info(),
              "frame": "1920x1080, depth 5, 4 spp, jittered; RMSE at 320x180 against a 4096-spp mode-3 reference",
              "environments": {"terrain": TERRAIN_SKY, "small_light": BOX_SKY}, "scenes": {}}
    for name in ("terrain", "small_light"):
        t = frame_times(r, L, name, a.blocks, a.repeats)
        mse, ref_spp = errors(r, name, 8, 16, 256)
        row = {"reference_spp": ref_spp}
        for mode in (2, 3):
            row["mode%d" % mode] = dict(t[mode], mse=mse[mode], rmse=mse[mode] ** 0.5,
                                        efficiency=1.0 / (mse[mode] * t[mode]["kernel_ms_median"]))
        row["efficiency_ratio_mode3_over_mode2"] = row["mode3"]["efficiency"] / row["mode2"]["efficiency"]
        result["scenes"][name] = row
        print(json.dumps({name: row}), flush=True)
    result["environment_table_builds"] = build_times(r, a.repeats)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))
    r.close()


if __name__ == "__main__":
    main()
