"""Light sampling (mode 3) against mode 2, on one GPU (DESIGN.md "Light sampling (mode 3)").

Everything runs in one process; modes 2 and 3 alternate in blocks.
1. cornell_small_light() and the original Cornell box at 1920x1080, depth 5, 4 spp, jittered:
   render-kernel time (CUDA events, L2 flushed before every frame), modes 2 and 3.
2. The same scenes at 320x180: RMSE of 8 seeds per mode at 4 spp against a converged mode-3
   reference (16 progressive frames of 256 spp), and efficiency = 1 / (MSE x 1080p kernel ms).
3. Emitter-table builds at ~1k, ~100k and ~1M emitters (every heightfield triangle emits): host wall
   time of CLDebugReadEmitters(0) with a stale table -- enqueueing the build (5 kernels, 3 memsets,
   2 CUB calls) on an idle stream, running it, reading the 16-byte header back and synchronising.
   At small sizes this is launch overhead, not build work.
Every arm's last 1080p frame is checked against the oracle on a band of rows.

    python profiles/experiments/nee_timing.py --out profiles/r05_nee_timing_b200.json
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
from oracle import oracle_instance_tree_py as ot  # noqa: E402
from oracle import oracle_nee_py as on  # noqa: E402

BAND = 8


def scene_of(name):
    if name == "small_light":
        v, c, n, tm = scenes.cornell_small_light(10)
        return v, c, n, tm, scenes.CORNELL_SMALL_LIGHT_MATERIALS
    v, c, n, tm = scenes.cornell(10)
    return v, c, n, tm, scenes.CORNELL_MATERIALS


def band_check(r, base, cam, w, h, mode, kw):
    y0 = h // 2 - BAND // 2
    args = dict(rows=(y0, y0 + BAND), aov=False, threads=os.cpu_count(), **kw)
    ref = on.render(base, cam, w, h, **args) if mode == 3 else ot.render(base, cam, w, h, mode=2, **args)
    got = r.read_image()
    return int(np.count_nonzero(got[y0:y0 + BAND].view(np.uint32) != ref["rgba"][y0:y0 + BAND].view(np.uint32)))


def timed(r, L, repeats):
    ms = []
    for k in range(repeats + 2):
        L.CLFlushL2()
        r.execute()
        if k >= 2:
            ms.append(r.kernel_ms())
    return ms


def frame_times(r, L, name, blocks, repeats):
    v, c, n, tm, mats = scene_of(name)
    r.build_meshes(v, c, n)
    base = r.download_kd()
    r.set_materials(mats, tm)
    w, h, spp = 1920, 1080, 4
    cam = cl.cam_matrix(cl.make_camera(**scenes.CORNELL_CAMERA), h)
    r.create_image(w, h)
    r.set_camera_matrix(cam)
    ms = {2: [], 3: []}
    for _ in range(blocks):
        for mode in (2, 3):
            r.set_params(mode=mode, depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER)
            ms[mode] += timed(r, L, repeats)
    out = {}
    for mode in (2, 3):
        r.set_params(mode=mode, depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER)
        r.execute()
        kw = dict(depth=5, spp=spp, seed=1, flags=cl.FLAG_JITTER, materials=mats, tri_material=tm)
        out[mode] = {"kernel_ms_median": round(float(np.median(ms[mode])), 4),
                     "kernel_ms_min": round(float(np.min(ms[mode])), 4), "frames": len(ms[mode]),
                     "band_words_differing_from_oracle": band_check(r, base, cam, w, h, mode, kw)}
    return out


def errors(r, name, seeds, ref_frames, ref_spp):
    v, c, n, tm, mats = scene_of(name)
    r.build_meshes(v, c, n)
    r.set_materials(mats, tm)
    w, h = 320, 180
    r.set_camera_matrix(cl.cam_matrix(cl.make_camera(**scenes.CORNELL_CAMERA), h))
    r.create_image(w, h)
    r.set_params(mode=3, depth=5, spp=ref_spp, seed=12345, flags=cl.FLAG_JITTER | cl.FLAG_ACCUMULATE)
    for _ in range(ref_frames):
        r.execute()
    ref = r.read_image()[..., :3].astype(np.float64)
    mse = {}
    for mode in (2, 3):
        r.set_params(mode=mode, depth=5, spp=4, seed=0, flags=cl.FLAG_JITTER)
        e = []
        for s in range(seeds):
            r.set_params(mode=mode, depth=5, spp=4, seed=s, flags=cl.FLAG_JITTER)
            r.execute()
            e.append(((r.read_image()[..., :3] - ref) ** 2).mean())
        mse[mode] = float(np.mean(e))
    return mse, ref_frames * ref_spp


def build_times(r, L, repeats):
    rows = []
    for n in (22, 224, 707):
        v, c, _ = scenes.heightfield(n, False)
        r.build_meshes(v, c)
        ms = []
        for _ in range(repeats + 1):
            r.set_materials(scenes.CORNELL_MATERIALS[3:])  # marks the table stale
            t0 = time.perf_counter()
            L.CLDebugReadEmitters(0, None, 0)  # builds it, reads the header back and synchronises
            ms.append((time.perf_counter() - t0) * 1e3)
        tab = r.read_emitters()
        twin = on.build_emitters(r.download_kd(), scenes.CORNELL_MATERIALS[3:])
        same = all(np.ascontiguousarray(tab[k]).tobytes() == np.ascontiguousarray(twin[k]).tobytes()
                   for k in ("header", "records", "cdf", "map"))
        rows.append({"emitters": int(tab["header"][0]), "call_wall_ms_median": round(float(np.median(ms[1:])), 4),
                     "equals_twin": bool(same)})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="nee_timing.json")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=10)
    a = ap.parse_args()
    r = cl.Renderer(0)
    L = r.L
    result = {"device": L.CLDeviceName().decode(), "nvidia_smi_name_power_limit_max_sm_clock": gpu_info(),
              "frame": "1920x1080, depth 5, 4 spp, jittered; RMSE at 320x180 against a 4096-spp mode-3 reference",
              "scenes": {}}
    for name in ("small_light", "cornell"):
        t = frame_times(r, L, name, a.blocks, a.repeats)
        mse, ref_spp = errors(r, name, 8, 16, 256)
        row = {"reference_spp": ref_spp}
        for mode in (2, 3):
            row["mode%d" % mode] = dict(t[mode], mse=mse[mode], rmse=mse[mode] ** 0.5,
                                        efficiency=1.0 / (mse[mode] * t[mode]["kernel_ms_median"]))
        row["efficiency_ratio_mode3_over_mode2"] = row["mode3"]["efficiency"] / row["mode2"]["efficiency"]
        result["scenes"][name] = row
        print(json.dumps({name: row}), flush=True)
    result["emitter_table_builds"] = build_times(r, L, a.repeats)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result))
    r.close()


if __name__ == "__main__":
    main()
