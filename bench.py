#!/usr/bin/env python
"""bench.py -- the render hot path on BASELINE.json's headline workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU)

Workload (BASELINE.json configs[2], the one the metric is quoted on): a
1920x1080 frame, 64 jittered samples per pixel, primary + 4 mirror bounces
(depth 5, the reference's bounce, src/kernel.cl:399-417) of the 999,698-triangle
synthetic heightfield, canonical camera (SURVEY.md section 8d).  A "step" is one
frame.  Rays = entries into the traversal loop (src/kernel.cl:311), counted on
the device by an instrumented frame before timing.

One JSON line on stdout (rank 0).
  value        Mrays/s with everything resident in HBM (device events around CLExecute, L2 flushed
               between frames outside the timed events, max over ranks)
  e2e          the same metric through the C ABI with host buffers: every step uploads the camera
               matrix, renders, and delivers ONE frame to pinned host memory -- in the reference's
               render-target format (RGBA8, src/GLHandler.c:177-185) through the pipelined read-back
               (CLReadImageAsync: frame k travels while frame k+1 renders; all frames have landed
               before the clock stops); --readback float4 / --readback-sync change that
  parity       the frame rendered with the timed parameters against the oracle's, word for word,
               and its sha256 (one per rank at N > 1: every rank holds the whole frame)
  roofline     the formal HBM bound of SURVEY.md section 8d (algorithmic bytes / kernel time /
               measured HBM peak) and, in `binding`, what really binds: the utilisation of every
               unit and the lane-issue efficiency from the ncu capture of the same workload
               (profiles/binding.json)
  cpu_baseline the oracle port on all host cores, the full frame at full spp (it is also the
               parity reference)
--config c1|c2|c4|c5 run the other BASELINE configs (c4: progressive, spread over GPUs by sample;
c5: animated, per-frame kd rebuild on the device, reports ms per frame p50/p99).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

# torchrun exports OMP_NUM_THREADS=1.  The (untimed) host kd build of every rank should still use the
# rank's share of the host cores -- 10M triangles on one thread take over a minute -- and libgomp reads
# the variable when it is first loaded, so it is corrected here, before anything that links it is imported.
if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("OMP_NUM_THREADS") == "1":
    os.environ["OMP_NUM_THREADS"] = str(max(1, len(os.sched_getaffinity(0)) // int(os.environ["WORLD_SIZE"])))

import numpy as np  # noqa: E402

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "Mrays/s (primary+bounce) 1080p 1M-tri scene"
UNIT = "Mrays/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed frames (default 5; 30 for c5)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # None: taken from --config (c3: 1920x1080, 64 spp, depth 5, grid 707)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--depth", type=int, default=None, help="bounces + 1")
    ap.add_argument("--grid", type=int, default=None, help="heightfield cells per side (707 -> 999,698 triangles)")
    ap.add_argument("--tree-depth", type=int, default=int(os.environ.get("CLPT_TREE_DEPTH", "22")))
    ap.add_argument("--builder", default=os.environ.get("CLPT_BUILDER", "sah"), choices=["ref", "sah"],
                    help="ref: the reference's heuristic at --tree-depth; sah: build_kd_sah (extension)")
    ap.add_argument("--sah-ci", type=float, default=1.0)
    ap.add_argument("--sah-bonus", type=float, default=0.9)
    ap.add_argument("--sah-bins", type=int, default=0, help="0: exact sweep over all triangle bounds")
    ap.add_argument("--mode", default="mirror", choices=["normal", "mirror", "path"],
                    help="normal: as shipped, first-hit normal colour (mode A); mirror: the reference's bounce "
                         "(mode B); path: diffuse BSDF extension (mode C)")
    ap.add_argument("--no-jitter", action="store_true", help="pixel-corner rays exactly as the reference generates them")
    ap.add_argument("--engine", type=int, default=int(os.environ.get("CLPT_ENGINE", "0")),
                    help="0 auto, 1 full occupancy, 2 fat-leaf variant")
    ap.add_argument("--tile-rows", type=int, default=None)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--anim-builder", default="gpu", choices=["gpu", "host"],
                    help="config c5: where the per-frame kd-tree is built")
    ap.add_argument("--readback", default="rgba8", choices=["rgba8", "float4"],
                    help="format of the end-to-end read-back: the reference's RGBA8 texture format, or the float4 frame")
    ap.add_argument("--readback-sync", action="store_true", help="blocking read-back instead of the pipelined one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="skip the word-for-word comparison of the rendered frame with the oracle")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the baseline sample")
    ap.add_argument("--config", default="c3", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="BASELINE.json configs[0..3]; c3 (the default) is the one the metric is quoted on")
    ap.add_argument("--progressive", action="store_true", default=None,
                    help="accumulate spp samples per frame (CLPT_FLAG_ACCUMULATE)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed frames, write what the last one computed as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    presets = {
        # the reference's own CPU-runnable case: 640x480, 1 spp, 1 bounce, ~1k triangles
        "c1": dict(width=640, height=480, spp=1, depth=2, grid=22),
        "c2": dict(width=1920, height=1080, spp=16, depth=5, grid=224),
        "c3": dict(width=1920, height=1080, spp=64, depth=5, grid=707, tile_rows=8),
        # 4K progressive accumulation (1 spp per frame) of a 10M-triangle scene
        "c4": dict(width=3840, height=2160, spp=1, depth=5, grid=2236, progressive=True),
        # animated: per-frame object transform + kd rebuild + re-upload, 1080p at 4 spp (run_animated)
        "c5": dict(width=1920, height=1080, spp=4, depth=2, grid=158),
    }
    for k, v in {**presets["c3"], "progressive": False, **presets[a.config]}.items():
        if getattr(a, k) is None:  # explicit flags win over the preset
            setattr(a, k, v)
    if a.steps is None:  # the animated loop reports p99 frame times: it wants more frames
        a.steps = 30 if a.config == "c5" and a.impl == "ours" else 5
    return a


def workload_config(a):
    return {
        "workload": f"{a.width}x{a.height}, {a.spp} spp jittered, {a.depth - 1} mirror bounces (depth {a.depth}), "
                    f"heightfield n={a.grid} ({2 * a.grid * a.grid} triangles), kd builder {a.builder}, canonical camera",
        "baseline_config": a.config, "progressive": bool(a.progressive),
        "width": a.width, "height": a.height, "spp": a.spp, "depth": a.depth, "triangles": 2 * a.grid * a.grid,
        "render_mode": a.mode, "kd_builder": ("reference heuristic (src/kd_tree.c:95-200) at depth %d, 25 bins" % a.tree_depth) if a.builder == "ref"
                      else "build_kd_sah ci=%g bonus=%g bins=%d" % (a.sah_ci, a.sah_bonus, a.sah_bins),
        "mode": "mirror (src/kernel.cl:399-417 enabled)",
        "sharding": ("progressive frames are spread over ranks by SAMPLE: every rank renders the whole frame with its "
                     "own sample indices into its own fixed-point sums (a step = ranks x spp samples per pixel); nothing "
                     "crosses GPUs per frame, the read-back adds the ranks' sums (ncclAllReduce, 64-bit integers)")
                    if a.progressive else
                    (f"row tiles of {a.tile_rows} rows, round-robin over ranks, scene replicated; frame assembled by "
                     + ("the render kernel storing into peer-mapped frames (NVLink), two flag-word barriers per frame"
                        if getattr(a, "direct_placement", 1) else "NCCL all-gather + de-interleave")),
        "l2": "flushed between timed frames (CLFlushL2, 256 MiB overwrite, outside the timed events)",
    }


def make_scene(a):
    import clpathtracer_b200 as cl
    from clpathtracer_b200 import scenes

    t0 = time.time()
    v, c, n = scenes.heightfield(a.grid, False)
    t1 = time.time()
    if a.builder == "sah":
        scene = cl.build_kd_sah(v, c, n, nbins=a.sah_bins, intersect_cost=a.sah_ci, empty_bonus=a.sah_bonus)
    else:
        scene = cl.build_kd(v, c, n, depth=a.tree_depth)
    t2 = time.time()
    cam = cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), a.height)
    return scene, cam, {"scene_gen_s": round(t1 - t0, 2), "kd_build_s": round(t2 - t1, 2), **scene.stats()}


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with NVML while the timed region runs."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.armed = index, threading.Event(), threading.Event()
        self.sm, self.reasons, self.max_mhz, self.err = [], set(), None, None

    def arm(self):
        """Start recording (the thread is started earlier: NVML takes a few hundred ms to come up)."""
        self.armed.set()

    def run(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag.is_set():
                if not self.armed.is_set():
                    time.sleep(0.002)
                    continue
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "error": self.err}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def algorithmic_bytes(counters, pixels):
    """SURVEY.md section 8d: 16 B per split visit, 36 B per leaf visit, 40 B per
    triangle test, 36 B per vn-shaded hit, 16 B per pixel stored."""
    return (16 * counters["splits"] + 36 * counters["leaves"] + 40 * counters["tris"] + 36 * counters["shade_vn"]
            + 16 * pixels)


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores():
    """Cores this process may run on.  torchrun exports OMP_NUM_THREADS=1; the CPU arms
    use the affinity mask instead so that they run on all host cores at every N."""
    from oracle import oracle_py as op

    return int(op.oracle().oracle_host_cores())


def oracle_mode(a):
    return {"normal": 0, "mirror": 1, "path": 2}[a.mode]


def oracle_flags(a):
    from oracle import oracle_py as op

    return 0 if a.no_jitter else op.FLAG_JITTER


def oracle_check_and_baseline(a, scene, cam, gpu_frame, target_seconds, want_baseline, world=1):
    """One run of the oracle port (all host cores) serves two purposes: it is the
    `cpu_baseline` sample, and its frame is compared WORD FOR WORD with the frame the
    GPU path just rendered with the timed parameters (`parity`).  The whole frame at
    full spp when that fits the time budget (the default workload: ~9 s on 16 cores),
    else the whole frame at fewer spp for the baseline and a band of rows at full spp
    for the comparison."""
    import hashlib

    from oracle import oracle_py as op

    cores = host_cores()
    # a progressive frame on `world` ranks is world x spp samples per pixel (spread by sample), added to
    # fixed-point sums; the check frame is the first frame after a reset, i.e. the mean of those samples
    flags = oracle_flags(a) | (op.FLAG_ACCUMULATE if a.progressive else 0)
    kw = dict(mode=oracle_mode(a), depth=a.depth, seed=a.seed, flags=flags, aov=False, threads=cores)
    spp_frame = a.spp * (world if a.progressive else 1)
    t0 = time.time()
    r1 = op.render(scene, cam, a.width, a.height, spp=1, **kw)
    t1 = time.time() - t0
    full = spp_frame == 1 or t1 * spp_frame <= 2.0 * target_seconds
    baseline, parity = None, {"checked": False}
    if full:
        if spp_frame == 1:
            ref, secs = r1, t1
        else:
            t0 = time.time()
            ref = op.render(scene, cam, a.width, a.height, spp=spp_frame, **kw)
            secs = time.time() - t0
        rays, spp, rows = ref["counters"]["rays"], spp_frame, (0, a.height)
    else:
        spp = max(1, int(min(spp_frame, target_seconds / max(t1, 1e-3))))
        if want_baseline and spp > 1:
            t0 = time.time()
            rb = op.render(scene, cam, a.width, a.height, spp=spp, **kw)
            secs, rays = time.time() - t0, rb["counters"]["rays"]
        else:
            secs, rays, spp = t1, r1["counters"]["rays"], 1
        band = max(8, int(a.height * target_seconds / max(t1 * spp_frame, 1e-3)) // 8 * 8)
        rows = (max(0, a.height // 2 - band // 2), min(a.height, a.height // 2 - band // 2 + band))
        ref = op.render(scene, cam, a.width, a.height, spp=spp_frame, rows=rows, **kw)
    if want_baseline:
        baseline = {"value": round(rays / secs / 1e6, 4), "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"same scene/camera/depth, full {a.width}x{a.height} frame at {spp} of {spp_frame} spp "
                              f"({rays} rays in {secs:.1f} s)",
                    "ms_per_frame_at_full_spp": round(secs / spp * spp_frame * 1e3, 1)}
    if gpu_frame is not None:
        want = ref["rgba"][rows[0]:rows[1]]
        got = gpu_frame[rows[0]:rows[1]]
        differ = int(np.count_nonzero(np.ascontiguousarray(got).view(np.uint32) != np.ascontiguousarray(want).view(np.uint32)))
        parity = {"checked": True, "words_differ": differ, "words": int(want.size), "rows": list(rows),
                  "oracle_sha256": hashlib.sha256(np.ascontiguousarray(want).tobytes()).hexdigest(),
                  "oracle": "oracle/oracle_kernel.c (CPU restatement of src/kernel.cl, -ffp-contract=off) on the same "
                            "scene, tree, camera, seed, spp and depth as the timed frames",
                  "reference_pin": "mirror bounce pinned at depth 2 and 5, 1 spp, by the reference's own kernel.cl run "
                                   "through the vendor OpenCL compiler (tests/test_reference_kernel.py, "
                                   "tests/golden/ref_kernel_stats_r02.json); jitter and multi-spp accumulation have no "
                                   "reference behaviour (extension, defined by the oracle)"}
    return baseline, parity


def run_reference(a):
    """--impl reference: the reference's algorithm on the host cores.  kernel.cl
    cannot be compiled here (no OpenCL), so this is the oracle port (kind 'port'),
    all host threads, each step one full frame at 1 spp of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as op

    scene, cam, info = make_scene(a)
    cores = host_cores()
    ref_spp = min(8, a.spp)
    kw = dict(mode=oracle_mode(a), depth=a.depth, spp=ref_spp, flags=oracle_flags(a), aov=False, threads=cores)
    for w in range(a.warmup):
        op.render(scene, cam, a.width, a.height, seed=a.seed, sample_base=w * ref_spp, **kw)
    rays, t0 = 0, time.time()
    for k in range(a.steps):
        last = op.render(scene, cam, a.width, a.height, seed=a.seed, sample_base=k * ref_spp, **kw)
        rays += last["counters"]["rays"]
    secs = time.time() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"frame": last["rgba"]})
    value = rays / secs / 1e6
    sample = (f"each step = the full {a.width}x{a.height} frame at {ref_spp} of {a.spp} spp, depth {a.depth}; the "
              f"reference's algorithm (CPU port of src/kernel.cl, oracle/oracle_kernel.c) walking THIS repository's "
              f"kd-tree ({workload_config(a)['kd_builder']}) -- the reference as shipped cannot render this workload "
              f"(no bounces, samples or accumulation) and its own DEPTH-15 tree is slower, see reference_tree")
    # the same port on the tree the reference's own builder makes (src/kd_tree.c, DEPTH 15 / 25 bins)
    import clpathtracer_b200 as cl
    from clpathtracer_b200 import scenes

    ref_tree = None
    if 2 * a.grid * a.grid <= 1_100_000:
        t0 = time.time()
        own = cl.build_kd(*scenes.heightfield(a.grid, False))
        t_build = time.time() - t0
        t0 = time.time()
        rr = op.render(own, cam, a.width, a.height, seed=a.seed, **dict(kw, spp=1))
        dt = time.time() - t0
        ref_tree = {"value": round(rr["counters"]["rays"] / dt / 1e6, 4), "unit": UNIT, "cores": cores,
                    "sample": f"one full frame at 1 of {a.spp} spp on the reference builder's own tree "
                              f"(DEPTH 15, 25 bins; {own.stats()['leaf_tri_refs'] / max(own.stats()['leaves'] - own.stats()['empty_leaves'], 1):.1f} "
                              f"triangles per non-empty leaf), {rr['counters']['rays']} rays in {dt:.1f} s",
                    "kd_build_s": round(t_build, 2)}
    emit({
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(secs / a.steps * 1e3, 2),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a),
        "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_tree": ref_tree,
        "scene": info,
    })


_REAL_STDOUT = None


def quiet_stdout():
    """Everything but the final JSON line goes to stderr (NCCL and friends print
    banners on stdout): fd 1 is pointed at fd 2 until emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, line)
    else:
        os.write(_REAL_STDOUT, line)


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each [..., channels] array as <out_dir>/<name>.npy in float32, so that two builds
    can be compared output for output.  When together they exceed DUMP_LIMIT_BYTES, every array keeps
    the same fraction of its pixels, at sorted indices drawn with seed 0: the same pixels for the same
    arguments."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {name: np.asarray(arr, dtype=np.float32) for name, arr in arrays.items()}
    keep_fraction = min(1.0, DUMP_LIMIT_BYTES / sum(a.nbytes for a in arrays.values()))
    for name, a in arrays.items():
        if keep_fraction < 1.0:
            pixels = a.reshape(-1, a.shape[-1])
            keep = int(len(pixels) * keep_fraction)
            a = pixels[np.sort(np.random.default_rng(0).choice(len(pixels), size=keep, replace=False))]
        np.save(out / f"{name}.npy", a)


def icosphere(subdiv=3):
    """Unit icosphere, outward-wound triangles."""
    t = (1 + 5 ** 0.5) / 2
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], dtype=np.float64)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                  [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                  [6, 2, 10], [8, 6, 7], [9, 8, 1]], dtype=np.int64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    for _ in range(subdiv):
        mid = {}
        verts = list(v)
        out = []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                p = verts[a] + verts[b]
                verts.append(p / np.linalg.norm(p))
                mid[k] = len(verts) - 1
            return mid[k]

        for a_, b_, c_ in f:
            ab, bc, ca = m(a_, b_), m(b_, c_), m(c_, a_)
            out += [[a_, ab, ca], [b_, bc, ab], [c_, ca, bc], [ab, bc, ca]]
        v, f = np.array(verts), np.array(out, dtype=np.int64)
    # the kernel keeps triangles whose (v1-v0)x(v2-v0) faces the ray origin side: outward here
    n = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    flip = (n * v[f[:, 0]]).sum(1) < 0
    f[flip] = f[flip][:, ::-1]
    return v.astype(np.float32), f


def run_animated(a):
    """BASELINE config 5: an object moved every frame by the reference's Euler
    integrator (PhysStep, src/physics.c:49-53); every frame rebuilds the kd-tree of
    terrain + object and renders it.  --anim-builder gpu (default): the mesh is uploaded
    and the tree built and re-laid-out ON THE DEVICE (CLBuildMeshes), by every rank for
    itself -- the build is deterministic, so the replicas are identical and nothing has to
    be broadcast; --anim-builder host: binned SAH build on the host cores + CLSetMeshes."""
    import ctypes as C

    import torch
    import torch.distributed as dist

    import clpathtracer_b200 as cl
    from clpathtracer_b200 import scenes

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = cl.lib()
    a.sah_bins = 32  # a per-frame rebuild wants the fast builder: binned planes, no clipping
    tv, tc, _ = scenes.heightfield(a.grid, False)
    sv, sf = icosphere(3)
    sv = sv * np.float32(0.12)
    sc = cl.corners_from_faces(sf + len(tv), False)
    corners = np.concatenate([tc, sc])
    pos, vel = cl.Vector4(), cl.Vector4()
    pos.s[:] = [0.0, 0.6, -0.4, 0.0]
    vel.s[:] = [0.25, 0.0, 0.35, 0.0]
    L.AddPhysObject(C.byref(pos), C.byref(vel))
    r = cl.Renderer(device=local)
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = np.zeros(128, dtype=np.uint8)
            L.CLDistGetUniqueId(raw.ctypes.data)
            idbuf = torch.from_numpy(raw.copy())
        idbuf = idbuf.cuda()
        dist.broadcast(idbuf, 0)
        raw = idbuf.cpu().numpy().copy()
        L.CLDistInit(rank, world, raw.ctypes.data, a.tile_rows)
    r.create_image(a.width, a.height)
    r.set_params(mode=cl.MODE_MIRROR, depth=a.depth, spp=a.spp, seed=a.seed, flags=cl.FLAG_JITTER)
    cam = cl.cam_matrix(cl.make_camera(**scenes.CANONICAL_CAMERA), a.height)
    host = torch.empty((a.height, a.width, 4), dtype=torch.uint8).pin_memory().numpy()
    verts = np.zeros((len(tv) + len(sv), 4), dtype=np.float32)
    verts[:len(tv), :3] = tv[:, :3]
    dt, g = 1.0 / 60.0, -1.5
    t_build, t_upload, t_render, t_frame, dev_build, dev_pack = [], [], [], [], [], []
    frames = a.warmup + a.steps
    import gc

    gc.disable()  # a collection in the middle of a frame is a 10+ ms outlier that is not the renderer's
    hosts = [host, torch.empty((a.height, a.width, 4), dtype=torch.uint8).pin_memory().numpy()]
    scene = None

    def one_frame(f, pipelined):
        nonlocal scene
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        vel.s[1] = vel.s[1] + g * dt
        L.PhysStep(dt)
        if pos.s[1] < 0.3 and vel.s[1] < 0:
            vel.s[1] = -vel.s[1]
        verts[len(tv):, :3] = sv + np.array(pos.s[:3], dtype=np.float32)
        if a.anim_builder == "gpu":
            t1 = time.perf_counter()
            if f == 0:
                r.build_meshes(verts, corners, None)      # the whole mesh crosses PCIe once
            else:
                r.update_vertices(len(tv), verts[len(tv):])  # then only the vertices that moved
                r.rebuild_meshes()
            t2 = time.perf_counter()
            b_ms, p_ms = r.build_ms()
            dev_build.append(b_ms), dev_pack.append(p_ms)
        else:
            scene = cl.build_kd_sah(verts, corners, None, nbins=a.sah_bins, intersect_cost=1.0, empty_bonus=0.9,
                                    clip=False)
            t1 = time.perf_counter()
            r.set_meshes(scene)
            t2 = time.perf_counter()
        r.set_camera_matrix(cam)
        r.execute()
        if rank == 0:
            if pipelined:  # frame f's copy to the host overlaps frame f + 1's rebuild
                r.read_image_async(hosts[f % 2])
                r.read_wait(1)
            else:
                r.read_image_rgba8(host)
        return t0, t1, t2, time.perf_counter()

    for f in range(frames):
        t0, t1, t2, t3 = one_frame(f, False)
        if f >= a.warmup:
            t_build.append(t1 - t0), t_upload.append(t2 - t1), t_render.append(t3 - t2), t_frame.append(t3 - t0)
    # the same frames as a stream: read-back pipelined one frame deep (CLReadImageAsync), frames per second is what counts
    t_stream = []
    for f in range(frames, 2 * frames):
        t0, _, _, t3 = one_frame(f, True)
        if f >= frames + a.warmup:
            t_stream.append(t3 - t0)
    r.read_wait(0)
    gc.enable()
    if a.dump_outputs:
        frame = r.read_image()
        if rank == 0:  # `delivered`: the RGBA8 texels the last streamed frame landed in host memory
            dump_outputs(a.dump_outputs, {"frame": frame, "delivered": hosts[(2 * frames - 1) % 2]})
    # self-check: the LAST frame (whatever tree the last rebuild made) against the oracle walking that tree
    parity = {"checked": False}
    if not a.no_parity_check:
        import hashlib

        from oracle import oracle_py as op

        frame = r.read_image()
        sha = hashlib.sha256(frame.tobytes()).hexdigest()
        if rank == 0:
            tree = r.download_kd() if a.anim_builder == "gpu" else scene
            ref = op.render(tree, cam, a.width, a.height, mode=1, depth=a.depth, spp=a.spp, seed=a.seed,
                            flags=op.FLAG_JITTER, aov=False, threads=host_cores())["rgba"]
            differ = int(np.count_nonzero(frame.view(np.uint32) != ref.view(np.uint32)))
            parity = {"checked": True, "words_differ": differ, "words": int(ref.size), "frame_sha256": sha,
                      "oracle": "oracle/oracle_kernel.c walking the tree of the last frame"
                                + (" (downloaded from the device, CLDownloadKd)" if a.anim_builder == "gpu" else "")}
    L.PhysTerminate()
    if world > 1:
        L.CLDistShutdown()
    r.close()
    ms = lambda x, q: round(float(np.percentile(x, q)) * 1e3, 3)  # noqa: E731
    if rank == 0:
        gpu = a.anim_builder == "gpu"
        breakdown = ({"transform(host)": ms(t_build, 50), "CLUpdateVertices+CLRebuildMeshes(upload of the moved vertices+device build+re-layout)": ms(t_upload, 50),
                      "  of which device build": round(float(np.median(dev_build)), 3),
                      "  of which device re-layout": round(float(np.median(dev_pack)), 3),
                      "camera+CLExecute+CLReadImageRGBA8": ms(t_render, 50)} if gpu else
                     {"transform+kd_build(host)": ms(t_build, 50), "CLSetMeshes(pack+upload)": ms(t_upload, 50),
                      "camera+CLExecute+CLReadImageRGBA8": ms(t_render, 50)})
        emit({"metric": "ms/frame, animated scene (per-frame object transform + kd rebuild + re-upload), 1080p 4 spp",
              "value": ms(t_frame, 50), "unit": "ms", "higher_is_better": False, "n_gpus": world, "steps": len(t_frame),
              "warmup": a.warmup, "p50_ms": ms(t_frame, 50), "p99_ms": ms(t_frame, 99), "max_ms": ms(t_frame, 100),
              "streamed_p50_ms": ms(t_stream, 50), "streamed_p99_ms": ms(t_stream, 99),
              "streamed": "the same loop with the read-back pipelined one frame deep (CLReadImageAsync + CLReadImageWait(1)): "
                          "ms per frame of a running animation; `value` is the latency of one frame, transform to pixels in host memory",
              "breakdown_p50_ms": breakdown, "kd_builder": "device (CLBuildMeshes)" if gpu else "host (build_kd_sah, binned)",
              "parity": parity,
              "config": dict(workload_config(a), triangles=int(len(corners) // 3)), "data": "synthetic", "dtype": "f32"})
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    quiet_stdout()
    if a.impl == "reference":
        return run_reference(a)
    if a.config == "c5":
        return run_animated(a)

    import torch
    import torch.distributed as dist

    import clpathtracer_b200 as cl

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
        a.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the render path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    scene, cam, info = make_scene(a)
    L = cl.lib()
    r = cl.Renderer(device=local)
    r.set_meshes(scene)
    r.set_camera_matrix(cam)
    L.CLSetEngine(a.engine)
    if world > 1:
        # the NCCL id is made by rank 0 and carried over torch.distributed (plumbing only)
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = (np.zeros(128, dtype=np.uint8))
            L.CLDistGetUniqueId(raw.ctypes.data)
            idbuf = torch.from_numpy(raw.copy())
        idbuf = idbuf.cuda()
        dist.broadcast(idbuf, 0)
        raw = idbuf.cpu().numpy().copy()
        L.CLDistInit(rank, world, raw.ctypes.data, a.tile_rows)
    r.create_image(a.width, a.height)
    a.direct_placement = int(L.CLDistDirectPlacement()) if world > 1 else 1
    flags = (0 if a.no_jitter else cl.FLAG_JITTER) | (cl.FLAG_ACCUMULATE if a.progressive else 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # instrumented frame: counts rays / node / triangle work for this rank's rows
    mode = {"normal": cl.MODE_NORMAL, "mirror": cl.MODE_MIRROR, "path": cl.MODE_PATH}[a.mode]
    r.set_params(mode=mode, depth=a.depth, spp=a.spp, seed=a.seed, flags=flags | cl.FLAG_COUNTERS)
    r.execute()
    counters = r.counters()
    r.set_params(mode=mode, depth=a.depth, spp=a.spp, seed=a.seed, flags=flags)
    totals = torch.tensor([counters[k] for k in ("rays", "splits", "leaves", "tris", "shade_vn", "capped")],
                          dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(totals)
    tot = dict(zip(("rays", "splits", "leaves", "tris", "shade_vn", "capped"), [int(x) for x in totals.tolist()]))
    rays_per_frame = tot["rays"]

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(a.warmup, 3)):
        r.execute()

    # ---- timed: device-resident ----
    barrier()
    sampler.arm()
    wall0 = time.time()
    step_ms, kern_ms = [], []
    for _ in range(a.steps):
        L.CLFlushL2()
        if world > 1:
            dist.barrier()
        L.CLEventRecord(0)
        r.execute()
        L.CLEventRecord(1)
        step_ms.append(L.CLEventElapsedMs(0, 1))
        kern_ms.append(r.kernel_ms())
    barrier()
    wall = time.time() - wall0
    clocks = sampler.result()
    launches = a.steps * L.CLLastLaunchCount()

    # ---- timed: end to end through the C ABI with host buffers ----
    # Every step: camera matrix host -> device, CLExecute, and the step's result -- ONE frame --
    # device -> pinned host memory.  The frame is delivered in the reference's render-target
    # format (RGBA8, src/GLHandler.c:177-185) unless --readback float4, through the pipelined
    # read-back (CLReadImageAsync: frame k travels while frame k+1 renders; every frame has
    # landed before the clock stops).  Across GPUs the frame is assembled on every rank and
    # read back by rank 0, the rank that owns the host buffer; a progressive frame lives in the
    # ranks' slabs, so its read-back is collective and every rank takes part.
    host_dtype = torch.uint8 if a.readback == "rgba8" else torch.float32
    host_frames = [torch.empty((a.height, a.width, 4), dtype=host_dtype).pin_memory() for _ in range(2)]
    host_np = [t.numpy() for t in host_frames]
    cam_host = np.ascontiguousarray(cam, dtype=np.float32)
    reader = rank == 0 or (a.progressive and world > 1)

    def e2e_step(k):
        r.set_camera_matrix(cam_host)   # 64 B host -> device (rides in the launch parameters)
        r.execute()
        if reader:
            if a.readback_sync:
                (r.read_image_rgba8 if a.readback == "rgba8" else r.read_image)(host_np[k & 1])
            else:
                r.read_image_async(host_np[k & 1])
                r.read_wait(1)          # frame k-1 has landed; frame k travels during the next step

    for k in range(2):                  # untimed: the read-back path's one-time set-up (second stream, staging)
        e2e_step(k)
    if reader:
        r.read_wait(0)
    barrier()
    e2e_t0 = time.time()
    e2e_each = []
    for k in range(a.steps):
        t_k = time.perf_counter()
        e2e_step(k)
        e2e_each.append(round((time.perf_counter() - t_k) * 1e3, 4))
    t_k = time.perf_counter()
    if reader:
        r.read_wait(0)
    t_drain = time.perf_counter() - t_k
    barrier()
    e2e_s = time.time() - e2e_t0
    if rank == 0:
        print(f"e2e steps (ms): {e2e_each}, drain {t_drain * 1e3:.3f} ms, total {e2e_s * 1e3:.3f} ms", file=sys.stderr)
    d2h_bytes = a.width * a.height * (4 if a.readback == "rgba8" else 16)
    if a.dump_outputs:
        frame = r.read_image()
        if rank == 0:  # `delivered`: what the last end-to-end step landed in host memory, in the --readback format
            dump_outputs(a.dump_outputs, {"frame": frame, "delivered": host_np[(a.steps - 1) & 1]})

    # ---- self-check frame: the timed parameters, read back once more (outside every timed region) ----
    import hashlib

    if a.progressive:
        L.CLResetAccumulation()
    r.execute()
    check_frame = r.read_image().copy()
    my_sha = hashlib.sha256(check_frame.tobytes()).hexdigest()
    shas = [my_sha]
    if world > 1:
        mine = torch.tensor(list(bytes.fromhex(my_sha)), dtype=torch.uint8, device="cuda")
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        shas = [bytes(x.cpu().tolist()).hex() for x in every]

    t = torch.tensor([sum(step_ms), sum(kern_ms), e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kernel_total_ms, e2e_ms = t.tolist()
    per_rank_kernel_ms = None
    if world > 1:  # how evenly the row tiles split the work: each rank's mean render-kernel time
        mine = torch.tensor([float(np.mean(kern_ms))], dtype=torch.float64, device="cuda")
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        per_rank_kernel_ms = [round(float(x.item()), 4) for x in every]

    if rank == 0:
        ms_per_step = total_ms / a.steps
        value = rays_per_frame / (ms_per_step * 1e-3) / 1e6
        e2e_value = rays_per_frame / (e2e_ms / a.steps * 1e-3) / 1e6
        peak, peak_src = hbm_peak()
        # roofline of the render kernel: algorithmic bytes of ONE launch on this rank / its duration
        my_rows = a.height if a.progressive else len(cl_rows(a, rank, world))
        my_bytes = algorithmic_bytes(counters, my_rows * a.width)
        kernel_ms = float(np.mean(kern_ms))
        achieved = my_bytes / (kernel_ms * 1e-3) / 1e9
        # What binds: one ncu --set full capture per workload (profiles/binding.json, made by
        # profiles/summarise_ncu.py from the .ncu-rep of the same command at N = 1).  DRAM traffic and
        # unit utilisations are properties of that captured launch; at N > 1 a launch covers 1/N of
        # the frame, so they are attached for reference and labelled, not scaled.
        traffic, binding = None, None
        bp = ROOT / "profiles" / "binding.json"
        key = a.config if a.mode == "mirror" and not a.no_jitter else ("modeA_ref" if a.builder == "ref" else "modeA_sah")
        if bp.exists():
            try:
                binding = json.loads(bp.read_text()).get(key)
            except Exception:
                binding = None
        if binding is not None:
            binding = dict(binding, captured_at_n_gpus=1,
                           note="lane_issue_efficiency = issue-slot utilisation x active threads per warp instruction / 32: "
                                "the share of the SMs' lane-issue capacity that does work; the busiest unit is the one "
                                "that binds this kernel, not HBM")
            if world == 1:
                traffic = binding.get("dram_bytes_per_launch")
        out = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            # by region the frame is fixed as N grows (strong); progressive frames are spread by sample:
            # every rank renders a whole frame per step, the step's sample count grows with N (weak)
            "scaling": "weak" if a.progressive else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a),
            "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": 64,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": round(e2e_ms / a.steps, 4),
                    "readback": {"format": a.readback, "pipelined": not a.readback_sync,
                                 "api": "CLReadImageAsync + CLReadImageWait" if not a.readback_sync else
                                        ("CLReadImageRGBA8" if a.readback == "rgba8" else "CLReadImage"),
                                 "readers": world if (a.progressive and world > 1) else 1,
                                 "note": "one frame per step reaches pinned host memory inside the timed region; "
                                         "RGBA8 is the reference's render-target format"}},
            "gpu_launches": launches,
            "per_rank_kernel_ms": per_rank_kernel_ms,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 5), "traffic": traffic, "peak_source": peak_src,
                         "kernel": "render_kernel<%d,false,%d>" % (mode, L.CLLastEngine() - 1),
                         "kernel_ms": round(kernel_ms, 4),
                         "note": "formal bound per SURVEY.md section 8d: algorithmic bytes / kernel time against the measured "
                                 "HBM copy bandwidth.  It does NOT bind (the scene is served by L1/L2; measured DRAM "
                                 "traffic is in `traffic`), so this fraction can exceed 1 and earns nothing by itself; "
                                 "`binding` names the unit that does bind and its utilisation",
                         "binding": binding,
                         "algorithmic_bytes_per_launch": my_bytes,
                         "bytes_per_ray": round(my_bytes / max(counters["rays"], 1), 1)},
            "rays_per_frame": rays_per_frame,
            "work_per_ray": {k: round(tot[k] / max(tot["rays"], 1), 3) for k in ("splits", "leaves", "tris")},
            "capped_rays": tot["capped"],
            "ms_per_frame": round(ms_per_step, 4), "wall_ms_per_step_incl_flush": round(wall / a.steps * 1e3, 3),
            "device": L.CLDeviceName().decode(), "scene": info,
            "engine": {1: "1 (8 resident blocks per SM)", 2: "2 (fat-leaf variant, 4 resident blocks)"}[L.CLLastEngine()],
        }
        want_baseline = world == 1 and not a.no_cpu_baseline
        if want_baseline or not a.no_parity_check:
            baseline, parity = oracle_check_and_baseline(a, scene, cam, None if a.no_parity_check else check_frame,
                                                         a.cpu_seconds, want_baseline, world)
        else:
            baseline, parity = None, {"checked": False}
        # every rank holds the whole frame: one sha per rank, to be compared with each other and,
        # across runs, with the N=1 line's
        if a.progressive:
            parity["check_frame"] = (f"the first progressive frame after a reset: the mean of ranks x spp = "
                                     f"{world * a.spp} samples per pixel (the oracle adds the same samples)")
        parity["frame_sha256"] = shas[0]
        parity["frame_sha256_per_rank"] = shas
        parity["ranks_agree"] = len(set(shas)) == 1
        if parity.get("checked") and parity["rows"] == [0, a.height]:
            parity["frame_equals_oracle"] = parity["words_differ"] == 0 and parity["oracle_sha256"] == shas[0]
        out["cpu_baseline"] = baseline
        out["parity"] = parity
        emit(out)
    if world > 1:
        L.CLDistShutdown()
    r.close()
    if world > 1:
        dist.destroy_process_group()


def cl_rows(a, rank, world):
    from clpathtracer_b200 import sharding

    return sharding.rows_of_rank(a.height, rank, world, a.tile_rows)


if __name__ == "__main__":
    main()
