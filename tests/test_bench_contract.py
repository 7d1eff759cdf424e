"""bench.py's JSON contract, on the arm that runs without a GPU: `--impl reference`
(the CPU port of the reference algorithm).  The GPU arm prints the same keys plus
roofline / gpu_launches / clocks; it is exercised on the GPU box by the driver."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_one_json_line(clpt, oracle, tmp_path):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", "c1", "--steps", "2",
                        "--warmup", "1", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["metric"].startswith("Mrays/s") and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["vs_baseline"] is None and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    # --dump-outputs: the frame of the last timed step (c1: 1 spp per step, step k renders sample k)
    from clpathtracer_b200 import scenes

    frame = np.load(tmp_path / "frame.npy")
    assert frame.dtype == np.float32 and frame.shape == (480, 640, 4)
    scene = clpt.build_kd_sah(*scenes.heightfield(22, False), nbins=0, intersect_cost=1.0, empty_bonus=0.9)
    cam = clpt.cam_matrix(clpt.make_camera(**scenes.CANONICAL_CAMERA), 480)
    kw = dict(mode=1, depth=2, spp=1, seed=0, flags=oracle.FLAG_JITTER, aov=False)
    assert np.array_equal(frame.view(np.uint32), oracle.render(scene, cam, 640, 480, sample_base=1, **kw)["rgba"].view(np.uint32))
    assert not np.array_equal(frame, oracle.render(scene, cam, 640, 480, sample_base=0, **kw)["rgba"])


def test_dump_outputs_samples_every_array_at_one_rate(tmp_path, monkeypatch):
    import bench

    frame = np.arange(30 * 20 * 4, dtype=np.uint8).reshape(30, 20, 4)
    bench.dump_outputs(tmp_path / "whole", {"frame": frame})  # 9600 bytes as float32: under the limit
    whole = np.load(tmp_path / "whole" / "frame.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, frame)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4800)   # 12800 bytes below: each array keeps 3/8 of its pixels
    for out in ("a", "b"):
        bench.dump_outputs(tmp_path / out, {"frame": frame, "delivered": frame[:10]})
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("frame", "delivered")}
    assert got["frame"].shape == (225, 4) and got["delivered"].shape == (75, 4)
    assert got["frame"].dtype == got["delivered"].dtype == np.float32
    rows = {tuple(p) for p in frame.reshape(-1, 4).astype(np.float32)}
    assert all(tuple(p) in rows for a in got.values() for p in a)  # whole pixels of the frame
    for n, a in got.items():                                      # the same ones every run
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{n}.npy"))
