"""bench.py's output contract.  CPU: the reference arm (`--impl reference`) runs the CPU oracle on a bounded sample of the workload
and must print the keys of the result line, with a `config` that names the WORKLOAD only (the same dict our arm prints for the same
flags: bench.workload_config); the --dump-outputs writer.  GPU: --steps sets the number of timed steps, and --dump-outputs writes
the same records for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--frames", "6", "--keyframes", "2",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "tracks/s" and line["higher_is_better"] is True
    assert line["metric"] == "frame-keyframe GN tracks/sec at 640x480"
    assert line["gpu_launches"] == 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"]
    assert cb["reference_faithful"]["cores"] == 3 and cb["reference_faithful"]["value"] > 0      # NUM_POSE_THREADS, src/ExternVariable.h:224
    # the workload, and nothing but the workload
    assert set(line["config"]) == {"workload", "width", "height", "keyframes_per_gpu", "frames_per_gpu", "pairs_per_gpu_per_step",
                                   "pairs_per_frame", "l2"}
    assert line["config"]["workload"] == "pair_sweep_640x480" and (line["config"]["width"], line["config"]["height"]) == (640, 480)
    assert line["implementation"]["sample_pairs_per_step"] <= line["config"]["pairs_per_gpu_per_step"]

    sys.path.insert(0, ROOT)
    import bench
    bench.W, bench.H = 640, 480
    want = bench.workload_config(bench.CONFIGS["pair_sweep"], 2, 6, line["config"]["pairs_per_frame"], line["config"]["pairs_per_gpu_per_step"])
    assert want == line["config"]
    # inputs of the default workload: 512 frames + 32 keyframes (image, 4-level depth and variance) + 4608 pair records
    assert bench.input_bytes_per_step(512, 32, 4608) == 271730688


def test_dump_outputs_writer(tmp_path):
    """One float32 / float64 .npy per field of the result record; a table above 64 MB is written as a fixed, seeded sample."""
    sys.path.insert(0, ROOT)
    import bench
    from egomotion_with_local_loop_closures_b200 import capi
    rec = np.zeros(400000, capi.RESULT_DTYPE)
    rec["status"] = np.arange(len(rec))
    rec["pose"] = np.random.default_rng(1).standard_normal((len(rec), 6))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rec)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted([n + ".npy" for n in capi.RESULT_DTYPE.names if n != "reserved"] + ["pair_index.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 * 10**6
    idx = np.load(tmp_path / "a" / "pair_index.npy")
    assert 100000 < len(idx) < len(rec) and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "status.npy"), idx)
    assert np.array_equal(np.load(tmp_path / "a" / "pose.npy"), rec["pose"][idx.astype(np.int64)])
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, np.load(tmp_path / "b" / n)), n


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    """Two runs of the pipelined path that differ only in --steps: the timed region's launches scale with the step count, and the
    records of the last timed step are identical (seeded inputs, run-to-run deterministic kernels)."""
    lines = []
    for steps in (2, 3):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--frames", "32", "--keyframes", "9", "--steps", str(steps),
                              "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(steps))],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads(out.stdout.strip().splitlines()[-1]))
    assert [l["steps"] for l in lines] == [2, 3] and lines[0]["config"]["pairs_per_gpu_per_step"] == 288
    assert "alternate" in lines[0]["implementation"]["pipelining"]
    assert lines[0]["gpu_launches"] > 0 and lines[1]["gpu_launches"] * 2 == lines[0]["gpu_launches"] * 3
    names = sorted(os.listdir(tmp_path / "2"))
    assert names == sorted(os.listdir(tmp_path / "3")) and "pose.npy" in names
    for n in names:
        a, b = np.load(tmp_path / "2" / n), np.load(tmp_path / "3" / n)
        assert a.dtype in (np.float32, np.float64) and len(a) == 288 and np.array_equal(a, b), n
    assert np.all(np.load(tmp_path / "2" / "n_iters.npy").sum(axis=1) > 0) and np.abs(np.load(tmp_path / "2" / "pose.npy")).max() > 0
