"""The bench.py contract: the reference arm (`--impl reference`) runs the oracle port on the host cores and prints ONE JSON
line with the contract's keys (no GPU needed); `--dump-outputs` writes the value path's results (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mkeypoints/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("Mkeypoints/s") and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "u8" and d["data"] == "synthetic" and d["steps"] == 1 and d["n_gpus"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and 1 <= cb["cores"] <= (os.cpu_count() or 1) and cb["value"] == d["value"] and cb["sample"]
    assert cb["single_thread_value"] > 0 and 0 < cb["parallel_efficiency"] <= 1.5
    assert d["config"]["frames_per_step_per_gpu"] == 256 and "semantics" in d["config"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_is_refused_outside_the_value_path(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(gpu_required, tmp_path):
    """--dump-outputs writes float32 arrays of what the value path returned in its last timed step; with the same inputs two
    runs (here with a different number of timed steps) write the same values, and the sampled frames are the oracle's."""
    import numpy as np
    import oracle as O
    import bench
    dirs = []
    for steps in (1, 2):
        d = tmp_path / ("s%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--frames", "64", "--batch", "64", "--repeat", "1", "--steps",
                            str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dirs.append(d)
    names = sorted(os.listdir(dirs[0]))
    assert names == ["descriptors.npy", "frame_index.npy", "keypoint_counts.npy", "keypoints.npy", "match_counts.npy", "matches.npy"]
    assert sum(os.path.getsize(dirs[0] / n) for n in names) <= 64 << 20
    out = [{n[:-4]: np.load(d / n) for n in names} for d in dirs]
    for n in out[0]:
        assert out[0][n].dtype in (np.float32, np.float64) and np.array_equal(out[0][n], out[1][n]), n
    assert out[0]["match_counts"].sum() > 0
    frames, _ = bench.make_stream(64, seed=11)
    j = len(out[0]["frame_index"]) - 1
    rc, ok, od, _ = O.extract(O.make_params(bench.NFEAT, bench.SCALE, bench.NLEVELS, 1, bench.FAST_TH), frames[int(out[0]["frame_index"][j])])
    n = int(out[0]["keypoint_counts"][j])
    assert rc == 0 and n == len(ok)
    assert np.array_equal(out[0]["keypoints"][j, :n, 0], ok["x"]) and np.array_equal(out[0]["keypoints"][j, :n, 5], ok["octave"])
    assert np.array_equal(out[0]["descriptors"][j, :n], od)
