"""bench.py's command line and JSON line; the reference arm runs without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--gib", "0.0625",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)  # a 64 MiB shard: the host generator is a Python loop
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]
    counts = np.load(tmp_path / "match_counts.npy")
    assert counts.dtype == np.float64 and counts.tolist() == [line["config"]["matches"], 0, line["config"]["matches"]]


def test_other_ranks_of_the_reference_arm_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly(tmp_path):
    """Runs of 2 and 3 timed steps on the same inputs launch 2 and 3 steps' worth of kernels in the timed
    region and dump the same arrays."""
    dumps, launches = [], []
    for steps in (2, 3):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0", "--gib", "0.5", "--no-e2e",
                              "--no-cpu", "--no-extras", "--dump-outputs", str(tmp_path / str(steps))],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        launches.append(line["gpu_launches"])
        dumps.append({f.stem: np.load(f) for f in sorted((tmp_path / str(steps)).iterdir())})
    assert launches[0] > 0 and launches[0] * 3 == launches[1] * 2, launches
    a, b = dumps
    assert sorted(a) == ["match_counts", "span_index", "spans"] and sorted(b) == sorted(a)
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["match_counts"][0] == line["config"]["matches_rank0"] == a["match_counts"][2]
    assert a["spans"].shape == (a["span_index"].shape[0], 2) and 0 < a["spans"].shape[0] < a["match_counts"][0]  # a sample
    assert (a["spans"][:, 0] < a["spans"][:, 1]).all()
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name in a:
        assert np.array_equal(a[name], b[name]), name
