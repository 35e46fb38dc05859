"""bench.py's reference arm runs without a GPU: its JSON line must carry the contract's keys, and under torchrun only
rank 0 may print (it is launched like the GPU arm).  Both arms write the outputs of their last timed step with
--dump-outputs, the same on every run of the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def _run(env_extra, args=("--impl", "reference", "--steps", "1", "--warmup", "0", "--map-points", "60000")):
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_line_has_the_contract_keys():
    lines = _run({})
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "registered_points_per_sec" and d["unit"] == "points/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("C2/C4") and d["config"]["scans_per_gpu_per_step"] == 512
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "scans" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0} or \
        (d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0)


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def _dumped_twice(tmp_path, args):
    """Runs bench.py twice with --dump-outputs; returns the JSON line and the arrays of the first run after checking that
    the second wrote the same float64 files."""
    lines = [_run({}, args + ("--dump-outputs", str(tmp_path / d))) for d in "ab"]
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "poses.npy" in names and "result_n_inlier.npy" in names
    out = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b), n
        out[n[:-4]] = a
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    S = len(out["poses"])
    assert out["poses"].shape == (S, 7) and all(a.shape == (S,) for k, a in out.items() if k != "poses")
    assert np.allclose(np.linalg.norm(out["poses"][:, :4], axis=1), 1.0)
    return json.loads(lines[0][0]), out


def test_reference_arm_dumps_its_last_step(tmp_path):
    line, out = _dumped_twice(tmp_path, ("--impl", "reference", "--steps", "2", "--warmup", "0", "--map-points", "60000"))
    assert line["steps"] == 2 and np.all(out["result_iters"] == 10)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path):
    line, out = _dumped_twice(tmp_path, ("--steps", "3", "--warmup", "1", "--scans-per-gpu", "16", "--map-points", "200000",
                                         "--configs", "none", "--no-cpu-baseline"))
    assert line["steps"] == 3 and len(out["poses"]) == 16 and np.all(out["result_iters"] == 10)
