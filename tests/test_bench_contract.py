"""The command-line contract of ``bench.py``.  CPU: ``--impl reference`` (the reference arm runs without a GPU) prints
one JSON line with the keys a caller reads, the CPU baseline described with both ways the reference can use the host
cores, and a rank != 0 process exits 0 without output.  GPU: ``--dump-outputs`` of the CUDA path."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra, *args):
    env = dict(os.environ, SACEO_REF_SECONDS="2", **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args],
                          capture_output=True, text=True, env=env, timeout=600, check=True)


def test_reference_arm_prints_one_contract_line():
    out = _run({}, "--shape", "hopper", "--steps", "2", "--warmup", "1").stdout.strip().splitlines()
    assert len(out) == 1
    line = json.loads(out[0])
    assert line["impl"] == "reference" and line["metric"] == "agent-updates/sec" and line["unit"] == "agent-updates/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 1
    assert line["value"] > 0 and abs(line["ms_per_step"] - 1e3 / line["value"]) < 1e-6
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"]
    assert cb["value"] == max(cb["single_process"], cb["process_pool"]) and cb["single_process"] > 0
    assert "train.py:130-152" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "WORLD_SIZE": "2"}, "--gpus", "2")
    assert r.stdout.strip() == ""


def test_reference_arm_refuses_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """--dump-outputs: float arrays within 64 MB; the same arrays from a second run with the same arguments; --steps sets
    the number of timed updates (launches scale with it) and the dump follows the last of them."""
    import numpy as np

    def bench(name, steps):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--agents", "5", "--replay-rows", "2000",
                            "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, check=True)
        lines = r.stdout.strip().splitlines()
        assert len(lines) == 1
        return json.loads(lines[0]), {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}

    line2, a = bench("a", 2)
    _, b = bench("b", 2)
    line3, c = bench("c", 3)
    assert line2["steps"] == 2 and line3["steps"] == 3
    per_step = line3["gpu_launches"] - line2["gpu_launches"]
    assert per_step > 0 and line2["gpu_launches"] - 2 * per_step in (0, 1)      # + one seeding launch per update call
    assert set(a) == {"losses", "alpha", "alpha_m", "alpha_v", "actor", "actor_m", "actor_v", "q", "q_m", "q_v", "qt"}
    assert sum(v.nbytes for v in a.values()) <= 64 * 10**6
    assert a["losses"].shape[0] == 5 and a["actor"].shape[0] == 5 and a["q"].shape[:2] == (5, 2)
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        assert np.linalg.norm(v - b[k]) <= 1e-5 * np.linalg.norm(v), k
    assert np.linalg.norm(a["losses"] - c["losses"]) > 1e-3 * np.linalg.norm(a["losses"])
    assert np.linalg.norm(a["actor"] - c["actor"]) > 0
