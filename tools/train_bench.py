"""Training throughput of ``train_population`` (all runs as one device population) next to ``train.main`` (one run after
the other): agent-environment-steps/s = runs x total_timesteps / wall time of the whole ``main`` call, which ends in a
device synchronisation.  Workload: ``sac_imit`` on the synthetic Ant shape (S=27, A=8) with the parser's default network
sizes.  For population mode it also reports where the wall time of the lockstep loop went: the runs' host code (of
which the per-run NumPy draws) and the batched device calls.  Writes one JSON.

    python tools/train_bench.py --out profiles/train_population_bench.json"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from sac_expert_b200.sac_eo import train as T  # noqa: E402
from sac_expert_b200.sac_eo import train_population as TP  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(0), "?")
    return {"name": name, "power_limit": power}


def timed(mode, runs, argv):
    with tempfile.TemporaryDirectory() as d:
        timings = {}
        argv = argv + ["--runs", str(runs), "--save_path", d]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if mode == "population":
            TP.main(argv, timings=timings)
        else:
            T.main(argv)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    return wall, timings


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "train_population_bench.json"))
    p.add_argument("--total_timesteps", type=int, default=3000)
    p.add_argument("--env_batch_size_init", type=int, default=1000)
    p.add_argument("--population_runs", type=int, nargs="+", default=[1, 8, 64, 256])
    p.add_argument("--sequential_runs", type=int, nargs="+", default=[8])
    a = p.parse_args()
    workload = lambda total, init: ["--env_type", "synthetic", "--env_name", "ant", "--alg_type", "sac_imit",
                                    "--actor_squash", "--total_timesteps", str(total), "--env_batch_size_init", str(init),
                                    "--seed", "1"]
    argv = workload(a.total_timesteps, a.env_batch_size_init)
    res = {"gpu": card(), "argv": argv, "unit": "agent-environment-steps/s", "results": []}
    timed("population", 1, workload(300, 200))            # warm-up: library load, first launches
    for mode, rs in (("population", a.population_runs), ("sequential", a.sequential_runs)):
        for R in rs:
            wall, tm = timed(mode, R, argv)
            row = {"mode": mode, "runs": R, "wall_s": round(wall, 3),
                   "agent_env_steps_per_s": round(R * a.total_timesteps / wall, 1)}
            if tm:
                row.update({"lockstep_rounds": tm["rounds"],
                            "share_host": round(tm["host"] / wall, 4), "share_host_draws": round(tm["draws"] / wall, 4),
                            "share_device_calls": round(tm["device"] / wall, 4),
                            "share_setup_and_output": round(1 - (tm["host"] + tm["device"]) / wall, 4)})
            print(json.dumps(row), flush=True)
            res["results"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
