"""Acting throughput of ``saceo_policy_act`` (``k_policy_forward``) for sets of expert policies: the reference's expert
shape on Ant dimensions (S = 27, A = 8, 3 x 256 elu, per-state std: 142,864 parameters, 0.57 MB per policy),
deterministic head, P in {1, 8, 64, 256, 1024} policies x rows in {1, 256} observations per policy.

Timing: CUDA events around ``--iters`` (>= 200) back-to-back launches after ``--warmup`` launches, replayed from a CUDA
graph so that the number is device time and not the Python binding's call overhead (``us_per_call_direct`` is the same
loop through ``PolicySet.actor_forward``, host overhead included).  Reported per point: microseconds per call,
policy-rows/s, and the unique weight bytes per call (P x 0.57 MB) over the call time as a share of 7.7 TB/s (HBM3e,
HGX B200 data sheet).  A weight set that fits the 126 MB L2 is read from L2 on every call after the first, so
``weights_fit_l2`` marks the points whose share of HBM bandwidth is an L2 figure.  Writes one JSON with the GPU name and
power limit read in the same run.

    python tools/policy_bench.py --out profiles/policy_forward_bench.json"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from sac_expert_b200 import lib as L  # noqa: E402
from sac_expert_b200.policy import PolicySet, PolicySpec  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "?", "max_sm_clock": "?"}
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def point(P, rows, iters, warmup):
    spec = PolicySpec(n_agents=P, S=27, A=8, hidden=(256, 256, 256), acts=("elu",) * 3, squash=False, per_state_std=True,
                      std_mult=0.3)
    ps = PolicySet(spec)
    g = torch.Generator(device="cuda").manual_seed(P * 1000 + rows)
    ps.params.normal_(0.0, 1.0 / 16.0, generator=g)             # ~ 1 / sqrt(fan-in) for the 256-wide layers
    obs = torch.randn(P, rows, spec.S, device="cuda", generator=g)
    out = torch.empty(P, rows, spec.A, device="cuda")
    lib = ps.lib

    def launch():
        st = torch.cuda.current_stream().cuda_stream
        L.check(lib.saceo_policy_act(C.byref(ps.cfg), ps.params.data_ptr(), ps.norm.data_ptr(), obs.data_ptr(), rows,
                                     None, out.data_ptr(), st))

    for _ in range(warmup):
        launch()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        for _ in range(iters):
            launch()
    graph.replay()                                              # warm the graph once
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    e1.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    # the same number of calls through the Python binding (allocation + ctypes call per call)
    x = obs.clone()
    for _ in range(warmup):
        ps.actor_forward(x)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        ps.actor_forward(x)
    e1.record()
    e1.synchronize()
    us_direct = e0.elapsed_time(e1) * 1e3 / iters
    wbytes = P * ps.n_params * 4
    return {"P": P, "rows": rows, "us_per_call": round(us, 3), "us_per_call_direct": round(us_direct, 3),
            "policy_rows_per_s": round(P * rows / (us * 1e-6), 1), "weight_bytes_per_call": wbytes,
            "weight_bytes_per_s": round(wbytes / (us * 1e-6), 1),
            "share_of_hbm_7p7TBps": round(wbytes / (us * 1e-6) / HBM_BYTES_PER_S, 4),
            "weights_fit_l2": wbytes <= L2_BYTES, "iters": iters}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "policy_forward_bench.json"))
    p.add_argument("--P", type=int, nargs="+", default=[1, 8, 64, 256, 1024])
    p.add_argument("--rows", type=int, nargs="+", default=[1, 256])
    p.add_argument("--iters", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    a = p.parse_args()
    if a.iters < 200:
        raise SystemExit("--iters must be at least 200")
    res = {"gpu": card(), "kernel": "k_policy_forward (saceo_policy_act)",
           "shape": {"S": 27, "A": 8, "hidden": [256, 256, 256], "act": "elu", "per_state_std": True, "n_params": 142864},
           "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S, "l2_bytes": L2_BYTES, "results": []}
    for rows in a.rows:
        for P in a.P:
            row = point(P, rows, a.iters, a.warmup)
            print(json.dumps(row), flush=True)
            res["results"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
