"""Cost of the dynamics-model depth: agent-fit-steps/s of model fitting and the SAC-EO update's ms per step for models
of 2x512 (the reference default, fused expert term), 3x512 and 4x200 (MBPO-style; every model pass on the per-layer
GEMM chain), one population at a time, CUDA-event timed.  The card's name and power limit are printed with the numbers.
    python tools/model_depth_bench.py [--agents 256] [--shape ant] [--fit-steps 20] [--update-steps 30] [--out FILE]"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sac_expert_b200 import lib as L
from sac_expert_b200.population import Population, PopulationSpec
from sac_expert_b200.synth import SHAPES, fill_synthetic

MODELS = {"2x512": (512, 512), "3x512": (512, 512, 512), "4x200": (200, 200, 200, 200)}

ap = argparse.ArgumentParser()
ap.add_argument("--agents", type=int, default=256)
ap.add_argument("--shape", default="ant")
ap.add_argument("--fit-steps", type=int, default=20)
ap.add_argument("--update-steps", type=int, default=30)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--mb", type=int, default=200)
ap.add_argument("--rows", type=int, default=20000)
ap.add_argument("--gemm-mode", type=int, default=L.GEMM_TCGEN05_BF16X3)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("model_depth_bench.py measures the GPU: no CUDA device")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(0), "?")
    return dict(name=name, power_limit=power)


def timed(pop, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(pop.stream):
        e0.record(pop.stream)
        fn()
        e1.record(pop.stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


S, A = SHAPES[a.shape][:2]
res = dict(card=card(), agents=a.agents, shape=a.shape, model_batch=a.mb, gemm_mode=a.gemm_mode, models={})
for name, hidden in MODELS.items():
    spec = PopulationSpec(n_agents=a.agents, S=S, A=A, B=256, E=20, num_models=2, replay_capacity=a.rows,
                          model_hidden=hidden, model_acts=("relu",) * len(hidden), gemm_mode=a.gemm_mode)
    pop = Population(spec)
    fill_synthetic(pop, seed=0, replay_rows=a.rows)
    pop.fit_bind(a.mb)
    g = torch.Generator(device="cuda").manual_seed(0)
    idx = torch.randint(0, a.rows, (a.fit_steps, a.agents, 2, a.mb), device="cuda", generator=g)
    pop.model_fit(idx[: a.warmup], want_losses=False)
    pop.update(a.warmup, use_device_rng=True, seed=1)
    torch.cuda.synchronize()
    fit_ms = timed(pop, lambda: pop.model_fit(idx, want_losses=False), a.fit_steps)
    upd_ms = timed(pop, lambda: pop.update(a.update_steps, num_timesteps=a.warmup, use_device_rng=True, seed=2),
                   a.update_steps)
    kernels = [k for k, _ in pop.profile_step(use_device_rng=True, seed=3)]
    res["models"][name] = dict(hidden=list(hidden), nm=int(pop.L.nm), fit_ms_per_step=fit_ms,
                               agent_fit_steps_per_s=a.agents / (fit_ms * 1e-3), update_ms_per_step=upd_ms,
                               expert_term="fused" if any(k.startswith("k_model_term") for k in kernels) else "gemm chain",
                               launches_per_update=len(kernels))
    pop.close()
    del pop
    torch.cuda.empty_cache()
print(json.dumps(res))
if a.out:
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
