#!/usr/bin/env python
"""bench.py - agent-updates/sec of the SAC-EO population update on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU update step (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as .npy files

A "step" is ONE `SAC_exp._update` for EVERY agent of the population resident on a GPU (gather ->
critics -> actor (+expert term) -> temperature -> Polyak).  Weak scaling: every rank holds
`--agents` agents (default 256), no data-path collective (agents are independent).  Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--shape", default="ant", choices=["hopper", "halfcheetah", "ant", "humanoid"])
    p.add_argument("--agents", type=int, default=256, help="agents per GPU (weak scaling, the default)")
    p.add_argument("--total-agents", type=int, default=None,
                   help="STRONG scaling: a fixed global population sharded over the ranks (agent i -> rank i %% world)")
    p.add_argument("--no-strong-record", action="store_true",
                   help="skip the 256-total-agents strong-scaling sub-record that multi-GPU runs add to the weak line")
    p.add_argument("--replay-rows", type=int, default=100_000)
    p.add_argument("--plain-sac", action="store_true", help="no expert term (BASELINE configs[1])")
    p.add_argument("--gemm-mode", type=int, default=None, help="0 fp32 SIMT, 1 tcgen05 hi/lo x3 (default)")
    p.add_argument("--tc-variant", type=int, default=0)
    p.add_argument("--no-fuse-forward", action="store_true")
    p.add_argument("--no-fuse-backward", action="store_true")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--no-ws", action="store_true", help="round-1 fused kernels instead of the warp-specialised TMA-fed ones")
    p.add_argument("--no-fork", action="store_true", help="whole update on one stream")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-seconds", type=float, default=16.0)
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last of them computed to DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    if a.dump_outputs and a.impl != "b200":
        p.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return a


def workload_name(a):
    from sac_expert_b200.synth import SHAPES
    S, A, B = SHAPES[a.shape]
    alg = "plain SAC" if a.plain_sac else "SAC-EO (2 MSEModels 2x512, E=20, eps=1e-3)"
    pop = (f"{a.total_agents}-agent population sharded over the GPUs" if getattr(a, "total_agents", None)
           else f"{a.agents}-agent population per GPU")
    return (f"{alg} {a.shape}-shaped (obs {S}, act {A}), actor/critics 2x256 relu, batch {B}, "
            f"{pop}, replay {a.replay_rows} rows/agent")


# ------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU baseline: the reference's update step, restated (oracle port), on the host cores
# ------------------------------------------------------------------------------------------
def cpu_update_rate(a, seconds, threads=None):
    """Times oracle.sac_eo_update (torch-CPU eager, autograd = tf.GradientTape, per-tensor Keras Adam,
    Polyak) for ONE agent at the benchmark's dimensions.  TensorFlow is not installable offline, so this is
    kind="port" (see DESIGN.md)."""
    import numpy as np
    import torch
    from oracle.sac_eo_oracle import NetCfg, draw_batch, make_problem, sac_eo_update, to_torch_state
    from sac_expert_b200.synth import SHAPES
    S, A, B = SHAPES[a.shape]
    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = NetCfg(S=S, A=A, num_models=0 if a.plain_sac else 2)
    st, replay, expert, hyper = make_problem(cfg, B, 20, 20000, seed=0)
    state = to_torch_state(st)
    n, t0 = 0, None
    deadline = None
    while True:
        batch = draw_batch(cfg, replay, expert, B, seed=n)      # includes the gather, like _update does
        out = sac_eo_update(cfg, state, batch, hyper)
        new = out["new"]
        for k in ("actor", "q1", "q2", "t1", "t2", "alpha", "adam_actor", "adam_q1", "adam_q2", "adam_alpha"):
            state[k] = new[k]
        n += 1
        if n == 3:                       # warm-up
            t0 = time.perf_counter(); deadline = t0 + seconds; n0 = n
        if deadline is not None and time.perf_counter() >= deadline:
            break
    dt = time.perf_counter() - t0
    return (n - n0) / dt, cores, n - n0


def _pool_worker(shape, plain_sac, seconds, q):
    """One single-threaded process = one independent agent, the reference's own parallel model (one process per seed
    through multiprocessing.Pool, train.py:130-152)."""
    import argparse
    # one thread per process, BLAS pools included (NumPy's QR in the problem builder would otherwise start one
    # OpenBLAS pool per process and the oversubscribed start-up takes half a minute)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    try:
        rate, _, n = cpu_update_rate(argparse.Namespace(shape=shape, plain_sac=plain_sac), seconds, threads=1)
        q.put((rate, n))
    except Exception as e:          # a dead worker must not hang the parent
        q.put((0.0, 0))
        raise e


def cpu_pool_rate(a, seconds, procs=None):
    """Aggregate agent-updates/s of `procs` single-threaded worker processes, each updating its own agent for `seconds`
    (spawned, so that a CUDA context in the parent is not inherited)."""
    import multiprocessing as mp
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_pool_worker, args=(a.shape, a.plain_sac, seconds, q)) for _ in range(procs)]
    saved = {v: os.environ.get(v) for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")}
    for v in saved:
        os.environ[v] = "1"                     # inherited by the spawned interpreters before they import NumPy / torch
    try:
        for p in ps:
            p.start()
    finally:
        for v, old in saved.items():
            if old is None:
                os.environ.pop(v, None)
            else:
                os.environ[v] = old
    import queue
    res = []
    deadline = time.perf_counter() + seconds + 150
    try:
        while len(res) < procs and time.perf_counter() < deadline:
            try:
                res.append(q.get(timeout=1.0))
            except queue.Empty:
                if not any(p.is_alive() for p in ps) and q.empty():
                    break                       # workers died without reporting: do not wait for the deadline
    finally:
        for p in ps:
            p.join(timeout=10)
            if p.is_alive():
                p.kill()
    res = [r for r in res if r[1] > 0]
    if not res:
        raise RuntimeError("no worker process reported a rate")
    return sum(r for r, _ in res), len(res), sum(n for _, n in res)


def cpu_baseline(a, seconds):
    """The reference's CPU update step on all host cores, both ways the reference can use them: (1) one agent, all cores
    as intra-op threads; (2) its multiprocessing model - one single-threaded process per core, independent agents.  The
    better aggregate is reported as the value; both are described."""
    r1, cores, n1 = cpu_update_rate(a, seconds / 2)
    try:
        r2, procs, n2 = cpu_pool_rate(a, seconds / 2, cores)
    except Exception as e:          # e.g. a sandbox without process spawning: keep the single-process figure
        r2, procs, n2 = 0.0, 0, 0
        print(f"# cpu pool baseline unavailable: {e}", file=sys.stderr)
    rate = max(r1, r2)
    probe = probe_reference()
    tf_res = None
    if probe["usable"]:               # the real reference (TensorFlow eager) is runnable here: cross-check + time it
        from oracle.tf_reference import crosscheck_and_time
        from sac_expert_b200.synth import SHAPES
        S_, A_, B_ = SHAPES[a.shape]
        tf_res = crosscheck_and_time(probe["reference_tree"], (S_, A_), B_, 20, seconds / 2)
    sample = (f"oracle/sac_eo_oracle.py (torch-CPU eager restatement of SAC_exp._update; TensorFlow probe: "
              f"tensorflow={probe['tensorflow']}, gym={probe['gym']}, reference tree={probe['reference_tree']}), "
              f"single-agent updates of the same shape: (1) one process, {cores} intra-op threads: {n1} updates in "
              f"{seconds / 2:.0f} s = {r1:.1f}/s; (2) {procs} single-threaded processes x independent agents (the "
              f"reference's mp.Pool model, train.py:130-152): {n2} updates in {seconds / 2:.0f} s = {r2:.1f}/s")
    out = {"value": rate, "unit": "agent-updates/s", "cores": cores, "kind": "port", "sample": sample,
           "single_process": r1, "process_pool": r2, "one_thread_process": (r2 / procs if procs else None),
           "os_cpu_count": os.cpu_count(), "reference_probe": probe}
    if tf_res is not None:
        out["tf_reference"] = tf_res
        if tf_res.get("ok"):
            out.update({"kind": "reference (TF eager)", "value": tf_res["updates_per_s"], "port_value": rate,
                        "sample": "the reference's own SAC_exp._update under TensorFlow eager, one process; oracle cross-check "
                                  "max rel err of the actor update %.2e; port: %s" % (tf_res["max_rel_dtheta_actor"], sample)})
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # K "steps", each a bounded sample (a fixed number of single-agent updates) of the population step
    per_step_budget = max(0.5, min(6.0, 80.0 / max(1, a.steps + a.warmup)))
    budget = float(os.environ.get("SACEO_REF_SECONDS", per_step_budget * (a.steps + a.warmup)))   # env: contract test only
    cb = cpu_baseline(a, budget)
    rate, cores = cb["value"], cb["cores"]
    line = {
        "impl": "reference", "metric": "agent-updates/sec", "value": rate, "unit": "agent-updates/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 / rate,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a)},
        "cpu_baseline": cb,
        "e2e": {"value": rate, "unit": "agent-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
def source_hash():
    """Hash of the CUDA sources + ABI header: profiles stamped with it are only used while it still matches."""
    import hashlib
    h = hashlib.sha256()
    base = os.path.join(ROOT, "sac_expert_b200", "csrc")
    for f in sorted(os.listdir(base)) + ["../../include/saceo.h"]:
        with open(os.path.join(base, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def probe_reference():
    """Is the REAL reference runnable here (TensorFlow + gym importable and the reference package under baseline/_ref or
    /root/reference)?  If so oracle/tf_reference.py cross-checks the oracle against the reference's own SAC_exp._update and
    times it; otherwise the torch-CPU restatement is the CPU arm (kind "port")."""
    info = {"tensorflow": False, "gym": False, "reference_tree": None}
    for cand in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if os.path.isdir(os.path.join(cand, "sac_eo")):
            info["reference_tree"] = cand
            break
    for mod in ("tensorflow", "gym"):
        try:
            m = __import__(mod)
            info[mod] = hasattr(m, "__version__")      # the three-function stand-ins under shims/ carry no version: not the real thing
        except Exception as e:          # ImportError or a broken install
            info[mod + "_error"] = type(e).__name__
    info["usable"] = bool(info["tensorflow"] and info["gym"] and info["reference_tree"])
    return info


def measure(pop, a, world, barrier, steps, warmup, torch, dist):
    """W warm-up updates, then `steps` timed updates bracketed by barrier + synchronize; CUDA events on the launching
    stream; MAX over ranks.  Returns (ms for all steps, launches in the timed region)."""
    for w in range(warmup):
        pop.update(1, num_timesteps=w, use_device_rng=True, seed=99)
    barrier()
    l0 = pop.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(pop.stream):
        e0.record(pop.stream)
    pop.update(steps, num_timesteps=warmup, use_device_rng=True, seed=99)
    with torch.cuda.stream(pop.stream):
        e1.record(pop.stream)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), pop.launches - l0


DUMP_BYTES = 64 * 10**6      # --dump-outputs writes at most this much (plus the .npy headers)
DUMP_AGENTS = 16             # agents whose parameter and optimiser tables are written
DUMP_PER_AGENT = ("losses", "alpha", "alpha_m", "alpha_v")
DUMP_TABLES = (("actor", "na"), ("actor_m", "na"), ("actor_v", "na"),
               ("q", "nc"), ("q_m", "nc"), ("q_v", "nc"), ("qt", "nc"))


def dump_outputs(pop, out_dir):
    """Writes the state one timed `pop.update` leaves behind, so that two builds run with the same arguments can be
    compared array for array: the per-agent losses the call returns and the temperature with its Adam moments, for every
    agent; the actor, both critics, both targets and their Adam moments (trimmed to the real parameter count, stride
    padding dropped) for a fixed sample of agents, drawn with numpy.random.default_rng(0), as many as fit DUMP_BYTES
    up to DUMP_AGENTS.  All float32."""
    import numpy as np
    import torch
    L, n = pop.L, pop.spec.n_agents
    out = {name: pop.losses if name == "losses" else pop.t[name] for name in DUMP_PER_AGENT}
    fixed = sum(v.numel() * 4 for v in out.values())
    per_agent = sum(pop.t[name][0, ..., :getattr(L, width)].numel() * 4 for name, width in DUMP_TABLES)
    count = min(n, DUMP_AGENTS, (DUMP_BYTES - fixed) // per_agent)
    agents = np.sort(np.random.default_rng(0).choice(n, size=count, replace=False))
    sel = torch.as_tensor(agents, device=pop.dev)
    out.update({name: pop.t[name][sel, ..., :getattr(L, width)] for name, width in DUMP_TABLES})
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())


def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sac_expert_b200 import lib
    from sac_expert_b200.parallel import agent_shard
    from sac_expert_b200.population import Population, PopulationSpec
    from sac_expert_b200.synth import (SHAPES, algorithmic_bytes, algorithmic_flops, fill_synthetic, kernel_compulsory_bytes,
                                       kernel_design_bytes)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    S, A, B = SHAPES[a.shape]
    gemm_mode = a.gemm_mode if a.gemm_mode is not None else lib.GEMM_TCGEN05_BF16X3
    strong = a.total_agents is not None
    n_local = len(agent_shard(a.total_agents, rank, world)) if strong else a.agents
    n_global = a.total_agents if strong else world * a.agents
    if n_local < 1:
        raise SystemExit("--total-agents must be >= the number of ranks")

    def make_pop(n):
        spec_ = PopulationSpec(n_agents=n, S=S, A=A, B=B, E=20, num_models=0 if a.plain_sac else 2,
                               replay_capacity=a.replay_rows, gemm_mode=gemm_mode, tc_variant=a.tc_variant,
                               fuse_forward=not a.no_fuse_forward, fuse_backward=not a.no_fuse_backward,
                               use_graph=not a.no_graph, ws_kernels=not a.no_ws, fork_actor=not a.no_fork, device=local)
        p_ = Population(spec_)
        fill_synthetic(p_, seed=1234 + rank)
        return spec_, p_

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                  # sampled across warm-up, the timed region and the end-to-end section
    spec, pop = make_pop(n_local)

    # ---- device-resident throughput ("value") ------------------------------------------------
    ms, launches = measure(pop, a, world, barrier, a.steps, a.warmup, torch, dist)
    losses = pop.losses.cpu().numpy()
    if not np.isfinite(losses).all():
        raise RuntimeError("non-finite losses after the timed region")
    if a.dump_outputs and rank == 0:     # before the end-to-end section below updates the same population again
        dump_outputs(pop, a.dump_outputs)
    value = n_global * a.steps / (ms * 1e-3)

    # ---- end-to-end through the host-buffer API ("e2e") -------------------------------------
    rng = np.random.default_rng(7 + rank)
    sizes = pop._host_size
    expert = np.stack([pop.t["expert_s"].cpu().numpy(), pop.t["expert_sp"].cpu().numpy()], 0) \
        if spec.num_models > 0 else None
    e2e_steps = max(3, min(a.steps, 20))
    for w in range(4):                         # warm-up: both pinned staging sets allocated, graphs instantiated
        idx = rng.integers(0, sizes[:, None], size=(n_local, B)).astype(np.int64)
        pop.update_host_async(w, 5, idx, expert, slot=w & 1)
        pop.wait_host(w & 1)
    barrier()
    t0 = time.perf_counter()
    prev = None
    for sidx in range(e2e_steps):
        idx = rng.integers(0, sizes[:, None], size=(n_local, B)).astype(np.int64)   # np.random.randint, buffers.py:135
        pop.update_host_async(sidx, 5, idx, expert, slot=sidx & 1)                  # H2D idx+expert rows, update, D2H losses
        if prev is not None:
            out = pop.wait_host(prev)          # the previous step's losses are consumed on the host while this one runs
        prev = sidx & 1
    out = pop.wait_host(prev)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = n_global * e2e_steps / float(dt.item())
    h2d = n_local * (B * 8 + (2 * spec.E * S * 4 if spec.num_models > 0 else 0))
    d2h = n_local * pop.L.n_losses * 4
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel device times, live: one un-graphed single-stream update with a CUDA event after every launch -----
    kern_us = {}
    if rank == 0:
        reps = 3
        for w in range(1 + reps):
            prof = pop.profile_step(w, True, seed=9)
            if w == 0:
                continue                       # first un-graphed step: lazy module loads
            for name, us in prof:
                # the weight-gradient contractions: dW1 (k_dw_planes), dW0 (k_dw0_planes), dW2 / fallbacks (k_gemm_*)
                key = "k_dw_planes+k_dw0_planes+k_gemm" if name.startswith(("k_gemm", "k_dw")) else name
                kern_us[key] = kern_us.get(key, 0.0) + us / reps

    # ---- strong-scaling sub-record: the SAME 256-agent population sharded over the ranks (BASELINE configs[2]) --------
    strong_rec = None
    if world > 1 and not strong and not a.no_strong_record:
        tot = 256
        pop.close()
        del pop
        torch.cuda.empty_cache()
        n2 = len(agent_shard(tot, rank, world))
        _, pop2 = make_pop(n2)
        ms2, _ = measure(pop2, a, world, barrier, a.steps, a.warmup, torch, dist)
        strong_rec = {"total_agents": tot, "agents_per_gpu": n2, "value": tot * a.steps / (ms2 * 1e-3), "unit": "agent-updates/s",
                      "ms_per_step": ms2 / a.steps, "scaling": "strong",
                      "note": "fixed 256-agent population, agent i on rank i % world, no data-path collective"}
        pop2.close()
        pop = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic, traffic_note = None, "no ncu DRAM-byte profile for this build and workload"
    tj = os.path.join(ROOT, "profiles", "r2_step_traffic.json")
    if os.path.exists(tj) and a.shape == "ant" and not a.plain_sac:
        tr = json.load(open(tj))          # ncu dram__bytes_{read,write}.sum summed over the launches of one step
        if tr.get("source_hash") == source_hash():
            traffic = (tr["dram_read_bytes_per_step"] + tr["dram_write_bytes_per_step"]) / tr["agents"] * n_local
            traffic_note = ("DRAM bytes per step from profiles/r2_step_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum of every launch of one step; capture command in the file's note), "
                            "taken with exactly these kernel sources (source hash %s)" % tr["source_hash"])
        else:
            traffic_note = ("profiles/r2_step_traffic.json was taken with other kernel sources (hash %s, now %s): not reported"
                            % (tr.get("source_hash"), source_hash()))
    per_agent = algorithmic_bytes(spec, L := pop_layout(spec, lib))
    bytes_step = per_agent * n_local
    step_s = ms / a.steps * 1e-3
    achieved = bytes_step / step_s / 1e9
    flops_step = algorithmic_flops(spec) * n_local
    tflops = flops_step / step_s / 1e12
    bf16_sust = float(peaks.get("bf16_tflops_sustained", 1400.0))
    line = {
        "metric": "agent-updates/sec", "value": value, "unit": "agent-updates/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "agents_per_gpu": n_local, "total_agents": n_global, "batch": B,
                   "gemm_engine": ("tcgen05 fp16 hi/lo x3 (fp32 accumulation in TMEM): warp-specialised fused 3-layer forward / backward "
                                   "kernels fed by cp.async.bulk from optimiser-maintained weight planes; TMA-fed bf16 hi/lo x3 weight-gradient kernels on activation plane images; "
                                   "expert term: 2x512 models on mma.sync m16n8k16 fp16 hi/lo x3 streamed from HBM (10 rows per model)"
                                   if gemm_mode == 1 and not a.no_ws else
                                   "tcgen05 16-bit hi/lo x3, round-1 fused kernels" if gemm_mode == 1 else "fp32 SIMT"),
                   "cuda_graph": not a.no_graph, "second_stream_branch": not a.no_fork, "rng": "in-kernel Philox4x32-10",
                   "l2_note": f"population state {bytes_step / 1e9:.2f} GB/step per GPU vs 126 MB L2; no explicit flush"
                              + ("" if bytes_step > 4 * 126e6 else " (NOTE: small population, partly L2-resident between steps)")},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "agent-updates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "note": "Population.update_host_async/wait_host: every step copies host np.random.randint indices + host expert "
                                            "rows H2D from pinned memory and the losses D2H; two pinned staging sets, so the host draws "
                                            "step t+1 while the device runs step t"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                     "achieved_note": "SURVEY.md 8d algorithmic bytes per step / CUDA-event step time",
                     "scope": f"whole update step ({int(launches) // max(a.steps, 1)} kernel launches); algorithmic bytes "
                              f"{per_agent / 1e6:.2f} MB/agent-update",
                     "algorithmic_tflops": tflops,
                     "tensor_note": (f"{tflops:.1f} algorithmic TFLOP/s = {tflops / (bf16_sust / 3):.3f} of the 3-pass-split tensor bound "
                                     f"(bf16 sustained {bf16_sust:.0f} / 3), {tflops / (bf16_sust / 2):.3f} of the TF32-equivalent bound")},
        "reference_probe": probe_reference(),
    }
    if a.shape == "humanoid":            # FLOP/B = 209: the tensor pipe bounds this shape (SURVEY.md 8d)
        line["roofline"].update({"bound": "tensor", "achieved": tflops, "peak": bf16_sust / 3, "unit": "TFLOP/s",
                                 "frac": tflops / (bf16_sust / 3),
                                 "peak_source": "MEASURED_PEAKS.json bf16 sustained / 3 (three 16-bit MMAs per fp32 product)",
                                 "hbm_frac": achieved / hbm_peak})
    if strong_rec:
        line["strong"] = strong_rec
    # per-kernel table from the live per-launch times (the dominant kernel first)
    kdes, kcomp = kernel_design_bytes(spec, L), kernel_compulsory_bytes(spec, L)
    tot_us = sum(kern_us.values()) or 1.0
    kernels = []
    for name, us in sorted(kern_us.items(), key=lambda kv: -kv[1])[:6]:
        ent = {"kernel": name, "us_per_step": us, "share": us / tot_us}
        if kdes.get(name):
            bw = kdes[name] * n_local / (us * 1e-6) / 1e9
            ent.update({"design_bytes_per_step": kdes[name] * n_local, "bandwidth_GBs": bw, "bandwidth_util": bw / hbm_peak})
        if kcomp.get(name):
            ach = kcomp[name] * n_local / (us * 1e-6) / 1e9
            ent.update({"algorithmic_bytes_per_step": kcomp[name] * n_local, "achieved": ach, "unit": "GB/s", "frac": ach / hbm_peak})
        kernels.append(ent)
    line["roofline"]["kernels"] = kernels
    line["roofline"]["kernels_note"] = (
        "saceo_profile_step: one update launched kernel by kernel on ONE stream (no graph, no second-stream branch), CUDA event "
        "after every launch, mean of 3; launch gaps are charged to the following kernel; un-graphed step total "
        f"{tot_us / 1e3:.2f} ms.  `frac` = SURVEY.md 8d compulsory bytes apportioned to the kernel that must move them (optimiser: "
        "theta/m/v/targets, model term: frozen model weights, gather: minibatch rows) over its time - a roofline fraction; "
        "`bandwidth_util` = the bytes the kernel moves BY DESIGN over its time - a utilisation, not a roofline fraction (the "
        "fused forward / backward / weight-gradient kernels have no compulsory traffic of their own)")
    if not a.no_cpu_baseline and world == 1:      # reported baseline: rank 0 at N = 1 only
        line["cpu_baseline"] = cpu_baseline(a, a.cpu_seconds)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def pop_layout(spec, lib):
    return lib.query_layout(spec.to_config())


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
