"""Shared helpers of the parity tests: build a device population from oracle problems, inject the
draws, and compare against the CPU oracle (oracle/ is the checker, never the thing under test)."""
import contextlib
from dataclasses import replace

import numpy as np
import torch

from oracle.sac_eo_oracle import NetCfg, draw_batch, make_problem, sac_eo_update, to_torch_state
from sac_expert_b200.population import Population, PopulationSpec


def rel(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def spec_from_cfg(cfg: NetCfg, n_agents, B, E, N, **kw) -> PopulationSpec:
    # tests default to the exact-fp32 engine launched kernel by kernel; the tensor-core engine / graphs are opted into
    from sac_expert_b200 import lib as _lib
    kw.setdefault("gemm_mode", _lib.GEMM_FP32_SIMT)
    kw.setdefault("use_graph", False)
    return PopulationSpec(n_agents=n_agents, S=cfg.S, A=cfg.A, actor_hidden=cfg.actor_hidden,
                          critic_hidden=cfg.critic_hidden, model_hidden=cfg.model_hidden,
                          actor_acts=cfg.actor_acts, critic_acts=cfg.critic_acts, model_acts=cfg.model_acts,
                          per_state_std=cfg.per_state_std, separate_reward_nn=cfg.separate_reward_nn,
                          num_models=cfg.num_models, delta_clip_pred=cfg.delta_clip_pred, B=B, E=E,
                          replay_capacity=N, std_mult=cfg.std_mult, **kw)


def build(cfg: NetCfg, n_agents, B, E, N, seed=0, perturb=0.05, eps=0.3, identity_norm=False, **kw):
    """-> (population, problems) with problems[i] = (state_np, replay, expert, hyper, batch)."""
    probs = []
    for i in range(n_agents):
        st, replay, expert, hyper = make_problem(cfg, B, E, N, seed=seed + 17 * i, perturb=perturb,
                                                 identity_norm=identity_norm)
        hyper["eps"] = eps
        hyper["gamma"] = 0.995 - 0.01 * i       # per-agent hyper-parameters differ
        batch = draw_batch(cfg, replay, expert, B, seed=seed + 1000 + i)
        probs.append((st, replay, expert, hyper, batch))
    return populate(cfg, probs, B, E, N, **kw), probs


def populate(cfg: NetCfg, probs, B, E, N, **kw) -> Population:
    """A device population holding problems[i] as agent i, with their draws injected."""
    pop = Population(spec_from_cfg(cfg, len(probs), B, E, N, **kw))
    for i, (st, replay, expert, hyper, batch) in enumerate(probs):
        pop.load_agent(i, st, hyper)
        pop.append_rows(i, replay["s"], replay["a"], replay["r"], replay["sp"], replay["d"])
        if cfg.num_models > 0:
            pop.set_expert(i, expert["sE"], expert["spE"])
    inject(pop, cfg, probs)
    return pop


@contextlib.contextmanager
def fp32_expert_term(on=True):
    """Populations updated inside the block run the expert term on the fp32 CUDA-core kernel (k_model_term) where the
    tensor-core kernel (k_model_term_mma) would run by default."""
    from sac_expert_b200 import lib as L
    lib = L.load()
    L.check(lib.saceo_test_set_mt_fp32(int(on)))
    try:
        yield
    finally:
        L.check(lib.saceo_test_set_mt_fp32(0))


# ------------------------------------------------------------------------------------------------------------------
# edge fixtures: make_problem results edited so that each branch edge of the element-wise stages is hit exactly, with
# values fp32 represents exactly (tests/test_edges_host.py proves on the CPU that every edge is really hit)
# ------------------------------------------------------------------------------------------------------------------
LOG_STD_EDGES = (-5.0, 2.0, -5.5, 2.5, -1.0, 0.5)      # boundaries, outside, interior; cycled over the action dims
ACT_LIMITS = (0.4, 1.0, 2.5)
SAT_MEAN = 12.0          # mean bias of the dims whose clamped log-std is 2 (std 7.39): tanh(z) rounds to +-1 on many rows
SAT_Z = 10.0             # fp64 |z| above which tanh rounds to +-1 in fp32 on every implementation (it does from ~9.01)
CONST_COLS = (1, 4)      # state columns with a zero normaliser std and every stored value equal to the mean
ALPHA_FLOOR_START = 1.2e-5
EDGES = ("head", "ties", "alpha_floor", "delta_clip", "eps0", "eps1")


def log_std_edges(A):
    return np.array([LOG_STD_EDGES[j % len(LOG_STD_EDGES)] for j in range(A)], np.float32)


def edit_problem(cfg: NetCfg, prob, edge: str, agent: int = 0):
    """Edits one make_problem result (st, replay, expert, hyper) in place so that ``edge`` is hit:
      head        clamped log-std (per-state: zero W2 log-std columns, b2 = LOG_STD_EDGES; state-independent: the
                  variable), saturated squash (mean bias +-SAT_MEAN where the clamped log-std is 2), per-dimension
                  act_limit, done flags on half the rows, CONST_COLS with s_std = 0
      ties        q2 := q1, t2 := t1, q2's Adam slots := q1's
      alpha_floor alpha 1.2e-5, very negative target entropy, lr_alpha large: the unclamped Adam step lands below 1e-5
      delta_clip  nothing here: the clip is chosen from the drawn batch (straddle_clip)
      eps0 / eps1 expert weight 0 / 1"""
    st, replay, expert, hyper = prob
    A = cfg.A
    if edge == "head":
        ls = log_std_edges(A)
        sgn = np.where(np.arange(A) % 2 == 0, 1.0, -1.0) * (1 - 2 * (agent % 2))
        mean_b = np.where(np.clip(ls, -5.0, 2.0) == 2.0, sgn * SAT_MEAN, 0.0).astype(np.float32)
        if cfg.per_state_std:
            st["actor"][4][:, A:] = 0.0
            st["actor"][5][A:] = ls
            st["actor"][5][:A] = mean_b
        else:
            st["actor"][6][0, :] = ls
            st["actor"][5][:] = mean_b
        st["act_limit"] = np.array([ACT_LIMITS[j % len(ACT_LIMITS)] for j in range(A)], np.float32)
        replay["d"][:] = (np.arange(len(replay["d"])) % 2 == 0).astype(np.float64)
        for c in CONST_COLS:
            st["s_std"][c] = 0.0
            for key in ("s", "sp"):
                replay[key][:, c] = st["s_mean"][c]
            for key in ("sE", "spE"):
                expert[key][:, c] = st["s_mean"][c]
    elif edge == "ties":
        for k in ("q", "t"):
            st[k + "2"] = [w.copy() for w in st[k + "1"]]
        st["adam_q2"] = dict(m=[w.copy() for w in st["adam_q1"]["m"]], v=[w.copy() for w in st["adam_q1"]["v"]],
                             t=st["adam_q1"]["t"])
    elif edge == "alpha_floor":
        st["alpha"] = np.float32(ALPHA_FLOOR_START)
        hyper["target_entropy"] = -1000.0
        hyper["lr_alpha"] = 1e-3
    elif edge == "eps0":
        hyper["eps"] = 0.0
    elif edge == "eps1":
        hyper["eps"] = 1.0
    elif edge != "delta_clip":
        raise ValueError(edge)


def edge_problems(cfg: NetCfg, edge: str, n_agents, B, E, N, seed=0, eps=0.3):
    """-> (cfg, problems) like build's, each problem edited by edit_problem; for "delta_clip" the returned cfg carries
    a delta_clip_pred that the fp64 model outputs of the expert rows straddle."""
    probs = []
    for i in range(n_agents):
        st, replay, expert, hyper = make_problem(cfg, B, E, N, seed=seed + 17 * i, perturb=0.05)
        hyper["eps"] = eps
        hyper["gamma"] = 0.995 - 0.01 * i
        edit_problem(cfg, (st, replay, expert, hyper), edge, i)
        batch = draw_batch(cfg, replay, expert, B, seed=seed + 1000 + i)
        probs.append((st, replay, expert, hyper, batch))
    if edge == "delta_clip":
        cfg = replace(cfg, delta_clip_pred=straddle_clip(np.concatenate(
            [np.concatenate([d.ravel() for d in expert_deltas(cfg, p)]) for p in probs])))
    return cfg, probs


def build_edge(cfg: NetCfg, edge: str, n_agents, B, E, N, seed=0, eps=0.3, **kw):
    """build() on edge_problems: -> (population, problems, cfg)."""
    cfg, probs = edge_problems(cfg, edge, n_agents, B, E, N, seed, eps)
    return populate(cfg, probs, B, E, N, **kw), probs, cfg


def straddle_clip(delta, margin=1e-4):
    """A clip (exact in fp32) between two neighbouring |delta| near their median, at least ``margin`` relative away
    from every |delta|, so that the clip mask does not depend on rounding."""
    a = np.unique(np.abs(np.asarray(delta, np.float64).ravel()))
    mid = len(a) // 2
    for k in sorted(range(int(0.3 * len(a)), int(0.7 * len(a))), key=lambda k: abs(k - mid)):
        c = float(np.float32(0.5 * (a[k] + a[k + 1])))
        if c - a[k] > margin * c and a[k + 1] - c > margin * c:
            return c
    raise AssertionError("no clip with a margin found")


def _t64(x):
    return torch.as_tensor(np.asarray(x)).to(torch.float64)


def actor_out64(cfg: NetCfg, st, s):
    """fp64 (mean, raw log-std) of the actor on states s, before the clamp."""
    from oracle.sac_eo_oracle import mlp, normalize
    th = [_t64(w) for w in st["actor"]]
    out = mlp(th, normalize(_t64(s), _t64(st["s_mean"]), _t64(st["s_std"])), cfg.actor_acts)
    if cfg.per_state_std:
        return out[:, :cfg.A], out[:, cfg.A:]
    return out, th[6] * torch.ones_like(out)


def actor_phase_z(cfg: NetCfg, prob):
    """fp64 pre-squash z of the actor-phase rows in the device's row order: the B minibatch rows (noise u2), then the
    E expert rows in permuted order (noise u3 | u4)."""
    st, batch = prob[0], prob[4]
    rows = [(batch["s"], batch["u2"])]
    if cfg.num_models == 1:
        rows.append((batch["sE"], batch["u3"]))
    elif cfg.num_models == 2:
        rows += [(batch["sE"][batch["I1"]], batch["u3"]), (batch["sE"][batch["I2"]], batch["u4"])]
    zs = []
    for s, u in rows:
        mean, ls = actor_out64(cfg, st, s)
        zs.append(mean + torch.exp(torch.clamp(ls, -5.0, 2.0)) * _t64(u))
    return torch.cat(zs).numpy()


def expert_deltas(cfg: NetCfg, prob):
    """fp64 model outputs (state-delta columns, before the clip) on the expert rows, one [rows, S] array per model."""
    from oracle.sac_eo_oracle import head, mlp, normalize
    st, batch = to_torch_state(prob[0], torch.float64), prob[4]
    sE = _t64(batch["sE"])
    parts = [(sE, batch["u3"], st["m1"])] if cfg.num_models == 1 else \
        [(sE[batch["I1"]], batch["u3"], st["m1"]), (sE[batch["I2"]], batch["u4"], st["m2"])]
    out = []
    for s, u, th in parts:
        c, _ = head(cfg, st["actor"], s, _t64(u), st)
        sa = torch.cat([normalize(s, st["m_s_mean"], st["m_s_std"]), normalize(c, st["m_a_mean"], st["m_a_std"])], -1)
        out.append(mlp(th, sa, cfg.model_acts)[:, :cfg.S].numpy())
    return out


def expert_term64(cfg: NetCfg, prob):
    """fp64 expert-observation term as the device splits it: (mdXa [nets, rows, A] = d(eps*MSE)/d(normalised expert
    action columns of each model's input), MSE)."""
    from oracle.sac_eo_oracle import denormalize, head, mlp, normalize
    st, batch, eps = to_torch_state(prob[0], torch.float64), prob[4], prob[3]["eps"]
    sE, spE = _t64(batch["sE"]), _t64(batch["spE"])
    idx = [np.arange(len(sE))] if cfg.num_models == 1 else [batch["I1"], batch["I2"]]
    us = [batch["u3"]] if cfg.num_models == 1 else [batch["u3"], batch["u4"]]
    xas, dl = [], 0.0
    for k, (I, u) in enumerate(zip(idx, us)):
        s = sE[I]
        with torch.no_grad():
            c, _ = head(cfg, st["actor"], s, _t64(u), st)
        xa = normalize(c, st["m_a_mean"], st["m_a_std"]).requires_grad_(True)
        sa = torch.cat([normalize(s, st["m_s_mean"], st["m_s_std"]), xa], -1)
        delta = mlp(st["m%d" % (k + 1)], sa, cfg.model_acts)[:, :cfg.S]
        if cfg.delta_clip_pred:
            delta = torch.clamp(delta, -cfg.delta_clip_pred, cfg.delta_clip_pred)
        pred = s + denormalize(delta, st["m_d_mean"], st["m_d_std"])
        dl = dl + ((spE[I] - pred) ** 2).sum(-1)
        xas.append(xa)
    mse = (0.5 * dl).mean()
    g = torch.autograd.grad(eps * mse, xas) if eps else [torch.zeros_like(x) for x in xas]
    return np.stack([x.numpy() for x in g]), float(mse.detach())


def alpha_unclamped(cfg: NetCfg, prob):
    """The fp64 temperature after its Adam step, before the 1e-5 floor (SAC_expert.py:341-348)."""
    import math
    from oracle.sac_eo_oracle import ADAM_B1, ADAM_B2, ADAM_EPS
    o = oracle_update(cfg, prob, torch.float64)
    ad, g = prob[0]["adam_alpha"], float(o["g_alpha"])
    t = ad["t"] + 1
    lr_t = prob[3]["lr_alpha"] * math.sqrt(1 - ADAM_B2 ** t) / (1 - ADAM_B1 ** t)
    m = ADAM_B1 * float(ad["m"]) + (1 - ADAM_B1) * g
    v = ADAM_B2 * float(ad["v"]) + (1 - ADAM_B2) * g * g
    return float(prob[0]["alpha"]) - lr_t * m / (math.sqrt(v) + ADAM_EPS)


def inject(pop, cfg, probs):
    B, E, A = pop.spec.B, (pop.spec.E if cfg.num_models > 0 else 0), cfg.A
    n = len(probs)
    idx = np.stack([p[4]["idx"] for p in probs])
    noise = np.zeros((n, 3 * B + E, A), np.float32)
    perm = np.zeros((n, max(E, 1)), np.int32)
    for i, p in enumerate(probs):
        b = p[4]
        noise[i, :B] = b["u1"]
        noise[i, B:2 * B] = b["u2"]
        if cfg.num_models == 1:
            noise[i, 2 * B:2 * B + E] = b["u3"]
            perm[i] = np.arange(E)
        elif cfg.num_models == 2:
            noise[i, 2 * B:2 * B + E] = np.concatenate([b["u3"], b["u4"]])
            perm[i] = np.concatenate([b["I1"], b["I2"]])
        noise[i, 2 * B + E:] = b["u5"]
    pop.set_draws(idx, noise, perm if E > 0 else None)


def oracle_update(cfg, prob, dtype=torch.float32):
    st, replay, expert, hyper, batch = prob
    return sac_eo_update(cfg, to_torch_state(st, dtype), batch, hyper)


def compare_update(pop, cfg, probs, tol=1e-3, verbose=False):
    """Runs ONE injected-draw update on the device and compares every tensor with the fp32 oracle.
    Returns the dict of worst relative errors."""
    L = pop.L
    pop.update(1, num_timesteps=0, use_device_rng=False)
    torch.cuda.synchronize()
    losses = pop.losses.cpu().numpy()
    g_q = pop.debug("g_q").cpu().numpy().reshape(pop.spec.n_agents, 2, L.nc_stride)
    g_a = pop.debug("g_actor").cpu().numpy().reshape(pop.spec.n_agents, L.na_stride)
    y = pop.debug("y").cpu().numpy().reshape(pop.spec.n_agents, pop.spec.B)
    worst = {}

    def upd(k, v):
        worst[k] = max(worst.get(k, 0.0), v)

    for i, prob in enumerate(probs):
        o = oracle_update(cfg, prob)
        o64 = oracle_update(cfg, prob, torch.float64)
        upd("oracle32_vs_64_g_actor", rel(np.concatenate([g.numpy().ravel() for g in o["g_actor"]]),
                                         np.concatenate([g.numpy().ravel() for g in o64["g_actor"]])))
        upd("y", rel(y[i], o["y"].numpy()))
        for j, k in enumerate(("L_q1", "L_q2", "L_pi", "mse", "p_loss", "alpha_loss")):
            ref = float(o[k])
            upd(k, abs(losses[i, j] - ref) / max(abs(ref), 1e-12) if ref != 0 else abs(losses[i, j]))
        upd("alpha", abs(losses[i, 6] - float(o["new"]["alpha"])) / abs(float(o["new"]["alpha"])))
        for net, key in ((0, "g_q1"), (1, "g_q2")):
            ref = np.concatenate([g.numpy().ravel() for g in o[key]])
            upd(key, rel(g_q[i, net, :ref.size], ref))
        ref = np.concatenate([g.numpy().ravel() for g in o["g_actor"]])
        upd("g_actor", rel(g_a[i, :ref.size], ref))
        upd("g_alpha", abs(g_a[i, -1] - float(o["g_alpha"])) / max(abs(float(o["g_alpha"])), 1e-12))
        for name in ("q1", "q2", "t1", "t2", "actor"):
            got = pop.get_net(i, name)
            new, old = o["new"][name], prob[0][name]
            for gw, nw, ow in zip(got, new, old):
                upd("theta_" + name, rel(gw, nw.numpy()))
                dref = nw.numpy() - np.asarray(ow)
                if np.linalg.norm(dref) > 0:
                    upd("dtheta_" + name, rel(gw - np.asarray(ow), dref))
        for name, (tm, tv) in (("q1", ("q_m", "q_v")), ("q2", ("q_m", "q_v")), ("actor", ("actor_m", "actor_v"))):
            for gw, nw in zip(pop.get_net(i, name, table=tm), o["new"]["adam_" + name]["m"]):
                upd("adam_m_" + name, rel(gw, nw.numpy()))
            for gw, nw in zip(pop.get_net(i, name, table=tv), o["new"]["adam_" + name]["v"]):
                upd("adam_v_" + name, rel(gw, nw.numpy()))
    if verbose:
        for k, v in worst.items():
            print(f"  {k:28s} {v:.3e}")
    return worst


def _engines():
    from sac_expert_b200 import lib as L
    tc = dict(gemm_mode=L.GEMM_TCGEN05_BF16X3)
    small = dict(actor_hidden=(64, 64), critic_hidden=(64, 64), model_hidden=(64, 64))
    # name -> (cfg, B, E, population keywords); the fused tcgen05 cases run graph + fork as bench.py does
    # the frozen models are tanh: with ReLU models an expert row whose hidden pre-activation lies within fp32 rounding of
    # 0 takes the branch its summation order picks (test_model_relu_tie_confined_to_one_row), which A = 17 / seed 5 hits
    mt = dict(model_acts=("tanh", "tanh"))
    update = {
        "fp32_S11_A6": (NetCfg(S=11, A=6, **small, **mt), 128, 8, dict(gemm_mode=L.GEMM_FP32_SIMT)),
        "tc_fused_ant": (NetCfg(S=27, A=8, **mt), 256, 20, dict(tc, use_graph=True)),
        "tc_fused_A17": (NetCfg(S=45, A=17, **mt), 256, 20, dict(tc, use_graph=True)),     # W2 rows straddle k_adam's float4s
        "tc_unfused_ant": (NetCfg(S=27, A=8, **mt), 256, 20, dict(tc, fuse_forward=False, fuse_backward=False)),
    }
    tanh = dict(actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"), model_acts=("tanh", "tanh"),
                actor_hidden=(32, 32), critic_hidden=(32, 32))
    # expert-term implementations: k_model_term_mma (default), k_model_term (fp32_expert_term), the GEMM chain with
    # k_model_loss (more expert rows per model than the fused kernels take)
    term = {
        "mma": (NetCfg(S=11, A=3, model_hidden=(512, 512), **tanh), 64, 20),
        "fp32": (NetCfg(S=11, A=3, model_hidden=(512, 512), **tanh), 64, 20),
        "chain": (NetCfg(S=11, A=3, model_hidden=(64, 64), **tanh), 160, 80),
    }
    return update, term


UPDATE_ENGINES, TERM_IMPLS = _engines()
