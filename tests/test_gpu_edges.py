"""GPU: the SAC-EO update and the acting entry points held to the oracle where their element-wise branches switch -
clamped log-stds, saturated squash, per-dimension act_limit, twin-critic ties, a straddled delta clip, the temperature
floor, expert weights 0 and 1, terminal rows and constant observation columns (the fixtures of tests/helpers.py,
proven to hit their edges by tests/test_edges_host.py).  Besides the norm bars of compare_update, each test asserts the
facts a norm hides: exact zeros, bitwise equalities and the values at the switching inputs."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from oracle.sac_eo_oracle import head, mlp, model_sample, normalize, q_value, to_torch_state
from tests.helpers import (CONST_COLS, SAT_Z, TERM_IMPLS, UPDATE_ENGINES, actor_out64, actor_phase_z, build_edge, compare_update,
                           edge_problems, expert_term64, fp32_expert_term, log_std_edges, oracle_update, populate, rel,
                           straddle_clip)

pytestmark = pytest.mark.gpu
TOL, GTOL = 1e-3, 2e-4      # north_star bar; gradients as RAGGED holds them
N, SEED, NA = 1000, 5, 2


def rup(x, m):
    return (x + m - 1) // m * m


def _np(pop, name, *shape):
    return pop.debug(name).cpu().numpy()[:int(np.prod(shape))].reshape(shape)


def _check_bar(w):
    bad = {k: v for k, v in w.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad
    assert max(w[k] for k in ("g_q1", "g_q2", "g_actor")) < GTOL, w


def _actor_offsets(pop):
    sizes = [int(np.prod(s)) for s in pop.shapes["actor"]]
    return int(np.sum(sizes[:4])), int(np.sum(sizes[:5]))       # W2, b2


def _update(engine, edge, per_state_std=True):
    cfg, B, E, kw = UPDATE_ENGINES[engine]
    pop, probs, cfg = build_edge(replace(cfg, per_state_std=per_state_std), edge, NA, B, E, N, seed=SEED, **kw)
    w = compare_update(pop, cfg, probs)
    torch.cuda.synchronize()
    return pop, probs, cfg, w


# ------------------------------------------------------------------------------------------------------------------
# the update
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_state_std", [True, False])
@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_head_edges_update(engine, per_state_std):
    """Clamped log-stds, saturated squash, act_limit != 1, done rows and constant columns in one update."""
    pop, probs, cfg, w = _update(engine, "head", per_state_std)
    _check_bar(w)
    n, A, B, E, S = NA, cfg.A, pop.spec.B, pop.spec.E, cfg.S
    R, Ao, lay = rup(B + E, 32), pop.L.Ao, pop.L
    ls = log_std_edges(A)
    outside, boundary = (ls < -5) | (ls > 2), (ls == -5) | (ls == 2)
    ga = _np(pop, "g_actor", n, lay.na_stride)
    oW2, ob2 = _actor_offsets(pop)
    h2 = cfg.actor_hidden[1]
    dao = _np(pop, "daOut", n, R, Ao)
    y = _np(pop, "y", n, B)
    Xc2 = _np(pop, "Xc2", n, B, rup(S + A, 4))
    Xpi = _np(pop, "Xpi", n, R, rup(S, 4))
    Xpi2 = _np(pop, "Xpi2", n, R, rup(S, 4))
    for i, p in enumerate(probs):
        st, hyper, batch = p[0], p[3], p[4]
        o = oracle_update(cfg, p, torch.float64)
        # clamp: outside [-5, 2] the log-std gradient is exactly 0; on the boundaries it is the oracle's
        if cfg.per_state_std:
            gw = ga[i, oW2:ob2].reshape(h2, Ao)[:, A:]
            gb = ga[i, ob2 + A:ob2 + Ao]
            rw, rb = o["g_actor"][4].numpy()[:, A:], o["g_actor"][5].numpy()[A:]
            assert (gw[:, outside] == 0).all() and (gb[outside] == 0).all()
            assert rel(gw[:, boundary], rw[:, boundary]) < TOL
        else:
            gb = ga[i, lay.na - A:lay.na]                           # k_lsv_reduce output
            rb = o["g_actor"][6].numpy()[0]
        assert (gb[outside] == 0).all()
        assert (gb[boundary] != 0).all() and rel(gb[boundary], rb[boundary]) < TOL
        # saturation: where fp64 |z| > 10, 1 - t*t is exactly 0 and the mean gradient is the g_nlp (-2t) term alone
        z = actor_phase_z(cfg, p)
        sat = np.abs(z) > SAT_Z
        t = np.sign(z).astype(np.float32)
        wpi = np.float32(1) - np.float32(hyper["eps"])
        g_nlp = np.float32(-np.float32(st["alpha"]) * wpi) / np.float32(B)
        mean_main = dao[i, :B, :A]
        want = (g_nlp * (np.float32(-2) * t[:B])).astype(np.float32)
        assert sat[:B].sum() > 0 and np.array_equal(mean_main[sat[:B]], want[sat[:B]])
        assert sat[B:].sum() > 0 and (dao[i, B:B + E, :A][sat[B:]] == 0).all()
        # terminal rows: y == r bitwise
        done = batch["d"] == 1
        assert done.any() and np.array_equal(y[i][done], batch["r"][done])
        # constant columns normalise to exactly 0
        for c in CONST_COLS:
            assert (Xc2[i, :, c] == 0).all() and (Xpi[i, :B, c] == 0).all() and (Xpi2[i, :B + E, c] == 0).all()
    pop.close()


@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_twin_critic_ties_update(engine):
    """q2 == q1: both critics take bitwise the same step, and the actor's min splits every tie equally."""
    pop, probs, cfg, w = _update(engine, "ties")
    _check_bar(w)
    n, B, A = NA, pop.spec.B, cfg.A
    g_q = _np(pop, "g_q", n, 2, pop.L.nc_stride)
    assert np.array_equal(g_q[:, 0], g_q[:, 1])
    for k in ("q", "qt", "q_m", "q_v"):
        t = pop.t[k].cpu().numpy()
        assert np.array_equal(t[:, 0], t[:, 1]), k
    losses = pop.losses.cpu().numpy()
    assert np.array_equal(losses[:, 0], losses[:, 1])
    cdQ = _np(pop, "cdQ", n, 2, B)
    cdXa = _np(pop, "cdXa", n, 2, B, A)
    for i, p in enumerate(probs):
        wpi = np.float32(1) - np.float32(p[3]["eps"])
        half = np.float32(np.float32(-wpi) / np.float32(B)) * np.float32(0.5)
        assert (cdQ[i] == half).all(), (cdQ[i, :, :4], half)
    assert np.array_equal(cdXa[:, 0], cdXa[:, 1])
    pop.close()


@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_alpha_floor_update(engine):
    pop, probs, cfg, w = _update(engine, "alpha_floor")
    _check_bar(w)
    alpha = pop.t["alpha"].cpu().numpy()
    assert (alpha == np.float32(1e-5)).all(), alpha
    losses = pop.losses.cpu().numpy()
    assert (losses[:, 6] == np.float32(1e-5)).all()
    for i, p in enumerate(probs):
        ref = float(oracle_update(cfg, p, torch.float64)["alpha_loss"])     # -alpha_pre * mean(-nlp3 + H)
        assert abs(losses[i, 5] - ref) < 1e-4 * abs(ref), (losses[i, 5], ref)
    pop.close()


# ------------------------------------------------------------------------------------------------------------------
# the expert-observation term: k_model_term_mma, k_model_term and the GEMM chain with k_model_loss
# ------------------------------------------------------------------------------------------------------------------
def _term(impl, edge):
    cfg, B, E = TERM_IMPLS[impl]
    with fp32_expert_term(impl == "fp32"):
        pop, probs, cfg = build_edge(cfg, edge, NA, B, E, N, seed=SEED)
        w = compare_update(pop, cfg, probs)
        torch.cuda.synchronize()
    return pop, probs, cfg, w


@pytest.mark.parametrize("edge", ["delta_clip", "eps0", "eps1"])
@pytest.mark.parametrize("impl", list(TERM_IMPLS))
def test_expert_term_edges(impl, edge):
    pop, probs, cfg, w = _term(impl, edge)
    _check_bar(w)
    n, B, E, A = NA, pop.spec.B, pop.spec.E, cfg.A
    nets, half = cfg.num_models, E // cfg.num_models
    md = _np(pop, "mdXa", n, 2, E, A)[:, :nets, :half]
    mse_part = _np(pop, "mse_part", n, 2)
    losses = pop.losses.cpu().numpy()
    for i, p in enumerate(probs):
        ref_md, ref_mse = expert_term64(cfg, p)
        assert abs(mse_part[i].sum() - ref_mse) < 1e-5 * ref_mse, (mse_part[i], ref_mse)
        if edge == "eps0":
            assert (md[i] == 0).all()
        else:
            err = rel(md[i], ref_md)
            print(f"MEASURED mdXa {impl} {edge} {err:.2e}")
            assert err < 1e-4, err
        if edge == "eps1":
            R, Ao = rup(B + E, 32), pop.L.Ao
            assert (_np(pop, "daOut", n, R, Ao)[i, :B] == 0).all()
            assert losses[i, 4] == losses[i, 3]
    pop.close()
    if edge == "delta_clip":        # the implementation named is the one that ran
        with fp32_expert_term(impl == "fp32"):
            pop, probs, cfg = build_edge(TERM_IMPLS[impl][0], edge, NA, B, E, N, seed=SEED)
            names = {k for k, _ in pop.profile_step(0, use_device_rng=False)}
        assert ("k_model_loss" in names) == (impl == "chain") and ("k_model_term" in names) == (impl != "chain"), names
        pop.close()


@pytest.mark.parametrize("edge", ["delta_clip", "eps1"])
def test_term_kernels_agree_on_edges(edge):
    """k_model_term_mma and k_model_term on the same edge problem: mdXa and the MSE to fp32 rounding."""
    outs = {}
    for impl in ("mma", "fp32"):
        pop, probs, cfg, w = _term(impl, edge)
        outs[impl] = (_np(pop, "mdXa", NA, 2 * pop.spec.E * cfg.A).copy(), _np(pop, "mse_part", NA, 2).copy())
        pop.close()
    assert rel(outs["mma"][0], outs["fp32"][0]) < 1e-5, rel(outs["mma"][0], outs["fp32"][0])
    assert np.allclose(outs["mma"][1], outs["fp32"][1], rtol=1e-5, atol=1e-9)


# ------------------------------------------------------------------------------------------------------------------
# the acting entry points (lockstep.py / train.py roll out on them)
# ------------------------------------------------------------------------------------------------------------------
ACT_ENGINES = ("fp32_S11_A6", "tc_fused_ant")


def _row_err(dev, ref):
    """max over rows of max |dev - ref| / max(|ref| of the row, rms of ref)."""
    dev, ref = np.asarray(dev, np.float64), np.asarray(ref, np.float64)
    dev, ref = dev.reshape(dev.shape[0], -1), ref.reshape(ref.shape[0], -1)
    den = np.maximum(np.abs(ref).max(1), np.sqrt((ref ** 2).mean()))
    return float((np.abs(dev - ref).max(1) / den).max())


@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("engine", ACT_ENGINES)
def test_actor_forward_edges(engine, noise):
    """Clamped, saturated actor with per-dimension act_limit at 1, 129 and B + 1 rows (a partial tile and a second
    B-row chunk)."""
    cfg, B, E, kw = UPDATE_ENGINES[engine]
    pop, probs, cfg = build_edge(cfg, "head", NA, B, E, N, seed=SEED, **kw)
    for rows in (1, 129, B + 1):
        rng = np.random.default_rng(rows)
        obs = np.stack([p[1]["s"][rng.integers(0, N, rows)] for p in probs])
        u = rng.standard_normal((NA, rows, cfg.A)).astype(np.float32) if noise else None
        out = pop.actor_forward(torch.from_numpy(obs), None if u is None else torch.from_numpy(u), want_neglogp=noise)
        act, nlp = out if noise else (out, None)
        act = act.cpu().numpy()
        for i, p in enumerate(probs):
            st = to_torch_state(p[0], torch.float64)
            s64 = torch.as_tensor(obs[i]).double()
            pi, nl = head(cfg, st["actor"], s64, None if u is None else torch.as_tensor(u[i]).double(), st,
                          deterministic=not noise)
            lim = p[0]["act_limit"]
            err = float((np.abs(act[i] - pi.numpy()) / lim).max())
            print(f"MEASURED actor_forward {engine} noise={noise} rows={rows} act {err:.2e}")
            assert err < 1e-4, (rows, err)
            # where fp64 |z| > 10 the action is exactly +-act_limit
            mean, raw = actor_out64(cfg, p[0], obs[i])
            z = (mean if u is None else mean + torch.exp(torch.clamp(raw, -5.0, 2.0)) * torch.as_tensor(u[i]).double()).numpy()
            sat = np.abs(z) > SAT_Z
            assert (sat.any() or rows == 1) and np.array_equal(act[i][sat], (np.sign(z) * lim)[sat].astype(np.float32))
            if noise:
                nerr = _row_err(nlp[i].cpu().numpy()[:, None], nl.numpy()[:, None])
                print(f"MEASURED actor_forward {engine} rows={rows} nlp {nerr:.2e}")
                assert nerr < 1e-4, (rows, nerr)
    pop.close()


@pytest.mark.parametrize("engine", ACT_ENGINES)
def test_critic_forward_target_scaled(engine):
    cfg, B, E, kw = UPDATE_ENGINES[engine]
    pop, probs, cfg = build_edge(cfg, "head", NA, B, E, N, seed=SEED, **kw)
    rows = B + 1
    rng = np.random.default_rng(7)
    obs = np.stack([p[1]["s"][rng.integers(0, N, rows)] for p in probs])
    act = np.stack([rng.uniform(-1, 1, (rows, cfg.A)).astype(np.float32) * p[0]["act_limit"] for p in probs])
    q = pop.critic_forward(obs, act, target=True, scale_ret=True).cpu().numpy()
    for i, p in enumerate(probs):
        assert p[0]["ret_std"] != 1
        st = to_torch_state(p[0], torch.float64)
        s64, a64 = torch.as_tensor(obs[i]).double(), torch.as_tensor(act[i]).double()
        for k, net in enumerate(("t1", "t2")):
            err = _row_err(q[i, k][:, None], q_value(cfg, st[net], s64, a64, st).numpy()[:, None])
            print(f"MEASURED critic_forward {engine} {net} {err:.2e}")
            assert err < 1e-4, err
    pop.close()


MODEL_EVAL = {     # name -> (engine, num_models, E, rows)
    "fp32_one_model": ("fp32_S11_A6", 1, 8, 19),
    "fp32_two_models": ("fp32_S11_A6", 2, 8, 19),
    "tc_bench_models_2E+3": ("tc_fused_ant", 2, 20, 43),
    "tc_one_model_2E+3": ("tc_fused_ant", 1, 20, 43),
    "tc_E160_rows400": ("tc_fused_ant", 2, 160, 400),
}


@pytest.mark.parametrize("name", list(MODEL_EVAL))
def test_model_eval_chunks_and_clip(name):
    """model_eval chunks by E: every row of every chunk against model_sample, with the delta clip straddled."""
    engine, nm, E, rows = MODEL_EVAL[name]
    cfg, B, _, kw = UPDATE_ENGINES[engine]
    cfg = replace(cfg, num_models=nm)
    _, probs = edge_problems(cfg, "head", NA, B, E, N, seed=SEED)     # constant observation columns included
    rng = np.random.default_rng(11)
    obs = np.stack([p[1]["s"][rng.integers(0, N, rows)] for p in probs])
    act = rng.uniform(-1, 1, (NA, rows, cfg.A)).astype(np.float32)
    deltas = []
    for i, p in enumerate(probs):
        st = to_torch_state(p[0], torch.float64)
        s64, a64 = torch.as_tensor(obs[i]).double(), torch.as_tensor(act[i]).double()
        sa = torch.cat([normalize(s64, st["m_s_mean"], st["m_s_std"]), normalize(a64, st["m_a_mean"], st["m_a_std"])], -1)
        for k in range(nm):
            deltas.append(mlp(st["m%d" % (k + 1)], sa, cfg.model_acts)[:, :cfg.S].numpy())
    cfg = replace(cfg, delta_clip_pred=straddle_clip(np.concatenate([d.ravel() for d in deltas])))
    pop = populate(cfg, probs, B, E, N, **kw)
    out = pop.model_eval(obs, act).cpu().numpy()
    for i, p in enumerate(probs):
        st = to_torch_state(p[0], torch.float64)
        s64, a64 = torch.as_tensor(obs[i]).double(), torch.as_tensor(act[i]).double()
        for k in range(nm):
            ref = model_sample(cfg, st["m%d" % (k + 1)], s64, a64, st).numpy()
            err = _row_err(out[i, k] - obs[i], ref - obs[i].astype(np.float64))
            print(f"MEASURED model_eval {name} model {k} {err:.2e}")
            assert err < 1e-4, err
    pop.close()
