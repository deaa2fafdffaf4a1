"""CPU: the edge fixtures of tests/test_gpu_edges.py really hit their branch edges in the fp64 oracle - clamped
log-stds on the intended dimensions, saturated squash, twin-critic ties, a straddled delta clip with a margin, the
temperature floor, terminal rows and constant observation columns.  A fixture that stops hitting its edge fails here,
instead of quietly passing on the GPU."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from oracle.sac_eo_oracle import q_forward, to_torch_state
from tests.helpers import (CONST_COLS, SAT_Z, TERM_IMPLS, UPDATE_ENGINES, actor_out64, actor_phase_z, alpha_unclamped,
                           edge_problems, expert_deltas, expert_term64, log_std_edges, oracle_update)

N = 600


def _problems(engine, edge, per_state_std=True):
    cfg, B, E, _ = UPDATE_ENGINES[engine]
    return edge_problems(replace(cfg, per_state_std=per_state_std), edge, 2, B, E, N, seed=5)


def _ls_slices(cfg, g):
    """(W2 log-std columns [h2, A], log-std bias or variable [A]) of a flat or listed actor gradient."""
    if cfg.per_state_std:
        return g[4][:, cfg.A:], g[5][cfg.A:]
    return None, g[6][0]


@pytest.mark.parametrize("per_state_std", [True, False])
@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_head_fixture_hits_clamp_saturation_done_and_constant_columns(engine, per_state_std):
    cfg, probs = _problems(engine, "head", per_state_std)
    A, B = cfg.A, probs[0][4]["s"].shape[0]
    ls = log_std_edges(A).astype(np.float64)
    outside, boundary = (ls < -5) | (ls > 2), (ls == -5) | (ls == 2)
    assert outside.sum() >= 2 and boundary.sum() >= 2 and (~outside & ~boundary).any()
    for p in probs:
        st, batch = p[0], p[4]
        # every row's raw log-std is exactly the edge value
        _, raw = actor_out64(cfg, st, batch["s"])
        assert np.array_equal(raw.numpy(), np.broadcast_to(ls, raw.shape))
        # the clamp gradient: exactly 0 outside [-5, 2], non-zero on the closed interval's boundaries
        o = oracle_update(cfg, p, torch.float64)
        gw, gb = _ls_slices(cfg, [g.numpy() for g in o["g_actor"]])
        assert (gb[outside] == 0).all() and (gb[boundary] != 0).all()
        if gw is not None:
            assert (gw[:, outside] == 0).all() and (np.abs(gw[:, boundary]).max(0) > 0).all()
        # saturated squash: >= 20 % of the rows of every log-std-2 dimension, minibatch and expert rows alike
        z = actor_phase_z(cfg, p)
        sat = np.clip(ls, -5, 2) == 2
        frac = (np.abs(z[:, sat]) > SAT_Z).mean(0)
        assert (frac >= 0.2).all(), frac
        assert (np.abs(z[B:, sat]) > SAT_Z).any()
        assert not np.allclose(st["act_limit"], st["act_limit"][0])
        # terminal rows and constant observation columns
        assert 0.3 < batch["d"].mean() < 0.7
        for c in CONST_COLS:
            assert st["s_std"][c] == 0
            for key in ("s", "sp", "sE", "spE"):
                assert (batch[key][:, c] == st["s_mean"][c]).all()
        y = o["y"].numpy()
        done = batch["d"] == 1
        assert np.array_equal(y[done], batch["r"][done].astype(np.float64))


@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_ties_fixture_ties_every_min(engine):
    cfg, probs = _problems(engine, "ties")
    for p in probs:
        o = oracle_update(cfg, p, torch.float64)
        new = o["new"]
        for a, b in (("q1", "q2"), ("t1", "t2")):
            assert all(torch.equal(x, y) for x, y in zip(new[a], new[b]))
        st = to_torch_state(p[0], torch.float64)
        s = torch.as_tensor(p[4]["s"]).double()
        qa = q_forward(cfg, new["q1"], s, o["a2"], st)
        qb = q_forward(cfg, new["q2"], s, o["a2"], st)
        assert torch.equal(qa, qb)                     # every reduce_min of the actor loss is a tie
        assert torch.equal(o["L_q1"], o["L_q2"])


@pytest.mark.parametrize("engine", list(UPDATE_ENGINES))
def test_alpha_floor_fixture_steps_below_the_floor(engine):
    cfg, probs = _problems(engine, "alpha_floor")
    for p in probs:
        o = oracle_update(cfg, p, torch.float64)
        assert float(o["g_alpha"]) > 0
        assert alpha_unclamped(cfg, p) < 1e-5
        o32 = oracle_update(cfg, p)
        assert float(o32["new"]["alpha"]) == float(np.float32(1e-5))


@pytest.mark.parametrize("impl", list(TERM_IMPLS))
def test_delta_clip_fixture_straddles_the_clip_with_a_margin(impl):
    cfg, B, E = TERM_IMPLS[impl]
    cfg, probs = edge_problems(cfg, "delta_clip", 2, B, E, N, seed=5)
    c = cfg.delta_clip_pred
    assert c > 0 and c == float(np.float32(c))
    for p in probs:
        d = np.abs(np.concatenate([x.ravel() for x in expert_deltas(cfg, p)]))
        assert (d > c).mean() > 0.2 and (d < c).mean() > 0.2
        assert (np.abs(d - c) > 1e-4 * c).all()


@pytest.mark.parametrize("edge", ["eps0", "eps1"])
@pytest.mark.parametrize("impl", list(TERM_IMPLS))
def test_eps_fixtures(impl, edge):
    cfg, B, E = TERM_IMPLS[impl]
    cfg, probs = edge_problems(cfg, edge, 2, B, E, N, seed=5)
    for p in probs:
        md, mse = expert_term64(cfg, p)
        o = oracle_update(cfg, p, torch.float64)
        if edge == "eps0":
            assert p[3]["eps"] == 0 and not md.any() and mse > 0
            assert float(o["p_loss"]) == float(o["L_pi"])
        else:
            assert p[3]["eps"] == 1 and np.abs(md).max() > 0
            assert float(o["p_loss"]) == float(o["mse"])
