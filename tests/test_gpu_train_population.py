"""GPU: ``train_population`` - all runs of one ``train.py`` invocation as one device population - computes, run for
run and bit for bit, what ``train.main`` computes one run after the other; the population calls it batches keep the
agents independent; runs that fall out of step raise ``LockstepError``."""
import os
import pickle

import numpy as np
import pytest
import torch

from tests.test_gpu_train import COMMON

pytestmark = pytest.mark.gpu


def _load(path):
    with open(path, "rb") as f:
        return pickle.load(f)


def _assert_same(got, want, where):
    """Bit-identical nested logs; wall-clock fields (``time_*``) and the output directory excepted."""
    if isinstance(want, dict):
        keep = lambda d: {k for k in d if not str(k).startswith("time_") and k != "save_path"}
        assert keep(got) == keep(want), where
        for k in keep(want):
            _assert_same(got[k], want[k], f"{where}/{k}")
    elif isinstance(want, (list, tuple)) and not np.isscalar(want):
        assert len(got) == len(want), where
        for i, (g, w) in enumerate(zip(got, want)):
            _assert_same(g, w, f"{where}[{i}]")
    else:
        g, w = np.asarray(got), np.asarray(want)
        assert g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes(), where


def _both(tmp_path, argv):
    from sac_expert_b200.sac_eo import train as T
    from sac_expert_b200.sac_eo import train_population as TP
    pop_dir, seq_dir = tmp_path / "population", tmp_path / "sequential"
    got = _load(TP.main(argv + ["--save_path", str(pop_dir)]))
    want = _load(T.main(argv + ["--save_path", str(seq_dir)]))
    assert os.listdir(pop_dir) and not [f for f in os.listdir(pop_dir) if f.startswith("TEMPLOG")]
    return got, want


@pytest.mark.parametrize("alg_type,extra", [("sac_imit", ["--scale_epsilon_by_true_MSE"]), ("sac", []), ("bc", [])])
def test_population_runs_equal_sequential_runs_bitwise(tmp_path, alg_type, extra):
    got, want = _both(tmp_path, COMMON + ["--alg_type", alg_type, "--runs", "3"] + extra)
    assert len(got) == len(want) == 3
    for r in range(3):
        assert set(got[r]) == {"param", "train", "final"}
        _assert_same(got[r], want[r], f"run {r}")
    assert not np.array_equal(got[0]["final"]["actor_weights"][0], got[1]["final"]["actor_weights"][0])


def test_one_run_population_equals_train_main(tmp_path):
    got, want = _both(tmp_path, COMMON + ["--alg_type", "sac_imit", "--runs", "1", "--scale_epsilon_by_true_MSE"])
    assert len(got) == len(want) == 1
    _assert_same(got[0], want[0], "run 0")


def test_population_calls_keep_agents_independent():
    """Four agents with different weights, replay rows and injected draws: two updates, a three-step model fit and one
    stochastic actor forward of the four-agent population equal, bit for bit, those of a one-agent population given
    agent r's inputs - nothing the batched calls compute for one agent depends on the population size."""
    from oracle.sac_eo_oracle import NetCfg, make_problem, draw_batch
    from sac_expert_b200 import lib
    from sac_expert_b200.population import Population
    from tests.helpers import inject, spec_from_cfg
    cfg = NetCfg(S=11, A=3)
    R, B, E, N, mb = 4, 256, 20, 3000, 50
    probs = []
    for i in range(R):
        st, replay, expert, hyper = make_problem(cfg, B, E, N, seed=5 + 17 * i, perturb=0.05)
        hyper.update(eps=0.3, gamma=0.995 - 0.01 * i)
        probs.append((st, replay, expert, hyper, draw_batch(cfg, replay, expert, B, seed=900 + i)))
    rng = np.random.default_rng(0)
    fit_idx = rng.integers(0, N, (3, R, 2, mb))
    obs = rng.standard_normal((R, 7, cfg.S)).astype(np.float32)
    noise = rng.standard_normal((R, 7, cfg.A)).astype(np.float32)

    def run(agents):
        pop = Population(spec_from_cfg(cfg, len(agents), B, E, N, gemm_mode=lib.GEMM_TCGEN05_BF16X3, use_graph=True))
        for j, i in enumerate(agents):
            st, replay, expert, hyper, _ = probs[i]
            pop.load_agent(j, st, hyper)
            pop.append_rows(j, replay["s"], replay["a"], replay["r"], replay["sp"], replay["d"])
            pop.set_expert(j, expert["sE"], expert["spE"])
        out = {}
        for step in range(2):
            inject(pop, cfg, [probs[i] for i in agents])
            out["losses%d" % step] = pop.update(1, num_timesteps=step, use_device_rng=False).clone()
        pop.fit_bind(mb)
        out["fit"] = pop.model_fit(fit_idx[:, agents])
        out["act"] = pop.actor_forward(torch.from_numpy(obs[agents]), torch.from_numpy(noise[agents]))
        for k in ("actor", "actor_m", "actor_v", "q", "q_m", "q_v", "qt", "alpha", "alpha_m", "alpha_v", "adam_t",
                  "model", "model_m", "model_v"):
            out[k] = pop.t[k]
        out = {k: v.cpu() for k, v in out.items()}
        out["fit"] = out["fit"].transpose(0, 1)                  # agent-major like the others
        pop.close()
        return out

    together = run(list(range(R)))
    for i in range(R):
        alone = run([i])
        for k, v in alone.items():
            assert torch.equal(together[k][i], v[0]), (i, k)
    assert not torch.equal(together["actor"][0], together["actor"][1])


def test_runs_out_of_step_raise_lockstep_error(tmp_path, monkeypatch):
    """Run 1's environment ends its episodes early: its trajectory, hence its replay append, is shorter than run 0's."""
    from sac_expert_b200.sac_eo import train_population as TP
    from sac_expert_b200.sac_eo.common.lockstep import LockstepError
    build = TP.build_run

    def build_run(inp, population=None, agent=0):
        alg = build(inp, population, agent)
        if agent == 1:
            alg.env._h = 25
        return alg
    monkeypatch.setattr(TP, "build_run", build_run)
    with pytest.raises(LockstepError, match=r"run 1 .*run 0|run 0 .*run 1"):
        TP.main(COMMON + ["--alg_type", "sac", "--runs", "2", "--save_path", str(tmp_path)])
