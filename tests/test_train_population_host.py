"""CPU: the lockstep scheduler of ``train_population`` driving the real training loop (``SAC.train_steps`` and the
``SAC_exp`` hooks) against a fake device population that records its calls.  Checks, without a GPU, that every run
consumes its NumPy stream exactly as the one-run schedule does and that one round of R runs costs one batched call."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from sac_expert_b200.sac_eo import train as T
from sac_expert_b200.sac_eo import train_population as TP
from sac_expert_b200.sac_eo.common import lockstep

ARGS = ["--env_type", "synthetic", "--env_name", "hopper", "--task_name", "12", "--actor_squash", "--actor_layers", "8", "8",
        "--critic_layers", "8", "8", "--model_layers", "8", "8", "--env_horizon", "12", "--env_batch_size_init", "20",
        "--total_timesteps", "45", "--model_num_epochs", "2", "--model_batch_size", "5", "--eval_freq", "30",
        "--eval_num_traj", "1", "--sac_batch_size", "8", "--expert_buffer_size", "6", "--seed", "5", "--runs", "3"]


class FakePop:
    """Stands in for ``Population``: outputs are cheap functions of the inputs and of per-agent state that every update
    and fit changes, so a run's logs depend on every draw it made.  ``calls`` records (entry point, agents)."""

    def __init__(self, spec):
        self.spec, n = spec, spec.n_agents
        self.t = {"alpha": torch.zeros(n), "model_logstd": torch.zeros(n, 2, spec.S)}
        self.model_batch, self.calls, self.nets = None, [], {}
        self.bias = np.zeros((n, spec.A), np.float32)

    def _log(self, name, n):
        self.calls.append((name, n))

    def set_net(self, agent, name, ws):
        self.nets[agent, name] = [np.array(w, np.float32) for w in ws]

    def get_net(self, agent, name):
        return self.nets[agent, name]

    def set_norm(self, agent, **kw):
        pass

    def set_hyper(self, agent, **kw):
        self._log("set_hyper", 1)

    def set_fit_hyper(self, agent, **kw):
        pass

    def fit_bind(self, model_batch, **kw):
        self._log("fit_bind", self.spec.n_agents)
        self.model_batch = model_batch

    def set_expert(self, agent, sE, spE):
        self._log("set_expert", 1)

    def set_expert_all(self, sE, spE):
        self._log("set_expert_all", len(sE))

    def append_rows(self, agent, s, a, r, sp, d):
        self._log("append_rows", 1)
        self.bias[agent] += 1e-3 * np.asarray(r, np.float32).mean()

    def append_all(self, s, a, r, sp, d):
        self._log("append_all", len(s))
        self.bias += 1e-3 * np.asarray(r, np.float32).mean(1)[:, None]

    def actor_forward(self, obs, noise=None):
        self._log("actor_forward", obs.shape[0])
        x = obs[..., :self.spec.A] + torch.from_numpy(self.bias)[:, None]
        return torch.tanh(x if noise is None else x + 0.1 * noise)

    def model_eval(self, obs, act):
        self._log("model_eval", obs.shape[0])
        out = obs.clone()
        out[..., :self.spec.A] += act + torch.from_numpy(self.bias)[:, None]
        return torch.stack([out, 2 * out], 1)

    def set_draws(self, idx=None, noise=None, perm=None):
        self._draws = (idx, noise)

    def update(self, n_steps, num_timesteps=0, use_device_rng=True):
        self._log("update", self.spec.n_agents)
        idx, noise = self._draws
        self.bias += 1e-2 * np.asarray(noise, np.float32).mean(1) + 1e-4 * np.asarray(idx).mean(1, keepdims=True)
        return torch.from_numpy(np.repeat(self.bias[:, :1], 8, 1))

    def bc_update(self, n_steps, use_device_rng=True):
        self._log("bc_update", self.spec.n_agents)
        self.bias += 1e-2 * np.asarray(self._draws[1], np.float32).mean(1)
        return torch.from_numpy(np.repeat(self.bias[:, :1], 8, 1))

    def model_fit(self, idx):
        self._log("model_fit", idx.shape[1])
        self.bias += 1e-4 * np.asarray(idx, np.float32).mean((0, 2, 3))[:, None]
        return torch.zeros(idx.shape[0], idx.shape[1], idx.shape[2])


class FakeShared:
    made = []

    def __init__(self, n):
        self.n, self.pop = n, None

    def get(self, spec):
        if self.pop is None:
            self.pop = FakePop(replace(spec, n_agents=self.n))
            FakeShared.made.append(self.pop)
        return self.pop


def _record(alg, params):
    """``_dump_and_save`` without files: keeps each checkpoint's train log (wall-clock fields dropped)."""
    train = {k: v for k, v in alg.logger.dump()["train"].items() if not k.startswith("time_")}
    alg.dumps = getattr(alg, "dumps", []) + [train]
    alg.logger.reset()


@pytest.mark.parametrize("alg_type,extra", [("sac_imit", ["--scale_epsilon_by_true_MSE", "--update_normalizers"]),
                                            ("sac", []), ("bc", [])])
def test_lockstep_consumes_each_runs_stream_like_a_one_run_schedule(tmp_path, monkeypatch, alg_type, extra):
    from sac_expert_b200.sac_eo.algs.SAC import SAC
    args = T.create_train_parser().parse_args(ARGS + ["--alg_type", alg_type, "--save_path", str(tmp_path)] + extra)
    monkeypatch.setattr(SAC, "_dump_and_save", _record)

    seq = []                                               # the one-run schedule, one run after the other
    for inp in T.build_inputs(args):
        alg = T.build_run(inp, FakeShared(1), 0)
        if alg_type != "sac":
            alg._bind_expert(FakeShared(1), 0)
        alg.train(inp["alg_kwargs"]["total_timesteps"], inp)
        seq.append((alg.dumps, np.random.get_state()))

    algs, streams, made = [], [], len(FakeShared.made)

    def build_run(inp, population=None, agent=0):
        algs.append(T.build_run(inp, population, agent))
        return algs[-1]

    def run_lockstep(runs, names, st, timings=None):
        streams.extend(st)
        return lockstep.run_lockstep(runs, names, st, timings)
    monkeypatch.setattr(TP, "SharedPopulation", FakeShared)
    monkeypatch.setattr(TP, "build_run", build_run)
    monkeypatch.setattr(TP, "run_lockstep", run_lockstep)
    TP.train_population(T.build_inputs(args))
    assert len(algs) == 3
    for r, alg in enumerate(algs):
        dumps, state = seq[r]
        assert len(alg.dumps) == len(dumps)
        for got, want in zip(alg.dumps, dumps):
            assert sorted(got) == sorted(want)
            for k in want:
                assert np.array_equal(got[k], want[k]), (r, k)
        have = streams[r].get_state()
        assert np.array_equal(have[1], state[1]) and have[2:] == state[2:], f"run {r}: stream consumed differently"
    pop = FakeShared.made[made]
    assert pop.spec.n_agents == 3 and {n for _, n in pop.calls} <= {1, 3}
    assert not [c for c in pop.calls if c[0] in ("append_rows", "set_expert")]
    assert [c for c in pop.calls if c[0] == "fit_bind"] == ([] if alg_type == "sac" else [("fit_bind", 3)])


def test_one_round_is_one_batched_call_per_request_kind(monkeypatch):
    """One step of R runs (act, update, replay append) issues one population call of each kind."""
    spec = type("Spec", (), {"n_agents": 4, "A": 2, "S": 3, "E": 2, "B": 5})()
    pop = FakePop(spec)
    from sac_expert_b200.sac_eo.common.lockstep import Request

    def step(r):
        rand = lockstep.np_random()
        obs = rand.normal(size=(1, 3)).astype(np.float32)
        act = yield Request("act", pop, r, (1, False), obs=obs, noise=rand.normal(size=(1, 2)).astype(np.float32))
        idx, noise = rand.randint(10, size=5), rand.normal(size=(15, 2)).astype(np.float32)
        losses = yield Request("update", pop, r, ("update", 3, (5,), (15, 2), None), bc=False, num_timesteps=3, idx=idx,
                               noise=noise, perm=None, expert=(obs, obs), eps=None)
        yield Request("append", pop, r, (1,), rows=(obs, act, np.ones(1), obs, np.zeros(1)))
        return float(losses[0])

    streams = [np.random.RandomState(r) for r in range(4)]
    out = lockstep.run_lockstep([step(r) for r in range(4)], list(range(4)), streams)
    assert len(out) == 4
    assert pop.calls == [("actor_forward", 4), ("set_expert_all", 4), ("update", 4), ("append_all", 4)]


def test_runs_out_of_step_raise_a_lockstep_error():
    spec = type("Spec", (), {"n_agents": 2, "A": 2, "S": 3})()
    pop = FakePop(spec)
    from sac_expert_b200.sac_eo.common.lockstep import LockstepError, Request

    def run(r, rows):
        yield Request("act", pop, r, (rows, True), obs=np.zeros((rows, 3), np.float32), noise=None)

    with pytest.raises(LockstepError, match=r"run 11 requested act\(2, True\).*run 10 requested act\(1, True\)"):
        lockstep.run_lockstep([run(0, 1), run(1, 2)], [10, 11], [np.random.RandomState(0)] * 2)
