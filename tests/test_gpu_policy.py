"""GPU: ``saceo_policy_act`` / ``PolicySet`` - acting for sets of policies of any depth (expert policies).  Parity with
the fp64 oracle over depths, widths, activations, both heads and both std parameterisations; bit-identical results
whatever the other policies of the set are; agreement with the training engine's ``actor_forward`` at depth 2; and
``train.main`` / ``train_population`` with an MPO-format ``--expert_file``."""
import os
import pickle

import numpy as np
import pytest
import torch

from oracle.sac_eo_oracle import NetCfg
from sac_expert_b200.policy import PolicySet, PolicySpec
from tests.policy_oracle import policy_sample
from tests.test_gpu_train import COMMON
from tests.test_gpu_train_population import _assert_same, _both, _load
from tests.test_policy_host import write_mpo_expert

pytestmark = pytest.mark.gpu


def _policy(rng, S, A, hidden, per_state_std):
    dims = [S] + list(hidden) + [2 * A if per_state_std else A]
    ws = []
    for i in range(len(dims) - 1):
        ws += [(1.2 * rng.standard_normal((dims[i], dims[i + 1])) / np.sqrt(dims[i])).astype(np.float32),
               (0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32)]
    if not per_state_std:
        ws.append((-0.7 + 0.3 * rng.standard_normal((1, A))).astype(np.float32))
    norm = dict(s_mean=(0.3 * rng.standard_normal(S)).astype(np.float32), s_std=rng.uniform(0.5, 2.0, S).astype(np.float32),
                act_limit=rng.uniform(0.5, 2.5, A).astype(np.float32))
    return ws, norm


def _near_zero_relu_rows(ws, norm, obs, hidden, acts):
    """Rows whose fp64 relu pre-activation lies within fp32 rounding of zero somewhere (a flip there is allowed)."""
    h = (obs.astype(np.float64) - norm["s_mean"]) / np.maximum(norm["s_std"].astype(np.float64), 1e-8)
    near = np.zeros(len(obs), bool)
    for l in range(len(hidden)):
        W, b = ws[2 * l].astype(np.float64), ws[2 * l + 1].astype(np.float64)
        z = h @ W + b
        if acts[l] == "relu":
            near |= (np.abs(z) <= 1e-5 * (np.abs(h) @ np.abs(W) + np.abs(b))).any(1)
        h = np.tanh(z) if acts[l] == "tanh" else np.maximum(z, 0) if acts[l] == "relu" else np.where(z > 0, z, np.expm1(z))
    return near


CASES = [  # S, A, hidden, acts, squash, per_state_std, std_mult, rows, P
    (11, 3, [37], ["tanh"], False, True, 0.3, 1, 1),
    (11, 3, [256, 300], ["relu", "elu"], True, True, 1.0, 7, 3),
    (27, 8, [1024, 37, 256], ["elu", "tanh", "relu"], False, False, 0.5, 33, 3),
    (17, 6, [300, 256, 37, 1024], ["tanh", "relu", "elu", "tanh"], True, False, 1.0, 257, 1),
    (27, 8, [256, 256, 256], ["elu", "elu", "elu"], False, True, 0.3, 1, 64),
    (3, 1, [37, 1024], ["relu", "relu"], False, True, 2.0, 257, 3),
    (11, 3, [37, 37, 37, 37], ["relu", "tanh", "elu", "relu"], True, True, 1.0, 33, 64),
]


@pytest.mark.parametrize("noisy", [False, True])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_policy_act_matches_the_fp64_oracle(case, noisy):
    S, A, hidden, acts, squash, pss, std_mult, rows, P = CASES[case]
    rng = np.random.default_rng(100 + case)
    spec = PolicySpec(n_agents=P, S=S, A=A, hidden=tuple(hidden), acts=tuple(acts), squash=squash, per_state_std=pss,
                      std_mult=std_mult)
    ps = PolicySet(spec)
    pols = [_policy(rng, S, A, hidden, pss) for _ in range(P)]
    for i, (ws, norm) in enumerate(pols):
        ps.set_net(i, "actor", ws)
        ps.set_norm(i, **norm)
        assert all(np.array_equal(a, b) for a, b in zip(ps.get_net(i, "actor"), ws))
    obs = (1.5 * rng.standard_normal((P, rows, S))).astype(np.float32)
    noise = rng.standard_normal((P, rows, A)).astype(np.float32) if noisy else None
    got = ps.actor_forward(torch.from_numpy(obs), None if noise is None else torch.from_numpy(noise)).cpu().numpy()
    assert got.shape == (P, rows, A) and np.all(np.isfinite(got))
    cfg = NetCfg(S=S, A=A, actor_hidden=tuple(hidden), actor_acts=tuple(acts), per_state_std=pss, std_mult=std_mult)
    skipped = 0
    for i, (ws, norm) in enumerate(pols):
        theta = [torch.from_numpy(w.astype(np.float64)) for w in ws]
        st = {k: v.astype(np.float64) for k, v in norm.items()}
        u = None if noise is None else torch.from_numpy(noise[i].astype(np.float64))
        want = policy_sample(cfg, theta, torch.from_numpy(obs[i].astype(np.float64)), u, st, squash).numpy()
        ok = ~_near_zero_relu_rows(ws, norm, obs[i], hidden, acts)
        skipped += int((~ok).sum())
        err = np.abs(got[i][ok] - want[ok]).max(initial=0.0) / max(np.abs(want[ok]).max(initial=0.0), 1e-30)
        assert err <= 1e-5, (i, err)
    assert skipped <= max(1, P * rows // 20)


def test_policy_results_do_not_depend_on_the_set():
    """Policy i inside a set of 4 is bit-identical to the same policy acted alone; two calls give identical bytes."""
    rng = np.random.default_rng(5)
    S, A, hidden, acts = 27, 8, (256, 300, 37), ("elu", "relu", "tanh")
    pols = [_policy(rng, S, A, hidden, True) for _ in range(4)]
    obs = rng.standard_normal((4, 33, S)).astype(np.float32)
    noise = rng.standard_normal((4, 33, A)).astype(np.float32)
    for squash in (False, True):
        spec = PolicySpec(n_agents=4, S=S, A=A, hidden=hidden, acts=acts, squash=squash, std_mult=0.3)
        ps = PolicySet(spec)
        for i, (ws, norm) in enumerate(pols):
            ps.set_net(i, "actor", ws); ps.set_norm(i, **norm)
        for nz in (None, noise):
            together = ps.actor_forward(torch.from_numpy(obs), None if nz is None else torch.from_numpy(nz)).cpu()
            again = ps.actor_forward(torch.from_numpy(obs), None if nz is None else torch.from_numpy(nz)).cpu()
            assert together.numpy().tobytes() == again.numpy().tobytes()
            for i, (ws, norm) in enumerate(pols):
                one = PolicySet(PolicySpec(n_agents=1, S=S, A=A, hidden=hidden, acts=acts, squash=squash, std_mult=0.3))
                one.set_net(0, "actor", ws); one.set_norm(0, **norm)
                alone = one.actor_forward(torch.from_numpy(obs[i:i + 1]),
                                          None if nz is None else torch.from_numpy(nz[i:i + 1])).cpu()
                assert torch.equal(alone[0], together[i]), (squash, i)
    with pytest.raises(NotImplementedError):
        ps.actor_forward(torch.from_numpy(obs), want_neglogp=True)


@pytest.mark.parametrize("per_state_std", [True, False])
def test_depth_two_squashed_policy_agrees_with_the_training_engine(per_state_std):
    from sac_expert_b200 import lib
    from sac_expert_b200.population import Population, PopulationSpec
    rng = np.random.default_rng(9)
    S, A, hidden, acts, P, rows = 11, 3, (256, 256), ("relu", "tanh"), 3, 40
    pols = [_policy(rng, S, A, hidden, per_state_std) for _ in range(P)]
    pop = Population(PopulationSpec(n_agents=P, S=S, A=A, actor_hidden=hidden, actor_acts=acts, per_state_std=per_state_std,
                                    num_models=0, B=64, E=2, replay_capacity=16, gemm_mode=lib.GEMM_FP32_SIMT))
    ps = PolicySet(PolicySpec(n_agents=P, S=S, A=A, hidden=hidden, acts=acts, squash=True, per_state_std=per_state_std))
    for i, (ws, norm) in enumerate(pols):
        pop.set_net(i, "actor", ws); pop.set_norm(i, **norm)
        ps.set_net(i, "actor", ws); ps.set_norm(i, **norm)
    obs = torch.from_numpy(rng.standard_normal((P, rows, S)).astype(np.float32))
    noise = torch.from_numpy(rng.standard_normal((P, rows, A)).astype(np.float32))
    for nz in (None, noise):
        want = pop.actor_forward(obs, nz).cpu().numpy()
        got = ps.actor_forward(obs, nz).cpu().numpy()
        assert np.abs(got - want).max() <= 1e-6 * np.abs(want).max()
    pop.close()


def test_trpo_update_through_a_gaussian_actor_equals_the_squashed_class():
    """The trust-region mirror accepts the reference's own on-policy actor class: the same weights and draws give the
    same update through a depth-2 ``GaussianActor`` as through a ``SquashedGaussianActor``."""
    from sac_expert_b200.sac_eo.actors.init_actor import init_actor
    from sac_expert_b200.sac_eo.algs.model_free.trpo import TRPO
    from sac_expert_b200.sac_eo.envs.synthetic import SyntheticEnv
    rng = np.random.default_rng(1)
    N = 80
    s = rng.standard_normal((N, 7)).astype(np.float32); a = rng.standard_normal((N, 2)).astype(np.float32)
    adv = rng.standard_normal(N).astype(np.float32)
    kw = dict(adv_center=True, adv_scale=True, delta_trpo=0.02, cg_it=5, trust_sub=1, trust_damp=0.01, kl_maxfactor=1.5,
              ent_reg=True, ent_targ=0.0, alpha_lr=0.01)
    out = []
    for squash in (True, False):
        np.random.seed(0)
        actor = init_actor(SyntheticEnv(7, 2), [32, 32], ["tanh"], 0.01, 0.7, "orthogonal", False, None,
                           actor_per_state_std=True, actor_squash=squash)
        log = TRPO(actor, kw).update((s, a, adv, None, None, None))
        out.append((actor.get_weights(), log, actor.neglogp(s, a).numpy(), actor.get_kl_info(s)))
    (w1, l1, n1, k1), (w2, l2, n2, k2) = out
    assert all(np.array_equal(x, y) for x, y in zip(w1, w2))
    assert l1 == l2 and np.array_equal(n1, n2) and np.array_equal(k1, k2)


# ---------------------------------------------------------------------------------------------- expert files
EXPERT = ["--expert_buffer_size", "120"]


def _expert_argv(tmp_path, alg_type, extra=()):
    return COMMON + ["--alg_type", alg_type, "--expert_path", str(tmp_path), "--expert_file", "expert.pkl"] + EXPERT + \
        list(extra)


def _host_rollout_J(tmp_path, argv):
    """expert_J_tot of ``_collect_expert_data`` recomputed on the host: the expert of the file through
    ``tests/policy_oracle.policy_sample`` in fp64, in the synthetic environment seeded like ``env_expert``."""
    from sac_expert_b200.sac_eo import train as T
    from sac_expert_b200.sac_eo.common.normalizer import RunningNormalizers
    from sac_expert_b200.sac_eo.common.train_utils import organize_rms_inputs
    from sac_expert_b200.sac_eo.envs import init_env
    args = T.create_train_parser().parse_args(argv + ["--save_path", str(tmp_path / "unused")])
    setup = T.build_inputs(args)[0]["setup_kwargs"]
    with open(tmp_path / "expert.pkl", "rb") as f:
        log = pickle.load(f)[0]
    kw, ws = log["param"]["actor_kwargs"], log["final"]["actor_weights"]
    env = init_env("synthetic", "hopper", "60")
    env.seed(setup["expert_seed"])
    s_rms = RunningNormalizers(11, 3, 0.995, organize_rms_inputs(log["final"])).s_rms
    hidden = tuple(kw["actor_layers"])
    acts = tuple(kw["actor_activations"]) * (len(hidden) if len(kw["actor_activations"]) == 1 else 1)
    cfg = NetCfg(S=11, A=3, actor_hidden=hidden, actor_acts=acts, per_state_std=bool(kw["actor_per_state_std"]),
                 std_mult=float(kw["actor_std_mult"]))
    theta = [torch.from_numpy(np.asarray(w, np.float64)) for w in ws]
    st = {"s_mean": np.asarray(s_rms.mean, np.float64), "s_std": np.asarray(s_rms.std, np.float64),
          "act_limit": np.ones(3)}
    J = []
    for _ in range(2):
        s, tot = env.reset(), 0.0
        for t in range(60):
            a = policy_sample(cfg, theta, torch.from_numpy(np.asarray(s, np.float64))[None], None, st,
                              bool(kw.get("actor_squash"))).numpy()[0].astype(np.float32)
            s, r, d, _ = env.step(np.clip(a, -1.0, 1.0))
            tot += r
        J.append(tot)
    return float(np.mean(J))


@pytest.mark.parametrize("alg_type", ["sac_imit", "bc"])
def test_train_main_rolls_out_an_mpo_expert_file(tmp_path, alg_type):
    from sac_expert_b200.sac_eo import train as T
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(256, 256, 256), act="elu", std_mult=0.3, seed=4)
    extra = ["--scale_epsilon_by_true_MSE"] if alg_type == "sac_imit" else []
    argv = _expert_argv(tmp_path, alg_type, extra)
    logs = _load(T.main(argv + ["--save_path", str(tmp_path / "out")]))
    tr = logs[0]["train"]
    got = float(np.ravel(tr["expert_J_tot"])[0])
    want = _host_rollout_J(tmp_path, argv)
    assert abs(got - want) <= 1e-4 * abs(want), (got, want)
    assert int(np.ravel(tr["expert_steps"])[0]) == 120
    key = "p_loss" if alg_type == "sac_imit" else "BC_MSE_loss"
    assert len(tr[key]) == 200 and np.all(np.isfinite(tr[key]))


def test_deep_squashed_expert_and_a_train_main_pickle_as_expert(tmp_path):
    from sac_expert_b200.sac_eo import train as T
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(64, 64, 64), act="relu", squash=True, seed=8)
    argv = _expert_argv(tmp_path, "sac_imit")
    first = T.main(argv + ["--save_path", str(tmp_path / "a")])
    tr = _load(first)[0]["train"]
    want = _host_rollout_J(tmp_path, argv)
    assert abs(float(np.ravel(tr["expert_J_tot"])[0]) - want) <= 1e-4 * abs(want)
    # the checkpoint pickle of that run is itself an expert file (a two-hidden-layer SquashedGaussianActor)
    second = T.main(COMMON + ["--alg_type", "bc", "--expert_path", os.path.dirname(first), "--expert_file",
                              os.path.basename(first), "--save_path", str(tmp_path / "b")] + EXPERT)
    tr2 = _load(second)[0]["train"]
    assert np.all(np.isfinite(tr2["BC_MSE_loss"])) and np.isfinite(float(np.ravel(tr2["expert_J_tot"])[0]))


def test_population_mode_with_an_expert_file_equals_train_main(tmp_path):
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(256, 256, 256), act="elu", std_mult=0.3, seed=4)
    got, want = _both(tmp_path, _expert_argv(tmp_path, "sac_imit", ["--scale_epsilon_by_true_MSE", "--runs", "3"]))
    assert len(got) == len(want) == 3
    for r in range(3):
        _assert_same(got[r], want[r], f"run {r}")
