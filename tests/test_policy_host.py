"""CPU: expert policies of any depth.  The layout arithmetic of ``saceo_policy_layout`` and its validation, the
``GaussianActor`` / ``init_actor`` / ``create_nn_weights`` generalisation, the depth limit at the training engine's
entry points, an MPO-format expert file loaded through ``train.build_run`` (it must reach the device layer as a
``PolicySpec``), and the any-depth policy oracle (``tests/policy_oracle.py``) against ``oracle.head`` /
``oracle.gaussian_sample`` at depth 2 and against a NumPy restatement at depth 3."""
import ctypes as C
import math
import os
import pickle

import numpy as np
import pytest
import torch

import __graft_entry__ as G
from sac_expert_b200 import lib as L
from sac_expert_b200.policy import PolicySpec, policy_layout
from sac_expert_b200.population import PopulationSpec
from sac_expert_b200.sac_eo import train as T
from sac_expert_b200.sac_eo.actors.continuous_actors import GaussianActor, SquashedGaussianActor
from sac_expert_b200.sac_eo.actors.init_actor import init_actor
from sac_expert_b200.sac_eo.common.nn_utils import _orthogonal, create_nn_weights
from sac_expert_b200.sac_eo.envs.synthetic import SyntheticEnv
from tests.test_train_population_host import ARGS, FakeShared


@pytest.fixture(scope="module")
def lib():
    G.build()
    return L.load()


def write_mpo_expert(path, S, A, hidden=(256, 256, 256), act="elu", std_mult=0.3, per_state_std=True, seed=0,
                     squash=None):
    """An expert pickle in the format of the reference's MPO logs (SURVEY.md §4): a list of one ``{param, final}``
    dict, ``param.actor_kwargs`` without ``actor_squash`` (a ``GaussianActor``) and the normaliser statistics in the
    old ``s_t / s_mean / s_var`` form.  ``squash=True`` writes a ``SquashedGaussianActor`` expert instead."""
    rng = np.random.default_rng(seed)
    dims = [S] + list(hidden) + [2 * A if per_state_std else A]
    ws = []
    for i in range(len(dims) - 1):
        ws += [(rng.standard_normal((dims[i], dims[i + 1])) / math.sqrt(dims[i])).astype(np.float32),
               (0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32)]
    if not per_state_std:
        ws.append((-0.5 + 0.2 * rng.standard_normal((1, A))).astype(np.float32))
    kw = dict(actor_layers=list(hidden), actor_activations=[act], actor_gain=0.01, actor_std_mult=std_mult,
              actor_init_type="orthogonal", actor_layer_norm=False, actor_per_state_std=per_state_std,
              actor_adversary_prob=0.0)
    if squash is not None:
        kw["actor_squash"] = squash
    final = {"actor_weights": ws}
    for p, d in (("s", S), ("a", A), ("delta", S)):
        final[p + "_t"] = 500
        final[p + "_mean"] = (0.5 * rng.standard_normal(d)).astype(np.float32)
        final[p + "_var"] = rng.uniform(0.3, 3.0, d).astype(np.float32)
    for p in ("r", "ret"):
        final[p + "_t"], final[p + "_mean"], final[p + "_var"] = 500, 0.5, 2.0
    with open(path, "wb") as f:
        pickle.dump([{"param": {"actor_kwargs": kw}, "final": final}], f)
    return ws, final


def _cfg(S, A, hidden, acts=None, per_state_std=True, squash=False, n=1):
    return PolicySpec(n_agents=n, S=S, A=A, hidden=tuple(hidden), acts=tuple(acts or ["relu"] * len(hidden)),
                      squash=squash, per_state_std=per_state_std).to_config()


def _count(S, A, hidden, per_state_std):
    dims = [S] + list(hidden) + [2 * A if per_state_std else A]
    return sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1)) + (0 if per_state_std else A)


# ---------------------------------------------------------------------------------------------- layout arithmetic
def test_layout_of_the_shipped_expert(lib):
    n, s, ns = policy_layout(PolicySpec(n_agents=1, S=3, A=1, hidden=(256, 256, 256), acts=("elu",) * 3))
    assert (n, s) == (133_122, 133_152) and ns % 4 == 0 and ns >= 2 * 3 + 1
    assert policy_layout(PolicySpec(n_agents=64, S=27, A=8, hidden=(256,) * 3, acts=("elu",) * 3))[0] == 142_864


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
@pytest.mark.parametrize("per_state_std", [True, False])
def test_layout_counts_every_depth(lib, depth, per_state_std):
    hidden = [37, 300, 5, 1024][:depth]
    n, s, ns = policy_layout(PolicySpec(n_agents=3, S=11, A=3, hidden=tuple(hidden), acts=("tanh",) * depth,
                                        per_state_std=per_state_std))
    assert n == _count(11, 3, hidden, per_state_std)
    assert s % 32 == 0 and n <= s < n + 32
    assert ns == 28                              # s_mean | s_std | act_limit = 25 floats, padded to 4


@pytest.mark.parametrize("edit,msg", [
    (dict(n_hidden=0), b"n_hidden"), (dict(n_hidden=9), b"n_hidden"), (dict(width=0), b"width"),
    (dict(width=1025), b"width"), (dict(act=3), b"activations"), (dict(S=0), b"S and A"), (dict(A=0), b"S and A"),
    (dict(n_policies=0), b"n_policies")])
def test_invalid_configurations_are_refused(lib, edit, msg):
    cfg = _cfg(4, 2, [16, 16])
    if "width" in edit:
        cfg.hidden[1] = edit["width"]
    elif "act" in edit:
        cfg.act[0] = edit["act"]
    else:
        for k, v in edit.items():
            setattr(cfg, k, v)
    n, s, ns = C.c_int64(), C.c_int64(), C.c_int32()
    assert lib.saceo_policy_layout(C.byref(cfg), C.byref(n), C.byref(s), C.byref(ns)) == -1
    assert msg in lib.saceo_last_error()
    dummy = C.c_void_p(16)
    assert lib.saceo_policy_act(C.byref(cfg), dummy, dummy, dummy, 1, None, dummy, None) == -1
    good = _cfg(4, 2, [16, 16])
    assert lib.saceo_policy_act(C.byref(good), dummy, dummy, dummy, 0, None, dummy, None) == -1     # rows < 1


def test_act_refuses_without_device(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = _cfg(4, 2, [16, 16, 16])
    dummy = C.c_void_p(16)
    assert lib.saceo_policy_act(C.byref(cfg), dummy, dummy, dummy, 1, None, dummy, None) == -3
    assert b"no CPU fallback" in lib.saceo_last_error()


def test_policy_spec_validates_on_the_host():
    with pytest.raises(ValueError):
        PolicySpec(n_agents=1, S=3, A=1, hidden=(8,) * 9, acts=("relu",) * 9).to_config()
    with pytest.raises(ValueError):
        PolicySpec(n_agents=1, S=3, A=1, hidden=(8, 8), acts=("relu", "gelu")).to_config()
    spec = PolicySpec(n_agents=1, S=3, A=2, hidden=(8, 4), acts=("relu", "elu"), per_state_std=False)
    assert spec.shapes() == [(3, 8), (8,), (8, 4), (4,), (4, 2), (2,), (1, 2)]


# ---------------------------------------------------------------------------------------------- actor classes
@pytest.mark.parametrize("layers", [[32], [32, 16, 8], [8, 8, 8, 8]])
@pytest.mark.parametrize("per_state_std", [True, False])
def test_init_actor_builds_a_gaussian_actor_of_any_depth(layers, per_state_std):
    env = SyntheticEnv(5, 2)
    a = init_actor(env, layers, ["elu"], 0.01, 0.3, "orthogonal", False, None, per_state_std, False)
    assert type(a) is GaussianActor and a.layers == tuple(layers) and a.activations == ("elu",) * len(layers)
    dims = [5] + layers + [4 if per_state_std else 2]
    want = []
    for i in range(len(dims) - 1):
        want += [(dims[i], dims[i + 1]), (dims[i + 1],)]
    want += [] if per_state_std else [(1, 2)]
    assert [w.shape for w in a.get_weights()] == want
    assert len(a.trainable) == len(want) and a.d == sum(int(np.prod(s)) for s in want)
    a.set_weights(a.get_weights(flat=True), from_flat=True)
    with pytest.raises(L.SaceoError):
        a.sample(np.zeros(5))                    # no device population bound: there is no CPU forward
    sq = init_actor(env, layers, ["elu"], 0.01, 0.3, "orthogonal", False, None, per_state_std, True)
    assert type(sq) is SquashedGaussianActor and isinstance(sq, GaussianActor)
    with pytest.raises(ValueError):
        init_actor(env, layers, ["elu"], 0.01, 0.3, "orthogonal", True, None, per_state_std, False)
    with pytest.raises(ValueError):
        init_actor(env, layers, ["elu"], 0.01, 0.3, "orthogonal", False, None, per_state_std, False, True)


def test_gaussian_actor_floors_the_state_independent_logstd():
    a = init_actor(SyntheticEnv(3, 2), [8, 8, 8], ["tanh"], 0.01, 1.0, "orthogonal", False, None, False, False)
    ws = a.get_weights()
    ws[-1] = np.array([[-20.0, 0.5]], np.float32)
    a.set_weights(ws)
    assert np.array_equal(a.get_weights()[-1], np.array([[np.log(1e-3), 0.5]], np.float32))


def _old_create_nn_weights(in_dim, out_dim, layers, gain, init_type="orthogonal", rng=None):
    """The three-layer loop ``create_nn_weights`` had before it learned other depths (frozen copy)."""
    rng = rng if rng is not None else np.random.default_rng(np.random.randint(2 ** 31))
    dims = [in_dim, layers[0], layers[1], out_dim]
    ws = []
    for l in range(3):
        rows, cols = dims[l], dims[l + 1]
        last = l == 2
        if init_type == "orthogonal":
            w = _orthogonal(rng, rows, cols, gain if (last and gain) else math.sqrt(2.0))
        elif init_type == "var":
            scale = gain if (last and gain) else 0.333
            lim = math.sqrt(3.0 * scale / cols)
            w = rng.uniform(-lim, lim, (rows, cols)).astype(np.float32)
        elif init_type == "uniform":
            lim = math.sqrt(6.0 / (rows + cols))
            w = rng.uniform(-lim, lim, (rows, cols)).astype(np.float32)
        else:
            raise ValueError("init_type must be orthogonal, var or uniform")
        ws += [w, np.zeros(cols, np.float32)]
    return ws


@pytest.mark.parametrize("init_type", ["orthogonal", "var", "uniform"])
@pytest.mark.parametrize("gain", [0.01, None])
def test_create_nn_weights_at_depth_two_is_unchanged(init_type, gain):
    np.random.seed(7)
    new = create_nn_weights(11, 6, (64, 48), gain, init_type)
    st_new = np.random.get_state()
    np.random.seed(7)
    old = _old_create_nn_weights(11, 6, (64, 48), gain, init_type)
    st_old = np.random.get_state()
    assert len(new) == len(old) == 6
    for a, b in zip(new, old):
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
    assert np.array_equal(st_new[1], st_old[1]) and st_new[2:] == st_old[2:]


def test_learners_off_the_training_engine_are_refused(tmp_path):
    base = [a for a in ARGS if a not in ("--runs", "3")] + ["--save_path", str(tmp_path), "--runs", "1"]
    no_squash = [a for a in base if a != "--actor_squash"]
    for alg_type in ("sac", "sac_imit", "bc"):
        inp = T.build_inputs(T.create_train_parser().parse_args(no_squash + ["--alg_type", alg_type]))[0]
        with pytest.raises(ValueError, match="--actor_squash"):
            T.build_run(inp, FakeShared(1), 0)
    deep = [a for a in base] + ["--actor_layers", "8", "8", "8", "--alg_type", "sac_imit"]
    inp = T.build_inputs(T.create_train_parser().parse_args(deep))[0]
    with pytest.raises(ValueError, match="exactly two hidden layers"):
        T.build_run(inp, FakeShared(1), 0)


def test_make_f_keeps_the_two_hidden_layer_limit():
    from sac_expert_b200.sac_eo.common.update_utils import make_F
    a = init_actor(SyntheticEnv(3, 2), [8, 8, 8], ["tanh"], 0.01, 1.0, "orthogonal", False, None, True, False)
    with pytest.raises(ValueError, match="exactly two hidden layers"):
        make_F(a, np.zeros((4, 3), np.float32))


# ---------------------------------------------------------------------------------------------- expert files
def _build_with_expert(tmp_path, extra, alg_type="sac_imit"):
    args = [a for a in ARGS if a not in ("--runs", "3")] + ["--runs", "1", "--save_path", str(tmp_path),
                                                            "--alg_type", alg_type, "--expert_path", str(tmp_path),
                                                            "--expert_file", "expert.pkl"] + extra
    inp = T.build_inputs(T.create_train_parser().parse_args(args))[0]
    alg = T.build_run(inp, FakeShared(1), 0)
    experts = FakeShared(1)
    alg._bind_expert(experts, 0)
    return alg, experts.pop


@pytest.mark.parametrize("alg_type", ["sac_imit", "bc"])
def test_mpo_expert_file_reaches_the_device_as_a_policy_spec(tmp_path, alg_type):
    ws, final = write_mpo_expert(tmp_path / "expert.pkl", 11, 3)
    alg, pop = _build_with_expert(tmp_path, [], alg_type)
    assert type(alg.expert) is GaussianActor
    assert pop.spec == PolicySpec(n_agents=1, S=11, A=3, hidden=(256, 256, 256), acts=("elu",) * 3, squash=False,
                                  per_state_std=True, std_mult=0.3, device=0)
    got = pop.nets[0, "actor"]
    assert len(got) == 8 and all(np.array_equal(g, w) for g, w in zip(got, ws))
    s_rms = alg.expert_normalizer.s_rms                  # old s_t / s_mean / s_var form (organize_rms_inputs)
    assert np.array_equal(s_rms.mean, final["s_mean"]) and np.array_equal(s_rms.std, np.sqrt(final["s_var"]))
    assert alg.expert.s_rms is s_rms


def test_state_independent_and_squashed_deep_experts(tmp_path):
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(32, 16), act="tanh", per_state_std=False, std_mult=0.5)
    _, pop = _build_with_expert(tmp_path, [])
    assert isinstance(pop.spec, PolicySpec) and not pop.spec.per_state_std and pop.spec.hidden == (32, 16)
    assert pop.nets[0, "actor"][-1].shape == (1, 3)
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(16, 16, 16), act="relu", squash=True)
    _, pop = _build_with_expert(tmp_path, [])
    assert isinstance(pop.spec, PolicySpec) and pop.spec.squash and pop.spec.hidden == (16, 16, 16)


def test_two_hidden_layer_squashed_expert_stays_on_the_population_path(tmp_path):
    write_mpo_expert(tmp_path / "expert.pkl", 11, 3, hidden=(8, 8), act="relu", squash=True)
    alg, pop = _build_with_expert(tmp_path, [])
    assert type(alg.expert) is SquashedGaussianActor
    assert isinstance(pop.spec, PopulationSpec) and pop.spec.actor_hidden == (8, 8) and pop.spec.num_models == 0


# ---------------------------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("per_state_std", [True, False])
def test_oracle_policy_sample_at_depth_two(per_state_std):
    from oracle.sac_eo_oracle import NetCfg, gaussian_sample, head
    from tests.policy_oracle import policy_sample
    cfg = NetCfg(S=5, A=2, actor_hidden=(16, 12), actor_acts=("tanh", "elu"), per_state_std=per_state_std, std_mult=0.4)
    rng = np.random.default_rng(3)
    dims = [5, 16, 12, cfg.Ao]
    theta = []
    for i in range(3):
        theta += [torch.from_numpy(rng.standard_normal((dims[i], dims[i + 1])) * 0.5),
                  torch.from_numpy(rng.standard_normal(dims[i + 1]) * 0.1)]
    if not per_state_std:
        theta.append(torch.from_numpy(rng.standard_normal((1, 2)) * 0.3))
    st = {"s_mean": rng.standard_normal(5), "s_std": rng.uniform(0.5, 2, 5), "act_limit": np.array([2.0, 0.5])}
    s = torch.from_numpy(rng.standard_normal((9, 5)))
    u = torch.from_numpy(rng.standard_normal((9, 2)))
    for noise in (None, u):
        sq = policy_sample(cfg, theta, s, noise, st, squash=True)
        ref = head(cfg, theta, s, noise, st, deterministic=noise is None)[0]
        assert sq.dtype == torch.float64 and torch.equal(sq, ref)
        assert torch.equal(policy_sample(cfg, theta, s, noise, st, squash=False), gaussian_sample(cfg, theta, s, noise, st))


@pytest.mark.parametrize("per_state_std", [True, False])
def test_oracle_policy_sample_at_depth_three(per_state_std):
    """The logstd variable of a state-independent-std actor is the tensor after the four dense layers."""
    from oracle.sac_eo_oracle import NetCfg
    from tests.policy_oracle import policy_sample
    A, std_mult = 2, 0.4
    cfg = NetCfg(S=5, A=A, actor_hidden=(16, 12, 8), actor_acts=("tanh", "elu", "relu"), per_state_std=per_state_std,
                 std_mult=std_mult)
    rng = np.random.default_rng(4)
    dims = [5, 16, 12, 8, cfg.Ao]
    ws = []
    for i in range(4):
        ws += [rng.standard_normal((dims[i], dims[i + 1])) * 0.5, rng.standard_normal(dims[i + 1]) * 0.1]
    if not per_state_std:
        ws.append(rng.standard_normal((1, A)) * 0.3)
    st = {"s_mean": rng.standard_normal(5), "s_std": rng.uniform(0.5, 2, 5), "act_limit": np.array([2.0, 0.5])}
    s, u = rng.standard_normal((9, 5)), rng.standard_normal((9, A))
    h = (s - st["s_mean"]) / st["s_std"]
    for l, act in enumerate(("tanh", "elu", "relu")):
        z = h @ ws[2 * l] + ws[2 * l + 1]
        h = np.tanh(z) if act == "tanh" else np.where(z > 0, z, np.expm1(z)) if act == "elu" else np.maximum(z, 0)
    out = h @ ws[6] + ws[7]
    mean = out[:, :A]
    raw = out[:, A:] if per_state_std else np.broadcast_to(ws[8], mean.shape)
    ls = (np.log(np.log1p(np.exp(raw))) - np.log(np.log(2.0)) if per_state_std else raw) + np.log(std_mult)
    gauss = mean + np.exp(np.maximum(ls, np.log(1e-3))) * u
    squashed = st["act_limit"] * np.tanh(mean + np.exp(np.clip(raw, -5, 2)) * u)
    theta = [torch.from_numpy(np.asarray(w)) for w in ws]
    s_t, u_t = torch.from_numpy(s), torch.from_numpy(u)
    assert np.allclose(policy_sample(cfg, theta, s_t, u_t, st, squash=False).numpy(), gauss, rtol=1e-12, atol=1e-12)
    assert np.allclose(policy_sample(cfg, theta, s_t, u_t, st, squash=True).numpy(), squashed, rtol=1e-12, atol=1e-12)
    assert np.allclose(policy_sample(cfg, theta, s_t, None, st, squash=False).numpy(), mean, rtol=1e-12, atol=1e-12)
