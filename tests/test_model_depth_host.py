"""CPU: dynamics models of 1 to 8 hidden layers - the layout the library derives for them, the configurations it
refuses, the reference-named model classes and the wiring of a deep model through train.py; actors and critics keep
their two hidden layers."""
import ctypes as C

import numpy as np
import pytest

import __graft_entry__ as G
from sac_expert_b200 import lib as L
from sac_expert_b200.population import PopulationSpec, net_shapes
from sac_expert_b200.sac_eo import train as T
from sac_expert_b200.sac_eo.envs.synthetic import SyntheticEnv
from sac_expert_b200.sac_eo.models.continuous_models import GaussianModel, MSEModel
from sac_expert_b200.sac_eo.models.init_world_models import init_world_models
from tests.test_train_population_host import ARGS, FakeShared


@pytest.fixture(scope="module")
def lib():
    G.build()
    return L.load()


def _nm(n_in, hidden, n_out):
    return sum(int(np.prod(sh)) for sh in net_shapes(n_in, hidden, n_out))


@pytest.mark.parametrize("hidden", [(40,), (64, 32, 48), (200,) * 3, (16, 24, 32, 8, 64, 8, 16, 24)])
@pytest.mark.parametrize("sep", [False, True])
def test_layout_counts_every_model_layer(lib, hidden, sep):
    S, A = 11, 3
    lay = L.query_layout(PopulationSpec(n_agents=4, S=S, A=A, model_hidden=hidden, model_acts=("tanh",) * len(hidden),
                                        separate_reward_nn=sep, reward_hidden=(32, 32) if sep else None,
                                        reward_acts=("relu", "relu") if sep else None).to_config())
    dims = [S + A] + list(hidden) + [S if sep else S + 1]
    assert lay.nm == sum(k * n + n for k, n in zip(dims[:-1], dims[1:])) == _nm(S + A, hidden, dims[-1])
    assert lay.nm_stride % 32 == 0 and lay.nm_stride >= lay.nm


def test_two_layer_layout_is_the_parents(lib):
    """A two-hidden-layer config yields the layout the fixed-depth ABI gave (nm formula of test_abi.py)."""
    S, A, Hm = 27, 8, 512
    lay = L.query_layout(PopulationSpec(n_agents=256, S=S, A=A).to_config())
    assert lay.nm == (S + A) * Hm + Hm + Hm * Hm + Hm + Hm * (S + 1) + (S + 1)
    deeper = L.query_layout(PopulationSpec(n_agents=256, S=S, A=A, model_hidden=(Hm,) * 3, model_acts=("relu",) * 3).to_config())
    assert deeper.nm == lay.nm + Hm * Hm + Hm
    assert deeper.workspace_bytes > lay.workspace_bytes       # one more activation and gradient buffer of the models


def test_model_depth_validation(lib):
    lay = L.Layout()
    ok = PopulationSpec(n_agents=1, S=4, A=2, model_hidden=(8,) * 8, model_acts=("elu",) * 8).to_config()
    assert lib.saceo_query_layout(C.byref(ok), C.byref(lay)) == 0
    for depth in (0, 9):
        cfg = PopulationSpec(n_agents=1, S=4, A=2).to_config()
        cfg.model_layers = depth
        assert lib.saceo_query_layout(C.byref(cfg), C.byref(lay)) == -1
        assert b"model_layers" in lib.saceo_last_error()
    narrow = PopulationSpec(n_agents=1, S=4, A=2, model_hidden=(8, 8, 0), model_acts=("relu",) * 3).to_config()
    assert lib.saceo_query_layout(C.byref(narrow), C.byref(lay)) == -1
    assert b"model hidden sizes" in lib.saceo_last_error()
    bad_act = PopulationSpec(n_agents=1, S=4, A=2, model_hidden=(8, 8, 8), model_acts=("relu",) * 3).to_config()
    bad_act.model_act[2] = 7
    assert lib.saceo_query_layout(C.byref(bad_act), C.byref(lay)) == -1
    with pytest.raises(ValueError, match="1 to 8"):
        PopulationSpec(n_agents=1, S=4, A=2, model_hidden=(8,) * 9, model_acts=("relu",) * 9).to_config()
    with pytest.raises(ValueError, match="one activation per"):
        PopulationSpec(n_agents=1, S=4, A=2, model_hidden=(8, 8, 8), model_acts=("relu", "relu")).to_config()


@pytest.mark.parametrize("cls", [MSEModel, GaussianModel])
def test_init_world_models_any_depth_keras_order(cls):
    env = SyntheticEnv(11, 3)
    models = init_world_models(env, [200, 200, 200, 200], ["relu"], 0.01, 1.0, None, [512, 512], ["relu"], 0.01, None,
                               2, cls is GaussianModel, {})
    S, A = 11, 3
    want = [(S + A, 200), (200,), (200, 200), (200,), (200, 200), (200,), (200, 200), (200,), (200, S + 1), (S + 1,)]
    for m in models:
        assert m.layers == (200,) * 4 and m.activations == ("relu",) * 4
        ws = m.get_weights()
        assert [w.shape for w in ws[:10]] == want
        assert m.trainable[:10] == ["W0", "b0", "W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4"]
        assert (len(ws), m.trainable[-1]) == ((11, "logstd") if cls is GaussianModel else (10, "b4"))
    with pytest.raises(ValueError, match="1 to 8"):
        MSEModel(env, [8] * 9, ["relu"], 0.01, [8, 8], ["relu"], 0.01, {})


def test_separate_reward_nn_with_a_deep_model():
    env = SyntheticEnv(5, 2)
    m = MSEModel(env, [32, 32, 32, 32], ["tanh"], 0.01, [16, 16], ["relu"], 0.01, {"separate_reward_nn": True})
    assert m.layers == (32,) * 4 and m.reward_layers == (16, 16)
    assert [w.shape for w in m.get_weights()][-2:] == [(32, 5), (5,)]
    with pytest.raises(ValueError, match="exactly two hidden layers"):       # the reward network keeps two
        MSEModel(env, [32, 32, 32, 32], ["tanh"], 0.01, [16, 16, 16], ["relu"], 0.01, {"separate_reward_nn": True})
    spec = PopulationSpec(n_agents=1, S=5, A=2, model_hidden=m.layers, model_acts=m.activations, separate_reward_nn=True,
                          reward_hidden=m.reward_layers, reward_acts=m.reward_activations)
    assert spec.reward_net() == ((16, 16), ("relu", "relu"))
    assert L.query_layout(spec.to_config()).nm == _nm(7, (32,) * 4, 5)
    with pytest.raises(ValueError, match="two hidden layers"):          # no fallback to the deep model's widths
        PopulationSpec(n_agents=1, S=5, A=2, model_hidden=m.layers, model_acts=m.activations, separate_reward_nn=True).reward_net()


def test_train_builds_a_deep_model_population(tmp_path):
    base = [a for a in ARGS if a not in ("--runs", "3")] + ["--save_path", str(tmp_path), "--runs", "1", "--alg_type", "sac_imit"]
    inp = T.build_inputs(T.create_train_parser().parse_args(base + ["--model_layers", "200", "200", "200", "200"]))[0]
    alg = T.build_run(inp, FakeShared(1), 0)
    assert alg.pop.spec.model_hidden == (200,) * 4 and alg.pop.spec.model_acts == ("relu",) * 4
    assert [w.shape for w in alg.models[0].get_weights()][:2] == [(14, 200), (200,)]


def test_actors_and_critics_keep_two_hidden_layers(tmp_path):
    from sac_expert_b200.sac_eo.critics.critics import QCritic
    with pytest.raises(ValueError, match="exactly two hidden layers"):
        QCritic(SyntheticEnv(4, 2), [8, 8, 8], ["relu"], 1.0)
    base = [a for a in ARGS if a not in ("--runs", "3")] + ["--save_path", str(tmp_path), "--runs", "1", "--alg_type", "sac_imit"]
    for flag in ("--actor_layers", "--critic_layers"):
        inp = T.build_inputs(T.create_train_parser().parse_args(base + [flag, "8", "8", "8"]))[0]
        with pytest.raises(ValueError, match="exactly two hidden layers"):
            T.build_run(inp, FakeShared(1), 0)
