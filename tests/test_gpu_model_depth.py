"""GPU: dynamics models of 1 to 8 hidden layers on both GEMM engines against the oracle - model evaluation, model fitting
(MSE and Gaussian NLL with the global-norm clip), the SAC-EO update with one and two models, behaviour cloning and the
on-policy expert gradient.  Models of any depth other than two run every pass on the per-layer GEMM chain; two-layer
models keep the fused kernels (the kernel sequence test)."""
import math

import numpy as np
import pytest
import torch

import oracle.sac_eo_oracle as O
from oracle.sac_eo_oracle import NetCfg, bc_update, model_sample, to_torch_state
from sac_expert_b200 import lib as L
from tests.helpers import build, compare_update, rel
from tests.test_gpu_model_fit import _run, _setup
from tests.test_gpu_trpo import _setup_expert

pytestmark = pytest.mark.gpu

ENGINES = {"fp32": L.GEMM_FP32_SIMT, "tc": L.GEMM_TCGEN05_BF16X3}
# depth -> (widths, activations): narrow, wide (tcgen05 tiles in the fitting passes), uneven and deep models
DEPTHS = {
    1: ((96,), ("tanh",)),
    3: ((256, 128, 64), ("tanh", "elu", "tanh")),
    4: ((200, 200, 200, 200), ("elu", "tanh", "elu", "tanh")),
    8: ((64, 48, 64, 32, 64, 48, 64, 40), ("tanh", "elu") * 4),
}
TANH = dict(actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"), actor_hidden=(64, 64), critic_hidden=(64, 64))
GRAD_TOL = 2e-4          # gradients of smooth activations, both engines (test_gpu_model_fit.py's full-size bound)


def init_net_any_depth(rng, n_in, hidden, n_out, gain):
    """oracle.init_net for any number of hidden layers (the oracle's builds two): orthogonal(sqrt 2) hidden kernels,
    orthogonal(gain) final kernel, zero biases, drawn in the same order."""
    dims = [n_in] + list(hidden) + [n_out]
    ws = []
    for l in range(len(hidden) + 1):
        ws.append(O.orthogonal(rng, (dims[l], dims[l + 1]), math.sqrt(2.0) if l < len(hidden) else gain))
        ws.append(np.zeros(dims[l + 1], np.float32))
    return ws


@pytest.fixture(autouse=True)
def _any_depth_problems(monkeypatch):
    """make_problem (and every helper built on it) draws models of the configured depth."""
    monkeypatch.setattr(O, "init_net", init_net_any_depth)


def _cfg(depth, **kw):
    hidden, acts = DEPTHS[depth]
    return NetCfg(model_hidden=hidden, model_acts=acts, **kw)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", DEPTHS)
def test_model_eval_any_depth(engine, depth):
    """saceo_model_eval: s + denorm(clip(delta)) of both models, rows staged in chunks of E, against fp64."""
    cfg = _cfg(depth, S=11, A=3, delta_clip_pred=3.0, **TANH)
    pop, probs = build(cfg, n_agents=2, B=32, E=20, N=200, seed=4, gemm_mode=ENGINES[engine])
    rows = 45
    obs = np.stack([p[1]["s"][:rows] for p in probs])
    act = np.stack([p[1]["a"][:rows] for p in probs])
    out = pop.model_eval(torch.from_numpy(obs), torch.from_numpy(act)).cpu().numpy()
    for i, p in enumerate(probs):
        st = to_torch_state(p[0], torch.float64)
        s64, a64 = torch.from_numpy(obs[i]).double(), torch.from_numpy(act[i]).double()
        for k in range(2):
            ref = model_sample(cfg, st["m%d" % (k + 1)], s64, a64, st).numpy()
            assert rel(out[i, k] - obs[i], ref - obs[i]) < GRAD_TOL, (i, k)
    pop.close()


def test_model_eval_relu_depth_3():
    """ReLU is continuous: the forward pass needs no flip allowance."""
    cfg = NetCfg(S=11, A=3, model_hidden=(128, 64, 96), model_acts=("relu",) * 3, **TANH)
    pop, probs = build(cfg, n_agents=2, B=32, E=20, N=200, seed=6, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    obs = np.stack([p[1]["s"][:30] for p in probs])
    act = np.stack([p[1]["a"][:30] for p in probs])
    out = pop.model_eval(torch.from_numpy(obs), torch.from_numpy(act)).cpu().numpy()
    for i, p in enumerate(probs):
        st = to_torch_state(p[0], torch.float64)
        ref = model_sample(cfg, st["m1"], torch.from_numpy(obs[i]).double(), torch.from_numpy(act[i]).double(), st).numpy()
        assert rel(out[i, 0] - obs[i], ref - obs[i]) < GRAD_TOL, i
    pop.close()


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("loss", ["mse", "gaussian_clip"])
def test_model_fit_any_depth(engine, depth, loss):
    """Three compounded joint fit steps of both models: losses, gradients, parameters, Adam slots (and logstd, clip norm)."""
    cfg = _cfg(depth, S=11, A=3)
    if loss == "mse":
        fit = dict(model_lr=1e-3, reward_loss_coef=0.7, delta_clip_loss=2.5)
    else:   # a clip well below the gradient norm, so that the clip scale is active
        fit = dict(model_lr=1e-3, reward_loss_coef=0.5, gaussian=True, scale_model_loss=True, model_max_grad_norm=0.05)
    pop, probs = _setup(cfg, 2, 200, 600, seed=31, fit=fit, gemm_mode=ENGINES[engine])
    w = _run(cfg, pop, probs, 200, steps=3, seed=7)
    assert w["grad"] < GRAD_TOL, w
    if loss != "mse":
        assert w["grad_logstd"] < GRAD_TOL and "gnorm" in w, w
        assert float(pop.debug("fit_gscale").cpu().max()) < 1.0        # the clip did scale the gradients
    pop.close()


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("num_models", [1, 2])
def test_update_any_depth(engine, depth, num_models):
    """One injected-draw SAC-EO update: the expert term runs through the per-layer chain on 10 (two models) or 20 (one
    model) rows per model; every loss, gradient and updated tensor against the fp32 oracle."""
    cfg = _cfg(depth, S=11, A=3, num_models=num_models, **TANH)
    pop, probs = build(cfg, n_agents=2, B=64, E=20, N=500, seed=13, gemm_mode=ENGINES[engine])
    w = compare_update(pop, cfg, probs)
    pop.close()
    bad = {k: v for k, v in w.items() if v > 1e-3 and not k.startswith("oracle32")}
    assert not bad, bad
    assert w["g_actor"] < GRAD_TOL, w


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", DEPTHS)
def test_bc_update_any_depth(engine, depth):
    cfg = _cfg(depth, S=6, A=3, num_models=2, delta_clip_pred=3.0, **TANH)
    pop, probs = build(cfg, n_agents=2, B=32, E=16, N=300, seed=3, gemm_mode=ENGINES[engine])
    frozen = pop.t["model"].clone()
    losses = pop.bc_update(1, use_device_rng=False).cpu().numpy()
    torch.cuda.synchronize()
    g_a = pop.debug("g_actor").cpu().numpy().reshape(2, pop.L.na_stride)
    assert torch.equal(pop.t["model"], frozen)
    for i, (st, replay, expert, hyper, batch) in enumerate(probs):
        o = bc_update(cfg, to_torch_state(st), batch, hyper)
        ref = np.concatenate([g.numpy().ravel() for g in o["g_actor"]])
        assert rel(g_a[i, :ref.size], ref) < GRAD_TOL, i
        assert abs(losses[i, 3] - float(o["mse"])) <= 1e-3 * abs(float(o["mse"])), i
    pop.close()


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("num_models", [1, 2])
def test_onpolicy_expert_grad_any_depth(engine, depth, num_models):
    """saceo_onpolicy_expert_grad through deep frozen models against autograd in fp64 (TRPO two-model / PPO one-model)."""
    hidden, acts = DEPTHS[depth]
    cfg, pop, probs = _setup_expert(True, ("tanh", "tanh"), num_models, gemm_mode=ENGINES[engine], model_hidden=hidden,
                                    model_acts=acts, E=16, act_limit=0.6 if num_models == 1 else None)
    grad, mse = pop.onpolicy_expert_grad(n_models=num_models, clip_actions=num_models == 1)
    grad, mse = grad.cpu().numpy(), mse.cpu().numpy()
    na = pop.L.na
    for i, (st, s, a, adv, batch) in enumerate(probs):
        th = O.to_torch_state(st, torch.float64)
        zero = [torch.zeros_like(t) for t in th["actor"]]
        if num_models == 2:
            g_ref, mse_ref, _, _ = O.trpo_expert_blend(cfg, th["actor"], zero, batch, 1.0, th)
        else:
            g_ref, mse_ref = O.ppo_expert_blend(cfg, th["actor"], zero, batch, 1.0, th)
        assert rel(grad[i, :na], O.flat(g_ref).numpy()) < GRAD_TOL, i
        assert np.all(grad[i, na:] == 0)
        assert abs(mse[i] - float(mse_ref)) <= 1e-4 * abs(float(mse_ref)), i
    pop.close()


def _kernels(depth):
    cfg = NetCfg(S=27, A=8, model_hidden=(512,) * depth, model_acts=("tanh",) * depth)
    pop, _ = build(cfg, n_agents=4, B=256, E=20, N=600, seed=1, gemm_mode=L.GEMM_TCGEN05_BF16X3, use_graph=True)
    names = [k for k, _ in pop.profile_step(use_device_rng=True, seed=3)]
    pop.close()
    return names


def test_profile_step_fused_term_only_for_two_hidden_layers():
    """Two-layer models take the fused expert term; a four-layer model never does, and its term is the GEMM chain
    (k_model_loss between the forward and the backward GEMMs)."""
    two, four = _kernels(2), _kernels(4)
    assert any(k.startswith("k_model_term") for k in two) and "k_model_loss" not in two
    assert not any(k.startswith("k_model_term") for k in four) and "k_model_loss" in four
    # everything but the expert term is the same sequence
    strip = lambda ks: [k for k in ks if not k.startswith("k_model_term") and k not in ("k_model_loss", "k_gemm_tc",
                                                                                        "k_gemm_skinny", "k_gemm_simt")]
    assert strip(two) == strip(four)


def test_train_population_four_layer_models_equal_train_main(tmp_path):
    """train_population with 2 runs of a 4-hidden-layer model reproduces train.main run for run, bit for bit."""
    from tests.test_gpu_train import COMMON
    from tests.test_gpu_train_population import _assert_same, _both
    got, want = _both(tmp_path, COMMON + ["--alg_type", "sac_imit", "--runs", "2", "--scale_epsilon_by_true_MSE",
                                          "--model_layers", "64", "64", "64", "64"])
    assert len(got) == len(want) == 2
    for r in range(2):
        _assert_same(got[r], want[r], f"run {r}")
    assert not np.array_equal(got[0]["final"]["actor_weights"][0], got[1]["final"]["actor_weights"][0])
