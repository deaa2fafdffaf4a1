"""GPU parity: one injected-draw SAC / SAC-EO update vs the CPU oracle (1e-3 relative, north_star)."""
import numpy as np
import pytest
import torch

from oracle.sac_eo_oracle import NetCfg
from tests.helpers import build, compare_update

pytestmark = pytest.mark.gpu

TOL = 1e-3   # BASELINE.json north_star: losses, gradients and parameters within 1e-3 relative

CASES = {
    "hopper_saceo": (NetCfg(S=11, A=3, actor_hidden=(64, 64), critic_hidden=(64, 64), model_hidden=(96, 96)), 64, 20),
    "state_indep_std_one_model": (NetCfg(S=7, A=2, actor_hidden=(32, 48), critic_hidden=(40, 32), model_hidden=(64, 32),
                                         per_state_std=False, num_models=1, actor_acts=("tanh", "tanh"),
                                         critic_acts=("elu", "tanh"), model_acts=("relu", "elu"),
                                         delta_clip_pred=0.05), 48, 10),
    "plain_sac_halfcheetah": (NetCfg(S=17, A=6, actor_hidden=(64, 64), critic_hidden=(64, 64), num_models=0), 64, 0),
    "sep_reward": (NetCfg(S=5, A=2, actor_hidden=(32, 32), critic_hidden=(32, 32), model_hidden=(32, 32),
                          separate_reward_nn=True), 32, 6),
}


@pytest.mark.parametrize("name", list(CASES))
def test_update_matches_oracle(name):
    cfg, B, E = CASES[name]
    pop, probs = build(cfg, n_agents=3, B=B, E=max(E, 2), N=500, seed=3)
    worst = compare_update(pop, cfg, probs, verbose=True)
    bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad


def test_full_size_hopper():
    cfg = NetCfg(S=11, A=3)   # 2x256 actor/critics, 2x512 models, B=256, E=20 (configs[0])
    pop, probs = build(cfg, n_agents=2, B=256, E=20, N=2000, seed=5)
    worst = compare_update(pop, cfg, probs, verbose=True)
    bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad


@pytest.mark.parametrize("shape", ["hopper", "ant"])
def test_full_size_tcgen05(shape):
    """Same parity bar with the tcgen05 bf16x3 engine on the 2x256 nets (B=256, E=20)."""
    from sac_expert_b200 import lib as L
    S, A = {"hopper": (11, 3), "ant": (27, 8)}[shape]
    cfg = NetCfg(S=S, A=A)
    pop, probs = build(cfg, n_agents=2, B=256, E=20, N=2000, seed=9, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    worst = compare_update(pop, cfg, probs, verbose=True)
    bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad


RAGGED = {
    # batch / expert sizes that do not line up with the 128-row tensor-core tiles or the 32-row slabs
    "B300_E6": (NetCfg(S=17, A=6, actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh")), 300, 6),
    "B129_one_model_state_indep_std": (NetCfg(S=11, A=3, per_state_std=False, num_models=1, actor_acts=("tanh", "tanh"),
                                              critic_acts=("tanh", "tanh")), 129, 20),
    "B144_plain_sac": (NetCfg(S=27, A=8, num_models=0, actor_acts=("elu", "elu"), critic_acts=("elu", "elu")), 144, 0),
    "B512_E32_A1": (NetCfg(S=3, A=1, actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"), model_hidden=(256, 256)), 512, 32),
    # 40 expert rows per model, more than the fused expert-term kernels take: the term runs as the GEMM chain
    "B160_E80_expert_term_gemms": (NetCfg(S=11, A=3, actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"),
                                          model_hidden=(64, 64), model_acts=("tanh", "tanh")), 160, 80),
    # the same with one model: its activations keep the two-model row stride of the model buffers
    "B160_E40_one_model_expert_term_gemms": (NetCfg(S=11, A=3, num_models=1, actor_acts=("tanh", "tanh"),
                                                    critic_acts=("tanh", "tanh"), model_hidden=(64, 64),
                                                    model_acts=("tanh", "tanh")), 160, 40),
    # 512-wide models: the chain's hidden-layer GEMMs run on the tensor cores (S = 17, A = 6: at S = 11, A = 3 one agent's
    # policy loss cancels to 2e-5 against terms of about 7, too close to zero for a relative tolerance)
    "B160_E80_expert_term_gemms_512": (NetCfg(S=17, A=6, actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"),
                                              model_acts=("tanh", "tanh")), 160, 80),
}


@pytest.mark.parametrize("name", list(RAGGED))
def test_ragged_sizes_tcgen05(name):
    """Partial row tiles, padded row strides, one-model / plain-SAC branches on the tensor-core engine (smooth activations:
    the tolerance is not blurred by ReLU mask flips, DESIGN.md section 4)."""
    from sac_expert_b200 import lib as L
    cfg, B, E = RAGGED[name]
    pop, probs = build(cfg, n_agents=3, B=B, E=max(E, 2), N=900, seed=13, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    worst = compare_update(pop, cfg, probs)
    bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad
    assert max(worst[k] for k in ("g_q1", "g_q2", "g_actor")) < 2e-4, worst
    pop.close()
