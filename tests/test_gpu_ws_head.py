"""GPU: the actor's output layer and first backward step on the tensor core (mlp_ws.cuh: k_mlp_fwd_ws with nout > 1,
k_mlp_bwd_ws with NG > 0).

Both read W2 from the W2 section of the actor's plane image, which k_adam rewrites after every update and
k_planes_build creates after a bind.  Covered at A = 3 / 8 / 17 (2A = 6 / 16 / 34 outputs: one and three 16-column
accumulator groups, and W2 rows that straddle the float4 groups of k_adam when 2A % 4 != 0):
  * after several graph-replayed updates, the tensor-core actor forward agrees with an exact-fp32 population holding
    the same weights - a stale or misplaced W2 plane element shows up here;
  * one update's actor gradients (dOut W2^T on the tensor core) agree with the fp32 oracle to 2e-4, the bound
    test_relu_mask_stability_operand_planes uses.
"""
import pytest
import torch

from oracle.sac_eo_oracle import NetCfg
from sac_expert_b200 import lib as L
from sac_expert_b200.population import Population, PopulationSpec
from sac_expert_b200.synth import fill_synthetic
from tests.helpers import build, compare_update, rel

pytestmark = pytest.mark.gpu
SHAPES = [(11, 3), (27, 8), (45, 17)]


@pytest.mark.parametrize("S,A", SHAPES)
def test_actor_forward_after_updates(S, A):
    n = 3
    tc = Population(PopulationSpec(n_agents=n, S=S, A=A, B=256, E=20, replay_capacity=600,
                                   gemm_mode=L.GEMM_TCGEN05_BF16X3, use_graph=True))
    ex = Population(PopulationSpec(n_agents=n, S=S, A=A, B=256, E=20, replay_capacity=600,
                                   gemm_mode=L.GEMM_FP32_SIMT, use_graph=False))
    fill_synthetic(tc, seed=11, replay_rows=500)
    fill_synthetic(ex, seed=11, replay_rows=500)
    obs = torch.randn(n, 300, S, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    a0 = tc.actor_forward(obs).clone()
    tc.update(4, num_timesteps=0, use_device_rng=True, seed=3)
    torch.cuda.synchronize()
    # first the forward on the planes k_adam wrote (reading tc.t below marks the tables as externally written)
    a1 = tc.actor_forward(obs).clone()
    assert rel(a1.cpu(), a0.cpu()) > 1e-4
    ex.t["actor"].copy_(tc.t["actor"])
    ref = ex.actor_forward(obs).clone()
    err = rel(a1.cpu(), ref.cpu())
    tc.close()
    ex.close()
    assert err < 1e-5, err


@pytest.mark.parametrize("S,A", SHAPES)
def test_actor_gradients_vs_oracle(S, A):
    cfg = NetCfg(S=S, A=A)
    pop, probs = build(cfg, n_agents=2, B=256, E=20, N=2000, seed=5, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    w = compare_update(pop, cfg, probs)
    pop.close()
    for k in ("g_actor", "L_pi"):
        assert w[k] < 2e-4, (k, w[k])
