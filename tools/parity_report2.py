import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.sac_eo_oracle import NetCfg
from sac_expert_b200 import lib as L
from tests.helpers import build, compare_update
for acts in (("tanh", "tanh"), ("relu", "relu")):
  for fuse in (True, False):
    cfg = NetCfg(S=27, A=8, actor_acts=acts, critic_acts=acts, model_acts=acts)
    worst = {}
    for seed in (5, 31, 77):
        pop, probs = build(cfg, n_agents=2, B=256, E=20, N=2000, seed=seed, gemm_mode=L.GEMM_TCGEN05_BF16X3,
                           fuse_forward=fuse, fuse_backward=fuse)
        w = compare_update(pop, cfg, probs)
        for k, v in w.items():
            worst[k] = max(worst.get(k, 0), v)
        pop.close()
    keys = ["y", "L_q1", "L_pi", "g_q1", "g_q2", "g_actor", "dtheta_q1", "dtheta_actor"]
    print(acts[0], "fused" if fuse else "unfused", " ".join(f"{k}={worst[k]:.1e}" for k in keys))
