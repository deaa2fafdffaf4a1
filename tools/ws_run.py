"""A few un-graphed updates of the bench population (for ncu captures of single kernels).  usage: ws_run.py [n] [updates]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sac_expert_b200.population import Population, PopulationSpec
from sac_expert_b200.synth import fill_synthetic
n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
k = int(sys.argv[2]) if len(sys.argv) > 2 else 5
pop = Population(PopulationSpec(n_agents=n, S=27, A=8, B=256, E=20, replay_capacity=2000, gemm_mode=1, use_graph=False))
fill_synthetic(pop, seed=1)
for w in range(k):
    pop.update(1, num_timesteps=w, use_device_rng=True, seed=3)
torch.cuda.synchronize()
print("ok", float(pop.losses.sum()))
