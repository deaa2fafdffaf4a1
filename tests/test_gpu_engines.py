"""GPU: engine-level consistency - fused tcgen05 kernels vs the unfused GEMM chain vs the exact fp32 engine,
the Humanoid-shaped wide-input case, and statistical checks of the in-kernel Philox draws (the reference's
NumPy streams cannot be reproduced on device, SURVEY.md §4 tier 4)."""
import numpy as np
import pytest
import torch

from oracle.sac_eo_oracle import NetCfg
from sac_expert_b200 import lib as L
from sac_expert_b200.population import Population, PopulationSpec
from sac_expert_b200.synth import fill_synthetic
from tests.helpers import build, compare_update, fp32_expert_term, rel

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _run(cfg, **kw):
    pop, probs = build(cfg, n_agents=2, B=256, E=20, N=1500, seed=31, **kw)
    pop.update(1, num_timesteps=0, use_device_rng=False)
    torch.cuda.synchronize()
    out = dict(g_q=pop.debug("g_q").cpu().numpy().copy(),
               g_a=pop.debug("g_actor").cpu().numpy().reshape(pop.spec.n_agents, -1).copy(),
               losses=pop.losses.cpu().numpy().copy(), actor=pop.t["actor"].cpu().numpy().copy(),
               q=pop.t["q"].cpu().numpy().copy())
    return out


def test_fused_vs_unfused_mlp_vs_fp32_engine():
    cfg = NetCfg(S=27, A=8)       # Ant-shaped, 2x256 nets, 2x512 models
    ref = _run(cfg, gemm_mode=L.GEMM_FP32_SIMT)
    fused = _run(cfg, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    plain = _run(cfg, gemm_mode=L.GEMM_TCGEN05_BF16X3, fuse_forward=False, fuse_backward=False)
    for name, got in (("fused", fused), ("unfused", plain)):
        # north_star tolerance (1e-3); the actor gradient runs through min(Q1,Q2) and tanh, which amplify the ~1e-5
        # per-GEMM error of the bf16x3 engine
        assert rel(got["g_q"], ref["g_q"]) < TOL, name
        assert rel(got["g_a"][:, :-1], ref["g_a"][:, :-1]) < TOL, name
        assert np.allclose(got["losses"], ref["losses"], rtol=TOL, atol=1e-6), name
    # the fused and the unfused tensor-core paths do the same bf16x3 arithmetic tile by tile
    assert rel(fused["g_q"], plain["g_q"]) < 2e-4 and rel(fused["g_a"][:, :-1], plain["g_a"][:, :-1]) < TOL


@pytest.mark.parametrize("B", [256, 260])
def test_wide_head_actor_fork_matches_one_stream(B):
    """A 2x256 actor with more outputs than the warp-specialised kernels take (per-state std, A = 20: 40 outputs) runs
    on the GEMM chain, which writes the hidden activations of every pass, the TD-target pass included.  The actor phase
    must then not run on a second stream next to it: graphed updates with and without fork_actor agree bit for bit, and
    the first one agrees with the oracle.  B = 260 leaves 4 rows past the last full 128-row tile."""
    cfg = NetCfg(S=17, A=20, model_acts=("tanh", "tanh"))
    outs = []
    for fork in (True, False):
        pop, probs = build(cfg, n_agents=2, B=B, E=20, N=1500, seed=23, gemm_mode=L.GEMM_TCGEN05_BF16X3,
                           use_graph=True, fork_actor=fork)
        worst = compare_update(pop, cfg, probs)
        bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
        assert not bad, (fork, bad)
        for step in range(1, 4):
            pop.update(1, num_timesteps=step, use_device_rng=False)
        torch.cuda.synchronize()
        out = {k: pop.t[k].cpu().numpy().copy() for k in ("actor", "q", "qt", "alpha")}
        out["losses"] = pop.losses.cpu().numpy().copy()
        outs.append(out)
        pop.close()
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k


def test_humanoid_shaped_batch_1024():
    """BASELINE configs[3]: obs 376, act 17, batch 1024 - multi-slab first layer in the fused kernels, 8 row tiles."""
    cfg = NetCfg(S=376, A=17)
    pop, probs = build(cfg, n_agents=1, B=1024, E=20, N=3000, seed=41, gemm_mode=L.GEMM_TCGEN05_BF16X3)
    worst = compare_update(pop, cfg, probs)
    bad = {k: v for k, v in worst.items() if v > TOL and not k.startswith("oracle32")}
    assert not bad, bad


def test_device_rng_statistics():
    n, B, E, A = 8, 256, 20, 8
    pop = Population(PopulationSpec(n_agents=n, S=27, A=A, B=B, E=E, replay_capacity=5000, gemm_mode=L.GEMM_TCGEN05_BF16X3))
    fill_synthetic(pop, seed=3, replay_rows=4000)
    draws = []
    for step in range(4):
        pop.update(1, num_timesteps=step, use_device_rng=True, seed=1234)
        torch.cuda.synchronize()
        idx = pop.debug("idx", torch.int64).cpu().numpy().reshape(n, B)
        noise = pop.debug("noise").cpu().numpy().reshape(n, 3 * B + E, A)
        perm = pop.debug("perm", torch.int32).cpu().numpy().reshape(n, E)
        assert idx.min() >= 0 and idx.max() < 4000
        for a in range(n):
            assert sorted(perm[a].tolist()) == list(range(E))
        draws.append((idx.copy(), noise.copy()))
    idx = np.concatenate([d[0].ravel() for d in draws])
    z = np.concatenate([d[1].ravel() for d in draws])
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert abs(np.mean(z ** 3)) < 0.03 and abs(np.mean(z ** 4) - 3.0) < 0.08
    from scipy import stats
    assert stats.kstest(z[:50000], "norm").pvalue > 1e-3
    assert stats.kstest(idx / 4000.0, "uniform").pvalue > 1e-3
    # streams differ between steps and agents, and are reproducible for a given (seed, step)
    assert not np.array_equal(draws[0][1], draws[1][1])
    assert not np.array_equal(draws[0][1][0], draws[0][1][1])
    assert np.isfinite(pop.losses.cpu().numpy()).all()


@pytest.mark.parametrize("seed", [5, 31, 77])
@pytest.mark.parametrize("fuse", [True, False])
def test_relu_mask_stability_operand_planes(seed, fuse):
    """ReLU nets on the tensor-core engine: forward passes use fp16 hi/lo planes so that activation masks and the
    min(Q1,Q2) selection agree with the fp32 oracle; with bf16 planes these seeds gave g_actor errors of 6e-3.
    Gradients are held to 2e-4 here (5x tighter than the 1e-3 bar) to catch a regression of the plane format."""
    cfg = NetCfg(S=27, A=8)
    # seed 31 holds an exact tie in a frozen MODEL (test_model_relu_tie_confined_to_one_row below): the fp32 CUDA-core expert
    # term keeps this test about the actor / critic operand planes
    with fp32_expert_term(seed == 31):
        pop, probs = build(cfg, n_agents=2, B=256, E=20, N=2000, seed=seed, gemm_mode=L.GEMM_TCGEN05_BF16X3,
                           fuse_forward=fuse, fuse_backward=fuse)
        w = compare_update(pop, cfg, probs)
    pop.close()
    for k in ("g_q1", "g_q2", "g_actor", "y", "L_pi"):
        assert w[k] < 2e-4, (k, w[k])
    assert max(w.values()) < TOL, w


def test_model_relu_tie_confined_to_one_row():
    """Seed 31 of the test above: one hidden pre-activation of one 2x512 ReLU model sits at 4.6e-8 of the magnitude of
    its summed terms - below fp32 epsilon, so the summation order alone decides the ReLU branch (the oracle, the fp32
    CUDA-core kernel and the tensor-core kernel are three orders).  The tensor-core expert term may take the other
    branch for THAT expert row; every other row must agree with the fp32 kernel to rounding, and the row that differs
    must be one whose fp64 pre-activations really contain such a tie."""
    cfg = NetCfg(S=27, A=8)
    n, E, SA, H = 2, 20, 35, 512
    outs = {}
    for kernel in ("mma", "fp32"):
        with fp32_expert_term(kernel == "fp32"):
            pop, probs = build(cfg, n_agents=n, B=256, E=E, N=2000, seed=31, gemm_mode=L.GEMM_TCGEN05_BF16X3)
            pop.update(1, num_timesteps=0, use_device_rng=False)
            torch.cuda.synchronize()
        outs[kernel] = pop.debug("mdXa").cpu().numpy().reshape(n, 2, E, cfg.A)[:, :, :E // 2].copy()
        if kernel == "mma":
            Xm = pop.debug("Xm").cpu().numpy().reshape(n, 2, E, SA)[:, :, :E // 2].astype(np.float64)
            th = pop.t["model"].cpu().numpy().astype(np.float64).reshape(n, 2, -1)
        pop.close()
    d = np.abs(outs["mma"] - outs["fp32"]).max(-1) / (np.abs(outs["fp32"]).max(-1) + 1e-30)       # [agent, model, row]
    bad = np.argwhere(d > 1e-5)
    assert len(bad) <= 1, d
    for a, m, r in bad:
        t = th[a, m]
        W0 = t[:SA * H].reshape(SA, H); b0 = t[SA * H:SA * H + H]; o = SA * H + H
        W1 = t[o:o + H * H].reshape(H, H); b1 = t[o + H * H:o + H * H + H]
        h1 = np.maximum(Xm[a, m, r] @ W0 + b0, 0)
        z2 = h1 @ W1 + b1
        scale = np.abs(h1) @ np.abs(W1) + np.abs(b1)
        assert (np.abs(z2) / scale).min() < 2e-7, (a, m, r, (np.abs(z2) / scale).min())


def test_host_buffer_paths_agree():
    """update_host (synchronous) vs update_host_async/wait_host (double-buffered, queued) vs update() with the same
    indices injected on the device: identical losses and parameters, bit for bit."""
    cfg = NetCfg(S=11, A=3, actor_hidden=(64, 64), critic_hidden=(64, 64), model_hidden=(64, 64))
    n, B, E, N, steps = 3, 64, 8, 500, 5
    rng = np.random.default_rng(3)
    idx = rng.integers(0, N, size=(steps, n, B)).astype(np.int64)
    outs = []
    for mode in ("sync", "async", "device"):
        pop, probs = build(cfg, n_agents=n, B=B, E=E, N=N, seed=4, gemm_mode=L.GEMM_FP32_SIMT)
        expert = np.stack([pop.t["expert_s"].cpu().numpy(), pop.t["expert_sp"].cpu().numpy()], 0)
        losses = []
        if mode == "sync":
            for s in range(steps):
                losses.append(pop.update_host(s, 11, idx[s], expert).copy())
        elif mode == "async":
            for s in range(steps):
                pop.update_host_async(s, 11, idx[s], expert, slot=s & 1)
                if s:
                    losses.append(pop.wait_host((s - 1) & 1).copy())
            losses.append(pop.wait_host((steps - 1) & 1).copy())
        else:
            for s in range(steps):
                pop.set_draws(idx=idx[s])
                losses.append(pop.update(1, num_timesteps=s, use_device_rng=2, seed=11).cpu().numpy().copy())
        torch.cuda.synchronize()
        outs.append((np.stack(losses), {k: pop.t[k].cpu().numpy().copy() for k in ("actor", "q", "qt", "alpha")}))
        pop.close()
    for other in outs[1:]:
        assert np.array_equal(outs[0][0], other[0])
        for k in outs[0][1]:
            assert np.array_equal(outs[0][1][k], other[1][k]), k


def test_profile_step_reports_every_launch():
    """saceo_profile_step: one real update, kernel by kernel, with per-launch device times; same result as update()."""
    cfg = NetCfg(S=11, A=3)
    outs = []
    for mode in ("profile", "plain"):
        pop, probs = build(cfg, n_agents=2, B=256, E=20, N=800, seed=6, gemm_mode=L.GEMM_TCGEN05_BF16X3)
        if mode == "profile":
            l0 = pop.launches
            prof = pop.profile_step(0, use_device_rng=False)
            assert len(prof) == pop.launches - l0 and len(prof) >= 20
            names = {n for n, _ in prof}
            assert {"k_mlp_fwd_ws", "k_mlp_bwd_ws", "k_adam", "k_model_term", "k_gather"} <= names
            assert all(us > 0 for _, us in prof) and sum(us for _, us in prof) < 1e6
        else:
            pop.update(1, num_timesteps=0, use_device_rng=False)
        torch.cuda.synchronize()
        outs.append({k: pop.t[k].cpu().numpy().copy() for k in ("actor", "q", "qt", "alpha")})
        pop.close()
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k


@pytest.mark.parametrize("hidden,acts,E,nm", [((512, 512), ("relu", "relu"), 20, 2), ((512, 512), ("tanh", "tanh"), 20, 2),
                                               ((64, 96), ("relu", "tanh"), 8, 2), ((96, 32), ("tanh", "relu"), 16, 1),
                                               ((256, 256), ("relu", "relu"), 32, 2), ((64, 64), ("relu", "relu"), 6, 2)])
def test_model_term_mma_matches_fp32_kernel(hidden, acts, E, nm):
    """Expert term, hidden layer on mma.sync tf32 hi/lo x3 (the default) against the fp32 CUDA-core kernel: the gradient
    w.r.t. the expert actions (mdXa) and the per-model MSE agree to fp32 rounding, and the whole update agrees with the
    oracle (compare_update)."""
    cfg = NetCfg(S=11, A=3, actor_hidden=(32, 32), critic_hidden=(32, 32), model_hidden=hidden, model_acts=acts, num_models=nm,
                 delta_clip_pred=3.0)
    outs = {}
    for kernel in ("mma", "fp32"):
        with fp32_expert_term(kernel == "fp32"):
            pop, probs = build(cfg, n_agents=3, B=64, E=E, N=600, seed=13)
            if kernel == "mma":
                w = compare_update(pop, cfg, probs)
                assert max(v for k, v in w.items() if not k.startswith("oracle32")) < TOL, w
            else:
                pop.update(1, num_timesteps=0, use_device_rng=False)
            torch.cuda.synchronize()
        outs[kernel] = (pop.debug("mdXa").cpu().numpy().copy(), pop.debug("mse_part").cpu().numpy().copy(),
                        pop.t["actor"].cpu().numpy().copy())
        pop.close()
    assert rel(outs["mma"][0], outs["fp32"][0]) < 1e-5, rel(outs["mma"][0], outs["fp32"][0])
    assert np.allclose(outs["mma"][1], outs["fp32"][1], rtol=1e-5, atol=1e-9)
    assert rel(outs["mma"][2], outs["fp32"][2]) < 1e-5
