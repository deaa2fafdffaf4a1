"""Synthetic MuJoCo-shaped population state, generated directly on the device (SURVEY.md §8d):
orthogonal(sqrt 2) hidden kernels / orthogonal(gain) final kernels, zero biases
(``/root/reference/sac_eo/common/nn_utils.py:24-46,86-138``), targets = copies of the live critics
(``critics/init_critic.py:34-35``), alpha = log(init_temperature) (``algs/SAC_expert.py:106``), replay rows
s,sp ~ N(0,1), a ~ U(-1,1), r ~ N(0,1), d ~ Bernoulli(0.01); non-identity normaliser statistics."""
from __future__ import annotations

import math

import torch

from .population import Population

SHAPES = {  # name -> (S, A, B)  (BASELINE.json configs)
    "hopper": (11, 3, 256),
    "halfcheetah": (17, 6, 256),
    "ant": (27, 8, 256),
    "humanoid": (376, 17, 1024),
}


def _orthogonal(gen, n, rows, cols, gain, dev):
    a = torch.randn(n, max(rows, cols), min(rows, cols), generator=gen, device=dev)
    q, r = torch.linalg.qr(a)
    q = q * torch.sign(torch.diagonal(r, dim1=-2, dim2=-1)).unsqueeze(-2)
    if rows < cols:
        q = q.transpose(-1, -2)
    return gain * q[:, :rows, :cols]


def _init_nets(gen, tab, n_in, hidden, n_out, gain, dev):
    """tab: [n, stride] flat tables; fills W blocks, leaves biases zero."""
    n = tab.shape[0]
    dims = [n_in] + list(hidden) + [n_out]
    o = 0
    for l in range(len(hidden) + 1):
        g = math.sqrt(2.0) if l < len(hidden) else gain
        w = _orthogonal(gen, n, dims[l], dims[l + 1], g, dev)
        tab[:, o:o + dims[l] * dims[l + 1]] = w.reshape(n, -1)
        o += dims[l] * dims[l + 1] + dims[l + 1]


def fill_synthetic(pop: Population, seed: int = 0, replay_rows: int | None = None, identity_norm: bool = False,
                   init_temperature: float = 0.1, gamma: float = 0.995, tau: float = 5e-3, lr_q: float = 3e-4,
                   lr_pi: float = 1e-4, lr_alpha: float = 1e-4, eps: float = 1e-3):
    sp, L, dev, t = pop.spec, pop.L, pop.dev, pop.t
    n, S, A = sp.n_agents, sp.S, sp.A
    gen = torch.Generator(device=dev).manual_seed(seed)
    t["actor"].zero_()
    _init_nets(gen, t["actor"], S, sp.actor_hidden, L.Ao, 0.01, dev)
    for k in range(2):
        q = torch.zeros(n, L.nc_stride, device=dev)
        _init_nets(gen, q, S + A, sp.critic_hidden, 1, 1.0, dev)
        t["q"][:, k] = q
        if sp.num_models > 0:
            m = torch.zeros(n, L.nm_stride, device=dev)
            _init_nets(gen, m, S + A, sp.model_hidden, L.model_out, 0.01, dev)
            t["model"][:, k] = m
    t["qt"].copy_(t["q"])
    for k in ("actor_m", "actor_v", "q_m", "q_v", "alpha_m", "alpha_v"):
        t[k].zero_()
    t["adam_t"].zero_()
    t["alpha"].fill_(math.log(init_temperature))
    hy = t["hyper"]
    hy.zero_()
    for i, v in enumerate((gamma, tau, lr_q, lr_pi, lr_alpha, eps, float(-A), 0.01)):
        hy[:, i] = v
    nm = t["norm"]
    if not identity_norm:
        r = lambda c: torch.randn(n, c, generator=gen, device=dev)
        u = lambda c: 0.5 + 1.5 * torch.rand(n, c, generator=gen, device=dev)
        nm[:, L.off_s_mean:L.off_s_mean + S] = 0.3 * r(S)
        nm[:, L.off_s_std:L.off_s_std + S] = u(S)
        nm[:, L.off_a_mean:L.off_a_mean + A] = 0.1 * r(A)
        nm[:, L.off_a_std:L.off_a_std + A] = u(A)
        nm[:, L.off_ret_std:L.off_ret_std + 1] = u(1)
        nm[:, L.off_m_s_mean:L.off_m_s_mean + S] = 0.3 * r(S)
        nm[:, L.off_m_s_std:L.off_m_s_std + S] = u(S)
        nm[:, L.off_m_a_mean:L.off_m_a_mean + A] = 0.1 * r(A)
        nm[:, L.off_m_a_std:L.off_m_a_std + A] = u(A)
        nm[:, L.off_m_d_mean:L.off_m_d_mean + S] = 0.03 * r(S)
        nm[:, L.off_m_d_std:L.off_m_d_std + S] = 0.2 * u(S)
    rows = replay_rows or sp.replay_capacity
    rows = min(rows, sp.replay_capacity)
    rep = t["replay"]
    for a0 in range(0, n, 16):        # chunked to bound temporaries
        a1 = min(n, a0 + 16)
        blk = rep[a0:a1, :rows]
        blk[..., L.off_s:L.off_s + S] = torch.randn(a1 - a0, rows, S, generator=gen, device=dev)
        blk[..., L.off_a:L.off_a + A] = 2 * torch.rand(a1 - a0, rows, A, generator=gen, device=dev) - 1
        blk[..., L.off_sp:L.off_sp + S] = torch.randn(a1 - a0, rows, S, generator=gen, device=dev)
        blk[..., L.off_r] = torch.randn(a1 - a0, rows, generator=gen, device=dev)
        d = (torch.rand(a1 - a0, rows, generator=gen, device=dev) < 0.01).double()
        rep[a0:a1].view(torch.float64)[:, :rows, L.off_d // 2] = d
    t["replay_size"].fill_(rows)
    t["replay_start"].zero_()
    pop._host_size[:] = rows
    pop._host_start[:] = 0
    if sp.num_models > 0:
        t["expert_s"].copy_(torch.randn(n, sp.E, S, generator=gen, device=dev))
        t["expert_sp"].copy_(torch.randn(n, sp.E, S, generator=gen, device=dev))
    if sp.fvp_rows > 0:
        t["fvp_states"].copy_(torch.randn(n, sp.fvp_rows, S, generator=gen, device=dev))
    torch.cuda.synchronize(dev)


def algorithmic_flops(sp) -> float:
    """Matmul FLOPs per agent-update (SURVEY.md §8d formula)."""
    S, A, B, E = sp.S, sp.A, sp.B, (sp.E if sp.num_models > 0 else 0)
    H, hm = sp.actor_hidden[0], list(sp.model_hidden)
    Ao = 2 * A if sp.per_state_std else A
    Pa = S * H + H * H + H * Ao
    Pc = (S + A) * H + H * H + H
    dm = [S + A] + hm + [S + 1]
    Pm = sum(k * n for k, n in zip(dm[:-1], dm[1:]))                        # model forward
    Bm = hm[-1] * S + sum(k * n for k, n in zip(hm[:-1], hm[1:])) + A * hm[0]   # model backward to the action columns
    f = 2 * B * (4 * Pa + 8 * Pc + 5 * H * H + H * Ao + 2 * A * H + 4 * H)
    if E:
        f += 2 * E * (2 * Pa + H * Ao + H * H + Pm + Bm)
    return float(f)


def algorithmic_bytes(sp, L) -> float:
    """Compulsory HBM bytes per agent-update (SURVEY.md §8d): theta,m,v read+write for 2 critics and the
    actor, targets read+write, models read, minibatch rows, expert rows."""
    S, A, B, E = sp.S, sp.A, sp.B, (sp.E if sp.num_models > 0 else 0)
    nm = L.nm if sp.num_models > 0 else 0
    return float(4 * (2 * 6 * L.nc + 2 * 2 * L.nc + 6 * L.na + sp.num_models * nm) + 4 * B * (2 * S + A + 2) + 4 * E * 2 * S)


def kernel_compulsory_bytes(sp, L) -> dict:
    """SURVEY.md 8d's compulsory bytes per agent-update, apportioned to the kernels that MUST move them: every
    parameter and optimiser slot once per update belongs to the optimiser kernel (theta, m, v read + write, targets read +
    write), the frozen model weights once to the expert-observation term, the minibatch rows to the gather.  The fused
    forward / backward / weight-gradient kernels have NO compulsory HBM traffic in that model (with perfect on-chip
    reuse the weights would be touched by the optimiser only): everything they move is overhead of the design, reported
    as ``bandwidth_util`` of ``kernel_design_bytes`` and never as a roofline fraction."""
    S, A, B = sp.S, sp.A, sp.B
    E = sp.E if sp.num_models > 0 else 0
    return {
        "k_adam": float(4 * (2 * 6 * L.nc + 2 * 2 * L.nc + 6 * L.na)),
        "k_model_term": float(4 * (sp.num_models * L.nm + E * 2 * S)) if sp.num_models > 0 else 0.0,
        "k_gather": float(4 * B * (2 * S + A + 2)),
    }


def kernel_design_bytes(sp, L) -> dict:
    """HBM bytes PER AGENT-UPDATE the launches of each hot kernel move BY DESIGN (weights of the nets each pass applies,
    input rows, saved activations, gradients written for the optimiser to read): the denominator of a bandwidth
    utilisation, not of a roofline fraction - summed over the kernels it is about 2.8x SURVEY.md 8d's compulsory bytes."""
    S, A, B, SA = sp.S, sp.A, sp.B, sp.S + sp.A
    E = sp.E if sp.num_models > 0 else 0
    R, H, Ao = B + E, sp.critic_hidden[0], L.Ao
    w = 4
    fwd = (  # actor(sp) | Q-target(sp,a') | Q(s,a) + saved h1,h2 | actor(s,sE) + saved | Q(s,pi) + saved | actor(s) alpha pass
        (L.na + B * S + B * Ao) + (2 * L.nc + B * SA + 2 * B) + (2 * L.nc + B * SA + 2 * B + 4 * B * H)
        + (L.na + R * S + R * Ao + 2 * R * sp.actor_hidden[0]) + (2 * L.nc + B * SA + 2 * B + 4 * B * H) + (L.na + B * S + B * Ao))
    bwd = (  # critic backward (dH2, dH1 out) | critic backward-to-action | actor backward
        (2 * L.nc + 4 * B * H + 4 * B * H + 2 * B) + (2 * L.nc + 4 * B * H + 2 * B * A + 2 * B)
        + (L.na + 2 * R * sp.actor_hidden[0] + 2 * R * sp.actor_hidden[0] + R * Ao))
    dw = (2 * (B * SA + 4 * B * H + L.nc)) + (R * S + 4 * R * sp.actor_hidden[0] + R * Ao + L.na)   # activations in, gradients out
    return {
        "k_mlp_fwd_ws": float(w * fwd), "k_mlp_bwd_ws": float(w * bwd),
        "k_model_term": float(w * (sp.num_models * L.nm + E * (2 * S + A))) if sp.num_models > 0 else 0.0,
        "k_adam": float(w * (2 * 11 * L.nc + 8 * L.na)),        # + the fp16 hi/lo weight planes of theta and of the targets
        "k_dw_planes+k_dw0_planes+k_gemm": float(w * dw), "k_gemm_tc+k_gemm_skinny": float(w * dw),
    }


kernel_algorithmic_bytes = kernel_design_bytes      # round-1 name
