"""Conjugate gradient / Fisher-vector product with the reference's call shapes
(``/root/reference/sac_eo/common/update_utils.py:4-24``, ``algs/model_free/trpo.py:179-187,200-227``).

    F = make_F(actor, s_all, trust_sub, trust_damp)      # TRPO._make_F
    v_flat = cg(F, pg_vec, cg_iters=20)                  # update_utils.cg
    vFv = np.dot(v_flat, F(v_flat))

``F`` runs J^T M J x / N + damp x on the device (tangent-forward and VJP GEMMs with the forward activations
resident); when ``cg`` receives such an ``F`` it runs the whole solve in one stream-ordered device call
(``saceo_cg_solve``) instead of one host round trip per iteration."""
import numpy as np
import torch

from ...population import Population, PopulationSpec
from .nn_utils import check_two_hidden


class _DeviceF:
    def __init__(self, actor, s_all, trust_sub=1, trust_damp=0.01, gemm_mode=0, device=0, models=None, expert=None):
        """``models`` / ``expert = (s_expert, sp_expert)``: additionally bind the frozen dynamics models and the expert
        rows, for the expert-observation blend of the on-policy updates (trpo.py:92-158, ppo.py:176-213)."""
        s_sub = np.asarray(s_all, np.float32)[::trust_sub]
        self.damp = float(trust_damp)
        mkw = {}
        if models:
            m0 = models[0]
            mkw = dict(num_models=len(models), E=len(expert[0]), model_hidden=m0.layers, model_acts=m0.activations,
                       separate_reward_nn=m0.separate_reward_nn, delta_clip_pred=float(m0.delta_clip_pred or 0.0))
        else:
            mkw = dict(num_models=0, E=0)
        spec = PopulationSpec(n_agents=1, S=actor.s_dim, A=actor.a_dim, actor_hidden=actor.layers,
                              critic_hidden=(8, 8), actor_acts=actor.activations, per_state_std=actor.per_state_std,
                              B=8, replay_capacity=8, fvp_rows=len(s_sub),
                              std_mult=actor.std_mult, gemm_mode=gemm_mode, device=device, **mkw)
        self.pop = Population(spec)
        self.pop.set_net(0, "actor", actor.get_weights())
        if getattr(actor, "s_rms", None) is not None:
            self.pop.set_norm(0, s_mean=actor.s_rms.mean, s_std=actor.s_rms.std)
        if models:
            for i, m in enumerate(models):
                self.pop.set_net(0, "m%d" % (i + 1), m.get_weights()[:6])
            m0 = models[0]
            if getattr(m0, "s_rms", None) is not None:        # the models' own normaliser set (SAC_expert.py:139-144)
                self.pop.set_norm(0, m_s_mean=m0.s_rms.mean, m_s_std=m0.s_rms.std, m_a_mean=m0.a_rms.mean,
                                  m_a_std=m0.a_rms.std, m_d_mean=m0.delta_rms.mean, m_d_std=m0.delta_rms.std)
            lim = getattr(actor, "act_high", None)
            if lim is not None:
                self.pop.set_norm(0, act_limit=np.asarray(lim, np.float32))
            self.pop.set_expert(0, np.asarray(expert[0], np.float32), np.asarray(expert[1], np.float32))
        self.pop.t["fvp_states"][0].copy_(torch.from_numpy(s_sub))
        self.n = self.pop.L.na

    def set_expert_draws(self, perm, u):
        """Expert shuffle and the ``actor.sample`` noise of the expert rows (in shuffled order) -> the u3 | u4 slots."""
        sp = self.pop.spec
        noise = np.zeros((1, 3 * sp.B + sp.E, sp.A), np.float32)
        noise[0, 2 * sp.B:2 * sp.B + sp.E] = np.asarray(u, np.float32)
        self.pop.set_draws(noise=noise, perm=np.asarray(perm, np.int32)[None])

    def _pad(self, x):
        v = torch.zeros(1, self.pop.L.na_stride)
        v[0, :self.n] = torch.as_tensor(np.asarray(x, np.float32))
        return v

    def __call__(self, x):
        return self.pop.fvp(self._pad(x), self.damp)[0, :self.n].cpu()

    def solve(self, b, cg_iters, residual_tol):
        x, vfv = self.pop.cg_solve(self._pad(b), iters=cg_iters, tol=residual_tol, damp=self.damp)
        return x[0, :self.n].cpu().numpy(), float(vfv[0])


def make_F(actor, s_all, trust_sub=1, trust_damp=0.01, **kw):
    """``TRPO._make_F`` (trpo.py:200-227) for a (Squashed)GaussianActor of two hidden layers (the training engine's)."""
    check_two_hidden(actor.layers)
    return _DeviceF(actor, s_all, trust_sub, trust_damp, **kw)


def cg(f_Ax, b, cg_iters=20, residual_tol=1e-10):
    """``cg`` (update_utils.py:4-24)."""
    if isinstance(f_Ax, _DeviceF):
        return f_Ax.solve(b, cg_iters, residual_tol)[0]
    p, r = b.copy(), b.copy()
    x = np.zeros_like(b)
    rdotr = r.dot(r)
    for _ in range(cg_iters):
        z = f_Ax(p)
        z = np.asarray(z.numpy() if hasattr(z, "numpy") else z)
        v = rdotr / p.dot(z)
        x += v * p
        r -= v * z
        newrdotr = r.dot(r)
        p = r + (newrdotr / rdotr) * p
        rdotr = newrdotr
        if rdotr < residual_tol:
            break
    return x.astype("float32")
