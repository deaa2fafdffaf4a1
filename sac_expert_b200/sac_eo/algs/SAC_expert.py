"""``SAC_exp`` - SAC with the expert-observation term and the adaptive weight, reference interface
(``/root/reference/sac_eo/algs/SAC_expert.py``).  ``_update(num_timesteps, expert_reg)`` is the seam the CUDA
path sits behind; ``expert_reg = (s_expert, a_expert, sp_expert, epsilon_coef, use_expert_actions)`` as built by
``_expert_preprocess`` (:375-424)."""
import time

import numpy as np
import torch

from .SAC import SAC
from ..common.lockstep import Request, inline, np_random
from ..common.samplers import trajectory_sampler_steps
from ..common.buffers import TrajectoryBuffer
from ..common.normalizer import RunningNormalizers


class SAC_exp(SAC):
    def __init__(self, idx, env, env_eval, env_expert, actor, expert, init_expert_rms_stats, v_critic, q_targets,
                 q_critics, models, alg_kwargs, mf_update_kwargs, population=None, agent=0):
        self.env_expert, self.expert, self.init_expert_rms_stats = env_expert, expert, init_expert_rms_stats
        self._kw_pre = alg_kwargs
        super().__init__(idx, env, env_eval, actor, v_critic, q_targets, q_critics, models, alg_kwargs, mf_update_kwargs,
                         population, agent)
        kw = self.alg_kwargs
        self.scale_epsilon_by_true_MSE, self.use_expert_actions = kw["scale_epsilon_by_true_MSE"], kw["use_expert_actions"]
        self.scale_max_disc, self.scale_median_disc, self.scale_total_disc = (kw["scale_max_disc"], kw["scale_median_disc"],
                                                                              kw["scale_total_disc"])
        self.exp_mult, self.min_mult, self.mult_coeff = kw["exp_mult"], kw["min_mult"], kw["mult_coeff"]
        self.expert_data = TrajectoryBuffer(self.s_dim, self.a_dim, self.gamma, self.lam, self.expert_buffer_size)
        self.model_data = TrajectoryBuffer(self.s_dim, self.a_dim, self.gamma, self.lam, int(kw["model_buffer_size"]))
        self.expert_normalizer = RunningNormalizers(self.s_dim, self.a_dim, self.gamma, init_expert_rms_stats)
        self.model_MSE_on_expert_data = []
        self.model_MSE_on_expert_counterfactual_action = []
        self.expert_reward = 1.0
        self.B = len(self.models)
        self._last_expert = None

    def _n_models(self):
        n = len(self.models)
        if n < 1:
            raise ValueError("SAC_exp needs at least one dynamics model")
        return min(n, 2)                      # only models[0] and models[1] are ever used (:325-326)

    def _expert_rows(self):
        kw = {**self._kw_pre}
        e = kw.get("expert_batch_size") or kw.get("expert_buffer_size") or 20
        return int(e)

    # ------------------------------------------------------------------ environment loop pieces (host)
    def _data_sinks(self):
        return [self.env_data, self.model_data]          # the per-step double add (SAC_expert.py:793-798)

    def _collect_expert_data_steps(self):
        """``_collect_expert_data`` (:156-209): deterministic rollouts of the expert policy into ``expert_data``."""
        t0 = time.time()
        cur, J_all = 0, []
        while cur < self.expert_buffer_size:
            horizon = min(self.expert_buffer_size - cur, self.env_horizon) if self.exp_batch_type == "steps" else self.env_horizon
            s, a, r, sp, d, J = yield from trajectory_sampler_steps(self.env_expert, self.expert, horizon, eval=True,
                                                                    deterministic=True, corruptor=self.corruptor)
            self.expert_data.add(s, a, r, sp, d)
            if horizon == self.env_horizon:
                J_all.append(J)
            cur = self.expert_data.steps_total if self.exp_batch_type == "steps" else self.expert_data.traj_total
        self.expert_reward = np.mean(J_all) if J_all else self.expert_reward
        self.logger.log_train({"expert_J_tot": self.expert_reward, "expert_steps": self.expert_data.steps_total,
                               "expert_traj": self.expert_data.traj_total, "time_expert_data": time.time() - t0})

    def _train_prologue_steps(self):
        self._set_rms()
        self._bind_expert()
        yield from self._collect_expert_data_steps()

    def _bind_expert(self, population=None, agent=0):
        """The expert policy is only ever rolled out (never updated): it gets a single-agent device population of its
        own for its forward passes, with its own normaliser statistics (``init_expert_rms_stats``, :128-133), or agent
        ``agent`` of the population a ``SharedPopulation`` holds for the experts of several runs.  A two-hidden-layer
        ``SquashedGaussianActor`` goes on the training engine's ``Population``; every other expert (a ``GaussianActor``,
        any depth) on a ``PolicySet``, which acts policies of any depth in one launch."""
        if self.expert is None or getattr(self.expert, "_pop", None) is not None:
            return
        from ...population import Population, PopulationSpec
        from ...policy import PolicySet, PolicySpec
        from ..actors.continuous_actors import SquashedGaussianActor
        e = self.expert
        if isinstance(e, SquashedGaussianActor) and len(e.layers) == 2:
            spec = PopulationSpec(n_agents=1, S=self.s_dim, A=self.a_dim, actor_hidden=e.layers, critic_hidden=(8, 8),
                                  model_hidden=(8, 8), actor_acts=e.activations, per_state_std=e.per_state_std, num_models=0,
                                  B=self.sac_batch_size, E=2, replay_capacity=16, std_mult=e.std_mult,
                                  gemm_mode=self.alg_kwargs["gemm_mode"], device=self.alg_kwargs["device"])
            make = Population
        else:
            spec = PolicySpec(n_agents=1, S=self.s_dim, A=self.a_dim, hidden=e.layers, acts=e.activations,
                              squash=isinstance(e, SquashedGaussianActor), per_state_std=e.per_state_std,
                              std_mult=e.std_mult, device=self.alg_kwargs["device"])
            make = PolicySet
        self._expert_pop = make(spec) if population is None else population.get(spec)
        e._bind(self._expert_pop, agent, "actor")
        e.set_rms(self.expert_normalizer)

    def _episode_start_steps(self):
        yield from self._update_models_steps()
        return (yield from self._expert_preprocess_steps())

    def _step_update_steps(self, num_timesteps, expert_reg):
        yield from self._update_steps(num_timesteps, expert_reg)

    # ------------------------------------------------------------------ hot path
    def _update_steps(self, num_timesteps, expert_reg):
        """``SAC_exp._update`` (:463-477)."""
        s_expert, _, sp_expert, epsilon, _ = expert_reg
        s_expert, sp_expert = np.asarray(s_expert, np.float32), np.asarray(sp_expert, np.float32)
        if len(s_expert) != self.pop.spec.E:
            raise ValueError(f"expert_reg carries {len(s_expert)} rows, the device population was built for {self.pop.spec.E}")
        # E*S floats: uploaded on every call (an identity / id() cache can go stale when the arrays are edited in
        # place or a freed array's id is reused by the next per-episode resample, :421-422)
        eps = None if float(epsilon) == self._last_expert else float(epsilon)
        self._last_expert = float(epsilon)
        self.last_losses = out = yield from self._device_update_steps(num_timesteps, expert_reg, expert=(s_expert, sp_expert),
                                                                      eps=eps)
        self.logger.log_train({"alpha_loss": out["alpha_loss"], "p_loss": out["p_loss"], "epsilon": epsilon})   # :351-356

    # ------------------------------------------------------------------ dynamics-model fitting (device)
    def _setup_model_fit(self):
        """``MBRLOnPolicyAlg._setup`` (mbrl_onpolicy_alg.py:35-59): one joint Adam over every model's tensors."""
        kw = self.alg_kwargs
        g = lambda k, d: kw[k] if kw.get(k) is not None else d
        self.model_lr, self.model_num_epochs = g("model_lr", 1e-3), int(g("model_num_epochs", 10))
        self.model_batch_size, self.model_batch_shuffle = int(g("model_batch_size", 200)), bool(g("model_batch_shuffle", True))
        self.model_max_updates, self.model_max_grad_norm = g("model_max_updates", 1e5), kw.get("model_max_grad_norm")
        self.model_holdout_ratio = g("model_holdout_ratio", 0.0)
        self.reset_model_optimizer = bool(g("reset_model_optimizer", False))
        if len(self.models) != self._n_models():
            raise NotImplementedError("the device joint optimiser covers the two models of the update path")
        gaussian = bool(getattr(self.models[0], "gaussian", False))
        if self.pop.model_batch is None:       # once per population: the first run of a shared one binds it for all
            self.pop.fit_bind(self.model_batch_size, use_grad_clip=self.model_max_grad_norm is not None, gaussian=gaussian)
        if getattr(self.models[0], "separate_reward_nn", False):      # the reward networks join the joint optimiser
            for k in range(self._n_models()):
                self.pop.set_net(self.agent, "r%d" % (k + 1), self.models[k]._reward_weights)
        if gaussian:                           # GaussianModel.logstd (continuous_models.py:24-25) joins the device optimiser
            for k in range(self._n_models()):
                self.pop.t["model_logstd"][self.agent, k].copy_(torch.from_numpy(np.asarray(self.models[k]._logstd, np.float32)[0]))
        self._fit_ready = True
        self._push_fit_hyper()

    def _push_fit_hyper(self):
        m = self.models[0]
        r_rms = getattr(m, "r_rms", None)
        self.pop.set_fit_hyper(self.agent, model_lr=self.model_lr, reward_loss_coef=getattr(m, "reward_loss_coef", 1.0),
                               delta_clip_loss=getattr(m, "delta_clip_loss", None), reward_clip_loss=getattr(m, "reward_clip_loss", None),
                               model_max_grad_norm=self.model_max_grad_norm,
                               scale_model_loss=float(getattr(m, "scale_model_loss", False)),
                               r_mean=float(np.ravel(r_rms.mean)[0]) if r_rms is not None else 0.0,
                               r_std=float(np.ravel(r_rms.std)[0]) if r_rms is not None else 1.0)

    def _apply_model_grads_steps(self, batch_idx):
        """``_apply_model_grads`` (mbrl_onpolicy_alg.py:301-319) for one or more minibatches.  The reference passes
        the gathered rows ``s_batch[B, mb, S]``...; the rows already live in the device replay table, so the device
        version takes the index matrix ``batch_idx[(steps,) B, mb]`` into ``model_data`` that produced them."""
        if not getattr(self, "_fit_ready", False):
            self._setup_model_fit()
        off = self.env_data.current_size - self.model_data.current_size
        if off < 0 or self.env_data.steps_total != self.model_data.steps_total:
            raise NotImplementedError("model_data must be a suffix window of the device-resident env_data rows")
        idx = np.asarray(batch_idx, np.int64)
        idx = idx.reshape((-1,) + idx.shape[-2:]) + off
        losses = yield Request("fit", self.pop, self.agent, idx.shape, idx=idx)
        self.last_model_losses = losses[-1, 0].cpu().numpy()
        return losses

    _apply_model_grads = inline(_apply_model_grads_steps)

    def _update_models_steps(self):
        """``SAC_exp._update_models`` (:480-609): holdout split, per-epoch (per-model) shuffles with the global NumPy
        RNG in the reference's order, ragged tail batch dropped, ``model_max_updates`` cap, optional optimiser
        reset, then the expert-data MSE bookkeeping.  All gradient steps of the call run back to back on the device."""
        if not getattr(self, "_fit_ready", False):
            self._setup_model_fit()
        self._sync_rms()
        self._push_fit_hyper()

        def shuffled(n):                       # one np.random.shuffle of arange(n): the reference's only RNG use here
            order = np.arange(n)
            np_random().shuffle(order)
            return order

        n_total = self.model_data.current_size
        # holdout rows are only withheld from training; the reference's holdout evaluation is commented out (:556-576)
        rows = shuffled(n_total)[: int(n_total * (1 - self.model_holdout_ratio))] if self.model_holdout_ratio > 0.0 \
            else np.arange(n_total)
        mb, nb = self.model_batch_size, len(rows) // self.model_batch_size      # ragged tail batch dropped (:538-540)
        budget = int(min(self.model_max_updates, self.model_num_epochs * nb))
        steps, ep = [], 0
        for ep in range(self.model_num_epochs):
            if self.model_batch_shuffle:       # every model sees its own order (:526-529)
                order = np.stack([shuffled(len(rows)) for _ in range(self.B)])
            else:                              # one order shared by all models (:530-532)
                order = np.repeat(shuffled(len(rows))[None], self.B, 0)
            epoch = rows[order[:, : nb * mb]].reshape(self.B, nb, mb).transpose(1, 0, 2)      # [nb, B, mb]
            steps.extend(epoch[: budget - len(steps)])
            if nb and len(steps) >= budget:
                break
        num_updates = len(steps)
        if steps:
            yield from self._apply_model_grads_steps(np.stack(steps))
        if self.reset_model_optimizer:
            yield Request("reset_fit", self.pop, self.agent, ())
        yield from self._expert_mse_bookkeeping_steps()
        self.logger.log_train({"model_loss_epochs": ep + 1, "model_updates": num_updates})
        return num_updates

    _update_models = inline(_update_models_steps)

    # ------------------------------------------------------------------ adaptive weight (host, once per episode)
    def _expert_mse_bookkeeping_steps(self):
        """MSE of the models on the expert transitions with expert actions and with one shared stochastic actor
        draw (:579-608); feeds ``scale_epsilon_by_true_MSE``."""
        sE, aE, spE, _ = self.expert_data.get_model_info()
        mse = lambda pred: float((0.5 * ((np.asarray(pred) - spE) ** 2).sum(-1)).mean())
        n = self._n_models()
        on_exp = []
        for k in range(n):
            on_exp.append(mse((yield from self.models[k]._sample_steps(sE, aE, deterministic=True)).numpy()))
        on_exp = np.mean(on_exp)
        self.model_MSE_on_expert_data.append(on_exp)
        if self.use_expert_actions:
            cf = on_exp
        else:
            a_cf = (yield from self.actor._sample_steps(sE, deterministic=False)).numpy()
            cf = []
            for k in range(n):
                cf.append(mse((yield from self.models[k]._sample_steps(sE, a_cf, deterministic=True)).numpy()))
            cf = np.mean(cf)
        self.model_MSE_on_expert_counterfactual_action.append(cf)
        return on_exp, cf

    _expert_mse_bookkeeping = inline(_expert_mse_bookkeeping_steps)

    def _calc_disc_steps(self, s_expert, a_expert, sp_expert):
        """Model-disagreement statistics over the expert rows (:427-460)."""
        if self.use_expert_actions:
            act = a_expert
        else:
            act = self.actor.tf_clip((yield from self.actor._sample_steps(s_expert, deterministic=False))).numpy()
        p0 = (yield from self.models[0]._sample_steps(s_expert, act, deterministic=True)).numpy()
        p1 = (yield from self.models[1]._sample_steps(s_expert, act, deterministic=True)).numpy()
        s_disc = np.linalg.norm(p0 - p1, axis=1)
        total = float(np.sum(s_disc))
        return s_disc / total, float(np.max(s_disc)), float(np.median(s_disc)), total

    _calc_disc = inline(_calc_disc_steps)

    def _expert_preprocess_steps(self):
        """``_expert_preprocess`` (:375-424): adaptive expert weight + optional expert minibatch."""
        eps = self.epsilon
        s_expert, a_expert, sp_expert, r_expert = self.expert_data.get_model_info()
        if self.scale_epsilon_by_true_MSE:
            eps = 1 / (self.epsilon * self.model_MSE_on_expert_counterfactual_action[-1] + 1)
            cur = self.current_reward
            if cur > 0:
                if self.min_mult:
                    eps = eps * (-min(self.mult_coeff * (cur / self.expert_reward) - 1, 0))
                if self.exp_mult:
                    eps = eps * np.exp(-self.mult_coeff * cur / self.expert_reward)
        elif self.scale_max_disc or self.scale_median_disc or self.scale_total_disc:
            _, mx, med, tot = yield from self._calc_disc_steps(s_expert, a_expert, sp_expert)
            eps = 1 / (self.epsilon * (mx if self.scale_max_disc else med if self.scale_median_disc else tot) + 1)
        if self.expert_batch_size:
            s_expert, a_expert, sp_expert, r_expert = self.expert_data.get_model_info(batch_size=self.expert_batch_size)
        return (s_expert, a_expert, sp_expert, eps, self.use_expert_actions)

    _expert_preprocess = inline(_expert_preprocess_steps)
