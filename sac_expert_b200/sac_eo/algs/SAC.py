"""``SAC`` - plain Soft Actor-Critic update with the reference's class interface
(``/root/reference/sac_eo/algs/SAC.py``): ``_update(num_timesteps)`` runs gather -> twin-Q critics ->
actor -> temperature -> Polyak for one agent as ONE stream-ordered device call.

What the reference keeps in tf.Variables / Keras optimizers / NumPy lives in a single-agent
``Population`` here (``n_agents = 1`` reproduces the reference's behaviour; use ``Population`` directly
for many agents).  The random draws are made on the HOST with the same calls, in the same order, as the
reference (``np.random.randint`` for the minibatch, ``np.random.normal`` for the three / five action-noise
draws, ``self.rng.shuffle`` for the expert split) and injected, so the NumPy RNG streams are consumed
identically.  ``train`` is the reference's environment loop (host Python) around that call."""
import time

import numpy as np
import torch

from ... import lib as _l
from ...population import Population, PopulationSpec
from ..common.buffers import TrajectoryBuffer
from ..common.lockstep import Request, inline, np_random
from ..common.logger import Logger
from ..common.nn_utils import check_two_hidden
from ..common.normalizer import RunningNormalizers
from ..common.samplers import trajectory_sampler_steps
from ..envs.synthetic import flatdim

_DEFAULTS = dict(gamma=0.995, lam=0.97, init_temperature=0.1, q_crit_lr=3e-4, mbpo_actor_lr=1e-4, mbpo_alpha_lr=1e-4,
                 sac_batch_size=256, soft_tau=5e-3, target_update_int=1, env_buffer_size=None, alg_seed=0,
                 init_rms_stats=None, only_model_normalizer=False, update_normalizers=False, random_act=False,
                 epsilon=1e-3, scale_epsilon_by_true_MSE=False, use_expert_actions=False, scale_max_disc=False,
                 scale_median_disc=False, scale_total_disc=False, exp_mult=False, min_mult=False, mult_coeff=1.0,
                 expert_buffer_size=20, expert_batch_size=None, model_buffer_size=100000, device_replay_capacity=100000,
                 gemm_mode=_l.GEMM_TCGEN05_BF16X3, device=0, save_path="./logs", checkpoint_file="TEMPLOG",
                 save_freq=None, eval_freq=None, eval_num_traj=5, env_horizon=1000, env_batch_type="steps",
                 env_batch_size_init=5000, env_batch_size=3000, exp_batch_type="steps", total_timesteps=5e5)


class SAC:
    _expert_term = False

    def __init__(self, idx, env, env_eval, actor, critics, q_targets, q_critics, models, alg_kwargs, mf_update_kwargs,
                 population=None, agent=0):
        self.env, self.env_eval = env, env_eval
        self.actor, self.critics, self.q_targets, self.q_critics, self.models = actor, critics, q_targets, q_critics, models
        self.s_dim, self.a_dim = flatdim(env.observation_space), flatdim(env.action_space)
        self._setup(alg_kwargs)
        self.logger = Logger()
        self.checkpoint_name = "%s_%d" % (self.checkpoint_file, idx)
        self.current_reward = 0
        self.normalizer = RunningNormalizers(self.s_dim, self.a_dim, self.gamma, self.init_rms_stats)
        self.model_normalizer = RunningNormalizers(self.s_dim, self.a_dim, self.gamma, self.init_rms_stats)
        self.env_data = TrajectoryBuffer(self.s_dim, self.a_dim, self.gamma, self.lam, self.env_buffer_size)
        self.target_entropy = -len(env.action_space.sample())              # SAC_expert.py:46
        self._build_population(population, agent)
        self._set_rms()

    # ------------------------------------------------------------------ setup
    def _setup(self, alg_kwargs):
        kw = dict(_DEFAULTS)
        kw.update({k: v for k, v in alg_kwargs.items() if v is not None or k not in _DEFAULTS})
        self.alg_kwargs = kw
        self.gamma, self.lam = kw["gamma"], kw["lam"]
        self.init_temperature = kw["init_temperature"]
        self.mbpo_lr, self.mbpo_actor_lr, self.mbpo_alpha_lr = kw["q_crit_lr"], kw["mbpo_actor_lr"], kw["mbpo_alpha_lr"]
        self.sac_batch_size = int(kw["sac_batch_size"])
        self.soft_tau, self.target_update_int = kw["soft_tau"], int(kw["target_update_int"])
        self.env_buffer_size = int(kw["env_buffer_size"]) if kw["env_buffer_size"] else None
        self.alg_seed = kw["alg_seed"]
        self.rng = np.random.default_rng(self.alg_seed)                    # base_onpolicy_alg.py:108-109
        self.init_rms_stats = kw["init_rms_stats"]
        self.only_model_normalizer = kw["only_model_normalizer"]
        self.update_normalizers, self.random_act = kw["update_normalizers"], kw["random_act"]
        self.epsilon = kw["epsilon"]
        self.expert_buffer_size = int(kw["expert_buffer_size"]) if kw["expert_buffer_size"] else None
        self.expert_batch_size = kw["expert_batch_size"]
        self.save_path, self.checkpoint_file = kw["save_path"], kw["checkpoint_file"]
        self.save_freq, self.eval_freq, self.eval_num_traj = kw["save_freq"], kw["eval_freq"], int(kw["eval_num_traj"])
        self.env_horizon, self.env_batch_type = int(kw["env_horizon"]), kw["env_batch_type"]
        self.env_batch_size_init, self.env_batch_size = int(kw["env_batch_size_init"]), int(kw["env_batch_size"])
        self.exp_batch_type = kw["exp_batch_type"]
        self._max_episode_steps = self.env_horizon               # base_onpolicy_alg.py:104
        self.corruptor = None                                    # state-noise corruption (common/corruptor.py) is out of scope
        self.last_eval = 0

    def _n_models(self):
        return 0

    def _expert_rows(self):
        return 0

    def _build_population(self, population=None, agent=0):
        """Binds the networks, the replay buffer and the per-agent records to agent ``agent`` of a device population:
        a new one-agent ``Population`` by default, or the population a ``SharedPopulation`` holds for several runs."""
        a, q, kw = self.actor, self.q_critics[0], self.alg_kwargs
        check_two_hidden(a.layers)           # the training engine's actor: two hidden layers (DESIGN.md §8)
        nm = self._n_models()
        m = self.models[0] if nm else None
        cap = self.env_buffer_size or int(kw["device_replay_capacity"])
        spec = PopulationSpec(
            n_agents=1, S=self.s_dim, A=self.a_dim, actor_hidden=a.layers, critic_hidden=q.layers,
            model_hidden=m.layers if m else (8, 8), actor_acts=a.activations, critic_acts=q.activations,
            model_acts=m.activations if m else ("relu", "relu"), per_state_std=a.per_state_std,
            separate_reward_nn=m.separate_reward_nn if m else False, num_models=nm,
            reward_hidden=getattr(m, "reward_layers", None) if m else None,
            reward_acts=getattr(m, "reward_activations", None) if m else None,
            delta_clip_pred=(m.delta_clip_pred or 0.0) if m else 0.0, B=self.sac_batch_size, E=max(self._expert_rows(), 2),
            target_update_int=self.target_update_int, replay_capacity=cap, std_mult=a.std_mult,
            gemm_mode=kw["gemm_mode"], device=kw["device"])
        self.pop = pop = Population(spec) if population is None else population.get(spec)
        self.agent = agent
        a._bind(pop, agent, "actor")
        for k, (live, tgt) in enumerate(zip(self.q_critics, self.q_targets)):
            live._bind(pop, agent, "q%d" % (k + 1))
            tgt._bind(pop, agent, "t%d" % (k + 1))
        for k in range(nm):
            self.models[k]._bind(pop, agent, "m%d" % (k + 1))
        pop.t["alpha"][agent] = float(np.log(self.init_temperature))      # raw, log-initialised (SAC_expert.py:106)
        pop.set_hyper(agent, gamma=self.gamma, tau=self.soft_tau, lr_q=self.mbpo_lr, lr_pi=self.mbpo_actor_lr,
                      lr_alpha=self.mbpo_alpha_lr, eps=self.epsilon, target_entropy=float(self.target_entropy))
        self.env_data.attach(pop, agent)

    def _set_rms(self):
        """Shares the normalisers with all networks (SAC_expert.py:135-153)."""
        self.actor.set_rms(self.normalizer)
        for net in list(self.q_critics) + list(self.q_targets):
            net.set_rms(self.normalizer)
        for m in self.models[: self._n_models()]:
            m.set_rms(self.model_normalizer if self.only_model_normalizer else self.normalizer)

    @property
    def alpha(self):
        return float(self.pop.t["alpha"][self.agent])

    # ------------------------------------------------------------------ the hot path
    def _draw(self, expert_reg=None):
        """Host draws in the reference's consumption order (SURVEY.md App. A)."""
        B, A = self.sac_batch_size, self.a_dim
        rand = np_random()
        idx = rand.randint(self.env_data.current_size, size=B)        # buffers.py:135
        u1 = rand.normal(size=(B, A))                                 # evaluate(sp), continuous_actors.py:350
        perm, u_exp = None, []
        if expert_reg is not None:
            E = len(expert_reg[0])
            if self._n_models() == 1:
                perm = np.arange(E)
            else:
                order = np.arange(E)
                self.rng.shuffle(order)                                    # SAC_expert.py:301-303
                sections = np.array_split(order, len(self.models))
                if len(sections[0]) != len(sections[1]):
                    raise ValueError("two-model expert term needs an even number of expert rows (SAC_expert.py:329-332)")
                perm = np.concatenate(sections[:2])
        u2 = rand.normal(size=(B, A))                                 # evaluate(s)
        if expert_reg is not None:
            if self._n_models() == 1:
                u_exp = [rand.normal(size=(len(perm), A))]
            else:
                h = len(perm) // 2
                u_exp = [rand.normal(size=(h, A)), rand.normal(size=(h, A))]   # sample(s_E_one/two)
        u5 = rand.normal(size=(B, A))                                 # evaluate(s) for the alpha step
        noise = np.concatenate([u1, u2] + u_exp + [u5], 0).astype(np.float32)
        return idx.astype(np.int64), noise, perm

    def _sync_rms(self):
        """Re-pushes normaliser statistics that changed since the last push (``update_rms`` / ``set_rms_stats``): the
        reference's networks see them live (SAC_expert.py:135-153, normalizer.py:126-190)."""
        for net in [self.actor] + list(self.q_critics) + list(self.q_targets) + list(self.models[: self._n_models()]):
            net._sync_rms()

    def _device_update_steps(self, num_timesteps, expert_reg=None, expert=None, eps=None):
        """One update of this agent; ``expert`` = (s_E, sp_E) rows and ``eps`` (None: unchanged) are uploaded first."""
        self._sync_rms()
        idx, noise, perm = self._draw(expert_reg)
        self.last_idx = idx
        perm = None if perm is None else perm.astype(np.int32)
        losses = yield Request("update", self.pop, self.agent,
                               ("update", int(num_timesteps), idx.shape, noise.shape, None if perm is None else perm.shape),
                               bc=False, num_timesteps=int(num_timesteps), idx=idx, noise=noise, perm=perm, expert=expert,
                               eps=eps)
        return dict(q1_loss=losses[0], q2_loss=losses[1], pi_loss=losses[2], mse_loss=losses[3], p_loss=losses[4],
                    alpha_loss=losses[5], alpha=losses[6], epsilon=losses[7])

    def _update_steps(self, num_timesteps):
        """``SAC._update`` (SAC.py:236-250)."""
        self.last_losses = yield from self._device_update_steps(num_timesteps)

    _update = inline(_update_steps)

    def _update_q_target(self):
        """Polyak averaging is fused into the critic Adam kernel, gated on
        ``num_timesteps % target_update_int == 0`` like SAC.py:246-248; nothing to do here."""

    # ------------------------------------------------------------------ environment loop (host; callers of the hot path)
    def _evaluate_steps(self, num_timesteps):
        """``_evaluate`` (base_onpolicy_alg.py:174-197)."""
        t0 = time.time()
        J = []
        for _ in range(self.eval_num_traj):
            J.append((yield from trajectory_sampler_steps(self.env_eval, self.actor, self.env_horizon, eval=True,
                                                          deterministic=True))[-1])
        self.logger.log_train({"J_tot_eval": np.mean(J), "steps_eval": num_timesteps - self.last_eval,
                               "time_eval": time.time() - t0})
        self.last_eval = num_timesteps

    def _data_sinks(self):
        return [self.env_data]

    def _collect_env_data_steps(self, num_timesteps, update_normalizers=True, only_model_normalizer=False):
        """``_collect_env_data`` (SAC_expert.py:625-683 / SAC.py): whole rollouts with the current actor before the
        per-step loop starts."""
        t0 = time.time()
        batch_size = self.env_batch_size_init if num_timesteps == 0 else self.env_batch_size
        steps_start, traj_start = self.env_data.steps_total, self.env_data.traj_total
        cur, J_all = 0, []
        while cur < batch_size:
            horizon = min(batch_size - cur, self.env_horizon) if self.env_batch_type == "steps" else self.env_horizon
            s, a, r, sp, d, J = yield from trajectory_sampler_steps(self.env, self.actor, horizon, eval=True,
                                                                    corruptor=self.corruptor)
            if update_normalizers:
                (self.model_normalizer if only_model_normalizer else self.normalizer).update_rms(s, a, r, sp)
            for sink in self._data_sinks():
                yield from sink._add_steps(s, a, r, sp, d)
            if horizon == self.env_horizon:
                J_all.append(J)
            cur = (self.env_data.steps_total - steps_start) if self.env_batch_type == "steps" \
                else (self.env_data.traj_total - traj_start)
        steps_new = self.env_data.steps_total - steps_start
        self.current_reward = np.mean(J_all) if J_all else float("nan")
        self.logger.log_train({"J_tot": self.current_reward, "steps": steps_new,
                               "traj": self.env_data.traj_total - traj_start, "time_env_data": time.time() - t0})
        return steps_new

    def _episode_start_steps(self):
        """Per-episode work before the first step (SAC_exp: model fitting + adaptive expert weight)."""
        return None
        yield

    def _step_update_steps(self, num_timesteps, episode_ctx):
        yield from self._update_steps(num_timesteps)

    def _dump_and_save(self, params):
        """``_dump_and_save`` (base_onpolicy_alg.py:366-374)."""
        self.logger.log_params(params)
        self.logger.log_final(self._dump_stats())
        self.logger.dump_and_save(self.save_path, self.checkpoint_name)
        self.logger.reset()

    def _train_prologue_steps(self):
        self._set_rms()
        return
        yield

    def train_steps(self, total_timesteps, params):
        """The reference's training loop (SAC_expert.py:685-824; SAC.py:254-385): initial data collection, then one
        environment step + one ``_update`` per iteration, per-episode bookkeeping, evaluation and checkpoints.  Host
        Python; every network call inside is a device request (``common/lockstep.py``).  Returns the checkpoint name."""
        total_timesteps = int(total_timesteps)
        yield from self._train_prologue_steps()
        pts = lambda f: np.concatenate((np.arange(0, total_timesteps, f)[1:], [total_timesteps]))
        checkpoints = np.array([total_timesteps]) if self.save_freq is None else pts(self.save_freq)
        evaluate = self.eval_freq is not None
        eval_points = pts(self.eval_freq) if evaluate else None
        checkpt_idx = eval_idx = 0
        num_timesteps = 0
        if evaluate:
            yield from self._evaluate_steps(num_timesteps)
        num_timesteps += yield from self._collect_env_data_steps(num_timesteps, update_normalizers=self.update_normalizers,
                                                only_model_normalizer=self.only_model_normalizer)
        new_traj = TrajectoryBuffer(self.s_dim, self.a_dim, self.gamma, self.lam)
        episode_step, episode, episode_reward, done = 0, 0, 0.0, True
        t0 = time.time()
        ctx = None
        while num_timesteps < total_timesteps:
            if done:
                if self.update_normalizers and episode > 0:
                    s_, a_, sp_, r_ = new_traj.get_model_info()
                    if self.only_model_normalizer:
                        self.model_normalizer.update_rms(s_, a_, r_, sp_)
                    else:
                        self.normalizer.update_rms(s_, a_, r_, sp_)
                        self.model_normalizer.update_rms(s_, a_, r_, sp_)
                    new_traj.reset()
                if episode > 0:
                    self.logger.log_train({"J_tot": episode_reward, "steps": episode_step, "traj": 1,
                                           "time_env_data": time.time() - t0})
                    self.current_reward = episode_reward
                obs = self.env.reset()
                done, episode_reward, episode_step = False, 0.0, 0
                episode += 1
                ctx = yield from self._episode_start_steps()
                t0 = time.time()
            a = np.asarray((yield from self.actor._sample_steps(obs, deterministic=not self.random_act)).numpy())   # :779
            yield from self._step_update_steps(num_timesteps, ctx)
            next_obs, r, done, _ = self.env.step(self.actor.clip(a))
            done_no_max = False if episode_step + 1 == self._max_episode_steps else done
            episode_reward += r
            row = (np.array([obs]), np.array([a]), np.array([r]), np.array([next_obs]), np.array([done_no_max]))
            for sink in self._data_sinks():
                yield from sink._add_steps(*row)
            if self.update_normalizers:
                new_traj.add(*row)
            obs = next_obs
            episode_step += 1
            num_timesteps += 1
            if evaluate and num_timesteps >= eval_points[eval_idx]:
                yield from self._evaluate_steps(num_timesteps)
                eval_idx += 1
            if num_timesteps >= checkpoints[checkpt_idx]:
                self._dump_and_save(params)
                checkpt_idx += 1
        self._dump_and_save(params)
        return self.checkpoint_name

    train = inline(train_steps)

    def _dump_stats(self):
        """{'actor_weights','critic_weights','rms_stats'} checkpoint payload (base_onpolicy_alg.py:351-364)."""
        return {"actor_weights": self.actor.get_weights(), "critic_weights": [c.get_weights() for c in self.critics],
                "rms_stats": self.normalizer.get_rms_stats()}
