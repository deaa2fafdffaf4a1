"""Learned dynamics models with the reference's interface
(``/root/reference/sac_eo/models/continuous_models.py``, ``base_world_model.py``): ``sample(s, a,
deterministic=True)`` = ``s + denorm_delta(MLP([norm(s), norm(a)])[:, :S])``.  Inside the SAC-EO update the
weights are frozen and only the gradient to the action input is needed; model FITTING runs on the device through
``SAC_exp._update_models`` / ``Population.model_fit`` (joint optimiser over both models, SURVEY.md §8f row 1)."""
import numpy as np
import torch

from ..common.device_net import DeviceNet
from ..common.lockstep import Request, inline
from ..common.nn_utils import broadcast_activations, check_two_hidden, create_nn_weights
from ..envs.synthetic import flatdim


class MSEModel(DeviceNet):
    gaussian = False

    def __init__(self, env, model_layers, model_activations, model_gain, reward_layers, reward_activations,
                 reward_gain, model_setup_kwargs, std_mult=1.0):
        super().__init__()
        self.s_dim, self.a_dim = flatdim(env.observation_space), flatdim(env.action_space)
        self.layers = check_two_hidden(model_layers)
        self.activations = broadcast_activations(model_layers, model_activations)
        self.separate_reward_nn = bool(model_setup_kwargs.get("separate_reward_nn", False))
        self.delta_clip_pred = model_setup_kwargs.get("delta_clip_pred", None)
        self.reward_clip_pred = model_setup_kwargs.get("reward_clip_pred", None)
        self.reward_loss_coef = model_setup_kwargs.get("reward_loss_coef", 1.0)
        self.delta_clip_loss = model_setup_kwargs.get("delta_clip_loss", None)
        self.reward_clip_loss = model_setup_kwargs.get("reward_clip_loss", None)
        self.scale_model_loss = bool(model_setup_kwargs.get("scale_model_loss", False))
        out = self.s_dim if self.separate_reward_nn else self.s_dim + 1
        self._host_weights = create_nn_weights(self.s_dim + self.a_dim, out, self.layers, model_gain)
        self.reward_layers = check_two_hidden(reward_layers) if self.separate_reward_nn else None
        self.reward_activations = broadcast_activations(reward_layers, reward_activations) if self.separate_reward_nn else None
        self._reward_weights = (create_nn_weights(self.s_dim + self.a_dim, 1, self.reward_layers, reward_gain)
                                if self.separate_reward_nn else None)
        self._logstd = np.ones((1, self.s_dim), np.float32) * np.log(std_mult) if self.gaussian else None
        self.trainable = ["W0", "b0", "W1", "b1", "W2", "b2"] + (["logstd"] if self.gaussian else [])

    def set_rms(self, normalizer):
        self._rms = normalizer.get_rms()
        self.s_rms, self.a_rms, self.r_rms, self.delta_rms, _ = self._rms
        self._push_rms()
        self._rms_pushed = self._rms_versions()

    def _push_rms(self):
        if self._pop is not None and self._rms is not None:
            self._pop.set_norm(self._agent, m_s_mean=self.s_rms.mean, m_s_std=self.s_rms.std, m_a_mean=self.a_rms.mean,
                               m_a_std=self.a_rms.std, m_d_mean=self.delta_rms.mean, m_d_std=self.delta_rms.std)

    def _device_logstd(self):
        """The trainable logstd lives in the device fit tables once the joint optimiser is bound."""
        if self.gaussian and self._pop is not None and "model_logstd" in self._pop.t:
            return self._pop.t["model_logstd"][self._agent, int(self._table[1]) - 1]
        return None

    def get_weights(self, flat=False):
        ws = super().get_weights(False)
        if not self.gaussian:
            return ws
        dev = self._device_logstd()
        if dev is not None:
            self._logstd = dev.detach().cpu().numpy()[None].astype(np.float32)
        return ws + [self._logstd.copy()]

    def set_weights(self, weights, from_flat=False, increment=False):
        if self.gaussian and not from_flat:
            self._logstd = np.asarray(weights[-1], np.float32).reshape(1, -1)
            weights = weights[:-1]
            dev = self._device_logstd()
            if dev is not None:
                dev.copy_(torch.from_numpy(self._logstd[0]))
        super().set_weights(weights, from_flat, increment)

    def _device_reward(self):
        """The reward network lives in the device fit tables once the joint optimiser is bound (separate_reward_nn)."""
        if self.separate_reward_nn and self._pop is not None and "reward_m" in self._pop.t:
            return "r%d" % int(self._table[1])
        return None

    def get_reward_weights(self):
        name = self._device_reward()
        if name is not None:
            self._reward_weights = self._pop.get_net(self._agent, name)
        return self._reward_weights

    def set_reward_weights(self, weights):
        if self.separate_reward_nn:
            self._reward_weights = [np.asarray(w, np.float32) for w in weights]
            name = self._device_reward()
            if name is not None:
                self._pop.set_net(self._agent, name, self._reward_weights)

    def _sample_steps(self, s, a, deterministic=True):
        if self.gaussian and not deterministic:
            raise NotImplementedError("stochastic GaussianModel rollouts are not on the SAC-EO update path")
        pop = self._need_device()
        self._sync_rms()
        net = int(self._table[1]) - 1
        s_, a_ = self._as_rows(s, self.s_dim), self._as_rows(np.asarray(a), self.a_dim)
        sp = yield Request("model", pop, self._agent, (s_.shape[0],), obs=s_, act=a_)
        out = sp[net]
        return out[0] if out.shape[0] == 1 else out

    sample = inline(_sample_steps)

    def get_loss(self, s, sp, a, r):
        raise NotImplementedError("per-model losses are evaluated inside the joint device step: use "
                                  "SAC_exp._apply_model_grads / Population.model_fit (returns the minibatch losses)")


class GaussianModel(MSEModel):
    gaussian = True
