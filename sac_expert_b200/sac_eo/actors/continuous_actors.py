"""``GaussianActor`` and ``SquashedGaussianActor`` with the reference's interface
(``/root/reference/sac_eo/actors/continuous_actors.py:9-234`` and ``:237-415`` on top of ``BaseActor``), backed by the
CUDA tables.

A ``GaussianActor`` (``_forward`` + ``sample``, :74-123: softplus std times ``std_mult``, floor log 1e-3, no squash) is
what the on-policy trust-region updates train and what the reference's MPO experts are; a ``SquashedGaussianActor``
(``sample`` :270-306, ``evaluate`` :327-379) is the SAC / SAC-EO learner.  Actors of any depth construct: a learner goes
on the two-hidden-layer training engine (``SAC._build_population`` / ``make_F`` check the depth), an expert that the
engine cannot host is acted through a ``PolicySet`` (``SAC_exp._bind_expert``).

Kept quirks: ``SquashedGaussianActor.evaluate``/``sample`` ignore ``std_mult``/``logstd_init`` and clip logstd to
[-5, 2] (:285-306, :345-376); its constructor takes ``(…, init_type, gain, …)`` in swapped order while ``init_actor``
passes ``(…, gain, init_type, …)`` positionally, so the two cancel (:240-246, ``init_actor.py:16-17``); the noise of every
stochastic call is drawn on the host with ``np.random.normal`` exactly like the reference, so the global NumPy RNG
stream is consumed identically."""
import numpy as np
import torch

from ..common.device_net import DeviceNet
from ..common.lockstep import Request, inline, np_random
from ..common.nn_utils import broadcast_activations, create_nn_weights
from ..envs.synthetic import flatdim


class GaussianActor(DeviceNet):
    def __init__(self, env, layers, activations, gain, init_type, layer_norm, std_mult=1.0, per_state_std=False,
                 output_norm=False):
        super().__init__()
        if layer_norm:
            raise ValueError("actor_layer_norm is not supported by the CUDA path (SURVEY.md App. D)")
        self.s_dim, self.a_dim = flatdim(env.observation_space), flatdim(env.action_space)
        self.layers = tuple(int(h) for h in layers)
        if not self.layers or min(self.layers) < 1:
            raise ValueError("an actor needs at least one hidden layer of positive width (got %r)" % (layers,))
        self.activations = broadcast_activations(layers, activations)
        self.per_state_std, self.output_norm, self.std_mult = bool(per_state_std), bool(output_norm), float(std_mult)
        self.act_low = np.asarray(env.action_space.low, np.float32)
        self.act_high = np.asarray(env.action_space.high, np.float32)
        self.act_limit = self.act_high
        out = 2 * self.a_dim if self.per_state_std else self.a_dim
        self._host_weights = create_nn_weights(self.s_dim, out, self.layers, gain, init_type)
        if not self.per_state_std:
            self._host_weights.append(np.zeros((1, self.a_dim), np.float32))       # logstd variable (:56-57)
        self.trainable = ["%s%d" % (k, l) for l in range(len(self.layers) + 1) for k in ("W", "b")] + \
            ([] if self.per_state_std else ["logstd"])
        self.d = int(sum(w.size for w in self._host_weights))

    # ---- plumbing ------------------------------------------------------------------------
    def set_rms(self, normalizer):
        self._rms = normalizer.get_rms()
        self.s_rms = self._rms[0]
        self._push_rms()
        self._rms_pushed = self._rms_versions()

    def _push_rms(self):
        if self._pop is not None:
            self._pop.set_norm(self._agent, act_limit=self.act_limit)
            if self._rms is not None:
                self._pop.set_norm(self._agent, s_mean=self.s_rms.mean, s_std=self.s_rms.std)

    def set_weights(self, weights, from_flat=False, increment=False, trpo_backtrack=False):
        super().set_weights(weights, from_flat, increment)
        if not self.per_state_std:                 # floor of the logstd variable (:230-233)
            ws = self._get_list()
            ws[-1] = np.maximum(ws[-1], np.log(1e-3)).astype(np.float32)
            self._set_list(ws)

    def _run(self, s, noise, want_nlp):
        pop = self._need_device()
        self._sync_rms()
        if pop.spec.n_agents != 1:
            raise ValueError("the class interface drives a single-agent population; use Population for many agents")
        x = self._as_rows(s, self.s_dim)
        obs = torch.from_numpy(x)[None]
        nz = None if noise is None else torch.from_numpy(np.asarray(noise, np.float32).reshape(1, -1, self.a_dim))
        return pop.actor_forward(obs, nz, want_neglogp=want_nlp), x.shape[0]

    # ---- reference interface -------------------------------------------------------------
    def _sample_steps(self, s, deterministic=False):
        x = self._as_rows(s, self.s_dim)
        n = x.shape[0]
        u = None if deterministic else np_random().normal(size=(n, self.a_dim))    # :297
        pop = self._need_device()
        self._sync_rms()
        act = yield Request("act", pop, self._agent, (n, u is None), obs=x,
                            noise=None if u is None else np.asarray(u, np.float32).reshape(n, self.a_dim))
        return act[0] if n == 1 else act                                           # squeeze like :302-303

    sample = inline(_sample_steps)

    def clip(self, a):
        return np.clip(a, self.act_low, self.act_high)

    def tf_clip(self, a):
        return torch.clamp(torch.as_tensor(a), torch.as_tensor(self.act_low), torch.as_tensor(self.act_high))

    # ---- trust-region interface (continuous_actors.py:137-192), on the two-hidden-layer engine ----------------------
    # _forward parameterisation (softplus std + logstd_init, floor log 1e-3), NOT the clipped one of
    # SquashedGaussianActor.evaluate / sample.
    def _gauss(self, s, **kw):
        from ..common.update_utils import make_F
        F = make_F(self, self._as_rows(s, self.s_dim))
        try:
            return F.pop.trpo_eval(**kw)
        finally:
            F.pop.close()

    def neglogp(self, s, a):
        a = np.asarray(a, np.float32).reshape(1, -1, self.a_dim)
        return self._host(self._gauss(s, act=a, want_nlp=True)["nlp"][0])

    def entropy(self, s):
        return self._host(self._gauss(s, want_rows=True)["rows"][0, :, 3])

    def get_kl_info(self, s):
        return self._host(self._gauss(s, want_kl_info=True)["kl_info"][0]).numpy()

    def kl(self, s, kl_info_ref, direction='forward'):
        if direction != 'forward':
            raise ValueError("only the forward KL is on the device path (the reverse branch reads self.logstd, :180-182)")
        ref = np.asarray(kl_info_ref, np.float32)[None]
        return self._host(self._gauss(s, kl_ref=ref, want_rows=True)["rows"][0, :, 1])


class SquashedGaussianActor(GaussianActor):
    def __init__(self, env, layers, activations, init_type, gain, layer_norm,
                 std_mult=1.0, per_state_std=False, output_norm=False):
        # positional swap, see module docstring: what arrives as `init_type` is the gain and vice versa
        super().__init__(env, layers, activations, init_type, gain, layer_norm, std_mult, per_state_std, output_norm)
        self.min_log_std, self.max_log_std = -5, 2

    def evaluate(self, s):
        n = self._as_rows(s, self.s_dim).shape[0]
        u = np_random().normal(size=(n, self.a_dim))                               # :350
        (act, nlp), n = self._run(s, u, True)
        act, nlp = self._host(act[0]), self._host(nlp[0])
        return (act[0], nlp[0]) if n == 1 else (act, nlp)
