"""A set of independent policies of any depth, acted on the device in one launch (``saceo_policy_act``).

An expert policy is only ever rolled out (``SAC_exp._collect_expert_data``, ``/root/reference/sac_eo/algs/
SAC_expert.py:156-209``), never trained, so it does not need the two-hidden-layer training engine of ``Population``:
``PolicySet`` holds the flat weights and the normaliser statistics of ``n_agents`` policies (a ``GaussianActor`` or a
``SquashedGaussianActor`` of 1 to 8 hidden layers, widths up to 1024) and answers ``actor_forward`` like a
``Population`` does, so the reference-compatible actor classes and ``common/lockstep.py`` serve it unchanged.  The field
is called ``n_agents`` so that a ``SharedPopulation`` can hold a ``PolicySet`` for the experts of several runs."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import lib as _l


@dataclass(frozen=True)
class PolicySpec:
    n_agents: int
    S: int
    A: int
    hidden: Tuple[int, ...]
    acts: Tuple[str, ...]
    squash: bool = False            # SquashedGaussianActor.sample head instead of GaussianActor._forward + .sample
    per_state_std: bool = True      # outputs 2A (mean, std); else A outputs + a logstd variable [1, A]
    std_mult: float = 1.0           # GaussianActor only
    device: int = 0

    def to_config(self) -> _l.PolicyConfig:
        if len(self.acts) != len(self.hidden):
            raise ValueError("one activation per hidden layer")
        if not 1 <= len(self.hidden) <= _l.POLICY_MAX_HIDDEN:
            raise ValueError(f"a policy has 1 to {_l.POLICY_MAX_HIDDEN} hidden layers (got {len(self.hidden)})")
        c = _l.PolicyConfig()
        c.abi_version, c.device, c.n_policies, c.S, c.A = _l.ABI_VERSION, self.device, self.n_agents, self.S, self.A
        c.n_hidden = len(self.hidden)
        for i, (h, a) in enumerate(zip(self.hidden, self.acts)):
            if a not in _l.ACT_IDS:
                raise ValueError("activations must be tanh, relu or elu")
            c.hidden[i], c.act[i] = int(h), _l.ACT_IDS[a]
        c.squash, c.per_state_std, c.std_mult = int(bool(self.squash)), int(bool(self.per_state_std)), float(self.std_mult)
        return c

    @property
    def Ao(self) -> int:
        return 2 * self.A if self.per_state_std else self.A

    def shapes(self) -> List[Tuple[int, ...]]:
        """Keras ``get_weights()`` shapes ``[W0, b0, ..., Wn, bn (, logstd)]`` (nn_utils.py:86-138, continuous_actors.py:56-57)."""
        dims = [self.S] + [int(h) for h in self.hidden] + [self.Ao]
        out = []
        for i in range(len(dims) - 1):
            out += [(dims[i], dims[i + 1]), (dims[i + 1],)]
        return out + ([] if self.per_state_std else [(1, self.A)])


def policy_layout(spec: PolicySpec) -> Tuple[int, int, int]:
    """(parameter count, per-policy stride, normaliser record stride) - host arithmetic, no GPU."""
    n, s, ns = C.c_int64(), C.c_int64(), C.c_int32()
    _l.check(_l.load().saceo_policy_layout(C.byref(spec.to_config()), C.byref(n), C.byref(s), C.byref(ns)))
    return n.value, s.value, ns.value


class PolicySet:
    """Device tables of ``spec.n_agents`` policies: ``params`` [P, param_stride] (flat Keras order) and ``norm``
    [P, norm_stride] (``s_mean | s_std | act_limit``, identity by default)."""

    def __init__(self, spec: PolicySpec):
        if not torch.cuda.is_available():
            raise _l.SaceoError("sac_expert_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.spec = spec
        self.lib = _l.load()
        self.cfg = spec.to_config()
        self.n_params, self.param_stride, self.norm_stride = policy_layout(spec)
        self.dev = torch.device("cuda", spec.device)
        n, S, A = spec.n_agents, spec.S, spec.A
        self.params = torch.zeros(n, self.param_stride, device=self.dev)
        self.norm = torch.zeros(n, self.norm_stride, device=self.dev)
        self.norm[:, S:2 * S] = 1.0
        self.norm[:, 2 * S:2 * S + A] = 1.0
        self._shapes = spec.shapes()
        self._off = {"s_mean": (0, S), "s_std": (S, S), "act_limit": (2 * S, A)}

    def close(self):
        pass

    def _check_name(self, name):
        if name != "actor":
            raise KeyError(f"a PolicySet holds actors only (got {name!r})")

    def set_net(self, agent: int, name: str, weights: Sequence[np.ndarray]):
        self._check_name(name)
        got = [tuple(np.shape(w)) for w in weights]
        if got != [tuple(s) for s in self._shapes]:
            raise ValueError(f"{name}: weight shapes {got} do not match {self._shapes}")
        flat = np.concatenate([np.asarray(w, np.float32).reshape(-1) for w in weights])
        self.params[agent, :flat.size].copy_(torch.from_numpy(flat))

    def get_net(self, agent: int, name: str) -> List[np.ndarray]:
        self._check_name(name)
        vec = self.params[agent, :self.n_params].cpu().numpy()
        out, o = [], 0
        for sh in self._shapes:
            k = int(np.prod(sh))
            out.append(np.array(vec[o:o + k], np.float32).reshape(sh))
            o += k
        return out

    def set_norm(self, agent: int, **stats):
        """``s_mean``, ``s_std`` (the policy's own observation normaliser) and ``act_limit``; other keys are refused."""
        for key, val in stats.items():
            if key not in self._off:
                raise KeyError(f"a PolicySet normaliser record holds s_mean, s_std and act_limit (got {key!r})")
            off, cnt = self._off[key]
            v = torch.as_tensor(np.broadcast_to(np.asarray(val, np.float32).reshape(-1), (cnt,)).copy())
            self.norm[agent, off:off + cnt].copy_(v)

    def actor_forward(self, obs: torch.Tensor, noise: Optional[torch.Tensor] = None, want_neglogp: bool = False):
        """``expert.sample`` for every policy: ``obs`` [P, rows, S], ``noise`` [P, rows, A] or None (deterministic)
        -> actions [P, rows, A] (device)."""
        if want_neglogp:
            raise NotImplementedError("a PolicySet only acts: neglogp / evaluate are not on the expert path")
        n, S, A = self.spec.n_agents, self.spec.S, self.spec.A
        obs = torch.as_tensor(obs).to(self.dev, torch.float32).contiguous().view(n, -1, S)
        rows = obs.shape[1]
        if noise is not None:
            noise = torch.as_tensor(noise).to(self.dev, torch.float32).contiguous().view(n, rows, A)
        act = torch.empty(n, rows, A, device=self.dev)
        st = torch.cuda.current_stream(self.dev).cuda_stream
        _l.check(self.lib.saceo_policy_act(C.byref(self.cfg), self.params.data_ptr(), self.norm.data_ptr(), obs.data_ptr(),
                                           rows, None if noise is None else noise.data_ptr(), act.data_ptr(), st))
        return act
