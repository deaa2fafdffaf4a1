"""fp64 restatement of ``expert.sample`` for actors of any depth - the checker of ``saceo_policy_act``.  TEST
INFRASTRUCTURE ONLY, like ``oracle/sac_eo_oracle.py``, whose building blocks (``mlp``, ``normalize``, the logstd
constants) it reuses unchanged.  ``oracle.head`` and ``oracle.gaussian_forward`` read the state-independent logstd
variable at ``theta[6]``, the position it has at two hidden layers; here it sits after the ``n_hidden + 1`` dense
layers, ``theta[2 (n_hidden + 1)]``.  Otherwise the operations and their order are those of ``head`` / ``gaussian_sample``,
so at two hidden layers ``policy_sample`` returns exactly what they return (tests/test_policy_host.py)."""
import math
from typing import Dict, Optional, Sequence

import torch

from oracle.sac_eo_oracle import MAX_LOG_STD, MIN_LOG_STD, NetCfg, mlp, normalize

Tensor = torch.Tensor


def _out(cfg: NetCfg, theta: Sequence[Tensor], s_: Tensor, st: Dict):
    dt = s_.dtype
    out = mlp(theta, normalize(s_, st["s_mean"], st["s_std"]).to(dt), cfg.actor_acts)
    if cfg.per_state_std:
        mean, o2 = torch.split(out, cfg.A, dim=-1)
        return mean, o2
    return out, theta[2 * (len(cfg.actor_hidden) + 1)] * torch.ones_like(out)


def gaussian_forward_any_depth(cfg: NetCfg, theta: Sequence[Tensor], s_: Tensor, st: Dict):
    """``GaussianActor._forward`` (continuous_actors.py:74-100): softplus std + logstd_init, floor log(1e-3)."""
    mean, raw = _out(cfg, theta, s_, st)
    if cfg.per_state_std:
        logstd = torch.log(torch.nn.functional.softplus(raw))
        logstd_init = math.log(cfg.std_mult) - math.log(math.log(2.0))   # :39-41
    else:
        logstd = raw
        logstd_init = math.log(cfg.std_mult)                             # :43-44
    logstd = logstd + logstd_init
    return mean, torch.maximum(logstd, torch.as_tensor(math.log(1e-3), dtype=s_.dtype))


def policy_sample(cfg: NetCfg, theta: Sequence[Tensor], s_: Tensor, u: Optional[Tensor], st: Dict, squash: bool) -> Tensor:
    """``expert.sample(s, deterministic=u is None)`` for an actor of ``len(cfg.actor_hidden)`` hidden layers:
    ``SquashedGaussianActor.sample`` (continuous_actors.py:270-306: logstd clipped to [-5, 2], ``act_limit tanh(z)``)
    when ``squash``, else ``GaussianActor.sample`` (:103-123: ``mean + exp(logstd) u``, no squash, no clip)."""
    if not squash:
        mean, logstd = gaussian_forward_any_depth(cfg, theta, s_, st)
        return mean if u is None else mean + torch.exp(logstd) * torch.as_tensor(u).to(mean.dtype)
    dt = s_.dtype
    mean, logstd = _out(cfg, theta, s_, st)
    logstd = torch.clamp(logstd, MIN_LOG_STD, MAX_LOG_STD)
    z = mean if u is None else mean + torch.exp(logstd) * u.to(dt)
    return torch.as_tensor(st["act_limit"], dtype=dt) * torch.tanh(z)
