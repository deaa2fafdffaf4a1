"""``trajectory_sampler`` with the reference's signature and return tuple
(``/root/reference/sac_eo/common/samplers.py:3-77``): one environment rollout with the current actor.  Host code; the
per-step ``actor.sample`` is the batched device forward (``saceo_actor_forward``)."""
import numpy as np

from .lockstep import run_inline


def trajectory_sampler(env, actor, horizon, s_init=None, eval=False, deterministic=False, corruptor=None):
    return run_inline(trajectory_sampler_steps(env, actor, horizon, s_init, eval, deterministic, corruptor))


def trajectory_sampler_steps(env, actor, horizon, s_init=None, eval=False, deterministic=False, corruptor=None):
    """``trajectory_sampler`` as a generator of its device requests (``common/lockstep.py``); an actor without
    ``_sample_steps`` (any object with the reference's ``sample``) is called directly."""
    sample_steps = getattr(actor, "_sample_steps", None)
    s_traj, a_traj, r_traj, sp_traj, d_traj = [], [], [], [], []
    J_tot = 0.0
    s = env.reset(s_init) if s_init is not None else env.reset()
    for t in range(int(horizon)):
        s_old = s
        a = (yield from sample_steps(s_old, deterministic=deterministic)) if sample_steps is not None \
            else actor.sample(s_old, deterministic=deterministic)
        a = np.asarray(a.numpy())
        s_true, r, d, _ = env.step(actor.clip(a))
        if corruptor is not None:
            s_store = corruptor.corrupt_samples(s_true)
            s = s_store if corruptor.s_noise_type == "all" else s_true
        else:
            s_store = s = s_true
        if eval:
            J_tot += r
        if t == horizon - 1:
            d = False                                   # time-limit truncation is not a terminal state (:52-53)
        s_traj.append(s_old); a_traj.append(a); r_traj.append(r); sp_traj.append(s_store); d_traj.append(d)
        if d:
            break
    out = (np.array(s_traj, np.float32), np.array(a_traj, np.float32), np.array(r_traj, np.float32),
           np.array(sp_traj, np.float32), np.array(d_traj))
    return out + (J_tot,) if eval else out
