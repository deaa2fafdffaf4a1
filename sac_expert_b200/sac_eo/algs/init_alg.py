"""``init_alg`` with the reference's signature (``/root/reference/sac_eo/algs/init_alg.py:9-34``).  Only the
algorithms whose update is the accelerated hot path are available.  ``population`` / ``agent``: bind the algorithm
to agent ``agent`` of the population a ``SharedPopulation`` holds instead of a one-agent population of its own."""
from ..actors.continuous_actors import SquashedGaussianActor
from .SAC import SAC
from .BC import BC
from .SAC_expert import SAC_exp


def init_alg(idx, env, env_eval, env_expert, actor, critics, q_targets, q_critics, models, alg_kwargs,
             mf_update_kwargs, expert, init_expert_rms_stats, population=None, agent=0):
    alg_type = alg_kwargs["alg_type"]
    if alg_type in ("sac", "sac_imit", "bc") and not isinstance(actor, SquashedGaussianActor):
        raise ValueError("alg_type %r trains a SquashedGaussianActor: pass --actor_squash (a GaussianActor is only "
                         "supported as the expert policy)" % alg_type)
    if alg_type == "sac":
        return SAC(idx, env, env_eval, actor, critics, q_targets, q_critics, models, alg_kwargs, mf_update_kwargs,
                   population, agent)
    if alg_type == "sac_imit":
        return SAC_exp(idx, env, env_eval, env_expert, actor, expert, init_expert_rms_stats, critics, q_targets,
                       q_critics, models, alg_kwargs, mf_update_kwargs, population, agent)
    if alg_type == "bc":
        return BC(idx, env, env_eval, env_expert, actor, expert, init_expert_rms_stats, critics, q_targets, q_critics,
                  models, alg_kwargs, mf_update_kwargs, population, agent)
    if alg_type == "mbrl":
        raise ValueError("alg_type 'mbrl' (on-policy model-based TRPO/PPO) is outside the accelerated hot path (SURVEY.md §2)")
    raise ValueError("invalid alg_type")
