"""Entry point for RL training - the reference's ``train.py`` (``/root/reference/sac_eo/train.py``) on the CUDA
path: same ``train(inputs_dict)`` contract (seeds, environments, actor / expert / critics / models, ``init_alg``,
``alg.train``), same seed derivation and multi-run aggregation in ``main``.  Differences: no TensorFlow device setup
(``train.py:29-31``), runs are executed one after the other in this process (one CUDA context; the reference forks one
process per run, :151), and ``--alg_seed`` works (the reference's parser omits it from ``setup_kwargs`` and raises
``KeyError`` at :41).  ``python -m sac_expert_b200.sac_eo.train --env_type synthetic --env_name hopper --actor_squash ...``"""
import copy
import os
import pickle
from datetime import datetime

import numpy as np

from .actors.init_actor import init_actor
from .algs.init_alg import init_alg
from .common.seeding import init_seeds
from .common.train_parser import create_train_parser
from .common.train_utils import gather_inputs, import_inputs, organize_rms_inputs
from .critics.init_critic import init_critics
from .envs import init_env
from .models.init_world_models import init_world_models


def build_run(inputs_dict, population=None, agent=0):
    """Seeds, environments, networks and algorithm of one run (train.py:33-106), in the reference's order, so the run
    consumes the global NumPy stream like the reference.  ``population`` / ``agent``: see ``init_alg``."""
    setup = inputs_dict["setup_kwargs"]
    idx = setup["idx"]
    inputs_dict["alg_kwargs"]["alg_seed"] = setup["algorithm_seed"]
    env_kwargs, actor_kwargs = inputs_dict["env_kwargs"], inputs_dict["actor_kwargs"]
    critic_kwargs, model_kwargs = inputs_dict["critic_kwargs"], inputs_dict["model_kwargs"]
    alg_kwargs, mf_update_kwargs = inputs_dict["alg_kwargs"], inputs_dict["mf_update_kwargs"]

    init_seeds(setup["setup_seed"])
    env, env_eval, env_expert = init_env(**env_kwargs), init_env(**env_kwargs), init_env(**env_kwargs)
    actor = init_actor(env, **actor_kwargs)
    if setup["expert_file"] is not None:
        with open(os.path.join(setup["expert_path"], setup["expert_file"]), "rb") as f:
            import_log = pickle.load(f)[0]
        expert_kwargs = import_log["param"]["actor_kwargs"]
        expert_kwargs["actor_weights"] = import_log["final"]["actor_weights"]
        for k in ("actor_adversary_prob",):
            expert_kwargs.pop(k, None)
        init_expert_rms_stats = organize_rms_inputs(import_log["final"])
    else:
        expert_kwargs = dict(actor_kwargs)
        expert_kwargs["actor_weights"] = None
        init_expert_rms_stats = None
    expert = init_actor(env, **expert_kwargs)
    critics, q_targets, q_critics = init_critics(env, **critic_kwargs)
    models = init_world_models(env, **model_kwargs, model_setup_kwargs=inputs_dict["model_setup_kwargs"])
    init_seeds(setup["eval_seed"], env_eval)
    init_seeds(setup["sim_seed"], env)
    init_seeds(setup["expert_seed"], env_expert)
    return init_alg(idx, env, env_eval, env_expert, actor, critics, q_targets, q_critics, models, alg_kwargs,
                    mf_update_kwargs, expert, init_expert_rms_stats, population, agent)


def train(inputs_dict):
    """Training on given seed (train.py:33-107)."""
    total_timesteps = inputs_dict["alg_kwargs"]["total_timesteps"]
    return build_run(inputs_dict).train(total_timesteps, inputs_dict)


def build_inputs(args):
    """The per-run input dicts of ``main`` (train.py:116-147)."""
    inputs_dict = gather_inputs(args)
    seeds = np.random.SeedSequence(args.seed).generate_state(5)
    per_run = [np.random.SeedSequence(s).generate_state(args.runs + args.runs_start)[args.runs_start:] for s in seeds]
    out = []
    for run in range(args.runs):
        setup = inputs_dict["setup_kwargs"]
        setup["idx"] = run + args.runs_start
        for key, arg, vals in (("setup_seed", args.setup_seed, per_run[0]), ("sim_seed", args.sim_seed, per_run[1]),
                               ("eval_seed", args.eval_seed, per_run[2]), ("expert_seed", args.expert_seed, per_run[3]),
                               ("algorithm_seed", args.alg_seed, per_run[4])):
            setup[key] = int(vals[run]) if arg is None else arg
        inputs_dict = import_inputs(inputs_dict)
        out.append(copy.deepcopy(inputs_dict))
    return out


def save_outputs(args, log_names):
    """Aggregates the per-run checkpoint files into one pickle and removes them (train.py:159-194); returns its path."""
    outputs = []
    os.makedirs(args.save_path, exist_ok=True)
    for name in log_names:                           # aggregate the per-run checkpoint files (train.py:159-168)
        with open(os.path.join(args.save_path, name), "rb") as f:
            outputs.append(pickle.load(f))
    save_env = args.env_name.split("-")[0].lower()
    if args.task_name is not None:
        save_env = "%s_%s" % (save_env, args.task_name.lower())
    parts = [args.env_type.lower(), save_env, args.alg_type, args.mf_algo] + ([args.save_file] if args.save_file else []) \
        + [datetime.today().strftime("%m%d%y_%H%M%S")]
    save_filefull = os.path.join(args.save_path, "_".join(parts))
    with open(save_filefull, "wb") as f:
        pickle.dump(outputs, f)
    for name in log_names:                           # remove the temporary per-run files (train.py:189-194)
        fn = os.path.join(args.save_path, name)
        if os.path.exists(fn):
            os.remove(fn)
    return save_filefull


def main(argv=None):
    start = datetime.now()
    args = create_train_parser().parse_args(argv)
    inputs_list = build_inputs(args)
    save_filefull = save_outputs(args, [train(inp) for inp in inputs_list])
    end = datetime.now()
    print("Time Elapsed: %s" % (end - start))
    return save_filefull


if __name__ == "__main__":
    main()
