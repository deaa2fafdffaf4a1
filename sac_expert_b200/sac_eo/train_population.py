"""``train.py`` with every run of the invocation trained at once as one device population.

Same command line, per-run seed derivation (``build_inputs``), checkpoint files and aggregated pickle as
``sac_expert_b200.sac_eo.train``, and run ``r`` computes exactly what sequential run ``r`` computes.  The R runs are
built one after the other with the code ``train.train`` uses; their networks and replay buffers are then agent ``r`` of
one shared ``Population`` (the experts of ``sac_imit`` / ``bc``: of one shared expert population).  The runs' training
loops, the unchanged ``alg.train`` loop, advance in lockstep (``common/lockstep.py``): every device call of a step -
acting, update, replay append, model fit and evaluation, expert rollout - is ONE batched population call for all R runs,
and run ``r`` draws from its own NumPy stream.  ``--cores`` (the reference's process-pool size) has no meaning here.

Supported: ``--alg_type sac | sac_imit | bc`` on ``--env_type synthetic``, like ``train.py``; the synthetic environment
ends episodes only at the horizon, so the runs stay in lockstep.  ``LockstepError`` names the run whose device request
differs if they ever do not.  ``python -m sac_expert_b200.sac_eo.train_population --env_type synthetic --runs 8 ...``"""
from datetime import datetime

import numpy as np

from ..population import SharedPopulation
from .algs.SAC_expert import SAC_exp
from .common.lockstep import run_lockstep
from .common.train_parser import create_train_parser
from .train import build_inputs, build_run, save_outputs


def train_population(inputs_list, timings=None):
    """Trains the runs of ``inputs_list`` as agents ``0 .. R-1`` of shared populations; returns their checkpoint names.
    ``timings``: see ``run_lockstep``."""
    R = len(inputs_list)
    pop, experts = SharedPopulation(R), SharedPopulation(R)
    algs, streams = [], []
    for r, inp in enumerate(inputs_list):
        alg = build_run(inp, pop, r)
        if isinstance(alg, SAC_exp):
            alg._bind_expert(experts, r)
        algs.append(alg)
        stream = np.random.RandomState()      # run r continues the global stream where its construction left it
        stream.set_state(np.random.get_state())
        streams.append(stream)
    runs = [alg.train_steps(inp["alg_kwargs"]["total_timesteps"], inp) for alg, inp in zip(algs, inputs_list)]
    return run_lockstep(runs, [inp["setup_kwargs"]["idx"] for inp in inputs_list], streams, timings)


def main(argv=None, timings=None):
    start = datetime.now()
    args = create_train_parser().parse_args(argv)
    save_filefull = save_outputs(args, train_population(build_inputs(args), timings))
    end = datetime.now()
    print("Time Elapsed: %s" % (end - start))
    return save_filefull


if __name__ == "__main__":
    main()
