"""Device requests of the training loop and the two schedules that serve them.

The environment loop (``SAC.train`` and the ``SAC_exp`` / ``BC`` hooks) is written once, as generators: wherever the
reference calls a network, it ``yield`` s a ``Request`` (act, model evaluation, update, replay append, model fit,
optimiser reset) and receives that request's result.  ``run_inline`` serves one loop on its own, one request at a time
- the class interface and ``train.py``.  ``run_lockstep`` drives R loops whose networks are agents ``0 .. R-1`` of shared
populations: it resumes every run up to its next request, checks that the R requests agree in kind and shape, and
issues ONE batched population call for all of them.

Every host draw of the loop goes through ``np_random()``: the global NumPy generator outside a lockstep schedule, the
run's own ``RandomState`` inside it, so each run consumes exactly the stream its sequential run would."""
import time

import numpy as np
import torch

_stream = np.random


def np_random():
    """The NumPy random stream of the run being resumed (``numpy.random`` itself outside ``run_lockstep``)."""
    return _stream


class LockstepError(RuntimeError):
    """The runs of one lockstep schedule stopped issuing the same device requests."""


class Request:
    """One device call of one run: ``kind`` selects the population entry point, ``shape`` is what must agree across
    the runs of a lockstep schedule, ``data`` holds this run's host inputs."""
    __slots__ = ("kind", "pop", "agent", "shape", "data")

    def __init__(self, kind, pop, agent, shape, **data):
        self.kind, self.pop, self.agent, self.shape, self.data = kind, pop, agent, tuple(shape), data

    def __repr__(self):
        return "%s%s" % (self.kind, self.shape)


def _stack(reqs, key, dtype=np.float32):
    return torch.from_numpy(np.stack([np.asarray(r.data[key], dtype) for r in reqs]))


def _act(pop, reqs):
    noise = None if reqs[0].data["noise"] is None else _stack(reqs, "noise")
    act = pop.actor_forward(_stack(reqs, "obs"), noise).cpu()
    return list(act)


def _model(pop, reqs):
    return list(pop.model_eval(_stack(reqs, "obs"), _stack(reqs, "act")).cpu())


def _update(pop, reqs):
    exp = [r for r in reqs if r.data["expert"] is not None]
    if len(exp) > 1 and len(exp) == pop.spec.n_agents:
        pop.set_expert_all(np.stack([r.data["expert"][0] for r in exp]), np.stack([r.data["expert"][1] for r in exp]))
    else:
        for r in exp:
            pop.set_expert(r.agent, *r.data["expert"])
    for r in reqs:                                   # changes once per episode at most
        if r.data["eps"] is not None:
            pop.set_hyper(r.agent, eps=r.data["eps"])
    d0 = reqs[0].data
    idx = None if d0["idx"] is None else np.stack([r.data["idx"] for r in reqs])
    perm = None if d0["perm"] is None else np.stack([r.data["perm"] for r in reqs])
    pop.set_draws(idx, np.stack([r.data["noise"] for r in reqs]), perm)
    if d0["bc"]:
        losses = pop.bc_update(1, use_device_rng=False)
    else:
        losses = pop.update(1, num_timesteps=d0["num_timesteps"], use_device_rng=False)
    return list(losses.cpu().numpy())


def _append(pop, reqs):
    if len(reqs) == 1:                               # one agent's buffer: the per-agent append
        pop.append_rows(reqs[0].agent, *reqs[0].data["rows"])
    else:
        pop.append_all(*[np.stack([r.data["rows"][k] for r in reqs]) for k in range(5)])
    return [None] * len(reqs)


def _fit(pop, reqs):
    losses = pop.model_fit(np.stack([r.data["idx"] for r in reqs], 1))      # [steps, n_agents, num_models, batch]
    return [losses[:, i:i + 1] for i in range(len(reqs))]


def _reset_fit(pop, reqs):
    pop.reset_model_optimizer()
    return [None] * len(reqs)


_RUN = dict(act=_act, model=_model, update=_update, append=_append, fit=_fit, reset_fit=_reset_fit)


def execute(reqs):
    """Serves the requests of every agent of one population (or one agent's replay append) with one population call;
    returns the per-request results in order."""
    pop = reqs[0].pop
    if len(reqs) != pop.spec.n_agents and not (len(reqs) == 1 and reqs[0].kind == "append"):
        raise ValueError("the class interface drives a single-agent population; use Population for many agents")
    return _RUN[reqs[0].kind](pop, reqs)


def run_inline(steps):
    """Runs one loop to completion, serving each request on its own; returns the loop's return value."""
    try:
        req = next(steps)
        while True:
            req = steps.send(execute([req])[0])
    except StopIteration as stop:
        return stop.value


def inline(steps_method):
    """The direct-call form of a generator method: ``_update = inline(_update_steps)`` runs ``self._update_steps(...)``
    (looked up by name, so subclass overrides apply) with ``run_inline``."""
    name = steps_method.__name__

    def call(self, *args, **kwargs):
        return run_inline(getattr(self, name)(*args, **kwargs))
    call.__doc__ = steps_method.__doc__
    return call


class _TimedStream:
    """A run's ``RandomState`` that adds the time spent in its draws to ``timings['draws']``."""

    def __init__(self, rs, timings):
        self._rs, self._t = rs, timings

    def __getattr__(self, name):
        fn = getattr(self._rs, name)

        def timed(*args, **kwargs):
            t0 = time.perf_counter()
            try:
                return fn(*args, **kwargs)
            finally:
                self._t["draws"] += time.perf_counter() - t0
        return timed


def run_lockstep(runs, names, streams, timings=None):
    """Drives the generators ``runs`` in lockstep.  Run ``r`` draws from ``streams[r]`` (a ``numpy.random.RandomState``)
    and its requests must target agent ``r`` of each population they use.  Every round resumes each run up to its next
    request; the R requests must have the same kind, population and shape, otherwise ``LockstepError`` names the first
    run that differs from run ``names[0]``.  The round is then served by one batched call.  Returns the runs' return
    values.  ``timings`` (a dict) receives the wall time spent in the runs' host code (``host``, which contains
    ``draws``) and in the batched calls (``device``, which ends in a device-to-host copy of the results)."""
    global _stream
    R = len(runs)
    if timings is not None:
        timings.update(host=0.0, device=0.0, draws=0.0, rounds=0)
        streams = [_TimedStream(s, timings) for s in streams]
    sent, out = [None] * R, [None] * R
    try:
        while True:
            t0 = time.perf_counter()
            reqs, done = [], []
            for r, gen in enumerate(runs):
                _stream = streams[r]
                try:
                    reqs.append(gen.send(sent[r]))
                except StopIteration as stop:
                    out[r] = stop.value
                    done.append(r)
                    reqs.append(None)
            _stream = np.random
            t1 = time.perf_counter()
            if len(done) == R:
                break
            if done:
                live = next(r for r in range(R) if reqs[r] is not None)
                raise LockstepError("run %s finished while run %s requested %r: the runs fell out of lockstep"
                                    % (names[done[0]], names[live], reqs[live]))
            a = reqs[0]
            for r, b in enumerate(reqs):
                if b.kind != a.kind or b.pop is not a.pop or b.shape != a.shape or b.agent != r:
                    raise LockstepError("run %s requested %r (agent %d) while run %s requested %r: the runs fell out of "
                                        "lockstep" % (names[r], b, b.agent, names[0], a))
            sent = execute(reqs)
            if timings is not None:
                t2 = time.perf_counter()
                timings["host"] += t1 - t0
                timings["device"] += t2 - t1
                timings["rounds"] += 1
    finally:
        _stream = np.random
    return out
