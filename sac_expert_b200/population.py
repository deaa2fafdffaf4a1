"""Population of independent SAC / SAC-EO agents resident on one B200.

This is the device-side state the reference keeps in ``tf.Variable`` s, Keras optimizer slots and
NumPy buffers (``/root/reference/sac_eo/algs/SAC_expert.py:28-116``), batched over ``n_agents``
(seeds x hyper-parameters) and laid out as flat per-agent tables (include/saceo.h).  PyTorch only
supplies the device allocations (``tensor.data_ptr()``) and the stream; every computation goes
through the C ABI in ``lib.py``.  ``n_agents == 1`` is the reference's single-agent behaviour and is
what the class mirrors in ``sac_expert_b200/sac_eo`` use.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import lib as _l
from .policy import PolicySet, PolicySpec

LOSS_NAMES = ("q1_loss", "q2_loss", "pi_loss", "mse_loss", "p_loss", "alpha_loss", "alpha", "epsilon")
HYPER_NAMES = ("gamma", "tau", "lr_q", "lr_pi", "lr_alpha", "eps", "target_entropy", "damp")


@dataclass
class PopulationSpec:
    n_agents: int
    S: int
    A: int
    actor_hidden: Tuple[int, int] = (256, 256)
    critic_hidden: Tuple[int, int] = (256, 256)
    model_hidden: Tuple[int, int] = (512, 512)
    actor_acts: Tuple[str, str] = ("relu", "relu")
    critic_acts: Tuple[str, str] = ("relu", "relu")
    model_acts: Tuple[str, str] = ("relu", "relu")
    per_state_std: bool = True
    separate_reward_nn: bool = False
    reward_hidden: Optional[Tuple[int, int]] = None     # separate_reward_nn: the reward network (default: model_hidden / model_acts)
    reward_acts: Optional[Tuple[str, str]] = None
    num_models: int = 2            # 0 = plain SAC
    delta_clip_pred: float = 0.0
    B: int = 256
    E: int = 20
    target_update_int: int = 1
    replay_capacity: int = 100_000
    fvp_rows: int = 0
    std_mult: float = 1.0
    gemm_mode: int = _l.GEMM_TCGEN05_BF16X3   # GEMM_FP32_SIMT: exact-fp32 CUDA-core engine (debugging / bit-faithful parity)
    tc_variant: int = 0            # tcgen05 tile variant (0: 128x256 1 CTA/SM, 1: 128x128 2 CTAs/SM)
    fuse_forward: bool = True      # fused 3-layer tcgen05 forward (activations resident in TMEM)
    fuse_backward: bool = True     # fused tcgen05 gradient chain dOut -> dH2 -> dH1 -> dXa
    use_graph: bool = True         # one update = one CUDA-graph replay
    ws_kernels: bool = True        # warp-specialised TMA-fed fused kernels on optimiser-maintained weight planes (round 2)
    fork_actor: bool = True        # critic-independent half of the actor phase on a second stream (needs ws_kernels)
    device: int = 0

    def to_config(self) -> _l.Config:
        c = _l.Config()
        c.abi_version = _l.ABI_VERSION
        c.device = self.device
        c.n_agents = self.n_agents
        c.S, c.A = self.S, self.A
        for i in range(2):
            c.actor_hidden[i] = self.actor_hidden[i]
            c.critic_hidden[i] = self.critic_hidden[i]
            c.model_hidden[i] = self.model_hidden[i]
            for dst, src in ((c.actor_act, self.actor_acts), (c.critic_act, self.critic_acts),
                             (c.model_act, self.model_acts)):
                if src[i] not in _l.ACT_IDS:
                    raise ValueError("activations must be tanh, relu or elu")   # nn_utils.py:18
                dst[i] = _l.ACT_IDS[src[i]]
        c.per_state_std = int(self.per_state_std)
        c.separate_reward_nn = int(self.separate_reward_nn)
        c.num_models = self.num_models
        c.delta_clip_pred = float(self.delta_clip_pred or 0.0)
        c.B, c.E = self.B, self.E
        c.target_update_int = self.target_update_int
        c.replay_capacity = self.replay_capacity
        c.fvp_rows = self.fvp_rows
        c.std_mult = self.std_mult
        c.gemm_mode = self.gemm_mode
        c.use_graph = int(self.use_graph)
        c.reserved[0] = self.tc_variant
        c.reserved[1] = 0 if self.fuse_forward else 1
        c.reserved[2] = 0 if self.fuse_backward else 1
        c.reserved[5] = 0 if self.ws_kernels else 1
        c.reserved[6] = 0 if self.fork_actor else 1
        return c


def net_shapes(n_in: int, hidden: Sequence[int], n_out: int) -> List[Tuple[int, ...]]:
    """Keras ``get_weights()`` shapes ``[W0,b0,W1,b1,W2,b2]`` (nn_utils.py:86-138)."""
    return [(n_in, hidden[0]), (hidden[0],), (hidden[0], hidden[1]), (hidden[1],), (hidden[1], n_out), (n_out,)]


def pack_flat(ws: Sequence[np.ndarray]) -> np.ndarray:
    """``list_to_flat`` (nn_utils.py:177-182)."""
    return np.concatenate([np.asarray(w, np.float32).reshape(-1) for w in ws])


def unpack_flat(vec: np.ndarray, shapes: Sequence[Tuple[int, ...]]) -> List[np.ndarray]:
    """``flat_to_list`` (nn_utils.py:162-175)."""
    out, o = [], 0
    for sh in shapes:
        n = int(np.prod(sh))
        out.append(np.array(vec[o:o + n], np.float32).reshape(sh))
        o += n
    return out


def backtrack_population(trial, n: int, kl_maxfactor: float, delta: float):
    """Control flow of ``TRPO._backtrack`` (trpo.py:251-301) for ``n`` agents at once, each with its own accept /
    shrink decisions.  ``trial(adj[n]) -> (stats[n, >=3], improve[n])`` applies ``theta_k + adj * eta * v`` for every
    agent and evaluates it (``stats[:, 1]`` = kl, ``stats[:, 2]`` = tv).  An agent accepts the first trial whose
    ``kl <= kl_maxfactor * delta`` and ``improve >= 0`` and keeps that ``adj`` from then on; otherwise its ``adj`` is
    divided by sqrt(2), at most ten times; an agent that has not accepted after the tenth shrink gets ``adj = 0`` (its
    old parameters).  Returns (adj, stats, improve, tv_pre, kl_pre) at the final parameters.  Pure host logic."""
    adj = np.ones(n)
    stats, improve = trial(adj)
    tv_pre, kl_pre = stats[:, 2].copy(), stats[:, 1].copy()
    done = np.zeros(n, bool)
    for _ in range(10):
        bad = ~done & ((stats[:, 1] > kl_maxfactor * delta) | (improve < 0))
        done |= ~bad
        if not bad.any():
            break
        adj = np.where(bad, adj / np.sqrt(2), adj)
        stats, improve = trial(adj)
    else:
        adj = np.where(done, adj, 0.0)                        # no policy update for the agents still failing
        stats, improve = trial(adj)
    return adj, stats, improve, tv_pre, kl_pre


class _DevBuf:
    """Zero-copy view of a library-owned device buffer through ``__cuda_array_interface__``."""

    def __init__(self, ptr: int, shape: Tuple[int, ...], typestr: str):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


class _Tables(dict):
    """The per-agent device tables by name.  Handing out a weight table (``actor``, ``q``, ``qt``) may be followed by a
    write the library cannot see (``tensor.copy_``, indexing assignment), so every such access marks the library's
    fp16 weight-plane images stale; they are rebuilt before the next kernel that reads them (``saceo_weights_changed``).
    The hot loop never looks the tables up, so it never pays for this."""
    _WEIGHTS = ("actor", "q", "qt")

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.dirty = True

    def __getitem__(self, key):
        if key in self._WEIGHTS:
            self.dirty = True
        return super().__getitem__(key)

    def items(self):
        self.dirty = True
        return super().items()

    def values(self):
        self.dirty = True
        return super().values()


class Population:
    def __init__(self, spec: PopulationSpec):
        if not torch.cuda.is_available():
            raise _l.SaceoError("sac_expert_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.spec = spec
        self.lib = _l.load()
        self.cfg = spec.to_config()
        self.L = _l.query_layout(self.cfg)
        self.dev = torch.device("cuda", spec.device)
        self.stream = torch.cuda.Stream(self.dev)
        n, L = spec.n_agents, self.L
        z = lambda *sh, dt=torch.float32: torch.zeros(*sh, dtype=dt, device=self.dev)
        self.t: Dict[str, torch.Tensor] = _Tables(
            actor=z(n, L.na_stride), actor_m=z(n, L.na_stride), actor_v=z(n, L.na_stride),
            q=z(n, 2, L.nc_stride), q_m=z(n, 2, L.nc_stride), q_v=z(n, 2, L.nc_stride), qt=z(n, 2, L.nc_stride),
            model=z(n, 2, L.nm_stride),
            alpha=z(n), alpha_m=z(n), alpha_v=z(n), adam_t=z(n, 4, dt=torch.int32),
            norm=z(n, L.norm_stride), hyper=z(n, L.hyper_stride),
            replay=z(n, spec.replay_capacity, L.row_words),
            replay_size=z(n, dt=torch.int32), replay_start=z(n, dt=torch.int32),
            expert_s=z(n, max(spec.E, 1), spec.S), expert_sp=z(n, max(spec.E, 1), spec.S),
        )
        if spec.fvp_rows > 0:
            self.t["fvp_states"] = z(n, spec.fvp_rows, spec.S)
        # identity normalisers by default (RunningNormalizer.__init__, normalizer.py:17-24)
        nm = self.t["norm"]
        for off, cnt in ((L.off_s_std, spec.S), (L.off_a_std, spec.A), (L.off_ret_std, 1), (L.off_m_s_std, spec.S),
                         (L.off_m_a_std, spec.A), (L.off_m_d_std, spec.S), (L.off_act_limit, spec.A)):
            nm[:, off:off + cnt] = 1.0
        self.shapes = dict(
            actor=net_shapes(spec.S, spec.actor_hidden, L.Ao) + ([] if spec.per_state_std else [(1, spec.A)]),
            q=net_shapes(spec.S + spec.A, spec.critic_hidden, 1),
            model=net_shapes(spec.S + spec.A, spec.model_hidden, L.model_out),
            reward=net_shapes(spec.S + spec.A, tuple(spec.reward_hidden or spec.model_hidden), 1),
        )
        self._host_size = np.zeros(n, np.int64)
        self._host_start = np.zeros(n, np.int64)
        if spec.separate_reward_nn and spec.num_models > 0:      # reward networks: fitted by model_fit, unused by the update
            nr = sum(int(np.prod(sh)) for sh in self.shapes["reward"])
            self.nr_stride = (nr + 31) // 32 * 32
            self.t["reward"] = torch.zeros(n, 2, self.nr_stride, device=self.dev)
        self.ctx = C.c_void_p()
        torch.cuda.synchronize(self.dev)
        _l.check(self.lib.saceo_create(C.byref(self.cfg), C.byref(self.ctx)))
        self._bind()
        self.losses = z(n, L.n_losses)
        self.model_batch = None          # set by fit_bind
        self._pin_idx = None
        self._pin_exp = None
        self._pin_loss = None

    # ------------------------------------------------------------------ plumbing
    def _bind(self):
        tb = _l.Tables()
        for name, _ in _l.Tables._fields_:
            tens = self.t.get(name)
            setattr(tb, name, tens.data_ptr() if tens is not None else None)
        _l.check(self.lib.saceo_bind(self.ctx, C.byref(tb)))

    def close(self):
        if getattr(self, "ctx", None) and self.ctx.value:
            torch.cuda.synchronize(self.dev)
            self.lib.saceo_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _enter(self):
        if self.t.dirty:          # a weight table was handed out since the last call: the weight planes may be stale
            self.lib.saceo_weights_changed(self.ctx)
            self.t.dirty = False
        self.stream.wait_stream(torch.cuda.current_stream(self.dev))
        return self.stream.cuda_stream

    def _exit(self):
        torch.cuda.current_stream(self.dev).wait_stream(self.stream)

    def debug(self, name: str, dtype=torch.float32) -> torch.Tensor:
        """View of a named library workspace buffer (tests / inspection)."""
        nb = C.c_int64()
        ptr = self.lib.saceo_debug_ptr(self.ctx, name.encode(), C.byref(nb))
        if not ptr:
            raise KeyError(name)
        item = torch.empty((), dtype=dtype).element_size()
        ts = {torch.float32: "<f4", torch.int64: "<i8", torch.int32: "<i4", torch.float64: "<f8"}[dtype]
        return torch.as_tensor(_DevBuf(ptr, (nb.value // item,), ts), device=self.dev)

    @property
    def launches(self) -> int:
        return int(self.lib.saceo_launch_count(self.ctx))

    # ------------------------------------------------------------------ state in / out
    def _net_table(self, name: str) -> Tuple[torch.Tensor, str, Optional[int]]:
        if name == "actor":
            return self.t["actor"], "actor", None
        if name in ("q1", "q2"):
            return self.t["q"], "q", int(name[1]) - 1
        if name in ("t1", "t2"):
            return self.t["qt"], "q", int(name[1]) - 1
        if name in ("m1", "m2"):
            return self.t["model"], "model", int(name[1]) - 1
        if name in ("r1", "r2"):      # reward networks of the models (separate_reward_nn, bound by fit_bind)
            return self.t["reward"], "reward", int(name[1]) - 1
        raise KeyError(name)

    def set_net(self, agent: int, name: str, weights: Sequence[np.ndarray], table: Optional[str] = None):
        tab, kind, net = self._net_table(name)
        if table is not None:   # Adam slot tables share the layout of their network
            tab = self.t[table]
        flat = pack_flat(weights)
        shapes = self.shapes[kind]
        if flat.size != sum(int(np.prod(s)) for s in shapes):
            raise ValueError(f"{name}: expected shapes {shapes}")
        dst = tab[agent] if net is None else tab[agent, net]
        dst[:flat.size].copy_(torch.from_numpy(flat))

    def get_net(self, agent: int, name: str, table: Optional[str] = None) -> List[np.ndarray]:
        tab, kind, net = self._net_table(name)
        if table is not None:
            tab = self.t[table]
        src = tab[agent] if net is None else tab[agent, net]
        return unpack_flat(src.detach().cpu().numpy(), self.shapes[kind])

    def set_norm(self, agent: int, **stats):
        """Normaliser record: s_mean,s_std,a_mean,a_std,ret_std and the model set m_* (normalizer.py)."""
        L, row = self.L, self.t["norm"][agent]
        for key, val in stats.items():
            off = getattr(L, "off_" + key)
            v = torch.as_tensor(np.atleast_1d(np.asarray(val, np.float32)))
            row[off:off + v.numel()].copy_(v)

    def set_hyper(self, agent: int, **hy):
        row = self.t["hyper"][agent]
        for key, val in hy.items():
            row[HYPER_NAMES.index(key)] = float(val)

    def load_agent(self, agent: int, st: Dict, hyper: Dict):
        """Loads one agent from the NumPy problem dict the oracle builders produce."""
        for name in ("actor", "q1", "q2", "t1", "t2"):
            self.set_net(agent, name, st[name])
        if self.spec.num_models > 0:
            for name in ("m1", "m2")[: max(self.spec.num_models, 1)]:
                self.set_net(agent, name, st[name])
        self.t["alpha"][agent] = float(st["alpha"])
        for k, (tm, tv) in (("actor", ("actor_m", "actor_v")), ("q1", ("q_m", "q_v")), ("q2", ("q_m", "q_v"))):
            ad = st.get("adam_" + k)
            if ad is not None:
                self.set_net(agent, k, ad["m"], table=tm)
                self.set_net(agent, k, ad["v"], table=tv)
                self.t["adam_t"][agent, {"q1": 0, "q2": 1, "actor": 2}[k]] = int(ad["t"])
        ad = st.get("adam_alpha")
        if ad is not None:
            self.t["alpha_m"][agent] = float(ad["m"])
            self.t["alpha_v"][agent] = float(ad["v"])
            self.t["adam_t"][agent, 3] = int(ad["t"])
        self.set_norm(agent, **{k: st[k] for k in ("s_mean", "s_std", "a_mean", "a_std", "ret_std", "m_s_mean",
                                                    "m_s_std", "m_a_mean", "m_a_std", "m_d_mean", "m_d_std",
                                                    "act_limit") if k in st})
        self.set_hyper(agent, **{k: hyper[k] for k in HYPER_NAMES if k in hyper})

    # ------------------------------------------------------------------ replay / expert rows
    def pack_rows(self, s, a, r, sp, d) -> np.ndarray:
        """Host-side AoS packing of replay rows: [s | a | sp | r | pad | d(f64) | pad]."""
        L = self.L
        n = len(r)
        rows = np.zeros((n, L.row_words), np.float32)
        rows[:, L.off_s:L.off_s + self.spec.S] = np.asarray(s, np.float32).reshape(n, -1)
        rows[:, L.off_a:L.off_a + self.spec.A] = np.asarray(a, np.float32).reshape(n, -1)
        rows[:, L.off_sp:L.off_sp + self.spec.S] = np.asarray(sp, np.float32).reshape(n, -1)
        rows[:, L.off_r] = np.asarray(r, np.float32)
        rows[:, L.off_d:L.off_d + 2] = np.asarray(d, np.float64).reshape(n, 1).view(np.float32)
        return rows

    def append_rows(self, agent: int, s, a, r, sp, d):
        """``TrajectoryBuffer.add`` (buffers.py:41-71) on the device table: append, and when the
        capacity is exceeded keep the LAST ``capacity`` rows (ring; logical index 0 = oldest)."""
        rows = self.pack_rows(s, a, r, sp, d)
        cap = self.spec.replay_capacity
        if len(rows) > cap:
            rows = rows[-cap:]
        size, start = int(self._host_size[agent]), int(self._host_start[agent])
        pos = (start + size) % cap
        first = min(len(rows), cap - pos)
        tab = self.t["replay"][agent]
        tab[pos:pos + first].copy_(torch.from_numpy(rows[:first]))
        if first < len(rows):
            tab[:len(rows) - first].copy_(torch.from_numpy(rows[first:]))
        over = max(0, size + len(rows) - cap)
        self._host_size[agent] = min(cap, size + len(rows))
        self._host_start[agent] = (start + over) % cap
        self.t["replay_size"][agent] = int(self._host_size[agent])
        self.t["replay_start"][agent] = int(self._host_start[agent])

    def append_all(self, s, a, r, sp, d):
        """``TrajectoryBuffer.add`` for EVERY agent in one device call (buffers.py:41-71; the per-step adds of the
        environment loop, SAC_expert.py:793-801): ``s, sp`` [n, k, S], ``a`` [n, k, A], ``r, d`` [n, k].  The packed rows
        travel through one pinned staging buffer and one H2D copy; the ring arithmetic (append behind the newest row,
        overwrite the oldest when full = keep the last ``capacity`` rows) runs on the device (``saceo_replay_append``).
        No host synchronisation; the host mirrors of size / start are advanced with the same arithmetic."""
        n, cap = self.spec.n_agents, self.spec.replay_capacity
        r = np.asarray(r, np.float32).reshape(n, -1)
        k = r.shape[1]
        if k < 1 or k > cap:
            raise ValueError("append_all: rows per agent must be in [1, replay_capacity]")
        rows = self.pack_rows(np.asarray(s).reshape(n * k, -1), np.asarray(a).reshape(n * k, -1), r.reshape(-1),
                              np.asarray(sp).reshape(n * k, -1), np.asarray(d).reshape(-1))
        pin = getattr(self, "_pin_rows", None)
        if pin is None or pin.shape[0] < n * k:
            self._pin_rows = pin = torch.empty(n * k, self.L.row_words, pin_memory=True)
            self._dev_rows = torch.empty(n * k, self.L.row_words, device=self.dev)
        pin[: n * k].numpy()[...] = rows
        st = self._enter()
        with torch.cuda.stream(self.stream):
            self._dev_rows[: n * k].copy_(pin[: n * k], non_blocking=True)
        _l.check(self.lib.saceo_replay_append(self.ctx, self._dev_rows.data_ptr(), k, st))
        self._exit()
        tot = self._host_size + k
        over = np.maximum(tot - cap, 0)
        self._host_size[:] = np.minimum(tot, cap)
        self._host_start[:] = (self._host_start + over) % cap

    def set_expert(self, agent: int, sE, spE):
        self.t["expert_s"][agent].copy_(torch.from_numpy(np.asarray(sE, np.float32)))
        self.t["expert_sp"][agent].copy_(torch.from_numpy(np.asarray(spE, np.float32)))

    def set_expert_all(self, sE, spE):
        """``set_expert`` for EVERY agent in one copy per table: ``sE, spE`` [n_agents, E, S]."""
        self.t["expert_s"].copy_(torch.from_numpy(np.asarray(sE, np.float32)))
        self.t["expert_sp"].copy_(torch.from_numpy(np.asarray(spE, np.float32)))

    # ------------------------------------------------------------------ hot path
    def gather(self, idx: torch.Tensor):
        """``get_offmodel_info`` for the given int64 indices [n_agents, B] -> (s, a, sp, r, d)."""
        sp_ = self.spec
        n, B = sp_.n_agents, sp_.B
        idx = idx.to(self.dev, torch.int64).contiguous()
        s = torch.empty(n, B, sp_.S, device=self.dev)
        a = torch.empty(n, B, sp_.A, device=self.dev)
        spn = torch.empty(n, B, sp_.S, device=self.dev)
        r = torch.empty(n, B, device=self.dev)
        d = torch.empty(n, B, device=self.dev, dtype=torch.float64)
        st = self._enter()
        _l.check(self.lib.saceo_gather(self.ctx, idx.data_ptr(), s.data_ptr(), a.data_ptr(), spn.data_ptr(),
                                       r.data_ptr(), d.data_ptr(), st))
        self._exit()
        return s, a, spn, r, d

    def set_draws(self, idx=None, noise=None, perm=None):
        ten = []
        for v, dt in ((idx, torch.int64), (noise, torch.float32), (perm, torch.int32)):
            ten.append(None if v is None else torch.as_tensor(v).to(self.dev, dt).contiguous())
        st = self._enter()
        _l.check(self.lib.saceo_set_draws(self.ctx, *[t.data_ptr() if t is not None else None for t in ten], st))
        self._exit()
        self._keep = ten

    def update(self, n_steps: int = 1, num_timesteps: int = 0, use_device_rng: bool = True, seed: int = 0):
        st = self._enter()
        _l.check(self.lib.saceo_update(self.ctx, n_steps, num_timesteps, int(use_device_rng), seed,
                                       self.losses.data_ptr(), st))
        self._exit()
        return self.losses

    def profile_step(self, num_timesteps: int = 0, use_device_rng: bool = True, seed: int = 0):
        """One real update launched kernel by kernel with a CUDA event after every launch.
        Returns [(kernel name, microseconds)] in launch order."""
        cap = 256
        names = C.create_string_buffer(cap * 32)
        us = (C.c_float * cap)()
        n = C.c_int32(0)
        st = self._enter()
        _l.check(self.lib.saceo_profile_step(self.ctx, num_timesteps, int(use_device_rng), seed, names, C.cast(us, C.c_void_p),
                                             cap, C.byref(n), st))
        self._exit()
        raw = names.raw
        return [(raw[i * 32:(i + 1) * 32].split(b"\0", 1)[0].decode(), float(us[i])) for i in range(n.value)]

    def bc_update(self, n_steps: int = 1, use_device_rng: bool = True, seed: int = 0):
        """``BC._update_actor`` (BC.py:309-363): actor step on the expert-observation MSE alone."""
        st = self._enter()
        _l.check(self.lib.saceo_bc_update(self.ctx, n_steps, int(use_device_rng), seed, self.losses.data_ptr(), st))
        self._exit()
        return self.losses

    def update_host(self, num_timesteps: int, seed: int, idx_host: Optional[np.ndarray] = None,
                    expert_host: Optional[np.ndarray] = None) -> np.ndarray:
        """One update through HOST buffers (pinned staging), synchronous - the per-step call of the
        reference-style ``alg._update``."""
        n, sp_ = self.spec.n_agents, self.spec
        if self._pin_loss is None:
            self._pin_loss = torch.empty(n, self.L.n_losses, pin_memory=True)
        ip = ep = None
        if idx_host is not None:
            if self._pin_idx is None:
                self._pin_idx = torch.empty(n, sp_.B, dtype=torch.int64, pin_memory=True)
            self._pin_idx.numpy()[...] = idx_host
            ip = self._pin_idx.data_ptr()
        if expert_host is not None:
            if self._pin_exp is None:
                self._pin_exp = torch.empty(2, n, sp_.E, sp_.S, pin_memory=True)
            self._pin_exp.numpy()[...] = expert_host
            ep = self._pin_exp.data_ptr()
        st = self._enter()
        _l.check(self.lib.saceo_update_host(self.ctx, num_timesteps, seed, ip, ep, self._pin_loss.data_ptr(), st))
        self._exit()
        return self._pin_loss.numpy()

    def update_host_async(self, num_timesteps: int, seed: int, idx_host: Optional[np.ndarray] = None,
                          expert_host: Optional[np.ndarray] = None, slot: int = 0) -> None:
        """Enqueues one update through HOST buffers without waiting for it.  ``slot`` (0/1) selects one of two pinned
        staging sets, so the caller can prepare step t+1 on the host (index draws, environment steps) while the
        device runs step t; ``wait_host(slot)`` returns that step's losses.  A slot must be waited for before reuse."""
        n, sp_ = self.spec.n_agents, self.spec
        if not hasattr(self, "_slots"):
            self._slots = [dict(loss=torch.empty(n, self.L.n_losses, pin_memory=True), idx=None, exp=None,
                                ev=torch.cuda.Event()) for _ in range(2)]
        sl = self._slots[slot]
        ip = ep = None
        if idx_host is not None:
            if sl["idx"] is None:
                sl["idx"] = torch.empty(n, sp_.B, dtype=torch.int64, pin_memory=True)
            sl["idx"].numpy()[...] = idx_host
            ip = sl["idx"].data_ptr()
        if expert_host is not None:
            if sl["exp"] is None:
                sl["exp"] = torch.empty(2, n, sp_.E, sp_.S, pin_memory=True)
            sl["exp"].numpy()[...] = expert_host
            ep = sl["exp"].data_ptr()
        st = self._enter()
        _l.check(self.lib.saceo_update_host_async(self.ctx, num_timesteps, seed, ip, ep, sl["loss"].data_ptr(), st))
        sl["ev"].record(self.stream)

    def wait_host(self, slot: int = 0) -> np.ndarray:
        """Blocks until the update enqueued with ``slot`` has finished; returns its losses [n_agents, n_losses] (host)."""
        sl = self._slots[slot]
        sl["ev"].synchronize()
        return sl["loss"].numpy()

    def update_phase(self, phase: int, num_timesteps: int = 0):
        st = self._enter()
        _l.check(self.lib.saceo_update_phase(self.ctx, phase, num_timesteps, st))
        self._exit()

    # ------------------------------------------------------------------ inference entry points
    def actor_forward(self, obs: torch.Tensor, noise: Optional[torch.Tensor] = None, want_neglogp: bool = False):
        n, sp_ = self.spec.n_agents, self.spec
        obs = obs.to(self.dev, torch.float32).contiguous().view(n, -1, sp_.S)
        rows = obs.shape[1]
        if noise is not None:
            noise = noise.to(self.dev, torch.float32).contiguous()
        act = torch.empty(n, rows, sp_.A, device=self.dev)
        nlp = torch.empty(n, rows, device=self.dev) if want_neglogp else None
        st = self._enter()
        _l.check(self.lib.saceo_actor_forward(self.ctx, obs.data_ptr(), rows,
                                              noise.data_ptr() if noise is not None else None, act.data_ptr(),
                                              nlp.data_ptr() if nlp is not None else None, st))
        self._exit()
        return (act, nlp) if want_neglogp else act

    def critic_forward(self, obs, act, target: bool = False, scale_ret: bool = False):
        n, sp_ = self.spec.n_agents, self.spec
        obs = torch.as_tensor(obs).to(self.dev, torch.float32).contiguous().view(n, -1, sp_.S)
        act = torch.as_tensor(act).to(self.dev, torch.float32).contiguous().view(n, -1, sp_.A)
        rows = obs.shape[1]
        q = torch.empty(n, 2, rows, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_critic_forward(self.ctx, int(target), obs.data_ptr(), act.data_ptr(), rows,
                                               int(scale_ret), q.data_ptr(), st))
        self._exit()
        return q

    def model_eval(self, obs, act):
        n, sp_ = self.spec.n_agents, self.spec
        obs = torch.as_tensor(obs).to(self.dev, torch.float32).contiguous().view(n, -1, sp_.S)
        act = torch.as_tensor(act).to(self.dev, torch.float32).contiguous().view(n, -1, sp_.A)
        rows = obs.shape[1]
        out = torch.zeros(n, 2, rows, sp_.S, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_model_eval(self.ctx, obs.data_ptr(), act.data_ptr(), rows, out.data_ptr(), st))
        self._exit()
        return out

    # ------------------------------------------------------------------ dynamics-model fitting
    def fit_bind(self, model_batch: int = 200, use_grad_clip: bool = False, gaussian: bool = False, std_mult: float = 1.0):
        """Allocates the joint model optimiser's slots (``self.model_optimizer``, mbrl_onpolicy_alg.py:48-49)
        and the fitting workspace for minibatches of ``model_batch`` rows (--model_batch_size).  ``gaussian``:
        ``GaussianModel`` loss with the trainable ``logstd`` variable initialised to log(std_mult)
        (continuous_models.py:24-25)."""
        n, L = self.spec.n_agents, self.L
        z = lambda *sh, dt=torch.float32: torch.zeros(*sh, dtype=dt, device=self.dev)
        self.t.update(model_m=z(n, 2, L.nm_stride), model_v=z(n, 2, L.nm_stride), model_t=z(n, dt=torch.int32),
                      fit_hyper=z(n, _l.FIT_HYPER))
        self.t["fit_hyper"][:, 0] = 1e-3      # --model_lr
        self.t["fit_hyper"][:, 1] = 1.0       # --reward_loss_coef
        self.t["fit_hyper"][:, 6] = 1.0       # identity r_rms
        if self.spec.separate_reward_nn:
            nr = sum(int(np.prod(sh)) for sh in self.shapes["reward"])
            self.nr_stride = (nr + 31) // 32 * 32
            keep = self.t.get("reward")
            self.t.update(reward=keep if keep is not None and keep.shape[-1] == self.nr_stride else z(n, 2, self.nr_stride),
                          reward_m=z(n, 2, self.nr_stride), reward_v=z(n, 2, self.nr_stride))
        if gaussian:
            self.t.update(model_logstd=torch.full((n, 2, self.spec.S), float(np.log(std_mult)), device=self.dev),
                          model_logstd_m=z(n, 2, self.spec.S), model_logstd_v=z(n, 2, self.spec.S))
        else:
            for k in ("model_logstd", "model_logstd_m", "model_logstd_v"):
                self.t.pop(k, None)
        ft = _l.FitTables()
        for name in _l.FitTables.POINTERS:
            setattr(ft, name, self.t[name].data_ptr() if name in self.t else None)
        if self.spec.separate_reward_nn:
            rh = tuple(self.spec.reward_hidden or self.spec.model_hidden)
            ra = tuple(self.spec.reward_acts or self.spec.model_acts)
            for i in range(2):
                if ra[i] not in _l.ACT_IDS:
                    raise ValueError("activations must be relu, tanh, or elu")
                ft.reward_hidden[i] = int(rh[i]); ft.reward_act[i] = _l.ACT_IDS[ra[i]]
            ft.reward_stride = self.nr_stride
        torch.cuda.synchronize(self.dev)
        _l.check(self.lib.saceo_fit_bind(self.ctx, C.byref(ft), int(model_batch), int(bool(use_grad_clip))))
        self.model_batch = int(model_batch)

    def set_fit_hyper(self, agent: int, **hy):
        """model_lr, reward_loss_coef, delta_clip_loss, reward_clip_loss, model_max_grad_norm (0/None = off), r_mean, r_std,
        scale_model_loss (Gaussian loss only)."""
        row = self.t["fit_hyper"][agent]
        for key, val in hy.items():
            row[_l.FIT_HYPER_NAMES.index(key)] = float(val or 0.0)

    def reset_model_optimizer(self):
        """``reset_model_optimizer`` (SAC_expert.py:551-553): fresh Adam slots and step count."""
        for k in ("model_m", "model_v", "model_t", "model_logstd_m", "model_logstd_v", "reward_m", "reward_v"):
            if k in self.t:
                self.t[k].zero_()

    def model_fit(self, idx, want_losses: bool = True) -> Optional[torch.Tensor]:
        """``_apply_model_grads`` for every entry of ``idx`` ([n_steps, n_agents, num_models, model_batch] or
        [n_agents, num_models, model_batch] logical replay rows).  Returns the per-model minibatch losses
        [n_steps, n_agents, num_models]."""
        n, nm = self.spec.n_agents, self.spec.num_models
        idx = torch.as_tensor(idx).to(self.dev, torch.int64).contiguous().view(-1, n, nm, self.model_batch)
        steps = idx.shape[0]
        losses = torch.zeros(steps, n, nm, device=self.dev) if want_losses else None
        st = self._enter()
        _l.check(self.lib.saceo_model_fit(self.ctx, steps, idx.data_ptr(), losses.data_ptr() if want_losses else None, st))
        self._exit()
        return losses

    # ------------------------------------------------------------------ CG / Fisher-vector
    def fvp(self, x: torch.Tensor, damp: float) -> torch.Tensor:
        x = x.to(self.dev, torch.float32).contiguous()
        out = torch.zeros_like(x)
        st = self._enter()
        _l.check(self.lib.saceo_fvp(self.ctx, x.data_ptr(), damp, out.data_ptr(), st))
        self._exit()
        return out

    def cg_solve(self, b: torch.Tensor, iters: int = 20, tol: float = 1e-10, damp: float = 0.01):
        b = b.to(self.dev, torch.float32).contiguous()
        x = torch.zeros_like(b)
        vfv = torch.zeros(self.spec.n_agents, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_cg_solve(self.ctx, b.data_ptr(), iters, tol, damp, x.data_ptr(), vfv.data_ptr(), st))
        self._exit()
        return x, vfv

    # ------------------------------------------------------------------ TRPO surrogate / line search
    def _opt(self, x, *shape):
        if x is None:
            return None
        return torch.as_tensor(x).to(self.dev, torch.float32).contiguous().view(*shape)

    def trpo_grad(self, act, adv, nlp_old=None, alpha=None):
        """Surrogate tape of ``TRPO.update`` (trpo.py:52-63) on the bound ``fvp_states``: returns
        (neg_pg [n, na_stride] flat gradients, stats [n, 8] = {mean(ratio adv), 0, tv, mean entropy, ...})."""
        n, N, A = self.spec.n_agents, self.spec.fvp_rows, self.spec.A
        act, adv = self._opt(act, n, N, A), self._opt(adv, n, N)
        nlp_old, alpha = self._opt(nlp_old, n, N), self._opt(alpha, n)
        grad = torch.zeros(n, self.L.na_stride, device=self.dev)
        stats = torch.zeros(n, 8, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_trpo_grad(self.ctx, act.data_ptr(), adv.data_ptr(),
                                          None if nlp_old is None else nlp_old.data_ptr(),
                                          None if alpha is None else alpha.data_ptr(), grad.data_ptr(), stats.data_ptr(), st))
        self._exit()
        return grad, stats

    def onpolicy_expert_grad(self, n_models: int = 2, clip_actions: bool = False):
        """Second tape of ``TRPO.update``'s expert branch / the MSE half of ``PPO._apply_actor_grad``'s (trpo.py:113-149,
        ppo.py:176-213): d MSE / d(actor trainable) through ``GaussianActor.sample`` and the frozen model(s), on the bound
        expert rows with the draws last injected by ``set_draws(noise=..., perm=...)`` (noise rows [2B, 2B+E)).
        Returns (grad [n, na_stride], mse [n])."""
        n = self.spec.n_agents
        grad = torch.empty(n, self.L.na_stride, device=self.dev)
        stats = torch.zeros(n, 8, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_onpolicy_expert_grad(self.ctx, int(n_models), int(bool(clip_actions)), grad.data_ptr(),
                                                     stats.data_ptr(), st))
        self._exit()
        return grad, stats[:, 0]

    def grad_blend(self, neg_pg, mse_grad, eps, max_grad_norm=None):
        """``grad_final = (1 - eps) neg_pg + eps MSE_grads`` per agent (trpo.py:150-158) + optional global-norm clip
        (ppo.py:226-231).  Returns (grad_final [n, na_stride], stats [n, 8]: [6] norm_pg, [7] norm_MSE as the reference
        logs them, [4] / [5] global norm before / after clipping)."""
        n = self.spec.n_agents
        eps = torch.as_tensor(np.broadcast_to(np.asarray(eps, np.float32), (n,)).copy()).to(self.dev)
        out = torch.empty(n, self.L.na_stride, device=self.dev)
        stats = torch.zeros(n, 8, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_grad_blend(self.ctx, neg_pg.data_ptr(), mse_grad.data_ptr(), eps.data_ptr(),
                                           float(max_grad_norm) if max_grad_norm is not None else 0.0, out.data_ptr(),
                                           stats.data_ptr(), st))
        self._exit()
        return out, stats

    def ppo_grad(self, act, adv, nlp_old, alpha=None, eps_clip=0.2, max_grad_norm=None):
        """Gradient of ``PPO._apply_actor_grad`` (ppo.py:132-147, :226-231) on the bound ``fvp_states``: clipped surrogate
        + entropy regulariser, then ``clip_by_global_norm``.  Returns (neg_pg [n, na_stride], stats [n, 8] with
        [4] / [5] = global norm before / after clipping)."""
        n, N, A = self.spec.n_agents, self.spec.fvp_rows, self.spec.A
        act, adv, nlp_old = self._opt(act, n, N, A), self._opt(adv, n, N), self._opt(nlp_old, n, N)
        alpha = self._opt(alpha, n)
        grad = torch.zeros(n, self.L.na_stride, device=self.dev)
        stats = torch.zeros(n, 8, device=self.dev)
        st = self._enter()
        _l.check(self.lib.saceo_ppo_grad(self.ctx, act.data_ptr(), adv.data_ptr(), nlp_old.data_ptr(),
                                         None if alpha is None else alpha.data_ptr(), float(eps_clip),
                                         float(max_grad_norm) if max_grad_norm is not None else 0.0,
                                         grad.data_ptr(), stats.data_ptr(), st))
        self._exit()
        return grad, stats

    def actor_adam(self, grad: torch.Tensor):
        """``actor_optimizer.apply_gradients`` (ppo.py:234): one Keras-Adam step of the actor optimiser with ``grad``
        [n, na_stride]; the learning rate is the per-agent ``actor_lr`` hyper-parameter."""
        grad = self._opt(grad, self.spec.n_agents, self.L.na_stride)
        st = self._enter()
        _l.check(self.lib.saceo_actor_adam(self.ctx, grad.data_ptr(), st))
        self._exit()

    def trpo_eval(self, act=None, adv=None, nlp_old=None, kl_ref=None, want_nlp=False, want_kl_info=False,
                  want_rows=False):
        """Line-search quantities of ``TRPO._backtrack`` (trpo.py:251-263) at the current actor parameters: dict with
        ``stats`` [n, 8] = {surr, kl, tv, ent, ...} and optionally ``nlp`` [n, N], ``kl_info`` [n, N, A, 2], ``rows``
        [n, N, 4] (per-row ratio adv, kl, |ratio - 1|, entropy)."""
        n, N, A = self.spec.n_agents, self.spec.fvp_rows, self.spec.A
        act, adv, nlp_old = self._opt(act, n, N, A), self._opt(adv, n, N), self._opt(nlp_old, n, N)
        kl_ref = self._opt(kl_ref, n, N, A, 2)
        res = {"stats": torch.zeros(n, 8, device=self.dev)}
        if want_nlp:
            res["nlp"] = torch.zeros(n, N, device=self.dev)
        if want_kl_info:
            res["kl_info"] = torch.zeros(n, N, A, 2, device=self.dev)
        ptr = lambda t: None if t is None else t.data_ptr()
        st = self._enter()
        _l.check(self.lib.saceo_trpo_eval(self.ctx, ptr(act), ptr(adv), ptr(nlp_old), ptr(kl_ref), ptr(res.get("nlp")),
                                          ptr(res.get("kl_info")), res["stats"].data_ptr(), st))
        self._exit()
        if want_rows:      # per-row {ratio adv, kl, |ratio - 1|, entropy} as the kernel left them in the workspace
            res["rows"] = self.debug("fTmp")[:n * N * 4].view(n, N, 4).clone()
        return res

    def actor_step(self, theta_ref: torch.Tensor, direction: torch.Tensor, scale):
        """``actor = theta_ref + scale[agent] * direction`` (``set_weights(..., increment=True)``,
        continuous_actors.py:211-233)."""
        n = self.spec.n_agents
        theta_ref, direction = self._opt(theta_ref, n, self.L.na_stride), self._opt(direction, n, self.L.na_stride)
        scale = self._opt(np.asarray(scale, np.float32) if not torch.is_tensor(scale) else scale, n)
        st = self._enter()
        _l.check(self.lib.saceo_actor_step(self.ctx, theta_ref.data_ptr(), direction.data_ptr(), scale.data_ptr(), st))
        self._exit()

    def trpo_update(self, act, adv, *, delta=0.01, cg_iters=20, trust_damp=0.01, kl_maxfactor=1.5, alpha=None,
                    adv_center=True, adv_scale=True, residual_tol=1e-10, expert_eps=None):
        """``TRPO.update`` (trpo.py:36-198) + ``TRPO._backtrack`` (:229-317) for every agent of the population on its
        bound ``fvp_states`` (trust_sub = 1): surrogate gradient, CG solve with the Fisher-vector product, step length
        ``sqrt(2 delta / vFv)`` and the back-tracking line search, each agent with its own accept / shrink decisions.
        ``adv`` [n, N] raw advantages (host); centred / scaled per agent with NumPy like the reference (:41-48, and a
        second time inside ``_backtrack`` :243-249).  ``expert_eps`` (scalar or [n]; None: the epsilon = 0 slice
        ``grad_final = neg_pg``): the two-model expert blend ``grad_final = (1 - eps) neg_pg + eps MSE_grads``
        (:113-158) on the bound expert rows with the draws last injected by ``set_draws(noise=..., perm=...)``.
        Returns one log dict per agent (``ent, tv_pre, kl_pre, tv, kl, adj, improve`` [+ ``mse, norm_pg, norm_MSE``])."""
        n, N = self.spec.n_agents, self.spec.fvp_rows
        adv = np.asarray(adv, np.float32).reshape(n, N)

        def norm(a):
            out = np.empty_like(a)
            for i in range(n):
                x = a[i]
                mean, std = np.mean(x), np.std(x) + 1e-8
                x = x - mean if adv_center else x
                out[i] = x / std if adv_scale else x
            return out

        adv1 = norm(adv)
        act = self._opt(act, n, N, self.spec.A)
        first = self.trpo_eval(act=act, want_nlp=True, want_kl_info=True)
        nlp_old, kl_ref = first["nlp"], first["kl_info"]
        ent = first["stats"][:, 3].cpu().numpy()
        neg_pg, _ = self.trpo_grad(act, adv1, nlp_old, alpha)
        extra = None
        if expert_eps is not None:
            g_mse, mse = self.onpolicy_expert_grad(n_models=2, clip_actions=False)
            neg_pg, bst = self.grad_blend(neg_pg, g_mse, expert_eps)
            extra = (mse.cpu().numpy(), bst.cpu().numpy())
        pg = -neg_pg
        theta_ref = self.t["actor"].clone()
        if delta == 0.0:
            eta = np.zeros(n, np.float32)
            v = torch.zeros_like(pg)
        else:
            v, vfv = self.cg_solve(pg, iters=cg_iters, tol=residual_tol, damp=trust_damp)
            vfv = vfv.cpu().numpy().astype(np.float64)
            zero = (pg[:, :self.L.na].abs().amax(dim=1) <= 1e-8).cpu().numpy()      # np.allclose(pg_vec, 0) per agent (:179)
            skip = zero | ~(vfv > 0)                          # pg_vec == 0 (:179-180): no step; CG of a zero vector is 0/0
            eta = np.where(skip, 0.0, np.sqrt(2 * delta / np.where(skip, 1.0, vfv))).astype(np.float32)
            v[torch.from_numpy(skip).to(self.dev)] = 0.0
        adv2 = self._opt(norm(adv1), n, N)
        surr_before = self.trpo_eval(act, adv2, nlp_old)["stats"][:, 0].cpu().numpy()

        def trial(scale):
            self.actor_step(theta_ref, v, scale)
            s = self.trpo_eval(act, adv2, nlp_old, kl_ref)["stats"].cpu().numpy()
            return s, s[:, 0] - surr_before

        adj, stats, improve, tv_pre, kl_pre = backtrack_population(lambda a: trial(eta * a), n, kl_maxfactor, delta)
        logs = [dict(ent=float(ent[i]), tv_pre=float(tv_pre[i]), kl_pre=float(kl_pre[i]), tv=float(stats[i, 2]),
                     kl=float(stats[i, 1]), adj=float(adj[i]), improve=float(improve[i])) for i in range(n)]
        if extra is not None:
            for i in range(n):
                logs[i].update(mse=float(extra[0][i]), norm_pg=float(extra[1][i, 6]), norm_MSE=float(extra[1][i, 7]))
        return logs



class SharedPopulation:
    """One ``n_agents`` population shared by objects that each describe a single agent: the first ``get(spec)``
    creates it from the one-agent ``spec`` with ``n_agents`` replaced, every later call must describe the same
    population.  Lets R algorithm objects built one after the other bind to agents 0 .. R-1 of one population.
    A ``PolicySpec`` (expert policies, ``policy.py``) makes it a ``PolicySet`` of ``n_agents`` policies instead."""

    def __init__(self, n_agents: int):
        self.n_agents, self.pop = int(n_agents), None

    def get(self, spec):
        spec = replace(spec, n_agents=self.n_agents)
        if self.pop is None:
            self.pop = PolicySet(spec) if isinstance(spec, PolicySpec) else Population(spec)
        elif spec != self.pop.spec:
            raise ValueError(f"a shared population needs one spec for every agent: {spec} != {self.pop.spec}")
        return self.pop
