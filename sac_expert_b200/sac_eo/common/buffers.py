"""``TrajectoryBuffer`` with the reference's interface (``/root/reference/sac_eo/common/buffers.py``): host
NumPy arrays (``s_all`` ... ``current_size``) with append + tail truncation, mirrored row-by-row into the
device replay table of one agent once ``attach`` ed.  Minibatch sampling keeps the reference's RNG call
(``np.random.randint(current_size, size=batch_size)``, :135) on the host and performs the five row gathers
on the device (bit-exact copies).  GAE / ``get_update_info`` belong to the on-policy path (out of scope)."""
import numpy as np
import torch

from ...lib import SaceoError
from .lockstep import Request, inline, np_random


class TrajectoryBuffer:
    def __init__(self, s_dim, a_dim, gamma, lam, buffer_size=None):
        self.s_dim, self.a_dim, self.gamma, self.lam, self.buffer_size = s_dim, a_dim, gamma, lam, buffer_size
        self._pop, self._agent = None, 0
        self.reset()

    _FIELDS = (("s", "s_dim", np.float32), ("a", "a_dim", np.float32), ("r", None, np.float32), ("sp", "s_dim", np.float32),
               ("d", None, np.float64), ("idx", None, np.float64))

    def reset(self):
        """Empty buffer.  The arrays the reference exposes (``s_all`` ... ``idx_all``, chronological order) are views
        ``store[lo:hi]`` of pre-allocated windows: ``add`` writes behind ``hi`` in amortised O(rows added) instead of
        re-concatenating every array (buffers.py:41-58 copies the whole buffer on every call - O(N) per environment
        step, SURVEY.md 8f-2); when the window reaches the end of the allocation the live rows slide to the front."""
        self._lo = self._hi = 0
        self._alloc(64)
        self.traj_total = self.steps_total = self.current_size = 0

    def _alloc(self, cap):
        old = getattr(self, "_store", None)
        self._store = {}
        for name, dim, dt in self._FIELDS:
            shape = (cap,) if dim is None else (cap, getattr(self, dim))
            arr = np.empty(shape, dt)
            if old is not None and self._hi > self._lo:
                arr[: self._hi - self._lo] = old[name][self._lo:self._hi]
            self._store[name] = arr
        self._hi -= self._lo
        self._lo = 0
        self._cap = cap

    def _view(self, name):
        return self._store[name][self._lo:self._hi]

    s_all = property(lambda self: self._view("s"))
    a_all = property(lambda self: self._view("a"))
    r_all = property(lambda self: self._view("r"))
    sp_all = property(lambda self: self._view("sp"))
    d_all = property(lambda self: self._view("d"))
    idx_all = property(lambda self: self._view("idx"))

    def attach(self, pop, agent=0):
        """Mirror this buffer into the device replay table of ``agent`` (existing rows are uploaded)."""
        if self.buffer_size and self.buffer_size > pop.spec.replay_capacity:
            raise ValueError("device replay_capacity is smaller than buffer_size")
        self._pop, self._agent = pop, agent
        if self.current_size:
            pop.append_rows(agent, self.s_all, self.a_all, self.r_all, self.sp_all, self.d_all)

    def _add_steps(self, s_traj, a_traj, r_traj, sp_traj, d_traj):
        s_traj = np.asarray(s_traj).reshape(-1, self.s_dim)
        a_traj = np.asarray(a_traj).reshape(-1, self.a_dim)
        r_traj, d_traj = np.atleast_1d(np.asarray(r_traj)), np.atleast_1d(np.asarray(d_traj))
        sp_traj = np.asarray(sp_traj).reshape(-1, self.s_dim)
        k = len(r_traj)
        if self._hi + k > self._cap:          # slide the live window to the front, growing the allocation if needed
            live = self._hi - self._lo
            keep = min(live, self.buffer_size) if self.buffer_size else live
            self._lo = self._hi - keep
            need = keep + k
            self._alloc(max(2 * self._cap, 2 * need) if (not self.buffer_size or self._cap < 2 * (self.buffer_size + k)) else self._cap)
        new = dict(s=s_traj, a=a_traj, r=r_traj, sp=sp_traj, d=d_traj, idx=np.ones(k) * self.traj_total)
        for name, _, _ in self._FIELDS:
            self._store[name][self._hi:self._hi + k] = new[name]
        self._hi += k
        if self.buffer_size and self._hi - self._lo > self.buffer_size:    # keep the LAST buffer_size rows (:60-66)
            self._lo = self._hi - self.buffer_size
        self.current_size = self._hi - self._lo
        self.traj_total += 1
        self.steps_total += k
        if self._pop is not None:
            if not self.buffer_size and self.current_size > self._pop.spec.replay_capacity:
                raise SaceoError("unbounded TrajectoryBuffer outgrew the device replay_capacity")
            yield Request("append", self._pop, self._agent, (k,), rows=(s_traj, a_traj, r_traj, sp_traj, d_traj))

    add = inline(_add_steps)

    def _device_gather(self, idx):
        if self._pop is None:
            raise SaceoError("TrajectoryBuffer is not attached to a device population; minibatch gathers have no CPU path")
        if len(idx) != self._pop.spec.B:
            raise ValueError(f"batch_size {len(idx)} != device batch {self._pop.spec.B}")
        full = np.zeros((self._pop.spec.n_agents, len(idx)), np.int64)
        full[self._agent] = idx
        out = self._pop.gather(torch.from_numpy(full))
        return [t[self._agent].cpu().numpy() for t in out]

    def get_offmodel_info(self, batch_size=None):
        if batch_size:
            idx = np_random().randint(self.current_size, size=batch_size)
            self.last_idx = idx
            s, a, sp, r, d = self._device_gather(idx)
            return s, a, sp, r, d
        return self.s_all, self.a_all, self.sp_all, self.r_all, self.d_all

    def get_model_info(self, batch_size=None):
        if batch_size:
            idx = np_random().randint(self.current_size, size=batch_size)
            if self._pop is not None and batch_size == self._pop.spec.B:
                s, a, sp, r, _ = self._device_gather(idx)
                return s, a, sp, r
            # small per-episode resample of the expert buffer (SAC_expert.py:421-422): host bookkeeping, not the
            # update hot path - the rows are re-uploaded as expert_reg afterwards
            return self.s_all[idx], self.a_all[idx], self.sp_all[idx], self.r_all[idx]
        return self.s_all, self.a_all, self.sp_all, self.r_all

    def get_states(self, batch_size=None):
        if batch_size:
            return self.get_offmodel_info(batch_size)[0]
        return self.s_all
