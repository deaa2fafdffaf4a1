"""Minimal gym-free environment stand-in with MuJoCo-shaped spaces (gym / dm_control are not installable
offline; the reference builds its spaces with ``gym.spaces.Box``, ``/root/reference/sac_eo/envs``).
The simulators are out of scope (SURVEY.md §2 row 16); this class only supplies ``observation_space`` /
``action_space`` and a cheap linear-dynamics ``step`` for smoke runs."""
import numpy as np

from ..common.lockstep import np_random


class Box:
    def __init__(self, low, high, shape):
        self.shape = tuple(shape)
        self.low = np.full(self.shape, low, np.float32)
        self.high = np.full(self.shape, high, np.float32)

    def sample(self):
        return np_random().uniform(self.low, self.high).astype(np.float32)


def flatdim(space) -> int:
    """``gym.spaces.utils.flatdim`` for Box spaces."""
    return int(np.prod(space.shape))


class SyntheticEnv:
    def __init__(self, s_dim, a_dim, seed=0, horizon=1000):
        self.observation_space = Box(-np.inf, np.inf, (s_dim,))
        self.action_space = Box(-1.0, 1.0, (a_dim,))     # RescaleAction(-1, 1), gym_wrapper.py:3-8
        rng = np.random.default_rng(seed)
        self._A = (np.eye(s_dim) * 0.95 + 0.02 * rng.standard_normal((s_dim, s_dim))).astype(np.float32)
        self._B = (0.1 * rng.standard_normal((a_dim, s_dim))).astype(np.float32)
        self._rng, self._h, self._t = rng, horizon, 0
        self.s = np.zeros(s_dim, np.float32)

    def seed(self, seed):
        self._rng = np.random.default_rng(seed)

    def reset(self, s_init=None):
        self._t = 0
        self.s = (self._rng.standard_normal(self.s.shape).astype(np.float32) if s_init is None
                  else np.asarray(s_init, np.float32))
        return self.s

    def step(self, a):
        a = np.asarray(a, np.float32)
        self.s = self.s @ self._A + a @ self._B + 0.01 * self._rng.standard_normal(self.s.shape).astype(np.float32)
        self._t += 1
        r = float(-np.sum(self.s ** 2) - 0.01 * np.sum(a ** 2))
        return self.s, r, self._t >= self._h, {}
