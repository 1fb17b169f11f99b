"""Reference for the dynamic-feature catalogue, built from the executable specification (gte.DeviceFeature).

`DynColumns` keeps, for N envs in lockstep, the History rows the reference would evaluate its
``dynamic_feature_functions`` on — per iteration the step's row and, where an episode restarted, the reset row —
evaluates the DeviceFeature callables on a History stand-in (vectorised over the envs: numpy applies the same IEEE fp64
operations element by element), casts to float32 (environments.py:153-154) and assembles windows whose rows before the
episode start read zero (the H3 normalisation, SURVEY.md §8a).  It is fed either from a golden's recorded reference
columns or from the CPU oracle's outputs (`CatalogueOracle`).
"""
from __future__ import annotations

import numpy as np

from gym_trading_env_b200.dynamic_features import KINDS, DeviceFeature

F32, F64 = np.float32, np.float64


class History:
    """The two rows of a reference History the catalogue reads: ``history[column, -1]`` and ``history[column, 0]``."""

    def __init__(self, first, last):
        self.first, self.last = first, last

    def __getitem__(self, key):
        column, row = key
        assert row in (0, -1)
        return (self.first if row == 0 else self.last)[column]


class DynColumns:
    def __init__(self, n_envs, windows, positions, v0, max_episode_duration):
        self.N, self.W = n_envs, (windows or 1)
        self.positions, self.v0 = np.asarray(positions, F64), float(v0)
        d = max_episode_duration if isinstance(max_episode_duration, (int, np.integer)) and max_episode_duration > 0 else None
        self.features = [DeviceFeature(k, d) if k == "episode_progress" else DeviceFeature(k)
                         for k in KINDS if k != "episode_progress" or d is not None]
        self.kinds = [f.kind for f in self.features]
        self.ring = np.zeros((self.W, n_envs, len(KINDS)), F32)     # row of iteration c in slot c % W, every kind
        self.c = 0
        self.final = None

    def _rows(self, pos_idx, real_position, valuation, reward, step):
        h = History({"portfolio_valuation": np.full(self.N, self.v0, F64)},
                    {"position": self.positions[pos_idx], "real_position": np.asarray(real_position, F64),
                     "portfolio_valuation": np.asarray(valuation, F64), "reward": np.asarray(reward, F64),
                     "step": np.asarray(step)})
        out = np.zeros((self.N, len(KINDS)), F32)
        for f in self.features:
            out[:, KINDS.index(f.kind)] = np.asarray(f(h), F64).astype(F32)
        return out

    def _reset_rows(self, pos_idx):
        pos_idx = np.asarray(pos_idx)
        return self._rows(pos_idx, self.positions[pos_idx], np.full(self.N, self.v0), np.zeros(self.N),
                          np.zeros(self.N, np.int64))

    def reset(self, pos_idx, mask=None):
        """Envs (re)started in place at the current iteration with these position indices."""
        m = np.ones(self.N, bool) if mask is None else np.asarray(mask, bool)
        self.ring[self.c % self.W][m] = self._reset_rows(pos_idx)[m]

    def step(self, pos_idx, real_position, valuation, reward, step, idx, ended, post_pos_idx):
        """One lockstep iteration: the step's row of every env (pos_idx = the position index the step ended in), then
        the reset row of the envs whose episode ended.  Keeps the terminal windows in self.final."""
        self.c += 1
        self.ring[self.c % self.W] = self._rows(np.asarray(pos_idx), real_position, valuation, reward, step)
        self.final = self.window(np.asarray(idx), np.asarray(idx) - np.asarray(step))
        self.reset(post_pos_idx, ended)

    def window(self, idx, ep_start):
        """[N, W, 5] rows idx-W+1 .. idx of every kind; rows before ep_start are zero."""
        W = self.W
        w = np.arange(W)
        slots = (self.c - (W - 1) + w) % W
        vals = self.ring[slots].transpose(1, 0, 2).copy()
        rows = np.asarray(idx)[:, None] - (W - 1) + w[None, :]
        vals[rows < np.asarray(ep_start)[:, None]] = 0
        return vals

    def select(self, vals, kinds):
        return vals[:, :, [KINDS.index(k) for k in kinds]]


def pos_after(actions, pos_before, positions):
    """The position index a step ends in (environments.py:213-215, :234): a value change of the target, else held."""
    a = np.asarray(actions, np.int64)
    p = np.asarray(positions, F64)
    cur = np.asarray(pos_before, np.int64)
    ok = (a >= 0) & (a < len(p))
    tgt = np.where(ok, a, cur)
    return np.where(ok & (p[tgt] != p[cur]), tgt, cur)


def with_dyn(static, dyn, windows):
    """Observation = static columns | dynamic columns; dyn is [N, W, nd]."""
    d = dyn if windows is not None else dyn[:, 0]
    return np.concatenate([static, d], axis=-1).astype(F32)


class CatalogueOracle:
    """The CPU oracle (default dynamic pair) with its dynamic columns replaced by a catalogue configuration."""

    def __init__(self, oracle_env, kinds, max_episode_duration):
        self.o, self.kinds = oracle_env, list(kinds)
        o = oracle_env
        self.ns = o.n_static
        self.cols = DynColumns(o.num_envs, o.windows, o.positions, o._e.v0, max_episode_duration)

    def _obs(self, vals):
        o = self.o
        static = o.obs[..., :self.ns]
        return with_dyn(static, self.cols.select(vals, self.kinds), o.windows)

    def reset(self, mask=None):
        o = self.o
        o.reset(mask)
        self.cols.reset(o.pos_idx.copy(), mask)
        self.obs = self._obs(self.cols.window(o.idx, o.ep_start))
        return self.obs

    def step(self, actions):
        o = self.o
        pos = pos_after(actions, o.pos_idx.copy(), o.positions)
        o.step(actions, want_final_obs=True)
        ended = (o.terminated | o.truncated).astype(bool)
        self.cols.step(pos, o.real_position, o.valuation, o.reward, o.info_step, o.info_idx, ended, o.pos_idx.copy())
        self.obs = self._obs(self.cols.window(o.idx, o.ep_start))
        self.final_obs = with_dyn(o.final_obs[..., :self.ns], self.cols.select(self.cols.final, self.kinds), o.windows)
        return self.obs
