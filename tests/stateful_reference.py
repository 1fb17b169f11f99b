"""Reference for the stateful dynamic features (current_drawdown, position_age).

`prefix_values` rebuilds every env's History prefix from recorded streams — the reset row, then one row per step, a new
History at every episode end, as `episode_reference.episode_histories` does but at every step — and evaluates the
DeviceFeature callables (the executable specification) on each prefix, cast to float32.

`StatefulColumns` is the same catalogue as `dyn_reference.DynColumns` plus the two stateful kinds, computed from a running
peak and age per env (what the device keeps in GteState.episode_acc) instead of whole prefixes; its windows read zero
before the episode start, as DynColumns' do.  `StatefulOracle` is `CatalogueOracle` over it.
"""
from __future__ import annotations

import numpy as np

from dyn_reference import CatalogueOracle, DynColumns
from gym_trading_env_b200.dynamic_features import KINDS, STATEFUL_KINDS, DeviceFeature

F32, F64 = np.float32, np.float64
ALL_KINDS = KINDS + STATEFUL_KINDS
STATEFUL = [DeviceFeature(k) for k in STATEFUL_KINDS]


def prefix_values(g, v0):
    """[K, N, 2] float32: the callables on each env's History prefix that ends with step k's row (before an auto-reset).
    g: arrays actions/position/valuation/terminated/truncated/post_pos_idx [K, N], plan [N, E, 3], positions [P]."""
    K, N = g["actions"].shape
    positions = np.asarray(g["positions"], F64)
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    out = np.zeros((K, N, len(STATEFUL)), F32)
    for i in range(N):
        rows = {"position": [positions[int(g["plan"][i, 0, 1])]], "portfolio_valuation": [float(v0)]}
        for k in range(K):
            rows["position"].append(g["position"][k, i])
            rows["portfolio_valuation"].append(g["valuation"][k, i])
            h = {c: np.asarray(v, F64) for c, v in rows.items()}
            out[k, i] = [np.float64(f(h)).astype(F32) for f in STATEFUL]
            if ended[k, i]:
                rows = {"position": [positions[int(g["post_pos_idx"][k, i])]], "portfolio_valuation": [float(v0)]}
    return out


class StatefulColumns(DynColumns):
    """DynColumns with the stateful kinds appended (columns in ALL_KINDS order).  `step_values` holds the stateful
    values of the last step's rows, before any reset."""

    def __init__(self, n_envs, windows, positions, v0, max_episode_duration):
        super().__init__(n_envs, windows, positions, v0, max_episode_duration)
        self.ring = np.zeros((self.W, n_envs, len(ALL_KINDS)), F32)
        self.peak = np.full(n_envs, self.v0)
        self.age = np.zeros(n_envs)
        self.prev = np.zeros(n_envs)
        self.row_values = np.zeros((n_envs, len(STATEFUL_KINDS)), F32)
        self.step_values = None

    def _rows(self, pos_idx, real_position, valuation, reward, step):
        return np.concatenate([super()._rows(pos_idx, real_position, valuation, reward, step), self.row_values], axis=1)

    def reset(self, pos_idx, mask=None):
        m = np.ones(self.N, bool) if mask is None else np.asarray(mask, bool)
        self.peak[m] = self.v0
        self.age[m] = 0.0
        self.prev[m] = self.positions[np.asarray(pos_idx)][m]
        self.row_values = np.zeros((self.N, len(STATEFUL_KINDS)), F32)        # the reset row reads 0.0 for both
        super().reset(pos_idx, mask)

    def fold(self, position, valuation):
        """One History row of every env: the running peak (compare-select) and age, and the row's stateful values."""
        position, valuation = np.asarray(position, F64), np.asarray(valuation, F64)
        self.peak = np.where(valuation > self.peak, valuation, self.peak)
        self.age = np.where(position != self.prev, 0.0, self.age + 1.0)
        self.prev = position
        self.row_values = np.stack([1.0 - valuation / self.peak, self.age], axis=1).astype(F32)
        self.step_values = self.row_values

    def step(self, pos_idx, real_position, valuation, reward, step, idx, ended, post_pos_idx):
        self.fold(self.positions[np.asarray(pos_idx)], valuation)
        super().step(pos_idx, real_position, valuation, reward, step, idx, ended, post_pos_idx)

    def select(self, vals, kinds):
        return vals[:, :, [ALL_KINDS.index(k) for k in kinds]]


class StatefulOracle(CatalogueOracle):
    """The CPU oracle with its dynamic columns replaced by a configuration that may hold the stateful kinds."""

    def __init__(self, oracle_env, kinds, max_episode_duration):
        super().__init__(oracle_env, kinds, max_episode_duration)
        o = oracle_env
        self.cols = StatefulColumns(o.num_envs, o.windows, o.positions, o._e.v0, max_episode_duration)
