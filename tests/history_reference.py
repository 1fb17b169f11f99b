"""The reference's History rows (environments.py:186-197 for reset(), :253-264 for step()) rebuilt from what the goldens
and the C oracle record — NO GPU code.

A History row, as `infos`, the tracked log (`track()` / `tracked_history()`) and `save_for_render()` expose it, holds:
``idx, step, position_index, position, real_position, portfolio_valuation, portfolio_distribution_* (6), reward`` and,
in this project, ``dataset_idx``.  ``data_<col>`` and ``date`` are lookups at (dataset_idx, idx).

* The step row: ``position_index`` is the action (hold -> -1, the reference's None; an action outside
  ``[0, len(positions))`` is a hold in the kernels, so -1 too); ``position`` is ``self._position`` after the market
  trade AND the limit orders; the distribution is ``portfolio.get_portfolio_distribution()`` (portfolio.py:49-57).
* The reset row: ``step`` 0, ``position_index = positions.index(position)`` (the FIRST index holding an equal value),
  ``position`` and ``real_position`` the position, ``portfolio_valuation = portfolio_initial_value``, reward and
  interest 0.

Rows are dicts of column -> [N] arrays (one entry per env).
"""
from __future__ import annotations

import numpy as np

DIST = ["asset", "fiat", "borrowed_asset", "borrowed_fiat", "interest_asset", "interest_fiat"]
COLS = (["idx", "step", "position_index", "position", "real_position", "portfolio_valuation"]
        + ["portfolio_distribution_" + d for d in DIST] + ["reward", "dataset_idx"])
INT_COLS = ("idx", "step", "position_index", "dataset_idx")


def pymax0(x):
    """Python's ``max(0, x)`` elementwise, as a float: 0 wins unless x > 0 (so -0.0 and NaN read +0.0)."""
    x = np.asarray(x, np.float64)
    return np.where(x > 0, x, 0.0)


def distribution(asset, fiat, interest_asset, interest_fiat):
    """``Portfolio.get_portfolio_distribution()`` (portfolio.py:49-57) as six [N] columns."""
    asset, fiat = np.asarray(asset, np.float64), np.asarray(fiat, np.float64)
    return {"portfolio_distribution_asset": pymax0(asset), "portfolio_distribution_fiat": pymax0(fiat),
            "portfolio_distribution_borrowed_asset": pymax0(-asset), "portfolio_distribution_borrowed_fiat": pymax0(-fiat),
            "portfolio_distribution_interest_asset": np.array(interest_asset, np.float64),
            "portfolio_distribution_interest_fiat": np.array(interest_fiat, np.float64)}


def valorisation(asset, fiat, interest_asset, interest_fiat, price):
    """``Portfolio.valorisation`` (portfolio.py:7-13) with Python floats, in its own operation order."""
    return np.array([sum([a * p, f, -ia * p, -ifi]) for a, f, ia, ifi, p in
                     zip(*(np.broadcast_arrays(*(np.asarray(x, np.float64) for x in
                                                 (asset, fiat, interest_asset, interest_fiat, price)))))])


def first_index(positions, pos_idx):
    """``positions.index(positions[k])`` for every k in `pos_idx`."""
    positions = [float(p) for p in positions]
    return np.array([positions.index(positions[int(k)]) for k in np.ravel(pos_idx)], np.int64).reshape(np.shape(pos_idx))


def action_index(actions, n_positions):
    a = np.asarray(actions, np.int64)
    return np.where((a >= 0) & (a < n_positions), a, -1)


def reset_row(positions, v0, idx, pos_idx, asset, fiat, dataset_idx, interest_asset=None, interest_fiat=None):
    """The row reset() writes (environments.py:186-197)."""
    positions = np.asarray(positions, np.float64)
    pos_idx = np.asarray(pos_idx, np.int64)
    z = np.zeros(pos_idx.shape, np.float64)
    pos = positions[pos_idx]
    row = {"idx": np.asarray(idx, np.int64), "step": np.zeros(pos_idx.shape, np.int64),
           "position_index": first_index(positions, pos_idx), "position": pos, "real_position": pos.copy(),
           "portfolio_valuation": z + v0, "reward": z.copy(), "dataset_idx": np.asarray(dataset_idx, np.int64)}
    row.update(distribution(asset, fiat, z if interest_asset is None else interest_asset,
                            z if interest_fiat is None else interest_fiat))
    return row


def step_row(positions, idx, step, actions, position, real_position, valuation, asset, fiat, interest_asset,
             interest_fiat, reward, dataset_idx):
    """The row step() adds (environments.py:253-264): the terminal values where the episode ended."""
    row = {"idx": np.asarray(idx, np.int64), "step": np.asarray(step, np.int64),
           "position_index": action_index(actions, len(positions)), "position": np.array(position, np.float64),
           "real_position": np.array(real_position, np.float64), "portfolio_valuation": np.array(valuation, np.float64),
           "reward": np.array(reward, np.float64), "dataset_idx": np.asarray(dataset_idx, np.int64)}
    row.update(distribution(asset, fiat, interest_asset, interest_fiat))
    return row


def where(mask, a, b):
    """Row `a` where `mask`, else row `b`."""
    return {c: np.where(mask, a[c], b[c]) for c in a}


# ---- goldens ------------------------------------------------------------------------------------------------------

class GoldenHistory:
    """History rows of every env of a golden run (oracle/ref_harness.py records the step row's values and the
    post-reset state of every step)."""

    def __init__(self, g):
        self.g = g
        p = g["params"]
        self.positions = [float(x) for x in g["positions"]]
        self.v0 = float(p["portfolio_initial_value"])
        self.K, self.N = g["actions"].shape
        self.multi = bool(p.get("multi_dataset", False))

    def dataset_before(self, k):
        """Dataset of each env's episode during step k (a dataset only changes at a reset)."""
        g = self.g
        if not self.multi:
            return np.zeros(self.N, np.int64)
        return (g["plan"][:, 0, 2] if k == 0 else g["post_dataset"][k - 1]).astype(np.int64)

    def initial_reset(self):
        g = self.g
        plan = g["plan"][:, 0]
        return reset_row(self.positions, self.v0, plan[:, 0], plan[:, 1], g["init_asset"], g["init_fiat"],
                         plan[:, 2] if self.multi else np.zeros(self.N, np.int64))

    def step(self, k):
        g = self.g
        return step_row(self.positions, g["idx"][k], g["step"][k], g["actions"][k], g["position"][k],
                        g["real_position"][k], g["valuation"][k], g["asset"][k], g["fiat"][k], g["interest_asset"][k],
                        g["interest_fiat"][k], g["reward"][k], self.dataset_before(k))

    def ended(self, k):
        return (self.g["terminated"][k] | self.g["truncated"][k]).astype(bool)

    def reset_after(self, k):
        """The reset row of the episode the auto-reset of step k started (meaningful where `ended(k)`)."""
        g = self.g
        return reset_row(self.positions, self.v0, g["post_idx"][k], g["post_pos_idx"][k], g["post_asset"][k],
                         g["post_fiat"][k], g["post_dataset"][k] if self.multi else np.zeros(self.N, np.int64),
                         g["post_interest_asset"][k], g["post_interest_fiat"][k])

    def infos_after(self, k):
        """History's last row after step k: the new episode's reset row where the episode ended (SAME_STEP)."""
        return where(self.ended(k), self.reset_after(k), self.step(k))

    def log(self, env, steps=None):
        """Every History row env `env` wrote, in order, with ``new_episode`` / ``terminated`` / ``truncated`` — what
        ``tracked_history()`` returns for it."""
        K = self.K if steps is None else steps
        rows = [_one(self.initial_reset(), env, new=True)]
        for k in range(K):
            rows.append(_one(self.step(k), env, term=self.g["terminated"][k, env], trunc=self.g["truncated"][k, env]))
            if self.ended(k)[env]:
                rows.append(_one(self.reset_after(k), env, new=True))
        return frame(rows)


def _one(row, env, new=False, term=False, trunc=False):
    r = {c: v[env] for c, v in row.items()}
    r.update(new_episode=bool(new), terminated=bool(term), truncated=bool(trunc))
    return r


def frame(rows):
    """A list of one-env rows -> dict of column arrays."""
    out = {}
    for c in COLS + ["new_episode", "terminated", "truncated"]:
        dt = np.int64 if c in INT_COLS else (bool if c in ("new_episode", "terminated", "truncated") else np.float64)
        out[c] = np.array([r[c] for r in rows], dtype=dt)
    return out


def episodes(log):
    """(start, stop) row ranges of the episodes of a log, and which of them finished."""
    starts = list(np.flatnonzero(log["new_episode"])) + [len(log["new_episode"])]
    eps = list(zip(starts[:-1], starts[1:]))
    done = [(a, b) for a, b in eps if log["terminated"][b - 1] or log["truncated"][b - 1]]
    return eps, done


# ---- the C oracle -------------------------------------------------------------------------------------------------

class OracleHistory:
    """History rows from an `oracle.OracleVecEnv` run driven alongside a device env: call `before_step()` then the
    oracle's step, then `after_step(actions)`; `after_reset(mask)` after a reset.  Limit orders are not replayed (the
    step row's position is the action's target unless the action holds or targets an equal value)."""

    def __init__(self, o, v0, log_ids=None):
        self.o, self.v0 = o, float(v0)
        self.positions = [float(x) for x in o.positions]
        self.rows = None           # the current History last row of every env
        self.log = [[] for _ in range(o.num_envs)]
        self.log_ids = range(o.num_envs) if log_ids is None else list(log_ids)     # the envs whose log is kept

    def current_reset_rows(self):
        o = self.o
        return reset_row(self.positions, self.v0, o.idx, o.pos_idx, o.asset, o.fiat, o.dataset_idx,
                         o.interest_asset, o.interest_fiat)

    def after_reset(self, mask=None):
        m = np.ones(self.o.num_envs, bool) if mask is None else np.asarray(mask, bool)
        new = self.current_reset_rows()
        self.rows = new if self.rows is None else where(m, new, self.rows)
        for i in self.log_ids:
            if m[i]:
                self.log[i].append(_one(new, i, new=True))

    def before_step(self):
        self._pre = (self.o.pos_idx.copy(), self.o.dataset_idx.copy())

    def after_step(self, actions, autoreset=True):
        o = self.o
        pre_pos, pre_ds = self._pre
        a = action_index(actions, len(self.positions))
        pos_tab = np.asarray(self.positions, np.float64)
        moved = (a >= 0) & (pos_tab[np.maximum(a, 0)] != pos_tab[pre_pos])
        position = pos_tab[np.where(moved, a, pre_pos)]
        fs = o.final_state
        st = step_row(self.positions, o.info_idx, o.info_step, actions, position, o.real_position, o.valuation,
                      fs[:, 0], fs[:, 1], fs[:, 2], fs[:, 3], o.reward, pre_ds)
        ended = (o.terminated | o.truncated).astype(bool)
        rs = self.current_reset_rows()
        reset_now = ended & autoreset
        self.rows = where(reset_now, rs, st)
        for i in self.log_ids:
            self.log[i].append(_one(st, i, term=o.terminated[i], trunc=o.truncated[i]))
            if reset_now[i]:
                self.log[i].append(_one(rs, i, new=True))
        return st

    def history(self, env):
        return frame(self.log[env])
