"""Reference for the episode-metric catalogue: the reference's per-episode History, rebuilt from recorded streams.

An episode's History (environments.py:186-197, :253-264) is its reset row — the start row and position of the reset,
valuation portfolio_initial_value, reward 0 — followed by one row per step.  `episode_histories` rebuilds it for every
finished episode of a golden (or of any run recorded in the same arrays): the reset row from the plan (first episode) or
the auto-reset's post_* columns, the step rows from the recorded position / valuation / reward / idx.  The DeviceMetric
callables evaluated on these Histories are the values the device must record, bit for bit.
"""
from __future__ import annotations

import numpy as np

from gym_trading_env_b200.episode_metrics import KINDS, DeviceMetric

METRICS = [DeviceMetric(k) for k in KINDS]


def episode_histories(g, v0):
    """Yield (env, terminal step index k, History dict) for every episode that ended within the recorded steps.
    g: arrays actions/position/valuation/reward/idx/terminated/truncated/post_idx/post_pos_idx/post_dataset [K, N],
    plan [N, E, 3], positions [P], price [n_ds, T]."""
    K, N = g["actions"].shape
    positions = np.asarray(g["positions"], np.float64)
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    for i in range(N):
        start, pidx, ds = (int(x) for x in g["plan"][i, 0])
        rows = {"position": [positions[pidx]], "portfolio_valuation": [float(v0)], "reward": [0.0],
                "close": [g["price"][ds, start]]}
        for k in range(K):
            rows["position"].append(g["position"][k, i])
            rows["portfolio_valuation"].append(g["valuation"][k, i])
            rows["reward"].append(g["reward"][k, i])
            rows["close"].append(g["price"][ds, g["idx"][k, i]])
            if ended[k, i]:
                yield i, k, {c: np.asarray(v, np.float64) for c, v in rows.items()}
                start, pidx, ds = int(g["post_idx"][k, i]), int(g["post_pos_idx"][k, i]), int(g["post_dataset"][k, i])
                rows = {"position": [positions[pidx]], "portfolio_valuation": [float(v0)], "reward": [0.0],
                        "close": [g["price"][ds, start]]}


def returns_of(h):
    """The two values the reference always records (environments.py:281-282), as fractions."""
    c, v = h["close"], h["portfolio_valuation"]
    return c[-1] / c[0] - 1, v[-1] / v[0] - 1


def record_of(h):
    """The 7 rows of GteStepOut.episode_record for a finished episode's History (every kind configured)."""
    mr, pr = returns_of(h)
    return np.array([mr, pr] + [float(m(h)) for m in METRICS], np.float64)
