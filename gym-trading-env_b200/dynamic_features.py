"""The device catalogue of dynamic features: what ``dynamic_feature_functions`` may hold.

The reference evaluates each function of ``TradingEnv(dynamic_feature_functions=[...])`` on the History after every
step and writes the result, fp64 cast to float32, into the observation's last columns (environments.py:43-48,
:153-154).  Arbitrary Python callbacks cannot run inside the CUDA step kernel, so this package accepts the kinds below,
each computed on the device in fp64 in the reference's operation order, bit for bit:

- ``position``: ``history["position", -1]``; in an episode's first (reset) row the position;
- ``real_position``: ``history["real_position", -1]``; reset row: the position;
- ``portfolio_return``: ``history["portfolio_valuation", -1] / history["portfolio_valuation", 0] - 1``; reset row 0.0;
- ``reward``: ``history["reward", -1]``, the step's reward (0 when terminated); reset row 0.0;
- ``episode_progress``: ``history["step", -1] / D``, D = the env's int ``max_episode_duration``; reset row 0.0.

Two STATEFUL kinds depend on the whole episode.  The step kernel keeps their running state per env in the episode
accumulators it also keeps for ``add_metric`` (so they take the two-launch form of a windowed step, as metrics do):

- ``current_drawdown``: ``1 - v[-1] / np.max(v)``, v = ``history["portfolio_valuation"]``; reset row 0.0;
- ``position_age``: the number of History rows since the position last changed (by value, as the ``position_changes``
  metric compares rows: -0.0 equals 0.0, and a limit order that undoes the step's trade is no change), counted back to
  the reset row when it never changed; reset row 0.0.  A raw count, exact in float32 up to 2^24 rows.

A :class:`DeviceFeature` is also callable on a reference ``History`` and returns exactly that expression: it is the
executable specification of the device column (the env itself never calls it).
"""
from __future__ import annotations

import numbers

import numpy as np

KINDS = ("position", "real_position", "portfolio_return", "reward", "episode_progress")
STATEFUL_KINDS = ("current_drawdown", "position_age")      # keep per-env state in the episode accumulators
KIND_CODES = {k: i + 1 for i, k in enumerate(KINDS + STATEFUL_KINDS)}   # enum GteDynKind (include/gte_b200.h)
MAX_DYN = len(KINDS)                                        # GTE_MAX_DYN: columns per env

# the reference's two default functions (environments.py:20-24), passed back in by name
_SENTINEL_KINDS = {"dynamic_feature_last_position_taken": "position", "dynamic_feature_real_position": "real_position"}


def _is_int(x):
    return isinstance(x, numbers.Integral) and not isinstance(x, bool)


class DeviceFeature:
    """One dynamic-feature column computed inside the CUDA step kernel (see the module docstring for the catalogue).
    ``max_episode_duration`` is required by, and only by, ``kind="episode_progress"``."""

    def __init__(self, kind, max_episode_duration=None):
        if kind not in KIND_CODES:
            raise ValueError(f"kind must be one of {list(KIND_CODES)}")
        if kind == "episode_progress":
            if not _is_int(max_episode_duration) or max_episode_duration < 1:
                raise ValueError(f"episode_progress needs an int max_episode_duration >= 1, got {max_episode_duration!r}")
            max_episode_duration = int(max_episode_duration)
        elif max_episode_duration is not None:
            raise ValueError(f"{kind} takes no max_episode_duration")
        self.kind, self.max_episode_duration = kind, max_episode_duration
        self.__name__ = f"dynamic_feature_{kind}"

    def __call__(self, history):
        k = self.kind
        if k == "position":
            return history["position", -1]
        if k == "real_position":
            return history["real_position", -1]
        if k == "portfolio_return":
            return history["portfolio_valuation", -1] / history["portfolio_valuation", 0] - 1
        if k == "reward":
            return history["reward", -1]
        if k == "current_drawdown":
            v = np.asarray(history["portfolio_valuation"], float)
            return 1 - v[-1] / np.max(v)
        if k == "position_age":
            p = np.asarray(history["position"], float)
            ch = np.flatnonzero(p[1:] != p[:-1])
            return float(len(p) - 1 - (ch[-1] + 1 if len(ch) else 0))
        return history["step", -1] / self.max_episode_duration

    def __eq__(self, other):
        return isinstance(other, DeviceFeature) and (self.kind, self.max_episode_duration) == \
            (other.kind, other.max_episode_duration)

    def __hash__(self):
        return hash((self.kind, self.max_episode_duration))

    def __repr__(self):
        if self.kind == "episode_progress":
            return f"DeviceFeature('episode_progress', max_episode_duration={self.max_episode_duration})"
        return f"DeviceFeature({self.kind!r})"


def portfolio_return_feature():
    """``valuation[-1] / valuation[0] - 1``: the episode's portfolio return so far."""
    return DeviceFeature("portfolio_return")


def reward_feature():
    """The step's reward (after the DeviceReward's scale and clip; 0 when the step terminated)."""
    return DeviceFeature("reward")


def episode_progress_feature(max_episode_duration):
    """``step / max_episode_duration``: how far the episode has run.  The env's own ``max_episode_duration`` must be the
    same int."""
    return DeviceFeature("episode_progress", max_episode_duration)


def current_drawdown_feature():
    """``1 - valuation[-1] / max(valuation)``: how far the portfolio is below the episode's best valuation so far."""
    return DeviceFeature("current_drawdown")


def position_age_feature():
    """History rows since the position last changed (0 on the row where it changed and on the reset row)."""
    return DeviceFeature("position_age")


def _kind_of(f):
    if isinstance(f, DeviceFeature):
        return f.kind
    kind = _SENTINEL_KINDS.get(getattr(f, "__name__", None))
    if kind is None:
        raise NotImplementedError(
            "dynamic_feature_functions may only hold the device catalogue: DeviceFeature(kind) for kind in "
            f"{list(KINDS + STATEFUL_KINDS)} (factories portfolio_return_feature(), reward_feature(), "
            "episode_progress_feature(D), current_drawdown_feature(), position_age_feature(); "
            "dynamic_feature_last_position_taken / dynamic_feature_real_position are 'position' / 'real_position'). "
            "Arbitrary Python callbacks over a History cannot run inside the CUDA step kernel and there is no CPU "
            f"fallback; got {f!r}")
    return kind


def parse_dynamic_features(functions, max_episode_duration):
    """``dynamic_feature_functions`` -> ``(n_dyn, dyn_kinds)`` of GteParams: one 4-bit kind code per column, column j in
    bits 4j..4j+3.  Host-only (no device needed).  Raises NotImplementedError for a function outside the catalogue and
    ValueError for a duplicate kind, more than MAX_DYN columns, or an episode_progress whose D is not the env's
    int ``max_episode_duration``."""
    fns = list(functions)
    if len(fns) > MAX_DYN:
        raise ValueError(f"at most {MAX_DYN} dynamic features (each kind of {list(KIND_CODES)} at most once), "
                         f"got {len(fns)}")
    kinds = [_kind_of(f) for f in fns]
    for k in set(kinds):
        if kinds.count(k) > 1:
            raise ValueError(f"dynamic feature {k!r} appears {kinds.count(k)} times; each kind at most once")
    for f in fns:
        if isinstance(f, DeviceFeature) and f.kind == "episode_progress":
            if not _is_int(max_episode_duration) or int(max_episode_duration) != f.max_episode_duration:
                raise ValueError(f"episode_progress_feature({f.max_episode_duration}) needs the env's "
                                 f"max_episode_duration to be the same int, got {max_episode_duration!r}")
    code = 0
    for j, k in enumerate(kinds):
        code |= KIND_CODES[k] << (4 * j)
    return len(kinds), code


def stateful_kinds_of(n_dyn, dyn_kinds):
    """The stateful kinds among the n_dyn columns of a dyn_kinds code (parse_dynamic_features)."""
    codes = {(dyn_kinds >> (4 * j)) & 15 for j in range(n_dyn)}
    return [k for k in STATEFUL_KINDS if KIND_CODES[k] in codes]
