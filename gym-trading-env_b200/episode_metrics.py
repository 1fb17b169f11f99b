"""The device catalogue of episode metrics: what ``TradingVectorEnv.add_metric(name, function)`` accepts.

The reference keeps, per env, the metrics of its most recently finished episode: "Market Return", "Portfolio Return" and
every ``function(history)`` registered with ``add_metric`` (environments.py:274-294).  Arbitrary Python callbacks cannot
run inside the CUDA step kernel, so this package accepts the kinds below.  Each is accumulated in the step kernel over
the episode's History (the reset row included) in IEEE fp64, in the reference's operation order, and recorded bit for
bit at the episode's end:

- ``position_changes``: ``int(np.sum(np.diff(np.asarray(h["position"], float)) != 0))``, the History rows whose position
  differs from the previous row's (a market trade undone by a limit order in the same step is no change);
- ``episode_length``: ``len(h["position"])``, the terminal step + 1;
- ``max_drawdown``: ``float(np.max(1 - v / np.maximum.accumulate(v)))``, ``v = h["portfolio_valuation"]``;
- ``episode_reward``: ``float(sum(h["reward"]))``, Python's left-to-right ``sum`` over the History's numpy column (not
  ``np.sum``, which adds pairwise);
- ``time_in_market``: ``float(np.mean(np.asarray(h["position"], float) != 0))``.

A :class:`DeviceMetric` is also callable on anything with column access (a reference ``History``, a
``tracked_history()`` DataFrame, a dict of arrays) and returns exactly that expression: it is the executable
specification of the device value (the env itself never calls it).
"""
from __future__ import annotations

import numpy as np

KINDS = ("position_changes", "episode_length", "max_drawdown", "episode_reward", "time_in_market")
KIND_INDEX = {k: i for i, k in enumerate(KINDS)}            # enum GteMetricKind (include/gte_b200.h)
INT_KINDS = ("position_changes", "episode_length")          # reported as Python ints
RECORD_RETURNS = ("Market Return", "Portfolio Return")      # rows 0 and 1 of the episode record, always kept


class DeviceMetric:
    """One episode metric computed inside the CUDA step kernel (see the module docstring for the catalogue)."""

    def __init__(self, kind):
        if kind not in KINDS:
            raise ValueError(f"kind must be one of {list(KINDS)}, got {kind!r}")
        self.kind = kind
        self.__name__ = f"metric_{kind}"

    def __call__(self, history):
        k = self.kind
        if k == "position_changes":
            return int(np.sum(np.diff(np.asarray(history["position"], float)) != 0))
        if k == "episode_length":
            return len(history["position"])
        if k == "max_drawdown":
            v = np.asarray(history["portfolio_valuation"], float)
            return float(np.max(1 - v / np.maximum.accumulate(v)))
        if k == "episode_reward":
            # sum() over the History's numpy column: one plain addition after another, left to right.  np.sum adds
            # pairwise, and since Python 3.12 sum() of plain Python floats is compensated; either can differ in the
            # last bits, so the column goes through float64 numpy scalars whatever container holds it
            return float(sum(np.asarray(history["reward"], float)))
        return float(np.mean(np.asarray(history["position"], float) != 0))

    def __eq__(self, other):
        return isinstance(other, DeviceMetric) and self.kind == other.kind

    def __hash__(self):
        return hash(("DeviceMetric", self.kind))

    def __repr__(self):
        return f"DeviceMetric({self.kind!r})"


def position_changes_metric():
    """How many History rows hold a different position than the row before (the reference README's metric)."""
    return DeviceMetric("position_changes")


def episode_length_metric():
    """``len(history["position"])``: the episode's rows, reset row included (the reference README's metric)."""
    return DeviceMetric("episode_length")


def max_drawdown_metric():
    """The largest fall of the portfolio valuation from its running peak, as a fraction of the peak."""
    return DeviceMetric("max_drawdown")


def episode_reward_metric():
    """The sum of the episode's rewards, added left to right as Python's ``sum`` does."""
    return DeviceMetric("episode_reward")


def time_in_market_metric():
    """The fraction of the episode's rows whose position is not 0."""
    return DeviceMetric("time_in_market")


def check_metric_function(function):
    """The kind of an ``add_metric`` function; NotImplementedError (listing the catalogue) for anything else."""
    if isinstance(function, DeviceMetric):
        return function.kind
    raise NotImplementedError(
        "add_metric only accepts the device catalogue: DeviceMetric(kind) for kind in "
        f"{list(KINDS)} (factories position_changes_metric(), episode_length_metric(), max_drawdown_metric(), "
        "episode_reward_metric(), time_in_market_metric()).  Arbitrary Python callbacks over a History cannot run "
        f"inside the CUDA step kernel and there is no CPU fallback; got {function!r}")


def metric_kinds_of(log_metrics):
    """``log_metrics`` (the ``{"name", "function"}`` entries of add_metric) -> GteParams.metric_kinds, bit 1 << kind."""
    bits = 0
    for m in log_metrics:
        bits |= 1 << KIND_INDEX[check_metric_function(m["function"])]
    return bits


def record_names(log_metrics):
    """Name -> row of the episode record, in the order of the reference's ``get_metrics()`` dict: the two returns, then
    each added name (a repeated name keeps its first place and takes the later function, as a dict assignment does)."""
    rows = {name: r for r, name in enumerate(RECORD_RETURNS)}
    for m in log_metrics:
        rows[m["name"]] = 2 + KIND_INDEX[m["function"].kind]
    return rows
