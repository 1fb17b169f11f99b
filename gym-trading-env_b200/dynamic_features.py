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

A :class:`DeviceFeature` is also callable on a reference ``History`` and returns exactly that expression: it is the
executable specification of the device column (the env itself never calls it).
"""
from __future__ import annotations

import numbers

KINDS = ("position", "real_position", "portfolio_return", "reward", "episode_progress")
KIND_CODES = {k: i + 1 for i, k in enumerate(KINDS)}       # enum GteDynKind (include/gte_b200.h)
MAX_DYN = len(KINDS)                                        # GTE_MAX_DYN

# the reference's two default functions (environments.py:20-24), passed back in by name
_SENTINEL_KINDS = {"dynamic_feature_last_position_taken": "position", "dynamic_feature_real_position": "real_position"}


def _is_int(x):
    return isinstance(x, numbers.Integral) and not isinstance(x, bool)


class DeviceFeature:
    """One dynamic-feature column computed inside the CUDA step kernel (see the module docstring for the catalogue).
    ``max_episode_duration`` is required by, and only by, ``kind="episode_progress"``."""

    def __init__(self, kind, max_episode_duration=None):
        if kind not in KINDS:
            raise ValueError(f"kind must be one of {list(KINDS)}")
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


def _kind_of(f):
    if isinstance(f, DeviceFeature):
        return f.kind
    kind = _SENTINEL_KINDS.get(getattr(f, "__name__", None))
    if kind is None:
        raise NotImplementedError(
            "dynamic_feature_functions may only hold the device catalogue: DeviceFeature(kind) for kind in "
            f"{list(KINDS)} (factories portfolio_return_feature(), reward_feature(), episode_progress_feature(D); "
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
        raise ValueError(f"at most {MAX_DYN} dynamic features (one per kind of {list(KINDS)}), got {len(fns)}")
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
