"""Episode-metric catalogue on the CPU: the History rebuilt from each golden is the one the reference saw, the
DeviceMetric callables are the reference's expressions on it, and bad configurations are refused on the host."""
from __future__ import annotations

import ctypes

import numpy as np
import pytest

from episode_reference import episode_histories, returns_of
from helpers import GOLDEN_NAMES, load_golden

import gym_trading_env_b200 as gte
from gym_trading_env_b200.episode_metrics import (KINDS, DeviceMetric, check_metric_function, metric_kinds_of,
                                                  record_names)


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_rebuilt_history_reproduces_the_recorded_returns(name):
    """Market and portfolio return of every finished episode, computed from the rebuilt History, equal the values the
    reference recorded at that step bit for bit: the reset row (start, position, dataset) and the step rows are the
    reference's own."""
    g = load_golden(name)
    n = 0
    for i, k, h in episode_histories(g, g["params"]["portfolio_initial_value"]):
        mr, pr = returns_of(h)
        assert _bits(mr) == _bits(g["market_return"][k, i]), f"{name} env {i} step {k} market return"
        assert _bits(pr) == _bits(g["portfolio_return"][k, i]), f"{name} env {i} step {k} portfolio return"
        assert len(h["position"]) == g["step"][k, i] + 1
        n += 1
    assert n == int((g["terminated"] | g["truncated"]).sum()) and n > 0


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_catalogue_equals_the_readme_lambdas(name):
    """position_changes and episode_length are the upstream README's own add_metric lambdas."""
    g = load_golden(name)
    for _, _, h in episode_histories(g, g["params"]["portfolio_initial_value"]):
        assert DeviceMetric("position_changes")(h) == np.sum(np.diff(h["position"]) != 0)
        assert DeviceMetric("episode_length")(h) == len(h["position"])
        v = h["portfolio_valuation"]
        dd = DeviceMetric("max_drawdown")(h)
        assert 0.0 <= dd < 1.0 and dd == float(np.max(1 - v / np.maximum.accumulate(v)))
        tim = DeviceMetric("time_in_market")(h)
        assert 0.0 <= tim <= 1.0
        r = 0
        for x in h["reward"]:
            r = r + x
        assert _bits(DeviceMetric("episode_reward")(h)) == _bits(r)


def test_position_changes_count_history_rows_not_trades():
    """limit_orders_persistent: a limit order moved the position in 26 steps; in 3 of them it undid the step's market
    trade, so the History row holds the previous position and the reference's np.diff counts no change there."""
    g = load_golden("limit_orders_persistent")
    positions = np.asarray(g["positions"], np.float64)
    K, N = g["actions"].shape
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    prev = positions[g["plan"][:, 0, 1]].copy()
    moved, undone, undone_at = 0, 0, []
    for k in range(K):
        a = g["actions"][k]
        market = np.where(a >= 0, positions[np.clip(a, 0, None)], prev)
        pos = g["position"][k]
        lim = pos != market
        moved += int(lim.sum())
        und = lim & (market != prev) & (pos == prev)
        undone += int(und.sum())
        undone_at += [(k, i) for i in np.flatnonzero(und)]
        prev = np.where(ended[k], positions[g["post_pos_idx"][k]], pos)
    assert (moved, undone) == (26, 3)
    # on exactly those steps a trade-counting metric would differ from the History-row count
    hist = {(i, k): h for i, k, h in episode_histories(g, g["params"]["portfolio_initial_value"])}
    for k0, i0 in undone_at:
        ends = [k for (i, k) in hist if i == i0 and k >= k0]
        if not ends:
            continue                              # the episode was still running when the recording stopped
        h = hist[(i0, min(ends))]
        trades = np.diff(h["position"]) != 0
        assert DeviceMetric("position_changes")(h) == int(trades.sum())


def test_device_metric_is_the_reference_expression():
    h = {"position": [0, 1, 1, 0, -1, -1], "portfolio_valuation": [1000.0, 1010.0, 990.0, 1020.0, 969.0, 1000.0],
         "reward": [0.0, 0.1, 0.2, 0.3, -0.1, 1e-17]}
    assert DeviceMetric("position_changes")(h) == 3
    assert DeviceMetric("episode_length")(h) == 6
    assert DeviceMetric("max_drawdown")(h) == max(1 - 990.0 / 1010.0, 1 - 969.0 / 1020.0)
    # left to right, one rounding per addition (not np.sum's pairwise order, not Python 3.12's compensated float sum)
    assert DeviceMetric("episode_reward")(h) == ((((0.0 + 0.1) + 0.2) + 0.3) - 0.1) + 1e-17
    assert DeviceMetric("time_in_market")(h) == 4 / 6
    assert gte.episode_reward_metric() == DeviceMetric("episode_reward")
    assert [f().kind for f in (gte.position_changes_metric, gte.episode_length_metric, gte.max_drawdown_metric,
                               gte.episode_reward_metric, gte.time_in_market_metric)] == list(KINDS)


def test_catalogue_parsing_errors():
    with pytest.raises(NotImplementedError, match="max_drawdown"):         # the message lists the catalogue
        check_metric_function(lambda history: 0)
    with pytest.raises(NotImplementedError):
        metric_kinds_of([{"name": "x", "function": np.sum}])
    with pytest.raises(ValueError):
        DeviceMetric("drawdown")
    log = [{"name": "Position Changes", "function": gte.position_changes_metric()},
           {"name": "Episode Length", "function": gte.episode_length_metric()},
           {"name": "Position Changes", "function": gte.time_in_market_metric()}]
    assert metric_kinds_of(log) == 0b10011
    # a repeated name keeps its place in the dict and takes the later function, as the reference's dict does
    assert record_names(log) == {"Market Return": 0, "Portfolio Return": 1, "Position Changes": 6, "Episode Length": 3}


def test_add_metric_after_reset_is_refused():
    """The host-side policy of add_metric, on a stand-in object (constructing an env needs a device)."""
    from gym_trading_env_b200.vector_env import TradingVectorEnv

    class Stub:
        _needs_first = False
    with pytest.raises(RuntimeError, match="before the first reset"):
        TradingVectorEnv.add_metric(Stub(), "Episode Length", gte.episode_length_metric())

    class Fresh:
        _needs_first = True
        log_metrics = []
    with pytest.raises(NotImplementedError):
        TradingVectorEnv.add_metric(Fresh(), "Position Changes", lambda h: 0)
    assert Fresh.log_metrics == []


_FAKE = 0x1000          # never dereferenced: the calls below must fail in host-side validation


def _structs(metric_kinds, acc=True, record=True):
    from gym_trading_env_b200 import _cabi
    p, d, s, o = _cabi.GteParams(), _cabi.GteData(), _cabi.GteState(), _cabi.GteStepOut()
    p.n_envs, p.n_positions, p.windows, p.n_static = 64, 3, 8, 4
    p.n_datasets, p.episodes_between_switch, p.t_stride, p.v0 = 1, 1, 100, 1000.0
    p.max_episode_duration, p.metric_kinds = -1, metric_kinds
    d.features, d.price, d.lengths = _FAKE, _FAKE, _FAKE
    for name, _ in _cabi.GteState._fields_:
        setattr(s, name, _FAKE)
    s.reset_plan, s.limit_price, s.limit_seq = None, None, None
    s.episode_acc = _FAKE if acc else None
    o.reward, o.terminated, o.truncated = _FAKE, _FAKE, _FAKE
    o.metric_partials, o.metrics_step, o.block_counter = _FAKE, _FAKE, _FAKE
    o.episode_record = _FAKE if record else None
    return p, d, s, o


@pytest.mark.parametrize("metric_kinds,acc,record,word", [
    (0x20, True, True, b"metric_kinds"),          # a bit outside the catalogue
    (-1, True, True, b"metric_kinds"),
    (0x1, False, True, b"episode_acc"),           # position_changes keeps state
    (0x1d, False, True, b"episode_acc"),
    (0x2, True, False, b"episode_record"),        # any kind needs the record
])
def test_bad_metric_configuration_is_rejected_before_any_cuda_call(metric_kinds, acc, record, word):
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s, o = _structs(metric_kinds, acc, record)
    rc = lib.gte_step(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), ctypes.c_void_p(_FAKE), ctypes.byref(o), 1, None)
    assert rc == -1
    msg = lib.gte_last_error()
    assert word in msg and b"metric_kinds" in msg, msg
    if record:                                     # gte_reset has no record: its check is the state's
        rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
        assert rc == -1 and word in lib.gte_last_error()


def test_episode_length_alone_needs_no_accumulators():
    """episode_length is the terminal step + 1: with it alone, episode_acc may be NULL (the metric check passes and the
    call fails on the next check, still on the host)."""
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s, o = _structs(0x2, acc=False, record=True)
    p.n_limit_positions = -1
    rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
    assert rc == -1 and b"metric_kinds" not in lib.gte_last_error() and b"n_limit_positions" in lib.gte_last_error()


def test_abi_constants_match_the_header():
    import os
    import re
    from gym_trading_env_b200 import _cabi
    hdr = open(os.path.join(_cabi.INCLUDE_DIR, "gte_b200.h")).read()
    for name in ("GTE_N_METRIC_KINDS", "GTE_METRIC_KINDS_ALL", "GTE_EPISODE_ACC_ROWS", "GTE_EPISODE_RECORD_ROWS"):
        assert int(re.search(rf"#define {name} (\w+)", hdr).group(1), 0) == getattr(_cabi, name)
    stateful = sum(1 << KINDS.index(k) for k in KINDS if k != "episode_length")
    assert _cabi.GTE_METRIC_KINDS_STATEFUL == stateful
    assert [k.upper() for k in KINDS] == re.findall(r"GTE_METRIC_(\w+) = \d", hdr)
