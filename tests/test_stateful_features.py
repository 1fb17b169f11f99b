"""CPU: the stateful dynamic features (current_drawdown, position_age): the DeviceFeature callables are the reference
expressions on hand-worked Histories, the running-state reference equals them on every History prefix of every golden,
and the parser and the C-ABI accept and refuse what they should."""
import ctypes
import os
import re

import numpy as np
import pytest

from helpers import GOLDEN_NAMES, load_golden
from stateful_reference import StatefulColumns, prefix_values

import gym_trading_env_b200 as gte
from gym_trading_env_b200.dynamic_features import (KIND_CODES, KINDS, STATEFUL_KINDS, DeviceFeature,
                                                   parse_dynamic_features)

DD, AGE = gte.current_drawdown_feature(), gte.position_age_feature()


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


def _h(position, valuation):
    return {"position": np.asarray(position, float), "portfolio_valuation": np.asarray(valuation, float)}


def test_factories_and_codes():
    assert DD == DeviceFeature("current_drawdown") and AGE == DeviceFeature("position_age")
    assert STATEFUL_KINDS == ("current_drawdown", "position_age")
    assert (KIND_CODES["current_drawdown"], KIND_CODES["position_age"]) == (6, 7)
    assert [KIND_CODES[k] for k in KINDS] == [1, 2, 3, 4, 5]


def test_reset_row_reads_positive_zero():
    h = _h([0.5], [1000.0])
    assert _bits(DD(h)) == _bits(0.0) and _bits(AGE(h)) == _bits(0.0)


def test_new_peak_and_drawdown_from_it():
    assert DD(_h([1, 1, 1], [1000.0, 1010.0, 990.0])) == 1 - 990.0 / 1010.0
    assert _bits(DD(_h([1, 1, 1, 1], [1000.0, 1010.0, 990.0, 1020.0]))) == _bits(0.0)      # a new peak
    assert DD(_h([1, 1, 1, 1, 1], [1000.0, 1010.0, 990.0, 1020.0, 969.0])) == 1 - 969.0 / 1020.0
    assert DD(_h([1, 1], [1000.0, 900.0])) == 1 - 900.0 / 1000.0                              # the reset row is the peak


def test_flat_position_held_and_changes():
    assert AGE(_h([1, 1, 1, 1], [1000.0] * 4)) == 3.0                  # held since the reset row
    assert AGE(_h([0, 1, 1, 1], [1000.0] * 4)) == 2.0
    assert AGE(_h([0, 1, 1, 0], [1000.0] * 4)) == 0.0                  # changed on the last row
    assert AGE(_h([0, 1, 0, 1, 1], [1000.0] * 5)) == 1.0


def test_negative_zero_equals_zero():
    assert AGE(_h([0.0, -0.0, 0.0, -0.0], [1000.0] * 4)) == 3.0


def _limit_order_undos(g):
    """(k, i) of the steps in which a limit order undid that step's market trade (History row = the previous position)."""
    positions = np.asarray(g["positions"], np.float64)
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    prev = positions[g["plan"][:, 0, 1]].copy()
    out = []
    for k in range(g["actions"].shape[0]):
        a = g["actions"][k]
        market = np.where(a >= 0, positions[np.clip(a, 0, None)], prev)
        pos = g["position"][k]
        out += [(k, i) for i in np.flatnonzero((pos != market) & (market != prev) & (pos == prev))]
        prev = np.where(ended[k], positions[g["post_pos_idx"][k]], pos)
    return out


def test_limit_order_that_undoes_the_trade_is_no_change():
    """limit_orders_persistent: in 3 steps a limit order undid the step's market trade.  The History row holds the
    previous position, so position_age keeps counting there (the step row is not a change)."""
    g = load_golden("limit_orders_persistent")
    undone = _limit_order_undos(g)
    assert len(undone) == 3
    vals = prefix_values(g, g["params"]["portfolio_initial_value"])
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    for k, i in undone:
        assert k > 0 and not ended[k - 1, i]
        assert vals[k, i, 1] == vals[k - 1, i, 1] + 1, (k, i)


@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_running_state_equals_the_callables_on_every_prefix(name):
    """The per-env peak and age the device keeps give, on every step of every golden, the callables' values on the
    whole History prefix, bit for bit (float32)."""
    g = load_golden(name)
    p = g["params"]
    K, N = g["actions"].shape
    expect = prefix_values(g, p["portfolio_initial_value"])
    cols = StatefulColumns(N, p["windows"], g["positions"], p["portfolio_initial_value"], p["max_episode_duration"])
    cols.reset(g["plan"][:, 0, 1].astype(np.int64))
    ended = (g["terminated"] | g["truncated"]).astype(bool)
    for k in range(K):
        cols.fold(g["position"][k], g["valuation"][k])
        assert cols.step_values.tobytes() == expect[k].tobytes(), f"{name} step {k}"
        cols.reset(g["post_pos_idx"][k].astype(np.int64), ended[k])
    assert (expect[..., 1] > 0).any() and (expect[..., 0] > 0).any()


def test_parse_accepts_the_stateful_kinds_in_any_order():
    assert parse_dynamic_features([DD], "max") == (1, 0x6)
    assert parse_dynamic_features([AGE], "max") == (1, 0x7)
    assert parse_dynamic_features([AGE, DD], "max") == (2, 0x67)
    pair = [gte.dynamic_feature_last_position_taken, gte.dynamic_feature_real_position]
    assert parse_dynamic_features(pair + [DD, AGE], "max") == (4, 0x7621)
    assert parse_dynamic_features([AGE, gte.reward_feature(), DD, gte.episode_progress_feature(9)], 9) == (4, 0x5647)
    five = [DeviceFeature("real_position"), gte.portfolio_return_feature(), gte.reward_feature(), DD, AGE]
    assert parse_dynamic_features(five, "max") == (5, 0x76432)


def test_parse_rejects_duplicates_a_sixth_column_and_lists_all_seven_kinds():
    with pytest.raises(ValueError, match="at most once"):
        parse_dynamic_features([DD, DD], "max")
    with pytest.raises(ValueError, match="at most once"):
        parse_dynamic_features([AGE, gte.reward_feature(), AGE], "max")
    with pytest.raises(ValueError, match="at most 5"):
        parse_dynamic_features([DeviceFeature(k) for k in KINDS[:4]] + [DD, AGE], "max")
    with pytest.raises(NotImplementedError) as e:
        parse_dynamic_features([lambda h: h["close", -1]], "max")
    for k in KINDS + STATEFUL_KINDS + ("current_drawdown_feature()", "position_age_feature()"):
        assert k in str(e.value), k
    with pytest.raises(ValueError):
        DeviceFeature("current_drawdown", max_episode_duration=10)


def _params(n_dyn, dyn_kinds):
    from gym_trading_env_b200 import _cabi
    p = _cabi.GteParams()
    p.n_envs, p.n_positions, p.windows, p.n_static = 64, 3, 8, 4
    p.n_dyn, p.dyn_kinds, p.max_episode_duration = n_dyn, dyn_kinds, 50
    p.n_datasets, p.episodes_between_switch, p.t_stride, p.v0 = 1, 1, 100, 1000.0
    return p


@pytest.mark.parametrize("n_dyn,dyn_kinds", [(1, 0x6), (1, 0x7), (2, 0x67), (4, 0x7621), (5, 0x76432)])
def test_stateful_kinds_need_episode_acc(n_dyn, dyn_kinds):
    """Without episode_acc the call is refused on the host naming dyn_kinds; with it the descriptor check passes (the
    call then fails on the NULL data pointers, still on the host)."""
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s = _params(n_dyn, dyn_kinds), _cabi.GteData(), _cabi.GteState()
    rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
    msg = lib.gte_last_error()
    assert rc == -1 and msg.split(b"bad argument: ")[1].startswith(b"dyn_kinds:") and b"episode_acc" in msg, msg
    s.episode_acc = 0x1000                     # never dereferenced
    rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
    msg = lib.gte_last_error()
    assert rc == -1 and b"dyn_kinds" not in msg and b"price" in msg, msg


def test_code_eight_is_outside_the_catalogue():
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s = _params(2, 0x81), _cabi.GteData(), _cabi.GteState()
    s.episode_acc = 0x1000
    assert lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None) == -1
    assert b"dyn_kinds: kind code outside 1..7" in lib.gte_last_error()


def test_ring_tile_of_five_f32_columns():
    from gym_trading_env_b200 import _cabi
    assert _cabi.ring_tile_bytes(64, 5, 0x76432) == 64 * 640
    assert _cabi.ring_tile_bytes(64, 4, 0x7621) == 64 * (3 * 128 + 32)


def test_header_constants_match_the_binding():
    from gym_trading_env_b200 import _cabi
    hdr = open(os.path.join(_cabi.INCLUDE_DIR, "gte_b200.h")).read()
    enum = dict((k, int(v)) for k, v in re.findall(r"GTE_DYN_(\w+) = (\d+)", hdr))
    assert enum == {k.upper(): KIND_CODES[k] for k in KIND_CODES}
    assert enum["CURRENT_DRAWDOWN"] == _cabi.GTE_DYN_CURRENT_DRAWDOWN and enum["POSITION_AGE"] == _cabi.GTE_DYN_POSITION_AGE
    assert int(re.search(r"#define GTE_EPISODE_ACC_ROWS (\d+)", hdr).group(1)) == _cabi.GTE_EPISODE_ACC_ROWS == 6
    assert int(re.search(r"GTE_ACC_POSITION_AGE = (\d+)", hdr).group(1)) == _cabi.GTE_ACC_POSITION_AGE == 5
    assert int(re.search(r"#define GTE_MAX_DYN (\d+)", hdr).group(1)) == _cabi.GTE_MAX_DYN == 5
