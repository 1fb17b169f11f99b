"""CPU: the dynamic-feature catalogue (gte.DeviceFeature) against the reference goldens, the host-side parser, and
the C-ABI's validation of GteParams.dyn_kinds."""
import ctypes

import numpy as np
import pytest

from dyn_reference import CatalogueOracle, DynColumns, pos_after
from gym_trading_env_b200.dynamic_features import (KINDS, DeviceFeature, episode_progress_feature,
                                                   parse_dynamic_features, portfolio_return_feature, reward_feature)
from helpers import assert_bits, load_golden, make_oracle

GOLDENS = ["c3_windows_leveraged", "w64_fixed_start_holds", "multi_dataset_k3", "c1_single_nowindow",
           "reward_clipped_log_return"]
CONFIGS = [[k] for k in KINDS] + [["real_position", "position"],
                                  ["episode_progress", "reward", "position", "portfolio_return", "real_position"]]
DEFAULT = ["position", "real_position"]


def _dyn(window_vals, cols, kinds, windows):
    d = cols.select(window_vals, kinds)
    return d if windows is not None else d[:, 0]


def golden_construction(g):
    """Per recorded iteration: (obs dynamic rows [N, W, 5], terminal obs dynamic rows), built from the golden's recorded
    reference columns through the DeviceFeature callables.  Yields the reset observation first (k = -1)."""
    p = g["params"]
    N, pos = p["n_envs"], g["positions"]
    cols = DynColumns(N, p["windows"], pos, p["portfolio_initial_value"], p["max_episode_duration"])
    start, cur = g["plan"][:, 0, 0], g["plan"][:, 0, 1].astype(np.int64)
    cols.reset(cur)
    yield -1, cols, cols.window(start, start), None
    for k in range(g["actions"].shape[0]):
        ended = (g["terminated"][k] | g["truncated"][k]).astype(bool)
        pa = pos_after(g["actions"][k], cur, pos)
        assert (pa[~ended] == g["post_pos_idx"][k][~ended]).all()
        cols.step(pa, g["real_position"][k], g["valuation"][k], g["reward"][k], g["step"][k], g["idx"][k], ended,
                  g["post_pos_idx"][k])
        post_idx = g["post_idx"][k]
        yield k, cols, cols.window(post_idx, post_idx - g["post_step"][k]), cols.final
        cur = g["post_pos_idx"][k].astype(np.int64)


@pytest.mark.parametrize("name", GOLDENS)
def test_construction_reproduces_the_goldens_default_columns(name):
    g = load_golden(name)
    W, ns = g["params"]["windows"], g["features"].shape[2]
    for k, cols, vals, final in golden_construction(g):
        if k < 0:
            assert_bits(_dyn(vals, cols, DEFAULT, W), g["obs0"][..., ns:], "reset obs")
            continue
        assert_bits(_dyn(vals, cols, DEFAULT, W), g["obs"][k][..., ns:], f"step {k} obs")
        assert_bits(_dyn(final, cols, DEFAULT, W), g["step_obs"][k][..., ns:], f"step {k} terminal obs")


def _configs_for(g):
    mdd = g["params"]["max_episode_duration"]
    return [c for c in CONFIGS if "episode_progress" not in c or mdd != "max"]


@pytest.mark.parametrize("name", GOLDENS)
def test_oracle_catalogue_matches_the_construction_and_the_golden(name):
    g = load_golden(name)
    p = g["params"]
    W, ns = p["windows"], g["features"].shape[2]
    for kinds in _configs_for(g):
        orc = CatalogueOracle(make_oracle(g), kinds, p["max_episode_duration"])
        assert orc.o.n_dyn == 2          # the oracle runs the default pair; its static columns are checked below
        for k, cols, vals, final in golden_construction(g):
            if k < 0:
                obs = orc.reset()
                assert_bits(obs[..., :ns], g["obs0"][..., :ns], f"{kinds} reset static")
                assert_bits(obs[..., ns:], _dyn(vals, cols, kinds, W), f"{kinds} reset dynamic")
                continue
            obs = orc.step(g["actions"][k])
            assert_bits(obs[..., :ns], g["obs"][k][..., :ns], f"{kinds} step {k} static")
            assert_bits(obs[..., ns:], _dyn(vals, cols, kinds, W), f"{kinds} step {k} dynamic")
            assert_bits(orc.final_obs[..., ns:], _dyn(final, cols, kinds, W), f"{kinds} step {k} terminal dynamic")


def test_configurations_exercise_every_reset_row_and_nonzero_values():
    """The catalogue columns are not trivially zero on the goldens: every kind takes non-zero values."""
    g = load_golden("c3_windows_leveraged")
    seen = np.zeros(len(KINDS), bool)
    for k, cols, vals, _ in golden_construction(g):
        seen |= (vals != 0).any(axis=(0, 1))
    assert seen.all()


def test_device_feature_is_the_reference_expression():
    class H:
        def __init__(self, rows):
            self.rows = rows

        def __getitem__(self, key):
            return self.rows[key[1]][key[0]]
    h = H([{"portfolio_valuation": 1000.0, "step": 0},
           {"position": 1.0, "real_position": 0.75, "portfolio_valuation": 1012.5, "reward": 0.01, "step": 7}])
    h.rows = {0: h.rows[0], -1: h.rows[1]}
    assert DeviceFeature("position")(h) == 1.0
    assert DeviceFeature("real_position")(h) == 0.75
    assert portfolio_return_feature()(h) == 1012.5 / 1000.0 - 1
    assert reward_feature()(h) == 0.01
    assert episode_progress_feature(720)(h) == 7 / 720


def test_parse_accepts_the_catalogue_in_any_order():
    import gym_trading_env_b200 as gte
    assert parse_dynamic_features([], "max") == (0, 0)
    assert parse_dynamic_features([DeviceFeature("position"), DeviceFeature("real_position")], "max") == (2, 0x21)
    sentinels = [gte.dynamic_feature_last_position_taken, gte.dynamic_feature_real_position]
    assert parse_dynamic_features(sentinels, "max") == (2, 0x21)
    assert parse_dynamic_features(sentinels[::-1], 30) == (2, 0x12)
    five = [gte.dynamic_feature_real_position, episode_progress_feature(720), reward_feature(),
            DeviceFeature("position"), portfolio_return_feature()]
    assert parse_dynamic_features(five, 720) == (5, 0x31452)
    assert parse_dynamic_features(five, np.int64(720)) == (5, 0x31452)
    assert parse_dynamic_features([reward_feature()], "max") == (1, 0x4)


def test_parse_rejects_what_the_device_cannot_compute():
    with pytest.raises(NotImplementedError, match="portfolio_return"):      # the message lists the catalogue
        parse_dynamic_features([lambda h: h["close", -1]], "max")
    with pytest.raises(ValueError, match="at most once"):
        parse_dynamic_features([reward_feature(), reward_feature()], "max")
    with pytest.raises(ValueError, match="at most once"):
        parse_dynamic_features([DeviceFeature("position"), DeviceFeature("position")], "max")
    with pytest.raises(ValueError):
        parse_dynamic_features([episode_progress_feature(720)], "max")
    with pytest.raises(ValueError):
        parse_dynamic_features([episode_progress_feature(720)], 700)
    with pytest.raises(ValueError):
        parse_dynamic_features([DeviceFeature(k) for k in KINDS[:4]] + [episode_progress_feature(9), reward_feature()], 9)
    with pytest.raises(ValueError):
        episode_progress_feature("max")
    with pytest.raises(ValueError):
        episode_progress_feature(0)
    with pytest.raises(ValueError):
        DeviceFeature("drawdown")


def _params(n_dyn, dyn_kinds, max_episode_duration=-1):
    from gym_trading_env_b200 import _cabi
    p = _cabi.GteParams()
    p.n_envs, p.n_positions, p.windows, p.n_static = 64, 3, 8, 4
    p.n_dyn, p.dyn_kinds, p.max_episode_duration = n_dyn, dyn_kinds, max_episode_duration
    p.n_datasets, p.episodes_between_switch, p.t_stride, p.v0 = 1, 1, 100, 1000.0
    return p


@pytest.mark.parametrize("n_dyn,dyn_kinds,mdd", [
    (6, 0x123456, 50),     # more columns than GTE_MAX_DYN
    (1, 0, 50),            # the legacy 0 only means n_dyn 0 or 2
    (3, 0, 50),
    (2, 0x71, 50),         # kind code outside 1..5
    (1, 0x0, 50),
    (2, 0x11, 50),         # duplicate
    (2, 0x321, 50),        # a non-zero kind beyond n_dyn
    (0, 0x1, 50),
    (1, 0x5, -1),          # episode_progress without an int max_episode_duration
    (-1, 0, 50),
])
def test_malformed_dyn_kinds_are_rejected_before_any_cuda_call(n_dyn, dyn_kinds, mdd):
    """Host-side validation in the style of test_bad_arguments_are_rejected_before_any_cuda_call: the state's pointers
    are all NULL, so any launch would fault; -1 and a message naming dyn_kinds come back instead."""
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s = _params(n_dyn, dyn_kinds, mdd), _cabi.GteData(), _cabi.GteState()
    rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
    assert rc == -1 and b"dyn_kinds" in lib.gte_last_error()


@pytest.mark.parametrize("n_dyn,dyn_kinds,mdd", [(0, 0, -1), (2, 0, -1), (2, 0x21, -1), (2, 0x12, -1),
                                                 (5, 0x34152, 50), (1, 0x3, -1)])
def test_wellformed_dyn_kinds_pass_the_descriptor_check(n_dyn, dyn_kinds, mdd):
    """A valid descriptor gets past the dyn_kinds check (and fails later, on the NULL data pointers)."""
    from gym_trading_env_b200 import _cabi
    lib = _cabi.load()
    p, d, s = _params(n_dyn, dyn_kinds, mdd), _cabi.GteData(), _cabi.GteState()
    rc = lib.gte_reset(ctypes.byref(p), ctypes.byref(d), ctypes.byref(s), None, 0, None)
    assert rc == -1 and b"dyn_kinds" not in lib.gte_last_error() and b"price" in lib.gte_last_error()


@pytest.mark.parametrize("windows,n_dyn,dyn_kinds,expect", [
    (64, 2, 0, 64 * 160), (64, 2, 0x21, 64 * 160), (64, 2, 0x12, 64 * 160), (8, 1, 0x1, 8 * 32),
    (8, 1, 0x4, 8 * 128), (64, 5, 0x34152, 64 * (4 * 128 + 32)), (0, 4, 0x5432, 512)])
def test_ring_tile_bytes(windows, n_dyn, dyn_kinds, expect):
    from gym_trading_env_b200 import _cabi
    assert _cabi.ring_tile_bytes(windows, n_dyn, dyn_kinds) == expect
