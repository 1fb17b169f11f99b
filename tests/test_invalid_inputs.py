"""CPU: the reference of the error-bit contract (invalid_inputs.py) on hand-built cases at every range edge, and against
the CPU oracle where the contract says an invalid input stands for a valid one."""
import numpy as np
import pytest

import invalid_inputs as V
import oracle as orc

P = 5
WIDTHS = [np.int8, np.int16, np.int32, np.int64]


# ---- actions -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", WIDTHS)
def test_hold_substitution_at_the_edges(dtype):
    info = np.iinfo(dtype)
    a = np.array([info.min, -2, -1, 0, P - 1, P, P + 1, info.max], dtype)
    for strict, bits in ((False, V.E_ACTION_RANGE), (True, V.E_ACTION_RANGE | V.E_NEGATIVE_ACTION)):
        valid, got = V.hold_substituted(a, P, strict)
        assert valid.dtype == a.dtype
        assert valid.tolist() == [-1, -1, -1, 0, P - 1, -1, -1, -1]
        assert got == bits
    neg = np.array([-1, info.min, 0], dtype)
    assert V.hold_substituted(neg, P, False)[1] == 0
    assert V.hold_substituted(neg, P, True)[1] == V.E_NEGATIVE_ACTION
    big = np.array([P, -1], dtype)
    assert V.hold_substituted(big, P, False)[1] == V.hold_substituted(big, P, True)[1] == V.E_ACTION_RANGE


@pytest.mark.parametrize("dtype", WIDTHS)
@pytest.mark.parametrize("strict", [False, True])
def test_hold_substitution_is_the_identity_on_valid_input(dtype, strict):
    a = np.random.default_rng(1).integers(-1, P, size=1000).astype(dtype)
    valid, bits = V.hold_substituted(a, P, strict)
    assert bits == 0 and valid.dtype == a.dtype and np.array_equal(valid, a)


# ---- reset plans -------------------------------------------------------------------------------------------------------
def test_clamped_plan_at_every_range_edge():
    W, lengths = 8, [100, 60]
    rows = [  # (start, position, dataset) -> expected (multi), flagged
        ((W - 2, 0, 0), (W - 1, 0, 0), True),
        ((W - 1, 0, 0), (W - 1, 0, 0), False),
        ((98, 1, 0), (98, 1, 0), False),                # T-2 of dataset 0
        ((99, 1, 0), (98, 1, 0), True),                 # T-1
        ((58, 1, 1), (58, 1, 1), False),                # T-2 of the shorter dataset 1
        ((59, 1, 1), (58, 1, 1), True),
        ((-(1 << 30), 2, 1), (W - 1, 2, 1), True),
        ((20, -1, 0), (20, 0, 0), True),
        ((20, P, 0), (20, P - 1, 0), True),
        ((20, P - 1, -1), (20, P - 1, 0), True),
        ((80, 0, 2), (58, 0, 1), True),                 # dataset n_ds -> the last one, whose T bounds the start
        ((1 << 30, P, 7), (58, P - 1, 1), True),
    ]
    plan = np.array([[r[0] for r in rows]], np.int32)
    got, bits = V.clamped_plan(plan, lengths, W, P, 2, multi=True)
    assert got[0].tolist() == [list(r[1]) for r in rows]
    assert bits[0].tolist() == [V.E_PLAN_RANGE if r[2] else 0 for r in rows]


def test_clamped_plan_single_dataset_and_no_window():
    plan = np.array([[[0, 0, 0], [0, 0, 1], [0, 0, -1], [98, 0, 0], [99, 0, 0], [-1, 0, 0]]], np.int32)
    got, bits = V.clamped_plan(plan, [100], None, P, 1, multi=False)
    assert got[0].tolist() == [[0, 0, 0], [0, 0, 0], [0, 0, 0], [98, 0, 0], [98, 0, 0], [0, 0, 0]]
    assert (bits[0] != 0).tolist() == [False, True, True, False, True, True]     # dataset ignored, still flagged


def test_wrapped_plan():
    plan = np.arange(2 * 3 * 3, dtype=np.int32).reshape(2, 3, 3)
    tiled, first = V.wrapped_plan(plan, 3)
    assert first is None and np.array_equal(tiled, plan)
    tiled, first = V.wrapped_plan(plan, 7)
    assert first == 3 and tiled.shape == (2, 7, 3)
    assert np.array_equal(tiled[:, 3:6], plan) and np.array_equal(tiled[:, 6], plan[:, 0])


def _series(T, seed):
    rng = np.random.default_rng(seed)
    price = 100.0 * np.exp(np.cumsum(rng.normal(0, 0.01, T)))
    feats = np.stack([np.arange(T) / 64.0, price], axis=1).astype(np.float32)
    return feats, price


def test_the_oracle_on_a_clamped_plan_equals_it_on_the_equivalent_valid_plan():
    W, T, N, E = 4, 120, 6, 4
    feats, price = _series(T, 3)
    bad = np.zeros((N, E, 3), np.int32)
    bad[:, :, 0] = 40
    bad[0, 0] = (-5, 0, 0)
    bad[1, 1] = (500, 1, 0)
    bad[2, 2] = (30, -3, 4)
    bad[3, 0] = (T - 1, 9, -1)
    valid = bad.copy()
    valid[0, 0], valid[1, 1], valid[2, 2], valid[3, 0] = (W - 1, 0, 0), (T - 2, 1, 0), (30, 0, 0), (T - 2, 2, 0)
    got, bits = V.clamped_plan(bad, [T], W, 3, 1, multi=False)
    assert np.array_equal(got, valid)
    assert np.argwhere(bits).tolist() == [[0, 0], [1, 1], [2, 2], [3, 0]]
    kw = dict(num_envs=N, positions=[-1, 0, 1], windows=W, trading_fees=1e-4, borrow_interest_rate=3e-6,
              max_episode_duration=6)
    a, b = orc.OracleVecEnv(feats, price, plan=got, **kw), orc.OracleVecEnv(feats, price, plan=valid, **kw)
    assert np.array_equal(a.reset().view(np.uint32), b.reset().view(np.uint32))
    rng = np.random.default_rng(0)
    for k in range(15):
        acts = rng.integers(-1, 3, size=N)
        sub, _ = V.hold_substituted(np.where(acts < 0, -7, acts), 3, True)   # negative holds, substituted
        a.step(sub)
        b.step(acts)
        for n in ("obs", "reward", "valuation", "terminated", "truncated", "asset", "fiat", "ep_start"):
            assert np.array_equal(getattr(a, n), getattr(b, n)), (k, n)


# ---- past the end -------------------------------------------------------------------------------------------------------
POS = [1.0, 0.0, -1.0, 2.0]
SIMPLE = ("simple_return", 1.0, -np.inf, np.inf)


def test_past_end_step_on_hand_built_portfolios():
    # long 1 with no fee / interest: asset 1, fiat 0 -> valuation = price
    r = V.past_end_step((1.0, 0.0, 0.0, 0.0), 0, -1, 120.0, 126.0, positions=POS, fee=0.0, rate=0.0, v0=100.0,
                        started_at_t2=False, reward=SIMPLE)
    assert r["valuation"] == 126.0 and r["reward"] == (126.0 - 120.0) / 120.0 and r["real_position"] == 1.0
    assert r["flags"] == V.E_PAST_END and r["truncated"] and not r["terminated"] and r["pos_idx"] == 0
    # an episode that started at T-2: the previous valuation is portfolio_initial_value
    r = V.past_end_step((1.0, 0.0, 0.0, 0.0), 0, -1, 120.0, 126.0, positions=POS, fee=0.0, rate=0.0, v0=100.0,
                        started_at_t2=True, reward=SIMPLE)
    assert r["reward"] == (126.0 - 100.0) / 100.0
    # a trade to flat at price[T-2]: the valuation freezes at that price
    r = V.past_end_step((1.0, 0.0, 0.0, 0.0), 0, 1, 120.0, 126.0, positions=POS, fee=0.0, rate=0.0, v0=100.0,
                        started_at_t2=False, reward=SIMPLE)
    assert r["pos_idx"] == 1 and r["valuation"] == 120.0 and r["reward"] == 0.0 and r["state"][0] == 0.0
    # an action past the positions is a hold; a valuation below the stop terminates with reward 0
    r = V.past_end_step((1.0, 0.0, 0.0, 0.0), 0, 9, 120.0, 60.0, positions=POS, fee=0.0, rate=0.0, v0=100.0,
                        started_at_t2=False, reward=SIMPLE)
    assert r["pos_idx"] == 0 and r["terminated"] and r["reward"] == 0.0


@pytest.mark.parametrize("action", [-1, 0, 1, 2, 3])
def test_past_end_step_is_the_oracles_ordinary_last_transition(action):
    """The oracle's own step from row T-2 to T-1 (an episode started at T-3) against past_end_step on the state it
    stepped from: what the contract says a past-end step computes."""
    T, N = 80, 1
    feats, price = _series(T, 5)
    plan = np.array([[[T - 3, 3, 0]] * 2], np.int32)
    kw = dict(num_envs=N, positions=POS, windows=4, trading_fees=1e-3, borrow_interest_rate=2e-5,
              reward_kind=1, plan=plan)
    o = orc.OracleVecEnv(feats, price, **kw)
    o.reset()
    o.step(np.array([0]))
    assert o.idx[0] == T - 2
    st = (o.asset[0], o.fiat[0], o.interest_asset[0], o.interest_fiat[0])
    pidx = int(o.pos_idx[0])
    o.step(np.array([action]))
    assert o.truncated[0] == 1 and o.info_idx[0] == T - 1
    r = V.past_end_step(st, pidx, action, price[T - 2], price[T - 1], positions=POS, fee=1e-3, rate=2e-5, v0=1000.0,
                        started_at_t2=False, reward=SIMPLE)
    assert r["valuation"] == o.valuation[0] and r["reward"] == o.reward[0]
    assert np.float64(r["real_position"]).view(np.uint64) == np.float64(o.real_position[0]).view(np.uint64)
