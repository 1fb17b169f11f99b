"""CPU checks of `history_reference`: the History rows it builds reproduce what every golden recorded from the reference's
own info dict, and its reset / step row semantics (signed zeros, duplicate positions) are the reference's expressions."""
from __future__ import annotations

import numpy as np
import pytest

import helpers as H
import history_reference as HR


@pytest.mark.parametrize("name", H.GOLDEN_NAMES)
def test_rows_reproduce_every_golden(name):
    """The step rows carry the golden's recorded info values bit for bit; the valuation is the reference's
    `valorisation` of the recorded terminal portfolio at price[idx]; the reset rows hold the recorded post-reset
    state and every env's log alternates episodes correctly."""
    g = H.load_golden(name)
    hist = HR.GoldenHistory(g)
    for k in range(hist.K):
        st = hist.step(k)
        for c, gk in (("idx", "idx"), ("step", "step"), ("position", "position"), ("real_position", "real_position"),
                      ("portfolio_valuation", "valuation"), ("reward", "reward")):
            H.assert_bits(st[c].astype(g[gk].dtype), g[gk][k], f"{name} step {k} {c}")
        ds = st["dataset_idx"]
        H.assert_bits(HR.valorisation(g["asset"][k], g["fiat"][k], g["interest_asset"][k], g["interest_fiat"][k],
                                      g["price"][ds, g["idx"][k]]), g["valuation"][k], f"{name} step {k} valorisation")
        assert (st["position_index"] == np.where(g["actions"][k] >= 0, g["actions"][k], -1)).all()
        ended = hist.ended(k)
        rs = hist.reset_after(k)
        assert (rs["idx"][ended] == g["post_idx"][k][ended]).all() and (rs["step"] == 0).all()
        assert (g["post_step"][k][ended] == 0).all()
        # an env that did not end keeps its episode's dataset
        if hist.multi:
            assert (g["post_dataset"][k][~ended] == ds[~ended]).all()
    for env in range(hist.N):
        log = hist.log(env)
        assert len(log["idx"]) == hist.K + int((g["terminated"][:, env] | g["truncated"][:, env]).sum()) + 1
        eps, done = HR.episodes(log)
        assert all(log["step"][a] == 0 and log["portfolio_valuation"][a] == hist.v0 for a, _ in eps)
        assert all((np.diff(log["step"][a:b]) == 1).all() for a, b in eps)


def test_limit_order_rows_are_exactly_the_26_steps_a_limit_order_moved():
    """In `limit_orders_persistent`, 26 step rows record a position that is not the action's target (or, on a hold,
    the previous position): those are the rows a device log must take from the post-step state, not the action."""
    g = H.load_golden("limit_orders_persistent")
    pos = np.asarray(g["positions"], np.float64)
    K, N = g["actions"].shape
    prev = np.concatenate([g["plan"][None, :, 0, 1], g["post_pos_idx"][:-1]]).astype(np.int64)     # pre-step index
    a = g["actions"]
    from_action = np.where(a >= 0, pos[np.maximum(a, 0)], pos[prev])
    moved = from_action != g["position"]
    assert int(moved.sum()) == 26
    # each of them executed a limit order: the recorded position is one of the orders' positions
    order_pos = {float(p) for p, _ in g["params"]["limit_orders"]}
    assert {float(x) for x in g["position"][moved]} <= order_pos


def test_distribution_is_pythons_max_with_zero_first():
    xs = np.array([1.5, 0.0, -0.0, -2.0, np.nan, 5e-324, -5e-324, np.inf, -np.inf])
    want = np.array([float(max(0, float(x))) for x in xs])
    H.assert_bits(HR.pymax0(xs), want, "max(0, x)")
    assert np.signbit(HR.pymax0(np.array([-0.0]))).sum() == 0
    d = HR.distribution(np.array([-0.0, 2.0]), np.array([0.0, -3.0]), np.array([-0.0, 0.1]), np.array([0.0, 0.0]))
    H.assert_bits(d["portfolio_distribution_asset"], np.array([0.0, 2.0]), "asset")
    H.assert_bits(d["portfolio_distribution_borrowed_asset"], np.array([0.0, 0.0]), "borrowed asset")
    H.assert_bits(d["portfolio_distribution_borrowed_fiat"], np.array([0.0, 3.0]), "borrowed fiat")
    assert np.signbit(d["portfolio_distribution_interest_asset"][0])          # interest is copied, not clipped


def test_reset_row_position_index_is_the_first_equal_value():
    """The reference's reset row records ``positions.index(self._position)`` (environments.py:189): with a value listed
    twice (0.0 and -0.0 compare equal) that is the first index, while position keeps the drawn value's sign."""
    positions = [-1, 0.0, 1, -0.0]
    assert positions.index(np.float64(-0.0)) == 1 and positions.index(-0.0) == 1
    row = HR.reset_row(positions, 1000.0, [5, 6, 7, 8], [0, 1, 2, 3], [0.0] * 4, [1000.0] * 4, [0] * 4)
    assert row["position_index"].tolist() == [0, 1, 2, 1]
    assert np.signbit(row["position"][3]) and not np.signbit(row["position"][1])
    H.assert_bits(row["real_position"], row["position"], "real_position = position")
    assert HR.first_index([2.0, 1.0, 2.0, 1.0], [0, 1, 2, 3]).tolist() == [0, 1, 0, 1]


def test_step_row_position_index_is_the_action_or_minus_one():
    assert HR.action_index([-1, 0, 3, 4, -7, 9], 4).tolist() == [-1, 0, 3, -1, -1, -1]


def test_oracle_history_matches_the_golden_rows():
    """`OracleHistory` (the builder for oracle-driven runs) gives the same rows as the golden builder on C3."""
    g = H.load_golden("c3_windows_leveraged")
    o = H.make_oracle(g)
    oh = HR.OracleHistory(o, g["params"]["portfolio_initial_value"])
    gh = HR.GoldenHistory(g)
    o.reset()
    oh.after_reset()
    for c in HR.COLS:
        H.assert_bits(oh.rows[c], gh.initial_reset()[c], f"reset {c}")
    for k in range(gh.K):
        oh.before_step()
        o.step(g["actions"][k])
        st = oh.after_step(g["actions"][k])
        want, want_info = gh.step(k), gh.infos_after(k)
        for c in HR.COLS:
            if c == "reward":
                H.assert_close64(st[c], want[c], f"step {k} {c}")
                continue
            H.assert_bits(st[c], want[c], f"step {k} {c}")
            H.assert_bits(oh.rows[c], want_info[c], f"infos {k} {c}")
    for env in range(gh.N):
        a, b = oh.history(env), gh.log(env)
        for c in ("idx", "step", "position_index", "position", "new_episode", "dataset_idx"):
            H.assert_bits(a[c], b[c], f"env {env} log {c}")
