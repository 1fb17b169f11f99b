"""CPU: the exact constructions of exact_edges.py hold, and the C oracle meets the contracts the device is tested
against with them — the termination threshold, the log reward within 1 ulp of its exact value, np.clip's signed-zero
ties and the signed zeros of a -0.0 position."""
import math

import numpy as np
import pytest

import exact_edges as X
import helpers as H

PAIRS = X.termination_pairs()


def _replay(b):
    """Run the oracle through the scenario; returns the per-step outputs stacked [K, N]."""
    o = X.make_oracle(b)
    o.reset()
    keys = ("reward", "terminated", "truncated", "valuation", "real_position")
    out = {k: [] for k in keys + ("obs",)}
    for k in range(b.actions.shape[0]):
        o.step(b.actions[k])
        for n in keys:
            out[n].append(np.array(getattr(o, n), copy=True))
        out["obs"].append((o.obs[:, -1] if b.windows else o.obs).copy())
    return {n: np.stack(v) for n, v in out.items()}


@pytest.mark.parametrize("v0,ratio", PAIRS)
def test_done_threshold_port_is_the_boundary(v0, ratio):
    """fl(thr / v0) <= ratio < fl(next_up(thr) / v0), or NaN: then only for ratio 0 and the subnormal ratio, where the
    step kernels divide."""
    thr = X.done_threshold(v0, ratio)
    if math.isnan(thr):
        assert ratio == 0.0 or (0.0 < ratio < 2.2250738585072014e-308), (v0, ratio)
        return
    assert thr / v0 <= ratio < X.next_up(thr) / v0
    assert thr == X.true_threshold(v0, ratio)


def test_the_grid_holds_the_off_by_one_ulp_thresholds():
    d = [X.ordinal(X.true_threshold(v0, r)) - X.ordinal(r * v0) for v0, r in PAIRS[1:17]]
    assert d.count(1) >= 8 and d.count(-1) >= 8, d
    assert math.isnan(X.done_threshold(1000.0, 0.0)) and math.isnan(X.done_threshold(1000.0, X.SUBNORMAL_RATIO))


def test_leveraged_ladder_reaches_zero_and_its_neighbours():
    (p_le, v_le), (p_gt, v_gt) = X.leveraged_bracket(0.0, 1000.0)
    assert X.bits(v_le) == 0 and p_le == 1000.0 and v_gt == X.next_up(1000.0) - 1000.0
    (p_le, v_le), (p_gt, v_gt) = X.leveraged_bracket(-250.0, 1000.0)
    assert v_le == -250.0 and v_gt > -250.0 and X.ordinal(v_gt) - X.ordinal(v_le) >= 1


@pytest.mark.parametrize("v0,ratio", PAIRS)
def test_oracle_replays_the_termination_ladders(v0, ratio):
    """The ladders give the intended first-step valuations, and the oracle's flags and rewards are the Python
    expressions', bit for bit."""
    b = X.build(X.grid_scenario(v0, ratio))
    r = _replay(b)
    e = b.expect
    H.assert_bits(r["valuation"], e["valuation"], "valuation")
    H.assert_bits(r["terminated"].astype(bool), e["terminated"], "terminated")
    H.assert_bits(r["truncated"].astype(bool), e["truncated"], "truncated")
    X.check_rewards(b, r["reward"], "oracle")
    # the first step's valuations are the targets: the threshold and its neighbours
    thr = X.true_threshold(v0, ratio)
    first = set(r["valuation"][0].tolist())
    if thr > 0.0:
        assert {thr, X.next_up(thr)} <= first and (X.next_down(thr) <= 0.0 or X.next_down(thr) in first)
    else:
        assert min(first) <= thr < max(first)
    assert r["terminated"][0].any() and not r["terminated"][0].all()


@pytest.mark.parametrize("sc", X.matrix_scenarios(), ids=lambda s: s.name)
@pytest.mark.parametrize("windows,n_ds", [(None, 1), (4, 2)])
def test_oracle_replays_the_matrix_scenarios(sc, windows, n_ds):
    b = X.build(sc, windows, n_ds)
    r = _replay(b)
    e = b.expect
    H.assert_bits(r["valuation"], e["valuation"], "valuation")
    H.assert_bits(r["terminated"].astype(bool), e["terminated"], "terminated")
    H.assert_bits(r["truncated"].astype(bool), e["truncated"], "truncated")
    X.check_rewards(b, r["reward"], "oracle")
    H.assert_bits(r["obs"][..., -2], e["position"], "position column")
    H.assert_bits(r["obs"][..., -1], e["real_position"], "real_position column")


def test_glibc_log_is_within_one_ulp_of_the_exact_log():
    """The reference's own log (the oracle's glibc log, and Python's) on every ladder ratio."""
    b = X.build(X.matrix_scenarios()[0])
    r = _replay(b)
    dist = X.check_rewards(b, r["reward"], "oracle")
    assert len(dist) > 200 and max(dist) <= 1
    for ln in b.sc.lanes:
        for prev, val in zip(ln.prices[:-1], ln.prices[1:]):
            assert X.ulps_apart(math.log(val / prev), X.exact_log(val, prev)) <= 1


def test_ladder_ratios_reach_the_hard_cases():
    ratios = set()
    for ln in X.log_ladder_lanes(1000.0):
        ratios |= {val / prev for prev, val in zip(ln.prices[:-1], ln.prices[1:])}
    for k in range(1, 5):
        assert 1.0 + k * 2.0 ** -52 in ratios and 1.0 - k * 2.0 ** -53 in ratios
    assert 1.0 in ratios and 1.0 + 2.0 ** -20 in ratios and 1.0 - 2.0 ** -20 in ratios
    lanes = X.clip_edge_lanes(1000.0, 100.0, -0.2, 0.5)
    xs = [100.0 * X.exact_log(v, p) for ln in lanes for p, v in zip(ln.prices[:-1], ln.prices[1:])]
    # within one price ulp of each bound (a price ulp moves 100 ln(q) by ~1.1e-14)
    assert min(abs(x + 0.2) for x in xs) < 1.2e-14 and min(abs(x - 0.5) for x in xs) < 1.2e-14
    assert any(x < -0.2 for x in xs) and any(-0.2 < x < 0 for x in xs) and any(x > 0.5 for x in xs)


def test_numpy_clip_keeps_x_on_signed_zero_ties():
    """The device's compare-select clip copies these semantics; if numpy changes them, this test says so."""
    for x, lo, hi in [(-0.0, 0.0, 1.0), (0.0, -1.0, -0.0), (0.0, -0.0, 0.0), (-0.0, -0.0, 0.0)]:
        got = float(np.clip(np.float64(x), lo, hi))
        assert X.bits(got) == X.bits(x) == X.bits(X.clip(x, lo, hi)), (x, lo, hi)


def test_signed_zeros_of_the_oracle():
    """A -0.0 position keeps its sign in the position column and real_position; the rewards of an unchanged
    valuation are +0.0, -0.0 with scale -1 (clip (0, 1) keeps it), and +0.0 under clip (-1, -0.0)."""
    scs = {s.name: s for s in X.matrix_scenarios()}
    b = X.build(scs["default log"])
    r = _replay(b)
    names = [ln.what for ln in b.sc.lanes]
    neg, pos = names.index("flat -0.0"), names.index("flat +0.0")
    assert (r["obs"][:, neg, -2].view(np.uint32) == 0x80000000).all()
    assert (r["obs"][:, pos, -2].view(np.uint32) == 0).all()
    assert (r["real_position"][:, neg].view(np.uint64) == 1 << 63).all()
    assert (r["real_position"][:, pos].view(np.uint64) == 0).all()
    assert (r["reward"][:, [neg, pos]].view(np.uint64) == 0).all()
    for name, sign in [("log x-1 clip (0, 1)", 1 << 63), ("-1 ulp threshold, simple x-1 clip (0, 1)", 1 << 63),
                       ("ratio 0 (divide), simple clip (-1, -0.0)", 0)]:
        b = X.build(scs[name])
        r = _replay(b)
        names = [ln.what for ln in b.sc.lanes]
        for lane in ("flat -0.0", "flat +0.0"):
            assert (r["reward"][:, names.index(lane)].view(np.uint64) == sign).all(), (name, lane)
