"""Exact constructions for the edge tests: price ladders that make an env's portfolio valuation a chosen double, and
the reference's expressions evaluated on them with Python floats (no GPU code).

With ``trading_fees=0``, ``borrow_interest_rate=0`` and a held position, an env's valuation is a function of the row's
price alone:

* long ladder: position 1, start price v0 -> asset = (1*v0)/v0 = 1.0, fiat = 0, every later valuation is the price;
* leveraged ladder: position 2, start price 2*v0 -> asset = 1.0, fiat = -v0, valuation = fl(p - v0), which reaches
  +0.0 and the values around it (and any negative target);
* flat lanes: position +0.0 or -0.0 -> asset = +-0.0, fiat = v0, valuation = v0 at every price.

A `Scenario` is one env configuration (v0, done ratio, reward) and a list of `Lane`s, one env each.  Every lane owns a
block of rows in one price series; its reset_plan row starts every episode at the block's start, so after an episode
ends (terminated, or truncated by max_episode_duration) the env replays the same block.  `simulate` evaluates the
reference's step (environments.py:233-267, portfolio.py) for such an env with Python floats in the reference's own
operation order, which is what the device and the C oracle have to reproduce.
"""
from __future__ import annotations

import math
import struct
from dataclasses import dataclass, field
from decimal import Decimal, localcontext

import numpy as np

INF = float("inf")


# ---- doubles --------------------------------------------------------------------------------------------------------
def next_up(x):
    return math.nextafter(x, INF)


def next_down(x):
    return math.nextafter(x, -INF)


def bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def ordinal(x):
    """Doubles in IEEE order as integers (-0.0 and +0.0 both map to 0): ordinal(next_up(x)) == ordinal(x) + 1."""
    b = bits(x)
    return b if b >= 0 else -(b & 0x7FFFFFFFFFFFFFFF)


def from_ordinal(n):
    b = n if n >= 0 else (-n) | (1 << 63)
    return struct.unpack("<d", struct.pack("<q", b if b < (1 << 63) else b - (1 << 64)))[0]


def ulps_apart(a, b):
    return abs(ordinal(a) - ordinal(b))


# ---- the reference's expressions --------------------------------------------------------------------------------------
def terminated(val, v0, ratio):
    """environments.py:246."""
    return val / v0 <= ratio


def true_threshold(v0, ratio):
    """The largest double x with fl(x / v0) <= ratio, by bisection over the doubles (IEEE division is monotonic in x)."""
    lo, hi = ordinal(-1.7976931348623157e308), ordinal(1.7976931348623157e308)
    if not terminated(from_ordinal(lo), v0, ratio):
        return math.nan
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if terminated(from_ordinal(mid), v0, ratio):
            lo = mid
        else:
            hi = mid
    return from_ordinal(hi) if terminated(from_ordinal(hi), v0, ratio) else from_ordinal(lo)


def done_threshold(v0, ratio):
    """Python port of done_threshold() in csrc/gte_step.cu: the threshold the step kernels compare the valuation with,
    or NaN when its search does not settle (the kernels then divide)."""
    if not (v0 > 0.0) or not math.isfinite(v0) or not math.isfinite(ratio):
        return math.nan
    x = ratio * v0
    k = 0
    while k < 64 and x / v0 <= ratio:
        x = next_up(x)
        k += 1
    for _ in range(128):
        if x / v0 <= ratio:
            return x if next_up(x) / v0 > ratio else math.nan
        x = next_down(x)
    return math.nan


def simple_return(v1, v0):
    return (v1 - v0) / v0


def clip(x, lo, hi):
    """np.clip as the kernels compute it: a compare-select that keeps x on ties (signed zeros included)."""
    x = lo if x < lo else x
    return hi if x > hi else x


def exact_log(val, prev):
    """ln(q) for q = fl(val / prev), computed at 60 digits and rounded once to a double."""
    q = val / prev
    with localcontext() as c:
        c.prec = 60
        return float(Decimal(q).ln())


def log_candidates(val, prev, scale, lo, hi):
    """Every reward a log within 1 ulp of the exact value leads to: clip(fl(scale * y)) for y = L - 1 ulp, L, L + 1 ulp,
    with L = exact_log(val, prev), as a set of bit patterns.  With scale 1 and no clip, that is exactly "within 1 ulp of the exact log"."""
    L = exact_log(val, prev)
    return {bits(clip(scale * y, lo, hi)) for y in (next_down(L), L, next_up(L))}


# ---- the leveraged ladder ---------------------------------------------------------------------------------------------
def leveraged_val(p, v0):
    return p - v0


def leveraged_bracket(t, v0, reach=8):
    """Prices p with fl(p - v0) the largest reachable valuation <= t and the smallest one > t, found among the
    neighbours of fl(t + v0).  Returns ((p_le, v_le), (p_gt, v_gt))."""
    c = ordinal(t + v0)
    cands = [from_ordinal(c + d) for d in range(-reach, reach + 1)]
    cands = [p for p in cands if p > 0.0 and math.isfinite(p)]
    le = [(p, leveraged_val(p, v0)) for p in cands if leveraged_val(p, v0) <= t]
    gt = [(p, leveraged_val(p, v0)) for p in cands if leveraged_val(p, v0) > t]
    assert le and gt, f"no reachable valuation around {t!r} for v0={v0!r}"
    best_le = max(le, key=lambda pv: ordinal(pv[1]))
    best_gt = min(gt, key=lambda pv: ordinal(pv[1]))
    # nothing between them: every price in between maps to one of the two (fl(p - v0) is monotonic in p)
    assert best_le[1] <= t < best_gt[1]
    return best_le, best_gt


# ---- scenarios ----------------------------------------------------------------------------------------------------------
@dataclass
class Lane:
    """One env: its position index, the block of rows it replays (start price first), the action it holds with."""
    pos_idx: int
    prices: list            # rows start .. start + L (the start row, then one row per step)
    action: int = -1        # -1 (hold) or an index whose position equals the held one by value
    dataset: int = 0
    what: str = ""


@dataclass
class Scenario:
    name: str
    v0: float
    ratio: float
    reward: tuple            # (kind, scale, lo, hi), kind "log_return" | "simple_return"
    lanes: list = field(default_factory=list)


POSITIONS = [1.0, 2.0, 0.0, -0.0]          # long, leveraged, flat, flat with a negative sign
LONG, LEVERED, FLAT, NEG_FLAT = 0, 1, 2, 3
STEPS = 10                                 # rows per episode after the start row (max_episode_duration = STEPS + 1)


def long_lane(v0, vals, what="", action=-1):
    return Lane(LONG, [v0] + list(vals), action, what=what)


def levered_lane(v0, prices, what="", action=-1):
    return Lane(LEVERED, [2.0 * v0] + list(prices), action, what=what)


def flat_lane(v0, negative, prices, what=""):
    # holds by naming the other zero: a value compare (:213-215) that never trades
    return Lane(NEG_FLAT if negative else FLAT, [v0] + list(prices), FLAT if negative else NEG_FLAT, what=what)


def pad(lane, steps=STEPS):
    """Fill the block to `steps` rows after the start with the start price (long: valuation v0; levered: v0)."""
    assert len(lane.prices) <= steps + 1
    lane.prices = lane.prices + [lane.prices[0]] * (steps + 1 - len(lane.prices))
    return lane


def boundary_lanes(v0, ratio):
    """Envs whose first-step valuation sits on the termination boundary: the threshold and both its neighbours
    (long ladder for positive valuations), or the leveraged ladder's values around the threshold."""
    thr = true_threshold(v0, ratio)
    lanes = []
    for t in (next_down(thr), thr, next_up(thr)):
        if t > 0.0:
            lanes.append(long_lane(v0, [t], what=f"val={t!r}"))
    if thr <= 0.0 or ratio <= 0.0:
        (p_le, v_le), (p_gt, v_gt) = leveraged_bracket(thr, v0)
        p_below = next_down(p_le)
        for p in (p_below, p_le, p_gt):
            lanes.append(levered_lane(v0, [p], what=f"val={leveraged_val(p, v0)!r}"))
    return [pad(x) for x in lanes]


def search_ulp_pairs(n, sign, seed=2024):
    """Seeded (v0, ratio) pairs with true_threshold = ratio*v0 + sign ulp and ratio in (0.05, 0.95)."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        v0 = float(rng.choice([1.0, 3.0, 10.0, 1000.0, 12345.0])) * float(rng.uniform(0.5, 2.0))
        ratio = float(rng.uniform(0.05, 0.95))
        t = true_threshold(v0, ratio)
        if ordinal(t) - ordinal(ratio * v0) == sign:
            out.append((v0, ratio))
    return out


SUBNORMAL_RATIO = 2.0 ** -1070


def termination_pairs():
    """The (v0, ratio) grid of the termination tests."""
    pairs = [(1000.0, 0.7)]
    pairs += search_ulp_pairs(8, +1, seed=1)
    pairs += search_ulp_pairs(8, -1, seed=2)
    pairs += [(1000.0, r) for r in (0.5, 1.0, 1.5, 0.9999999999999999)]
    pairs += [(1000.0, -0.25), (1000.0, 0.0), (1000.0, SUBNORMAL_RATIO)]
    pairs += [(v0, 0.7) for v0 in (1.0, 3.0, 0.1, 1e6)]
    return pairs


def log_ladder_lanes(v0, steps=STEPS, seed=7):
    """Long ladders whose step ratios put the log reward where a sloppy log loses accuracy: 1 +- k ulp (k = 1..4),
    1 +- 2^-20, +-0.1 % and +-30 % moves, and seeded small moves; every price far above the termination threshold
    of a ratio below 1.4 (the ladder runs at 2..4 v0)."""
    base = 2.0 ** math.ceil(math.log2(v0)) * 2.0       # a power of two: base * (1 + k 2^-52) is exact
    seq = []
    for k in range(1, 5):
        up, dn = base, base
        for _ in range(k):
            up, dn = next_up(up), next_down(dn)
        seq += [up, base, dn, base]
    seq += [base * (1 + 2.0 ** -20), base, base * (1 - 2.0 ** -20), base]
    seq += [base * 1.001, base, base * 0.999, base, base * 1.3, base, base * 0.7, base]
    seq += [base, base]                                   # unchanged price: reward +0.0
    rng = np.random.default_rng(seed)
    p = base
    for r in rng.normal(0.0, 1e-4, size=160):
        p = p * math.exp(float(r))
        seq.append(p)
    for r in rng.integers(-6, 7, size=40):             # a few ulps around the previous price
        seq.append(from_ordinal(ordinal(seq[-1]) + int(r)))
    lanes = []
    for j in range(0, len(seq), steps):
        chunk = seq[j:j + steps]
        lanes.append(pad(long_lane(v0, chunk, what=f"log ladder {j // steps}")))
    return lanes


def clip_edge_lanes(v0, scale, lo, hi, steps=STEPS):
    """Long ladders whose log reward lands next to the clip bounds: scale * ln(q) within a few ulps of lo and hi."""
    base = 2.0 ** math.ceil(math.log2(v0)) * 2.0
    seq = []
    for bound in (lo, hi):
        p1 = base * math.exp(bound / scale)
        for d in range(-3, 4):
            seq += [from_ordinal(ordinal(p1) + d), base]
    return [pad(long_lane(v0, seq[j:j + steps], what=f"clip edge {j // steps}")) for j in range(0, len(seq), steps)]


def zero_lanes(v0, steps=STEPS):
    """Signed zeros: the flat lanes (position +0.0 and -0.0), and a long lane that makes new peaks and returns to v0."""
    rising = [v0 * 1.5, v0 * 2.0, v0 * 2.0, v0 * 2.5]
    return [pad(flat_lane(v0, False, [v0 * 1.1, v0 * 0.9], "flat +0.0")),
            pad(flat_lane(v0, True, [v0 * 1.1, v0 * 0.9], "flat -0.0")),
            pad(long_lane(v0, rising + [v0], what="new peaks"))]


# ---- the price series and the reset plan --------------------------------------------------------------------------
def layout(lanes, windows, n_datasets=1, lead=3):
    """Price series per dataset and the reset plan: lane i lives in dataset i % n_datasets; every block is preceded
    by max(windows - 1, lead) ordinary rows (the window before an episode start).  Dataset k gets k extra tail rows,
    so multi-dataset series have different lengths."""
    W0 = max((windows or 1) - 1, lead)
    series = [[] for _ in range(n_datasets)]
    starts = []
    for i, ln in enumerate(lanes):
        ln.dataset = i % n_datasets
        s = series[ln.dataset]
        s += [100.0 + 0.25 * k for k in range(W0)]
        starts.append(len(s))
        s += ln.prices
    for k, s in enumerate(series):
        s += [100.0] * (2 + k)
    return [np.asarray(s, np.float64) for s in series], starts


def plan_of(lanes, starts, episodes):
    plan = np.zeros((len(lanes), episodes, 3), np.int32)
    for i, ln in enumerate(lanes):
        plan[i, :, 0], plan[i, :, 1], plan[i, :, 2] = starts[i], ln.pos_idx, ln.dataset
    return plan


# ---- the reference's step, with Python floats -----------------------------------------------------------------------
def simulate(sc, lanes, starts, series_len, n_steps, steps=STEPS):
    """Per step k and env i: terminated, truncated, valuation, the reward (exact for simple_return; for log_return the
    set of rewards a log within 1 ulp leads to, see log_candidates) and the dynamic columns of the row the observation
    ends with (after an auto-reset: the new episode's first row).  The reward column is not among them: it is the f32
    cast of whatever reward the env computed."""
    kind, scale, lo, hi = sc.reward
    N = len(lanes)
    out = dict(terminated=np.zeros((n_steps, N), bool), truncated=np.zeros((n_steps, N), bool),
               valuation=np.zeros((n_steps, N)), reward=np.zeros((n_steps, N)), reward_set=[[None] * N for _ in range(n_steps)],
               position=np.zeros((n_steps, N), np.float32), real_position=np.zeros((n_steps, N), np.float32),
               portfolio_return=np.zeros((n_steps, N), np.float32), current_drawdown=np.zeros((n_steps, N), np.float32),
               position_age=np.zeros((n_steps, N), np.float32), real_position64=np.zeros((n_steps, N)))
    for i, ln in enumerate(lanes):
        pos = POSITIONS[ln.pos_idx]
        T = series_len[ln.dataset]
        step = 0
        for k in range(n_steps):
            if step == 0:                                  # reset (:179-183): TargetPortfolio
                p_s = ln.prices[0]
                asset, fiat = (pos * sc.v0) / p_s, (1.0 - pos) * sc.v0
                ia = ifi = 0.0
                prev, peak, age = sc.v0, sc.v0, 0.0
            step += 1
            idx = starts[i] + step
            p = ln.prices[step]
            na, nf = -asset, -fiat                        # update_interest with rate 0
            ia, ifi = (na if na > 0.0 else 0.0) * 0.0, (nf if nf > 0.0 else 0.0) * 0.0
            val = asset * p
            val = val + fiat
            val = val + (-ia) * p
            val = val + (-ifi)
            done = terminated(val, sc.v0, sc.ratio)
            trunc = idx >= T - 1 or step >= steps
            with np.errstate(divide="ignore", invalid="ignore"):
                rp = float(np.float64((asset - ia) * p) / np.float64(val))
            rew = 0.0
            rset = {bits(0.0)}
            if not done:
                if kind == "simple_return":
                    rew = clip(scale * simple_return(val, prev), lo, hi)
                    rset = {bits(rew)}
                else:
                    rset = log_candidates(val, prev, scale, lo, hi)
                    rew = clip(scale * exact_log(val, prev), lo, hi)
            peak = val if val > peak else peak
            age += 1.0
            out["terminated"][k, i], out["truncated"][k, i] = done, trunc
            out["valuation"][k, i], out["reward"][k, i], out["reward_set"][k][i] = val, rew, rset
            out["real_position64"][k, i] = rp
            if done or trunc:                              # the observation shows the new episode's first row
                out["position"][k, i] = out["real_position"][k, i] = np.float32(pos)
                step = 0
            else:
                out["position"][k, i], out["real_position"][k, i] = np.float32(pos), np.float32(rp)
                out["portfolio_return"][k, i] = np.float32(val / sc.v0 - 1.0)
                out["current_drawdown"][k, i] = np.float32(1.0 - val / peak)
                out["position_age"][k, i] = np.float32(age)
            prev = val
    return out


# ---- the scenarios the tests run --------------------------------------------------------------------------------------
N_STEPS = STEPS + 2          # every lane ends one episode (truncated at the latest) and replays its block once more
NO_CLIP = (-INF, INF)


def grid_scenario(v0, ratio):
    """One (v0, ratio) pair of the termination grid: the boundary lanes, with the simple return (an exact reward)."""
    return Scenario(f"v0={v0!r} ratio={ratio!r}", v0, ratio, ("simple_return", 1.0) + NO_CLIP, boundary_lanes(v0, ratio))


def matrix_scenarios():
    """The scenarios every step path and instantiation runs: termination (a plain, a +1 ulp, a -1 ulp threshold and
    the divide fallback), the log ladders at scale 1 and at scale 100 next to the clip bounds, and the signed zeros."""
    up, dn = search_ulp_pairs(1, +1, seed=1)[0], search_ulp_pairs(1, -1, seed=2)[0]
    return [
        Scenario("default log", 1000.0, 0.7, ("log_return", 1.0) + NO_CLIP,
                 boundary_lanes(1000.0, 0.7) + log_ladder_lanes(1000.0) + zero_lanes(1000.0)),
        Scenario("+1 ulp threshold, log x100 clipped", up[0], up[1], ("log_return", 100.0, -0.2, 0.5),
                 boundary_lanes(*up) + log_ladder_lanes(up[0])[:6] + clip_edge_lanes(up[0], 100.0, -0.2, 0.5)),
        Scenario("-1 ulp threshold, simple x-1 clip (0, 1)", dn[0], dn[1], ("simple_return", -1.0, 0.0, 1.0),
                 boundary_lanes(*dn) + zero_lanes(dn[0]) + log_ladder_lanes(dn[0])[:3]),
        Scenario("ratio 0 (divide), simple clip (-1, -0.0)", 1000.0, 0.0, ("simple_return", 1.0, -1.0, -0.0),
                 boundary_lanes(1000.0, 0.0) + zero_lanes(1000.0)),
        Scenario("log x-1 clip (0, 1)", 1000.0, 0.7, ("log_return", -1.0, 0.0, 1.0),
                 zero_lanes(1000.0) + log_ladder_lanes(1000.0)[:3]),
    ]


@dataclass
class Built:
    sc: Scenario
    windows: object
    series: list             # f64 price per dataset
    features: list           # f32 [T, 2] static features per dataset
    plan: np.ndarray
    starts: list
    actions: np.ndarray      # int64 [N_STEPS, N]
    expect: dict

    @property
    def n_envs(self):
        return len(self.sc.lanes)


def build(sc, windows=None, n_datasets=1, n_steps=N_STEPS):
    lanes = [Lane(ln.pos_idx, list(ln.prices), ln.action, what=ln.what) for ln in sc.lanes]
    series, starts = layout(lanes, windows, n_datasets)
    sc = Scenario(sc.name, sc.v0, sc.ratio, sc.reward, lanes)
    feats = [np.stack([np.arange(len(s)) / 64.0, s], axis=1).astype(np.float32) for s in series]
    plan = plan_of(lanes, starts, n_steps + 2)
    actions = np.tile(np.array([ln.action for ln in lanes], np.int64), (n_steps, 1))
    expect = simulate(sc, lanes, starts, [len(s) for s in series], n_steps)
    return Built(sc, windows, series, feats, plan, starts, actions, expect)


def env_kwargs(b):
    """Constructor arguments shared by the device env and the oracle."""
    return dict(positions=list(POSITIONS), windows=b.windows, trading_fees=0, borrow_interest_rate=0,
                portfolio_initial_value=b.sc.v0, max_episode_duration=STEPS + 1)


def stacked(b):
    """[n_datasets, T_max] prices / [n_datasets, T_max, 2] features and the lengths, for the oracle."""
    T = max(len(s) for s in b.series)
    price = np.ones((len(b.series), T))
    feats = np.zeros((len(b.series), T, 2), np.float32)
    for k, (s, f) in enumerate(zip(b.series, b.features)):
        price[k, :len(s)], feats[k, :len(s)] = s, f
    return feats, price, np.array([len(s) for s in b.series], np.int32)


def make_oracle(b):
    import oracle as orc
    feats, price, lengths = stacked(b)
    kind, scale, lo, hi = b.sc.reward
    return orc.OracleVecEnv(feats, price, lengths, num_envs=b.n_envs, done_ratio=b.sc.ratio, plan=b.plan,
                            multi_dataset=len(b.series) > 1, reward_kind=0 if kind == "log_return" else 1,
                            reward_scale=scale, reward_clip=(lo, hi), **env_kwargs(b))


def check_rewards(b, reward, what, k=None):
    """Device / oracle rewards [K, N] against the expectation: bit for bit for the simple return, one of the rewards a
    log within 1 ulp leads to for the log return.  Returns the ulp distances of the unclipped scale-1 log rewards."""
    kind, scale, lo, hi = b.sc.reward
    dist = []
    for k in range(reward.shape[0]):
        for i in range(reward.shape[1]):
            got = float(reward[k, i])
            ok = b.expect["reward_set"][k][i]
            assert bits(got) in ok, (f"{what}: step {k} env {i} ({b.sc.lanes[i].what}): reward {got!r} not in "
                                     f"{sorted(struct.unpack('<d', struct.pack('<q', x))[0] for x in ok)}")
            if kind == "log_return" and scale == 1.0 and not b.expect["terminated"][k, i]:
                dist.append(ulps_apart(got, b.expect["reward"][k, i]))
    return dist
