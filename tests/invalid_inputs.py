"""CPU reference of the error-bit contract (include/gte_b200.h, GteErrorBit and GteState.error_flag): what the step and
reset kernels must do with an invalid action, an out-of-range or exhausted reset plan and a step past the end of the
data, written from the header's words (no GPU code).

* bit 1  an action >= n_positions is a hold;
* bit 16 with strict_actions, a negative action other than -1 is flagged (and is a hold, as every negative action is);
* bit 4  a reset-plan row outside the data / position list is clamped: start into [W-1, T_ds-2] (0 for windows=None),
         position into [0, P), dataset into [0, n_ds); a single-dataset env ignores the dataset field but still flags it;
* bit 8  a plan whose episodes ran out wraps around to its first row;
* bit 2  a step past the end of the data is an ordinary transition from row T-2 to row T-1 from the env's current
         portfolio, reported as truncated; the stored row stays at T-1.
"""
from __future__ import annotations

import math

import numpy as np

E_ACTION_RANGE, E_PAST_END, E_PLAN_RANGE, E_PLAN_EXHAUSTED, E_NEGATIVE_ACTION = 1, 2, 4, 8, 16


def hold_substituted(actions, P, strict):
    """(the valid action array the kernel acts on, the exact error bits of the step).  Every entry that is not an index
    into the positions becomes -1 (hold); the array keeps its dtype."""
    a = np.asarray(actions)
    wide = a.astype(np.int64)
    too_big = wide >= P
    below = wide < -1
    bits = (E_ACTION_RANGE if too_big.any() else 0) | (E_NEGATIVE_ACTION if (strict and below.any()) else 0)
    valid = np.where(too_big | (wide < 0), -1, wide).astype(a.dtype)
    return valid, bits


def clamped_plan(plan, lengths, W, P, n_ds, multi):
    """(the plan the reset kernels act on, bit 4 per row [N, E]).  W: windows (None = 0 rows before the start)."""
    plan = np.asarray(plan, np.int64)
    lengths = np.asarray(lengths, np.int64)
    start, pos, ds = plan[..., 0], plan[..., 1], plan[..., 2]
    bad = (pos < 0) | (pos >= P) | (ds < 0) | (ds >= n_ds)
    pos_c = np.clip(pos, 0, P - 1)
    ds_c = np.clip(ds, 0, n_ds - 1) if multi else np.zeros_like(ds)
    lo = (W - 1) if W else 0
    hi = lengths[ds_c] - 2
    bad |= (start < lo) | (start > hi)
    start_c = np.minimum(np.maximum(start, lo), hi)
    out = np.stack([start_c, pos_c, ds_c], axis=-1).astype(np.int32)
    return out, np.where(bad, E_PLAN_RANGE, 0).astype(np.int32)


def wrapped_plan(plan, episodes):
    """(the plan tiled to `episodes` rows per env — what an exhausted plan replays —, the ordinal of the first reset that
    wraps around and sets bit 8, or None when `episodes` fit the plan)."""
    plan = np.asarray(plan, np.int32)
    E = plan.shape[1]
    tiled = np.ascontiguousarray(plan[:, np.arange(episodes) % E])
    return tiled, (E if episodes > E else None)


def past_end_step(state, pos_idx, action, price_t2, price_t1, *, positions, fee, rate, v0, started_at_t2, reward,
                  done_ratio=0.7):
    """One step past the end of the data (bit 2) of an env whose portfolio is `state` = (asset, fiat, interest_asset,
    interest_fiat) at position index `pos_idx`: the transition from row T-2 (price_t2) to row T-1 (price_t1).
    `started_at_t2`: the episode started at row T-2, so the step counter is back at the episode's first step and the
    previous valuation is portfolio_initial_value.  reward = (kind, scale, lo, hi) as in exact_edges.Scenario.
    Returns dict(reward, reward_bits, valuation, real_position, pos_idx, state, flags, terminated, truncated):
    reward_bits is the set of reward bit patterns the contract allows (exact for the simple return, a log within 1 ulp
    of the exact one for the log return, exact_edges.log_candidates)."""
    import oracle as orc
    import exact_edges as X
    s = np.asarray(state, np.float64)
    val0 = orc.valorisation(s, price_t2)
    prev = float(v0) if started_at_t2 else val0
    new_pos = pos_idx
    if 0 <= action < len(positions) and positions[action] != positions[pos_idx]:
        s = orc.trade_to_position(s, positions[action], price_t2, fee)
        new_pos = action
    s = orc.update_interest(s, rate)
    val = orc.valorisation(s, price_t1)
    with np.errstate(divide="ignore", invalid="ignore"):
        rp = float(np.float64((s[0] - s[2]) * price_t1) / np.float64(val))
    kind, scale, lo, hi = reward
    done = X.terminated(val, v0, done_ratio)
    if done:
        rew, rbits = 0.0, {X.bits(0.0)}
    elif kind == "simple_return":
        rew = X.clip(scale * X.simple_return(val, prev), lo, hi)
        rbits = {X.bits(rew)}
    else:
        rew = X.clip(scale * math.log(val / prev), lo, hi)
        rbits = X.log_candidates(val, prev, scale, lo, hi)
    return dict(reward=rew, reward_bits=rbits, valuation=val, real_position=rp, pos_idx=new_pos, state=s,
                flags=E_PAST_END, terminated=done, truncated=True)
