"""Shared test plumbing: golden fixtures, env factories, and the step-by-step comparison.

The same `replay_golden` drives the CPU oracle (`-m "not gpu"`) and the CUDA path (`-m gpu`), so
both are held to the outputs of the reference's own code recorded in tests/golden/*.npz — run unmodified except for the one
documented H3 normalisation (oracle/ref_harness.py zeroes each env's private dynamic-feature columns before every
reset(), fixtures with normalize_dyn=True; `raw_stale_dynamic_rows` is the raw reference and pins the oracle's faithful mode).
"""
from __future__ import annotations

import json
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_NAMES = sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))
# fp64 tolerance stated by BASELINE.json north_star (valuation, reward): 1e-12 relative, plus an
# absolute floor because log-returns can be ~1e-16 (SURVEY.md §8c)
RTOL, ATOL = 1e-12, 1e-15


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    g = {k: z[k] for k in z.files}
    g["params"] = json.loads(str(g["params"]))
    return g


def env_kwargs(g):
    p = g["params"]
    return dict(positions=[float(x) for x in g["positions"]], windows=p["windows"],
                trading_fees=p["trading_fees"], borrow_interest_rate=p["borrow_interest_rate"],
                portfolio_initial_value=p["portfolio_initial_value"],
                initial_position=p["initial_position"], max_episode_duration=p["max_episode_duration"])


def make_oracle(g, dyn_mode=None, plan=True, **over):
    import oracle as orc
    p = g["params"]
    if dyn_mode is None:
        dyn_mode = 1 if p.get("normalize_dyn", True) else 0
    kw = env_kwargs(g)
    kw.update(num_envs=p["n_envs"], dynamic_features=p.get("dynamic_features", True),
              plan=g["plan"] if plan else None, multi_dataset=p.get("multi_dataset", False),
              episodes_between_dataset_switch=p.get("episodes_between_dataset_switch", 1), dyn_mode=dyn_mode)
    if "reward" in p:
        r = p["reward"]
        clip = r["reward_clip"]
        kw.update(reward_kind=r["reward_kind"], reward_scale=r["reward_scale"],
                  reward_clip=(-np.inf if clip[0] is None else clip[0], np.inf if clip[1] is None else clip[1]))
    if p.get("limit_orders"):
        kw.update(high=g["high"], low=g["low"])
    kw.update(over)
    return orc.OracleVecEnv(g["features"], g["price"], g["lengths"], **kw)


def series_from_golden(g):
    import gym_trading_env_b200 as gte
    out = []
    for k, T in enumerate(g["lengths"]):
        info = {}
        if "high" in g:
            info = {"high": np.ascontiguousarray(g["high"][k, :T]), "low": np.ascontiguousarray(g["low"][k, :T])}
        out.append(gte.SeriesArrays(np.ascontiguousarray(g["features"][k, :T]),
                                    np.ascontiguousarray(g["price"][k, :T]),
                                    [f"feature_{j}" for j in range(g["features"].shape[2])], info, None))
    return out


def make_device_env(g, plan=True, **over):
    import gym_trading_env_b200 as gte
    p = g["params"]
    kw = env_kwargs(g)
    kw.update(num_envs=p["n_envs"], reset_plan=g["plan"] if plan else None, verbose=0, debug_outputs=True)
    if not p.get("dynamic_features", True):
        kw["dynamic_feature_functions"] = []
    if "reward" in p:
        r = p["reward"]
        kw["reward_function"] = gte.DeviceReward("simple_return" if r["reward_kind"] == 1 else "log_return",
                                                 r["reward_scale"], tuple(r["reward_clip"]))
    kw.update(over)
    series = series_from_golden(g)
    if p.get("multi_dataset", False):
        return gte.MultiDatasetTradingVectorEnv(
            datasets=series, episodes_between_dataset_switch=p.get("episodes_between_dataset_switch", 1), **kw)
    return gte.TradingVectorEnv(series[0], **kw)


class OracleAdapter:
    def __init__(self, env):
        self.e = env

    def reset(self):
        return self.e.reset().copy()

    def step(self, a, want_final_obs=False):
        e = self.e
        e.step(a, want_final_obs=want_final_obs)
        return dict(obs=e.obs, idx=e.info_idx, step=e.info_step, valuation=e.valuation, reward=e.reward,
                    terminated=e.terminated, truncated=e.truncated, real_position=e.real_position,
                    pre_reset=e.final_state.T, post_asset=e.asset, post_fiat=e.fiat,
                    post_interest_asset=e.interest_asset, post_interest_fiat=e.interest_fiat,
                    post_idx=e.idx, post_step=e.step_, post_pos_idx=e.pos_idx, post_dataset=e.dataset_idx,
                    metrics=e.metrics, final_obs=e.final_obs if want_final_obs else None)


class DeviceAdapter:
    def __init__(self, env):
        self.e = env

    def reset(self):
        obs, _ = self.e.reset()
        return obs.cpu().numpy()

    def step(self, a, want_final_obs=False):
        import torch
        e = self.e
        e.step(torch.as_tensor(a, dtype=torch.int64, device=e.device))
        c = lambda t: t.cpu().numpy()   # noqa: E731
        return dict(obs=c(e._obs), idx=c(e._info_idx), step=c(e._info_step), valuation=c(e._valuation),
                    reward=c(e._reward), terminated=c(e._terminated), truncated=c(e._truncated),
                    real_position=c(e._real_position), pre_reset=c(e._pre_reset_portfolio),
                    post_asset=c(e._asset), post_fiat=c(e._fiat), post_interest_asset=c(e._interest_asset),
                    post_interest_fiat=c(e._interest_fiat), post_idx=c(e.idx), post_step=c(e._step),
                    post_pos_idx=c(e._pos_idx), post_dataset=c(e._dataset_idx), metrics=c(e._metrics_step),
                    final_obs=None)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def assert_bits(a, b, what):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.tobytes() != b.astype(a.dtype).tobytes():
        bb = b.astype(a.dtype)
        bad = np.argwhere(a != bb)
        if len(bad) == 0 and a.dtype.kind == "f":         # equal values, different bits: signed zeros or NaN payloads
            bad = np.argwhere((np.signbit(a) != np.signbit(bb)) | (np.isnan(a) != np.isnan(bb)))
        if len(bad) == 0:
            raise AssertionError(f"{what}: the bytes differ")
        raise AssertionError(f"{what}: {len(bad)} elements differ bitwise, first at {bad[:3].tolist()}: "
                             f"{a[tuple(bad[0])]!r} vs {b[tuple(bad[0])]!r}")


def assert_close64(a, b, what):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b)
    tol = RTOL * np.abs(b) + ATOL
    if not (err <= tol).all():
        i = int(np.argmax(err - tol))
        raise AssertionError(f"{what}: |{a.flat[i]!r} - {b.flat[i]!r}| = {err.flat[i]:.3e} > {tol.flat[i]:.3e}")


def _add_planned_orders(adapter, g, env_ids, cursor):
    """Re-add the golden's limit orders for the envs that were just reset (a reset clears them, :168)."""
    orders = g["params"].get("limit_orders") or []
    for j, (lpos, _factor) in enumerate(orders):
        limits = np.array([g["limit_plan"][i, cursor[i], j] for i in env_ids])
        adapter.e.add_limit_order(float(lpos), limits, persistent=True, env_ids=np.asarray(env_ids))
    for i in env_ids:
        cursor[i] += 1


def replay_golden(adapter, g, *, exact_money=True, check_final_obs=False, max_steps=None):
    """Replay the golden action stream and compare every recorded quantity, step by step."""
    obs0 = adapter.reset()
    has_orders = bool(g["params"].get("limit_orders"))
    order_cursor = np.zeros(g["actions"].shape[1], dtype=np.int64)
    if has_orders:
        _add_planned_orders(adapter, g, list(range(g["actions"].shape[1])), order_cursor)
    assert_bits(obs0, g["obs0"], "reset obs")
    K = g["actions"].shape[0] if max_steps is None else min(max_steps, g["actions"].shape[0])
    money = assert_bits if exact_money else assert_close64
    stats = dict(steps=0, reward_bit_mismatch=0, episodes=0)
    for k in range(K):
        r = adapter.step(g["actions"][k], want_final_obs=check_final_obs)
        w = f"step {k}"
        assert_bits(r["obs"], g["obs"][k], f"{w} obs")                          # bit-exact
        assert_bits(r["idx"], g["idx"][k], f"{w} idx")
        assert_bits(r["step"], g["step"][k], f"{w} step")
        assert_bits(r["terminated"], g["terminated"][k], f"{w} terminated")
        assert_bits(r["truncated"], g["truncated"][k], f"{w} truncated")
        assert_close64(r["valuation"], g["valuation"][k], f"{w} valuation")      # 1e-12 rel (north_star)
        assert_close64(r["reward"], g["reward"][k], f"{w} reward")
        money(r["valuation"], g["valuation"][k], f"{w} valuation(bits)")
        money(r["real_position"], g["real_position"][k], f"{w} real_position")
        for j, nm in enumerate(["asset", "fiat", "interest_asset", "interest_fiat"]):
            money(r["pre_reset"][j], g[nm][k], f"{w} {nm} (terminal)")
            money(r["post_" + nm], g["post_" + nm][k], f"{w} post_{nm}")
        assert_bits(r["post_idx"], g["post_idx"][k], f"{w} post idx")
        assert_bits(r["post_step"], g["post_step"][k], f"{w} post step")
        assert_bits(r["post_pos_idx"], g["post_pos_idx"][k], f"{w} post position index")
        assert_bits(r["post_dataset"], g["post_dataset"][k], f"{w} post dataset")
        if check_final_obs and r["final_obs"] is not None:
            assert_bits(r["final_obs"], g["step_obs"][k], f"{w} terminal obs")
        ended = (g["terminated"][k] | g["truncated"][k]).astype(bool)
        m = r["metrics"]
        assert m[0] == ended.sum(), f"{w} episodes metric"
        assert m[1] == g["terminated"][k].sum() and m[2] == (g["truncated"][k].astype(bool) & ended).sum()
        np.testing.assert_allclose(m[3], np.nansum(g["portfolio_return"][k]), rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(m[4], np.nansum(g["market_return"][k]), rtol=1e-10, atol=1e-12)
        assert m[5] == g["step"][k][ended].sum(), f"{w} episode length metric"
        np.testing.assert_allclose(m[6], g["reward"][k].sum(), rtol=1e-9, atol=1e-12)
        if has_orders and ended.any():
            _add_planned_orders(adapter, g, np.flatnonzero(ended).tolist(), order_cursor)
        stats["reward_bit_mismatch"] += int((r["reward"] != g["reward"][k]).sum())
        stats["episodes"] += int(ended.sum())
        stats["steps"] += g["actions"].shape[1]
    return stats
