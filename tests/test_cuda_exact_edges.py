"""GPU: the exactness claims of the step kernels at their edges, on every step path and kernel instantiation.

The inputs are the exact constructions of exact_edges.py (valid data only: finite positive prices, in-range plan rows,
actions in [-1, n_positions)).  Checked against the reference's expressions evaluated with Python floats:

* termination: `valuation <= done_thr` is `valuation / v0 <= ratio` bit for bit at the threshold and both its
  neighbours, over a grid of (v0, ratio) pairs that includes thresholds one ulp off ratio * v0 and the divide fallback;
  the divide path (GTE_NO_DONE_THRESHOLD=1, in a subprocess) gives the same bits;
* the log reward is within 1 ulp of the exact log of q = fl(val / prev) (scale and clip exact on top of it); the simple
  return is bit-exact; the reward column and the f32 reward wire are the f32 cast of the device's own fp64 reward;
* signed zeros: rewards of an unchanged valuation, scale -1 and clips at signed-zero ties, a -0.0 position in the
  position column, real_position and the info, and -0.0 == 0.0 for position_changes / position_age.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

import exact_edges as X
import helpers as H

pytestmark = pytest.mark.gpu

WIN = 4
INSTANCES = {            # name -> (dynamic feature kinds, episode metrics, datasets)
    "pair": (["position", "real_position"], [], 1),
    "catalogue": (["reward", "position", "portfolio_return", "real_position"], [], 1),
    "metrics": (["position", "real_position"], ["position_changes", "episode_reward"], 1),
    "catalogue+stateful": (["position", "real_position", "reward", "current_drawdown", "position_age"],
                           ["position_changes"], 1),
    "two datasets": (["position", "real_position"], [], 2),
}
PATHS = {                # name -> (windows, constructor arguments); "plain" / "plain_row" are the bases
    "plain": (WIN, dict(n_chunks=1)),
    "chunks": (WIN, dict(n_chunks=3)),
    "graph": (WIN, dict(cuda_graph=True)),
    "fused": (WIN, dict()),
    "rollout": (WIN, dict()),
    "rollout_keep": (WIN, dict()),
    "hybrid_copy": (WIN, dict(output="hybrid", host_io="copy")),
    "async": (WIN, dict(output="hybrid")),
    "plain_row": (None, dict(n_chunks=1)),
    "hybrid_mapped": (None, dict(output="hybrid", host_io="mapped")),
    "hybrid_server": (None, dict(output="hybrid", host_io="server")),
    "f32_wire": (None, dict(output="hybrid", host_io="copy", reward_wire="f32")),
}
SCENARIOS = X.matrix_scenarios()


def _np(x):
    return x if isinstance(x, np.ndarray) else x.cpu().numpy()


def _make_env(b, inst="pair", **kw):
    import gym_trading_env_b200 as gte
    kinds, metrics, _ = INSTANCES[inst]
    kind, scale, lo, hi = b.sc.reward
    series = [gte.SeriesArrays(f, s, ["feature_0", "feature_1"], {}, None) for s, f in zip(b.series, b.features)]
    args = dict(X.env_kwargs(b), num_envs=b.n_envs, reset_plan=b.plan, done_valuation_ratio=b.sc.ratio,
                reward_function=gte.DeviceReward(kind, scale, (lo, hi)), verbose=0, debug_outputs=True,
                dynamic_feature_functions=[gte.DeviceFeature(k) for k in kinds], **kw)
    env = (gte.MultiDatasetTradingVectorEnv(datasets=series, **args) if len(series) > 1
           else gte.TradingVectorEnv(series[0], **args))
    for m in metrics:
        env.add_metric(m, gte.DeviceMetric(m))
    return env


def _run(b, inst, path):
    """Drive one env through the scenario on one step path.  Every env is closed (and a resident server kernel stopped)
    before the next one is built."""
    windows, kw = PATHS[path]
    env = _make_env(b, inst, **kw)
    try:
        acts = b.actions
        dev = env.device
        res = dict(reward=[], terminated=[], truncated=[], obs=[], valuation=[])
        env.reset()
        if path in ("fused", "plain"):
            acc = bool(INSTANCES[inst][1]) or "position_age" in INSTANCES[inst][0]
            expect = 2 if (path == "plain" or acc) else 1
            assert env.launches_per_step == expect, (path, inst, env.launches_per_step)
        if path.startswith("rollout"):
            out = env.rollout(torch.as_tensor(acts, device=dev), keep_obs=path == "rollout_keep")
            res = {n: _np(out[n]) for n in ("reward", "terminated", "truncated", "valuation")}
            res["obs"] = _np(out["obs"]).copy() if path == "rollout_keep" else None
        else:
            for k in range(acts.shape[0]):
                if path == "async":
                    env.step_async(acts[k].astype(np.int8))
                    o, r, te, tr, _ = env.step_wait()
                elif env.output == "hybrid":
                    o, r, te, tr, _ = env.step(acts[k].astype(np.int8))
                else:
                    o, r, te, tr, _ = env.step(torch.as_tensor(acts[k], device=dev))
                if path == "f32_wire":      # the wire carries the f32 cast of the device's fp64 reward
                    r64 = _np(env.reward_device).copy()
                    assert r.dtype == np.float32
                    H.assert_bits(r, r64.astype(np.float32), f"f32 reward wire, step {k}")
                    r = r64
                res["reward"].append(np.array(_np(r), np.float64, copy=True))
                res["terminated"].append(np.array(_np(te), bool, copy=True))
                res["truncated"].append(np.array(_np(tr), bool, copy=True))
                res["obs"].append(_np(o).copy())
                if env.output == "torch":
                    res["valuation"].append(_np(env._valuation).copy())
            res = {n: (np.stack(v) if v else None) for n, v in res.items()}
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        res["last_obs"] = _np(env._obs).copy()
        res["episode_metrics"] = ({n: _np(v).copy() for n, v in env.get_episode_metrics().items()}
                                  if INSTANCES[inst][1] else None)
        env.check_errors()
        return res
    finally:
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        env.close()


def _expected_columns(b, inst, reward):
    """The dynamic columns of the observation's last row [K, N, n_dyn] (the reward column from the device's reward)."""
    e = b.expect
    ended = e["terminated"] | e["truncated"]
    cols = []
    for kind in INSTANCES[inst][0]:
        if kind == "reward":
            cols.append(np.where(ended, np.float32(0.0), reward.astype(np.float32)))
        else:
            cols.append(e[kind])
    return np.stack(cols, axis=-1)


def _check(b, inst, res, what):
    e = b.expect
    H.assert_bits(res["terminated"], e["terminated"], f"{what}: terminated")
    H.assert_bits(res["truncated"], e["truncated"], f"{what}: truncated")
    X.check_rewards(b, res["reward"], what)
    if res["valuation"] is not None:
        H.assert_bits(res["valuation"], e["valuation"], f"{what}: valuation")
    n_dyn = len(INSTANCES[inst][0])
    want = _expected_columns(b, inst, res["reward"])
    last = lambda o: o[..., -1, :] if b.windows else o     # noqa: E731
    if res["obs"] is not None:
        H.assert_bits(last(res["obs"])[..., -n_dyn:], want, f"{what}: dynamic columns")
    H.assert_bits(last(res["last_obs"])[..., -n_dyn:], want[-1], f"{what}: last observation")
    m = res["episode_metrics"]
    if m is not None and "position_changes" in m:
        ended_once = (e["terminated"] | e["truncated"]).any(axis=0)
        H.assert_bits(m["position_changes"][ended_once], np.zeros(ended_once.sum()), f"{what}: position_changes")


_BASES = {}


def _base(sc_i, inst, windows):
    key = (sc_i, inst, windows)
    if key not in _BASES:
        b = X.build(SCENARIOS[sc_i], windows, INSTANCES[inst][2])
        _BASES[key] = (b, _run(b, inst, "plain" if windows else "plain_row"))
    return _BASES[key]


# ---- 1. termination boundary ------------------------------------------------------------------------------------------
def _grid_run(v0, ratio):
    b = X.build(X.grid_scenario(v0, ratio))
    return b, _run(b, "pair", "plain_row")


@pytest.mark.parametrize("v0,ratio", X.termination_pairs())
def test_termination_boundary(v0, ratio):
    """terminated == (val / v0 <= ratio) at the threshold and its neighbours; reward +0.0 where terminated."""
    b, res = _grid_run(v0, ratio)
    _check(b, "pair", res, f"v0={v0!r} ratio={ratio!r}")
    term = res["terminated"][0]
    assert term.any() and not term.all()
    assert (res["reward"][0][term].view(np.uint64) == 0).all()


_DUMP = """
import sys
sys.path[:0] = {paths!r}
import numpy as np, exact_edges as X, test_cuda_exact_edges as T
out = {{}}
for j, (v0, ratio) in enumerate(X.termination_pairs()):
    b, res = T._grid_run(v0, ratio)
    for n in ("reward", "terminated", "truncated", "valuation", "obs"):
        out[f"grid{{j}}_{{n}}"] = res[n]
for i in range(len(T.SCENARIOS)):
    b, res = T._base(i, "pair", None)
    for n in ("reward", "terminated", "truncated", "valuation", "obs"):
        out[f"sc{{i}}_{{n}}"] = res[n]
np.savez({path!r}, **out)
"""


def test_divide_path_gives_the_same_bits():
    """GTE_NO_DONE_THRESHOLD=1 (read once per process, hence the subprocess): every step divides, as the reference."""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "divide.npz")
        code = _DUMP.format(paths=[here, root, os.path.join(root, "oracle")], path=path)
        env = dict(os.environ, GTE_NO_DONE_THRESHOLD="1")
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
        p = subprocess.run(cmd, env=env, cwd=root, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        z = np.load(path)
        got = {k: z[k] for k in z.files}
    for j, (v0, ratio) in enumerate(X.termination_pairs()):
        b, res = _grid_run(v0, ratio)
        for n in ("reward", "terminated", "truncated", "valuation", "obs"):
            H.assert_bits(got[f"grid{j}_{n}"], res[n], f"divide path, v0={v0!r} ratio={ratio!r}: {n}")
    for i in range(len(SCENARIOS)):
        b, res = _base(i, "pair", None)
        for n in ("reward", "terminated", "truncated", "valuation", "obs"):
            H.assert_bits(got[f"sc{i}_{n}"], res[n], f"divide path, {SCENARIOS[i].name}: {n}")


# ---- 2. log reward within one ulp -------------------------------------------------------------------------------------
def test_log_reward_within_one_ulp():
    b, res = _base(0, "pair", None)
    dist = X.check_rewards(b, res["reward"], "log ladder")
    counts = np.bincount(dist, minlength=2)
    print(f"\nlog_return on the ladders: {counts[0]} rewards 0 ulp, {counts[1]} 1 ulp from the exact log "
          f"(of {len(dist)})")
    assert len(dist) > 200 and max(dist) <= 1
    b, res = _base(1, "pair", None)            # scale 100, next to the clip bounds
    X.check_rewards(b, res["reward"], "log x100 clipped")
    rew = res["reward"][~b.expect["terminated"]]
    assert (rew == -0.2).any() and (rew == 0.5).any() and ((rew > -0.2) & (rew < 0.5)).any()


# ---- 3. signed zeros --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("inst", ["pair", "catalogue+stateful"])
def test_signed_zeros(inst):
    """A -0.0 position: 0x80000000 in the position column against 0 for +0.0, real_position -0.0 (the zero numerator of
    ddiv), the info's portfolio distribution as the reference's max(0, x); -0.0 == 0.0 for the position compare, so
    no position change and an age that keeps counting; rewards +0.0 / -0.0 as the Python expressions give them."""
    sc = SCENARIOS[0]
    b = X.build(sc, None)
    env = _make_env(b, inst)
    try:
        names = [ln.what for ln in b.sc.lanes]
        neg, pos = names.index("flat -0.0"), names.index("flat +0.0")
        peak = names.index("new peaks")
        obs, info = env.reset()
        o = _np(obs)
        kinds = INSTANCES[inst][0]
        c_pos, c_rp = 2 + kinds.index("position"), 2 + kinds.index("real_position")
        assert o[neg, c_pos].view(np.uint32) == 0x80000000 and o[pos, c_pos].view(np.uint32) == 0
        assert o[neg, c_rp].view(np.uint32) == 0x80000000 and o[pos, c_rp].view(np.uint32) == 0
        for k in range(5):
            obs, rew, term, trunc, info = env.step(torch.as_tensor(b.actions[k], device=env.device))
            o, r = _np(obs), _np(rew)
            assert o[neg, c_pos].view(np.uint32) == 0x80000000 and o[pos, c_pos].view(np.uint32) == 0, k
            assert o[neg, c_rp].view(np.uint32) == 0x80000000 and o[pos, c_rp].view(np.uint32) == 0, k
            rp = _np(env._real_position)
            assert rp[neg].view(np.uint64) == 1 << 63 and rp[pos].view(np.uint64) == 0, k
            assert r[neg].view(np.uint64) == 0 and r[pos].view(np.uint64) == 0, k
            i_rp, i_pos = _np(info["real_position"]), _np(info["position"])
            assert i_rp[neg].view(np.uint64) == 1 << 63 and i_rp[pos].view(np.uint64) == 0, k
            assert i_pos[neg].view(np.uint64) == 1 << 63 and i_pos[pos].view(np.uint64) == 0, k
            for part, want in [("asset", 0.0), ("fiat", sc.v0), ("borrowed_asset", 0.0), ("borrowed_fiat", 0.0),
                               ("interest_asset", 0.0), ("interest_fiat", 0.0)]:
                d = _np(info["portfolio_distribution_" + part])
                H.assert_bits(d[[neg, pos]], np.array([float(want)] * 2), f"step {k} distribution {part}")
            if "position_age" in kinds:
                c_age, c_dd = 2 + kinds.index("position_age"), 2 + kinds.index("current_drawdown")
                assert o[neg, c_age] == k + 1 and o[pos, c_age] == k + 1, k
                # val == v0 and (the first four steps of the rising lane) a new peak or its repeat: drawdown +0.0
                assert o[[neg, pos], c_dd].view(np.uint32).tolist() == [0, 0], k
                assert k == 4 or o[peak, c_dd].view(np.uint32) == 0, k
    finally:
        env.close()


def test_signed_zero_rewards_on_the_reward_kinds():
    """Unchanged valuation: +0.0 for both kinds; scale -1 gives -0.0 and clip (0, 1) keeps it; clip (-1, -0.0) keeps
    +0.0 — on the device, bit for bit."""
    cases = [(0, 0), (4, 1 << 63), (2, 1 << 63), (3, 0)]
    for sc_i, sign in cases:
        b, res = _base(sc_i, "pair", None)
        names = [ln.what for ln in b.sc.lanes]
        for lane in ("flat -0.0", "flat +0.0"):
            col = res["reward"][:, names.index(lane)]
            assert (col.view(np.uint64) == sign).all(), (SCENARIOS[sc_i].name, lane, col)


# ---- 4. every step path and instantiation -----------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("inst", list(INSTANCES))
def test_every_path_and_instantiation(inst, path):
    """Each scenario against the expectations, and bit for bit the plain two-launch path's flags, rewards and
    observations."""
    windows = PATHS[path][0]
    for i, sc in enumerate(SCENARIOS):
        b, base = _base(i, inst, windows)
        what = f"{sc.name} / {inst} / {path}"
        res = base if path in ("plain", "plain_row") else _run(b, inst, path)
        _check(b, inst, res, what)
        for n in ("reward", "terminated", "truncated", "last_obs"):
            H.assert_bits(res[n], base[n], f"{what}: {n} against the plain path")
        if res["obs"] is not None:
            H.assert_bits(res["obs"], base["obs"], f"{what}: obs against the plain path")
