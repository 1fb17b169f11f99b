"""GPU: `infos`, the tracked History log and `save_for_render` against the reference's History rows.

Expected rows come from `history_reference` (the goldens' recorded info values, or the C oracle's state).  Every
comparison is bit-exact except `reward` (within the suite's fp64 tolerance).  Covered:

* `infos` on every golden after reset() and after every step, every key: ``data_<col>`` and ``date`` through frames
  with OHLC info columns and a DatetimeIndex (ragged lengths and their own dates per dataset);
* the tracked log of every env of every golden: every step row (the position after the limit orders) and every reset
  row; `save_for_render` for a finished, the latest finished and a running episode;
* masked resets (also in consecutive calls), ``autoreset=False`` with an explicit reset of the ended envs, duplicate
  position values (``positions.index`` in the reset row) and past-end steps, against the oracle;
* identical `infos` bits on every step path and kernel instantiation; an oracle block at scale;
* an out-of-range action on a tracked env: a hold, ``position_index`` -1 in the log and in `infos`.
"""
import numpy as np
import pandas as pd
import pytest
import torch

import helpers as H
import history_reference as HR

pytestmark = pytest.mark.gpu

def _np(x):
    return x if isinstance(x, np.ndarray) else x.cpu().numpy()


def _dated_series(g):
    """The golden's datasets as frames with open / high / low / close / a per-dataset "volume" info column and an hourly
    DatetimeIndex starting at a different date for each dataset."""
    import gym_trading_env_b200 as gte
    out = []
    for k, T in enumerate(g["lengths"]):
        close = np.ascontiguousarray(g["price"][k, :T])
        hi = g["high"][k, :T] if "high" in g else close * 1.002
        lo = g["low"][k, :T] if "low" in g else close * 0.998
        info = {"open": close * 1.001, "high": np.ascontiguousarray(hi), "low": np.ascontiguousarray(lo), "close": close,
                "volume": np.arange(T, dtype=np.float64) * 0.5 + 1000.0 * k}
        index = pd.date_range(f"{2000 + k}-01-01", periods=T, freq="h").values
        out.append(gte.SeriesArrays(np.ascontiguousarray(g["features"][k, :T]), close,
                                    [f"feature_{j}" for j in range(g["features"].shape[2])], info, index))
    return out


def _golden_env(g, **over):
    import gym_trading_env_b200 as gte
    p = g["params"]
    kw = H.env_kwargs(g)
    kw.update(num_envs=p["n_envs"], reset_plan=g["plan"], verbose=0, debug_outputs=True, name="golden")
    if not p.get("dynamic_features", True):
        kw["dynamic_feature_functions"] = []
    if "reward" in p:
        r = p["reward"]
        kw["reward_function"] = gte.DeviceReward("simple_return" if r["reward_kind"] == 1 else "log_return",
                                                 r["reward_scale"], tuple(r["reward_clip"]))
    kw.update(over)
    series = _dated_series(g)
    if p.get("multi_dataset", False):
        return gte.MultiDatasetTradingVectorEnv(
            datasets=series, episodes_between_dataset_switch=p.get("episodes_between_dataset_switch", 1), **kw), series
    return gte.TradingVectorEnv(series[0], **kw), series


def _check_infos(infos, want, series, what, reward=True, lookups=True):
    """Every key of `infos` against a History row `want` (dict of [N] arrays)."""
    for c in HR.COLS:
        if c == "reward":
            if reward:
                H.assert_close64(_np(infos[c]), want[c], f"{what} infos {c}")
            continue
        got = _np(infos[c])
        H.assert_bits(got, want[c].astype(got.dtype), f"{what} infos {c}")
    if not lookups:
        return
    ds, idx = want["dataset_idx"], want["idx"]
    for c in series[0].info:
        exp = np.array([series[d].info[c][i] for d, i in zip(ds, idx)])
        H.assert_bits(_np(infos["data_" + c]), exp, f"{what} infos data_{c}")
    if series[0].index is not None:
        exp = np.array([series[d].index[i] for d, i in zip(ds, idx)])
        assert np.array_equal(infos["date"], exp), f"{what} infos date"


def _readd_orders(env, g, env_ids, cursor):
    class _A:
        e = env
    H._add_planned_orders(_A, g, env_ids, cursor)


def _replay(g, env, series, on_step=None):
    """reset() then every golden step, limit orders re-added as the golden did; `on_step(k, infos)` after each step."""
    hist = HR.GoldenHistory(g)
    has_orders = bool(g["params"].get("limit_orders"))
    cursor = np.zeros(hist.N, np.int64)
    _, infos = env.reset()
    if has_orders:
        _readd_orders(env, g, list(range(hist.N)), cursor)
    _check_infos(infos, hist.initial_reset(), series, "reset", reward=False)
    for k in range(hist.K):
        _, _, _, _, infos = env.step(torch.as_tensor(g["actions"][k], device=env.device))
        if on_step is not None:
            on_step(k, infos, hist)
        ended = hist.ended(k)
        if has_orders and ended.any():
            _readd_orders(env, g, np.flatnonzero(ended).tolist(), cursor)
    return hist


def _variants(name):
    g = H.load_golden(name)
    return ["auto"] if g["params"]["windows"] is None else ["auto", "generic"]


@pytest.mark.parametrize("name,variant", [(n, v) for n in H.GOLDEN_NAMES for v in _variants(n)])
def test_infos_are_the_reference_rows_on_every_golden(name, variant):
    g = H.load_golden(name)
    env, series = _golden_env(g, obs_variant=variant)
    try:
        def check(k, infos, hist):
            want = hist.infos_after(k)
            _check_infos(infos, want, series, f"{name} step {k}", reward=False)
            # `reward` is the step's reward in every env (what step() returned), the reset row's 0 is not reported
            H.assert_close64(_np(infos["reward"]), g["reward"][k], f"{name} step {k} infos reward")
        _replay(g, env, series, check)
    finally:
        env.close()


@pytest.mark.parametrize("name", H.GOLDEN_NAMES)
def test_tracked_history_is_the_reference_log_on_every_golden(name):
    g = H.load_golden(name)
    env, series = _golden_env(g)
    try:
        N = g["actions"].shape[1]
        env.track(range(N), max_steps=g["actions"].shape[0] + 2)
        hist = _replay(g, env, series)
        for i in range(N):
            got, want = env.tracked_history(i), hist.log(i)
            assert len(got) == len(want["idx"]), f"{name} env {i}: {len(got)} rows vs {len(want['idx'])}"
            for c in HR.COLS + ["new_episode", "terminated", "truncated"]:
                if c == "reward":
                    H.assert_close64(got[c].to_numpy(), want[c], f"{name} env {i} log {c}")
                else:
                    H.assert_bits(got[c].to_numpy(), want[c], f"{name} env {i} log {c}")
            ds, idx = want["dataset_idx"], want["idx"]
            H.assert_bits(got["data_close"].to_numpy(), np.array([series[d].price[j] for d, j in zip(ds, idx)]),
                          f"{name} env {i} log data_close")
            assert np.array_equal(got["date"].to_numpy(), np.array([series[d].index[j] for d, j in zip(ds, idx)]))
    finally:
        env.close()


@pytest.mark.parametrize("name", ["limit_orders_persistent", "multi_dataset_k3"])
@pytest.mark.parametrize("which", ["finished", "latest"])
def test_save_for_render_writes_the_reference_episode_rows(name, which, tmp_path):
    g = H.load_golden(name)
    env, series = _golden_env(g)
    try:
        N = g["actions"].shape[1]
        env.track(range(N), max_steps=g["actions"].shape[0] + 2)
        hist = _replay(g, env, series)
        for i in range(N):
            log = hist.log(i)
            eps, done = HR.episodes(log)
            if which == "finished":
                e = len(done) // 2
                path = env.save_for_render(dir=str(tmp_path / f"{which}_{i}"), which=i, episode=e)
                a, b = done[e]
            else:
                # the default: the latest finished episode
                path = env.save_for_render(dir=str(tmp_path / f"{which}_{i}"), which=i)
                a, b = done[-1] if done else eps[-1]
            df = pd.read_pickle(path)
            ds = int(log["dataset_idx"][a])
            srs = series[ds]
            assert len(df) == b - a, f"{name} env {i}: {len(df)} rows vs {b - a}"
            exp_dates = srs.index[log["idx"][a:b]]
            assert np.array_equal(df.index.values, np.sort(exp_dates))
            for c in HR.COLS:
                if c == "dataset_idx":
                    continue
                got = df[c].to_numpy()
                if c == "reward":
                    H.assert_close64(got, log[c][a:b], f"{name} env {i} render {c}")
                else:
                    H.assert_bits(got, log[c][a:b].astype(got.dtype), f"{name} env {i} render {c}")
            for c in srs.info:                       # the market frame is this episode's dataset's frame
                H.assert_bits(df[c].to_numpy(), srs.info[c][log["idx"][a:b]], f"{name} env {i} market {c}")
                H.assert_bits(df["data_" + c].to_numpy(), srs.info[c][log["idx"][a:b]], f"{name} env {i} data_{c}")
    finally:
        env.close()


def test_save_for_render_of_a_running_episode_before_any_finished(tmp_path):
    g = H.load_golden("multi_dataset_k3")
    env, series = _golden_env(g)
    try:
        env.track([0], max_steps=64)
        first_end = int(np.flatnonzero(g["terminated"][:, 0] | g["truncated"][:, 0])[0])
        hist = HR.GoldenHistory(g)
        env.reset()
        for k in range(first_end):
            env.step(torch.as_tensor(g["actions"][k], device=env.device))
        log = hist.log(0, steps=first_end)
        df = pd.read_pickle(env.save_for_render(dir=str(tmp_path), which=0))
        assert len(df) == first_end + 1
        for c in ("idx", "step", "position", "portfolio_valuation", "position_index"):
            H.assert_bits(df[c].to_numpy(), log[c].astype(df[c].dtype), f"running render {c}")
        srs = series[int(log["dataset_idx"][0])]
        H.assert_bits(df["close"].to_numpy(), srs.price[log["idx"]], "running render market close")
    finally:
        env.close()


# ---- oracle-driven: masked resets, autoreset=False, duplicate positions, past-end steps ------------------------------

def _gbm(T, seed):
    import gym_trading_env_b200 as gte
    return gte.frame_to_arrays(gte.make_gbm_ohlcv(T, seed=seed))


def _plan(N, E, T, W, duration, n_pos, seed, n_ds=1, lengths=None):
    rng = np.random.default_rng(seed)
    plan = np.zeros((N, E, 3), np.int32)
    plan[:, :, 2] = rng.integers(0, n_ds, size=(N, E)) if n_ds > 1 else 0
    Ts = np.asarray(lengths if lengths is not None else [T])[plan[:, :, 2]]
    plan[:, :, 0] = (W - 1) + (rng.random((N, E)) * (Ts - duration - 2 * W)).astype(np.int32)
    plan[:, :, 1] = rng.integers(0, n_pos, size=(N, E))
    return plan


def _oracle_pair(N, *, positions, windows=4, duration=15, seed=3, E=64, autoreset=True, series=None, **kw):
    import gym_trading_env_b200 as gte
    import oracle as orc
    srs = series or _gbm(1500, seed)
    plan = _plan(N, E, srs.length, windows or 1, duration, len(positions), seed)
    common = dict(positions=positions, windows=windows, trading_fees=1e-4, borrow_interest_rate=3e-6,
                  portfolio_initial_value=1000.0, max_episode_duration=duration)
    dev = gte.TradingVectorEnv(srs, num_envs=N, seed=seed, reset_plan=plan, verbose=0, debug_outputs=True,
                               autoreset=autoreset, **common, **kw)
    o = orc.OracleVecEnv(srs.features, srs.price, num_envs=N, seed=seed, plan=plan, **common)
    return dev, o, HR.OracleHistory(o, 1000.0), [srs]


def _check_log(dev, oh, ids, what):
    for j, i in enumerate(ids):
        got, want = dev.tracked_history(j), oh.history(i)
        assert len(got) == len(want["idx"]), f"{what} env {i}: {len(got)} rows vs {len(want['idx'])}"
        for c in HR.COLS + ["new_episode", "terminated", "truncated"]:
            if c == "reward":
                H.assert_close64(got[c].to_numpy(), want[c], f"{what} env {i} log {c}")
            else:
                H.assert_bits(got[c].to_numpy(), want[c], f"{what} env {i} log {c}")


@pytest.mark.parametrize("positions", [[-1, 0, 0.5, 1, 2], [-1, 0.0, 1, -0.0]], ids=["distinct", "signed_zero_twice"])
def test_masked_resets_touch_only_the_masked_envs(positions):
    """reset(mask) in the middle of a run, twice in consecutive iterations: the reset envs' infos and logs get the
    reset row (``positions.index`` of the drawn value), the others keep their last step row."""
    N, K = 300, 80
    dev, o, oh, series = _oracle_pair(N, positions=positions)
    ids = list(range(0, N, 7))
    try:
        dev.track(ids, max_steps=4 * K)
        _, infos = dev.reset()
        o.reset()
        oh.after_reset()
        _check_infos(infos, oh.rows, series, "reset", reward=False)
        rng = np.random.default_rng(1)
        for k in range(K):
            a = rng.integers(-1, len(positions), size=N)
            oh.before_step()
            o.step(a)
            oh.after_step(a)
            _, _, _, _, infos = dev.step(torch.as_tensor(a, device=dev.device))
            _check_infos(infos, oh.rows, series, f"step {k}", reward=False)
            if k in (20, 21, 50):
                m = rng.random(N) < 0.3
                _, infos = dev.reset(options={"mask": m})
                o.reset(m)
                oh.after_reset(m)
                _check_infos(infos, oh.rows, series, f"masked reset after step {k}", reward=False)
        _check_log(dev, oh, ids, "masked")
    finally:
        dev.close()


def test_autoreset_false_then_reset_of_the_ended_envs():
    """autoreset=False: after a step the ended envs report their terminal step row; reset(mask=ended) then gives them
    the reset row and leaves everything else alone.  With a reset plan the run equals the oracle's auto-reset run."""
    N, K = 257, 90
    dev, o, oh, series = _oracle_pair(N, positions=[-1, 0, 1, 2], autoreset=False)
    ids = [0, 3, 100, 256]
    try:
        dev.track(ids, max_steps=4 * K)
        dev.reset()
        o.reset()
        oh.after_reset()
        rng = np.random.default_rng(2)
        for k in range(K):
            a = rng.integers(0, 4, size=N)
            oh.before_step()
            o.step(a)
            st = oh.after_step(a, autoreset=False)
            _, _, te, tr, infos = dev.step(torch.as_tensor(a, device=dev.device))
            _check_infos(infos, st, series, f"step {k}")
            ended = _np(te) | _np(tr)
            if ended.any():
                _, infos = dev.reset(options={"mask": ended})
                oh.after_reset(ended)
                _check_infos(infos, oh.rows, series, f"reset of the ended envs after step {k}", reward=False)
        _check_log(dev, oh, ids, "autoreset=False")
    finally:
        dev.close()


def test_past_end_steps_stay_on_the_last_row():
    """Episodes planned to start at T-3 (autoreset=False): the steps past the end set error bit 2, infos stay on row T-1
    (idx, data_close, date) and the tracked row is what infos reports."""
    import gym_trading_env_b200 as gte
    srs = _gbm(300, 4)
    T, N = srs.length, 64
    plan = np.zeros((N, 4, 3), np.int32)
    plan[:, :, 0] = T - 3
    plan[:, :, 1] = np.arange(N)[:, None] % 3
    dev = gte.TradingVectorEnv(srs, num_envs=N, positions=[-1, 0, 1], windows=4, trading_fees=1e-4,
                               borrow_interest_rate=3e-6, reset_plan=plan, autoreset=False, debug_outputs=True, verbose=0)
    try:
        dev.track(range(N), max_steps=16)
        dev.reset()
        rng = np.random.default_rng(3)
        for k in range(5):
            a = rng.integers(-1, 3, size=N)
            _, _, _, tr, infos = dev.step(torch.as_tensor(a, device=dev.device))
            flag = int(dev._error_flag.item())
            assert (flag & 2) == (2 if k >= 2 else 0), (k, flag)
            idx = _np(infos["idx"])
            assert (idx == min(T - 1, T - 3 + k + 1)).all()
            H.assert_bits(_np(infos["data_close"]), srs.price[idx], f"past-end step {k} data_close")
            assert np.array_equal(infos["date"], srs.index[idx])
            if k >= 1:
                assert _np(tr).all()
            dev._error_flag.zero_()
            for j in range(N):
                row = dev.tracked_history(j).iloc[-1]
                for c in HR.COLS:
                    v = _np(infos[c])[j]
                    assert np.asarray(row[c]).astype(v.dtype).tobytes() == np.asarray(v).tobytes(), (k, j, c, row[c], v)
    finally:
        dev.close()


# ---- every step path gives the same infos -----------------------------------------------------------------------

INSTANCES = {            # name -> (dynamic feature kinds, episode metrics, datasets)
    "pair": (["position", "real_position"], [], 1),
    "catalogue": (["reward", "position", "portfolio_return", "real_position"], [], 1),
    "metrics": (["position", "real_position"], ["position_changes", "episode_reward"], 1),
    "catalogue+stateful": (["position", "real_position", "reward", "current_drawdown", "position_age"],
                           ["position_changes"], 1),
    "two datasets": (["position", "real_position"], [], 2),
}
PATHS = {                # name -> (windows, constructor arguments); "plain" / "plain_row" are the bases
    "plain": (4, dict(n_chunks=1)),
    "fast": (4, dict()),
    "chunks": (4, dict(n_chunks=3)),
    "graph": (4, dict(cuda_graph=True)),
    "numpy": (4, dict(output="numpy")),
    "hybrid_copy": (4, dict(output="hybrid", host_io="copy")),
    "async": (4, dict(output="hybrid")),
    "rollout": (4, dict()),
    "rollout_stepped": (4, dict(debug_outputs=True)),
    "plain_row": (None, dict(n_chunks=1)),
    "hybrid_mapped": (None, dict(output="hybrid", host_io="mapped")),
    "hybrid_server": (None, dict(output="hybrid", host_io="server")),
}

def _path_env(inst, path, N=160):
    import gym_trading_env_b200 as gte
    kinds, metrics, n_ds = INSTANCES[inst]
    windows, kw = PATHS[path]
    series = [_gbm(700 + 90 * d, 20 + d) for d in range(n_ds)]
    positions = [-1, 0, 0.5, 1, 2]
    plan = _plan(N, 64, None, windows or 1, 12, len(positions), 9, n_ds=n_ds, lengths=[s.length for s in series])
    args = dict(positions=positions, windows=windows, trading_fees=1e-4, borrow_interest_rate=3e-6,
                max_episode_duration=12, num_envs=N, reset_plan=plan, verbose=0, seed=9,
                dynamic_feature_functions=[gte.DeviceFeature(k) for k in kinds], **kw)
    env = (gte.MultiDatasetTradingVectorEnv(datasets=series, **args) if n_ds > 1 else gte.TradingVectorEnv(series[0], **args))
    for m in metrics:
        env.add_metric(m, gte.DeviceMetric(m))
    return env


def _snapshot(env, infos):
    keys = [k for k in infos if k not in ("reward", "episode_metrics")]
    out = {k: np.array(_np(infos[k]), copy=True) for k in keys}
    out["reward"] = np.array(_np(infos["reward"]), np.float64, copy=True)
    if env.log_metrics:
        em, gm = infos["episode_metrics"], env.get_metrics()
        assert set(em) == set(gm) and all(np.array_equal(_np(em[n]), _np(gm[n]), equal_nan=True) for n in em)
    return out


def _path_run(inst, path, K=40):
    env = _path_env(inst, path)
    acts = np.random.default_rng(4).integers(-1, 5, size=(K, env.num_envs))
    snaps = []
    try:
        _, infos = env.reset()
        snaps.append(_snapshot(env, infos))
        if path == "rollout":
            env.rollout(torch.as_tensor(acts, device=env.device))
            snaps.append(_snapshot(env, env.infos))
        elif path == "rollout_stepped":
            env.track([0])                      # a tracked env takes the stepped form of rollout()
            env.rollout(torch.as_tensor(acts, device=env.device))
            snaps.append(_snapshot(env, env.infos))
        else:
            for k in range(K):
                if path == "async":
                    env.step_async(acts[k].astype(np.int8))
                    *_, infos = env.step_wait()
                elif env.output != "torch":
                    *_, infos = env.step(acts[k].astype(np.int8))
                else:
                    *_, infos = env.step(torch.as_tensor(acts[k], device=env.device))
                snaps.append(_snapshot(env, infos))
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        env.check_errors()
        return snaps
    finally:
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        env.close()


_BASE = {}


@pytest.mark.parametrize("inst", list(INSTANCES))
@pytest.mark.parametrize("path", [p for p in PATHS if p not in ("plain", "plain_row")])
def test_every_step_path_gives_the_same_infos(inst, path):
    base = "plain_row" if PATHS[path][0] is None else "plain"
    if (inst, base) not in _BASE:
        _BASE[(inst, base)] = _path_run(inst, base)
    ref, got = _BASE[(inst, base)], _path_run(inst, path)
    if path.startswith("rollout"):
        ref = [ref[0], ref[-1]]
    assert len(ref) == len(got)
    for k, (a, b) in enumerate(zip(ref, got)):
        assert set(a) == set(b)
        for c in a:
            if c == "date":
                assert np.array_equal(a[c], b[c]), f"{inst} {path} snapshot {k} date"
            else:
                H.assert_bits(b[c], a[c], f"{inst} {path} snapshot {k} {c}")


# ---- at scale -----------------------------------------------------------------------------------------------------

def test_infos_at_the_c3_shape_match_the_oracle_every_step():
    """~3000 envs, W = 64, Philox resets, leverage: infos against the oracle after every one of 220 steps (info_kernel
    on a grid of several waves)."""
    import gym_trading_env_b200 as gte
    import oracle as orc
    srs = _gbm(5000, 13)
    pos = [-3, -2, -1, 0, 1, 2, 3]
    kw = dict(positions=pos, windows=64, trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000,
              max_episode_duration=60)
    N = 3000
    dev = gte.TradingVectorEnv(srs, num_envs=N, seed=17, verbose=0, **kw)
    o = orc.OracleVecEnv(srs.features, srs.price, num_envs=N, seed=17, threads=8, **kw)
    oh = HR.OracleHistory(o, 1000.0, log_ids=())
    try:
        _, infos = dev.reset()
        o.reset()
        oh.after_reset()
        _check_infos(infos, oh.rows, [srs], "reset", reward=False)
        rng = np.random.default_rng(6)
        for k in range(220):
            a = rng.integers(-1, len(pos), size=N)
            oh.before_step()
            o.step(a)
            oh.after_step(a)
            _, _, _, _, infos = dev.step(torch.as_tensor(a, device=dev.device))
            _check_infos(infos, oh.rows, [srs], f"step {k}", reward=False, lookups=(k % 20 == 0))
    finally:
        dev.close()


def test_infos_of_a_block_inside_a_65536_env_run():
    import gym_trading_env_b200 as gte
    import oracle as orc
    srs = _gbm(4000, 14)
    pos = [-1, 0, 0.5, 1, 2]
    kw = dict(positions=pos, windows=16, trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000,
              max_episode_duration=40)
    N, lo, n = 65536, 40000, 128
    dev = gte.TradingVectorEnv(srs, num_envs=N, seed=23, verbose=0, **kw)
    o = orc.OracleVecEnv(srs.features, srs.price, num_envs=n, seed=23, env_id_offset=lo, **kw)
    oh = HR.OracleHistory(o, 1000.0, log_ids=())
    try:
        _, infos = dev.reset()
        o.reset()
        oh.after_reset()
        rng = np.random.default_rng(8)
        for k in range(100):
            a = rng.integers(-1, len(pos), size=N)
            oh.before_step()
            o.step(a[lo:lo + n])
            oh.after_step(a[lo:lo + n])
            _, _, _, _, infos = dev.step(torch.as_tensor(a, device=dev.device))
            sub = {c: _np(infos[c])[lo:lo + n] for c in HR.COLS if c != "reward"}
            for c in sub:
                H.assert_bits(sub[c], oh.rows[c].astype(sub[c].dtype), f"block step {k} {c}")
            H.assert_bits(_np(infos["data_close"])[lo:lo + n], srs.price[oh.rows["idx"]], f"block step {k} data_close")
    finally:
        dev.close()


# ---- out-of-range actions on a tracked env ----------------------------------------------------------------------

def test_out_of_range_action_on_a_tracked_env_is_a_recorded_hold():
    """An action >= len(positions) sets error bit 1 and is a hold: the tracked row and infos read position_index -1 and
    the previous position, exactly as an explicit hold does in a twin env."""
    import gym_trading_env_b200 as gte
    srs = _gbm(600, 5)
    N = 8
    mk = lambda: gte.TradingVectorEnv(srs, num_envs=N, positions=[-1, 0, 1], windows=4, seed=2, debug_outputs=True,  # noqa: E731
                                      verbose=0, max_episode_duration=30)
    bad, ok = mk(), mk()
    try:
        for e in (bad, ok):
            e.track(range(N), max_steps=32)
            e.reset()
        a = np.array([[1] * N, [3, 7, -1, 0, 2, 100, 3, 1], [0] * N])
        for k in range(3):
            bi = bad.step(torch.as_tensor(a[k], device=bad.device))[-1]
            oi = ok.step(torch.as_tensor(np.where(a[k] >= 3, -1, a[k]), device=ok.device))[-1]
            assert (int(bad._error_flag.item()) & 1) == (1 if k >= 1 else 0)
            for c in HR.COLS:
                H.assert_bits(_np(bi[c]), _np(oi[c]), f"step {k} infos {c}")
        assert (_np(bad.infos["position_index"]) == np.array([0] * N)).all()
        for j in range(N):
            hb, ho = bad.tracked_history(j), ok.tracked_history(j)
            for c in HR.COLS:
                H.assert_bits(hb[c].to_numpy(), ho[c].to_numpy(), f"env {j} log {c}")
            assert hb["position_index"].iloc[2] == (-1 if a[1, j] >= 3 or a[1, j] < 0 else a[1, j])
    finally:
        bad.close()
        ok.close()
