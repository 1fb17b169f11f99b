"""GPU: the stateful dynamic features (current_drawdown, position_age) on the device.  Every golden's observations hold the
values the DeviceFeature callables give on the reference's History; every gather variant and work unit, every step path
and the usual state changes (masked resets, autoreset=False, dataset rotation, checkpoints) keep them right; they change
no other output and share the max_drawdown metric's peak without disturbing it; nothing is written outside episode_acc;
and the full-size C5 shard holds up."""
import numpy as np
import pytest
import torch

import helpers as H
from stateful_reference import StatefulColumns, StatefulOracle
from test_cuda_dynamic_features import _series, _plan

pytestmark = pytest.mark.gpu

PAIR_ST = ["position", "real_position", "current_drawdown", "position_age"]
F32_5 = ["real_position", "portfolio_return", "reward", "current_drawdown", "position_age"]
MIXED = ["position_age", "reward", "current_drawdown", "position", "episode_progress"]
FEES = dict(trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000)


def _features(kinds, duration=None):
    import gym_trading_env_b200 as gte
    return [gte.episode_progress_feature(duration) if k == "episode_progress" else gte.DeviceFeature(k) for k in kinds]


def _np(x):
    return x if isinstance(x, np.ndarray) else x.cpu().numpy()


# ---- goldens ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", H.GOLDEN_NAMES)
def test_golden_replay_with_the_stateful_columns(name):
    """The default pair plus both stateful kinds: static columns as recorded, dynamic columns as the reference rebuilds
    them from the golden's recorded positions and valuations, bit for bit — observations and terminal observations."""
    g = H.load_golden(name)
    p = g["params"]
    W, ns = p["windows"], g["features"].shape[2]
    positions = np.asarray(g["positions"], np.float64)
    env = H.make_device_env(g, dynamic_feature_functions=_features(PAIR_ST), final_obs=True)
    assert env._episode_acc.shape == (6, p["n_envs"])
    cols = StatefulColumns(p["n_envs"], W, positions, p["portfolio_initial_value"], p["max_episode_duration"])
    cols.reset(g["plan"][:, 0, 1].astype(np.int64))
    start = g["plan"][:, 0, 0]

    def expect(static, vals):
        d = cols.select(vals, PAIR_ST)
        return np.concatenate([static, d if W is not None else d[:, 0]], axis=-1)

    obs, _ = env.reset()
    H.assert_bits(_np(obs), expect(g["obs0"][..., :ns], cols.window(start, start)), f"{name} reset obs")
    orders = bool(p.get("limit_orders"))
    cursor = np.zeros(p["n_envs"], np.int64)
    if orders:
        H._add_planned_orders(H.DeviceAdapter(env), g, list(range(p["n_envs"])), cursor)
    for k in range(g["actions"].shape[0]):
        obs = env.step(torch.as_tensor(g["actions"][k], device=env.device))[0]
        ended = (g["terminated"][k] | g["truncated"][k]).astype(bool)
        match = g["position"][k][:, None] == positions[None, :]
        assert match.any(axis=1).all()
        cols.step(match.argmax(axis=1), g["real_position"][k], g["valuation"][k], g["reward"][k], g["step"][k],
                  g["idx"][k], ended, g["post_pos_idx"][k].astype(np.int64))
        post = g["post_idx"][k]
        H.assert_bits(_np(obs), expect(g["obs"][k][..., :ns], cols.window(post, post - g["post_step"][k])),
                      f"{name} step {k} obs")
        if ended.any():
            H.assert_bits(_np(env.final_obs)[ended], expect(g["step_obs"][k][..., :ns], cols.final)[ended],
                          f"{name} step {k} terminal obs")
            if orders:
                H._add_planned_orders(H.DeviceAdapter(env), g, np.flatnonzero(ended).tolist(), cursor)
    env.check_errors()


# ---- against the CPU oracle -------------------------------------------------------------------------------------
def _pair(kinds, n_envs, *, windows, duration=40, positions=(-1, 0, 0.5, 1, 2), series=None, seed=5, multi=False,
          plan=None, **dev_kw):
    import gym_trading_env_b200 as gte
    import oracle as orc
    series = series or [_series(1500, 3)]
    kw = dict(positions=list(positions), windows=windows, max_episode_duration=duration, **FEES)
    dkw = dict(kw, num_envs=n_envs, seed=seed, verbose=0, dynamic_feature_functions=_features(kinds, duration),
               reset_plan=plan, **dev_kw)
    if multi:
        dev = gte.MultiDatasetTradingVectorEnv(datasets=series, episodes_between_dataset_switch=2, **dkw)
    else:
        dev = gte.TradingVectorEnv(series[0], **dkw)
    tmax = max(s.length for s in series)
    feats = np.zeros((len(series), tmax, series[0].features.shape[1]), np.float32)
    price = np.ones((len(series), tmax))
    for k, s in enumerate(series):
        feats[k, :s.length], price[k, :s.length] = s.features, s.price
    o = orc.OracleVecEnv(feats, price, np.array([s.length for s in series]), num_envs=n_envs, seed=seed,
                         multi_dataset=multi, episodes_between_dataset_switch=2, threads=8 if n_envs > 20000 else 1,
                         plan=plan, **kw)
    return dev, StatefulOracle(o, kinds, duration)


def _run(kinds, n_envs, K=30, *, check_final=False, **kw):
    dev, ref = _pair(kinds, n_envs, **kw)
    obs, _ = dev.reset()
    H.assert_bits(_np(obs), ref.reset(), "reset obs")
    rng = np.random.default_rng(11)
    P = len(dev.positions)
    for k in range(K):
        a = rng.integers(-1, P, size=n_envs)
        got = dev.step(torch.as_tensor(a, device=dev.device) if dev.output == "torch" else a)
        ref.step(a)
        H.assert_bits(_np(got[0]), ref.obs, f"{kinds} step {k} obs")
        ended = (ref.o.terminated | ref.o.truncated).astype(bool)
        if check_final and ended.any():
            H.assert_bits(_np(dev.final_obs)[ended], ref.final_obs[ended], f"{kinds} step {k} final_obs")
    dev.check_errors()
    if dev.windows is not None:
        assert dev.launches_per_step == 2
    return dev, ref


@pytest.mark.parametrize("kinds", [PAIR_ST, F32_5, MIXED], ids=["pair+stateful", "five-f32", "mixed"])
@pytest.mark.parametrize("windows,variant", [(None, "auto"), (None, "generic"), (8, "generic"), (8, "vec"), (8, "tma"),
                                             (64, "auto"), (64, "generic"), (64, "vec"), (64, "tma")])
def test_every_gather_variant(kinds, windows, variant):
    dev, _ = _run(kinds, 300, K=30 if windows != 64 else 50, windows=windows, obs_variant=variant,
                  duration=40 if windows != 64 else 30)
    if variant == "auto" and windows is not None:
        assert dev.obs_variant in ("tma", "vec")


@pytest.mark.parametrize("kinds", [["current_drawdown"], ["position_age"], F32_5], ids=["dd", "age", "five-f32"])
@pytest.mark.parametrize("n_envs", [40, 1000, 9000, 70_000, 300_000])
def test_work_units_and_claimed_tiles(kinds, n_envs):
    """Batch sizes that select the 8-, 16- and 32-env work units and the claimed-tiles gather."""
    _run(kinds, n_envs, K=12 if n_envs < 100_000 else 6, windows=16, duration=10, series=[_series(3000, 6)])


def test_five_f32_columns_take_the_largest_ring_tile():
    dev, _ = _run(F32_5, 500, K=20, windows=64, duration=30)
    assert dev._dyn_ring.shape[1] == 64 * 640
    assert dev._episode_acc.shape == (6, 500)


def test_final_obs_keeps_the_terminal_observation():
    _run(F32_5, 200, K=45, windows=8, duration=15, final_obs=True, check_final=True, plan=_plan(200, 8, 15, 1500, 5))


def test_multi_dataset_rotation():
    series = [_series(T, 40 + k) for k, T in enumerate([600, 750, 680])]
    dev, _ = _run(MIXED, 333, K=60, windows=8, duration=20, series=series, multi=True)
    assert len(np.unique(dev._dataset_idx.cpu().numpy())) == 3


@pytest.mark.parametrize("variant", ["generic", "vec", "tma"])
def test_masked_reset_in_the_middle_of_a_run(variant):
    dev, ref = _pair(PAIR_ST, 203, windows=12, duration=50, obs_variant=variant)
    obs, _ = dev.reset()
    H.assert_bits(_np(obs), ref.reset(), "reset obs")
    rng = np.random.default_rng(1)
    for k in range(60):
        if k in (7, 8, 30):
            mask = rng.random(203) < 0.3
            obs, _ = dev.reset(options={"mask": mask})
            H.assert_bits(_np(obs), ref.reset(mask=mask), f"masked reset before step {k}")
        a = rng.integers(-1, 5, size=203)
        dev.step(torch.as_tensor(a, device=dev.device))
        ref.step(a)
        H.assert_bits(_np(dev._obs), ref.obs, f"step {k} obs")


def test_autoreset_false_then_explicit_resets():
    """The stateful columns of every observation against the reference fed from the device's own per-step History rows
    (position index, valuation); an ended env restarts only through an explicit masked reset."""
    N, W = 250, 8
    dev, _ = _pair(F32_5, N, windows=W, duration=15, autoreset=False, debug_outputs=True)
    positions = np.asarray(dev.positions, np.float64)
    cols = StatefulColumns(N, W, positions, 1000.0, 15)
    c = lambda t: t.cpu().numpy()   # noqa: E731
    obs, _ = dev.reset()
    cols.reset(c(dev._pos_idx))
    sel = lambda: cols.select(cols.window(c(dev.idx), c(dev._ep_start)), F32_5[3:])   # noqa: E731
    H.assert_bits(c(obs)[..., -2:], sel(), "reset obs")
    rng = np.random.default_rng(4)
    restarts = 0
    for k in range(50):
        a = rng.integers(-1, 5, size=N)
        obs = dev.step(torch.as_tensor(a, device=dev.device))[0]
        pidx = c(dev._pos_idx)
        cols.step(pidx, c(dev._real_position), c(dev._valuation), c(dev._reward), c(dev._info_step), c(dev._info_idx),
                  np.zeros(N, bool), pidx)
        H.assert_bits(c(obs)[..., -2:], sel(), f"step {k} obs")
        ended = (dev._terminated | dev._truncated).cpu().numpy().astype(bool)
        if ended.any():
            obs, _ = dev.reset(options={"mask": ended})
            cols.reset(c(dev._pos_idx), ended)
            H.assert_bits(c(obs)[..., -2:], sel(), f"explicit reset after step {k}")
            restarts += int(ended.sum())
    assert restarts > N


# ---- every step path gives the same bits ------------------------------------------------------------------------
K_RUN = 60


def _env(windows, kinds=PAIR_ST, N=1000, **kw):
    import gym_trading_env_b200 as gte
    return gte.TradingVectorEnv(_series(1500, 3), positions=[-1, 0, 0.5, 1, 2], windows=windows,
                                max_episode_duration=15, num_envs=N, seed=7, verbose=0,
                                dynamic_feature_functions=_features(kinds), **FEES, **kw)


def _actions(N=1000):
    return np.random.default_rng(5).integers(-1, 5, size=(K_RUN, N))


def _drive(env, path):
    acts = _actions(env.num_envs)
    env.reset()
    dev = env.device
    if path.startswith("rollout"):
        out = env.rollout(torch.as_tensor(acts, device=dev), keep_obs=path.endswith("keep"))
        obs = [o.clone() for o in out["obs"]] if path.endswith("keep") else None
    else:
        obs = []
        for k in range(K_RUN):
            if path == "async":
                env.step_async(acts[k].astype(np.int8))
                o = env.step_wait()[0]
            else:
                a = acts[k] if env.output != "torch" else torch.as_tensor(acts[k], device=dev)
                o = env.step(a)[0]
            obs.append(torch.as_tensor(np.array(o, copy=True)) if isinstance(o, np.ndarray) else o.clone())
    torch.cuda.synchronize()
    env._lib.gte_serve_stop()
    last = env._obs.cpu().numpy() if obs is None else _np(obs[-1]).copy()
    return [_np(o) for o in obs] if obs else None, last, env._episode_acc.cpu().numpy()


@pytest.mark.parametrize("windows,paths", [
    (8, [dict(), dict(n_chunks=3), "rollout_keep", "rollout", dict(output="hybrid", host_io="copy"), "async",
         dict(cuda_graph=True)]),
    (None, [dict(), "rollout_keep", "rollout", dict(output="hybrid", host_io="copy"),
            dict(output="hybrid", host_io="mapped"), dict(output="hybrid", host_io="server")]),
])
def test_every_step_path_gives_the_same_bits(windows, paths):
    base = _env(windows)
    obs0, last0, acc0 = _drive(base, "step")
    for p in paths[1:]:
        kw = p if isinstance(p, dict) else (dict(output="hybrid") if p == "async" else {})
        env = _env(windows, **kw)
        obs, last, acc = _drive(env, p if isinstance(p, str) else "step")
        H.assert_bits(last, last0, f"last obs via {p}")
        H.assert_bits(acc, acc0, f"accumulators via {p}")
        if obs is not None:
            for k in range(K_RUN):
                H.assert_bits(obs[k], obs0[k], f"obs {k} via {p}")


@pytest.mark.parametrize("windows,N", [(8, 1000), (64, 4096), (None, 1000)])
def test_stateful_columns_change_no_other_output(windows, N):
    """Against the same run with the default pair only: reward, flags, valuation, the static and the pair's columns,
    bit for bit (the two-launch form without them, n_chunks=1, as the same-order reference of the batch sums)."""
    a, b = _env(windows, ["position", "real_position"], N=N, n_chunks=1), _env(windows, N=N)
    ns = a._n_static
    oa, _ = a.reset()
    ob, _ = b.reset()
    assert torch.equal(oa.view(torch.int32), ob[..., :ns + 2].contiguous().view(torch.int32))
    acts = _actions(N)
    for k in range(K_RUN):
        act = torch.as_tensor(acts[k], device=a.device)
        ra, rb = a.step(act), b.step(act)
        assert torch.equal(ra[0].view(torch.int32), rb[0][..., :ns + 2].contiguous().view(torch.int32)), k
        for x, y in zip(ra[1:4], rb[1:4]):
            assert torch.equal(x, y), k
        assert torch.equal(a._valuation, b._valuation), k
    for n, v in a.get_metrics().items():
        assert torch.equal(v, b.get_metrics()[n]), n


@pytest.mark.parametrize("windows", [8, None])
def test_shared_peak_leaves_the_max_drawdown_record_unchanged(windows):
    """With add_metric(max_drawdown) as well, the episode record and the metric's accumulator rows are bit-identical to
    the metrics-only run: the shared peak is updated once per step."""
    import gym_trading_env_b200 as gte
    a, b = _env(windows, ["position", "real_position"]), _env(windows, ["position", "real_position", "current_drawdown"])
    for e in (a, b):
        e.add_metric("max_drawdown", gte.max_drawdown_metric())
        e.add_metric("episode_reward", gte.episode_reward_metric())
    assert a._episode_acc.shape == (5, 1000) and b._episode_acc.shape == (5, 1000)
    _drive(a, "step")
    _drive(b, "step")
    H.assert_bits(b._episode_record.cpu().numpy(), a._episode_record.cpu().numpy(), "episode record")
    H.assert_bits(b._episode_acc.cpu().numpy(), a._episode_acc.cpu().numpy(), "accumulators")


@pytest.mark.parametrize("kinds,rows", [(PAIR_ST, 6), (["current_drawdown", "reward"], 5)])
def test_state_dict_round_trip_mid_episode(kinds, rows):
    a, b = _env(16, kinds, N=300), _env(16, kinds, N=300)
    assert a._episode_acc.shape == (rows, 300)
    a.reset(); b.reset()
    acts = torch.as_tensor(_actions(300), device=a.device)
    for k in range(33):
        a.step(acts[k])
    snap = a.state_dict()
    assert snap["episode_acc"].shape == (rows, 300) and "episode_record" not in snap
    b.load_state_dict(snap)
    b._launch_obs()
    assert torch.equal(b._obs.view(torch.int32), a._obs.view(torch.int32))
    for k in range(33, K_RUN):
        oa, ob = a.step(acts[k])[0], b.step(acts[k])[0]
        assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), k
    H.assert_bits(b._episode_acc.cpu().numpy(), a._episode_acc.cpu().numpy(), "accumulators after the round trip")


@pytest.mark.parametrize("N", [1, 1000, 4097])
@pytest.mark.parametrize("windows", [None, 8])
def test_no_write_outside_episode_acc(N, windows):
    """current_drawdown alone: a [5, N] buffer with 1 KiB guard bands of a NaN payload on both sides (row 5, the age row,
    would be the band after it) stays untouched outside [5, N]."""
    env = _env(windows, ["current_drawdown", "position"], N=N)
    assert env._episode_acc.shape == (5, N) and env._episode_record is None
    G = 128
    sentinel = np.array([0x7FF00000DEADBEEF], np.uint64).view(np.float64)[0]
    big = torch.from_numpy(np.full(5 * N + 2 * G, sentinel)).to(env.device)
    env._episode_acc = big[G:G + 5 * N].view(5, N)
    env._S.episode_acc = env._episode_acc.data_ptr()
    env.reset()
    acts = _actions(N)
    for k in range(40):
        env.step(torch.as_tensor(acts[k], device=env.device))
    env.rollout(torch.as_tensor(acts[:10], device=env.device))
    torch.cuda.synchronize()
    h = big.cpu().numpy().view(np.uint64)
    s = np.array([sentinel]).view(np.uint64)[0]
    assert (h[:G] == s).all() and (h[-G:] == s).all()
    assert (h[G + 1 * N:G + 5 * N] == s).all()            # rows 1..4 belong to metrics that are not configured
    env.check_errors()


def test_full_size_c5_shard_with_five_f32_columns():
    """The C5 shard shape (2^21 envs, W=64, 7 positions, D=720) with the five-f32-column configuration for 1 500
    iterations (two full episodes), a 128-env block against the reference along the way."""
    import gym_trading_env_b200 as gte
    import oracle as orc
    N, W, D, K = 1 << 21, 64, 720, 1500
    pos = [-3, -2, -1, 0, 1, 2, 3]
    s = gte.frame_to_arrays(gte.make_gbm_ohlcv(100_000, seed=0))
    kw = dict(positions=pos, windows=W, max_episode_duration=D, **FEES)
    dev = gte.TradingVectorEnv(s, num_envs=N, seed=3, verbose=0, dynamic_feature_functions=_features(F32_5, D), **kw)
    lo, n = 1_048_544, 128
    ref = StatefulOracle(orc.OracleVecEnv(s.features, s.price, num_envs=n, seed=3, env_id_offset=lo, **kw), F32_5, D)
    obs, _ = dev.reset()
    H.assert_bits(obs[lo:lo + n].cpu().numpy(), ref.reset(), "reset obs block")
    g = torch.Generator(device=dev.device); g.manual_seed(9)
    episodes = 0
    for k in range(K):
        act = torch.randint(0, len(pos), (N,), generator=g, device=dev.device)
        obs = dev.step(act)[0]
        ref.step(act[lo:lo + n].cpu().numpy())
        episodes += int(ref.o.terminated.sum() + ref.o.truncated.sum())
        if k % 25 == 0 or k >= K - 3 or (ref.o.terminated | ref.o.truncated).any():
            H.assert_bits(obs[lo:lo + n].cpu().numpy(), ref.obs, f"step {k} obs block")
    dev.check_errors()
    assert episodes >= 2 * n * 0.5
    assert dev.launches_per_step == 2
