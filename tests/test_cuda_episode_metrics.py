"""GPU: the episode-metric catalogue (add_metric with gte.DeviceMetric) on the device.  Every golden's finished episodes
are recorded bit for bit as the DeviceMetric callables evaluate on the reference's History; every step path records
the same bits; metrics change no other output; resets, autoreset=False, datasets rotation and checkpoints keep the
accumulators right; nothing is written outside the two buffers; and the full-size C5 shard holds up."""
import numpy as np
import pytest
import torch

import helpers as H
from episode_reference import episode_histories, record_of

pytestmark = pytest.mark.gpu

KINDS = ["position_changes", "episode_length", "max_drawdown", "episode_reward", "time_in_market"]
FEES = dict(trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000)


def _add_all(env):
    import gym_trading_env_b200 as gte
    for k in KINDS:
        env.add_metric(k, gte.DeviceMetric(k))


def _rec(env):
    return env._episode_record.cpu().numpy()


REWARD_ROW = 2 + KINDS.index("episode_reward")


@pytest.mark.parametrize("name", H.GOLDEN_NAMES)
def test_golden_replay_records_the_reference_metrics(name):
    """Every record row of every finished episode, bit for bit against the DeviceMetric callables on the History the
    reference saw.  The log-return reward itself may differ from the recorded one in its last bit (the device's log
    against numpy's; the golden replay holds rewards to 1e-12 relative), so episode_reward is held bit for bit to the
    left-to-right sum of the device's own per-step rewards, and to 1e-12 relative to the sum of the recorded ones."""
    g = H.load_golden(name)
    env = H.make_device_env(g)
    _add_all(env)
    v0 = g["params"]["portfolio_initial_value"]
    expect = {(i, k): record_of(h) for i, k, h in episode_histories(g, v0)}
    rewards = np.zeros_like(g["reward"])
    env.reset()
    orders = bool(g["params"].get("limit_orders"))
    cursor = np.zeros(g["actions"].shape[1], np.int64)
    if orders:
        H._add_planned_orders(H.DeviceAdapter(env), g, list(range(g["actions"].shape[1])), cursor)
    prev = _rec(env)
    assert np.isnan(prev).all()
    for k in range(g["actions"].shape[0]):
        env.step(torch.as_tensor(g["actions"][k], device=env.device))
        rec = _rec(env)
        rewards[k] = env._reward.cpu().numpy()
        ended = (g["terminated"][k] | g["truncated"][k]).astype(bool)
        for i in range(rec.shape[1]):
            if ended[i]:
                other = np.arange(7) != REWARD_ROW
                H.assert_bits(rec[other, i], expect[(i, k)][other], f"{name} step {k} env {i} record")
                H.assert_close64(rec[REWARD_ROW, i], expect[(i, k)][REWARD_ROW], f"{name} step {k} env {i} reward sum")
            else:
                H.assert_bits(rec[:, i], prev[:, i], f"{name} step {k} env {i} untouched")
        if orders and ended.any():
            H._add_planned_orders(H.DeviceAdapter(env), g, np.flatnonzero(ended).tolist(), cursor)
        prev = rec
    own = {(i, k): record_of(h)[REWARD_ROW] for i, k, h in episode_histories(dict(g, reward=rewards), v0)}
    last = {}
    for (i, k), r in own.items():
        last[i] = max(last.get(i, -1), k)
    for i, k in last.items():
        H.assert_bits(prev[REWARD_ROW, i], own[(i, k)], f"{name} env {i} reward sum of the device's rewards")
    m = env.get_episode_metrics()
    assert list(m) == ["Market Return", "Portfolio Return"] + KINDS
    i = int(np.flatnonzero(~np.isnan(prev[0]))[0])
    one = env.get_episode_metrics(i)
    assert one["Market Return"] == f"{100 * prev[0, i]:5.2f}%" and one["episode_length"] == int(prev[3, i])
    assert isinstance(one["position_changes"], int) and isinstance(one["max_drawdown"], float)


# ---- one random run through every step path ---------------------------------------------------------------------
def _series(T=1500, seed=3):
    import gym_trading_env_b200 as gte
    return gte.frame_to_arrays(gte.make_gbm_ohlcv(T, seed=seed))


def _env(windows, metrics=True, N=1000, **kw):
    import gym_trading_env_b200 as gte
    env = gte.TradingVectorEnv(_series(), positions=[-1, 0, 0.5, 1, 2], windows=windows, max_episode_duration=15,
                               num_envs=N, seed=7, verbose=0, **FEES, **kw)
    if metrics:
        _add_all(env)
    return env


K_RUN = 60


def _actions(N=1000):
    return np.random.default_rng(5).integers(-1, 5, size=(K_RUN, N))


def _drive(env, path):
    acts = _actions(env.num_envs)
    env.reset()
    dev = env.device
    if path.startswith("rollout"):
        env.rollout(torch.as_tensor(acts, device=dev), keep_obs=path.endswith("keep"))
    elif path == "async":
        for k in range(K_RUN):
            env.step_async(acts[k].astype(np.int8))
            env.step_wait()
    else:
        for k in range(K_RUN):
            a = acts[k] if env.output != "torch" else torch.as_tensor(acts[k], device=dev)
            env.step(a)
    torch.cuda.synchronize()
    m = env.get_episode_metrics()                     # stops a resident server kernel first
    return _rec(env), env._episode_acc.cpu().numpy(), m


@pytest.mark.parametrize("windows,paths", [
    (8, [dict(), dict(n_chunks=3), "rollout_keep", "rollout", dict(output="hybrid", host_io="copy"), "async",
         dict(cuda_graph=True)]),
    (None, [dict(), "rollout_keep", "rollout", dict(output="hybrid", host_io="mapped"),
            dict(output="hybrid", host_io="server")]),
])
def test_every_step_path_records_the_same_bits(windows, paths):
    base = _env(windows)
    assert base.launches_per_step == (1 if windows is None else 2)
    rec0, acc0, _ = _drive(base, "step")
    assert (~np.isnan(rec0[0])).sum() > 900                      # most envs finished an episode
    for p in paths[1:]:
        kw = p if isinstance(p, dict) else (dict(output="hybrid") if p == "async" else {})
        env = _env(windows, **kw)
        rec, acc, _ = _drive(env, p if isinstance(p, str) else "step")
        H.assert_bits(rec, rec0, f"record via {p}")
        H.assert_bits(acc, acc0, f"accumulators via {p}")


@pytest.mark.parametrize("windows,N", [(8, 1000), (64, 4096), (None, 1000)])
def test_metrics_change_no_other_output(windows, N):
    """Against the same run without metrics: obs, rewards and flags every step, and the state, bit for bit.  Without
    metrics a small windowed batch takes the fused launch, whose CTAs fold the batch sums (get_metrics) in another
    order; the same run in the two-launch form (n_chunks=1) is the bit-for-bit reference for those."""
    a, a1, b = _env(windows, metrics=False, N=N), _env(windows, metrics=False, N=N, n_chunks=1), _env(windows, N=N)
    if windows is not None:
        assert b.launches_per_step == 2 and a1.launches_per_step == 2     # the fused launch is not taken with metrics
    oa, _ = a.reset()
    a1.reset()
    ob, _ = b.reset()
    assert torch.equal(oa.view(torch.int32), ob.view(torch.int32))
    acts = _actions(N)
    for k in range(K_RUN):
        act = torch.as_tensor(acts[k], device=a.device)
        ra, ra1, rb = a.step(act), a1.step(act), b.step(act)
        for r in (ra, ra1):
            assert torch.equal(r[0].view(torch.int32), rb[0].view(torch.int32)), k
            for x, y in zip(r[1:4], rb[1:4]):
                assert torch.equal(x, y), k
    sa, sa1, sb = a.state_dict(), a1.state_dict(), b.state_dict()
    assert set(sb) - set(sa) == {"episode_acc", "episode_record"}
    for n in sa:
        assert torch.equal(sa1[n], sb[n]), n
        if n != "metrics_total":
            assert torch.equal(sa[n], sb[n]), n
    H.assert_close64(sb["metrics_total"].cpu().numpy(), sa["metrics_total"].cpu().numpy(), "metrics_total, fused form")
    for n, v in a1.get_metrics().items():
        assert torch.equal(v, b.get_metrics()[n]), n


# ---- resets, autoreset=False, datasets, checkpoints: a History rebuilt from the device's own per-step outputs ------
class Recorder:
    """Each env's History (position from the actions: no limit orders here), fed from per-step outputs."""

    def __init__(self, env):
        self.env, self.pos = env, np.asarray(env.positions, np.float64)
        self.price = [s.price for s in env._series]
        self.rows = [None] * env.num_envs
        self.expect = np.full((7, env.num_envs), np.nan)
        self.restart(np.ones(env.num_envs, bool))

    def restart(self, mask):
        e = self.env
        idx, pidx, ds = e.idx.cpu().numpy(), e._pos_idx.cpu().numpy(), e._dataset_idx.cpu().numpy()
        for i in np.flatnonzero(mask):
            self.rows[i] = dict(ds=ds[i], position=[self.pos[pidx[i]]], portfolio_valuation=[1000.0], reward=[0.0],
                                close=[self.price[ds[i]][idx[i]]])

    def step(self, a, autoreset=True):
        e = self.env
        val, rew, idx = e._valuation.cpu().numpy(), e._reward.cpu().numpy(), e._info_idx.cpu().numpy()
        ended = (e._terminated | e._truncated).cpu().numpy().astype(bool)
        for i in range(e.num_envs):
            r = self.rows[i]
            r["position"].append(self.pos[a[i]] if a[i] >= 0 else r["position"][-1])
            r["portfolio_valuation"].append(val[i])
            r["reward"].append(rew[i])
            r["close"].append(self.price[r["ds"]][idx[i]])
            if ended[i]:
                self.expect[:, i] = record_of({c: np.asarray(v, np.float64) for c, v in r.items() if c != "ds"})
        if autoreset:
            self.restart(ended)
        return ended


def _check_against_recorder(env, rec, what):
    H.assert_bits(_rec(env), rec.expect, what)


def test_masked_reset_mid_run_starts_new_accumulators_and_keeps_the_record():
    env = _env(8, N=700, debug_outputs=True)
    env.reset()
    rec = Recorder(env)
    acts = _actions(700)
    for k in range(K_RUN):
        env.step(torch.as_tensor(acts[k], device=env.device))
        rec.step(acts[k])
        if k == 23:
            mask = np.arange(700) % 3 == 0
            env.reset(options={"mask": mask})
            rec.restart(mask)
            _check_against_recorder(env, rec, "record after the masked reset")
    _check_against_recorder(env, rec, "record at the end")


def test_autoreset_false_then_explicit_resets():
    env = _env(8, N=500, debug_outputs=True, autoreset=False)
    env.reset()
    rec = Recorder(env)
    acts = _actions(500)
    for k in range(K_RUN):
        env.step(torch.as_tensor(acts[k], device=env.device))
        ended = rec.step(acts[k], autoreset=False)
        if ended.any():
            env.reset(options={"mask": ended})
            rec.restart(ended)
    _check_against_recorder(env, rec, "autoreset=False")


def test_multi_dataset_rotation():
    import gym_trading_env_b200 as gte
    env = gte.MultiDatasetTradingVectorEnv(datasets=[_series(900, s) for s in (1, 2, 3)], episodes_between_dataset_switch=2,
                                           positions=[-1, 0, 0.5, 1, 2], windows=8, max_episode_duration=15, num_envs=600,
                                           seed=7, verbose=0, debug_outputs=True, **FEES)
    _add_all(env)
    env.reset()
    rec = Recorder(env)
    acts = _actions(600)
    for k in range(K_RUN):
        env.step(torch.as_tensor(acts[k], device=env.device))
        rec.step(acts[k])
    assert len(np.unique(env._dataset_idx.cpu().numpy())) == 3
    _check_against_recorder(env, rec, "multi-dataset")


def test_state_dict_round_trip_mid_episode():
    a, b = _env(16, N=300), _env(16, N=300)
    a.reset(); b.reset()
    acts = torch.as_tensor(_actions(300), device=a.device)
    for k in range(33):
        a.step(acts[k])
    b.load_state_dict(a.state_dict())
    for k in range(33, K_RUN):
        a.step(acts[k]); b.step(acts[k])
    H.assert_bits(_rec(b), _rec(a), "record after the round trip")
    H.assert_bits(b._episode_acc.cpu().numpy(), a._episode_acc.cpu().numpy(), "accumulators after the round trip")


@pytest.mark.parametrize("N", [1, 1000, 4097])
@pytest.mark.parametrize("windows", [None, 8])
def test_no_write_outside_the_metric_buffers(N, windows):
    """Guard bands of 1 KiB of a NaN payload around episode_acc and episode_record (as test_cuda_edge_cases does for the
    other buffers): no kernel writes outside [rows, N]."""
    env = _env(windows, N=N)
    G = 128
    sentinel = np.array([0x7FF00000DEADBEEF], np.uint64).view(np.float64)[0]
    bufs = {}
    for name, rows in (("_episode_acc", 5), ("_episode_record", 7)):
        big = torch.from_numpy(np.full(rows * N + 2 * G, sentinel)).to(env.device)
        inner = big[G:G + rows * N].view(rows, N)
        inner.copy_(getattr(env, name))
        setattr(env, name, inner)
        bufs[name] = big
    env._S.episode_acc, env._O.episode_record = env._episode_acc.data_ptr(), env._episode_record.data_ptr()
    env.reset()
    acts = _actions(N)
    for k in range(40):
        env.step(torch.as_tensor(acts[k], device=env.device))
    env.rollout(torch.as_tensor(acts[:10], device=env.device))
    torch.cuda.synchronize()
    for name, big in bufs.items():
        h = big.cpu().numpy().view(np.uint64)
        s = np.array([sentinel]).view(np.uint64)[0]
        assert (h[:G] == s).all() and (h[-G:] == s).all(), name
    env.check_errors()


def test_full_size_c5_shard_with_all_five_metrics():
    """The C5 shard shape (2^21 envs, W=64, 7 positions, D=720) for 1 500 iterations: a 128-env block against the
    History fed from the CPU oracle, and every env's record satisfies the catalogue's invariants."""
    import gym_trading_env_b200 as gte
    import oracle as orc
    N, W, D, K = 1 << 21, 64, 720, 1500
    pos = [-3, -2, -1, 0, 1, 2, 3]
    s = gte.frame_to_arrays(gte.make_gbm_ohlcv(100_000, seed=0))
    kw = dict(positions=pos, windows=W, max_episode_duration=D, **FEES)
    dev = gte.TradingVectorEnv(s, num_envs=N, seed=3, verbose=0, **kw)
    _add_all(dev)
    lo, n = 1_048_544, 128
    ref = orc.OracleVecEnv(s.features, s.price, num_envs=n, seed=3, env_id_offset=lo, **kw)
    dev.reset()
    ref.reset()
    posv = np.asarray(pos, np.float64)
    rows = [None] * n
    expect = np.full((7, n), np.nan)

    def restart(m):
        for i in np.flatnonzero(m):
            rows[i] = dict(position=[posv[ref.pos_idx[i]]], portfolio_valuation=[1000.0], reward=[0.0],
                           close=[s.price[ref.idx[i]]])
    restart(np.ones(n, bool))
    g = torch.Generator(device=dev.device); g.manual_seed(9)
    for k in range(K):
        act = torch.randint(0, len(pos), (N,), generator=g, device=dev.device)
        dev.step(act)
        a = act[lo:lo + n].cpu().numpy()
        ref.step(a)
        ended = (ref.terminated | ref.truncated).astype(bool)
        for i in range(n):
            r = rows[i]
            r["position"].append(posv[a[i]])
            r["portfolio_valuation"].append(ref.valuation[i])
            r["reward"].append(ref.reward[i])
            r["close"].append(s.price[ref.info_idx[i]])
            if ended[i]:
                expect[:, i] = record_of({c: np.asarray(v, np.float64) for c, v in r.items()})
        restart(ended)
    rec = _rec(dev)
    H.assert_bits(rec[:, lo:lo + n], expect, "C5 block record")
    dev.check_errors()
    done = ~np.isnan(rec[0])
    assert done.all()
    length, changes, dd, tim = rec[3], rec[2], rec[4], rec[6]
    step = dev._step.cpu().numpy()
    assert (length >= 2).all() and (length <= D).all() and (changes <= length - 1).all() and (changes >= 0).all()
    assert (dd >= 0).all() and (dd < 1).all() and (tim >= 0).all() and (tim <= 1).all()
    assert (length == np.round(length)).all() and (changes == np.round(changes)).all()
    assert step.max() < D
