"""GPU: the error-bit contract (include/gte_b200.h GteErrorBit) on every step path and kernel instantiation, against the
CPU reference of invalid_inputs.py.

* invalid actions: a run with out-of-range / negative actions of every host width is bit for bit the run with those
  entries replaced by -1 (obs, rewards, flags, valuations, state, dynamic-feature ring, episode accumulators and record,
  batch metrics); the error bits are exactly the expected ones — in the torch error_flag tensor (sticky until
  check_errors()), in the host result-block header, and as the documented exception on the very step that carried the
  bad action, whose results are still delivered; the next valid step raises nothing;
* reset plans: a plan with rows out of range is bit for bit the run of the clamped plan, plus bit 4; an exhausted plan is
  the run of the plan tiled to the episodes actually started, plus bit 8 from the reset that wrapped around — through
  the first gte_reset and the auto-resets of the plain, fused, persistent rollout and windows=None server / mapped paths;
* past-end steps (autoreset=False): bit 2 and truncated, the stored row stays at T-1, reward / valuation / real_position
  as the contract's transition from T-2 to T-1, the observation window inside the data, fused = two-launch, and the
  info columns inside the data; a masked reset rejoins the CPU oracle.  Every table the kernels index by row is first
  re-homed between NaN-filled guard bands, so no read leaves memory the test owns, whatever the kernels do.
"""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
import invalid_inputs as V
import test_cuda_exact_edges as XE
from dyn_reference import DynColumns

pytestmark = pytest.mark.gpu

POS = [-1.0, 0.0, 0.5, 1.0, 2.0]
P = len(POS)
FEES = dict(trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000)
PATHS = dict(XE.PATHS, numpy=(XE.WIN, dict(output="numpy")))
HOST_PATHS = ("hybrid_copy", "hybrid_mapped", "hybrid_server", "f32_wire", "async", "numpy")
WIDTHS = [np.int8, np.int16, np.int32, np.int64]
STATE = ["_asset", "_fiat", "_interest_asset", "_interest_fiat", "_pos_idx", "_step", "_ep_start", "_dataset_idx",
         "_plan_cursor", "_dyn_ring", "_ring_clock", "_valuation", "_metrics_step", "_metrics_total"]


def _np(x):
    return np.array(x, copy=True) if isinstance(x, np.ndarray) else x.detach().cpu().numpy().copy()


def _series(T, seed):
    import gym_trading_env_b200 as gte
    return gte.frame_to_arrays(gte.make_gbm_ohlcv(T, seed=seed, sigma=0.01))


def _env(inst, path, N, *, strict=False, plan=None, duration=5, T=400, **over):
    import gym_trading_env_b200 as gte
    kinds, metrics, n_ds = XE.INSTANCES[inst]
    windows, kw = PATHS[path]
    args = dict(positions=POS, windows=windows, max_episode_duration=duration, num_envs=N, seed=3, verbose=0,
                strict_actions=strict, reset_plan=plan, debug_outputs=True,
                dynamic_feature_functions=[gte.DeviceFeature(k) for k in kinds], **FEES, **kw)
    args.update(over)
    series = [_series(T + 60 * k, 10 + k) for k in range(n_ds)]
    env = (gte.MultiDatasetTradingVectorEnv(datasets=series, **args) if n_ds > 1
           else gte.TradingVectorEnv(series[0], **args))
    for m in metrics:
        env.add_metric(m, gte.DeviceMetric(m))
    return env


def _snap(env, obs, reward, term, trunc):
    s = {"obs": _np(obs), "reward": _np(reward), "terminated": _np(term).view(np.uint8),
         "truncated": _np(trunc).view(np.uint8)}
    for n in STATE:
        s[n] = _np(getattr(env, n))
    for n in ("_episode_acc", "_episode_record"):
        if getattr(env, n) is not None:
            s[n] = _np(getattr(env, n))
    return s


def _same(a, b, what):
    assert a.keys() == b.keys(), what
    for n in a:
        H.assert_bits(a[n], b[n], f"{what}: {n}")


def _raises(bits):
    if bits & (V.E_ACTION_RANGE | V.E_NEGATIVE_ACTION | V.E_PAST_END):
        return pytest.raises(IndexError)
    if bits & V.E_PLAN_RANGE:
        return pytest.raises(ValueError)
    if bits & V.E_PLAN_EXHAUSTED:
        return pytest.raises(RuntimeError)
    return contextlib.nullcontext()


def _host_step(env, path, a, bits):
    """One host-path step that must raise for `bits` with the step's results delivered: (obs, reward, term, trunc,
    the result block's error word)."""
    with _raises(bits):
        if path == "async":
            env.step_async(a)
            k = (env._async["n"] - 1) & 1
            env.step_wait()
        else:
            env.step(a)
    blk = env._async["sets"][k] if path == "async" else env._host
    obs = env._host["obs"] if path == "numpy" else env._obs
    return obs, env._last_reward_host, blk["terminated"], blk["truncated"], int(blk["error"][0])


# ---- a. invalid actions -------------------------------------------------------------------------------------------------
SCHEDULE = ["none", "high", "none", "neg", "both", "none", "both", "none"]    # per step: which invalid values appear


def _bad_actions(N, dtype, seed):
    """[K, N] actions of one width: random valid entries, and per SCHEDULE invalid ones on envs around the 32-env and
    256-env tile boundaries and a few random envs."""
    info = np.iinfo(dtype)
    rng = np.random.default_rng(seed)
    acts = rng.integers(-1, P, size=(len(SCHEDULE), N)).astype(dtype)
    edge = [i for i in (0, 1, 31, 32, 33, 63, 255, 256, 257, 511, 512, 999) if i < N]
    for k, kind in enumerate(SCHEDULE):
        vals = {"none": [], "high": [P, P + 1, info.max], "neg": [-2, info.min, -1],
                "both": [P, info.min, P + 1, -2, info.max, -1]}[kind]
        if not vals:
            continue
        envs = sorted(set(edge) | set(rng.choice(N, size=max(1, N // 50), replace=False).tolist()))
        for j, i in enumerate(envs):
            acts[k, i] = vals[(j + k) % len(vals)]
    return acts


def _run_actions(inst, path, N, strict, acts):
    """Drive one env through the action rows; returns the per-step snapshots and checks the flag delivery on the way."""
    env = _env(inst, path, N, strict=strict)
    host = path in HOST_PATHS
    snaps = []
    try:
        env.reset()
        if path.startswith("rollout"):
            exp = 0
            for a in acts:
                exp |= V.hold_substituted(a, P, strict)[1]
            out = env.rollout(torch.as_tensor(acts.astype(np.int64), device=env.device), keep_obs=path == "rollout_keep")
            torch.cuda.synchronize()
            s = _snap(env, out["obs"] if "obs" in out else env._obs, out["reward"], out["terminated"], out["truncated"])
            s["valuation_k"] = _np(out["valuation"])
            snaps.append(s)
            assert int(env.error_flag.item()) == exp, (int(env.error_flag.item()), exp)
            with _raises(exp):
                env.check_errors()
            env.step(torch.full((N,), -1, dtype=torch.int64, device=env.device))
            env.check_errors()                                   # cleared: the next valid step raises nothing
            return snaps
        sticky = 0
        for k, a in enumerate(acts):
            bits = V.hold_substituted(a, P, strict)[1]
            if host:
                obs, rew, te, tr, word = _host_step(env, path, a, bits)
                assert word == bits, (k, word, bits)             # the result block's error word, this step's bits only
            else:
                obs, rew, te, tr, _ = env.step(torch.as_tensor(a.astype(np.int64), device=env.device))
                sticky |= bits
                assert int(env.error_flag.item()) == sticky, (k, int(env.error_flag.item()), sticky)
                if k in (4, len(acts) - 1):                      # sticky until check_errors(), which raises and clears
                    with _raises(sticky):
                        env.check_errors()
                    sticky = 0
            torch.cuda.synchronize()
            snaps.append(_snap(env, obs, rew, te, tr))
        if host:
            assert int(env._error_flag.item()) == 0
        env.check_errors()
        return snaps
    finally:
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        env.close()


def _check_actions(inst, path, N, strict, seed=0):
    host = path in HOST_PATHS
    rows = []
    for k in range(len(SCHEDULE)):                               # host paths: every width in turn; torch paths: int64
        dt = WIDTHS[k % 4] if host else np.int64
        rows.append(_bad_actions(N, dt, seed + 7 * k)[k])
    if not host:
        rows = np.stack(rows)
    sub = [V.hold_substituted(a, P, strict)[0] for a in rows]
    assert any(V.hold_substituted(a, P, strict)[1] for a in rows)
    got = _run_actions(inst, path, N, strict, rows)
    want = _run_actions(inst, path, N, strict, sub if host else np.stack(sub))
    for k, (g, w) in enumerate(zip(got, want)):
        _same(g, w, f"{inst} / {path} / N={N} strict={strict}, step {k}: invalid actions against holds")


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("inst", list(XE.INSTANCES))
def test_invalid_actions_equal_holds_on_every_path(inst, path):
    for strict in (False, True):
        _check_actions(inst, path, 257, strict)


@pytest.mark.parametrize("N", [1, 33, 257, 1000])
@pytest.mark.parametrize("path", ["plain", "fused", "hybrid_mapped", "async"])
def test_invalid_actions_at_env_counts_across_the_tiles(path, N):
    _check_actions("pair", path, N, True, seed=N)


# ---- b. reset plans -----------------------------------------------------------------------------------------------------
PLAN_PATHS = ["plain", "fused", "rollout", "hybrid_mapped", "hybrid_server"]
BAD_FIELDS = ["start<W-1", "start>T-2", "start<<0", "pos=-1", "pos=P", "ds=-1", "ds=n_ds", "all"]


def _plan(N, E, lengths, W, n_ds, seed):
    """A valid plan with one bad field (or all of them) in a third of its rows, episode 0 (the first gte_reset) included."""
    rng = np.random.default_rng(seed)
    lo = (W or 1) - 1
    plan = np.zeros((N, E, 3), np.int32)
    plan[:, :, 2] = rng.integers(0, n_ds, size=(N, E))
    plan[:, :, 0] = rng.integers(lo, min(lengths) - 30, size=(N, E))
    plan[:, :, 1] = rng.integers(0, P, size=(N, E))
    for i in range(N):
        for j in range(E):
            f = (i + 2 * j) % (3 * len(BAD_FIELDS) // 2)
            if f >= len(BAD_FIELDS):
                continue
            name, T = BAD_FIELDS[f], lengths[plan[i, j, 2]]
            if name in ("start<W-1", "all"):
                plan[i, j, 0] = lo - 1 if lo > 0 else -1
            if name == "start>T-2":
                plan[i, j, 0] = T - 1 + (i % 3) * 1000
            if name == "start<<0":
                plan[i, j, 0] = -(1 << 30)
            if name in ("pos=-1", "all"):
                plan[i, j, 1] = -1
            if name == "pos=P":
                plan[i, j, 1] = P
            if name == "ds=-1":
                plan[i, j, 2] = -1
            if name in ("ds=n_ds", "all"):
                plan[i, j, 2] = n_ds
    return plan


def _run_plan(inst, path, plan, K, acts):
    """(snapshots, plan cursor after the reset and after every step, error word per step (host) / sticky flag)"""
    N = plan.shape[0]
    env = _env(inst, path, N, plan=plan)
    host = path in HOST_PATHS
    try:
        env.reset()
        cursors = [_np(env._plan_cursor)]
        words = [int(env._error_flag.item())]
        snaps = []
        if path == "rollout":
            out = env.rollout(torch.as_tensor(acts, device=env.device))
            torch.cuda.synchronize()
            snaps.append(_snap(env, env._obs, out["reward"], out["terminated"], out["truncated"]))
            snaps[-1]["valuation_k"] = _np(out["valuation"])
            cursors.append(_np(env._plan_cursor))
            words.append(int(env._error_flag.item()))
            return env, snaps, cursors, words
        for k in range(K):
            if host:
                word = [None]
                try:
                    env.step(acts[k].astype(np.int8))
                except (ValueError, RuntimeError) as e:
                    word[0] = e
                blk = env._host
                obs, rew, te, tr = env._obs, env._last_reward_host, blk["terminated"], blk["truncated"]
                words.append((int(blk["error"][0]), type(word[0])))
            else:
                obs, rew, te, tr, _ = env.step(torch.as_tensor(acts[k], device=env.device))
                words.append(int(env.error_flag.item()))
            torch.cuda.synchronize()
            cursors.append(_np(env._plan_cursor))
            snaps.append(_snap(env, obs, rew, te, tr))
        return env, snaps, cursors, words
    finally:
        torch.cuda.synchronize()
        env._lib.gte_serve_stop()
        env.close()


def _expected_bits(cursors, row_bits, E):
    """Per step (index 0 = the first gte_reset): the bits of the resets that step performed, from the plan cursors."""
    out = []
    prev = np.zeros_like(cursors[0])
    for cur in cursors:
        b = 0
        for i in np.nonzero(cur > prev)[0]:
            for c in range(prev[i], cur[i]):                     # reset number c consumed row c % E
                b |= int(row_bits[i, c % E])
                if c >= E:
                    b |= V.E_PLAN_EXHAUSTED
        out.append(b)
        prev = cur
    return out


@pytest.mark.parametrize("path", PLAN_PATHS)
@pytest.mark.parametrize("inst", ["pair", "metrics", "catalogue+stateful", "two datasets"])
def test_reset_plans_clamp_and_wrap_as_the_reference(inst, path):
    N, E, K = 257, 3, 14
    n_ds = XE.INSTANCES[inst][2]
    W = PATHS[path][0]
    lengths = [400 + 60 * k for k in range(n_ds)]
    bad = _plan(N, E, lengths, W, n_ds, seed=len(inst))
    clamped, row_bits = V.clamped_plan(bad, lengths, W, P, n_ds, multi=n_ds > 1)
    assert row_bits[:, 0].any() and row_bits[:, 1:].any()
    acts = np.random.default_rng(2).integers(-1, P, size=(K, N))
    _, got, cur_b, words_b = _run_plan(inst, path, bad, K, acts)
    _, want, cur_c, words_c = _run_plan(inst, path, clamped, K, acts)
    for k, (g, w) in enumerate(zip(got, want)):
        _same(g, w, f"{inst} / {path}, step {k}: out-of-range plan against the clamped plan")
    for c_b, c_c in zip(cur_b, cur_c):
        H.assert_bits(c_b, c_c, "plan cursors")
    started = int(cur_c[-1].max())
    assert started > E                                           # the plan wrapped around (short clamped episodes)
    tiled, first = V.wrapped_plan(clamped, started)
    assert first == E
    _, tiled_snaps, cur_t, words_t = _run_plan(inst, path, tiled, K, acts)
    for k, (g, w) in enumerate(zip(tiled_snaps, want)):
        g = dict(g, _plan_cursor=w["_plan_cursor"])              # the tiled plan's cursor runs over more rows
        _same(g, w, f"{inst} / {path}, step {k}: exhausted plan against the tiled plan")
    exp_bad = _expected_bits(cur_c, row_bits, E)
    exp_clamped = _expected_bits(cur_c, np.zeros_like(row_bits), E)
    wrap_step = next(k for k, c in enumerate(cur_c) if (c > E).any())
    assert all(b & V.E_PLAN_EXHAUSTED == 0 for b in exp_clamped[:wrap_step]) and exp_clamped[wrap_step] & V.E_PLAN_EXHAUSTED
    exp_tiled = [0] * len(cur_t)
    if path in HOST_PATHS:
        # the first gte_reset's bits reach the host with the first step's result block; every step's word is its own
        for words, exp in ((words_b, exp_bad), (words_c, exp_clamped), (words_t, exp_tiled)):
            assert words[0] == exp[0]
            exp = [exp[0] | exp[1]] + exp[2:]
            for k, ((word, raised), e) in enumerate(zip(words[1:], exp)):
                assert word == e, (k, word, e)
                cls = ValueError if e & V.E_PLAN_RANGE else RuntimeError if e & V.E_PLAN_EXHAUSTED else type(None)
                assert raised is cls, (k, raised, e)
    else:
        # torch mode: the bits are sticky (nobody calls check_errors() here)
        for words, exp in ((words_b, exp_bad), (words_c, exp_clamped), (words_t, exp_tiled)):
            sticky = [int(np.bitwise_or.reduce(exp[:k + 1])) for k in range(len(exp))]
            if path == "rollout":
                sticky = [sticky[0], sticky[-1]]
            assert words == sticky, (words, sticky)


# ---- c. past-end steps --------------------------------------------------------------------------------------------------
PAYLOAD = 0x7FF4DEAD                      # a NaN as float32, and (twice) as float64
GUARD = 64 << 10
DUR = 20


def _rehome(env):
    """Every table the kernels index by row (window tables at their shifted base, features, price, high / low) moves
    between GUARD bytes of NaN payload on each side; returns the guard buffers."""
    bands = []

    def home(t):
        nbytes = t.numel() * t.element_size()
        big = torch.empty(2 * GUARD + nbytes + (-nbytes) % 16, dtype=torch.uint8, device=env.device)
        big.view(torch.int32).fill_(PAYLOAD)
        view = big[GUARD:GUARD + nbytes].view(t.dtype).view(t.shape)
        view.copy_(t)
        bands.append(big)
        return view

    env._features = home(env._features)
    env._price = home(env._price)
    for c, t in enumerate(env._window_tables):
        if t is not None:
            shift = env._window_ptrs[c] - t.data_ptr()
            env._window_tables[c] = home(t)
            env._window_ptrs[c] = env._window_tables[c].data_ptr() + shift
    if getattr(env, "_high", None) is not None:
        env._high, env._low = home(env._high), home(env._low)
    env._build_structs()
    return bands


def _past_env(N, windows, *, n_ds=1, variant="auto", n_chunks=0, seed=0, **kw):
    """An env (autoreset=False) whose plan starts every episode 0 at T-3 (every 7th env at T-2) and episodes 1, 2 at
    ordinary rows; its tables re-homed between guard bands."""
    import gym_trading_env_b200 as gte
    lengths = [300 + 120 * k for k in range(n_ds)]               # dataset 0 is the shorter one and not the last
    series = [_series(T, 20 + k) for k, T in enumerate(lengths)]
    rng = np.random.default_rng(seed)
    plan = np.zeros((N, 3, 3), np.int32)
    plan[:, :, 2] = (np.arange(N) % n_ds)[:, None]
    T = np.asarray(lengths)[plan[:, 0, 2]]
    plan[:, 0, 0] = np.where(np.arange(N) % 7 == 3, T - 2, T - 3)
    plan[:, 1:, 0] = rng.integers((windows or 1) - 1, min(lengths) - DUR - 10, size=(N, 2))
    plan[:, :, 1] = rng.integers(0, P, size=(N, 3))
    args = dict(positions=POS, windows=windows, max_episode_duration=DUR, num_envs=N, verbose=0, reset_plan=plan,
                autoreset=False, debug_outputs=True, obs_variant=variant, n_chunks=n_chunks, **FEES, **kw)
    env = (gte.MultiDatasetTradingVectorEnv(datasets=series, **args) if n_ds > 1 else gte.TradingVectorEnv(series[0], **args))
    return env, _rehome(env), series, plan


STATE_IN = ["_asset", "_fiat", "_interest_asset", "_interest_fiat", "_pos_idx", "_step", "_ep_start", "_dataset_idx"]


def _state(env):
    return {n: _np(getattr(env, n)) for n in STATE_IN}


def _check_past_step(env, k, pre, acts, series, out, cols, windows, sample):
    """Steps 1-4 of the contract check for one step (in the order that keeps a wrong stored row from reaching any
    further read)."""
    obs, rew, trunc, flag = out
    lengths = np.array([s.length for s in series])
    T = lengths[pre["_dataset_idx"]]
    past = pre["_ep_start"] + pre["_step"] >= T - 1
    ended = past | (pre["_ep_start"] + pre["_step"] + 1 >= T - 1)
    # 1. bit 2 and truncated
    assert flag == (V.E_PAST_END if past.any() else 0), (k, flag)
    assert np.asarray(trunc, bool)[ended].all(), f"step {k}: truncated"
    # 2. the stored row and the info row stay at T-1
    post = _state(env)
    idx = post["_ep_start"] + post["_step"]
    H.assert_bits(idx[ended], (T - 1)[ended], f"step {k}: stored row ep_start + step")
    H.assert_bits(_np(env._info_idx)[ended], (T - 1)[ended], f"step {k}: info idx")
    H.assert_bits(_np(env._info_step)[ended], (T - 1 - post["_ep_start"])[ended], f"step {k}: info step")
    # 3. reward, valuation, real_position as the transition T-2 -> T-1 from the current portfolio
    rew, val, rp = np.asarray(rew, np.float64), _np(env._valuation), _np(env._real_position)
    for i in np.nonzero(past & sample)[0]:
        s = V.past_end_step([pre[n][i] for n in STATE_IN[:4]], int(pre["_pos_idx"][i]), int(acts[i]),
                            series[pre["_dataset_idx"][i]].price[T[i] - 2], series[pre["_dataset_idx"][i]].price[T[i] - 1],
                            positions=POS, fee=FEES["trading_fees"], rate=FEES["borrow_interest_rate"],
                            v0=FEES["portfolio_initial_value"], started_at_t2=pre["_ep_start"][i] == T[i] - 2,
                            reward=("log_return", 1.0, -np.inf, np.inf))
        what = f"step {k} env {i}"
        assert H_bits(rew[i]) in s["reward_bits"], (what, rew[i], s["reward"])
        H.assert_bits(np.array([val[i], rp[i]]), np.array([s["valuation"], s["real_position"]]), what)
        assert post["_pos_idx"][i] == s["pos_idx"], what
    # 4. the observation: static rows idx-W+1 .. idx of the tables, dynamic columns from the device's own outputs
    pidx = post["_pos_idx"]
    cols.step(pidx, rp, val, rew, _np(env._info_step), idx, np.zeros(len(idx), bool), pidx)
    W = windows or 1
    rows = idx[:, None] - (W - 1) + np.arange(W)[None, :]
    static = np.zeros(rows.shape + (series[0].features.shape[1],), np.float32)
    for d, s in enumerate(series):
        m = post["_dataset_idx"] == d
        static[m] = s.features[rows[m]]
    dyn = cols.select(cols.window(idx, post["_ep_start"]), ["position", "real_position"])
    want = np.concatenate([static, dyn], axis=-1)
    H.assert_bits(np.asarray(obs), want if windows else want[:, 0], f"step {k}: observation")
    assert not (np.asarray(obs).view(np.uint32) == PAYLOAD).any(), f"step {k}: a guard band reached the observation"


def H_bits(x):
    import exact_edges as X
    return X.bits(float(x))


def _drive_past(env, driver, a):
    """One step of the given driver; returns (obs, reward, truncated, error bits of the step)."""
    if driver in ("numpy", "hybrid"):
        with contextlib.suppress(IndexError):
            env.step(a.astype(np.int16))
        hb = env._host
        return hb["obs"] if driver == "numpy" else _np(env._obs), hb["reward"].copy(), hb["truncated"].copy(), int(hb["error"][0])
    obs, rew, _, tr, _ = env.step(torch.as_tensor(a, device=env.device))
    flag = int(env.error_flag.item())
    if flag:
        with pytest.raises(IndexError):
            env.check_errors()
    return _np(obs), _np(rew), _np(tr), flag


def _past_end_run(N, windows, *, driver="torch", variant="auto", n_ds=1, twin=False, **kw):
    import oracle as orc
    out_kw = {"numpy": dict(output="numpy"), "hybrid": dict(output="hybrid"), "graph": dict(cuda_graph=True)}.get(driver, {})
    env, bands, series, plan = _past_env(N, windows, n_ds=n_ds, variant=variant, **out_kw, **kw)
    other = _past_env(N, windows, n_ds=n_ds, variant=variant, n_chunks=1, **kw) if twin else None
    assert not twin or other[0].launches_per_step == 2
    try:
        env.reset()
        if other:
            other[0].reset()
        cols = DynColumns(N, windows, POS, FEES["portfolio_initial_value"], DUR)
        cols.reset(_np(env._pos_idx))
        rng = np.random.default_rng(1)
        sample = np.ones(N, bool) if N <= 4096 else (rng.random(N) < 2000 / N)
        sample[:64] = sample[-64:] = True
        W = windows or 1
        for k in range(2 + W + 2):                               # to the last row, then W + 2 past-end steps
            pre = _state(env)
            acts = rng.integers(-1, P, size=N)
            out = _drive_past(env, driver, acts)
            _check_past_step(env, k, pre, acts, series, out, cols, windows, sample)
            if other:                                            # 5. the two-launch form gives the same bits
                o = _drive_past(other[0], "torch", acts)
                for j, n in enumerate(("obs", "reward", "truncated", "flag")):
                    H.assert_bits(np.asarray(o[j]), np.asarray(out[j]), f"step {k}: two-launch {n}")
                # (the metric sums are reduced over other CTA shapes: only the counts are bit-exact)
                same = [n for n in STATE if not n.startswith("_metrics")] + ["_real_position", "_info_idx", "_info_step"]
                _same({n: _np(getattr(other[0], n)) for n in same}, {n: _np(getattr(env, n)) for n in same},
                      f"step {k}: two-launch state")
                H.assert_bits(_np(other[0]._metrics_step)[:3], _np(env._metrics_step)[:3], f"step {k}: two-launch counts")
        assert (_np(env._metrics_step)[2] == N) and (_np(env._metrics_step)[0] == N)     # counted like any truncation
        # 6. only now: the info columns look rows up on the host and on the device
        ds, T = _np(env._dataset_idx), np.array([s.length for s in series])[_np(env._dataset_idx)]
        inf = env.infos
        want_close = np.array([series[d].price[t - 1] for d, t in zip(ds, T)])
        H.assert_bits(_np(inf["data_close"]), want_close, "infos data_close")
        H.assert_bits(_np(inf["data_high"]), np.array([series[d].info["high"][t - 1] for d, t in zip(ds, T)]), "data_high")
        if "date" in inf.KEYS:
            assert (inf["date"] == np.array([series[d].index[t - 1] for d, t in zip(ds, T)])).all()
        assert not np.isnan(_np(env._valuation)).any() and not np.isnan(_np(env._reward)).any()
        # a masked reset of the ended envs rejoins the oracle (plan rows 1.. from here on)
        lengths = np.array([s.length for s in series])
        feats = np.zeros((n_ds, lengths.max(), series[0].features.shape[1]), np.float32)
        price = np.ones((n_ds, lengths.max()))
        for d, s in enumerate(series):
            feats[d, :s.length], price[d, :s.length] = s.features, s.price
        o = orc.OracleVecEnv(feats, price, lengths, num_envs=N, positions=POS, windows=windows, plan=plan[:, 1:],
                             multi_dataset=n_ds > 1, max_episode_duration=DUR, **FEES)
        mask = _np(env._truncated).astype(bool)
        assert mask.all()
        obs, _ = env.reset(options={"mask": mask})
        H.assert_bits(_np(obs), o.reset(), "masked reset rejoins the oracle")
        for k in range(4):
            a = rng.integers(-1, P, size=N)
            if driver in ("numpy", "hybrid"):
                obs = env.step(a.astype(np.int64))[0]
            else:
                obs = env.step(torch.as_tensor(a, device=env.device))[0]
            o.step(a)
            H.assert_bits(_np(obs), o.obs, f"after the reset, step {k}: obs")
            H.assert_bits(_np(env._valuation), o.valuation, f"after the reset, step {k}: valuation")
        env.check_errors()
        torch.cuda.synchronize()
        for big in bands:                                        # the guard bands are read-only to the kernels
            assert bool((big[:GUARD].view(torch.int32) == PAYLOAD).all())
            assert bool((big[-GUARD:].view(torch.int32) == PAYLOAD).all())
    finally:
        torch.cuda.synchronize()
        env.close()
        if other:
            other[0].close()


@pytest.mark.parametrize("windows,variant", [(None, "auto"), (8, "tma"), (8, "vec"), (8, "generic"), (64, "tma"),
                                             (64, "vec"), (64, "generic")])
def test_past_end_steps_stay_inside_the_data(windows, variant):
    _past_end_run(1000, windows, variant=variant, twin=windows is not None)


def test_past_end_steps_claimed_tiles_gather():
    _past_end_run(150_016, 8, variant="tma", twin=True)


@pytest.mark.parametrize("driver", ["graph", "numpy", "hybrid"])
def test_past_end_steps_on_the_other_step_paths(driver):
    _past_end_run(1000, 8, driver=driver)


def test_past_end_steps_on_a_shorter_dataset_that_is_not_the_last():
    _past_end_run(1000, 8, n_ds=2, twin=True)
    _past_end_run(333, None, n_ds=2)


@pytest.mark.parametrize("windows", [None, 8])
def test_past_end_steps_in_the_persistent_rollout_kernel(windows):
    """gte_rollout with autoreset=0 (the state stays in registers across its iterations) against the same steps taken one
    call at a time."""
    from gym_trading_env_b200 import _cabi
    N = 1000
    K = 2 + (windows or 1) + 2
    env, bands, series, _ = _past_env(N, windows, n_chunks=1)
    ref, _, _, _ = _past_env(N, windows, n_chunks=1)
    try:
        env.reset()
        ref.reset()
        acts = torch.as_tensor(np.random.default_rng(3).integers(-1, P, size=(K, N)), device=env.device)
        want = {n: [] for n in ("reward", "terminated", "truncated", "valuation")}
        for k in range(K):
            ref.step(acts[k])
            for n in want:
                want[n].append(_np(getattr(ref, "_" + n)))
        got = {n: torch.zeros(K, N, dtype=torch.float64 if n in ("reward", "valuation") else torch.uint8,
                              device=env.device) for n in want}
        o = _cabi.GteStepOut()
        C.memmove(C.byref(o), C.byref(env._O), C.sizeof(o))
        o.reward, o.terminated, o.truncated = got["reward"].data_ptr(), got["terminated"].data_ptr(), got["truncated"].data_ptr()
        o.valuation = got["valuation"].data_ptr()
        o.real_position = o.info_idx = o.info_step = o.pre_reset_portfolio = None
        env._tick += K
        _cabi.check(env._lib.gte_rollout(C.byref(env._P), C.byref(env._D), C.byref(env._S), C.c_void_p(acts.data_ptr()),
                                         K, C.byref(o), C.c_void_p(env._obs.data_ptr()), 0, 0, env._obs_variant,
                                         env._stream()), "gte_rollout")
        torch.cuda.synchronize()
        assert int(env._error_flag.item()) == V.E_PAST_END
        T = np.array([s.length for s in series])[_np(env._dataset_idx)]
        H.assert_bits(_np(env._ep_start) + _np(env._step), T - 1, "rollout: stored row")
        for n in want:
            H.assert_bits(_np(got[n]), np.stack(want[n]).view(_np(got[n]).dtype), f"rollout: {n}")
        # (the rollout folds its sums in another order; its valuations went to got["valuation"])
        same = [n for n in STATE if n not in ("_metrics_total", "_valuation")]
        _same({n: _np(getattr(env, n)) for n in same} | {"obs": _np(env._obs)},
              {n: _np(getattr(ref, n)) for n in same} | {"obs": _np(ref._obs)},
              "rollout against single steps")
        for big in bands:
            assert bool((big[:GUARD].view(torch.int32) == PAYLOAD).all())
    finally:
        torch.cuda.synchronize()
        env._error_flag.zero_()
        env.close()
        ref.close()
