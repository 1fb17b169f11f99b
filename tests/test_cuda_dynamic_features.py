"""GPU: the dynamic-feature catalogue (gte.DeviceFeature) on the device, bit for bit against the CPU oracle whose
dynamic columns are rebuilt from the catalogue's executable specification (tests/dyn_reference.py) — every gather
variant, window shape, work-unit size, the fused and the two-launch forms, multi-dataset, final_obs, masked resets,
CUDA graphs, rollout, the host-output modes and checkpoints."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers as H
from dyn_reference import CatalogueOracle

pytestmark = pytest.mark.gpu

KINDS = ["position", "real_position", "portfolio_return", "reward", "episode_progress"]
ALL5 = ["episode_progress", "reward", "position", "portfolio_return", "real_position"]
CONFIGS = [[k] for k in KINDS] + [["real_position", "position"], ALL5]
IDS = ["+".join(c) for c in CONFIGS]
FEES = dict(trading_fees=1e-4, borrow_interest_rate=3e-6, portfolio_initial_value=1000)


def _features(kinds, duration):
    import gym_trading_env_b200 as gte
    return [gte.episode_progress_feature(duration) if k == "episode_progress" else gte.DeviceFeature(k) for k in kinds]


def _series(T, seed, n_features=8):
    import gym_trading_env_b200 as gte
    s = gte.frame_to_arrays(gte.make_gbm_ohlcv(T, seed=seed))
    if n_features != s.features.shape[1]:
        f = np.ascontiguousarray(np.resize(s.features.T, (n_features, s.length)).T)
        s = gte.SeriesArrays(f, s.price, [f"feature_{j}" for j in range(n_features)], {}, None)
    return s


def _np(x):
    return x if isinstance(x, np.ndarray) else x.cpu().numpy()


def _plan(n_envs, windows, duration, T, n_pos, episodes=40, seed=0):
    """Recorded episode starts (reset_plan): the final_obs mode resets through gte_reset, whose Philox draws are keyed
    by a later tick than the in-kernel auto-reset's."""
    rng = np.random.default_rng(seed)
    lo = (windows or 1) - 1
    plan = np.zeros((n_envs, episodes, 3), np.int32)
    plan[:, :, 0] = rng.integers(lo, T - duration - lo, size=(n_envs, episodes))
    plan[:, :, 1] = rng.integers(0, n_pos, size=(n_envs, episodes))
    return plan


def _pair(kinds, n_envs, *, windows, duration=40, positions=(-1, 0, 0.5, 1, 2), series=None, seed=5, multi=False,
          plan=None, **dev_kw):
    """A device env with the catalogue and the oracle reference of the same shape."""
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
    return dev, CatalogueOracle(o, kinds, duration)


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
        H.assert_bits(dev._valuation.cpu().numpy(), ref.o.valuation, f"step {k} valuation")
        ended = (ref.o.terminated | ref.o.truncated).astype(bool)
        if check_final and ended.any():
            H.assert_bits(_np(dev.final_obs)[ended], ref.final_obs[ended], f"{kinds} step {k} final_obs")
    dev.check_errors()
    assert ref.o.metrics[0] >= 0
    return dev, ref


@pytest.mark.parametrize("kinds", CONFIGS, ids=IDS)
@pytest.mark.parametrize("windows,variant", [(None, "auto"), (None, "generic"), (8, "auto"), (8, "generic"),
                                             (8, "vec"), (8, "tma"), (64, "auto"), (64, "vec"), (64, "tma")])
def test_catalogue_matches_the_oracle_in_every_variant(kinds, windows, variant):
    dev, _ = _run(kinds, 300, K=30 if windows != 64 else 50, windows=windows, obs_variant=variant,
                  duration=40 if windows != 64 else 30)
    if variant == "auto" and windows is not None:
        assert dev.obs_variant == "tma"


@pytest.mark.parametrize("kinds", [["real_position", "position"], ALL5], ids=["swapped", "all5"])
def test_window_off_the_16_byte_grid_runs_the_generic_gather(kinds):
    """windows=5 with F = 10: 200-byte windows are not a multiple of 16 -> no window tables, the generic gather."""
    ns = 10 - len(kinds)
    dev, _ = _run(kinds, 257, K=40, windows=5, series=[_series(1500, 4, n_features=ns)])
    assert dev._resolved_variant == 1 and dev.obs_variant == "generic"


@pytest.mark.parametrize("kinds", [["position"], ["reward"], ALL5], ids=["position", "reward", "all5"])
@pytest.mark.parametrize("n_envs", [40, 1000, 9000, 70_000, 300_000])
def test_work_units_fused_and_two_launches(kinds, n_envs):
    """Batch sizes that select the 8-, 16- and 32-env work units, the fused single launch and two launches (the
    claimed-tiles gather from ~150k envs on)."""
    dev, _ = _run(kinds, n_envs, K=12 if n_envs < 100_000 else 6, windows=16, duration=10,
                  series=[_series(3000, 6)])
    assert dev.obs_variant == "tma"
    if n_envs >= 300_000:
        assert dev.launches_per_step == 2


def test_multi_dataset_rotation():
    series = [_series(T, 40 + k) for k, T in enumerate([600, 750, 680])]
    _run(ALL5, 333, K=60, windows=8, duration=20, series=series, multi=True)


@pytest.mark.parametrize("kinds", [["reward", "episode_progress"], ALL5], ids=["reward+progress", "all5"])
def test_final_obs_keeps_the_terminal_observation(kinds):
    _run(kinds, 200, K=45, windows=8, duration=15, final_obs=True, check_final=True,
         plan=_plan(200, 8, 15, 1500, 5))


@pytest.mark.parametrize("variant", ["generic", "vec", "tma"])
def test_masked_reset_in_the_middle_of_a_run(variant):
    dev, ref = _pair(ALL5, 203, windows=12, duration=50, obs_variant=variant)
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


@pytest.mark.parametrize("windows", [None, 16])
def test_cuda_graph_replay(windows):
    _run(ALL5, 500, K=30, windows=windows, duration=20, cuda_graph=True)


@pytest.mark.parametrize("windows", [None, 8])
@pytest.mark.parametrize("keep_obs", [True, False])
def test_rollout_equals_the_oracle(windows, keep_obs):
    dev, ref = _pair(ALL5, 500, windows=windows, duration=20)
    dev.reset()
    ref.reset()
    rng = np.random.default_rng(2)
    acts = rng.integers(0, 5, size=(35, 500))
    out = dev.rollout(torch.as_tensor(acts, device=dev.device), keep_obs=keep_obs)
    for k in range(35):
        ref.step(acts[k])
        if keep_obs:
            H.assert_bits(out["obs"][k].cpu().numpy(), ref.obs, f"rollout obs {k}")
    H.assert_bits(dev._obs.cpu().numpy(), ref.obs, "rollout last obs")


@pytest.mark.parametrize("output,host_io", [("numpy", "auto"), ("hybrid", "copy"), ("hybrid", "mapped"),
                                            ("hybrid", "server"), ("numpy", "server")])
def test_host_output_modes_with_one_row_observations(output, host_io):
    dev, _ = _run(ALL5, 1000, K=40, windows=None, duration=20, output=output, host_io=host_io)


def test_host_output_modes_windowed():
    _run(ALL5, 1000, K=30, windows=8, duration=20, output="hybrid", host_io="copy")


def test_state_dict_round_trip_mid_episode():
    import gym_trading_env_b200 as gte
    s = _series(900, 9)
    kw = dict(positions=[-1, 0, 1, 2], windows=16, max_episode_duration=25, num_envs=300, seed=4, verbose=0,
              dynamic_feature_functions=_features(ALL5, 25), **FEES)
    a, b = gte.TradingVectorEnv(s, **kw), gte.TradingVectorEnv(s, **kw)
    a.reset(); b.reset()
    g = torch.Generator(device=a.device); g.manual_seed(3)
    acts = torch.randint(0, 4, (70, 300), generator=g, device=a.device)
    for k in range(33):
        a.step(acts[k])
    assert a._dyn_ring.shape[1] == 16 * (4 * 128 + 32)
    snap = a.state_dict()
    b.load_state_dict(snap)
    b._launch_obs()
    assert torch.equal(b._obs.view(torch.int32), a._obs.view(torch.int32))
    for k in range(33, 70):
        oa = a.step(acts[k])[0]
        ob = b.step(acts[k])[0]
        assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), k


@pytest.mark.parametrize("windows,n_envs", [(None, 700), (8, 700), (64, 4096), (64, 300_000)])
def test_explicit_default_pair_is_the_default_env(windows, n_envs):
    """[DeviceFeature("position"), DeviceFeature("real_position")] is the default configuration: same observations bit
    for bit, same gather variant, same launches per step."""
    import gym_trading_env_b200 as gte
    s = _series(3000, 8)
    kw = dict(positions=[-3, -2, -1, 0, 1, 2, 3], windows=windows, max_episode_duration=20, num_envs=n_envs, seed=1,
              verbose=0, **FEES)
    a = gte.TradingVectorEnv(s, **kw)
    b = gte.TradingVectorEnv(s, dynamic_feature_functions=[gte.DeviceFeature("position"),
                                                           gte.DeviceFeature("real_position")], **kw)
    assert a._dyn_ring.shape == b._dyn_ring.shape
    assert a.obs_variant == b.obs_variant and a.launches_per_step == b.launches_per_step
    oa, _ = a.reset()
    ob, _ = b.reset()
    assert torch.equal(oa.view(torch.int32), ob.view(torch.int32))
    g = torch.Generator(device=a.device); g.manual_seed(5)
    for k in range(25):
        act = torch.randint(0, 7, (n_envs,), generator=g, device=a.device)
        oa = a.step(act)[0]
        ob = b.step(act)[0]
        assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), k


def test_full_size_c5_shard_with_all_five_columns():
    """The C5 shard shape (2^21 envs, W=64, 7 positions, D=720) with all five columns for 1 500 iterations (two full
    episodes), a 128-env block checked against the oracle along the way."""
    import gym_trading_env_b200 as gte
    import oracle as orc
    N, W, D, K = 1 << 21, 64, 720, 1500
    pos = [-3, -2, -1, 0, 1, 2, 3]
    s = gte.frame_to_arrays(gte.make_gbm_ohlcv(100_000, seed=0))
    kw = dict(positions=pos, windows=W, max_episode_duration=D, **FEES)
    dev = gte.TradingVectorEnv(s, num_envs=N, seed=3, verbose=0, dynamic_feature_functions=_features(ALL5, D), **kw)
    assert dev.obs_variant == "tma"
    lo, n = 1_048_544, 128                 # straddles the middle of the batch, a multiple of 32
    ref = CatalogueOracle(orc.OracleVecEnv(s.features, s.price, num_envs=n, seed=3, env_id_offset=lo, **kw), ALL5, D)
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
    H.assert_bits(dev._valuation[lo:lo + n].cpu().numpy(), ref.o.valuation, "valuation block")
    dev.check_errors()
    assert episodes >= 2 * n * 0.5


@pytest.mark.parametrize("env_var", ["GTE_TMA_DYN=2", "GTE_FUSED=0"])
def test_tma_cases_with_claimed_tiles_and_without_the_fused_launch(env_var):
    """The TMA cases of this file again with the claimed-tiles gather forced on for every batch (GTE_TMA_DYN=2) and
    with the fused single launch switched off (GTE_FUSED=0)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    k, v = env_var.split("=")
    env = dict(os.environ, **{k: v})
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider",
           "-k", "(every_variant and (auto or tma)) or work_units or final_obs or rollout or explicit_default",
           os.path.abspath(__file__)]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
