"""gymnasium-VectorEnv-shaped host classes over the CUDA library (the drop-in boundary, SURVEY.md §8b).

``TradingVectorEnv`` keeps the constructor surface of the reference ``TradingEnv``
(`/root/reference/src/gym_trading_env/environments.py:79-93`) and ``MultiDatasetTradingVectorEnv``
that of ``MultiDatasetTradingEnv`` (`:365-371`), plus ``num_envs`` / ``device`` / ``seed``.
``reset(seed, options) -> (obs, infos)`` and ``step(actions) -> (obs, rewards, terminations,
truncations, infos)`` follow gymnasium's vector API with SAME-STEP in-place auto-reset: where an
episode ended, reward/flags are the terminal step's and obs/state are those of the fresh episode.

Everything numeric happens in ``libgte_b200.so`` (hand-written sm_100a kernels) through ctypes on raw
``tensor.data_ptr()`` pointers; PyTorch only owns device memory and streams.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import glob as _glob
import os
from collections.abc import Mapping
from pathlib import Path

import numpy as np
import torch

from . import _cabi
from .dynamic_features import (DeviceFeature, current_drawdown_feature, episode_progress_feature,  # noqa: F401
                               parse_dynamic_features, portfolio_return_feature, position_age_feature, reward_feature,
                               stateful_kinds_of)
from . import episode_metrics as _em
from .episode_metrics import (DeviceMetric, episode_length_metric, episode_reward_metric,  # noqa: F401
                              max_drawdown_metric, position_changes_metric, time_in_market_metric)
from .data import SeriesArrays, build_window_tables, frame_to_arrays, load_frame, reconcile_series


# host action arrays cross PCIe in their own width and are widened by the step kernel's load (GteParams.action_bytes)
_WIRE_ACTION_DTYPES = (np.dtype(np.int8), np.dtype(np.int16), np.dtype(np.int32), np.dtype(np.int64))


# ---- names the reference exports and callers pass back in (identity-compared, never called) -------
def basic_reward_function(history=None):
    """Sentinel for the reference's ``basic_reward_function`` (environments.py:17-18):
    ``log(valuation[-1] / valuation[-2])``.  Selects the fused device log-return reward."""
    raise NotImplementedError("basic_reward_function is evaluated inside the CUDA step kernel")


def dynamic_feature_last_position_taken(history=None):
    """Sentinel for environments.py:20-21 (position taken at the last step)."""
    raise NotImplementedError("evaluated inside the CUDA step kernel")


def dynamic_feature_real_position(history=None):
    """Sentinel for environments.py:23-24 (real position of the portfolio)."""
    raise NotImplementedError("evaluated inside the CUDA step kernel")


_DEFAULT_DYNAMIC = [dynamic_feature_last_position_taken, dynamic_feature_real_position]


class DeviceReward:
    """A reward functor fused into the CUDA step kernel:
    ``reward = clip(scale * f(valuation[-1], valuation[-2]), lo, hi)`` with ``f`` the log-return
    (``kind="log_return"``, the reference's ``basic_reward_function``, environments.py:17-18) or the simple
    return ``(v[-1]-v[-2])/v[-2]`` (``kind="simple_return"``).  Covers the variants the reference's callers
    pass as Python callbacks — ``np.clip(log_return, -0.002, 0.005)`` (luckymodel/envs/env.py:16-18),
    ``100 * log_return`` (luckymodel/scripts/test_env.py:20-22), ``max(0, simple_return)`` (env.py:19) —
    without a CPU fallback.  Evaluated only when the step did not terminate (environments.py:265-267)."""

    KINDS = {"log_return": _cabi.REWARD_LOG_RETURN, "simple_return": _cabi.REWARD_SIMPLE_RETURN}

    def __init__(self, kind="log_return", scale=1.0, clip=None):
        if kind not in self.KINDS:
            raise ValueError(f"kind must be one of {list(self.KINDS)}")
        self.kind, self.scale = kind, float(scale)
        lo, hi = (-np.inf, np.inf) if clip is None else clip
        self.lo = -np.inf if lo is None else float(lo)
        self.hi = np.inf if hi is None else float(hi)
        if not self.lo <= self.hi:
            raise ValueError("clip must be (lo, hi) with lo <= hi")

    def __repr__(self):
        return f"DeviceReward(kind={self.kind!r}, scale={self.scale}, clip=({self.lo}, {self.hi}))"


def log_return_reward(scale=1.0, clip=None):
    """``clip(scale * log(v[-1]/v[-2]), *clip)`` on the device."""
    return DeviceReward("log_return", scale, clip)


def simple_return_reward(scale=1.0, clip=None):
    """``clip(scale * (v[-1]-v[-2])/v[-2], *clip)`` on the device."""
    return DeviceReward("simple_return", scale, clip)


def _fn_name(f):
    return getattr(f, "__name__", None)


# ---- gymnasium's VectorEnv base class and spaces when importable, else duck-typed stand-ins ---------
# (SURVEY.md §8b: "inherit from gymnasium.vector.VectorEnv only if importable"; gymnasium is absent from the build image)
try:
    import gymnasium as _gym
    from gymnasium import spaces as _spaces
    _VectorEnvBase = _gym.vector.VectorEnv
    _Discrete, _Box, _MultiDiscrete = _spaces.Discrete, _spaces.Box, _spaces.MultiDiscrete
except Exception:  # noqa: BLE001
    _gym, _VectorEnvBase = None, object

    class _Discrete:
        def __init__(self, n):
            self.n, self.shape, self.dtype = int(n), (), np.dtype(np.int64)

        def __repr__(self):
            return f"Discrete({self.n})"

    class _MultiDiscrete:
        def __init__(self, nvec):
            self.nvec = np.asarray(nvec, dtype=np.int64)
            self.shape, self.dtype = self.nvec.shape, np.dtype(np.int64)

        def __repr__(self):
            return f"MultiDiscrete({self.nvec.tolist()})"

    class _Box:
        def __init__(self, low, high, shape, dtype=np.float32):
            self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), np.dtype(dtype)

        def __repr__(self):
            return f"Box({self.low}, {self.high}, {self.shape}, {self.dtype})"


class _SparseFlags:
    """Host side of the sparse flag wire (include/gte_b200.h, result block): `terminated` / `truncated` as persistent
    bool arrays that are PATCHED from the list of envs whose episode ended in the iteration (a few thousand entries)
    instead of being copied densely every step (2 bytes per env over PCIe).  Falls back to the dense bytes — which
    gte_step_host then fetched in the same call — when more episodes ended at once than the list holds."""

    def __init__(self, n, host_block):
        toff, uoff, eoff, _ = _cabi.host_result_layout(n)
        cap = _cabi.host_result_ended_cap(n)
        self.n_ended = host_block[eoff + 8:eoff + 12].view(np.uint32)
        self.entries = host_block[eoff + 32:eoff + 32 + 4 * cap].view(np.uint32)
        self.dense_term = host_block[toff:toff + n].view(np.bool_)
        self.dense_trunc = host_block[uoff:uoff + n].view(np.bool_)
        self.terminated, self.truncated = np.zeros(n, np.bool_), np.zeros(n, np.bool_)
        self.prev = np.zeros(0, np.int64)                 # env indices set by the previous update (None: unknown -> clear all)

    def update(self):
        if self.prev is None:
            self.terminated.fill(False); self.truncated.fill(False)
        elif self.prev.size:
            self.terminated[self.prev] = False; self.truncated[self.prev] = False
        n = int(self.n_ended[0])
        if n > self.entries.size:                          # a burst of episode ends: the dense bytes were fetched as well
            self.terminated[:] = self.dense_term; self.truncated[:] = self.dense_trunc
            self.prev = None
        else:
            e = self.entries[:n]
            idx = (e & np.uint32(0x3fffffff)).astype(np.int64)
            self.terminated[idx[(e >> np.uint32(31)) != 0]] = True
            self.truncated[idx[((e >> np.uint32(30)) & np.uint32(1)) != 0]] = True
            self.prev = idx
        return self.terminated, self.truncated


def shard_envs(total_envs: int, rank: int, world_size: int):
    """Env-index range owned by `rank`: [offset, offset+count) — contiguous, sizes differ by <= 1."""
    base, rem = divmod(int(total_envs), int(world_size))
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


class LazyInfos(Mapping):
    """History's last row (environments.py:186-197 after a reset, :253-264 after a step) for every env, as a dict of
    [N] columns computed on first access after each step/reset (one `gte_info` launch; the ``data_*`` columns and
    ``date`` are looked up from the staged frames).  Same keys as the reference's info dict: ``idx, step, date,
    position_index, position, real_position, data_<every numeric non-feature column>, portfolio_valuation,
    portfolio_distribution_*, reward`` — plus ``dataset_idx`` and ``episode_metrics``.  Values are CUDA tensors, except
    ``date`` (numpy datetime64, a host-side lookup) and, in the host-output modes, ``reward``.

    As in a SAME_STEP vector env the row describes the CURRENT state: for an env whose episode just ended it is the
    row `reset()` wrote for the new episode.  ``position_index`` is what the reference records: the action of the step
    (hold or out of range -> -1, the reference's None) for envs that stepped, ``positions.index(position)`` (the first
    index holding an equal value) for envs that were just reset; after a masked `reset()` the envs outside the mask keep
    their step row — read it before overwriting the action buffer passed to `step()`.  ``reward`` is the reward the
    last `step()` returned, for every env (also where the row is a reset row, whose History reward is 0)."""

    BASE_KEYS = ["idx", "step", "position_index", "position", "real_position", "portfolio_valuation",
                 "dataset_idx", "portfolio_distribution_asset", "portfolio_distribution_fiat",
                 "portfolio_distribution_borrowed_asset", "portfolio_distribution_borrowed_fiat",
                 "portfolio_distribution_interest_asset", "portfolio_distribution_interest_fiat",
                 "reward", "episode_metrics"]
    _DIST = ["asset", "fiat", "borrowed_asset", "borrowed_fiat", "interest_asset", "interest_fiat"]

    def __init__(self, env):
        self._env = env
        self._version = -1
        self._cache = {}
        series = env._series
        cols = [c for c in series[0].info if all(c in srs.info for srs in series)]      # History's data_<column> (:131-134)
        if "close" not in cols:
            cols.append("close")                                                          # the price column always exists
        self._data_cols = cols
        self.KEYS = self.BASE_KEYS + ["data_" + c for c in cols]
        if all(srs.index is not None for srs in series):
            self.KEYS.append("date")

    def _materialise(self):
        if self._version != self._env._tick:
            self._env._launch_info()
            self._version = self._env._tick
            self._cache = {}

    def __getitem__(self, key):
        e = self._env
        if key == "reward":               # host-output modes: the step's rewards are in the pinned result block
            return e._last_reward_host if (e.output != "torch" and e._last_reward_host is not None) else e._reward
        if key == "episode_metrics":
            return e.get_metrics()
        if key not in self.KEYS:
            raise KeyError(key)
        self._materialise()
        if key in self._cache:
            return self._cache[key]
        if key.startswith("portfolio_distribution_"):
            return e._info_dist[self._DIST.index(key[len("portfolio_distribution_"):])]
        if key == "data_close":
            return e._info_t["data_close"]
        if key == "position_index":
            v = self._cache[key] = e._info_position_index()
            return v
        if key.startswith("data_"):
            col = e._info_column(key[5:])                                   # f64 [n_datasets, t_stride] on the device
            v = self._cache[key] = col[e._info_t["dataset_idx"].long(), e._info_t["idx"].long()]
            return v
        if key == "date":
            idx, ds = e._info_t["idx"].cpu().numpy(), e._info_t["dataset_idx"].cpu().numpy()
            out = np.empty(idx.shape, dtype=e._series[0].index.dtype)
            for k, srs in enumerate(e._series):
                m = ds == k
                if m.any():
                    out[m] = srs.index[idx[m]]
            self._cache[key] = out
            return out
        return e._info_t[key]

    def __iter__(self):
        return iter(self.KEYS)

    def __len__(self):
        return len(self.KEYS)


class TradingVectorEnv(_VectorEnvBase):
    """N independent reference-semantics ``TradingEnv`` instances advanced in lockstep on one B200.

    Reference parameters (same names, defaults and meaning as environments.py:79-93): ``df, positions,
    dynamic_feature_functions, reward_function, windows, trading_fees, borrow_interest_rate,
    portfolio_initial_value, initial_position, max_episode_duration, verbose, name, render_mode``.

    Extra keyword-only parameters: ``num_envs``; ``device``; ``seed`` (keys the Philox stream that
    replaces the reference's global ``np.random`` draws at reset, hazard H2); ``env_id_offset``
    (global id of env 0 when sharded over GPUs); ``done_valuation_ratio`` (0.7 = this fork's stop
    rule, environments.py:246; 0.0 = upstream "valuation <= 0"); ``reset_plan`` — int32
    ``[N, E, 3]`` of (start row, position index, dataset index) consumed by successive resets
    instead of the RNG (record-and-replay for parity tests); ``obs_variant`` in
    {"auto","generic","vec","tma"}; ``output`` "torch" (CUDA tensors, default), "numpy" (everything
    in pinned host buffers, host<->device copies inside `step`) or "hybrid" (host actions in, reward /
    terminated / truncated on the host, observations stay device-resident for the policy's forward pass:
    one blocking ``gte_step_host`` C call per step — ONE copy per direction beside the gather kernel, or,
    for small batches, no copy at all: the step kernel reads / writes the pinned host memory itself;
    ``host_io`` = "auto" | "copy" | "mapped" | "server" picks the mechanism — "server" (windows=None, batches up to
    256 x SMs envs) keeps a kernel RESIDENT that answers each `step()` through mapped host memory, with no kernel
    launch or driver call per step: the lowest step latency for a host policy; any other call on the env (reset,
    infos, rollout ...) or 2 ms without a step make it leave, and the next step launches it again); ``autoreset`` (True = in-place); ``cuda_graph``
    (capture one lockstep iteration and replay it: removes the launch overhead at small N; actions
    are then read from the env's own buffer); ``n_chunks`` (0 = the library's choice: ONE fused launch per
    iteration — every CTA advances its own envs, then gathers their windows — while the batch fits a single wave
    (~100k envs), else two plain launches; 1 = always two plain launches; k > 1 cuts the envs into k ranges and
    runs the step kernel of range c+1 beside the gather of range c on a side stream — measured: no gain on B200,
    kept as an option);
    ``debug_outputs`` (also write the terminal step's idx/step/real_position/portfolio, +48 B/env);
    ``final_obs`` (gymnasium's SAME_STEP ``final_obs``: ``env.final_obs`` keeps, for every env whose episode
    ended in this step, the observation ``step()`` itself returned before the in-place reset
    (environments.py:272); costs a second gather, off by default); ``strict_actions`` (False: every negative
    action means "hold", the reference's ``position_index=None``; True: only -1 does, any other negative index raises
    IndexError — the reference's ``positions[-k]`` would silently index from the end of the list).

    ``sparse_flags`` (None = automatic: on from 2^18 envs): in the "hybrid" mode with the copy engines, `terminated` /
    `truncated` cross PCIe as the list of envs whose episode ended (a few thousand entries) and are patched into
    persistent bool arrays on the host — 8.1 instead of 10 bytes per env-step, lossless; a burst of more than N/32
    simultaneous episode ends falls back to the dense bytes inside the same call.

    ``reward_wire`` ("f64" = default, lossless; "f32" = opt-in, LOSSY): in the "hybrid" mode with the copy engines the
    rewards cross PCIe rounded to float32 (numpy's cast of the fp64 reward, round-to-nearest-even) — what a trainer that
    keeps float32 rewards anyway (stable-baselines3's buffers) would do on the host; with the sparse flags 5.1 instead of
    9.1 bytes per env-step come back.  ``step()`` then returns a float32 reward array; the fp64 rewards stay on the
    device (``env.reward_device``).

    Host actions (``output`` "numpy" / "hybrid") may be int8 / int16 / int32 / int64: they cross PCIe in that width
    (``Discrete(P)`` fits int8 for every supported P, which is what :meth:`pinned_actions` hands out by default) and
    are widened by the step kernel's own load — lossless, 8x fewer host-to-device bytes than gymnasium's int64.

    ``reward_function`` must be :func:`basic_reward_function` or a :class:`DeviceReward` from the fused
    catalogue (log / simple return with scale and clip), and ``dynamic_feature_functions`` a list of up to five
    :class:`DeviceFeature` columns, each kind at most once, in any order (``position``, ``real_position`` — also
    spelled :func:`dynamic_feature_last_position_taken` / :func:`dynamic_feature_real_position` —
    ``portfolio_return``, ``reward``, ``episode_progress``, and the stateful ``current_drawdown`` and
    ``position_age``, which keep per-env state in the episode accumulators; see ``dynamic_features.py``):
    arbitrary Python callbacks over a History cannot run inside the kernel and there is deliberately no CPU fallback
    (NotImplementedError).

    Returned tensors are persistent buffers overwritten by the next call: copy what you keep.
    """

    metadata = {"render_modes": ["logs"]}

    def __init__(self, df, positions=[0, 1], dynamic_feature_functions=_DEFAULT_DYNAMIC,
                 reward_function=basic_reward_function, windows=None, trading_fees=0,
                 borrow_interest_rate=0, portfolio_initial_value=1000, initial_position="random",
                 max_episode_duration="max", verbose=1, name="Stock", render_mode="logs", *,
                 num_envs=1, device=None, seed=0, env_id_offset=0, done_valuation_ratio=0.7,
                 reset_plan=None, obs_variant="auto", output="torch", autoreset=True,
                 debug_outputs=False, cuda_graph=False, n_chunks=0, final_obs=False, strict_actions=False,
                 host_io="auto", sparse_flags=None, reward_wire="f64", _multi_dataset=False,
                 _episodes_between_dataset_switch=1):
        self._lib = _cabi.load()                      # fails loudly when the CUDA library is missing
        if not torch.cuda.is_available():
            raise RuntimeError("gym_trading_env_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")

        # --- reference constructor checks (environments.py:94-110) ---
        self.max_episode_duration = max_episode_duration
        self.name, self.verbose = name, verbose
        self.positions = list(positions)
        self.windows = windows
        self.trading_fees = trading_fees
        self.borrow_interest_rate = borrow_interest_rate
        self.portfolio_initial_value = float(portfolio_initial_value)
        self.initial_position = initial_position
        assert self.initial_position in self.positions or self.initial_position == "random", \
            "The 'initial_position' parameter must be 'random' or a position mentionned in the 'position' (default is [0, 1]) parameter."
        assert render_mode is None or render_mode in self.metadata["render_modes"]
        self.render_mode = render_mode
        if isinstance(reward_function, DeviceReward):
            self._reward_spec = reward_function
        elif reward_function is basic_reward_function or _fn_name(reward_function) == "basic_reward_function":
            self._reward_spec = DeviceReward()
        else:
            raise NotImplementedError(
                "reward_function must be basic_reward_function (log-return, environments.py:17-18) or a "
                "DeviceReward (log_return_reward / simple_return_reward with scale and clip): arbitrary Python "
                "callbacks over a History cannot run inside the CUDA step kernel and there is no CPU fallback")
        self.reward_function = reward_function
        dyn = list(dynamic_feature_functions)
        self._n_dyn, self._dyn_kinds = parse_dynamic_features(dyn, max_episode_duration)
        self.dynamic_feature_functions = dyn
        if not (1 <= len(self.positions) <= _cabi.GTE_MAX_POSITIONS):
            raise ValueError(f"between 1 and {_cabi.GTE_MAX_POSITIONS} positions are supported")
        if windows is not None and (int(windows) != windows or windows < 1):
            raise ValueError("windows must be None or a positive int")
        if max_episode_duration != "max" and (not isinstance(max_episode_duration, (int, np.integer))
                                              or max_episode_duration < 2):
            raise ValueError("max_episode_duration must be 'max' or an int >= 2")
        if output not in ("torch", "numpy", "hybrid"):
            raise ValueError("output must be 'torch', 'numpy' or 'hybrid'")
        if obs_variant not in _cabi.OBS_VARIANTS:
            raise ValueError(f"obs_variant must be one of {list(_cabi.OBS_VARIANTS)}")

        self.num_envs = int(num_envs)
        if self.num_envs < 1:
            raise ValueError("num_envs must be >= 1")
        self.seed = int(seed)
        self.env_id_offset = int(env_id_offset)
        self.done_valuation_ratio = float(done_valuation_ratio)
        self.output = output
        if host_io not in _cabi.IO_MODES:
            raise ValueError(f"host_io must be one of {list(_cabi.IO_MODES)}")
        self.host_io = host_io
        self.strict_actions = bool(strict_actions)
        # host-output wire of the flags: None = sparse (the list of ended envs) for batches of 2^18 envs and more
        self.sparse_flags = (int(num_envs) >= (1 << 18)) if sparse_flags is None else bool(sparse_flags)
        if reward_wire not in ("f64", "f32"):
            raise ValueError("reward_wire must be 'f64' (lossless, default) or 'f32' (lossy, opt-in)")
        if reward_wire == "f32" and output != "hybrid":
            raise ValueError("reward_wire='f32' is a wire format of output='hybrid'")
        self.reward_wire = reward_wire
        self.autoreset = bool(autoreset)
        self.debug_outputs = bool(debug_outputs)
        self.cuda_graph = bool(cuda_graph)
        self.n_chunks = int(n_chunks)
        self.keep_final_obs = bool(final_obs)
        self.final_obs = None
        self._graph = None
        self._copy_in = None
        self._pin_ident = {}                 # id(array) -> (array, pointer, itemsize) of pinned action arrays seen by step()
        self._last_actions = None            # the actions of the last step (infos["position_index"]); None after a reset
        self._last_reward_host = None        # host-output modes: the reward array the last step returned
        self._async = None                   # step_async / step_wait: two wire sets + the queue of iterations in flight
        self._relay = None                   # enable_result_relay(): multi-GPU routing of result bytes through peer GPUs
        self._track_ids = None
        self._limit_price = None
        self._red_stream = None              # enable_metric_allreduce(): side stream of the per-iteration all-reduce
        self._kernel_events = None           # bench.py: list collecting (start, after step, after gather) CUDA events
        self._kernel_events_every = 1        # ... on every k-th iteration
        self._obs_variant = _cabi.OBS_VARIANTS[obs_variant]
        self._multi = bool(_multi_dataset)
        self._k_switch = int(_episodes_between_dataset_switch)
        self._tick = 0
        self._needs_first = True
        self.log_metrics = []
        self._episode_acc = None             # f64 [5 or 6, N] running state of each env's episode (add_metric, stateful
                                             # dynamic features), or None
        self._episode_record = None          # add_metric(): f64 [7, N] metrics of each env's last finished episode

        series = df if isinstance(df, (list, tuple)) else [df]
        series = [s if isinstance(s, SeriesArrays) else frame_to_arrays(s) for s in series]
        self._set_series(series)
        self._alloc_state(reset_plan)
        self._build_structs()

        F = self._n_static + self._n_dyn
        shape = (F,) if windows is None else (int(windows), F)
        self.single_observation_space = _Box(-np.inf, np.inf, shape=shape, dtype=np.float32)
        self.observation_space = _Box(-np.inf, np.inf, shape=(self.num_envs,) + shape, dtype=np.float32)
        self.single_action_space = _Discrete(len(self.positions))
        self.action_space = _MultiDiscrete([len(self.positions)] * self.num_envs)
        self.closed = False
        if _gym is not None:                    # a real gymnasium.vector.VectorEnv: say how episodes restart (SAME_STEP)
            mode = getattr(getattr(_gym.vector, "AutoresetMode", None), "SAME_STEP", None)
            if mode is not None:
                self.metadata = dict(self.metadata, autoreset_mode=mode)

    # ------------------------------------------------------------------ data staging (_set_df, :128-143)
    def _set_series(self, series):
        n_ds = len(series)
        if not (1 <= n_ds <= _cabi.GTE_MAX_DATASETS):
            raise ValueError(f"between 1 and {_cabi.GTE_MAX_DATASETS} datasets are supported")
        ns = series[0].features.shape[1]
        for s in series:
            if s.features.shape[1] != ns:
                raise ValueError("every dataset must have the same number of feature columns")
        self._n_static = ns
        if ns + self._n_dyn == 0:
            raise ValueError("no feature column (name containing 'feature') and no dynamic feature")
        self._series = series
        self._feature_names = list(series[0].feature_names) + [f"dynamic_feature__{i}" for i in range(self._n_dyn)]
        lengths = np.array([s.length for s in series], dtype=np.int32)
        W0 = 0 if self.windows is None else int(self.windows) - 1
        for T in lengths:
            if self.max_episode_duration != "max":
                if int(T) - int(self.max_episode_duration) - W0 <= W0:     # np.random.randint(low, high) needs low < high (:174)
                    raise ValueError(f"dataset of {T} rows is too short for windows={self.windows}, "
                                     f"max_episode_duration={self.max_episode_duration}")
            elif int(T) < W0 + 2:
                raise ValueError(f"dataset of {T} rows is too short for windows={self.windows}")
        t_stride = int(lengths.max())
        self._t_stride, self._lengths_np, self._n_ds = t_stride, lengths, n_ds
        feats = np.zeros((n_ds, t_stride, ns), dtype=np.float32)
        price = np.ones((n_ds, t_stride), dtype=np.float64)
        for k, s in enumerate(series):
            feats[k, :s.length] = s.features
            price[k, :s.length] = s.price
        dev = self.device
        self._features = torch.from_numpy(feats).to(dev)
        self._price = torch.from_numpy(price).to(dev)
        self._lengths = torch.from_numpy(lengths).to(dev)
        self._build_window_tables(feats)

    def _build_window_tables(self, feats):
        """16-byte-aligned copies of the reference's own `_obs_array` layout [t, F] (dynamic columns
        zero, environments.py:135-141), one per alignment class a window start can fall in."""
        self._window_tables = [None] * 4
        self._window_ptrs = [0] * 4
        self._window_ds_stride = 0
        if self.windows is None:
            return
        F = self._n_static + self._n_dyn
        row_bytes = 4 * F
        if (int(self.windows) * row_bytes) % 16 != 0:
            return
        tables, shifts, ds_stride = build_window_tables(feats, self._n_dyn)
        for c, host in tables.items():
            t = torch.from_numpy(host).to(self.device)
            assert t.data_ptr() % 16 == 0
            self._window_tables[c] = t
            self._window_ptrs[c] = t.data_ptr() + shifts[c]
        self._window_ds_stride = ds_stride

    # ------------------------------------------------------------------ device state
    def _alloc_state(self, reset_plan):
        N, dev = self.num_envs, self.device
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)   # noqa: E731
        i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)     # noqa: E731
        W = 1 if self.windows is None else int(self.windows)
        F = self._n_static + self._n_dyn
        self._asset, self._fiat, self._interest_asset, self._interest_fiat = f64(N), f64(N), f64(N), f64(N)
        self._pos_idx, self._step, self._ep_start, self._dataset_idx = i32(N), i32(N), i32(N), i32(N)
        self._plan_cursor, self._ds_episodes = i32(N), i32(N)
        self._ds_used = torch.zeros(N, dtype=torch.int64, device=dev)
        # dynamic-feature ring: one GTE_RING_TILE_BYTES_DYN block per tile of 32 envs, slots indexed by the
        # device-resident iteration clock (layout: include/gte_b200.h)
        # (unused without dynamic columns: then sized as for the default pair, the shape state_dict() has always had)
        tile = _cabi.ring_tile_bytes(W, self._n_dyn or 2, self._dyn_kinds)
        self._dyn_ring = torch.zeros((N + 31) // 32, tile, dtype=torch.uint8, device=dev)
        # stateful dynamic features keep their running state in the episode accumulators: only the rows they touch
        # (row GTE_ACC_POSITION_AGE only with position_age), so that a later add_metric() reuses the same buffer
        stateful = stateful_kinds_of(self._n_dyn, self._dyn_kinds)
        if stateful:
            rows = _cabi.GTE_ACC_POSITION_AGE + ("position_age" in stateful)
            self._episode_acc = f64(rows, N)
        self._ring_clock = torch.zeros(1, dtype=torch.int64, device=dev)
        self._error_flag = i32(1)
        self._tick_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self._reset_plan = None
        if reset_plan is not None:
            plan = torch.as_tensor(np.ascontiguousarray(reset_plan), dtype=torch.int32)
            if plan.dim() != 3 or plan.shape[0] != N or plan.shape[2] != 3:
                raise ValueError("reset_plan must be int32 [num_envs, E, 3]")
            self._reset_plan = plan.to(dev).contiguous()
        obs_shape = (N, F) if self.windows is None else (N, W, F)
        self._obs = torch.zeros(obs_shape, dtype=torch.float32, device=dev)
        # reward | terminated | truncated | error flag live in ONE block (GTE_HOST_RESULT_* layout): what a host policy
        # needs back from an iteration leaves the device with a single copy
        toff, uoff, eoff, nbytes = _cabi.host_result_layout(N)
        self._result_block = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        self._reward = self._result_block[:8 * N].view(torch.float64)
        self._terminated = self._result_block[toff:toff + N]
        self._truncated = self._result_block[uoff:uoff + N]
        self._error_out = self._result_block[eoff:eoff + 4].view(torch.int32)
        self._valuation, self._real_position = f64(N), f64(N)
        self._info_idx, self._info_step = i32(N), i32(N)
        self._pre_reset_portfolio = f64(4, N)
        self._metric_partials = f64(_cabi.GTE_MAX_PARTIAL_ROWS, _cabi.GTE_N_METRICS)
        self._metrics_step, self._metrics_total = f64(_cabi.GTE_N_METRICS), f64(_cabi.GTE_N_METRICS)
        self._block_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self._actions_dev = torch.zeros(N, dtype=torch.int64, device=dev)
        self._actions_raw = self._actions_dev.view(torch.uint8)          # the same bytes, for narrow host actions
        # lazily computed info columns
        self._info_t = {"idx": i32(N), "step": i32(N), "position_index": i32(N), "dataset_idx": i32(N),
                        "position": f64(N), "real_position": f64(N), "portfolio_valuation": f64(N),
                        "data_close": f64(N)}
        self._info_dist = f64(6, N)
        self._host = None
        self.infos = LazyInfos(self)

    def _build_structs(self):
        p = _cabi.GteParams()
        p.n_envs, p.n_positions = self.num_envs, len(self.positions)
        p.windows = 0 if self.windows is None else int(self.windows)
        p.n_static, p.n_dyn, p.dyn_kinds = self._n_static, self._n_dyn, self._dyn_kinds
        p.max_episode_duration = -1 if self.max_episode_duration == "max" else int(self.max_episode_duration)
        p.n_datasets = self._n_ds
        p.initial_position_idx = -1 if self.initial_position == "random" else self.positions.index(self.initial_position)
        p.episodes_between_switch = self._k_switch
        p.plan_episodes = 0 if self._reset_plan is None else int(self._reset_plan.shape[1])
        p.multi_dataset = int(self._multi)
        p.t_stride, p.env_id_offset, p.seed = self._t_stride, self.env_id_offset, self.seed & (2**64 - 1)
        p.fee, p.rate = float(self.trading_fees), float(self.borrow_interest_rate)
        p.v0, p.done_ratio = self.portfolio_initial_value, self.done_valuation_ratio
        p.reward_kind = DeviceReward.KINDS[self._reward_spec.kind]
        p.reward_scale, p.reward_lo, p.reward_hi = self._reward_spec.scale, self._reward_spec.lo, self._reward_spec.hi
        p.strict_actions = int(self.strict_actions)
        for i, x in enumerate(self.positions):
            p.positions[i] = float(x)
        d = _cabi.GteData()
        d.features = self._features.data_ptr() if self._n_static else None
        d.price, d.lengths = self._price.data_ptr(), self._lengths.data_ptr()
        for c in range(4):
            d.window_table[c] = self._window_ptrs[c] or None
        d.window_table_ds_stride = self._window_ds_stride
        s = _cabi.GteState()
        s.asset, s.fiat = self._asset.data_ptr(), self._fiat.data_ptr()
        s.interest_asset, s.interest_fiat = self._interest_asset.data_ptr(), self._interest_fiat.data_ptr()
        s.pos_idx, s.step, s.ep_start = self._pos_idx.data_ptr(), self._step.data_ptr(), self._ep_start.data_ptr()
        s.dataset_idx = self._dataset_idx.data_ptr()
        s.dyn_ring, s.ring_clock = self._dyn_ring.data_ptr(), self._ring_clock.data_ptr()
        s.plan_cursor, s.ds_used, s.ds_episodes = self._plan_cursor.data_ptr(), self._ds_used.data_ptr(), self._ds_episodes.data_ptr()
        s.reset_plan = None if self._reset_plan is None else self._reset_plan.data_ptr()
        s.error_flag = self._error_flag.data_ptr()
        s.tick = self._tick_dev.data_ptr()
        s.episode_acc = None if self._episode_acc is None else self._episode_acc.data_ptr()
        o = _cabi.GteStepOut()
        o.reward, o.terminated, o.truncated = self._reward.data_ptr(), self._terminated.data_ptr(), self._truncated.data_ptr()
        o.valuation = self._valuation.data_ptr()
        if self.debug_outputs:          # terminal-step info columns, only materialised for tests / final_info
            o.real_position = self._real_position.data_ptr()
            o.info_idx, o.info_step = self._info_idx.data_ptr(), self._info_step.data_ptr()
            o.pre_reset_portfolio = self._pre_reset_portfolio.data_ptr()
        o.metric_partials, o.metrics_step = self._metric_partials.data_ptr(), self._metrics_step.data_ptr()
        o.metrics_total, o.block_counter = self._metrics_total.data_ptr(), self._block_counter.data_ptr()
        o.error_out = self._error_out.data_ptr()
        i = _cabi.GteInfo()
        t = self._info_t
        i.idx, i.step, i.position_index, i.dataset_idx = (t["idx"].data_ptr(), t["step"].data_ptr(),
                                                          t["position_index"].data_ptr(), t["dataset_idx"].data_ptr())
        i.position, i.real_position = t["position"].data_ptr(), t["real_position"].data_ptr()
        i.portfolio_valuation, i.data_close = t["portfolio_valuation"].data_ptr(), t["data_close"].data_ptr()
        i.distribution = self._info_dist.data_ptr()
        self._P, self._D, self._S, self._O, self._I = p, d, s, o, i
        self._resolved_variant = self._lib.gte_obs_variant_for(C.byref(p), C.byref(d))
        # arguments of the per-step call that never change, built once (the Python side of a step is what bounds
        # small batches: ~20 us per call before this, a ~10 us kernel behind it)
        self._fast_args = (C.byref(p), C.byref(d), C.byref(s), C.byref(o), C.c_void_p(self._obs.data_ptr()))
        self._term_b, self._trunc_b = self._terminated.view(torch.bool), self._truncated.view(torch.bool)
        self._n_shape = torch.Size((self.num_envs,))
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _launch_reset(self, mask_ptr, first):
        self._tick += 1
        _cabi.check(self._lib.gte_reset(C.byref(self._P), C.byref(self._D), C.byref(self._S), mask_ptr,
                                        int(first), self._stream()), "gte_reset")

    def _launch_obs(self, variant=None):
        v = self._obs_variant if variant is None else variant
        _cabi.check(self._lib.gte_gather_obs(C.byref(self._P), C.byref(self._D), C.byref(self._S),
                                             C.c_void_p(self._obs.data_ptr()), v, self._stream()), "gte_gather_obs")

    def _launch_info(self):
        _cabi.check(self._lib.gte_info(C.byref(self._P), C.byref(self._D), C.byref(self._S), C.byref(self._I),
                                       self._stream()), "gte_info")

    def _launch_step(self, actions_ptr, autoreset=None):
        ar = self.autoreset if autoreset is None else autoreset
        self._tick += 1
        _cabi.check(self._lib.gte_step(C.byref(self._P), C.byref(self._D), C.byref(self._S), actions_ptr,
                                       C.byref(self._O), int(ar), self._stream()), "gte_step")

    def _launch_step_obs(self, actions_ptr, n_chunks=None):
        """One lockstep iteration in one C call: step kernel(s) + gather kernel(s), chunk-pipelined."""
        self._tick += 1
        _cabi.check(self._lib.gte_step_obs(C.byref(self._P), C.byref(self._D), C.byref(self._S), actions_ptr,
                                           C.byref(self._O), C.c_void_p(self._obs.data_ptr()), int(self.autoreset),
                                           self._obs_variant, self.n_chunks if n_chunks is None else n_chunks,
                                           self._stream()), "gte_step_obs")

    def _capture_graph(self):
        """Capture one lockstep iteration (actions read from self._actions_dev) into a CUDA graph.
        Kernel arguments are all pointers/constants; the Philox tick lives on the device."""
        g = torch.cuda.CUDAGraph()
        cap = torch.cuda.Stream(device=self.device)
        cap.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.graph(g, stream=cap):
            self._launch_step_obs(C.c_void_p(self._actions_dev.data_ptr()))
        self._tick -= 1                       # the capture itself executed nothing
        torch.cuda.current_stream(self.device).wait_stream(cap)
        self._graph = g

    def _host_buffers(self):
        """Pinned host side of the "numpy" / "hybrid" modes: ONE result block (reward | terminated | truncated | error
        flag, the layout of the device block) and one action staging buffer per wire dtype."""
        if self._host is None:
            N = self.num_envs
            toff, uoff, eoff, nbytes = _cabi.host_result_layout(N)
            blk = torch.zeros(nbytes, dtype=torch.uint8, pin_memory=True)
            r = blk.numpy()
            self._host = {"results": blk, "reward": r[:8 * N].view(np.float64),
                          "terminated": r[toff:toff + N].view(np.bool_), "truncated": r[uoff:uoff + N].view(np.bool_),
                          "error": r[eoff:eoff + 4].view(np.int32), "actions": {}, "pinned": {}}
            if self.output == "numpy":
                self._host["obs_t"] = torch.empty(self._obs.shape, dtype=self._obs.dtype, pin_memory=True)
                self._host["obs"] = self._host["obs_t"].numpy()
            self._copy_in = torch.cuda.Stream(device=self.device)
            io = _cabi.GteHostIO()
            io.results, io.dev_results = blk.data_ptr(), self._result_block.data_ptr()
            io.dev_actions, io.mode = self._actions_raw.data_ptr(), _cabi.IO_MODES[self.host_io]
            # large batches (copy engines): the flags come back as the list of envs whose episode ended, 8.1 instead of
            # 10 bytes per env over PCIe, and are patched into persistent bool arrays on the host
            self._host["sparse"] = _SparseFlags(N, r) if (self.sparse_flags and self.output == "hybrid") else None
            io.sparse_flags = int(self._host["sparse"] is not None)
            if self.reward_wire == "f32":                    # opt-in lossy wire: float32 rewards, 4 bytes per env
                self._host["reward_f32_t"] = torch.zeros(N, dtype=torch.float32, pin_memory=True)
                self._host["reward_f32"] = self._host["reward_f32_t"].numpy()
                self._host["reward_f32_dev"] = torch.zeros(N, dtype=torch.float32, device=self.device)
                io.reward_f32_host = self._host["reward_f32_t"].data_ptr()
                io.dev_reward_f32 = self._host["reward_f32_dev"].data_ptr()
            if self.output == "numpy":                       # the observation batch is delivered to the host as well
                io.obs_host, io.obs_bytes = self._host["obs_t"].data_ptr(), self._obs.numel() * 4
            self._io, self._io_mode_used = io, C.c_int(0)
            self._io_ref, self._io_mode_ref = C.byref(io), C.byref(self._io_mode_used)
            # recorded by gte_step_host right behind the step kernel: lets the metric all-reduce run beside the gather
            self._step_done = torch.cuda.Event()
            self._step_done.record(torch.cuda.current_stream(self.device))
        return self._host

    @staticmethod
    def _is_pinned(hb, a):
        """Whether a numpy array lives in pinned (page-locked) memory — asked of the driver once per buffer.  A positive
        answer is cached TOGETHER WITH a reference to the array, so the buffer cannot be freed (and its address handed
        to pageable memory) while the cache says "pinned"; a negative answer is never cached."""
        ent = hb["pinned"].get(a.ctypes.data)
        if ent is not None:
            return True
        if a.flags.writeable and torch.from_numpy(a).is_pinned():
            if len(hb["pinned"]) < 64:
                hb["pinned"][a.ctypes.data] = a
            return True
        return False

    def _stage_host_actions(self, actions):
        """numpy / list actions -> (array in PINNED memory, its dtype one of int8/16/32/64).  Arrays handed out by
        :meth:`pinned_actions` (or any other pinned array) are used in place; everything else goes through one
        staging copy into a pinned buffer of the same width (other integer dtypes: widened to int64)."""
        hb = self._host_buffers()
        a = np.asarray(actions)
        if a.shape != (self.num_envs,):
            raise ValueError(f"actions must have shape ({self.num_envs},), got {a.shape}")
        if a.dtype in _WIRE_ACTION_DTYPES and a.flags.c_contiguous:
            if self._is_pinned(hb, a):
                return a
        dt = a.dtype if a.dtype in _WIRE_ACTION_DTYPES else np.dtype(np.int64)
        buf = hb["actions"].get(dt)
        if buf is None:
            t = torch.empty(self.num_envs, dtype=torch.from_numpy(np.empty(0, dt)).dtype, pin_memory=True)
            buf = hb["actions"][dt] = t.numpy()
            hb["actions"][("t", dt)] = t                      # keeps the pinned allocation alive
        buf[...] = a
        return buf

    # ------------------------------------------------------------------ gymnasium vector API
    def reset(self, seed=None, options=None):
        """Reset every env (environments.py:163-199); ``options={"mask": bool[N]}`` resets a subset.
        ``seed`` re-keys the Philox stream (the reference ignores gymnasium's seed, hazard H2)."""
        with torch.cuda.device(self.device):
            if seed is not None:
                self.seed = int(seed)
                self._P.seed = self.seed & (2**64 - 1)
                self._graph = None        # captured kernel nodes hold GteParams (and with it the old seed) by value
            if self._needs_first:                                  # MultiDatasetTradingEnv.__init__ draw (:378)
                self._launch_reset(None, first=True)
                self._needs_first = False
            mask_ptr, keep = None, None
            if options is not None and options.get("mask") is not None:
                keep = torch.as_tensor(options["mask"]).to(self.device).to(torch.uint8).contiguous()
                if keep.shape != (self.num_envs,):
                    raise ValueError("options['mask'] must have shape [num_envs]")
                mask_ptr = C.c_void_p(keep.data_ptr())
            self._launch_reset(mask_ptr, first=False)
            self._launch_obs()
            if keep is None:
                self._last_actions = None
            elif self._last_actions is not None:
                # the envs outside the mask keep their last step row; the reset envs read step == 0 (the reset row)
                la = self._last_actions
                self._last_actions = la.copy() if isinstance(la, np.ndarray) else la.clone()
            if self._track_ids is not None:
                self._track_append(after_reset=True, mask=keep)
            return self._emit_obs(), self.infos

    def step(self, actions):
        """One lockstep iteration (environments.py:233-272) with in-place auto-reset."""
        if (type(actions) is torch.Tensor and self.output == "torch" and actions.dtype is torch.int64 and actions.is_cuda
                and actions.shape == self._n_shape and actions.device == self.device and actions.is_contiguous()
                and self._track_ids is None and not self.keep_final_obs and not self.cuda_graph
                and self._red_stream is None and self._kernel_events is None
                and torch.cuda.current_device() == self._dev_index):
            # the common on-device loop: one C call, nothing else
            a = self._fast_args
            self._tick += 1
            self._last_actions = actions
            rc = self._lib.gte_step_obs(a[0], a[1], a[2], actions.data_ptr(), a[3], a[4], self.autoreset,
                                        self._obs_variant, self.n_chunks,
                                        torch.cuda.current_stream(self.device).cuda_stream)
            if rc:
                _cabi.check(rc, "gte_step_obs")
            return self._obs, self._reward, self._term_b, self._trunc_b, self.infos
        host_in = not (isinstance(actions, torch.Tensor) and actions.is_cuda)
        if (host_in and self.output != "torch" and self._track_ids is None and not self.keep_final_obs
                and not self.cuda_graph and self._kernel_events is None and self.autoreset):
            if self._relay is not None:
                if self._async is not None and self._async["pending"]:
                    raise RuntimeError("step() while step_async() iterations are in flight: call step_wait() first")
                self.step_async(actions)
                return self.step_wait()
            return self._step_host(actions)
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream(self.device)
            if host_in:
                src = self._stage_host_actions(actions)
                # H2D on its own stream, in the array's own width (the step kernel widens while loading).  Out-of-range
                # actions are flagged by the kernel (positions[position_index] would raise, :234) and the flag rides
                # back with the results in the host-output modes.
                self._copy_in.wait_stream(main)              # the last step kernel may still be reading the buffer
                nb = src.dtype.itemsize
                with torch.cuda.stream(self._copy_in):
                    self._actions_raw[:nb * self.num_envs].copy_(torch.from_numpy(src.view(np.uint8)), non_blocking=True)
                main.wait_stream(self._copy_in)
                act, act_bytes = self._actions_dev, nb
            else:
                act, act_bytes = actions, 8
                if act.dtype != torch.int64 or not act.is_contiguous() or act.shape != (self.num_envs,) \
                        or act.device != self.device:
                    act = act.to(device=self.device, dtype=torch.int64).contiguous().view(self.num_envs)
            if self._track_ids is not None or (self.cuda_graph and act_bytes != 8):
                if act_bytes != 8:               # the History log / the captured graph read the actions as int64
                    nt = {1: torch.int8, 2: torch.int16, 4: torch.int32}[act_bytes]
                    wide = self._actions_raw[:act_bytes * self.num_envs].view(nt).to(torch.int64)
                    self._actions_dev.copy_(wide)
                    act, act_bytes = self._actions_dev, 8
            if self._track_ids is not None:
                # pre-step state of the tracked envs: the auto-reset overwrites the position and clears the limit orders
                lim = None if self._limit_price is None else self._limit_price[self._track_ids].clone()
                self._track_pre = (self._pos_idx[self._track_ids].clone(), self._dataset_idx[self._track_ids].clone(), lim)
            self._P.action_bytes = act_bytes
            self._last_actions = src if host_in else act
            try:
                ret = self._step_launch(act, main)
            finally:
                self._P.action_bytes = 0
            if self._track_ids is not None:
                self._track_append(after_reset=False, actions=act)
            return ret

    def _step_host(self, actions):
        """output="hybrid" / "numpy" with host actions: ONE blocking C call (gte_step_host) — host actions in, step
        kernel, reward / terminated / truncated / error flag back in one pinned block, gather enqueued; returns as soon
        as the block has landed ("numpy": and the observation batch, delivered into pinned host memory too)."""
        ent = self._pin_ident.get(id(actions))
        if ent is not None and ent[0] is actions:            # a pinned array seen before (kept alive by the cache)
            ptr, nb = ent[1], ent[2]
            self._last_actions = actions
        else:
            a = self._stage_host_actions(actions)
            ptr, nb = a.ctypes.data, a.dtype.itemsize
            if a is actions and len(self._pin_ident) < 64:
                self._pin_ident[id(actions)] = (actions, ptr, nb)
            self._last_actions = a
        hb, red = self._host, self._red_stream
        if hb is None:
            hb = self._host_buffers()
        io = self._io
        if red is not None and self._red_snapshot is not None:
            torch.cuda.current_stream(self.device).wait_event(self._red_snapshot)   # metrics_step is about to be overwritten
        io.actions = ptr
        if red is not None:
            io.step_done_event = self._step_done.cuda_event
        self._P.action_bytes = nb
        self._tick += 1
        f = self._fast_args
        try:
            if torch.cuda.current_device() == self._dev_index:
                rc = self._lib.gte_step_host(f[0], f[1], f[2], self._io_ref, f[3], f[4], 1, self._obs_variant,
                                             self._io_mode_ref, torch.cuda.current_stream(self.device).cuda_stream)
            else:
                with torch.cuda.device(self.device):
                    rc = self._lib.gte_step_host(f[0], f[1], f[2], self._io_ref, f[3], f[4], 1, self._obs_variant,
                                                 self._io_mode_ref, torch.cuda.current_stream(self.device).cuda_stream)
        finally:
            self._P.action_bytes = 0
        if rc:
            _cabi.check(rc, "gte_step_host")
        if red is not None:
            self._issue_metric_allreduce(None, after=self._step_done)
        reward = hb["reward"]
        if self.reward_wire == "f32":
            reward = hb["reward_f32"]
            if self._io_mode_used.value != _cabi.IO_COPY:    # small batches answer through mapped memory in fp64: same dtype out
                np.copyto(reward, hb["reward"], casting="same_kind")
        self._last_reward_host = reward
        if hb["error"][0]:
            self._raise_on_flag(int(hb["error"][0]))
        term, trunc = hb["terminated"], hb["truncated"]
        if hb["sparse"] is not None and self._io_mode_used.value == _cabi.IO_COPY:
            term, trunc = hb["sparse"].update()
        return (hb["obs"] if self.output == "numpy" else self._obs), reward, term, trunc, self.infos

    # ------------------------------------------------------------------ step_async / step_wait (host policy, pipelined)
    def _async_sets(self):
        """Two independent wire sets (pinned result block, device result block, device + pinned action staging, one
        GteHostIO each) for step_async / step_wait."""
        if self._async is None:
            N, dev = self.num_envs, self.device
            toff, uoff, eoff, nbytes = _cabi.host_result_layout(N)
            sets = []
            for k_set in range(2):
                host = self._relay.host_block(k_set) if self._relay is not None else None
                if host is None:
                    host = torch.zeros(nbytes, dtype=torch.uint8, pin_memory=True)
                devb = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
                dact = torch.zeros(N * 8, dtype=torch.uint8, device=dev)
                r = host.numpy()
                io = _cabi.GteHostIO()
                io.results, io.dev_results, io.dev_actions = host.data_ptr(), devb.data_ptr(), dact.data_ptr()
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                io.sparse_flags = int(self.sparse_flags)
                if self._relay is not None:
                    io.reward_host_count = self._relay.own_count
                r32 = r32d = None
                if self.reward_wire == "f32":
                    r32 = torch.zeros(N, dtype=torch.float32, pin_memory=True)
                    r32d = torch.zeros(N, dtype=torch.float32, device=dev)
                    io.reward_f32_host, io.dev_reward_f32 = r32.data_ptr(), r32d.data_ptr()
                sets.append({"io": io, "r32": (r32, r32d), "io_ref": C.byref(io), "host": host, "dev": devb, "dact": dact, "event": ev,
                             "sparse": _SparseFlags(N, r) if self.sparse_flags else None,
                             "stage": {}, "reward": r[:8 * N].view(np.float64) if r32 is None else r32.numpy(),
                             "terminated": r[toff:toff + N].view(np.bool_), "truncated": r[uoff:uoff + N].view(np.bool_),
                             "error": r[eoff:eoff + 4].view(np.int32)})
            self._async = {"sets": sets, "pending": [], "n": 0}
        return self._async

    def enable_result_relay(self, group=None, plan=None, verbose=False, calibrate_rounds=2):
        """COLLECTIVE (every rank of the ``torch.distributed`` job, or of ``group``): balance the device-to-host result
        bytes of a multi-GPU host-policy job over the GPUs' PCIe links in proportion to the bandwidth each link gets while
        all ranks copy (measured here in ``calibrate_rounds`` short rounds: the even load, then the planned split; 2 suits a
        caller that steps one iteration at a time, 4 one that keeps two in flight with step_async).  A rank on a slow link then ships
        the tail of its fp64 rewards over NVLink to a peer GPU whose copy engine writes them into this rank's (shared,
        pinned) result block — lossless, no kernel, no NCCL call per step (``relay.py``, ``gte_relay_*``).  Afterwards
        every ``step()`` / ``step_async()`` is a collective too: all ranks must make the same calls in the same order.
        ``plan`` = {sender rank: (peer rank, envs)} overrides the measurement (also: ``GTE_RELAY_FORCE``).  Returns the
        plan and the measured bandwidths; an empty plan (links within 20 % of each other) changes nothing."""
        from .relay import ResultRelay
        if self.output != "hybrid" or self.reward_wire != "f64" or not self.autoreset:
            raise ValueError("the result relay serves output='hybrid' with the lossless fp64 reward wire and autoreset")
        if self._async is not None and self._async["pending"]:
            raise RuntimeError("step_async() iterations are in flight: call step_wait() first")
        if self._relay is not None:
            self._relay.close()
        self._async = None                                 # wire sets are rebuilt (a sender's result blocks move to shared memory)
        with torch.cuda.device(self.device):
            self._relay = ResultRelay(self, group=group, plan=plan, verbose=verbose, calibrate_rounds=calibrate_rounds)
        desc = self._relay.describe()
        if not self._relay.plan:                           # nothing to balance (or the set-up failed somewhere): the plain path
            self._relay.close()
            self._relay = None
        return desc

    def result_relay_state(self):
        """The relay's current plan, the measurements behind it and the adjustments the running job has made (or None)."""
        return self._relay.describe() if self._relay is not None else None

    def step_async(self, actions):
        """Enqueue one lockstep iteration for host actions and return at once (`output="hybrid"`): the action copy, the
        transition, the copy of the result block and the gather are all in flight when this returns; :meth:`step_wait`
        hands out the results.  Up to TWO iterations may be in flight — ``step_async(a[k+1])`` before ``step_wait()`` of
        iteration k — so that the device-to-host copy of iteration k runs under iteration k+1 (what a caller that does
        not need iteration k's rewards to choose iteration k+1's actions wants: scripted or replayed actions, a policy
        that reads the device-resident observations).  A pinned ``actions`` array is read in place: do not overwrite it
        before the matching ``step_wait()``."""
        if self.output != "hybrid" or self._track_ids is not None or self.keep_final_obs or self.cuda_graph or not self.autoreset:
            raise ValueError("step_async() needs output='hybrid' with autoreset, without tracking / final_obs / CUDA graphs")
        st = self._async_sets()
        if len(st["pending"]) >= 2:
            raise RuntimeError("two iterations are already in flight: call step_wait() first")
        k = st["n"] & 1
        ws = st["sets"][k]
        if self._relay is not None and (self._relay.count & 1) != k:
            raise RuntimeError("result relay: wire sets out of step with the relay's iteration count")
        self._host_buffers()
        a = np.asarray(actions)
        if a.shape != (self.num_envs,):
            raise ValueError(f"actions must have shape ({self.num_envs},), got {a.shape}")
        pinned = False
        if a.dtype in _WIRE_ACTION_DTYPES and a.flags.c_contiguous:
            pinned = self._is_pinned(self._host, a)
        if not pinned:                                   # this set's own staging buffer: free since its last step_wait()
            dt = a.dtype if a.dtype in _WIRE_ACTION_DTYPES else np.dtype(np.int64)
            buf = ws["stage"].get(dt)
            if buf is None:
                t = torch.empty(self.num_envs, dtype=torch.from_numpy(np.empty(0, dt)).dtype, pin_memory=True)
                buf = ws["stage"][dt] = t.numpy()
                ws["stage"][("t", dt)] = t
            buf[...] = a
            a = buf
        io = ws["io"]
        io.actions = a.ctypes.data
        red, relay = self._red_stream, self._relay
        if relay is not None:
            io.reward_host_count = relay.own_count        # (the running job may have moved the split)
            relay.before_begin()                          # this rank's share of its senders' iteration, enqueued first
        if red is not None:
            if self._red_snapshot is not None:
                torch.cuda.current_stream(self.device).wait_event(self._red_snapshot)
        if red is not None or relay is not None:
            io.step_done_event = ws["event"].cuda_event
        self._P.action_bytes = a.dtype.itemsize
        self._tick += 1
        self._last_actions = a
        f = self._fast_args
        try:
            with torch.cuda.device(self.device):
                rc = self._lib.gte_step_host_begin(f[0], f[1], f[2], ws["io_ref"], f[3], f[4], 1, self._obs_variant,
                                                   torch.cuda.current_stream(self.device).cuda_stream)
        finally:
            self._P.action_bytes = 0
        if rc:
            _cabi.check(rc, "gte_step_host_begin")
        if relay is not None:
            relay.after_begin(k, ws["dev"].data_ptr(), ws["event"].cuda_event)
        if red is not None:
            self._issue_metric_allreduce(None, after=ws["event"])
        st["pending"].append(k)
        st["n"] += 1

    def step_wait(self):
        """Results of the OLDEST iteration enqueued by :meth:`step_async`: ``(obs, reward, terminated, truncated,
        infos)`` — numpy views of that iteration's pinned result block (valid until the second ``step_async`` from
        now); ``obs`` is the device-resident observation tensor, which the newest enqueued iteration writes."""
        st = self._async
        if st is None or not st["pending"]:
            raise RuntimeError("step_wait() without a pending step_async()")
        k = st["pending"].pop(0)
        ws = st["sets"][k]
        with torch.cuda.device(self.device):
            rc = self._lib.gte_step_host_end(ws["io_ref"])
        if rc:
            _cabi.check(rc, "gte_step_host_end")
        if self._relay is not None:
            self._relay.wait(k)                           # the tail of the rewards comes through a peer GPU's link
        self._last_reward_host = ws["reward"]
        if ws["error"][0]:
            self._raise_on_flag(int(ws["error"][0]))
        term, trunc = ws["sparse"].update() if ws["sparse"] is not None else (ws["terminated"], ws["truncated"])
        return self._obs, ws["reward"], term, trunc, self.infos

    def _step_launch(self, act, main):
        if self._red_stream is not None and self._red_snapshot is not None:
            main.wait_event(self._red_snapshot)             # metrics_step is about to be overwritten
        if self.keep_final_obs and self.autoreset:
            # step without the in-kernel reset, gather the terminal observations, keep those of the ended envs,
            # then reset exactly those envs and gather again (what a SAME_STEP vector env returns)
            if self.final_obs is None:
                self.final_obs = torch.zeros_like(self._obs)
            self._launch_step(C.c_void_p(act.data_ptr()), autoreset=False)
            self._launch_obs()
            ended = (self._terminated | self._truncated)
            shape = (self.num_envs,) + (1,) * (self._obs.dim() - 1)
            torch.where(ended.view(shape).bool(), self._obs, self.final_obs, out=self.final_obs)
            self._launch_reset(C.c_void_p(ended.data_ptr()), first=False)
            self._tick -= 1                                 # one public call = one info version
            self._launch_obs()
        elif self.cuda_graph:
            if act.data_ptr() != self._actions_dev.data_ptr():
                self._actions_dev.copy_(act, non_blocking=True)
            if self._graph is None:
                self._capture_graph()
            self._tick += 1
            self._graph.replay()
        elif self.windows is not None and (self._red_stream is not None or self.output == "hybrid") and not (
                self._kernel_events is not None and self._tick % self._kernel_events_every == 0):
            # the all-reduce (and, in the hybrid mode, the result copy) is issued between the two kernels so that it
            # overlaps the gather
            self._launch_step(C.c_void_p(act.data_ptr()))
            self._issue_metric_allreduce(main)
            if self.output == "hybrid":
                return self._results_to_host(main, before_gather=True)
            self._launch_obs()
        elif self._kernel_events is not None and self.windows is not None and self._tick % self._kernel_events_every == 0:
            # (bench.py, every k-th iteration) the same two kernels as gte_step_obs, issued as two calls so that
            # CUDA events can bracket each of them without perturbing the other iterations
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
            self._launch_step(C.c_void_p(act.data_ptr()))
            ev[1].record()
            self._issue_metric_allreduce(main)
            self._launch_obs()
            ev[2].record()
            self._kernel_events.append(ev)
        else:
            self._launch_step_obs(C.c_void_p(act.data_ptr()))
            self._issue_metric_allreduce(main)
        if self.output in ("numpy", "hybrid"):
            return self._results_to_host(main, before_gather=False)
        return self._obs, self._reward, self._terminated.view(torch.bool), self._truncated.view(torch.bool), self.infos

    def _results_to_host(self, main, before_gather):
        """The general host-output path (device actions, tracking, final_obs, CUDA graphs ...): ONE device-to-host copy
        of the result block (+ the observation batch in the "numpy" mode), then the error flag is checked."""
        hb = self._host_buffers()
        if before_gather:                                   # hybrid: the block leaves beside the gather kernel
            self._copy_in.wait_stream(main)
            with torch.cuda.stream(self._copy_in):
                hb["results"].copy_(self._result_block, non_blocking=True)
            self._launch_obs()
            self._copy_in.synchronize()
        else:
            hb["results"].copy_(self._result_block, non_blocking=True)
            if self.output == "numpy":
                hb["obs_t"].copy_(self._obs, non_blocking=True)
            main.synchronize()
        self._last_reward_host = hb["reward"]
        if hb["error"][0]:
            self._raise_on_flag(int(hb["error"][0]))
        obs = hb["obs"] if self.output == "numpy" else self._obs
        return obs, hb["reward"], hb["terminated"], hb["truncated"], self.infos

    def _emit_obs(self):
        if self.output == "numpy":
            h = self._host_buffers()
            h["obs_t"].copy_(self._obs, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            return h["obs"]
        return self._obs

    def close(self, **kwargs):
        self.close_extras(**kwargs)
        self.closed = True

    def close_extras(self, **kwargs):
        if getattr(self, "_async", None) is not None:
            while self._async["pending"]:                 # let the iterations in flight land before the buffers go
                self._lib.gte_step_host_end(self._async["sets"][self._async["pending"].pop(0)]["io_ref"])
            self._async = None
        if getattr(self, "_relay", None) is not None:    # collective, like enable_result_relay()
            self._relay.close()
            self._relay = None
        if getattr(self, "host_io", None) == "server" and getattr(self, "_lib", None) is not None:
            self._lib.gte_serve_stop()           # the resident server kernel, if it is still waiting for requests
        self._host = None
        self._pin_ident = {}
        self._graph = None

    def add_limit_order(self, position, limit, persistent=False, env_ids=None):
        """``TradingEnv.add_limit_order(position, limit, persistent)`` (environments.py:227-231) for every env, or
        for ``env_ids``: at each following step, after the index has advanced, an env whose position differs from
        ``position`` and whose bar contains the price (``low <= limit <= high``) rebalances to ``position`` AT THE
        LIMIT PRICE (:217-223).  ``limit`` is a scalar or one value per selected env.  Orders are tried in the order
        in which their positions first received one (the reference iterates its dict in insertion order) and are
        cleared by reset() and by the in-kernel auto-reset, like ``self._limit_orders = {}`` (:168) — re-add them
        for the envs whose episode ended.  Only ``persistent=True`` is supported: the reference's non-persistent
        branch deletes from the dict it is iterating and raises RuntimeError as soon as such an order executes."""
        if not persistent:
            raise NotImplementedError(
                "persistent=False is not supported: in the reference a non-persistent order raises RuntimeError "
                "('dictionary changed size during iteration', environments.py:220-223) when it executes")
        if position not in self.positions:
            raise ValueError("position must be one of `positions`")
        if any("high" not in srs.info or "low" not in srs.info for srs in self._series):
            raise ValueError("limit orders need 'high' and 'low' columns in every dataset (environments.py:221)")
        N, P, dev = self.num_envs, len(self.positions), self.device
        if self._limit_price is None:
            hi = np.ones((self._n_ds, self._t_stride), dtype=np.float64)
            lo = np.ones((self._n_ds, self._t_stride), dtype=np.float64)
            for k, srs in enumerate(self._series):
                hi[k, :srs.length], lo[k, :srs.length] = srs.info["high"], srs.info["low"]
            self._high, self._low = torch.from_numpy(hi).to(dev), torch.from_numpy(lo).to(dev)
            self._limit_price = torch.full((N, P), float("nan"), dtype=torch.float64, device=dev)
            self._limit_seq_host = []
            self._limit_seq = torch.zeros(P, dtype=torch.int32, device=dev)
            self._D.high, self._D.low = self._high.data_ptr(), self._low.data_ptr()
            self._S.limit_price, self._S.limit_seq = self._limit_price.data_ptr(), self._limit_seq.data_ptr()
            self._graph = None                                   # kernel arguments changed: re-capture
        pk = self.positions.index(position)
        if pk not in self._limit_seq_host:
            self._limit_seq_host.append(pk)
            self._limit_seq[:len(self._limit_seq_host)] = torch.tensor(self._limit_seq_host, dtype=torch.int32, device=dev)
            self._P.n_limit_positions = len(self._limit_seq_host)
            self._graph = None
        lim = torch.as_tensor(limit, dtype=torch.float64, device=dev)
        if env_ids is None:
            self._limit_price[:, pk] = lim
        else:
            ids = torch.as_tensor(np.asarray(env_ids), dtype=torch.int64, device=dev)
            self._limit_price[ids, pk] = lim

    def rollout(self, actions, keep_obs=False):
        """Advance K lockstep iterations from a device tensor of actions ``[K, N]`` (int64) without touching the
        host between them; returns dict of device tensors ``reward [K, N]`` (f64), ``terminated`` / ``truncated``
        ``[K, N]`` (bool), ``valuation [K, N]`` (terminal-step valuation) and, with ``keep_obs``, ``obs [K, N, ...]``.
        The open-loop driver for pre-computed action streams (replay, random-policy baselines, benchmarks)."""
        if not (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dim() == 2
                and actions.shape[1] == self.num_envs):
            raise ValueError("rollout() needs a CUDA int64 tensor of shape [K, num_envs]")
        actions = actions.to(torch.int64).contiguous()
        K, N, dev = actions.shape[0], self.num_envs, self.device
        out = {"reward": torch.empty(K, N, dtype=torch.float64, device=dev),
               "terminated": torch.empty(K, N, dtype=torch.bool, device=dev),
               "truncated": torch.empty(K, N, dtype=torch.bool, device=dev),
               "valuation": torch.empty(K, N, dtype=torch.float64, device=dev)}
        if keep_obs:
            out["obs"] = torch.empty((K,) + tuple(self._obs.shape), dtype=torch.float32, device=dev)
        if self._track_ids is None and not self.keep_final_obs and self._red_stream is None and self.autoreset:
            # one C call enqueues all K iterations (gte_rollout); the observation windows are only gathered for the
            # iterations whose observation is kept
            term8 = torch.empty(K, N, dtype=torch.uint8, device=dev)
            trunc8 = torch.empty(K, N, dtype=torch.uint8, device=dev)
            o = _cabi.GteStepOut()
            C.memmove(C.byref(o), C.byref(self._O), C.sizeof(o))
            o.reward, o.terminated, o.truncated = out["reward"].data_ptr(), term8.data_ptr(), trunc8.data_ptr()
            o.valuation = out["valuation"].data_ptr()
            o.real_position = o.info_idx = o.info_step = o.pre_reset_portfolio = None
            obs_buf = out["obs"] if keep_obs else self._obs
            self._tick += K
            self._last_actions = actions[-1]
            _cabi.check(self._lib.gte_rollout(C.byref(self._P), C.byref(self._D), C.byref(self._S),
                                              C.c_void_p(actions.data_ptr()), K, C.byref(o),
                                              C.c_void_p(obs_buf.data_ptr()), int(keep_obs), 1,
                                              self._obs_variant or 0, self._stream()), "gte_rollout")
            out["terminated"], out["truncated"] = term8.view(torch.bool), trunc8.view(torch.bool)
            # the persistent one-iteration outputs keep meaning "the last iteration"
            self._reward.copy_(out["reward"][-1]); self._valuation.copy_(out["valuation"][-1])
            self._terminated.copy_(term8[-1]); self._truncated.copy_(trunc8[-1])
            if keep_obs:
                self._obs.copy_(out["obs"][-1])
            return out
        saved, self.output = self.output, "torch"
        try:
            for k in range(K):
                obs, rew, term, trunc, _ = self.step(actions[k])
                out["reward"][k].copy_(rew)
                out["terminated"][k].copy_(term)
                out["truncated"][k].copy_(trunc)
                out["valuation"][k].copy_(self._valuation)
                if keep_obs:
                    out["obs"][k].copy_(obs)
        finally:
            self.output = saved
        return out

    # ------------------------------------------------------------------ History of tracked envs (utils/history.py)
    def track(self, env_indices, max_steps=100_000):
        """Keep a device-side per-step log — the reference's ``History`` rows (environments.py:186-197,
        253-264) — for a FEW selected envs (rendering / debugging; needs ``debug_outputs=True``).
        Rows are appended on the device after every reset()/step() with no host synchronisation."""
        if not self.debug_outputs:
            raise ValueError("track() needs debug_outputs=True (the terminal-step info columns)")
        ids = torch.as_tensor(list(env_indices), dtype=torch.int64, device=self.device)
        if ids.numel() == 0 or int(ids.min()) < 0 or int(ids.max()) >= self.num_envs:
            raise ValueError("env_indices out of range")
        self._track_ids = ids
        self._track_log = torch.zeros(int(max_steps), ids.numel(), len(self._TRACK_COLS), dtype=torch.float64,
                                      device=self.device)
        self._track_len = 0

    _TRACK_COLS = ["idx", "step", "position_index", "position", "real_position", "portfolio_valuation",
                   "portfolio_distribution_asset", "portfolio_distribution_fiat",
                   "portfolio_distribution_borrowed_asset", "portfolio_distribution_borrowed_fiat",
                   "portfolio_distribution_interest_asset", "portfolio_distribution_interest_fiat",
                   "reward", "terminated", "truncated", "dataset_idx", "new_episode",
                   # state after the in-place auto-reset (used to rebuild the reset() row of the next episode)
                   "_post_idx", "_post_pos_idx", "_post_asset", "_post_fiat", "_post_ds",
                   # 0 where a masked reset() left the env alone: no History row
                   "_present"]

    def _first_position_index(self, pidx):
        """``positions.index(positions[pidx])``: the FIRST index holding an equal value (environments.py:189) — what the
        reference records in a reset row when ``positions`` lists a value twice (e.g. 0.0 and -0.0)."""
        if getattr(self, "_pos_first", None) is None:
            first = [self.positions.index(p) for p in self.positions]
            self._pos_first = torch.tensor(first, dtype=torch.int32, device=self.device)
        return self._pos_first[pidx.long()]

    def _track_append(self, after_reset, actions=None, mask=None):
        if self._track_ids is None or self._track_len >= self._track_log.shape[0]:
            return
        i = self._track_ids
        z = torch.zeros(i.numel(), dtype=torch.float64, device=self.device)
        pos_tab = torch.tensor(self.positions, dtype=torch.float64, device=self.device)
        dist = lambda a, f: [torch.where(a > 0, a, z), torch.where(f > 0, f, z),         # noqa: E731  max(0, x)
                             torch.where(-a > 0, -a, z), torch.where(-f > 0, -f, z)]      # (portfolio.py:49-57)
        if after_reset:       # the row reset() writes (environments.py:186-197)
            pidx = self._pos_idx[i].long()
            pos = pos_tab[pidx]
            a, f = self._asset[i], self._fiat[i]
            present = z + 1 if mask is None else mask[i].double()
            cols = [(self._ep_start[i] + self._step[i]).double(), self._step[i].double(),
                    self._first_position_index(pidx).double(), pos, pos,
                    torch.full_like(z, self.portfolio_initial_value), *dist(a, f),
                    self._interest_asset[i], self._interest_fiat[i],
                    z, z, z, self._dataset_idx[i].double(), z + 1, z, z, z, z, z, present]
        else:                 # the row step() adds (:253-264): terminal values where the episode ended
            pf = self._pre_reset_portfolio[:, i]
            a, f = pf[0], pf[1]
            a_i = actions[i]
            pre_pos, pre_ds, pre_lim = self._track_pre
            # the position after the step, before any auto-reset, replayed from the pre-step state with the step
            # kernel's comparisons (no arithmetic): an action outside [0, len(positions)) is a hold (:234)
            valid = (a_i >= 0) & (a_i < len(self.positions))
            target = torch.where(valid, a_i, torch.zeros_like(a_i))
            cur = pre_pos.long()
            cur = torch.where(valid & (pos_tab[target] != pos_tab[cur]), target, cur)          # :213-215
            if pre_lim is not None and self._limit_seq_host:                                    # :217-223
                row = self._info_idx[i].long()
                hi, lo = self._high[pre_ds.long(), row], self._low[pre_ds.long(), row]
                for pk in self._limit_seq_host:
                    lim = pre_lim[:, pk]
                    hit = (lim == lim) & (pos_tab[pk] != pos_tab[cur]) & (lim <= hi) & (lim >= lo)
                    cur = torch.where(hit, torch.full_like(cur, pk), cur)
            cols = [self._info_idx[i].double(), self._info_step[i].double(),
                    torch.where(valid, a_i, torch.full_like(a_i, -1)).double(), pos_tab[cur], self._real_position[i],
                    self._valuation[i], *dist(a, f), pf[2], pf[3],
                    self._reward[i], self._terminated[i].double(), self._truncated[i].double(),
                    pre_ds.double(), z,
                    (self._ep_start[i] + self._step[i]).double(), self._pos_idx[i].double(), self._asset[i], self._fiat[i],
                    self._dataset_idx[i].double(), z + 1]
        self._track_log[self._track_len] = torch.stack(cols, dim=1)
        self._track_len += 1

    def tracked_history(self, which=0):
        """The log of tracked env number `which` as a pandas DataFrame with the reference's History
        column names (+ terminated / truncated / new_episode / date / data_close when known)."""
        import pandas as pd
        if self._track_ids is None:
            raise ValueError("no env is tracked: call track([...]) first")
        rows = self._track_log[:self._track_len, which].cpu().numpy()
        cols = self._TRACK_COLS
        c = {n: k for k, n in enumerate(cols)}
        out = []
        for r in rows:
            if not r[c["_present"]]:
                continue
            out.append(r)
            if not r[c["new_episode"]] and (r[c["terminated"]] or r[c["truncated"]]) and self.autoreset:
                # the row reset() writes for the episode the auto-reset started (environments.py:186-197)
                n = np.zeros(len(cols))
                pos = self.positions[int(r[c["_post_pos_idx"]])]
                a, f = r[c["_post_asset"]], r[c["_post_fiat"]]
                n[c["idx"]], n[c["position_index"]] = r[c["_post_idx"]], self.positions.index(pos)
                n[c["position"]] = n[c["real_position"]] = float(pos)
                n[c["portfolio_valuation"]] = self.portfolio_initial_value
                # Python's max(0, x) (portfolio.py:49-57): the first argument wins a tie, so -0.0 reads +0.0
                n[c["portfolio_distribution_asset"]], n[c["portfolio_distribution_fiat"]] = max(0.0, a), max(0.0, f)
                n[c["portfolio_distribution_borrowed_asset"]], n[c["portfolio_distribution_borrowed_fiat"]] = max(0.0, -a), max(0.0, -f)
                n[c["dataset_idx"]], n[c["new_episode"]], n[c["_present"]] = r[c["_post_ds"]], 1.0, 1.0
                out.append(n)
        df = pd.DataFrame(np.array(out).reshape(-1, len(cols)), columns=cols)
        df = df[[n for n in cols if not n.startswith("_")]]
        for c in ("idx", "step", "position_index", "dataset_idx"):
            df[c] = df[c].astype(np.int64)
        for c in ("terminated", "truncated", "new_episode"):
            df[c] = df[c].astype(bool)
        ds, idx = df["dataset_idx"].to_numpy(), df["idx"].to_numpy()
        df["data_close"] = np.array([self._series[d].price[i] for d, i in zip(ds, idx)])
        if all(s.index is not None for s in self._series):
            df["date"] = np.array([self._series[d].index[i] for d, i in zip(ds, idx)])
        return df

    def save_for_render(self, dir="render_logs", which=0, episode=-1):
        """``TradingEnv.save_for_render`` (environments.py:296-307) for tracked env number `which`: the History rows of
        one episode joined with the market frame on the date index, pickled to ``{dir}/{name}_{timestamp}.pkl`` — the
        file the reference's ``Renderer`` (renderer.py:51-58) loads.  `episode` indexes the FINISHED episodes of the
        log (-1 = the latest; the reference object only ever holds its current episode), falling back to the running
        episode when none has finished.  Returns the path."""
        import datetime
        import pandas as pd
        h = self.tracked_history(which)
        starts = list(np.flatnonzero(h["new_episode"].to_numpy())) + [len(h)]
        episodes = [(a, b) for a, b in zip(starts[:-1], starts[1:])]
        finished = [(a, b) for a, b in episodes if bool(h["terminated"].iloc[b - 1] or h["truncated"].iloc[b - 1])]
        a, b = finished[episode] if finished else episodes[-1]
        ep = h.iloc[a:b]
        srs = self._series[int(ep["dataset_idx"].iloc[0])]
        assert all(c in srs.info for c in ("open", "high", "low", "close")), \
            "Your DataFrame needs to contain columns : open, high, low, close to render !"        # :297
        if srs.index is None:
            raise ValueError("save_for_render needs a DatetimeIndex (History's 'date' column, environments.py:188)")
        market = pd.DataFrame({**{n: srs.features[:, j] for j, n in enumerate(srs.feature_names)}, **srs.info},
                              index=pd.DatetimeIndex(srs.index, name="date"))
        idx = ep["idx"].to_numpy()
        hist = ep.drop(columns=["terminated", "truncated", "new_episode", "dataset_idx", "data_close"])
        for c, col in srs.info.items():                                          # History's data_<info column> (:131-134)
            hist["data_" + c] = col[idx]
        hist = hist.set_index("date").sort_index()
        render_df = market.join(hist, how="inner")                               # :304
        os.makedirs(dir, exist_ok=True)
        path = f"{dir}/{self.name}_{datetime.datetime.now().strftime('%Y-%m-%d_%H-%M-%S')}.pkl"
        render_df.to_pickle(path)
        return path

    def _info_column(self, name):
        """A numeric non-feature column of the staged frames (History's ``data_<name>``) as f64 [n_datasets, t_stride] on
        the device, uploaded on first use."""
        cols = self.__dict__.setdefault("_info_cols_dev", {})
        if name not in cols:
            host = np.ones((self._n_ds, self._t_stride), dtype=np.float64)
            for k, srs in enumerate(self._series):
                host[k, :srs.length] = srs.price if name == "close" and name not in srs.info else srs.info[name]
            cols[name] = torch.from_numpy(host).to(self.device)
        return cols[name]

    def _info_position_index(self):
        """``position_index`` as the reference records it: the step's action (hold = None -> -1) for envs that stepped
        (:257), ``positions.index(position)`` on the row reset() writes (:189)."""
        state = self._info_t["position_index"]
        if len(set(self.positions)) < len(self.positions):      # a value listed twice: the first index holding it
            state = self._first_position_index(state)
        la = self._last_actions
        if la is None:
            return state
        if isinstance(la, np.ndarray):
            act = torch.from_numpy(np.ascontiguousarray(la)).to(self.device)
        else:
            act = la
        act = act.to(torch.int64)
        act = torch.where((act >= 0) & (act < len(self.positions)), act, torch.full_like(act, -1)).to(torch.int32)
        return torch.where(self._info_t["step"] > 0, act, state)

    # ------------------------------------------------------------------ metrics / errors / state
    def add_metric(self, name, function):
        """``TradingEnv.add_metric(name, function)`` (environments.py:274-276): record ``function`` over every env's
        episode.  ``function`` must be a :class:`DeviceMetric` from the device catalogue (``episode_metrics.py``:
        position_changes, episode_length, max_drawdown, episode_reward, time_in_market), accumulated in the step kernel
        and recorded bit for bit at each episode's end; anything else raises NotImplementedError.  Call it before the
        first ``reset()``, as the reference's usage does: the accumulators must run from an episode's reset row.  A
        repeated name: the later function wins, as in the reference's metric dict."""
        if not self._needs_first:
            raise RuntimeError("add_metric() after reset(): episode metrics must be added before the first reset(), "
                               "so that their accumulators run from every episode's reset row")
        _em.check_metric_function(function)
        self.log_metrics.append({"name": name, "function": function})
        kinds = _em.metric_kinds_of(self.log_metrics)
        N, f64 = self.num_envs, dict(dtype=torch.float64, device=self.device)
        if self._episode_record is None:
            self._episode_record = torch.full((_cabi.GTE_EPISODE_RECORD_ROWS, N), float("nan"), **f64)
            self._O.episode_record = self._episode_record.data_ptr()
        if kinds & _cabi.GTE_METRIC_KINDS_STATEFUL and self._episode_acc is None:
            # rows 0..4: row GTE_ACC_POSITION_AGE is only read by the position_age dynamic feature
            self._episode_acc = torch.zeros(_cabi.GTE_ACC_POSITION_AGE, N, **f64)
            self._S.episode_acc = self._episode_acc.data_ptr()
        self._P.metric_kinds = kinds
        self._graph = None                                   # kernel arguments changed: re-capture

    def get_episode_metrics(self, env_index=None):
        """The metrics of each env's most recently finished episode (``add_metric``).  ``env_index=None``: a dict
        name -> f64 [N] CUDA tensor ("Market Return", "Portfolio Return" as fractions, then each added name), NaN
        for an env that has not finished an episode yet; the tensors are views of a buffer that later steps overwrite.
        ``env_index=i``: the reference's ``get_metrics()`` dict of env i (environments.py:285-294) — the two returns
        as its ``f"{100*x:5.2f}%"`` strings, the added metrics as Python numbers; raises if env i has not finished an
        episode.  The record is kept across ``reset()``, as the reference keeps ``results_metrics``."""
        if self._episode_record is None:
            raise RuntimeError("no episode metric is configured: call add_metric(name, DeviceMetric) before reset()")
        with torch.cuda.device(self.device):
            self._lib.gte_serve_stop()                   # a resident server kernel owns the state while it runs
        rows = _em.record_names(self.log_metrics)
        if env_index is None:
            return {name: self._episode_record[r] for name, r in rows.items()}
        i = int(env_index)
        if not 0 <= i < self.num_envs:
            raise IndexError(f"env_index {env_index} out of range for {self.num_envs} envs")
        rec = self._episode_record[:, i].cpu().numpy()
        if np.isnan(rec[0]):
            raise RuntimeError(f"env {i} has not finished an episode yet")
        out = {}
        for name, r in rows.items():
            if r < 2:
                out[name] = f"{100 * float(rec[r]):5.2f}%"
            else:
                out[name] = int(rec[r]) if _em.KINDS[r - 2] in _em.INT_KINDS else float(rec[r])
        return out

    def get_metrics(self, total=True):
        """Numeric episode metrics (environments.py:279-283) as a name -> 0-d tensor dict."""
        t = self._metrics_total if total else self._metrics_step
        return {n: t[i] for i, n in enumerate(_cabi.METRIC_NAMES)}

    def allreduce_metrics(self, total=False, async_op=False):
        """Sum the metric vector over all ranks (NCCL over NVLink when torch.distributed is initialised).
        The only cross-GPU exchange on this path: envs never interact (SURVEY.md §8e)."""
        import torch.distributed as dist
        t = self._metrics_total if total else self._metrics_step
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist.all_reduce(t, op=dist.ReduceOp.SUM, async_op=async_op)
        return None

    def enable_metric_allreduce(self):
        """Sum the metric vector of EVERY lockstep iteration over all ranks (SURVEY.md §8e: the path's only
        collective, 8 doubles over NCCL / NVLink) into ``global_metrics_step`` / ``global_metrics_total``.  The
        exchange rides a side stream: right after the step kernel the 64 bytes are snapshotted by the copy engine,
        the all-reduce then runs beside the window gather (or beside the next step kernel once an SM has room),
        and the next iteration only waits for the snapshot — never for the collective."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("enable_metric_allreduce() needs an initialised torch.distributed process group")
        f64 = dict(dtype=torch.float64, device=self.device)
        self._red_stream = torch.cuda.Stream(device=self.device)
        self.global_metrics_step, self.global_metrics_total = torch.zeros(8, **f64), torch.zeros(8, **f64)
        self._red_snapshot = None

    def _issue_metric_allreduce(self, main, after=None):
        if self._red_stream is None:
            return
        import torch.distributed as dist
        ev = after                                       # gte_step_host recorded it right behind the step kernel
        if ev is None:
            ev = torch.cuda.Event()
            ev.record(main)                              # the step kernel (which wrote metrics_step) is the last thing on main
        with torch.cuda.stream(self._red_stream):
            self._red_stream.wait_event(ev)
            self.global_metrics_step.copy_(self._metrics_step, non_blocking=True)     # 64 B device-to-device copy
            snap = torch.cuda.Event()
            snap.record()
            dist.all_reduce(self.global_metrics_step)
            self.global_metrics_total.add_(self.global_metrics_step)
        self._red_snapshot = snap

    def wait_metric_allreduce(self):
        """Make the current stream wait for the all-reduces issued so far (before reading ``global_metrics_*``)."""
        if self._red_stream is not None:
            torch.cuda.current_stream(self.device).wait_stream(self._red_stream)

    @property
    def error_flag(self):
        """The sticky in-kernel error bits (include/gte_b200.h ``GteErrorBit``) as a 1-element int32 CUDA tensor that
        every step refreshes — a device-resident loop can fold it into its own bookkeeping (or `.item()` it every k
        steps) instead of calling :meth:`check_errors`; the host-output modes raise by themselves."""
        return self._error_out

    def check_errors(self):
        """Synchronising check of the in-kernel error flags (device-resident actions are not validated on the host)."""
        self._raise_on_flag(int(self._error_flag.item()))

    def pinned_actions(self, dtype=None):
        """A pinned [N] numpy array to fill and pass to `step()` (no staging copy).  ``dtype`` None = the narrowest
        signed integer that holds ``Discrete(len(positions))`` — int8 for every supported position list: one byte per
        env over PCIe instead of gymnasium's eight, widened losslessly by the step kernel; int16 / int32 / int64 on request."""
        dt = np.dtype(np.int8 if dtype is None else dtype)
        if dt not in _WIRE_ACTION_DTYPES:
            raise ValueError("pinned_actions: dtype must be int8, int16, int32 or int64")
        t = torch.empty(self.num_envs, dtype=torch.from_numpy(np.empty(0, dt)).dtype, pin_memory=True)
        a = t.numpy()
        hb = self._host_buffers()
        hb["pinned"][a.ctypes.data] = a
        hb["actions"][("handed", a.ctypes.data)] = t          # keeps the allocation alive as long as the env
        return a

    def _raise_on_flag(self, flag):
        """Raise for the sticky in-kernel error bits (include/gte_b200.h GteErrorBit) and clear them."""
        self._error_flag.zero_()
        if flag & _cabi.E_ACTION_RANGE:
            raise IndexError("an action >= len(positions) was passed to step() (treated as hold)")
        if flag & _cabi.E_NEGATIVE_ACTION:
            raise IndexError("a negative action other than -1 was passed to step() (strict_actions=True; treated as hold)")
        if flag & _cabi.E_PAST_END:
            raise IndexError("an env was stepped past the end of its data without a reset")
        if flag & _cabi.E_PLAN_RANGE:
            raise ValueError("reset_plan holds a row outside the dataset / position list (clamped)")
        if flag & _cabi.E_PLAN_EXHAUSTED:
            raise RuntimeError("reset_plan exhausted: more episodes were started than the plan holds (it wrapped around)")

    def state_dict(self):
        """Env state as tensors (checkpoint/resume: SURVEY.md §5)."""
        names = ["asset", "fiat", "interest_asset", "interest_fiat", "pos_idx", "step", "ep_start", "dataset_idx",
                 "dyn_ring", "ring_clock", "plan_cursor", "ds_used", "ds_episodes",
                 "metrics_total", "tick_dev"]
        # episode metrics (add_metric) and stateful dynamic features: the accumulators and the record, only when configured
        names += [n for n in ("episode_acc", "episode_record") if getattr(self, "_" + n) is not None]
        return {n: getattr(self, "_" + n).clone() for n in names}

    def load_state_dict(self, d):
        for n, v in d.items():
            getattr(self, "_" + n).copy_(v)
        self._tick += 1                    # invalidates the lazily computed infos
        self._needs_first = False

    @property
    def reward_device(self):
        """The fp64 rewards of the last `step()` as a device tensor (kept exact whatever `reward_wire` says)."""
        return self._reward

    @property
    def idx(self):
        return self._ep_start + self._step

    @property
    def chunks(self):
        """Env ranges one `step()` is pipelined over (step kernel of range c+1 beside gather of range c)."""
        return self.n_chunks if self.n_chunks > 0 else int(self._lib.gte_default_chunks(self.num_envs))

    @property
    def launches_per_step(self):
        """Kernel launches one `step()` of the on-device loop issues: 1 (windows=None, or transition + gather fused
        into one launch for batches that fit a single wave, no episode metric and no stateful dynamic feature), else 2
        per env range."""
        return int(self._lib.gte_step_obs_launches(C.byref(self._P), C.byref(self._D), self._obs_variant, self.n_chunks))

    @property
    def obs_variant(self):
        v = self._obs_variant or self._resolved_variant
        return {v_: k for k, v_ in _cabi.OBS_VARIANTS.items()}[v]


class MultiDatasetTradingVectorEnv(TradingVectorEnv):
    """Batched ``MultiDatasetTradingEnv`` (environments.py:309-400): every dataset matched by
    ``dataset_dir`` is loaded, preprocessed and kept device-resident; each env carries its own dataset
    index and least-used rotation state (`next_dataset`, :380-391) and switches every
    ``episodes_between_dataset_switch`` episodes inside the in-kernel auto-reset.

    ``dataset_dir`` is a glob like the reference's (``"data/*.pkl"``); ``.csv`` / ``.parquet`` files are accepted too.
    The datasets may have different lengths (each keeps its own T) and their columns in different orders: feature
    columns are matched by name against the first dataset, non-numeric columns are ignored, and a dataset whose feature
    set differs is refused by name (``reconcile_series``).  ``datasets=[DataFrame | SeriesArrays, ...]`` may be given
    instead of ``dataset_dir``.
    """

    def __init__(self, dataset_dir=None, *args, preprocess=lambda df: df, episodes_between_dataset_switch=1,
                 datasets=None, **kwargs):
        self.dataset_dir = dataset_dir
        self.preprocess = preprocess
        self.episodes_between_dataset_switch = int(episodes_between_dataset_switch)
        if self.episodes_between_dataset_switch < 1:
            raise ValueError("episodes_between_dataset_switch must be >= 1")
        if datasets is None:
            self.dataset_pathes = sorted(_glob.glob(self.dataset_dir))
            if len(self.dataset_pathes) == 0:
                raise FileNotFoundError(f"No dataset found with the path : {self.dataset_dir}")   # :376
            # :391 read_pickle -> preprocess; .csv / .parquet files are read the way the reference's examples do
            frames = [self.preprocess(load_frame(p)) for p in self.dataset_pathes]
            self.dataset_names = [Path(p).name for p in self.dataset_pathes]
        else:
            frames = [d if isinstance(d, SeriesArrays) else self.preprocess(d) for d in datasets]
            self.dataset_names = [f"dataset_{k}" for k in range(len(frames))]
        # ragged lengths are fine (per-dataset T); feature columns are matched by NAME across the datasets
        datasets = reconcile_series([d if isinstance(d, SeriesArrays) else frame_to_arrays(d) for d in frames],
                                    self.dataset_names)
        super().__init__(list(datasets), *args, _multi_dataset=True,
                         _episodes_between_dataset_switch=self.episodes_between_dataset_switch, **kwargs)
