"""B200-native batched implementation of Gym-Trading-Env's per-step simulation hot path.

Scope (SURVEY.md §8): `TradingEnv.step` + `Portfolio` math + log-return reward + done/truncated
flags + windowed `_get_obs` + in-place auto-reset, for N independent envs in lockstep, as
hand-written sm_100a CUDA kernels behind a C-ABI library (`include/gte_b200.h`).

    import gym_trading_env_b200 as gte
    env = gte.TradingVectorEnv(df, positions=[-1, 0, 1], windows=64, num_envs=65536, ...)
    obs, infos = env.reset()
    obs, reward, terminated, truncated, infos = env.step(actions)     # CUDA tensors
"""
from .data import (SeriesArrays, build_window_tables, frame_to_arrays, load_frame, make_gbm_arrays,  # noqa: F401
                   make_gbm_ohlcv, reconcile_series, window_table_classes)

__version__ = "0.1.0"

_LAZY = {"TradingVectorEnv", "MultiDatasetTradingVectorEnv", "basic_reward_function",
         "dynamic_feature_last_position_taken", "dynamic_feature_real_position", "shard_envs", "LazyInfos",
         "DeviceReward", "log_return_reward", "simple_return_reward"}
_FEATURES = {"DeviceFeature", "parse_dynamic_features", "portfolio_return_feature", "reward_feature",
             "episode_progress_feature", "current_drawdown_feature", "position_age_feature"}
_METRICS = {"DeviceMetric", "position_changes_metric", "episode_length_metric", "max_drawdown_metric",
            "episode_reward_metric", "time_in_market_metric"}


def __getattr__(name):          # torch / the CUDA library are only imported when an env class is used
    if name in _FEATURES:             # host-only: importable without torch or a device
        from . import dynamic_features
        return getattr(dynamic_features, name)
    if name in _METRICS:              # host-only as well
        from . import episode_metrics
        return getattr(episode_metrics, name)
    if name in _LAZY:
        from . import vector_env
        return getattr(vector_env, name)
    if name == "SB3VecEnv":
        from .sb3_adapter import SB3VecEnv
        return SB3VecEnv
    if name == "bind_host_to_gpu":
        from .hostbind import bind_host_to_gpu
        return bind_host_to_gpu
    if name == "build":
        from ._cabi import build
        return build
    raise AttributeError(name)


def register():
    """Register the batched envs with gymnasium (ids ``TradingEnv-B200-v0`` / ``MultiDatasetTradingEnv-B200-v0``,
    vector entry points), mirroring the reference's registration (src/gym_trading_env/__init__.py:3-14).
    Raises ImportError when gymnasium is not installed (it is not part of this image)."""
    from gymnasium.envs.registration import register as _register
    _register(id="TradingEnv-B200-v0", vector_entry_point="gym_trading_env_b200.vector_env:TradingVectorEnv",
              disable_env_checker=True, order_enforce=False)
    _register(id="MultiDatasetTradingEnv-B200-v0",
              vector_entry_point="gym_trading_env_b200.vector_env:MultiDatasetTradingVectorEnv",
              disable_env_checker=True, order_enforce=False)
