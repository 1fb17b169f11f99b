"""ctypes binding of ``libgte_b200.so`` — the only way Python reaches the GPU in this package.

The structures mirror ``include/gte_b200.h`` field for field.  There is NO fallback: if the CUDA
library is missing or fails to load, :func:`load` raises and every env constructor fails loudly.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import re
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG, "csrc")
LIB_PATH = os.path.join(_CSRC, "libgte_b200.so")
INCLUDE_DIR = os.path.join(os.path.dirname(_PKG), "include")
SOURCES = ["gte_step.cu", "gte_obs.cu", "gte_relay.cu", "gte_cabi.cu"]
HEADERS = ["gte_device.cuh", "gte_step_env.cuh", "gte_tma.cuh", "gte_launch.h", os.path.join(INCLUDE_DIR, "gte_b200.h")]

GTE_VERSION = 203                 # include/gte_b200.h GTE_VERSION this binding was written against
GTE_MAX_POSITIONS = 64
GTE_MAX_DATASETS = 64
GTE_N_METRICS = 8
GTE_STEP_THREADS = 256
GTE_MAX_PARTIAL_ROWS = 4096
GTE_MAX_DYN = 5
GTE_N_METRIC_KINDS = 5            # enum GteMetricKind: metric_kinds bit 1 << kind
GTE_METRIC_KINDS_ALL = 0x1f
GTE_METRIC_KINDS_STATEFUL = 0x1d  # every kind but episode_length keeps state in episode_acc
GTE_EPISODE_ACC_ROWS = 6
GTE_ACC_POSITION_AGE = 5          # the episode_acc row read only with position_age: [5, N] suffices without it
GTE_EPISODE_RECORD_ROWS = 7
GTE_DYN_CURRENT_DRAWDOWN, GTE_DYN_POSITION_AGE = 6, 7   # enum GteDynKind: the stateful kinds (keep state in episode_acc)


def ring_tile_bytes(windows: int, n_dyn: int, dyn_kinds: int) -> int:
    """Bytes of one 32-env tile of the dynamic-feature ring (GTE_RING_TILE_BYTES_DYN): W rows x 32 f32 values per f32
    kind, plus W rows x 32 u8 position indices when "position" (kind 1) is a column; dyn_kinds 0 = the default pair."""
    W = max(int(windows), 1)
    n_pos = sum(((dyn_kinds >> (4 * j)) & 15) == 1 for j in range(n_dyn)) if dyn_kinds else 1
    return W * (128 * (n_dyn - n_pos) + 32 * n_pos)
REWARD_LOG_RETURN, REWARD_SIMPLE_RETURN = 0, 1
OBS_AUTO, OBS_GENERIC, OBS_VEC, OBS_TMA = 0, 1, 2, 3
OBS_VARIANTS = {"auto": OBS_AUTO, "generic": OBS_GENERIC, "vec": OBS_VEC, "tma": OBS_TMA}
METRIC_NAMES = ["episodes", "terminated", "truncated", "sum_portfolio_return", "sum_market_return",
                "sum_episode_length", "sum_reward", "reserved"]


class GteParams(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("n_positions", C.c_int32), ("windows", C.c_int32),
        ("n_static", C.c_int32), ("n_dyn", C.c_int32), ("max_episode_duration", C.c_int32),
        ("n_datasets", C.c_int32), ("initial_position_idx", C.c_int32),
        ("episodes_between_switch", C.c_int32), ("plan_episodes", C.c_int32),
        ("multi_dataset", C.c_int32), ("reward_kind", C.c_int32),
        ("n_limit_positions", C.c_int32), ("action_bytes", C.c_int32),
        ("strict_actions", C.c_int32), ("dyn_kinds", C.c_int32),
        ("t_stride", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("fee", C.c_double), ("rate", C.c_double), ("v0", C.c_double), ("done_ratio", C.c_double),
        ("reward_scale", C.c_double), ("reward_lo", C.c_double), ("reward_hi", C.c_double),
        ("positions", C.c_double * GTE_MAX_POSITIONS),
        ("metric_kinds", C.c_int32), ("pad_metric", C.c_int32),
    ]


class GteData(C.Structure):
    _fields_ = [
        ("features", C.c_void_p), ("price", C.c_void_p), ("lengths", C.c_void_p),
        ("high", C.c_void_p), ("low", C.c_void_p),
        ("window_table", C.c_void_p * 4), ("window_table_ds_stride", C.c_int64),
    ]


class GteState(C.Structure):
    _fields_ = [
        ("asset", C.c_void_p), ("fiat", C.c_void_p), ("interest_asset", C.c_void_p),
        ("interest_fiat", C.c_void_p), ("pos_idx", C.c_void_p), ("step", C.c_void_p),
        ("ep_start", C.c_void_p), ("dataset_idx", C.c_void_p),
        ("dyn_ring", C.c_void_p), ("ring_clock", C.c_void_p),
        ("plan_cursor", C.c_void_p), ("ds_used", C.c_void_p), ("ds_episodes", C.c_void_p),
        ("reset_plan", C.c_void_p), ("limit_price", C.c_void_p), ("limit_seq", C.c_void_p),
        ("error_flag", C.c_void_p), ("tick", C.c_void_p), ("episode_acc", C.c_void_p),
    ]


class GteStepOut(C.Structure):
    _fields_ = [
        ("reward", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p),
        ("valuation", C.c_void_p), ("real_position", C.c_void_p), ("info_idx", C.c_void_p),
        ("info_step", C.c_void_p), ("pre_reset_portfolio", C.c_void_p),
        ("metric_partials", C.c_void_p), ("metrics_step", C.c_void_p),
        ("metrics_total", C.c_void_p), ("block_counter", C.c_void_p), ("error_out", C.c_void_p),
        ("seq_out", C.c_void_p), ("seq_value", C.c_uint32), ("ended_cap", C.c_uint32),
        ("ended_list", C.c_void_p), ("ended_counter", C.c_void_p), ("ended_n_out", C.c_void_p),
        ("reward_f32", C.c_void_p), ("episode_record", C.c_void_p),
    ]


class GteHostIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("results", C.c_void_p), ("dev_actions", C.c_void_p), ("dev_results", C.c_void_p),
        ("step_done_event", C.c_void_p), ("obs_host", C.c_void_p), ("obs_bytes", C.c_int64),
        ("reward_f32_host", C.c_void_p), ("dev_reward_f32", C.c_void_p), ("reward_host_count", C.c_int64),
        ("mode", C.c_int32), ("sparse_flags", C.c_int32),
    ]


IO_AUTO, IO_COPY, IO_MAPPED, IO_SERVER = 0, 1, 2, 3
IO_MODES = {"auto": IO_AUTO, "copy": IO_COPY, "mapped": IO_MAPPED, "server": IO_SERVER}
E_ACTION_RANGE, E_PAST_END, E_PLAN_RANGE, E_PLAN_EXHAUSTED, E_NEGATIVE_ACTION = 1, 2, 4, 8, 16


def host_result_layout(n: int):
    """(term offset, trunc offset, error offset, total bytes) of gte_step_host's result block (GTE_HOST_RESULT_*):
    reward f64[N] | header 32 B (error i32, sequence u32, n_ended u32, cap u32, counter u32, pad) | ended u32[cap] |
    terminated u8[N] | truncated u8[N]."""
    cap = host_result_ended_cap(n)
    err = n * 8
    term = err + 32 + 4 * cap
    return term, term + n, err, (term + 2 * n + 7) // 8 * 8


def host_result_ended_cap(n: int) -> int:
    return (max(n // 32, 1024) + 3) // 4 * 4


def host_result_sparse_bytes(n: int) -> int:
    """Bytes of the sparse prefix (reward | header | ended list)."""
    return n * 8 + 32 + 4 * host_result_ended_cap(n)


class GteInfo(C.Structure):
    _fields_ = [
        ("idx", C.c_void_p), ("step", C.c_void_p), ("position_index", C.c_void_p),
        ("dataset_idx", C.c_void_p), ("position", C.c_void_p), ("real_position", C.c_void_p),
        ("portfolio_valuation", C.c_void_p), ("data_close", C.c_void_p), ("distribution", C.c_void_p),
    ]


EXPORTS = ["gte_version", "gte_last_error", "gte_build_id", "gte_reset", "gte_step", "gte_gather_obs", "gte_step_obs",
           "gte_step_host", "gte_step_host_begin", "gte_step_host_end", "gte_serve_stop", "gte_relay_supported", "gte_relay_alloc", "gte_relay_open",
           "gte_relay_release", "gte_relay_push", "gte_relay_serve", "gte_relay_unblock", "gte_host_register", "gte_host_unregister", "gte_rollout", "gte_info", "gte_obs_variant_for", "gte_default_chunks", "gte_struct_size",
           "gte_step_obs_launches"]


def source_hash() -> str:
    """Hash of every CUDA source / header the library is compiled from: the build line bakes it into the binary
    (``gte_build_id()``), so a stale ``libgte_b200.so`` — mtimes mean nothing after a checkout or a copy to the GPU
    box — is recognised by content, not by date."""
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        path = f if os.path.isabs(f) else os.path.join(_CSRC, f)
        h.update(os.path.basename(path).encode() + b"\0")
        with open(path, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def nvcc_command(out_path: str = LIB_PATH):
    """The exact build line (sm_100a only; -fmad=false keeps fp64 math FMA-free, -lineinfo for ncu)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
            "-fmad=false", f'-DGTE_BUILD_ID="{source_hash()}"', "-Xcompiler", "-fPIC", "-shared", "-o", out_path] + \
           [os.path.join(_CSRC, s) for s in SOURCES]


def built_id(path: str = LIB_PATH):
    """The source hash baked into an existing library file (read from the file, not through dlopen), or None."""
    try:
        with open(path, "rb") as fh:
            m = re.search(rb"GTE_BUILD_ID=([0-9a-f]{16})", fh.read())
        return m.group(1).decode() if m else None
    except OSError:
        return None


def needs_build() -> bool:
    return built_id() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into csrc/libgte_b200.so with nvcc (cross-compiles without a GPU)."""
    if force or needs_build():
        cmd = nvcc_command()
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB_PATH


_lib = None


def load():
    """Load the CUDA library or raise — there is deliberately no CPU / PyTorch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  gym_trading_env_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.gte_version.restype = C.c_int
    lib.gte_last_error.restype = C.c_char_p
    lib.gte_build_id.restype = C.c_char_p
    if lib.gte_version() != GTE_VERSION:
        raise RuntimeError(f"{LIB_PATH} is ABI version {lib.gte_version()}, this binding expects {GTE_VERSION} — rebuild it")
    if os.path.exists(os.path.join(_CSRC, SOURCES[0])) and lib.gte_build_id().decode() != source_hash():
        raise RuntimeError(f"{LIB_PATH} was built from other sources (build id {lib.gte_build_id().decode()}, "
                           f"sources {source_hash()}) — rebuild it: python -c 'import __graft_entry__ as g; g.build()'")
    P = C.POINTER
    lib.gte_reset.argtypes = [P(GteParams), P(GteData), P(GteState), C.c_void_p, C.c_int, C.c_void_p]
    lib.gte_step.argtypes = [P(GteParams), P(GteData), P(GteState), C.c_void_p, P(GteStepOut), C.c_int, C.c_void_p]
    lib.gte_gather_obs.argtypes = [P(GteParams), P(GteData), P(GteState), C.c_void_p, C.c_int, C.c_void_p]
    lib.gte_step_obs.argtypes = [P(GteParams), P(GteData), P(GteState), C.c_void_p, P(GteStepOut), C.c_void_p,
                                 C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.gte_step_host.argtypes = [P(GteParams), P(GteData), P(GteState), P(GteHostIO), P(GteStepOut), C.c_void_p,
                                  C.c_int, C.c_int, P(C.c_int), C.c_void_p]
    lib.gte_rollout.argtypes = [P(GteParams), P(GteData), P(GteState), C.c_void_p, C.c_int, P(GteStepOut), C.c_void_p,
                                C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.gte_info.argtypes = [P(GteParams), P(GteData), P(GteState), P(GteInfo), C.c_void_p]
    lib.gte_obs_variant_for.argtypes = [P(GteParams), P(GteData)]
    lib.gte_step_obs_launches.argtypes = [P(GteParams), P(GteData), C.c_int, C.c_int]
    lib.gte_step_obs_launches.restype = C.c_int
    lib.gte_step_host_begin.argtypes = [P(GteParams), P(GteData), P(GteState), P(GteHostIO), P(GteStepOut), C.c_void_p,
                                        C.c_int, C.c_int, C.c_void_p]
    lib.gte_step_host_begin.restype = C.c_int
    lib.gte_step_host_end.argtypes = [P(GteHostIO)]
    lib.gte_step_host_end.restype = C.c_int
    lib.gte_serve_stop.argtypes = []
    lib.gte_serve_stop.restype = C.c_int
    lib.gte_relay_supported.argtypes = []
    lib.gte_relay_alloc.argtypes = [C.c_int64, P(C.c_void_p), C.c_void_p]
    lib.gte_relay_open.argtypes = [C.c_void_p, P(C.c_void_p)]
    lib.gte_relay_release.argtypes = [C.c_void_p, C.c_int]
    lib.gte_relay_push.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.gte_relay_serve.argtypes = [C.c_int, C.c_void_p, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.gte_relay_unblock.argtypes = [C.c_void_p, C.c_uint32]
    lib.gte_relay_unblock.restype = C.c_int
    lib.gte_host_register.argtypes = [C.c_void_p, C.c_int64]
    lib.gte_host_unregister.argtypes = [C.c_void_p]
    for name in ("gte_relay_supported", "gte_relay_alloc", "gte_relay_open", "gte_relay_release", "gte_relay_push",
                 "gte_relay_serve", "gte_host_register", "gte_host_unregister"):
        getattr(lib, name).restype = C.c_int
    lib.gte_default_chunks.argtypes = [C.c_int]
    lib.gte_default_chunks.restype = C.c_int
    for name in ("gte_reset", "gte_step", "gte_gather_obs", "gte_step_obs", "gte_step_host", "gte_step_host_begin", "gte_step_host_end", "gte_serve_stop", "gte_relay_supported", "gte_relay_alloc", "gte_relay_open",
           "gte_relay_release", "gte_relay_push", "gte_relay_serve", "gte_relay_unblock", "gte_host_register", "gte_host_unregister", "gte_rollout", "gte_info",
                 "gte_obs_variant_for"):
        getattr(lib, name).restype = C.c_int
    lib.gte_struct_size.argtypes = [C.c_int]
    lib.gte_struct_size.restype = C.c_int
    for which, st in enumerate((GteParams, GteData, GteState, GteStepOut, GteInfo, GteHostIO)):
        if lib.gte_struct_size(which) != C.sizeof(st):
            raise RuntimeError(f"ABI mismatch: {st.__name__} is {C.sizeof(st)} bytes here, "
                               f"{lib.gte_struct_size(which)} in {LIB_PATH} — rebuild the library")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc == 0:
        return
    msg = load().gte_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: {msg}")
