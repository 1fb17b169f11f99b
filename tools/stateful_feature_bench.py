"""Cost of the stateful dynamic features (current_drawdown, position_age) on the device: ms per lockstep iteration
(step + observation gather) at the C5 shard shape (2^21 envs, W=64, 7 positions, D=720) and at C3 (65 536 envs), in
three configurations:

- ``pair``: the default pair (position, real_position);
- ``pair+stateful``: the default pair plus both stateful kinds;
- ``five-f32``: real_position, portfolio_return, reward, current_drawdown, position_age — five f32 ring blocks, the
  largest ring tile (W x 640 bytes).

    python tools/stateful_feature_bench.py [--out FILE.json] [--repeats 5] [--min-seconds 0.3]

In one process, the configurations of a workload are timed in turn, alternating, each region >= --min-seconds of device
time between CUDA events after a warm-up, median of --repeats regions.  The gather variant each configuration takes
and its launches per step are reported with it.  The GPU's name, power limit and maximum SM clock are read with a
read-only nvidia-smi query and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from episode_metrics_bench import WORKLOADS, gpu_identity  # noqa: E402

CONFIGS = {
    "pair": ["position", "real_position"],
    "pair+stateful": ["position", "real_position", "current_drawdown", "position_age"],
    "five-f32": ["real_position", "portfolio_return", "reward", "current_drawdown", "position_age"],
}
W, D = 64, 720


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--min-seconds", type=float, default=0.3)
    ap.add_argument("--workloads", default="c5,c3")
    args = ap.parse_args()
    import torch
    import gym_trading_env_b200 as gte
    assert torch.cuda.is_available(), "needs a CUDA device"
    ident = gpu_identity()
    print(f"GPU: {ident}", flush=True)
    series = gte.frame_to_arrays(gte.make_gbm_ohlcv(100_000, seed=0))
    results = []
    for wname in args.workloads.split(","):
        wl = WORKLOADS[wname]
        N = wl["envs"]
        envs = {}
        for name, kinds in CONFIGS.items():
            env = gte.TradingVectorEnv(series, positions=wl["positions"], windows=W, trading_fees=1e-4,
                                       borrow_interest_rate=3e-6, portfolio_initial_value=1000, max_episode_duration=D,
                                       num_envs=N, seed=2024, verbose=0,
                                       dynamic_feature_functions=[gte.DeviceFeature(k) for k in kinds])
            env.reset()
            envs[name] = env
        gen = torch.Generator(device="cuda")
        gen.manual_seed(1234)
        acts = torch.randint(0, len(wl["positions"]), (8, N), generator=gen, device="cuda", dtype=torch.int64)
        steps = {}
        for name, env in envs.items():                      # warm-up + calibration: >= min_seconds per region
            for k in range(20):
                env.step(acts[k % 8])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(20):
                env.step(acts[k % 8])
            e1.record()
            torch.cuda.synchronize()
            steps[name] = max(50, int(args.min_seconds * 1e3 / (e0.elapsed_time(e1) / 20)) + 1)
        times = {name: [] for name in envs}
        for r in range(args.repeats):                       # configurations alternate
            for name, env in envs.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for k in range(steps[name]):
                    env.step(acts[k % 8])
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / steps[name])
        for name, env in envs.items():
            env.check_errors()
            ms = statistics.median(times[name])
            row = dict(workload=wname, n_envs=N, config=name, kinds=CONFIGS[name], obs_variant=env.obs_variant,
                       launches_per_step=env.launches_per_step, ring_tile_bytes=int(env._dyn_ring.shape[1]),
                       steps_per_region=steps[name], repeats=args.repeats, ms_per_iter=ms, ms_min=min(times[name]),
                       ms_max=max(times[name]), env_steps_per_s=N / (ms * 1e-3))
            results.append(row)
            print(f"{wname} {name}: {ms:.4f} ms/iter (min {row['ms_min']:.4f}, max {row['ms_max']:.4f})  "
                  f"[{env.obs_variant}, {env.launches_per_step} launch(es), ring tile {row['ring_tile_bytes']} B]",
                  flush=True)
        del envs
        torch.cuda.empty_cache()
    doc = dict(gpu=ident, windows=W, max_episode_duration=D, results=results)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
