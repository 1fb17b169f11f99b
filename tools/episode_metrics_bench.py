"""Cost of the episode-metric catalogue on the device: ms per lockstep iteration (step + observation gather) with no
episode metric and with all five (add_metric), at the C5 shard shape (2^21 envs, W=64, 7 positions, D=720, the default
dynamic pair) and at C3 (65 536 envs).

    python tools/episode_metrics_bench.py [--out FILE.json] [--repeats 5] [--min-seconds 0.3]

In one process: the HBM copy peak (as tools/hbm_probe.py measures it: the best of 10 copies of 2.5 GiB), then both
configurations of a workload timed in turn, alternating, each region >= --min-seconds of device time between CUDA
events after a warm-up, median of --repeats regions.  The metrics add up to 80 bytes per env-step of state traffic
(5 f64 accumulators read and written) to bench.algorithmic_bytes' count, reported beside it.  The GPU's name, power
limit and maximum SM clock are read with a read-only nvidia-smi query and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = {
    "c5": dict(envs=1 << 21, positions=[-3, -2, -1, 0, 1, 2, 3]),
    "c3": dict(envs=65_536, positions=[-1, 0, 0.5, 1]),
}
CONFIGS = {            # name -> the add_metric kinds
    "none": [],
    "all5": ["position_changes", "episode_length", "max_drawdown", "episode_reward", "time_in_market"],
}
W, D = 64, 720
ACC_BYTES = 2 * 8 * 5     # five f64 accumulator rows, read and written every step


def gpu_identity():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def hbm_copy_peak(torch):
    n = (5 * 1024 ** 3) // 4
    a = torch.empty(n, dtype=torch.float32, device="cuda")
    src, dst = a[: n // 2], a[n // 2: 2 * (n // 2)]
    for _ in range(3):
        dst.copy_(src)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a
    torch.cuda.empty_cache()
    return 2 * src.numel() * 4 / (best * 1e-3)          # bytes / s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--min-seconds", type=float, default=0.3)
    ap.add_argument("--workloads", default="c5,c3")
    args = ap.parse_args()
    import torch
    import bench
    import gym_trading_env_b200 as gte
    assert torch.cuda.is_available(), "needs a CUDA device"
    ident = gpu_identity()
    peak = hbm_copy_peak(torch)
    print(f"GPU: {ident}\nHBM copy peak: {peak / 1e12:.3f} TB/s", flush=True)
    series = gte.frame_to_arrays(gte.make_gbm_ohlcv(100_000, seed=0))
    ns = series.features.shape[1]
    results = []
    for wname in args.workloads.split(","):
        wl = WORKLOADS[wname]
        N = wl["envs"]
        envs = {}
        for nd, kinds in CONFIGS.items():
            env = gte.TradingVectorEnv(series, positions=wl["positions"], windows=W, trading_fees=1e-4,
                                       borrow_interest_rate=3e-6, portfolio_initial_value=1000, max_episode_duration=D,
                                       num_envs=N, seed=2024, verbose=0)
            for k in kinds:
                env.add_metric(k, gte.DeviceMetric(k))
            env.reset()
            envs[nd] = env
        gen = torch.Generator(device="cuda")
        gen.manual_seed(1234)
        acts = torch.randint(0, len(wl["positions"]), (8, N), generator=gen, device="cuda", dtype=torch.int64)
        steps = {}
        for nd, env in envs.items():                        # warm-up + calibration: >= min_seconds per region
            for k in range(20):
                env.step(acts[k % 8])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(20):
                env.step(acts[k % 8])
            e1.record()
            torch.cuda.synchronize()
            per = e0.elapsed_time(e1) / 20
            steps[nd] = max(50, int(args.min_seconds * 1e3 / per) + 1)
        times = {nd: [] for nd in envs}
        for r in range(args.repeats):                       # configurations alternate
            for nd, env in envs.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for k in range(steps[nd]):
                    env.step(acts[k % 8])
                e1.record()
                torch.cuda.synchronize()
                times[nd].append(e0.elapsed_time(e1) / steps[nd])
        for nd, env in envs.items():
            env.check_errors()
            ms = statistics.median(times[nd])
            step_b, obs_b = bench.algorithmic_bytes(W, ns, 2)
            nbytes = step_b + obs_b + (ACC_BYTES if CONFIGS[nd] else 0)
            rate = N / (ms * 1e-3)
            row = dict(workload=wname, n_envs=N, metrics=nd, kinds=CONFIGS[nd], obs_variant=env.obs_variant,
                       launches_per_step=env.launches_per_step, steps_per_region=steps[nd], repeats=args.repeats,
                       ms_per_iter=ms, ms_min=min(times[nd]), ms_max=max(times[nd]), env_steps_per_s=rate,
                       algorithmic_bytes_per_env_step=nbytes, achieved_tb_s=rate * nbytes / 1e12,
                       fraction_of_copy_peak=rate * nbytes / peak)
            results.append(row)
            print(f"{wname} metrics={nd}: {ms:.4f} ms/iter (min {row['ms_min']:.4f}, max {row['ms_max']:.4f}), "
                  f"{rate / 1e9:.3f} G env-steps/s, {nbytes} B/env-step, {row['achieved_tb_s']:.3f} TB/s = "
                  f"{row['fraction_of_copy_peak']:.3f} of copy peak  [{env.obs_variant}, "
                  f"{env.launches_per_step} launch(es)]", flush=True)
        del envs
        torch.cuda.empty_cache()
    for wname in args.workloads.split(","):
        t = {r["metrics"]: r["ms_per_iter"] for r in results if r["workload"] == wname}
        print(f"{wname}: all five metrics cost {100 * (t['all5'] / t['none'] - 1):+.1f} % per iteration", flush=True)
    doc = dict(gpu=ident, hbm_copy_peak_tb_s=peak / 1e12, windows=W, max_episode_duration=D, n_static=ns,
               results=results)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
