"""What track_metrics=True costs per step: the extra fe_episode_metrics launch after the step, on the c2 workload
(1 Mi envs, W = 60, bench.make_series) for the device-resident step_into, step_lazy and a 32-step CapturedRollout
replay, with and without the metrics.  The two envs alternate block by block in one process; each number is the median
of the timed blocks (CUDA events, ms per step).  Prints the card name and power limit of the same run.

    python tools/episode_metrics_cost.py --out profiles/r04_episode_metrics_cost.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card() -> dict:
    import torch

    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = (x.strip() for x in q.split(","))
    except Exception as e:  # the measurement stands without it, but say so
        out["power_limit"] = f"unavailable ({e})"
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--window", type=int, default=60)
    ap.add_argument("--steps", type=int, default=64, help="steps per timed block (a multiple of 32)")
    ap.add_argument("--blocks", type=int, default=9)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_episode_metrics_cost.json"))
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    N, W, K = args.envs, args.window, args.steps
    prices, seg_start, seg_len, meta = bench.make_series("c2", W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    envs = {on: TimeSeriesEnv("cost", num_intervals=W, device_id=0, series=series, num_envs=N, seed=bench.ACTION_SEED,
                              random_reset="all", random_offset=True, track_metrics=on) for on in (False, True)}
    g = torch.Generator(device="cuda").manual_seed(bench.ACTION_SEED)
    ring = [torch.rand((N, 1), generator=g, device="cuda") * 2 - 1 for _ in range(8)]
    obs = torch.empty((N, W, 5), dtype=torch.float32, device="cuda")
    rewards = torch.empty(N, dtype=torch.float32, device="cuda")
    dones = torch.empty(N, dtype=torch.int32, device="cuda")
    rolls = {on: env.capture_rollout(lambda o: ring[0], 32) for on, env in envs.items()}

    legs = {
        "step_into": lambda env, on, i: env.step_into(ring[i % 8], obs, rewards, dones),
        "step_lazy": lambda env, on, i: env.step_lazy(ring[i % 8]),
        "captured_replay_32": lambda env, on, i: rolls[on].replay(refresh_obs=False) if i % 32 == 0 else None,
    }
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    result = {"card": card(), "workload": "c2", "envs": N, "window": W, "steps_per_block": K, "blocks": args.blocks,
              "series": meta, "legs": {}}
    for leg, fn in legs.items():
        times = {False: [], True: []}
        for on, env in envs.items():   # warm-up
            for i in range(K):
                fn(env, on, i)
        for b in range(args.blocks):
            for on, env in envs.items():
                if on:
                    env.clear_metrics()
                torch.cuda.synchronize()
                ev0.record()
                for i in range(K):
                    fn(env, on, i)
                ev1.record()
                ev1.synchronize()
                times[on].append(ev0.elapsed_time(ev1) / K)
        off_ms, on_ms = float(np.median(times[False])), float(np.median(times[True]))
        result["legs"][leg] = {"ms_per_step_off": off_ms, "ms_per_step_on": on_ms,
                               "overhead_pct": 100.0 * (on_ms - off_ms) / off_ms,
                               "spread_ms_off": [min(times[False]), max(times[False])],
                               "spread_ms_on": [min(times[True]), max(times[True])]}
        print(leg, json.dumps(result["legs"][leg]), flush=True)
    s = envs[True].metrics_summary()
    result["episodes_recorded_last_block"] = int(s["episodes"].item())
    print(json.dumps(result["card"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
