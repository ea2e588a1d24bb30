"""What computing the rules on the device costs against a signal table, on three workloads (bench.make_series):

    c2  1023 days of 252 bars, W = 60, 1024 mixed rules (momentum, MA crossover, Bollinger, constant): 1 047 552 envs
    c3  30 assets, 1023 days of 252 bars, W = 128, 64 cross-sectional momentum rules (w in 5..130, n in 1..10, the shape
        of the r10 workload): 65 472 envs
    c4  10 M minute bars, 25 640 days of 390 bars, W = 60, 256 mixed rules: 6 563 840 envs; the table is 10.2 GB

each in evaluate mode, one full episode per env, and three legs:

    (r)  evaluate_rules(rules)                                   the values computed in the kernel, no table
    (t)  rule_table(rules) (fe_rule_table), then evaluate_signal / evaluate_portfolio_signal on it
    (t0) evaluate_signal / evaluate_portfolio_signal on a table built beforehand

The three reports must be identical.  Each number is the median of the timed blocks (host clock around work that ends
in a device synchronise, ms per report); the legs alternate block by block in one process.  Memory is counted from
shapes: the staged running sums (StagedSeries.rule_sums()) against the table.  The one-time staging of those sums
(fe_rule_sums_build) is timed with device events.  Prints the card name and power limit of
the same run.

    python tools/rule_backtest_cost.py --out profiles/r11_rule_backtest_cost.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from episode_metrics_cost import card  # noqa: E402

WORKLOADS = {"c2": (60, 1024), "c3": (128, 64), "c4": (60, 256)}   # (W, rules)


def mixed_rules(S: int, seed: int = 0):
    """S single-asset rules, a quarter each of momentum (w in 1..399), MA crossover (fast in 1..49, slow in 50..1999),
    Bollinger (w in 2..399, k in 0.5..3) and constant +-1, parameters from a seeded generator."""
    from finenvs_b200 import rules as R

    rng = np.random.default_rng(seed)
    q = S // 4
    return R.concat(R.momentum(rng.integers(1, 400, q)), R.ma_cross(rng.integers(1, 50, q), rng.integers(50, 2000, q)),
                    R.bollinger(rng.integers(2, 400, q), rng.uniform(0.5, 3.0, q)),
                    R.constant(np.where(np.arange(S - 3 * q) % 2 == 0, 1.0, -1.0)))


def xs_rules(S: int, A: int, seed: int = 0):
    from finenvs_b200 import rules as R

    rng = np.random.default_rng(seed)
    return R.xs_momentum(rng.integers(5, 131, S), rng.integers(1, max(A // 3, 1) + 1, S))


def run(workload: str, blocks: int) -> dict:
    import torch

    import bench
    from finenvs_b200 import _lib
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    W, S = WORKLOADS[workload]
    prices, seg_start, seg_len, _ = bench.make_series(workload, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    D, A, T = series.num_segments, series.num_assets, series.num_rows
    N = S * D
    rules = xs_rules(S, A) if A > 1 else mixed_rules(S)
    envs = {leg: TimeSeriesEnv("cost", num_intervals=W, device_id=0, series=series, num_envs=N, evaluate=True,
                               track_metrics=True, seed=bench.ACTION_SEED) for leg in ("r", "t", "t0")}
    sums = series.rule_sums()
    table0 = envs["t0"].rule_table(rules)

    def evaluate(env, table):
        return env.evaluate_signal(table) if A == 1 else env.evaluate_portfolio_signal(table)

    def leg_t():
        env = envs["t"]
        return evaluate(env, env.rule_table(rules))

    legs = {"r": lambda: envs["r"].evaluate_rules(rules), "t": leg_t, "t0": lambda: evaluate(envs["t0"], table0)}
    reports = {k: f() for k, f in legs.items()}   # warm-up of every shape, and the results to compare

    def identical(x, y):
        return (all(torch.equal(reports[x]["metrics"][k], reports[y]["metrics"][k]) for k in reports[x]["metrics"])
                and torch.equal(reports[x]["returns"], reports[y]["returns"]))

    same = {"r==t0": bool(identical("r", "t0")), "t==t0": bool(identical("t", "t0"))}
    steps = reports["r"]["steps"]
    mean_return = {k: float(r["metrics"]["return"].mean()) for k, r in reports.items()}
    del reports
    times = {k: [] for k in legs}
    for _ in range(blocks):
        for k, f in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: statistics.median(v) for k, v in times.items()}
    # the one-time staging of the running sums (fe_rule_sums_build), timed with device events into a second buffer
    L, buf, stream = _lib.lib(), torch.empty_like(sums), torch.cuda.current_stream()
    staging = []
    for _ in range(blocks + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(L.fe_rule_sums_build(series.prices.data_ptr(), T, A, buf.data_ptr(), 0, stream.cuda_stream),
                   "fe_rule_sums_build")
        e1.record()
        torch.cuda.synchronize()
        staging.append(e0.elapsed_time(e1))
    assert torch.equal(buf, sums)
    names = {"r": "evaluate_rules (fe_backtest_rules: values computed in the kernel)",
             "t": "rule_table (fe_rule_table) + evaluate on that table",
             "t0": "evaluate on a table built beforehand"}
    kinds = np.bincount(rules.records["kind"], minlength=5).tolist()
    return {
        "workload": {"series": workload, "assets": A, "rows": T, "window": W, "days": D, "rules": S, "envs": N,
                     "steps": steps, "rule_kinds [const, momentum, ma_cross, bollinger, xs_momentum]": kinds},
        "staging_ms": {"fe_rule_sums_build_median": round(statistics.median(staging[1:]), 3),
                       "first_call": round(staging[0], 3)},
        "bytes": {"staged_sums": sums.numel(), "table": table0.numel() * 4,
                  "table_over_sums": round(table0.numel() * 4 / sums.numel(), 1)},
        "legs": {k: {"what": names[k], "ms_median": round(med[k], 3), "ms_blocks": [round(x, 3) for x in times[k]],
                     "mean_episode_return": round(mean_return[k], 4)} for k in legs},
        "r_over_t0": round(med["r"] / med["t0"], 3),
        "r_over_t": round(med["r"] / med["t"], 3),
        "reports_identical": same,
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3,c4")
    ap.add_argument("--blocks", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(), "blocks": args.blocks, "workloads": {}}
    for w in args.workloads.split(","):
        res["workloads"][w] = run(w, args.blocks)
        torch.cuda.empty_cache()
        print(json.dumps({w: res["workloads"][w]}, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
