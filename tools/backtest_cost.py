"""What a signal backtest costs: evaluate_signal (one fused fe_backtest launch) against the per-step loops a user could
write without it, on the c2 series (bench.make_series("c2", 60): 1023 days of 252 bars) with S = 1024 momentum columns,
i.e. 1 047 552 envs in evaluate mode, one full 252-step episode each.

    (a)  evaluate_signal(signal)                                         one launch + one host read
    (a') evaluate_signal(signal, targets=True): the same table read as target positions (long / short while the
         momentum is positive / negative)
    (a") the same with a trailing stop and a take-profit per column (exits)
    (b)  per step: torch row lookup -> step_lazy (+ fe_episode_metrics, + its evaluate-mode host read of n_terminated)
    (b') per step: torch row lookup and target -> share delta -> step_lazy (+ the same), the loop a user has for (a')
    (c)  per step: torch row lookup -> step_into (+ fe_episode_metrics), one "all terminated" read at the end

Each leg ends with a report (returns + each env's first-episode metrics) and leaves the env where it started (every env
finished its episode and restarted on its day), so the legs alternate block by block in one process.  The reports of
(a), (b) and (c) must be identical, and so must those of (a') and (b').  Each number is the median of the timed blocks
(host clock around work that ends in a device synchronise, ms per backtest).  Bytes per env-step are counted from
shapes.  Prints the card name and power limit of the same run.

    python tools/backtest_cost.py --out profiles/r06_backtest_targets_cost.json
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from episode_metrics_cost import card  # noqa: E402


def momentum_signal(series, S: int, seed: int = 0):
    """(S, T) f32: sign of the rolling sum of close-to-close log-returns over the last w rows, w in 2..65 drawn per
    column from a seeded generator (0 while fewer than w rows exist)."""
    import torch

    dev = series.logret.device
    g = torch.Generator(device=dev).manual_seed(seed)
    windows = torch.randint(2, 66, (S,), generator=g, device=dev)
    c = torch.cumsum((series.logret[:, 0] + series.logret[:, 3]).double(), 0)   # 100 * log(C_t / C_0)
    idx = torch.arange(c.numel(), device=dev)
    out = torch.empty((S, c.numel()), dtype=torch.float32, device=dev)
    for s in range(S):
        w = int(windows[s])
        prev = torch.where(idx >= w, c[(idx - w).clamp_min(0)], torch.zeros_like(c))
        out[s] = torch.sign(c - prev).float()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--signals", type=int, default=1024)
    ap.add_argument("--window", type=int, default=60)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_backtest_targets_cost.json"))
    args = ap.parse_args()

    import torch

    import bench
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    S, W = args.signals, args.window
    prices, seg_start, seg_len, _ = bench.make_series("c2", W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    D = series.num_segments
    N = S * D
    sig = momentum_signal(series, S)
    cols = (torch.arange(N, device="cuda") // D).to(torch.int32)
    legs_all = ("a", "a_targets", "a_targets_exits", "b", "b_targets", "c")
    envs = {leg: TimeSeriesEnv("cost", num_intervals=W, device_id=0, series=series, num_envs=N, evaluate=True,
                               track_metrics=True, seed=bench.ACTION_SEED) for leg in legs_all}
    # per column a trailing stop and a take-profit, log-uniform in [2, 60] currency units (5 shares of a ~100 price)
    g = torch.Generator(device="cuda").manual_seed(1)
    exits = (2.0 * torch.exp(torch.rand((S, 2), generator=g, device="cuda", dtype=torch.float64) * math.log(30.0)))
    ms = float(envs["b_targets"].max_shares)
    scale = torch.tensor(ms + 0.5, dtype=torch.float32, device="cuda")
    K = int(series.seg_len.max()) - W
    obs = torch.empty((N, W, 5), dtype=torch.float32, device="cuda")
    rew = torch.empty(N, dtype=torch.float32, device="cuda")
    done = torch.empty(N, dtype=torch.int32, device="cuda")

    def lookup(env):
        rows = series.seg_start[env._seg.long()] + env._ptr.long() + W - 1
        return sig[cols.long(), rows].reshape(N, 1)

    def target_actions(env):
        """The header's target -> delta rule in the same f32 operations as fe_backtest_targets_kernel."""
        T = torch.round(lookup(env) * scale).clamp(-ms, ms)
        return (T - (env._long - env._short).reshape(N, 1)) / scale

    def leg_a():
        return envs["a"].evaluate_signal(sig)

    def leg_a_targets():
        return envs["a_targets"].evaluate_signal(sig, targets=True)

    def leg_a_targets_exits():
        return envs["a_targets_exits"].evaluate_signal(sig, targets=True, exits=exits)

    def leg_b():
        env = envs["b"]
        for _ in range(K):
            info = env.step_lazy(lookup(env))[3]
            if "returns" in info:
                return info
        raise RuntimeError("not every env terminated")

    def leg_b_targets():
        env = envs["b_targets"]
        for _ in range(K):
            info = env.step_lazy(target_actions(env))[3]
            if "returns" in info:
                return info
        raise RuntimeError("not every env terminated")

    def leg_c():
        env = envs["c"]
        for _ in range(K):
            env.step_into(lookup(env), obs, rew, done)
        return env.record_evaluation_metrics()

    legs = {"a": leg_a, "a_targets": leg_a_targets, "a_targets_exits": leg_a_targets_exits, "b": leg_b,
            "b_targets": leg_b_targets, "c": leg_c}
    reports = {k: f() for k, f in legs.items()}   # warm-up of every shape, and the results to compare

    def identical(x, others):
        return all(torch.equal(reports[x]["metrics"][k].cpu(), reports[o]["metrics"][k].cpu())
                   and torch.equal(reports[x]["returns"], reports[o]["returns"]) for o in others
                   for k in reports[x]["metrics"])

    same, same_targets = identical("a", ("b", "c")), identical("a_targets", ("b_targets",))
    mean_return = {k: float(r["metrics"]["return"].mean()) for k, r in reports.items()}
    times = {k: [] for k in legs}
    for _ in range(args.blocks):
        for k, f in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: statistics.median(v) for k, v in times.items()}
    # bytes from shapes: per env-step the bar (4 x f64) and the signal value; per env and launch the state read and
    # written once (seg, ptr, cash, long, short, margin, terminated, ep_return; metrics: 6 f64 + 2 i32 + emitted) and
    # one 60-byte record
    state = 4 + 4 + 4 + 4 + 4 + 8 + 1 + 4 + 6 * 8 + 2 * 4 + 1
    per_step = 32 + 4 + (2 * state + 60) / K
    names = {"a": "evaluate_signal (fused fe_backtest launch)",
             "a_targets": "evaluate_signal(targets=True) (fused fe_backtest_targets launch)",
             "a_targets_exits": "evaluate_signal(targets=True, exits) (fused fe_backtest_targets launch)",
             "b": "lookup -> step_lazy -> fe_episode_metrics per step, host read per step",
             "b_targets": "lookup -> target to delta -> step_lazy -> fe_episode_metrics per step, host read per step",
             "c": "lookup -> step_into -> fe_episode_metrics per step"}
    res = {
        "card": card(),
        "workload": {"series": "c2", "window": W, "days": D, "signals": S, "envs": N, "steps": K,
                     "signal_table_bytes": sig.numel() * 4},
        "blocks": args.blocks,
        "exits": "per column: trailing stop and take-profit log-uniform in [2, 60] (seeded)",
        "legs": {k: {"what": names[k], "ms_median": round(med[k], 3), "ms_blocks": [round(x, 3) for x in times[k]],
                     "G_env_steps_per_s": round(N * K / (med[k] * 1e-3) / 1e9, 3),
                     "mean_episode_return": round(mean_return[k], 4)} for k in legs},
        "speedup_a_over_b": round(med["b"] / med["a"], 2),
        "speedup_a_over_c": round(med["c"] / med["a"], 2),
        "speedup_a_targets_over_b_targets": round(med["b_targets"] / med["a_targets"], 2),
        "a_targets_over_a": round(med["a_targets"] / med["a"], 3),
        "a_targets_exits_over_a": round(med["a_targets_exits"] / med["a"], 3),
        "bytes_per_env_step_a": round(per_step, 2),
        "achieved_GB_per_s_a": round(N * K * per_step / (med["a"] * 1e-3) / 1e9, 1),
        "reports_identical": bool(same),
        "target_reports_identical": bool(same_targets),
    }
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
