"""Generates tests/golden/*.npz by running the REAL reference (hmomin/FinEnvs) in this container.

Run:  python tests/golden/make_golden.py        (needs /root/reference; CPU only)

Each trace stores the inputs (flat series exactly as the reference built it, per-step actions,
seed for the injected Philox redraws) and the reference's outputs after every step (rewards,
dones, full state; the observation tensor on selected steps plus a per-env f64 row-sum on all
steps).  The GPU box has no reference checkout, so these files are what pins the oracle and the
CUDA path there.  The dummy CSV inputs are stored as arrays (not as files) and re-serialised by
the tests.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_harness as rh  # noqa: E402
from parity_utils import day_labels, gbm_ohlc  # noqa: E402


def digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(np.nan_to_num(a, nan=-12345.0)).tobytes()).hexdigest()


def csv_arrays(path: str) -> dict:
    import pandas as pd

    df = pd.read_csv(path, names=["Date", "Time", "Open", "High", "Low", "Close", "Volume"])
    return {
        "csv_date": df["Date"].to_numpy().astype("S10"),
        "csv_time": df["Time"].to_numpy().astype("S5"),
        "csv_ohlc": df[["Open", "High", "Low", "Close"]].to_numpy(np.float64),
        "csv_volume": df["Volume"].to_numpy(np.int64),
    }


def trace(csv: str, window: int, steps: int, seed: int, *, evaluate=False, widen=None, action_fn=None,
          scripted=None, store_all_obs=False, max_obs_steps=10, params=None, obs_at=None) -> dict:
    """`params`: (max_shares, starting_balance, per_share_commission, initial_margin_requirement,
    maintenance_margin_requirement) when they differ from the reference's defaults (time_series_env.py:20-26).
    `obs_at`: the steps whose full observation is stored (default: the first two, the first steps with dones, the last)."""
    ref_kw = {}
    if params is not None:
        ref_kw = dict(max_shares=int(params[0]), starting_balance=float(params[1]), per_share_commission=float(params[2]),
                      initial_margin_requirement=float(params[3]), maintenance_margin_requirement=float(params[4]))
    r = rh.RefEnv(csv, "dummy", window, seed=seed, evaluate=evaluate, **ref_kw)
    fs = rh.flat_series_from_ref(r)
    out = {
        "window": window, "seed": seed, "evaluate": int(evaluate),
        "params": np.array(params if params is not None else (5, 10000.0, 0.01, 1.5, 0.25), dtype=np.float64),
        "prices": fs.prices, "logret": fs.logret, "seg_start": fs.seg_start, "seg_len_raw": fs.seg_len_raw,
        "pe_shape": np.array(r.env.price_environments.shape),
        "pe_digest": digest(r.env.price_environments.numpy()),
        "le_digest": digest(r.env.log_return_environments.numpy()),
    }
    if widen:
        seg_init = (np.arange(widen) % fs.num_segments).astype(np.int32)
        r.widen(seg_init)
    st0 = r.state()
    out["seg_init"] = st0["seg"]
    out["obs_reset"] = r.reset()
    N = int(r.env.num_envs)
    rng = np.random.default_rng(seed + 1)
    if scripted is not None:
        steps = len(scripted)
    acts, rews, dones, states, obs_sums, obs_kept, obs_steps, infos, info_steps = [], [], [], [], [], [], [], [], []
    for t in range(steps):
        if scripted is not None:
            a = np.asarray(scripted[t], np.float32)
        elif action_fn is not None:
            a = action_fn(rng, N)
        else:
            a = rng.uniform(-1, 1, N).astype(np.float32)
        o, rw, d, info = r.step(a)
        acts.append(a); rews.append(rw); dones.append(d)
        s = r.state()
        states.append(np.stack([s["seg"].astype(np.float64), s["ptr"].astype(np.float64), s["cash"].astype(np.float64),
                                s["long_sh"].astype(np.float64), s["short_sh"].astype(np.float64), s["margin"]]))
        obs_sums.append(o.reshape(N, -1).sum(axis=1))
        if obs_at is not None:
            keep = t in obs_at
        else:
            keep = store_all_obs or t < 2 or (d.any() and len(obs_steps) < max_obs_steps) or t == steps - 1
        if keep:
            obs_kept.append(o); obs_steps.append(t)
        if info:
            infos.append(info["returns"]); info_steps.append(t)
    out.update(actions=np.stack(acts), rewards=np.stack(rews), dones=np.stack(dones), states=np.stack(states),
               obs_sums=np.stack(obs_sums), obs=np.stack(obs_kept), obs_steps=np.array(obs_steps),
               draw_log=np.array(r.draw_log, dtype=np.int64).reshape(-1, 3))
    if infos:
        out.update(info_returns=np.stack(infos), info_steps=np.array(info_steps))
    r.close()
    nd = int(np.stack(dones).sum())
    print(f"  {os.path.basename(os.path.dirname(csv))} W={window} N={N} steps={steps} dones={nd} "
          f"draws={len(r.draw_log)} obs_kept={len(obs_steps)}")
    return out


def short_biased(frac):
    def f(rng, n):
        a = rng.uniform(-1, 1, n)
        m = rng.uniform(0, 1, n) < frac
        a[m] = -np.abs(a[m])
        return a.astype(np.float32)
    return f


def main():
    import tempfile

    os.chdir(HERE)
    # ---- the three dummy CSV fixtures of the reference (finenvs/data/{IBM,OIH,SPY}/dummy.csv)
    csvs = {n: os.path.join(rh.data_dir(n), "dummy.csv") for n in ("IBM", "OIH", "SPY")}
    np.savez_compressed("dummy_csv.npz", **{f"{n}_{k}": v for n, p in csvs.items() for k, v in csv_arrays(p).items()})

    # ---- SURVEY App. B known-answer trace
    kat = trace(csvs["IBM"], 390, 0, 0, store_all_obs=True,
                scripted=[[1, -1, 0.3], [1, -1, -0.3], [-1, 1, 0.05], [0.5, 0.5, 0.5], [-0.2, 0.9, -1]])
    np.savez_compressed("kat_ibm_w390.npz", **kat)

    # ---- dummy CSVs, several windows, training mode (last env redraws) and evaluate mode
    for name, W, steps, seed, ev in [
        ("IBM", 60, 450, 3, False), ("IBM", 4, 420, 4, False),
        ("OIH", 390, 200, 5, False), ("OIH", 60, 450, 6, False), ("OIH", 4, 300, 7, False),
        ("SPY", 60, 450, 8, False), ("SPY", 390, 400, 9, False),
        ("OIH", 60, 450, 10, True), ("SPY", 4, 800, 11, True),
    ]:
        t = trace(csvs[name], W, steps, seed, evaluate=ev, max_obs_steps=4 if W == 390 else 10)
        np.savez_compressed(f"trace_{name.lower()}_w{W}{'_eval' if ev else ''}.npz", **t)

    # ---- widened N on a real CSV (env i -> segment i mod D); 100 steps and three full observations keep it under 1 MB
    t = trace(csvs["OIH"], 60, 100, 12, widen=256, obs_at=(0, 19, 24))
    np.savez_compressed("trace_oih_w60_n256.npz", **t)

    # ---- adversarial GBM: big intrabar spikes + short-biased actions => margin calls at High and
    # Close, releases, bankruptcies, blocked entries, ragged days (NaN padding dones)
    with tempfile.TemporaryDirectory() as td:
        rng = np.random.default_rng(20260101)
        bars = [40, 25, 40, 33, 40, 12, 40, 40, 1, 40, 38, 40]
        dates, times = day_labels(len(bars), bars)
        for tag, sigma, frac, seed in [("s15", 0.15, 0.6, 13), ("s03", 0.03, 0.9, 14), ("s08", 0.08, 0.3, 15)]:
            ohlc = gbm_ohlc(rng, sum(bars), sigma)
            p = os.path.join(td, f"adv_{tag}.csv")
            rh.write_csv(p, dates, times, ohlc)
            t = trace(p, 8, 300, seed, widen=96, action_fn=short_biased(frac), max_obs_steps=12)
            np.savez_compressed(f"trace_adv_{tag}_w8_n96.npz", **t)

    # ---- every constructor parameter off its default (time_series_env.py:20-26), ragged days, actions beyond [-1, 1]
    with tempfile.TemporaryDirectory() as td:
        for tag, seed, W, sigma, s0, params, ev in [
            ("p1", 31, 5, 0.08, 40.0, (40, 500.0, 0.37, 2.25, 0.4), False),
            ("p2", 32, 3, 0.2, 3.0, (1, 250000.0, 0.0, 1.0, 0.1), True),
            ("p3", 33, 9, 0.02, 900.0, (12, 20000.0, 0.05, 1.2, 0.3), False),
        ]:
            rng = np.random.default_rng(seed)
            bars = [W + 3, 20, 1, 14, 31, 2, 9, 20, 5]
            dates, times = day_labels(len(bars), bars)
            p = os.path.join(td, f"par_{tag}.csv")
            rh.write_csv(p, dates, times, gbm_ohlc(rng, sum(bars), sigma, s0=s0))
            bias = {"p1": -0.4, "p2": 0.3, "p3": 0.0}[tag]
            t = trace(p, W, 220, seed, evaluate=ev, widen=64, params=params, max_obs_steps=8,
                      action_fn=lambda r, n, b=bias: np.clip(r.normal(b, 0.8, n), -1.3, 1.3).astype(np.float32))
            np.savez_compressed(f"trace_par_{tag}_w{W}_n64.npz", **t)

    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f"{f}: {os.path.getsize(f) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
