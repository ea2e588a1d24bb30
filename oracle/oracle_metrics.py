"""Numpy restatement of the per-episode trading metrics (fe_episode_metrics, csrc/fe_metrics.cu; definition in
include/finenvs_b200.h and DESIGN.md §4.11).

The same float64 operations in the same order, each one IEEE-rounded (numpy's element-wise ufuncs contract nothing),
so the records match the kernel's bit for bit.  The aggregate sums are exact (math.fsum); the kernel adds them with
atomics in an arbitrary order, so tests compare those within a relative bound and the counts exactly.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np

RECORD_KEYS = ("key", "env", "len", "return", "sharpe", "mdd", "mdd_rel", "hit_rate")


def episode_metrics(rewards: np.ndarray, dones: np.ndarray, starting_balance: float, *, first_step: int = 1,
                    env_id_base: int = 0, total_envs: Optional[int] = None, evaluate: bool = False
                    ) -> Tuple[Dict[str, np.ndarray], Dict[str, float]]:
    """rewards (T, N) f32 | f64, dones (T, N) of one rollout starting from zero running state; row t is step ordinal
    first_step + t.  evaluate: an env records only its first episode.  Returns (records sorted by key, aggregates)."""
    r_all = np.asarray(rewards).astype(np.float64)
    d_all = np.asarray(dones) != 0
    T, N = r_all.shape
    total = N if total_envs is None else int(total_envs)
    gid = env_id_base + np.arange(N, dtype=np.int64)
    ln = np.zeros(N, np.int32)
    pos = np.zeros(N, np.int32)
    s, mean, m2, peak, mdd, mdd_rel = (np.zeros(N) for _ in range(6))
    emitted = np.zeros(N, bool)
    sb = np.float64(starting_balance)
    out = {k: [] for k in RECORD_KEYS}
    for t in range(T):
        r, done = r_all[t], d_all[t]
        ln = ln + 1
        dlen = ln.astype(np.float64)
        s = s + r
        d = r - mean
        mean = mean + d / dlen
        m2 = m2 + d * (r - mean)
        pos = pos + (r > 0)
        peak = np.maximum(peak, s)
        dd = peak - s
        mdd = np.maximum(mdd, dd)
        mdd_rel = np.maximum(mdd_rel, dd / (sb + peak))
        if done.any():
            emit = done & ~emitted if evaluate else done
            if evaluate:
                emitted |= done
            e = np.nonzero(emit)[0]
            with np.errstate(divide="ignore", invalid="ignore"):
                sharpe = np.where((ln[e] < 2) | (m2[e] == 0.0), 0.0, mean[e] / np.sqrt(m2[e] / dlen[e]))
            out["key"].append((first_step + t) * total + gid[e])
            out["env"].append(gid[e])
            out["len"].append(ln[e])
            out["return"].append(s[e])
            out["sharpe"].append(sharpe)
            out["mdd"].append(mdd[e])
            out["mdd_rel"].append(mdd_rel[e])
            out["hit_rate"].append(pos[e] / dlen[e])
            for a in (s, mean, m2, peak, mdd, mdd_rel):
                a[done] = 0.0
            ln[done] = 0
            pos[done] = 0
    dtypes = {"key": np.int64, "env": np.int64, "len": np.int32}
    rec = {k: (np.concatenate(v) if v else np.zeros(0, dtypes.get(k, np.float64))).astype(dtypes.get(k, np.float64))
           for k, v in out.items()}
    order = np.argsort(rec["key"], kind="stable")
    rec = {k: v[order] for k, v in rec.items()}
    agg = {
        "episodes": int(rec["key"].size),
        "sum_len": int(rec["len"].astype(np.int64).sum()),
        "sum_return": math.fsum(rec["return"]),
        "sum_sharpe": math.fsum(rec["sharpe"]),
        "sum_sharpe_sq": math.fsum(rec["sharpe"] * rec["sharpe"]),
        "sum_mdd": math.fsum(rec["mdd"]),
        "max_mdd": float(rec["mdd"].max()) if rec["mdd"].size else 0.0,
        "sum_hit_rate": math.fsum(rec["hit_rate"]),
    }
    return rec, agg


def abs_sums(rec: Dict[str, np.ndarray]) -> Dict[str, float]:
    """Σ|x| of each summed field: the scale an order-dependent f64 sum's error is bounded by."""
    return {"sum_return": math.fsum(np.abs(rec["return"])), "sum_sharpe": math.fsum(np.abs(rec["sharpe"])),
            "sum_sharpe_sq": math.fsum(rec["sharpe"] * rec["sharpe"]), "sum_mdd": math.fsum(rec["mdd"]),
            "sum_hit_rate": math.fsum(rec["hit_rate"])}
