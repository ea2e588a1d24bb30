"""Numpy restatement of the device rules (include/finenvs_b200.h, "rule backtests"; csrc/fe_step.cu: fe_rule_sums_kernel,
rule_window, rule_sign_ts, rule_sign_xs, rule_value): the same IEEE f64 operations in the same order, so every staged
sum and every rule value matches the device bit for bit.  Vectorised over rows and assets; `rows` selects the rows to
evaluate (all by default).

`records` are rule records (finenvs_b200.rules.RECORD, or any structured array with its field names); `closes` is the
(T, A) float64 array prices[:, :, 3] ((T,) is taken as A = 1)."""
from __future__ import annotations

import numpy as np

BLOCK = 1024
MAX_LOOKBACK = 65536
CONST, MOMENTUM, MA_CROSS, BOLLINGER, XS_MOMENTUM = 0, 1, 2, 3, 4


def _closes(closes) -> np.ndarray:
    c = np.asarray(closes, dtype=np.float64)
    return c[:, None] if c.ndim == 1 else c


def rule_sums(closes) -> dict:
    """fe_rule_sums_build: per block of BLOCK rows and asset, base = the first finite close (0 if none), then inclusive
    running sums of d = C - base (0 for a non-finite close) and d * d, and the running count of non-finite closes."""
    c = _closes(closes)
    T, A = c.shape
    B = -(-T // BLOCK)
    pad = np.full((B * BLOCK, A), np.nan)
    pad[:T] = c
    blk = pad.reshape(B, BLOCK, A)
    fin = np.isfinite(blk)
    first = np.argmax(fin, axis=1)                                        # (B, A): first finite row of the block
    base = np.where(fin.any(axis=1), np.take_along_axis(blk, first[:, None, :], axis=1)[:, 0, :], 0.0)
    with np.errstate(invalid="ignore"):
        d = np.where(fin, blk - base[:, None, :], 0.0)
    s1 = np.cumsum(d, axis=1).reshape(-1, A)[:T]                          # sequential: one rounding per row
    s2 = np.cumsum(d * d, axis=1).reshape(-1, A)[:T]
    nf = np.cumsum(~fin, axis=1, dtype=np.int32).reshape(-1, A)[:T]
    return {"s1": s1, "s2": s2, "base": base, "nf": nf}


def sums_bytes(sums: dict) -> bytes:
    """The staged buffer's bytes (the header's layout), to compare with the device's."""
    return b"".join(np.ascontiguousarray(sums[k]).tobytes() for k in ("s1", "s2", "base", "nf"))


def window(sums: dict, r: np.ndarray, k: int):
    """rule_window over rows r-k+1 .. r of every asset (r >= k-1): (t1, t2, ok, ref), each (len(r), A): the sums of
    C - ref and (C - ref)^2 with ref the base of r's block, and whether the window's closes are all finite."""
    s1, s2, nf, base = sums["s1"], sums["s2"], sums["nf"], sums["base"]
    r = np.asarray(r, dtype=np.int64)
    lo, hi = r - k + 1, r
    bh, bl = hi // BLOCK, lo // BLOCK
    ref = base[bh]
    t1 = np.zeros_like(ref)
    t2 = np.zeros_like(ref)
    bad = np.zeros(ref.shape, dtype=np.int32)
    pieces = int((bh - bl).max()) + 1 if r.size else 0
    for j in range(pieces):
        live = (bh - j >= bl)[:, None]
        b = np.maximum(bh - j, bl)
        b0 = b * BLOCK
        e = hi if j == 0 else np.minimum(b0 + BLOCK - 1, hi)              # = b0 + BLOCK - 1 where live
        s0 = np.maximum(lo, b0)
        p1, p2, c = s1[e], s2[e], nf[e]
        sub = (s0 > b0)[:, None]
        prev = np.maximum(s0 - 1, 0)
        p1 = np.where(sub, p1 - s1[prev], p1)
        p2 = np.where(sub, p2 - s2[prev], p2)
        c = np.where(sub, c - nf[prev], c)
        if j > 0:
            dl = base[b] - ref
            n = (e - s0 + 1).astype(np.float64)[:, None]
            p2 = (p2 + (2.0 * dl) * p1) + n * (dl * dl)
            p1 = p1 + n * dl
        t1 = np.where(live, t1 + p1, t1)
        t2 = np.where(live, t2 + p2, t2)
        bad = np.where(live, bad | c, bad)
    return t1, t2, bad == 0, ref


def window_error_scale(sums: dict, r: np.ndarray, k: int) -> np.ndarray:
    """The block-local magnitude M that bounds the window variance's rounding error (the header's accuracy statement):
    M = (1/k) * sum over the window's block pieces of (the staged sum of d^2 at the piece's last row, plus the one
    before its first row when the piece does not start its block, plus, for pieces shifted to ref, |2 dl * p1| and
    n dl^2).  These are the magnitudes of every addend the window's sums are formed from.  (len(r), A)."""
    s1, s2, base = sums["s1"], sums["s2"], sums["base"]
    r = np.asarray(r, dtype=np.int64)
    lo, hi = r - k + 1, r
    bh, bl = hi // BLOCK, lo // BLOCK
    ref = base[bh]
    out = np.zeros_like(ref)
    for j in range(int((bh - bl).max()) + 1 if r.size else 0):
        live = (bh - j >= bl)[:, None]
        b = np.maximum(bh - j, bl)
        b0 = b * BLOCK
        e = hi if j == 0 else np.minimum(b0 + BLOCK - 1, hi)
        s0 = np.maximum(lo, b0)
        sub = (s0 > b0)[:, None]
        prev = np.maximum(s0 - 1, 0)
        p1 = np.where(sub, s1[e] - s1[prev], s1[e])
        mag = s2[e] + np.where(sub, s2[prev], 0.0)
        if j > 0:
            dl = base[b] - ref
            n = (e - s0 + 1).astype(np.float64)[:, None]
            mag = mag + 2.0 * np.abs(dl * p1) + n * dl * dl
        out = np.where(live, out + mag, out)
    return out / float(k)


def window_stats(closes, sums: dict, r: np.ndarray, k: int):
    """The mean and population standard deviation of the k closes ending at rows r, as the device forms them for
    BOLLINGER (mean = ref + t1 / k; sd = sqrt(max(t2 / k - (t1 / k)^2, 0))): for the accuracy checks."""
    t1, t2, ok, ref = window(sums, r, k)
    m = t1 / float(k)
    var = t2 / float(k) - m * m
    return ref + m, np.sqrt(np.where(var > 0.0, var, 0.0)), ok


def _lookback_ok(w) -> bool:
    return 1 <= int(w) <= MAX_LOOKBACK


def signs(rec, closes, sums: dict, rows=None) -> np.ndarray:
    """s in {-1, 0, +1} of one rule record at `rows`, (len(rows), A) int."""
    c = _closes(closes)
    T, A = c.shape
    r = np.arange(T, dtype=np.int64) if rows is None else np.asarray(rows, dtype=np.int64)
    out = np.zeros((r.size, A), dtype=np.int64)
    kind, w, w2, k = int(rec["kind"]), int(rec["lookback"]), int(rec["lookback2"]), float(rec["k"])
    if kind == CONST:
        out[:] = 1
    elif kind == MOMENTUM and _lookback_ok(w):
        m = r >= w
        c0, c1 = c[r[m]], c[r[m] - w]
        fin = np.isfinite(c0) & np.isfinite(c1)
        out[m] = np.where(fin, np.where(c0 > c1, 1, np.where(c0 < c1, -1, 0)), 0)
    elif kind == MA_CROSS and _lookback_ok(w) and _lookback_ok(w2) and w < w2:
        m = r >= w2 - 1
        f1, _, okf, _ = window(sums, r[m], w)
        l1, _, oks, _ = window(sums, r[m], w2)
        mf, ms = f1 / float(w), l1 / float(w2)
        out[m] = np.where(okf & oks, np.where(mf > ms, 1, np.where(mf < ms, -1, 0)), 0)
    elif kind == BOLLINGER and _lookback_ok(w) and w >= 2 and k > 0.0 and np.isfinite(k):
        m = r >= w - 1
        t1, t2, ok, ref = window(sums, r[m], w)
        n = float(w)
        mean = t1 / n
        var = t2 / n - mean * mean
        band = k * np.sqrt(np.where(var > 0.0, var, 0.0))
        x = c[r[m]] - ref
        out[m] = np.where(ok, np.where(x > mean + band, -1, np.where(x < mean - band, 1, 0)), 0)
    elif kind == XS_MOMENTUM and _lookback_ok(w) and 1 <= w2 <= A // 2:
        m = r >= w
        c0, c1 = c[r[m]], c[r[m] - w]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            q = c0 / c1
        ok = np.isfinite(c0) & np.isfinite(c1) & (c1 != 0.0) & np.isfinite(q)
        idx = np.arange(A)
        # rank[a] = #{b ranked : q_b > q_a, or q_b == q_a and b < a}
        beats = ok[:, :, None] & ((q[:, :, None] > q[:, None, :]) |
                                  ((q[:, :, None] == q[:, None, :]) & (idx[:, None] < idx[None, :])))
        rank = beats.sum(axis=1)
        cnt = ok.sum(axis=1)[:, None]
        s = np.where(rank < w2, 1, np.where(rank >= cnt - w2, -1, 0))
        out[m] = np.where(ok & (cnt >= 2 * w2), s, 0)
    return out


def values(rec, closes, sums: dict, rows=None) -> np.ndarray:
    """v = +size, -size or +0.0f (after long_only) of one rule at `rows`: (len(rows), A) float32."""
    s = signs(rec, closes, sums, rows)
    if int(rec["long_only"]):
        s = np.maximum(s, 0)
    size = np.float32(rec["size"])
    return np.where(s > 0, size, np.where(s < 0, -size, np.float32(0.0))).astype(np.float32)


def rule_table(records, closes, rows=None, sums: dict | None = None) -> np.ndarray:
    """fe_rule_table: (R, len(rows), A) float32."""
    sums = rule_sums(closes) if sums is None else sums
    return np.stack([values(rec, closes, sums, rows) for rec in np.atleast_1d(records)])
