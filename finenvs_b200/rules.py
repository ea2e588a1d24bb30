"""Rule sets for TimeSeriesEnv.backtest_rules() / evaluate_rules() / rule_table(): classic trading rules evaluated on
the device from the staged closes, one rule per signal column, instead of a signal table built in torch.

A rule gives s in {-1, 0, +1} at every row r of the series (per asset in a portfolio), from the closes of rows <= r only;
long_only maps s to max(s, 0) and the value is s * size (an action, or with targets=True a target position).  The kinds
and their exact arithmetic are defined in include/finenvs_b200.h ("rule backtests"):

    constant(size=1.0)                  +1 everywhere (with targets=True buy-and-hold; size=-1: short-and-hold)
    momentum(w)                         sign(C[r] - C[r-w])
    ma_cross(fast, slow)                sign(mean of the last `fast` closes - mean of the last `slow` closes)
    bollinger(w, k)                     -1 above mean + k sd of the last w closes, +1 below mean - k sd, else 0
    xs_momentum(w, n)                   portfolios: +1 for the n assets with the largest C[r] / C[r-w], -1 for the n
                                        smallest, 0 for the others

Every builder takes scalars or arrays that broadcast elementwise (numpy rules), and flattens the result in C order, so
a grid is ma_cross(fast[:, None], slow[None, :]).  size= and long_only= broadcast with the parameters.  concat() joins
rule sets; column c of the result is rule c.  Values are checked here, before anything reaches the device.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib

CONST, MOMENTUM, MA_CROSS, BOLLINGER, XS_MOMENTUM = (_lib.RULE_CONST, _lib.RULE_MOMENTUM, _lib.RULE_MA_CROSS,
                                                     _lib.RULE_BOLLINGER, _lib.RULE_XS_MOMENTUM)
KIND_NAMES = {CONST: "constant", MOMENTUM: "momentum", MA_CROSS: "ma_cross", BOLLINGER: "bollinger",
              XS_MOMENTUM: "xs_momentum"}
MAX_LOOKBACK = _lib.RULE_MAX_LOOKBACK

# the FeRule record (include/finenvs_b200.h) as a numpy structured dtype
RECORD = np.dtype({"names": [f for f, _ in _lib.FeRule._fields_],
                   "formats": ["<i4", "<i4", "<i4", "<i4", "<f8", "<f4", "<i4"],
                   "offsets": [getattr(_lib.FeRule, f).offset for f, _ in _lib.FeRule._fields_],
                   "itemsize": ctypes.sizeof(_lib.FeRule)})


class RuleSet:
    """An array of rule records, one per signal column (`records`: a (R,) array of dtype RECORD)."""

    __slots__ = ("records",)

    def __init__(self, records: np.ndarray):
        records = np.ascontiguousarray(records)
        if records.dtype != RECORD or records.ndim != 1 or records.size < 1:
            raise ValueError("a RuleSet holds a non-empty 1-D array of rules.RECORD records")
        check_records(records)
        self.records = records

    def __len__(self) -> int:
        return int(self.records.size)

    def __repr__(self) -> str:
        kinds = np.bincount(self.records["kind"], minlength=len(KIND_NAMES))
        return "RuleSet(" + ", ".join(f"{n} {KIND_NAMES[k]}" for k, n in enumerate(kinds) if n) + ")"

    def needs_assets(self) -> int:
        """The fewest assets an env needs to run every rule of the set (xs_momentum with n needs 2n)."""
        xs = self.records["kind"] == XS_MOMENTUM
        return int(2 * self.records["lookback2"][xs].max()) if xs.any() else 1


def _ints(name: str, x, lo: int, hi: int) -> np.ndarray:
    a = np.asarray(x)
    if a.dtype == bool or not (np.issubdtype(a.dtype, np.integer) or
                               (np.issubdtype(a.dtype, np.floating) and np.all(np.isfinite(a)) and
                                np.all(a == np.round(a)))):
        raise ValueError(f"{name} must be integers in [{lo}, {hi}]; got {x!r}")
    if a.size and (a.min() < lo or a.max() > hi):
        raise ValueError(f"{name} must be integers in [{lo}, {hi}]; got values in [{a.min()}, {a.max()}]")
    return a.astype(np.int64)


def _build(kind: int, size, long_only, lookback=0, lookback2=0, k=0.0) -> RuleSet:
    size_a = np.asarray(size, dtype=np.float64)
    if not np.all(np.isfinite(size_a)) or np.any(np.abs(size_a) > np.finfo(np.float32).max):
        raise ValueError(f"size must be finite float32 values; got {size!r}")
    lo_a = np.asarray(long_only)
    if lo_a.dtype != bool and not np.issubdtype(lo_a.dtype, np.integer):
        raise ValueError(f"long_only must be booleans; got {long_only!r}")
    arrays = np.broadcast_arrays(np.asarray(lookback), np.asarray(lookback2), np.asarray(k, dtype=np.float64), size_a,
                                 lo_a)
    rec = np.zeros(arrays[0].size, dtype=RECORD)
    rec["kind"] = kind
    rec["lookback"], rec["lookback2"], rec["k"] = (a.ravel() for a in arrays[:3])
    rec["size"] = arrays[3].ravel().astype(np.float32)
    rec["long_only"] = arrays[4].ravel() != 0
    return RuleSet(rec)


def constant(size=1.0, *, long_only=False) -> RuleSet:
    """s = +1 at every row (every asset)."""
    return _build(CONST, size, long_only)


def momentum(w, *, size=1.0, long_only=False) -> RuleSet:
    """s = sign(C[r] - C[r-w]), 1 <= w <= MAX_LOOKBACK; 0 when equal, for a non-finite close, or while r < w."""
    return _build(MOMENTUM, size, long_only, lookback=_ints("w", w, 1, MAX_LOOKBACK))


def ma_cross(fast, slow, *, size=1.0, long_only=False) -> RuleSet:
    """s = sign(M_fast - M_slow), M_k the mean of the last k closes (rows r-k+1 .. r), 1 <= fast < slow <=
    MAX_LOOKBACK; 0 when equal, while r < slow - 1, or when the slow window holds a non-finite close."""
    f = _ints("fast", fast, 1, MAX_LOOKBACK - 1)
    sl = _ints("slow", slow, 2, MAX_LOOKBACK)
    if np.any(np.broadcast_to(f, np.broadcast_shapes(f.shape, sl.shape)) >= sl):
        raise ValueError("ma_cross needs fast < slow")
    return _build(MA_CROSS, size, long_only, lookback=f, lookback2=sl)


def bollinger(w, k, *, size=1.0, long_only=False) -> RuleSet:
    """Fade the band: s = -1 when C[r] > M_w + k sd_w, +1 when C[r] < M_w - k sd_w, else 0 (sd_w the population
    standard deviation of the last w closes), 2 <= w <= MAX_LOOKBACK, k finite and > 0."""
    kk = np.asarray(k, dtype=np.float64)
    if not np.all(np.isfinite(kk) & (kk > 0)):
        raise ValueError(f"k must be finite and > 0; got {k!r}")
    return _build(BOLLINGER, size, long_only, lookback=_ints("w", w, 2, MAX_LOOKBACK), k=kk)


def xs_momentum(w, n, *, size=1.0, long_only=False) -> RuleSet:
    """Portfolios: rank the assets by C_a[r] / C_a[r-w] (descending, ties to the lower asset index); s = +1 for the first
    n, -1 for the last n, 0 otherwise.  1 <= w <= MAX_LOOKBACK, n >= 1; the env needs at least 2n assets.  An asset
    whose ratio is not finite (a non-finite close, or C_a[r-w] == 0) gets 0 and is not ranked; with fewer than 2n
    ranked assets every asset gets 0."""
    return _build(XS_MOMENTUM, size, long_only, lookback=_ints("w", w, 1, MAX_LOOKBACK), lookback2=_ints("n", n, 1, 16))


def concat(*sets: RuleSet) -> RuleSet:
    """One rule set of the given sets' rules, in order."""
    if not sets or not all(isinstance(s, RuleSet) for s in sets):
        raise ValueError("concat takes one or more RuleSets")
    return RuleSet(np.concatenate([s.records for s in sets]))


def check_records(rec: np.ndarray, num_assets: int | None = None) -> None:
    """Refuse records the device would evaluate to 0 because a field is out of range (the kernels are total, but such a
    record is a mistake), and, for an env of num_assets assets, rules it cannot run."""
    kind, w, w2, k = rec["kind"], rec["lookback"], rec["lookback2"], rec["k"]

    def bad(mask, what):
        if np.any(mask):
            c = int(np.flatnonzero(mask)[0])
            raise ValueError(f"rule {c} ({KIND_NAMES.get(int(kind[c]), f'kind {int(kind[c])}')}): {what}")

    bad(~np.isin(kind, list(KIND_NAMES)), f"unknown kind (one of {sorted(KIND_NAMES)})")
    uses_w = kind != CONST
    bad(uses_w & ((w < 1) | (w > MAX_LOOKBACK)), f"lookback outside [1, {MAX_LOOKBACK}]")
    bad((kind == MA_CROSS) & ((w2 <= w) | (w2 > MAX_LOOKBACK)), f"slow lookback outside [fast + 1, {MAX_LOOKBACK}]")
    bad((kind == BOLLINGER) & (w < 2), "w must be >= 2")
    bad((kind == BOLLINGER) & ~(np.isfinite(k) & (k > 0)), "k must be finite and > 0")
    bad((kind == XS_MOMENTUM) & (w2 < 1), "n must be >= 1")
    bad(~np.isfinite(rec["size"]), "size must be finite")
    bad(~np.isin(rec["long_only"], (0, 1)), "long_only must be 0 or 1")
    bad(rec["reserved"] != 0, "reserved must be 0")
    if num_assets is not None:
        xs = kind == XS_MOMENTUM
        if num_assets == 1:
            bad(xs, "xs_momentum needs a portfolio env (num_assets >= 2)")
        bad(xs & (w2 > num_assets // 2), f"n must be <= num_assets / 2 = {num_assets // 2}")
