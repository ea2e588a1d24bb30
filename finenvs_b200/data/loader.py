"""Series loader and one-time HBM staging.

Replaces the reference's loader (finenvs/environments/time_series_env.py:80-216) with a vectorised
pass that produces the FLAT layout the step kernel reads:

    prices   (T, 4) f64   O,H,L,C of every kept bar                        (:169-177)
    logret   (T, 4) f32|f64   100*log-returns, computed on the GPU          (:179-194)
    seg_start (D,) i64    first row of segment d = first bar of the day - W history rows (:141-152)
    seg_len   (D,) i32    rows of segment d, with the NaN end-of-day probe folded in (:486-496)

instead of the reference's two NaN-padded, history-duplicating (D, L, 4) tensors (:196-216).  Row j
of the reference's `*_environments[d]` is row `seg_start[d] + j` here.  The O(D*T) per-day boolean
scans of :127-152 become one first/last-occurrence pass over the Date column.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from glob import glob

import numpy as np
import torch

from .. import _lib

MARKET_OPEN_S = (9 * 60 + 30) * 60   # between_time("9:30", "15:59") :90-91, both ends inclusive
MARKET_CLOSE_S = (15 * 60 + 59) * 60

PACKAGE_DATA_DIR = os.path.dirname(os.path.abspath(__file__))


# ----------------------------------------------------------------------------- file lookup ----
def get_data_dir_name(data_dir_name: str) -> str:
    """:47-51 — a name containing "data" is used verbatim as a path, anything else names an
    instrument directory under the package data dir (or $FINENVS_DATA_DIR)."""
    if "data" not in data_dir_name:
        base = os.environ.get("FINENVS_DATA_DIR", PACKAGE_DATA_DIR)
        data_dir_name = os.path.join(base, data_dir_name)
    return data_dir_name


def determine_file_key(key_attempt: str) -> str:
    """:53-58"""
    possible_keys = ["dummy", "train", "valid", "test"]
    for possible_key in possible_keys:
        if possible_key in key_attempt:
            return possible_key
    raise Exception("dataset_key expected to be one of: " + str(possible_keys))


def find_file_by_key(data_dir_name: str, key_string: str) -> str:
    """:60-73 — exactly one `*<key>*.csv` must exist."""
    filenames = glob(os.path.join(data_dir_name, "*" + key_string + "*.csv"))
    if len(filenames) == 0:
        raise Exception(f"No file was found in {data_dir_name} with key ({key_string})")
    if len(filenames) > 1:
        raise Exception(f"More than one file was found in {data_dir_name} with key ({key_string})")
    return filenames[0]


# ----------------------------------------------------------------------------- host tables ----
@dataclass
class HostSeries:
    prices: np.ndarray       # (T, 4) f64
    seg_start: np.ndarray    # (D,) i64
    seg_len_raw: np.ndarray  # (D,) i32 = W + bars of the day


def _seconds_of_day(times) -> np.ndarray:
    """Seconds since midnight of "HH:MM[:SS]" strings.  A trading file has at most a few thousand DISTINCT times:
    they are factorised (one hash pass) and only the distinct strings are parsed."""
    import pandas as pd

    codes, uniques = pd.factorize(times)
    parts = pd.Series(uniques).astype(str).str.split(":", expand=True)
    secs = parts[0].astype(np.int64) * 3600 + parts[1].astype(np.int64) * 60
    if parts.shape[1] > 2:
        secs = secs + parts[2].fillna(0).astype(float).astype(np.int64)
    return secs.to_numpy()[codes]


def _first_last_rows(dates: np.ndarray):
    """First and last row of every distinct value of `dates`, in order of first appearance."""
    n = len(dates)
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    if dates.dtype.kind in "iu":
        # integer keys (the native reader's date hashes): days are runs of equal keys; one comparison pass finds them
        starts = np.flatnonzero(np.concatenate(([True], dates[1:] != dates[:-1])))
        if len(np.unique(dates[starts])) == len(starts):       # every day is ONE run (any normal file)
            return starts.astype(np.int64), np.concatenate((starts[1:] - 1, [n - 1])).astype(np.int64)
        _, first, inv = np.unique(dates, return_index=True, return_inverse=True)   # a date that comes back later
        last = np.zeros(len(first), np.int64)
        np.maximum.at(last, inv, np.arange(n, dtype=np.int64))
        order = np.argsort(first, kind="stable")
        return first[order].astype(np.int64), last[order]
    import pandas as pd

    inv, uniques = pd.factorize(dates)          # codes in order of first appearance
    idx = np.arange(n, dtype=np.int64)
    first = np.full(len(uniques), n, dtype=np.int64)
    last = np.zeros(len(uniques), dtype=np.int64)
    np.minimum.at(first, inv, idx)
    np.maximum.at(last, inv, idx)
    return first, last


def segment_table(dates: np.ndarray, window: int):
    """First/last row of every distinct Date (:141-152), backtracked by W rows of history; days
    whose history would start before row 0 are skipped (:134).  Order = first appearance.  One pass over the
    rows (the reference scans the whole frame once per day)."""
    first, last = _first_last_rows(np.asarray(dates))
    start = first - window
    keep = start >= 0
    return start[keep], (last[keep] - start[keep] + 1).astype(np.int32)


FE_ECSV = -5   # include/finenvs_b200.h: a record outside the native reader's format


def read_csv_native(path: str, num_threads: int = 0):
    """The CSV through the library's memory-mapped multi-threaded reader (csrc/fe_csv.cu, fe_csv_open / fe_csv_read):
    (date_key (T,) i64, sec_of_day (T,) i32, ohlc (T, 4) f64), prices bit-identical to pandas.read_csv's, or None when
    the file uses CSV syntax the native reader does not handle (quotes, header lines, missing values, other time formats)."""
    import ctypes as C

    L = _lib.lib()
    handle, rows = C.c_void_p(), C.c_int64()
    _lib.check(L.fe_csv_open(os.fsencode(path), num_threads, C.byref(handle), C.byref(rows)), f"fe_csv_open({path})")
    try:
        T = rows.value
        date_key = np.empty(T, np.int64)
        secs = np.empty(T, np.int32)
        ohlc = np.empty((T, 4), np.float64)
        rc = L.fe_csv_read(handle, date_key.ctypes.data, secs.ctypes.data, ohlc.ctypes.data)
    finally:
        L.fe_csv_close(handle)
    if rc == FE_ECSV:
        return None
    _lib.check(rc, "fe_csv_read")
    return date_key, secs, ohlc


def read_csv_pandas(path: str):
    """The reference's own reader (:80-88): same three arrays as read_csv_native, dates as strings."""
    import pandas as pd

    df = pd.read_csv(path, names=["Date", "Time", "Open", "High", "Low", "Close", "Volume"])
    return (df["Date"].to_numpy(), _seconds_of_day(df["Time"]),
            np.ascontiguousarray(df[["Open", "High", "Low", "Close"]].to_numpy(dtype=np.float64)))


def read_market_csv(path: str, window: int, reader: str = "auto") -> HostSeries:
    """read_data :80-88 + force_market_hours :90-91 + determine_environment_bounds :127-152.
    reader: "native" (fe_csv_*; raises on syntax it does not handle), "pandas", or "auto" (native, pandas for such files)."""
    if reader not in ("auto", "native", "pandas"):
        raise ValueError("reader must be 'auto', 'native' or 'pandas'")
    cols = read_csv_native(path) if reader != "pandas" else None
    if cols is None:
        if reader == "native":
            raise Exception(f"{path}: CSV syntax outside the native reader's format (use reader='pandas')")
        cols = read_csv_pandas(path)
    dates, secs, ohlc = cols
    keep = (secs >= MARKET_OPEN_S) & (secs <= MARKET_CLOSE_S)
    prices = np.ascontiguousarray(ohlc[keep])
    seg_start, seg_len_raw = segment_table(dates[keep], window)
    if len(seg_start) == 0:
        raise Exception(f"{path}: no trading day has {window} bars of history before it")
    return HostSeries(prices, seg_start, seg_len_raw)


def regular_segments(num_rows: int, bars_per_segment: int, window: int):
    """Segment table for a synthetic series cut into equal days (BASELINE configs 2-5)."""
    firsts = np.arange(0, num_rows - bars_per_segment + 1, bars_per_segment, dtype=np.int64)
    start = firsts - window
    keep = start >= 0
    start = start[keep]
    return start, np.full(len(start), window + bars_per_segment, dtype=np.int32)


# ---------------------------------------------------------------------------------- staging ----
@dataclass
class StagedSeries:
    """The series resident in HBM (device tensors) + the small host-side facts about it."""

    prices: torch.Tensor      # (T, 4) f64, or (T, A, 4) time-major for an A-asset portfolio
    logret: torch.Tensor      # same shape, f32 or f64 (matches the observation dtype)
    seg_start: torch.Tensor   # (D,) i64
    seg_len: torch.Tensor     # (D,) i32 effective
    seg_len_raw: torch.Tensor  # (D,) i32
    window: int
    logret64: torch.Tensor | None = None  # kept only when asked (loader parity tests)
    _obs_table: torch.Tensor | None = None  # observation-layout table of the gather kernel (built on first use)
    _obs_table_tried: bool = False
    _rule_sums: torch.Tensor | None = None  # running sums of the closes for device-side rules (built on first use)

    @property
    def num_rows(self) -> int:
        return int(self.prices.shape[0])

    @property
    def num_segments(self) -> int:
        return int(self.seg_start.shape[0])

    @property
    def num_assets(self) -> int:
        return 1 if self.prices.dim() == 2 else int(self.prices.shape[1])

    @property
    def device(self) -> torch.device:
        return self.prices.device

    def nbytes(self) -> int:
        extra = sum(t.numel() for t in (self._obs_table, self._rule_sums) if t is not None)
        return extra + sum(t.numel() * t.element_size() for t in (self.prices, self.logret, self.seg_start, self.seg_len))

    # the table only pays while it stays L2-resident beside the observation stream (csrc/fe_step.cu: gather_table_resident)
    OBS_TABLE_MAX_BYTES = 64 << 20

    def obs_table(self) -> torch.Tensor | None:
        """The log-returns in OBSERVATION layout (5 values per row, shifted copies so that every window start is
        16-byte aligned) that the gather kernel's TMA gather4 reads — replaces the per-step (N, L, 4) gather + cat of
        time_series_env.py:423-445 on the read side.  Built once per series on first use (fe_obs_table_build); None for
        multi-asset series, windows that are not a legal TMA row, or series too long for the table to stay in L2."""
        if self._obs_table_tried:
            return self._obs_table
        self._obs_table_tried = True
        if self.num_assets != 1:
            return None
        L = _lib.lib()
        f64 = int(self.logret.dtype == torch.float64)
        nbytes = int(L.fe_obs_table_bytes(self.num_rows, self.window, f64))
        if nbytes == 0 or nbytes > self.OBS_TABLE_MAX_BYTES:
            return None
        with torch.cuda.device(self.device):
            table = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            _lib.check(L.fe_obs_table_build(self.logret.data_ptr(), self.num_rows, self.window, f64, table.data_ptr(),
                                            torch.cuda.current_stream(self.device).cuda_stream), "fe_obs_table_build")
        self._obs_table = table
        return table

    def rule_sums(self) -> torch.Tensor:
        """Per asset, block-local running sums of the closes and their squares (include/finenvs_b200.h, "rule
        backtests"), from which the device evaluates moving-average and band rules in O(1 + lookback / 1024) loads
        per value.  Built once per series on first use (fe_rule_sums_build): fe_rule_sums_bytes(T, A) bytes, about 20
        per row and asset."""
        if self._rule_sums is None:
            L = _lib.lib()
            T, A = self.num_rows, self.num_assets
            with torch.cuda.device(self.device):
                sums = torch.empty(int(L.fe_rule_sums_bytes(T, A)), dtype=torch.uint8, device=self.device)
                _lib.check(L.fe_rule_sums_build(self.prices.data_ptr(), T, A, sums.data_ptr(), self.device.index,
                                                torch.cuda.current_stream(self.device).cuda_stream), "fe_rule_sums_build")
            self._rule_sums = sums
        return self._rule_sums


def stage_series(prices, seg_start, seg_len_raw, window: int, device: str, obs_dtype=torch.float32,
                 keep_logret64: bool = False) -> StagedSeries:
    """Upload OHLC once (pinned staging buffer -> HBM), derive log-returns and the effective segment
    lengths on the GPU (fe_log_returns / fe_effective_len)."""
    L = _lib.lib()
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("stage_series needs a CUDA device (no CPU path)")
    prices_h = torch.as_tensor(np.ascontiguousarray(prices, dtype=np.float64)) if not torch.is_tensor(prices) else prices
    if prices_h.dim() not in (2, 3) or prices_h.shape[-1] != 4:
        raise ValueError(f"prices must be (T, 4) or (T, A, 4) O,H,L,C; got {tuple(prices_h.shape)}")
    T = int(prices_h.shape[0])
    A = 1 if prices_h.dim() == 2 else int(prices_h.shape[1])
    if not 1 <= A <= 32:
        raise ValueError("1 <= num_assets <= 32")
    seg_start_h = torch.as_tensor(np.ascontiguousarray(seg_start, dtype=np.int64))
    raw_h = torch.as_tensor(np.ascontiguousarray(seg_len_raw, dtype=np.int32))
    if seg_start_h.numel() == 0:
        raise ValueError("empty segment table")
    if int(seg_start_h.min()) < 0 or int((seg_start_h + raw_h.long()).max()) > T:
        raise ValueError("segment table reaches outside the series")
    if int(raw_h.min()) < window + 1:
        raise ValueError("every segment needs W history rows plus at least one bar")
    with torch.cuda.device(dev):
        if prices_h.device.type == "cpu":
            prices_d = prices_h.to(torch.float64).contiguous().pin_memory().to(dev, non_blocking=True)
        else:
            prices_d = prices_h.to(dev, torch.float64).contiguous()
        seg_start_d = seg_start_h.to(dev)
        raw_d = raw_h.to(dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        lr64 = torch.empty(prices_d.shape, dtype=torch.float64, device=dev)
        want32 = obs_dtype == torch.float32
        lr32 = torch.empty(prices_d.shape, dtype=torch.float32, device=dev) if want32 else None
        _lib.check(L.fe_log_returns(prices_d.data_ptr(), T, A, lr64.data_ptr(), lr32.data_ptr() if want32 else None,
                                    stream), "fe_log_returns")
        seg_len_d = torch.empty_like(raw_d)
        _lib.check(L.fe_effective_len(lr64.data_ptr(), seg_start_d.data_ptr(), raw_d.data_ptr(), raw_d.numel(), window, A,
                                      seg_len_d.data_ptr(), stream), "fe_effective_len")
        torch.cuda.current_stream(dev).synchronize()
    logret = lr32 if want32 else lr64
    return StagedSeries(prices_d, logret, seg_start_d, seg_len_d, raw_d, window,
                        lr64 if (keep_logret64 or not want32) else None)
