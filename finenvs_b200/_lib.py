"""ctypes binding of libfinenvs_b200.so (the C ABI declared in include/finenvs_b200.h).

No torch types cross this boundary: tensors are passed as `data_ptr()` integers and the current
stream as its raw handle.  There is no fallback: if the shared library has not been built the
import fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfinenvs_b200.so")

RESET_KEEP, RESET_LAST, RESET_ALL = 0, 1, 2
VARIANT_AUTO, VARIANT_TILE, VARIANT_DIRECT, VARIANT_PORTFOLIO, VARIANT_PIPE, VARIANT_SPLIT, VARIANT_GATHER = 0, 1, 2, 3, 4, 6, 8
ABI_VERSION = 3


class FeParams(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int64),
        ("env_id_base", C.c_int64),
        ("total_envs", C.c_int64),
        ("num_rows", C.c_int64),
        ("window", C.c_int32),
        ("num_segments", C.c_int32),
        ("num_assets", C.c_int32),
        ("max_shares", C.c_int32),
        ("starting_balance", C.c_double),
        ("commission", C.c_double),
        ("imr", C.c_double),
        ("mmr", C.c_double),
        ("seed", C.c_uint64),
        ("reset_mode", C.c_int32),
        ("random_offset", C.c_int32),
        ("evaluate", C.c_int32),
        ("out_f64", C.c_int32),
        ("variant", C.c_int32),
        ("device", C.c_int32),
    ]


class FeSeries(C.Structure):
    _fields_ = [("prices", C.c_void_p), ("logret", C.c_void_p), ("seg_start", C.c_void_p), ("seg_len", C.c_void_p),
                ("obs_table", C.c_void_p)]


class FeState(C.Structure):
    _fields_ = [
        ("seg", C.c_void_p),
        ("ptr", C.c_void_p),
        ("cash", C.c_void_p),
        ("long_sh", C.c_void_p),
        ("short_sh", C.c_void_p),
        ("margin", C.c_void_p),
        ("terminated", C.c_void_p),
        ("ep_return", C.c_void_p),
        ("ep_len", C.c_void_p),
        ("sched", C.c_void_p),
    ]


FE_ES_MAX_LAYERS = 4


class FeEsNet(C.Structure):
    _fields_ = [("num_layers", C.c_int32), ("dims", C.c_int32 * (FE_ES_MAX_LAYERS + 1))]


# FeStats as a flat tensor: 4 x u64 then 2 x f64 = 48 bytes
STATS_BYTES = 48

# FeMetricsSummary as a flat tensor: 2 x u64 then 6 x f64 = 64 bytes
METRICS_SUMMARY_KEYS = ("episodes", "sum_len", "sum_return", "sum_sharpe", "sum_sharpe_sq", "sum_mdd", "max_mdd",
                        "sum_hit_rate")
METRICS_SUMMARY_BYTES = 64

# FE_TARGET_MAX_SHARES: the largest max_shares of a target-position backtest (the D -> action -> D round trip is exact)
TARGET_MAX_SHARES = 1 << 20


# rule backtests (include/finenvs_b200.h, "rule backtests"): FE_RULE_* kinds, the longest lookback, the staging block
RULE_CONST, RULE_MOMENTUM, RULE_MA_CROSS, RULE_BOLLINGER, RULE_XS_MOMENTUM = 0, 1, 2, 3, 4
RULE_MAX_LOOKBACK = 65536
RULE_BLOCK = 1024


class FeRule(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lookback", C.c_int32), ("lookback2", C.c_int32), ("long_only", C.c_int32),
                ("k", C.c_double), ("size", C.c_float), ("reserved", C.c_int32)]


class FeMetricsState(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in (
        "len", "pos", "sum", "mean", "m2", "peak", "mdd", "mdd_rel", "emitted",
        "fin_key", "fin_env", "fin_len", "fin_return", "fin_sharpe", "fin_mdd", "fin_mdd_rel", "fin_hit_rate", "summary")]

_PROTOTYPES = {
    "fe_version": (C.c_int, []),
    "fe_error_string": (C.c_char_p, [C.c_int]),
    "fe_tile_envs": (C.c_int, [C.c_int32, C.c_int32, C.c_int32]),
    "fe_pipe_envs": (C.c_int, [C.c_int32, C.c_int32, C.c_int32]),
    "fe_step_kernel_name": (C.c_char_p, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState)]),
    "fe_obs_table_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "fe_obs_table_build": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "fe_log_returns": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_effective_len": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                   C.c_void_p]),
    "fe_observe": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p]),
    "fe_step": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "fe_step_captured": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_step_host": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                               C.c_void_p]),
    "fe_step_host_packed": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                      C.c_void_p]),
    "fe_reset_all": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_uint64, C.c_int32,
                               C.c_void_p]),
    "fe_returns_advantages": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                        C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_observe_lazy": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "fe_step_lazy": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "fe_materialize": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_gather_obs": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                C.c_void_p, C.c_void_p]),
    "fe_gather_obs_kernel_name": (C.c_char_p, [C.POINTER(FeParams), C.POINTER(FeSeries)]),
    "fe_episode_metrics": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeMetricsState), C.c_void_p, C.c_void_p, C.c_uint64,
                                     C.c_void_p, C.c_int64, C.c_void_p]),
    "fe_backtest": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState), C.POINTER(FeMetricsState),
                              C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p,
                              C.c_void_p, C.c_int32, C.c_void_p]),
    "fe_backtest_targets": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState),
                                      C.POINTER(FeMetricsState), C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "fe_backtest_portfolio": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState),
                                        C.POINTER(FeMetricsState), C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_void_p, C.c_int32, C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_int32, C.c_void_p]),
    "fe_rule_sums_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "fe_rule_sums_build": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "fe_backtest_rules": (C.c_int, [C.POINTER(FeParams), C.POINTER(FeSeries), C.POINTER(FeState),
                                    C.POINTER(FeMetricsState), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_void_p]),
    "fe_rule_table": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                C.c_int32, C.c_void_p]),
    "fe_es_params_padded": (C.c_int64, [C.POINTER(FeEsNet)]),
    "fe_es_packed_index": (C.c_int64, [C.POINTER(FeEsNet), C.c_int32, C.c_int32, C.c_int32]),
    "fe_es_perturb": (C.c_int, [C.POINTER(FeEsNet), C.c_uint64, C.c_uint64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "fe_es_forward": (C.c_int, [C.POINTER(FeEsNet), C.c_void_p, C.c_void_p, C.c_float, C.c_int64, C.c_int64, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_uint64, C.c_uint64,
                                C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "fe_es_forward_kernel_name": (C.c_char_p, [C.POINTER(FeEsNet), C.c_int32, C.c_int32]),
    "fe_es_gradient_scratch": (C.c_int64, [C.POINTER(FeEsNet), C.c_int64]),
    "fe_es_gradient": (C.c_int, [C.POINTER(FeEsNet), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_es_store": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_void_p,
                              C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_philox": (None, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]),
    "fe_csv_open": (C.c_int, [C.c_char_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "fe_csv_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_csv_close": (None, [C.c_void_p]),
}

EXPORTS = tuple(_PROTOTYPES)

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
                "finenvs_b200 has no CPU or pure-PyTorch fallback."
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = L.fe_version()
        if got != ABI_VERSION:
            raise ImportError(f"libfinenvs_b200.so ABI {got} != binding ABI {ABI_VERSION}; rebuild")
        _lib = L
    return _lib


class FeError(RuntimeError):
    pass


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().fe_error_string(code)
        raise FeError(f"{what} failed ({code}): {msg.decode() if msg else '?'}")


def philox(seed: int, env_id: int, step: int, kind: int = 0):
    out = (C.c_uint32 * 4)()
    lib().fe_philox(seed, env_id, step, kind, out)
    return [int(x) for x in out]
