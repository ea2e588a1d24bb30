"""Signal backtests without a GPU: fe_backtest's argument checks (rejected before any CUDA call) and the default mapping
of envs to signal columns."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def _params(lib, N=1 << 10, assets=1, evaluate=0, num_envs=None):
    return lib.FeParams(N if num_envs is None else num_envs, 0, N, 4096, 60, 16, assets, 5, 10000.0, 0.01, 1.5, 0.25, 1,
                        lib.RESET_KEEP if evaluate else lib.RESET_ALL, 0, evaluate, 0, lib.VARIANT_AUTO, 0)


def test_backtest_argument_errors(built):
    L = built.lib()
    p = _params(built)
    s = built.FeSeries(16, 16, 16, 16, None)
    st = built.FeState(16, 16, 16, 16, 16, 16, None, 16, 16, None)
    m = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
    P, S, ST, M = (ctypes.byref(x) for x in (p, s, st, m))
    # (p, s, st, m, capacity, stats, signal, num_signals, column, first_step, num_steps, rewards, dones, history, stream)
    good = [P, S, ST, M, 8, None, 16, 4, 16, 1, 10, 16, 16, 0, None]

    def call(**over):
        names = ("p", "s", "st", "m", "cap", "stats", "signal", "nsig", "col", "first", "steps", "rew", "done", "hist",
                 "stream")
        args = dict(zip(names, good))
        args.update(over)
        return L.fe_backtest(*(args[n] for n in names))

    for name in ("p", "s", "st", "m", "signal", "col", "rew", "done"):
        assert call(**{name: None}) == -1, name
    assert call(steps=0) == -1 and call(steps=-3) == -1
    assert call(nsig=0) == -1
    assert call(cap=-1) == -1
    assert call(p=ctypes.byref(_params(built, assets=2))) == -1            # portfolio envs are out of scope
    assert call(p=ctypes.byref(_params(built, num_envs=0))) == -1
    assert call(p=ctypes.byref(_params(built, evaluate=1))) == -1          # evaluate needs the terminated flags ...
    st_eval = built.FeState(16, 16, 16, 16, 16, 16, 16, 16, None, None)
    assert call(p=ctypes.byref(_params(built, evaluate=1)), st=ctypes.byref(st_eval)) == -1   # ... and the emitted flags
    for k, (field, _) in enumerate(built.FeMetricsState._fields_):
        if field == "emitted":
            continue
        mm = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
        setattr(mm, field, None)
        assert call(m=ctypes.byref(mm)) == -1, field
    # training-mode statistics need the running episode return and length
    st_no_len = built.FeState(16, 16, 16, 16, 16, 16, None, 16, None, None)
    assert call(st=ctypes.byref(st_no_len), stats=16) == -1
    # misaligned series pointers are FE_EALIGN, also before any CUDA call
    assert call(s=ctypes.byref(built.FeSeries(8, 16, 16, 16, None))) == -2


def test_default_columns_are_global_id_over_segments():
    from finenvs_b200.environments.time_series_env import default_signal_columns

    D, S = 7, 5
    whole = default_signal_columns(0, S * D, D, S)
    assert whole.dtype == torch.int32 and whole.tolist() == [g // D for g in range(S * D)]
    assert torch.bincount(whole.long()).tolist() == [D] * S    # every (strategy, day) pair is one env
    parts = torch.cat([default_signal_columns(0, 12, D, S), default_signal_columns(12, S * D - 12, D, S)])
    assert torch.equal(parts, whole)                            # shard-invariant


def test_default_columns_need_enough_signals():
    from finenvs_b200.environments.time_series_env import default_signal_columns

    assert default_signal_columns(0, 14, 7, 2).max().item() == 1
    with pytest.raises(ValueError, match="signal table has 2 rows"):
        default_signal_columns(0, 15, 7, 2)
    with pytest.raises(ValueError):
        default_signal_columns(14, 1, 7, 2)
