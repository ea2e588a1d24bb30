"""Portfolio backtests without a GPU: fe_backtest_portfolio's argument checks, each rejected with its code before any
CUDA call (a CUDA call on a machine without a device would return a positive CUDA error instead)."""
import ctypes

import pytest

from test_backtest_host import _params


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


NAMES = ("p", "s", "st", "m", "cap", "stats", "signal", "nsig", "col", "targets", "exits", "first", "steps", "rew", "done",
         "hist", "stream")


@pytest.fixture
def call(built):
    L = built.lib()
    keep = []

    def byref(x):
        keep.append(x)
        return ctypes.byref(x)

    good = dict(zip(NAMES, [byref(_params(built, assets=5)), byref(built.FeSeries(16, 16, 16, 16, None)),
                            byref(built.FeState(16, 16, 16, 16, 16, 16, None, 16, 16, None)),
                            byref(built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))), 8, None, 16, 4, 16, 1, None, 1,
                            10, 16, 16, 0, None]))

    def run(**over):
        args = dict(good)
        args.update({k: (byref(v) if isinstance(v, ctypes.Structure) else v) for k, v in over.items()})
        return L.fe_backtest_portfolio(*(args[n] for n in NAMES))

    return run


def test_null_pointers_and_sizes(built, call):
    for name in ("p", "s", "st", "m", "signal", "col", "rew", "done"):
        assert call(**{name: None}) == -1, name
    assert call(steps=0) == -1 and call(steps=-3) == -1
    assert call(nsig=0) == -1 and call(nsig=-1) == -1
    assert call(cap=-1) == -1
    assert call(p=_params(built, assets=5, num_envs=0)) == -1


def test_num_assets_range(built, call):
    assert call(p=_params(built, assets=0)) == -1
    assert call(p=_params(built, assets=33)) == -1
    assert call(p=_params(built, assets=-1)) == -1


def test_state_and_metrics_pointers(built, call):
    assert call(p=_params(built, assets=5, evaluate=1)) == -1                         # evaluate needs the terminated flags
    st_eval = built.FeState(16, 16, 16, 16, 16, 16, 16, 16, None, None)
    assert call(p=_params(built, assets=5, evaluate=1), st=st_eval) == -1            # ... and the emitted flags
    for field, _ in built.FeMetricsState._fields_:
        if field == "emitted":
            continue
        mm = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
        setattr(mm, field, None)
        assert call(m=mm) == -1, field
    st_no_len = built.FeState(16, 16, 16, 16, 16, 16, None, 16, None, None)
    assert call(st=st_no_len, stats=16) == -1                                         # stats outside evaluate: ep_len


def test_targets_and_exits(built, call):
    assert call(targets=0, exits=16) == -1                                            # exits need targets
    for ms in (0, -5, built.TARGET_MAX_SHARES + 1, 1 << 30):                          # trade mode does not check
        q = _params(built, assets=5)
        q.max_shares = ms
        assert call(p=q, targets=1) == -1, ms
        assert call(p=q, targets=1, exits=16) == -1, ms
    q = _params(built, assets=5)
    q.max_shares = built.TARGET_MAX_SHARES
    assert call(p=q, targets=1, exits=12) == -2                                       # accepted max_shares, misaligned
    for bad in (4, 12, 20):
        assert call(targets=1, exits=bad) == -2, bad
    assert call(targets=0, exits=4) == -1                                             # exits without targets first


def test_alignment(built, call):
    assert call(s=built.FeSeries(8, 16, 16, 16, None)) == -2
    assert call(s=built.FeSeries(16, 8, 16, 16, None)) == -2
