"""Target-position backtests without a GPU: fe_backtest_targets' argument checks (rejected before any CUDA call) and the
exact round trip share delta D -> action D / scale -> rint(action * scale) = D that makes a target backtest equal to
stepping with the caller's actions."""
import ctypes

import numpy as np
import pytest

from test_backtest_host import _params


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def test_backtest_targets_argument_errors(built):
    L = built.lib()
    p = _params(built)
    s = built.FeSeries(16, 16, 16, 16, None)
    st = built.FeState(16, 16, 16, 16, 16, 16, None, 16, 16, None)
    m = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
    P, S, ST, M = (ctypes.byref(x) for x in (p, s, st, m))
    names = ("p", "s", "st", "m", "cap", "stats", "signal", "nsig", "col", "exits", "first", "steps", "rew", "done",
             "hist", "stream")
    good = [P, S, ST, M, 8, None, 16, 4, 16, 16, 1, 10, 16, 16, 0, None]

    def call(**over):
        args = dict(zip(names, good))
        args.update(over)
        return L.fe_backtest_targets(*(args[n] for n in names))

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
    for field, _ in built.FeMetricsState._fields_:
        if field == "emitted":
            continue
        mm = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
        setattr(mm, field, None)
        assert call(m=ctypes.byref(mm)) == -1, field
    st_no_len = built.FeState(16, 16, 16, 16, 16, 16, None, 16, None, None)
    assert call(st=ctypes.byref(st_no_len), stats=16) == -1
    # max_shares outside [1, FE_TARGET_MAX_SHARES]: the round trip below is proven for that range only
    for ms in (0, -5, built.TARGET_MAX_SHARES + 1, 1 << 30):
        q = _params(built)
        q.max_shares = ms
        assert call(p=ctypes.byref(q)) == -1, ms
    q = _params(built)
    q.max_shares = built.TARGET_MAX_SHARES
    # exits: NULL is "no exits"; a misaligned table is FE_EALIGN, as are misaligned series pointers
    assert call(p=ctypes.byref(q), exits=12) == -2
    assert call(exits=4) == -2 and call(exits=20) == -2
    assert call(s=ctypes.byref(built.FeSeries(8, 16, 16, 16, None))) == -2


def _round_trip(ms: int, D: np.ndarray) -> np.ndarray:
    """The kernel's operations in f32: a = D / scale (TargetRule), then rint(a * scale) (env_compute_core)."""
    scale = np.float32(float(ms) + 0.5)            # Consts::scale = (float)((double)max_shares + 0.5)
    with np.errstate(all="raise"):
        a = D / scale                              # __fdiv_rn
        return np.rint(a * scale)                  # __fmul_rn, rintf (half to even)


def _sample_max_shares():
    edges = [m for k in range(21) for m in (2 ** k - 1, 2 ** k, 2 ** k + 1) if 1 <= m <= 1 << 20]
    rng = np.random.default_rng(0)
    return sorted(set(range(1, 65)) | set(edges) | set(rng.integers(1, (1 << 20) + 1, 40).tolist()))


def test_delta_round_trip_is_exact():
    """rint(f32(f32(D / scale) * scale)) == D for every integer |D| <= 2^21, at every accepted max_shares.

    The proof: for 1 <= ms <= 2^20, ms + 0.5 needs at most 22 significant bits, so scale is exact in f32 (checked for
    every ms below).  Each of the two roundings has relative error <= u = 2^-24, so |rint argument - D| <= |D|(2u + u^2)
    < 0.26 < 0.5 for |D| <= 2^21, whatever the scale: rint returns D.  The exhaustive check over every D at a sample of
    max_shares (all of 1..64, every power of two and its neighbours, random ones) confirms the bound numerically."""
    ms_all = np.arange(1, (1 << 20) + 1, dtype=np.float64)
    assert np.array_equal(ms_all.astype(np.float32).astype(np.float64) + 0.5,
                          (ms_all + 0.5).astype(np.float32).astype(np.float64))
    u = 2.0 ** -24
    assert 2 ** 21 * (2 * u + u * u) < 0.5
    D = np.arange(-(1 << 21), (1 << 21) + 1, dtype=np.float32)
    assert np.array_equal(D.astype(np.int64), np.arange(-(1 << 21), (1 << 21) + 1))   # every integer is exact in f32
    for ms in _sample_max_shares():
        back = _round_trip(ms, D)
        bad = np.flatnonzero(back != D)
        assert bad.size == 0, (ms, D[bad[:4]], back[bad[:4]])


def test_large_deltas_still_clamp_to_max_shares():
    """Beyond 2^21 (a position that trade-mode steps built up past 2 x max_shares) the round trip may be off by a share,
    but never by enough to change the sign or bring |rint(a * scale)| below max_shares: the step's clamp gives +-ms."""
    rng = np.random.default_rng(1)
    D = np.concatenate([np.arange((1 << 21) + 1, (1 << 21) + 200_000), rng.integers(1 << 21, 1 << 40, 200_000)])
    D = np.concatenate([D, -D]).astype(np.float32)
    for ms in (1, 5, 1000, (1 << 20) - 1, 1 << 20):
        back = _round_trip(ms, D)
        assert np.array_equal(np.clip(back, -ms, ms), np.sign(D) * np.float32(ms)), ms
