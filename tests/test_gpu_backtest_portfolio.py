"""Portfolio signal backtests (backtest_portfolio / evaluate_portfolio_signal, fe_backtest_portfolio_kernel in
csrc/fe_step.cu) against the step loop they replace: read the A table values from the env's state, turn them into actions
(trade mode: the values; target mode: per-asset share deltas in the same f32 / f64 operations), step_into.  Bit for bit on
an adversarial series (margin calls, bankruptcies, entries the shared cash cannot pay for), the A = 1 cross-check against
backtest(), composition, the numpy oracle, known answers, the evaluate report, sharding, overflow, argument checks and
the c3 population at full size."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import oracle_metrics as om
from parity_utils import gbm_ohlc
from test_gpu_backtest import _assert_same, _bits, _columns, _env
from test_gpu_backtest import _series as _series1
from test_gpu_backtest import _signal as _signal1
from test_gpu_backtest_targets import _exits
from test_gpu_episode_metrics import _assert_records_equal, _np

W = 8
MODES = ("trade", "targets", "exits")


def _series(A, dtype, seed=5, window=W, logret64=False):
    """A assets at sigma = 0.15 per bar (margin calls, bankruptcies) on 120 ragged days of 1..59 bars.  Prices start at
    300 .. 1320, so max_shares of every asset costs more than the 10 000 of cash: entries are blocked and retried."""
    from finenvs_b200.data import loader

    rng = np.random.default_rng(seed)
    bars = rng.integers(1, 60, 120)
    T = int(bars.sum()) + window
    prices = np.stack([np.round(gbm_ohlc(rng, T, 0.15, s0=300.0 + 170.0 * (a % 7)), 4) for a in range(A)], axis=1)
    firsts = window + np.concatenate([[0], np.cumsum(bars)[:-1]])
    seg_start, seg_len = firsts - window, (bars + window).astype(np.int32)
    series = loader.stage_series(prices, seg_start, seg_len, window, "cuda:0", dtype, keep_logret64=logret64)
    return series, (prices, seg_start, seg_len)


def _signal(S, T, A, seed=11):
    """(S, T, A) f32 values, 60 % negative, 10 % exact zeros, some beyond [-1, 1]."""
    return _signal1(S, T * A, seed).view(S, T, A)


def _lookup(env, signal, cols):
    rows = env.series.seg_start[env._seg.long()] + env._ptr.long() + env.num_intervals - 1
    return signal[cols.long(), rows]   # (N, A)


def _actions(env, signal, cols, mode, exits=None):
    """The header's definition from the env's state before the step: (N, A) actions and the exit mask (or None)."""
    v = _lookup(env, signal, cols)
    if mode == "trade":
        return v.contiguous(), None
    N, A = env.num_envs, env.num_assets
    ms = float(env.max_shares)
    scale = torch.tensor(ms + 0.5, dtype=torch.float32, device=v.device)
    T = torch.round(v * scale).clamp(-ms, ms)
    hit = None
    if exits is not None:
        total, peak = env._m_f64[0], env._m_f64[3]
        e = exits[cols.long()]
        hit = ((peak - total) >= e[:, 0]) | (total >= e[:, 1])
        T = torch.where(hit[:, None], torch.zeros_like(T), T)
    a = (T - (env._long - env._short).view(N, A)) / scale
    return a.contiguous(), hit


def _loop(env, signal, cols, K, mode="trade", exits=None):
    """K x (actions -> step_into -> fe_episode_metrics): (K, N) rewards, dones, and the number of env-steps at which an
    exit flattened held positions."""
    N, A = env.num_envs, env.num_assets
    R = torch.empty((K, N), dtype=env.obs_dtype, device="cuda")
    D = torch.empty((K, N), dtype=torch.int32, device="cuda")
    obs = torch.empty((N, env.num_intervals, env.num_obs), dtype=env.obs_dtype, device="cuda")
    flattened = torch.zeros((), dtype=torch.int64, device="cuda")
    for t in range(K):
        a, hit = _actions(env, signal, cols, mode, exits)
        if hit is not None:
            held = ((env._long.view(N, A) != 0) | (env._short.view(N, A) != 0)).any(1)
            flattened += (hit & held).sum()
        env.step_into(a, obs, R[t], D[t])
    return R, D, int(flattened)


def _run(env, signal, K, cols, mode, exits=None, history=True):
    return env.backtest_portfolio(signal, K, cols, history=history, targets=mode != "trade",
                                  exits=exits if mode == "exits" else None)


def _check(A, dtype, reset, random_offset, evaluate, track_stats, K, mode, window=W, N=2003, S=6, seed=5):
    series, _ = _series(A, dtype, seed=seed, window=window)
    kw = dict(random_reset=reset, random_offset=random_offset, evaluate=evaluate, track_stats=track_stats,
              metrics_capacity=64 * N)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    sig, cols = _signal(S, series.num_rows, A), _columns(N, S)
    ex = _exits(S) if mode == "exits" else None
    for e in (a, b):   # trade-mode steps first: the run starts mid-episode with positions beyond max_shares
        _loop(e, sig, cols, 7)
    assert int(((a._long > a.max_shares) | (a._short > a.max_shares)).sum()) > 0
    out = _run(a, sig, K, cols, mode, ex)
    R, D, flattened = _loop(b, sig, cols, K, mode, ex)
    assert out["steps"] == K and out["rewards"].dtype == dtype
    assert torch.equal(_bits(out["rewards"]), _bits(R)) and torch.equal(out["dones"], D)
    _assert_same(a, b, f"A={A} K={K} {mode}")
    return D, flattened


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("K", [1, 5, 150])
@pytest.mark.parametrize("track_stats", [False, True])
@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("random_offset", [False, True])
@pytest.mark.parametrize("reset", ["keep", "last", "all"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_portfolio_backtest_equals_the_step_loop(dtype, reset, random_offset, evaluate, track_stats, K, mode):
    N = 2003   # not a multiple of the 8 envs (warps) of a block
    D, flattened = _check(5, dtype, reset, random_offset, evaluate, track_stats, K, mode, N=N)
    if K == 150:
        assert int(D.sum()) > 2 * N   # several episodes per env
        if mode == "exits":
            assert flattened > 0      # exits flattened held positions


@pytest.mark.gpu
@pytest.mark.parametrize("A,window,dtype,mode,evaluate", [
    (2, 8, torch.float32, "trade", False), (2, 8, torch.float64, "exits", True),
    (30, 128, torch.float32, "exits", False), (30, 128, torch.float64, "targets", True),
    (32, 16, torch.float32, "targets", False), (32, 16, torch.float64, "trade", True),
    (32, 60, torch.float32, "exits", True)])
def test_other_asset_counts_equal_the_step_loop(A, window, dtype, mode, evaluate):
    _check(A, dtype, "all", True, evaluate, True, 60, mode, window=window, N=777, seed=A + window)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_one_asset_equals_backtest(dtype, mode):
    """An (S, T, 1) table through backtest_portfolio (the warp-per-env kernel) equals the (S, T) table through backtest()
    (the thread-per-env kernel): two independent implementations of the same definition."""
    N, S, K = 3001, 6, 150
    series, _ = _series1(dtype)
    kw = dict(track_stats=True, metrics_capacity=64 * N)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    sig, cols = _signal1(S, series.num_rows), _columns(N, S)
    ex = _exits(S) if mode == "exits" else None
    oa = _run(a, sig[..., None].contiguous(), K, cols, mode, ex)
    ob = b.backtest(sig, K, cols, history=True, targets=mode != "trade", exits=ex)
    # equal values; a zero reward may differ in sign (the portfolio step sums the assets' rewards over the warp, and
    # -0.0 + 0.0 is +0.0), which changes nothing downstream: the state and metrics compare bit for bit
    assert torch.equal(oa["rewards"], ob["rewards"]) and torch.equal(oa["dones"], ob["dones"])
    _assert_same(a, b, f"A=1 {mode}")


@pytest.mark.gpu
def test_portfolio_backtests_compose_and_interleave_with_steps():
    N, S, A = 2003, 6, 5
    series, _ = _series(A, torch.float32, seed=6)
    sig, cols, ex = _signal(S, series.num_rows, A, seed=2), _columns(N, S, seed=4), _exits(S, seed=5)
    one, two, mixed, ref = (_env(series, N, track_stats=True) for _ in range(4))
    _run(one, sig, 70, cols, "exits", ex, history=False)
    _run(two, sig, 23, cols, "exits", ex, history=False)
    _run(two, sig, 47, cols, "exits", ex, history=False)
    _assert_same(two, one, "K1 + K2")
    obs = torch.empty((N, W, 5 * A), device="cuda")
    r, d = torch.empty(N, device="cuda"), torch.empty(N, dtype=torch.int32, device="cuda")
    for k in (5, 11, 1, 30):
        _run(mixed, sig, k, cols, "exits", ex, history=False)
        for _ in range(3):
            mixed.step_into(_actions(mixed, sig, cols, "exits", ex)[0], obs, r, d)
    _loop(ref, sig, cols, 5 + 11 + 1 + 30 + 4 * 3, "exits", ex)
    _assert_same(mixed, ref, "interleaved")


@pytest.mark.gpu
def test_portfolio_records_match_the_numpy_oracle():
    """oracle.OracleEnv (multi-asset feo_step_multi) stepped with target actions computed from its own state, the exits'
    running P&L and peak rebuilt from its rewards; records from oracle_metrics."""
    from oracle import oracle as orc

    N, S, K, A = 1024, 6, 160, 4
    series, (prices, seg_start, seg_len) = _series(A, torch.float64, seed=8, logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    env = _env(series, N, metrics_capacity=64 * N)
    ref = orc.OracleEnv(fs, num_envs=N, seed=9, reset_mode=orc.RESET_ALL, random_offset=True, out_f64=True)
    sig, cols, ex = _signal(S, series.num_rows, A, seed=5), _columns(N, S, seed=6), _exits(S, seed=7)
    sig_h, cols_h, ex_h = sig.cpu().numpy(), cols.cpu().numpy(), ex.cpu().numpy()
    out = env.backtest_portfolio(sig, K, cols, history=True, targets=True, exits=ex)
    scale = np.float32(5.5)
    run_sum, run_peak = np.zeros(N), np.zeros(N)
    R, Dn = np.empty((K, N)), np.empty((K, N), np.int32)
    blocked_before = np.zeros((N, A), bool)
    blocked = retried = margin_calls = bankrupt = exited = 0
    for t in range(K):
        seg0, ptr0 = ref.seg.copy(), ref.ptr.copy()
        v = sig_h[cols_h, fs.seg_start[seg0] + ptr0 + W - 1]                     # (N, A)
        T = np.clip(np.rint(v * scale), np.float32(-5), np.float32(5))
        hit = ((run_peak - run_sum) >= ex_h[cols_h, 0]) | (run_sum >= ex_h[cols_h, 1])
        T = np.where(hit[:, None], np.float32(0), T).astype(np.float32)
        delta = (T - (ref.long_sh - ref.short_sh)).astype(np.float32)
        a = (delta / scale).astype(np.float32)
        flat0 = (ref.long_sh == 0) & (ref.short_sh == 0)
        short0 = ref.short_sh.copy()
        bar = prices[fs.seg_start[seg0] + ptr0 + W]                             # (N, A, 4): the bar this step trades on
        _, R[t], Dn[t], _ = ref.step(a, want_obs=False)
        held = (Dn[t] == 0)[:, None]
        exited += int(np.sum(hit & ~flat0.all(1)))
        retried += int(np.sum(blocked_before & (delta != 0)))
        # an entry the shared cash could not pay for: the asset is still flat although its target asked for a position
        blocked_now = held & flat0 & (T != 0) & (ref.long_sh == 0) & (ref.short_sh == 0)
        blocked += int(np.sum(blocked_now))
        blocked_before = blocked_now
        margin_calls += int(np.sum((short0 > 0) & (delta == 0) & (bar[..., 1] > 1.2 * bar[..., 0])))
        bankrupt += int(np.sum((Dn[t] == 1) & (ptr0 + 1 + W < fs.seg_len[seg0])))
        run_sum = run_sum + R[t]
        run_peak = np.maximum(run_peak, run_sum)
        run_sum[Dn[t] == 1] = 0.0
        run_peak[Dn[t] == 1] = 0.0
    assert np.array_equal(out["rewards"].cpu().numpy(), R) and np.array_equal(out["dones"].cpu().numpy(), Dn)
    for key in ("seg", "ptr", "cash"):
        assert np.array_equal(getattr(ref, key), getattr(env, "_" + key).cpu().numpy().reshape(-1)), key
    assert np.array_equal(ref.long_sh.reshape(-1), env._long.cpu().numpy())
    assert np.array_equal(ref.short_sh.reshape(-1), env._short.cpu().numpy())
    assert np.array_equal(ref.margin.reshape(-1).view(np.int64), env._margin.cpu().numpy().view(np.int64))
    assert min(blocked, retried, bankrupt, margin_calls, exited) > 0, (blocked, retried, bankrupt, margin_calls, exited)
    rec, agg = om.episode_metrics(R, Dn, env.starting_balance)
    _assert_records_equal(_np(env.episode_metrics()), rec, "oracle")
    s = {k: v.item() for k, v in env.metrics_summary().items()}
    assert s["episodes"] == agg["episodes"] and s["max_mdd"] == agg["max_mdd"]


# ------------------------------------------------------------------ known answers on a 3-asset day series ----
W_D = 2
_DAYS = [[101.0, 103.0, 102.5], [99.0, 98.0, 97.25], [100.0, 100.0, 104.0]]
_SCALE = (4.0, 4.0, 5.0)                               # asset a's prices are _SCALE[a] x the day's
_COMM = float(np.float32(5.0) * np.float32(0.01))     # one asset's five shares of commission (f32 product, :363-365)
_CLOSE3 = float(np.float32(15.0) * np.float32(0.01))  # the closing commission on 3 x 5 shares (:288-289)


def _day_series3(dtype=torch.float64):
    """Days of three bars each with Open = previous Close (no overnight gaps), W = 2 history rows, three assets whose
    prices are _SCALE times the same path."""
    from finenvs_b200.data import loader

    closes = [100.0, 100.0]
    rows = [[100.0, 100.5, 99.5, 100.0], [100.0, 100.5, 99.5, 100.0]]
    for day in _DAYS:
        for c in day:
            o = closes[-1]
            rows.append([o, max(o, c) + 0.5, min(o, c) - 0.5, c])
            closes.append(c)
    one = np.array(rows)
    prices = np.stack([one * f for f in _SCALE], axis=1)   # (T, 3, 4)
    days = len(_DAYS)
    seg_start = np.array([3 * d for d in range(days)], dtype=np.int64)
    seg_len = np.full(days, W_D + 3, dtype=np.int32)
    return loader.stage_series(prices, seg_start, seg_len, W_D, "cuda:0", dtype), prices


def _pos(env):
    return (env._long - env._short).view(env.num_envs, env.num_assets)


@pytest.mark.gpu
def test_buy_and_hold_from_every_start():
    """Target +1 on every asset: every asset at max_shares after the first step, held to the last Close of the day,
    whatever the start offset; the episode return is the closed-form P&L."""
    series, prices = _day_series3()
    T = series.num_rows
    zeros = torch.zeros(9, dtype=torch.int32, device="cuda")
    table = torch.ones((1, T, 3), device="cuda")
    envs = []
    for _ in range(2):
        env = _env(series, 9, evaluate=True, random_reset=None, random_offset=True)
        env._seg.copy_(torch.arange(9, device="cuda", dtype=torch.int32) // 3)   # (day, offset) = (i // 3, i % 3)
        env._ptr.copy_(torch.arange(9, device="cuda", dtype=torch.int32) % 3)
        envs.append(env)
    first, env = envs
    first.backtest_portfolio(table, 1, zeros, targets=True)
    going_on = torch.arange(9, device="cuda") % 3 != 2   # offset 2 starts on the last bar: its episode ends at once
    assert bool((_pos(first)[going_on] == 5).all()) and bool((_pos(first)[~going_on] == 0).all())
    rep = env.evaluate_portfolio_signal(table, zeros, targets=True)
    ss = series.seg_start.cpu().numpy()
    want = [sum(5 * (prices[ss[i // 3] + W_D + 2, a, 3] - prices[ss[i // 3] + W_D + i % 3, a, 0]) for a in range(3))
            - 3 * _COMM - _CLOSE3 for i in range(9)]
    np.testing.assert_allclose(rep["metrics"]["return"].cpu().numpy(), want, rtol=1e-12)
    np.testing.assert_array_equal(rep["metrics"]["len"].cpu().numpy(), [3 - i % 3 for i in range(9)])


@pytest.mark.gpu
def test_an_entry_the_cash_cannot_pay_for_stays_flat_and_is_retried():
    """4 500 of cash pays for 5 shares of assets 0 and 1 (2 000 each at the first Open) but not then for asset 2
    (2 500): asset 2 stays flat on every step of the day although its target asks for 5 shares every time."""
    series, _ = _day_series3()
    env = _env(series, 3, random_reset=None, random_offset=False, starting_balance=4500.0)
    cols = torch.zeros(3, dtype=torch.int32, device="cuda")
    table = torch.ones((1, series.num_rows, 3), device="cuda")
    for t in range(2):
        before = _pos(env)[0].clone()
        env.backtest_portfolio(table, 1, cols, targets=True)
        assert _pos(env)[0].tolist() == [5.0, 5.0, 0.0], t
        assert float(before[2]) == 0.0   # the target (5) differs from the position: the entry is asked for again


@pytest.mark.gpu
def test_flip_takes_two_steps_per_asset():
    """+1 then -1 on day 0: every asset goes 5, 0 (the sell of the longs; the short entry sees no sell order), then
    short 5 on the third bar, which ends the day."""
    series, prices = _day_series3()
    sig = torch.full((1, series.num_rows, 3), -1.0, device="cuda")
    sig[0, W_D - 1] = 1.0
    env = _env(series, 3, random_reset=None, random_offset=False, starting_balance=20000.0, evaluate=True)
    cols = torch.zeros(3, dtype=torch.int32, device="cuda")
    net, rew = [], []
    for _ in range(3):
        out = env.backtest_portfolio(sig, 1, cols, history=True, targets=True)
        net.append(_pos(env)[0].tolist())
        rew.append(float(out["rewards"][0, 0]))
    O, C = prices[W_D:W_D + 3, :, 0], prices[W_D:W_D + 3, :, 3]
    assert net == [[5.0] * 3, [0.0] * 3, [0.0] * 3]   # the third step ends the day, which closes the shorts
    assert rew[0] == pytest.approx(5 * (C[0] - O[0]).sum() - 3 * _COMM, rel=1e-12)
    assert rew[1] == pytest.approx(-3 * _COMM, rel=1e-12)
    assert rew[2] == pytest.approx(-5 * (C[2] - O[2]).sum() - 3 * _COMM - _CLOSE3, rel=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["stop", "take"])
def test_portfolio_exit_flattens_every_asset_until_the_episode_ends(kind):
    """Day 1 falls on its first bar (a stop of 10 on the portfolio P&L triggers), day 0 rises (a take-profit of 4
    triggers): the next step sells every asset at the Open, the rest of the day pays nothing, and the next episode
    trades again."""
    series, prices = _day_series3()
    day = 1 if kind == "stop" else 0
    ex = torch.tensor([[10.0, math.inf]] if kind == "stop" else [[math.inf, 4.0]], dtype=torch.float64, device="cuda")
    env = _env(series, 3, random_reset=None, random_offset=False)
    cols = torch.zeros(3, dtype=torch.int32, device="cuda")
    table = torch.ones((1, series.num_rows, 3), device="cuda")
    r, d, pos = [], [], []
    for _ in range(6):
        out = env.backtest_portfolio(table, 1, cols, history=True, targets=True, exits=ex)
        r.append(float(out["rewards"][0, day]))
        d.append(int(out["dones"][0, day]))
        pos.append(_pos(env)[day].tolist())
    s0 = int(series.seg_start[day]) + W_D
    first = 5 * (prices[s0, :, 3] - prices[s0, :, 0]).sum() - 3 * _COMM
    assert (first < -10) if kind == "stop" else (first > 4)
    assert r[0] == pytest.approx(first, rel=1e-12) and pos[0] == [5.0] * 3
    assert r[1] == pytest.approx(-3 * _COMM, rel=1e-12) and pos[1] == [0.0] * 3 and r[2] == 0.0
    assert d == [0, 0, 1, 0, 0, 1]
    assert r[3] == r[0] and r[4] == r[1] and r[5] == 0.0


@pytest.mark.gpu
def test_evaluate_portfolio_signal_equals_evaluate_policy():
    N, S, A = 600, 3, 5
    series, _ = _series(A, torch.float32, seed=12)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    K = int(series.seg_len.max()) - W
    cols = _columns(N, S, seed=1)
    for seed in (21, 22):
        sig = _signal(S, series.num_rows, A, seed=seed)
        got = a.evaluate_portfolio_signal(sig, cols)
        want = b.evaluate_policy(lambda obs: _lookup(b, sig, cols).contiguous(), steps_per_replay=K)
        assert got["steps"] == want["steps"] == K
        assert list(got) == ["returns", "steps", "metrics"]
        assert torch.equal(_bits(got["returns"]), _bits(want["returns"]))
        _assert_records_equal(_np(got["metrics"]), _np(want["metrics"]), f"signal {seed}")
        assert a.metrics_summary()["episodes"].item() == 0 and int(a._m_emitted.sum()) == 0 and int(a._stats[1]) == 0
        assert a.step_count == b.step_count


@pytest.mark.gpu
def test_portfolio_shards_give_the_records_of_one_population():
    A = 3
    series, _ = _series(A, torch.float64, seed=13)
    D, S, K = series.num_segments, 7, 90
    N = S * D
    sig, ex = _signal(S, series.num_rows, A, seed=9), _exits(S, seed=3)
    whole = _env(series, N)
    whole.backtest_portfolio(sig, K, targets=True, exits=ex)
    parts = []
    for base, n in ((0, 411), (411, N - 411)):
        env = _env(series, n, env_id_base=base, total_envs=N)
        env.backtest_portfolio(sig, K, targets=True, exits=ex)
        parts.append(env.episode_metrics())
    cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    order = torch.argsort(cat["key"])
    _assert_records_equal(_np({k: v[order] for k, v in cat.items()}), _np(whole.episode_metrics()), "shards")
    ref = _env(series, N)   # the default columns: (strategy, day) = (gid // D, gid % D)
    _loop(ref, sig, torch.arange(N, device="cuda", dtype=torch.int32) // D, K, "exits", ex)
    _assert_same(whole, ref, "default columns")


@pytest.mark.gpu
def test_portfolio_overflow_is_counted_not_written():
    from finenvs_b200 import _lib

    N, S, K, cap, guard, A = 1024, 3, 120, 100, 64, 4
    series, _ = _series(A, torch.float32, seed=14)
    sig, cols = _signal(S, series.num_rows, A, seed=7), _columns(N, S, seed=8)
    env = _env(series, N, metrics_capacity=cap)
    out = env.backtest_portfolio(sig, K, cols, history=True)
    n = int(out["dones"].sum())
    assert n > cap and env.metrics_summary()["episodes"].item() == n
    with pytest.raises(RuntimeError, match="metrics_capacity"):
        env.episode_metrics()

    # raw ABI with guard entries behind the list
    env = _env(series, N)
    f64 = torch.zeros((6, N), dtype=torch.float64, device="cuda")
    i32 = torch.zeros((2, N), dtype=torch.int32, device="cuda")
    li = torch.full((2, cap + guard), -7, dtype=torch.int64, device="cuda")
    ll = torch.full((cap + guard,), -7, dtype=torch.int32, device="cuda")
    lf = torch.full((5, cap + guard), -7.0, dtype=torch.float64, device="cuda")
    summ = torch.zeros(8, dtype=torch.int64, device="cuda")
    st = _lib.FeMetricsState(i32[0].data_ptr(), i32[1].data_ptr(), *(f64[k].data_ptr() for k in range(6)), None,
                             li[0].data_ptr(), li[1].data_ptr(), ll.data_ptr(), *(lf[k].data_ptr() for k in range(5)),
                             summ.data_ptr())
    R = torch.empty((K, N), device="cuda")
    Dn = torch.empty((K, N), dtype=torch.int32, device="cuda")
    _lib.check(env._L.fe_backtest_portfolio(env._pp, env._ps, env._pst, ctypes.byref(st), cap, None, sig.data_ptr(), S,
                                            cols.data_ptr(), 0, None, 1, K, R.data_ptr(), Dn.data_ptr(), 1,
                                            env._stream()), "fe_backtest_portfolio")
    rec, agg = om.episode_metrics(R.cpu().numpy(), Dn.cpu().numpy(), env.starting_balance)
    assert summ[0].item() == agg["episodes"] == n
    assert (li[:, cap:] == -7).all() and (ll[cap:] == -7).all() and (lf[:, cap:] == -7.0).all()
    keys = li[0, :cap].cpu().numpy()
    pos = np.minimum(np.searchsorted(rec["key"], keys), rec["key"].size - 1)
    assert (rec["key"][pos] == keys).all() and np.unique(keys).size == cap
    got = {"key": keys, "env": li[1, :cap].cpu().numpy(), "len": ll[:cap].cpu().numpy(),
           **{k: lf[j, :cap].cpu().numpy() for j, k in enumerate(("return", "sharpe", "mdd", "mdd_rel", "hit_rate"))}}
    _assert_records_equal(got, {k: v[pos] for k, v in rec.items()}, "raw list")


@pytest.mark.gpu
def test_portfolio_argument_validation():
    from finenvs_b200.agents.PPO.buffer import Buffer

    N, S, A = 256, 2, 3
    series, _ = _series(A, torch.float32, seed=15)
    T = series.num_rows
    env = _env(series, N)
    cols = _columns(N, S)
    sig = _signal(S, T, A)
    ex = torch.ones((S, 2), dtype=torch.float64, device="cuda")
    for bad in (sig[:, :-1], sig[..., :-1], sig.double(), sig.cpu(), sig.transpose(1, 2).contiguous().transpose(1, 2),
                sig[:, :, 0], sig[None], torch.ones((S, T, A + 1), device="cuda")):
        with pytest.raises(ValueError):
            env.backtest_portfolio(bad, 3, cols)
    for bad in (cols + S, cols - cols - 1, cols[:-1], cols.float()):
        with pytest.raises(ValueError):
            env.backtest_portfolio(sig, 3, bad)
    with pytest.raises(ValueError):   # default columns: global id // 120 days reaches 2, S = 1 is too small
        env.backtest_portfolio(sig[:1].contiguous(), 3)
    with pytest.raises(ValueError):
        env.backtest_portfolio(sig, 0, cols)
    with pytest.raises(ValueError, match="targets"):
        env.backtest_portfolio(sig, 3, cols, exits=ex)
    for bad in (ex[:1], ex.float(), ex.cpu(), -ex, ex * math.nan):
        with pytest.raises(ValueError):
            env.backtest_portfolio(sig, 3, cols, targets=True, exits=bad.contiguous())
    with pytest.raises(RuntimeError, match="track_metrics"):
        _env(series, N, track_metrics=False).backtest_portfolio(sig, 3, cols)
    with pytest.raises(RuntimeError, match="evaluate"):
        env.evaluate_portfolio_signal(sig, cols)
    bound = _env(series, N)
    Buffer(2, 0.99, 0, capacity=4).bind_env(bound)
    with pytest.raises(RuntimeError, match="bind_env"):
        bound.backtest_portfolio(sig, 3, cols)
    big = _env(series, N, max_shares=(1 << 20) + 1)
    with pytest.raises(ValueError, match="max_shares"):
        big.backtest_portfolio(sig, 3, cols, targets=True)
    big.backtest_portfolio(sig, 3, cols)   # trade mode has no such bound
    assert env.step_count == 0 and env.metrics_summary()["episodes"].item() == 0   # nothing ran
    assert int(env._m_i32.abs().sum()) == 0


@pytest.mark.gpu
def test_full_size_c3():
    """c3 (30 assets, W = 128; 1023 days of 252 bars) with 64 cross-sectional momentum columns: 65 472 envs in evaluate
    mode, one full episode each, in all three modes.  The records equal the step loop's on a contiguous slice."""
    import bench
    from finenvs_b200.data import loader
    from tools.backtest_cost import portfolio_momentum_signal

    Wc, S, sl = 128, 64, 8192
    prices, seg_start, seg_len, _ = bench.make_series("c3", Wc)
    series = loader.stage_series(prices, seg_start, seg_len, Wc, "cuda:0", torch.float32)
    D, A = series.num_segments, series.num_assets
    assert (D, A) == (1023, 30)
    N = S * D
    sig = portfolio_momentum_signal(series, S)
    assert sig.shape == (S, series.num_rows, A)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    cols = torch.arange(N, device="cuda", dtype=torch.int32) // D
    g = torch.Generator(device="cuda").manual_seed(1)
    ex = (2.0 * torch.exp(torch.rand((S, 2), generator=g, device="cuda", dtype=torch.float64) * math.log(30.0)))
    lo = 20_000
    for mode in MODES:
        a = _env(series, N, **kw)
        rep = a.evaluate_portfolio_signal(sig, targets=mode != "trade", exits=ex if mode == "exits" else None)
        assert rep["steps"] == 252 and rep["metrics"]["key"].numel() == N
        b = _env(series, N, **kw)
        _loop(b, sig, cols, rep["steps"], mode, ex if mode == "exits" else None)
        want = b._first_episode_metrics()
        _assert_records_equal(_np({k: v[lo:lo + sl] for k, v in rep["metrics"].items()}),
                              _np({k: v[lo:lo + sl] for k, v in want.items()}), f"c3 slice {mode}")
        assert torch.equal(_bits(rep["returns"]), _bits(b._ep_return))
        del a, b
        torch.cuda.empty_cache()
