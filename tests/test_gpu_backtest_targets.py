"""Target-position backtests (backtest(targets=True, exits=...), fe_backtest_targets_kernel in csrc/fe_step.cu) against
the step loop a user would write: read the table value from the env's state, turn the target position into a share
delta in the same f32 / f64 operations, step_into.  Bit for bit on the adversarial series of test_gpu_backtest.py, with
and without trailing stops and take-profits; composition, the numpy oracle, known answers, sharding, overflow,
argument checks and the c2 population at full size."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import oracle_metrics as om
from test_gpu_backtest import W, _assert_same, _bits, _columns, _day_series, _env, _momentum_signal, _series, _signal
from test_gpu_episode_metrics import _assert_records_equal, _np


def _exits(S, seed=4):
    """(S, 2) f64 (trailing stop, take-profit) from 0.01 to 1000 on a log scale; row 0 both +inf, row 1 only a stop,
    row 2 only a take-profit, row 3 tiny thresholds that trigger on most days."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ex = torch.exp(torch.rand((S, 2), generator=g, device="cuda", dtype=torch.float64) * math.log(1e5)) * 0.01
    ex[0] = math.inf
    ex[1, 1] = math.inf
    ex[2, 0] = math.inf
    ex[3] = 0.01
    return ex.contiguous()


def _target_actions(env, signal, cols, exits=None):
    """The header's definition from the env's state before the step: (N, 1) actions and the exit mask (or None)."""
    rows = env.series.seg_start[env._seg.long()] + env._ptr.long() + env.num_intervals - 1
    v = signal[cols.long(), rows]
    ms = float(env.max_shares)
    scale = torch.tensor(ms + 0.5, dtype=torch.float32, device=v.device)
    T = torch.round(v * scale).clamp(-ms, ms)
    hit = None
    if exits is not None:
        total, peak = env._m_f64[0], env._m_f64[3]
        e = exits[cols.long()]
        hit = ((peak - total) >= e[:, 0]) | (total >= e[:, 1])
        T = torch.where(hit, torch.zeros_like(T), T)
    a = (T - (env._long - env._short)) / scale
    return a.reshape(env.num_envs, 1).contiguous(), hit


def _target_loop(env, signal, cols, K, exits=None):
    """K x (target actions -> step_into -> fe_episode_metrics); (K, N) rewards, dones and the number of steps at which
    an exit flattened a held position."""
    N = env.num_envs
    R = torch.empty((K, N), dtype=env.obs_dtype, device="cuda")
    D = torch.empty((K, N), dtype=torch.int32, device="cuda")
    obs = torch.empty((N, env.num_intervals, env.num_obs), dtype=env.obs_dtype, device="cuda")
    flattened = torch.zeros((), dtype=torch.int64, device="cuda")
    for t in range(K):
        a, hit = _target_actions(env, signal, cols, exits)
        if hit is not None:
            flattened += (hit & ((env._long != 0) | (env._short != 0))).sum()
        env.step_into(a, obs, R[t], D[t])
    return R, D, int(flattened)


def _warm(envs, signal, cols, steps=7):
    """Trade-mode steps first (a table value is a trade there), so the backtest starts mid-episode from positions of
    up to 7 x max_shares."""
    from test_gpu_backtest import _step_loop

    for e in envs:
        _step_loop(e, signal, cols, steps)


@pytest.mark.gpu
@pytest.mark.parametrize("exits", [False, True])
@pytest.mark.parametrize("K", [1, 5, 150])
@pytest.mark.parametrize("track_stats", [False, True])
@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("random_offset", [False, True])
@pytest.mark.parametrize("reset", ["keep", "last", "all"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_targets_equal_the_step_loop(dtype, reset, random_offset, evaluate, track_stats, K, exits):
    N, S = 5003, 6
    series, _ = _series(dtype)
    kw = dict(random_reset=reset, random_offset=random_offset, evaluate=evaluate, track_stats=track_stats,
              metrics_capacity=64 * N)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    sig, cols = _signal(S, series.num_rows), _columns(N, S)
    ex = _exits(S) if exits else None
    _warm((a, b), sig, cols)
    assert int(((a._long > a.max_shares) | (a._short > a.max_shares)).sum()) > 0   # beyond one step's reach
    out = a.backtest(sig, K, cols, history=True, targets=True, exits=ex)
    R, D, flattened = _target_loop(b, sig, cols, K, ex)
    assert out["steps"] == K and out["rewards"].dtype == dtype
    assert torch.equal(_bits(out["rewards"]), _bits(R)) and torch.equal(out["dones"], D)
    _assert_same(a, b, f"K={K}")
    if K == 150:
        assert int(D.sum()) > 2 * N
        if exits:
            assert flattened > N // 20, flattened   # exits flattened held positions


@pytest.mark.gpu
@pytest.mark.parametrize("evaluate", [False, True])
def test_infinite_exits_equal_no_exits(evaluate):
    N, S, K = 5003, 4, 120
    series, _ = _series(torch.float64, seed=16)
    a, b = (_env(series, N, evaluate=evaluate, track_stats=True) for _ in range(2))
    sig, cols = _signal(S, series.num_rows, seed=3), _columns(N, S, seed=2)
    inf = torch.full((S, 2), math.inf, dtype=torch.float64, device="cuda")
    oa = a.backtest(sig, K, cols, history=True, targets=True, exits=inf)
    ob = b.backtest(sig, K, cols, history=True, targets=True)
    assert torch.equal(_bits(oa["rewards"]), _bits(ob["rewards"])) and torch.equal(oa["dones"], ob["dones"])
    _assert_same(a, b, "inf exits")


@pytest.mark.gpu
def test_target_backtests_compose_and_interleave_with_steps():
    N, S = 5003, 6
    series, _ = _series(torch.float32, seed=6)
    sig, cols, ex = _signal(S, series.num_rows, seed=2), _columns(N, S, seed=4), _exits(S, seed=5)
    one, two, mixed, ref = (_env(series, N, track_stats=True) for _ in range(4))
    one.backtest(sig, 70, cols, targets=True, exits=ex)
    two.backtest(sig, 23, cols, targets=True, exits=ex)
    two.backtest(sig, 47, cols, targets=True, exits=ex)
    _assert_same(two, one, "K1 + K2")
    obs = torch.empty((N, W, 5), device="cuda")
    r, d = torch.empty(N, device="cuda"), torch.empty(N, dtype=torch.int32, device="cuda")
    for k in (5, 11, 1, 30):
        mixed.backtest(sig, k, cols, targets=True, exits=ex)
        for _ in range(3):
            mixed.step_into(_target_actions(mixed, sig, cols, ex)[0], obs, r, d)
    _target_loop(ref, sig, cols, 5 + 11 + 1 + 30 + 4 * 3, ex)
    _assert_same(mixed, ref, "interleaved")


@pytest.mark.gpu
def test_target_records_match_the_numpy_oracle():
    """oracle.OracleEnv stepped with actions computed from its own state; the exits' running P&L and peak rebuilt from
    its rewards."""
    from oracle import oracle as orc

    N, S, K = 2048, 6, 160
    series, (prices, seg_start, seg_len) = _series(torch.float64, seed=8, logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    env = _env(series, N, metrics_capacity=64 * N)
    ref = orc.OracleEnv(fs, num_envs=N, seed=9, reset_mode=orc.RESET_ALL, random_offset=True, out_f64=True)
    sig, cols, ex = _signal(S, series.num_rows, seed=5), _columns(N, S, seed=6), _exits(S, seed=7)
    sig_h, cols_h, ex_h = sig.cpu().numpy(), cols.cpu().numpy(), ex.cpu().numpy()
    out = env.backtest(sig, K, cols, history=True, targets=True, exits=ex)
    scale = np.float32(5.5)
    run_sum, run_peak = np.zeros(N), np.zeros(N)
    R, Dn = np.empty((K, N)), np.empty((K, N), np.int32)
    blocked_before = np.zeros(N, bool)
    blocked = retried = margin_calls = bankrupt = exited = 0
    for t in range(K):
        seg0, ptr0 = ref.seg.copy(), ref.ptr.copy()
        v = sig_h[cols_h, fs.seg_start[seg0] + ptr0 + W - 1]
        T = np.clip(np.rint(v * scale), np.float32(-5), np.float32(5))
        hit = ((run_peak - run_sum) >= ex_h[cols_h, 0]) | (run_sum >= ex_h[cols_h, 1])
        T = np.where(hit, np.float32(0), T).astype(np.float32)
        net0 = ref.long_sh - ref.short_sh
        delta = (T - net0).astype(np.float32)
        a = (delta / scale).astype(np.float32)
        flat0 = (ref.long_sh == 0) & (ref.short_sh == 0)
        short0 = ref.short_sh.copy()
        bar = prices[fs.seg_start[seg0] + ptr0 + W]   # the bar this step trades on
        _, R[t], Dn[t], _ = ref.step(a, want_obs=False)
        held = Dn[t] == 0
        exited += int(np.sum(hit & ~flat0))
        retried += int(np.sum(blocked_before & (delta != 0)))   # the target is asked for again at the next step
        # an entry the cash could not pay for: still flat although the target asked for a position (all-or-nothing)
        blocked_now = held & flat0 & (T != 0) & (ref.long_sh == 0) & (ref.short_sh == 0)
        blocked += int(np.sum(blocked_now))
        blocked_before = blocked_now
        # a short held (at its target) through a bar whose High is 20 % above its Open
        margin_calls += int(np.sum((short0 > 0) & (delta == 0) & (bar[:, 1] > 1.2 * bar[:, 0])))
        bankrupt += int(np.sum((Dn[t] == 1) & (ptr0 + 1 + W < fs.seg_len[seg0])))
        run_sum = run_sum + R[t]
        run_peak = np.maximum(run_peak, run_sum)
        run_sum[Dn[t] == 1] = 0.0
        run_peak[Dn[t] == 1] = 0.0
    assert np.array_equal(out["rewards"].cpu().numpy(), R) and np.array_equal(out["dones"].cpu().numpy(), Dn)
    assert min(blocked, retried, bankrupt, margin_calls, exited) > 0, (blocked, retried, bankrupt, margin_calls, exited)
    rec, agg = om.episode_metrics(R, Dn, env.starting_balance)
    _assert_records_equal(_np(env.episode_metrics()), rec, "oracle")
    s = {k: v.item() for k, v in env.metrics_summary().items()}
    assert s["episodes"] == agg["episodes"] and s["max_mdd"] == agg["max_mdd"]


W_D = 2   # _day_series' window
_DAYS = [[101.0, 103.0, 102.5], [99.0, 98.0, 97.25], [100.0, 100.0, 104.0]]
_COMM = float(np.float32(5.0) * np.float32(0.01))   # five shares of commission, an f32 product (:363-365)


@pytest.mark.gpu
def test_buy_and_hold_from_every_start():
    """Target +1 everywhere at the default balance of 10 000: one entry of 5 shares at the first traded Open, held to
    the last Close of the day, whatever the start offset (trade mode would buy 5 more on every bar)."""
    series, prices = _day_series(_DAYS)
    T = series.num_rows
    env = _env(series, 9, evaluate=True, random_reset=None, random_offset=True)
    env._seg.copy_(torch.arange(9, device="cuda", dtype=torch.int32) // 3)   # (day, offset) = (i // 3, i % 3)
    env._ptr.copy_(torch.arange(9, device="cuda", dtype=torch.int32) % 3)
    zeros = torch.zeros(9, dtype=torch.int32, device="cuda")
    rep = env.evaluate_signal(torch.ones((1, T), device="cuda"), zeros, targets=True)
    ss = series.seg_start.cpu().numpy()
    want = [5 * (prices[ss[i // 3] + W_D + 2, 3] - prices[ss[i // 3] + W_D + i % 3, 0]) - 2 * _COMM for i in range(9)]
    np.testing.assert_allclose(rep["metrics"]["return"].cpu().numpy(), want, rtol=1e-12)
    np.testing.assert_array_equal(rep["metrics"]["len"].cpu().numpy(), [3 - i % 3 for i in range(9)])



def _one_env(series, **kw):
    env = _env(series, 3, random_reset=None, random_offset=False, **kw)
    return env, torch.zeros(3, dtype=torch.int32, device="cuda")


@pytest.mark.gpu
def test_flip_takes_two_steps():
    """+1 then -1 on day 0: positions 5, 0 (the sell of the longs; the short entry sees no sell order), then -5."""
    series, prices = _day_series(_DAYS)
    sig = torch.full((1, series.num_rows), -1.0, device="cuda")
    sig[0, W_D - 1] = 1.0                      # the row the first step of day 0 reads
    env, cols = _one_env(series, evaluate=True)
    net, rew = [], []
    for _ in range(3):
        out = env.backtest(sig, 1, cols, history=True, targets=True)
        net.append(float(env._long[0] - env._short[0]))
        rew.append(float(out["rewards"][0, 0]))
    O = prices[W_D:W_D + 3, 0]
    C = prices[W_D:W_D + 3, 3]
    assert net[:2] == [5.0, 0.0] and net[2] == 0.0            # the third step ends the day, which closes the short
    assert rew[0] == pytest.approx(5 * (C[0] - O[0]) - _COMM, rel=1e-12)
    assert rew[1] == pytest.approx(-_COMM, rel=1e-12)          # sold at the Open, flat through the bar
    assert rew[2] == pytest.approx(-5 * (C[2] - O[2]) - 2 * _COMM, rel=1e-12)   # short 5 through the last bar


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["stop", "take"])
def test_exit_goes_flat_until_the_episode_ends(kind):
    """Day 1 falls on its first bar (a stop of 10 triggers), day 0 rises (a take-profit of 4 triggers): the next step
    sells at the Open, the rest of the day pays nothing, and the next episode (the same day again, reset "keep")
    trades afresh."""
    series, prices = _day_series(_DAYS)
    day = 1 if kind == "stop" else 0
    ex = torch.tensor([[10.0, math.inf]] if kind == "stop" else [[math.inf, 4.0]], dtype=torch.float64, device="cuda")
    env = _env(series, 3, random_reset=None, random_offset=False)
    cols = torch.zeros(3, dtype=torch.int32, device="cuda")
    out = env.backtest(torch.ones((1, series.num_rows), device="cuda"), 6, cols, history=True, targets=True, exits=ex)
    r = out["rewards"][:, day].cpu().numpy()
    s0 = int(series.seg_start[day]) + W_D
    first = 5 * (prices[s0, 3] - prices[s0, 0]) - _COMM
    assert (first < -10) if kind == "stop" else (first > 4)
    assert r[0] == pytest.approx(first, rel=1e-12)
    assert r[1] == pytest.approx(-_COMM, rel=1e-12) and r[2] == 0.0
    assert out["dones"][:, day].tolist() == [0, 0, 1, 0, 0, 1]
    assert r[3] == r[0] and r[4] == r[1] and r[5] == 0.0       # trading again in the next episode


@pytest.mark.gpu
def test_target_shards_give_the_records_of_one_population():
    series, _ = _series(torch.float64, seed=13)
    D, S, K = series.num_segments, 7, 90
    N = S * D
    sig, ex = _signal(S, series.num_rows, seed=9), _exits(S, seed=3)
    whole = _env(series, N)
    whole.backtest(sig, K, targets=True, exits=ex)
    parts = []
    for base, n in ((0, 611), (611, N - 611)):
        env = _env(series, n, env_id_base=base, total_envs=N)
        env.backtest(sig, K, targets=True, exits=ex)
        parts.append(env.episode_metrics())
    cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    order = torch.argsort(cat["key"])
    _assert_records_equal(_np({k: v[order] for k, v in cat.items()}), _np(whole.episode_metrics()), "shards")
    ref = _env(series, N)
    _target_loop(ref, sig, torch.arange(N, device="cuda", dtype=torch.int32) // D, K, ex)
    _assert_same(whole, ref, "default columns")


@pytest.mark.gpu
def test_target_overflow_is_counted_not_written():
    from finenvs_b200 import _lib

    N, S, K, cap, guard = 1024, 6, 120, 100, 64
    series, _ = _series(torch.float32, seed=14)
    sig, cols, ex = _signal(S, series.num_rows, seed=7), _columns(N, S, seed=8), _exits(S, seed=9)
    env = _env(series, N, metrics_capacity=cap)
    out = env.backtest(sig, K, cols, history=True, targets=True, exits=ex)
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
    _lib.check(env._L.fe_backtest_targets(env._pp, env._ps, env._pst, ctypes.byref(st), cap, None, sig.data_ptr(), S,
                                          cols.data_ptr(), ex.data_ptr(), 1, K, R.data_ptr(), Dn.data_ptr(), 1,
                                          env._stream()), "fe_backtest_targets")
    assert torch.equal(R, out["rewards"]) and torch.equal(Dn, out["dones"])
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
def test_target_argument_validation():
    from finenvs_b200.agents.PPO.buffer import Buffer

    N, S = 256, 2
    series, _ = _series(torch.float32, seed=15)
    env = _env(series, N)
    cols, sig = _columns(N, S), _signal(S, series.num_rows)
    ex = torch.full((S, 2), 50.0, dtype=torch.float64, device="cuda")
    for bad in (ex[:1], torch.ones((S, 3), dtype=torch.float64, device="cuda"), ex[:, :1], ex.float(), ex.cpu(),
                ex.t().contiguous().t(), ex[None], [[1.0, 1.0]] * S):
        with pytest.raises(ValueError, match="exits"):
            env.backtest(sig, 3, cols, targets=True, exits=bad)
    for v in (0.0, -1.0, math.nan, -math.inf):
        bad = ex.clone()
        bad[1, 1] = v
        with pytest.raises(ValueError, match="> 0"):
            env.backtest(sig, 3, cols, targets=True, exits=bad)
    with pytest.raises(ValueError, match="targets=True"):
        env.backtest(sig, 3, cols, exits=ex)
    with pytest.raises(ValueError, match="targets=True"):
        _env(series, N, evaluate=True).evaluate_signal(sig, cols, exits=ex)
    with pytest.raises(ValueError, match="max_shares"):
        _env(series, N, max_shares=(1 << 20) + 1).backtest(sig, 3, cols, targets=True)
    with pytest.raises(RuntimeError, match="track_metrics"):
        _env(series, N, track_metrics=False).backtest(sig, 3, cols, targets=True, exits=ex)
    for lazy in (False, True):
        bound = _env(series, N)
        Buffer(2, 0.99, 0, capacity=4).bind_env(bound, lazy=lazy)
        with pytest.raises(RuntimeError, match="bind_env"):
            bound.backtest(sig, 3, cols, targets=True, exits=ex)
    assert env.step_count == 0 and env.metrics_summary()["episodes"].item() == 0   # nothing ran


@pytest.mark.gpu
def test_target_portfolio_envs_are_rejected():
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv
    from parity_utils import gbm_ohlc

    rng = np.random.default_rng(3)
    prices = np.stack([np.round(gbm_ohlc(rng, 400, 0.02), 4) for _ in range(2)], axis=1)
    seg_start, seg_len = loader.regular_segments(400, 40, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    env = TimeSeriesEnv("p", num_intervals=W, device_id=0, series=series, num_envs=64, seed=1, track_metrics=True)
    ex = torch.full((1, 2), math.inf, dtype=torch.float64, device="cuda")
    with pytest.raises(NotImplementedError):
        env.backtest(torch.zeros((1, series.num_rows), device="cuda"), 3, torch.zeros(64, dtype=torch.int32,
                     device="cuda"), targets=True, exits=ex)


@pytest.mark.gpu
def test_targets_full_size_c2():
    """c2 (1023 days of 252 bars, W = 60) with 1024 momentum targets (long while momentum is positive, short while
    negative): 1 047 552 envs, one full episode each.  evaluate_signal's records equal the step loop's on a contiguous
    65 536-env slice, and every env's return is identical."""
    import bench
    from finenvs_b200.data import loader

    Wc, S, sl = 60, 1024, 65536
    prices, seg_start, seg_len, _ = bench.make_series("c2", Wc)
    series = loader.stage_series(prices, seg_start, seg_len, Wc, "cuda:0", torch.float32)
    D = series.num_segments
    N = S * D
    sig = _momentum_signal(series.logret[:, 0] + series.logret[:, 3], S)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    a = _env(series, N, **kw)
    rep = a.evaluate_signal(sig, targets=True)
    assert rep["steps"] == 252 and rep["metrics"]["key"].numel() == N
    b = _env(series, N, **kw)
    _target_loop(b, sig, torch.arange(N, device="cuda", dtype=torch.int32) // D, rep["steps"])
    want = b._first_episode_metrics()
    lo = 300_000
    _assert_records_equal(_np({k: v[lo:lo + sl] for k, v in rep["metrics"].items()}),
                          _np({k: v[lo:lo + sl] for k, v in want.items()}), "c2 slice")
    assert torch.equal(_bits(rep["returns"]), _bits(b._ep_return))
