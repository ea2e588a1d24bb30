"""Signal backtests (TimeSeriesEnv.backtest / evaluate_signal, fe_backtest_kernel in csrc/fe_step.cu) against the step
loop they replace: row lookup from the env's state, step_into, fe_episode_metrics.  State, stats, metrics and records bit
for bit on the adversarial series of test_gpu_episode_metrics.py, composition, the numpy oracle, known answers, the
evaluate report, sharding, list overflow, argument checks, and the c2 population at full size."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import oracle_metrics as om
from parity_utils import gbm_ohlc
from test_gpu_episode_metrics import _assert_records_equal, _np

W = 8
_STATE = ("_seg", "_ptr", "_cash", "_long", "_short", "_margin", "_terminated", "_ep_return", "_ep_len", "_m_f64",
          "_m_i32", "_m_emitted")


def _series(dtype, seed=5, logret64=False):
    """sigma = 0.15 bars (margin calls, bankruptcies) on 200 ragged days of 1..59 bars; also the raw arrays."""
    from finenvs_b200.data import loader

    rng = np.random.default_rng(seed)
    bars = rng.integers(1, 60, 200)
    prices = np.round(gbm_ohlc(rng, int(bars.sum()) + W, 0.15), 4)
    firsts = W + np.concatenate([[0], np.cumsum(bars)[:-1]])
    seg_start, seg_len = firsts - W, (bars + W).astype(np.int32)
    return loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype, keep_logret64=logret64), (prices, seg_start, seg_len)


def _env(series, N, **kw):
    from finenvs_b200.environments import TimeSeriesEnv

    args = dict(num_intervals=series.window, device_id=0, series=series, num_envs=N, seed=9, random_reset="all",
                random_offset=True, obs_dtype=series.logret.dtype, track_metrics=True)
    args.update(kw)
    return TimeSeriesEnv("backtest", **args)


def _signal(S, T, seed=11):
    """(S, T) f32 actions, 60 % short, 10 % exact zeros, some beyond [-1, 1] (clamped like step()'s)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.rand((S, T), generator=g, device="cuda") * 2.4 - 1.2
    short = torch.rand((S, T), generator=g, device="cuda") < 0.6
    zero = torch.rand((S, T), generator=g, device="cuda") < 0.1
    return torch.where(zero, 0.0, torch.where(short, -a.abs(), a)).contiguous()


def _columns(N, S, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, S, (N,), generator=g, device="cuda", dtype=torch.int32)


def _lookup(env, signal, cols):
    rows = env.series.seg_start[env._seg.long()] + env._ptr.long() + env.num_intervals - 1
    return signal[cols.long(), rows].reshape(env.num_envs, 1).contiguous()


def _step_loop(env, signal, cols, K):
    """The reference: K x (lookup -> step_into -> fe_episode_metrics); (K, N) rewards and dones."""
    N = env.num_envs
    R = torch.empty((K, N), dtype=env.obs_dtype, device="cuda")
    D = torch.empty((K, N), dtype=torch.int32, device="cuda")
    obs = torch.empty((N, env.num_intervals, env.num_obs), dtype=env.obs_dtype, device="cuda")
    for t in range(K):
        env.step_into(_lookup(env, signal, cols), obs, R[t], D[t])
    return R, D


def _bits(t):
    return t.view(torch.int64 if t.element_size() == 8 else torch.int32 if t.element_size() == 4 else torch.uint8)


def _assert_same(a, b, what=""):
    """env a (backtests) against env b (the step loop): everything bit for bit, f64 sums within 1e-12 of their scale."""
    assert a.step_count == b.step_count, what
    for name in _STATE:
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), (what, name)
        if x is not None:
            bad = (_bits(x) != _bits(y)).nonzero()
            assert bad.numel() == 0, f"{what} {name}: {bad.numel()} mismatches, first {bad[0].tolist()}"
    if b._stats is not None:
        sa, sb = a._stats.cpu(), b._stats.cpu()
        assert sa[:3].tolist() == sb[:3].tolist(), (what, "stats counts", sa[:3], sb[:3])
        fa, fb = sa.view(torch.float64), sb.view(torch.float64)
        bound = 1e-12 * (int(sb[0]) * float(fb[5])) ** 0.5   # sum |x| <= sqrt(n * sum x^2)
        assert abs(float(fa[4]) - float(fb[4])) <= bound and abs(float(fa[5]) - float(fb[5])) <= 1e-12 * float(fb[5]), what
    ra, rb = _np(a.episode_metrics()), _np(b.episode_metrics())
    _assert_records_equal(ra, rb, what)
    sa = {k: v.item() for k, v in a.metrics_summary().items()}
    sb = {k: v.item() for k, v in b.metrics_summary().items()}
    assert sa["episodes"] == sb["episodes"] and sa["sum_len"] == sb["sum_len"] and sa["max_mdd"] == sb["max_mdd"], what
    for k, bound in om.abs_sums(rb).items():
        assert abs(sa[k] - sb[k]) <= 1e-12 * bound, (what, k, sa[k], sb[k])


def _warm(envs, signal, cols, steps=7):
    """A few identical steps first, so the backtest starts mid-episode with positions, stats and metrics running."""
    for e in envs:
        _step_loop(e, signal, cols, steps)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5, 150])
@pytest.mark.parametrize("track_stats", [False, True])
@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("random_offset", [False, True])
@pytest.mark.parametrize("reset", ["keep", "last", "all"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_backtest_equals_the_step_loop(dtype, reset, random_offset, evaluate, track_stats, K):
    N, S = 5003, 3
    series, _ = _series(dtype)
    kw = dict(random_reset=reset, random_offset=random_offset, evaluate=evaluate, track_stats=track_stats,
              metrics_capacity=64 * N)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    sig, cols = _signal(S, series.num_rows), _columns(N, S)
    _warm((a, b), sig, cols)
    out = a.backtest(sig, K, cols, history=True)
    R, D = _step_loop(b, sig, cols, K)
    assert out["steps"] == K and out["rewards"].dtype == dtype
    assert torch.equal(_bits(out["rewards"]), _bits(R)) and torch.equal(out["dones"], D)
    _assert_same(a, b, f"K={K}")
    if K == 150:
        assert int(D.sum()) > 2 * N   # several episodes per env


@pytest.mark.gpu
def test_backtests_compose_and_interleave_with_steps():
    N, S = 5003, 4
    series, _ = _series(torch.float32, seed=6)
    sig, cols = _signal(S, series.num_rows, seed=2), _columns(N, S, seed=4)
    one, two, mixed, ref = (_env(series, N, track_stats=True) for _ in range(4))
    one.backtest(sig, 70, cols)
    two.backtest(sig, 23, cols)
    two.backtest(sig, 47, cols)
    _assert_same(two, one, "K1 + K2")
    obs = torch.empty((N, W, 5), device="cuda")
    r, d = torch.empty(N, device="cuda"), torch.empty(N, dtype=torch.int32, device="cuda")
    for k in (5, 11, 1, 30):
        mixed.backtest(sig, k, cols)
        for _ in range(3):
            mixed.step_into(_lookup(mixed, sig, cols), obs, r, d)
    _step_loop(ref, sig, cols, 5 + 11 + 1 + 30 + 4 * 3)
    _assert_same(mixed, ref, "interleaved")


@pytest.mark.gpu
def test_records_match_the_numpy_oracle():
    from oracle import oracle as orc

    N, S, K = 2048, 5, 160
    series, (prices, seg_start, seg_len) = _series(torch.float64, seed=8, logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    env = _env(series, N, metrics_capacity=64 * N)
    ref = orc.OracleEnv(fs, num_envs=N, seed=9, reset_mode=orc.RESET_ALL, random_offset=True, out_f64=True)
    sig, cols = _signal(S, series.num_rows, seed=5), _columns(N, S, seed=6)
    sig_h, cols_h = sig.cpu().numpy(), cols.cpu().numpy()
    out = env.backtest(sig, K, cols, history=True)
    R, Dn = np.empty((K, N)), np.empty((K, N), np.int32)
    blocked = margin_calls = bankrupt = 0
    for t in range(K):
        seg0, ptr0 = ref.seg.copy(), ref.ptr.copy()
        a = sig_h[cols_h, fs.seg_start[seg0] + ptr0 + W - 1]
        flat0 = (ref.long_sh == 0) & (ref.short_sh == 0)
        short0 = ref.short_sh.copy()
        want = np.clip(np.rint(a.astype(np.float32) * np.float32(5.5)), -5, 5)
        bar = prices[fs.seg_start[seg0] + ptr0 + W]   # the bar this step trades on
        _, R[t], Dn[t], _ = ref.step(a, want_obs=False)
        held = Dn[t] == 0
        # an entry the cash could not pay for: still flat although the rule asked for a position (all-or-nothing)
        blocked += int(np.sum(held & flat0 & (want != 0) & (ref.long_sh == 0) & (ref.short_sh == 0)))
        # a short held through a bar whose High is 20 % above its Open: 1.25 x High > the 1.5 x Open margin
        margin_calls += int(np.sum((short0 > 0) & (want == 0) & (bar[:, 1] > 1.2 * bar[:, 0])))
        # done before the end of the day: cash went negative
        bankrupt += int(np.sum((Dn[t] == 1) & (ptr0 + 1 + W < fs.seg_len[seg0])))
    assert np.array_equal(out["rewards"].cpu().numpy(), R) and np.array_equal(out["dones"].cpu().numpy(), Dn)
    assert blocked > 0 and bankrupt > 0 and margin_calls > 0, (blocked, bankrupt, margin_calls)
    rec, agg = om.episode_metrics(R, Dn, env.starting_balance)
    _assert_records_equal(_np(env.episode_metrics()), rec, "oracle")
    s = {k: v.item() for k, v in env.metrics_summary().items()}
    assert s["episodes"] == agg["episodes"] and s["max_mdd"] == agg["max_mdd"]


def _day_series(bars, dtype=torch.float64):
    """Hand-built days of three bars each with Open = previous Close (no overnight gaps), W = 2 history rows."""
    from finenvs_b200.data import loader

    Wd, days = 2, len(bars)
    closes = [100.0, 100.0]
    rows = [[100.0, 100.5, 99.5, 100.0], [100.0, 100.5, 99.5, 100.0]]
    for day in bars:
        for c in day:
            o = closes[-1]
            rows.append([o, max(o, c) + 0.5, min(o, c) - 0.5, c])
            closes.append(c)
    prices = np.array(rows)
    seg_start = np.array([Wd + 3 * d - Wd for d in range(days)], dtype=np.int64)
    seg_len = np.full(days, Wd + 3, dtype=np.int32)
    return loader.stage_series(prices, seg_start, seg_len, Wd, "cuda:0", dtype), prices


@pytest.mark.gpu
def test_known_answers():
    days = [[101.0, 103.0, 102.5], [99.0, 98.0, 97.25], [100.0, 100.0, 104.0]]
    series, prices = _day_series(days)
    kw = dict(evaluate=True, random_reset=None, random_offset=False, starting_balance=600.0)
    T = series.num_rows

    # all zero: no position, zero rewards, Sharpe 0
    env = _env(series, 3, **kw)
    out = env.backtest(torch.zeros((1, T), device="cuda"), 3, history=True)
    assert (out["rewards"] == 0).all() and (env._long == 0).all() and (env._short == 0).all()
    m = env.episode_metrics()
    assert m["len"].tolist() == [3, 3, 3] and (m["sharpe"] == 0).all() and (m["return"] == 0).all()

    # all +1: five shares bought at the first Open (600 buys one lot of 5 at ~100; the next entries are blocked), held,
    # closed at the end: 5 * (last Close - first Open) - two commissions of 5 x 0.01 (an f32 product, :363-365)
    comm = float(np.float32(5.0) * np.float32(0.01))
    env = _env(series, 3, **kw)
    rep = env.evaluate_signal(torch.ones((1, T), device="cuda"))
    want = [5 * (d[-1] - o) - 2 * comm for d, o in zip(days, (100.0, 102.5, 97.25))]
    assert rep["steps"] == 3
    np.testing.assert_allclose(rep["metrics"]["return"].cpu().numpy(), want, rtol=1e-12)
    np.testing.assert_allclose(rep["returns"].cpu().numpy(), want, rtol=1e-6)

    # non-zero at exactly one row r (the first bar of day 0): the trade happens at the Open of row r + 1
    r = 2
    sig = torch.zeros((1, T), device="cuda")
    sig[0, r] = 1.0
    env = _env(series, 3, **kw)
    out = env.backtest(sig, 3, torch.zeros(3, dtype=torch.int32, device="cuda"), history=True)
    rew = out["rewards"][:, 0].cpu().numpy()
    O3, C3, C4 = prices[3, 0], prices[3, 3], prices[4, 3]
    assert rew[0] == 0.0                                         # the bar of row r itself is not traded
    assert rew[1] == pytest.approx(5 * (C3 - O3) - comm, rel=1e-12)
    assert rew[2] == pytest.approx(5 * (C4 - prices[4, 0]) - comm, rel=1e-12)
    assert (out["rewards"][:, 1:] == 0).all()                    # the other days never see row r


@pytest.mark.gpu
def test_evaluate_signal_equals_evaluate_policy():
    N, S = 600, 3
    series, _ = _series(torch.float32, seed=12)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    a, b = _env(series, N, **kw), _env(series, N, **kw)
    K = int(series.seg_len.max()) - W
    cols = _columns(N, S, seed=1)
    for seed in (21, 22):
        sig = _signal(S, series.num_rows, seed=seed)
        got = a.evaluate_signal(sig, cols)
        want = b.evaluate_policy(lambda obs: _lookup(b, sig, cols), steps_per_replay=K)
        assert got["steps"] == want["steps"] == K
        assert list(got) == ["returns", "steps", "metrics"]
        assert torch.equal(_bits(got["returns"]), _bits(want["returns"]))
        _assert_records_equal(_np(got["metrics"]), _np(want["metrics"]), f"signal {seed}")
        assert a.metrics_summary()["episodes"].item() == 0 and int(a._m_emitted.sum()) == 0 and int(a._stats[1]) == 0
        assert a.step_count == b.step_count


@pytest.mark.gpu
def test_shards_give_the_records_of_one_population():
    series, _ = _series(torch.float64, seed=13)
    D, S, K = series.num_segments, 7, 90
    N = S * D
    sig = _signal(S, series.num_rows, seed=9)
    whole = _env(series, N)
    whole.backtest(sig, K)
    parts = []
    for base, n in ((0, 611), (611, N - 611)):
        env = _env(series, n, env_id_base=base, total_envs=N)
        env.backtest(sig, K)
        parts.append(env.episode_metrics())
    cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    order = torch.argsort(cat["key"])
    _assert_records_equal(_np({k: v[order] for k, v in cat.items()}), _np(whole.episode_metrics()), "shards")
    # the default columns: (strategy, day) = (gid // D, gid % D)
    ref = _env(series, N)
    _step_loop(ref, sig, torch.arange(N, device="cuda", dtype=torch.int32) // D, K)
    _assert_same(whole, ref, "default columns")


@pytest.mark.gpu
def test_overflow_is_counted_not_written():
    from finenvs_b200 import _lib

    N, S, K, cap, guard = 1024, 3, 120, 100, 64
    series, _ = _series(torch.float32, seed=14)
    sig, cols = _signal(S, series.num_rows, seed=7), _columns(N, S, seed=8)
    env = _env(series, N, metrics_capacity=cap)
    out = env.backtest(sig, K, cols, history=True)
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
    _lib.check(env._L.fe_backtest(env._pp, env._ps, env._pst, ctypes.byref(st), cap, None, sig.data_ptr(), S,
                                  cols.data_ptr(), 1, K, R.data_ptr(), Dn.data_ptr(), 1, env._stream()), "fe_backtest")
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
def test_argument_validation():
    from finenvs_b200.agents.PPO.buffer import Buffer

    N, S = 256, 2
    series, _ = _series(torch.float32, seed=15)
    T = series.num_rows
    env = _env(series, N)
    cols = _columns(N, S)
    sig = _signal(S, T)
    for bad in (sig[:, :-1], sig.double(), sig.cpu(), sig.t().contiguous().t(), sig[None]):
        with pytest.raises(ValueError):
            env.backtest(bad, 3, cols)
    for bad in (cols + S, cols - cols - 1, cols[:-1], cols.float()):
        with pytest.raises(ValueError):
            env.backtest(sig, 3, bad)
    with pytest.raises(ValueError):   # default columns: global id // 200 days reaches 1, S = 1 is too small
        _env(series, 256).backtest(sig[:1].contiguous(), 3)
    with pytest.raises(ValueError):
        env.backtest(sig, 0, cols)
    with pytest.raises(RuntimeError, match="track_metrics"):
        _env(series, N, track_metrics=False).backtest(sig, 3, cols)
    with pytest.raises(RuntimeError, match="evaluate"):
        env.evaluate_signal(sig, cols)
    for lazy in (False, True):
        bound = _env(series, N)
        Buffer(2, 0.99, 0, capacity=4).bind_env(bound, lazy=lazy)
        with pytest.raises(RuntimeError, match="bind_env"):
            bound.backtest(sig, 3, cols)
    assert env.step_count == 0 and env.metrics_summary()["episodes"].item() == 0   # nothing ran


@pytest.mark.gpu
def test_portfolio_envs_are_rejected():
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    rng = np.random.default_rng(3)
    prices = np.stack([np.round(gbm_ohlc(rng, 400, 0.02), 4) for _ in range(2)], axis=1)
    seg_start, seg_len = loader.regular_segments(400, 40, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    env = TimeSeriesEnv("p", num_intervals=W, device_id=0, series=series, num_envs=64, seed=1, track_metrics=True)
    with pytest.raises(NotImplementedError):
        env.backtest(torch.zeros((1, series.num_rows), device="cuda"), 3, torch.zeros(64, dtype=torch.int32, device="cuda"))


def _momentum_signal(logret_close, S, seed=0):
    """Sign of a rolling sum of close-to-close log-returns, window 2..65 varying by column (tools/backtest_cost.py)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    windows = torch.randint(2, 66, (S,), generator=g, device="cuda")
    c = torch.cumsum(logret_close.double(), 0)
    T = c.numel()
    idx = torch.arange(T, device="cuda")
    out = torch.empty((S, T), dtype=torch.float32, device="cuda")
    for s in range(S):
        w = int(windows[s])
        prev = torch.where(idx >= w, c[(idx - w).clamp_min(0)], torch.zeros_like(c))
        out[s] = torch.sign(c - prev).float()
    return out


@pytest.mark.gpu
def test_full_size_c2():
    """c2 (1023 days of 252 bars, W = 60) with 1024 momentum columns: 1 047 552 envs, one full episode each.  The
    backtest's records equal the step loop's on a contiguous 65 536-env slice (the loop steps the whole population)."""
    import bench
    from finenvs_b200.data import loader

    Wc, S, sl = 60, 1024, 65536
    prices, seg_start, seg_len, _ = bench.make_series("c2", Wc)
    series = loader.stage_series(prices, seg_start, seg_len, Wc, "cuda:0", torch.float32)
    D = series.num_segments
    N = S * D
    lr = series.logret[:, 0] + series.logret[:, 3]   # 100 * log(C_t / C_{t-1})
    sig = _momentum_signal(lr, S)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    a = _env(series, N, **kw)
    rep = a.evaluate_signal(sig)
    assert rep["steps"] == 252 and rep["metrics"]["key"].numel() == N
    b = _env(series, N, **kw)
    cols = torch.arange(N, device="cuda", dtype=torch.int32) // D
    _step_loop(b, sig, cols, rep["steps"])
    want = b._first_episode_metrics()
    lo = 300_000
    _assert_records_equal(_np({k: v[lo:lo + sl] for k, v in rep["metrics"].items()}),
                          _np({k: v[lo:lo + sl] for k, v in want.items()}), "c2 slice")
    assert torch.equal(_bits(rep["returns"]), _bits(b._ep_return))
