"""Rules computed on the device (finenvs_b200.rules; fe_rule_sums_build, fe_rule_table, fe_backtest_rules in
csrc/fe_step.cu) against their definitions: the staged sums and every rule value equal the numpy oracle bit for bit, and
backtest_rules / evaluate_rules equal the table path (backtest / backtest_portfolio / evaluate_*signal on rule_table)
bit for bit, in every mode, with known answers, shards, refusals and the c2 / c3 workloads at full size."""
import math

import numpy as np
import pytest
import torch

from oracle import oracle_rules as orl
from test_gpu_backtest import _assert_same, _bits, _columns, _env
from test_gpu_backtest import _series as _series1
from test_gpu_backtest_portfolio import _series as _series_a
from test_gpu_backtest_targets import _exits
from test_gpu_episode_metrics import _assert_records_equal, _np

W = 8
MODES = ("trade", "targets", "exits")


def _rules(A):
    """Every kind, lookbacks 1, W - 1, W, W + 1, across a staging block (1500, 2047) and past the series (MAX), sizes,
    long_only; xs_momentum for portfolios."""
    from finenvs_b200 import rules as R

    M = R.MAX_LOOKBACK
    sets = [R.constant(), R.constant(-0.5), R.momentum([1, W - 1, W, W + 1, 1500, M], size=[1, 1, 0.7, 1, 1, 1]),
            R.momentum(3, long_only=True), R.ma_cross([1, W - 1, W, 20], [W - 1 + 1, W, W + 1, 2047]),
            R.ma_cross(1, M), R.bollinger([2, W - 1, W, W + 1, 1500, M], [0.5, 1.0, 1.5, 2.0, 1.0, 1.0]),
            R.bollinger(W, 1.0, long_only=True, size=0.3)]
    if A > 1:
        sets.append(R.xs_momentum([1, W - 1, W, W + 1, 1500, M], [1, 1, A // 2, 2 if A >= 4 else 1, 1, 1]))
        sets.append(R.xs_momentum(W, 1, long_only=True))
    return R.concat(*sets)


def _closes(series):
    p = series.prices.cpu().numpy()
    return p[:, 3] if p.ndim == 2 else p[:, :, 3]


def _series(A, dtype=torch.float32, seed=5):
    return _series1(dtype, seed=seed)[0] if A == 1 else _series_a(A, dtype, seed=seed)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 5, 30, 32])
def test_sums_and_rule_table_equal_the_oracle(A):
    series = _series(A)
    env = _env(series, 64)
    rs = _rules(A)
    c = _closes(series)
    want_sums = orl.rule_sums(c)
    got = series.rule_sums().cpu().numpy().tobytes()
    assert got == orl.sums_bytes(want_sums)
    table = env.rule_table(rs)
    assert table.shape == ((len(rs), series.num_rows) if A == 1 else (len(rs), series.num_rows, A))
    want = orl.rule_table(rs.records, c, sums=want_sums)
    got = table.cpu().numpy().reshape(want.shape)
    for j in range(len(rs)):
        bad = np.nonzero(got[j].view(np.int32) != want[j].view(np.int32))
        assert bad[0].size == 0, f"rule {j} {rs.records[j]}: {bad[0].size} values differ, first at row {bad[0][0]}"
    # every kind produced all three signs somewhere, so the comparison bites
    for kind in set(rs.records["kind"].tolist()) - {0}:
        vals = got[rs.records["kind"] == kind]
        assert (vals > 0).any() and (vals < 0).any() and (vals == 0).any(), kind


@pytest.mark.gpu
def test_max_lookback_on_the_c4_series():
    """FE_RULE_MAX_LOOKBACK on the 10 M-row c4 series: staged sums bit for bit, and the values at 4 000 rows (the first
    rows with the lookback, a staging block's edges, the end) bit for bit."""
    import bench
    from finenvs_b200 import rules as R
    from finenvs_b200.data import loader

    M = R.MAX_LOOKBACK
    prices, seg_start, seg_len, _ = bench.make_series("c4", 60)
    series = loader.stage_series(prices, seg_start, seg_len, 60, "cuda:0", torch.float32)
    env = _env(series, 64)
    rs = R.concat(R.momentum([M, M - 1]), R.ma_cross([1, 7800], M), R.bollinger([M, 7800], [1.0, 2.0]))
    c = prices[:, 3]
    sums = orl.rule_sums(c)
    assert series.rule_sums().cpu().numpy().tobytes() == orl.sums_bytes(sums)
    T = c.shape[0]
    rng = np.random.default_rng(2)
    rows = np.unique(np.concatenate([np.arange(M - 3, M + 3), [M + 1023, M + 1024, 1 << 22, T - 1025, T - 1024, T - 1],
                                     rng.integers(0, T, 3980)]))
    table = env.rule_table(rs)[:, torch.from_numpy(rows).cuda()].cpu().numpy()
    want = orl.rule_table(rs.records, c, rows=rows, sums=sums)[:, :, 0]
    assert np.array_equal(table.view(np.int32), want.view(np.int32))
    assert (table[:2, rows < M - 1] == 0).all() and (table[2:4, rows < M - 1] == 0).all()   # no lookback yet
    assert (table != 0).any(axis=1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 6])
def test_out_of_range_records_give_zero(A):
    """Records the Python layer refuses are total on the device: fe_rule_table writes 0 and reads nothing outside the
    series."""
    from finenvs_b200 import _lib, rules as R

    series = _series(A)
    good = R.momentum(3).records[0]
    bad = []
    for fields in ({"kind": 5}, {"kind": -7}, {"lookback": 0}, {"lookback": -2_000_000_000}, {"lookback": 65537},
                   {"lookback": 2**31 - 1}, {"kind": 2, "lookback2": 3}, {"kind": 2, "lookback2": 1 << 30},
                   {"kind": 2, "lookback": 0, "lookback2": 5}, {"kind": 3, "lookback": 1, "k": 1.0},
                   {"kind": 3, "k": 0.0}, {"kind": 3, "k": -1.0}, {"kind": 3, "k": math.nan}, {"kind": 3, "k": math.inf},
                   {"kind": 4, "lookback2": 0}, {"kind": 4, "lookback2": A // 2 + 1}, {"kind": 4, "lookback": 0,
                                                                                         "lookback2": 1}):
        r = good.copy()
        for k, v in fields.items():
            r[k] = v
        bad.append(r)
    recs = torch.from_numpy(np.array(bad, dtype=R.RECORD).view(np.uint8)).cuda()
    T = series.num_rows
    table = torch.full((len(bad), T, A), 7.0, device="cuda")
    L = _lib.lib()
    _lib.check(L.fe_rule_table(series.prices.data_ptr(), series.rule_sums().data_ptr(), T, A, recs.data_ptr(), len(bad),
                               table.data_ptr(), 0, torch.cuda.current_stream().cuda_stream), "fe_rule_table")
    torch.cuda.synchronize()
    assert (table == 0).all() and not torch.signbit(table).any()


def _pair(A, dtype, N=2003, seed=5, **kw):
    series = _series(A, dtype, seed=seed)
    kw.setdefault("metrics_capacity", 64 * N)
    return series, _env(series, N, **kw), _env(series, N, **kw)


def _table_run(env, table, K, cols, mode, ex, history=True):
    targets, exits = mode != "trade", ex if mode == "exits" else None
    if env.num_assets == 1:
        return env.backtest(table, K, cols, history=history, targets=targets, exits=exits)
    return env.backtest_portfolio(table, K, cols, history=history, targets=targets, exits=exits)


def _check(a, b, rs, K, mode, cols, what):
    """backtest_rules on env a against the table path on env b: rewards, dones, then everything _assert_same checks."""
    S = len(rs)
    ex = _exits(S) if mode == "exits" else None
    table = b.rule_table(rs)
    out = a.backtest_rules(rs, K, cols, history=True, targets=mode != "trade", exits=ex if mode == "exits" else None)
    ref = _table_run(b, table, K, cols, mode, ex)
    assert out["steps"] == ref["steps"] == K
    assert torch.equal(_bits(out["rewards"]), _bits(ref["rewards"])) and torch.equal(out["dones"], ref["dones"]), what
    _assert_same(a, b, what)


# one case per (assets, dtype, mode, reset); offsets, evaluate, stats and K cycle through their combinations
_COMBOS = [(o, e, s, k) for k in (1, 5, 150) for o in (False, True) for e in (False, True) for s in (False, True)]
_CASES = [(A, dt, mode, reset, *_COMBOS[j % len(_COMBOS)])
          for j, (A, dt, mode, reset) in enumerate((A, dt, mode, reset) for A in (1, 5) for dt in ("f32", "f64")
                                                   for mode in MODES for reset in ("keep", "last", "all"))]


@pytest.mark.gpu
@pytest.mark.parametrize("A,dt,mode,reset,random_offset,evaluate,track_stats,K", _CASES)
def test_backtest_rules_equals_the_table_path(A, dt, mode, reset, random_offset, evaluate, track_stats, K):
    dtype = torch.float32 if dt == "f32" else torch.float64
    series, a, b = _pair(A, dtype, random_reset=reset, random_offset=random_offset, evaluate=evaluate,
                         track_stats=track_stats)
    rs = _rules(A)
    cols = _columns(a.num_envs, len(rs))
    # a few identical table-path steps first, so the run starts mid-episode with positions and metrics running
    table = b.rule_table(rs)
    for e in (a, b):
        _table_run(e, table, 7, cols, "trade", None, history=False)
    _check(a, b, rs, K, mode, cols, f"A={A} {dt} {mode} {reset} K={K}")
    # and a second run: backtests compose
    _check(a, b, rs, 3, mode, cols, f"A={A} {dt} {mode} {reset} again")


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 4])
def test_every_lane_of_a_warp_runs_another_rule(A):
    """Column c = env % R with R = 32 rules of every kind: neighbouring envs (the lanes of one warp at A = 1, of
    neighbouring warps at A > 1) run different kinds and lookbacks."""
    from finenvs_b200 import rules as R

    sets = [R.constant(), R.momentum([1, 2, 9, 40, 1100]), R.ma_cross([1, 2, 3, 5, 8], [4, 9, 30, 60, 1200]),
            R.bollinger([2, 5, 9, 30, 1100], [0.5, 1.0, 1.5, 2.0, 2.5]), R.momentum(4, long_only=True)]
    if A > 1:
        sets.append(R.xs_momentum([1, 3, 9, 30, 1100], [1, 2, 1, 2, 1]))
    rs = R.concat(*sets)
    rs = R.RuleSet(rs.records[np.arange(32) % len(rs)])
    series, a, b = _pair(A, torch.float32, N=3001)
    cols = (torch.arange(a.num_envs, device="cuda") % 32).to(torch.int32)
    for mode in MODES:
        _check(a, b, rs, 40, mode, cols, f"A={A} mixed lanes {mode}")


def _one_day(closes, opens):
    """One asset, one segment: W history rows then the bars."""
    from finenvs_b200.data import loader

    T = len(closes)
    p = np.zeros((T, 4))
    p[:, 0], p[:, 3] = opens, closes
    p[:, 1] = np.maximum(opens, closes) + 0.5
    p[:, 2] = np.minimum(opens, closes) - 0.5
    return loader.stage_series(p, np.array([0]), np.array([T], dtype=np.int32), W, "cuda:0", torch.float64)


@pytest.mark.gpu
def test_known_answers():
    """CONST with targets is buy-and-hold (the table of ones), and an MA crossing at a constructed row X trades at row
    X + 1's Open: flat before, max_shares long after, paid at that Open."""
    from finenvs_b200 import rules as R

    T, X = 40, 25
    closes = np.full(T, 100.0)
    closes[X:] = 104.0 + np.arange(T - X)
    opens = closes.copy()
    opens[X + 1] = 101.25
    series = _one_day(closes, opens)
    kw = dict(random_reset="keep", random_offset=False, metrics_capacity=64)
    a, b = _env(series, 1, **kw), _env(series, 1, **kw)
    a.backtest_rules(R.constant(), 20, targets=True)
    b.backtest(torch.ones((1, T), device="cuda"), 20, targets=True)
    _assert_same(a, b, "buy-and-hold")
    assert float(a._long[0]) == a.max_shares
    env = _env(series, 1, **kw)
    rule = R.ma_cross(2, 5)
    assert env.rule_table(rule)[0, X - 1].item() == 0 and env.rule_table(rule)[0, X].item() == 1.0
    for _ in range(T - W - 1):
        row = int(series.seg_start[env._seg[0]] + env._ptr[0]) + W - 1    # the row this step reads
        cash = float(env._cash[0])
        env.backtest_rules(rule, 1, targets=True)
        held = float(env._long[0])
        if row < X:
            assert held == 0, row
        elif row == X:
            assert held == env.max_shares
            paid = cash - float(env._cash[0])
            assert paid == pytest.approx(env.max_shares * (101.25 + env.per_share_commission), rel=1e-6)
            break
    else:
        raise AssertionError("the crossing never traded")


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 5])
def test_evaluate_rules_equals_evaluate_signal(A):
    series = _series(A)
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    a, b = _env(series, 700, **kw), _env(series, 700, **kw)
    rs = _rules(A)
    cols = _columns(700, len(rs), seed=1)
    table = b.rule_table(rs)
    for targets in (False, True):
        got = a.evaluate_rules(rs, cols, targets=targets)
        want = (b.evaluate_signal if A == 1 else b.evaluate_portfolio_signal)(table, cols, targets=targets)
        assert got["steps"] == want["steps"] and list(got) == list(want) == ["returns", "steps", "metrics"]
        assert torch.equal(_bits(got["returns"]), _bits(want["returns"]))
        _assert_records_equal(_np(got["metrics"]), _np(want["metrics"]), f"A={A} targets={targets}")
        assert a.step_count == b.step_count


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 3])
def test_shards_give_the_records_of_one_population(A):
    series = _series(A, torch.float64, seed=13)
    rs = _rules(A)
    D, S, K = series.num_segments, len(rs), 90
    N = S * D
    ex = _exits(S, seed=3)
    whole = _env(series, N)
    whole.backtest_rules(rs, K, targets=True, exits=ex)
    parts = []
    for base, n in ((0, 411), (411, N - 411)):
        env = _env(series, n, env_id_base=base, total_envs=N)
        env.backtest_rules(rs, K, targets=True, exits=ex)
        parts.append(env.episode_metrics())
    cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    order = torch.argsort(cat["key"])
    _assert_records_equal(_np({k: v[order] for k, v in cat.items()}), _np(whole.episode_metrics()), f"shards A={A}")


@pytest.mark.gpu
def test_argument_refusals_launch_nothing():
    from finenvs_b200 import rules as R

    series1, a1, _ = _pair(1, torch.float32, N=300)
    series5, a5, _ = _pair(5, torch.float32, N=300)
    before = {id(e): (e.step_count, e._ptr.clone(), e._cash.clone(), e.metrics_summary()["episodes"].item())
              for e in (a1, a5)}
    rs = R.momentum(5)

    def ones(shape):
        return torch.ones(shape, dtype=torch.float64, device="cuda")

    c0 = torch.zeros(300, dtype=torch.int32, device="cuda")

    cases = [
        (a1, lambda e: e.backtest_rules(torch.ones(3, 10), 5), ValueError, "RuleSet"),
        (a1, lambda e: e.backtest_rules(R.xs_momentum(5, 1), 5), ValueError, "portfolio env"),
        (a5, lambda e: e.backtest_rules(R.xs_momentum(5, 3), 5), ValueError, "num_assets / 2 = 2"),
        (a1, lambda e: e.backtest_rules(rs, 0, c0), ValueError, "num_steps"),
        (a5, lambda e: e.backtest_rules(rs, 5, c0, exits=ones((1, 2))), ValueError, "exits need targets"),
        (a1, lambda e: e.backtest_rules(rs, 5, c0, targets=True, exits=ones((2, 2))), ValueError, r"\(1, 2\) tensor"),
        (a1, lambda e: e.backtest_rules(rs, 5, c0, targets=True, exits=-ones((1, 2))), ValueError, "> 0"),
        (a1, lambda e: e.backtest_rules(rs, 5), ValueError, "default columns"),
        (a1, lambda e: e.backtest_rules(rs, 5, columns=torch.full((300,), 1, device="cuda")), ValueError, "columns"),
        (a5, lambda e: e.backtest_rules(rs, 5, columns=torch.zeros(299, dtype=torch.int32)), ValueError, "columns"),
        (a1, lambda e: e.evaluate_rules(rs, c0), RuntimeError, "evaluate=True"),
        (a5, lambda e: e.rule_table(R.xs_momentum(5, 3)), ValueError, "num_assets / 2"),
    ]
    for env, f, exc, msg in cases:
        with pytest.raises(exc, match=msg):
            f(env)
    torch.cuda.synchronize()
    for e in (a1, a5):
        n, ptr, cash, eps = before[id(e)]
        assert e.step_count == n and torch.equal(e._ptr, ptr) and torch.equal(e._cash, cash)
        assert e.metrics_summary()["episodes"].item() == eps


def _mixed_rules(S, A, seed=0):
    """S rules of every kind with lookbacks drawn from a seeded generator (xs_momentum only for portfolios)."""
    from finenvs_b200 import rules as R

    rng = np.random.default_rng(seed)
    q = S // (5 if A > 1 else 4)
    sets = [R.momentum(rng.integers(1, 400, q)), R.ma_cross(rng.integers(1, 50, q), rng.integers(50, 2000, q)),
            R.bollinger(rng.integers(2, 400, q), rng.uniform(0.5, 3.0, q))]
    if A > 1:
        sets.append(R.xs_momentum(rng.integers(1, 400, q), rng.integers(1, A // 2 + 1, q)))
    rest = S - q * len(sets)
    sets.append(R.constant(np.where(np.arange(rest) % 2 == 0, 1.0, -1.0)))
    return R.concat(*sets)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_full_size(workload):
    """c2 (W = 60, 1023 days of 252 bars) with 1024 mixed rules, 1 047 552 envs, and c3 (30 assets, W = 128) with 64
    xs_momentum rules, 65 472 envs: evaluate_rules equals the evaluate report of the rule table, in trade and target
    mode."""
    import bench
    from finenvs_b200 import rules as R
    from finenvs_b200.data import loader

    Wc, S = (60, 1024) if workload == "c2" else (128, 64)
    prices, seg_start, seg_len, _ = bench.make_series(workload, Wc)
    series = loader.stage_series(prices, seg_start, seg_len, Wc, "cuda:0", torch.float32)
    D, A = series.num_segments, series.num_assets
    N = S * D
    rng = np.random.default_rng(4)
    rs = (_mixed_rules(S, A) if workload == "c2" else
          R.xs_momentum(rng.integers(5, 131, S), rng.integers(1, A // 3 + 1, S)))
    kw = dict(evaluate=True, random_reset=None, random_offset=False)
    for targets in (False, True):
        a = _env(series, N, **kw)
        got = a.evaluate_rules(rs, targets=targets)
        del a
        b = _env(series, N, **kw)
        table = b.rule_table(rs)
        want = (b.evaluate_signal if A == 1 else b.evaluate_portfolio_signal)(table, targets=targets)
        del b, table
        torch.cuda.empty_cache()
        assert got["steps"] == want["steps"] == 252 and got["metrics"]["key"].numel() == N
        assert torch.equal(_bits(got["returns"]), _bits(want["returns"]))
        _assert_records_equal(_np(got["metrics"]), _np(want["metrics"]), f"{workload} targets={targets}")
