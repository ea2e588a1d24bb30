"""Rules computed on the device, checked without a GPU: the FeRule record and its mirrors, the builders of
finenvs_b200.rules (packing, broadcasting, refusals), hand-computed values of every kind through the numpy oracle (the
definition the device matches bit for bit), no look-ahead, the accuracy of the staged window sums on a 10 M-row series,
and the argument checks of fe_backtest_rules / fe_rule_table / fe_rule_sums_build, each rejected before any CUDA call."""
import ctypes
import math
import os

import numpy as np
import pytest

from oracle import oracle_rules as orl
from parity_utils import ROOT
from test_backtest_host import _params

NAN = float("nan")


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


# ------------------------------------------------------------------------------------------------ the record ----
def test_record_layout(built):
    from finenvs_b200 import rules

    assert ctypes.sizeof(built.FeRule) == 32 and rules.RECORD.itemsize == 32
    assert [(f, built.FeRule.__dict__[f].offset) for f, _ in built.FeRule._fields_] == [
        ("kind", 0), ("lookback", 4), ("lookback2", 8), ("long_only", 12), ("k", 16), ("size", 24), ("reserved", 28)]
    assert [rules.RECORD.fields[f][1] for f, _ in built.FeRule._fields_] == [0, 4, 8, 12, 16, 24, 28]
    assert (built.RULE_MAX_LOOKBACK, built.RULE_BLOCK) == (orl.MAX_LOOKBACK, orl.BLOCK) == (65536, 1024)
    hdr = open(os.path.join(ROOT, "include", "finenvs_b200.h")).read()
    for name, v in (("FE_RULE_CONST", 0), ("FE_RULE_MOMENTUM", 1), ("FE_RULE_MA_CROSS", 2), ("FE_RULE_BOLLINGER", 3),
                    ("FE_RULE_XS_MOMENTUM", 4), ("FE_RULE_MAX_LOOKBACK", 65536), ("FE_RULE_BLOCK", 1024)):
        assert f"#define {name} {v}\n" in hdr, name


def test_sums_bytes(built):
    L = built.lib()
    assert L.fe_rule_sums_bytes(10, 1) == 10 * 20 + 8
    assert L.fe_rule_sums_bytes(1025, 3) == 1025 * 3 * 20 + 2 * 3 * 8
    assert L.fe_rule_sums_bytes(0, 1) == 0 and L.fe_rule_sums_bytes(5, 0) == 0 and L.fe_rule_sums_bytes(5, 33) == 0
    s = orl.rule_sums(np.arange(1025 * 3, dtype=np.float64).reshape(1025, 3))
    assert len(orl.sums_bytes(s)) == L.fe_rule_sums_bytes(1025, 3)


# ------------------------------------------------------------------------------------------------ builders ----
def test_builders_pack_and_broadcast():
    from finenvs_b200 import rules

    g = rules.ma_cross(np.array([5, 10])[:, None], np.array([20, 50, 100])[None, :], size=0.5)
    assert len(g) == 6
    assert g.records["kind"].tolist() == [rules.MA_CROSS] * 6
    assert g.records["lookback"].tolist() == [5, 5, 5, 10, 10, 10]
    assert g.records["lookback2"].tolist() == [20, 50, 100] * 2
    assert g.records["size"].tolist() == [0.5] * 6 and g.records["long_only"].tolist() == [0] * 6
    m = rules.momentum([1, 2, 3], size=[1.0, -1.0, 2.0], long_only=[True, False, True])
    assert m.records["lookback"].tolist() == [1, 2, 3]
    assert m.records["size"].tolist() == [1.0, -1.0, 2.0] and m.records["long_only"].tolist() == [1, 0, 1]
    b = rules.bollinger(20, [1.5, 2.0])
    assert b.records["lookback"].tolist() == [20, 20] and b.records["k"].tolist() == [1.5, 2.0]
    x = rules.xs_momentum([20, 60], 3)
    assert x.records["lookback2"].tolist() == [3, 3] and x.needs_assets() == 6
    c = rules.constant(-1.0)
    assert len(c) == 1 and c.records["kind"][0] == rules.CONST and c.records["size"][0] == -1.0
    allr = rules.concat(c, m, g, b, x)
    assert len(allr) == 14 and allr.records["kind"].tolist() == [0, 1, 1, 1] + [2] * 6 + [3, 3, 4, 4]
    assert allr.needs_assets() == 6 and rules.concat(m, g).needs_assets() == 1
    assert (allr.records["reserved"] == 0).all()
    assert "6 ma_cross" in repr(allr)
    assert rules.momentum(np.float64(7.0)).records["lookback"][0] == 7     # integral floats are accepted


def test_builder_refusals():
    from finenvs_b200 import rules

    M = rules.MAX_LOOKBACK
    for bad in (0, -1, M + 1, 2.5, np.nan, True, [1, 0]):
        with pytest.raises(ValueError, match="w must be integers"):
            rules.momentum(bad)
    with pytest.raises(ValueError, match="fast < slow"):
        rules.ma_cross(20, 20)
    with pytest.raises(ValueError, match="fast < slow"):
        rules.ma_cross([5, 30], 20)
    with pytest.raises(ValueError, match="slow must be integers"):
        rules.ma_cross(5, M + 1)
    with pytest.raises(ValueError, match="w must be integers"):
        rules.bollinger(1, 2.0)
    for k in (0.0, -1.0, np.inf, np.nan):
        with pytest.raises(ValueError, match="k must be finite and > 0"):
            rules.bollinger(20, k)
    with pytest.raises(ValueError, match="n must be integers"):
        rules.xs_momentum(20, 0)
    for size in (np.nan, np.inf, 1e39):
        with pytest.raises(ValueError, match="size must be finite"):
            rules.momentum(5, size=size)
    with pytest.raises(ValueError, match="long_only must be booleans"):
        rules.momentum(5, long_only=0.5)
    with pytest.raises(ValueError):
        rules.momentum([1, 2, 3], size=[1.0, 2.0])                          # does not broadcast
    with pytest.raises(ValueError, match="concat"):
        rules.concat()
    with pytest.raises(ValueError, match="non-empty"):
        rules.RuleSet(np.zeros(0, dtype=rules.RECORD))


def test_record_checks():
    """check_records refuses every field the device would evaluate to 0, and rules the env cannot run."""
    from finenvs_b200 import rules

    def rec(**f):
        r = rules.momentum(5).records.copy()
        for k, v in f.items():
            r[k] = v
        return r

    for fields, msg in (({"kind": 5}, "unknown kind"), ({"kind": -1}, "unknown kind"),
                        ({"lookback": 0}, r"lookback outside \[1, 65536\]"), ({"lookback": 65537}, "lookback outside"),
                        ({"kind": 2, "lookback2": 5}, "slow lookback"), ({"kind": 2, "lookback2": 65537}, "slow lookback"),
                        ({"kind": 3, "lookback": 1, "k": 1.0}, "w must be >= 2"), ({"kind": 3, "k": 0.0}, "k must be"),
                        ({"kind": 3, "k": np.inf}, "k must be"), ({"kind": 4, "lookback2": 0}, "n must be >= 1"),
                        ({"size": np.nan}, "size must be finite"), ({"long_only": 2}, "long_only"),
                        ({"reserved": 1}, "reserved")):
        with pytest.raises(ValueError, match=msg):
            rules.RuleSet(rec(**fields))
    x = rules.xs_momentum(5, 2)
    rules.check_records(x.records, 4)
    rules.check_records(rules.momentum(5).records, 1)
    with pytest.raises(ValueError, match="portfolio env"):
        rules.check_records(x.records, 1)
    with pytest.raises(ValueError, match="num_assets / 2 = 1"):
        rules.check_records(x.records, 3)
    r = rec(lookback=0)                                                   # CONST ignores its lookbacks
    r["kind"] = 0
    rules.RuleSet(r)


# ------------------------------------------------------------------------------------------------ known answers ----
C12 = np.array([10, 11, 11, 9, NAN, 12, 12, 13, 10, 10, 11, 14], dtype=np.float64)


def _signs(rs, closes=C12):
    return orl.signs(rs.records[0], closes, orl.rule_sums(closes))[:, 0].tolist()


def test_known_answers_single_asset():
    from finenvs_b200 import rules

    assert _signs(rules.constant()) == [1] * 12
    assert _signs(rules.momentum(1)) == [0, 1, 0, -1, 0, 0, 0, 1, -1, 0, 1, 1]          # equal closes, NaN, row 0
    assert _signs(rules.momentum(3)) == [0, 0, 0, -1, 0, 1, 1, 0, -1, -1, -1, 1]
    assert _signs(rules.ma_cross(1, 2)) == [0, 1, 0, -1, 0, 0, 0, 1, -1, 0, 1, 1]       # equal means give 0
    assert _signs(rules.ma_cross(1, 3)) == [0, 0, 1, -1, 0, 0, 0, 1, -1, -1, 1, 1]      # windows over the NaN give 0
    assert _signs(rules.bollinger(3, 1.0)) == [0, 0, 0, 1, 0, 0, 0, -1, 1, 0, -1, -1]
    assert _signs(rules.bollinger(2, 0.5)) == [0, -1, 0, 1, 0, 0, 0, -1, 1, 0, -1, -1]     # sd 0 (equal closes): 0
    assert _signs(rules.momentum(12)) == [0] * 12                                         # the lookback never exists
    assert _signs(rules.bollinger(12, 1.0)) == [0] * 12


def test_values_size_long_only_and_zero_sign():
    from finenvs_b200 import rules

    s = orl.rule_sums(C12)
    v = orl.values(rules.momentum(1, size=0.5, long_only=True).records[0], C12, s)[:, 0]
    assert v.tolist() == [0, 0.5, 0, 0, 0, 0, 0, 0.5, 0, 0, 0.5, 0.5]
    v = orl.values(rules.momentum(1, size=-2.0).records[0], C12, s)[:, 0]
    assert v.tolist() == [0, -2.0, 0, 2.0, 0, 0, 0, -2.0, 2.0, 0, -2.0, -2.0]
    assert not np.signbit(v[v == 0]).any()                                                # 0 is +0.0f, whatever the size
    assert v.dtype == np.float32


XS = np.array([[10, 20, 30, 40], [11, 22, 30, 36], [12.1, 22, NAN, 36], [12.1, 0, 30, 36], [12.1, 5, 30, 36]],
              dtype=np.float64)


def test_known_answers_cross_sectional():
    """Ties go to the lower asset index; a non-finite close or a zero C[r-w] takes the asset out of the ranking; with
    fewer than 2n ranked assets the row is 0."""
    from finenvs_b200 import rules

    s = orl.rule_sums(XS)
    one = orl.signs(rules.xs_momentum(1, 1).records[0], XS, s).tolist()
    assert one == [[0, 0, 0, 0], [1, 0, 0, -1], [1, 0, 0, -1], [1, -1, 0, 0], [1, 0, 0, -1]]
    two = orl.signs(rules.xs_momentum(1, 2).records[0], XS, s).tolist()
    assert two == [[0, 0, 0, 0], [1, 1, -1, -1], [0] * 4, [0] * 4, [0] * 4]
    # the time-series kinds apply to each asset's own closes; CONST gives every asset `size`
    mom = orl.signs(rules.momentum(1).records[0], XS, s).tolist()
    assert mom == [[0] * 4, [1, 1, 0, -1], [1, 0, 0, 0], [0, -1, 0, 0], [0, 1, 0, 0]]
    assert orl.values(rules.constant(0.25).records[0], XS, s).tolist() == [[0.25] * 4] * 5
    # n > A / 2 is total on the device: 0 everywhere
    r = rules.xs_momentum(1, 3).records[0]
    assert (orl.signs(r, XS, s) == 0).all()


def test_no_look_ahead():
    """Every value at row r is unchanged when the closes of rows > r change (sums included)."""
    from finenvs_b200 import rules

    rng = np.random.default_rng(3)
    T, A = 2600, 6
    c = 100.0 * np.exp(np.cumsum(rng.normal(0, 0.01, (T, A)), axis=0))
    rs = rules.concat(rules.constant(), rules.momentum([1, 7, 1500]), rules.ma_cross([3, 20], [50, 1100]),
                      rules.bollinger([2, 30, 2000], 1.5), rules.xs_momentum([1, 40], [1, 3]))
    base = orl.rule_table(rs.records, c)
    for r in (0, 1, 1023, 1024, 1500, 2047, 2048, 2599):
        d = c.copy()
        d[r + 1:] = rng.uniform(1, 500, d[r + 1:].shape)
        d[r + 1:r + 3] = np.nan
        got = orl.rule_table(rs.records, d, rows=np.arange(r + 1))
        assert np.array_equal(got.view(np.int32), base[:, :r + 1].view(np.int32)), r


# ------------------------------------------------------------------------------------------------ accuracy ----
U = 2.0 ** -53


@pytest.fixture(scope="module")
def c4_like():
    """A c4-shaped series: 10 M minute bars, GBM sigma 0.0005 from 100, 4-decimal prices (75.7 .. 791.9)."""
    rng = np.random.default_rng(17)
    c = np.round(100.0 * np.exp(np.cumsum(rng.normal(0, 0.0005, 10_000_000))), 4)
    return c, orl.rule_sums(c)


def _reference_var(c, rows, k):
    """Population variance of the k closes ending at each row: exact for k = 2 ((C[r] - C[r-1]) / 2 squared; the
    subtraction is exact), else numpy's two-pass form (pairwise sums; relative error a few ulps)."""
    if k == 2:
        return ((c[rows] - c[rows - 1]) / 2) ** 2
    win = np.lib.stride_tricks.sliding_window_view(c, k)
    out = np.empty(rows.size)
    step = max(1, (4 << 20) // k)
    for i in range(0, rows.size, step):
        w = win[rows[i:i + step] - k + 1]
        out[i:i + w.shape[0]] = ((w - w.mean(axis=1, keepdims=True)) ** 2).mean(axis=1)
    return out


@pytest.mark.parametrize("k", [2, 20, 390, 7800, 65536])
def test_window_variance_error_is_bounded_by_block_local_magnitudes(c4_like, k):
    """The guarantee of the staged sums (the header's "Accuracy"): the window variance the device forms,
    t2 / k - (t1 / k)^2, is within 128 u M of the exact variance, M = orl.window_error_scale (the magnitudes of the
    staged terms the window is formed from, all local to the window's blocks).  Checked on every row of a c4-shaped
    series for k <= 390 and on every staging block's last row for the longer windows (the rows whose prefix sums are
    largest).  The bound is the same constant at row 0 and at row 10 M; what it scales with, M, is the local price
    level and drift, not the row index.  The relative error of the standard deviation is NOT bounded: a window whose
    variance is far below u M (two equal or nearly equal closes late in a block) gets an absolute, not a relative,
    error.  Window means hold a relative bound."""
    c, s = c4_like
    T = c.size
    rows = np.arange(k - 1, T) if k <= 390 else np.arange(1023, T, 1024)
    rows = rows[rows >= k - 1]
    mean, sd, ok = orl.window_stats(c, s, rows, k)
    assert ok.all()
    var = sd[:, 0] ** 2
    want = _reference_var(c, rows, k)
    M = orl.window_error_scale(s, rows, k)[:, 0]
    err = np.abs(var - want)
    assert np.all(err <= 128 * U * M), (k, rows[np.argmax(err - 128 * U * M)])
    ratio = np.where(M > 0, err / np.where(M > 0, M, 1.0) / U, 0.0)
    for lo, hi in ((0, 100_000), (T - 100_000, T)):                      # the same constant at both ends
        sel = (rows >= lo) & (rows < hi)
        assert ratio[sel].max() <= 128
    win = np.lib.stride_tricks.sliding_window_view(c, k)
    step = max(1, (4 << 20) // k)
    m_ref = np.concatenate([win[rows[i:i + step] - k + 1].mean(axis=1) for i in range(0, rows.size, step)])
    assert np.max(np.abs(mean[:, 0] - m_ref) / m_ref) <= 1e-14

# ------------------------------------------------------------------------------------------------ C ABI ----
NAMES = ("p", "s", "st", "m", "cap", "stats", "sums", "rules", "nrules", "col", "targets", "exits", "first", "steps",
         "rew", "done", "hist", "stream")


@pytest.fixture
def call(built):
    L = built.lib()
    keep = []

    def byref(x):
        keep.append(x)
        return ctypes.byref(x)

    good = dict(zip(NAMES, [byref(_params(built, assets=5)), byref(built.FeSeries(16, 16, 16, 16, None)),
                            byref(built.FeState(16, 16, 16, 16, 16, 16, None, 16, 16, None)),
                            byref(built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))), 8, None, 16, 16, 4, 16, 1,
                            None, 1, 10, 16, 16, 0, None]))

    def run(**over):
        args = dict(good)
        args.update({k: (byref(v) if isinstance(v, ctypes.Structure) else v) for k, v in over.items()})
        return L.fe_backtest_rules(*(args[n] for n in NAMES))

    return run


def test_backtest_rules_null_pointers_and_sizes(built, call):
    for name in ("p", "s", "st", "m", "sums", "rules", "col", "rew", "done"):
        assert call(**{name: None}) == -1, name
    assert call(steps=0) == -1 and call(steps=-3) == -1
    assert call(nrules=0) == -1 and call(nrules=-1) == -1
    assert call(cap=-1) == -1
    assert call(p=_params(built, assets=5, num_envs=0)) == -1
    for a in (0, 33, -1):
        assert call(p=_params(built, assets=a)) == -1


def test_backtest_rules_state_and_metrics(built, call):
    assert call(p=_params(built, assets=5, evaluate=1)) == -1
    st_eval = built.FeState(16, 16, 16, 16, 16, 16, 16, 16, None, None)
    assert call(p=_params(built, assets=5, evaluate=1), st=st_eval) == -1
    for field, _ in built.FeMetricsState._fields_:
        if field == "emitted":
            continue
        mm = built.FeMetricsState(*([16] * 8 + [None] + [16] * 9))
        setattr(mm, field, None)
        assert call(m=mm) == -1, field
    assert call(st=built.FeState(16, 16, 16, 16, 16, 16, None, 16, None, None), stats=16) == -1


def test_backtest_rules_targets_exits_alignment(built, call):
    assert call(targets=0, exits=16) == -1
    for ms in (0, -5, built.TARGET_MAX_SHARES + 1):
        q = _params(built, assets=1)
        q.max_shares = ms
        assert call(p=q, targets=1) == -1, ms
    for bad in (4, 12):
        assert call(targets=1, exits=bad) == -2, bad
        assert call(rules=bad) == -2 and call(sums=bad) == -2
    assert call(s=built.FeSeries(8, 16, 16, 16, None)) == -2


def test_rule_table_and_sums_refusals(built):
    L = built.lib()
    args = dict(prices=16, sums=16, T=100, A=1, rules=16, R=3, table=16, device=0, stream=None)
    order = ("prices", "sums", "T", "A", "rules", "R", "table", "device", "stream")

    def tab(**over):
        a = dict(args, **over)
        return L.fe_rule_table(*(a[k] for k in order))

    for name in ("prices", "sums", "rules", "table"):
        assert tab(**{name: None}) == -1, name
    for over in ({"R": 0}, {"R": -2}, {"T": 0}, {"A": 0}, {"A": 33}):
        assert tab(**over) == -1, over
    assert tab(prices=12) == -2 and tab(sums=4) == -2 and tab(rules=20) == -2 and tab(table=6) == -2
    assert L.fe_rule_sums_build(None, 100, 1, 16, 0, None) == -1
    assert L.fe_rule_sums_build(16, 100, 1, None, 0, None) == -1
    assert L.fe_rule_sums_build(16, 0, 1, 16, 0, None) == -1
    assert L.fe_rule_sums_build(16, 100, 33, 16, 0, None) == -1
    assert L.fe_rule_sums_build(8, 100, 1, 16, 0, None) == -2
    assert L.fe_rule_sums_build(16, 100, 1, 24, 0, None) == -2
