"""Outputs and inputs past element 2^31: the step kernels, fe_step_host, fe_step_lazy + fe_materialize, the PPO
storage kernels, the signal and rule backtests with their tables, fe_rule_table and the ES kernels at the population
sizes the library is built for (bench's c4 population on one GPU, the reference's W = 390 f64 window, c5's whole ES
population, the c3 portfolio shape), each checked past the boundary against a plain reference.  (fe_log_returns and
fe_rule_sums_build pass 2^31 only beyond 537 M rows x assets, which no workload here comes near.)  One `int` in an
offset would make the top envs write over other envs' windows; the slices checked here start before and end after
element 2^31, byte 2^31 and byte 2^32 of their output, and the last slice is the population's last tile.  Also
fe_es_gradient past 65 535 slabs of 512 pairs (gridDim.y's limit).

Each test checks the free device memory first and skips, naming the GB it needs, when the device has less; every full
tensor stays on the device (host copies are slices)."""
import gc

import numpy as np
import pytest
import torch

from parity_utils import assert_bits_equal, gbm_ohlc
from test_gpu_es_kernels import ROUTES, _eps_known_answer, _grad_f64, _inputs, _max_err, _weights, forward_reference, gamma
from test_gpu_backtest import _assert_same, _bits, _signal
from test_gpu_backtest import _env as _bt_env
from test_gpu_backtest_targets import _exits
from test_gpu_episode_metrics import _assert_records_equal, _np
from test_gpu_parity import _c1_series, _check_obs_properties, _env

pytestmark = pytest.mark.gpu

E31, B31, B32 = 1 << 31, 1 << 31, 1 << 32
SLICE = 4096
GUARD = 64 << 10              # sentinel bytes on either side of a step's observation
SENTINEL = 1234.5


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


@pytest.fixture(autouse=True)
def _free_between_cases(request):
    if torch.cuda.is_available():
        torch.cuda.reset_peak_memory_stats()
    yield
    if torch.cuda.is_available():
        print(f"\n[peak] {request.node.name}: max_memory_allocated {torch.cuda.max_memory_allocated() / 1e9:.1f} GB")
    gc.collect()
    torch.cuda.empty_cache()


def _need(gb):
    free, _ = torch.cuda.mem_get_info()
    if free < gb * 1e9:
        pytest.skip(f"needs {gb:.0f} GB of free device memory; {free / 1e9:.1f} GB free")


def _straddles(first, count, unit_bytes, boundary):
    """Units [first, first + count) of `unit_bytes` each: the first starts before `boundary` (a byte offset) and the last
    ends after it."""
    return first * unit_bytes < boundary < (first + count) * unit_bytes


def _slice_starts(n, unit_bytes, itemsize, count=SLICE):
    """Starts of `count`-unit slices of an (n, ...) output with `unit_bytes` per unit that straddle element 2^31,
    byte 2^31 and byte 2^32, and of the last `count` units.  Asserts that each really straddles its boundary."""
    starts = {}
    for name, b in (("element_2^31", E31 * itemsize), ("byte_2^31", B31), ("byte_2^32", B32)):
        first = min(max(0, b // unit_bytes - count // 2), n - count)
        assert _straddles(first, count, unit_bytes, b), (name, first)
        starts[name] = first
    starts["last"] = n - count
    assert n * unit_bytes > E31 * itemsize                     # the whole output passes element 2^31
    return starts


# ---------------------------------------------------------------------------------------------------------------------
# step kernels
# ---------------------------------------------------------------------------------------------------------------------
def _c4_series(W):
    from finenvs_b200.data import loader

    T, bars = 10_000_000, 390
    prices = np.round(gbm_ohlc(np.random.default_rng(20260101), T, 0.0005), 4)
    seg_start, seg_len = loader.regular_segments(T, bars, W)
    return prices, seg_start, seg_len


# id: (series, envs, W, obs dtype, variant, kernel_name())
STEP_CASES = {
    "gather_c2_8Mi": ("c2", 8 << 20, 60, torch.float32, "auto", "fe_gather_kernel<float>"),
    "pipe_cached_c2_8Mi": ("c2", 8 << 20, 60, torch.float32, "pipe", "fe_pipe_kernel<float,cached>"),
    "split_c2_8Mi": ("c2", 8 << 20, 60, torch.float32, "split", "fe_book_kernel + fe_stream_kernel<float>"),
    "pipe_stream_c4_8Mi": ("c4", 8 << 20, 60, torch.float32, "auto", "fe_pipe_kernel<float,stream>"),
    "tile_w390_f64": ("c2", 1_179_648, 390, torch.float64, "tile", "fe_tile_kernel<double>"),
    "direct_w390_f64": ("c2", 1_179_648, 390, torch.float64, "direct", "fe_direct_kernel<double>"),
    "gather_f64_7Mi": ("c2", 7 << 20, 60, torch.float64, "gather", "fe_gather_kernel<double>"),
    "portfolio_c3": ("c3", 131_072, 128, torch.float32, "auto",
                     "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<float>"),
}
STEPS, PROPERTY_STEPS = 40, (0, 19, 39)


def _stage(kind, W, dtype):
    from oracle import oracle as orc
    from finenvs_b200.data import loader

    if kind == "c2":
        prices, seg_start, seg_len = _c1_series(W)
    elif kind == "c4":
        prices, seg_start, seg_len = _c4_series(W)
    else:   # bench's c3 series: 30 assets, 1024 days of 252 bars
        import bench

        prices, seg_start, seg_len, _ = bench.make_series("c3", W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype, keep_logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    return series, fs


def _guarded(numel, dtype):
    """(buffer, view of numel elements inside it) with GUARD sentinel bytes on either side."""
    g = GUARD // torch.empty((), dtype=dtype).element_size()
    buf = torch.full((numel + 2 * g,), SENTINEL, dtype=dtype, device="cuda")
    return buf, buf[g: g + numel], g


def _guards_intact(buf, g):
    return bool((buf[:g] == SENTINEL).all()) and bool((buf[-g:] == SENTINEL).all())


@pytest.mark.parametrize("case", list(STEP_CASES))
def test_step_kernel_past_2_31(lib, case):
    """40 steps with random resets and offsets into a NaN-prefilled, guarded output: every slice's state, rewards, dones
    and whole observation equal, bit for bit, an oracle of the same global env ids; every env's window passes the gather
    property on three steps (a window never written stays NaN); the guard bands are intact."""
    from oracle import oracle as orc

    kind, N, W, dtype, variant, kernel = STEP_CASES[case]
    f64 = dtype == torch.float64
    itemsize = 8 if f64 else 4
    A = 30 if kind == "c3" else 1
    per_env = W * A * 5 * itemsize
    _need(N * per_env * 1.15 / 1e9 + 4)
    series, fs = _stage(kind, W, dtype)
    env = _env(series, num_envs=N, seed=17, random_reset="all", random_offset=True, obs_dtype=dtype, variant=variant)
    assert env.kernel_name() == kernel
    starts = _slice_starts(N, per_env, itemsize)
    refs = {k: orc.OracleEnv(fs, num_envs=SLICE, env_id_base=b, total_envs=N, seed=17, reset_mode=orc.RESET_ALL,
                             random_offset=True, out_f64=f64) for k, b in starts.items()}
    for k, b in starts.items():
        assert np.array_equal(env._seg[b: b + SLICE].cpu().numpy(), refs[k].seg), k
        assert np.array_equal(env._ptr[b: b + SLICE].cpu().numpy(), refs[k].ptr), k
    buf, flat, g = _guarded(N * W * A * 5, dtype)
    obs = flat.view(N, W, 5 * A)
    assert obs.numel() > E31
    rewards = torch.empty(N, dtype=dtype, device="cuda")
    dones = torch.empty(N, dtype=torch.int32, device="cuda")
    rng = np.random.default_rng(N + W)
    n_done = dict.fromkeys(starts, 0)
    for t in range(STEPS):
        a = rng.uniform(-1, 1, (N, A)).astype(np.float32)
        obs.fill_(float("nan"))
        rewards.fill_(float("nan"))
        dones.fill_(-1)
        ptr0, seg0 = env._ptr.clone() + 1, env._seg.clone()
        env.step_into(torch.from_numpy(a).cuda(), obs, rewards, dones)
        for k, b in starts.items():
            sl = slice(b, b + SLICE)
            o_ref, r_ref, d_ref, _ = refs[k].step(a[sl])
            ctx = f"{k} t={t}"
            assert_bits_equal(d_ref, dones[sl].cpu().numpy(), f"dones {ctx}")
            assert_bits_equal(r_ref, rewards[sl].cpu().numpy(), f"rewards {ctx}")
            for key, t_gpu in (("seg", env._seg), ("ptr", env._ptr), ("cash", env._cash)):
                assert_bits_equal(getattr(refs[k], key), t_gpu[sl].cpu().numpy(), f"{key} {ctx}")
            for key, t_gpu in (("long_sh", env._long), ("short_sh", env._short), ("margin", env._margin)):
                assert_bits_equal(getattr(refs[k], key).reshape(-1), t_gpu[b * A: (b + SLICE) * A].cpu().numpy(),
                                  f"{key} {ctx}")
            assert_bits_equal(o_ref, obs[sl].cpu().numpy(), f"obs {ctx}")
            n_done[k] += int(d_ref.sum())
        if t in PROPERTY_STEPS:
            _check_obs_properties(env, obs, ptr0, seg0)
        assert _guards_intact(buf, g), f"guard band overwritten at t={t}"
    assert all(v > 0 for v in n_done.values()), n_done


def test_step_host_and_lazy_past_2_31(lib):
    """The 8 Mi-env c2 gather case through fe_step_host (pageable actions: the chunked path's observation offsets; plain
    and bit-packed dones) and through fe_step_lazy + fe_materialize: equal to a step_into twin, and every env's window
    of the materialised observation passes the gather property."""
    N, W = 8 << 20, 60
    _need(3 * N * W * 5 * 4 / 1e9 + 6)
    series, _ = _stage("c2", W, torch.float32)
    kw = dict(num_envs=N, seed=23, random_reset="all", random_offset=True)
    dense, host, lazy = _env(series, **kw), _env(series, **kw), _env(series, **kw)
    assert dense.kernel_name() == "fe_gather_kernel<float>"
    starts = _slice_starts(N, W * 5 * 4, 4)
    obs = torch.empty((N, W, 5), device="cuda")
    rewards = torch.empty(N, device="cuda")
    dones = torch.empty(N, dtype=torch.int32, device="cuda")
    g = torch.Generator().manual_seed(5)
    n_done = 0
    for t in range(6):
        a = torch.rand((N, 1), generator=g) * 2 - 1
        ptr0, seg0 = dense._ptr.clone() + 1, dense._seg.clone()
        dense.step_into(a.cuda(), obs, rewards, dones)
        packed = t % 2 == 1
        o_h, r_h, d_h, _ = host.step_host(a, packed_dones=packed)
        if packed:
            d_h = host.unpack_dones(d_h)
        assert torch.equal(o_h, obs), t
        assert torch.equal(r_h, rewards.cpu()) and torch.equal(d_h, dones.cpu()), t
        del o_h
        lo, r_l, d_l, _ = lazy.step_lazy(a.cuda())
        assert torch.equal(r_l, rewards) and torch.equal(d_l, dones), t
        o_l = lo.materialize()
        for b in starts.values():
            assert torch.equal(o_l[b: b + SLICE], obs[b: b + SLICE]), (t, b)
        _check_obs_properties(lazy, o_l, ptr0, seg0)
        assert torch.equal(o_l, obs), t
        del o_l, lo
        for k in ("_seg", "_ptr", "_cash", "_long", "_short", "_margin"):
            assert torch.equal(getattr(dense, k), getattr(host, k)) and torch.equal(getattr(dense, k), getattr(lazy, k)), k
        n_done += int(dones.sum())
    assert n_done > 0


# ---------------------------------------------------------------------------------------------------------------------
# PPO storage
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rew_dtype", [torch.float32, torch.float64])
def test_returns_advantages_past_2_31(lib, rew_dtype):
    """fe_returns_advantages on (T, N) = (2049, 1 048 579): row 2048 starts past element 2^31, so every column has
    rows past it.  1 024 columns (the first, the last and spread ones) equal oracle_rollout bit for bit over all T."""
    from oracle import oracle_rollout as orr

    T, N, gam = 2049, 1_048_579, 0.99
    assert (T - 1) * N > E31
    rsize = torch.empty((), dtype=rew_dtype).element_size()
    _need(T * N * (rsize + 4 + 4 + 4 + 4 + 5) / 1e9 + 4)      # + the f32 and bool temporaries of the dones draw
    gen = torch.Generator(device="cuda").manual_seed(T + rsize)
    rewards = torch.randn((T, N), generator=gen, device="cuda", dtype=rew_dtype)
    dones = (torch.rand((T, N), generator=gen, device="cuda") < 0.02).to(torch.int32)
    values = torch.randn((T, N), generator=gen, device="cuda")
    last = torch.randn((N,), generator=gen, device="cuda")
    ret = torch.full((T, N), float("nan"), device="cuda")
    adv = torch.full((T, N), float("nan"), device="cuda")
    lib.check(lib.lib().fe_returns_advantages(rewards.data_ptr(), int(rew_dtype == torch.float64), dones.data_ptr(),
                                              values.data_ptr(), last.data_ptr(), N, T, gam, ret.data_ptr(),
                                              adv.data_ptr(), torch.cuda.current_stream().cuda_stream),
              "fe_returns_advantages")
    cols = torch.unique(torch.cat([torch.tensor([0, 1, N // 2, N - 2, N - 1]),
                                   torch.randperm(N, generator=torch.Generator().manual_seed(1))[:1019]])).cuda()
    want_r, want_a = orr.returns_and_advantages(rewards[:, cols].cpu().numpy(), dones[:, cols].cpu().numpy(),
                                                values[:, cols].cpu().numpy(), last[cols].cpu().numpy(), gam)
    assert_bits_equal(want_r, ret[:, cols].cpu().numpy(), "returns")
    assert_bits_equal(want_a, adv[:, cols].cpu().numpy(), "advantages")


# id: (series, kernel)
GATHER_OBS = {"tma_c2": ("c2", "fe_gather_obs_kernel<float>"), "warp_c4": ("c4", "fe_materialize_kernel<float>")}


@pytest.mark.parametrize("case", list(GATHER_OBS))
def test_gather_obs_past_2_31(lib, case):
    """fe_gather_obs with a shuffled int64 index of 7 200 000 samples at W = 60 f32 (2.16 G output values) against
    torch indexing of the staged log-returns, chunked; the TMA table path on the c2 series and the warp path on the
    c4 series."""
    from finenvs_b200.agents.PPO.buffer import Buffer

    kind, kernel = GATHER_OBS[case]
    W, N, B = 60, 1 << 20, 7_200_000
    _need(B * W * 5 * 4 * 1.1 / 1e9 + 4)
    series, _ = _stage(kind, W, torch.float32)
    env = _env(series, num_envs=N, seed=3, random_reset="all", random_offset=True)
    Buffer(2, 0.99, 0).bind_env(env, lazy=True)
    assert env.gather_obs_kernel_name() == kernel
    row0, pf = [], []
    lo = env.reset_lazy()
    row0.append(lo.row0)
    pf.append(lo.posfeat)
    gen = torch.Generator(device="cuda").manual_seed(9)
    for _ in range(3):
        lo, _, _, _ = env.step_lazy(torch.rand((N, 1), generator=gen, device="cuda") * 2 - 1)
        row0.append(lo.row0)
        pf.append(lo.posfeat)
    row0, pf = torch.cat(row0), torch.cat(pf)
    index = torch.randint(0, row0.numel(), (B,), generator=gen, device="cuda", dtype=torch.int64)
    index[-1] = row0.numel() - 1
    buf, flat, g = _guarded(B * W * 5, torch.float32)
    flat.fill_(float("nan"))
    out = flat.view(B, W, 5)
    assert out.numel() > E31
    env.gather_obs(row0, pf, index, out)
    assert _guards_intact(buf, g)
    starts = _slice_starts(B, W * 5 * 4, 4)
    table = series.logret
    steps = torch.arange(W, device="cuda")[None, :]
    chunk = 1 << 18
    for lo_ in range(0, B, chunk):
        idx = index[lo_: lo_ + chunk]
        o = out[lo_: lo_ + chunk]
        assert torch.equal(o[..., :4], table[row0[idx][:, None] + steps]), lo_
        assert torch.equal(o[..., 4], pf[idx][:, None].expand(-1, W)), lo_
    r0_h, pf_h, lr = row0.cpu().numpy(), pf.cpu().numpy(), series.logret.cpu().numpy()
    for b in starts.values():   # the slices around the boundaries once more, on the host
        idx = index[b: b + SLICE].cpu().numpy()
        r0, p = r0_h[idx], pf_h[idx]
        want = np.concatenate([lr[r0[:, None] + np.arange(W)[None, :]], np.repeat(p[:, None, None], W, 1)], 2)
        assert_bits_equal(want, out[b: b + SLICE].cpu().numpy(), f"gather_obs slice at {b}")


# ---------------------------------------------------------------------------------------------------------------------
# backtests and rule tables
# ---------------------------------------------------------------------------------------------------------------------
def _bench_series(kind, W):
    import bench
    from finenvs_b200.data import loader

    prices, seg_start, seg_len, _ = bench.make_series(kind, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32, keep_logret64=True)
    return series, (prices, seg_start, seg_len)


def _oracle_trade_run(fs, signal_h, cols_h, base, total, K, W):
    """(K, n) rewards and dones of an oracle of global ids [base, base + n) driven with the table's actions, looked up
    from the oracle's own state before each step (backtest()'s definition)."""
    from oracle import oracle as orc

    n = cols_h.shape[0]
    ref = orc.OracleEnv(fs, num_envs=n, env_id_base=base, total_envs=total, seed=9, reset_mode=orc.RESET_ALL,
                        random_offset=True, out_f64=False)
    R, D = np.empty((K, n), np.float32), np.empty((K, n), np.int32)
    for t in range(K):
        a = signal_h[cols_h, fs.seg_start[ref.seg] + ref.ptr + W - 1]
        _, R[t], D[t], _ = ref.step(a, want_obs=False)
    return R, D


def test_backtest_history_past_2_31(lib):
    """The c2 population (1 047 552 envs) for K = 2 100 steps with history: the (K, N) rewards and dones pass element
    2^31 at row 2 050 (inside the row, at env 2 048) and byte 2^32 at row 1 025 (env 1 024), so slice [0, 4096) straddles
    both.  Its history and that of the last 4 096 envs equal an oracle driven with the table's actions, and their
    episode records equal oracle_metrics on those histories."""
    from oracle import oracle as orc
    from oracle import oracle_metrics as om

    W, K, S = 60, 2100, 4
    series, (prices, seg_start, seg_len) = _bench_series("c2", W)
    N = 1024 * series.num_segments
    assert N == 1_047_552 and K * N > E31
    assert _straddles(2050 * N, SLICE, 4, E31 * 4) and _straddles(1025 * N, SLICE, 4, B32)
    _need(K * N * 8 * 1.1 / 1e9 + 8)
    env = _bt_env(series, N, metrics_capacity=40 * N)   # about 25 episodes per env: the random table bankrupts often
    sig = _signal(S, series.num_rows, seed=21)
    cols = (torch.arange(N, device="cuda") % S).to(torch.int32)
    out = env.backtest(sig, K, cols, history=True)
    R, D = out["rewards"], out["dones"]
    assert R.shape == (K, N) and R.numel() > E31
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    sig_h = sig.cpu().numpy()
    rec = _np(env.episode_metrics())
    for b in (0, N - SLICE):
        Rr, Dr = _oracle_trade_run(fs, sig_h, (b + np.arange(SLICE)) % S, b, N, K, W)
        assert_bits_equal(Dr, D[:, b: b + SLICE].cpu().numpy(), f"dones of [{b}, {b + SLICE})")
        assert_bits_equal(Rr, R[:, b: b + SLICE].cpu().numpy(), f"rewards of [{b}, {b + SLICE})")
        want, _ = om.episode_metrics(Rr, Dr, env.starting_balance, env_id_base=b, total_envs=N)
        m = (rec["env"] >= b) & (rec["env"] < b + SLICE)
        _assert_records_equal({k: v[m] for k, v in rec.items()}, want, f"records of [{b}, {b + SLICE})")
        assert int(Dr.sum()) > 4 * SLICE


def _fill_table(S, shape, seed):
    """A (S, *shape) f32 signal table filled column by column by test_gpu_backtest._signal (seeded, on the device)."""
    n = int(np.prod(shape))
    sig = torch.empty((S, *shape), device="cuda")
    for c in range(S):
        sig[c] = _signal(1, n, seed=seed + c)[0].view(shape)
    return sig


def _twin_backtests(series, sig, big_cols, N, K, run):
    """`run(env, table, columns, targets, exits)` on the full table and on its compact copy of the columns `big_cols`
    (env i runs column big_cols[i // (N / 4)], remapped in the copy): histories, state, records and summaries equal,
    in trade mode and in targets mode with exits.  Returns the trade run's history on the full table."""
    S = sig.shape[0]
    per = N // len(big_cols)
    idx = torch.arange(N, device="cuda") // per
    cols_big = torch.tensor(big_cols, device="cuda", dtype=torch.int32)[idx]
    cols_small = idx.to(torch.int32)
    small = sig[list(big_cols)].contiguous()
    ex = _exits(S)
    ex_small = ex[list(big_cols)].contiguous()
    first = None
    for targets in (False, True):
        a = _bt_env(series, N, metrics_capacity=32 * N, track_stats=True)
        b = _bt_env(series, N, metrics_capacity=32 * N, track_stats=True)
        oa = run(a, sig, cols_big, targets, ex if targets else None)
        ob = run(b, small, cols_small, targets, ex_small if targets else None)
        assert torch.equal(_bits(oa["rewards"]), _bits(ob["rewards"])) and torch.equal(oa["dones"], ob["dones"])
        _assert_same(a, b, "targets" if targets else "trade")
        assert int(ob["dones"].sum()) > N
        if first is None:
            first = oa
    return first


def test_signal_table_backtest_past_2_31(lib):
    """The c4 series (10 M rows) with a 216-column signal table (2.16 G floats): column 214 straddles element 2^31 and
    column 215 lies past it.  Envs on columns {0, 107, 214, 215} run backtest() in trade mode and in targets mode with
    exits, bit-identical to a twin on a compact 4-column copy; the column-215 envs also equal the oracle."""
    from oracle import oracle as orc

    W, S, K, N = 60, 216, 400, 4 * SLICE
    series, (prices, seg_start, seg_len) = _bench_series("c4", W)
    T = series.num_rows
    _need(S * T * 4 * 1.1 / 1e9 + 6)
    assert S * T > E31 and _straddles(214, 1, T, E31) and 215 * T > E31
    sig = _fill_table(S, (T,), seed=100)

    def run(env, table, cols, targets, exits):
        return env.backtest(table, K, cols, history=True, targets=targets, exits=exits)

    out = _twin_backtests(series, sig, (0, 107, 214, 215), N, K, run)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    b = 3 * SLICE
    Rr, Dr = _oracle_trade_run(fs, sig[215:216].cpu().numpy(), np.zeros(SLICE, np.int64), b, N, K, W)
    assert_bits_equal(Dr, out["dones"][:, b:].cpu().numpy(), "dones of the column-215 envs")
    assert_bits_equal(Rr, out["rewards"][:, b:].cpu().numpy(), "rewards of the column-215 envs")


def test_portfolio_signal_table_backtest_past_2_31(lib):
    """bench's c3 series (258 048 rows x 30 assets) with a 280-column portfolio table (7 741 440 values per column,
    2.17 G floats): column 277 straddles element 2^31.  Envs on columns {0, 138, 277, 279} run backtest_portfolio() in
    trade mode and in targets mode with exits, bit-identical to a twin on a compact 4-column copy."""
    W, S, K, N = 128, 280, 300, 4 * 1024
    series, _ = _bench_series("c3", W)
    T, A = series.num_rows, series.num_assets
    assert T * A == 7_741_440
    _need(S * T * A * 4 * 1.1 / 1e9 + 6)
    assert S * T * A > E31 and _straddles(277, 1, T * A, E31)
    sig = _fill_table(S, (T, A), seed=300)

    def run(env, table, cols, targets, exits):
        return env.backtest_portfolio(table, K, cols, history=True, targets=targets, exits=exits)

    _twin_backtests(series, sig, (0, 138, 277, 279), N, K, run)


def _rule_set(kind):
    """216 momentum / MA-cross / Bollinger rules for c4; 280 rules ending in 70 xs_momentum rules for c3."""
    from finenvs_b200 import rules as R

    n = 72 if kind == "c4" else 70
    sets = [R.momentum(list(range(2, 2 + n))), R.ma_cross(list(range(1, 1 + n)), list(range(80, 80 + n))),
            R.bollinger(list(range(10, 10 + n)), [0.5 + 0.02 * i for i in range(n)])]
    if kind == "c3":
        sets.append(R.xs_momentum(list(range(1, 1 + n)), [1 + i % 15 for i in range(n)]))
    return R.concat(*sets)


@pytest.mark.parametrize("kind", ["c4", "c3"])
def test_rule_table_past_2_31(lib, kind):
    """fe_rule_table on the c4 series (216 rules) and on bench's c3 series (280 rules, the last ones xs_momentum: the
    warp path): the table passes element 2^31 inside rule S - 2 (c4) / S - 3 (c3); about 4 000 sampled rows of the last
    rules, those around the boundary included, equal oracle_rules bit for bit."""
    from oracle import oracle_rules as orl

    W = 60 if kind == "c4" else 128
    series, (prices, _, _) = _bench_series(kind, W)
    rs = _rule_set(kind)
    S, T, A = len(rs), series.num_rows, series.num_assets
    assert S == (216 if kind == "c4" else 280)
    _need(S * T * A * 4 * 1.1 / 1e9 + 6)
    assert S * T * A > E31
    first = E31 // (T * A) - 1                     # the rule before the one that straddles 2^31, and every later one
    assert _straddles(first + 1, 1, T * A, E31)
    env = _bt_env(series, 64)
    table = env.rule_table(rs)
    c = prices[..., 3]
    sums = orl.rule_sums(c)
    rng = np.random.default_rng(T)
    b_row = (E31 - (first + 1) * T * A) // A      # the row of rule first + 1 at element 2^31
    rows = np.unique(np.concatenate([np.arange(b_row - 3, b_row + 4), [0, 1, 100, T - 2, T - 1],
                                     rng.integers(0, T, 3980)]))
    got = table[first:, torch.from_numpy(rows).cuda()].cpu().numpy().reshape(S - first, rows.size, A)
    want = orl.rule_table(rs.records[first:], c, rows=rows, sums=sums)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    assert (got != 0).any(axis=(1, 2)).all()


# ---------------------------------------------------------------------------------------------------------------------
# ES
# ---------------------------------------------------------------------------------------------------------------------
def _eps_boundaries(pairs, P):
    """The half-element offsets 2^30, 2^31, 2^32 an eps matrix of `pairs` rows of P halves passes (2^31 always)."""
    out = [b for b in (1 << 30, 1 << 31, 1 << 32) if (pairs - 2) * P > b]
    assert (1 << 31) in out
    return out


def _check_eps_rows(lib, net, pairs):
    """eps rows of the pairs on both sides of 2^30, 2^31 and 2^32 halves (bytes 2^31, 2^32, 2^33) that the matrix
    passes, and of the last pair, equal the known answer (fp16 rounding of an f64 Box-Muller: at most one code apart, at
    most 0.1 % of the values)."""
    P = net.params_padded
    rng = np.random.default_rng(pairs)
    checks = []
    for b in _eps_boundaries(pairs, P):
        p = b // P
        assert _straddles(p - 1, 3, P, b)
        checks += [(p - 1, rng.integers(0, P, 64)), (p, np.arange(P)), (p + 1, rng.integers(0, P, 64))]
    checks.append((pairs - 1, np.arange(P)))
    e = net._eps
    mism = n = 0
    for p, qs in checks:
        row = e[p].cpu().numpy()
        for q in qs:
            want = _eps_known_answer(lib, net.seed, net.generation, p, int(q))
            n += 1
            if row[q] != want:
                mism += 1
                assert abs(int(np.array(row[q]).view(np.int16)) - int(np.array(want).view(np.int16))) <= 1, (p, q)
    assert mism <= 0.001 * n, (mism, n)


def _gradient_check(lib, net, pairs, seed):
    """fe_es_gradient against _grad_f64 with the gamma(512 + slabs) bound; two calls give the same bits.  The last pair
    weighs 0.05 * pairs: that keeps the bound within about 10 % of what unit weights give (so the other slabs are held
    to it as before), yet leaving the last slab out moves the result outside the bound."""
    L = lib.lib()
    P = net.params_padded
    slabs = (pairs + 511) // 512
    w = _weights("normal", pairs, seed)
    w[-1] = 0.05 * pairs
    scratch = torch.full((int(L.fe_es_gradient_scratch(net._pnet, pairs)),), float("nan"), device="cuda")
    assert scratch.numel() == slabs * P
    outs = []
    for _ in range(2):
        g = torch.full((P,), float("nan"), device="cuda")
        lib.check(L.fe_es_gradient(net._pnet, net._eps.data_ptr(), w.data_ptr(), pairs, scratch.data_ptr(), g.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream), "fe_es_gradient")
        outs.append(g)
    assert torch.equal(outs[0], outs[1])
    ref, mag = _grad_f64(net._eps, w)
    err = (outs[0].double() - ref).abs()
    bound = gamma(512 + slabs) * mag
    assert bool((err <= bound).all()), float((err - bound).max())
    assert bool(((mag == 0) <= (outs[0] == 0)).all())
    ref_short, _ = _grad_f64(net._eps[: (slabs - 1) * 512], w[: (slabs - 1) * 512])
    assert not bool(((outs[0].double() - ref_short).abs() <= bound).all())


# id: (shape, pairs, eval envs, sampled envs): the fast kernel at 7 Mi envs (eps 9.1 G halves, dense obs 2.2 G values),
# the streaming and generic kernels at pair counts where eps passes 2^31 halves
ES_CASES = {
    "fast_300_8_1_7Mi": ((300, 8, 1), 7 << 19, 7, 1 << 16),
    "stream_300_256_256_1": ((300, 256, 256, 1), 16_001, 1, 1 << 13),
    "generic_400_64_2": ((400, 64, 2), 90_001, 7, 1 << 14),
}


@pytest.mark.parametrize("case", list(ES_CASES))
def test_es_kernels_past_2_31(lib, case):
    """fe_es_perturb rows around 2^31 and 2^32 halves and the last pair against the known answer; fe_es_forward, lazy
    and dense, on sampled envs (the pairs whose eps rows straddle the boundaries, in both halves of the population, the
    top pairs and the eval envs) within the f64-reference bound; fe_es_gradient against the f64 sum."""
    from finenvs_b200.agents.networks import ParallelMLP

    shape, pairs, num_eval, sample = ES_CASES[case]
    N = 2 * pairs + num_eval
    net0 = lib.FeEsNet(len(shape) - 1, (lib.C.c_int32 * (lib.FE_ES_MAX_LAYERS + 1))(*shape))
    P = int(lib.lib().fe_es_params_padded(lib.C.byref(net0)))
    assert pairs * P > E31
    _need((pairs * P * 2 + N * shape[0] * 4 * 2.2) / 1e9 + 8)
    torch.manual_seed(11)
    sigma = 0.05
    net = ParallelMLP(N, num_eval, shape, noise_std_dev=sigma, device_id=0, seed=1234567, action_noise_std=0.0)
    net.perturb_parameters()
    _check_eps_rows(lib, net, pairs)
    W = shape[0] // 5
    handles, X = _inputs("series", N, W, shape[0], seed=7)
    lazy_name, dense_name = ROUTES[shape][0], ROUTES[shape][1]
    assert net.forward_kernel_name(lazy=True) == lazy_name and net.forward_kernel_name(lazy=False) == dense_name
    outs = {"lazy": net.forward(handles), "dense": net.forward(X)}
    # sampled envs: the pairs whose rows straddle the boundaries (+ and - halves), the top pairs, the eval envs
    special = []
    for b in _eps_boundaries(pairs, P):
        p = b // P
        special += [p - 1, p, p + 1, pairs + p - 1, pairs + p, pairs + p + 1]
    special += list(range(pairs - 8, pairs)) + list(range(2 * pairs - 8, N))
    rand = torch.randperm(N, generator=torch.Generator().manual_seed(pairs))[:sample]
    rows = torch.unique(torch.cat([torch.tensor(special), rand])).cuda()
    ref, bnd = forward_reference(net, X, sigma, pairs, num_eval, rows)
    for m, a in outs.items():
        got = a[rows].double()
        err = (got - ref).abs()
        assert bool((err <= 2 * bnd).all()), (m, float((err - 2 * bnd).max()))
        assert float(err.max()) <= _max_err("series"), (m, float(err.max()))
    del outs, handles, X, ref, bnd
    _gradient_check(lib, net, pairs, seed=pairs)


def test_gradient_past_65535_slabs(lib):
    """A 5-1 network at 65 535 * 512 + 1 pairs: 65 536 slabs, one more than gridDim.y can launch (the parent of this
    test's kernel change refused the launch with cudaErrorInvalidConfiguration); the partial kernel walks the slabs past
    the grid.  At this many pairs gamma(512 + slabs) is about 3.9e-3, so the f64 bound is loose: what this test pins is
    that the last slab, which only the block-stride walk reaches, is summed (its one pair outweighs the bound), that
    every partial is written (the scratch starts as NaN), and that two calls give the same bits."""
    from finenvs_b200.agents.networks import ParallelMLP

    pairs = 65535 * 512 + 1
    _need(pairs * 48 * 2 / 1e9 + 4)
    net = ParallelMLP(2 * pairs, 0, (5, 1), device_id=0, seed=77, action_noise_std=0.0)
    assert net.params_padded == 48
    assert (pairs + 511) // 512 == 65536
    net.perturb_parameters()
    _gradient_check(lib, net, pairs, seed=5)
