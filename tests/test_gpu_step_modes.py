"""Every step kernel against the oracle in the modes a reference user runs — "last" (training), "keep", "all" without
offsets, evaluate with "keep" (the reference's evaluate) and evaluate with "all" + offsets — at populations where the
persistent kernels run several tiles per block with a ragged last tile; the other step entry points (lazy, host,
captured) against a twin driven by step_into in "last" and evaluate mode; reset_all() in the middle of a run; and the
staging kernels (log-returns, effective segment lengths) for portfolios.

Comparisons are bit-exact unless a comment says otherwise.  Where the oracle is given `series.logret64` it steps on
the log-return table the GPU computed: test_log_returns_portfolio_vs_numpy pins that table for A > 1 and
test_gpu_parity.py::test_log_returns_kernel_vs_reference_values for A = 1."""
import functools
import math

import numpy as np
import pytest
import torch

from parity_utils import CudaAdapter, assert_bits_equal, gbm_ohlc

pytestmark = pytest.mark.gpu

SEED = 31
STEPS = 84               # every env finishes >= 2 episodes (<= 40 bars each); evaluate mode sees "all terminated" twice
OBS_EVERY = 10
U64 = 2.0 ** -53


# (variant, dtype, W, N, A, kernel name, tile width of the pipe kernel or None)
KERNELS = [
    pytest.param("tile", torch.float32, 16, 3001, 1, "fe_tile_kernel<float>", None, id="tile-f32-W16-N3001"),
    pytest.param("direct", torch.float64, 16, 2999, 1, "fe_direct_kernel<double>", None, id="direct-f64-W16-N2999"),
    pytest.param("split", torch.float32, 60, 20011, 1, "fe_book_kernel + fe_stream_kernel<float>", None,
                 id="split-f32-W60-N20011"),
    pytest.param("pipe", torch.float32, 26, 40003, 1, "fe_pipe_kernel<float,cached>", 32, id="pipe32-f32-W26-N40003"),
    pytest.param("pipe", torch.float64, 130, 9001, 1, "fe_pipe_kernel<double,cached>", 4, id="pipe4-f64-W130-N9001"),
    pytest.param("gather", torch.float32, 60, 40003, 1, "fe_gather_kernel<float>", None, id="gather1-f32-W60-N40003"),
    pytest.param("gather", torch.float64, 60, 20011, 1, "fe_gather_kernel<double>", None, id="gather2-f64-W60-N20011"),
    pytest.param("portfolio", torch.float32, 12, 5003, 3, "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<float>",
                 None, id="portfolio-A3-f32-W12-N5003"),
    pytest.param("portfolio", torch.float64, 8, 1001, 32, "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<double>",
                 None, id="portfolio-A32-f64-W8-N1001"),
]

# (random_reset, evaluate, random_offset)
MODES = [
    pytest.param("last", False, False, id="last"),
    pytest.param("keep", False, False, id="keep"),
    pytest.param("all", False, False, id="all"),
    pytest.param("keep", True, False, id="eval-keep"),
    pytest.param("all", True, True, id="eval-all-offset"),
]


# ------------------------------------------------------------------ series builders ----------------------------------
def _prices(W, A, seed, days=160, sigma=0.08, s0=500.0):
    """Ragged days of 5..40 bars (envs end at different steps).  sigma = 0.08 at a price level of a few hundred lets a
    short-biased policy reach its margin limit within an episode, so margin calls and bankruptcies happen."""
    rng = np.random.default_rng(seed)
    bars = rng.integers(5, 41, days)
    T = W + int(bars.sum())
    if A == 1:
        prices = gbm_ohlc(rng, T, sigma, s0=s0)
    else:
        prices = np.stack([gbm_ohlc(rng, T, sigma, s0=s0 * (1 + 0.3 * a)) for a in range(A)], axis=1)
    firsts = W + np.concatenate([[0], np.cumsum(bars)[:-1]])
    return prices, firsts - W, (bars + W).astype(np.int32)


@functools.lru_cache(maxsize=None)
def _series(W, A, dtype):
    """(staged series, oracle series on the GPU's log-return table), one per shape for the whole module."""
    from oracle import oracle as orc
    from finenvs_b200.data import loader

    prices, seg_start, seg_len = _prices(W, A, seed=W * 7 + A)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype, keep_logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    assert np.array_equal(series.seg_len.cpu().numpy(), fs.seg_len)
    assert int(fs.seg_len.max()) - W <= 40
    return series, fs


def _short_biased(rng, n, A):
    a = rng.uniform(-1, 1, (n, A))
    m = rng.uniform(0, 1, (n, A)) < 0.6
    a[m] = -np.abs(a[m])
    return a.astype(np.float32)


def _env(series, W, N, dtype, variant="auto", mode="last", evaluate=False, offset=False, base=0, total=None):
    from finenvs_b200.environments import TimeSeriesEnv

    return TimeSeriesEnv("modes", num_intervals=W, device_id=0, series=series, num_envs=N, seed=SEED, random_reset=mode,
                         random_offset=offset, evaluate=evaluate, obs_dtype=dtype, variant=variant, track_stats=True,
                         env_id_base=base, total_envs=total)


def _oracle(fs, N, dtype, mode="last", evaluate=False, offset=False, base=0, total=None):
    from oracle import oracle as orc

    return orc.OracleEnv(fs, num_envs=N, seed=SEED, reset_mode={"keep": 0, "last": 1, "all": 2}[mode], random_offset=offset,
                         evaluate=evaluate, out_f64=dtype == torch.float64, env_id_base=base, total_envs=total)


def _reorder_bound(n, abs_sum):
    """|any order's f64 sum of n terms - the exact sum| <= gamma_n * sum|x| (Higham, Accuracy and Stability, §4.2)."""
    nu = n * U64
    return nu / (1 - nu) * abs_sum


# ------------------------------------------------------------------ the env, seen like the oracle --------------------
class ModeAdapter(CudaAdapter):
    """CudaAdapter that also returns the evaluate-mode state (terminated flags, episode returns) and the stats block."""

    def state(self):
        st = super().state()
        if self.env.evaluate:
            st["terminated"] = self.env._terminated.cpu().numpy()
            st["ep_return"] = self.env._ep_return.cpu().numpy()
        return st

    def stats(self):
        return {k: v.item() for k, v in self.env.stats().items()}


class LockStep:
    """env and oracle stepped together with short-biased actions.  Asserts state, rewards, dones, info and the stats
    block every step (the observation every OBS_EVERY steps) and records what happened (dones, bankruptcies, info
    steps, segment changes) so that each test can prove its scenario occurred."""

    def __init__(self, env, ref, act_seed=7):
        self.ad, self.ref = ModeAdapter(env), ref
        self.env = env
        self.N, self.A, self.W = ref.N, ref.A, ref.series.window
        self.f64 = env.obs_dtype == torch.float64
        self.evaluate = bool(env.evaluate)
        self.rng = np.random.default_rng(act_seed)
        self.t = 0
        # expected stats since the last clear
        self.n_done = self.n_term = self.sum_len = 0
        self.fin = []
        self.er = np.zeros(self.N, np.float32)
        self.el = np.zeros(self.N, np.int64)
        # what happened
        self.total_done = self.bankrupt = 0
        self.info_steps = []
        self.seg_changed = np.zeros(self.N, bool)
        self.check_state("init")
        assert_bits_equal(ref.reset(), self.ad.reset(), "reset obs")

    def check_state(self, ctx):
        st, ref = self.ad.state(), self.ref
        for key in ("seg", "ptr", "cash", "long_sh", "short_sh", "margin"):
            assert_bits_equal(getattr(ref, key).reshape(-1), st[key], f"{key} {ctx}")
        if self.evaluate:
            assert_bits_equal(ref.terminated, st["terminated"], f"terminated {ctx}")
            assert_bits_equal(ref.ep_return, st["ep_return"], f"ep_return {ctx}")

    def check_stats(self, ctx):
        s = self.ad.stats()
        assert s["n_done"] == self.n_done, f"n_done {ctx}: {s['n_done']} vs {self.n_done}"
        assert s["n_terminated"] == self.n_term, f"n_terminated {ctx}: {s['n_terminated']} vs {self.n_term}"
        if not self.evaluate:
            assert s["sum_len"] == self.sum_len, f"sum_len {ctx}: {s['sum_len']} vs {self.sum_len}"

    def step(self):
        ref, t = self.ref, self.t
        seg0, ptr0, term0 = ref.seg.copy(), ref.ptr.copy(), ref.terminated.copy()
        a = _short_biased(self.rng, self.N, self.A)
        want = t % OBS_EVERY == 0
        o_ref, r_ref, d_ref, i_ref = ref.step(a if self.A > 1 else a.reshape(-1), want_obs=want)
        o, r, d, info = self.ad.step(a)
        assert_bits_equal(d_ref, d, f"dones t={t}")
        assert_bits_equal(r_ref, r, f"rewards t={t}")
        self.check_state(f"t={t}")
        if want:
            assert_bits_equal(o_ref, o, f"obs t={t}")
        assert set(info) == set(i_ref), f"info at t={t}: {sorted(info)} vs the oracle's {sorted(i_ref)}"
        if i_ref:
            assert_bits_equal(i_ref["returns"], info["returns"], f"info['returns'] t={t}")
            self.info_steps.append(t)
        done = d_ref.astype(bool)
        self.n_done += int(done.sum())
        if self.evaluate:
            self.n_term += int((done & (term0 == 0)).sum())
        else:   # the kernel's running episode return: er = f32(f64(er) + reward)
            self.er = (self.er.astype(np.float64) + r_ref.astype(np.float64)).astype(np.float32)
            self.el += 1
            self.sum_len += int(self.el[done].sum())
            self.fin.extend(self.er[done].astype(np.float64).tolist())
            self.er[done] = 0.0
            self.el[done] = 0
        if i_ref:   # record_evaluation_metrics() zeroed the stats block
            self.n_done = self.n_term = 0
        self.check_stats(f"t={t}")
        self.total_done += int(done.sum())
        self.bankrupt += int((done & (ptr0 + 1 + self.W < ref.series.seg_len[seg0])).sum())
        self.seg_changed |= ref.seg != seg0
        self.t += 1

    def reset_all(self, redraw):
        o = self.env.reset_all(redraw=bool(redraw)).cpu().numpy()
        o_ref = self.ref.reset_all(redraw=bool(redraw))
        assert_bits_equal(o_ref, o, f"reset_all(redraw={redraw}) obs")
        self.check_state(f"after reset_all(redraw={redraw})")
        if self.evaluate:
            assert not self.env._terminated.any() and not self.env._ep_return.any()
        self.n_done = self.n_term = self.sum_len = 0
        self.fin = []
        self.er[:] = 0.0
        self.el[:] = 0
        self.check_stats("after reset_all")

    def check_sums(self):
        if self.evaluate:
            return
        s = self.ad.stats()
        x = np.asarray(self.fin)
        assert len(x) == self.n_done
        for key, v in (("sum_return", x), ("sum_return_sq", x * x)):   # f32 x f32 is exact in f64
            if self.f64:   # the host repeats the kernel's arithmetic: only the order of the device's additions differs
                assert abs(s[key] - math.fsum(v)) <= _reorder_bound(len(v), math.fsum(np.abs(v))), key
            else:
                # f32 rewards are already rounded, so the host's running returns differ from the kernel's in the last
                # bits: the tolerance of test_track_stats_matches_host_accounting, relative to sum|x| (the sum cancels)
                assert abs(s[key] - math.fsum(v)) <= 1e-6 * math.fsum(np.abs(v)), key

    def assert_scenario(self, mode, redraws=True):
        """What the case is about really happened."""
        assert self.total_done >= 2 * self.N, "every env finishes at least two episodes"
        assert self.bankrupt > 0, "a done came from bankruptcy"
        if self.evaluate:
            assert len(self.info_steps) >= 2, f"'all terminated' fired at {self.info_steps}"
        if mode == "keep" or not redraws:
            assert not self.seg_changed.any(), "no env may redraw"
        elif mode == "last":
            assert self.seg_changed[-1], "the global last env redrew its segment"
            assert not self.seg_changed[:-1].any(), "only the global last env redraws"


# ------------------------------------------------------------------ 1. mode matrix -----------------------------------
@pytest.mark.parametrize("mode,evaluate,offset", MODES)
@pytest.mark.parametrize("variant,dtype,W,N,A,kname,pipe_envs", KERNELS)
def test_step_kernel_mode_vs_oracle(variant, dtype, W, N, A, kname, pipe_envs, mode, evaluate, offset):
    from finenvs_b200 import _lib

    series, fs = _series(W, A, dtype)
    env = _env(series, W, N, dtype, variant, mode, evaluate, offset)
    assert env.kernel_name() == kname
    if pipe_envs is not None:
        assert _lib.lib().fe_pipe_envs(W, int(dtype == torch.float64), 0) == pipe_envs
    if variant in ("pipe", "gather", "split"):
        te = pipe_envs or 32
        assert N > 4 * 148 * te and N % te != 0   # several tiles per block on 148 SMs, rings wrap, ragged last tile
    run = LockStep(env, _oracle(fs, N, dtype, mode, evaluate, offset))
    for _ in range(STEPS):
        run.step()
    run.check_sums()
    run.assert_scenario(mode)


@pytest.mark.parametrize("holds_last", [True, False], ids=["holds-last", "not-last"])
@pytest.mark.parametrize("variant,dtype,W,N,A,kname", [
    pytest.param("gather", torch.float32, 60, 40003, 1, "fe_gather_kernel<float>", id="gather"),
    pytest.param("portfolio", torch.float32, 12, 5003, 3, "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<float>",
                 id="portfolio")])
def test_last_mode_shard_vs_oracle(variant, dtype, W, N, A, kname, holds_last):
    """A shard [base, base + N) of a larger population in "last" mode: the redraw belongs to the global last id.  base is
    not a multiple of 32; the shard either ends the population (its last env, in a ragged tile, redraws) or does not
    (nobody on it may ever redraw)."""
    series, fs = _series(W, A, dtype)
    base = 1237
    total = base + N + (0 if holds_last else 4099)
    env = _env(series, W, N, dtype, variant, "last", base=base, total=total)
    assert env.kernel_name() == kname
    run = LockStep(env, _oracle(fs, N, dtype, "last", base=base, total=total))
    for _ in range(STEPS):
        run.step()
    run.check_sums()
    run.assert_scenario("last", redraws=holds_last)


# ------------------------------------------------------------------ 2. other entry points vs a step_into twin -------
def _twin_pair(A, evaluate):
    """Gather (A = 1, W = 60, f32, 40 003 envs) or the portfolio kernel (A = 3, W = 12, f32, 20 011 envs: more than one
    16 384-env chunk of step_host's copy pipeline); "last" in training, "keep" in evaluate mode."""
    W, N, variant = (60, 40003, "gather") if A == 1 else (12, 20011, "portfolio")
    series, _ = _series(W, A, torch.float32)
    mode = "keep" if evaluate else "last"
    a, b = (_env(series, W, N, torch.float32, variant, mode, evaluate) for _ in range(2))
    return a, b


_STATE = ("_seg", "_ptr", "_cash", "_long", "_short", "_margin", "_terminated", "_ep_return", "_ep_len")


def _assert_twins_equal(x, y, ctx):
    for k in _STATE:
        u, v = getattr(x, k), getattr(y, k)
        assert (u is None) == (v is None), k
        if u is not None:
            assert torch.equal(u, v), f"{k} {ctx}"
    sx, sy = x.stats(), y.stats()
    for k in ("n_done", "n_terminated", "sum_len"):
        assert int(sx[k]) == int(sy[k]), f"stats {k} {ctx}: {int(sx[k])} vs {int(sy[k])}"
    # two kernels add the same terms in different orders: each sum is within gamma_n * sum|terms| of the exact one.
    # The squares are >= 0, so sum|x^2| is sum_return_sq itself, and sum|x| <= sqrt(n * sum x^2).
    n, sq = int(sx["n_done"]), float(sx["sum_return_sq"])
    for k, abs_sum in (("sum_return", math.sqrt(n * sq)), ("sum_return_sq", sq)):
        assert abs(float(sx[k]) - float(sy[k])) <= 2 * _reorder_bound(n, abs_sum), f"stats {k} {ctx}"


@pytest.mark.parametrize("evaluate", [False, True], ids=["last", "eval-keep"])
@pytest.mark.parametrize("entry", ["lazy", "host-pinned", "host-pinned-packed", "host-pageable", "host-pageable-packed"])
@pytest.mark.parametrize("A", [1, 3], ids=["gather", "portfolio"])
def test_entry_point_equals_step_into(A, entry, evaluate):
    """step_lazy (+ materialize), step_host with pinned actions (zero-copy: the persistent and portfolio kernels read the
    actions over PCIe) and with pageable actions (chunked copy pipeline on side streams), each with int32 and bit-packed
    dones, against a twin stepped with step() == step_into() + the evaluate bookkeeping."""
    if entry == "lazy" and A > 1:
        pytest.skip("lazy observations are single-asset")
    twin, env = _twin_pair(A, evaluate)
    N = env.num_envs
    if entry.startswith("host-pageable"):
        assert N > 16384   # at least two chunks
    rng = np.random.default_rng(11)
    info_steps = []
    total_done = 0
    for t in range(STEPS):
        a = torch.from_numpy(_short_biased(rng, N, A))
        o1, r1, d1, i1 = twin.step(a.cuda())
        want = t % OBS_EVERY == 0
        if entry == "lazy":
            lo, r2, d2, i2 = env.step_lazy(a.cuda())
            if want:
                assert torch.equal(lo.materialize(), o1), f"obs t={t}"
            r2, d2 = r2.cpu(), d2.cpu()
        else:
            packed = entry.endswith("packed")
            o2, r2, d2, i2 = env.step_host(a.pin_memory() if "pinned" in entry else a, packed_dones=packed)
            if packed:
                assert d2.dtype == torch.uint8 and d2.numel() == 4 * ((N + 31) // 32)
                d2 = env.unpack_dones(d2)
            if want:
                assert torch.equal(o2, o1), f"obs t={t}"
        assert torch.equal(r2, r1.cpu()) and torch.equal(d2, d1.cpu()), f"rewards / dones t={t}"
        assert set(i1) == set(i2), f"info t={t}"
        if i1:
            assert torch.equal(i1["returns"], i2["returns"]), f"returns t={t}"
            info_steps.append(t)
        _assert_twins_equal(twin, env, f"t={t}")
        total_done += int(d1.sum())
    assert total_done >= 2 * N
    if evaluate:
        assert len(info_steps) >= 2
    else:
        assert int(env.stats()["n_done"]) == total_done


@pytest.mark.parametrize("A", [1, 3], ids=["gather", "portfolio"])
def test_captured_rollout_across_all_terminated(A):
    """A CapturedRollout in evaluate mode replayed across the "all terminated" step (terminated envs collect zero
    reward, nothing resets inside the graph) equals step_into() with the same actions; each env is counted once in
    n_terminated, and the returns handed out by the evaluate bookkeeping agree."""
    twin, env = _twin_pair(A, True)
    N, W = env.num_envs, env.num_intervals

    def policy(obs):
        x = obs.reshape(N, W, A, 5)
        return (torch.tanh(x[:, -1, :, 3] * 40.0 + x[:, 0, :, 4] * 3.0) - 0.3).clamp(-1.0, 1.0).float()

    K = 48
    roll = env.capture_rollout(policy, K)
    obs = twin.reset()
    r = torch.empty(N, dtype=torch.float32, device="cuda")
    d = torch.empty(N, dtype=torch.int32, device="cuda")
    for rep in range(2):
        o_g, r_g, d_g = roll.replay()
        for t in range(K):
            obs = torch.empty_like(obs)
            twin.step_into(roll.actions[t], obs, r, d)
            assert torch.equal(r_g[t], r) and torch.equal(d_g[t], d), (rep, t)
        assert torch.equal(o_g, obs), rep
        _assert_twins_equal(twin, env, f"replay {rep}")
        # 48 steps pass the longest episode (40 bars): every env terminated, each counted once
        assert int(env.stats()["n_terminated"]) == N and bool(env._terminated.all())
        i1, i2 = twin.record_evaluation_metrics(), env.record_evaluation_metrics()
        assert torch.equal(i1["returns"], i2["returns"]) and float(i2["returns"].abs().sum()) > 0
        _assert_twins_equal(twin, env, f"after the evaluate reset {rep}")
        assert int(env.stats()["n_terminated"]) == 0 and not bool(env._terminated.any())


# ------------------------------------------------------------------ 3. reset_all() vs the oracle ---------------------
@pytest.mark.parametrize("redraw", [0, 1])
@pytest.mark.parametrize("mode,evaluate", [pytest.param("all", False, id="all"), pytest.param("last", False, id="last"),
                                           pytest.param("keep", True, id="eval-keep")])
@pytest.mark.parametrize("variant,dtype,W,N,A", [
    pytest.param("tile", torch.float32, 16, 3001, 1, id="tile"),
    pytest.param("gather", torch.float32, 60, 40003, 1, id="gather"),
    pytest.param("portfolio", torch.float32, 12, 5003, 3, id="portfolio")])
def test_reset_all_mid_run_vs_oracle(variant, dtype, W, N, A, mode, evaluate, redraw):
    """reset_all() after 45 steps (kind-1 draws keyed by a non-zero step ordinal; in evaluate mode in the middle of the
    second evaluation, so terminated flags and returns are set), then 45 more steps in lock-step."""
    series, fs = _series(W, A, dtype)
    env = _env(series, W, N, dtype, variant, mode, evaluate)
    run = LockStep(env, _oracle(fs, N, dtype, mode, evaluate))
    for _ in range(45):
        run.step()
    assert env.step_count == 45
    if evaluate:
        assert len(run.info_steps) == 1 and bool(env._terminated.any()) and bool(env._ep_return.any())
    seg_before = run.ref.seg.copy()
    run.reset_all(redraw)
    if redraw:
        assert not np.array_equal(run.ref.seg, seg_before)
    else:
        assert np.array_equal(run.ref.seg, seg_before) and not run.ref.ptr.any()
    for _ in range(45):
        run.step()
    run.check_sums()
    if evaluate:   # the next "all terminated" came from the fresh episodes, at the oracle's step
        assert len(run.info_steps) == 2 and run.info_steps[1] >= 45


# ------------------------------------------------------------------ 4. staging for A > 1 -----------------------------
@pytest.mark.parametrize("A", [3, 32])
def test_log_returns_portfolio_vs_numpy(A):
    """fe_log_returns on a (T, A, 4) series against a float64 numpy restatement of feo_log_returns: col 0 =
    100*log(O_t / C_{t-1}) of the same asset (O_0 on the first row), cols 1..3 = 100*log(H|L|C / O).  Tolerances of
    test_log_returns_kernel_vs_reference_values; the f32 table is the f64 one rounded once."""
    from finenvs_b200.data import loader

    W = 8
    prices, seg_start, seg_len = _prices(W, A, seed=A, days=40)
    s = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32, keep_logret64=True)
    prev_close = np.concatenate([prices[:1, :, 0], prices[:-1, :, 3]], axis=0)
    want = np.empty_like(prices)
    want[..., 0] = 100.0 * np.log(prices[..., 0] / prev_close)
    want[..., 1:] = 100.0 * np.log(prices[..., 1:] / prices[..., :1])
    got = s.logret64.cpu().numpy()
    assert got.shape == prices.shape
    np.testing.assert_allclose(got, want, rtol=4e-16, atol=2e-14)
    assert_bits_equal(got.astype(np.float32), s.logret.cpu().numpy(), "f32 table")


@pytest.mark.parametrize("A", [1, 3])
def test_effective_len_nan_rows(A):
    """fe_effective_len (one warp per segment, lane l scans rows W+1+l, W+33+l, ...) equals feo_effective_len: the first
    NaN in column 0 of asset 0 at a row k > W ends the segment at k.  A zero or negative price makes the NaN."""
    from oracle import oracle as orc
    from finenvs_b200.data import loader

    W, bars, days = 10, 60, 10
    rng = np.random.default_rng(40 + A)
    T = W + bars * days
    shp = (T, 4) if A == 1 else (T, A, 4)
    prices = gbm_ohlc(rng, T, 0.01) if A == 1 else np.stack([gbm_ohlc(rng, T, 0.01, s0=50.0 + a) for a in range(A)], axis=1)
    assert prices.shape == shp
    firsts = W + bars * np.arange(days)
    seg_start, seg_len = firsts - W, np.full(days, W + bars, np.int32)
    a0 = (lambda r: (r,)) if A == 1 else (lambda r: (r, 0))

    def bad_open(d, k, asset=0):   # log(O / C_prev) and log(x / O) of row k: NaN in every column of that row
        prices[(int(seg_start[d]) + k,) + (() if A == 1 else (asset,)) + (0,)] = -1.0

    want = np.full(days, W + bars, np.int32)
    bad_open(0, W)                                   # row W: the first bar's own row, never tested -> ignored
    bad_open(1, W + 1); want[1] = W + 1
    bad_open(2, W + 40); want[2] = W + 40            # lane 7, second pass of the warp
    bad_open(3, W + 1 + 30); bad_open(3, W + 1 + 32 + 2); want[3] = W + 31   # lane 30 pass 1 beats lane 2 pass 2
    bad_open(4, W + bars - 1); want[4] = W + bars - 1                         # the segment's last row
    prices[a0(int(seg_start[5]) + W + 5) + (1,)] = -1.0                      # High < 0: NaN in column 1 only
    if A > 1:
        bad_open(6, W + 5, asset=1)                                          # another asset's NaN
    s = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float64, keep_logret64=True)
    lr = s.logret64.cpu().numpy().reshape(T, A, 4)
    assert np.isnan(lr[int(seg_start[5]) + W + 5, 0, 1]) and not np.isnan(lr[int(seg_start[5]) + W + 5, 0, 0])
    if A > 1:
        assert np.isnan(lr[int(seg_start[6]) + W + 5, 1, 0])
    fs = orc.series_from_prices(prices, seg_start, seg_len, W)   # the oracle's own log-returns and feo_effective_len
    got = s.seg_len.cpu().numpy()
    assert_bits_equal(fs.seg_len, got, "seg_len vs feo_effective_len")
    assert_bits_equal(want, got, "seg_len")
