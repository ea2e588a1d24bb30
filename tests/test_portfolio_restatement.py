"""A > 1 (portfolio extension): two INDEPENDENT restatements must agree.

`oracle/fe_oracle.c: feo_step_multi` (explicit casts, scalar C) against `tests/portfolio_restatement.py` (torch dtype
promotion, built on one real reference TimeSeriesEnv per asset).  First the torch restatement is pinned where a
reference exists: at A = 1 it must reproduce the reference's own step() bit for bit.  Then both are stepped in lock-step
for A in {2, 5, 30} on violent series (sigma up to 0.15, short-biased actions, ragged days) that reach margin calls at
High and Close, margin releases, blocked long and short entries and bankruptcies — the branches where the definition's
"one cash movement per phase / greedy walk over the assets" could be misread.

Runs where the reference checkout exists (this container); the CUDA portfolio kernels are compared with feo_step_multi
on the GPU box (tests/test_gpu_parity.py), so agreement here carries over to them.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from oracle import ref_harness as rh
from parity_utils import assert_bits_equal, day_labels, gbm_ohlc
from portfolio_restatement import PortfolioRestatement, butterfly_sum

needs_reference = pytest.mark.skipif(not rh.available(), reason="reference checkout not present")


def _asset_csvs(tmp_path, A, bars, sigmas, seed, s0=lambda a: 20.0 + 13.0 * a):
    rng = np.random.default_rng(seed)
    dates, times = day_labels(len(bars), bars)
    paths = []
    for a in range(A):
        d = tmp_path / f"asset{a}"
        d.mkdir()
        p = str(d / "series.csv")
        rh.write_csv(p, dates, times, gbm_ohlc(rng, sum(bars), sigmas[a % len(sigmas)], s0=s0(a)))
        paths.append(p)
    return paths


def _short_biased(frac, spread=1.0):
    def act(r, shape):
        a = r.uniform(-spread, spread, shape)
        m = r.uniform(0, 1, shape) < frac
        a[m] = -np.abs(a[m])
        return a.astype(np.float32)
    return act


def _build(paths, W, N, **ref_kw):
    refs = [rh.RefEnv(p, "dummy", W, seed=7, evaluate=True, **ref_kw) for p in paths]
    flats = [rh.flat_series_from_ref(r) for r in refs]
    for f in flats[1:]:
        assert np.array_equal(f.seg_start, flats[0].seg_start) and np.array_equal(f.seg_len_raw, flats[0].seg_len_raw)
    A = len(paths)
    if A == 1:
        fs = flats[0]
    else:
        fs = orc.series_from_prices(np.stack([f.prices for f in flats], axis=1), flats[0].seg_start, flats[0].seg_len_raw, W,
                                    logret=np.stack([f.logret for f in flats], axis=1))
    port = PortfolioRestatement([r.env for r in refs], N)
    return refs, fs, port


def _state(port):
    return {"cash": port.cash.numpy().reshape(-1).copy(), "long": port.long_shares.numpy().copy(),
            "short": port.short_shares.numpy().copy(), "margin": port.margin.numpy().astype(np.float64).copy(),
            "ptr": port.e[0].env_pointers.numpy().astype(np.int32).copy()}


def test_butterfly_sum_is_the_warp_order():
    x = torch.tensor(np.random.default_rng(0).normal(0, 1e6, (64, 30)))
    want = np.empty(64)
    for i in range(64):
        w = np.zeros(32)
        w[:30] = x[i].numpy()
        for off in (16, 8, 4, 2, 1):
            w = w + w[np.arange(32) ^ off]
        want[i] = w[0]
    assert np.array_equal(butterfly_sum(x).numpy().reshape(-1), want)
    one = torch.tensor([[3.25], [-0.5]])
    assert torch.equal(butterfly_sum(one), one)


@needs_reference
@pytest.mark.parametrize("sigma,frac,seed", [(0.12, 0.7, 31), (0.03, 0.9, 32), (0.15, 0.55, 33)])
def test_restatement_equals_the_real_reference_at_one_asset(tmp_path, sigma, frac, seed):
    """The pin: same torch ops in the same order as time_series_env.py:277-521 when A = 1."""
    bars = [30, 7, 30, 22, 1, 30, 30, 16]
    W, N, steps = 6, 96, 260
    (path,) = _asset_csvs(tmp_path, 1, bars, [sigma], seed, s0=lambda a: 100.0)
    refs, fs, port = _build([path], W, N)
    real = rh.RefEnv(path, "dummy", W, seed=7, evaluate=True)      # the unmodified reference, stepped through ITS step()
    real.widen(np.arange(N) % fs.num_segments)
    try:
        assert_bits_equal(real.reset(), port.observe().numpy(), "reset obs")
        rng = np.random.default_rng(seed + 1)
        act = _short_biased(frac)
        terminated = np.zeros(N, bool)      # `real` runs in evaluate mode (no redraw): :527-528 zero the rewards of
        n_done = 0                          # envs whose first episode is over; the restatement has no such bookkeeping
        for t in range(steps):
            a = act(rng, (N, 1))
            ro, rr, rd, info = real.step(a)
            po, pr, pd_ = port.step(torch.from_numpy(a))
            assert_bits_equal(rd, pd_.numpy(), f"dones t={t}")
            assert_bits_equal(rr, np.where(terminated, 0.0, pr.numpy()), f"rewards t={t}")
            terminated |= rd.astype(bool)
            if info:
                terminated[:] = False       # :531-534 all episodes over: metrics cleared
            n_done += int(rd.sum())
            assert_bits_equal(ro, po.numpy(), f"obs t={t}")
            s = real.state()
            assert_bits_equal(s["cash"], port.cash.numpy().reshape(-1), f"cash t={t}")
            assert_bits_equal(s["long_sh"], port.long_shares.numpy().reshape(-1), f"long t={t}")
            assert_bits_equal(s["short_sh"], port.short_shares.numpy().reshape(-1), f"short t={t}")
            assert_bits_equal(s["margin"], port.margin.numpy().astype(np.float64).reshape(-1), f"margin t={t}")
            assert_bits_equal(s["ptr"], port.e[0].env_pointers.numpy().astype(np.int32), f"ptr t={t}")
        assert n_done > 2 * N
    finally:
        real.close()
        for r in refs:
            r.close()


@needs_reference
@pytest.mark.parametrize("A,sigmas,frac,seed,params", [
    (2, [0.12, 0.05], 0.7, 41, {}),
    (5, [0.15, 0.02, 0.08, 0.12, 0.05], 0.6, 42, {}),
    (30, [0.10, 0.03, 0.15, 0.06], 0.65, 43, {}),
    (5, [0.12, 0.08], 0.5, 44, dict(max_shares=40, starting_balance=2500.0, per_share_commission=0.37,
                                    initial_margin_requirement=2.25, maintenance_margin_requirement=0.4)),
    (30, [0.2, 0.1], 0.8, 45, dict(max_shares=12, starting_balance=900.0, per_share_commission=0.05,
                                   initial_margin_requirement=1.2, maintenance_margin_requirement=0.3)),
])
def test_two_restatements_agree_for_several_assets(tmp_path, A, sigmas, frac, seed, params):
    bars = [30, 7, 30, 22, 1, 30, 30, 16]
    W, N, steps = 6, 64, 200
    paths = _asset_csvs(tmp_path, A, bars, sigmas, seed)
    refs, fs, port = _build(paths, W, N, **params)
    okw = {}
    if params:
        okw = dict(max_shares=params["max_shares"], starting_balance=params["starting_balance"],
                   commission=params["per_share_commission"], imr=params["initial_margin_requirement"],
                   mmr=params["maintenance_margin_requirement"])
    o = orc.OracleEnv(fs, num_envs=N, evaluate=False, reset_mode=orc.RESET_KEEP, seg_init=np.arange(N) % fs.num_segments,
                      out_f64=True, **okw)
    try:
        assert o.multi and o.A == A
        assert_bits_equal(o.reset(), port.observe().numpy(), "reset obs")
        rng = np.random.default_rng(seed + 1)
        act = _short_biased(frac, spread=1.2)
        seen = dict(done=0, blocked_long=0, blocked_short=0, margin_call=0, bankrupt=0, short_open=0)
        for t in range(steps):
            a = act(rng, (N, A))
            before = _state(port)
            po, pr, pd_ = port.step(torch.from_numpy(a))
            oo, orr, od, _ = o.step(a)
            assert_bits_equal(od, pd_.numpy(), f"dones t={t}")
            assert_bits_equal(orr, pr.numpy(), f"rewards t={t}")
            assert_bits_equal(oo, po.numpy(), f"obs t={t}")
            s = _state(port)
            assert_bits_equal(o.cash, s["cash"], f"cash t={t}")
            assert_bits_equal(o.long_sh.reshape(N, A), s["long"], f"long t={t}")
            assert_bits_equal(o.short_sh.reshape(N, A), s["short"], f"short t={t}")
            assert_bits_equal(o.margin.reshape(N, A), s["margin"], f"margin t={t}")
            assert_bits_equal(o.ptr, s["ptr"], f"ptr t={t}")
            # which rare branches did this step reach (evidence that the comparison is not vacuous)
            ms = params.get("max_shares", 5)
            want = np.clip(np.rint(a * np.float32(ms + 0.5)), -ms, ms)
            alive = od == 0
            grew_long = s["long"] - before["long"]
            grew_short = s["short"] - before["short"]
            seen["done"] += int(od.sum())
            seen["blocked_long"] += int(((want > before["short"]) & (grew_long == 0) & (before["long"] == 0) & alive[:, None]).sum())
            seen["blocked_short"] += int(((-want > before["long"]) & (grew_short == 0) & (before["short"] == 0) & alive[:, None]).sum())
            seen["short_open"] += int((grew_short > 0).sum())
            seen["margin_call"] += int((s["margin"] > before["margin"]).sum())
            seen["bankrupt"] += int((od.astype(bool) & (s["ptr"] == 0) & (before["ptr"] + 1 + W < fs.seg_len[np.arange(N) % fs.num_segments])).sum())
        assert seen["done"] > 0 and seen["short_open"] > 0 and seen["margin_call"] > 0, seen
        assert seen["bankrupt"] > 0 or (A < 5 and not params), seen
        print("branches reached:", seen)
        if params or A >= 30:   # with the default balance two or five assets never exhaust the account
            assert seen["blocked_long"] + seen["blocked_short"] > 0, seen
    finally:
        for r in refs:
            r.close()
