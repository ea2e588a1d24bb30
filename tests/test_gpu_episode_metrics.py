"""Per-episode trading metrics (TimeSeriesEnv(track_metrics=True), fe_episode_metrics in csrc/fe_metrics.cu) against
the numpy restatement oracle/oracle_metrics.py: bit-exact records and aggregates on an adversarial series, the same
records from every step path and from a sharded population, evaluate mode's first-episode report, list overflow, no
launch when the feature is off, and a 1 Mi-env run on the c2 series."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import oracle_metrics as om
from parity_utils import gbm_ohlc

W = 8


def _adv_series(dtype, seed=5):
    """sigma = 0.15 bars (margin calls, bankruptcies) on 200 ragged days of 1..59 bars."""
    from finenvs_b200.data import loader

    rng = np.random.default_rng(seed)
    bars = rng.integers(1, 60, 200)
    prices = np.round(gbm_ohlc(rng, int(bars.sum()) + W, 0.15), 4)
    firsts = W + np.concatenate([[0], np.cumsum(bars)[:-1]])
    seg_start, seg_len = firsts - W, (bars + W).astype(np.int32)
    return loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype)


def _env(series, N, **kw):
    from finenvs_b200.environments import TimeSeriesEnv

    args = dict(num_intervals=series.window, device_id=0, series=series, num_envs=N, seed=9, random_reset="all",
                random_offset=True, obs_dtype=series.logret.dtype, track_metrics=True)
    args.update(kw)
    return TimeSeriesEnv("metrics", **args)


def _actions(T, N, seed=11):
    """(T, N, 1) f32 on the device, 60 % of them short (the adversarial branches need short positions)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.rand((T, N, 1), generator=g, device="cuda") * 2 - 1
    short = torch.rand((T, N, 1), generator=g, device="cuda") < 0.6
    return torch.where(short, -a.abs(), a).contiguous()


def _np(rec):
    return {k: v.cpu().numpy() for k, v in rec.items()}


def _assert_records_equal(got, want, what=""):
    assert set(got) == set(want)
    for k in om.RECORD_KEYS:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.dtype == b.dtype and a.shape == b.shape, (what, k, a.dtype, b.dtype, a.shape, b.shape)
        if a.dtype == np.float64:
            a, b = a.view(np.int64), b.view(np.int64)   # bit for bit
        bad = np.nonzero(a != b)[0]
        assert bad.size == 0, f"{what} {k}: {bad.size} mismatches, first at {bad[0]}: {got[k][bad[0]]!r} vs {want[k][bad[0]]!r}"


def _assert_summary(summary, rec, agg):
    s = {k: v.item() for k, v in summary.items()}
    assert s["episodes"] == agg["episodes"] and s["sum_len"] == agg["sum_len"]
    assert s["max_mdd"] == agg["max_mdd"]
    scale = om.abs_sums(rec)
    for k, bound in scale.items():   # f64 atomics in arbitrary order: within 1e-12 of the magnitude summed
        assert abs(s[k] - agg[k]) <= 1e-12 * bound, (k, s[k], agg[k], bound)


def _rollout(env, A, T):
    N = env.num_envs
    R = torch.empty((T, N), dtype=env.obs_dtype, device="cuda")
    D = torch.empty((T, N), dtype=torch.int32, device="cuda")
    env.reset()
    for t in range(T):
        _, r, d, _ = env.step(A[t])
        R[t], D[t] = r, d
    return R.cpu().numpy(), D.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_records_and_aggregates_match_the_oracle(dtype):
    N, T = 5003, 600
    env = _env(_adv_series(dtype), N, metrics_capacity=64 * N)
    R, D = _rollout(env, _actions(T, N), T)
    rec, agg = om.episode_metrics(R, D, env.starting_balance)
    assert np.bincount(rec["env"], minlength=N).min() >= 2
    assert (rec["mdd"] > 0).any() and (rec["return"] < 0).any() and (rec["return"] > 0).any()
    _assert_records_equal(_np(env.episode_metrics()), rec, str(dtype))
    _assert_summary(env.metrics_summary(), rec, agg)
    env.clear_metrics()
    assert env.episode_metrics()["key"].numel() == 0 and env.metrics_summary()["episodes"].item() == 0


@pytest.mark.gpu
def test_every_step_path_gives_the_same_records():
    from finenvs_b200.agents.PPO.buffer import Buffer

    N, T, chunk = 2051, 96, 32
    series = _adv_series(torch.float32)
    A = _actions(T, N, seed=3)
    out = {}

    env = _env(series, N)
    env.reset()
    for t in range(T):
        env.step(A[t])
    out["step"] = env.episode_metrics()

    env = _env(series, N)
    env.reset_lazy()
    for t in range(T):
        env.step_lazy(A[t])
    out["step_lazy"] = env.episode_metrics()

    env = _env(series, N)
    A_host = A.cpu()
    for t in range(T):
        env.step_host(A_host[t].contiguous(), packed_dones=True)
    out["step_host_packed"] = env.episode_metrics()

    env = _env(series, N)
    buf = Buffer(2, 0.99, 0, capacity=T)
    buf.bind_env(env, lazy=True)
    s = env.reset()
    for t in range(T):
        n, r, d, _ = env.step(A[t])
        buf.store(s, A[t], r, d, A[t], A[t])
        s = n
    out["bound_buffer"] = env.episode_metrics()

    env = _env(series, N)
    calls = [0]

    def policy(obs):   # called once in the warm-up, then once per captured step
        k = max(calls[0] - 1, 0)
        calls[0] += 1
        return A[k % chunk]

    roll = env.capture_rollout(policy, chunk)
    assert calls[0] == chunk + 1
    cap = []
    for rep in range(T // chunk):
        roll.replay()
        cap.append(env.episode_metrics())
        env.clear_metrics()
    # each replay feeds A[0:chunk] again: compare against eager stepping with the same schedule
    merged = {k: torch.cat([c[k] for c in cap]) for k in cap[0]}
    env2 = _env(series, N)
    env2.reset()
    for t in range(T):
        env2.step(A[t % chunk])
    _assert_records_equal(_np(merged), _np(env2.episode_metrics()), "captured")

    ref = _np(out["step"])
    assert ref["key"].size > N
    for name, rec in out.items():
        _assert_records_equal(_np(rec), ref, name)


@pytest.mark.gpu
def test_shards_give_the_records_of_one_population():
    N, T = 3001, 200
    series = _adv_series(torch.float64)
    A = _actions(T, N, seed=4)
    whole = _env(series, N)
    whole.reset()
    for t in range(T):
        whole.step(A[t])
    parts = []
    for base, n in ((0, 1500), (1500, 1501)):
        env = _env(series, n, env_id_base=base, total_envs=N)
        env.reset()
        for t in range(T):
            env.step(A[t, base:base + n])
        parts.append(env.episode_metrics())
    cat = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    order = torch.argsort(cat["key"])
    _assert_records_equal(_np({k: v[order] for k, v in cat.items()}), _np(whole.episode_metrics()), "shards")


@pytest.mark.gpu
def test_evaluate_policy_reports_each_envs_first_episode():
    from finenvs_b200.data import loader

    rng = np.random.default_rng(21)
    bars, days, N, steps = 40, 24, 300, 64   # every env's first episode ends within one 64-step replay
    prices = np.round(gbm_ohlc(rng, bars * days, 0.08), 4)
    seg_start, seg_len = loader.regular_segments(bars * days, bars, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    env = _env(series, N, evaluate=True, random_reset=None, random_offset=False)
    assert env.metrics_capacity == N

    def policy(obs):
        return torch.tanh(obs[:, -1, 3:4] * 3.0 + obs[:, -2, 0:1])

    first_step = 1
    roll = None
    for checkpoint in range(2):
        res = env.evaluate_policy(policy, steps_per_replay=steps, rollout=roll)
        roll = res["rollout"]
        assert res["steps"] == steps   # one replay: its static rewards / dones hold the whole trace
        R, D = roll.rewards.cpu().numpy(), roll.dones.cpu().numpy()
        rec, agg = om.episode_metrics(R, D, env.starting_balance, first_step=first_step, evaluate=True)
        assert rec["key"].size == N   # exactly one record per env, none carried over from the previous checkpoint
        by_env = np.argsort(rec["env"], kind="stable")
        _assert_records_equal(_np(res["metrics"]), {k: v[by_env] for k, v in rec.items()}, f"checkpoint {checkpoint}")
        np.testing.assert_allclose(res["metrics"]["return"].cpu().numpy(), res["returns"].cpu().numpy(), rtol=1e-4, atol=1e-2)
        # the metric reset emptied the list, the summary and the first-episode flags
        assert env.metrics_summary()["episodes"].item() == 0 and int(env._m_emitted.sum().item()) == 0
        first_step += steps


@pytest.mark.gpu
def test_overflow_is_counted_not_written():
    from finenvs_b200 import _lib

    N, T, cap = 1024, 120, 100
    env = _env(_adv_series(torch.float32), N, metrics_capacity=cap)
    R, D = _rollout(env, _actions(T, N, seed=8), T)
    rec, agg = om.episode_metrics(R, D, env.starting_balance)
    assert agg["episodes"] > cap
    assert env.metrics_summary()["episodes"].item() == agg["episodes"]
    with pytest.raises(RuntimeError, match="metrics_capacity"):
        env.episode_metrics()

    # raw ABI with guard entries behind the list; the step ordinal from a device counter
    guard, dev = 64, "cuda:0"
    p = env._params
    f64 = torch.zeros((6, N), dtype=torch.float64, device=dev)
    i32 = torch.zeros((2, N), dtype=torch.int32, device=dev)
    li = torch.full((2, cap + guard), -7, dtype=torch.int64, device=dev)
    ll = torch.full((cap + guard,), -7, dtype=torch.int32, device=dev)
    lf = torch.full((5, cap + guard), -7.0, dtype=torch.float64, device=dev)
    summ = torch.zeros(8, dtype=torch.int64, device=dev)
    st = _lib.FeMetricsState(i32[0].data_ptr(), i32[1].data_ptr(), *(f64[k].data_ptr() for k in range(6)), None,
                             li[0].data_ptr(), li[1].data_ptr(), ll.data_ptr(), *(lf[k].data_ptr() for k in range(5)),
                             summ.data_ptr())
    Rd, Dd = torch.from_numpy(R).to(dev), torch.from_numpy(D).to(dev)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    L = _lib.lib()
    for t in range(T):
        counter.fill_(t + 1)
        _lib.check(L.fe_episode_metrics(ctypes.byref(p), ctypes.byref(st), Rd[t].data_ptr(), Dd[t].data_ptr(), 0,
                                        counter.data_ptr(), cap, torch.cuda.current_stream().cuda_stream), "fe_episode_metrics")
    assert summ[0].item() == agg["episodes"]
    assert (li[:, cap:] == -7).all() and (ll[cap:] == -7).all() and (lf[:, cap:] == -7.0).all()
    # the entries that were written are oracle records (which ones won a slot depends on warp timing)
    keys = li[0, :cap].cpu().numpy()
    pos = np.minimum(np.searchsorted(rec["key"], keys), rec["key"].size - 1)
    assert (rec["key"][pos] == keys).all() and np.unique(keys).size == cap
    got = {"key": keys, "env": li[1, :cap].cpu().numpy(), "len": ll[:cap].cpu().numpy(),
           **{k: lf[j, :cap].cpu().numpy() for j, k in enumerate(("return", "sharpe", "mdd", "mdd_rel", "hit_rate"))}}
    _assert_records_equal(got, {k: v[pos] for k, v in rec.items()}, "raw list")


def _kernel_names(env, steps):
    from torch.profiler import ProfilerActivity, profile

    A = _actions(steps, env.num_envs, seed=1)
    env.reset()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for t in range(steps):
            env.step(A[t])
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


@pytest.mark.gpu
def test_no_launch_when_off():
    series = _adv_series(torch.float32)
    off = _kernel_names(_env(series, 4096, track_metrics=False), 10)
    assert any("fe_" in n for n in off) and not any("fe_episode_metrics_kernel" in n for n in off)
    on = _kernel_names(_env(series, 4096), 10)
    assert sum("fe_episode_metrics_kernel" in n for n in on) >= 10


@pytest.mark.gpu
def test_full_size_c2_one_mi_envs():
    import bench
    from finenvs_b200.data import loader

    N, T, S, Wc = 1 << 20, 300, 65536, 60
    prices, seg_start, seg_len, _ = bench.make_series("c2", Wc)
    series = loader.stage_series(prices, seg_start, seg_len, Wc, "cuda:0", torch.float32)
    env = _env(series, N, seed=bench.ACTION_SEED)
    g = torch.Generator(device="cuda").manual_seed(5)
    R = torch.empty((T, S), dtype=torch.float32, device="cuda")
    D = torch.empty((T, S), dtype=torch.int32, device="cuda")
    env.reset_lazy()
    for t in range(T):
        _, r, d, _ = env.step_lazy(torch.rand((N, 1), generator=g, device="cuda") * 2 - 1)
        R[t], D[t] = r[:S], d[:S]
    rec, _ = om.episode_metrics(R.cpu().numpy(), D.cpu().numpy(), env.starting_balance, total_envs=N)
    got = env.episode_metrics()
    sl = got["env"] < S
    assert rec["key"].size > 1000
    _assert_records_equal(_np({k: v[sl] for k, v in got.items()}), rec, "c2 slice")
    assert env.metrics_summary()["episodes"].item() == got["key"].numel()
