"""PPO rollout buffer that stores observations as 12-byte handles (Buffer.bind_env(env, lazy=True)) and builds shuffled
minibatches with fe_gather_obs (csrc/fe_step.cu): path policy, argument checks, bit-exactness against the dense
observations step() returns, a lock-step rollout against the dense buffer, and the reference's own PPO agent."""
import ctypes
import os

import numpy as np
import pytest
import torch

from baseline import reference as ref


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def _params(lib, W, f64=0, A=1, rows=258048, N=1 << 20):
    return lib.FeParams(N, 0, N, rows, W, 1024, A, 5, 10000.0, 0.01, 1.5, 0.25, 1, lib.RESET_ALL, 1, 0, f64, lib.VARIANT_AUTO, 0)


# ---------------------------------------------------------------------------------------------- host only
def test_gather_obs_path_policy(built):
    L = built.lib()

    def name(W, f64=0, A=1, rows=258048, table=True):
        p = _params(built, W, f64, A, rows)
        s = built.FeSeries(16, 16, 16, 16, 4096 if table else None)   # only obs_table == NULL matters to the policy
        return L.fe_gather_obs_kernel_name(ctypes.byref(p), ctypes.byref(s)).decode()

    for W in (24, 60, 100, 128):
        assert name(W) == "fe_gather_obs_kernel<float>", W
    for W in (50, 60):
        assert name(W, f64=1) == "fe_gather_obs_kernel<double>", W
    assert name(61) == "fe_materialize_kernel<float>"                  # 20 * 61 bytes is not a multiple of 16
    assert name(54, f64=1) == "fe_materialize_kernel<double>"          # half of 2160 bytes is not a whole 80-byte pitch
    assert name(60, table=False) == "fe_materialize_kernel<float>"
    assert name(60, rows=10_000_000) == "fe_materialize_kernel<float>"   # an 800 MB table would not stay in L2
    assert name(60, A=2).startswith("none")


def test_gather_obs_argument_errors(built):
    L = built.lib()
    p = _params(built, 60)
    s = built.FeSeries(16, 16, 16, 16, None)
    P, S = ctypes.byref(p), ctypes.byref(s)
    assert L.fe_gather_obs(None, S, 16, 16, None, 4, 16, None) == -1
    assert L.fe_gather_obs(P, None, 16, 16, None, 4, 16, None) == -1
    assert L.fe_gather_obs(P, S, None, 16, None, 4, 16, None) == -1
    assert L.fe_gather_obs(P, S, 16, None, None, 4, 16, None) == -1
    assert L.fe_gather_obs(P, S, 16, 16, None, 4, None, None) == -1
    assert L.fe_gather_obs(P, S, 16, 16, None, -1, 16, None) == -1
    assert L.fe_gather_obs(P, S, 16, 16, None, 4, 24, None) == -2      # output not 16-byte aligned
    assert L.fe_gather_obs(P, ctypes.byref(built.FeSeries(16, 16, 16, 16, 4104)), 16, 16, None, 4, 16, None) == -2
    pa = _params(built, 60, A=2)
    assert L.fe_gather_obs(ctypes.byref(pa), S, 16, 16, None, 4, 16, None) == -1
    assert L.fe_gather_obs(P, S, 16, 16, None, 0, 16, None) == 0        # nothing to do: no launch (fake pointers untouched)
    assert L.fe_gather_obs(P, S, 16, 16, 16, 0, 16, None) == 0


# ---------------------------------------------------------------------------------------------- GPU
def _series(W, dtype, bars=None, days=30, seed=2):
    from finenvs_b200.data import loader
    from parity_utils import gbm_ohlc

    bars = bars or W + 40
    rng = np.random.default_rng(seed)
    prices = np.round(gbm_ohlc(rng, bars * days, 0.02), 4)
    seg_start, seg_len = loader.regular_segments(bars * days, bars, W)
    return loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype)


def _twins(W, dtype, N, seed=5, series=None):
    from finenvs_b200.environments import TimeSeriesEnv

    series = series or _series(W, dtype)
    kw = dict(num_intervals=W, device_id=0, series=series, num_envs=N, seed=seed, random_reset="all", random_offset=True,
              obs_dtype=dtype)
    return TimeSeriesEnv("a", **kw), TimeSeriesEnv("b", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("W", [4, 8, 24, 60, 61, 100, 128, 390])
def test_gather_obs_equals_indexing_the_dense_observations(built, W, dtype):
    """fe_gather_obs over the handles of a few steps == the dense observations step() returned, indexed; with and
    without the observation-layout table (TMA / LSU path); duplicates, ragged counts, identity order == fe_materialize."""
    from finenvs_b200 import _lib

    N, T = 1000, 4
    dense_env, lazy_env = _twins(W, dtype, N)
    series = lazy_env.series
    table = series.obs_table()
    f64 = int(dtype == torch.float64)
    can_tma = built.lib().fe_obs_table_bytes(series.num_rows, W, f64) > 0
    assert (table is not None) == can_tma
    g = torch.Generator(device="cuda").manual_seed(W)
    dense = [dense_env.reset()]
    lo = lazy_env.reset_lazy()
    row0, pf = [lo.row0], [lo.posfeat]
    for t in range(T):
        a = torch.rand((N, 1), generator=g, device="cuda") * 2 - 1
        o, r, d, _ = dense_env.step(a)
        lo, r2, d2, _ = lazy_env.step_lazy(a)
        assert torch.equal(r, r2) and torch.equal(d, d2)
        dense.append(o)
        row0.append(lo.row0)
        pf.append(lo.posfeat)
    dense, row0, pf = torch.cat(dense), torch.cat(row0), torch.cat(pf)
    M = dense.shape[0]
    L = built.lib()
    for with_table in (True, False):
        fs = _lib.FeSeries(series.prices.data_ptr(), series.logret.data_ptr(), series.seg_start.data_ptr(),
                           series.seg_len.data_ptr(), table.data_ptr() if (with_table and table is not None) else None)
        kname = L.fe_gather_obs_kernel_name(lazy_env._pp, ctypes.byref(fs)).decode()
        assert kname.startswith("fe_gather_obs_kernel" if (with_table and can_tma) else "fe_materialize_kernel"), kname

        def gather(index, count):
            out = torch.full((count, W, 5), float("nan"), dtype=dtype, device="cuda")
            _lib.check(L.fe_gather_obs(lazy_env._pp, ctypes.byref(fs), row0.data_ptr(), pf.data_ptr(),
                                       index.data_ptr() if index is not None else None, count, out.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream), "fe_gather_obs")
            return out

        for count in (1, 3, 5, 4097):
            idx = torch.randint(0, M, (count,), generator=g, device="cuda")
            if count > 3:
                idx[count // 2:count // 2 + 3] = idx[0]       # duplicates
            assert torch.equal(gather(idx, count), dense[idx]), (with_table, count)
        assert torch.equal(gather(None, M), dense), with_table             # identity order
        for t in range(T + 1):   # fe_materialize on one step's handles == fe_gather_obs without an index == step()'s tensor
            out = torch.empty((N, W, 5), dtype=dtype, device="cuda")
            _lib.check(L.fe_materialize(lazy_env._pp, ctypes.byref(fs), row0[t * N:].data_ptr(), pf[t * N:].data_ptr(),
                                        out.data_ptr(), torch.cuda.current_stream().cuda_stream), "fe_materialize")
            assert torch.equal(out, dense[t * N:(t + 1) * N]), (with_table, t)


def _lockstep(dtype, W=60, N=3000, T=5, rollouts=2, flat_obs=False):
    from finenvs_b200.agents.PPO.buffer import Buffer, LazyStates
    from finenvs_b200.environments import TimeSeriesEnv

    series = _series(W, dtype)
    kw = dict(num_intervals=W, device_id=0, series=series, num_envs=N, seed=9, random_reset="all", random_offset=True,
              obs_dtype=dtype, flat_obs=flat_obs)
    env_d, env_l = TimeSeriesEnv("d", **kw), TimeSeriesEnv("l", **kw)
    buf_d, buf_l = Buffer(4, 0.97, 0, capacity=2), Buffer(4, 0.97, 0, capacity=2)   # both grow inside the first rollout
    buf_d.bind_env(env_d)
    buf_l.bind_env(env_l, lazy=True)
    if series.obs_table() is not None:
        assert env_l.gather_obs_kernel_name().startswith("fe_gather_obs_kernel")
    assert env_l.kernel_name() == env_d.kernel_name()     # the step kernel's own choice is untouched
    s_d, s_l = env_d.reset(), env_l.reset()
    assert torch.equal(s_d, s_l)
    g = torch.Generator(device="cuda").manual_seed(3)
    n_done = 0
    for rollout in range(rollouts):
        for t in range(T):
            a = torch.rand((N, 1), generator=g, device="cuda") * 2 - 1
            lp = torch.rand((N, 1), generator=g, device="cuda")
            v = torch.rand((N, 1), generator=g, device="cuda")
            n_d, r_d, d_d, _ = env_d.step(a)
            n_l, r_l, d_l, _ = env_l.step(a)
            assert torch.equal(n_d, n_l) and torch.equal(r_d, r_l) and torch.equal(d_d, d_l), (rollout, t)
            n_done += int(d_d.sum())
            buf_d.store(s_d, a, r_d, d_d, lp, v)
            buf_l.store(s_l, a, r_l, d_l, lp, v)
            s_d, s_l = n_d, n_l
        for k in ("_seg", "_ptr", "_cash", "_long", "_short", "_margin"):
            assert torch.equal(getattr(env_d, k), getattr(env_l, k)), k
        last = torch.rand((N, 1), generator=g, device="cuda")
        buf_d.prepare_training_data(last)
        buf_l.prepare_training_data(last)
        for k in ("returns", "advantages"):
            assert torch.equal(buf_d.container[k], buf_l.container[k]), k
        st = buf_l.container["states"]
        assert isinstance(st, LazyStates) and st.shape == buf_d.container["states"].shape and len(st) == T * N
        assert st.dtype == dtype and st.device == torch.device("cuda:0")
        assert torch.equal(st.materialize(), buf_d.container["states"])
        torch.manual_seed(100 + rollout)
        b_d = buf_d.get_batches()
        torch.manual_seed(100 + rollout)
        b_l = buf_l.get_batches()
        idx_d, idx_l = buf_d.get_mini_batch_indices(), buf_l.get_mini_batch_indices()
        for i_d, i_l in zip(idx_d, idx_l):
            assert torch.equal(b_l["states"][i_l, :], b_d["states"][i_d, :])
            assert torch.equal(b_l["states"][i_l], b_d["states"][i_d])
            for k in ("actions", "log_probs", "advantages", "returns"):
                assert torch.equal(b_l[k][i_l], b_d[k][i_d]), k
        assert torch.equal(b_l["states"][10:300], b_d["states"][10:300])
        assert torch.equal(b_l["states"][5:900:7, ...], b_d["states"][5:900:7])
        buf_d.clear()
        buf_l.clear()
    assert n_done > 0, "no episode ended: the rollout did not exercise dones and redraws"
    return buf_l, env_l


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_lockstep_rollout_dense_vs_handles(built, dtype):
    _lockstep(dtype)


@pytest.mark.gpu
def test_lockstep_rollout_short_window_flat_obs(built):
    _lockstep(torch.float32, W=8, N=1000, T=7, flat_obs=True)


@pytest.mark.gpu
def test_lazy_store_errors_and_storage_bound(built):
    from finenvs_b200.agents.PPO.buffer import Buffer
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv
    from parity_utils import gbm_ohlc

    W, N, T = 60, 2000, 6
    env, _ = _twins(W, torch.float64, N)
    buf = Buffer(2, 0.99, 0, capacity=4)
    buf.bind_env(env, lazy=True)
    s = env.reset()
    a = torch.zeros((N, 1), device="cuda")
    for t in range(T):
        n, r, d, _ = env.step(a)
        with pytest.raises(ValueError):
            buf.store(s.clone(), a, r, d, a, a)          # not the tensor the env returned
        buf.store(s, a, r, d, a, a)
        s = n
    cap = buf.capacity
    assert cap >= T
    nbytes = buf._row0.numel() * buf._row0.element_size() + buf._posfeat.numel() * buf._posfeat.element_size()
    assert nbytes <= (cap + 1) * N * 16
    # multi-asset envs have no handles
    rng = np.random.default_rng(0)
    bars, days, A = 100, 10, 2
    prices = np.stack([np.round(gbm_ohlc(rng, bars * days, 0.02), 4) for _ in range(A)], axis=1)
    seg_start, seg_len = loader.regular_segments(bars * days, bars, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    penv = TimeSeriesEnv("p", num_intervals=W, device_id=0, series=series, num_envs=64, seed=1)
    with pytest.raises(NotImplementedError):
        Buffer(2, 0.99, 0).bind_env(penv, lazy=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_full_size_c2_one_mi_envs(built, dtype):
    """1 Mi envs on the c2 series: a few lazily stored steps, then a 1 Mi-sample random gather == the dense observations."""
    import bench
    from finenvs_b200.agents.PPO.buffer import Buffer
    from finenvs_b200.data import loader

    W, N, T = 60, 1 << 20, 3
    prices, seg_start, seg_len, _ = bench.make_series("c2", W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dtype)
    env_l, env_d = _twins(W, dtype, N, seed=4, series=series)
    buf = Buffer(16, 0.99, 0, capacity=T)
    buf.bind_env(env_l, lazy=True)
    assert env_l.gather_obs_kernel_name().startswith("fe_gather_obs_kernel")
    s_l, s_d = env_l.reset(), env_d.reset()
    kept = [s_d]
    for t in range(T):
        a = torch.rand((N, 1), device="cuda") * 2 - 1
        n_l, r_l, d_l, _ = env_l.step(a)
        n_d, r_d, d_d, _ = env_d.step(a)
        assert torch.equal(n_l, n_d) and torch.equal(r_l, r_d) and torch.equal(d_l, d_d)
        buf.store(s_l, a, r_l, d_l, a, a)
        s_l = n_l
        if t < T - 1:
            kept.append(n_d)
        del n_d
    buf.prepare_training_data(torch.zeros((N, 1), device="cuda"))
    dense = torch.cat(kept)
    del kept
    idx = torch.randint(0, T * N, (N,), device="cuda")
    assert torch.equal(buf.container["states"][idx], dense[idx])


@pytest.mark.gpu
@pytest.mark.skipif(not ref.available(), reason="baseline/_ref (the reference tree) is absent")
def test_reference_ppo_lstm_agent_trains_with_a_lazy_buffer(built, tmp_path, monkeypatch):
    """The loop of test_gpu_reference_agents.py with the reference's PPOAgentLSTM, its buffer replaced by a Buffer bound
    lazily: the agent's own train() consumes LazyStates minibatches."""
    ref.import_reference()
    monkeypatch.setenv("FINENVS_DATA_DIR", os.path.join(ref.REF_DST, "finenvs", "data"))
    monkeypatch.chdir(tmp_path)
    from finenvs.agents.PPO.PPO_agent import PPOAgentLSTM

    from finenvs_b200.agents.PPO.buffer import Buffer
    from finenvs_b200.environments import TimeSeriesEnv

    torch.manual_seed(602585557)
    env = TimeSeriesEnv(instrument_name="SPY", dataset_key="dummy", num_intervals=4)
    env_args = env.get_env_args()
    num_envs = env_args["num_envs"]
    batch_size = num_envs * 64
    agent = PPOAgentLSTM(env_args=env_args, num_epochs=4, num_mini_batches=4, hidden_dim=1024, model_save_interval=0,
                         write_to_csv=False)
    old = agent.buffer
    agent.buffer = Buffer(getattr(old, "num_mini_batches", 4), getattr(old, "gamma", 0.99), 0)
    agent.buffer.bind_env(env, lazy=True)
    states = env.reset()
    trained = 0
    for it in range(150):
        (actions, log_probs, values) = agent.step(states)
        (next_states, rewards, dones, _) = env.step(actions)
        agent.store(states, actions, rewards, dones, log_probs, values)
        states = next_states
        if agent.get_buffer_size() >= batch_size:
            before = [p.detach().clone() for p in agent.actor.parameters()]
            agent.train(states)
            trained += 1
            assert any(not torch.equal(a, b) for a, b in zip(before, agent.actor.parameters())), "train() changed nothing"
            assert agent.get_buffer_size() == 0
    assert trained == 2
    assert all(torch.isfinite(p).all() for p in agent.actor.parameters())
    assert all(torch.isfinite(p).all() for p in agent.critic.parameters())
