"""Per-episode trading metrics without a GPU: the numpy restatement on a hand-computed trace, fe_episode_metrics'
argument checks (rejected before any CUDA call) and the cross-rank reduction of the summary over gloo."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle_metrics as om


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def test_oracle_hand_computed_trace():
    # env 0: a 2-step episode of zero rewards (sharpe 0), then 4 steps whose equity rises to +30 and ends at -15
    # env 1: +1 / -1 alternating, done every second step (three episodes; evaluate keeps only the first)
    rewards = np.array([[0, 1], [0, -1], [10, 1], [20, -1], [-50, 1], [5, -1]], np.float32)
    dones = np.array([[0, 0], [1, 1], [0, 0], [0, 1], [0, 0], [1, 1]], np.int32)
    rec, agg = om.episode_metrics(rewards, dones, 100.0, env_id_base=4, total_envs=10)
    assert rec["key"].tolist() == [2 * 10 + 4, 2 * 10 + 5, 4 * 10 + 5, 6 * 10 + 4, 6 * 10 + 5]
    assert rec["env"].tolist() == [4, 5, 5, 4, 5]
    assert rec["len"].tolist() == [2, 2, 2, 4, 2]
    assert rec["return"].tolist() == [0.0, 0.0, 0.0, -15.0, 0.0]
    # the second episode of env 0: mean -3.75, population variance 2968.75 / 4
    assert rec["sharpe"][0] == 0.0
    assert rec["sharpe"][3] == pytest.approx(-3.75 / math.sqrt(742.1875), rel=1e-15)
    assert rec["mdd"][3] == 50.0 and rec["mdd_rel"][3] == 50.0 / 130.0 and rec["hit_rate"][3] == 0.75
    assert rec["mdd"][0] == 0.0 and rec["hit_rate"][0] == 0.0
    # env 1: +1 then -1: peak 1, drawdown 1 (relative to equity 101), sharpe 0 / 1
    for k in (1, 2, 4):
        assert rec["sharpe"][k] == 0.0 and rec["mdd"][k] == 1.0 and rec["mdd_rel"][k] == 1.0 / 101.0
        assert rec["hit_rate"][k] == 0.5
    assert agg["episodes"] == 5 and agg["sum_len"] == 12 and agg["max_mdd"] == 50.0
    assert agg["sum_mdd"] == 53.0 and agg["sum_return"] == -15.0 and agg["sum_hit_rate"] == 2.25
    ev, ev_agg = om.episode_metrics(rewards, dones, 100.0, env_id_base=4, total_envs=10, evaluate=True)
    assert ev["key"].tolist() == [24, 25] and ev_agg["episodes"] == 2


def _state(lib, cap_ptrs=True, emitted=None):
    f = [16] * 8 + [emitted] + ([16] * 9 if cap_ptrs else [None] * 8 + [16])
    return lib.FeMetricsState(*f)


def test_metrics_argument_errors(built):
    L = built.lib()
    N = 1 << 10
    p = built.FeParams(N, 0, N, 4096, 60, 16, 1, 5, 10000.0, 0.01, 1.5, 0.25, 1, built.RESET_ALL, 1, 0, 0,
                       built.VARIANT_AUTO, 0)
    P, M = ctypes.byref(p), ctypes.byref(_state(built))
    assert L.fe_episode_metrics(None, M, 16, 16, 1, None, 8, None) == -1
    assert L.fe_episode_metrics(P, None, 16, 16, 1, None, 8, None) == -1
    assert L.fe_episode_metrics(P, M, None, 16, 1, None, 8, None) == -1
    assert L.fe_episode_metrics(P, M, 16, None, 1, None, 8, None) == -1
    assert L.fe_episode_metrics(P, M, 16, 16, 1, None, -1, None) == -1
    assert L.fe_episode_metrics(P, ctypes.byref(_state(built, cap_ptrs=False)), 16, 16, 1, None, 8, None) == -1
    for k in range(len(built.FeMetricsState._fields_)):
        if built.FeMetricsState._fields_[k][0] == "emitted":
            continue
        s = _state(built)
        setattr(s, built.FeMetricsState._fields_[k][0], None)
        assert L.fe_episode_metrics(P, ctypes.byref(s), 16, 16, 1, None, 8, None) == -1, built.FeMetricsState._fields_[k][0]
    pe = built.FeParams(N, 0, N, 4096, 60, 16, 1, 5, 10000.0, 0.01, 1.5, 0.25, 1, built.RESET_KEEP, 0, 1, 0,
                        built.VARIANT_AUTO, 0)
    assert L.fe_episode_metrics(ctypes.byref(pe), M, 16, 16, 1, None, 8, None) == -1   # evaluate needs the emitted flags
    p0 = built.FeParams(0, 0, N, 4096, 60, 16, 1, 5, 10000.0, 0.01, 1.5, 0.25, 1, built.RESET_ALL, 1, 0, 0,
                        built.VARIANT_AUTO, 0)
    assert L.fe_episode_metrics(ctypes.byref(p0), M, 16, 16, 1, None, 8, None) == -1


def test_summary_layout(built):
    assert ctypes.sizeof(built.FeMetricsState) == 18 * 8
    assert built.METRICS_SUMMARY_BYTES == 2 * 8 + 6 * 8 and len(built.METRICS_SUMMARY_KEYS) == 8


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from finenvs_b200 import parallel as par

    par.init_distributed("gloo")
    f = lambda x: torch.tensor(x, dtype=torch.float64)
    summary = {"episodes": torch.tensor(3 + rank), "sum_len": torch.tensor(40 * (rank + 1)), "sum_return": f(1.5 * rank),
               "sum_sharpe": f(0.25), "sum_sharpe_sq": f(0.125), "sum_mdd": f(2.0 + rank), "max_mdd": f([7.0, 5.0][rank]),
               "sum_hit_rate": f(1.0)}
    out = par.all_reduce_episode_metrics(summary)
    assert out == {"episodes": 7, "sum_len": 120, "sum_return": 1.5, "sum_sharpe": 0.5, "sum_sharpe_sq": 0.25,
                   "sum_mdd": 5.0, "sum_hit_rate": 2.0, "max_mdd": 7.0}
    dist.destroy_process_group()


def test_all_reduce_episode_metrics_gloo():
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
