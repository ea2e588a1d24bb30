#!/usr/bin/env python
"""PPO rollout storage (SURVEY.md 8f-3): finenvs_b200.agents.PPO.Buffer against the reference's storage scheme.

    python tools/ppo_storage.py [--envs 65536] [--window 60] [--steps 64]

One rollout = `steps` x (random actions -> env.step -> buffer.store) + prepare_training_data.  Compared:
  reference scheme  buffer.py:33-63 / :80-100 restated here for the comparison: every key re-grown with
                    torch.cat(dim=1) per step, returns/advantages by the Python loop of ~6 torch ops per time step
                    (same env, same observations; f32 to keep the memory comparable — the reference stores f64)
  Buffer            pre-allocated time-major storage, observations written in place by the step kernel (bind_env),
                    returns/advantages by one launch of fe_returns_advantages
Prints one JSON line: ms per rollout for both, bytes the returns kernel moves and its GB/s, max |difference| of the returns.

    python tools/ppo_storage.py --states dense|handles|both [--envs 1048576] [--steps 64] [--dtype f32|f64]

Observation storage of the Buffer instead: `dense` (bind_env(env): (T+1, N, W, 5) values, shuffle() copies them) against
`handles` (bind_env(env, lazy=True): 12-byte handles, minibatches gathered by fe_gather_obs).  Per mode: ms per rollout
with store, ms for one epoch (get_batches() + materialising every minibatch), torch.cuda.max_memory_allocated (a mode
that runs out of memory is recorded as such).  Then fe_gather_obs alone: 1 Mi random indices into 64 x 1 Mi handles on
the same series (f32 and f64): TMA path against the warp-per-sample path (fe_materialize_kernel) on the same handles in
identity order, GB written per second and its fraction of the measured 6522.7 GB/s; and step() of an unbound env
against the lazily bound step() (fe_step_lazy + fe_gather_obs).  One JSON line, with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--window", type=int, default=60)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--rollouts", type=int, default=3)
    ap.add_argument("--states", choices=("dense", "handles", "both"), default=None)
    ap.add_argument("--dtype", choices=("f32", "f64"), default="f32")
    args = ap.parse_args()
    if args.states is not None:
        return storage_modes(args)

    import bench
    from finenvs_b200.agents.PPO import Buffer
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    W, N, T = args.window, args.envs, args.steps
    prices, seg_start, seg_len, _ = bench.make_series("c2", W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    kw = dict(num_intervals=W, device_id=0, series=series, num_envs=N, seed=1, random_reset="all", random_offset=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.rand((N, 1), generator=g, device="cuda") * 2 - 1 for _ in range(T)]
    vals = [torch.rand((N, 1), generator=g, device="cuda") for _ in range(T + 1)]
    gamma = 0.99

    def ev():
        return torch.cuda.Event(enable_timing=True)

    # ---- reference scheme
    env = TimeSeriesEnv("ref", **kw)
    ref_ms, ref_returns = [], None
    for _ in range(args.rollouts):
        cont = {}
        s0 = env.reset()
        torch.cuda.synchronize()
        t0, t1, t2 = ev(), ev(), ev()
        t0.record()
        for t in range(T):
            s1, r, d, _ = env.step(acts[t])
            for key, x in (("states", s0), ("actions", acts[t]), ("rewards", r.unsqueeze(-1)), ("dones", d.unsqueeze(-1)),
                           ("values", vals[t])):
                x = x.unsqueeze(1)                                   # buffer.py:58-63 time axis at dim 1
                cont[key] = x if key not in cont else torch.cat((cont[key], x), dim=1)   # :51-56
            s0 = s1
        t1.record()
        rewards, dones, values = cont["rewards"], cont["dones"], cont["values"]           # (N, T, 1)
        returns = torch.zeros_like(rewards)
        cur = vals[T]
        for t in reversed(range(T)):                                                      # :90-98
            cur = rewards[:, t, :] + (1 - dones[:, t, :]) * gamma * cur
            returns[:, t, :] = cur
        adv = returns - values
        t2.record()
        torch.cuda.synchronize()
        ref_ms.append((t0.elapsed_time(t1), t1.elapsed_time(t2)))
        ref_returns = returns.transpose(0, 1).contiguous()
        del cont, returns, adv

    # ---- Buffer
    env = TimeSeriesEnv("buf", **kw)
    buf = Buffer(16, gamma, 0, capacity=T)
    buf.bind_env(env)
    our_ms = []
    zeros = torch.zeros((N, 1), device="cuda")
    for _ in range(args.rollouts):
        buf.clear()
        s0 = env.reset()
        torch.cuda.synchronize()
        t0, t1, t2 = ev(), ev(), ev()
        t0.record()
        for t in range(T):
            s1, r, d, _ = env.step(acts[t])
            buf.store(s0, acts[t], r, d, zeros, vals[t])
            s0 = s1
        t1.record()
        buf.compute_returns_and_advantages(vals[T])
        t2.record()
        torch.cuda.synchronize()
        our_ms.append((t0.elapsed_time(t1), t1.elapsed_time(t2)))
    ours = buf.container["returns"]
    bytes_moved = T * N * (4 + 4 + 4 + 4 + 4) + 4 * N    # rewards, dones, values read; returns, advantages written
    out = {
        "workload": f"{N} envs, W={W}, {T}-step rollouts, f32",
        "reference_scheme_ms": {"rollout_store": ref_ms[-1][0], "returns_advantages": ref_ms[-1][1]},
        "buffer_ms": {"rollout_store": our_ms[-1][0], "returns_advantages": our_ms[-1][1]},
        "returns_kernel_bytes": bytes_moved, "returns_kernel_GBps": bytes_moved / (our_ms[-1][1] * 1e-3) / 1e9,
        "returns_max_abs_diff_vs_reference_scheme": float((ours - ref_returns).abs().max()),
        "same_env_trajectory": True,
    }
    print(json.dumps(out), flush=True)


HBM_MEASURED_GBPS = 6522.7   # measured copy bandwidth of the B200 (DESIGN.md)


def _card():
    import subprocess

    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # pragma: no cover
        out = f"unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out}


def _time_ms(fn, iters=20, warmup=3):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def storage_modes(args):
    import gc

    import bench
    from finenvs_b200.agents.PPO import Buffer
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    W, N, T = args.window, args.envs, args.steps
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    prices, seg_start, seg_len, _ = bench.make_series("c2", W)
    series = {dt: loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", dt) for dt in (torch.float32, torch.float64)}
    kw = dict(num_intervals=W, device_id=0, num_envs=N, seed=1, random_reset="all", random_offset=True)
    out = {"workload": f"c2 series, {N} envs, W={W}, {T}-step rollouts, {args.dtype}, 16 minibatches", "card": _card()}
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((T, N, 1), generator=g, device="cuda") * 2 - 1
    zeros = torch.zeros((N, 1), device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    modes = ("dense", "handles") if args.states == "both" else (args.states,)
    for mode in modes:
        gc.collect()            # a bound env and its buffer reference each other: free the previous mode's storage
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        rec, env, buf, batch, s0, s1 = {}, None, None, None, None, None
        try:
            env = TimeSeriesEnv(mode, series=series[dtype], obs_dtype=dtype, **kw)
            buf = Buffer(16, 0.99, 0, capacity=T)
            buf.bind_env(env, lazy=(mode == "handles"))
            rollout_ms, epoch_ms = [], []
            for r in range(args.rollouts):
                buf.clear()
                s0 = env.reset()
                torch.cuda.synchronize()
                t0, t1, t2 = ev(), ev(), ev()
                t0.record()
                for t in range(T):
                    s1, rew, d, _ = env.step(acts[t])
                    buf.store(s0, acts[t], rew, d, zeros, zeros)
                    s0 = s1
                t1.record()
                buf.prepare_training_data(zeros)
                torch.cuda.synchronize()
                t1b = ev()
                t1b.record()
                batch = buf.get_batches()
                for idx in buf.get_mini_batch_indices():
                    mb = batch["states"][idx, :]
                    del mb
                t2.record()
                torch.cuda.synchronize()
                rollout_ms.append(t0.elapsed_time(t1))
                epoch_ms.append(t1b.elapsed_time(t2))
            rec = {"rollout_with_store_ms": rollout_ms, "epoch_get_batches_and_16_minibatches_ms": epoch_ms,
                   "max_memory_allocated_GB": torch.cuda.max_memory_allocated() / 1e9}
        except torch.cuda.OutOfMemoryError as e:
            rec = {"out_of_memory": str(e).splitlines()[0],
                   "max_memory_allocated_GB_before_failure": torch.cuda.max_memory_allocated() / 1e9}
        env = buf = batch = s0 = s1 = None   # what the failed mode allocated must not count against the next one
        out[mode] = rec
        gc.collect()
        torch.cuda.empty_cache()

    # ---- fe_gather_obs alone: 1 Mi random samples out of a 64 x 1 Mi-handle rollout
    from finenvs_b200 import _lib

    kern = {}
    M, B = 64 << 20, 1 << 20
    for dt in (torch.float32, torch.float64):
        name = "f64" if dt == torch.float64 else "f32"
        env = TimeSeriesEnv("kernel", series=series[dt], obs_dtype=dt, **{**kw, "num_envs": 1024})
        Buffer(16, 0.99, 0).bind_env(env, lazy=True)     # builds the gather FeSeries with the observation-layout table
        rows = series[dt].num_rows
        row0 = torch.randint(0, rows - W, (M,), generator=g, device="cuda")
        pf = torch.rand((M,), generator=g, device="cuda", dtype=dt)
        idx = torch.randint(0, M, (B,), generator=g, device="cuda")
        sel_row0, sel_pf = row0[idx], pf[idx]
        obs = torch.empty((B, W, 5), dtype=dt, device="cuda")
        ref_obs = torch.empty_like(obs)
        stream = torch.cuda.current_stream().cuda_stream

        def launch(series_ptr, r0, p, index, o):
            _lib.check(env._L.fe_gather_obs(env._pp, series_ptr, r0.data_ptr(), p.data_ptr(),
                                            index.data_ptr() if index is not None else None, B, o.data_ptr(), stream),
                       "fe_gather_obs")

        bytes_out = B * W * 5 * obs.element_size()
        res = {"tma_kernel": env._L.fe_gather_obs_kernel_name(env._pp, env._pgs).decode(),
               "lsu_kernel": env._L.fe_gather_obs_kernel_name(env._pp, env._ps).decode(), "bytes_written": bytes_out}
        for label, sp, r0, p, index in (("tma_random_index", env._pgs, row0, pf, idx),
                                        ("lsu_identity_baseline", env._ps, sel_row0, sel_pf, None),
                                        ("tma_identity", env._pgs, sel_row0, sel_pf, None),
                                        ("lsu_random_index", env._ps, row0, pf, idx)):
            ms = _time_ms(lambda: launch(sp, r0, p, index, obs))
            res[label] = {"ms": ms, "GBps_written": bytes_out / (ms * 1e-3) / 1e9,
                          "fraction_of_measured_hbm": bytes_out / (ms * 1e-3) / 1e9 / HBM_MEASURED_GBPS}
        launch(env._pgs, row0, pf, idx, obs)
        launch(env._ps, sel_row0, sel_pf, None, ref_obs)
        res["tma_random_equals_lsu_identity"] = bool(torch.equal(obs, ref_obs))
        kern[name] = res
        del row0, pf, idx, sel_row0, sel_pf, obs, ref_obs
        torch.cuda.empty_cache()
    out["fe_gather_obs"] = kern

    # ---- step(): unbound vs bound lazily (fe_step_lazy + fe_gather_obs), same population
    step = {}
    for label in ("plain", "lazy_bound"):
        env = TimeSeriesEnv(label, series=series[dtype], obs_dtype=dtype, **kw)
        if label == "lazy_bound":
            Buffer(16, 0.99, 0, capacity=4).bind_env(env, lazy=True)
        env.reset()
        step[label] = {"ms": _time_ms(lambda: env.step(acts[0])), "kernel": env.kernel_name()}
        del env
    step["lazy_bound"]["gather_kernel"] = kern["f64" if dtype == torch.float64 else "f32"]["tma_kernel"]
    out["step_ms"] = step
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
