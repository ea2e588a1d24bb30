#!/usr/bin/env python
"""bench.py — env-steps/s of the fused trading-env step kernel (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of envs: one fe_step launch over this GPU's envs.
Default workload = BASELINE config 2 (single asset, 1 Mi envs per GPU, W=60, synthetic GBM daily bars).
N>1 is launched by torchrun, one rank per GPU; envs are sharded (weak scaling: 1 Mi envs per GPU), the
series is replicated, the step needs no collective.  Rank 0 prints ONE JSON line.

Timing: W warm-up steps, then exactly K timed steps right behind them, split into `blocks` blocks that run back to
back (a CUDA event on the launch stream at every block boundary, barrier + synchronize before the warm-up and after
the K steps, max over ranks per block); `value` / `ms_per_step` come from the MEDIAN block's time per step, `timing`
also gives min and max — a 20-step block is 5 ms, one block alone is at the mercy of a clock ramp.
The default K = 200 (ten 20-step blocks) gave 4.712, 4.718 and 4.714 G env-steps/s in three c2 runs on one B200 at
1000 W.  Longer windows are not steadier: the per-step time rises from 0.222 ms over steps 10-210 to about 0.25 ms
towards step 600 (median SM clock 1957 MHz against 1965 at K = 200), so K = 600 gave 4.31 - 4.36 across three runs.

--dump-outputs DIR: after the timed steps, rank 0 writes what the timed call (step_into) returned in the last
step as float32 .npy files: rewards.npy (N,), dones.npy (N,) as 0/1, obs.npy (N, W, 5A).  An array larger than
its share of 48 MB in all is replaced by the rows of a fixed, seeded sample of envs (sorted env indices drawn
with DUMP_SEED).  Series, actions and env seeds are fixed, so the same arguments give the same inputs on every
run and two builds can be compared output for output.

value    = device-resident throughput through TimeSeriesEnv.step_into (caller-owned outputs, actions in HBM).
public_step = the same loop through the drop-in call TimeSeriesEnv.step(actions) (allocates obs/rewards/dones).
e2e      = the same metric through the host-buffer C-ABI call fe_step_host_packed (TimeSeriesEnv.step_host(packed_dones=True)):
           per step 4N bytes of actions pinned-host -> HBM and 4N (rewards f32) + N/8 (dones, 1 bit per env) bytes HBM ->
           pinned host; the observation stays in HBM for the policy.  e2e.int32_dones = the same through fe_step_host
           (dones as int32: 8N bytes back).
roofline = DRAM bytes per launch / average launch duration (live, CUDA events), against MEASURED_PEAKS.json hbm_gbs.
           DRAM bytes = the ncu-measured dram__bytes_read+write of this kernel and configuration (profiles/traffic.json,
           `traffic`) when recorded, else the algorithmic bytes that must cross DRAM.  Beside it: `dram_algorithmic_*`
           (DESIGN.md: 2264 B per env-step at A=1, W=60, f32 obs, MINUS the 960 B of window reads while the table is
           L2-resident: those never reach DRAM, and counting them gave round 1 a "fraction" of 1.34) and `algorithmic_*`
           (all 2264 B).
also     = the other BASELINE workloads measured in the same process (N=1: c4, c3, c5 and c1; N>1: c4 and c5), same protocol;
           c1 = the reference's native size (1024 envs), the configuration cpu_baseline times the reference on (at least
           300 timed steps: a step there takes microseconds);
           c5 = the ES population rollout (policy forward + env step + return bookkeeping per step, EvoAgent.train() per
           generation; perturbations are stored as fp16 where the reference draws f32).
collectives (N>1) = device time of the NCCL collectives the path uses outside the step (episode statistics
           all-reduce, ES fitness all-gather, ES gradient all-reduce).
cpu_baseline / --impl reference = the reference's OWN TimeSeriesEnv.step (unmodified, from baseline/_ref,
           device_id=-1) on the box's host cores, thread count forced: at its native 1024 envs, widened to 65 536, and at
           the GPU arm's own 1 Mi envs (`same_config_run`, ~2.6 s per step; skipped on hosts with < 64 GB free); `value` is
           the BEST of the all-thread runs (conservative); the C/OpenMP oracle port is reported beside it as `cpu_port`.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
SERIES_SEED = 20260101
ACTION_SEED = 1234
DUMP_SEED = 4321
DUMP_BYTES = {"obs": 32 << 20, "rewards": 8 << 20, "dones": 8 << 20}   # --dump-outputs: 48 MB in all
L2_RESIDENT_BYTES = 48 << 20   # the library's own threshold for the "cached" flavour (fe_step.cu: pick_pipe_stages)


# ------------------------------------------------------------------------------ workloads ----
def algorithmic_bytes_per_env_step(W: int, A: int = 1, obs_bytes: int = 4) -> int:
    """SURVEY.md §8(d): window read + obs write + OHLC row + state r/w + tables + action + reward + done."""
    window_read = W * 4 * A * obs_bytes
    obs_write = W * 5 * A * obs_bytes
    ohlc = 32 * A
    cash = 8
    per_asset_state = A * (8 + 8 + 16)   # long, short (f32 r+w), margin (f64 r+w)
    pointer = 8
    tables = 12                           # segment id 4 r, seg_start 8 r (seg_len shares the line)
    return window_read + obs_write + ohlc + cash + per_asset_state + pointer + tables + 4 * A + obs_bytes + 4


def window_read_bytes(W: int, A: int = 1, obs_bytes: int = 4) -> int:
    return W * 4 * A * obs_bytes


WORKLOAD_ASSETS = {"c1": 1, "c2": 1, "c4": 1, "c3": 30}
WORKLOAD_DEFAULTS = {"c1": (1024, 60), "c2": (1 << 20, 60), "c4": (1 << 20, 60), "c3": (65536, 128)}   # (envs per GPU, window)
WORKLOAD_SERIES = {"c1": (1024 * 252, 252, 0.01), "c2": (1024 * 252, 252, 0.01), "c3": (1024 * 252, 252, 0.01), "c4": (10_000_000, 390, 0.0005)}

WORKLOAD_NAMES = {
    "c1": "single-asset synthetic GBM daily-bar TimeSeriesEnv, 1024 envs, 60-step window, random actions (the reference's native size)",
    "c3": "30-asset portfolio-allocation env, 65536 envs, 128-step window, transaction costs, 1 B200",
    "c2": "single-asset env, 1M envs, 60-step window, fused step kernel on 1 B200 vs reference",
    "c4": "synthetic minute-bar series of 10M timesteps, 1M envs per GPU with random start offsets, env-sharded",
    "c5": "ES population rollout (finenvs_b200.agents.ES.EvoAgent) with 512Ki envs per GPU (4M across 8), fitness over NCCL",
}


_SERIES_CACHE: dict = {}


def make_series(workload: str, W: int):
    """Synthetic GBM OHLC (SURVEY.md §8d recipe) + segment table.  The 10 M-row c4 series (320 MB, seconds of host time)
    is kept for the second workload that uses it (also.c5)."""
    if (workload, W) in _SERIES_CACHE:
        return _SERIES_CACHE[(workload, W)]
    out = _make_series(workload, W)
    if workload == "c4":
        _SERIES_CACHE[(workload, W)] = out
    return out


def _make_series(workload: str, W: int):
    from finenvs_b200.data import loader
    from parity_utils import gbm_ohlc

    rng = np.random.default_rng(SERIES_SEED)
    T, bars, sigma = WORKLOAD_SERIES[workload]
    if workload == "c3":     # 30 independent GBM assets, time-major (T, A, 4)
        prices = np.stack([np.round(gbm_ohlc(rng, T, sigma, s0=20.0 + 7 * a), 4) for a in range(WORKLOAD_ASSETS["c3"])], axis=1)
    else:
        prices = np.round(gbm_ohlc(rng, T, sigma), 4)
    seg_start, seg_len = loader.regular_segments(T, bars, W)
    return prices, seg_start, seg_len, {"rows": T, "bars_per_segment": bars, "sigma": sigma}


def workload_config(workload: str, envs: int, window: int, world: int):
    return {"workload": WORKLOAD_NAMES[workload], "envs_per_gpu": envs, "total_envs": envs * world,
            "window": window, "assets": WORKLOAD_ASSETS[workload], "obs_dtype": "float32",
            "reset": "all envs redraw (segment, offset), Philox",
            "parallelism": f"env-sharded x{world}, series replicated, no per-step collective",
            "l2": "per-step working set (obs >= 1.2 GB + state) >> 126 MB L2: no flush needed",
            **dict(zip(("rows", "bars_per_segment", "sigma"), WORKLOAD_SERIES[workload]))}


# ------------------------------------------------------------------------------ clocks -------
class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)   # NVML queries take driver locks: poll gently, the timed legs last seconds in total

    def __enter__(self):
        if self._nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._t is not None:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------ CPU legs -----
def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def force_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs must use the cores the box has.  Call before torch / the
    oracle library initialise their OpenMP runtimes (and set them explicitly afterwards as well)."""
    n = str(host_threads())
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[k] = n


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_port_throughput(W: int, workload: str, sample_envs: int, steps: int, warmup: int, budget_s: float | None):
    """The oracle port (oracle/fe_oracle.c, the reference's algorithm restated in C + OpenMP) stepped on all host
    threads over a bounded sample of the workload.  Returns (env-steps/s, seconds per step, threads, steps timed)."""
    from oracle import oracle as orc

    prices, seg_start, seg_len, _ = make_series(workload, W)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W)
    env = orc.OracleEnv(fs, num_envs=sample_envs, seed=ACTION_SEED, reset_mode=orc.RESET_ALL, random_offset=True,
                        out_f64=False)
    orc.lib().feo_set_num_threads(host_threads())
    threads = orc.lib().feo_num_threads()
    rng = np.random.default_rng(ACTION_SEED)
    A = WORKLOAD_ASSETS[workload]
    acts = [rng.uniform(-1, 1, sample_envs * A).astype(np.float32) for _ in range(4)]
    obs = np.empty((sample_envs, W, 5 * A), np.float32)
    rewards = np.empty(sample_envs, np.float32)
    dones = np.empty(sample_envs, np.int32)
    import ctypes as C

    def one(i):
        env.step_count += 1
        fn = orc.lib().feo_step_multi if env.multi else orc.lib().feo_step
        fn(C.byref(env.p), C.byref(env.s), C.byref(env.st), orc._p(acts[i % 4]), orc._p(obs),
           orc._p(rewards), orc._p(dones), env.step_count, None)

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    done_steps = 0
    for i in range(steps):
        one(i)
        done_steps += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s and done_steps >= 3:
            break
    dt = time.perf_counter() - t0
    return sample_envs * done_steps / dt, dt / done_steps, threads, done_steps


class ReferenceRunner:
    """The UNMODIFIED reference env (baseline/_ref, finenvs/environments/time_series_env.py:14-536) on the host cores.

    Inputs = BASELINE config 1 as SURVEY §8d restates it: the c2 GBM daily-bar series written as a reference-format
    CSV (1024 dates x 252 one-minute-labelled bars), W=60 => D=1023 days, N=1024 envs natively; widened to more envs by
    re-assigning the state tensors exactly as SURVEY App. C.4 does (env i on day i mod D).  Actions: pre-generated
    torch.rand((N,1), CPU generator seed 1234)*2-1 (BASELINE.md §3)."""

    def __init__(self, W: int = 60):
        import datetime
        import tempfile

        import torch
        from baseline import reference as ref

        ref.import_reference()
        from finenvs.environments.time_series_env import TimeSeriesEnv as RefEnv

        self.torch = torch
        self.W = W
        prices, _, _, _ = make_series("c2", W)
        T, bars, _ = WORKLOAD_SERIES["c2"]
        self._tmp = tempfile.mkdtemp(prefix="fe_refbench_", suffix="_data")   # the path must contain "data" (:47-51)
        day0 = datetime.date(1998, 1, 2)
        t0 = time.perf_counter()
        with open(os.path.join(self._tmp, "dummy.csv"), "w") as f:
            lines = []
            for d in range(T // bars):
                date = (day0 + datetime.timedelta(days=d)).strftime("%m/%d/%Y")
                for j in range(bars):
                    o, h, l, c = prices[d * bars + j]
                    lines.append(f"{date},{9 + (30 + j) // 60:02d}:{(30 + j) % 60:02d},{o:.4f},{h:.4f},{l:.4f},{c:.4f},0\n")
            f.writelines(lines)
        torch.manual_seed(ACTION_SEED)
        self.env = RefEnv(self._tmp, "dummy", num_intervals=W, device_id=-1)
        self.construct_s = time.perf_counter() - t0
        self.native_envs = int(self.env.num_envs)
        self.D = self.native_envs - 1

    def close(self):
        import shutil

        shutil.rmtree(self._tmp, ignore_errors=True)

    def widen(self, N: int):
        torch, e = self.torch, self.env
        e.env_indices = torch.arange(N, dtype=torch.int64) % self.D
        e.num_envs = N
        e.env_pointers = torch.zeros((N,), dtype=torch.int64)
        e.env_spots = torch.arange(0, e.num_intervals).repeat(N, 1)
        e.cash = e.starting_balance * torch.ones((N, 1))
        e.long_shares = torch.zeros((N, 1))
        e.short_shares = torch.zeros((N, 1))
        e.margin = torch.zeros((N, 1))
        if hasattr(e, "current_close_prices"):   # :426 reset() keys "no step yet" on this attribute
            del e.current_close_prices

    def run(self, N: int, threads: int, steps: int, warmup: int, budget_s: float | None):
        """(env-steps/s, seconds per step, steps timed) of TimeSeriesEnv.step at N envs with `threads` torch threads."""
        torch = self.torch
        torch.set_num_threads(threads)
        self.widen(N)
        g = torch.Generator().manual_seed(ACTION_SEED)
        acts = [torch.rand((N, 1), generator=g) * 2 - 1 for _ in range(4)]
        self.env.reset()
        for i in range(warmup):
            self.env.step(acts[i % 4])
        t0 = time.perf_counter()
        n = 0
        for i in range(steps):
            self.env.step(acts[i % 4])
            n += 1
            if budget_s is not None and time.perf_counter() - t0 > budget_s and n >= 3:
                break
        dt = time.perf_counter() - t0
        return N * n / dt, dt / n, n


def host_mem_available_gb() -> float:
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def reference_baseline(W: int, steps: int, warmup: int, budget_each_s: float, with_single_thread: bool, port_workload: str,
                       widened_envs: int = 65536, full_envs: int = 0):
    """All CPU numbers of one run: the real reference at C1 (N=1024), widened to N=65 536 and — full_envs > 0, the host has
    the memory (the step makes ~25 GB of transient copies at 1 Mi envs) — at the GPU arm's own population; and the C port."""
    import torch
    from baseline import reference as ref

    ncpu = host_threads()
    out = {"cores": ncpu, "cpu_count": os.cpu_count(), "cpu_model": cpu_model(), "torch": torch.__version__, "runs": []}
    best = None
    if ref.available():
        rr = ReferenceRunner(W)
        out["reference_constructor_s"] = rr.construct_s
        sizes = [rr.native_envs] + ([widened_envs] if widened_envs > rr.native_envs else [])
        plan = [(n, ncpu) for n in sizes] + ([(n, 1) for n in sizes] if with_single_thread else [])
        if full_envs > max(sizes) and host_mem_available_gb() >= 64.0:
            plan.append((full_envs, ncpu))   # the exact configuration of the GPU arm: ~2.6 s per step, all threads only
        for N, th in plan:
            wu = warmup if N <= 4096 else 1
            v, sps, n = rr.run(N, th, steps if N <= 4096 else (max(3, min(steps, 8)) if N <= 65536 else 3), wu, budget_each_s)
            run = {"impl": "reference TimeSeriesEnv.step (torch eager, device_id=-1)", "envs": N, "threads": th, "value": v,
                   "ms_per_step": sps * 1e3, "steps": n}
            out["runs"].append(run)
            if th == ncpu and (best is None or v > best["value"]):
                best = run
            if N == full_envs and th == ncpu:
                out["same_config_run"] = run
        rr.close()
    sample = min(WORKLOAD_DEFAULTS[port_workload][0], 262144 // WORKLOAD_ASSETS[port_workload] // (2 if port_workload == "c3" else 1))
    pv, psps, pth, pn = cpu_port_throughput(WORKLOAD_DEFAULTS[port_workload][1], port_workload, sample, 10_000, 3, min(budget_each_s, 8.0))
    out["cpu_port"] = {"value": pv, "unit": UNIT, "cores": pth, "kind": "port", "ms_per_step": psps * 1e3,
                       "sample": f"{sample} envs per step, {pn} steps, oracle/fe_oracle.c (OpenMP, {pth} threads), workload {port_workload}"}
    out["best"] = best
    return out


def cpu_baseline_block(rb: dict) -> dict:
    best = rb["best"]
    if best is None:   # no reference tree on this box: the port is all there is
        p = rb["cpu_port"]
        return {**p, "cpu_port": p, "note": "baseline/_ref absent: oracle port only"}
    return {"value": best["value"], "unit": UNIT, "cores": best["threads"], "kind": "reference", "tree": "baseline/_ref",
            "sample": (f"unmodified reference TimeSeriesEnv.step, c2 series as CSV, W=60, {best['envs']} envs per step "
                       f"({'C1 native' if best['envs'] <= 4096 else 'widened, SURVEY App. C.4'}), {best['steps']} steps, "
                       f"torch.set_num_threads({best['threads']}); best of the all-thread runs"),
            "ms_per_step": best["ms_per_step"], "cpu_count": rb["cpu_count"], "cpu_model": rb["cpu_model"], "torch": rb["torch"],
            "runs": rb["runs"], "cpu_port": rb["cpu_port"],
            **({"same_config_run": rb["same_config_run"]} if "same_config_run" in rb else
               {"not_timed": "the reference step at the GPU arm's full population (~25 GB of transient copies per step at 1 Mi envs)"})}


def run_reference_arm(args, rank: int):
    """--impl reference: the reference's own CPU implementation on the box's host cores."""
    if rank != 0:
        return
    force_host_threads()
    full = args.envs if (args.workload == "c2" and args.ref_widened_envs > 0) else 0
    rb = reference_baseline(60, args.steps, args.warmup, 45.0, True, args.workload, args.ref_widened_envs, full)
    cb = cpu_baseline_block(rb)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
        "config": workload_config(args.workload, args.envs, args.window, args.gpus),
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ GPU arm ------
class Timer:
    """Exactly `steps` timed steps in back-to-back blocks right behind the warm-up, a CUDA event at every block boundary,
    barrier + synchronize before the warm-up and after the last block, max over ranks per block."""

    def __init__(self, torch, dist, dev, world):
        self.torch, self.dist, self.dev, self.world = torch, dist, dev, world

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def blocks(self, fn, steps: int, warmup: int, nblocks: int, wall: bool = False):
        """Returns [(ms, steps)] per block; the block sizes differ by at most one and add up to `steps`."""
        torch = self.torch
        stream = torch.cuda.current_stream()
        nblocks = max(1, min(nblocks, steps))
        sizes = [steps // nblocks + (b < steps % nblocks) for b in range(nblocks)]
        events = [torch.cuda.Event(enable_timing=True) for _ in range(nblocks + 1)]
        self.sync_all()
        k = 0
        for _ in range(warmup):   # still queued when the first event is recorded: the device never idles in between
            fn(k)
            k += 1
        walls = [time.perf_counter()]
        events[0].record(stream)
        for b, n in enumerate(sizes):
            for _ in range(n):
                fn(k)
                k += 1
            events[b + 1].record(stream)
            walls.append(time.perf_counter())
        self.sync_all()
        ms = [events[b].elapsed_time(events[b + 1]) for b in range(nblocks)]
        if wall:   # a host-synchronous call: the wall clock is the larger of the two
            ms = [max(t, (walls[b + 1] - walls[b]) * 1e3) for b, t in enumerate(ms)]
        v = torch.tensor(ms, dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(v, op=self.dist.ReduceOp.MAX)
        return [(float(x), n) for x, n in zip(v.tolist(), sizes)]


def summarize(blocks, total_envs: int):
    per_step = [ms / n for ms, n in blocks]
    med, lo, hi = float(np.median(per_step)), float(min(per_step)), float(max(per_step))
    return {"value": total_envs / (med * 1e-3), "ms_per_step": med,
            "timing": {"blocks": len(blocks), "timed_steps": sum(n for _, n in blocks),
                       "steps_per_block": [n for _, n in blocks], "ms_per_step_median": med,
                       "ms_per_step_min": lo, "ms_per_step_max": hi}}


def dump_sample(n: int, row_bytes: int, budget: int):
    """Sorted indices of a fixed, seeded sample of n rows that fits `budget` bytes; None when all n rows fit."""
    k = max(1, budget // row_bytes)
    if k >= n:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))


def dump_outputs(out_dir: str, torch, outputs: dict):
    """--dump-outputs: the timed call's outputs of its last step as float32 .npy files (module docstring)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        idx = dump_sample(t.shape[0], t[0].numel() * 4, DUMP_BYTES[name])
        if idx is not None:
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def load_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def roofline_block(workload: str, W: int, N: int, A: int, kernel_s: float, table_bytes: int, kernel_name: str):
    peak, peak_src = load_peak()
    alg = algorithmic_bytes_per_env_step(W, A)
    resident = table_bytes <= L2_RESIDENT_BYTES
    dram_alg = alg - (window_read_bytes(W, A) if resident else 0)
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(f"{workload}_w{W}_n{N}")
    except Exception:
        pass
    alg_dram_gbs = dram_alg * N / kernel_s / 1e9
    # what DRAM carried: the ncu-measured bytes of this exact configuration when recorded, else the algorithmic bytes that
    # must cross DRAM.  (c3's 124 MB table is about the size of L2: part of its window reads are hits, which only the
    # measurement can tell.)
    achieved = traffic / kernel_s / 1e9 if traffic else alg_dram_gbs
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "basis": ("ncu dram__bytes_read+write of this kernel and configuration (profiles/traffic.json) / live launch time" if traffic
                      else "algorithmic bytes that must cross DRAM / live launch time"),
            "peak_source": f"of {peak_src}",
            "dram_algorithmic_bytes_per_env_step": dram_alg, "dram_algorithmic_achieved": alg_dram_gbs,
            "dram_algorithmic_frac": alg_dram_gbs / peak,
            "note": ("log-return table is L2-resident: the window reads (W*16*A B per env-step) never reach DRAM and are not part of "
                     "dram_algorithmic_*; algorithmic_* counts them" if resident else
                     "log-return table >= L2: dram_algorithmic_* = algorithmic_*"),
            "algorithmic_bytes_per_env_step": alg, "algorithmic_achieved": alg * N / kernel_s / 1e9,
            "algorithmic_frac": alg * N / kernel_s / 1e9 / peak,
            "kernel": kernel_name, "kernel_ms": kernel_s * 1e3,
            "dram_gbs": (traffic / kernel_s / 1e9) if traffic else None,
            "dram_frac": (traffic / kernel_s / 1e9 / peak) if traffic else None}


def measure_workload(torch, par, loader, timer, workload, N, W, rank, world, local_rank, steps, warmup, nblocks, variant,
                     full: bool, dump_dir: str | None = None):
    """One workload on this rank's GPU.  full=True adds the public step() and the host-buffer (e2e) legs;
    dump_dir: rank 0 writes the device-resident leg's last outputs there (--dump-outputs)."""
    dev = f"cuda:{local_rank}"
    A = WORKLOAD_ASSETS[workload]
    total = N * world
    prices, seg_start, seg_len, meta = make_series(workload, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, dev, torch.float32)
    del prices
    env = par.make_sharded_env(total, rank, world, "bench", num_intervals=W, device_id=local_rank, series=series,
                               seed=ACTION_SEED, random_reset="all", random_offset=True, variant=variant)
    assert env.num_envs == N
    g = torch.Generator(device=dev).manual_seed(ACTION_SEED + rank)
    ring = [torch.rand((N, A), generator=g, device=dev) * 2 - 1 for _ in range(8)]   # inputs resident in HBM
    obs = torch.empty((N, W, 5 * A), dtype=torch.float32, device=dev)
    rewards = torch.empty(N, dtype=torch.float32, device=dev)
    dones = torch.empty(N, dtype=torch.int32, device=dev)

    out = {}
    dev_blocks = timer.blocks(lambda i: env.step_into(ring[i % 8], obs, rewards, dones), steps, warmup, nblocks)
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, torch, {"obs": obs, "rewards": rewards, "dones": dones})
    res = summarize(dev_blocks, total)
    kernel_s = res["ms_per_step"] * 1e-3   # only fe_step launches sit between the events
    table_bytes = int(series.logret.numel() * series.logret.element_size())
    res["roofline"] = roofline_block(workload, W, N, A, kernel_s, table_bytes, env.kernel_name())
    res["episodes_finished_last_step"] = int(dones.sum().item())
    launches_per_step = 2 if " + " in env.kernel_name() else 1
    launches = launches_per_step * steps
    out.update(res)
    if full:
        del obs
        held = []

        def public_step(i):
            held.clear()
            held.append(env.step(ring[i % 8]))   # fresh obs / rewards / dones every call, like the reference

        pub = summarize(timer.blocks(public_step, steps, warmup, nblocks), total)
        held.clear()
        out["public_step"] = {"value": pub["value"], "unit": UNIT, "ms_per_step": pub["ms_per_step"], "timing": pub["timing"],
                              "api": "TimeSeriesEnv.step(actions) -> (obs, rewards, dones, info): allocates its outputs"}
        launches += launches_per_step * steps
        ring_host = [a.cpu().pin_memory() for a in ring[:4]]
        check = [0.0]

        # step_host returns the same pinned result buffers every call (documented): a host-side consumer wraps them once
        _, r_h, d_h, _ = env.step_host(ring_host[0], packed_dones=True)
        r_np, d_np = r_h.numpy(), d_h.numpy()

        def host_step(i):
            env.step_host(ring_host[i % 4], packed_dones=True)
            check[0] += float(r_np[0]) + int(d_np[0])   # the host reads the step's result

        e2e = summarize(timer.blocks(host_step, steps, warmup, nblocks, wall=True), total)
        h2d, d2h = env.host_bytes_per_step(packed_dones=True)
        out["e2e"] = {"value": e2e["value"], "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "ms_per_step": e2e["ms_per_step"], "timing": e2e["timing"],
                      "api": "TimeSeriesEnv.step_host(packed_dones=True) -> fe_step_host_packed (pinned host buffers; rewards f32, "
                             "dones 1 bit per env)"}
        launches += launches_per_step * steps   # the persistent kernels pack the dones themselves

        _, r_h, d_h, _ = env.step_host(ring_host[0])
        r_np32, d_np32 = r_h.numpy(), d_h.numpy()

        def host_step_i32(i):
            env.step_host(ring_host[i % 4])
            check[0] += float(r_np32[0]) + int(d_np32[0])

        e2e32 = summarize(timer.blocks(host_step_i32, steps, warmup, nblocks, wall=True), total)
        h2d32, d2h32 = env.host_bytes_per_step()
        out["e2e"]["int32_dones"] = {"value": e2e32["value"], "ms_per_step": e2e32["ms_per_step"], "h2d_bytes_per_step": h2d32,
                                     "d2h_bytes_per_step": d2h32, "api": "TimeSeriesEnv.step_host -> fe_step_host"}
        launches += launches_per_step * steps
    out["gpu_launches"] = launches
    out["meta"] = meta
    del env, series, ring
    torch.cuda.empty_cache()
    return out


def measure_es_rollout(rank: int, world: int, local_rank: int):
    """BASELINE config 5 at this GPU count: 512 Ki envs per GPU (4 Mi on 8), each env its own ES population member, the
    reference's ES loop (examples/isaac_gym/ES_MLP_Isaac_Gym.py:30-38) on the drop-ins: policy forward + env step + return
    bookkeeping per step, EvoAgent.train() (fitness all-gather, gradient all-reduce over NCCL when world > 1) per
    generation.  tools/es_rollout.py is the same loop as a script."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import es_rollout

    steps, gens, n = 64, 3, 524288
    rec = es_rollout.run(rank, world, local_rank, envs_per_gpu=n, steps=steps, generations=gens, make_series=make_series)
    g = rec["generations"]
    med = float(np.median([x["ms_per_step"] for x in g]))
    return {"workload": WORKLOAD_NAMES["c5"], "envs_per_gpu": n, "total_envs": n * world, "window": rec["window"], "assets": 1,
            "value": n * world / (med * 1e-3), "unit": UNIT, "ms_per_step": med,
            "what_a_step_is": "policy forward (perturbed MLP per env, window read straight from the staged 10 M-row series) + env step "
                              "+ return bookkeeping: 3 launches, no observation tensor, no host sync",
            "train_ms_per_generation": float(np.median([x["train_ms"] for x in g])), "steps_per_generation": steps,
            "generations": gens, "episodes_ranked_per_generation": g[-1]["episodes_ranked"],
            "parameters_identical_on_all_ranks": all(x["parameters_identical_on_all_ranks"] for x in g),
            "network_shape": rec["network_shape"], "perturbation_storage": rec["perturbation_storage"],
            "fitness_gather": rec["fitness_gather"], "kernels_per_step": rec["kernels_per_step"],
            "gpu_launches": 3 * steps * gens}


def measure_collectives(torch, dist, par, dev, world, N):
    """Device time (CUDA events, max over ranks) of the collectives the path uses outside the step."""
    def timed(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    stats = torch.zeros(5, dtype=torch.float64, device=dev)
    fit = torch.rand(N, device=dev)
    out = {"world": world, "unit": "us", "backend": dist.get_backend()}
    out["episode_stats_all_reduce_5xf64"] = timed(lambda: dist.all_reduce(stats, op=dist.ReduceOp.SUM))
    out[f"es_fitness_all_gather_{N}xf32_per_rank"] = timed(lambda: par.all_gather_fitness(fit, N * world))
    for name, n in (("300-8-1", 2417), ("300-256-256-1", 143105)):
        grad = torch.zeros(n, device=dev)
        out[f"es_gradient_all_reduce_{name}_{n}xf32"] = timed(lambda: dist.all_reduce(grad, op=dist.ReduceOp.SUM))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per measured leg (module docstring: Timing)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4"])
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: 1 Mi; c3: 65536)")
    ap.add_argument("--window", type=int, default=None, help="default 60; c3: 128")
    ap.add_argument("--variant", default="auto")
    ap.add_argument("--blocks", type=int, default=None,
                    help="how many blocks the K timed steps are split into (default: K // 20, at least 3 and at most 10)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-widened-envs", type=int, default=65536,
                    help="second size the unmodified reference is timed at (SURVEY App. C.4 widening); 0 = native N=1024 only")
    ap.add_argument("--no-also", action="store_true", help="skip the other workloads / collectives")
    ap.add_argument("--no-c5", action="store_true", help="skip the ES population rollout (also.c5)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to its GPU's NUMA-local CPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed call's outputs of its last step to DIR/<name>.npy (float32, a seeded sample of "
                         "envs where an array exceeds its share of 48 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU arm's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3)
    args.envs = args.envs or WORKLOAD_DEFAULTS[args.workload][0]
    args.window = args.window or WORKLOAD_DEFAULTS[args.workload][1]
    nblocks = args.blocks or max(3, min(10, args.steps // 20))

    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist

    from finenvs_b200 import parallel as par
    from finenvs_b200.data import loader

    prev_affinity = None
    if not args.no_numa_bind:   # before the CUDA context and any pinned allocation exist
        prev_affinity = par.bind_to_gpu_numa(int(os.environ.get("LOCAL_RANK", "0")))
    rank, world, local_rank = par.init_distributed("nccl")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    timer = Timer(torch, dist, dev, world)

    sampler = ClockSampler(local_rank)
    with sampler:
        main_res = measure_workload(torch, par, loader, timer, args.workload, args.envs, args.window, rank, world, local_rank,
                                    args.steps, args.warmup, nblocks, args.variant, full=True, dump_dir=args.dump_outputs)
    also, collectives = {}, None
    if not args.no_also:
        others = [w for w in (("c4", "c3") if world == 1 else ("c4",)) if w != args.workload]
        for w in others:
            n, win = WORKLOAD_DEFAULTS[w]
            r = measure_workload(torch, par, loader, timer, w, n, win, rank, world, local_rank, args.steps, args.warmup,
                                 nblocks, "auto", full=False)
            also[w] = {"workload": WORKLOAD_NAMES[w], "envs_per_gpu": n, "window": win, "assets": WORKLOAD_ASSETS[w],
                       "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "timing": r["timing"],
                       "kernel": r["roofline"]["kernel"], "frac": r["roofline"]["frac"], "dram_frac": r["roofline"]["dram_frac"],
                       "algorithmic_frac": r["roofline"]["algorithmic_frac"], "roofline": r["roofline"],
                       "gpu_launches": r["gpu_launches"]}
        if not args.no_c5:
            also["c5"] = measure_es_rollout(rank, world, local_rank)
        if world == 1 and args.workload != "c1":
            # BASELINE config 1, the size the reference itself runs at (cpu_baseline times the reference on exactly this):
            # launch-bound, so what counts is the public step() and the host-buffer call, not a roofline
            n, win = WORKLOAD_DEFAULTS["c1"]
            r = measure_workload(torch, par, loader, timer, "c1", n, win, rank, world, local_rank, max(args.steps, 300), args.warmup,
                                 3, "auto", full=True)
            also["c1"] = {"workload": WORKLOAD_NAMES["c1"], "envs_per_gpu": n, "window": win, "assets": 1, "value": r["value"],
                          "unit": UNIT, "ms_per_step": r["ms_per_step"], "kernel": r["roofline"]["kernel"],
                          "public_step": {k: r["public_step"][k] for k in ("value", "ms_per_step", "api")},
                          "e2e": {k: r["e2e"][k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "api")},
                          "note": "launch-bound: one kernel launch per step; CUDA-graph replay of policy + step: tools/graph_rollout.py",
                          "gpu_launches": r["gpu_launches"]}
        _SERIES_CACHE.clear()
        if world > 1:
            collectives = measure_collectives(torch, dist, par, dev, world, args.envs)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32/f64", "data": "synthetic", "config": workload_config(args.workload, args.envs, args.window, world),
        "timing": main_res["timing"],
        "roofline": main_res["roofline"],
        "e2e": main_res["e2e"],
        "public_step": main_res["public_step"],
        # kernels of this library inside the timed regions (device, public step() and e2e legs; + the `also` workloads):
        # one per step, two where the step is a bookkeeping + a streaming launch (portfolio, split)
        "gpu_launches": main_res["gpu_launches"] + sum(a["gpu_launches"] for a in also.values()),
        "clocks": sampler.summary(),
        "episodes_finished_last_step": main_res["episodes_finished_last_step"],
    }
    if also:
        line["also"] = also
    if collectives:
        line["collectives"] = collectives
    line["host"] = {"numa_bound_cpus": len(os.sched_getaffinity(0)) if prev_affinity is not None else None,
                    "cpu_count": os.cpu_count()}
    if prev_affinity is not None:
        os.sched_setaffinity(0, prev_affinity)   # the CPU baseline uses every host core
    if world == 1 and not args.no_cpu_baseline:
        full = args.envs if (args.workload == "c2" and args.ref_widened_envs > 0) else 0
        rb = reference_baseline(60, 30, 3, 10.0, False, args.workload, args.ref_widened_envs, full)
        line["cpu_baseline"] = cpu_baseline_block(rb)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
