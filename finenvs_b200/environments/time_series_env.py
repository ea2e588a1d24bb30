"""TimeSeriesEnv — drop-in for the reference's finenvs/environments/time_series_env.py:14-536.

Same constructor arguments, attributes and `reset()` / `step(actions)` / `get_env_args()` contract
(torch tensors in and out, so finenvs/agents run unchanged), but the series is staged once into
HBM as a flat table and every `step` is ONE launch of the sm_100a kernel in csrc/fe_step.cu,
reached through the C ABI of include/finenvs_b200.h.  There is no CPU path.

Keyword-only arguments after `device_id` are extensions (SURVEY.md App. D); their defaults
reproduce the reference's behaviour, except `obs_dtype` (float32; pass torch.float64 for the
reference's dtype) and the redraw RNG (counter-based Philox instead of torch's global generator).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from .. import _lib
from ..base_object import BaseObject
from ..data import loader
from ..device_utils import require_cuda_device

try:  # gym is metadata only (:218-234); the reference needs it, we do not
    from gym import spaces as _spaces
except Exception:  # pragma: no cover - gym is not installed in the target image
    class _Box:
        def __init__(self, low, high, shape=None, dtype=None):
            self.low, self.high, self.dtype = low, high, dtype
            self.shape = shape if shape is not None else np.shape(low)

    class _spaces:  # type: ignore
        Box = _Box

_RESET_MODES = {"keep": _lib.RESET_KEEP, "last": _lib.RESET_LAST, "all": _lib.RESET_ALL}
_VARIANTS = {"auto": _lib.VARIANT_AUTO, "tile": _lib.VARIANT_TILE, "direct": _lib.VARIANT_DIRECT,
             "portfolio": _lib.VARIANT_PORTFOLIO, "pipe": _lib.VARIANT_PIPE, "split": _lib.VARIANT_SPLIT,
             "gather": _lib.VARIANT_GATHER}


def default_signal_columns(env_id_base: int, num_envs: int, num_segments: int, num_signals: int) -> torch.Tensor:
    """The signal column each env of the shard [env_id_base, env_id_base + num_envs) trades in TimeSeriesEnv.backtest()
    by default: global id // num_segments.  Env g starts on segment g % num_segments, so with total_envs = S x D every
    (strategy, day) pair is one env, whatever the sharding.  (num_envs,) int32 on the CPU; ValueError when a column
    falls outside [0, num_signals)."""
    gid = torch.arange(int(env_id_base), int(env_id_base) + int(num_envs), dtype=torch.int64)
    cols = gid // int(num_segments)
    if num_envs > 0 and int(cols[-1]) >= num_signals:
        raise ValueError(f"the default columns (global id // {num_segments} segments) reach {int(cols[-1])}, but the "
                         f"signal table has {num_signals} rows; pass columns= or more signals")
    return cols.to(torch.int32)


class LazyObs:
    """An observation that has not been materialised: obs[i, j, 0:4] = logret[row0[i] + j], obs[i, j, 4] = posfeat[i]
    (time_series_env.py:428-445).  12 bytes per env instead of W x 20; consumers that read the window straight from
    the staged series (finenvs_b200.agents.networks.ParallelMLP.forward) never need the tensor."""

    __slots__ = ("env", "row0", "posfeat")

    def __init__(self, env: "TimeSeriesEnv", row0: torch.Tensor, posfeat: torch.Tensor):
        self.env, self.row0, self.posfeat = env, row0, posfeat

    @property
    def logret(self) -> torch.Tensor:
        return self.env.series.logret

    @property
    def window(self) -> int:
        return self.env.num_intervals

    @property
    def shape(self):
        return self.env._obs_shape

    def materialize(self) -> torch.Tensor:
        """The tensor step() would have returned for this observation."""
        e = self.env
        obs = torch.empty(self.shape, dtype=e.obs_dtype, device=e._dev)
        _lib.check(e._L.fe_materialize(e._pp, e._ps, self.row0.data_ptr(), self.posfeat.data_ptr(), obs.data_ptr(), e._stream()),
                   "fe_materialize")
        return obs


class CapturedRollout:
    """`num_steps` iterations of `actions = policy(obs); obs, rewards, dones = env.step(actions)` recorded ONCE in a
    CUDA graph and replayed with a single launch (SURVEY.md 8f-4).  The loop it replaces is the reference's evaluation
    loop (examples/time_series/PPO_LSTM_testing_SPY.py:43-52), whose cost for a few thousand envs is Python and launch
    overhead, not the step.  The step ordinal lives in device memory (fe_step_captured), so a replay continues the
    env exactly where eager stepping would be: results are identical to calling env.step() num_steps times.

    Static tensors (overwritten by every replay): `obs` (N, W, 5) current observation, `rewards` (num_steps, N),
    `dones` (num_steps, N) int32, `actions` (num_steps, N, num_acts)."""

    def __init__(self, env: "TimeSeriesEnv", policy, num_steps: int):
        if num_steps < 1:
            raise ValueError("num_steps must be >= 1")
        self.env, self.policy, self.num_steps = env, policy, int(num_steps)
        dev, N = env._dev, env.num_envs
        self.obs = torch.empty(env._obs_shape, dtype=env.obs_dtype, device=dev)
        self.rewards = torch.empty((num_steps, N), dtype=env.obs_dtype, device=dev)
        self.dones = torch.empty((num_steps, N), dtype=torch.int32, device=dev)
        self.actions = torch.empty((num_steps, N, env.num_acts), dtype=torch.float32, device=dev)
        self._counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.graph = torch.cuda.CUDAGraph()
        # warm-up on a side stream (lazy initialisation inside the policy / the library must not be captured), on a
        # snapshot of the env state that is restored afterwards
        snap = env.state_snapshot()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            env._observe_into(self.obs)
            self._counter.fill_(env.step_count)
            self._record(1)
        torch.cuda.current_stream(dev).wait_stream(side)
        env.load_state_snapshot(snap)
        with torch.cuda.graph(self.graph):
            self._record(self.num_steps)
        env.load_state_snapshot(snap)   # capture does not execute, but keep the contract explicit

    def _record(self, steps: int) -> None:
        env = self.env
        for t in range(steps):
            a = self.policy(self.obs)
            self.actions[t].copy_(a.reshape(env.num_envs, env.num_acts))
            _lib.check(
                env._L.fe_step_captured(env._pp, env._ps, env._pst, self.actions[t].data_ptr(), self.obs.data_ptr(),
                                        self.rewards[t].data_ptr(), self.dones[t].data_ptr(), env._stats_ptr,
                                        self._counter.data_ptr(), env._stream()),
                "fe_step_captured",
            )
            env._launch_metrics(self.rewards[t].data_ptr(), self.dones[t].data_ptr(), self._counter.data_ptr())

    def replay(self, refresh_obs: Optional[bool] = None):
        """Run the captured num_steps steps.  `refresh_obs=True` first rebuilds `obs` from the env's current state
        (what env.reset() returns); False continues from the observation the previous replay left (what the eager
        loop does: the observation returned by a step is built before the auto-reset, :321).  Default: refresh only
        if this is the first replay or something else stepped / reset the env in between."""
        env = self.env
        if refresh_obs is None:
            refresh_obs = getattr(self, "_resume_at", None) != (env.step_count, env._epoch)
        if refresh_obs:
            env._observe_into(self.obs)
        self._counter.fill_(env.step_count)
        self.graph.replay()
        env.step_count += self.num_steps
        self._resume_at = (env.step_count, env._epoch)
        return self.obs, self.rewards, self.dones


class TimeSeriesEnv(BaseObject):
    _obs_ring = None      # Buffer bound with bind_env(env): observations are written into its states slots
    _handle_ring = None   # Buffer bound with bind_env(env, lazy=True): it keeps the observations' handles

    def __init__(
        self,
        instrument_name: str,
        dataset_key: str = "dummy",
        num_intervals: int = 390,
        max_shares: int = 5,
        starting_balance: float = 10000,
        per_share_commission: float = 0.01,
        initial_margin_requirement: float = 1.5,
        maintenance_margin_requirement: float = 0.25,
        evaluate: bool = False,
        device_id: int = 0,
        *,
        num_envs: Optional[int] = None,
        obs_dtype: torch.dtype = torch.float32,
        seed: Optional[int] = None,
        random_reset: Optional[str] = None,
        random_offset: bool = False,
        series: Optional[loader.StagedSeries] = None,
        env_id_base: int = 0,
        total_envs: Optional[int] = None,
        track_stats: bool = False,
        variant: str = "auto",
        flat_obs: bool = False,
        num_eval_envs: Optional[int] = None,
        track_metrics: bool = False,
        metrics_capacity: Optional[int] = None,
    ):
        """Reference arguments: :15-29.  Extensions:

        num_envs      envs on this device (default: one per trading day, +1 evaluation env when
                      training, :246-257).  Env i starts on segment (global id) mod D.
        obs_dtype     torch.float32 (default) or torch.float64 (reference dtype) for obs and rewards.
        seed          Philox key of the segment redraws; default torch.initial_seed().
        random_reset  "last" (reference training: only the last env redraws its day, :504-513),
                      "keep" (reference evaluate: same day again), "all" (every finished env redraws).
        random_offset redraws also draw the start offset inside the segment.
        series        an already staged series (share one copy between envs / skip the CSV).
        env_id_base, total_envs   this env object is a shard [base, base+num_envs) of a global
                      population (multi-GPU); draws are keyed by global id, so results do not
                      depend on the sharding.
        track_stats   accumulate episode count / return / length on the device (stats()).
        variant       "auto" | "gather" | "pipe" | "tile" | "direct" | "split" | "portfolio" kernel variant (auto: for
                      populations of >= 4 tiles per SM (18 944 envs on a B200) with windows of >= 24 rows the persistent
                      kernels — gather while the series is short enough for its observation-layout table to stay in L2
                      and 5*W*itemsize is a multiple of 16, else pipe; else tile; direct when the window does not fit
                      in shared memory; portfolio whenever the series has more than one asset).
        flat_obs      return observations as (N, W*num_obs) — the 2-D input the ES agent's ParallelMLP needs
                      (parallel_mlp.py:98-103); same memory, only the shape differs.
        num_eval_envs reported in get_env_args() for the ES agent (evo_agent.py:53); the last
                      num_eval_envs envs are the evaluation envs by the reference's convention.
        track_metrics record per-episode trading metrics on the device after every step (fe_episode_metrics: length,
                      return, per-step Sharpe ratio, max drawdown absolute and relative to peak equity, hit rate; see
                      episode_metrics(), metrics_summary()).  Off: no extra launch.
        metrics_capacity  entries of the finished-episode list (default: num_envs in evaluate mode, where an env records
                      only its first episode between metric resets; else max(8 * num_envs, 65536)).
        """
        if obs_dtype not in (torch.float32, torch.float64):
            raise ValueError("obs_dtype must be torch.float32 or torch.float64")
        self.instrument_name = instrument_name
        self.num_intervals = int(num_intervals)
        self.max_shares = max_shares
        self.starting_balance = starting_balance
        self.per_share_commission = per_share_commission
        self.initial_margin_requirement = initial_margin_requirement
        self.maintenance_margin_requirement = maintenance_margin_requirement
        self.log_return_scale_factor = 100
        self.evaluate = evaluate
        self.obs_dtype = obs_dtype
        self.device = require_cuda_device(device_id)
        self._dev = torch.device(self.device)
        self._L = _lib.lib()
        if series is None:
            self.data_dir_name = loader.get_data_dir_name(instrument_name)
            self.file_key = loader.determine_file_key(dataset_key)
            self.filename = loader.find_file_by_key(self.data_dir_name, self.file_key)
            host = loader.read_market_csv(self.filename, self.num_intervals)
            series = loader.stage_series(host.prices, host.seg_start, host.seg_len_raw, self.num_intervals,
                                         self.device, obs_dtype)
        else:
            if series.window != self.num_intervals:
                raise ValueError(f"series was staged for W={series.window}, env asks W={self.num_intervals}")
            if series.device != self._dev:
                raise ValueError(f"series lives on {series.device}, env on {self._dev}")
            if series.logret.dtype != obs_dtype:
                raise ValueError(f"series log-returns are {series.logret.dtype}, obs_dtype is {obs_dtype}")
        self.series = series
        self.num_assets = series.num_assets   # extension: A > 1 = portfolio env sharing one cash account
        self.values_per_interval = 4
        self.set_spaces()
        if random_reset is None:
            random_reset = "keep" if evaluate else "last"
        if random_reset not in _RESET_MODES:
            raise ValueError(f"random_reset must be one of {sorted(_RESET_MODES)}")
        self.random_reset = random_reset
        self.random_offset = bool(random_offset)
        self.seed = int(torch.initial_seed() if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
        self.track_stats = bool(track_stats)
        self.flat_obs = bool(flat_obs)
        self.num_eval_envs = num_eval_envs
        self.track_metrics = bool(track_metrics)
        self._metrics_capacity = metrics_capacity
        self.set_environment_params(num_envs, env_id_base, total_envs, _VARIANTS[variant])

    # ------------------------------------------------------------------ metadata (:218-243) ----
    def set_spaces(self) -> None:
        self.num_obs = (self.values_per_interval + 1) * self.num_assets
        self.num_acts = self.num_assets
        self.action_space = _spaces.Box(np.ones(self.num_acts) * -1.0, np.ones(self.num_acts) * +1.0, dtype=np.float64)
        self.observation_space = _spaces.Box(
            np.ones((self.num_intervals, self.num_obs)) * -np.inf,
            np.ones((self.num_intervals, self.num_obs)) * +np.inf,
            dtype=np.float64,
        )

    def get_env_args(self) -> Dict:
        env_args = {
            "env_name": self.instrument_name,
            "num_envs": self.num_envs,
            "num_observations": self.num_obs * (self.num_intervals if self.flat_obs else 1),
            "num_actions": self.num_acts,
            "sequence_length": self.num_intervals,
        }
        if self.num_eval_envs is not None:
            env_args["num_eval_envs"] = self.num_eval_envs
        return env_args

    # ------------------------------------------------------------------ state (:245-275) -------
    def set_environment_params(self, num_envs=None, env_id_base=0, total_envs=None, variant=0) -> None:
        D = self.series.num_segments
        if num_envs is None:
            num_envs = D if self.evaluate else D + 1  # :246-257
        N = int(num_envs)
        if N <= 0:
            raise ValueError("num_envs must be positive")
        total = int(N if total_envs is None else total_envs)
        base = int(env_id_base)
        if base < 0 or base + N > total:
            raise ValueError("shard [env_id_base, env_id_base+num_envs) must lie inside total_envs")
        self.num_envs, self.env_id_base, self.total_envs = N, base, total
        dev = self._dev
        gid = torch.arange(base, base + N, device=dev, dtype=torch.int64)
        self._seg = (gid % D).to(torch.int32)
        self._ptr = torch.zeros(N, dtype=torch.int32, device=dev)
        self._cash = torch.full((N,), float(self.starting_balance), dtype=torch.float32, device=dev)
        A = self.num_assets
        self._long = torch.zeros(N * A, dtype=torch.float32, device=dev)
        self._short = torch.zeros(N * A, dtype=torch.float32, device=dev)
        self._margin = torch.zeros(N * A, dtype=torch.float64, device=dev)
        need_ep = self.evaluate or self.track_stats
        self._terminated = torch.zeros(N, dtype=torch.uint8, device=dev) if self.evaluate else None
        self._ep_return = torch.zeros(N, dtype=torch.float32, device=dev) if need_ep else None
        self._ep_len = torch.zeros(N, dtype=torch.int32, device=dev) if self.track_stats else None
        self._stats = torch.zeros(_lib.STATS_BYTES // 8, dtype=torch.int64, device=dev) if need_ep else None
        self._stats_ptr = self._stats.data_ptr() if self._stats is not None else None   # never reallocated (zeroed in place)
        self.step_count = 0
        self._epoch = 0   # bumped by everything that changes the state other than a step (reset_all, snapshots)
        self._params = _lib.FeParams(
            N, base, total, self.series.num_rows, self.num_intervals, D, A, int(self.max_shares),
            float(self.starting_balance), float(self.per_share_commission), float(self.initial_margin_requirement),
            float(self.maintenance_margin_requirement), self.seed, _RESET_MODES[self.random_reset],
            int(self.random_offset), int(self.evaluate), int(self.obs_dtype == torch.float64), variant,
            dev.index if dev.index is not None else torch.cuda.current_device(),
        )
        self._sched = torch.zeros(4, dtype=torch.int32, device=dev)   # gather kernel: tile / arrival counters (FeState.sched)
        s = self.series
        # the observation-layout table is only built for envs that can use it (large populations or variant="gather")
        want_table = variant == _lib.VARIANT_GATHER or (variant == _lib.VARIANT_AUTO and A == 1 and N >= 4096 and self.num_intervals >= 24)
        table = s.obs_table() if want_table else None
        self._cseries = _lib.FeSeries(s.prices.data_ptr(), s.logret.data_ptr(), s.seg_start.data_ptr(), s.seg_len.data_ptr(),
                                      table.data_ptr() if table is not None else None)
        self._cstate = _lib.FeState(
            self._seg.data_ptr(), self._ptr.data_ptr(), self._cash.data_ptr(), self._long.data_ptr(),
            self._short.data_ptr(), self._margin.data_ptr(),
            self._terminated.data_ptr() if self._terminated is not None else None,
            self._ep_return.data_ptr() if self._ep_return is not None else None,
            self._ep_len.data_ptr() if self._ep_len is not None else None,
            self._sched.data_ptr() if table is not None else None,
        )
        self._pp, self._ps, self._pst = C.byref(self._params), C.byref(self._cseries), C.byref(self._cstate)
        self._pm = self._alloc_metrics() if self.track_metrics else None
        if self.random_reset == "last" and base + N == total:
            # :253-257 the extra (evaluation) env starts on a drawn day
            r = _lib.philox(self.seed, total - 1, 0, 1)
            self._seg[-1] = (r[0] * D) >> 32
        elif self.random_reset == "all":
            self._launch_reset_all(redraw=True)

    def _alloc_metrics(self):
        N, dev = self.num_envs, self._dev
        cap = self._metrics_capacity
        cap = int((N if self.evaluate else max(8 * N, 1 << 16)) if cap is None else cap)
        if cap < 1:
            raise ValueError("metrics_capacity must be >= 1")
        self.metrics_capacity = cap
        # running state (FeMetricsState): sum, mean, m2, peak, mdd, mdd_rel as f64 rows; len, pos as int32 rows
        self._m_f64 = torch.zeros((6, N), dtype=torch.float64, device=dev)
        self._m_i32 = torch.zeros((2, N), dtype=torch.int32, device=dev)
        self._m_emitted = torch.zeros(N, dtype=torch.uint8, device=dev) if self.evaluate else None
        self._m_summary = torch.zeros(_lib.METRICS_SUMMARY_BYTES // 8, dtype=torch.int64, device=dev)
        # finished-episode list: key, env (i64); len (i32); return, sharpe, mdd, mdd_rel, hit_rate (f64)
        self._m_fin_i64 = torch.empty((2, cap), dtype=torch.int64, device=dev)
        self._m_fin_len = torch.empty(cap, dtype=torch.int32, device=dev)
        self._m_fin_f64 = torch.empty((5, cap), dtype=torch.float64, device=dev)
        f, i, L = self._m_f64, self._m_i32, self._m_fin_f64
        self._cmetrics = _lib.FeMetricsState(
            i[0].data_ptr(), i[1].data_ptr(), *(f[k].data_ptr() for k in range(6)),
            self._m_emitted.data_ptr() if self._m_emitted is not None else None,
            self._m_fin_i64[0].data_ptr(), self._m_fin_i64[1].data_ptr(), self._m_fin_len.data_ptr(),
            *(L[k].data_ptr() for k in range(5)), self._m_summary.data_ptr())
        return C.byref(self._cmetrics)

    def _launch_metrics(self, rewards_ptr: int, dones_ptr: int, counter_ptr: Optional[int] = None) -> None:
        """fe_episode_metrics on one step's device rewards / dones (track_metrics=True; a no-op otherwise).  The step
        ordinal is step_count, or *counter_ptr inside a CapturedRollout."""
        if self._pm is None:
            return
        _lib.check(self._L.fe_episode_metrics(self._pp, self._pm, rewards_ptr, dones_ptr, self.step_count, counter_ptr,
                                              self.metrics_capacity, self._stream()), "fe_episode_metrics")

    def _zero_metrics_running(self) -> None:
        self._m_f64.zero_()
        self._m_i32.zero_()
        if self._m_emitted is not None:
            self._m_emitted.zero_()

    def reset_evaluation_metrics(self) -> None:
        """:271-275; with track_metrics also the episode metrics (running state, "first episode recorded" flags, list
        and summary), so that the next evaluation records each env's first episode afresh."""
        # in place: CapturedRollout graphs and FeState / FeMetricsState hold these device addresses
        self._terminated.zero_()
        self._ep_return.zero_()
        self._stats.zero_()
        if self._pm is not None:
            self._zero_metrics_running()
            self._m_summary.zero_()

    # reference-named views of the state (same memory; reference shapes (N,1) / (N,))
    @property
    def env_indices(self) -> torch.Tensor:
        return self._seg.long()

    @property
    def env_pointers(self) -> torch.Tensor:
        return self._ptr.long()

    @property
    def env_spots(self) -> torch.Tensor:
        """(N, W) row indices of the window; the reference stores this tensor (:261), here it is derived."""
        return self._ptr.long().unsqueeze(1) + torch.arange(self.num_intervals, device=self._dev)

    @property
    def cash(self) -> torch.Tensor:
        return self._cash.view(-1, 1)

    @property
    def long_shares(self) -> torch.Tensor:
        return self._long.view(self.num_envs, self.num_assets)

    @property
    def short_shares(self) -> torch.Tensor:
        return self._short.view(self.num_envs, self.num_assets)

    @property
    def margin(self) -> torch.Tensor:
        return self._margin.view(self.num_envs, self.num_assets)

    @property
    def terminated_episodes(self) -> torch.Tensor:
        return self._terminated.bool()

    @property
    def episode_returns(self) -> torch.Tensor:
        return self._ep_return

    # ------------------------------------------------------------------ the hot path ------------
    def _stream(self) -> int:
        return torch.cuda.current_stream(self._dev).cuda_stream

    @property
    def _obs_shape(self) -> Tuple[int, ...]:
        """(N, W * num_obs) with flat_obs, else (N, W, num_obs)."""
        W = self.num_intervals
        return (self.num_envs, W * self.num_obs) if self.flat_obs else (self.num_envs, W, self.num_obs)

    def _new_obs(self, for_reset: bool = False) -> torch.Tensor:
        # a fresh tensor every call: the PPO buffer keeps references to past observations (buffer.py:44-56)
        ring = getattr(self, "_obs_ring", None)
        if ring is not None:  # a rollout buffer bound with Buffer.bind_env: write straight into its storage
            return ring.next_obs_slot(self._obs_shape, self.obs_dtype, for_reset)
        return torch.empty(self._obs_shape, dtype=self.obs_dtype, device=self._dev)

    def reset(self) -> torch.Tensor:
        """:423-435 — materialises the current observation; touches no state (reference semantics)."""
        if self._handle_ring is not None:
            return self._observe_via_handle(None, for_reset=True)
        obs = self._new_obs(for_reset=True)
        self._observe_into(obs)
        return obs

    def _prepare_actions(self, actions: torch.Tensor) -> torch.Tensor:
        if not torch.is_tensor(actions):
            raise TypeError("actions must be a torch.Tensor")
        if actions.numel() != self.num_envs * self.num_acts:
            raise ValueError(f"actions must be (num_envs, num_acts) = ({self.num_envs}, {self.num_acts}); "
                             f"got {tuple(actions.shape)}")
        if actions.device != self._dev or actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.to(device=self._dev, dtype=torch.float32, non_blocking=True).contiguous()
        return actions

    def step(self, actions: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, dict]:
        """:277-296 — one kernel launch, no host synchronisation in training mode."""
        actions = self._prepare_actions(actions)
        rewards = torch.empty(self.num_envs, dtype=self.obs_dtype, device=self._dev)
        dones = torch.empty(self.num_envs, dtype=torch.int32, device=self._dev)
        if self._handle_ring is not None:
            obs = self._observe_via_handle((actions, rewards, dones), for_reset=False)
        else:
            obs = self._new_obs()
            self.step_into(actions, obs, rewards, dones)
        info_dict = self.record_evaluation_metrics() if self.evaluate else {}
        return (obs, rewards, dones, info_dict)

    def step_into(self, actions: torch.Tensor, obs: torch.Tensor, rewards: torch.Tensor, dones: torch.Tensor) -> None:
        """step() into caller-owned output tensors (zero allocation; CUDA-graph capturable)."""
        self.step_count += 1
        _lib.check(
            self._L.fe_step(self._pp, self._ps, self._pst, actions.data_ptr(), obs.data_ptr(), rewards.data_ptr(),
                            dones.data_ptr(), self._stats_ptr, self.step_count, self._stream()),
            "fe_step",
        )
        self._launch_metrics(rewards.data_ptr(), dones.data_ptr())

    def _new_lazy(self) -> LazyObs:
        if self.num_assets != 1:
            raise NotImplementedError("lazy observations are implemented for single-asset envs")
        return LazyObs(self, torch.empty(self.num_envs, dtype=torch.int64, device=self._dev),
                       torch.empty(self.num_envs, dtype=self.obs_dtype, device=self._dev))

    def _observe_lazy(self, row0: torch.Tensor, posfeat: torch.Tensor) -> None:
        _lib.check(self._L.fe_observe_lazy(self._pp, self._ps, self._pst, row0.data_ptr(), posfeat.data_ptr(),
                                           self._stream()), "fe_observe_lazy")

    def _step_lazy(self, actions: torch.Tensor, row0: torch.Tensor, posfeat: torch.Tensor, rewards: torch.Tensor,
                   dones: torch.Tensor) -> None:
        self.step_count += 1
        _lib.check(
            self._L.fe_step_lazy(self._pp, self._ps, self._pst, actions.data_ptr(), row0.data_ptr(), posfeat.data_ptr(),
                                 rewards.data_ptr(), dones.data_ptr(), self._stats_ptr, self.step_count, self._stream()),
            "fe_step_lazy",
        )
        self._launch_metrics(rewards.data_ptr(), dones.data_ptr())

    def reset_lazy(self) -> LazyObs:
        """reset() returning a LazyObs handle instead of the tensor."""
        lo = self._new_lazy()
        self._observe_lazy(lo.row0, lo.posfeat)
        return lo

    def step_lazy(self, actions: torch.Tensor) -> Tuple[LazyObs, torch.Tensor, torch.Tensor, dict]:
        """step() without materialising the observation: same state transition, rewards and dones; the observation
        comes back as a LazyObs handle (`.materialize()` gives exactly the tensor step() returns)."""
        actions = self._prepare_actions(actions)
        lo = self._new_lazy()
        rewards = torch.empty(self.num_envs, dtype=self.obs_dtype, device=self._dev)
        dones = torch.empty(self.num_envs, dtype=torch.int32, device=self._dev)
        self._step_lazy(actions, lo.row0, lo.posfeat, rewards, dones)
        info_dict = self.record_evaluation_metrics() if self.evaluate else {}
        return (lo, rewards, dones, info_dict)

    # ------------------------------------------------------------------ rollout buffer that keeps handles ----
    def _bind_handle_ring(self, ring) -> None:
        """Buffer.bind_env(env, lazy=True): reset() / step() write each observation's handle into the buffer's next handle
        slot (fe_observe_lazy / fe_step_lazy) and return the dense tensor fe_gather_obs builds from it.  fe_gather_obs
        calls get their own FeSeries carrying the series' observation-layout table (built here once per series when it
        stays L2-resident) so that they take the TMA path; the step kernel's FeSeries, and with it `auto`, is unchanged."""
        if self.num_assets != 1:
            raise NotImplementedError("lazy observations are implemented for single-asset envs")
        s = self.series
        table = s.obs_table()
        self._gather_cseries = _lib.FeSeries(s.prices.data_ptr(), s.logret.data_ptr(), s.seg_start.data_ptr(),
                                             s.seg_len.data_ptr(), table.data_ptr() if table is not None else None)
        self._pgs = C.byref(self._gather_cseries)
        self._obs_ring, self._handle_ring = None, ring

    def gather_obs_kernel_name(self) -> str:
        """Which kernel fe_gather_obs launches for this env once bound to a buffer with bind_env(env, lazy=True)."""
        return self._L.fe_gather_obs_kernel_name(self._pp, self._pgs).decode()

    def gather_obs(self, row0: torch.Tensor, posfeat: torch.Tensor, index: Optional[torch.Tensor], out: torch.Tensor) -> None:
        """out[b] = the observation of handle index[b] (index None: handle b), b < out.shape[0] (fe_gather_obs).  The index
        values must lie in [0, row0.numel())."""
        _lib.check(self._L.fe_gather_obs(self._pp, self._pgs, row0.data_ptr(), posfeat.data_ptr(),
                                         index.data_ptr() if index is not None else None, out.shape[0], out.data_ptr(),
                                         self._stream()), "fe_gather_obs")

    def _observe_via_handle(self, step_args, for_reset: bool) -> torch.Tensor:
        row0, posfeat = self._handle_ring.next_handle_slot(self.num_envs, self.obs_dtype, for_reset)
        if step_args is None:
            self._observe_lazy(row0, posfeat)
        else:
            actions, rewards, dones = step_args
            self._step_lazy(actions, row0, posfeat, rewards, dones)
        obs = torch.empty(self._obs_shape, dtype=self.obs_dtype, device=self._dev)
        self.gather_obs(row0, posfeat, None, obs)
        self._handle_ring.hand_out(obs)
        return obs

    def step_host(self, actions_host: torch.Tensor, packed_dones: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, dict]:
        """step() for a host-resident policy, through fe_step_host: `actions_host` is a CPU tensor
        (pinned for full speed); rewards and dones come back as pinned CPU tensors, already complete when the
        call returns (the pinned buffers are reused by the next step_host call; copy them to keep them);
        the observation stays in HBM.  Per step: 4N bytes host->device, 8N (f32) device->host.
        packed_dones=True (fe_step_host_packed): dones come back bit-packed — a uint8 tensor of 4*ceil(N/32) bytes, bit
        (i % 8) of byte i // 8 is env i's flag; `unpack_dones()` expands it — N/8 instead of 4N bytes on the wire."""
        if actions_host.device.type != "cpu" or actions_host.dtype != torch.float32 or not actions_host.is_contiguous():
            raise ValueError("actions_host must be a contiguous float32 CPU tensor")
        if actions_host.numel() != self.num_envs * self.num_acts:
            raise ValueError(f"actions must have {self.num_envs * self.num_acts} elements")
        if not hasattr(self, "_host_bufs"):
            self._host_bufs = (
                torch.empty(self.num_envs * self.num_acts, dtype=torch.float32, device=self._dev),
                torch.empty(self.num_envs, dtype=self.obs_dtype, device=self._dev),
                torch.empty(self.num_envs, dtype=torch.int32, device=self._dev),
                torch.empty(self.num_envs, dtype=self.obs_dtype).pin_memory(),
                torch.empty(self.num_envs, dtype=torch.int32).pin_memory(),
                torch.zeros(4 * ((self.num_envs + 31) // 32), dtype=torch.uint8).pin_memory(),
            )
            self._host_ptrs = tuple(t.data_ptr() for t in self._host_bufs)   # the buffers live as long as the env
        _, _, _, rewards, dones, done_bits = self._host_bufs
        p_a, p_r, p_d, p_rh, p_dh, p_bh = self._host_ptrs
        obs = self._new_obs()
        self.step_count += 1
        fn = self._L.fe_step_host_packed if packed_dones else self._L.fe_step_host
        out_dones = done_bits if packed_dones else dones
        _lib.check(
            fn(self._pp, self._ps, self._pst, actions_host.data_ptr(), p_a, obs.data_ptr(), p_r, p_d, p_rh,
               p_bh if packed_dones else p_dh, self._stats_ptr, self.step_count, self._stream()),
            "fe_step_host_packed" if packed_dones else "fe_step_host",
        )
        self._launch_metrics(p_r, p_d)   # the device copies of rewards and dones (int32 flags with either wire format)
        info_dict = self.record_evaluation_metrics() if self.evaluate else {}
        return (obs, rewards, out_dones, info_dict)

    def unpack_dones(self, done_bits: torch.Tensor) -> torch.Tensor:
        """(N,) int32 flags from the bit-packed form step_host(packed_dones=True) returns."""
        bits = np.unpackbits(done_bits.numpy(), bitorder="little")[: self.num_envs]
        return torch.from_numpy(bits.astype(np.int32))

    def host_bytes_per_step(self, packed_dones: bool = False) -> Tuple[int, int]:
        """(host->device, device->host) bytes one step_host() call moves over PCIe."""
        osz = 8 if self.obs_dtype == torch.float64 else 4
        dones = 4 * ((self.num_envs + 31) // 32) if packed_dones else 4 * self.num_envs
        return 4 * self.num_envs * self.num_acts, osz * self.num_envs + dones

    # ------------------------------------------------------------------ captured rollouts (8f-4) ----
    def _observe_into(self, obs: torch.Tensor) -> None:
        _lib.check(self._L.fe_observe(self._pp, self._ps, self._pst, obs.data_ptr(), self._stream()), "fe_observe")

    _STATE_FIELDS = ("_seg", "_ptr", "_cash", "_long", "_short", "_margin", "_terminated", "_ep_return", "_ep_len", "_stats",
                     "_m_f64", "_m_i32", "_m_emitted", "_m_summary")

    def state_snapshot(self) -> dict:
        """Copy of the per-env state (device tensors) + the step ordinal; load_state_snapshot() restores it in place."""
        snap = {k: getattr(self, k).clone() for k in self._STATE_FIELDS if getattr(self, k, None) is not None}
        snap["step_count"] = self.step_count
        return snap

    def load_state_snapshot(self, snap: dict) -> None:
        for k in self._STATE_FIELDS:
            if k in snap:
                getattr(self, k).copy_(snap[k])
        self.step_count = snap["step_count"]
        self._epoch += 1

    def capture_rollout(self, policy, num_steps: int) -> CapturedRollout:
        """Record `num_steps` x (policy -> step) in a CUDA graph; see CapturedRollout."""
        return CapturedRollout(self, policy, num_steps)

    def evaluate_policy(self, policy, steps_per_replay: int = 32, max_steps: Optional[int] = None,
                        rollout: Optional[CapturedRollout] = None) -> Dict:
        """The reference's evaluation loop (PPO_LSTM_testing_SPY.py:43-52: step until info has "returns") with the
        "all envs terminated" test (:531) read once per `steps_per_replay` graph-replayed steps instead of once per
        step.  Terminated envs collect zero reward (:527-528), so running past the end changes nothing: the returned
        {"returns": (N,) f32} equals what the per-step loop returns.  With track_metrics the result also holds
        "metrics": each env's first episode (the backtest report of the checkpoint), per-env tensors in env order.
        Metrics are reset afterwards (:532-534) — in place, so `rollout` (a CapturedRollout of this env, e.g. the one
        returned in the result) can be passed back in to evaluate the next checkpoint of the same policy object
        without capturing again."""
        if not self.evaluate:
            raise RuntimeError("evaluate_policy needs an env constructed with evaluate=True")
        roll = rollout if rollout is not None else self.capture_rollout(policy, steps_per_replay)
        if roll.env is not self:
            raise ValueError("rollout was captured on another env")
        steps = 0
        while max_steps is None or steps < max_steps:
            roll.replay(refresh_obs=(steps == 0))
            steps += roll.num_steps
            if int(self._stats[1].item()) >= self.num_envs:
                info = {"returns": self._ep_return.clone(), "steps": steps, "rollout": roll}
                if self._pm is not None:
                    info["metrics"] = self._first_episode_metrics()
                self.reset_evaluation_metrics()
                return info
        return {"steps": steps, "rollout": roll}

    def record_evaluation_metrics(self) -> Dict:
        """:523-536 — the per-env bookkeeping ran inside the kernel; here only the "all terminated"
        test (:531), which like the reference's torch.all() costs one host read per step."""
        n_terminated = int(self._stats[1].item())
        if n_terminated >= self.num_envs:
            info_dict = {"returns": self._ep_return.clone()}   # the reference hands out the old tensor and rebinds (:532-534)
            if self._pm is not None:
                info_dict["metrics"] = self._first_episode_metrics()
            self.reset_evaluation_metrics()
            return info_dict
        return {}

    # ------------------------------------------------------------------ extensions --------------
    def _launch_reset_all(self, redraw: bool) -> None:
        _lib.check(self._L.fe_reset_all(self._pp, self._ps, self._pst, self.step_count, int(redraw), self._stream()),
                   "fe_reset_all")

    def reset_all(self, redraw: Optional[bool] = None, lazy: bool = False):
        """Fresh episode for every env (the reset the ES loop expects, cf. isaac_gym_env.py:55-58)."""
        if redraw is None:
            redraw = self.random_reset == "all"
        self._epoch += 1
        self._launch_reset_all(redraw)
        if self._stats is not None:
            self._stats.zero_()
        if self._pm is not None:   # fe_reset_all also clears the terminated flags the emitted flags follow
            self._zero_metrics_running()
        return self.reset_lazy() if lazy else self.reset()

    def kernel_name(self) -> str:
        """Which kernel step() launches for this env's shape (diagnostics)."""
        return self._L.fe_step_kernel_name(self._pp, self._ps, self._pst).decode()

    def stats(self) -> Dict[str, torch.Tensor]:
        """Device-side episode statistics accumulated since the last clear (track_stats=True)."""
        if self._stats is None:
            raise RuntimeError("construct the env with track_stats=True")
        f = self._stats.view(torch.float64)
        return {"n_done": self._stats[0], "n_terminated": self._stats[1], "sum_len": self._stats[2],
                "sum_return": f[4], "sum_return_sq": f[5]}

    def clear_stats(self) -> None:
        if self._stats is not None:
            self._stats.zero_()

    # ------------------------------------------------------------------ episode metrics (track_metrics) ----
    def _require_metrics(self) -> None:
        if self._pm is None:
            raise RuntimeError("construct the env with track_metrics=True")

    def episode_metrics(self) -> Dict[str, torch.Tensor]:
        """Every episode finished since the last clear_metrics() (evaluate mode: since the last metric reset), sorted
        by key = step ordinal * total_envs + global env id, i.e. in (step, env) order: {"key", "env" (global id),
        "len", "return" (cumulative P&L), "sharpe" (per-step mean / std of the rewards, not annualised), "mdd" (max
        drawdown of the cumulative P&L), "mdd_rel" (the same relative to peak equity starting_balance + peak),
        "hit_rate" (share of steps with a positive reward)}.  Reads the episode count (one host sync); raises
        RuntimeError when more episodes finished than metrics_capacity."""
        self._require_metrics()
        n = int(self._m_summary[0].item())
        if n > self.metrics_capacity:
            raise RuntimeError(f"{n} episodes finished but metrics_capacity={self.metrics_capacity}")
        order = torch.argsort(self._m_fin_i64[0, :n])
        f = self._m_fin_f64[:, :n][:, order]
        return {"key": self._m_fin_i64[0, :n][order], "env": self._m_fin_i64[1, :n][order],
                "len": self._m_fin_len[:n][order], "return": f[0], "sharpe": f[1], "mdd": f[2], "mdd_rel": f[3],
                "hit_rate": f[4]}

    def _first_episode_metrics(self) -> Dict[str, torch.Tensor]:
        """evaluate: every env has recorded exactly its first episode; the records in env order."""
        m = self.episode_metrics()
        order = torch.argsort(m["env"])
        return {k: v[order] for k, v in m.items()}

    def metrics_summary(self) -> Dict[str, torch.Tensor]:
        """Aggregates of every episode recorded since the last clear (no list needed, overflowed episodes included):
        device scalars episodes, sum_len (int64) and sum_return, sum_sharpe, sum_sharpe_sq, sum_mdd, max_mdd,
        sum_hit_rate (f64).  finenvs_b200.parallel.all_reduce_episode_metrics combines them over ranks."""
        self._require_metrics()
        s, f = self._m_summary, self._m_summary.view(torch.float64)
        return {k: (s[j] if j < 2 else f[j]) for j, k in enumerate(_lib.METRICS_SUMMARY_KEYS)}

    def clear_metrics(self) -> None:
        """Empty the finished-episode list and zero the summary (episodes in progress keep their running state)."""
        self._require_metrics()
        self._m_summary.zero_()

    # ------------------------------------------------------------------ signal backtests (DESIGN §4.12) ----
    def backtest(self, signal: torch.Tensor, num_steps: int, columns: Optional[torch.Tensor] = None,
                 history: bool = False, *, targets: bool = False, exits: Optional[torch.Tensor] = None) -> Dict:
        """Advance every env `num_steps` steps with actions read from a signal table, in ONE launch (fe_backtest).

        `signal` is a float32 (S, series.num_rows) tensor on the env's device: one row ("column") per rule-based
        strategy, one action per row of the staged series, mapped like step()'s actions.  Env i trades column
        `columns[i]` (default: default_signal_columns, global id // num_segments).  At every step env i's action is
        signal[columns[i], seg_start[seg] + ptr + W - 1] with the state before the step: the last row of the window the
        env observes.  The trade executes at the next bar's Open, so there is no look-ahead by construction.

        With targets=True (fe_backtest_targets) that value v is the net position to hold instead of a trade:
        T = clamp(rint(v * (max_shares + 0.5)), +-max_shares) shares, and the action is the delta (T - (long - short)) /
        (max_shares + 0.5), which step() maps back to exactly that delta (clamped to +-max_shares).  So +1 everywhere is
        buy-and-hold wherever the episode starts, and sign(momentum) is "long while momentum is positive".  `exits`, a
        contiguous float64 (S, 2) tensor on the env's device, adds per column a trailing stop [:, 0] and a take-profit
        [:, 1] in reward units: T is 0 on every step at which the episode's P&L is that far below its running peak
        (peak starts at 0), or at least the take-profit.  Thresholds must be > 0; +inf disables one.  The exit is not
        latched, but once flat the rewards are 0, so the env stays flat until its episode ends.  The env's rules still
        apply: a flip from long to short takes two steps, and an entry the cash cannot pay for is retried.  Needs
        max_shares <= 2**20.

        The result is bit-identical to `num_steps` step_into() calls with those actions (for targets, computed from the
        env's state before each step in the same f32 / f64 operations): per-env state, redraws, stats, episode metrics
        (records, running state, summary counts; the f64 sums up to their order of addition).  Unlike step() in evaluate
        mode it does not test for "all terminated" or reset the evaluation metrics on the way (evaluate_signal() does
        that once, at the end).  Needs track_metrics=True and a single-asset series.  Records are keyed by global env id,
        so shards of one population (env_id_base / total_envs) produce the records of the whole and
        parallel.all_reduce_episode_metrics combines their summaries.

        Returns {"steps": num_steps}, plus "rewards" / "dones" (num_steps, N) when history=True."""
        self._require_metrics()
        if self.num_assets != 1:
            raise NotImplementedError("signal backtests are implemented for single-asset envs")
        if self._obs_ring is not None or self._handle_ring is not None:
            raise RuntimeError("a rollout buffer is bound to this env (bind_env): a backtest would leave the observation "
                               "it holds stale")
        K = int(num_steps)
        if K < 1:
            raise ValueError("num_steps must be >= 1")
        if not torch.is_tensor(signal) or signal.dim() != 2 or signal.shape[1] != self.series.num_rows:
            raise ValueError(f"signal must be a (S, {self.series.num_rows}) tensor (one row per strategy, one value per "
                             f"series row); got {tuple(signal.shape) if torch.is_tensor(signal) else type(signal)}")
        if signal.dtype != torch.float32 or signal.device != self._dev or not signal.is_contiguous():
            raise ValueError(f"signal must be a contiguous float32 tensor on {self._dev}; got {signal.dtype} on "
                             f"{signal.device}{'' if signal.is_contiguous() else ', not contiguous'}")
        S = signal.shape[0]
        if S < 1 or S > 0x7FFFFFFF:
            raise ValueError("signal must have between 1 and 2**31 - 1 rows")
        if columns is None:
            cols = default_signal_columns(self.env_id_base, self.num_envs, self.series.num_segments, S).to(self._dev)
        else:
            if (not torch.is_tensor(columns) or columns.shape != (self.num_envs,) or columns.dtype.is_floating_point
                    or columns.dtype.is_complex or columns.dtype == torch.bool):
                raise ValueError(f"columns must be an integer ({self.num_envs},) tensor")
            lo, hi = torch.stack(torch.aminmax(columns)).tolist()   # one host read
            if lo < 0 or hi >= S:
                raise ValueError(f"columns must lie in [0, {S}); got [{lo}, {hi}]")
            cols = columns.to(device=self._dev, dtype=torch.int32).contiguous()
        if exits is not None:
            if not targets:
                raise ValueError("exits need targets=True (they flatten a target position)")
            if not torch.is_tensor(exits) or exits.shape != (S, 2):
                raise ValueError(f"exits must be a ({S}, 2) tensor (trailing stop, take-profit per signal row); got "
                                 f"{tuple(exits.shape) if torch.is_tensor(exits) else type(exits)}")
            if exits.dtype != torch.float64 or exits.device != self._dev or not exits.is_contiguous():
                raise ValueError(f"exits must be a contiguous float64 tensor on {self._dev}; got {exits.dtype} on "
                                 f"{exits.device}{'' if exits.is_contiguous() else ', not contiguous'}")
            if not bool((exits > 0).all()):   # one host read; NaN fails the comparison too
                raise ValueError("exit thresholds must be > 0 (+inf disables one); got a value <= 0 or NaN")
        if targets and not 1 <= self.max_shares <= _lib.TARGET_MAX_SHARES:
            raise ValueError(f"target backtests need 1 <= max_shares <= {_lib.TARGET_MAX_SHARES}")
        shape = (K, self.num_envs) if history else (self.num_envs,)
        rewards = torch.empty(shape, dtype=self.obs_dtype, device=self._dev)
        dones = torch.empty(shape, dtype=torch.int32, device=self._dev)
        if targets:
            _lib.check(
                self._L.fe_backtest_targets(self._pp, self._ps, self._pst, self._pm, self.metrics_capacity,
                                            self._stats_ptr, signal.data_ptr(), S, cols.data_ptr(),
                                            exits.data_ptr() if exits is not None else None, self.step_count + 1, K,
                                            rewards.data_ptr(), dones.data_ptr(), int(bool(history)), self._stream()),
                "fe_backtest_targets",
            )
        else:
            _lib.check(
                self._L.fe_backtest(self._pp, self._ps, self._pst, self._pm, self.metrics_capacity, self._stats_ptr,
                                    signal.data_ptr(), S, cols.data_ptr(), self.step_count + 1, K, rewards.data_ptr(),
                                    dones.data_ptr(), int(bool(history)), self._stream()),
                "fe_backtest",
            )
        self.step_count += K
        self._epoch += 1   # a CapturedRollout's observation is stale now
        out = {"steps": K}
        if history:
            out["rewards"], out["dones"] = rewards, dones
        return out

    def evaluate_signal(self, signal: torch.Tensor, columns: Optional[torch.Tensor] = None, *, targets: bool = False,
                        exits: Optional[torch.Tensor] = None) -> Dict:
        """The evaluate-mode report of a signal table, the counterpart of evaluate_policy(): one backtest() launch of
        max(seg_len) - W steps (enough for every env to finish its current episode from any pointer; terminated envs
        collect zero reward, so running past the end changes nothing), then one host read of the terminated count.
        `targets` / `exits` are backtest()'s (target positions, trailing stop and take-profit per signal row).
        Returns {"returns": (N,) f32, "steps", "metrics": each env's first episode in env order} and resets the
        evaluation metrics, as evaluate_policy() does.  Needs evaluate=True and track_metrics=True."""
        if not self.evaluate:
            raise RuntimeError("evaluate_signal needs an env constructed with evaluate=True")
        self._require_metrics()
        if getattr(self, "_signal_steps", None) is None:
            self._signal_steps = int(self.series.seg_len.max().item()) - self.num_intervals
        steps = self.backtest(signal, self._signal_steps, columns, targets=targets, exits=exits)["steps"]
        if int(self._stats[1].item()) >= self.num_envs:
            info = {"returns": self._ep_return.clone(), "steps": steps, "metrics": self._first_episode_metrics()}
            self.reset_evaluation_metrics()
            return info
        return {"steps": steps}
