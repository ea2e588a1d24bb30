/*
 * finenvs_b200.h — C ABI of the B200-native trading-env step.
 *
 * The reference (hmomin/FinEnvs) has no native layer: its hot path is ~660 torch-eager ops inside
 * finenvs/environments/time_series_env.py.  Each entry point below replaces the reference METHOD(s)
 * named in its comment (file = finenvs/environments/time_series_env.py); the Python class
 * finenvs_b200.environments.TimeSeriesEnv binds them with ctypes and keeps the reference's
 * reset()/step() surface.
 *
 * Conventions
 *   - plain pointers + sizes, no torch / C++ types; every `*_dev` / struct pointer member is a DEVICE
 *     pointer owned by the caller (the library allocates nothing persistent and frees nothing);
 *   - `stream` is a cudaStream_t (CUstream) passed as void*; calls only enqueue work and never
 *     synchronise, except fe_step_host which returns after its device->host copies completed;
 *   - return 0 on success, a negative FE_E* code for a rejected argument, or a positive cudaError_t;
 *   - no exceptions cross the boundary; there is NO CPU fallback: without a CUDA device every compute
 *     entry point returns a cudaError.
 */
#ifndef FINENVS_B200_H
#define FINENVS_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FE_ABI_VERSION 3

/* argument errors */
#define FE_EINVAL (-1)   /* null pointer / non-positive size / unsupported num_assets */
#define FE_EALIGN (-2)   /* pointer not 16-byte aligned */
#define FE_ESMEM (-3)    /* window too large for the requested kernel variant */
#define FE_EIO (-4)      /* fe_csv_open: the file cannot be opened or mapped */
#define FE_ECSV (-5)     /* fe_csv_read: a record is outside the format the native reader handles (the caller falls back to pandas) */
#define FE_EDRIVER (-6)  /* gather variant: the driver's tensor-map encoder is unavailable or rejected the table */

/* FeParams.reset_mode */
#define FE_RESET_KEEP 0  /* finished envs restart on the same segment (reference evaluate=True, :504) */
#define FE_RESET_LAST 1  /* only the globally-last env redraws its segment (reference training mode, :504-513) */
#define FE_RESET_ALL 2   /* extension: every finished env redraws its segment */

/* FeParams.variant */
#define FE_VARIANT_AUTO 0   /* portfolio when num_assets > 1; gather / pipe for large populations; else tile when the window fits in shared memory, else direct */
#define FE_VARIANT_TILE 1   /* cp.async.bulk in -> smem interleave -> cp.async.bulk out */
#define FE_VARIANT_DIRECT 2 /* warp-per-env global->global copy (any window) */
#define FE_VARIANT_PORTFOLIO 3 /* warp-per-env bookkeeping kernel + block-per-env streaming kernel; always used when num_assets > 1 */
#define FE_VARIANT_PIPE 4   /* persistent warp-specialised pipeline (bookkeeper / mover warps, multi-stage rings) */
#define FE_VARIANT_SPLIT 6  /* two launches: thread-per-env bookkeeping, then warp-per-env streaming with fully coalesced stores */
#define FE_VARIANT_GATHER 8 /* persistent pipeline whose windows arrive by TMA gather4 from the observation-layout table
                               (FeSeries.obs_table, fe_obs_table_build; needs FeState.sched) and leave by bulk stores */
/* (5 and 7 were the round-1 "scatter" and "rows" experiments; both measured slower everywhere and were removed) */

typedef struct FeParams {
    int64_t num_envs;        /* envs held by this GPU (a shard) */
    int64_t env_id_base;     /* global id of local env 0 (keys the redraw RNG; results do not depend on sharding) */
    int64_t total_envs;      /* global env count; the reference's evaluation env is id total_envs-1 (:250-257) */
    int64_t num_rows;        /* T: rows of the flat series */
    int32_t window;          /* W = num_intervals (:19) */
    int32_t num_segments;    /* D: trading days / segments */
    int32_t num_assets;      /* A: 1 for the reference env; 2..32 = portfolio extension (series (T,A,4), obs (N,W,A,5)) */
    int32_t max_shares;      /* :20 */
    double starting_balance; /* :21 */
    double commission;       /* per_share_commission :22 */
    double imr;              /* initial_margin_requirement :25 */
    double mmr;              /* maintenance_margin_requirement :26 */
    uint64_t seed;           /* Philox key for segment / offset redraws */
    int32_t reset_mode;      /* FE_RESET_* */
    int32_t random_offset;   /* extension: a redraw also draws the start offset inside the segment */
    int32_t evaluate;        /* reference evaluate=True (:523-536): needs state.terminated / ep_return */
    int32_t out_f64;         /* 1: obs/rewards are double (reference dtype); 0: float */
    int32_t variant;         /* FE_VARIANT_* */
    int32_t device;          /* CUDA device ordinal the pointers live on */
} FeParams;

/* Series staged once into HBM (replaces the two NaN-padded (D,L,4) tensors of :196-216). */
typedef struct FeSeries {
    const double *prices;     /* (T, A, 4) f64 O,H,L,C, time-major  (:169-177) */
    const void *logret;       /* (T, A, 4) 100*log-returns, float when !out_f64 else double (:179-194) */
    const int64_t *seg_start; /* (D,) first row of segment d: first bar of the day minus W history rows (:141-152) */
    const int32_t *seg_len;   /* (D,) rows in segment d with the NaN probe of :486-496 folded in */
    const void *obs_table;    /* optional (NULL: none): the log-returns in observation layout for the gather variant,
                                 fe_obs_table_bytes() bytes filled by fe_obs_table_build(); single-asset series only */
} FeSeries;

/* Per-env state, structure of arrays (replaces the tensors of :245-275). */
typedef struct FeState {
    int32_t *seg;        /* (N,)   env -> segment            (env_indices :246) */
    int32_t *ptr;        /* (N,)   time pointer              (env_pointers :258; env_spots[i,j] == ptr[i]+j) */
    float *cash;         /* (N,)   :264 */
    float *long_sh;      /* (N,A)  :267 */
    float *short_sh;     /* (N,A)  :268 */
    double *margin;      /* (N,A)  :269 (f64 from the first step on, :383) */
    uint8_t *terminated; /* (N,)   evaluate only :272 (may be NULL otherwise) */
    float *ep_return;    /* (N,)   evaluate: :275; training: running episode return when stats != NULL */
    int32_t *ep_len;     /* (N,)   running episode length when stats != NULL (may be NULL) */
    unsigned int *sched; /* optional (NULL: none) 4 zero-initialised words of scratch owned by this env: the gather variant's
                            tile counter (its blocks claim tiles), block and bookkeeper arrival counters; the last block out
                            rewinds them.  Launches that share it must not run concurrently — an env's steps never do. */
} FeState;

/* Device-side episode statistics, accumulated with one atomic per thread block (extension; the
 * values all-reduced over NCCL by finenvs_b200.parallel).  May be NULL. */
typedef struct FeStats {
    unsigned long long n_done;       /* envs finished (all steps since last clear) */
    unsigned long long n_terminated; /* evaluate: envs terminated since the metrics were reset (:529-531) */
    unsigned long long sum_len;      /* sum of finished episode lengths */
    unsigned long long pad;
    double sum_return;               /* sum of finished episode returns */
    double sum_return_sq;
} FeStats;

int fe_version(void);
const char *fe_error_string(int code);

/* Shared-memory bytes per env the tile variant needs for (window, out_f64), and the envs-per-block it
 * would pick (0 = does not fit, the direct variant is used). */
int fe_tile_envs(int32_t window, int32_t out_f64, int32_t device);
/* Envs per tile (<= 32, multiple of 4) the pipe variant would use for (window, out_f64) in its "cached"
 * (stream_flavour = 0: series L2-resident, register prefetch) or "stream" (1: cp.async in-ring) flavour;
 * 0 if the window does not fit (the tile / direct variants are used instead). */
int fe_pipe_envs(int32_t window, int32_t out_f64, int32_t stream_flavour);

/* Name of the kernel fe_step / fe_observe will launch for these parameters, this series and this state (s / st may be
 * NULL: as if obs_table / sched were NULL).  Diagnostics, bench.py. */
const char *fe_step_kernel_name(const FeParams *p, const FeSeries *s, const FeState *st);

/* Observation-layout table of the gather variant (replaces the (N,L,4) gather + cat of get_log_return_observations /
 * reset, :423-445, on the read side): the (T,4) log-returns as 5-value rows [lr0..lr3, hole for the position feature],
 * in P = 4 (float) / 2 (double) copies shifted by one row each so that every window start is 16-byte aligned for the TMA
 * engine.  fe_obs_table_bytes: buffer size for (num_rows, window, dtype), 0 when this window has no gather variant
 * (a window's 5*W*sizeof(value) bytes must be a multiple of 16 and <= 2048, or <= 4096 with W <= 128 and half of them a
 * multiple of 80: those windows are fetched in two parts — f32 up to 102 rows in one part, e.g. 128 in two; f64 up to 51 in
 * one, 60 or 100 in two).  fe_obs_table_build fills a 16-byte aligned buffer of
 * that size from logret_dev (T,4) of the same dtype.  Worth it while the table stays L2-resident (<= 64 MB: ~800 k rows). */
int64_t fe_obs_table_bytes(int64_t num_rows, int32_t window, int32_t out_f64);
int fe_obs_table_build(const void *logret_dev, int64_t num_rows, int32_t window, int32_t out_f64, void *table_dev, void *stream);

/* generate_log_return_dataset (:179-194): logret[t,a,0] = 100*log(O_t/C_{t-1}) (row 0: O_0/O_0),
 * logret[t,a,1..3] = 100*log(H|L|C / O).  Either output may be NULL. */
int fe_log_returns(const double *prices_dev, int64_t num_rows, int32_t num_assets, double *logret64_dev,
                   float *logret32_dev, void *stream);

/* find_nan_spots (:486-496) folded into the segment table:
 * seg_len[d] = min(raw_len[d], first k >= W+1 with isnan(logret64[seg_start[d]+k, 0, 0])). */
int fe_effective_len(const double *logret64_dev, const int64_t *seg_start_dev, const int32_t *raw_len_dev,
                     int32_t num_segments, int32_t window, int32_t num_assets, int32_t *seg_len_dev, void *stream);

/* reset() (:423-445): materialise the current observation (N, W, 5A); touches no state. */
int fe_observe(const FeParams *p, const FeSeries *s, const FeState *st, void *obs_dev, void *stream);

/* step() (:277-296) and everything it calls (:298-536) as ONE kernel.
 * actions (N,A) float in [-1,1]; obs (N,W,5A); rewards (N,); dones (N,) int32.
 * step_counter: ordinal of this step (1 for the first step after construction / reset_all). */
int fe_step(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, void *obs_dev,
            void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t step_counter, void *stream);

/* fe_step whose step ordinal lives in device memory: the launch first increments *step_counter_dev, then steps
 * with the new value.  Nothing in the launch depends on a host-side scalar that changes from step to step, so a
 * policy -> step loop can be captured once in a CUDA graph and replayed (evaluation sweeps, small populations whose
 * step is launch-bound; replaces the Python loop of examples/time_series/PPO_LSTM_testing_SPY.py:43-52). */
int fe_step_captured(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, void *obs_dev,
                     void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t *step_counter_dev, void *stream);

/* Lazy observations (extension): an observation is fully described by the 12-byte handle (row0, posfeat):
 * obs[i,j,0:4] = logret[row0[i]+j], obs[i,j,4] = posfeat[i] (:428-445).  fe_step_lazy / fe_observe_lazy are fe_step /
 * fe_observe writing the handle instead of the (N,W,5) tensor (single-asset envs); fe_materialize builds the tensor
 * from a handle (identical to what fe_step would have written).  Used by the fused ES policy (fe_es_forward). */
int fe_observe_lazy(const FeParams *p, const FeSeries *s, const FeState *st, int64_t *obs_row0_dev, void *obs_posfeat_dev,
                    void *stream);
int fe_step_lazy(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, int64_t *obs_row0_dev,
                 void *obs_posfeat_dev, void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t step_counter,
                 void *stream);
int fe_materialize(const FeParams *p, const FeSeries *s, const int64_t *obs_row0_dev, const void *obs_posfeat_dev,
                   void *obs_dev, void *stream);
/* obs[b] = the observation described by handle index[b] (index_dev == NULL: handle b), b < count; (count, W, 5) written
 * contiguously to obs_dev (16-byte aligned).  Bit-identical to what fe_step / fe_materialize write for the same handle.
 * Single-asset series only.  Index values are the caller's responsibility (like fe_materialize's handles).  A rollout
 * buffer keeps the 12-byte handles and builds shuffled minibatches with this call.  Two paths: while s->obs_table is
 * staged for this window and L2-resident (as for the gather variant), windows arrive by TMA gather4 (four samples, or
 * two for windows fetched in two parts, per instruction) and leave by bulk stores; otherwise a warp per sample copies
 * from s->logret.  fe_materialize is this call with index_dev == NULL and count = p->num_envs.  count == 0: nothing is
 * launched. */
int fe_gather_obs(const FeParams *p, const FeSeries *s, const int64_t *row0_dev, const void *posfeat_dev,
                  const int64_t *index_dev, int64_t count, void *obs_dev, void *stream);
const char *fe_gather_obs_kernel_name(const FeParams *p, const FeSeries *s); /* which path; host-only, for tests */

/* Same step driven from HOST buffers (the call a non-torch embedder makes).  When actions_host, rewards_host and
 * dones_host are all pinned (cudaHostAlloc / cudaHostRegister), the step kernel itself reads the actions from and
 * writes rewards / dones to host memory over PCIe (zero-copy: no separate upload or download); otherwise the envs
 * are cut into chunks whose upload, kernel and download are pipelined over three streams (also with pinned buffers for
 * the tile / direct variants above 32 Ki envs, whose blocks would wait on PCIe holding their shared memory).  Either way the call
 * returns after the results are in rewards_host / dones_host; rewards_dev / dones_dev hold the same values; the
 * observation stays in HBM (obs_dev) for the policy.  actions_dev is scratch (N*A floats). */
int fe_step_host(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_host,
                 float *actions_dev, void *obs_dev, void *rewards_dev, int32_t *dones_dev, void *rewards_host,
                 int32_t *dones_host, FeStats *stats_dev, uint64_t step_counter, void *stream);
/* fe_step_host with the dones bit-packed on the wire: dones_bits_host holds ceil(N/32) little-endian 32-bit words,
 * bit (i % 32) of word i / 32 = done flag of env i (4 bytes per env -> 1 bit: 12 -> 8.1 bytes per env-step over PCIe,
 * which is what bounds 8 ranks sharing one host).  dones_dev still receives the int32 flags.  The words are built by the
 * step kernel (one ballot per 32-env tile), staged in actions_dev and leave for the host in full 128-byte lines; with the
 * gather variant that uses the arrival counters of FeState.sched. */
int fe_step_host_packed(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_host,
                        float *actions_dev, void *obs_dev, void *rewards_dev, int32_t *dones_dev, void *rewards_host,
                        uint32_t *dones_bits_host, FeStats *stats_dev, uint64_t step_counter, void *stream);

/* Extension (mirrors isaac_gym_env.py:55-58 reset_all): fresh episode for every env; with redraw != 0
 * each env draws (segment[, offset]) from Philox(seed, global env id, step_counter). */
int fe_reset_all(const FeParams *p, const FeSeries *s, const FeState *st, uint64_t step_counter, int32_t redraw,
                 void *stream);

/* The redraw RNG evaluated on the host (Philox4x32-10; key = seed, counter = (env id, step, kind)):
 * lets callers reproduce / pre-compute draws.  kind: 0 step-time reset, 1 reset_all / constructor. */
void fe_philox(uint64_t seed, uint64_t env_id, uint64_t step, uint32_t kind, uint32_t out[4]);

/* Market-data CSV reader of the loader (host code, no GPU work): replaces pandas.read_csv of read_data()
 * (finenvs/environments/time_series_env.py:80-88) for records `Date,Time,Open,High,Low,Close,Volume`.
 * fe_csv_open maps the file, cuts it into one chunk per thread (num_threads <= 0: all hardware threads) and counts the
 * records (non-empty lines); fe_csv_read fills caller-owned arrays of num_rows entries: date_key = 64-bit FNV-1a hash of
 * the Date string (the reference compares dates as strings, :98, :141-152), sec_of_day = seconds since midnight of the
 * Time field (for between_time("9:30", "15:59"), :90-91), ohlc = (num_rows, 4) float64 converted exactly like pandas'
 * default converter (bit-identical prices).  FE_ECSV = some record is outside this format.  fe_csv_close unmaps. */
int fe_csv_open(const char *path, int32_t num_threads, void **handle, int64_t *num_rows);
int fe_csv_read(void *handle, int64_t *date_key, int32_t *sec_of_day, double *ohlc);
void fe_csv_close(void *handle);

/* ---- callers of the step (SURVEY.md 8f) --------------------------------------------------------------- */

/* PPO rollout returns (finenvs/agents/PPO/buffer.py:80-100, compute_returns_and_advantages) over a TIME-MAJOR
 * rollout: rewards (T,N) float or double (rewards_f64), dones (T,N) int32, values (T,N) float, last_values (N,)
 * float -> returns (T,N) float, advantages (T,N) float.  returns[t] = rewards[t] + (1-dones[t])*gamma*returns[t+1]
 * with the reference's dtype promotion (DESIGN.md, "PPO rollout storage"). */
int fe_returns_advantages(const void *rewards_dev, int32_t rewards_f64, const int32_t *dones_dev, const float *values_dev,
                          const float *last_values_dev, int64_t num_envs, int32_t num_steps, double gamma,
                          float *returns_dev, float *advantages_dev, void *stream);

/* ---- per-episode trading metrics (extension; DESIGN.md §4.11) ---------------------------------------------
 * An episode of env i runs from a reset to the step whose done flag is 1, that step's reward included.  r is the
 * reward the step returned (float or double, promoted to double); all accumulation is in double, per step in this order:
 *     len += 1;  sum += r  (cumulative P&L);
 *     d = r - mean;  mean += d / len;  m2 += d * (r - mean)   (Welford);
 *     pos += (r > 0);  peak = max(peak, sum)  (peak starts at 0);
 *     mdd = max(mdd, peak - sum);  mdd_rel = max(mdd_rel, (peak - sum) / (starting_balance + peak)).
 * At done one record is emitted and the running state is zeroed:
 *     key = step_ordinal * total_envs + global env id (sorting by key gives (step, env) order, as fe_es_store);
 *     sharpe = mean / sqrt(m2 / len), 0 when len < 2 or m2 == 0 — the per-step ratio, not annualised;
 *     hit_rate = pos / len.
 * With FeParams.evaluate an env records only its first episode after its `emitted` flag was cleared (terminated envs
 * keep stepping with zero reward and must not record again).  Every product, quotient and sum is one IEEE-rounded f64
 * operation (no FMA contraction), so a numpy restatement with the same operations in the same order matches bit for
 * bit. */
typedef struct FeMetricsSummary {
    unsigned long long episodes; /* finished episodes recorded since the last clear; also the next list slot (> capacity:
                                    the list overflowed, the entries past capacity were not written) */
    unsigned long long sum_len;
    double sum_return;
    double sum_sharpe;
    double sum_sharpe_sq;
    double sum_mdd;
    double max_mdd;              /* atomic max on the bit pattern (mdd >= 0) */
    double sum_hit_rate;
} FeMetricsSummary;

typedef struct FeMetricsState {
    /* running state of the current episode, (N,) each, zero-initialised */
    int32_t *len;
    int32_t *pos;
    double *sum;
    double *mean;
    double *m2;
    double *peak;
    double *mdd;
    double *mdd_rel;
    uint8_t *emitted;            /* (N,) evaluate only: the env has recorded its first episode (may be NULL otherwise) */
    /* finished-episode list, `capacity` entries each, filled in slot order (sort by key for (step, env) order) */
    int64_t *fin_key;
    int64_t *fin_env;            /* global env id */
    int32_t *fin_len;
    double *fin_return;          /* sum */
    double *fin_sharpe;
    double *fin_mdd;
    double *fin_mdd_rel;
    double *fin_hit_rate;
    FeMetricsSummary *summary;   /* aggregates of every recorded episode, overflowed ones included */
} FeMetricsState;

/* Advance the metrics of p->num_envs envs by one step's rewards (float, or double when p->out_f64) and dones (int32),
 * the device outputs of any step entry point.  The step ordinal is *step_counter_dev when that is not NULL (the counter
 * fe_step_captured increments, so the launch can be captured in a CUDA graph right after it), else step_counter.
 * Finished episodes take slots with one atomic per 1024-env block; slots >= capacity are counted, not written. */
int fe_episode_metrics(const FeParams *p, const FeMetricsState *m, const void *rewards_dev, const int32_t *dones_dev,
                       uint64_t step_counter, const uint64_t *step_counter_dev, int64_t capacity, void *stream);

/* ---- signal backtests (extension; DESIGN.md §4.12) ----------------------------------------------------------
 * A signal table signal_dev (num_signals, p->num_rows) float holds one row ("column") per rule-based strategy and one
 * value per row of the staged flat series; values are actions, mapped exactly like fe_step's (rint(a * (max_shares +
 * 0.5)), clamped).  Env i trades column column_dev[i] in [0, num_signals) (the caller's responsibility, like
 * fe_gather_obs' index).  fe_backtest advances every env num_steps steps in ONE launch and is bit-identical to
 * num_steps calls of fe_step + fe_episode_metrics with step ordinals first_step, first_step + 1, ... in which env i's
 * action at each step is
 *     a_i = signal[column[i], seg_start[seg_i] + ptr_i + W - 1]        (seg_i, ptr_i: the state BEFORE the step)
 * i.e. the last row of the window the env observes; the trade executes at the next row's Open, so a signal computed from
 * rows <= r never trades on row r's prices: no look-ahead by construction.  Identical are the per-env state, the Philox
 * redraws, the FeStats counts, the metrics' running state, the records of the finished-episode list (same keys and values;
 * which records win a slot on overflow depends on warp timing, as with fe_episode_metrics) and the summary counts and
 * max_mdd; f64 sums are the same values added in another order.  rewards_dev / dones_dev: (num_steps, N) histories when
 * history != 0, else (N,) holding the last step.  No observation is written.  Single-asset series only (num_assets == 1);
 * evaluate mode needs m->emitted, FeStats (stats_dev, may be NULL) as fe_step. */
int fe_backtest(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m, int64_t metrics_capacity,
                FeStats *stats_dev, const float *signal_dev, int32_t num_signals, const int32_t *column_dev,
                uint64_t first_step, int32_t num_steps, void *rewards_dev, int32_t *dones_dev, int32_t history, void *stream);

/* Target-position backtests: as fe_backtest, but the table value v = signal[column[i], row] (same row) is the net
 * position env i should hold, and exits_dev (num_signals, 2) double, or NULL, holds per column c a trailing stop
 * exits[c][0] and a take-profit exits[c][1] in reward units (the episode's P&L).  Per env and step, on the state before
 * the step, f32 unless noted (scale = (float)(max_shares + 0.5), ms = max_shares; sum, peak: the metrics' running
 * state of the current episode):
 *     T = clamp(rintf(v * scale), -ms, ms)                          target net position in shares
 *     if exits_dev && ((peak - sum) >= exits[c][0] || sum >= exits[c][1])   (f64)
 *         T = +0.0f                                                  go flat
 *     D = T - (long - short)                                         share delta that reaches the target
 *     a = D / scale                                                  (IEEE-rounded), the action of the step
 * The step maps a back to clamp(rint(a * scale), -ms, ms) = clamp(D, -ms, ms): for |D| <= 2^21 the two rounding errors
 * stay below 2^21 * 2^-23 = 0.25 shares (max_shares <= FE_TARGET_MAX_SHARES keeps scale exact; larger max_shares are
 * FE_EINVAL), and beyond that bound they cannot bring |a * scale| below ms.  So a target backtest is bit-identical to
 * fe_step calls with these actions computed by the caller, and follows the env's rules: a flip from +ms to -ms takes two
 * steps (the first sells the longs, the short entry sees no sell order), an entry the cash cannot pay for is retried on
 * the next step, and the exit rule is evaluated every step without latching: once flat the rewards are 0, sum and peak
 * stay put and the env stays flat until its episode ends; the next episode trades again.  A threshold of +inf never
 * triggers.  exits_dev must be 8-byte aligned (FE_EALIGN); the other checks are fe_backtest's. */
#define FE_TARGET_MAX_SHARES (1 << 20)
int fe_backtest_targets(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m,
                        int64_t metrics_capacity, FeStats *stats_dev, const float *signal_dev, int32_t num_signals,
                        const int32_t *column_dev, const double *exits_dev, uint64_t first_step, int32_t num_steps,
                        void *rewards_dev, int32_t *dones_dev, int32_t history, void *stream);

/* Portfolio backtests (any 1 <= num_assets <= 32): the signal table signal_dev (num_signals, p->num_rows, A) float is
 * time-major like the series, so the A values of one column at one row are 4A contiguous bytes.  At every step env i
 * reads, with the state before the step,
 *     v[a] = signal[column[i], seg_start[seg_i] + ptr_i + W - 1, a]          a = 0 .. A-1
 * and, per asset, applies fe_backtest's rule (targets == 0: v[a] is asset a's action) or fe_backtest_targets' rule
 * (targets != 0: v[a] is asset a's target net position, T_a = clamp(rintf(v[a] * scale), -ms, ms), action
 * (T_a - (long_a - short_a)) / scale).  exits_dev (num_signals, 2) double, targets only: a trailing stop and a
 * take-profit per column on the episode's portfolio P&L (the metrics' running sum / peak of the env, the sum over its
 * assets); when either triggers, every asset's target is 0 for that step (not latched).  The portfolio env's rules
 * apply: long entries, then short entries, are all-or-nothing per asset and greedy in asset order (an asset the cash
 * left by the earlier ones cannot pay for stays flat and is retried on the next step), a flip from long to short takes
 * two steps per asset, and margin calls and bankruptcy act on the whole account.  The run is bit-identical to
 * num_steps calls of fe_step + fe_episode_metrics with actions[i, a] computed that way (the same per-env and per-asset
 * state, redraws, FeStats counts, metrics state, records, summary counts and max_mdd; f64 sums in another order), and
 * at A = 1 to fe_backtest / fe_backtest_targets.  Checks: fe_backtest's (except num_assets), exits_dev without
 * targets is FE_EINVAL, a misaligned exits_dev FE_EALIGN, targets with max_shares outside [1, FE_TARGET_MAX_SHARES]
 * FE_EINVAL; every refusal happens before any CUDA call. */
int fe_backtest_portfolio(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m,
                          int64_t metrics_capacity, FeStats *stats_dev, const float *signal_dev, int32_t num_signals,
                          const int32_t *column_dev, int32_t targets, const double *exits_dev, uint64_t first_step,
                          int32_t num_steps, void *rewards_dev, int32_t *dones_dev, int32_t history, void *stream);

/* ---- rule backtests (extension; DESIGN.md §4.12, "Rules computed on the device") ---------------------------
 * A rule is a 32-byte FeRule record; a rule set is an array of them indexed by column, and its value at a row r of the
 * staged series (the row fe_backtest reads, seg_start + ptr + W - 1 before the step) for asset a is computed from the
 * closes C[j] = prices[j, a, 3] (f64) of rows j <= r only:
 *     s in {-1, 0, +1} by kind (0 while r is too small for the lookback, i.e. a row before 0 would be needed):
 *       FE_RULE_CONST         +1
 *       FE_RULE_MOMENTUM      (lookback w >= 1) sign(C[r] - C[r-w]); 0 when equal or either close is not finite
 *       FE_RULE_MA_CROSS      (lookback f, lookback2 sl, 1 <= f < sl) sign(M_f - M_sl), M_k the mean of C over r-k+1 .. r
 *       FE_RULE_BOLLINGER     (lookback w >= 2, k > 0) -1 if C[r] > M_w + k sd_w, +1 if C[r] < M_w - k sd_w, else 0
 *                             (sd_w: population standard deviation of the same w closes)
 *       FE_RULE_XS_MOMENTUM   (lookback w >= 1, lookback2 n, 1 <= n <= A/2; portfolios) rank the assets by
 *                             q_a = C_a[r] / C_a[r-w], descending, ties to the lower asset index: +1 for the first n,
 *                             -1 for the last n, 0 otherwise.  An asset whose q is not finite (a non-finite close, or
 *                             C_a[r-w] == 0) takes no rank and gets 0, and the others are ranked among themselves; when
 *                             fewer than 2n assets have a finite q, every asset gets 0.
 *     long_only != 0 maps s to max(s, 0); the value is v = +size, -size or +0.0f for s = +1, -1, 0, and goes into
 *     fe_backtest_portfolio's rule unchanged (an action, or with targets a target net position).
 * Time-series kinds apply per asset to the asset's own closes; CONST gives every asset `size`.  Any window containing a
 * non-finite close gives 0 (MA_CROSS, BOLLINGER).  Every value is a function of (rule, row, asset) alone, computed with
 * IEEE f64 basic operations and sqrt in a fixed order (no FMA), so a numpy restatement (oracle/oracle_rules.py) matches
 * bit for bit.  Evaluation is total: an unknown kind, a lookback outside [1, FE_RULE_MAX_LOOKBACK], or a parameter
 * outside the ranges above gives 0 and reads nothing, so no record can make a kernel read outside the series.
 *
 * Window means and deviations come from running sums staged once per series by fe_rule_sums_build: per asset, the
 * series is cut into blocks of FE_RULE_BLOCK rows; each block has a base (its first finite close, 0 if none) and holds
 * inclusive running sums, restarted at the block's first row, of d = C - base and d*d (d = 0 for a non-finite close,
 * which is counted instead).  A window sum is assembled from at most 1 + lookback / FE_RULE_BLOCK block pieces, each
 * shifted to the base of the window's last block (a single prefix sum over 10 M rows would cancel catastrophically).
 * Accuracy: the window variance (BOLLINGER's sd_w^2, formed as t2/w - (t1/w)^2 from those sums) has an ABSOLUTE error
 * of at most a small multiple of u * M (u = 2^-53), where M, the sum of the magnitudes of the staged terms the window
 * is formed from divided by w, is set by the prices and their drift inside the window's blocks, not by the row index
 * (measured on every row of a 10 M-row series: below 51 u M; oracle_rules.window_error_scale computes M).  The error is
 * not relative: a window whose variance is far below u M, such as two nearly equal closes late in a block, can carry a
 * large relative error in sd_w, and a window of equal closes can get sd_w of order sqrt(u M) instead of 0.  Window
 * means hold a relative error of a few ulps.  The buffer holds, for
 * T rows, A assets and B = ceil(T / FE_RULE_BLOCK) blocks: sum d (T, A) f64, sum d*d (T, A) f64, base (B, A) f64,
 * non-finite count (T, A) int32 — fe_rule_sums_bytes() bytes, 16-byte aligned. */
#define FE_RULE_CONST 0
#define FE_RULE_MOMENTUM 1
#define FE_RULE_MA_CROSS 2
#define FE_RULE_BOLLINGER 3
#define FE_RULE_XS_MOMENTUM 4
#define FE_RULE_MAX_LOOKBACK 65536
#define FE_RULE_BLOCK 1024

typedef struct FeRule {
    int32_t kind;       /* FE_RULE_* */
    int32_t lookback;   /* w (MOMENTUM, BOLLINGER, XS_MOMENTUM) or the fast f (MA_CROSS) */
    int32_t lookback2;  /* the slow sl (MA_CROSS) or n (XS_MOMENTUM); 0 otherwise */
    int32_t long_only;  /* != 0: s -> max(s, 0) */
    double k;           /* BOLLINGER band width in standard deviations; 0 otherwise */
    float size;         /* v = s * size */
    int32_t reserved;   /* 0 */
} FeRule;

int64_t fe_rule_sums_bytes(int64_t num_rows, int32_t num_assets);
int fe_rule_sums_build(const double *prices_dev, int64_t num_rows, int32_t num_assets, void *sums_dev, int32_t device,
                       void *stream);

/* fe_backtest_portfolio with every value computed by rule column_dev[i] of rules_dev (num_rules FeRule records,
 * 8-byte aligned) from the staged closes instead of loaded from a table: at A = 1 the thread-per-env loop of
 * fe_backtest / fe_backtest_targets, at A > 1 the warp-per-env loop of fe_backtest_portfolio, each fed by the rule.
 * The run is bit-identical to fe_backtest_portfolio (at A = 1 also fe_backtest / fe_backtest_targets) with the table
 * fe_rule_table writes for the same rules: everything those calls guarantee, f64 sums up to their order of addition.
 * rule_sums_dev: fe_rule_sums_build's buffer for s->prices.  Checks: fe_backtest_portfolio's, plus a NULL rules_dev /
 * rule_sums_dev or num_rules < 1 FE_EINVAL and a misaligned one FE_EALIGN; every refusal happens before any CUDA call.
 * Records are not checked here: the caller validates them (an out-of-range field evaluates to 0). */
int fe_backtest_rules(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m,
                      int64_t metrics_capacity, FeStats *stats_dev, const void *rule_sums_dev, const FeRule *rules_dev,
                      int32_t num_rules, const int32_t *column_dev, int32_t targets, const double *exits_dev,
                      uint64_t first_step, int32_t num_steps, void *rewards_dev, int32_t *dones_dev, int32_t history,
                      void *stream);

/* The (num_rules, num_rows, num_assets) float table the rules define: table[c, r, a] = the value of rules_dev[c] at row r
 * for asset a, computed by the same device function as fe_backtest_rules.  FE_EINVAL for a NULL pointer or a
 * non-positive size, num_assets outside 1..32; FE_EALIGN for a misaligned pointer. */
int fe_rule_table(const double *prices_dev, const void *rule_sums_dev, int64_t num_rows, int32_t num_assets,
                  const FeRule *rules_dev, int32_t num_rules, float *table_dev, int32_t device, void *stream);

/* ---- ES rollout path (finenvs/agents/networks/parallel_mlp.py, finenvs/agents/ES/evo_agent.py) -------------
 * Population layout of the reference (parallel_mlp.py:121-136): envs [0, T/2) use theta + sigma*eps[p], envs
 * [T/2, T) use theta - sigma*eps[p - T/2] (T = num_envs - num_eval_envs, even), the last num_eval_envs envs use
 * theta.  Perturbations are stored per PAIR as fp16 in the packed layout
 *     index(layer l, input j (j == in_l: bias), output o) = off[l] + ((o/8)*(in_l+1) + j)*8 + o%8,
 * off[l+1] = off[l] + ceil(out_l/8)*(in_l+1)*8; theta and the gradient use the same layout in f32. */
#define FE_ES_MAX_LAYERS 4
typedef struct FeEsNet {
    int32_t num_layers;                 /* weight layers: len(shape) - 1 (parallel_mlp.py:46-50) */
    int32_t dims[FE_ES_MAX_LAYERS + 1]; /* shape: (num_observations, *hidden_dims, num_actions); tanh after every layer */
} FeEsNet;

/* P_pad: packed values per network; index of one parameter in the packed layout (-1: invalid). */
int64_t fe_es_params_padded(const FeEsNet *net);
int64_t fe_es_packed_index(const FeEsNet *net, int32_t layer, int32_t input, int32_t output);

/* perturb_parameters (:112-155): eps[pair, q] ~ N(0,1) as a pure function of (seed, generation, pair_id_base + pair,
 * q): Philox4x32-10 + Box-Muller.  eps_dev: (num_pairs, P_pad) fp16, 16-byte aligned.  generation < 2^31. */
int fe_es_perturb(const FeEsNet *net, uint64_t seed, uint64_t generation, int64_t pair_id_base, int64_t num_pairs,
                  void *eps_dev, void *stream);

/* forward (:84-109) for every env: actions (N, num_actions) = MLP(theta +- sigma*eps)(obs) [+ N(0, action_noise_std)
 * exploration noise, reference semantics: none for eval envs, none at all when num_eval_envs == 0].
 * Observations: dense obs_dev (N, dims[0]) f32, or — obs_dev == NULL — lazy handles (obs_row0_dev, obs_posfeat_dev)
 * from fe_step_lazy plus the staged log-return table logret_dev (T,4) f32 and window (dims[0] == window*5). */
int fe_es_forward(const FeEsNet *net, const float *theta_packed_dev, const void *eps_dev, float sigma, int64_t num_envs,
                  int64_t num_eval_envs, const float *obs_dev, const void *logret_dev, const int64_t *obs_row0_dev,
                  const float *obs_posfeat_dev, int32_t window, float action_noise_std, uint64_t seed,
                  uint64_t step_counter, int64_t env_id_base, float *actions_dev, int32_t device, void *stream);
/* Which forward kernel fe_es_forward launches for this network (host-only, for tests): "fe_es_forward_fast_kernel<lazy>",
 * "fe_es_forward_stream_kernel<dense> U=2" (U: pairs per warp), "fe_es_forward_kernel<lazy,theta_smem>" /
 * "...,theta_global>", or "none (FE_ESMEM: ...)".  lazy: observations come as handles; obs_aligned: the dense
 * observation pointer is 16-byte aligned (ignored when lazy).  "" for an invalid network. */
const char *fe_es_forward_kernel_name(const FeEsNet *net, int32_t lazy, int32_t obs_aligned);

/* update_parameters' reduction (:176-218): grad_packed[q] = sum_p pair_weights[p] * eps[p, q] (pair_weights =
 * fitness(+) - fitness(-)); deterministic.  scratch_dev: fe_es_gradient_scratch(net, num_pairs) floats. */
int64_t fe_es_gradient_scratch(const FeEsNet *net, int64_t num_pairs);
int fe_es_gradient(const FeEsNet *net, const void *eps_dev, const float *pair_weights_dev, int64_t num_pairs,
                   float *scratch_dev, float *grad_packed_dev, void *stream);

/* EvoAgent.step/.store accounting (evo_agent.py:90-112) without host synchronisation: cur_steps += 1,
 * cur_returns += rewards; every done env appends (key, env, return) to the finished list (capacity entries; overflow
 * is counted, not written), adds its step count to counters[1], and is zeroed.  counters[0] = finished episodes.
 * key = step_ordinal * total_envs + env_id_base + env: sorting by key gives the reference's list order. */
int fe_es_store(const void *rewards_dev, int32_t rewards_f64, const int32_t *dones_dev, int64_t num_envs,
                int64_t env_id_base, int64_t total_envs, uint64_t step_ordinal, float *cur_returns_dev,
                float *cur_steps_dev, int64_t capacity, unsigned long long *counters_dev, int64_t *fin_key_dev,
                int64_t *fin_env_dev, float *fin_ret_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FINENVS_B200_H */
