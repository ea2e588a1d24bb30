// fe_metrics.cu — per-episode trading metrics (P&L, Sharpe ratio, drawdown, hit rate) on the device.
//
// fe_episode_metrics_kernel runs right after a step, one thread per env.  The running state is structure-of-arrays
// (every load and store coalesced over the env dimension): 6 doubles + 2 int32 read and written once per step, plus the
// step's reward and done flag — ~128 bytes per env-step against the step's ~2.3 kB at W = 60.  Finished episodes are
// reduced per block (slots inside the block in env order) and appended to a caller-owned list, and folded into a small
// aggregate block, with one atomic per block and field: all of them land on one 64-byte line, and one atomic per warp
// and field (the fe_es_store_kernel scheme) serialised there (c2, 1 Mi envs: ~5 000 warps with a finished episode per
// step).
// The definition (op order) is in include/finenvs_b200.h and its one implementation in fe_metrics.cuh (fe_backtest_kernel
// uses it too); every product, quotient and sum is an explicit __d*_rn intrinsic (the TU is also built with -fmad=false),
// so a numpy restatement reproduces the records bit for bit.
#include "finenvs_b200.h"
#include "fe_common.cuh"
#include "fe_metrics.cuh"

#include <cuda_runtime.h>
#include <stdint.h>

namespace {

constexpr unsigned kAll = 0xFFFFFFFFu;
constexpr int kThreads = 1024;
constexpr int kWarps = kThreads / 32;   // = 32: warp 0 reduces one lane per warp

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(kAll, v, o));
    return v;
}

template <typename RewT>
__global__ void __launch_bounds__(kThreads)
fe_episode_metrics_kernel(const RewT *__restrict__ rewards, const int32_t *__restrict__ dones, const int64_t N,
                          const int64_t env_id_base, const int64_t total_envs, const double starting_balance,
                          const FeMetricsState m, const uint64_t step_counter, const uint64_t *__restrict__ step_counter_dev,
                          const int64_t capacity) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int emit = 0;
    int32_t len = 0;
    double sum = 0.0, sharpe = 0.0, mdd = 0.0, mdd_rel = 0.0, hit = 0.0;
    if (i < N) {
        const double r = (double)rewards[i];
        const EpisodeRun e = episode_advance(RunInMemory{m, i}, r, starting_balance);
        len = e.len; sum = e.sum; mdd = e.mdd; mdd_rel = e.mdd_rel;
        if (dones[i] != 0) {
            emit = 1;
            if (m.emitted) {   // evaluate: only the first episode after the flags were cleared
                emit = !m.emitted[i];
                m.emitted[i] = 1;
            }
            sharpe = episode_sharpe(e);
            hit = episode_hit_rate(e);
            episode_store(m, i, EpisodeRun{});
        } else {
            episode_store(m, i, e);
        }
    }
    __shared__ double s_sum[6][kWarps];                 // return, sharpe, sharpe^2, mdd, hit_rate, max mdd
    __shared__ unsigned long long s_cnt[2][kWarps];     // episodes, len
    __shared__ unsigned long long s_off[kWarps];        // first slot of each warp
    const unsigned ballot = __ballot_sync(kAll, emit);
    if (ballot) {
        unsigned long long wlen = emit ? (unsigned long long)len : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wlen += __shfl_xor_sync(kAll, wlen, o);
        const double wret = warp_sum(emit ? sum : 0.0);
        const double wsh = warp_sum(emit ? sharpe : 0.0);
        const double wsh2 = warp_sum(emit ? __dmul_rn(sharpe, sharpe) : 0.0);
        const double wmdd = warp_sum(emit ? mdd : 0.0);
        const double whit = warp_sum(emit ? hit : 0.0);
        double wmax = emit ? mdd : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wmax = fmax(wmax, __shfl_xor_sync(kAll, wmax, o));
        if (lane == 0) {
            s_sum[0][warp] = wret; s_sum[1][warp] = wsh; s_sum[2][warp] = wsh2; s_sum[3][warp] = wmdd;
            s_sum[4][warp] = whit; s_sum[5][warp] = wmax;
            s_cnt[0][warp] = (unsigned long long)__popc(ballot); s_cnt[1][warp] = wlen;
        }
    } else if (lane == 0) {
        for (int k = 0; k < 6; ++k) s_sum[k][warp] = 0.0;
        s_cnt[0][warp] = 0; s_cnt[1][warp] = 0;
    }
    __syncthreads();
    if (warp == 0) {   // lane w holds warp w's partials
        const unsigned long long cnt = s_cnt[0][lane];
        unsigned long long incl = cnt;   // inclusive prefix over the warps: slots in env order inside the block
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(kAll, incl, o);
            if (lane >= o) incl += v;
        }
        const unsigned long long total = __shfl_sync(kAll, incl, 31);
        if (total) {
            unsigned long long blen = s_cnt[1][lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) blen += __shfl_xor_sync(kAll, blen, o);
            double b[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) b[k] = warp_sum(s_sum[k][lane]);
            double bmax = s_sum[5][lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) bmax = fmax(bmax, __shfl_xor_sync(kAll, bmax, o));
            unsigned long long base = 0;
            if (lane == 0) {
                FeMetricsSummary *sm = m.summary;
                base = atomicAdd(&sm->episodes, total);
                atomicAdd(&sm->sum_len, blen);
                atomicAdd(&sm->sum_return, b[0]);
                atomicAdd(&sm->sum_sharpe, b[1]);
                atomicAdd(&sm->sum_sharpe_sq, b[2]);
                atomicAdd(&sm->sum_mdd, b[3]);
                atomicAdd(&sm->sum_hit_rate, b[4]);
                // mdd >= 0: the order of non-negative doubles is the order of their bit patterns
                atomicMax(reinterpret_cast<unsigned long long *>(&sm->max_mdd), (unsigned long long)__double_as_longlong(bmax));
            }
            base = __shfl_sync(kAll, base, 0);
            s_off[lane] = base + incl - cnt;
        }
    }
    __syncthreads();
    if (emit) {
        const int64_t slot = (int64_t)s_off[warp] + __popc(ballot & ((1u << lane) - 1u));
        if (slot < capacity) {
            const uint64_t step = step_counter_dev ? *step_counter_dev : step_counter;
            const int64_t gid = env_id_base + i;
            episode_write_record(m, slot, (int64_t)step * total_envs + gid, gid, len, sum, sharpe, mdd, mdd_rel, hit);
        }
    }
}

} // namespace

extern "C" int fe_episode_metrics(const FeParams *p, const FeMetricsState *m, const void *rewards_dev,
                                  const int32_t *dones_dev, uint64_t step_counter, const uint64_t *step_counter_dev,
                                  int64_t capacity, void *stream) {
    if (!p || !rewards_dev || !dones_dev || p->num_envs <= 0) return FE_EINVAL;
    if (int rc = check_metrics_state(p, m, capacity)) return rc;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    FeMetricsState ms = *m;
    if (!p->evaluate) ms.emitted = nullptr;
    const unsigned blocks = (unsigned)((p->num_envs + kThreads - 1) / kThreads);
    cudaStream_t q = (cudaStream_t)stream;
    return with_out_type(p->out_f64, [&](auto out_type) {
        using OutT = decltype(out_type);
        fe_episode_metrics_kernel<OutT><<<blocks, kThreads, 0, q>>>((const OutT *)rewards_dev, dones_dev, p->num_envs,
                                                                    p->env_id_base, p->total_envs, p->starting_balance, ms,
                                                                    step_counter, step_counter_dev, capacity);
        return (int)cudaGetLastError();
    });
}
