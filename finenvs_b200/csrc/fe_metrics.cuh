// fe_metrics.cuh — the per-episode metrics update (include/finenvs_b200.h, DESIGN.md §4.11), shared by
// fe_episode_metrics_kernel (fe_metrics.cu: one step, running state in memory) and fe_backtest_kernel (fe_step.cu: K
// steps, running state in registers).  Every product, quotient and sum is an explicit __d*_rn intrinsic.
#ifndef FE_METRICS_CUH
#define FE_METRICS_CUH
#include "finenvs_b200.h"

#include <cuda_runtime.h>
#include <stdint.h>

namespace {

// running state of env i's current episode
struct EpisodeRun {
    int32_t len, pos;
    double sum, mean, m2, peak, mdd, mdd_rel;
};

// the previous running state, each field read where the update needs it: from the state arrays (fe_episode_metrics_kernel)
// or from registers (fe_backtest_kernel)
struct RunInMemory {
    const FeMetricsState &m;
    const int64_t i;
    __device__ __forceinline__ int32_t len() const { return m.len[i]; }
    __device__ __forceinline__ int32_t pos() const { return m.pos[i]; }
    __device__ __forceinline__ double sum() const { return m.sum[i]; }
    __device__ __forceinline__ double mean() const { return m.mean[i]; }
    __device__ __forceinline__ double m2() const { return m.m2[i]; }
    __device__ __forceinline__ double peak() const { return m.peak[i]; }
    __device__ __forceinline__ double mdd() const { return m.mdd[i]; }
    __device__ __forceinline__ double mdd_rel() const { return m.mdd_rel[i]; }
};
struct RunInRegisters {
    const EpisodeRun &e;
    __device__ __forceinline__ int32_t len() const { return e.len; }
    __device__ __forceinline__ int32_t pos() const { return e.pos; }
    __device__ __forceinline__ double sum() const { return e.sum; }
    __device__ __forceinline__ double mean() const { return e.mean; }
    __device__ __forceinline__ double m2() const { return e.m2; }
    __device__ __forceinline__ double peak() const { return e.peak; }
    __device__ __forceinline__ double mdd() const { return e.mdd; }
    __device__ __forceinline__ double mdd_rel() const { return e.mdd_rel; }
};

__device__ __forceinline__ void episode_store(const FeMetricsState &m, int64_t i, const EpisodeRun &e) {
    m.len[i] = e.len; m.pos[i] = e.pos;
    m.sum[i] = e.sum; m.mean[i] = e.mean; m.m2[i] = e.m2; m.peak[i] = e.peak; m.mdd[i] = e.mdd; m.mdd_rel[i] = e.mdd_rel;
}

// one step with reward r, in the header's operation order
template <typename Run>
__device__ __forceinline__ EpisodeRun episode_advance(const Run &a, double r, double starting_balance) {
    EpisodeRun e;
    e.len = a.len() + 1;
    const double dlen = (double)e.len;
    e.sum = __dadd_rn(a.sum(), r);
    const double d = __dsub_rn(r, a.mean());
    e.mean = __dadd_rn(a.mean(), __ddiv_rn(d, dlen));
    e.m2 = __dadd_rn(a.m2(), __dmul_rn(d, __dsub_rn(r, e.mean)));
    e.pos = a.pos() + (r > 0.0 ? 1 : 0);
    e.peak = fmax(a.peak(), e.sum);
    const double dd = __dsub_rn(e.peak, e.sum);
    e.mdd = fmax(a.mdd(), dd);
    e.mdd_rel = fmax(a.mdd_rel(), __ddiv_rn(dd, __dadd_rn(starting_balance, e.peak)));
    return e;
}

// the record fields of a finished episode (the per-step ratio, not annualised)
__device__ __forceinline__ double episode_sharpe(const EpisodeRun &e) {
    return (e.len < 2 || e.m2 == 0.0) ? 0.0 : __ddiv_rn(e.mean, __dsqrt_rn(__ddiv_rn(e.m2, (double)e.len)));
}
__device__ __forceinline__ double episode_hit_rate(const EpisodeRun &e) { return __ddiv_rn((double)e.pos, (double)e.len); }

__device__ __forceinline__ void episode_write_record(const FeMetricsState &m, int64_t slot, int64_t key, int64_t gid,
                                                     int32_t len, double sum, double sharpe, double mdd, double mdd_rel,
                                                     double hit) {
    m.fin_key[slot] = key;
    m.fin_env[slot] = gid;
    m.fin_len[slot] = len;
    m.fin_return[slot] = sum;
    m.fin_sharpe[slot] = sharpe;
    m.fin_mdd[slot] = mdd;
    m.fin_mdd_rel[slot] = mdd_rel;
    m.fin_hit_rate[slot] = hit;
}

// host: the pointers fe_episode_metrics and fe_backtest need (FE_EINVAL when one is missing)
inline int check_metrics_state(const FeParams *p, const FeMetricsState *m, int64_t capacity) {
    if (!m || capacity < 0) return FE_EINVAL;
    if (!m->len || !m->pos || !m->sum || !m->mean || !m->m2 || !m->peak || !m->mdd || !m->mdd_rel || !m->summary)
        return FE_EINVAL;
    if (!m->fin_key || !m->fin_env || !m->fin_len || !m->fin_return || !m->fin_sharpe || !m->fin_mdd || !m->fin_mdd_rel ||
        !m->fin_hit_rate)
        return FE_EINVAL;
    if (p->evaluate && !m->emitted) return FE_EINVAL;
    return 0;
}

} // namespace
#endif // FE_METRICS_CUH
