// fe_rollout.cu — the callers on either side of the env step (SURVEY.md §8f): PPO rollout storage.
//
// fe_returns_advantages: the reverse discounted-return scan of finenvs/agents/PPO/buffer.py:80-100
// (a Python loop of ~6 torch ops per time step there) as ONE kernel over a TIME-MAJOR (T, N) rollout —
// the layout in which the env writes one (N, ...) slab per step.  One thread per env walks t = T-1 .. 0;
// every load and store is coalesced over the env dimension; the loads of the next kUnroll time steps do not
// depend on the running value, so they are issued ahead of the dependent multiply-add chain.
// Arithmetic follows the reference dtype for dtype (DESIGN.md §4.6): f32 products/sums for f32
// rewards; for f64 rewards the running value is f64 after the first iteration and each stored return is
// rounded once.  No FMA contraction (explicit __*_rn intrinsics; the TU is also built with -fmad=false).
#include "finenvs_b200.h"
#include "fe_common.cuh"

#include <cuda_runtime.h>
#include <stdint.h>

namespace {

constexpr int kUnroll = 8;

template <typename RewT>
__global__ void __launch_bounds__(256)
fe_returns_kernel(const RewT *__restrict__ rewards, const int32_t *__restrict__ dones, const float *__restrict__ values,
                  const float *__restrict__ last_values, const int64_t N, const int T, const float gamma,
                  float *__restrict__ returns, float *__restrict__ advantages) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float cur32 = last_values[i];   // buffer.py:90
    double cur64 = 0.0;
    bool wide = false;              // f64 rewards: the running value is f64 from the first iteration on
    int t = T - 1;
    while (t >= 0) {
        const int n = t + 1 < kUnroll ? t + 1 : kUnroll;
        RewT r[kUnroll];
        int32_t d[kUnroll];
        float v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            if (u < n) {
                const int64_t idx = (int64_t)(t - u) * N + i;
                r[u] = rewards[idx];
                d[u] = dones[idx];
                v[u] = values[idx];
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            if (u < n) {
                const int64_t idx = (int64_t)(t - u) * N + i;
                const float keep = __fmul_rn((float)(1 - d[u]), gamma);   // (1 - dones) * gamma: int32 tensor x python float
                float ret;
                if constexpr (sizeof(RewT) == 4) {
                    cur32 = __fadd_rn(r[u], __fmul_rn(keep, cur32));      // :94-97
                    ret = cur32;
                } else {
                    const double prod = wide ? __dmul_rn((double)keep, cur64) : (double)__fmul_rn(keep, cur32);
                    cur64 = __dadd_rn(r[u], prod);
                    wide = true;
                    ret = __double2float_rn(cur64);                       // :98 store into the f32 returns tensor
                }
                returns[idx] = ret;
                advantages[idx] = __fsub_rn(ret, v[u]);                   // :100
            }
        }
        t -= n;
    }
}

} // namespace

extern "C" int fe_returns_advantages(const void *rewards_dev, int32_t rewards_f64, const int32_t *dones_dev,
                                     const float *values_dev, const float *last_values_dev, int64_t num_envs,
                                     int32_t num_steps, double gamma, float *returns_dev, float *advantages_dev,
                                     void *stream) {
    if (!rewards_dev || !dones_dev || !values_dev || !last_values_dev || !returns_dev || !advantages_dev) return FE_EINVAL;
    if (num_envs <= 0 || num_steps <= 0) return FE_EINVAL;
    DeviceGuard guard(pointer_device(rewards_dev));
    if (guard.rc) return guard.rc;
    const unsigned blocks = (unsigned)((num_envs + 255) / 256);
    cudaStream_t q = (cudaStream_t)stream;
    return with_out_type(rewards_f64 != 0, [&](auto rew_type) {
        using RewT = decltype(rew_type);
        fe_returns_kernel<RewT><<<blocks, 256, 0, q>>>((const RewT *)rewards_dev, dones_dev, values_dev, last_values_dev,
                                                       num_envs, num_steps, (float)gamma, returns_dev, advantages_dev);
        return (int)cudaGetLastError();
    });
}
