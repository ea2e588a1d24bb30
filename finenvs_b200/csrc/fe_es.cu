// fe_es.cu — the ES rollout path around the env step (SURVEY.md §8f-2): the reference's ParallelMLP
// (finenvs/agents/networks/parallel_mlp.py) and EvoAgent.store (finenvs/agents/ES/evo_agent.py:96-112) as
// sm_100a kernels sized for millions of envs per GPU.
//
// The reference keeps one full perturbed copy of the network PER ENV (parallel_mlp.py:112-155: N x params f32,
// 2.3 TB at 4 Mi envs with the default net) and multiplies through it with batched matmuls.  Here:
//   * a mirrored PAIR (env p uses theta + sigma*eps_p, env p + N/2 uses theta - sigma*eps_p, :121-136) shares one
//     stored perturbation, kept as fp16 in a layout the forward kernel streams with 16-byte loads
//     (pairs x P_pad halves: 1.3 GB for 512 Ki envs x a 300-8-1 net, instead of 5 GB f32 per-env copies);
//   * eps is a pure function of (seed, generation, GLOBAL pair id, parameter index) — Philox4x32-10 + Box-Muller,
//     fe_es_perturb — so results do not depend on how pairs are sharded over GPUs;
//   * fe_es_forward evaluates both envs of a pair in one warp: the shared theta sits in shared memory, each lane
//     owns a strided slice of the layer's inputs, the four dot-product families (theta.x+, theta.x-, eps.x+,
//     eps.x-) are FMA chains in registers, and a butterfly reduce-scatter leaves one output per lane pair.
//     With LAZY observations (fe_step_lazy) the kernel gathers the env's window straight from the staged series:
//     the (N, W*5) observation tensor — 53 % of the step kernel's HBM traffic — is never written or read;
//   * fe_es_gradient is the fitness-weighted column sum of eps (parallel_mlp.py:176-218) in one pass over eps;
//   * fe_es_store keeps the per-env running returns and appends finished episodes to a device list with no host
//     synchronisation (evo_agent.py:96-112 does nonzero + cat + .item() per step).
// Packed parameter layout (theta f32, eps fp16, gradient f32): per layer l with (in, out): ceil(out/8) chunks of
// 8 outputs; chunk c holds rows j = 0..in (row `in` is the bias, its input is the constant 1), 8 values per row:
//     index(l, j, o) = off[l] + ((o / 8) * (in + 1) + j) * 8 + (o % 8).
#include "finenvs_b200.h"
#include "fe_common.cuh"

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace {

constexpr int kEsWarps = 8;
constexpr int kEsThreads = kEsWarps * 32;
constexpr uint64_t kEsKey = 0x9E3779B97F4A7C15ull; // separates the ES streams from the env's redraw streams
constexpr unsigned kAll = 0xFFFFFFFFu;

struct EsLayout {
    int L;
    int in[FE_ES_MAX_LAYERS], out[FE_ES_MAX_LAYERS];
    int64_t off[FE_ES_MAX_LAYERS + 1]; // off[L] = P_pad
    int max_dim;
};

bool make_layout(const FeEsNet *net, EsLayout &lay) {
    if (!net || net->num_layers < 1 || net->num_layers > FE_ES_MAX_LAYERS) return false;
    lay.L = net->num_layers;
    lay.off[0] = 0;
    lay.max_dim = 0;
    for (int l = 0; l <= lay.L; ++l) {
        if (net->dims[l] < 1) return false;
        if (net->dims[l] > lay.max_dim) lay.max_dim = net->dims[l];
    }
    for (int l = 0; l < lay.L; ++l) {
        lay.in[l] = net->dims[l];
        lay.out[l] = net->dims[l + 1];
        lay.off[l + 1] = lay.off[l] + (int64_t)((lay.out[l] + 7) / 8) * (lay.in[l] + 1) * 8;
    }
    return true;
}

// two standard normals from two 32-bit draws (Box-Muller on 24-bit uniforms, u1 in (0,1], u2 in [0,1))
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float &z0, float &z1) {
    const float u1 = (float)((a >> 8) + 1u) * 5.9604644775390625e-8f;
    const float u2 = (float)(b >> 8) * 5.9604644775390625e-8f;
    const float r = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    z0 = r * cs;
    z1 = r * sn;
}

// ------------------------------------------------------------------------------------------
// perturbations (parallel_mlp.py:112-155): eps[pair, q] ~ N(0, 1); the network uses theta +- sigma * eps
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
fe_es_perturb_kernel(const int64_t total8, const int64_t num_pairs, const int64_t pair_id_base, const uint64_t seed,
                     const uint64_t generation, __half *__restrict__ eps) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= num_pairs * total8) return;
    const int64_t pair = idx / total8, q8 = idx - pair * total8;
    float z[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        uint32_t r[4];
        philox4x32_10(seed ^ kEsKey, (uint64_t)(pair_id_base + pair), (generation << 32) | (uint64_t)(q8 * 2 + h), 1u, r);
        box_muller(r[0], r[1], z[4 * h + 0], z[4 * h + 1]);
        box_muller(r[2], r[3], z[4 * h + 2], z[4 * h + 3]);
    }
    __half2 h2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h2[i] = __floats2half2_rn(z[2 * i], z[2 * i + 1]);
    *reinterpret_cast<uint4 *>(eps + idx * 8) = *reinterpret_cast<const uint4 *>(h2);
}

__device__ __forceinline__ void halves8_to_floats(const uint4 v, float e[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        __half2 h;
        *reinterpret_cast<uint32_t *>(&h) = w[i];
        const float2 f = __half22float2(h);
        e[2 * i] = f.x;
        e[2 * i + 1] = f.y;
    }
}

// one level of the butterfly reduce-scatter: 2*kHalf live values -> kHalf (exchange with lane ^ 2*kHalf)
template <int kHalf> __device__ __forceinline__ void butterfly_step(float (&v)[16], const int lane) {
    const bool upper = (lane & (2 * kHalf)) != 0;
#pragma unroll
    for (int i = 0; i < kHalf; ++i) {
        const float keep = upper ? v[i + kHalf] : v[i];
        const float send = upper ? v[i] : v[i + kHalf];
        v[i] = keep + __shfl_xor_sync(kAll, send, 2 * kHalf);
    }
}

// ------------------------------------------------------------------------------------------
// forward (parallel_mlp.py:84-109): actions = tanh(... tanh(x W1' + b1') ...) with W' = W +- sigma * eps, per env
// ------------------------------------------------------------------------------------------
template <bool kLazy, bool kThetaSmem>
__global__ void __launch_bounds__(kEsThreads)
fe_es_forward_kernel(const EsLayout lay, const float *__restrict__ theta, const __half *__restrict__ eps, const float sigma,
                     const int64_t num_pairs, const int64_t num_eval, const float *__restrict__ obs,
                     const float *__restrict__ logret, const int64_t *__restrict__ row0, const float *__restrict__ posfeat,
                     const int W, const float noise_std, const uint64_t seed, const uint64_t step,
                     const int64_t env_id_base, float *__restrict__ actions) {
    extern __shared__ __align__(16) float es_smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t P = lay.off[lay.L];
    const int stride = (lay.max_dim + 1 + 3) & ~3; // one sign's activations (+ the constant-1 bias input)
    float *th = es_smem;
    float *bufA = es_smem + (kThetaSmem ? P : 0) + (size_t)warp * 4 * stride;
    float *bufB = bufA + 2 * stride;
    if (kThetaSmem) {
        for (int64_t q = tid; q < P; q += kEsThreads) th[q] = theta[q];
        __syncthreads();
    }
    const float *thbase = kThetaSmem ? th : theta;
    const int I = lay.in[0], OL = lay.out[lay.L - 1];
    const int64_t units = num_pairs + num_eval;
    for (int64_t unit = (int64_t)blockIdx.x * kEsWarps + warp; unit < units; unit += (int64_t)gridDim.x * kEsWarps) {
        const bool is_eval = unit >= num_pairs;
        const int64_t e0 = is_eval ? 2 * num_pairs + (unit - num_pairs) : unit; // :121-136 positives first,
        const int64_t e1 = is_eval ? e0 : unit + num_pairs;                      // negatives second, eval envs last
        const float sg = is_eval ? 0.0f : sigma;
        // ---- inputs of layer 0 into bufA: [0][.] = env e0, [1][.] = env e1
        if (kLazy) {
#pragma unroll
            for (int sgn = 0; sgn < 2; ++sgn) {
                const int64_t e = sgn ? e1 : e0;
                const float4 *src = reinterpret_cast<const float4 *>(logret) + row0[e];
                const float pfe = posfeat[e];
                float *x = bufA + sgn * stride;
                for (int r = lane; r < W; r += 32) {
                    const float4 v = __ldg(src + r);
                    x[r * 5 + 0] = v.x; x[r * 5 + 1] = v.y; x[r * 5 + 2] = v.z; x[r * 5 + 3] = v.w;
                    x[r * 5 + 4] = pfe;
                }
            }
        } else {
            for (int j = lane; j < I; j += 32) {
                bufA[j] = __ldg(obs + e0 * I + j);
                bufA[stride + j] = __ldg(obs + e1 * I + j);
            }
        }
        if (lane == 0) { bufA[I] = 1.0f; bufA[stride + I] = 1.0f; }
        __syncwarp();
        float *xin = bufA, *xout = bufB;
        for (int l = 0; l < lay.L; ++l) {
            const int in1 = lay.in[l] + 1, out = lay.out[l];
            const float *thl = thbase + lay.off[l];
            const __half *epl = eps + (is_eval ? 0 : unit * P) + lay.off[l];
            for (int c = 0; c * 8 < out; ++c) {
                float a0[8], a1[8], b0[8], b1[8];
#pragma unroll
                for (int o = 0; o < 8; ++o) { a0[o] = 0.0f; a1[o] = 0.0f; b0[o] = 0.0f; b1[o] = 0.0f; }
#pragma unroll 2
                for (int j = lane; j < in1; j += 32) {
                    const size_t q = ((size_t)c * in1 + j) * 8;
                    const float4 t03 = *reinterpret_cast<const float4 *>(thl + q);
                    const float4 t47 = *reinterpret_cast<const float4 *>(thl + q + 4);
                    const float t[8] = {t03.x, t03.y, t03.z, t03.w, t47.x, t47.y, t47.z, t47.w};
                    float e[8];
                    uint4 ev = make_uint4(0u, 0u, 0u, 0u);
                    if (!is_eval) ev = __ldg(reinterpret_cast<const uint4 *>(epl + q));
                    halves8_to_floats(ev, e);
                    const float xp = xin[j], xm = xin[stride + j];
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        a0[o] = fmaf(t[o], xp, a0[o]);
                        a1[o] = fmaf(t[o], xm, a1[o]);
                        b0[o] = fmaf(e[o], xp, b0[o]);
                        b1[o] = fmaf(e[o], xm, b1[o]);
                    }
                }
                float v[16];
#pragma unroll
                for (int o = 0; o < 8; ++o) {
                    v[o] = fmaf(sg, b0[o], a0[o]);       // (theta + sigma eps) . x+
                    v[8 + o] = fmaf(-sg, b1[o], a1[o]);  // (theta - sigma eps) . x-
                }
                // butterfly reduce-scatter: 16 partial sums x 32 lanes -> lanes 2m, 2m+1 hold the total of value m
                butterfly_step<8>(v, lane);
                butterfly_step<4>(v, lane);
                butterfly_step<2>(v, lane);
                butterfly_step<1>(v, lane);
                v[0] += __shfl_xor_sync(kAll, v[0], 1);
                const int m = lane >> 1, o = c * 8 + (m & 7);
                if ((lane & 1) == 0 && o < out) xout[(m >> 3) * stride + o] = tanhf(v[0]);
            }
            if (lane == 0) { xout[out] = 1.0f; xout[stride + out] = 1.0f; }
            __syncwarp();
            float *tmp = xin; xin = xout; xout = tmp;
        }
        // ---- actions (+ exploration noise, parallel_mlp.py:104-109: none for the eval envs; with no eval envs the
        //      reference's `action_noise[-0:, :] = 0` zeroes ALL of it)
        for (int f = lane; f < 2 * OL; f += 32) {
            const int sgn = f >= OL, o = f - sgn * OL;
            if (sgn && is_eval) continue;
            const int64_t e = sgn ? e1 : e0;
            float a = xin[sgn * stride + o];
            if (noise_std > 0.0f && !is_eval && num_eval > 0) {
                uint32_t r[4]; // one Philox block = four normals: actions 4b .. 4b+3 of this (env, step)
                philox4x32_10(seed ^ kEsKey, (uint64_t)(env_id_base + e), step | ((uint64_t)(o >> 2) << 48), 0u, r);
                float z[4];
                box_muller(r[0], r[1], z[0], z[1]);
                box_muller(r[2], r[3], z[2], z[3]);
                a = fmaf(noise_std, (o & 2) ? ((o & 1) ? z[3] : z[2]) : ((o & 1) ? z[1] : z[0]), a);
            }
            actions[e * OL + o] = a;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// forward, fast path: first layer 5*R inputs (R <= 63 window rows x 5 features) -> <= 8 outputs — the shape of the ES
// population rollout on the trading env (BASELINE config 5: 300-8-1).  ncu on the generic kernel above
// (profiles/r01_es_forward_generic_ncu.txt): 1.08 ms per 512 Ki envs, 1.65 TB/s, stalled on its own eps loads
// (long scoreboard 10.6 of 12.7 stall cycles per issue, <= 1 KB in flight per warp).  Here
//   * every warp owns a ring of kFastStages shared-memory stages; a unit's perturbation (P_pad fp16, contiguous) and
//     its two observation windows arrive by 1-D bulk async copies (cp.async.bulk, UBLKCP) issued kFastStages-1 units
//     ahead and completing on the stage's mbarrier: ~14 KB in flight per warp, no register staging;
//   * lane r owns window rows r and r+32, i.e. inputs 5r..5r+4: the first layer's theta rows of a lane never change,
//     so they live in registers for the whole kernel (80 floats) — shared memory only feeds eps and x;
//   * the lazy window (W x 16 B straight from the staged series) is consumed as it lies: the 4->5 interleave with the
//     position feature never happens anywhere.
// The remaining (tiny) layers read theta from shared memory and eps from the stage.  Dense observations take the
// same path (their rows are 5 consecutive floats), with the same FMA order, so lazy == dense bit for bit.
// ------------------------------------------------------------------------------------------
#ifndef FE_ES_FAST_WARPS
#define FE_ES_FAST_WARPS 12
#endif
#ifndef FE_ES_FAST_STAGES
#define FE_ES_FAST_STAGES 2
#endif
constexpr int kFastWarps = FE_ES_FAST_WARPS;
constexpr int kFastThreads = kFastWarps * 32;
constexpr int kFastStages = FE_ES_FAST_STAGES;

struct FastShape {
    int rows;        // R: window rows (in[0] == 5 * R)
    int x_bytes;     // one env's layer-0 inputs as staged: lazy R*16, dense R*20
    int eps_bytes;   // P_pad * 2
    int stage_bytes; // eps + 2 x + pf pair, rounded to 128
    int act_stride;  // floats per sign in the activation buffers of layers >= 1
    int tail_in_regs; // exactly two layers and <= 8 actions: the second layer runs out of the butterfly's registers
    int theta_bytes; // P_pad * 4 rounded to 128
};
__host__ __device__ inline size_t fast_smem_bytes(const FastShape &f) {
    return 256 + (size_t)f.theta_bytes + (size_t)kFastWarps * ((size_t)kFastStages * f.stage_bytes + (size_t)4 * f.act_stride * 4);
}

template <bool kLazy>
__global__ void __launch_bounds__(kFastThreads, 1)
fe_es_forward_fast_kernel(const EsLayout lay, const FastShape fs, const float *__restrict__ theta,
                          const __half *__restrict__ eps, const float sigma, const int64_t num_pairs, const int64_t num_eval,
                          const float *__restrict__ obs, const float *__restrict__ logret, const int64_t *__restrict__ row0,
                          const float *__restrict__ posfeat, const float noise_std, const uint64_t seed, const uint64_t step,
                          const int64_t env_id_base, float *__restrict__ actions) {
    extern __shared__ __align__(128) unsigned char fsm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t P = lay.off[lay.L];
    const int R = fs.rows, I = lay.in[0], out0 = lay.out[0], OL = lay.out[lay.L - 1];
    float *th = reinterpret_cast<float *>(fsm + 256);
    unsigned char *ring = fsm + 256 + fs.theta_bytes + (size_t)warp * kFastStages * fs.stage_bytes;
    const int stride = fs.act_stride;
    float *bufA = reinterpret_cast<float *>(fsm + 256 + fs.theta_bytes + (size_t)kFastWarps * kFastStages * fs.stage_bytes) +
                  (size_t)warp * 4 * stride;
    float *bufB = bufA + 2 * stride;
    const uint32_t bar0 = smem_u32(fsm) + (uint32_t)warp * kFastStages * 8u;
    for (int64_t q = tid; q < P; q += kFastThreads) th[q] = theta[q];
    if (lane == 0)
        for (int s = 0; s < kFastStages; ++s) mbar_init(bar0 + 8u * s, 1);
    mbar_fence_init();
    __syncthreads();

    // lane-stationary first-layer theta: window rows lane and lane + 32 (inputs 5r .. 5r+4, packed index j*8 + o).
    // "Row" R is the bias: its first input is the constant 1 (packed row j = I), the other four do not exist.
    float t0[2][5][8];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
        const int r = lane + 32 * sl;
#pragma unroll
        for (int i = 0; i < 5; ++i)
#pragma unroll
            for (int o = 0; o < 8; ++o) t0[sl][i][o] = (r < R || (r == R && i == 0)) ? th[(size_t)(5 * r + i) * 8 + o] : 0.0f;
    }

    const int64_t units = num_pairs + num_eval;
    const int64_t gw = (int64_t)blockIdx.x * kFastWarps + warp, nw = (int64_t)gridDim.x * kFastWarps;
    const int nloc = gw < units ? (int)((units - gw + nw - 1) / nw) : 0;
    auto env_of = [&](int64_t u, int sgn) -> int64_t { // :121-136 positives first, negatives second, eval envs last
        if (u >= num_pairs) return 2 * num_pairs + (u - num_pairs);
        return sgn ? u + num_pairs : u;
    };
    // registers of lanes 0/1 describing the NEXT unit to issue (loaded one iteration early: no stall on row0)
    int64_t n_src = 0;
    float n_pf = 0.0f;
    auto preload = [&](int k) {
        if (k < nloc && lane < 2) {
            const int64_t e = env_of(gw + (int64_t)k * nw, lane);
            if (kLazy) { n_src = __ldg(row0 + e); n_pf = __ldg(posfeat + e); }
            else n_src = e;
        }
    };
    int st_i = 0; // stage the next issue goes to
    auto issue = [&](int k) {
        if (k >= nloc) return;
        const int64_t u = gw + (int64_t)k * nw;
        const bool is_eval = u >= num_pairs;
        unsigned char *stage = ring + (size_t)st_i * fs.stage_bytes;
        const uint32_t bar = bar0 + 8u * (uint32_t)st_i;
        st_i = st_i + 1 == kFastStages ? 0 : st_i + 1;
        if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)((is_eval ? 0 : fs.eps_bytes) + 2 * fs.x_bytes));
        __syncwarp();
        if (lane == 0 && !is_eval) bulk_load(smem_u32(stage), eps + u * P, (uint32_t)fs.eps_bytes, bar);
        if (lane < 2) {
            const void *src = kLazy ? (const void *)(reinterpret_cast<const float4 *>(logret) + n_src)
                                    : (const void *)(obs + n_src * I);
            bulk_load(smem_u32(stage + fs.eps_bytes + lane * fs.x_bytes), src, (uint32_t)fs.x_bytes, bar);
            if (kLazy) reinterpret_cast<float *>(stage + fs.eps_bytes + 2 * fs.x_bytes)[lane] = n_pf;
        }
    };
    for (int k = 0; k < kFastStages - 1; ++k) { preload(k); issue(k); }
    preload(kFastStages - 1);

    const int m = lane >> 1, om = m & 7;                 // after the butterfly: lanes 2m, 2m+1 hold value m = sign*8 + output
    const int off1 = (int)lay.off[1];
    int st_c = 0;
    uint32_t ph_c = 0;
    for (int k = 0; k < nloc; ++k) {
        issue(k + kFastStages - 1); // into the stage consumed in iteration k - 1
        preload(k + kFastStages);
        const int64_t unit = gw + (int64_t)k * nw;
        const bool is_eval = unit >= num_pairs;
        const float sg = is_eval ? 0.0f : sigma;
        const unsigned char *stage = ring + (size_t)st_c * fs.stage_bytes;
        mbar_wait(bar0 + 8u * (uint32_t)st_c, ph_c);
        if (++st_c == kFastStages) { st_c = 0; ph_c ^= 1u; }
        __syncwarp();
        const unsigned char *xs = stage + fs.eps_bytes;
        // ---- layer 0
        float a0[8], a1[8], b0[8], b1[8];
#pragma unroll
        for (int o = 0; o < 8; ++o) { a0[o] = 0.0f; a1[o] = 0.0f; b0[o] = 0.0f; b1[o] = 0.0f; }
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
            const int r = lane + 32 * sl;
            if (r <= R) {
                const bool row = r < R;
                float xp[5], xm[5];
                if (kLazy) {
                    const float4 p4 = *reinterpret_cast<const float4 *>(xs + (size_t)r * 16);
                    const float4 m4 = *reinterpret_cast<const float4 *>(xs + fs.x_bytes + (size_t)r * 16);
                    const float2 pf = *reinterpret_cast<const float2 *>(xs + 2 * fs.x_bytes);
                    xp[0] = p4.x; xp[1] = p4.y; xp[2] = p4.z; xp[3] = p4.w; xp[4] = pf.x;
                    xm[0] = m4.x; xm[1] = m4.y; xm[2] = m4.z; xm[3] = m4.w; xm[4] = pf.y;
                } else {
                    const float *pp = reinterpret_cast<const float *>(xs) + 5 * r;
                    const float *pm = reinterpret_cast<const float *>(xs + fs.x_bytes) + 5 * r;
#pragma unroll
                    for (int i = 0; i < 5; ++i) { xp[i] = pp[i]; xm[i] = pm[i]; }
                }
#pragma unroll
                for (int i = 0; i < 5; ++i) { // the bias "row": (1, 0, 0, 0, 0) whatever lies behind the window
                    xp[i] = row ? xp[i] : (i == 0 ? 1.0f : 0.0f);
                    xm[i] = row ? xm[i] : (i == 0 ? 1.0f : 0.0f);
                }
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    float e[8];
                    uint4 ev = make_uint4(0u, 0u, 0u, 0u);
                    if (!is_eval && (row || i == 0)) ev = *reinterpret_cast<const uint4 *>(stage + (size_t)(5 * r + i) * 16);
                    halves8_to_floats(ev, e);
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        a0[o] = fmaf(t0[sl][i][o], xp[i], a0[o]);
                        a1[o] = fmaf(t0[sl][i][o], xm[i], a1[o]);
                        b0[o] = fmaf(e[o], xp[i], b0[o]);
                        b1[o] = fmaf(e[o], xm[i], b1[o]);
                    }
                }
            }
        }
        float v[16];
#pragma unroll
        for (int o = 0; o < 8; ++o) {
            v[o] = fmaf(sg, b0[o], a0[o]);       // (theta + sigma eps) . x+
            v[8 + o] = fmaf(-sg, b1[o], a1[o]);  // (theta - sigma eps) . x-
        }
        butterfly_step<8>(v, lane);
        butterfly_step<4>(v, lane);
        butterfly_step<2>(v, lane);
        butterfly_step<1>(v, lane);
        v[0] += __shfl_xor_sync(kAll, v[0], 1);
        const int64_t e0 = env_of(unit, 0), e1 = env_of(unit, 1);
        if (fs.tail_in_regs) {
            // ---- second (= last) layer with <= 8 outputs, straight from the butterfly's registers: lane pair m holds
            // hidden unit om of sign m>>3 (hidden "unit" out0 is the constant 1 feeding the bias row); the dot product
            // over the 8 lane pairs of one sign is three xor-shuffles per output
            const float h = om < out0 ? tanhf(v[0]) : (om == out0 ? 1.0f : 0.0f);
            const float sgs = (m >> 3) ? -sg : sg;
            float t[8], e[8];
            {
                float4 t03 = make_float4(0.f, 0.f, 0.f, 0.f), t47 = t03;
                uint4 ev = make_uint4(0u, 0u, 0u, 0u);
                if (om <= out0) {
                    t03 = *reinterpret_cast<const float4 *>(th + off1 + om * 8);
                    t47 = *reinterpret_cast<const float4 *>(th + off1 + om * 8 + 4);
                    if (!is_eval) ev = *reinterpret_cast<const uint4 *>(stage + (size_t)(off1 + om * 8) * 2);
                }
                t[0] = t03.x; t[1] = t03.y; t[2] = t03.z; t[3] = t03.w; t[4] = t47.x; t[5] = t47.y; t[6] = t47.z; t[7] = t47.w;
                halves8_to_floats(ev, e);
            }
            float bias_t = 0.0f, bias_e = 0.0f; // out0 == 8: the bias row has no lane pair of its own
#pragma unroll
            for (int o2 = 0; o2 < 8; ++o2) {
                if (o2 < OL) {
                    float pacc = fmaf(sgs, e[o2], t[o2]) * h;
                    pacc += __shfl_xor_sync(kAll, pacc, 2);
                    pacc += __shfl_xor_sync(kAll, pacc, 4);
                    pacc += __shfl_xor_sync(kAll, pacc, 8);
                    if (out0 == 8) {
                        bias_t = th[off1 + 64 + o2];
                        bias_e = is_eval ? 0.0f : __half2float(*reinterpret_cast<const __half *>(stage + (size_t)(off1 + 64 + o2) * 2));
                        pacc += fmaf(sgs, bias_e, bias_t);
                    }
                    float a = tanhf(pacc);
                    const bool writer = (lane & 15) == 0 && !(lane == 16 && is_eval);
                    if (writer) {
                        const int64_t e = lane ? e1 : e0;
                        if (noise_std > 0.0f && !is_eval && num_eval > 0) {
                            uint32_t rr[4];
                            philox4x32_10(seed ^ kEsKey, (uint64_t)(env_id_base + e), step | ((uint64_t)(o2 >> 2) << 48), 0u, rr);
                            float z[4];
                            box_muller(rr[0], rr[1], z[0], z[1]);
                            box_muller(rr[2], rr[3], z[2], z[3]);
                            a = fmaf(noise_std, (o2 & 2) ? ((o2 & 1) ? z[3] : z[2]) : ((o2 & 1) ? z[1] : z[0]), a);
                        }
                        actions[e * OL + o2] = a;
                    }
                }
            }
            __syncwarp(); // every lane is done with this stage
            continue;
        }
        {
            if ((lane & 1) == 0 && om < out0) bufA[(m >> 3) * stride + om] = tanhf(v[0]);
            if (lane == 0) { bufA[out0] = 1.0f; bufA[stride + out0] = 1.0f; }
        }
        __syncwarp();
        // ---- layers 1 .. L-1 (general shapes): theta from shared memory, eps from the stage
        float *xin = bufA, *xout = bufB;
        for (int l = 1; l < lay.L; ++l) {
            const int in1 = lay.in[l] + 1, out = lay.out[l];
            const float *thl = th + lay.off[l];
            const unsigned char *epl = stage + (size_t)lay.off[l] * 2;
            for (int c = 0; c * 8 < out; ++c) {
                float c0[8], c1[8], d0[8], d1[8];
#pragma unroll
                for (int o = 0; o < 8; ++o) { c0[o] = 0.0f; c1[o] = 0.0f; d0[o] = 0.0f; d1[o] = 0.0f; }
                for (int j = lane; j < in1; j += 32) {
                    const size_t q = ((size_t)c * in1 + j) * 8;
                    const float4 t03 = *reinterpret_cast<const float4 *>(thl + q);
                    const float4 t47 = *reinterpret_cast<const float4 *>(thl + q + 4);
                    const float t[8] = {t03.x, t03.y, t03.z, t03.w, t47.x, t47.y, t47.z, t47.w};
                    float e[8];
                    uint4 ev = make_uint4(0u, 0u, 0u, 0u);
                    if (!is_eval) ev = *reinterpret_cast<const uint4 *>(epl + q * 2);
                    halves8_to_floats(ev, e);
                    const float xp = xin[j], xm = xin[stride + j];
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        c0[o] = fmaf(t[o], xp, c0[o]);
                        c1[o] = fmaf(t[o], xm, c1[o]);
                        d0[o] = fmaf(e[o], xp, d0[o]);
                        d1[o] = fmaf(e[o], xm, d1[o]);
                    }
                }
                float w[16];
#pragma unroll
                for (int o = 0; o < 8; ++o) {
                    w[o] = fmaf(sg, d0[o], c0[o]);
                    w[8 + o] = fmaf(-sg, d1[o], c1[o]);
                }
                butterfly_step<8>(w, lane);
                butterfly_step<4>(w, lane);
                butterfly_step<2>(w, lane);
                butterfly_step<1>(w, lane);
                w[0] += __shfl_xor_sync(kAll, w[0], 1);
                const int o = c * 8 + om;
                if ((lane & 1) == 0 && o < out) xout[(m >> 3) * stride + o] = tanhf(w[0]);
            }
            if (lane == 0) { xout[out] = 1.0f; xout[stride + out] = 1.0f; }
            __syncwarp();
            float *tmp = xin; xin = xout; xout = tmp;
        }
        // ---- actions (+ exploration noise; same semantics and streams as the generic kernel)
        for (int f = lane; f < 2 * OL; f += 32) {
            const int sgn = f >= OL, o = f - sgn * OL;
            if (sgn && is_eval) continue;
            const int64_t e = sgn ? e1 : e0;
            float a = xin[sgn * stride + o];
            if (noise_std > 0.0f && !is_eval && num_eval > 0) {
                uint32_t r[4];
                philox4x32_10(seed ^ kEsKey, (uint64_t)(env_id_base + e), step | ((uint64_t)(o >> 2) << 48), 0u, r);
                float z[4];
                box_muller(r[0], r[1], z[0], z[1]);
                box_muller(r[2], r[3], z[2], z[3]);
                a = fmaf(noise_std, (o & 2) ? ((o & 1) ? z[3] : z[2]) : ((o & 1) ? z[1] : z[0]), a);
            }
            actions[e * OL + o] = a;
        }
        __syncwarp(); // every lane is done with this stage and the activation buffers
    }
}

// ------------------------------------------------------------------------------------------
// forward, streaming path: any tanh MLP whose layers have <= 319 inputs (e.g. the reference's default 256-256 hidden
// layers, evo_agent.py:16).  The generic kernel above reads eps and theta with plain loads, one 8-output chunk of one
// pair at a time: 5.7 ms per step for 64 Ki envs x a 300-256-256-1 policy (9.5 GB of eps, 1.67 TB/s).  Here a warp
// owns U pairs at a time and walks the network chunk by chunk (8 outputs x (in+1) rows):
//   * the chunk's theta rows of a lane (<= 10 rows x 8 outputs) are loaded ONCE into registers and reused for the
//     warp's U pairs (theta traffic from L2 / L1 drops by U and leaves the shared-memory pipe to eps and x);
//   * a pair's eps chunk ((in+1) x 16 bytes, contiguous in the packed layout) arrives by one bulk async copy into the
//     warp's ring, issued kStStages-1 (pair, chunk) steps ahead, completing on the stage's mbarrier;
//   * activations of the U pairs live in shared memory as (x+, x-) float2 per input.
// ------------------------------------------------------------------------------------------
#ifndef FE_ES_ST_WARPS
#define FE_ES_ST_WARPS 12
#endif
#ifndef FE_ES_ST_STAGES
#define FE_ES_ST_STAGES 2
#endif
#ifndef FE_ES_ST_MAXU
#define FE_ES_ST_MAXU 4
#endif
constexpr int kStWarps = FE_ES_ST_WARPS;
constexpr int kStThreads = kStWarps * 32;
constexpr int kStStages = FE_ES_ST_STAGES;
constexpr int kStRows = 10;   // rows per lane: in + 1 <= 320
constexpr int kStMaxU = FE_ES_ST_MAXU;

struct StreamShape {
    int U;            // pairs per warp per group
    int stage_bytes;  // largest eps chunk, rounded to 128
    int strideA, strideB; // float2 entries per pair in the two activation buffers (inputs of even / odd layers)
    int chunks[FE_ES_MAX_LAYERS + 1]; // cumulative chunk counts: chunks[l] = chunks of layers < l
};
__host__ __device__ inline size_t stream_smem_bytes(const StreamShape &f) {
    return 256 + (size_t)kStWarps * ((size_t)kStStages * f.stage_bytes + (size_t)f.U * (f.strideA + f.strideB) * 8);
}

template <bool kLazy>
__global__ void __launch_bounds__(kStThreads, 1)
fe_es_forward_stream_kernel(const EsLayout lay, const StreamShape fs, const float *__restrict__ theta,
                            const __half *__restrict__ eps, const float sigma, const int64_t num_pairs, const int64_t num_eval,
                            const float *__restrict__ obs, const float *__restrict__ logret, const int64_t *__restrict__ row0,
                            const float *__restrict__ posfeat, const int W, const float noise_std, const uint64_t seed,
                            const uint64_t step, const int64_t env_id_base, float *__restrict__ actions) {
    extern __shared__ __align__(128) unsigned char ssm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t P = lay.off[lay.L];
    const int U = fs.U, I = lay.in[0], OL = lay.out[lay.L - 1];
    const size_t warp_bytes = (size_t)kStStages * fs.stage_bytes + (size_t)U * (fs.strideA + fs.strideB) * 8;
    unsigned char *ring = ssm + 256 + (size_t)warp * warp_bytes;
    float2 *actA = reinterpret_cast<float2 *>(ring + (size_t)kStStages * fs.stage_bytes); // [U][strideA]
    float2 *actB = actA + (size_t)U * fs.strideA;                                         // [U][strideB]
    const uint32_t bar0 = smem_u32(ssm) + (uint32_t)warp * kStStages * 8u;
    if (lane == 0)
        for (int s = 0; s < kStStages; ++s) mbar_init(bar0 + 8u * s, 1);
    mbar_fence_init();
    __syncthreads();

    const int64_t units = num_pairs + num_eval;
    const int m = lane >> 1, om = m & 7;
    auto env_of = [&](int64_t u, int sgn) -> int64_t { // :121-136 positives first, negatives second, eval envs last
        if (u >= num_pairs) return 2 * num_pairs + (u - num_pairs);
        return sgn ? u + num_pairs : u;
    };
    uint32_t gi = 0, gc = 0; // steps issued / consumed by this warp since the kernel started (stage = g % S)
    for (int64_t first = ((int64_t)blockIdx.x * kStWarps + warp) * U; first < units; first += (int64_t)gridDim.x * kStWarps * U) {
        const int nu = (int)(units - first < U ? units - first : U);
        // the steps of a group in consumption order: for every layer, for every chunk, for every pair of the warp;
        // (il, ic, iu) walks that order one step ahead of the consumer by kStStages - 1 steps
        int il = 0, ic = 0, iu = 0;
        auto issue = [&]() {
            if (il >= lay.L) return;
            const int in1 = lay.in[il] + 1;
            const int64_t unit = first + iu;
            const uint32_t bar = bar0 + 8u * (gi % kStStages);
            unsigned char *stage = ring + (size_t)(gi % kStStages) * fs.stage_bytes;
            ++gi;
            if (lane == 0) {
                if (unit < num_pairs) {
                    mbar_arrive_expect_tx(bar, (uint32_t)in1 * 16u);
                    bulk_load(smem_u32(stage), eps + unit * P + lay.off[il] + (int64_t)ic * in1 * 8, (uint32_t)in1 * 16u, bar);
                } else {
                    mbar_arrive(bar); // evaluation env: no perturbation to fetch
                }
            }
            if (++iu == nu) {
                iu = 0;
                if (++ic * 8 >= lay.out[il]) { ic = 0; ++il; }
            }
        };
        for (int k = 0; k < kStStages - 1; ++k) issue();
        // ---- inputs of layer 0: actA[u][j] = (x of the + env, x of the - env), entry I = the constant 1 of the bias row
        for (int u = 0; u < nu; ++u) {
            const int64_t unit = first + u, e0 = env_of(unit, 0), e1 = env_of(unit, 1);
            float2 *x = actA + (size_t)u * fs.strideA;
            if (kLazy) {
                const float4 *s0 = reinterpret_cast<const float4 *>(logret) + row0[e0];
                const float4 *s1 = reinterpret_cast<const float4 *>(logret) + row0[e1];
                const float p0 = posfeat[e0], p1 = posfeat[e1];
                for (int r = lane; r < W; r += 32) {
                    const float4 a = __ldg(s0 + r), b = __ldg(s1 + r);
                    x[r * 5 + 0] = make_float2(a.x, b.x); x[r * 5 + 1] = make_float2(a.y, b.y);
                    x[r * 5 + 2] = make_float2(a.z, b.z); x[r * 5 + 3] = make_float2(a.w, b.w);
                    x[r * 5 + 4] = make_float2(p0, p1);
                }
            } else {
                for (int j = lane; j < I; j += 32) x[j] = make_float2(__ldg(obs + e0 * I + j), __ldg(obs + e1 * I + j));
            }
            if (lane == 0) x[I] = make_float2(1.0f, 1.0f);
        }
        __syncwarp();
        float2 *xin = actA, *xout = actB;
        int sin_stride = fs.strideA, sout_stride = fs.strideB;
        for (int l = 0; l < lay.L; ++l) {
            const int in1 = lay.in[l] + 1, out = lay.out[l];
            for (int c = 0; c * 8 < out; ++c) {
                // the chunk's theta rows of this lane, reused for the warp's nu pairs
                float t[kStRows][8];
                const float *thc = theta + lay.off[l] + (int64_t)c * in1 * 8;
#pragma unroll
                for (int r = 0; r < kStRows; ++r) {
                    const int j = lane + 32 * r;
                    float4 t03 = make_float4(0.f, 0.f, 0.f, 0.f), t47 = t03;
                    if (j < in1) {
                        t03 = __ldg(reinterpret_cast<const float4 *>(thc + (size_t)j * 8));
                        t47 = __ldg(reinterpret_cast<const float4 *>(thc + (size_t)j * 8 + 4));
                    }
                    t[r][0] = t03.x; t[r][1] = t03.y; t[r][2] = t03.z; t[r][3] = t03.w;
                    t[r][4] = t47.x; t[r][5] = t47.y; t[r][6] = t47.z; t[r][7] = t47.w;
                }
                for (int u = 0; u < nu; ++u) {
                    issue();
                    const int64_t unit = first + u;
                    const bool is_eval = unit >= num_pairs;
                    const float sg = is_eval ? 0.0f : sigma;
                    const unsigned char *stage = ring + (size_t)(gc % kStStages) * fs.stage_bytes;
                    mbar_wait(bar0 + 8u * (gc % kStStages), (gc / kStStages) & 1u);
                    ++gc;
                    const float2 *x = xin + (size_t)u * sin_stride;
                    float a0[8], a1[8], b0[8], b1[8];
#pragma unroll
                    for (int o = 0; o < 8; ++o) { a0[o] = 0.0f; a1[o] = 0.0f; b0[o] = 0.0f; b1[o] = 0.0f; }
#pragma unroll
                    for (int r = 0; r < kStRows; ++r) {
                        const int j = lane + 32 * r;
                        if (j < in1) {
                            float e[8];
                            uint4 ev = make_uint4(0u, 0u, 0u, 0u);
                            if (!is_eval) ev = *reinterpret_cast<const uint4 *>(stage + (size_t)j * 16);
                            halves8_to_floats(ev, e);
                            const float2 xv = x[j];
#pragma unroll
                            for (int o = 0; o < 8; ++o) {
                                a0[o] = fmaf(t[r][o], xv.x, a0[o]);
                                a1[o] = fmaf(t[r][o], xv.y, a1[o]);
                                b0[o] = fmaf(e[o], xv.x, b0[o]);
                                b1[o] = fmaf(e[o], xv.y, b1[o]);
                            }
                        }
                    }
                    float v[16];
#pragma unroll
                    for (int o = 0; o < 8; ++o) {
                        v[o] = fmaf(sg, b0[o], a0[o]);       // (theta + sigma eps) . x+
                        v[8 + o] = fmaf(-sg, b1[o], a1[o]);  // (theta - sigma eps) . x-
                    }
                    butterfly_step<8>(v, lane);
                    butterfly_step<4>(v, lane);
                    butterfly_step<2>(v, lane);
                    butterfly_step<1>(v, lane);
                    v[0] += __shfl_xor_sync(kAll, v[0], 1);
                    const int o = c * 8 + om;
                    if ((lane & 1) == 0 && o < out) {
                        float *dst = reinterpret_cast<float *>(xout + (size_t)u * sout_stride + o) + (m >> 3);
                        *dst = tanhf(v[0]);
                    }
                    __syncwarp(); // every lane is done with this eps stage
                }
            }
            if (lane < nu) xout[(size_t)lane * sout_stride + out] = make_float2(1.0f, 1.0f);
            __syncwarp();
            float2 *tp = xin; xin = xout; xout = tp;
            const int ts = sin_stride; sin_stride = sout_stride; sout_stride = ts;
        }
        // ---- actions (+ exploration noise; same semantics and streams as the generic kernel)
        for (int u = 0; u < nu; ++u) {
            const int64_t unit = first + u;
            const bool is_eval = unit >= num_pairs;
            for (int f = lane; f < 2 * OL; f += 32) {
                const int sgn = f >= OL, o = f - sgn * OL;
                if (sgn && is_eval) continue;
                const int64_t e = env_of(unit, sgn);
                const float2 xv = xin[(size_t)u * sin_stride + o];
                float a = sgn ? xv.y : xv.x;
                if (noise_std > 0.0f && !is_eval && num_eval > 0) {
                    uint32_t r[4];
                    philox4x32_10(seed ^ kEsKey, (uint64_t)(env_id_base + e), step | ((uint64_t)(o >> 2) << 48), 0u, r);
                    float z[4];
                    box_muller(r[0], r[1], z[0], z[1]);
                    box_muller(r[2], r[3], z[2], z[3]);
                    a = fmaf(noise_std, (o & 2) ? ((o & 1) ? z[3] : z[2]) : ((o & 1) ? z[1] : z[0]), a);
                }
                actions[e * OL + o] = a;
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// gradient (parallel_mlp.py:176-218): grad[q] = sum over pairs of w[pair] * eps[pair, q], w = f+ - f-.
// Deterministic two-stage sum: slabs of pairs -> partial[slab, q]; then the slabs in order.
// ------------------------------------------------------------------------------------------
constexpr int kGradThreads = 128;
constexpr int kGradSlab = 512; // pairs per block

__global__ void __launch_bounds__(kGradThreads)
fe_es_grad_partial_kernel(const int64_t total8, const int64_t num_pairs, const __half *__restrict__ eps,
                          const float *__restrict__ w, float *__restrict__ partial) {
    const int64_t q8 = (int64_t)blockIdx.x * kGradThreads + threadIdx.x;
    if (q8 >= total8) return;
    const int64_t p0 = (int64_t)blockIdx.y * kGradSlab;
    const int64_t p1 = p0 + kGradSlab < num_pairs ? p0 + kGradSlab : num_pairs;
    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = 0.0f;
#pragma unroll 4
    for (int64_t p = p0; p < p1; ++p) {
        float e[8];
        halves8_to_floats(__ldg(reinterpret_cast<const uint4 *>(eps + (p * total8 + q8) * 8)), e);
        const float wp = __ldg(w + p);
#pragma unroll
        for (int o = 0; o < 8; ++o) acc[o] = fmaf(wp, e[o], acc[o]);
    }
    float4 *dst = reinterpret_cast<float4 *>(partial + ((int64_t)blockIdx.y * total8 + q8) * 8);
    dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

__global__ void __launch_bounds__(256)
fe_es_grad_reduce_kernel(const int64_t total, const int64_t slabs, const float *__restrict__ partial, float *__restrict__ grad) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= total) return;
    float s = 0.0f;
    for (int64_t y = 0; y < slabs; ++y) s += partial[y * total + q];
    grad[q] = s;
}

// ------------------------------------------------------------------------------------------
// episode accounting (evo_agent.py:90-112): running return / step count per env, finished episodes appended to a
// device list (key = step ordinal * total_envs + global env id, so sorting by key restores the reference's order)
// ------------------------------------------------------------------------------------------
template <typename RewT>
__global__ void __launch_bounds__(256)
fe_es_store_kernel(const RewT *__restrict__ rewards, const int32_t *__restrict__ dones, const int64_t N,
                   const int64_t env_id_base, const int64_t total_envs, const uint64_t step_ordinal,
                   float *__restrict__ cur_returns, float *__restrict__ cur_steps, const int64_t capacity,
                   unsigned long long *__restrict__ counters, int64_t *__restrict__ fin_key, int64_t *__restrict__ fin_env,
                   float *__restrict__ fin_ret) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int done = 0;
    float ret = 0.0f, steps = 0.0f;
    if (i < N) {
        // :99 current_returns (f32) += rewards: computed in the promoted dtype, rounded once
        if constexpr (sizeof(RewT) == 8) ret = __double2float_rn(__dadd_rn((double)cur_returns[i], rewards[i]));
        else ret = __fadd_rn(cur_returns[i], rewards[i]);
        steps = cur_steps[i] + 1.0f; // :93 current_timesteps += 1 (EvoAgent.step)
        done = dones[i] != 0;
        cur_returns[i] = done ? 0.0f : ret;   // :110-111
        cur_steps[i] = done ? 0.0f : steps;
    }
    // one counter update per warp; slots inside the warp in lane (= env) order
    const unsigned ballot = __ballot_sync(kAll, done);
    if (ballot == 0) return;
    float wsteps = done ? steps : 0.0f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wsteps += __shfl_xor_sync(kAll, wsteps, o);
    unsigned long long base = 0;
    if (lane == 0) {
        base = atomicAdd(&counters[0], (unsigned long long)__popc(ballot));
        atomicAdd(&counters[1], (unsigned long long)wsteps); // :103-104 total_timesteps
    }
    base = __shfl_sync(kAll, base, 0);
    if (done) {
        const int64_t slot = (int64_t)base + __popc(ballot & ((1u << lane) - 1u));
        if (slot < capacity) {
            fin_key[slot] = (int64_t)step_ordinal * total_envs + env_id_base + i;
            fin_env[slot] = i;
            fin_ret[slot] = ret;
        }
    }
}

// ------------------------------------------------------------------------------------------
// forward routing: which of the three kernels runs a network, and its launch shape.  A host function of the layout
// alone (no device attribute), shared by fe_es_forward and fe_es_forward_kernel_name so the two cannot disagree.
// ------------------------------------------------------------------------------------------
enum EsKern { ES_FAST, ES_STREAM, ES_GENERIC, ES_ERR_SMEM };
struct EsRoute {
    EsKern kern;
    size_t smem;     // dynamic shared memory of the launch
    FastShape fast;  // ES_FAST
    StreamShape stream; // ES_STREAM
    bool theta_smem; // ES_GENERIC: theta staged in shared memory (else read from global memory)
};

// obs_aligned: dense observations start on a 16-byte boundary (always true for lazy handles)
EsRoute route_forward(const EsLayout &lay, const bool lazy, const bool obs_aligned) {
    EsRoute rt{};
    const int64_t P = lay.off[lay.L];
    // ---- fast path: 5R -> <= 8 first layer (R <= 63), inputs 16-byte granular, ring fits in shared memory
    const bool no_fast = env_override("FE_ES_NO_FAST") != 0; // A/B runs (experiment builds only)
    if (!no_fast && lay.out[0] <= 8 && lay.in[0] % 5 == 0 && lay.in[0] / 5 <= 63 &&
        (lazy || (lay.in[0] % 4 == 0 && obs_aligned))) {
        FastShape &f = rt.fast;
        f.rows = lay.in[0] / 5;
        f.x_bytes = lazy ? f.rows * 16 : f.rows * 20;
        f.eps_bytes = (int)(P * 2);
        f.stage_bytes = (f.eps_bytes + 2 * f.x_bytes + 16 + 127) & ~127;
        int md = 1;
        for (int l = 1; l <= lay.L; ++l) md = lay.out[l - 1] > md ? lay.out[l - 1] : md;
        f.act_stride = (md + 1 + 3) & ~3;
        f.tail_in_regs = lay.L == 2 && lay.out[1] <= 8;
        f.theta_bytes = (int)((P * 4 + 127) & ~(int64_t)127);
        rt.smem = fast_smem_bytes(f);
        if (rt.smem <= kSmemMax) {
            rt.kern = ES_FAST;
            return rt;
        }
    }
    // ---- streaming path: every layer has <= 319 inputs, eps chunks 16-byte granular (always), ring + activations fit
    const bool no_stream = env_override("FE_ES_NO_STREAM") != 0;
    bool stream_ok = !no_stream;
    for (int l = 0; l < lay.L; ++l) stream_ok = stream_ok && lay.in[l] + 1 <= 32 * kStRows;
    if (stream_ok) {
        StreamShape &f = rt.stream;
        int max_in1 = 0, a = 0, b = 0;
        f.chunks[0] = 0;
        for (int l = 0; l < lay.L; ++l) {
            if (lay.in[l] + 1 > max_in1) max_in1 = lay.in[l] + 1;
            f.chunks[l + 1] = f.chunks[l] + (lay.out[l] + 7) / 8;
            // buffer A holds the inputs of even layers (and the outputs of odd ones), buffer B the others
            const int need_in = lay.in[l] + 1, need_out = lay.out[l] + 1;
            if (l % 2 == 0) { a = need_in > a ? need_in : a; b = need_out > b ? need_out : b; }
            else { b = need_in > b ? need_in : b; a = need_out > a ? need_out : a; }
        }
        f.stage_bytes = (max_in1 * 16 + 127) & ~127;
        f.strideA = (a + 1) & ~1;
        f.strideB = (b + 1) & ~1;
        f.U = kStMaxU;
        while (f.U > 1 && stream_smem_bytes(f) > kSmemMax) --f.U;
        rt.smem = stream_smem_bytes(f);
        if (rt.smem <= kSmemMax) {
            rt.kern = ES_STREAM;
            return rt;
        }
    }
    // ---- generic kernel: theta in shared memory while the block stays small enough for >= 2 blocks per SM
    const int stride = (lay.max_dim + 1 + 3) & ~3;
    const size_t act_bytes = (size_t)kEsWarps * 4 * stride * sizeof(float);
    rt.theta_smem = act_bytes + (size_t)P * sizeof(float) <= 100 * 1024;
    rt.smem = act_bytes + (rt.theta_smem ? (size_t)P * sizeof(float) : 0);
    rt.kern = rt.smem <= kSmemMax ? ES_GENERIC : ES_ERR_SMEM;
    return rt;
}

} // namespace

extern "C" {

int64_t fe_es_params_padded(const FeEsNet *net) {
    EsLayout lay;
    return make_layout(net, lay) ? lay.off[lay.L] : -1;
}

int64_t fe_es_packed_index(const FeEsNet *net, int32_t layer, int32_t input, int32_t output) {
    EsLayout lay;
    if (!make_layout(net, lay) || layer < 0 || layer >= lay.L) return -1;
    if (input < 0 || input > lay.in[layer] || output < 0 || output >= lay.out[layer]) return -1;
    return lay.off[layer] + ((int64_t)(output / 8) * (lay.in[layer] + 1) + input) * 8 + (output % 8);
}

int fe_es_perturb(const FeEsNet *net, uint64_t seed, uint64_t generation, int64_t pair_id_base, int64_t num_pairs,
                  void *eps_dev, void *stream) {
    EsLayout lay;
    if (!make_layout(net, lay) || !eps_dev || num_pairs <= 0 || pair_id_base < 0 || generation >> 31) return FE_EINVAL;
    if ((uintptr_t)eps_dev & 15) return FE_EALIGN;
    DeviceGuard guard(pointer_device(eps_dev));
    if (guard.rc) return guard.rc;
    const int64_t total8 = lay.off[lay.L] / 8, n = num_pairs * total8;
    fe_es_perturb_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(total8, num_pairs, pair_id_base, seed,
                                                                                        generation, (__half *)eps_dev);
    return (int)cudaGetLastError();
}

int fe_es_forward(const FeEsNet *net, const float *theta_packed_dev, const void *eps_dev, float sigma, int64_t num_envs,
                  int64_t num_eval_envs, const float *obs_dev, const void *logret_dev, const int64_t *obs_row0_dev,
                  const float *obs_posfeat_dev, int32_t window, float action_noise_std, uint64_t seed,
                  uint64_t step_counter, int64_t env_id_base, float *actions_dev, int32_t device, void *stream) {
    EsLayout lay;
    if (!make_layout(net, lay) || !theta_packed_dev || !actions_dev) return FE_EINVAL;
    const int64_t train = num_envs - num_eval_envs;
    if (num_envs <= 0 || num_eval_envs < 0 || train < 0 || (train & 1)) return FE_EINVAL; // mirrored sampling :24-27
    if (train > 0 && !eps_dev) return FE_EINVAL;
    const bool lazy = obs_dev == nullptr;
    if (lazy) {
        if (!logret_dev || !obs_row0_dev || !obs_posfeat_dev || window <= 0 || window * 5 != lay.in[0]) return FE_EINVAL;
        if ((uintptr_t)logret_dev & 15) return FE_EALIGN;
    }
    if (((uintptr_t)eps_dev | (uintptr_t)theta_packed_dev) & 15) return FE_EALIGN;
    const EsRoute rt = route_forward(lay, lazy, lazy || ((uintptr_t)obs_dev & 15) == 0);
    if (rt.kern == ES_ERR_SMEM) return FE_ESMEM;
    DeviceGuard guard(device);
    if (guard.rc) return guard.rc;
    int num_sms = 0;
    if (const int rc = device_sm_count(device, &num_sms)) return rc;
    const int64_t units = train / 2 + num_eval_envs;
    return with_flag(lazy, [&](auto lazy_obs) {
        constexpr bool kLazy = decltype(lazy_obs)::value;
        if (rt.kern == ES_FAST) {
            constexpr auto kern = fe_es_forward_fast_kernel<kLazy>;
            if (const int rc = opt_in_smem<kern>(device)) return rc;
            int64_t blocks = (units + kFastWarps - 1) / kFastWarps;
            if (blocks > num_sms) blocks = num_sms;
            kern<<<(unsigned)blocks, kFastThreads, rt.smem, (cudaStream_t)stream>>>(
                lay, rt.fast, theta_packed_dev, (const __half *)eps_dev, sigma, train / 2, num_eval_envs, obs_dev,
                (const float *)logret_dev, obs_row0_dev, obs_posfeat_dev, action_noise_std, seed, step_counter, env_id_base,
                actions_dev);
            return (int)cudaGetLastError();
        }
        if (rt.kern == ES_STREAM) {
            constexpr auto kern = fe_es_forward_stream_kernel<kLazy>;
            if (const int rc = opt_in_smem<kern>(device)) return rc;
            int64_t blocks = (units + (int64_t)kStWarps * rt.stream.U - 1) / ((int64_t)kStWarps * rt.stream.U);
            if (blocks > num_sms) blocks = num_sms;
            kern<<<(unsigned)blocks, kStThreads, rt.smem, (cudaStream_t)stream>>>(
                lay, rt.stream, theta_packed_dev, (const __half *)eps_dev, sigma, train / 2, num_eval_envs, obs_dev,
                (const float *)logret_dev, obs_row0_dev, obs_posfeat_dev, window, action_noise_std, seed, step_counter,
                env_id_base, actions_dev);
            return (int)cudaGetLastError();
        }
        return with_flag(rt.theta_smem, [&](auto theta_smem) {
            constexpr auto kern = fe_es_forward_kernel<kLazy, decltype(theta_smem)::value>;
            if (const int rc = opt_in_smem<kern>(device)) return rc;
            int per_sm = (int)(kSmemMax / (rt.smem + 1024));
            if (per_sm > 8) per_sm = 8;
            if (per_sm < 1) per_sm = 1;
            int64_t blocks = (units + kEsWarps - 1) / kEsWarps;
            if (blocks > (int64_t)num_sms * per_sm) blocks = (int64_t)num_sms * per_sm;
            kern<<<(unsigned)blocks, kEsThreads, rt.smem, (cudaStream_t)stream>>>(
                lay, theta_packed_dev, (const __half *)eps_dev, sigma, train / 2, num_eval_envs, obs_dev,
                (const float *)logret_dev, obs_row0_dev, obs_posfeat_dev, window, action_noise_std, seed, step_counter,
                env_id_base, actions_dev);
            return (int)cudaGetLastError();
        });
    });
}

const char *fe_es_forward_kernel_name(const FeEsNet *net, int32_t lazy, int32_t obs_aligned) {
    EsLayout lay;
    if (!make_layout(net, lay)) return "";
    const bool lz = lazy != 0;
    const EsRoute rt = route_forward(lay, lz, lz || obs_aligned != 0);
    // one name per (input form, U) for whatever kStMaxU the build uses (FE_ES_ST_MAXU); filled once, thread-safely
    static const struct StreamNames {
        char s[2][kStMaxU][48];
        StreamNames() {
            for (int l = 0; l < 2; ++l)
                for (int u = 0; u < kStMaxU; ++u)
                    snprintf(s[l][u], sizeof s[l][u], "fe_es_forward_stream_kernel<%s> U=%d", l ? "lazy" : "dense", u + 1);
        }
    } stream_names;
    switch (rt.kern) {
    case ES_FAST: return lz ? "fe_es_forward_fast_kernel<lazy>" : "fe_es_forward_fast_kernel<dense>";
    case ES_STREAM: return stream_names.s[lz][rt.stream.U - 1];
    case ES_GENERIC:
        return rt.theta_smem ? (lz ? "fe_es_forward_kernel<lazy,theta_smem>" : "fe_es_forward_kernel<dense,theta_smem>")
                             : (lz ? "fe_es_forward_kernel<lazy,theta_global>" : "fe_es_forward_kernel<dense,theta_global>");
    default: return "none (FE_ESMEM: the network's activations do not fit in shared memory)";
    }
}

int64_t fe_es_gradient_scratch(const FeEsNet *net, int64_t num_pairs) {
    EsLayout lay;
    if (!make_layout(net, lay) || num_pairs <= 0) return -1;
    return ((num_pairs + kGradSlab - 1) / kGradSlab) * lay.off[lay.L];
}

int fe_es_gradient(const FeEsNet *net, const void *eps_dev, const float *pair_weights_dev, int64_t num_pairs,
                   float *scratch_dev, float *grad_packed_dev, void *stream) {
    EsLayout lay;
    if (!make_layout(net, lay) || !eps_dev || !pair_weights_dev || !scratch_dev || !grad_packed_dev || num_pairs <= 0)
        return FE_EINVAL;
    if (((uintptr_t)eps_dev | (uintptr_t)scratch_dev) & 15) return FE_EALIGN;
    DeviceGuard guard(pointer_device(eps_dev));
    if (guard.rc) return guard.rc;
    const int64_t total = lay.off[lay.L], total8 = total / 8, slabs = (num_pairs + kGradSlab - 1) / kGradSlab;
    const dim3 grid((unsigned)((total8 + kGradThreads - 1) / kGradThreads), (unsigned)slabs);
    fe_es_grad_partial_kernel<<<grid, kGradThreads, 0, (cudaStream_t)stream>>>(total8, num_pairs, (const __half *)eps_dev,
                                                                               pair_weights_dev, scratch_dev);
    fe_es_grad_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(total, slabs, scratch_dev,
                                                                                               grad_packed_dev);
    return (int)cudaGetLastError();
}

int fe_es_store(const void *rewards_dev, int32_t rewards_f64, const int32_t *dones_dev, int64_t num_envs,
                int64_t env_id_base, int64_t total_envs, uint64_t step_ordinal, float *cur_returns_dev,
                float *cur_steps_dev, int64_t capacity, unsigned long long *counters_dev, int64_t *fin_key_dev,
                int64_t *fin_env_dev, float *fin_ret_dev, void *stream) {
    if (!rewards_dev || !dones_dev || !cur_returns_dev || !cur_steps_dev || !counters_dev || !fin_key_dev || !fin_env_dev ||
        !fin_ret_dev || num_envs <= 0 || capacity < 0)
        return FE_EINVAL;
    DeviceGuard guard(pointer_device(rewards_dev));
    if (guard.rc) return guard.rc;
    const unsigned blocks = (unsigned)((num_envs + 255) / 256);
    return with_out_type(rewards_f64 != 0, [&](auto rew_type) {
        using RewT = decltype(rew_type);
        fe_es_store_kernel<RewT><<<blocks, 256, 0, (cudaStream_t)stream>>>(
            (const RewT *)rewards_dev, dones_dev, num_envs, env_id_base, total_envs, step_ordinal, cur_returns_dev,
            cur_steps_dev, capacity, counters_dev, fin_key_dev, fin_env_dev, fin_ret_dev);
        return (int)cudaGetLastError();
    });
}

} // extern "C"
