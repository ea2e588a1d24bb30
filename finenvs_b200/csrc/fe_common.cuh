// fe_common.cuh — pieces shared by the translation units of libfinenvs_b200.so.
#ifndef FE_COMMON_CUH
#define FE_COMMON_CUH
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <type_traits>

namespace {

// ------------------------------------------------------------------------------------------
// Philox4x32-10 keyed (seed) with counter (env id, step | kind<<63): the redraw RNG
// (replaces torch.randint at :253 / :511; identical on host, see fe_philox)
// ------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t env_id, uint64_t step,
                                                       uint32_t kind, uint32_t out[4]) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)env_id, c1 = (uint32_t)(env_id >> 32), c2 = (uint32_t)step,
             c3 = ((uint32_t)(step >> 32) & 0x7FFFFFFFu) | (kind << 31);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// ------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + 1-D bulk async copies (TMA engine, no tensor map needed)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// Whole-warp wait (call converged): every lane makes ONE attempt; only if the phase is still open does lane 0 keep
// waiting while the others sit in __syncwarp.  Measured (tools/mbar_wait_probe.cu, phase already complete): 75 cycles,
// against 130 for a try_wait loop run by all lanes and 190 for `if (lane == 0) wait; __syncwarp()`.
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (!__all_sync(0xFFFFFFFFu, ok)) {
        if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity);
        __syncwarp();
    }
}
// global -> shared, completes `bytes` on the mbarrier
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// shared -> global
__device__ __forceinline__ void bulk_store(void *dst, uint32_t src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes)
                 : "memory");
}
// L2 eviction priorities for the TMA engine's requests: the observation stream is written once and never read by this
// kernel (evict_first), the series tables are re-read by every env (evict_last).  Without them the 1.26 GB written per
// step pushed the 20 MB observation-layout table out of L2 again and again: ncu showed 297 MB of DRAM reads per launch.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_store_hint(void *dst, uint32_t src_smem, uint32_t bytes, uint64_t policy) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src_smem),
                 "r"(bytes), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// host side: current-device discipline of the entry points
// ------------------------------------------------------------------------------------------
// RAII: make `device` current for the duration of an entry point and put the caller's device back afterwards (an env
// on cuda:1 inside a process whose current device is cuda:0 must not change where the caller's next allocation lands)
struct DeviceGuard {
    int prev = -1, rc = 0;
    bool switched = false;
    explicit DeviceGuard(int device) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) { rc = (int)e; return; }
        if (prev != device) {
            e = cudaSetDevice(device);
            if (e != cudaSuccess) { rc = (int)e; return; }
            switched = true;
        }
    }
    ~DeviceGuard() { if (switched) (void)cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};

// entry points without a device argument: the device that owns `ptr` (a device pointer the caller passed)
inline int pointer_device(const void *ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess || a.type != cudaMemoryTypeDevice) {
        (void)cudaGetLastError();
        int cur = 0;
        (void)cudaGetDevice(&cur);
        return cur;
    }
    return a.device;
}

// ------------------------------------------------------------------------------------------
// host side: kernel set-up
// ------------------------------------------------------------------------------------------
// dynamic shared memory every large-smem kernel opts in to
constexpr int kSmemMax = 226 * 1024;

// SM count of `device`, queried once per device
inline int device_sm_count(int device, int *out) {
    static std::atomic<int> num_sms[16];
    const int dev = device & 15;
    int n = num_sms[dev].load(std::memory_order_relaxed);
    if (!n) {
        cudaError_t e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
        if (e != cudaSuccess) return (int)e;
        num_sms[dev].store(n, std::memory_order_relaxed);
    }
    *out = n;
    return 0;
}

// cudaFuncSetAttribute(max dynamic shared memory) once per (kernel instantiation, device); safe to race: the attribute
// call is idempotent and the flag is only set after it succeeded
template <auto Kern> int opt_in_smem(int device) {
    static std::atomic<uint32_t> done_mask{0};
    const uint32_t bit = 1u << (device & 15);
    if (done_mask.load(std::memory_order_acquire) & bit) return 0;
    cudaError_t e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
    if (e != cudaSuccess) return (int)e;
    done_mask.fetch_or(bit, std::memory_order_release);
    return 0;
}

// Template arguments chosen at run time: f is called with a value of the chosen type (f(float{}) / f(double{}) for the
// output dtype, f(std::true_type{}) / f(std::false_type{}) for a flag), so the launch it makes is written once.
template <class F> int with_out_type(bool f64, F &&f) { return f64 ? f(double{}) : f(float{}); }
template <class F> int with_flag(bool b, F &&f) { return b ? f(std::true_type{}) : f(std::false_type{}); }

} // namespace
#endif // FE_COMMON_CUH
