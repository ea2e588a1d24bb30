// fe_step.cu — the vectorised trading-env step of hmomin/FinEnvs as hand-written sm_100a CUDA.
//
// One launch per step does what finenvs/environments/time_series_env.py:277-536 does in ~660
// torch-eager ops: advance the time pointer, read the current OHLC bar, map the action to trades
// with cash / position / margin / commission bookkeeping, build the observation window, compute
// the reward, detect episode end, auto-reset (with counter-based redraws) and keep the
// evaluate-mode metrics.  The arithmetic follows the reference op for op, dtype for dtype
// (SURVEY.md App. A): f32 state, f64 temporaries rounded once, no FMA contraction (every
// product/sum below is an explicit __*_rn intrinsic, and the TU is built with -fmad=false).
//
// Data movement (the part that costs time: ~2.2 KB per env-step at W=60, <100 flops):
//   tile variant   — each env's W x 16 B log-return window is fetched with one 1-D bulk async
//                    copy (cp.async.bulk, SASS UBLKCP) into shared memory, completing on an
//                    mbarrier; the block interleaves the position feature (4 -> 5 values per row,
//                    conflict-free stride-5 STS) into an output tile that is contiguous in the
//                    (N, W, 5) observation tensor and leaves with one bulk async store.
//   direct variant — warp-per-env global->global copy for windows that do not fit in smem.
//
// The C ABI is declared in include/finenvs_b200.h.
#include "finenvs_b200.h"
#include "fe_common.cuh"
#include "fe_metrics.cuh"

#include <cuda.h> // CUtensorMap (types only; cuTensorMapEncodeTiled is resolved at run time, libcuda is not linked)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <mutex>
#include <vector>

namespace {

constexpr int kThreads = 128;          // threads per block (both variants)
constexpr int kMaxTileEnvs = kThreads; // one bookkeeping thread per env of the tile
constexpr int kSmemHeader = 16;        // mbarrier (8 B) + pad

// ------------------------------------------------------------------------------------------
// exact (never contracted) arithmetic helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float d2f(double a) { return __double2float_rn(a); }
// torch.relu keeps NaN (clamp_min), unlike fmax
__device__ __forceinline__ float relu32(float x) { return x < 0.0f ? 0.0f : x; }
__device__ __forceinline__ double relu64(double x) { return x < 0.0 ? 0.0 : x; }

struct Consts {
    float ms, scale, cf, imrf, SBf;
    double c, imr, mmr1, SB;
    // optional second destination of rewards / dones (fe_step_host's zero-copy mode: mapped pinned host memory)
    void *rewards_mirror;
    int32_t *dones_mirror;
    // fe_step_host_packed: 1 bit per env, one word per 32-env tile, written by the persistent kernels' bookkeepers.
    // dones_bits_out is where they write it.  Writing the words straight to mapped host memory means 32 Ki separate 4-byte
    // PCIe writes per 1 Mi-env step (partial cache lines for the host: measured 0.32 ms per step against 0.27 ms with int32
    // dones), so the words go to a staging buffer in HBM and leave in 128-byte lines: the gather kernel's
    // blocks copy the staging buffer to dones_bits_host (dones_bits_host != nullptr) once all bookkeeping is done, the
    // other kernels are followed by fe_flush_bits_kernel.
    uint32_t *dones_bits_out;
    uint32_t *dones_bits_host;
};

Consts make_consts(const FeParams &p) {
    Consts k;
    k.ms = (float)p.max_shares;
    k.scale = (float)((double)p.max_shares + 0.5); // :299  f32 tensor * python float
    k.cf = (float)p.commission;                    // :364
    k.imrf = (float)p.imr;                         // :377-378
    k.SBf = (float)p.starting_balance;             // :499
    k.c = p.commission;
    k.imr = p.imr;
    k.mmr1 = 1.0 + p.mmr;                          // :462
    k.SB = p.starting_balance;
    k.rewards_mirror = nullptr;
    k.dones_mirror = nullptr;
    k.dones_bits_out = nullptr;
    k.dones_bits_host = nullptr;
    return k;
}

__device__ __forceinline__ void draw_segment(const FeParams &p, const FeSeries &s, int64_t gid, uint64_t step,
                                             uint32_t kind, int32_t &seg, int32_t &off) {
    uint32_t r[4];
    philox4x32_10(p.seed, (uint64_t)gid, step, kind, r);
    seg = (int32_t)__umulhi(r[0], (uint32_t)p.num_segments);
    off = 0;
    if (p.random_offset) {
        // valid start pointers are 0 .. seg_len - W - 1 (one bar must remain to step onto)
        const int32_t span = __ldg(s.seg_len + seg) - p.window;
        off = span > 0 ? (int32_t)__umulhi(r[1], (uint32_t)span) : 0;
    }
}

// ------------------------------------------------------------------------------------------
// per-env bookkeeping: everything of step() except moving the window
// ------------------------------------------------------------------------------------------
struct EnvResult {
    int64_t row0;   // first row of the observation window in the flat series
    double posfeat; // (long - short) * close / starting_balance  (:428-431)
    int done;
    int newly_terminated;
    double fin_return; // episode return of an env that finished this step (stats)
    int fin_len;
};

// reset() (:423-435): no state change, current window + position feature
__device__ __forceinline__ EnvResult env_observe(const FeParams &p, const FeSeries &s, const FeState &st,
                                                 const Consts &k, int64_t i) {
    EnvResult r;
    r.row0 = __ldg(s.seg_start + st.seg[i]) + st.ptr[i];
    const double C = __ldg(s.prices + (r.row0 + p.window - 1) * 4 + 3);
    const float net = fsub(st.long_sh[i], st.short_sh[i]);
    r.posfeat = __ddiv_rn(dmul((double)net, C), k.SB);
    r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0;
    return r;
}

// The loads of one env-step, split from the arithmetic so that a caller can issue them ahead of time (the gather
// variant's bookkeeper warps keep the loads of the next two tiles in flight while they compute the current one: under a
// saturated write stream a dependent HBM load costs several thousand cycles, and the chain state -> segment table ->
// price row was what bounded the persistent kernels' bookkeeping at ~0.16 ms per 1 Mi envs).
struct EnvLoads {   // per-env state + action (first hop)
    int32_t seg, ptr;
    float cash, lng, sht, act;
    double margin;
};
struct EnvBar {     // current bar of the env (second / third hop: needs seg and ptr)
    int32_t len;
    int64_t row0;   // first row of the window AFTER the time pointer advanced
    double O, H, L, C;
};
__device__ __forceinline__ EnvLoads env_load_state(const FeState &st, const float *__restrict__ actions, int64_t i) {
    EnvLoads e;
    e.act = __ldg(actions + i);
    e.seg = st.seg[i];
    e.ptr = st.ptr[i];
    e.cash = st.cash[i];
    e.lng = st.long_sh[i];
    e.sht = st.short_sh[i];
    e.margin = st.margin[i];
    return e;
}
__device__ __forceinline__ EnvBar env_load_bar(const FeParams &p, const FeSeries &s, const EnvLoads &e) {
    EnvBar b;
    b.len = __ldg(s.seg_len + e.seg);
    b.row0 = __ldg(s.seg_start + e.seg) + e.ptr + 1; // :281-282 advance time
    // :323-342 current bar = last row of the window: O,H,L,C as two 16-byte loads
    const double2 *px = reinterpret_cast<const double2 *>(s.prices + (b.row0 + p.window - 1) * 4);
    const double2 oh = __ldg(px), lc = __ldg(px + 1);
    b.O = oh.x; b.H = oh.y; b.L = lc.x; b.C = lc.y;
    return b;
}

// The trading arithmetic of one env-step, written once.  Whatever it reads or writes besides `ld` / `bar` goes through
// `io`: GlobalEnvIO (the state arrays and outputs, for the step kernels) or BacktestEnvIO (registers across the K steps
// of fe_backtest_kernel).
template <typename IO>
__device__ __forceinline__ EnvResult env_compute_core(const FeParams &p, const FeSeries &s, const Consts &k, int64_t i,
                                                      const EnvLoads &ld, const EnvBar &bar, bool track, uint64_t step,
                                                      IO &io) {
    EnvResult res;
    const int W = p.window;
    // :298-302 action -> integer share delta (round half to even, then clamp)
    float d = rintf(fmul(ld.act, k.scale));
    d = d < -k.ms ? -k.ms : (d > k.ms ? k.ms : d);
    int32_t seg = ld.seg;
    int32_t ptr = ld.ptr + 1;
    const int32_t len = bar.len;
    res.row0 = bar.row0;
    const double O = bar.O, H = bar.H, L = bar.L, C = bar.C;
    float cash = ld.cash;
    float lng = ld.lng;
    float sht = ld.sht;
    double margin = ld.margin;
    float comm = 0.0f; // :305
    // :344-351
    float pos = d < 0.0f ? 0.0f : d;
    float neg = d > 0.0f ? 0.0f : d;
    const double Omc = dsub(O, k.c), Opc = dadd(O, k.c);
    { // :353-361 sell longs (+ :363-365)
        const float nl = relu32(fadd(lng, neg));
        const float sold = fsub(lng, nl);
        neg = fadd(neg, sold);
        comm = fadd(comm, fmul(sold, k.cf));
        cash = d2f(dadd((double)cash, dmul((double)sold, Omc)));
        lng = nl;
    }
    { // :367-383 cover shorts, re-mark margin to imr * short * open
        const float ns = relu32(fsub(sht, pos));
        const float bought = fsub(sht, ns);
        pos = fsub(pos, bought);
        comm = fadd(comm, fmul(bought, k.cf));
        cash = d2f(dsub((double)cash, dmul((double)bought, Opc)));
        sht = ns;
        const double nm = dmul((double)fmul(k.imrf, sht), O);
        cash = d2f(dsub((double)cash, dsub(nm, margin)));
        margin = nm;
    }
    // :385-392 all-or-nothing long entry
    if (dsub((double)cash, dmul((double)pos, Opc)) < 0.0) pos = 0.0f;
    // :394-399
    comm = fadd(comm, fmul(pos, k.cf));
    cash = d2f(dsub((double)cash, dmul((double)pos, Opc)));
    lng = fadd(lng, pos);
    { // :401-410 all-or-nothing short entry, :412-421 open short
        float q = -neg;
        float sc = fmul(q, k.cf);
        double req = dmul(k.imr, dmul((double)q, O));
        if (dsub(dsub((double)cash, req), (double)sc) < 0.0) {
            q = -0.0f; // neg = 0 -> -neg
            sc = fmul(q, k.cf);
            req = dmul(k.imr, dmul((double)q, O));
        }
        comm = fadd(comm, fmul(q, k.cf));
        cash = d2f(dsub((double)cash, dadd(req, (double)sc)));
        margin = dadd(margin, req);
        sht = fadd(sht, q);
    }
    // :321 -> reset(): the observation is built NOW, before rewards / dones / auto-reset
    res.posfeat = __ddiv_rn(dmul((double)fsub(lng, sht), C), k.SB);
    // :447-457 rewards
    int done = cash < 0.0f; // :448
    double rew;
    {
        // :459-468 maintenance margin at High
        const double mc1 = relu64(dsub(dmul(dmul((double)sht, H), k.mmr1), margin));
        cash = d2f(dsub((double)cash, mc1));
        margin = dadd(margin, mc1);
        done |= cash < 0.0f;
        // :470-475 margin release at Low
        const double rel = relu64(dsub(margin, dmul(dmul((double)sht, L), k.imr)));
        margin = dsub(margin, rel);
        cash = d2f(dadd((double)cash, rel));
        // :451 maintenance margin at Close
        const double mc2 = relu64(dsub(dmul(dmul((double)sht, C), k.mmr1), margin));
        cash = d2f(dsub((double)cash, mc2));
        margin = dadd(margin, mc2);
        done |= cash < 0.0f;
        rew = dadd(-mc1, -mc2);
        if (done) { lng = 0.0f; sht = 0.0f; } // :452-453
        rew = dadd(rew, dmul((double)fsub(lng, sht), dsub(C, O))); // :454-455
        rew = dsub(rew, (double)comm);                              // :456
    }
    // :477-496 time limit / NaN padding == pointer ran into the end of the (effective) segment
    done |= (ptr + W >= len);
    // :288-289 closing commission on whatever is still held
    rew = dsub(rew, (double)fmul(fmul(done ? 1.0f : 0.0f, fadd(sht, lng)), k.cf));
    // :498-521 auto-reset
    if (done) {
        cash = k.SBf; margin = 0.0; lng = 0.0f; sht = 0.0f; ptr = 0;
        const int64_t gid = p.env_id_base + i;
        if (p.reset_mode == FE_RESET_ALL || (p.reset_mode == FE_RESET_LAST && gid == p.total_envs - 1)) {
            draw_segment(p, s, gid, step, 0u, seg, ptr);
            io.set_seg(seg);
        }
    }
    res.done = done;
    res.newly_terminated = 0; res.fin_return = 0.0; res.fin_len = 0;
    if (p.evaluate) { // :523-536
        const int was = io.terminated();
        if (was) rew = 0.0;                                             // :527-528
        if (done && !was) { io.set_terminated(); res.newly_terminated = 1; } // :529
        io.set_ep_return(d2f(dadd((double)io.ep_return(), rew)));       // :530  f32 += f64
    } else if (track) { // extension: running episode return / length for the NCCL-reduced statistics
        const float er = d2f(dadd((double)io.ep_return(), rew));
        const int32_t el = io.ep_len() + 1;
        if (done) { res.fin_return = (double)er; res.fin_len = el; }
        io.set_ep_return(done ? 0.0f : er);
        io.set_ep_len(done ? 0 : el);
    }
    io.finish(ptr, cash, lng, sht, margin, rew, done);
    return res;
}

// the step kernels' accessor: env i's slots of the state arrays, its reward / done outputs (and their mirrors)
template <typename OutT>
struct GlobalEnvIO {
    const FeState &st;
    const Consts &k;
    const int64_t i;
    OutT *__restrict__ rewards;
    int32_t *__restrict__ dones;
    __device__ __forceinline__ void set_seg(int32_t v) { st.seg[i] = v; }
    __device__ __forceinline__ int terminated() const { return st.terminated[i]; }
    __device__ __forceinline__ void set_terminated() { st.terminated[i] = 1; }
    __device__ __forceinline__ float ep_return() const { return st.ep_return[i]; }
    __device__ __forceinline__ void set_ep_return(float v) { st.ep_return[i] = v; }
    __device__ __forceinline__ int32_t ep_len() const { return st.ep_len[i]; }
    __device__ __forceinline__ void set_ep_len(int32_t v) { st.ep_len[i] = v; }
    __device__ __forceinline__ void finish(int32_t ptr, float cash, float lng, float sht, double margin, double rew, int done) {
        st.ptr[i] = ptr; st.cash[i] = cash; st.long_sh[i] = lng; st.short_sh[i] = sht; st.margin[i] = margin;
        rewards[i] = (OutT)rew;
        dones[i] = done; // :296 dones.int()
        if (k.rewards_mirror) reinterpret_cast<OutT *>(k.rewards_mirror)[i] = (OutT)rew;
        if (k.dones_mirror) k.dones_mirror[i] = done;
    }
};

template <typename OutT>
__device__ __forceinline__ EnvResult env_compute(const FeParams &p, const FeSeries &s, const FeState &st, const Consts &k,
                                                 int64_t i, const EnvLoads &ld, const EnvBar &bar, OutT *__restrict__ rewards,
                                                 int32_t *__restrict__ dones, bool track, uint64_t step) {
    GlobalEnvIO<OutT> io{st, k, i, rewards, dones};
    return env_compute_core(p, s, k, i, ld, bar, track, step, io);
}

template <typename OutT>
__device__ __forceinline__ EnvResult env_step(const FeParams &p, const FeSeries &s, const FeState &st,
                                              const Consts &k, int64_t i, const float *__restrict__ actions,
                                              OutT *__restrict__ rewards, int32_t *__restrict__ dones,
                                              bool track, uint64_t step) {
    const EnvLoads ld = env_load_state(st, actions, i);
    const EnvBar bar = env_load_bar(p, s, ld);
    return env_compute<OutT>(p, s, st, k, i, ld, bar, rewards, dones, track, step);
}

// one atomic per warp for the episode statistics
__device__ __forceinline__ void accumulate_stats(FeStats *stats, const EnvResult &r, bool active) {
    if (stats == nullptr) return;
    const unsigned full = 0xFFFFFFFFu;
    const int done = active ? r.done : 0;
    const int nterm = active ? r.newly_terminated : 0;
    const unsigned nd = __reduce_add_sync(full, (unsigned)done);
    const unsigned nt = __reduce_add_sync(full, (unsigned)nterm);
    if (nd == 0 && nt == 0) return;
    unsigned sl = __reduce_add_sync(full, (unsigned)(done ? r.fin_len : 0));
    double sr = done ? r.fin_return : 0.0;
    double sq = sr * sr;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(full, sr, o);
        sq += __shfl_xor_sync(full, sq, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (nd) atomicAdd(&stats->n_done, (unsigned long long)nd);
        if (nt) atomicAdd(&stats->n_terminated, (unsigned long long)nt);
        if (sl) atomicAdd(&stats->sum_len, (unsigned long long)sl);
        if (nd) { atomicAdd(&stats->sum_return, sr); atomicAdd(&stats->sum_return_sq, sq); }
    }
}

// ------------------------------------------------------------------------------------------
// tile variant
// ------------------------------------------------------------------------------------------
template <typename OutT> struct Row4;
template <> struct Row4<float> { float4 v; };
template <> struct Row4<double> { double2 a, b; };

// smem layout: [mbarrier 16 B][posfeat E x OutT, padded to 16 B][in tile E*W*4 OutT][out tile E*W*5 OutT]
template <typename OutT> __host__ __device__ constexpr size_t tile_pf_bytes(int E) {
    return ((size_t)E * sizeof(OutT) + 15) & ~(size_t)15;
}
template <typename OutT> __host__ __device__ inline size_t tile_smem_bytes(int E, int W) {
    return kSmemHeader + tile_pf_bytes<OutT>(E) + (size_t)E * W * 9 * sizeof(OutT);
}

template <typename OutT, bool kObserve>
__global__ void __launch_bounds__(kThreads)
fe_tile_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const float *__restrict__ actions,
               OutT *__restrict__ obs, OutT *__restrict__ rewards, int32_t *__restrict__ dones, FeStats *stats,
               const uint64_t step_arg, const uint64_t *__restrict__ step_dev, const int E) {
    extern __shared__ __align__(128) unsigned char smem[];
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int W = p.window;
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * E;
    const int nvalid = (int)min((int64_t)E, p.num_envs - env0);
    OutT *pf = reinterpret_cast<OutT *>(smem + kSmemHeader);
    unsigned char *in_tile = smem + kSmemHeader + tile_pf_bytes<OutT>(E);
    OutT *out_tile = reinterpret_cast<OutT *>(in_tile + (size_t)E * W * 4 * sizeof(OutT));
    const uint32_t bar = smem_u32(smem);
    const uint32_t row_bytes = 4 * sizeof(OutT);
    const uint32_t win_bytes = (uint32_t)W * row_bytes;

    if (tid == 0) {
        mbar_init(bar, (uint32_t)nvalid);
        mbar_fence_init();
    }
    __syncthreads();

    // ---- one thread per env: fetch its window asynchronously, do the bookkeeping meanwhile ----
    const bool active = tid < nvalid;
    EnvResult r;
    r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0;
    if (active) {
        const int64_t i = env0 + tid;
        // window start is known before any arithmetic: launch the copy first
        const int64_t row0 = __ldg(s.seg_start + st.seg[i]) + st.ptr[i] + (kObserve ? 0 : 1);
        mbar_arrive_expect_tx(bar, win_bytes);
        bulk_load(smem_u32(in_tile + (size_t)tid * win_bytes),
                  reinterpret_cast<const unsigned char *>(s.logret) + (size_t)row0 * row_bytes, win_bytes, bar);
        if (kObserve) r = env_observe(p, s, st, k, i);
        else r = env_step<OutT>(p, s, st, k, i, actions, rewards, dones, stats != nullptr, step);
        pf[tid] = (OutT)r.posfeat;
    }
    if (!kObserve && tid < ((nvalid + 31) & ~31)) accumulate_stats(stats, r, active);
    __syncthreads(); // pf visible
    mbar_wait(bar, 0); // all windows landed

    // ---- interleave: row (4 values) + position feature -> 5 values, rows are contiguous in both tiles
    const int nrows = nvalid * W;
    const float invW = 1.0f / (float)W;
    const Row4<OutT> *in_rows = reinterpret_cast<const Row4<OutT> *>(in_tile);
    for (int row = tid; row < nrows; row += blockDim.x) {
        const int e = __float2int_rz(((float)row + 0.5f) * invW);
        const Row4<OutT> v = in_rows[row];
        OutT *o = out_tile + (size_t)row * 5;
        if constexpr (sizeof(OutT) == 4) {
            o[0] = v.v.x; o[1] = v.v.y; o[2] = v.v.z; o[3] = v.v.w;
        } else {
            o[0] = v.a.x; o[1] = v.a.y; o[2] = v.b.x; o[3] = v.b.y;
        }
        o[4] = pf[e];
    }
    // ---- out tile -> obs[env0 : env0+nvalid] (contiguous): one bulk async store
    const size_t out_bytes = (size_t)nrows * 5 * sizeof(OutT);
    OutT *dst = obs + (size_t)env0 * W * 5;
    if ((out_bytes & 15) == 0) {
        fence_proxy_async_smem(); // generic-proxy smem writes -> visible to the async proxy
        __syncthreads();
        if (tid == 0) {
            bulk_store(dst, smem_u32(out_tile), (uint32_t)out_bytes);
            bulk_commit();
            bulk_wait_read_all(); // smem must outlive the read side of the store
        }
    } else { // ragged tail block whose byte count is not a multiple of 16
        __syncthreads();
        for (int f = tid; f < nrows * 5; f += blockDim.x) dst[f] = out_tile[f];
    }
}

// ------------------------------------------------------------------------------------------
// pipe variant: persistent, warp-specialised (the fast path; windows up to 512 rows)
//
// One block per SM loops over tiles of TE consecutive envs.  Roles:
//   bookkeeper warps (kPipeBook): one lane per env at full lane utilisation; run the per-env arithmetic and
//       publish {row0, position feature} of a tile into a ring of Q descriptors (mbarriers desc_full /
//       desc_free).  They run up to Q tiles ahead, so their load -> lookup -> load -> arithmetic latency
//       chain is off the critical path.
//   mover warps (kPipeMove): gather the tile's window rows with coalesced 16-byte loads straight into
//       registers (RPT rows per thread, the loads of tile t+1 are issued before tile t is written, so
//       their L2/HBM latency hides behind a whole tile of work), interleave the position feature while
//       storing into the out ring (conflict-free stride-5 STS), and one thread issues ONE bulk async store
//       (UBLKCP.G.S) per tile; up to S_OUT stores stay in flight.
// History (profiles/r01_pipe_*.txt): a first version fetched every env's window with its own bulk async
// copy into an in-ring; ncu showed the block pinned on the copy-issue loop — one UBLKCP per ~85 cycles
// per SM whatever the stage counts (7085 copies per SM per step => 0.32 ms floor), the same wall the
// tile variant hits.  Register gathers have no such per-copy cost and halve the shared-memory traffic.
// ------------------------------------------------------------------------------------------
#ifndef FE_PIPE_BOOK
#define FE_PIPE_BOOK 6
#endif
#ifndef FE_PIPE_MOVE
#define FE_PIPE_MOVE 8
#endif
#ifndef FE_PIPE_SOUT
#define FE_PIPE_SOUT 2
#endif
#ifndef FE_PIPE_SIN
#define FE_PIPE_SIN 4   /* in-ring stages of the "stream" flavour (series larger than L2) */
#endif
#ifndef FE_PIPE_RPT
#define FE_PIPE_RPT 8   /* f32 rows per mover thread per tile (f64: half) */
#endif
constexpr int kPipeBook = FE_PIPE_BOOK;
constexpr int kPipeMove = FE_PIPE_MOVE;
constexpr int kPipeThreads = (kPipeBook + kPipeMove) * 32;
constexpr int kMovers = kPipeMove * 32;
constexpr int kPipeQ = 8;                // descriptor ring depth
constexpr int kPipeSOut = FE_PIPE_SOUT;  // out-tile stages
// Two flavours, chosen per launch from the size of the log-return table (pick_pipe_stages):
//   kSIn == 0  "cached": the table is L2-resident, one tile of register prefetch covers the L2 latency and the
//              rows never touch shared memory on the way in (measured c2: 0.28 ms vs 0.35 ms for kSIn == 3);
//   kSIn  > 0  "stream": the table lives in HBM; rows arrive through an in-ring of kSIn stages filled with
//              16-byte cp.async (LDGSTS), ~kSIn x 30 KB in flight per SM (measured c4: 0.376 ms vs 0.43 ms).
constexpr int kPipeSInStream = FE_PIPE_SIN;
template <typename OutT> struct PipeRows { static constexpr int value = sizeof(OutT) == 4 ? FE_PIPE_RPT : (FE_PIPE_RPT + 1) / 2; }; // rows / thread / tile

// smem: [mbarriers desc_full[Q], desc_free[Q], in_full[S_IN]] (256 B) [descriptors Q x TE x (8 + 8) B]
//       [in ring S_IN x TE*W*4 OutT] [out ring S_OUT x TE*W*5 OutT]
template <typename OutT> __host__ __device__ inline size_t pipe_smem_bytes(int TE, int W, int sin) {
    return 256 + (size_t)kPipeQ * TE * 16 + (size_t)TE * W * sizeof(OutT) * (4 * sin + 5 * kPipeSOut);
}
// 16-byte async copy global -> shared (LDGSTS), and "arrive on the mbarrier once my copies have landed"
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ Row4<float> ldg_row(const Row4<float> *p) {
    Row4<float> r;
    r.v = __ldg(reinterpret_cast<const float4 *>(p));
    return r;
}
__device__ __forceinline__ Row4<double> ldg_row(const Row4<double> *p) {
    Row4<double> r;
    r.a = __ldg(reinterpret_cast<const double2 *>(p));
    r.b = __ldg(reinterpret_cast<const double2 *>(p) + 1);
    return r;
}

template <typename OutT, bool kObserve, int kPipeSIn>
__global__ void __launch_bounds__(kPipeThreads, 1)
fe_pipe_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const float *__restrict__ actions,
               OutT *__restrict__ obs, OutT *__restrict__ rewards, int32_t *__restrict__ dones, FeStats *stats,
               const uint64_t step_arg, const uint64_t *__restrict__ step_dev, const int TE) {
    constexpr int RPT = PipeRows<OutT>::value;
    extern __shared__ __align__(128) unsigned char smem[];
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int W = p.window;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles_all = (p.num_envs + TE - 1) / TE;
    const int ntiles = (int)((ntiles_all - blockIdx.x + gridDim.x - 1) / gridDim.x); // tiles blockIdx.x, +gridDim.x, ...
    const uint32_t bars = smem_u32(smem);
    auto desc_full = [&](int q) { return bars + 8u * q; };
    auto desc_free = [&](int q) { return bars + 8u * (kPipeQ + q); };
    auto in_full = [&](int si) { return bars + 8u * (2 * kPipeQ + si); };
    int64_t *d_row0 = reinterpret_cast<int64_t *>(smem + 256);                       // [Q][TE]
    double *d_pf = reinterpret_cast<double *>(smem + 256 + (size_t)kPipeQ * TE * 8); // [Q][TE], OutT in the low bytes
    const size_t in_stage = (size_t)TE * W * 4 * sizeof(OutT), out_stage = (size_t)TE * W * 5 * sizeof(OutT);
    unsigned char *in_ring = smem + 256 + (size_t)kPipeQ * TE * 16;
    unsigned char *out_ring = in_ring + kPipeSIn * in_stage;

    if (tid == 0) {
        for (int q = 0; q < kPipeQ; ++q) { mbar_init(desc_full(q), 1); mbar_init(desc_free(q), 1); }
        for (int si = 0; si < kPipeSIn; ++si) mbar_init(in_full(si), kMovers);
        mbar_fence_init();
    }
    __syncthreads();

    if (warp < kPipeBook) {
        // ------------------------------------------------------------------ bookkeepers
        // Zero-copy launches (fe_step_host: the actions sit in mapped host memory, k.rewards_mirror is set): the action and
        // state loads of this warp's NEXT tile are issued before the current tile's arithmetic, which takes the ~2 us PCIe
        // read out of every tile's dependency chain (as in the gather kernel, where it is measured).
        const bool ahead = !kObserve && k.rewards_mirror != nullptr;
        auto tile_env = [&](int t) { return ((int64_t)blockIdx.x + (int64_t)t * gridDim.x) * TE + lane; };
        auto tile_active = [&](int t) { return t < ntiles && lane < TE && tile_env(t) < p.num_envs; };
        EnvLoads ld, ld_next;
        ld.seg = 0; ld.ptr = 0; ld.cash = 0.0f; ld.lng = 0.0f; ld.sht = 0.0f; ld.act = 0.0f; ld.margin = 0.0;
        ld_next = ld;
        if (ahead && tile_active(warp)) ld = env_load_state(st, actions, tile_env(warp));
        for (int t = warp; t < ntiles; t += kPipeBook) {
            const int q = t % kPipeQ;
            if (ahead && tile_active(t + kPipeBook)) ld_next = env_load_state(st, actions, tile_env(t + kPipeBook));
            mbar_wait(desc_free(q), ((t / kPipeQ) & 1) ^ 1); // first lap passes immediately
            const int64_t env0 = ((int64_t)blockIdx.x + (int64_t)t * gridDim.x) * TE;
            const int nvalid = (int)min((int64_t)TE, p.num_envs - env0);
            EnvResult r;
            r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0; r.row0 = 0; r.posfeat = 0.0;
            const bool active = lane < nvalid;
            if (active) {
                const int64_t i = env0 + lane;
                if (kObserve) r = env_observe(p, s, st, k, i);
                else {
                    if (!ahead) ld = env_load_state(st, actions, i);
                    r = env_compute<OutT>(p, s, st, k, i, ld, env_load_bar(p, s, ld), rewards, dones, stats != nullptr, step);
                }
                d_row0[q * TE + lane] = r.row0;
                reinterpret_cast<OutT *>(d_pf + q * TE)[lane] = (OutT)r.posfeat;
            }
            ld = ld_next;
            if (!kObserve && k.dones_bits_out) { // only set when TE == 32: the tile is one word of the bit-packed dones
                const unsigned word = __ballot_sync(0xFFFFFFFFu, active && r.done);
                if (lane == 0) k.dones_bits_out[env0 >> 5] = word;
            }
            if (!kObserve) accumulate_stats(stats, r, active);
            __syncwarp();
            if (lane == 0) mbar_arrive(desc_full(q)); // release: descriptor visible to the movers
        }
    } else {
        // ------------------------------------------------------------------ movers
        const int mtid = tid - kPipeBook * 32;
        int e_u[RPT], j_u[RPT]; // tile row mtid + u*kMovers = window row j_u of env e_u: the same in every tile
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            e_u[u] = (mtid + u * kMovers) / W;
            j_u[u] = (mtid + u * kMovers) - e_u[u] * W;
        }
        const Row4<OutT> *series_rows = reinterpret_cast<const Row4<OutT> *>(s.logret);
        auto tile_rows = [&](int t) {
            const int64_t env0 = ((int64_t)blockIdx.x + (int64_t)t * gridDim.x) * TE;
            return (int)min((int64_t)TE, p.num_envs - env0) * W;
        };
        // fetch tile t's rows: row r of the tile = env r / W, window row r % W.  Either straight into registers
        // (kPipeSIn == 0) or with 16-byte async copies into in-ring stage t % S_IN, arriving on in_full when landed.
        auto gather = [&](int t, Row4<OutT>(&buf)[RPT]) {
            const int q = t % kPipeQ;
            mbar_wait(desc_full(q), (t / kPipeQ) & 1);
            const int nrows = tile_rows(t);
            const uint32_t stage = kPipeSIn > 0 ? smem_u32(in_ring + (t % (kPipeSIn > 0 ? kPipeSIn : 1)) * in_stage) : 0u;
#pragma unroll
            for (int u = 0; u < RPT; ++u) {
                const int r = mtid + u * kMovers;
                if (r < nrows) {
                    const Row4<OutT> *src = series_rows + d_row0[q * TE + e_u[u]] + j_u[u];
                    if constexpr (kPipeSIn == 0) {
                        buf[u] = ldg_row(src);
                    } else {
                        cp_async16(stage + (uint32_t)r * sizeof(Row4<OutT>), src);
                        if constexpr (sizeof(OutT) == 8)
                            cp_async16(stage + (uint32_t)r * sizeof(Row4<OutT>) + 16, reinterpret_cast<const char *>(src) + 16);
                    }
                }
            }
            if constexpr (kPipeSIn > 0) cp_async_arrive_noinc(in_full(t % (kPipeSIn > 0 ? kPipeSIn : 1)));
        };
        Row4<OutT> cur[RPT], nxt[RPT];
        constexpr int kAhead = kPipeSIn > 0 ? kPipeSIn : 1;
        if constexpr (kPipeSIn == 0) {
            if (ntiles > 0) gather(0, cur);
        } else {
            for (int t = 0; t < kAhead && t < ntiles; ++t) gather(t, nxt);
        }
        for (int t = 0; t < ntiles; ++t) {
            const int q = t % kPipeQ, so = t % kPipeSOut;
            const int64_t env0 = ((int64_t)blockIdx.x + (int64_t)t * gridDim.x) * TE;
            const int nrows = tile_rows(t);
            if constexpr (kPipeSIn == 0) {
                if (t + 1 < ntiles) gather(t + 1, nxt); // in flight while this tile is written
            } else {
                mbar_wait(in_full(t % kAhead), (t / kAhead) & 1);
                const Row4<OutT> *in_rows = reinterpret_cast<const Row4<OutT> *>(in_ring + (t % kAhead) * in_stage);
#pragma unroll
                for (int u = 0; u < RPT; ++u) {
                    const int r = mtid + u * kMovers;
                    if (r < nrows) cur[u] = in_rows[r];
                }
            }
            if (t >= kPipeSOut) { // the store that last used out[so] must have finished reading shared memory
                if (mtid == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPipeSOut - 1) : "memory");
                named_bar_sync(1, kMovers);
            }
            OutT *out_tile = reinterpret_cast<OutT *>(out_ring + so * out_stage);
            const OutT *pf = reinterpret_cast<const OutT *>(d_pf + q * TE);
#pragma unroll
            for (int u = 0; u < RPT; ++u) {
                const int r = mtid + u * kMovers;
                if (r < nrows) {
                    OutT *o = out_tile + (size_t)r * 5;
                    if constexpr (sizeof(OutT) == 4) {
                        o[0] = cur[u].v.x; o[1] = cur[u].v.y; o[2] = cur[u].v.z; o[3] = cur[u].v.w;
                    } else {
                        o[0] = cur[u].a.x; o[1] = cur[u].a.y; o[2] = cur[u].b.x; o[3] = cur[u].b.y;
                    }
                    o[4] = pf[e_u[u]];
                }
            }
            const size_t out_bytes = (size_t)nrows * 5 * sizeof(OutT);
            OutT *dst = obs + (size_t)env0 * W * 5;
            if ((out_bytes & 15) == 0) {
                fence_proxy_async_smem();
                named_bar_sync(1, kMovers); // out tile complete, descriptor consumed
                if (mtid == 0) {
                    bulk_store_hint(dst, smem_u32(out_tile), (uint32_t)out_bytes, l2_policy_evict_first());
                    bulk_commit();
                }
            } else { // ragged last tile
                named_bar_sync(1, kMovers);
                for (int f = mtid; f < nrows * 5; f += kMovers) dst[f] = out_tile[f];
                named_bar_sync(1, kMovers);
            }
            if constexpr (kPipeSIn == 0) {
                if (mtid == 0) mbar_arrive(desc_free(q));
#pragma unroll
                for (int u = 0; u < RPT; ++u) cur[u] = nxt[u];
            } else {
                // the barrier above also means every mover finished reading in-stage t % S_IN: refill it, and only
                // then release the descriptor (the refill of tile t+S_IN reads ITS descriptor, not this one)
                if (mtid == 0) mbar_arrive(desc_free(q));
                if (t + kAhead < ntiles) gather(t + kAhead, nxt);
            }
        }
        if (mtid == 0) bulk_wait_read_all();
    }
}

// ------------------------------------------------------------------------------------------
// gather variant: the window gather done by the TMA engine (round 2; the fast path when the series is L2-resident).
//
// Read side.  cp.async.bulk.tensor ... tile::gather4 (SASS UTMALDG.2D.GATHER4) fetches FOUR rows of a 2-D tensor, chosen
// by row index, with one instruction.  The tensor map used here has a row pitch (80 B) far smaller than its row length
// (one whole window): "row i" is the window that starts at series row i, so ONE instruction brings the windows of
// four consecutive envs into shared memory.  The table it reads is the series in OBSERVATION layout — 5 values per
// row, the four log-returns plus a hole for the position feature — so the bytes land exactly as the (N, W, 5) tensor
// wants them and the only thing threads still write is the position-feature column (W values per env).  Window
// starts must be 16-byte aligned for the TMA engine and a 20-byte row is not: the table holds P = 4 (f32; 2 for f64)
// copies shifted by one row each, copy k serving the windows whose first row is k mod P (fe_obs_table_build; 20.6 MB
// for the 258 k-row series of BASELINE config 2, L2-resident).
// Write side.  One bulk async store (UBLKCP.G.S) per 4-env unit, straight from the slot the gather filled.
// Why this shape (tools/tma_rate_probe.cu, tools/tma_gather_probe.cu, profiles/r02_*): a thread pays ~470 cycles of
// issue latency per TMA load whatever its size, but loads issued by DIFFERENT warps overlap (1 warp: 750 cycles per
// gather4, 8 warps: 110, 16 warps: 72 = 67 B/clk/SM), so the movers are many warps with one small unit each rather
// than one producer with big tiles; shared-memory destinations of tensor copies must be 128-byte aligned, which is why
// a unit is one gather4 (4 x 20W bytes, padded to a 128-byte pitch) and leaves with its own store.
// Roles per block (one block per SM, persistent):
//   bookkeeper warps (kGaBook)  as in the pipe variant: one lane per env runs env_step(), publishes
//                               {tensor row index, position feature} of a 32-env tile into a ring of kGaQ descriptors;
//   mover warps (kGaMove)       warp-autonomous, no block-wide barrier anywhere: mover m owns units m, m + kGaMove, ...
//                               (unit u = tile u / 8, group u % 8) and a private ring of S slots.  Per unit: wait for the
//                               slot's mbarrier (gather landed) -> 4W position-feature stores -> proxy fence -> lane 0
//                               issues the bulk store, releases the descriptor, waits until the store has read the slot
//                               and issues the gather of unit i + S into it.
// ------------------------------------------------------------------------------------------
#ifndef FE_GATHER_BOOK
#define FE_GATHER_BOOK 6 /* measured c2: 6 -> 0.2525 ms, 8 -> 0.2655 ms (profiles/r02_gather_allwait.txt) */
#endif
#ifndef FE_GATHER_MOVE
#define FE_GATHER_MOVE 12
#endif
#ifndef FE_GATHER_STAGES
#define FE_GATHER_STAGES 3 /* slots per mover when they fit (else 2) */
#endif
#ifndef FE_GATHER_FLUSH_SPINS
#define FE_GATHER_FLUSH_SPINS 2000 /* x 100 ns: how long a block waits for the grid's bookkeeping before it leaves the packed dones to the last block out */
#endif
constexpr int kGaBook = FE_GATHER_BOOK;
constexpr int kGaMove = FE_GATHER_MOVE;
constexpr int kGaThreads = (kGaBook + kGaMove) * 32;
constexpr int kGaQ = 32;          // descriptor ring depth in tiles (movers keep a descriptor until its unit is stored)
constexpr int kGaMaxStages = 4;
constexpr int kGaBarBytes = 1280; // desc_full[Q], desc_free[Q], full[kGaMove][kGaMaxStages]; last 16 bytes: claim lock + sequence
constexpr int kGaPitch = 80;      // tensor row pitch of the observation-layout table: P * row bytes for both dtypes

static_assert((2 * kGaQ + kGaMove * kGaMaxStages) * 8 + 16 <= kGaBarBytes, "mbarrier area too small");
__host__ __device__ inline int ga_row_bytes(bool f64) { return f64 ? 40 : 20; }
__host__ __device__ inline int ga_phase_shift(bool f64) { return f64 ? 1 : 2; } // log2 P, P = 16 / gcd(16, row bytes)
// tensor rows per shifted copy: enough for every window start, plus slack so that the last windows stay inside the copy
__host__ __device__ inline int64_t ga_rows_per_phase(int64_t num_rows, int W, bool f64) {
    const int P = 1 << ga_phase_shift(f64);
    return (num_rows + P - 1) / P + (W + P - 1) / P + 8;
}
__host__ __device__ inline size_t ga_table_bytes(int64_t num_rows, int W, bool f64) {
    return (size_t)(1 << ga_phase_shift(f64)) * (size_t)ga_rows_per_phase(num_rows, W, f64) * kGaPitch + 4096;
}
// A TMA box row is at most 256 8-byte elements and a multiple of 16 bytes.  Windows of up to 2048 bytes are one box row
// (one gather4 = the windows of 4 envs).  Longer windows — 60 rows of f64, the reference's own dtype, are 2400 bytes — are
// fetched in TWO parts: the second half of a window is the tensor row (half window bytes / 80) pitches further on, so one
// gather4 with the indices (a, a + d, b, b + d) lands the complete windows of 2 envs contiguously; units are then 2 envs.
// That needs half a window to be a whole number of pitches.  0 = this window has no gather variant.
__host__ __device__ inline int ga_parts(int W, bool f64) {
    const int wb = ga_row_bytes(f64) * W;
    if (W <= 0 || (wb % 16) != 0) return 0;
    if (wb <= 2048) return 1;
    if (wb <= 4096 && ((wb / 2) % kGaPitch) == 0 && W <= 128) return 2; // W <= 128: four rounds of position-feature stores
    return 0;
}
__host__ __device__ inline bool ga_window_ok(int W, bool f64) { return ga_parts(W, f64) != 0; }
__host__ __device__ inline uint32_t ga_slot_pitch(int W, bool f64) { // one unit: 4 envs (one part) or 2 envs (two parts)
    const int parts = ga_parts(W, f64);
    return ((4u / (uint32_t)(parts ? parts : 1)) * ga_row_bytes(f64) * W + 127u) & ~127u;
}
template <typename OutT> __host__ __device__ inline size_t gather_desc_bytes() { // tile id + 32 x {row index, feature} per slot
    return ((size_t)kGaQ * (4 + 32 * (4 + sizeof(OutT))) + 127) & ~(size_t)127;
}
template <typename OutT> __host__ __device__ inline size_t gather_smem_bytes(int W, int S) {
    return kGaBarBytes + gather_desc_bytes<OutT>() + (size_t)kGaMove * S * ga_slot_pitch(W, sizeof(OutT) == 8);
}

__device__ __forceinline__ void tma_gather4(uint32_t dst_smem, const CUtensorMap *map, int r0, int r1, int r2, int r3, uint32_t bar,
                                            uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%2, %3, %4, %5, %6}], [%7], %8;"
        ::"r"(dst_smem), "l"(map), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar), "l"(policy)
        : "memory");
}

#ifdef FE_GATHER_CLOCKS
// experiment builds: cycles spent per phase by block 0's mover 0 / bookkeeper 0 (tools/gather_clocks.py)
__device__ unsigned long long fe_gather_clk[16];
__device__ unsigned long long fe_gather_block_ns[3 * 160]; // per block: start, all movers done, smid (globaltimer ns)
__device__ __forceinline__ unsigned long long ga_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define GA_CLK(var) const long long var = clock64()
#define GA_ACC(slot, a, b) acc[slot] += (b) - (a)
#else
#define GA_CLK(var)
#define GA_ACC(slot, a, b)
#endif

template <typename OutT, bool kObserve, int kParts>
__global__ void __launch_bounds__(kGaThreads, 1)
fe_gather_kernel(const __grid_constant__ CUtensorMap tmap, const FeParams p, const FeSeries s, const FeState st, const Consts k,
                 const float *__restrict__ actions, OutT *__restrict__ obs, OutT *__restrict__ rewards,
                 int32_t *__restrict__ dones, FeStats *stats, const uint64_t step_arg, const uint64_t *__restrict__ step_dev,
                 const int S, const int rows_per_phase, unsigned int *__restrict__ sched) {
    constexpr bool kF64 = sizeof(OutT) == 8;
    constexpr int kUnitEnvs = 4 / kParts;        // envs per unit (one gather4, one bulk store)
    constexpr int kTileUnits = 32 / kUnitEnvs;   // units per 32-env tile: 8 or 16
    constexpr int kUnitShift = kParts == 1 ? 3 : 4;
    static_assert(kParts == 1 || kParts == 2, "a window is fetched in one or two parts");
    extern __shared__ __align__(128) unsigned char smem[];
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int W = p.window;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ntiles_all = (int)((p.num_envs + 31) / 32);
    const uint32_t bars = smem_u32(smem);
    auto desc_full = [&](int q) { return bars + 8u * q; };
    auto desc_free = [&](int q) { return bars + 8u * (kGaQ + q); };
    auto slot_full = [&](int m, int si) { return bars + 8u * (2 * kGaQ + m * kGaMaxStages + si); };
    unsigned int *claim = reinterpret_cast<unsigned int *>(smem + kGaBarBytes - 16);         // [0] lock, [1] next sequence number
    int32_t *d_tile = reinterpret_cast<int32_t *>(smem + kGaBarBytes);                         // [Q] tile id, -1 = no more tiles
    int32_t *d_row = d_tile + kGaQ;                                                            // [Q][32] tensor row index
    OutT *d_pf = reinterpret_cast<OutT *>(smem + kGaBarBytes + (size_t)kGaQ * (4 + 32 * 4));   // [Q][32]
    unsigned char *ring = smem + kGaBarBytes + gather_desc_bytes<OutT>();
    const uint32_t pitch = ga_slot_pitch(W, kF64);

#ifdef FE_GATHER_CLOCKS
    if (tid == 0 && blockIdx.x < 160) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        fe_gather_block_ns[3 * blockIdx.x] = ga_globaltimer();
        fe_gather_block_ns[3 * blockIdx.x + 2] = smid;
        fe_gather_block_ns[3 * blockIdx.x + 1] = 0;
    }
#endif
    if (tid == 0) {
        for (int q = 0; q < kGaQ; ++q) { mbar_init(desc_full(q), 1); mbar_init(desc_free(q), kTileUnits); }
        for (int m = 0; m < kGaMove; ++m)
            for (int si = 0; si < kGaMaxStages; ++si) mbar_init(slot_full(m, si), 1);
        claim[0] = 0; claim[1] = 0;
        mbar_fence_init();
    }
    __syncthreads();

    if (warp < kGaBook) {
        // ------------------------------------------------------------------ bookkeepers
        // Tiles are CLAIMED, not pre-assigned: SMs differ by ~15 % in how fast they move this traffic (position relative
        // to the L2 slices / the two dies), and with a static round-robin the slowest SM set the kernel time (232 ... 273 us
        // per block, profiles/r02_gather_sweeps.txt, sweep 5).  A claim = (next sequence number of this block, next tile of the
        // grid), taken together under a block-local lock so that sequence order = tile order: once a sequence slot says
        // "no more tiles", every later one does.
        const int shift = ga_phase_shift(kF64);
#ifdef FE_GATHER_CLOCKS
        long long acc[16] = {0};
        int ntl = 0;
#endif
        // With the actions in mapped host memory (fe_step_host: k.rewards_mirror is set) the action load is a PCIe read of
        // ~2 us.  There a claim is taken one tile AHEAD of the tile being computed and the first-hop loads of the claimed
        // tile (action and per-env state) are issued at once, in flight while the current tile is computed, so that the
        // read no longer sits in every tile's dependency chain (measured c2, 1 Mi envs, zero-copy: kernel 0.253 -> 0.2305 ms,
        // the device-resident time; profiles/r02_e2e_probes.txt, call 3).  Device-resident launches claim tile by tile: holding
        // a second claim cost them 0.5 % (tail balance).
        const bool ahead = !kObserve && k.rewards_mirror != nullptr;
        auto take_claim = [&](int &n, int &t) { // sequence slot of this block, tile of the grid (>= ntiles_all: none left)
            n = 0; t = 0;
            if (lane == 0) {
                while (atomicCAS(&claim[0], 0u, 1u) != 0u) {}
                n = (int)claim[1];
                claim[1] = (unsigned)n + 1;
                t = (int)atomicAdd(&sched[0], 1u);
                __threadfence_block();
                atomicExch(&claim[0], 0u);
            }
            n = __shfl_sync(0xFFFFFFFFu, n, 0);
            t = __shfl_sync(0xFFFFFFFFu, t, 0);
        };
        auto first_hop = [&](int t, EnvLoads &ld) {
            const int64_t i = (int64_t)t * 32 + lane;
            if (!kObserve && t < ntiles_all && i < p.num_envs) ld = env_load_state(st, actions, i);
        };
        int n, t, n_next = 0, t_next = 0;
        EnvLoads ld, ld_next;
        ld.seg = 0; ld.ptr = 0; ld.cash = 0.0f; ld.lng = 0.0f; ld.sht = 0.0f; ld.act = 0.0f; ld.margin = 0.0;
        ld_next = ld;
        take_claim(n, t);
        first_hop(t, ld);
        for (;;) {
            const int q = n & (kGaQ - 1);
            if (ahead && t < ntiles_all) { // the next claim and its loads, before this tile's wait and arithmetic
                take_claim(n_next, t_next);
                first_hop(t_next, ld_next);
            }
            GA_CLK(c0);
            if (lane == 0) mbar_wait(desc_free(q), ((n / kGaQ) & 1) ^ 1); // first lap passes immediately
            __syncwarp();
            GA_CLK(c1);
            GA_ACC(8, c0, c1);
            if (t >= ntiles_all) { // nothing left: tell the movers and stop
                if (lane == 0) { d_tile[q] = -1; mbar_arrive(desc_full(q)); }
                break;
            }
            const int64_t i = (int64_t)t * 32 + lane;
            const bool active = i < p.num_envs;
            EnvResult r;
            r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0; r.row0 = 0; r.posfeat = 0.0;
            if (active) {
                if (kObserve) r = env_observe(p, s, st, k, i);
                else r = env_compute<OutT>(p, s, st, k, i, ld, env_load_bar(p, s, ld), rewards, dones, stats != nullptr, step);
            }
            // window starting at series row row0 = copy (row0 mod P), tensor row (row0 div P) of that copy
            d_row[q * 32 + lane] = (int32_t)((r.row0 & ((1 << shift) - 1)) * rows_per_phase + (r.row0 >> shift));
            d_pf[q * 32 + lane] = (OutT)r.posfeat;
            if (lane == 0) d_tile[q] = t;
            if (!kObserve && k.dones_bits_out) { // tile t = envs [32t, 32t + 32) = word t of the bit-packed dones
                const unsigned word = __ballot_sync(0xFFFFFFFFu, active && r.done);
                if (lane == 0) k.dones_bits_out[t] = word;
            }
            if (!kObserve) accumulate_stats(stats, r, active);
            __syncwarp();
            if (lane == 0) mbar_arrive(desc_full(q)); // release: descriptor visible to the movers
            GA_CLK(c2);
            GA_ACC(9, c1, c2);
#ifdef FE_GATHER_CLOCKS
            ++ntl;
#endif
            if (ahead) { n = n_next; t = t_next; ld = ld_next; }
            else { take_claim(n, t); first_hop(t, ld); }
        }
        // Bit-packed dones (fe_step_host_packed): the words sit in the staging buffer; once EVERY bookkeeper warp of the grid
        // has finished (counter sched[2]; the grid is persistent, one block per SM, so waiting on it cannot deadlock) each
        // block sends its 1 / gridDim.x share to the host as full 128-byte lines — the movers are still draining their
        // last units meanwhile.  (One block sending all 128 KB took 8 us of tail: a single SM's stores to system memory.)
        if (!kObserve && k.dones_bits_host) {
            if (lane == 0) {
                __threadfence();
                atomicAdd(&sched[2], 1u);
            }
            if (warp == 0) {
                // The wait normally lasts a few microseconds (the tile counter runs out for every block at the same moment).
                // Should part of the grid not be resident (fewer SMs available than the device reports), the blocks that
                // are would wait for blocks that cannot start: after ~0.2 ms the block gives up, flags it in sched[3], and
                // the last block out — by then every word is staged — sends everything.
                int ok = 1;
                if (lane == 0) {
                    const unsigned want = gridDim.x * (unsigned)kGaBook;
                    int spins = 0;
                    while (ld_acquire_gpu(&sched[2]) < want) {
                        if (++spins > FE_GATHER_FLUSH_SPINS) { ok = 0; break; }
                        __nanosleep(100);
                    }
                    if (!ok) atomicOr(&sched[3], 1u);
                }
                ok = __shfl_sync(0xFFFFFFFFu, ok, 0);
                const int per = (((ntiles_all + (int)gridDim.x - 1) / (int)gridDim.x) + 31) & ~31; // whole lines per block
                const int w_begin = (int)blockIdx.x * per;
                const int w_end = !ok ? w_begin : w_begin + per < ntiles_all ? w_begin + per : ntiles_all;
                constexpr int kBatch = 8; // loads in batches ahead of the stores: one L2 round trip per batch, not per word
                for (int w0 = w_begin + lane; w0 < w_end; w0 += kBatch * 32) {
                    uint32_t v[kBatch];
#pragma unroll
                    for (int j = 0; j < kBatch; ++j) v[j] = w0 + 32 * j < w_end ? __ldcg(k.dones_bits_out + w0 + 32 * j) : 0u;
#pragma unroll
                    for (int j = 0; j < kBatch; ++j)
                        if (w0 + 32 * j < w_end) k.dones_bits_host[w0 + 32 * j] = v[j];
                }
            }
        }
#ifdef FE_GATHER_CLOCKS
        if (blockIdx.x == 0 && tid == 0) { fe_gather_clk[8] = acc[8]; fe_gather_clk[9] = acc[9]; fe_gather_clk[10] = ntl; }
#endif
    } else {
        // ------------------------------------------------------------------ movers
#ifdef FE_GATHER_CLOCKS
        long long acc[16] = {0};
        const long long mover_t0 = clock64();
#endif
        const int m = warp - kGaBook;
        const uint32_t row_b = (uint32_t)ga_row_bytes(kF64) * W, unit_b = kUnitEnvs * row_b; // row_b: one window
        const int part_rows = (int)(row_b / 2) / kGaPitch; // two parts: tensor rows from a window's first half to its second
        unsigned char *slots = ring + (size_t)m * S * pitch;
        // position-feature column: env e of a unit owns rows [eW, (e+1)W) of the slot; this lane writes rows eW + lane + 32k
        constexpr int kRounds = (kParts == 1 && kF64) ? 2 : 4; // ceil(W / 32) for the largest W ga_parts() admits (51 / 102 / 128)
        uint32_t round_mask = 0;              // bit k: lane + 32k < W
#pragma unroll
        for (int kk = 0; kk < kRounds; ++kk) round_mask |= (uint32_t)(lane + 32 * kk < W) << kk;
        const uint32_t env_stride = (uint32_t)W * 5; // values per env
        const uint64_t keep = l2_policy_evict_last(), stream_out = l2_policy_evict_first();
        // unit i of this mover = group (m + i * kGaMove) % kTileUnits of the block's sequence slot (m + i * kGaMove) / kTileUnits
        static_assert((kGaQ & (kGaQ - 1)) == 0, "kGaQ must be a power of two");
        int iss_u = m, iss_si = 0; // lane 0: next unit to issue (unit number within the block, slot)
        int issued = 0;            // lane 0: units whose gather has been issued
        bool open = true;          // lane 0: more units may follow (no "no more tiles" slot seen yet)
        auto issue = [&]() {       // lane 0: gather of the next unit into slot iss_si
            const int n = iss_u >> kUnitShift, g = iss_u & (kTileUnits - 1), q = n & (kGaQ - 1);
            GA_CLK(c0);
            mbar_wait(desc_full(q), (n / kGaQ) & 1);
            GA_CLK(c1);
            GA_ACC(4, c0, c1);
            if (d_tile[q] < 0) { open = false; return; }
            int4 rows4;
            if constexpr (kParts == 1) {
                rows4 = *reinterpret_cast<const int4 *>(d_row + q * 32 + 4 * g);
            } else { // (first half, second half) of env 2g, then of env 2g + 1
                const int2 r2 = *reinterpret_cast<const int2 *>(d_row + q * 32 + 2 * g);
                rows4 = make_int4(r2.x, r2.x + part_rows, r2.y, r2.y + part_rows);
            }
#ifdef FE_GATHER_NOLOAD
            if (rows4.x == -12345)
#endif
            {
                mbar_arrive_expect_tx(slot_full(m, iss_si), unit_b);
                tma_gather4(smem_u32(slots + (size_t)iss_si * pitch), &tmap, rows4.x, rows4.y, rows4.z, rows4.w, slot_full(m, iss_si),
                            keep);
            }
#ifdef FE_GATHER_NOLOAD
            mbar_arrive(slot_full(m, iss_si));
#endif
            ++issued;
            iss_u += kGaMove;
            iss_si = iss_si + 1 == S ? 0 : iss_si + 1;
            GA_CLK(c2);
            GA_ACC(5, c1, c2);
        };
        if (lane == 0)
            for (int i = 0; i < S && open; ++i) issue();
        // Per unit: lane 0 waits until the gather has landed (one lane, then __syncwarp: a try_wait run by all 32 lanes on a
        // per-thread address is serialised lane by lane, ~30 cycles each) -> the warp writes the 4W position features ->
        // proxy fence -> lane 0 issues the bulk store, hands the descriptor entries back, waits until the store has read
        // the slot and issues the next gather into it.
        int u = m, si = 0;
        uint32_t slot_phase = 0; // bit si: parity the mover waits for on slot_full(m, si)
        int n_iss = __shfl_sync(0xFFFFFFFFu, issued, 0);
        for (int i = 0; i < n_iss; ++i) {
            const int n = u >> kUnitShift, g = u & (kTileUnits - 1), q = n & (kGaQ - 1);
            GA_CLK(c0);
            if (lane == 0) mbar_wait(slot_full(m, si), (slot_phase >> si) & 1u); // the unit's windows have landed
            __syncwarp();
            GA_CLK(c1);
            GA_ACC(0, c0, c1);
            unsigned char *slot = slots + (size_t)si * pitch;
            const OutT *pf = d_pf + q * 32 + kUnitEnvs * g;
            OutT *col = reinterpret_cast<OutT *>(slot) + 5 * lane + 4; // position-feature slot of row `lane` of env 0
#ifdef FE_GATHER_NOPF
            if (pf[0] == (OutT)12345.678)
#endif
#pragma unroll
            for (int e = 0; e < kUnitEnvs; ++e) {
                const OutT v = pf[e];
#pragma unroll
                for (int kk = 0; kk < kRounds; ++kk)
                    if (round_mask & (1u << kk)) col[e * env_stride + 160 * kk] = v;
            }
            GA_CLK(c1b);
            GA_ACC(1, c1, c1b);
#ifndef FE_GATHER_NOFENCE
            fence_proxy_async_smem(); // generic-proxy writes -> visible to the bulk store
#endif
            __syncwarp();
            GA_CLK(c2);
            GA_ACC(11, c1b, c2);
            if (lane == 0) {
                const int64_t env0 = (int64_t)d_tile[q] * 32 + kUnitEnvs * g;
                const int64_t left = p.num_envs - env0;
                const int nv = left >= kUnitEnvs ? kUnitEnvs : (left > 0 ? (int)left : 0); // fewer only in the ragged last tile
#ifdef FE_GATHER_NOSTORE
                if (nv > 4)
#else
                if (nv > 0)
#endif
                {
                    bulk_store_hint(obs + (size_t)env0 * W * 5, smem_u32(slot), (uint32_t)nv * row_b, stream_out);
                    bulk_commit();
                }
                mbar_arrive(desc_free(q)); // this unit's descriptor entries are consumed
                GA_CLK(c3);
                GA_ACC(2, c2, c3);
                if (open) {
                    bulk_wait_read_all(); // the store has read the slot: refill it
                    GA_CLK(c4);
                    GA_ACC(3, c3, c4);
                    issue();
                }
            }
            __syncwarp();
            n_iss = __shfl_sync(0xFFFFFFFFu, issued, 0); // every issued unit gets stored; none follows once the stream closed
            slot_phase ^= 1u << si;
            u += kGaMove;
            si = si + 1 == S ? 0 : si + 1;
        }
        if (lane == 0) bulk_wait_read_all();
#ifdef FE_GATHER_CLOCKS
        if (lane == 0 && blockIdx.x < 160) atomicMax(&fe_gather_block_ns[3 * blockIdx.x + 1], ga_globaltimer());
        if (blockIdx.x == 0 && m == 0 && lane == 0) { for (int c = 0; c < 6; ++c) fe_gather_clk[c] = acc[c]; fe_gather_clk[6] = issued; fe_gather_clk[11] = acc[11]; fe_gather_clk[12] = 0; fe_gather_clk[13] = clock64() - mover_t0; }
#endif
    }
    // the last block out rewinds the counters for the next launch (every block's claims, and its wait on sched[2], precede
    // its arrival here)
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        unsigned send_all = 0;
        if (atomicAdd(&sched[1], 1u) == gridDim.x - 1) {
            __threadfence();
            send_all = ld_acquire_gpu(&sched[3]);
            sched[0] = 0;
            sched[1] = 0;
            sched[2] = 0;
            sched[3] = 0;
            __threadfence();
        }
        claim[2] = send_all;
    }
    if (!kObserve && k.dones_bits_host) { // only after a block gave up its wait above
        __syncthreads();
        if (claim[2])
            for (int w = tid; w < ntiles_all; w += kGaThreads) k.dones_bits_host[w] = __ldcg(k.dones_bits_out + w);
    }
}

// series (T, 4) -> observation-layout table: P copies of the (T, 5) layout, copy k starting at series row k, placed
// k * 80 * rows_per_phase bytes into the buffer (so that every window start is a multiple of the 80-byte tensor pitch)
template <typename OutT>
__global__ void __launch_bounds__(256)
fe_obs_table_kernel(const OutT *__restrict__ logret, const int64_t num_rows, const int64_t rows_per_phase,
                    unsigned char *__restrict__ table) {
    constexpr bool kF64 = sizeof(OutT) == 8;
    const int shift = ga_phase_shift(kF64);
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t r = idx >> shift;
    const int kk = (int)(idx & ((1 << shift) - 1));
    if (r >= num_rows || r < kk) return;
    OutT *dst = reinterpret_cast<OutT *>(table + (size_t)kk * kGaPitch * rows_per_phase + (size_t)(r - kk) * ga_row_bytes(kF64));
    const OutT *src = logret + r * 4;
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
    dst[4] = (OutT)0; // the hole the movers fill with the position feature
}

// ------------------------------------------------------------------------------------------
// direct variant: any window; thread-per-env bookkeeping, then warp-per-env copy
// ------------------------------------------------------------------------------------------
template <typename OutT, bool kObserve>
__global__ void __launch_bounds__(kThreads)
fe_direct_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const float *__restrict__ actions,
                 OutT *__restrict__ obs, OutT *__restrict__ rewards, int32_t *__restrict__ dones, FeStats *stats,
                 const uint64_t step_arg, const uint64_t *__restrict__ step_dev) {
    __shared__ int64_t sh_row0[kThreads];
    const uint64_t step = step_dev ? *step_dev : step_arg;
    __shared__ OutT sh_pf[kThreads];
    const int W = p.window;
    const int tid = threadIdx.x;
    const int64_t env0 = (int64_t)blockIdx.x * kThreads;
    const int nvalid = (int)min((int64_t)kThreads, p.num_envs - env0);
    const bool active = tid < nvalid;
    EnvResult r;
    r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0; r.row0 = 0; r.posfeat = 0.0;
    if (active) {
        const int64_t i = env0 + tid;
        if (kObserve) r = env_observe(p, s, st, k, i);
        else r = env_step<OutT>(p, s, st, k, i, actions, rewards, dones, stats != nullptr, step);
    }
    sh_row0[tid] = r.row0;
    sh_pf[tid] = (OutT)r.posfeat;
    if (!kObserve) accumulate_stats(stats, r, active);
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5;
    const OutT *lr = reinterpret_cast<const OutT *>(s.logret);
    const int nvals = W * 5;
    for (int e = warp; e < nvalid; e += kThreads / 32) {
        const OutT *src = lr + sh_row0[e] * 4;
        OutT *dst = obs + (size_t)(env0 + e) * nvals;
        const OutT pfe = sh_pf[e];
        for (int f = lane; f < nvals; f += 32) {
            const int j = f / 5, c = f - j * 5;
            dst[f] = c == 4 ? pfe : __ldg(src + j * 4 + c);
        }
    }
}

// ------------------------------------------------------------------------------------------
// lazy variant: the step WITHOUT materialising the observation.  An observation of this env is fully described by
// (row0, position feature): obs[i, j, 0:4] = logret[row0[i] + j], obs[i, j, 4] = posfeat[i] (:437-445, :428-434).
// Consumers that read the window straight from the staged series (the fused ES policy kernel, fe_es.cu) take the
// 12-byte handle instead of the W x 20-byte tensor; fe_materialize turns a handle into the tensor.
// ------------------------------------------------------------------------------------------
template <typename OutT, bool kObserve>
__global__ void __launch_bounds__(kThreads)
fe_lazy_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const float *__restrict__ actions,
               int64_t *__restrict__ row0_out, OutT *__restrict__ pf_out, OutT *__restrict__ rewards,
               int32_t *__restrict__ dones, FeStats *stats, const uint64_t step_arg, const uint64_t *__restrict__ step_dev) {
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const bool active = i < p.num_envs;
    EnvResult r;
    r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0; r.row0 = 0; r.posfeat = 0.0;
    if (active) {
        if (kObserve) r = env_observe(p, s, st, k, i);
        else r = env_step<OutT>(p, s, st, k, i, actions, rewards, dones, stats != nullptr, step);
        row0_out[i] = r.row0;
        pf_out[i] = (OutT)r.posfeat;
    }
    if (!kObserve) accumulate_stats(stats, r, active);
}

// handles -> tensor (fe_gather_obs, LSU path): warp per sample, same element order as the direct variant; sample b is
// handle index[b] (index == NULL: handle b)
template <typename OutT>
__global__ void __launch_bounds__(kThreads)
fe_materialize_kernel(const int64_t N, const int W, const OutT *__restrict__ logret, const int64_t *__restrict__ row0,
                      const OutT *__restrict__ pf, const int64_t *__restrict__ index, OutT *__restrict__ obs) {
    const int lane = threadIdx.x & 31;
    const int64_t e = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
    if (e >= N) return;
    const int64_t h = index ? index[e] : e;
    const OutT *src = logret + row0[h] * 4;
    OutT *dst = obs + (size_t)e * W * 5;
    const OutT pfe = pf[h];
    for (int f = lane; f < W * 5; f += 32) {
        const int j = f / 5, c = f - j * 5;
        dst[f] = c == 4 ? pfe : __ldg(src + j * 4 + c);
    }
}

// handles -> tensor (fe_gather_obs, TMA path): the gather variant's movers without its bookkeepers.  Every warp is
// autonomous: it owns the 32-sample tiles gw, gw + NW, ... (gw = global warp id, NW = warps in the grid) and a private
// ring of S slots.  Lane l of the warp holds the handle of sample l of the tile being stored (as {tensor row index,
// position feature}) and, loaded one tile ahead, of the next one.  A unit = one gather4 = 4 samples (2 for windows
// fetched in two parts); per unit: wait for the slot's mbarrier -> the position-feature column -> proxy fence -> one
// bulk store of the unit's contiguous output bytes -> (once the store has read the slot) the gather of unit i + S.
// In the ragged last tile the missing samples repeat the last valid handle, so a gather4 always has 4 valid rows, and
// the store covers only the valid samples.
constexpr int kGoMaxWarps = 16;
constexpr int kGoBarBytes = kGoMaxWarps * kGaMaxStages * 8; // one mbarrier per slot

template <typename OutT, int kParts>
__global__ void __launch_bounds__(kGoMaxWarps * 32)
fe_gather_obs_kernel(const __grid_constant__ CUtensorMap tmap, const int64_t count, const int W, const int64_t *__restrict__ row0,
                     const OutT *__restrict__ pf, const int64_t *__restrict__ index, OutT *__restrict__ obs, const int S,
                     const int rows_per_phase) {
    constexpr bool kF64 = sizeof(OutT) == 8;
    constexpr int kUnitEnvs = 4 / kParts;      // samples per unit
    constexpr int kTileUnits = 32 / kUnitEnvs; // units per 32-sample tile: 8 or 16 (> S: a refill is at most one tile ahead)
    constexpr int kRounds = (kParts == 1 && kF64) ? 2 : 4; // ceil(W / 32) for the largest W ga_parts() admits
    static_assert(kParts == 1 || kParts == 2, "a window is fetched in one or two parts");
    extern __shared__ __align__(128) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const uint32_t pitch = ga_slot_pitch(W, kF64);
    const uint32_t bars = smem_u32(smem) + 8u * (uint32_t)(warp * S);
    unsigned char *slots = smem + kGoBarBytes + (size_t)warp * S * pitch;
    const uint32_t row_b = (uint32_t)ga_row_bytes(kF64) * W, unit_b = kUnitEnvs * row_b; // row_b: one window
    const int part_rows = (int)(row_b / 2) / kGaPitch; // two parts: tensor rows from a window's first half to its second
    const int shift = ga_phase_shift(kF64);
    const int64_t gw = (int64_t)blockIdx.x * nwarps + warp, NW = (int64_t)gridDim.x * nwarps;
    const int64_t ntiles = (count + 31) / 32;
    if (gw >= ntiles) return;
    const int64_t my_tiles = (ntiles - gw + NW - 1) / NW;
    const int64_t last_tile = gw + (my_tiles - 1) * NW;
    const int last_units = (int)(((count - last_tile * 32 < 32 ? count - last_tile * 32 : 32) + kUnitEnvs - 1) / kUnitEnvs);
    const int64_t n_units = (my_tiles - 1) * kTileUnits + last_units;

    if (lane == 0) {
        for (int si = 0; si < S; ++si) mbar_init(bars + 8u * si, 1);
        mbar_fence_init();
    }
    __syncwarp();

    auto load = [&](int64_t k, int &row, OutT &v) { // handle of sample `lane` of this warp's k-th tile
        int64_t b = (gw + k * NW) * 32 + lane;
        if (b >= count) b = count - 1;
        const int64_t h = index ? __ldg(index + b) : b;
        const int64_t r0 = __ldg(row0 + h);
        v = __ldg(pf + h);
        row = (int)((r0 & ((1 << shift) - 1)) * rows_per_phase + (r0 >> shift)); // copy (row0 mod P), row (row0 div P)
    };
    int cur_row = 0, nxt_row = 0;
    OutT cur_pf = 0, nxt_pf = 0;
    int64_t kc = 0; // tile (of this warp's) whose units are being stored
    load(0, cur_row, cur_pf);
    if (my_tiles > 1) load(1, nxt_row, nxt_pf);
    const uint64_t keep = l2_policy_evict_last(), stream_out = l2_policy_evict_first();

    auto issue = [&](int64_t j) { // whole warp (shuffles); lane 0 issues the gather of unit j into slot j % S
        const int src = (j / kTileUnits == kc) ? cur_row : nxt_row;
        const int g = (int)(j % kTileUnits);
        int4 rows4;
        if constexpr (kParts == 1) {
            rows4 = make_int4(__shfl_sync(0xFFFFFFFFu, src, 4 * g), __shfl_sync(0xFFFFFFFFu, src, 4 * g + 1),
                              __shfl_sync(0xFFFFFFFFu, src, 4 * g + 2), __shfl_sync(0xFFFFFFFFu, src, 4 * g + 3));
        } else { // (first half, second half) of sample 2g, then of sample 2g + 1
            const int a = __shfl_sync(0xFFFFFFFFu, src, 2 * g), b = __shfl_sync(0xFFFFFFFFu, src, 2 * g + 1);
            rows4 = make_int4(a, a + part_rows, b, b + part_rows);
        }
        if (lane == 0) {
            const int si = (int)(j % S);
            mbar_arrive_expect_tx(bars + 8u * si, unit_b);
            tma_gather4(smem_u32(slots + (size_t)si * pitch), &tmap, rows4.x, rows4.y, rows4.z, rows4.w, bars + 8u * si, keep);
        }
    };
    for (int64_t j = 0; j < S && j < n_units; ++j) issue(j);

    // position-feature column: sample e of a unit owns rows [eW, (e+1)W) of the slot; this lane writes rows eW + lane + 32k
    uint32_t round_mask = 0; // bit k: lane + 32k < W
#pragma unroll
    for (int kk = 0; kk < kRounds; ++kk) round_mask |= (uint32_t)(lane + 32 * kk < W) << kk;
    const uint32_t env_stride = (uint32_t)W * 5; // values per sample
    for (int64_t j = 0; j < n_units; ++j) {
        if (j / kTileUnits != kc) { // next tile: its handles arrived a tile ago; fetch the one after it
            kc = j / kTileUnits;
            cur_row = nxt_row; cur_pf = nxt_pf;
            if (kc + 1 < my_tiles) load(kc + 1, nxt_row, nxt_pf);
        }
        const int si = (int)(j % S), g = (int)(j % kTileUnits);
        if (lane == 0) mbar_wait(bars + 8u * si, (uint32_t)((j / S) & 1)); // the unit's windows have landed
        __syncwarp();
        unsigned char *slot = slots + (size_t)si * pitch;
        OutT *col = reinterpret_cast<OutT *>(slot) + 5 * lane + 4; // position-feature slot of row `lane` of sample 0
#pragma unroll
        for (int e = 0; e < kUnitEnvs; ++e) {
            const OutT v = __shfl_sync(0xFFFFFFFFu, cur_pf, kUnitEnvs * g + e);
#pragma unroll
            for (int kk = 0; kk < kRounds; ++kk)
                if (round_mask & (1u << kk)) col[e * env_stride + 160 * kk] = v;
        }
        fence_proxy_async_smem(); // generic-proxy writes -> visible to the bulk store
        __syncwarp();
        if (lane == 0) {
            const int64_t b0 = (gw + kc * NW) * 32 + (int64_t)kUnitEnvs * g;
            const int nv = count - b0 >= kUnitEnvs ? kUnitEnvs : (int)(count - b0); // fewer only in the ragged last tile
            bulk_store_hint(obs + (size_t)b0 * W * 5, smem_u32(slot), (uint32_t)nv * row_b, stream_out);
            bulk_commit();
            if (j + S < n_units) bulk_wait_read_all(); // the store has read the slot: it can be refilled
        }
        __syncwarp();
        if (j + S < n_units) issue(j + S);
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); // stores complete before the warp exits
}

// ------------------------------------------------------------------------------------------
// split variant: bookkeeping and streaming as two launches (what made the portfolio path 25 % faster).
//   fe_book_kernel    one THREAD per env at full occupancy runs env_step() and leaves {row0, position feature} as a
//                     header inside the env's slice of the observation tensor (row0 in its first 8 bytes, the feature
//                     at element 4 = its final place in window row 0);
//   fe_stream_kernel  one WARP per env, no shared memory, no barriers: lane l produces output elements l, l+32, ... of
//                     the env's W*5 values — element f is column f%5 of window row f/5, i.e. input element f - f/5 or
//                     the position feature — so every store instruction writes 128 contiguous bytes and every load
//                     instruction reads ~104 contiguous bytes of the staged series; ceil(5W/32) independent loads per
//                     lane are in flight at once and 48 warps per SM hide the L2 / HBM latency.
// ------------------------------------------------------------------------------------------
template <typename OutT, bool kObserve>
__global__ void __launch_bounds__(kThreads)
fe_book_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const float *__restrict__ actions,
               OutT *__restrict__ obs, OutT *__restrict__ rewards, int32_t *__restrict__ dones, FeStats *stats,
               const uint64_t step_arg, const uint64_t *__restrict__ step_dev) {
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const bool active = i < p.num_envs;
    EnvResult r;
    r.done = 0; r.newly_terminated = 0; r.fin_return = 0.0; r.fin_len = 0; r.row0 = 0; r.posfeat = 0.0;
    if (active) {
        if (kObserve) r = env_observe(p, s, st, k, i);
        else r = env_step<OutT>(p, s, st, k, i, actions, rewards, dones, stats != nullptr, step);
        OutT *slice = obs + (size_t)i * p.window * 5;
        if constexpr (sizeof(OutT) == 8) {
            reinterpret_cast<int64_t *>(slice)[0] = r.row0;
        } else { // the slice is only 4-byte aligned when W is odd: two words
            reinterpret_cast<uint32_t *>(slice)[0] = (uint32_t)((uint64_t)r.row0 & 0xFFFFFFFFu);
            reinterpret_cast<uint32_t *>(slice)[1] = (uint32_t)((uint64_t)r.row0 >> 32);
        }
        slice[4] = (OutT)r.posfeat;
    }
    if (!kObserve) accumulate_stats(stats, r, active);
}

constexpr int kStreamThreads = 256;
constexpr int kStreamSlots = 15;                   // output elements per lane and batch whose loads are in flight together
constexpr int kStreamSpan = 32 * kStreamSlots;     // 480 output elements = 96 window rows: a multiple of 5, so the
constexpr int kStreamSpanIn = kStreamSpan / 5 * 4; // (row, column) pattern of a lane's slots is the same in every batch
template <typename OutT>
__global__ void __launch_bounds__(kStreamThreads)
fe_stream_kernel(const int64_t N, const int W, const OutT *__restrict__ logret, OutT *__restrict__ obs) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * kStreamThreads + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kStreamThreads) >> 5;
    const int n = W * 5;
    // slot u of this lane is output element g = lane + 32u of a batch: input element g - g/5, or the position feature
    int off[kStreamSlots];
#pragma unroll
    for (int u = 0; u < kStreamSlots; ++u) {
        const int g = lane + 32 * u;
        off[u] = g % 5 == 4 ? -1 : g - g / 5;
    }
    const int nfull = n / kStreamSpan, tail = n - nfull * kStreamSpan; // elements of the last, partial batch
    auto header = [&](int64_t e, int64_t &row0, OutT &pf) {
        const OutT *slice = obs + (size_t)e * n;
        if constexpr (sizeof(OutT) == 8) {
            row0 = reinterpret_cast<const int64_t *>(slice)[0];
        } else {
            const uint32_t lo = reinterpret_cast<const uint32_t *>(slice)[0], hi = reinterpret_cast<const uint32_t *>(slice)[1];
            row0 = (int64_t)(((uint64_t)hi << 32) | lo);
        }
        pf = slice[4];
    };
    int64_t row0 = 0, row0_next = 0;
    OutT pf = 0, pf_next = 0;
    if (warp0 < N) header(warp0, row0, pf);
    for (int64_t e = warp0; e < N; e += nwarps) {
        // the next env's header travels while this env's window does (a warp's envs are nwarps apart: other slices)
        if (e + nwarps < N) header(e + nwarps, row0_next, pf_next);
        OutT *out = obs + (size_t)e * n + lane;
        const OutT *src = logret + row0 * 4;
        __syncwarp(); // every lane holds this env's header before any lane overwrites it
        for (int b = 0; b < nfull; ++b, out += kStreamSpan, src += kStreamSpanIn) {
            OutT v[kStreamSlots];
#pragma unroll
            for (int u = 0; u < kStreamSlots; ++u) v[u] = off[u] >= 0 ? __ldg(src + off[u]) : pf;
#pragma unroll
            for (int u = 0; u < kStreamSlots; ++u) out[32 * u] = v[u];
        }
        if (tail > 0) {
            OutT v[kStreamSlots];
#pragma unroll
            for (int u = 0; u < kStreamSlots; ++u) v[u] = (off[u] >= 0 && lane + 32 * u < tail) ? __ldg(src + off[u]) : pf;
#pragma unroll
            for (int u = 0; u < kStreamSlots; ++u)
                if (lane + 32 * u < tail) out[32 * u] = v[u];
        }
        row0 = row0_next;
        pf = pf_next;
    }
}

// ------------------------------------------------------------------------------------------
// portfolio variant (A > 1 assets, one cash account): EXTENSION, the reference is single-asset (:223).
// Semantics (DESIGN.md §3, §4.4): the reference's phases in the reference's order; inside a phase the
// cash moves ONCE: by the f64 butterfly sum of the per-asset deltas where these do not depend on cash (sales,
// covers, margin re-mark / calls / release; bankruptcy is tested on the result), and by a greedy walk over
// the assets in index order with an f64 running cash where they do (long and short entries: an entry is
// legal if the cash left by the assets before it pays for it); A = 1 is the reference exactly.  One WARP per
// env does the bookkeeping with lane = asset (fe_portfolio_book_kernel): every per-asset quantity is
// lane-local, only the f32 cash chain is serial (all lanes keep an identical copy of cash); per-env sums
// (reward, share count) are xor-butterfly warp reductions.  fe_portfolio_stream_kernel then streams the
// (W, A, 4) window in chunks, one block per env: bulk copy in -> interleave 4->5 -> bulk store, double buffered.
// ------------------------------------------------------------------------------------------
constexpr int kPortThreads = 128;
constexpr unsigned kFull = 0xFFFFFFFFu;

__device__ __forceinline__ double warp_sum64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = dadd(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum32(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fadd(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// executed by all 32 lanes of the env's warp; lane >= A is a neutral asset (no shares, no action, price 1).
// Cash-independent phases are butterfly sums; for the two greedy entry walks the per-asset costs are exchanged
// through two 32-double scratch rows in shared memory (broadcast LDS, whose addresses do not depend on the cash
// chain, so the loads run ahead of it) and the serial part is one DADD + compare per asset.  (A first version walked
// every phase with __shfl_sync inside the loops: ncu showed ~10 k instructions per env in this warp,
// WARPSYNC.COLLECTIVE wrappers around every shuffle.)
template <typename OutT>
__device__ __forceinline__ void portfolio_step(const FeParams &p, const FeSeries &s, const FeState &st, const Consts &k,
                                               const int64_t i, const int32_t seg_in, const int32_t ptr_in,
                                               const int64_t row0, const float *__restrict__ actions,
                                               OutT *__restrict__ rewards, int32_t *__restrict__ dones, FeStats *stats,
                                               const uint64_t step, OutT *pf_smem, double *scratch) {
    const int A = p.num_assets, W = p.window;
    const int lane = threadIdx.x & 31;
    const bool act = lane < A;
    const int64_t ia = i * A + lane;
    double *xa = scratch, *xb = scratch + 32; // two 32-double rows; __syncwarp() orders the exchanges
    double O = 1.0, H = 1.0, L = 1.0, C = 1.0, margin = 0.0;
    float lng = 0.0f, sht = 0.0f, d = 0.0f;
    if (act) {
        const double2 *px = reinterpret_cast<const double2 *>(s.prices + ((row0 + W - 1) * A + lane) * 4);
        const double2 oh = __ldg(px), lc = __ldg(px + 1);
        O = oh.x; H = oh.y; L = lc.x; C = lc.y;
        lng = st.long_sh[ia]; sht = st.short_sh[ia]; margin = st.margin[ia];
        d = rintf(fmul(__ldg(actions + ia), k.scale));                       // :298-302
        d = d < -k.ms ? -k.ms : (d > k.ms ? k.ms : d);
    }
    float cash = st.cash[i];
    const int32_t len = __ldg(s.seg_len + seg_in);
    float comm = 0.0f;
    float pos = d < 0.0f ? 0.0f : d, neg = d > 0.0f ? 0.0f : d;             // :344-351
    const double Omc = dsub(O, k.c), Opc = dadd(O, k.c);
    { // :353-361 sell longs ; :367-374 cover shorts ; :375-383 re-mark margin.  The three cash deltas of an asset do not
      // depend on cash: each phase adds the butterfly sum of its per-asset deltas to cash and rounds once
        const float nl = relu32(fadd(lng, neg));
        const float sold = fsub(lng, nl);
        neg = fadd(neg, sold);
        comm = fadd(comm, fmul(sold, k.cf));
        lng = nl;
        cash = d2f(dadd((double)cash, warp_sum64(act ? dmul((double)sold, Omc) : 0.0)));
        const float ns = relu32(fsub(sht, pos));
        const float bought = fsub(sht, ns);
        pos = fsub(pos, bought);
        comm = fadd(comm, fmul(bought, k.cf));
        sht = ns;
        cash = d2f(dsub((double)cash, warp_sum64(act ? dmul((double)bought, Opc) : 0.0)));
        const double nm = dmul((double)fmul(k.imrf, sht), O);
        cash = d2f(dsub((double)cash, warp_sum64(act ? dsub(nm, margin) : 0.0)));
        margin = nm;
    }
    { // :385-399 long entries, greedy in asset order
        xa[lane] = dmul((double)pos, Opc);
        __syncwarp();
        unsigned blocked_mask = 0;
        double c = (double)cash;
        for (int a = 0; a < A; ++a) {
            const double ca = xa[a];
            const bool blocked = dsub(c, ca) < 0.0;
            if (!blocked) c = dsub(c, ca);
            blocked_mask |= (blocked ? 1u : 0u) << a;
        }
        cash = d2f(c);
        if ((blocked_mask >> lane) & 1u) pos = 0.0f;
        comm = fadd(comm, fmul(pos, k.cf));
        lng = fadd(lng, pos);
        __syncwarp();
    }
    { // :401-421 short entries, greedy in asset order
        float q = -neg;
        float sc = fmul(q, k.cf);
        double req = dmul(k.imr, dmul((double)q, O));
        xa[lane] = req;
        xb[lane] = (double)sc;
        __syncwarp();
        unsigned blocked_mask = 0;
        double c = (double)cash;
        for (int a = 0; a < A; ++a) {
            const double ra = xa[a], sa = xb[a];
            const bool blocked = dsub(dsub(c, ra), sa) < 0.0;
            if (!blocked) c = dsub(c, dadd(ra, sa));
            blocked_mask |= (blocked ? 1u : 0u) << a;
        }
        cash = d2f(c);
        if ((blocked_mask >> lane) & 1u) { q = -0.0f; sc = fmul(q, k.cf); req = dmul(k.imr, dmul((double)q, O)); }
        comm = fadd(comm, fmul(q, k.cf));
        margin = dadd(margin, req);
        sht = fadd(sht, q);
        __syncwarp();
    }
    // :428-431 position feature, built before rewards / dones / reset
    if (act) pf_smem[lane] = (OutT)__ddiv_rn(dmul((double)fsub(lng, sht), C), k.SB);
    int done = cash < 0.0f;                                                  // :448
    const double mc1 = relu64(dsub(dmul(dmul((double)sht, H), k.mmr1), margin)); // :459-468 at High
    margin = dadd(margin, mc1);
    const double rel = relu64(dsub(margin, dmul(dmul((double)sht, L), k.imr)));  // :470-475 at Low
    margin = dsub(margin, rel);
    const double mc2 = relu64(dsub(dmul(dmul((double)sht, C), k.mmr1), margin)); // :451 at Close
    margin = dadd(margin, mc2);
    cash = d2f(dsub((double)cash, warp_sum64(act ? mc1 : 0.0)));                 // all margin calls at High, then :465
    done |= cash < 0.0f;
    cash = d2f(dadd((double)cash, warp_sum64(act ? rel : 0.0)));
    cash = d2f(dsub((double)cash, warp_sum64(act ? mc2 : 0.0)));
    done |= cash < 0.0f;
    double r = dadd(-mc1, -mc2);
    if (done) { lng = 0.0f; sht = 0.0f; }                                    // :452-453
    r = dadd(r, dmul((double)fsub(lng, sht), dsub(C, O)));                   // :454-455
    r = dsub(r, (double)comm);                                               // :456
    double rew = warp_sum64(act ? r : 0.0);
    const float nsh = warp_sum32(act ? fadd(sht, lng) : 0.0f);               // :288
    int32_t seg = seg_in, ptr = ptr_in;
    done |= (ptr + W >= len);                                                // :477-496
    rew = dsub(rew, (double)fmul(fmul(done ? 1.0f : 0.0f, nsh), k.cf));      // :288-289
    if (done) {                                                              // :498-521
        cash = k.SBf; margin = 0.0; lng = 0.0f; sht = 0.0f; ptr = 0;
        const int64_t gid = p.env_id_base + i;
        if (p.reset_mode == FE_RESET_ALL || (p.reset_mode == FE_RESET_LAST && gid == p.total_envs - 1))
            draw_segment(p, s, gid, step, 0u, seg, ptr);
    }
    if (act) { st.long_sh[ia] = lng; st.short_sh[ia] = sht; st.margin[ia] = margin; }
    if (lane == 0) {
        if (p.evaluate) {                                                    // :523-536
            const int was = st.terminated[i];
            if (was) rew = 0.0;
            if (done && !was) { st.terminated[i] = 1; if (stats) atomicAdd(&stats->n_terminated, 1ULL); }
            st.ep_return[i] = d2f(dadd((double)st.ep_return[i], rew));
            if (done && stats) atomicAdd(&stats->n_done, 1ULL);
        } else if (stats) {
            const float er = d2f(dadd((double)st.ep_return[i], rew));
            const int32_t el = st.ep_len[i] + 1;
            if (done) {
                atomicAdd(&stats->n_done, 1ULL);
                atomicAdd(&stats->sum_len, (unsigned long long)el);
                atomicAdd(&stats->sum_return, (double)er);
                atomicAdd(&stats->sum_return_sq, (double)er * (double)er);
            }
            st.ep_return[i] = done ? 0.0f : er;
            st.ep_len[i] = done ? 0 : el;
        }
        st.seg[i] = seg; st.ptr[i] = ptr; st.cash[i] = cash;
        rewards[i] = (OutT)rew;
        dones[i] = done;
        if (k.rewards_mirror) reinterpret_cast<OutT *>(k.rewards_mirror)[i] = (OutT)rew;
    if (k.dones_mirror) k.dones_mirror[i] = done;
    }
}

// stream kernel smem: [2 mbarriers 16 B][pf 32 x OutT -> 256 B][unused 768 B][in[2]: CH*4 OutT each][out[2]: CH*5 OutT each]
constexpr int kPortHeader = 16 + 256 + 768;
template <typename OutT> __host__ __device__ inline size_t port_smem_bytes(int CH) {
    return kPortHeader + (size_t)2 * CH * 9 * sizeof(OutT);
}

// ------------------------------------------------------------------------------------------
// portfolio kernels (A > 1): bookkeeping and streaming as two launches.  A first, fused form (one block per env: warp 0
// bookkeeping, then the whole block streaming; profiles/r01_v4_portfolio_fused_ncu.txt) ran at 0.82 of the HBM
// roofline: warp 0's serial cash chain (8 passes over the A assets, each a cvt -> DADD -> cvt dependency) holds its
// block's streaming back for several microseconds per env (11.9 of 21.6 stall cycles per issue were barrier waits).  Here fe_portfolio_book_kernel runs the bookkeeping with one WARP per env at full occupancy
// (~0.05 ms for 65 536 envs) and leaves each env's {row0, position features} as a header INSIDE the env's slice of the
// observation tensor (the position features already at their final place in window row 0); fe_portfolio_stream_kernel
// then reads the header and streams the window exactly as before, with nothing serial in front of it.
// ------------------------------------------------------------------------------------------
constexpr int kBookWarps = 4;

template <typename OutT, bool kObserve>
__global__ void __launch_bounds__(kBookWarps * 32)
fe_portfolio_book_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k,
                         const float *__restrict__ actions, OutT *__restrict__ obs, OutT *__restrict__ rewards,
                         int32_t *__restrict__ dones, FeStats *stats, const uint64_t step_arg,
                         const uint64_t *__restrict__ step_dev) {
    __shared__ double scratch[kBookWarps][64];
    __shared__ OutT pf_s[kBookWarps][32];
    const uint64_t step = step_dev ? *step_dev : step_arg;
    const int W = p.window, A = p.num_assets;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * kBookWarps + warp;
    if (i >= p.num_envs) return; // whole warps leave together; no block-wide barrier below
    const int32_t seg = st.seg[i];
    const int32_t ptr = st.ptr[i] + (kObserve ? 0 : 1);
    const int64_t row0 = __ldg(s.seg_start + seg) + ptr;
    OutT *pf = pf_s[warp];
    if (kObserve) {
        if (lane < A) {
            const double C = __ldg(s.prices + ((row0 + W - 1) * A + lane) * 4 + 3);
            const float net = fsub(st.long_sh[i * A + lane], st.short_sh[i * A + lane]);
            pf[lane] = (OutT)__ddiv_rn(dmul((double)net, C), k.SB);
        }
    } else {
        portfolio_step<OutT>(p, s, st, k, i, seg, ptr, row0, actions, rewards, dones, stats, step, pf, scratch[warp]);
    }
    __syncwarp();
    // header: row0 in the first 8 bytes of the env's slice (two words for f32 obs: the slice is only 4-byte aligned
    // when W*A is odd), position feature of asset a at its final place, element (row 0, asset a, column 4)
    OutT *slice = obs + (size_t)i * W * A * 5;
    if (lane == 0) {
        if constexpr (sizeof(OutT) == 8) {
            reinterpret_cast<int64_t *>(slice)[0] = row0;
        } else {
            reinterpret_cast<uint32_t *>(slice)[0] = (uint32_t)((uint64_t)row0 & 0xFFFFFFFFu);
            reinterpret_cast<uint32_t *>(slice)[1] = (uint32_t)((uint64_t)row0 >> 32);
        }
    }
    if (lane < A) slice[(size_t)lane * 5 + 4] = pf[lane];
}

template <typename OutT>
__global__ void __launch_bounds__(kPortThreads)
fe_portfolio_stream_kernel(const FeParams p, const FeSeries s, OutT *__restrict__ obs, const int CH) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int W = p.window, A = p.num_assets;
    const int tid = threadIdx.x;
    const int64_t i = blockIdx.x;
    const int P = W * A;                         // (row, asset) pairs of one env's window
    const int nchunks = (P + CH - 1) / CH;
    OutT *pf = reinterpret_cast<OutT *>(smem + 16);
    unsigned char *in0 = smem + kPortHeader;
    const size_t in_bytes = (size_t)CH * 4 * sizeof(OutT), out_bytes = (size_t)CH * 5 * sizeof(OutT);
    unsigned char *out0 = in0 + 2 * in_bytes;
    const uint32_t bar0 = smem_u32(smem);
    OutT *dst = obs + (size_t)i * P * 5;
    // the header left by fe_portfolio_book_kernel; every thread reads row0 before anything overwrites it
    int64_t row0;
    if constexpr (sizeof(OutT) == 8) {
        row0 = reinterpret_cast<const int64_t *>(dst)[0];
    } else {
        const uint32_t lo = reinterpret_cast<const uint32_t *>(dst)[0], hi = reinterpret_cast<const uint32_t *>(dst)[1];
        row0 = (int64_t)(((uint64_t)hi << 32) | lo);
    }
    if (tid < A) pf[tid] = dst[(size_t)tid * 5 + 4];
    const unsigned char *src = reinterpret_cast<const unsigned char *>(s.logret) + (size_t)row0 * A * 4 * sizeof(OutT);
    const bool bulk_out = (P & 3) == 0;          // then every chunk of every env is 16-byte aligned and sized
    if (tid == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        mbar_fence_init();
    }
    __syncthreads(); // header consumed, pf visible, barriers initialised
    auto load_chunk = [&](int c) { // thread 0 only
        const int n = min(CH, P - c * CH);
        const uint32_t bytes = (uint32_t)n * 4 * sizeof(OutT);
        const uint32_t bar = bar0 + 8 * (c & 1);
        mbar_arrive_expect_tx(bar, bytes);
        bulk_load(smem_u32(in0 + (c & 1) * in_bytes), src + (size_t)c * in_bytes, bytes, bar);
    };
    if (tid == 0) {
        load_chunk(0);
        if (nchunks > 1) load_chunk(1);
    }
    const float invA = 1.0f / (float)A;
    for (int c = 0; c < nchunks; ++c) {
        const int sidx = c & 1;
        const int n = min(CH, P - c * CH);
        mbar_wait(bar0 + 8 * sidx, (c >> 1) & 1);
        if (c >= 2) { // out[sidx] is being read by the store of chunk c-2: allow only chunk c-1's store in flight
            if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            __syncthreads();
        }
        const Row4<OutT> *in_rows = reinterpret_cast<const Row4<OutT> *>(in0 + sidx * in_bytes);
        OutT *out_tile = reinterpret_cast<OutT *>(out0 + sidx * out_bytes);
        const int g0 = c * CH;
        for (int r = tid; r < n; r += kPortThreads) {
            const int g = g0 + r;
            const int a = g - __float2int_rz(((float)g + 0.5f) * invA) * A;
            const Row4<OutT> v = in_rows[r];
            OutT *o = out_tile + (size_t)r * 5;
            if constexpr (sizeof(OutT) == 4) {
                o[0] = v.v.x; o[1] = v.v.y; o[2] = v.v.z; o[3] = v.v.w;
            } else {
                o[0] = v.a.x; o[1] = v.a.y; o[2] = v.b.x; o[3] = v.b.y;
            }
            o[4] = pf[a];
        }
        OutT *d = dst + (size_t)g0 * 5;
        if (bulk_out) {
            fence_proxy_async_smem();
            __syncthreads(); // out tile complete, in tile fully consumed
            if (tid == 0) {
                bulk_store_hint(d, smem_u32(out_tile), (uint32_t)((size_t)n * 5 * sizeof(OutT)), l2_policy_evict_first());
                bulk_commit();
                if (c + 2 < nchunks) load_chunk(c + 2);
            }
        } else {
            __syncthreads();
            for (int f = tid; f < n * 5; f += kPortThreads) d[f] = out_tile[f];
            __syncthreads();
            if (tid == 0 && c + 2 < nchunks) load_chunk(c + 2);
        }
    }
    if (tid == 0) bulk_wait_read_all();
}

// ------------------------------------------------------------------------------------------
// reset_all, log-returns, effective segment length
// ------------------------------------------------------------------------------------------
__global__ void fe_reset_all_kernel(const FeParams p, const FeSeries s, const FeState st, const uint64_t step,
                                    const int redraw) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.num_envs) return;
    st.cash[i] = (float)p.starting_balance;
    for (int a = 0; a < p.num_assets; ++a) {
        st.margin[i * p.num_assets + a] = 0.0;
        st.long_sh[i * p.num_assets + a] = 0.0f;
        st.short_sh[i * p.num_assets + a] = 0.0f;
    }
    int32_t ptr = 0;
    if (redraw) {
        int32_t seg;
        draw_segment(p, s, p.env_id_base + i, step, 1u, seg, ptr);
        st.seg[i] = seg;
    }
    st.ptr[i] = ptr;
    if (st.terminated) st.terminated[i] = 0;
    if (st.ep_return) st.ep_return[i] = 0.0f;
    if (st.ep_len) st.ep_len[i] = 0;
}

// :179-194.  log() here is CUDA's double-precision log (<= 1 ulp), the reference's is torch's.
__global__ void fe_log_returns_kernel(const double *__restrict__ prices, const int64_t num_rows, const int A,
                                      double *__restrict__ lr64, float *__restrict__ lr32) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; // (t, a)
    if (idx >= num_rows * A) return;
    const int64_t t = idx / A;
    const double *px = prices + idx * 4;
    const double o = px[0];
    const double prev_close = t == 0 ? o : prices[(idx - A) * 4 + 3];
    double v[4];
    v[0] = dmul(100.0, log(__ddiv_rn(o, prev_close)));
#pragma unroll
    for (int c = 1; c < 4; ++c) v[c] = dmul(100.0, log(__ddiv_rn(px[c], o)));
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        if (lr64) lr64[idx * 4 + c] = v[c];
        if (lr32) lr32[idx * 4 + c] = (float)v[c];
    }
}

// :486-496 folded into the table: one warp per segment scans for the first NaN in column 0
__global__ void fe_effective_len_kernel(const double *__restrict__ lr64, const int64_t *__restrict__ seg_start,
                                        const int32_t *__restrict__ raw_len, const int D, const int W, const int A,
                                        int32_t *__restrict__ seg_len) {
    const int d = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (d >= D) return;
    const int64_t start = seg_start[d];
    const int n = raw_len[d];
    int best = n;
    for (int kk = W + 1 + lane; kk < n; kk += 32) {
        const double v = lr64[(size_t)(start + kk) * A * 4];
        if (v != v) { best = kk; break; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if (lane == 0) seg_len[d] = best;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
int check_common(const FeParams *p, const FeSeries *s, const FeState *st) {
    if (!p || !s || !st) return FE_EINVAL;
    if (p->num_envs <= 0 || p->window <= 0 || p->num_segments <= 0 || p->num_rows <= 0) return FE_EINVAL;
    if (p->num_assets < 1 || p->num_assets > 32) return FE_EINVAL;
    if (!s->prices || !s->logret || !s->seg_start || !s->seg_len) return FE_EINVAL;
    if (!st->seg || !st->ptr || !st->cash || !st->long_sh || !st->short_sh || !st->margin) return FE_EINVAL;
    if (p->evaluate && (!st->terminated || !st->ep_return)) return FE_EINVAL;
    if (((uintptr_t)s->prices | (uintptr_t)s->logret | (uintptr_t)s->obs_table) & 15) return FE_EALIGN;
    if ((uintptr_t)st->sched & 7) return FE_EALIGN;
    return 0;
}

// check_common for the entry points that step: accumulating FeStats outside evaluate mode reads and writes the
// episode returns and lengths
int check_step(const FeParams *p, const FeSeries *s, const FeState *st, const FeStats *stats) {
    const int rc = check_common(p, s, st);
    if (rc) return rc;
    return stats && !p->evaluate && (!st->ep_return || !st->ep_len) ? FE_EINVAL : 0;
}

// Tile shape.  Measured on B200 (tools/sweep_tile.sh, 1 Mi envs, W=60): the step is latency-bound per
// block (state loads -> table lookup -> window copy -> interleave -> store), so MANY SMALL blocks in
// flight beat few large ones: 4 envs x 32 threads (23 blocks/SM) runs 0.35 ms where 32 envs x 128
// threads (3 blocks/SM) runs 0.46 ms.  E is kept a multiple of 4 so that every full tile's byte count
// (E*W*20) is a multiple of 16 for any W (bulk-copy granularity).
int pick_tile_envs(int W, bool f64, int *threads_out = nullptr) {
    const size_t sz = f64 ? 8 : 4;
    const size_t per_env = (size_t)W * 9 * sz + sz;
    long e_max = (long)((kSmemMax - kSmemHeader - 16) / per_env) & ~3L;
    if (e_max < 4) return 0;
    long e = 4;
    while (e * W < 192 && e < kMaxTileEnvs) e += 4; // tiny windows: keep >= ~200 rows per block
    if (e > e_max) e = e_max;
    long rows = e * W;
    int threads = (int)(((rows / 8) + 31) & ~31L);
    if (threads < 32) threads = 32;
    if (threads > kThreads) threads = kThreads;
    while (threads < e) threads += 32;
    if (threads_out) *threads_out = threads;
    return (int)e;
}

// envs per tile of the pipe variant: up to 32 (one bookkeeper lane each), a multiple of 4 (16-byte store
// granularity), with TE*W rows fitting the movers' register staging; 0 = window too large, use the tile variant
int pick_pipe_envs(int W, bool f64, int sin) {
    const int max_rows = kMovers * (f64 ? PipeRows<double>::value : PipeRows<float>::value);
    int te = (max_rows / W) & ~3;
    if (te > 32) te = 32;
    while (te >= 4 && (f64 ? pipe_smem_bytes<double>(te, W, sin) : pipe_smem_bytes<float>(te, W, sin)) > (size_t)kSmemMax) te -= 4;
    return te < 4 ? 0 : te;
}
// in-ring stages: 0 ("cached" flavour) while the log-return table is comfortably L2-resident (126 MB L2, shared
// with the observation stream passing through it), else the "stream" flavour
int pick_pipe_stages(const FeParams &p, bool f64) {
    const size_t table = (size_t)p.num_rows * p.num_assets * 4 * (f64 ? 8 : 4);
    return table <= ((size_t)48 << 20) ? 0 : kPipeSInStream;
}
// slots per mover of the gather variant (3 when they fit, else 2); 0 = this window has no gather variant
int pick_gather_stages(int W, bool f64) {
    if (!ga_window_ok(W, f64)) return 0;
    for (int S = FE_GATHER_STAGES; S >= 2; --S)
        if ((f64 ? gather_smem_bytes<double>(W, S) : gather_smem_bytes<float>(W, S)) <= (size_t)kSmemMax) return S;
    return 0;
}
// the observation-layout table is worth reading only while it stays L2-resident next to the observation stream
bool gather_table_resident(const FeParams &p, bool f64) { return ga_table_bytes(p.num_rows, p.window, f64) <= ((size_t)64 << 20); }

// Which kernel a launch uses.  `auto`: portfolio when A > 1; for populations that give every SM a few tiles and windows
// of >= 24 rows a persistent kernel — gather when the caller staged the observation-layout table (FeSeries.obs_table),
// the window is a legal TMA row and that table is L2-resident, else pipe (measured on c2, tools/window_sweep.sh ->
// profiles/r01_v4_window_sweep.txt: W = 4 / 16: tile 0.19 / 0.24 ms vs pipe 0.73 / 0.37 ms — with so few rows per env the
// bookkeeper warps are the bottleneck, while the tile variant gives every env its own thread; W = 60 / 128 / 390: pipe
// 0.27 / 0.27 / 0.23 vs tile 0.36 / 0.38 / 0.29); split for windows too long for the pipe rings; else tile while the
// window fits in shared memory; else direct.
enum StepKernel { K_PORTFOLIO, K_SPLIT, K_GATHER, K_PIPE, K_TILE, K_DIRECT, K_ERR_SMEM, K_ERR_TABLE };
struct StepChoice {
    StepKernel kern;
    int te;      // envs per tile (pipe / tile)
    int sin;     // pipe: in-ring stages (0 = cached flavour)
    int S;       // gather: slots per mover
    int threads; // tile: threads per block
};
StepChoice choose_kernel(const FeParams &p, bool gather_ready, bool f64, int sms) {
    StepChoice c = {K_DIRECT, 0, 0, 0, kThreads};
    if (p.num_assets > 1 || p.variant == FE_VARIANT_PORTFOLIO) { c.kern = K_PORTFOLIO; return c; }
    if (p.variant == FE_VARIANT_SPLIT) { c.kern = K_SPLIT; return c; }
    // small populations: a persistent grid needs a few tiles per SM to hide its prologue
    const bool worth_persistent = p.num_envs >= (int64_t)4 * sms * 32;
    if (p.variant == FE_VARIANT_GATHER || p.variant == FE_VARIANT_AUTO) {
        c.S = pick_gather_stages(p.window, f64);
        if (p.variant == FE_VARIANT_GATHER) {
            c.kern = !gather_ready ? K_ERR_TABLE : c.S == 0 ? K_ERR_SMEM : K_GATHER;
            return c;
        }
        const bool no_gather = env_override("FE_NO_GATHER") != 0; // sweeps: "auto" never picks gather
        if (!no_gather && gather_ready && c.S > 0 && worth_persistent && p.window >= 24 && gather_table_resident(p, f64)) {
            c.kern = K_GATHER;
            return c;
        }
    }
    if (p.variant == FE_VARIANT_PIPE || p.variant == FE_VARIANT_AUTO) {
        const int ov_sin = env_override("FE_PIPE_FLAVOUR"); // sweeps: 1 = cached, 2 = stream
        c.sin = ov_sin == 1 ? 0 : ov_sin == 2 ? kPipeSInStream : pick_pipe_stages(p, f64);
        c.te = pick_pipe_envs(p.window, f64, c.sin);
        if (c.te == 0 && p.variant == FE_VARIANT_PIPE) { c.kern = K_ERR_SMEM; return c; }
        if (c.te > 0 && (p.variant == FE_VARIANT_PIPE || (worth_persistent && p.window >= 24))) { c.kern = K_PIPE; return c; }
        // windows too long for the pipe variant's rings (> 512 rows f32, > 256 f64): the split variant's warp-per-env
        // streaming (W = 1024, 64 Ki envs: 0.26 ms vs 0.66 ms for tile)
        if (c.te == 0 && p.variant == FE_VARIANT_AUTO) { c.kern = K_SPLIT; return c; }
    }
    c.te = p.variant == FE_VARIANT_DIRECT ? 0 : pick_tile_envs(p.window, f64, &c.threads);
    if (p.variant == FE_VARIANT_TILE && c.te == 0) { c.kern = K_ERR_SMEM; return c; }
    if (c.te > 0) {
        const int ov_e = env_override("FE_TILE_ENVS"), ov_t = env_override("FE_TILE_THREADS");
        const size_t sz = f64 ? 8 : 4;
        if (ov_e >= 4 && kSmemHeader + 16 + (size_t)(ov_e & ~3) * (p.window * 9 * sz + sz) <= (size_t)kSmemMax) c.te = ov_e & ~3;
        if (ov_t >= 32 && ov_t <= kThreads) c.threads = ov_t & ~31;
        if (c.te > c.threads) c.te = c.threads;
        c.kern = K_TILE;
    }
    return c;
}

// Geometry and tensor map of the observation-layout table, shared by the gather step and gather_obs: `rpp` tensor rows
// per shifted copy, each window read in `parts` box rows of `inner_bytes` at an 80-byte pitch — the rows overlap, row i
// is the window starting i pitches into a shifted copy.  The map is encoded by the driver (cuTensorMapEncodeTiled,
// resolved through the runtime so that libcuda is not a link dependency) and cached: a step costs no driver call.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
struct TmapEntry {
    const void *base;
    int64_t rows;
    int inner_bytes, device;
    CUtensorMap map;
};
struct ObsTableMap {
    CUtensorMap map;
    int64_t rpp;
    int parts;
};
int gather_tensor_map(const FeParams &p, const FeSeries &s, bool f64, ObsTableMap *out) {
    out->rpp = ga_rows_per_phase(p.num_rows, p.window, f64);
    out->parts = ga_parts(p.window, f64);
    const int64_t total_rows = out->rpp << ga_phase_shift(f64);
    if (total_rows >= ((int64_t)1 << 31)) return FE_EINVAL;
    const void *table = s.obs_table;
    const int inner_bytes = ga_row_bytes(f64) * p.window / out->parts, device = p.device;
    static std::mutex mu;
    static std::vector<TmapEntry> cache;
    static EncodeTiledFn encode = nullptr;
    std::lock_guard<std::mutex> lock(mu);
    for (const TmapEntry &e : cache)
        if (e.base == table && e.rows == total_rows && e.inner_bytes == inner_bytes && e.device == device) { out->map = e.map; return 0; }
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
        if (e != cudaSuccess) return (int)e;
        if (!fn || q != cudaDriverEntryPointSuccess) return FE_EDRIVER;
        encode = (EncodeTiledFn)fn;
    }
    TmapEntry n;
    n.base = table; n.rows = total_rows; n.inner_bytes = inner_bytes; n.device = device;
    const cuuint64_t dims[2] = {(cuuint64_t)(inner_bytes / 8), (cuuint64_t)total_rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kGaPitch};
    const cuuint32_t box[2] = {(cuuint32_t)(inner_bytes / 8), 1}, elem_strides[2] = {1, 1};
    const CUresult r = encode(&n.map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void *>(table), dims, strides, box, elem_strides,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return FE_EDRIVER;
    if (cache.size() >= 64) cache.erase(cache.begin());
    cache.push_back(n);
    out->map = n.map;
    return 0;
}

template <typename OutT, bool kObserve>
int launch(const FeParams &p, const FeSeries &s, const FeState &st, const float *actions, void *obs, void *rewards,
           int32_t *dones, FeStats *stats, uint64_t step, cudaStream_t stream, const uint64_t *step_dev = nullptr,
           void *rewards_mirror = nullptr, int32_t *dones_mirror = nullptr, uint32_t *dones_bits_mirror = nullptr,
           uint32_t *dones_bits_stage = nullptr, int *packed_inline = nullptr) {
    Consts k = make_consts(p);
    k.rewards_mirror = rewards_mirror;
    k.dones_mirror = dones_mirror;
    int sms = 0;
    int rc = device_sm_count(p.device, &sms);
    if (rc) return rc;
    const StepChoice c = choose_kernel(p, s.obs_table && st.sched, sizeof(OutT) == 8, sms);
    // the persistent kernels with 32-env tiles pack the dones themselves (one ballot per tile); otherwise the caller runs
    // fe_pack_dones_kernel after the step
    const bool inline_pack = dones_bits_mirror && dones_bits_stage && (c.kern == K_GATHER || (c.kern == K_PIPE && c.te == 32));
    const int pack_mode = env_override("FE_PACK_MODE"); // sweeps: 1 = words straight to the host, 2 = flush by a second kernel
    if (inline_pack) {
        k.dones_bits_out = pack_mode == 1 ? dones_bits_mirror : dones_bits_stage;
        if (c.kern == K_GATHER && pack_mode == 0) k.dones_bits_host = dones_bits_mirror; // sent by the kernel itself
    }
    // 0: the caller packs dones_dev after the step; 1: packed and already sent to the host; 2: packed into the staging buffer
    if (packed_inline) *packed_inline = !inline_pack ? 0 : (pack_mode == 1 || (c.kern == K_GATHER && pack_mode == 0)) ? 1 : 2;
    switch (c.kern) {
    case K_ERR_SMEM: return FE_ESMEM;
    case K_ERR_TABLE: return FE_EINVAL;
    case K_PORTFOLIO: {
        if ((uintptr_t)obs & 15) return FE_EALIGN;
        const int P = p.window * p.num_assets;
        int CH = 512; // pairs per chunk (8 KB in + 10 KB out, x2 stages); C3: 128 -> 1.492 ms, 256 -> 1.480, 512 -> 1.472, 1024 -> 1.471
        const int ov_ch = env_override("FE_PORT_CHUNK");
        if (ov_ch >= 4) CH = ov_ch & ~3;
        if (CH > ((P + 3) & ~3)) CH = (P + 3) & ~3;
        const size_t smem = port_smem_bytes<OutT>(CH);
        if (smem > (size_t)kSmemMax) return FE_ESMEM;
        constexpr auto skern = fe_portfolio_stream_kernel<OutT>;
        if ((rc = opt_in_smem<skern>(p.device))) return rc;
        fe_portfolio_book_kernel<OutT, kObserve><<<(unsigned)((p.num_envs + kBookWarps - 1) / kBookWarps), kBookWarps * 32, 0, stream>>>(
            p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones, stats, step, step_dev);
        skern<<<(unsigned)p.num_envs, kPortThreads, smem, stream>>>(p, s, (OutT *)obs, CH);
        break;
    }
    case K_SPLIT: {
        if ((uintptr_t)obs & 7) return FE_EALIGN;
        fe_book_kernel<OutT, kObserve><<<(unsigned)((p.num_envs + kThreads - 1) / kThreads), kThreads, 0, stream>>>(
            p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones, stats, step, step_dev);
        const int ov_b = env_override("FE_STREAM_BLOCKS_PER_SM");
        int64_t blocks = (int64_t)sms * (ov_b > 0 ? ov_b : 6); // 48 warps per SM
        const int64_t need = (p.num_envs * 32 + kStreamThreads - 1) / kStreamThreads;
        if (blocks > need) blocks = need;
        fe_stream_kernel<OutT><<<(unsigned)blocks, kStreamThreads, 0, stream>>>(p.num_envs, p.window, (const OutT *)s.logret, (OutT *)obs);
        break;
    }
    case K_GATHER: {
        if ((uintptr_t)obs & 15) return FE_EALIGN;
        ObsTableMap tab;
        if ((rc = gather_tensor_map(p, s, sizeof(OutT) == 8, &tab))) return rc;
        const int64_t ntiles = (p.num_envs + 31) / 32;
        const unsigned blocks = (unsigned)(ntiles < sms ? ntiles : sms);
        const size_t smem = gather_smem_bytes<OutT>(p.window, c.S);
        return with_flag(tab.parts == 2, [&](auto two_parts) {
            constexpr auto kern = fe_gather_kernel<OutT, kObserve, decltype(two_parts)::value ? 2 : 1>;
            if (const int r = opt_in_smem<kern>(p.device)) return r;
            kern<<<blocks, kGaThreads, smem, stream>>>(tab.map, p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones, stats,
                                                       step, step_dev, c.S, (int)tab.rpp, st.sched);
            return (int)cudaGetLastError();
        });
    }
    case K_PIPE: {
        if ((uintptr_t)obs & 15) return FE_EALIGN;
        const int64_t ntiles = (p.num_envs + c.te - 1) / c.te;
        const unsigned blocks = (unsigned)(ntiles < sms ? ntiles : sms);
        return with_flag(c.sin != 0, [&](auto stream_flavour) {
            constexpr auto kern = fe_pipe_kernel<OutT, kObserve, decltype(stream_flavour)::value ? kPipeSInStream : 0>;
            if (const int r = opt_in_smem<kern>(p.device)) return r;
            kern<<<blocks, kPipeThreads, pipe_smem_bytes<OutT>(c.te, p.window, c.sin), stream>>>(
                p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones, stats, step, step_dev, c.te);
            return (int)cudaGetLastError();
        });
    }
    case K_TILE: {
        if ((uintptr_t)obs & 15) return FE_EALIGN;
        const size_t smem = tile_smem_bytes<OutT>(c.te, p.window);
        constexpr auto kern = fe_tile_kernel<OutT, kObserve>;
        if ((rc = opt_in_smem<kern>(p.device))) return rc;
        const int64_t blocks = (p.num_envs + c.te - 1) / c.te;
        kern<<<(unsigned)blocks, c.threads, smem, stream>>>(p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones,
                                                             stats, step, step_dev, c.te);
        break;
    }
    case K_DIRECT: {
        const int64_t blocks = (p.num_envs + kThreads - 1) / kThreads;
        fe_direct_kernel<OutT, kObserve><<<(unsigned)blocks, kThreads, 0, stream>>>(
            p, s, st, k, actions, (OutT *)obs, (OutT *)rewards, dones, stats, step, step_dev);
        break;
    }
    }
    return (int)cudaGetLastError();
}

// handles -> tensor (fe_gather_obs / fe_materialize).  TMA path while the gather variant could serve this window from an
// L2-resident observation-layout table; the warp-per-sample copy otherwise (and for an output or table that is not 16-byte
// aligned, which only fe_materialize accepts).
enum ObsPath { OBS_NONE, OBS_TMA, OBS_LSU };
ObsPath choose_obs_path(const FeParams &p, const FeSeries &s) {
    if (p.num_assets != 1) return OBS_NONE;
    const bool f64 = p.out_f64 != 0;
    return s.obs_table && ga_parts(p.window, f64) > 0 && gather_table_resident(p, f64) ? OBS_TMA : OBS_LSU;
}

template <typename OutT>
int gather_obs(const FeParams &p, const FeSeries &s, const int64_t *row0, const void *pf, const int64_t *index, int64_t count,
               void *obs, cudaStream_t stream) {
    constexpr bool f64 = sizeof(OutT) == 8;
    if (choose_obs_path(p, s) != OBS_TMA || (((uintptr_t)obs | (uintptr_t)s.obs_table) & 15)) {
        const int64_t blocks = (count * 32 + kThreads - 1) / kThreads;
        fe_materialize_kernel<OutT><<<(unsigned)blocks, kThreads, 0, stream>>>(count, p.window, (const OutT *)s.logret, row0,
                                                                               (const OutT *)pf, index, (OutT *)obs);
        return (int)cudaGetLastError();
    }
    int sms = 0;
    int rc = device_sm_count(p.device, &sms);
    if (rc) return rc;
    ObsTableMap tab;
    if ((rc = gather_tensor_map(p, s, f64, &tab))) return rc;
    // 3 slots per warp when at least 8 warps of them fit in shared memory, else 2; up to 16 warps per block and, for short
    // windows whose rings are small, up to 4 blocks per SM
    const size_t pitch = ga_slot_pitch(p.window, f64), room = (size_t)kSmemMax - kGoBarBytes;
    int S = 3;
    if (room / (S * pitch) < 8) S = 2;
    const int warps = (int)(room / (S * pitch) < (size_t)kGoMaxWarps ? room / (S * pitch) : kGoMaxWarps);
    const size_t smem = kGoBarBytes + (size_t)warps * S * pitch;
    int per_sm = (int)((size_t)(228 * 1024) / (smem + 1024));
    per_sm = per_sm < 1 ? 1 : per_sm > 4 ? 4 : per_sm;
    const int64_t need = ((count + 31) / 32 + warps - 1) / warps;
    const unsigned blocks = (unsigned)(need < (int64_t)sms * per_sm ? need : (int64_t)sms * per_sm);
    return with_flag(tab.parts == 2, [&](auto two_parts) {
        constexpr auto kern = fe_gather_obs_kernel<OutT, decltype(two_parts)::value ? 2 : 1>;
        if (const int r = opt_in_smem<kern>(p.device)) return r;
        kern<<<blocks, warps * 32, smem, stream>>>(tab.map, count, p.window, row0, (const OutT *)pf, index, (OutT *)obs, S,
                                                   (int)tab.rpp);
        return (int)cudaGetLastError();
    });
}

// step ordinal kept on the device (fe_step_captured): one thread bumps it ahead of the step kernel
__global__ void fe_bump_kernel(uint64_t *counter) { *counter += 1; }

// ------------------------------------------------------------------------------------------
// signal backtest (fe_backtest, fe_backtest_targets): K steps of every env in one launch, one thread per env.  The
// action of each step comes from the env's column of a signal table: the value itself (TradeRule) or the delta to a
// target position (TargetRule); the step is env_compute_core (the trading arithmetic of every step
// kernel) and the metrics update is the one of fe_episode_metrics_kernel (fe_metrics.cuh).  The env state and the
// metrics' running state stay in registers for the whole launch and are written back once; no observation is built.
// ------------------------------------------------------------------------------------------
constexpr int kBtThreads = 256;
constexpr int kBtWarps = kBtThreads / 32;

// env i's state in registers (env_compute_core's accessor for the backtest), plus the reward / done of the last step
struct BacktestEnvIO {
    int32_t seg, ptr;
    float cash, lng, sht;
    double margin;
    int term;
    float eret;
    int32_t elen;
    double rew;
    int done;
    __device__ __forceinline__ void set_seg(int32_t v) { seg = v; }
    __device__ __forceinline__ int terminated() const { return term; }
    __device__ __forceinline__ void set_terminated() { term = 1; }
    __device__ __forceinline__ float ep_return() const { return eret; }
    __device__ __forceinline__ void set_ep_return(float v) { eret = v; }
    __device__ __forceinline__ int32_t ep_len() const { return elen; }
    __device__ __forceinline__ void set_ep_len(int32_t v) { elen = v; }
    __device__ __forceinline__ void finish(int32_t ptr_, float cash_, float lng_, float sht_, double margin_, double rew_,
                                           int done_) {
        ptr = ptr_; cash = cash_; lng = lng_; sht = sht_; margin = margin_; rew = rew_; done = done_;
    }
};

// reduction over the block; the result is valid in thread 0.  Every thread of the block must call it.
template <typename T, typename Op>
__device__ __forceinline__ T bt_block_reduce(T v, Op op, T *sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    __syncthreads();   // the previous call's readers are done with sh
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < kBtWarps; ++w) v = op(v, sh[w]);
    return v;
}

// The action rules of a backtest step: the table value v of env i's column at the step's row -> the action fed to
// env_compute_core.  load(c) runs once per launch with env i's column c.
struct TradeRule {   // fe_backtest: v is the action
    __device__ __forceinline__ void load(int32_t) {}
    __device__ __forceinline__ float action(float v, const BacktestEnvIO &, const EpisodeRun &) const { return v; }
};
struct TargetRule {  // fe_backtest_targets: v is a target net position (include/finenvs_b200.h)
    const double *__restrict__ exits;   // (num_signals, 2) trailing stop, take-profit; nullptr: no exits
    float ms, scale;
    double stop, take;
    __device__ __forceinline__ void load(int32_t c) {
        if (exits) { stop = __ldg(exits + 2 * (int64_t)c); take = __ldg(exits + 2 * (int64_t)c + 1); }
    }
    __device__ __forceinline__ float action(float v, const BacktestEnvIO &e, const EpisodeRun &run) const {
        float T = rintf(fmul(v, scale));
        T = T < -ms ? -ms : (T > ms ? ms : T);
        if (exits && (dsub(run.peak, run.sum) >= stop || run.sum >= take)) T = 0.0f;
        // env_compute_core maps the quotient back to exactly D (the header's round-trip bound, max_shares <= 2^20)
        return __fdiv_rn(fsub(T, fsub(e.lng, e.sht)), scale);
    }
};

// the backtest loop of both entry points; Rule turns each step's table value into the action.  The structs are taken
// by value: with references the compiler numbered fe_backtest_kernel's accumulators differently and its SASS changed.
template <typename OutT, typename Rule>
__device__ __forceinline__ void
backtest_run(const FeParams p, const FeSeries s, const FeState st, const Consts k, const FeMetricsState m,
             const int64_t capacity, FeStats *stats, const float *__restrict__ signal, const int32_t *__restrict__ column,
             const uint64_t first_step, const int K, OutT *__restrict__ rewards, int32_t *__restrict__ dones,
             const int history, Rule rule) {
    constexpr unsigned kAll = 0xFFFFFFFFu;
    const int64_t N = p.num_envs;
    const int64_t i = (int64_t)blockIdx.x * kBtThreads + threadIdx.x;
    const int64_t gid = p.env_id_base + i;
    const bool active = i < N;
    const bool track = stats != nullptr;
    const int lane = threadIdx.x & 31;
    BacktestEnvIO e{};
    EpisodeRun run{};
    int emitted = 0;
    const float *sig = signal;
    if (active) {
        e.seg = st.seg[i]; e.ptr = st.ptr[i]; e.cash = st.cash[i]; e.lng = st.long_sh[i]; e.sht = st.short_sh[i];
        e.margin = st.margin[i];
        if (p.evaluate) e.term = st.terminated[i];
        if (p.evaluate || track) e.eret = st.ep_return[i];
        if (!p.evaluate && track) e.elen = st.ep_len[i];
        run.len = m.len[i]; run.pos = m.pos[i];
        run.sum = m.sum[i]; run.mean = m.mean[i]; run.m2 = m.m2[i]; run.peak = m.peak[i]; run.mdd = m.mdd[i];
        run.mdd_rel = m.mdd_rel[i];
        if (m.emitted) emitted = m.emitted[i];
        const int32_t c = column[i];
        sig = signal + (int64_t)c * p.num_rows;
        rule.load(c);
    }
    // FeStats and FeMetricsSummary contributions, flushed once per block after the loop; only the slot counter
    // (summary->episodes) is touched inside it, once per warp and step with a finished episode
    unsigned long long st_done = 0, st_term = 0, st_len = 0;
    double st_ret = 0.0, st_sq = 0.0;
    unsigned long long ms_cnt = 0, ms_len = 0;
    double ms_ret = 0.0, ms_sh = 0.0, ms_sh2 = 0.0, ms_mdd = 0.0, ms_hit = 0.0, ms_max = 0.0;
    for (int t = 0; t < K; ++t) {
        const uint64_t step = first_step + (uint64_t)t;
        int emit = 0;
        int32_t len = 0;
        double sum = 0.0, sharpe = 0.0, mdd = 0.0, mdd_rel = 0.0, hit = 0.0;
        if (active) {
            EnvLoads ld;
            ld.seg = e.seg; ld.ptr = e.ptr; ld.cash = e.cash; ld.lng = e.lng; ld.sht = e.sht; ld.margin = e.margin;
            const EnvBar bar = env_load_bar(p, s, ld);
            // row seg_start + ptr + W - 1: the last row of the window the env observed before this step (bar.row0 is the
            // window after the advance).  The trade executes at the next row's Open: no look-ahead.
            ld.act = rule.action(__ldg(sig + bar.row0 + p.window - 2), e, run);
            const EnvResult r = env_compute_core(p, s, k, i, ld, bar, track, step, e);
            const OutT ro = (OutT)e.rew;
            if (history) {
                rewards[(int64_t)t * N + i] = ro;
                dones[(int64_t)t * N + i] = e.done;
            } else if (t == K - 1) {
                rewards[i] = ro;
                dones[i] = e.done;
            }
            if (track && r.done) {   // accumulate_stats
                st_done += 1;
                st_len += (unsigned long long)r.fin_len;
                st_ret += r.fin_return;
                st_sq += r.fin_return * r.fin_return;
            }
            st_term += (unsigned long long)r.newly_terminated;
            const EpisodeRun nx = episode_advance(RunInRegisters{run}, (double)ro, p.starting_balance);
            len = nx.len; sum = nx.sum; mdd = nx.mdd; mdd_rel = nx.mdd_rel;
            if (e.done) {
                emit = 1;
                if (m.emitted) {   // evaluate: only the first episode after the flags were cleared
                    emit = !emitted;
                    emitted = 1;
                }
                sharpe = episode_sharpe(nx);
                hit = episode_hit_rate(nx);
                run = EpisodeRun{};
            } else {
                run = nx;
            }
        }
        const unsigned ballot = __ballot_sync(kAll, emit);
        if (ballot) {
            const int leader = __ffs(ballot) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(&m.summary->episodes, (unsigned long long)__popc(ballot));
            base = __shfl_sync(kAll, base, leader);
            if (emit) {
                const int64_t slot = (int64_t)base + __popc(ballot & ((1u << lane) - 1u));
                if (slot < capacity)
                    episode_write_record(m, slot, (int64_t)step * p.total_envs + gid, gid, len, sum, sharpe, mdd, mdd_rel, hit);
                ms_cnt += 1;
                ms_len += (unsigned long long)len;
                ms_ret = __dadd_rn(ms_ret, sum);
                ms_sh = __dadd_rn(ms_sh, sharpe);
                ms_sh2 = __dadd_rn(ms_sh2, __dmul_rn(sharpe, sharpe));
                ms_mdd = __dadd_rn(ms_mdd, mdd);
                ms_hit = __dadd_rn(ms_hit, hit);
                ms_max = fmax(ms_max, mdd);
            }
        }
    }
    if (active) {
        st.seg[i] = e.seg; st.ptr[i] = e.ptr; st.cash[i] = e.cash; st.long_sh[i] = e.lng; st.short_sh[i] = e.sht;
        st.margin[i] = e.margin;
        if (p.evaluate) st.terminated[i] = (uint8_t)e.term;
        if (p.evaluate || track) st.ep_return[i] = e.eret;
        if (!p.evaluate && track) st.ep_len[i] = e.elen;
        episode_store(m, i, run);
        if (m.emitted) m.emitted[i] = (uint8_t)emitted;
    }
    __shared__ unsigned long long sh_u[kBtWarps];
    __shared__ double sh_d[kBtWarps];
    const auto add_u = [](unsigned long long a, unsigned long long b) { return a + b; };
    const auto add_d = [](double a, double b) { return __dadd_rn(a, b); };
    const auto max_d = [](double a, double b) { return fmax(a, b); };
    if (track) {
        const unsigned long long nd = bt_block_reduce(st_done, add_u, sh_u);
        const unsigned long long nt = bt_block_reduce(st_term, add_u, sh_u);
        const unsigned long long sl = bt_block_reduce(st_len, add_u, sh_u);
        const double sr = bt_block_reduce(st_ret, add_d, sh_d);
        const double sq = bt_block_reduce(st_sq, add_d, sh_d);
        if (threadIdx.x == 0) {
            if (nd) atomicAdd(&stats->n_done, nd);
            if (nt) atomicAdd(&stats->n_terminated, nt);
            if (sl) atomicAdd(&stats->sum_len, sl);
            if (nd) { atomicAdd(&stats->sum_return, sr); atomicAdd(&stats->sum_return_sq, sq); }
        }
    }
    const unsigned long long cnt = bt_block_reduce(ms_cnt, add_u, sh_u);
    const unsigned long long blen = bt_block_reduce(ms_len, add_u, sh_u);
    const double bret = bt_block_reduce(ms_ret, add_d, sh_d);
    const double bsh = bt_block_reduce(ms_sh, add_d, sh_d);
    const double bsh2 = bt_block_reduce(ms_sh2, add_d, sh_d);
    const double bmdd = bt_block_reduce(ms_mdd, add_d, sh_d);
    const double bhit = bt_block_reduce(ms_hit, add_d, sh_d);
    const double bmax = bt_block_reduce(ms_max, max_d, sh_d);
    if (threadIdx.x == 0 && cnt) {
        FeMetricsSummary *sm = m.summary;
        atomicAdd(&sm->sum_len, blen);
        atomicAdd(&sm->sum_return, bret);
        atomicAdd(&sm->sum_sharpe, bsh);
        atomicAdd(&sm->sum_sharpe_sq, bsh2);
        atomicAdd(&sm->sum_mdd, bmdd);
        atomicAdd(&sm->sum_hit_rate, bhit);
        // mdd >= 0: the order of non-negative doubles is the order of their bit patterns
        atomicMax(reinterpret_cast<unsigned long long *>(&sm->max_mdd), (unsigned long long)__double_as_longlong(bmax));
    }
}

template <typename OutT>
__global__ void __launch_bounds__(kBtThreads)
fe_backtest_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const FeMetricsState m,
                   const int64_t capacity, FeStats *stats, const float *__restrict__ signal, const int32_t *__restrict__ column,
                   const uint64_t first_step, const int K, OutT *__restrict__ rewards, int32_t *__restrict__ dones,
                   const int history) {
    backtest_run<OutT>(p, s, st, k, m, capacity, stats, signal, column, first_step, K, rewards, dones, history, TradeRule{});
}

template <typename OutT>
__global__ void __launch_bounds__(kBtThreads)
fe_backtest_targets_kernel(const FeParams p, const FeSeries s, const FeState st, const Consts k, const FeMetricsState m,
                           const int64_t capacity, FeStats *stats, const float *__restrict__ signal,
                           const int32_t *__restrict__ column, const double *__restrict__ exits, const uint64_t first_step,
                           const int K, OutT *__restrict__ rewards, int32_t *__restrict__ dones, const int history) {
    const TargetRule rule{exits, k.ms, k.scale, 0.0, 0.0};
    backtest_run<OutT>(p, s, st, k, m, capacity, stats, signal, column, first_step, K, rewards, dones, history, rule);
}

// fe_backtest (kTargets = false, exits == nullptr) and fe_backtest_targets: validation and launch
template <bool kTargets>
int backtest_entry(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m, int64_t capacity,
                   FeStats *stats, const float *signal, int32_t num_signals, const int32_t *column, const double *exits,
                   uint64_t first_step, int32_t num_steps, void *rewards, int32_t *dones, int32_t history, void *stream) {
    int rc = check_step(p, s, st, stats);
    if (rc) return rc;
    if (p->num_assets != 1 || !signal || num_signals < 1 || !column || num_steps < 1 || !rewards || !dones) return FE_EINVAL;
    if (kTargets && (p->max_shares < 1 || p->max_shares > FE_TARGET_MAX_SHARES)) return FE_EINVAL;
    if ((uintptr_t)exits & 7) return FE_EALIGN;
    if ((rc = check_metrics_state(p, m, capacity))) return rc;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    const Consts k = make_consts(*p);
    FeMetricsState ms = *m;
    if (!p->evaluate) ms.emitted = nullptr;
    const unsigned blocks = (unsigned)((p->num_envs + kBtThreads - 1) / kBtThreads);
    cudaStream_t q = (cudaStream_t)stream;
    return with_out_type(p->out_f64, [&](auto out_type) {
        using OutT = decltype(out_type);
        if constexpr (kTargets)
            fe_backtest_targets_kernel<OutT><<<blocks, kBtThreads, 0, q>>>(*p, *s, *st, k, ms, capacity, stats, signal, column,
                                                                           exits, first_step, num_steps, (OutT *)rewards, dones,
                                                                           history);
        else
            fe_backtest_kernel<OutT><<<blocks, kBtThreads, 0, q>>>(*p, *s, *st, k, ms, capacity, stats, signal, column,
                                                                   first_step, num_steps, (OutT *)rewards, dones, history);
        return (int)cudaGetLastError();
    });
}

// side streams of fe_step_host (created once per device, never destroyed: they live as long as the process)
constexpr int kHostStreams = 3;
struct HostPipe {
    cudaStream_t s[kHostStreams];
    cudaEvent_t start, done[kHostStreams];
    bool ok;
};
HostPipe *host_pipe(int device) { // the device must be current (DeviceGuard)
    static HostPipe pipes[16];
    static std::once_flag once[16];
    HostPipe *hp = &pipes[device & 15];
    std::call_once(once[device & 15], [hp] {
        hp->ok = true;
        for (int k = 0; k < kHostStreams; ++k) {
            if (cudaStreamCreateWithFlags(&hp->s[k], cudaStreamNonBlocking) != cudaSuccess) hp->ok = false;
            if (cudaEventCreateWithFlags(&hp->done[k], cudaEventDisableTiming) != cudaSuccess) hp->ok = false;
        }
        if (cudaEventCreateWithFlags(&hp->start, cudaEventDisableTiming) != cudaSuccess) hp->ok = false;
    });
    return hp->ok ? hp : nullptr;
}

// dones (N,) int32 -> bit i of the little-endian word i / 32 (the wire format of fe_step_host_packed)
__global__ void __launch_bounds__(256) fe_pack_dones_kernel(const int32_t *__restrict__ dones, const int64_t n, uint32_t *__restrict__ bits) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned word = __ballot_sync(0xFFFFFFFFu, i < n && dones[i] != 0);
    if ((threadIdx.x & 31) == 0 && i < n) bits[i >> 5] = word;
}

// staging buffer (HBM) -> mapped host memory: consecutive threads, consecutive words, so the bits cross PCIe in full lines
__global__ void __launch_bounds__(256) fe_flush_bits_kernel(const uint32_t *__restrict__ stage, const int64_t nwords, uint32_t *__restrict__ host) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < nwords) host[w] = stage[w];
}

} // namespace

extern "C" {

int fe_version(void) { return FE_ABI_VERSION; }

const char *fe_error_string(int code) {
    switch (code) {
    case 0: return "ok";
    case FE_EINVAL: return "finenvs_b200: invalid argument (null pointer, non-positive size, num_assets outside 1..32, or the gather variant without FeSeries.obs_table / FeState.sched)";
    case FE_EALIGN: return "finenvs_b200: pointer not 16-byte aligned";
    case FE_ESMEM: return "finenvs_b200: window does not fit the requested kernel variant";
    case FE_EIO: return "finenvs_b200: cannot open or map the file";
    case FE_ECSV: return "finenvs_b200: CSV record outside the format of the native reader";
    case FE_EDRIVER: return "finenvs_b200: the CUDA driver could not encode the tensor map of the observation-layout table";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "finenvs_b200: unknown error";
    }
}

int fe_tile_envs(int32_t window, int32_t out_f64, int32_t device) {
    (void)device;
    return window > 0 ? pick_tile_envs(window, out_f64 != 0) : 0;
}

int fe_pipe_envs(int32_t window, int32_t out_f64, int32_t stream_flavour) {
    return window > 0 ? pick_pipe_envs(window, out_f64 != 0, stream_flavour ? kPipeSInStream : 0) : 0;
}

const char *fe_step_kernel_name(const FeParams *p, const FeSeries *s, const FeState *st) {
    if (!p) return "";
    const bool f64 = p->out_f64 != 0;
    int sms = 148;
    (void)device_sm_count(p->device, &sms);
    const StepChoice c = choose_kernel(*p, s && s->obs_table && st && st->sched, f64, sms);
    switch (c.kern) {
    case K_PORTFOLIO:
        return f64 ? "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<double>" : "fe_portfolio_book_kernel + fe_portfolio_stream_kernel<float>";
    case K_SPLIT: return f64 ? "fe_book_kernel + fe_stream_kernel<double>" : "fe_book_kernel + fe_stream_kernel<float>";
    case K_GATHER: return f64 ? "fe_gather_kernel<double>" : "fe_gather_kernel<float>";
    case K_PIPE:
        return c.sin == 0 ? (f64 ? "fe_pipe_kernel<double,cached>" : "fe_pipe_kernel<float,cached>")
                          : (f64 ? "fe_pipe_kernel<double,stream>" : "fe_pipe_kernel<float,stream>");
    case K_TILE: return f64 ? "fe_tile_kernel<double>" : "fe_tile_kernel<float>";
    case K_DIRECT: return f64 ? "fe_direct_kernel<double>" : "fe_direct_kernel<float>";
    case K_ERR_TABLE: return "none (the gather variant needs FeSeries.obs_table and FeState.sched)";
    default: return "none (window does not fit the requested variant)";
    }
}

int64_t fe_obs_table_bytes(int64_t num_rows, int32_t window, int32_t out_f64) {
    if (num_rows <= 0 || window <= 0 || pick_gather_stages(window, out_f64 != 0) == 0) return 0;
    if ((ga_rows_per_phase(num_rows, window, out_f64 != 0) << ga_phase_shift(out_f64 != 0)) >= ((int64_t)1 << 31)) return 0;
    return (int64_t)ga_table_bytes(num_rows, window, out_f64 != 0);
}

int fe_obs_table_build(const void *logret_dev, int64_t num_rows, int32_t window, int32_t out_f64, void *table_dev, void *stream) {
    if (!logret_dev || !table_dev || ((uintptr_t)table_dev & 15)) return !logret_dev || !table_dev ? FE_EINVAL : FE_EALIGN;
    const bool f64 = out_f64 != 0;
    if (fe_obs_table_bytes(num_rows, window, out_f64) == 0) return FE_ESMEM;
    cudaStream_t q = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(table_dev, 0, ga_table_bytes(num_rows, window, f64), q);
    if (e != cudaSuccess) return (int)e;
    const int64_t rpp = ga_rows_per_phase(num_rows, window, f64);
    const int64_t threads = num_rows << ga_phase_shift(f64);
    const unsigned blocks = (unsigned)((threads + 255) / 256);
    return with_out_type(f64, [&](auto out_type) {
        using OutT = decltype(out_type);
        fe_obs_table_kernel<OutT><<<blocks, 256, 0, q>>>((const OutT *)logret_dev, num_rows, rpp, (unsigned char *)table_dev);
        return (int)cudaGetLastError();
    });
}

int fe_log_returns(const double *prices_dev, int64_t num_rows, int32_t num_assets, double *logret64_dev,
                   float *logret32_dev, void *stream) {
    if (!prices_dev || num_rows <= 0 || num_assets <= 0) return FE_EINVAL;
    const int64_t n = num_rows * num_assets;
    fe_log_returns_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(prices_dev, num_rows, num_assets,
                                                                                         logret64_dev, logret32_dev);
    return (int)cudaGetLastError();
}

int fe_effective_len(const double *logret64_dev, const int64_t *seg_start_dev, const int32_t *raw_len_dev,
                     int32_t num_segments, int32_t window, int32_t num_assets, int32_t *seg_len_dev, void *stream) {
    if (!logret64_dev || !seg_start_dev || !raw_len_dev || !seg_len_dev || num_segments <= 0) return FE_EINVAL;
    const int64_t threads = (int64_t)num_segments * 32;
    fe_effective_len_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        logret64_dev, seg_start_dev, raw_len_dev, num_segments, window, num_assets, seg_len_dev);
    return (int)cudaGetLastError();
}

int fe_observe(const FeParams *p, const FeSeries *s, const FeState *st, void *obs_dev, void *stream) {
    int rc = check_common(p, s, st);
    if (rc) return rc;
    if (!obs_dev) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    return with_out_type(p->out_f64, [&](auto out_type) {
        return launch<decltype(out_type), true>(*p, *s, *st, nullptr, obs_dev, nullptr, nullptr, nullptr, 0, (cudaStream_t)stream);
    });
}

int fe_step(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, void *obs_dev,
            void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t step_counter, void *stream) {
    int rc = check_step(p, s, st, stats_dev);
    if (rc) return rc;
    if (!actions_dev || !obs_dev || !rewards_dev || !dones_dev) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    return with_out_type(p->out_f64, [&](auto out_type) {
        return launch<decltype(out_type), false>(*p, *s, *st, actions_dev, obs_dev, rewards_dev, dones_dev, stats_dev,
                                                 step_counter, (cudaStream_t)stream);
    });
}

int fe_step_captured(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, void *obs_dev,
                     void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t *step_counter_dev, void *stream) {
    int rc = check_step(p, s, st, stats_dev);
    if (rc) return rc;
    if (!actions_dev || !obs_dev || !rewards_dev || !dones_dev || !step_counter_dev) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    fe_bump_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_counter_dev);
    if ((rc = (int)cudaGetLastError())) return rc;
    return with_out_type(p->out_f64, [&](auto out_type) {
        return launch<decltype(out_type), false>(*p, *s, *st, actions_dev, obs_dev, rewards_dev, dones_dev, stats_dev, 0,
                                                 (cudaStream_t)stream, step_counter_dev);
    });
}

int fe_observe_lazy(const FeParams *p, const FeSeries *s, const FeState *st, int64_t *obs_row0_dev, void *obs_posfeat_dev,
                    void *stream) {
    int rc = check_common(p, s, st);
    if (rc) return rc;
    if (!obs_row0_dev || !obs_posfeat_dev || p->num_assets != 1) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    const Consts k = make_consts(*p);
    const unsigned blocks = (unsigned)((p->num_envs + kThreads - 1) / kThreads);
    return with_out_type(p->out_f64, [&](auto out_type) {
        using OutT = decltype(out_type);
        fe_lazy_kernel<OutT, true><<<blocks, kThreads, 0, (cudaStream_t)stream>>>(
            *p, *s, *st, k, nullptr, obs_row0_dev, (OutT *)obs_posfeat_dev, nullptr, nullptr, nullptr, 0, nullptr);
        return (int)cudaGetLastError();
    });
}

int fe_step_lazy(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_dev, int64_t *obs_row0_dev,
                 void *obs_posfeat_dev, void *rewards_dev, int32_t *dones_dev, FeStats *stats_dev, uint64_t step_counter,
                 void *stream) {
    int rc = check_step(p, s, st, stats_dev);
    if (rc) return rc;
    if (!actions_dev || !obs_row0_dev || !obs_posfeat_dev || !rewards_dev || !dones_dev || p->num_assets != 1) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    const Consts k = make_consts(*p);
    const unsigned blocks = (unsigned)((p->num_envs + kThreads - 1) / kThreads);
    return with_out_type(p->out_f64, [&](auto out_type) {
        using OutT = decltype(out_type);
        fe_lazy_kernel<OutT, false><<<blocks, kThreads, 0, (cudaStream_t)stream>>>(
            *p, *s, *st, k, actions_dev, obs_row0_dev, (OutT *)obs_posfeat_dev, (OutT *)rewards_dev, dones_dev, stats_dev,
            step_counter, nullptr);
        return (int)cudaGetLastError();
    });
}

int fe_backtest(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m, int64_t metrics_capacity,
                FeStats *stats_dev, const float *signal_dev, int32_t num_signals, const int32_t *column_dev,
                uint64_t first_step, int32_t num_steps, void *rewards_dev, int32_t *dones_dev, int32_t history, void *stream) {
    return backtest_entry<false>(p, s, st, m, metrics_capacity, stats_dev, signal_dev, num_signals, column_dev, nullptr,
                                 first_step, num_steps, rewards_dev, dones_dev, history, stream);
}

int fe_backtest_targets(const FeParams *p, const FeSeries *s, const FeState *st, const FeMetricsState *m,
                        int64_t metrics_capacity, FeStats *stats_dev, const float *signal_dev, int32_t num_signals,
                        const int32_t *column_dev, const double *exits_dev, uint64_t first_step, int32_t num_steps,
                        void *rewards_dev, int32_t *dones_dev, int32_t history, void *stream) {
    return backtest_entry<true>(p, s, st, m, metrics_capacity, stats_dev, signal_dev, num_signals, column_dev, exits_dev,
                                first_step, num_steps, rewards_dev, dones_dev, history, stream);
}

int fe_materialize(const FeParams *p, const FeSeries *s, const int64_t *obs_row0_dev, const void *obs_posfeat_dev,
                   void *obs_dev, void *stream) {
    if (!p || !s || !s->logret || !obs_row0_dev || !obs_posfeat_dev || !obs_dev) return FE_EINVAL;
    if (p->num_envs <= 0 || p->window <= 0 || p->num_assets != 1) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    return with_out_type(p->out_f64, [&](auto out_type) {
        return gather_obs<decltype(out_type)>(*p, *s, obs_row0_dev, obs_posfeat_dev, nullptr, p->num_envs, obs_dev,
                                              (cudaStream_t)stream);
    });
}

int fe_gather_obs(const FeParams *p, const FeSeries *s, const int64_t *row0_dev, const void *posfeat_dev,
                  const int64_t *index_dev, int64_t count, void *obs_dev, void *stream) {
    if (!p || !s || !s->logret || !row0_dev || !posfeat_dev || !obs_dev || count < 0) return FE_EINVAL;
    if (p->window <= 0 || p->num_assets != 1) return FE_EINVAL;
    if (((uintptr_t)obs_dev | (uintptr_t)s->obs_table) & 15) return FE_EALIGN;
    if (count == 0) return 0;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    return with_out_type(p->out_f64, [&](auto out_type) {
        return gather_obs<decltype(out_type)>(*p, *s, row0_dev, posfeat_dev, index_dev, count, obs_dev, (cudaStream_t)stream);
    });
}

const char *fe_gather_obs_kernel_name(const FeParams *p, const FeSeries *s) {
    if (!p || !s) return "";
    const bool f64 = p->out_f64 != 0;
    switch (choose_obs_path(*p, *s)) {
    case OBS_TMA: return f64 ? "fe_gather_obs_kernel<double>" : "fe_gather_obs_kernel<float>";
    case OBS_LSU: return f64 ? "fe_materialize_kernel<double>" : "fe_materialize_kernel<float>";
    default: return "none (handles exist for single-asset series only)";
    }
}

// Host-buffer step, pipelined: the envs are cut into chunks (multiples of 1024 envs, so every chunk's slice of
// every array keeps its alignment); chunk c's action upload, kernel and result download run on side stream
// c % kHostStreams, so the upload of chunk c+1 and the download of chunk c-1 overlap the kernel of chunk c
// (two copy engines + SMs busy at once).  Redraws are keyed by global env id, so chunking changes no result.
// dones travel either as int32 per env (dones_host) or bit-packed, 1 bit per env (dones_bits_host): exactly one of the
// two is non-NULL.
static int step_host_impl(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_host, float *actions_dev,
                          void *obs_dev, void *rewards_dev, int32_t *dones_dev, void *rewards_host, int32_t *dones_host,
                          uint32_t *dones_bits_host, FeStats *stats_dev, uint64_t step_counter, void *stream) {
    if (!p || !s || !st || !actions_host || !actions_dev || !rewards_host || (!dones_host == !dones_bits_host)) return FE_EINVAL;
    int rc = check_step(p, s, st, stats_dev);
    if (rc) return rc;
    if (!obs_dev || !rewards_dev || !dones_dev) return FE_EINVAL;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    cudaStream_t q = (cudaStream_t)stream;
    const int64_t n = p->num_envs;
    const int A = p->num_assets;
    const size_t osz = p->out_f64 ? 8 : 4;
    const void *dones_any = dones_host ? (const void *)dones_host : (const void *)dones_bits_host;
    // Zero-copy mode: when all three host buffers are pinned (mapped into the device's address space), the step
    // kernel reads the actions from them and writes rewards / dones to them directly over PCIe — 12 bytes per env
    // (8.1 with bit-packed dones, which a small kernel writes after the step) spread over the whole kernel, no
    // copy-engine hop, no head (upload) or tail (download) outside the kernel.
    // rewards_dev / dones_dev are written as well (device-side consumers); actions_dev is left untouched.
    // (Tried instead: copy-engine upload of the actions in chunks behind the already running kernel, each chunk
    // followed by a 4-byte copy bumping an arrival counter the envs poll.  Same speed on one GPU (0.317 ms per
    // 1 Mi-env step) and on eight (0.67 vs 0.68 ms: with 8 ranks the host side of PCIe, not the read latency, is the
    // limit), more machinery, and a kernel that waits for copies queued after it deadlocks under anything that
    // serialises launches (ncu, CUDA_LAUNCH_BLOCKING=1) — dropped.)
    int sms = 0;
    if ((rc = device_sm_count(p->device, &sms))) return rc;
    if (!env_override("FE_HOST_NO_ZEROCOPY")) {
        cudaPointerAttributes aa, ar, ad;
        const bool ok = cudaPointerGetAttributes(&aa, actions_host) == cudaSuccess && aa.type == cudaMemoryTypeHost &&
                        aa.devicePointer && cudaPointerGetAttributes(&ar, rewards_host) == cudaSuccess &&
                        ar.type == cudaMemoryTypeHost && ar.devicePointer &&
                        cudaPointerGetAttributes(&ad, dones_any) == cudaSuccess && ad.type == cudaMemoryTypeHost &&
                        ad.devicePointer;
        (void)cudaGetLastError(); // an unregistered pointer leaves a sticky-free error on old drivers
        // Only for the persistent (and the portfolio) kernels: their bookkeeper warps run tiles ahead, which hides the
        // PCIe read latency, and they write rewards / dones 32 envs (128 bytes) per store.  A tile / direct block would
        // sit on its shared memory while it waits for its actions and write 16-byte PCIe packets (measured W = 60,
        // 1 Mi envs: 1.04 ms zero-copy, 0.77 ms with a copy-engine upload + zero-copy writes, vs 0.36 ms
        // device-resident): those take the chunked copy pipeline below.
        // Small populations are the exception: there the whole step is a few microseconds and the three copies, two events
        // and their stream hops of the chunked path cost more than the PCIe round trips (1024 envs: C call 25.6 -> 20.0 us, bit-packed
        // 35.0 -> 24.8 us; profiles/r02_e2e_probe_small_populations.txt), so tile / direct launches of <= 32 Ki envs go zero-copy too.
        const StepKernel kk = choose_kernel(*p, s->obs_table && st->sched, p->out_f64 != 0, sms).kern;
        const bool small = n <= 32768;
        if (ok && ((kk != K_TILE && kk != K_DIRECT) || small)) {
            const float *a = (const float *)aa.devicePointer;
            int32_t *dmirror = dones_host ? (int32_t *)ad.devicePointer : nullptr;
            uint32_t *bmirror = dones_bits_host ? (uint32_t *)ad.devicePointer : nullptr;
            // the actions are read from the host: actions_dev (>= 4 bytes per env) is free to stage the packed bits
            uint32_t *stage = reinterpret_cast<uint32_t *>(actions_dev);
            int packed_inline = 0;
            rc = with_out_type(p->out_f64, [&](auto out_type) {
                return launch<decltype(out_type), false>(*p, *s, *st, a, obs_dev, rewards_dev, dones_dev, stats_dev, step_counter,
                                                         q, nullptr, ar.devicePointer, dmirror, bmirror, stage, &packed_inline);
            });
            if (rc) return rc;
            if (dones_bits_host && packed_inline != 1) {
                const int64_t nwords = (n + 31) / 32;
                if (packed_inline == 0 && small) { // a handful of words: straight to the host, one launch less
                    fe_pack_dones_kernel<<<(unsigned)((n + 255) / 256), 256, 0, q>>>(dones_dev, n, (uint32_t *)ad.devicePointer);
                } else {
                    if (packed_inline == 0)
                        fe_pack_dones_kernel<<<(unsigned)((n + 255) / 256), 256, 0, q>>>(dones_dev, n, stage);
                    fe_flush_bits_kernel<<<(unsigned)((nwords + 255) / 256), 256, 0, q>>>(stage, nwords, (uint32_t *)ad.devicePointer);
                }
                if ((rc = (int)cudaGetLastError())) return rc;
            }
            return (int)cudaStreamSynchronize(q);
        }
    }
    const int ov_chunks = env_override("FE_HOST_CHUNKS");
    int chunks = ov_chunks > 0 ? ov_chunks : 4;
    int64_t per = ((n + chunks - 1) / chunks + 1023) & ~(int64_t)1023;
    if (per < 16384) per = 16384; // below this a chunk's kernel is shorter than the launch + copy set-up it would hide
    chunks = (int)((n + per - 1) / per);
    HostPipe *hp = nullptr;
    if (chunks > 1) {
        hp = host_pipe(p->device);
        if (!hp) return (int)cudaGetLastError();
        cudaError_t e = cudaEventRecord(hp->start, q);
        if (e != cudaSuccess) return (int)e;
    }
    for (int c = 0; c < chunks; ++c) {
        const int64_t off = (int64_t)c * per, cnt = off + per <= n ? per : n - off;
        cudaStream_t cs = hp ? hp->s[c % kHostStreams] : q;
        cudaError_t e;
        if (hp && c < kHostStreams && (e = cudaStreamWaitEvent(cs, hp->start, 0)) != cudaSuccess) return (int)e;
        e = cudaMemcpyAsync(actions_dev + off * A, actions_host + off * A, (size_t)cnt * A * sizeof(float),
                            cudaMemcpyHostToDevice, cs);
        if (e != cudaSuccess) return (int)e;
        FeParams pc = *p;
        pc.num_envs = cnt;
        pc.env_id_base = p->env_id_base + off;
        if (pc.variant == FE_VARIANT_GATHER) pc.variant = FE_VARIANT_AUTO;
        FeState sc = *st;
        sc.sched = nullptr; // the chunks run concurrently on side streams: they cannot share the gather kernel's tile counter
        sc.seg += off; sc.ptr += off; sc.cash += off;
        sc.long_sh += off * A; sc.short_sh += off * A; sc.margin += off * A;
        if (sc.terminated) sc.terminated += off;
        if (sc.ep_return) sc.ep_return += off;
        if (sc.ep_len) sc.ep_len += off;
        const size_t obs_off = (size_t)off * p->window * 5 * A * osz;
        rc = with_out_type(p->out_f64, [&](auto out_type) {
            return launch<decltype(out_type), false>(pc, *s, sc, actions_dev + off * A, (char *)obs_dev + obs_off,
                                                     (char *)rewards_dev + off * osz, dones_dev + off, stats_dev, step_counter, cs);
        });
        if (rc) return rc;
        e = cudaMemcpyAsync((char *)rewards_host + off * osz, (char *)rewards_dev + off * osz, (size_t)cnt * osz,
                            cudaMemcpyDeviceToHost, cs);
        if (e != cudaSuccess) return (int)e;
        if (dones_host) {
            e = cudaMemcpyAsync(dones_host + off, dones_dev + off, (size_t)cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, cs);
        } else {
            // the chunk's actions are consumed: its slice of actions_dev (>= cnt * 4 bytes) is scratch for the packed bits
            uint32_t *bits_dev = reinterpret_cast<uint32_t *>(actions_dev + off * A);
            fe_pack_dones_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, cs>>>(dones_dev + off, cnt, bits_dev);
            if ((rc = (int)cudaGetLastError())) return rc;
            e = cudaMemcpyAsync(dones_bits_host + (off >> 5), bits_dev, (size_t)((cnt + 31) / 32) * 4, cudaMemcpyDeviceToHost, cs);
        }
        if (e != cudaSuccess) return (int)e;
    }
    if (hp) { // the caller's stream continues only after every side stream has finished
        for (int k = 0; k < kHostStreams && k < chunks; ++k) {
            cudaError_t e = cudaEventRecord(hp->done[k], hp->s[k]);
            if (e != cudaSuccess) return (int)e;
            if ((e = cudaStreamWaitEvent(q, hp->done[k], 0)) != cudaSuccess) return (int)e;
        }
    }
    return (int)cudaStreamSynchronize(q);
}

int fe_step_host(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_host, float *actions_dev,
                 void *obs_dev, void *rewards_dev, int32_t *dones_dev, void *rewards_host, int32_t *dones_host,
                 FeStats *stats_dev, uint64_t step_counter, void *stream) {
    if (!dones_host) return FE_EINVAL;
    return step_host_impl(p, s, st, actions_host, actions_dev, obs_dev, rewards_dev, dones_dev, rewards_host, dones_host, nullptr,
                          stats_dev, step_counter, stream);
}

int fe_step_host_packed(const FeParams *p, const FeSeries *s, const FeState *st, const float *actions_host, float *actions_dev,
                        void *obs_dev, void *rewards_dev, int32_t *dones_dev, void *rewards_host, uint32_t *dones_bits_host,
                        FeStats *stats_dev, uint64_t step_counter, void *stream) {
    if (!dones_bits_host) return FE_EINVAL;
    return step_host_impl(p, s, st, actions_host, actions_dev, obs_dev, rewards_dev, dones_dev, rewards_host, nullptr, dones_bits_host,
                          stats_dev, step_counter, stream);
}

int fe_reset_all(const FeParams *p, const FeSeries *s, const FeState *st, uint64_t step_counter, int32_t redraw,
                 void *stream) {
    int rc = check_common(p, s, st);
    if (rc) return rc;
    DeviceGuard guard(p->device);
    if (guard.rc) return guard.rc;
    fe_reset_all_kernel<<<(unsigned)((p->num_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*p, *s, *st, step_counter,
                                                                                                 redraw);
    return (int)cudaGetLastError();
}

#ifdef FE_GATHER_CLOCKS
int fe_debug_gather_clocks(unsigned long long out[16]) { return (int)cudaMemcpyFromSymbol(out, fe_gather_clk, 128); }
int fe_debug_gather_blocks(unsigned long long out[480]) { return (int)cudaMemcpyFromSymbol(out, fe_gather_block_ns, 480 * 8); }
#endif

void fe_philox(uint64_t seed, uint64_t env_id, uint64_t step, uint32_t kind, uint32_t out[4]) {
    philox4x32_10(seed, env_id, step, kind, out);
}

} // extern "C"
