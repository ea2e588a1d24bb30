"""The ES kernels of csrc/fe_es.cu against float64 references written here, at the shapes and edges where each of them
branches: the three forward kernels (fast, streaming, generic) and their launch shapes, the two-stage gradient over
many 512-pair slabs, the episode store at scale and on overflow, and the perturbation stream's exact layout.

Forward tolerances are derived per output, not fixed.  Every kernel sums a dot product as FMA chains of at most
ceil((in + 1) / 32) + 5 terms per lane, one fmaf(sigma, eps.x, theta.x) and a 5-level butterfly, so with
u = 2^-24 and gamma(n) = n u / (1 - n u) the pre-activation error of a layer is at most
    gamma(ceil((in + 1) / 32) + 12) * (sum|theta_i x_i| + sigma sum|eps_i x_i| + |b| + sigma |eps_b|) + sum|w'_i| e_i
where e_i bounds the error of the layer's inputs; tanh passes an error d on as at most d (1 - y^2) + d^2, and tanhf
adds at most 2 ulp.  The test asserts |kernel - reference| <= 2 e_L.  That bound is worst-case: its propagated part
grows by sum|w| per hidden layer, so for wide multi-layer networks it is about 1000 times the measured error and its
median is held below 2e-3 there (1e-4 elsewhere) rather than 1e-5.  Every case therefore also meets an empirical cap
on the measured error (_max_err)."""
import ctypes
import math
import zlib

import numpy as np
import pytest
import torch

U = 2.0 ** -24
FE_EINVAL, FE_ESMEM = -1, -3
FAST, STREAM, GEN = "fe_es_forward_fast_kernel", "fe_es_forward_stream_kernel", "fe_es_forward_kernel"


def gamma(n):
    return n * U / (1 - n * U)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def _fe_net(_lib, shape):
    return _lib.FeEsNet(len(shape) - 1, (ctypes.c_int32 * (_lib.FE_ES_MAX_LAYERS + 1))(*shape))


def kernel_name(_lib, shape, lazy, aligned=True):
    return _lib.lib().fe_es_forward_kernel_name(ctypes.byref(_fe_net(_lib, shape)), int(lazy), int(aligned)).decode()


# shape: (lazy handles, dense aligned, dense at a 4-byte offset); None: the shape has no lazy form (in % 5 != 0)
ROUTES = {
    (300, 8, 1): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=3"),     # BASELINE config 5
    (5, 1): (f"{FAST}<lazy>", f"{STREAM}<dense> U=4", f"{STREAM}<dense> U=4"),     # R = 1: 20-byte rows are not 16-byte granular
    (20, 5): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=4"),
    (155, 8, 1): (f"{FAST}<lazy>", f"{STREAM}<dense> U=4", f"{STREAM}<dense> U=4"),   # R = 31
    (160, 8, 1): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=4"),         # R = 32: bias row on lane 0's second slot
    (165, 8, 1): (f"{FAST}<lazy>", f"{STREAM}<dense> U=4", f"{STREAM}<dense> U=4"),   # R = 33
    (315, 8, 1): (f"{FAST}<lazy>", f"{STREAM}<dense> U=3", f"{STREAM}<dense> U=3"),   # R = 63: the last fast shape
    (320, 8, 1): (f"{GEN}<lazy,theta_smem>", f"{GEN}<dense,theta_smem>", f"{GEN}<dense,theta_smem>"),   # R = 64, in + 1 > 320
    (300, 4): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=3"),            # L = 1
    (300, 8, 12): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=3"),        # 9..16 actions: not in registers
    (300, 8, 8, 8, 2): (f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<dense> U=3"),   # L = 4
    (300, 9, 1): (f"{STREAM}<lazy> U=3", f"{STREAM}<dense> U=3", f"{STREAM}<dense> U=3"),   # 9 first-layer outputs
    (315, 9, 1): (f"{STREAM}<lazy> U=3", f"{STREAM}<dense> U=3", f"{STREAM}<dense> U=3"),
    (300, 256, 256, 1): (f"{STREAM}<lazy> U=2", f"{STREAM}<dense> U=2", f"{STREAM}<dense> U=2"),   # the reference default
    (300, 300, 300, 1): (f"{STREAM}<lazy> U=1", f"{STREAM}<dense> U=1", f"{STREAM}<dense> U=1"),
    (300, 64, 64, 1): (f"{STREAM}<lazy> U=3", f"{STREAM}<dense> U=3", f"{STREAM}<dense> U=3"),
    (60, 16, 4, 2): (f"{STREAM}<lazy> U=4", f"{STREAM}<dense> U=4", f"{STREAM}<dense> U=4"),
    (60, 64, 32, 16, 3): (f"{STREAM}<lazy> U=4", f"{STREAM}<dense> U=4", f"{STREAM}<dense> U=4"),
    (319, 16, 1): (None, f"{STREAM}<dense> U=3", f"{STREAM}<dense> U=3"),              # in + 1 = 320: the streaming limit
    (400, 12, 2): (f"{GEN}<lazy,theta_smem>", f"{GEN}<dense,theta_smem>", f"{GEN}<dense,theta_smem>"),
    (400, 64, 2): (f"{GEN}<lazy,theta_global>", f"{GEN}<dense,theta_global>", f"{GEN}<dense,theta_global>"),
    (1000, 256, 1): (f"{GEN}<lazy,theta_global>", f"{GEN}<dense,theta_global>", f"{GEN}<dense,theta_global>"),
}


def test_forward_routing_table(lib):
    """fe_es_forward_kernel_name is the routing fe_es_forward launches with (one host function serves both): which
    kernel, and the streaming kernel's pairs per warp U.  Pinned here so that a change of a shared-memory limit or a
    threshold shows up as a change of coverage."""
    for shape, (lazy, dense, off4) in ROUTES.items():
        if lazy is not None:
            assert kernel_name(lib, shape, True) == lazy, shape
            assert kernel_name(lib, shape, True, aligned=False) == lazy, shape   # handles have no dense pointer
        assert kernel_name(lib, shape, False) == dense, shape
        assert kernel_name(lib, shape, False, aligned=False) == off4, shape
    for shape in ((1900, 4, 1), (1900, 4, 1, 1)):
        assert kernel_name(lib, shape, True).startswith("none (FE_ESMEM")
    net = lib.FeEsNet(0, (ctypes.c_int32 * (lib.FE_ES_MAX_LAYERS + 1))(300, 8, 1, 0, 0))
    assert lib.lib().fe_es_forward_kernel_name(ctypes.byref(net), 1, 1) == b""


# ---------------------------------------------------------------------------------------------------------------------
# forward values
# ---------------------------------------------------------------------------------------------------------------------
class _Handles:
    """The lazy observation handle ParallelMLP.forward reads (what TimeSeriesEnv.step_lazy returns), built directly."""

    def __init__(self, logret, row0, posfeat, window):
        self.logret, self.row0, self.posfeat, self.window = logret, row0, posfeat, window
        self.shape = (row0.numel(), 5 * window)


def _logret_table(kind, rows, seed):
    """A (rows, 4) f32 log-return table on the GPU: staged from a GBM series ("series") or drawn directly."""
    if kind == "series":
        from finenvs_b200.data import loader
        from parity_utils import gbm_ohlc

        rng = np.random.default_rng(seed)
        bars = 50
        prices = np.round(gbm_ohlc(rng, rows, 0.02), 4)
        seg_start, seg_len = loader.regular_segments(rows, bars, 1)
        return loader.stage_series(prices, seg_start, seg_len, 1, "cuda:0", torch.float32).logret
    g = torch.Generator(device="cuda").manual_seed(seed)
    scale = {"n1": 1.0, "n30": 30.0, "zeros": 0.0}[kind]
    return (torch.randn((rows, 4), generator=g, device="cuda") * scale).contiguous()


def _inputs(kind, N, W, in0, seed):
    """(handles or None, dense f32 inputs).  The dense rows of a window are built here by indexing the table, never by a
    step or materialise kernel: obs[e, 5j + c] = logret[row0[e] + j, c] (c < 4), obs[e, 5j + 4] = posfeat[e]."""
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    if W is None:
        scale = {"n1": 1.0, "n30": 30.0, "zeros": 0.0, "series": 1.0}[kind]
        return None, (torch.randn((N, in0), generator=g, device="cuda") * scale).contiguous()
    rows = max(4 * W + 64, 4096, min(2 * N, 1 << 20))
    table = _logret_table(kind, rows, seed)
    row0 = torch.randint(0, rows - W + 1, (N,), generator=g, device="cuda", dtype=torch.int64)
    pf = torch.rand((N,), generator=g, device="cuda") * 2 - 1
    if kind == "zeros":
        pf.zero_()
    win = table[row0[:, None] + torch.arange(W, device="cuda")[None, :]]            # (N, W, 4)
    dense = torch.cat([win, pf[:, None, None].expand(N, W, 1)], 2).reshape(N, 5 * W).contiguous()
    return _Handles(table, row0, pf, W), dense


def _mlp_f64(x, Ws, Bs, ew, eb, s):
    """One sign of a population slice in f64: x (n, in0); Ws/Bs shared f64 layers; ew/eb per-env unit perturbations
    (n, in, out) / (n, 1, out) or None (evaluation envs); s = +-sigma.  Returns (actions, error bound)."""
    e = torch.zeros_like(x)
    for li, (W, b) in enumerate(zip(Ws, Bs)):
        ax = x.abs()
        if ew is None:
            wp, bp = W.expand(x.shape[0], *W.shape), b
            mag = ax @ W.abs() + b.abs()
        else:
            wp, bp = W + s * ew[li], b + s * eb[li][:, 0]
            mag = ax @ W.abs() + abs(s) * torch.einsum("ni,nio->no", ax, ew[li].abs()) + b.abs() + abs(s) * eb[li][:, 0].abs()
        z = torch.einsum("ni,nio->no", x, wp) + bp
        depth = math.ceil((W.shape[0] + 1) / 32) + 12
        pre = gamma(depth) * mag + torch.einsum("ni,nio->no", e, wp.abs())
        y = torch.tanh(z)
        e = pre * (1 - y * y) + pre * pre + 4 * U * (y.abs() + pre)
        x = y
    return x, e


def forward_reference(net, X, sigma, num_pairs, num_eval, rows=None, drop=None):
    """f64 actions and bounds of the envs `rows` (default: all) of `net` on inputs X (N, in0) f32 (GPU).
    `drop`: input index of layer 0 left out of the reference (a deliberately wrong reference)."""
    N = X.shape[0]
    rows = torch.arange(N, device="cuda") if rows is None else rows
    Ws = [w.double() for w in net.weight_layers]
    Bs = [b.double()[0] for b in net.bias_layers]
    s = float(np.float32(sigma))
    Xd = X.double()
    if drop is not None:
        if drop == "bias":
            Bs[0] = torch.zeros_like(Bs[0])
        else:
            Xd[:, drop] = 0.0
    params = sum(w.numel() + b.numel() for w, b in zip(Ws, Bs))
    chunk = max(1, min(16384, (1 << 27) // params))
    out = torch.empty((rows.numel(), Ws[-1].shape[1]), dtype=torch.float64, device="cuda")
    bnd = torch.empty_like(out)
    for c0 in range(0, rows.numel(), chunk):
        r = rows[c0: c0 + chunk]
        tr = r < 2 * num_pairs
        if tr.any():
            rt = r[tr]
            pair = torch.where(rt < num_pairs, rt, rt - num_pairs)
            sgn = torch.where(rt < num_pairs, 1.0, -1.0).double()
            ew, eb = net.unpack(net._eps[pair].double())
            # +-sigma per env: fold the sign into the perturbation (exact)
            ew = [w * sgn[:, None, None] for w in ew]
            eb = [b * sgn[:, None, None] for b in eb]
            y, e = _mlp_f64(Xd[rt], Ws, Bs, ew, eb, s)
            out[c0: c0 + r.numel()][tr], bnd[c0: c0 + r.numel()][tr] = y, e
        if (~tr).any():
            y, e = _mlp_f64(Xd[r[~tr]], Ws, Bs, None, None, 0.0)
            out[c0: c0 + r.numel()][~tr], bnd[c0: c0 + r.numel()][~tr] = y, e
    return out, bnd


# units (pairs + eval envs) one past a full wave of the kernel's warps: fast and streaming run one block of 12 warps
# per SM (a streaming warp takes U units at a time); the generic kernel runs 8 warps per block, and a (400, 12, 2)
# block (78 KB of shared memory) fits twice per SM
WAVES = {"wave_fast": lambda sms: sms * 12 + 1, "wave_stream4": lambda sms: sms * 12 * 4 + 1,
         "wave_generic": lambda sms: sms * 2 * 8 + 1}


# id: (shape, pairs, eval envs, modes, input kind, sigma); modes: "lazy", "dense", "off4" (dense at a 4-byte offset)
FWD = {
    # fast path, lazy: R at the lane-slot boundaries x first-layer widths (second layer in registers)
    **{f"fast_R{R}_w{w}": ((5 * R, w, 1), p, e, ("lazy",), "series", 0.02)
       for (R, w), (p, e) in zip([(R, w) for R in (1, 4, 31, 32, 33, 60, 63) for w in (1, 5, 8)],
                                  [(1, 0), (2, 1), (13, 7), (40, 0), (37, 1), (64, 7)] * 4)},
    "fast_L1": ((300, 4), 13, 7, ("lazy", "dense"), "series", 0.3),
    "fast_L2_tail_regs": ((300, 5, 3), 41, 1, ("lazy", "dense"), "series", 0.3),
    "fast_L2_12_actions": ((300, 8, 12), 41, 7, ("lazy", "dense"), "series", 0.3),
    "fast_L3": ((300, 8, 8, 2), 29, 1, ("lazy", "dense"), "n30", 0.3),
    "fast_L4": ((300, 8, 8, 8, 2), 29, 7, ("lazy", "dense"), "series", 0.02),
    "fast_sigma0": ((300, 8, 1), 100, 7, ("lazy", "dense"), "series", 0.0),
    "fast_zeros": ((300, 8, 1), 100, 1, ("lazy", "dense"), "zeros", 0.3),
    "fast_n30": ((300, 8, 1), 500, 0, ("lazy", "dense"), "n30", 0.3),
    "fast_dense_off4": ((300, 8, 1), 100, 7, ("lazy", "off4"), "series", 0.3),
    "fast_R31_dense_streams": ((155, 8, 1), 100, 7, ("lazy", "dense"), "series", 0.3),
    "fast_R33_dense_streams": ((165, 8, 1), 99, 1, ("lazy", "dense"), "n1", 0.3),
    "fast_wave_plus_one": ((300, 8, 1), "wave_fast", 0, ("lazy", "dense"), "series", 0.02),
    # streaming
    "stream_default_odd_pairs": ((300, 256, 256, 1), 13, 1, ("lazy", "dense"), "series", 0.02),   # U = 2, 13 % 2 = 1
    "stream_default_7_eval": ((300, 256, 256, 1), 5, 7, ("dense",), "n1", 0.3),
    "stream_in319": ((319, 16, 1), 29, 7, ("dense", "off4"), "n1", 0.3),
    "stream_R63_9_out": ((315, 9, 1), 62, 1, ("lazy", "dense"), "series", 0.3),
    "stream_4_layers": ((60, 64, 32, 16, 3), 100, 7, ("lazy", "dense"), "n1", 0.3),
    "stream_U1": ((300, 300, 300, 1), 6, 1, ("dense",), "n1", 0.3),
    "stream_U4_mod1": ((60, 16, 4, 2), 13, 7, ("lazy", "dense"), "series", 0.3),
    "stream_U4_mod2": ((60, 16, 4, 2), 14, 1, ("lazy", "dense"), "n30", 0.3),
    "stream_U4_mod3": ((60, 16, 4, 2), 15, 7, ("lazy", "dense"), "zeros", 0.02),
    "stream_U4_wave_plus_one": ((60, 16, 4, 2), "wave_stream4", 1, ("lazy", "dense"), "series", 0.02),
    "stream_U3_pairs_2": ((300, 64, 64, 1), 2, 7, ("dense",), "n1", 0.0),
    # generic
    "generic_lazy_R64": ((320, 8, 1), 13, 7, ("lazy", "dense"), "series", 0.3),
    "generic_theta_smem": ((400, 12, 2), 13, 1, ("dense", "lazy"), "n1", 0.3),
    "generic_theta_global": ((400, 64, 2), 13, 7, ("dense",), "n30", 0.3),
    "generic_1000_256": ((1000, 256, 1), 3, 1, ("dense",), "n1", 0.02),
    "generic_wave_plus_one": ((400, 12, 2), "wave_generic", 0, ("dense",), "n1", 0.02),
}


# Empirical cap on |kernel - reference| of every forward case.  Measured on one B200 (1000 W): at most 2.3e-6 over
# all cases with O(1) inputs, the wide 300-256-256-1, 300-300-300-1 and 1000-256-1 networks included; 2.2e-5 for
# 300-8-1 on N(0, 30) inputs, whose pre-activations are 30 times larger.  A 1e-4 error in any layer fails it.
def _max_err(kind):
    return 1e-4 if kind == "n30" else 1e-5


def _median_cap(shape):
    # a worst-case bound: about 1.5e-5 at the median for 300-8-1 on O(1) inputs, 5e-5 for 300-8-8-8-2.  Its
    # propagated part grows by sum|w| per hidden layer (about 18 for a 256-wide one) while the actual error does not, so
    # wide multi-layer networks get the looser cap; self-check 2 shows the bound still sees a single missing input
    # term there
    return 1e-4 if sum(shape[1:-1]) <= 64 and shape[0] <= 400 else 2e-3


def _run_case(lib, shape, num_pairs, num_eval, modes, kind, sigma, seed, sample=None):
    from finenvs_b200.agents.networks import ParallelMLP

    N = 2 * num_pairs + num_eval
    torch.manual_seed(seed)
    net = ParallelMLP(N, num_eval, shape, noise_std_dev=sigma, device_id=0, seed=seed, action_noise_std=0.0)
    net.perturb_parameters()
    W = shape[0] // 5 if shape[0] % 5 == 0 and "lazy" in modes else None
    handles, X = _inputs(kind, N, W, shape[0], seed)
    outs = {}
    for mode in modes:
        if mode == "lazy":
            want = kernel_name(lib, shape, True)
            if shape in ROUTES:
                assert want == ROUTES[shape][0]
            assert net.forward_kernel_name(lazy=True) == want
            outs[mode] = (net.forward(handles), want)
        elif mode == "dense":
            want = kernel_name(lib, shape, False)
            if shape in ROUTES:
                assert want == ROUTES[shape][1]
            assert net.forward_kernel_name(lazy=False) == want
            outs[mode] = (net.forward(X), want)
        else:
            buf = torch.empty(X.numel() + 4, dtype=torch.float32, device="cuda")
            Xo = buf[1: 1 + X.numel()].view(X.shape)
            Xo.copy_(X)
            assert Xo.data_ptr() % 16 == 4 and Xo.is_contiguous()
            want = kernel_name(lib, shape, False, aligned=False)
            assert net.forward_kernel_name(lazy=False, obs_aligned=False) == want
            outs[mode] = (net.forward(Xo), want)
    # same kernel for two input forms -> same bits (dense rows are the window as it lies in the series)
    names = {m: w for m, (_, w) in outs.items()}
    if "lazy" in outs:
        for m in outs:
            if m != "lazy" and names[m].replace("<dense", "<lazy") == names["lazy"]:
                assert torch.equal(outs[m][0], outs["lazy"][0]), (m, names[m])
    rows = None
    if sample is not None:
        rows = torch.randperm(N, generator=torch.Generator().manual_seed(seed), device="cpu")[:sample].sort().values.cuda()
    ref, bnd = forward_reference(net, X, sigma, num_pairs, num_eval, rows)
    for m, (a, want) in outs.items():
        got = (a if rows is None else a[rows]).double()
        err = (got - ref).abs()
        worst = int((err - 2 * bnd).argmax())
        assert bool((err <= 2 * bnd).all()), (m, want, float(err.flatten()[worst]), float(bnd.flatten()[worst]))
    # self-check 1: the bound is tight enough to mean something
    assert float(bnd.median()) < _median_cap(shape), float(bnd.median())
    # the measured error against an empirical cap, far below the worst-case bound of the wide networks
    worst_err = max(float(((a if rows is None else a[rows]).double() - ref).abs().max()) for a, _ in outs.values())
    assert worst_err <= _max_err(kind), worst_err
    # self-check 2: a reference missing one input term of layer 0 fails the same comparison
    drop = "bias" if kind == "zeros" else shape[0] - 1
    bad, _ = forward_reference(net, X, sigma, num_pairs, num_eval, rows, drop=drop)
    a = next(iter(outs.values()))[0]
    got = (a if rows is None else a[rows]).double()
    assert not bool(((got - bad).abs() <= 2 * bnd).all()), "the bound cannot see a missing input term"
    return net, outs, worst_err


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(FWD))
def test_forward_vs_f64(lib, case):
    shape, pairs, num_eval, modes, kind, sigma = FWD[case]
    if isinstance(pairs, str):
        pairs = WAVES[pairs](torch.cuda.get_device_properties(0).multi_processor_count) - num_eval
    _run_case(lib, shape, pairs, num_eval, modes, kind, sigma, seed=zlib.crc32(case.encode()) % 1000 + 1)


@pytest.mark.gpu
def test_forward_config5_population(lib):
    """BASELINE config 5: 512 Ki envs x 300-8-1 on a long staged series; 64 Ki sampled envs against the reference,
    lazy == dense on every env."""
    _run_case(lib, (300, 8, 1), 1 << 18, 0, ("lazy", "dense"), "series", 0.05, seed=5, sample=1 << 16)


@pytest.mark.gpu
def test_forward_esmem_raises_without_a_launch(lib):
    from finenvs_b200.agents.networks import ParallelMLP

    net = ParallelMLP(4, 0, (1900, 4, 1), device_id=0, seed=1, action_noise_std=0.0)
    net.perturb_parameters()
    assert net.forward_kernel_name(lazy=False).startswith("none (FE_ESMEM")
    x = torch.randn((4, 1900), device="cuda")
    torch.cuda.synchronize()
    with pytest.raises(lib.FeError, match=rf"\({FE_ESMEM}\)"):
        net.forward(x)
    torch.cuda.synchronize()     # nothing was launched, nothing faulted


def test_forward_cases_reach_every_kernel(lib):
    """The forward value cases above (each asserts its kernel name) cover every kernel and launch shape; host-only."""
    reached = {kernel_name(lib, (300, 8, 1), lazy) for lazy in (True, False)}      # test_forward_config5_population
    for shape, _, _, modes, _, _ in FWD.values():
        reached |= {kernel_name(lib, shape, m == "lazy", aligned=m != "off4") for m in modes}
    want = [f"{FAST}<lazy>", f"{FAST}<dense>", f"{STREAM}<lazy> U=4", f"{STREAM}<dense> U=4", f"{STREAM}<lazy> U=2",
            f"{STREAM}<dense> U=1", f"{STREAM}<dense> U=3", f"{GEN}<lazy,theta_smem>", f"{GEN}<dense,theta_smem>",
            f"{GEN}<dense,theta_global>"]
    missing = [w for w in want if w not in reached]
    assert not missing, missing


# ---------------------------------------------------------------------------------------------------------------------
# gradient
# ---------------------------------------------------------------------------------------------------------------------
def _grad_f64(eps, w):
    """g[q] = sum_p w_p eps_pq and sum_p |w_p eps_pq| in f64, chunked over pairs."""
    g = torch.zeros(eps.shape[1], dtype=torch.float64, device="cuda")
    a = torch.zeros_like(g)
    wd = w.double()
    for p0 in range(0, eps.shape[0], 8192):
        e = eps[p0: p0 + 8192].double()
        g += wd[p0: p0 + 8192] @ e
        a += wd[p0: p0 + 8192].abs() @ e.abs()
    return g, a


def _weights(kind, pairs, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "normal":
        return torch.randn((pairs,), generator=g, device="cuda")
    # EvoAgent: one episode per env, centred ranks in [-0.5, 0.5], pair weight = rank(+) - rank(-)
    n = 2 * pairs
    pos = torch.empty(n, dtype=torch.float32, device="cuda")
    pos[torch.randperm(n, generator=g, device="cuda")] = torch.arange(n, dtype=torch.float32, device="cuda")
    r = pos / max(n - 1, 1) - 0.5
    return (r[:pairs] - r[pairs:]).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,pairs", [((60, 8, 1), p) for p in (1, 511, 512, 513, 1025, 10001, 1 << 18)]
                         + [((300, 256, 1), p) for p in (1, 513, 10001)] + [((300, 8, 1), 1 << 18)])
@pytest.mark.parametrize("wkind", ["normal", "ranks"])
def test_gradient_vs_f64(lib, shape, pairs, wkind):
    """fe_es_gradient: 512-pair slabs (ragged last slab, up to 512 of them) then the slabs in order; P_pad below 1024
    (one x-block of the partial kernel) and far above it.  Deterministic: two calls give the same bits."""
    from finenvs_b200.agents.networks import ParallelMLP

    L = lib.lib()
    net = ParallelMLP(2 * pairs, 0, shape, device_id=0, seed=pairs + len(shape), action_noise_std=0.0)
    net.perturb_parameters()
    w = _weights(wkind, pairs, pairs)
    P = net.params_padded
    slabs = (pairs + 511) // 512
    scratch = torch.full((int(L.fe_es_gradient_scratch(net._pnet, pairs)),), float("nan"), device="cuda")
    assert scratch.numel() == slabs * P
    outs = []
    for _ in range(2):
        g = torch.full((P,), float("nan"), device="cuda")
        lib.check(L.fe_es_gradient(net._pnet, net._eps.data_ptr(), w.data_ptr(), pairs, scratch.data_ptr(), g.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream), "fe_es_gradient")
        outs.append(g)
    assert torch.equal(outs[0], outs[1])
    ref, mag = _grad_f64(net._eps, w)
    err = (outs[0].double() - ref).abs()
    bound = gamma(512 + slabs) * mag
    assert bool((err <= bound).all()), float((err - bound).max())
    # padding columns of the packed layout carry eps = 0 -> exactly 0
    assert bool(((mag == 0) <= (outs[0] == 0)).all())
    # the reduction does not get slabs wrong: dropping the last slab's pairs would move the result out of the bound
    if slabs > 1:
        ref_short, _ = _grad_f64(net._eps[: (slabs - 1) * 512], w[: (slabs - 1) * 512])
        assert not bool(((outs[0].double() - ref_short).abs() <= bound).all())


@pytest.mark.gpu
def test_update_parameters_adam_step_vs_f64(lib):
    """One generation update through ParallelMLP.update_parameters at 10 001 pairs against an f64 restatement of
    oracle_es.update_parameters.  Adam's first step is ~lr * sign(g), so the bound follows the update's own
    sensitivity: |h(g + d) - h(g - d)| with h(g) = m / (sqrt(v) + 1e-8) and d the bound on the f32 gradient."""
    from finenvs_b200.agents.networks import ParallelMLP

    pairs, E, lr, l2 = 10001, 3, 0.01, 0.005
    N = 2 * pairs + E
    torch.manual_seed(2)
    net = ParallelMLP(N, E, (60, 16, 2), learning_rate=lr, noise_std_dev=0.02, l2_coefficient=l2, device_id=0, seed=7,
                      action_noise_std=0.0)
    net.perturb_parameters()
    fit = torch.randn((N,), device="cuda")
    W0 = [w.clone() for w in net.weight_layers]
    B0 = [b.clone() for b in net.bias_layers]
    diff = (fit[:pairs] - fit[pairs: 2 * pairs]).contiguous()
    g, mag = _grad_f64(net._eps, diff)
    slabs = (pairs + 511) // 512
    net.update_parameters(fit)
    gw, gb = net.unpack(g / pairs)
    mw, mb = net.unpack(mag / pairs)
    b1, b2 = 0.9, 0.999
    alpha = math.sqrt(1 - b2) / (1 - b1) * lr

    def h(x):
        m, v = (1 - b1) * x, (1 - b2) * x * x
        return m / (v.sqrt() + 1e-8)

    for i in range(len(W0)):
        for new, old, gm, am in ((net.weight_layers[i], W0[i], gw[i], mw[i]), (net.bias_layers[i], B0[i], gb[i], mb[i])):
            old = old.double()
            gfull = gm - l2 * old
            d = (gamma(512 + slabs) * am + 4 * U * (gm.abs() + l2 * old.abs())) * (1 + 4 * U) + 1e-30
            upd = alpha * h(gfull)
            spread = alpha * (h(gfull + d) - h(gfull - d))
            bound = spread + 16 * U * upd.abs() + U * (old + upd).abs()
            err = (new.double() - (old + upd)).abs()
            assert bool((err <= bound).all()), float((err - bound).max())
            assert float((new.double() - old).abs().max()) > 0.5 * lr      # a real step was taken
    # the step above is ~lr * sign(g); Adam's moments pin the gradient's scale: m = 0.1 g, v = 0.001 g^2 after one step
    for i in range(len(W0)):
        for m_, v_, old, gm, am in ((net.first_moment_weights[i], net.second_moment_weights[i], W0[i], gw[i], mw[i]),
                                    (net.first_moment_biases[i], net.second_moment_biases[i], B0[i], gb[i], mb[i])):
            old = old.double()
            gfull = gm - l2 * old
            d = (gamma(512 + slabs) * am + 4 * U * (gm.abs() + l2 * old.abs())) * (1 + 4 * U)
            assert bool(((m_.double() - (1 - b1) * gfull).abs() <= (1 - b1) * d + 4 * U * (1 - b1) * gfull.abs()).all())
            assert bool(((v_.double() - (1 - b2) * gfull ** 2).abs()
                         <= (1 - b2) * (2 * gfull.abs() * d + d * d) + 6 * U * (1 - b2) * gfull ** 2).all())
            assert float(gfull.abs().max()) > 100 * float(d.max())        # the bound is far below the gradient


# ---------------------------------------------------------------------------------------------------------------------
# episode store
# ---------------------------------------------------------------------------------------------------------------------
def _store(lib, rew, dones, base, total, ordinal, cur_r, cur_s, cap, counters, key, env, ret):
    return lib.lib().fe_es_store(rew.data_ptr(), int(rew.dtype == torch.float64), dones.data_ptr(), rew.numel(), base, total,
                                 ordinal, cur_r.data_ptr(), cur_s.data_ptr(), cap, counters.data_ptr(), key.data_ptr(),
                                 env.data_ptr(), ret.data_ptr(), torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 31, 33, 257, 100003, 1 << 20])
@pytest.mark.parametrize("f64", [False, True])
def test_store_vs_accounting(lib, N, f64):
    """fe_es_store over many steps (no dones, all dones, random dones) against oracle_es.Accounting, which performs the
    same f32 / f64 operations: the key-sorted (env, return) list, both counters and the running arrays, exactly.
    The population is a shard (env_id_base > 0 of total_envs > N), so keys carry the global env id."""
    from oracle import oracle_es as oes

    T, base, total = 55, 3 * N + 5, 7 * N + 11
    rng = np.random.default_rng(N + f64)
    acc = oes.Accounting(N)
    cap = int(N * T * 0.12) + 2 * N + 64
    cur_r = torch.zeros(N, device="cuda")
    cur_s = torch.zeros(N, device="cuda")
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    key = torch.full((cap,), -1, dtype=torch.int64, device="cuda")
    env = torch.full((cap,), -1, dtype=torch.int64, device="cuda")
    ret = torch.full((cap,), float("nan"), device="cuda")
    exact_steps, keys = 0, []
    dt = np.float64 if f64 else np.float32
    for t in range(T):
        r = (rng.standard_normal(N) * 3).astype(dt)
        if t in (0, 10):
            d = np.zeros(N, np.int32)
        elif t in (20, 21):
            d = np.ones(N, np.int32)
        else:
            d = (rng.random(N) < 0.07).astype(np.int32)
        idx = np.nonzero(d)[0]
        exact_steps += int((acc.cur_steps[idx].astype(np.int64) + 1).sum())
        keys.append((t + 1) * total + base + idx)
        acc.step_and_store(r, d)
        assert _store(lib, torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda(), base, total, t + 1, cur_r, cur_s, cap,
                      counters, key, env, ret) == 0
    n = int(counters[0])
    assert n == len(acc.fin_ret) and int(counters[1]) == exact_steps
    if exact_steps < 1 << 24:        # Accounting sums the step counts in f32
        assert int(counters[1]) == int(acc.total_timesteps)
    k = key[:n].cpu().numpy()
    order = np.argsort(k, kind="stable")
    assert np.array_equal(k[order], np.concatenate(keys))
    assert np.array_equal(env[:n].cpu().numpy()[order], acc.dones)                  # local env index
    assert np.array_equal(ret[:n].cpu().numpy()[order], acc.fin_ret)
    assert np.array_equal(cur_r.cpu().numpy(), acc.cur_ret) and np.array_equal(cur_s.cpu().numpy(), acc.cur_steps)
    assert bool((key[n:] == -1).all()) and bool((env[n:] == -1).all())


@pytest.mark.gpu
def test_store_overflow_is_counted_not_written(lib):
    from finenvs_b200.agents.ES import EvoAgent

    N, cap, guard = 4099, 1000, 64
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    key = torch.full((cap + guard,), -7, dtype=torch.int64, device="cuda")
    env = torch.full((cap + guard,), -7, dtype=torch.int64, device="cuda")
    ret = torch.full((cap + guard,), -7.0, device="cuda")
    cur_r, cur_s = torch.zeros(N, device="cuda"), torch.zeros(N, device="cuda")
    ones = torch.ones(N, dtype=torch.int32, device="cuda")
    rew = torch.ones(N, device="cuda")
    for t in range(3):
        assert _store(lib, rew, ones, 0, N, t + 1, cur_r, cur_s, cap, counters, key, env, ret) == 0
    assert int(counters[0]) == 3 * N and int(counters[1]) == 3 * N
    assert bool((key[cap:] == -7).all()) and bool((env[cap:] == -7).all()) and bool((ret[cap:] == -7.0).all())
    k, e = key[:cap], env[:cap]
    assert bool((k >= N).all()) and bool((k < 4 * N).all()) and bool((e == k % N).all()) and bool((ret[:cap] == 1.0).all())
    assert k.unique().numel() == cap
    agent = EvoAgent({"env_name": "x", "num_envs": N - 1, "num_eval_envs": 2, "num_observations": 4, "num_actions": 1},
                     hidden_dims=(4,), write_to_csv=False, device_id=0, max_finished=cap, seed=1)
    dones = torch.ones(N - 1, dtype=torch.int32, device="cuda")
    agent.store(torch.ones(N - 1, device="cuda"), dones)
    with pytest.raises(RuntimeError, match="max_finished"):
        agent.dones


# ---------------------------------------------------------------------------------------------------------------------
# perturbation stream
# ---------------------------------------------------------------------------------------------------------------------
ES_KEY = 0x9E3779B97F4A7C15


def _eps_known_answer(lib, seed, generation, pair_id, q):
    """eps[pair, q] restated: Philox4x32-10 (the host fe_philox) keyed by seed ^ ES_KEY, counter (global pair id,
    generation << 32 | 2 * (q // 8) + (q % 8) // 4, kind 1); Box-Muller on 24-bit uniforms in f64, rounded to fp16."""
    q8, k = divmod(q, 8)
    r = lib.philox(seed ^ ES_KEY, pair_id, (generation << 32) | (2 * q8 + k // 4), 1)
    a, b = (r[0], r[1]) if k % 4 < 2 else (r[2], r[3])
    u1 = ((a >> 8) + 1) * 2.0 ** -24
    u2 = (b >> 8) * 2.0 ** -24
    rad = math.sqrt(-2.0 * math.log(u1))
    z = rad * (math.cos(2 * math.pi * u2) if k % 2 == 0 else math.sin(2 * math.pi * u2))
    return np.float16(z)


@pytest.mark.gpu
@pytest.mark.parametrize("generation,pair_id_base", [(1, 0), (2**31 - 1, 600), (5, 123456789)])
def test_perturbation_stream_known_answer(lib, generation, pair_id_base):
    L = lib.lib()
    shape, pairs, seed = (300, 8, 1), 700, 0x1234_5678_9ABC
    net = _fe_net(lib, shape)
    P = int(L.fe_es_params_padded(ctypes.byref(net)))
    eps = torch.zeros((pairs, P), dtype=torch.float16, device="cuda")
    assert L.fe_es_perturb(ctypes.byref(net), seed, generation, pair_id_base, pairs, eps.data_ptr(),
                           torch.cuda.current_stream().cuda_stream) == 0
    e = eps.cpu().numpy()
    rng = np.random.default_rng(generation)
    samples = [(int(p), int(q)) for p, q in zip(rng.integers(0, pairs, 3000), rng.integers(0, P, 3000))]
    samples += [(0, 0), (pairs - 1, P - 1), (0, P - 1), (pairs - 1, 0)] + [(pairs - 1, q) for q in range(P - 16, P)]
    mism = 0
    for p, q in samples:
        want = _eps_known_answer(lib, seed, generation, pair_id_base + p, q)
        got = e[p, q]
        if got != want:
            mism += 1
            assert abs(int(np.array(got).view(np.int16)) - int(np.array(want).view(np.int16))) <= 1, (p, q, got, want)
    assert mism <= 0.001 * len(samples), mism


@pytest.mark.gpu
def test_perturb_rejects_generation_2_pow_31(lib):
    L = lib.lib()
    net = _fe_net(lib, (20, 4, 1))
    eps = torch.zeros((2, int(L.fe_es_params_padded(ctypes.byref(net)))), dtype=torch.float16, device="cuda")
    for g in (2**31, 2**32 + 1):
        assert L.fe_es_perturb(ctypes.byref(net), 1, g, 0, 2, eps.data_ptr(), torch.cuda.current_stream().cuda_stream) == FE_EINVAL
    assert not bool(eps.any())
