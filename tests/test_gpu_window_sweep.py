"""Every step and observation kernel at every window shape it configures itself for.

Each step kernel picks its geometry from the window W and the dtype: the gather kernel its TMA part count, slot count and
pitch; the pipe kernel its envs per tile (TE) and register rows; the tile kernel its envs per block and shared memory; the
split kernel's stream pass a 480-element span plus a tail; the portfolio stream kernel its 512-pair chunks and bulk or
plain stores.  A wrong constant breaks only the windows that reach it, so the cases here are DERIVED from the library:
W = 1 ... WMAX is enumerated per dtype through the host-only calls fe_obs_table_bytes, fe_pipe_envs and fe_tile_envs, and
every window where a kernel's configuration changes (with its neighbours) becomes a case.  If a change moves a boundary,
the sweep moves with it.  What the ABI does not expose (the split span, the portfolio chunk, the descriptor ring depths,
the stream grid, the tile kernel's thread count and fe_gather_obs's launch formula) is read out of fe_step.cu and
fe_common.cuh: a constant by its name, a formula by the source line that holds it, so a changed line fails the host test
instead of silently leaving its mirror here behind.

Every step case forces its variant, asserts kernel_name(), runs lock-step with oracle.OracleEnv on the log-returns the
GPU staged, and compares bit for bit the state, rewards, dones and the whole observation (the reset's included), written
through step_into / fe_observe into a NaN-prefilled buffer with guard bands.  Each asserts that its scenario happened:
a ragged last tile, episodes ending and redrawing their segment and offset, several tiles per persistent block.
test_window_sweep_reaches_every_configuration (host only, no GPU) regenerates the configuration classes from the library
and checks that the case lists below reach every one of them."""
import functools
import os
import re

import numpy as np
import pytest
import torch

from parity_utils import ROOT, gbm_ohlc
from test_gpu_large_offsets import _guarded, _guards_intact
from test_gpu_parity import _env

WMAX = 4096                   # windows enumerated per dtype (the longest tile window is 1606 rows of f32)
STREAM_ROWS = {False: 3_300_000, True: 1_700_000}   # log-return tables above the 48 MB of pick_pipe_stages()
STEPS = 8
BARS = 5                      # bars per segment: with random offsets every env ends an episode within STEPS steps
DTYPES = (False, True)        # out_f64


# ---------------------------------------------------------------------------------------------------------------------
# what the ABI does not expose, read out of the kernel sources
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _source():
    csrc = os.path.join(ROOT, "finenvs_b200", "csrc")
    return "".join(open(os.path.join(csrc, f)).read() for f in ("fe_common.cuh", "fe_step.cu"))


@functools.lru_cache(maxsize=None)
def _const(name):
    """The value of `constexpr int <name> = <expression>;` in fe_common.cuh / fe_step.cu (names in the expression
    resolved the same way)."""
    found = re.findall(rf"constexpr int {name} = ([^;]+);", _source())
    assert len(found) == 1, f"constexpr int {name} in fe_common.cuh / fe_step.cu: {found}"
    expr = re.sub(r"\b(k[A-Za-z0-9]+)\b", lambda m: str(_const(m.group(1))), found[0])
    assert re.fullmatch(r"[0-9 ()*+/-]+", expr), (name, expr)
    return int(eval(expr, {"__builtins__": {}}))


def _line(pattern):
    """The integers a regular expression captures from the one source line it must match."""
    found = re.findall(pattern, _source())
    assert len(found) == 1, f"{pattern!r} matches {len(found)} lines of fe_common.cuh / fe_step.cu"
    return tuple(int(v) for v in (found[0] if isinstance(found[0], tuple) else (found[0],)))


def split_span():
    """kStreamSpan: output elements one fe_stream_kernel batch covers."""
    return _const("kStreamSpan")


def split_warps_per_sm():
    """fe_stream_kernel's grid in launch(): `blocks = (int64_t)sms * 6` blocks of kStreamThreads threads."""
    return _line(r"int64_t blocks = \(int64_t\)sms \* (\d+);")[0] * _const("kStreamThreads") // 32


def port_chunk():
    """CH in launch()'s K_PORTFOLIO case: (row, asset) pairs per fe_portfolio_stream_kernel chunk."""
    return _line(r"int CH = (\d+);")[0]


def gather_queue():
    """kGaQ: the gather kernel's descriptor ring depth, in 32-env tiles."""
    return _const("kGaQ")


def pipe_queue():
    """kPipeQ: the pipe kernel's descriptor ring depth, in tiles."""
    return _const("kPipeQ")


def tile_threads(e, W):
    """Threads per block of the tile kernel (pick_tile_envs): rows / 8 rounded up to whole warps, at least one warp,
    at most kThreads, and at least one thread per env."""
    (per,) = _line(r"int threads = \(int\)\(\(\(rows / (\d+)\) \+ 31\) & ~31L\);\s+"
                   r"if \(threads < 32\) threads = 32;\s+if \(threads > kThreads\) threads = kThreads;\s+"
                   r"while \(threads < e\) threads \+= 32;")
    threads = min(max(((e * W // per) + 31) & ~31, 32), _const("kThreads"))
    while threads < e:
        threads += 32
    return threads


# ---------------------------------------------------------------------------------------------------------------------
# configuration classes, from the library's host-only calls
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _L():
    """The library, built first: the case lists are made at collection, before any fixture runs, and ctypes keeps the
    library it loads for the whole session, so a stale one must never be the first one loaded (build() does nothing when
    the library is newer than its sources)."""
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib.lib()


def _tname(f64):
    return "double" if f64 else "float"


def _itemsize(f64):
    return 8 if f64 else 4


@functools.lru_cache(maxsize=None)
def gather_windows(f64):
    """Windows that have a gather variant (fe_obs_table_bytes > 0 for a short series)."""
    return tuple(W for W in range(1, WMAX + 1) if _L().fe_obs_table_bytes(4096, W, int(f64)) > 0)


def gather_parts(W, f64):
    """TMA parts of a gather window: one box row of at most 2048 bytes (ga_parts in fe_step.cu), else two."""
    return 1 if 5 * W * _itemsize(f64) <= 2048 else 2


def _runs(f):
    """[(value, first W, last W)] of f over W = 1 ... WMAX."""
    out = []
    for W in range(1, WMAX + 1):
        v = f(W)
        if out and out[-1][0] == v:
            out[-1][2] = W
        else:
            out.append([v, W, W])
    return [tuple(r) for r in out]


@functools.lru_cache(maxsize=None)
def pipe_classes(f64, stream):
    """[(TE, first W, last W)] of the pipe variant (TE > 0)."""
    return tuple(r for r in _runs(lambda W: _L().fe_pipe_envs(W, int(f64), int(stream))) if r[0] > 0)


@functools.lru_cache(maxsize=None)
def tile_classes(f64):
    """[(envs per block, first W, last W)] of the tile variant (> 0), and the first window past the last one."""
    runs = [r for r in _runs(lambda W: _L().fe_tile_envs(W, int(f64), 0)) if r[0] > 0]
    return tuple(runs), runs[-1][2] + 1


def split_class(W):
    """(tail class, has whole batches) of fe_stream_kernel at window W: tail 0, a tail inside the first 32-element slot
    row of a batch, or a longer one."""
    n = 5 * W
    tail = n % split_span()
    return ("none" if tail == 0 else "short" if tail < 32 else "long", n >= split_span())


def portfolio_class(A, W):
    """(chunks: 1, 2 or 3+, store path) of fe_portfolio_stream_kernel."""
    P = A * W
    chunks = -(-P // port_chunk())
    return (min(chunks, 3), "bulk" if P % 4 == 0 else "plain")


def pipe_store(W, nvalid, f64):
    """How the pipe kernel writes a tile of nvalid envs: one bulk store when its bytes are a multiple of 16."""
    return "bulk" if nvalid * W * 5 * _itemsize(f64) % 16 == 0 else "plain"


def _ragged_pipe(W, te, f64, want):
    """A ragged last-tile size (1 .. TE-1) whose store takes path `want` if any does, else the other path."""
    sizes = range(1, te)
    return next((n for n in sizes if pipe_store(W, n, f64) == want), next(iter(sizes)))


# ---------------------------------------------------------------------------------------------------------------------
# case lists (ids stable without a GPU; populations come from the SM count at run time)
# ---------------------------------------------------------------------------------------------------------------------
def _dt(f64):
    return "f64" if f64 else "f32"


def gather_cases():
    return [(f64, W) for f64 in DTYPES for W in gather_windows(f64)]


def gather_ring_cases():
    """The smallest and largest window of each part count, per dtype."""
    out = []
    for f64 in DTYPES:
        for parts in (1, 2):
            ws = [W for W in gather_windows(f64) if gather_parts(W, f64) == parts]
            out += [(f64, ws[0]), (f64, ws[-1])]
    return out


def pipe_cases():
    """(f64, stream, TE, W, ragged last tile): first and last window of every TE class in the cached flavour (plain
    store on the first, bulk on the last where the window allows it), the last windows again in the stream flavour
    (plain store where it can be had)."""
    out = []
    for f64 in DTYPES:
        for stream in (False, True):
            for te, lo, hi in pipe_classes(f64, stream):
                if not stream:
                    out.append((f64, stream, te, lo, _ragged_pipe(lo, te, f64, "plain")))
                    if hi != lo:
                        out.append((f64, stream, te, hi, _ragged_pipe(hi, te, f64, "bulk")))
                else:
                    out.append((f64, stream, te, hi, _ragged_pipe(hi, te, f64, "plain")))
    return out


@functools.lru_cache(maxsize=None)
def tile_shapes(f64):
    """[((envs per block, threads per block), first W, last W)] of the tile variant: the thread count also changes
    inside a class of equal env counts (the 4-env class runs from W = 48 to the longest tile window)."""
    last = tile_classes(f64)[0][-1][2]
    runs = _runs(lambda W: (_L().fe_tile_envs(W, int(f64), 0), tile_threads(_L().fe_tile_envs(W, int(f64), 0), W))
                 if W <= last else None)
    return tuple(r for r in runs if r[0] is not None)


def tile_cases():
    """(f64, envs per block, W): first and last window of every (envs, threads) shape; the last one is the longest
    window with a tile."""
    out = []
    for f64 in DTYPES:
        for (te, _), lo, hi in tile_shapes(f64):
            out += [(f64, te, lo)] + ([(f64, te, hi)] if hi != lo else [])
    return out


SPLIT_WINDOWS = (1, 95, 96, 97, 192)                 # 5W mod 480: 5, 475, 0, 5 and 0


def split_auto_windows(f64):
    """Windows too long for the pipe rings, which `auto` streams with split: the first one past the last pipe class, and
    f32 600 and 1024, f64 300 where they lie past it."""
    past = pipe_classes(f64, False)[-1][2] + 1
    return tuple(sorted({past} | {W for W in ((300,) if f64 else (600, 1024)) if W > past}))


def split_cases():
    return ([(f64, W, "split") for f64 in DTYPES for W in SPLIT_WINDOWS] +
            [(f64, W, "auto") for f64 in DTYPES for W in split_auto_windows(f64)])


PORTFOLIO_SHAPES = ((2, 60), (5, 7), (32, 16), (3, 171), (31, 32), (3, 205), (32, 48), (7, 221), (31, 41))


def portfolio_cases():
    return [(f64, A, W) for f64 in DTYPES for A, W in PORTFOLIO_SHAPES]


LSU_WINDOWS = {False: (1, 3, 61, 130, 390), True: (1, 27, 54, 101, 257)}


def gather_obs_cases():
    """(f64, W, path, large): every gather window through the TMA path (a count large enough for two passes of every
    warp at the extreme windows of each part count), and a sample of other windows through the warp-per-sample path."""
    ext = set(gather_ring_cases())
    return ([(f64, W, "tma", (f64, W) in ext) for f64, W in gather_cases()] +
            [(f64, W, "lsu", False) for f64 in DTYPES for W in LSU_WINDOWS[f64]])


def population_sizes(te, sms):
    """Fewer tiles than blocks, exactly one per block, and one more (in 32-env tiles, and in TE-env tiles)."""
    return sorted({1, 31, 33, 32 * sms - 1, 32 * sms + 1, te - 1, te + 1, te * sms - 1, te * sms + 1} - {0})


def population_cases():
    """(kernel, f64, W, TE): the gather kernel and the pipe kernel at TE 32 and TE 4, one window each."""
    classes = pipe_classes(False, False)
    first, last = classes[0], classes[-1]              # TE 32 and TE 4
    gather_w = next(W for W in gather_windows(False) if W >= 60)
    return [("gather", False, gather_w, 32), ("pipe", False, first[2], first[0]), ("pipe", False, last[1], last[0])]


def _ids(cases, fmt):
    return [fmt(*c) for c in cases]


# ---------------------------------------------------------------------------------------------------------------------
# the coverage claim (host only)
# ---------------------------------------------------------------------------------------------------------------------
def test_window_sweep_reaches_every_configuration():
    """The library's own configuration classes, regenerated from its host-only calls, each reached by a case below."""
    for f64 in DTYPES:
        legal = gather_windows(f64)
        assert len(legal) >= 20 and all(5 * W * _itemsize(f64) % 16 == 0 for W in legal)
        assert {W for g, W in gather_cases() if g == f64} == set(legal)
        assert {W for g, W, p, _ in gather_obs_cases() if g == f64 and p == "tma"} == set(legal)
        assert {W for g, W, p, _ in gather_obs_cases() if g == f64 and p == "lsu"}.isdisjoint(legal)
        assert {gather_parts(W, f64) for W in legal} == {1, 2}
        assert {gather_parts(W, f64) for g, W in gather_ring_cases() if g == f64} == {1, 2}
        for stream in (False, True):
            classes = pipe_classes(f64, stream)
            assert classes and len({c[0] for c in classes}) == len(classes)
            got = {(te, W) for g, s, te, W, _ in pipe_cases() if g == f64 and s == stream}
            for te, lo, hi in classes:
                assert (te, hi) in got and (stream or (te, lo) in got), (f64, stream, te)
                assert _L().fe_pipe_envs(hi + 1, int(f64), int(stream)) != te
            stores = {pipe_store(W, nv, f64) for g, s, te, W, nv in pipe_cases() if g == f64 and s == stream}
            assert stores == {"bulk", "plain"}, (f64, stream)
        for g, s, te, W, nv in pipe_cases():
            assert 0 < nv < te and _L().fe_pipe_envs(W, int(g), int(s)) == te
        classes, past = tile_classes(f64)
        assert _L().fe_tile_envs(past, int(f64), 0) == 0
        tiles = {(te, W) for g, te, W in tile_cases() if g == f64}
        assert tiles >= {(te, lo) for te, lo, _ in classes} | {(classes[-1][0], past - 1)}
        assert {(te, tile_threads(te, W)) for te, W in tiles} == {shape for shape, _, _ in tile_shapes(f64)}
        assert {split_class(W) for g, W, _ in split_cases() if g == f64} == \
            {("none", True), ("short", False), ("short", True), ("long", False), ("long", True)}
        for W in split_auto_windows(f64):
            assert _L().fe_pipe_envs(W, int(f64), 0) == 0       # `auto` has no pipe variant for it
        assert {portfolio_class(A, W) for g, A, W in portfolio_cases() if g == f64} == \
            {(c, s) for c in (1, 2, 3) for s in ("bulk", "plain")}
        assert {A for g, A, W in portfolio_cases() if g == f64} >= {2, 3, 7, 31, 32}
    # fe_gather_obs's grid at the two-pass windows, from the launch formula read out of gather_obs()
    for f64, W, path, large in gather_obs_cases():
        if large:
            assert 0 < gather_obs_grid_warps(W, f64, 1) <= 4 * 16
    # the populations the GPU cases run at reach what they claim at any SM count
    for sms in (1, 2, 132, 148, 160):
        for f64, W in gather_cases():
            N = _gather_population(sms)
            assert N % 2 == 1 and (N % 32) % 2 == 1 and -(-N // 32) >= 3 * sms
        for f64, W in gather_ring_cases():
            assert -(-_ring_population(sms) // 32) > gather_queue() * sms
        for f64, stream, te, W, nv in pipe_cases():
            N = _pipe_population(te, nv, sms)
            assert N % te == nv and -(-N // te) > pipe_queue() * sms
        for f64, te, W in tile_cases():
            assert _tile_population(te, sms) % te != 0 and _tile_population(te, sms) > 2 * te * sms
        assert _split_population(sms) >= 3 * split_warps_per_sm() * sms
        for _, _, _, te in population_cases():
            ns = population_sizes(te, sms)
            assert {1, 31, 33, 32 * sms - 1, 32 * sms + 1} <= set(ns)


# ---------------------------------------------------------------------------------------------------------------------
# populations (sms = the device's SM count)
# ---------------------------------------------------------------------------------------------------------------------
def _gather_population(sms):
    return 3 * 32 * sms + 17                 # 3 tiles per SM and a ragged tail of 17 envs (N % 32 odd)


def _ring_population(sms):
    return (gather_queue() + 8) * 32 * sms + 13   # more tiles per block than the descriptor ring holds


def _pipe_population(te, nvalid, sms):
    return (pipe_queue() + 2) * te * sms + nvalid


def _tile_population(te, sms):
    return 3 * te * sms + max(1, te // 2 - 1)


def _split_population(sms):
    return 3 * split_warps_per_sm() * sms + 37


def _portfolio_population(sms):
    return 2 * sms + 7


# ---------------------------------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


@pytest.fixture(scope="module")
def sms(lib):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _torch_dtype(f64):
    return torch.float64 if f64 else torch.float32


@functools.lru_cache(maxsize=None)
def _prices(T, A, sigma, seed):
    rng = np.random.default_rng(seed)
    if A == 1:
        return np.round(gbm_ohlc(rng, T, sigma), 4)
    return np.stack([np.round(gbm_ohlc(rng, T, sigma, s0=20.0 + 7 * a), 4) for a in range(A)], axis=1)


def _regular(T, W, bars):
    firsts = np.arange(W, T - bars + 1, bars, dtype=np.int64)
    return firsts - W, np.full(len(firsts), W + bars, np.int32)


def _stage(prices, seg_start, seg_len, W, f64):
    from oracle import oracle as orc
    from finenvs_b200.data import loader

    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", _torch_dtype(f64), keep_logret64=True)
    fs = orc.series_from_prices(prices, seg_start, seg_len, W, logret=series.logret64.cpu().numpy())
    return series, fs


@functools.lru_cache(maxsize=None)
def _short_series(W, f64, A=1, days=64, bars=BARS):
    """`days` segments of `bars` steps after a W-row window, staged once per (W, dtype, A, days, bars)."""
    T = W + days * bars
    seg_start, seg_len = _regular(T, W, bars)
    return _stage(_prices(T, A, 0.05, 1000 * A + W), seg_start, seg_len, W, f64)


def _long_series(W, f64, bars=24):
    """A series whose log-return table is above 48 MB (the pipe kernel's stream flavour); the prices are generated once
    for both dtypes and re-staged per window."""
    T = STREAM_ROWS[f64]
    prices = _prices(STREAM_ROWS[False], 1, 0.002, 77)[:T]
    seg_start, seg_len = _regular(T, W, bars)
    return _stage(prices, seg_start, seg_len, W, f64)


def _same_bits(want, got, what):
    """Bit-level equality (parity_utils.assert_bits_equal compares values: it takes -0.0 for 0.0 and any NaN for any)."""
    want, got = np.ascontiguousarray(want), np.ascontiguousarray(got)
    assert want.dtype == got.dtype and want.size == got.size, (what, want.dtype, got.dtype, want.shape, got.shape)
    u = {1: np.uint8, 4: np.uint32, 8: np.uint64}[want.itemsize]
    a, b = want.reshape(-1).view(u), got.reshape(-1).view(u)
    if not np.array_equal(a, b):
        bad = np.flatnonzero(a != b)
        raise AssertionError(f"{what}: {bad.size} of {a.size} elements differ, first at flat index {bad[0]}: "
                             f"{want.reshape(-1)[bad[0]]!r} (oracle) vs {got.reshape(-1)[bad[0]]!r}")


def _lockstep(series, fs, N, f64, variant, kernel, *, steps=STEPS, obs_steps=None, packed_steps=(), min_done=None,
              seed=5):
    """Lock-step of the CUDA env (variant forced) with the oracle, bit for bit, into a guarded NaN-prefilled output.
    obs_steps: the steps (0 = the reset) whose whole observation is compared (default: all).  packed_steps: steps
    taken through step_host(packed_dones=True) with pinned actions instead of step_into.  Returns the episode ends."""
    from oracle import oracle as orc

    dtype = _torch_dtype(f64)
    A, W = series.num_assets, series.window
    env = _env(series, num_envs=N, seed=seed, random_reset="all", random_offset=True, obs_dtype=dtype, variant=variant)
    assert env.kernel_name() == kernel, (env.kernel_name(), kernel)
    ref = orc.OracleEnv(fs, num_envs=N, seed=seed, reset_mode=orc.RESET_ALL, random_offset=True, out_f64=f64)
    obs_steps = set(range(steps + 1)) if obs_steps is None else set(obs_steps)
    buf, flat, g = _guarded(N * W * 5 * A, dtype)
    obs = flat.view(N, W, 5 * A)
    rewards = torch.empty(N, dtype=dtype, device="cuda")
    dones = torch.empty(N, dtype=torch.int32, device="cuda")
    seg0 = env._seg.cpu().numpy()
    _same_bits(ref.seg, seg0, "seg after the initial redraw")
    _same_bits(ref.ptr, env._ptr.cpu().numpy(), "ptr after the initial redraw")
    obs.fill_(float("nan"))
    env._observe_into(obs)
    if 0 in obs_steps:
        _same_bits(ref.reset(), obs.cpu().numpy(), "reset observation")
    assert _guards_intact(buf, g), "guard band overwritten by the reset observation"
    rng = np.random.default_rng(N + 7 * W + A)
    n_done, redrawn = 0, np.zeros(N, bool)
    for t in range(1, steps + 1):
        a = rng.uniform(-1.1, 1.1, (N, A)).astype(np.float32)
        want = t in obs_steps
        o_ref, r_ref, d_ref, _ = ref.step(a if A > 1 else a.reshape(-1), want_obs=want)
        ctx = f"t={t}"
        if t in packed_steps:
            o, r_h, bits, _ = env.step_host(torch.from_numpy(a).pin_memory(), packed_dones=True)
            assert bits.dtype == torch.uint8 and bits.numel() == 4 * ((N + 31) // 32)
            d_dev = env._host_bufs[2].cpu().numpy()
            _same_bits(d_ref, env.unpack_dones(bits).numpy(), f"packed dones {ctx}")
            _same_bits(d_ref, d_dev, f"device dones of step_host {ctx}")
            _same_bits(r_ref, r_h.numpy(), f"rewards of step_host {ctx}")
            if want:
                _same_bits(o_ref, o.cpu().numpy(), f"observation of step_host {ctx}")
            del o
        else:
            obs.fill_(float("nan"))
            rewards.fill_(float("nan"))
            dones.fill_(-1)
            env.step_into(torch.from_numpy(a).cuda(), obs, rewards, dones)
            _same_bits(d_ref, dones.cpu().numpy(), f"dones {ctx}")
            _same_bits(r_ref, rewards.cpu().numpy(), f"rewards {ctx}")
            if want:
                _same_bits(o_ref, obs.cpu().numpy(), f"observation {ctx}")
            assert _guards_intact(buf, g), f"guard band overwritten at {ctx}"
        for key, t_gpu in (("seg", env._seg), ("ptr", env._ptr), ("cash", env._cash), ("long_sh", env._long),
                           ("short_sh", env._short), ("margin", env._margin)):
            _same_bits(getattr(ref, key).reshape(-1), t_gpu.cpu().numpy(), f"{key} {ctx}")
        n_done += int(d_ref.sum())
        redrawn |= ref.seg != seg0
        del o_ref
    assert n_done >= (N if min_done is None else min_done), (n_done, N)
    assert redrawn.any(), "no env redrew its segment"
    return n_done


def _gather_kernel(f64):
    return f"fe_gather_kernel<{_tname(f64)}>"


def _pipe_kernel(f64, stream):
    return f"fe_pipe_kernel<{_tname(f64)},{'stream' if stream else 'cached'}>"


# ---- 1. gather step --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f64,W", gather_cases(), ids=_ids(gather_cases(), lambda f, W: f"{_dt(f)}-W{W}"))
def test_gather_step_every_window(lib, sms, f64, W):
    """3 tiles per SM and a ragged tail of 17 envs; steps 3 and 6 go through step_host with bit-packed dones (packed by
    the kernel's bookkeepers)."""
    N = _gather_population(sms)
    assert N % 32 != 0 and -(-N // 32) >= 3 * sms
    series, fs = _short_series(W, f64)
    _lockstep(series, fs, N, f64, "gather", _gather_kernel(f64), packed_steps=(3, 6))


@pytest.mark.gpu
@pytest.mark.parametrize("f64,W", gather_ring_cases(), ids=_ids(gather_ring_cases(), lambda f, W: f"{_dt(f)}-W{W}"))
def test_gather_step_descriptor_ring_wraps(lib, sms, f64, W):
    """More than SMs x 32 tiles of 32 envs: every block laps its 32-tile descriptor ring; observations compared on the
    reset and the last step."""
    N = _ring_population(sms)
    assert -(-N // 32) > gather_queue() * sms
    series, fs = _short_series(W, f64, bars=3)
    _lockstep(series, fs, N, f64, "gather", _gather_kernel(f64), steps=4, obs_steps=(0, 4))


# ---- 2. pipe step ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f64,stream,te,W,nvalid", pipe_cases(),
                         ids=_ids(pipe_cases(), lambda f, s, te, W, nv:
                                  f"{_dt(f)}-{'stream' if s else 'cached'}-TE{te}-W{W}-{pipe_store(W, nv, f)}"))
def test_pipe_step_every_tile_class(lib, sms, f64, stream, te, W, nvalid):
    """More tiles per block than the descriptor ring holds; the ragged last tile of nvalid envs leaves through the
    store path in the id.  Steps 3 and 6 go through step_host with bit-packed dones (packed by the bookkeepers at
    TE = 32, by fe_pack_dones_kernel otherwise)."""
    N = _pipe_population(te, nvalid, sms)
    assert N % te == nvalid and -(-N // te) > pipe_queue() * sms
    if stream:
        series, fs = _long_series(W, f64)
        min_done = 1
    else:
        series, fs = _short_series(W, f64)
        min_done = None
    _lockstep(series, fs, N, f64, "pipe", _pipe_kernel(f64, stream), packed_steps=(3, 6), min_done=min_done)


# ---- 3. tile step ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f64,te,W", tile_cases(),
                         ids=_ids(tile_cases(), lambda f, te, W: f"{_dt(f)}-E{te}-T{tile_threads(te, W)}-W{W}"))
def test_tile_step_every_block_shape(lib, sms, f64, te, W):
    N = _tile_population(te, sms)
    assert N % te != 0
    series, fs = _short_series(W, f64)
    _lockstep(series, fs, N, f64, "tile", f"fe_tile_kernel<{_tname(f64)}>")


@pytest.mark.gpu
@pytest.mark.parametrize("f64", DTYPES, ids=_dt)
def test_tile_refuses_the_first_window_past_it(lib, f64):
    W = tile_classes(f64)[1]
    series, _ = _short_series(W, f64, days=4)
    env = _env(series, num_envs=8, obs_dtype=_torch_dtype(f64), variant="tile")
    assert env.kernel_name().startswith("none"), env.kernel_name()
    with pytest.raises(lib.FeError):
        env.step(torch.zeros((8, 1), device="cuda"))


# ---- 4. split step ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f64,W,variant", split_cases(),
                         ids=_ids(split_cases(), lambda f, W, v: f"{_dt(f)}-W{W}-{v}-tail{5 * W % split_span()}"))
def test_split_step_every_stream_tail(lib, sms, f64, W, variant):
    """Every warp of the stream grid streams at least three envs (the next-header prefetch runs)."""
    N = _split_population(sms)
    series, fs = _short_series(W, f64)
    steps = STEPS if W < 512 else 6
    _lockstep(series, fs, N, f64, variant, f"fe_book_kernel + fe_stream_kernel<{_tname(f64)}>", steps=steps)


# ---- 5. portfolio step -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f64,A,W", portfolio_cases(),
                         ids=_ids(portfolio_cases(), lambda f, A, W: f"{_dt(f)}-A{A}-W{W}-P{A * W}"))
def test_portfolio_step_every_chunk_shape(lib, sms, f64, A, W):
    N = _portfolio_population(sms)
    series, fs = _short_series(W, f64, A=A)
    _lockstep(series, fs, N, f64, "auto", f"fe_portfolio_book_kernel + fe_portfolio_stream_kernel<{_tname(f64)}>")


# ---- 6. fe_gather_obs / fe_materialize -------------------------------------------------------------------------------
GATHER_OBS_LAUNCH = (  # gather_obs() in fe_step.cu, the lines that size the TMA path's grid
    r"room = \(size_t\)kSmemMax - kGoBarBytes;\s+int S = (\d+);\s+if \(room / \(S \* pitch\) < (\d+)\) S = (\d+);\s+"
    r"const int warps = \(int\)\(room / \(S \* pitch\) < \(size_t\)kGoMaxWarps \? room / \(S \* pitch\) : kGoMaxWarps\);\s+"
    r"const size_t smem = kGoBarBytes \+ \(size_t\)warps \* S \* pitch;\s+"
    r"int per_sm = \(int\)\(\(size_t\)\((\d+) \* 1024\) / \(smem \+ (\d+)\)\);\s+"
    r"per_sm = per_sm < 1 \? 1 : per_sm > (\d+) \? \d+ : per_sm;\s+"
    r"const int64_t need = \(\(count \+ 31\) / 32 \+ warps - 1\) / warps;\s+"
    r"const unsigned blocks = \(unsigned\)\(need < \(int64_t\)sms \* per_sm \? need : \(int64_t\)sms \* per_sm\);")
SLOT_PITCH = r"return \(\((\d+)u / \(uint32_t\)\(parts \? parts : 1\)\) \* ga_row_bytes\(f64\) \* W \+ (\d+)u\) & ~\d+u;"


def gather_obs_grid_warps(W, f64, sms):
    """Warps in the grid fe_gather_obs launches on the TMA path for a count large enough to fill it: gather_obs()'s
    formula, with its numbers read from the source."""
    s3, slots_min, s2, sm_kb, block_extra, per_sm_max = _line(GATHER_OBS_LAUNCH)
    envs, align = _line(SLOT_PITCH)
    pitch = ((envs // gather_parts(W, f64)) * (40 if f64 else 20) * W + align) & ~align
    room = _const("kSmemMax") - _const("kGoBarBytes")
    S = s3 if room // (s3 * pitch) >= slots_min else s2
    warps = min(room // (S * pitch), _const("kGoMaxWarps"))
    per_sm = min(max((sm_kb * 1024) // (_const("kGoBarBytes") + warps * S * pitch + block_extra), 1), per_sm_max)
    return warps * sms * per_sm


@pytest.mark.gpu
@pytest.mark.parametrize("f64,W,path,large", gather_obs_cases(),
                         ids=_ids(gather_obs_cases(), lambda f, W, p, big: f"{_dt(f)}-W{W}-{p}{'-2pass' if big else ''}"))
def test_gather_obs_every_window(lib, sms, f64, W, path, large):
    """fe_gather_obs with a random index with duplicates (count % 4 in 1..3) equals indexing the dense observations a
    step_into twin produced; fe_materialize of the last handle equals the last dense observation."""
    from finenvs_b200.agents.PPO.buffer import Buffer

    dtype = _torch_dtype(f64)
    series, _ = _short_series(W, f64)
    N = 4 * 32 * sms + 5
    kw = dict(num_envs=N, seed=13, random_reset="all", random_offset=True, obs_dtype=dtype)
    dense_env, lazy = _env(series, **kw), _env(series, **kw)
    Buffer(2, 0.99, 0).bind_env(lazy, lazy=True)
    kernel = "fe_gather_obs_kernel" if path == "tma" else "fe_materialize_kernel"
    assert lazy.gather_obs_kernel_name() == f"{kernel}<{_tname(f64)}>"
    lo = lazy.reset_lazy()
    row0, pf, dense = [lo.row0], [lo.posfeat], [dense_env.reset()]
    gen = torch.Generator(device="cuda").manual_seed(W + 100 * int(f64))
    for _ in range(3):
        a = torch.rand((N, 1), generator=gen, device="cuda") * 2 - 1
        o = torch.empty((N, W, 5), dtype=dtype, device="cuda")
        r = torch.empty(N, dtype=dtype, device="cuda")
        d = torch.empty(N, dtype=torch.int32, device="cuda")
        dense_env.step_into(a, o, r, d)
        lo, r_l, d_l, _ = lazy.step_lazy(a)
        assert torch.equal(r_l, r) and torch.equal(d_l, d)
        row0.append(lo.row0)
        pf.append(lo.posfeat)
        dense.append(o)
    assert torch.equal(lo.materialize(), dense[-1])
    row0, pf, dense = torch.cat(row0), torch.cat(pf), torch.cat(dense)
    if large:   # every warp of the grid takes at least two 32-sample tiles
        count = 2 * 32 * gather_obs_grid_warps(W, f64, sms) + 64
    else:
        count = 2 * N
    count = count - count % 4 + 1 + (W // 4 + int(f64)) % 3
    assert count % 4 in (1, 2, 3)
    index = torch.randint(0, row0.numel(), (count,), generator=gen, device="cuda", dtype=torch.int64)
    index[count // 2] = index[0]
    index[-1] = index[1]
    buf, flat, g = _guarded(count * W * 5, dtype)
    flat.fill_(float("nan"))
    out = flat.view(count, W, 5)
    lazy.gather_obs(row0, pf, index, out)
    assert _guards_intact(buf, g)
    chunk = max(1, (1 << 26) // (W * 5))
    for b in range(0, count, chunk):
        assert torch.equal(out[b: b + chunk], dense[index[b: b + chunk]]), f"samples [{b}, {b + chunk})"


# ---- 7. populations --------------------------------------------------------------------------------------------------
def _population_ids():
    return _ids(population_cases(), lambda k, f, W, te: f"{k}-{_dt(f)}-W{W}-TE{te}")


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,f64,W,te", population_cases(), ids=_population_ids())
def test_step_populations_around_one_tile_per_block(lib, sms, kernel, f64, W, te):
    """N in {1, 31, 33, 32 SMs - 1, 32 SMs + 1} and the same counts in TE-env tiles: fewer tiles than blocks, exactly
    one per block, and one more."""
    if kernel == "gather":
        name = _gather_kernel(f64)
    else:
        assert lib.lib().fe_pipe_envs(W, int(f64), 0) == te
        name = _pipe_kernel(f64, False)
    series, fs = _short_series(W, f64)
    for N in population_sizes(te, sms):
        _lockstep(series, fs, N, f64, kernel, name, packed_steps=(4,) if kernel == "gather" else ())
