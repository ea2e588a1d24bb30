"""The C-ABI library loads and exports every symbol include/finenvs_b200.h declares (no compute
calls: this runs without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from parity_utils import ROOT


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as ge

    ge.build()
    from finenvs_b200 import _lib

    return _lib


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "finenvs_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(fe_[a-z_0-9]+)\s*\(", hdr)))


def test_every_declared_symbol_is_exported_and_bound(built):
    names = _declared_symbols()
    assert len(names) >= 10
    raw = ctypes.CDLL(built.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in the header but not exported"
    assert sorted(built.EXPORTS) == names, "ctypes binding and header disagree"
    assert built.lib().fe_version() == built.ABI_VERSION


def test_struct_layouts_match_the_header(built):
    # sizes implied by the header's field lists (LP64): a silent mismatch would corrupt every call
    assert ctypes.sizeof(built.FeParams) == 4 * 8 + 4 * 4 + 4 * 8 + 8 + 6 * 4
    assert ctypes.sizeof(built.FeSeries) == 5 * 8
    assert ctypes.sizeof(built.FeState) == 10 * 8
    assert built.STATS_BYTES == 6 * 8


def test_error_strings_and_argument_validation(built):
    L = built.lib()
    assert L.fe_error_string(0) == b"ok"
    assert b"invalid" in L.fe_error_string(-1)
    assert b"aligned" in L.fe_error_string(-2)
    # null params are rejected before any CUDA call is made
    assert L.fe_step(None, None, None, None, None, None, None, None, 1, None) == -1
    assert L.fe_observe(None, None, None, None, None) == -1
    assert L.fe_log_returns(None, 0, 1, None, None, None) == -1


def test_host_philox_matches_oracle_and_known_answer(built):
    from oracle import oracle as orc

    # Philox4x32-10 known answer (Random123 kat_vectors): ctr=0, key=0
    assert built.philox(0, 0, 0, 0) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    rng = np.random.default_rng(0)
    for _ in range(200):
        seed, env, step = (int(x) for x in rng.integers(0, 2**63 - 1, 3))
        kind = int(rng.integers(0, 2))
        assert built.philox(seed, env, step, kind) == [int(x) for x in orc.philox(seed, env, step, kind)]


def test_tile_sizes(built):
    L = built.lib()
    # small tiles (many blocks in flight) measured fastest; always a multiple of 4 (16-byte bulk-copy granularity)
    assert L.fe_tile_envs(60, 0, 0) == 4 and L.fe_tile_envs(60, 1, 0) == 4
    assert L.fe_tile_envs(390, 0, 0) == 4      # the reference default window
    assert L.fe_tile_envs(4, 0, 0) == 48       # tiny windows: more envs per block
    for w in (1, 3, 8, 16, 128, 1500):
        assert L.fe_tile_envs(w, 0, 0) % 4 == 0 and L.fe_tile_envs(w, 0, 0) > 0
    assert L.fe_tile_envs(1500, 1, 0) == 0     # f64 rows: does not fit -> direct variant
    assert L.fe_tile_envs(2000, 0, 0) == 0
    assert L.fe_tile_envs(0, 0, 0) == 0


def test_env_has_no_cpu_fallback(built):
    import torch

    from finenvs_b200.environments import TimeSeriesEnv

    if not torch.cuda.is_available():   # the default device is cuda:0: only refused where there is none
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            TimeSeriesEnv("IBM", "dummy")
    with pytest.raises(RuntimeError, match="no CPU fallback"):   # an explicit CPU device is refused everywhere
        TimeSeriesEnv("IBM", "dummy", device_id=-1)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "finenvs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), f"{f} mentions the oracle"


def test_kernel_choice_policy(built):
    """choose_kernel() (fe_step.cu) through fe_step_kernel_name: a pure host function, so the `auto` policy that
    DESIGN.md's window sweep justifies is pinned here without a GPU."""
    L = built.lib()

    def name(N=1 << 20, W=60, A=1, rows=258048, f64=0, variant=built.VARIANT_AUTO, table=False):
        p = built.FeParams(N, 0, N, rows, W, 1024, A, 5, 10000.0, 0.01, 1.5, 0.25, 1, built.RESET_ALL, 1, 0, f64, variant, 0)
        s = built.FeSeries(16, 16, 16, 16, 4096 if table else None)    # only obs_table / sched == NULL matter to the policy
        st = built.FeState(16, 16, 16, 16, 16, 16, None, None, None, 4096 if table else None)
        return L.fe_step_kernel_name(ctypes.byref(p), ctypes.byref(s), ctypes.byref(st)).decode()

    assert name(table=True) == "fe_gather_kernel<float>"                      # BASELINE config 2 with the staged obs table
    assert name() == "fe_pipe_kernel<float,cached>"                           # ... without it: the round-1 kernel
    assert name(rows=10_000_000) == "fe_pipe_kernel<float,stream>"            # config 4: table larger than L2
    assert name(rows=10_000_000, table=True) == "fe_pipe_kernel<float,stream>"   # an obs table of 800 MB would not stay in L2
    assert name(rows=1_000_000, table=True) == "fe_pipe_kernel<float,cached>"
    assert name(f64=1) == "fe_pipe_kernel<double,cached>"
    assert name(f64=1, table=True) == "fe_gather_kernel<double>"              # 40 * 60 bytes: two TMA rows of 1200 = 15 * 80 bytes
    assert name(f64=1, W=50, table=True) == "fe_gather_kernel<double>"
    assert name(f64=1, W=54, table=True) == "fe_pipe_kernel<double,cached>"   # 2160 bytes: half a window is not a whole pitch
    assert name(W=61, table=True) == "fe_pipe_kernel<float,cached>"           # 20 * 61 is not a multiple of 16
    assert name(W=100, table=True) == "fe_gather_kernel<float>" and name(W=108, table=True) == "fe_pipe_kernel<float,cached>"
    assert name(W=128, N=1 << 19, table=True) == "fe_gather_kernel<float>"    # two parts of 1280 bytes
    assert name(W=136, N=1 << 19, table=True) == "fe_pipe_kernel<float,cached>"   # two-part windows stop at 128 rows
    assert name(N=1024) == "fe_tile_kernel<float>" == name(N=1024, table=True)   # config 1: too few tiles per SM
    assert name(W=4, N=1 << 22) == "fe_tile_kernel<float>" and name(W=16, table=True) == "fe_tile_kernel<float>"   # few rows per env
    assert name(W=24) == "fe_pipe_kernel<float,cached>" and name(W=512, N=1 << 17) == "fe_pipe_kernel<float,cached>"
    assert name(W=24, table=True) == "fe_gather_kernel<float>"
    assert name(W=1024, N=1 << 16).startswith("fe_book_kernel + fe_stream_kernel")       # beyond the pipe rings
    assert name(W=300, f64=1, N=1 << 17).startswith("fe_book_kernel + fe_stream_kernel")  # f64 rings hold 256 rows
    assert name(W=2000, N=64).startswith("fe_book_kernel + fe_stream_kernel")
    assert name(A=30, W=128, N=65536).startswith("fe_portfolio_book_kernel + fe_portfolio_stream_kernel")   # config 3
    assert name(variant=built.VARIANT_TILE) == "fe_tile_kernel<float>"
    assert name(variant=built.VARIANT_DIRECT) == "fe_direct_kernel<float>"
    assert name(variant=built.VARIANT_SPLIT).startswith("fe_book_kernel")
    assert name(N=64, variant=built.VARIANT_PIPE) == "fe_pipe_kernel<float,cached>"
    assert name(N=64, variant=built.VARIANT_GATHER, table=True) == "fe_gather_kernel<float>"
    assert name(variant=built.VARIANT_GATHER).startswith("none (the gather variant needs")
    assert name(W=61, variant=built.VARIANT_GATHER, table=True).startswith("none")
    assert name(W=4000, variant=built.VARIANT_TILE).startswith("none")        # does not fit in shared memory
    assert name(W=4000, variant=built.VARIANT_PIPE).startswith("none")
    for bad in (5, 7):   # the round-1 scatter / rows experiments are gone: unknown variants fall through to tile / direct
        assert name(variant=bad) in ("fe_tile_kernel<float>", "fe_direct_kernel<float>")


def test_obs_table_geometry(built):
    """fe_obs_table_bytes: which windows have a gather variant and how large its table is (host arithmetic only)."""
    L = built.lib()
    assert L.fe_obs_table_bytes(258048, 60, 0) == 4 * (258048 // 4 + 15 + 8) * 80 + 4096      # 20.6 MB for config 2
    assert L.fe_obs_table_bytes(258048, 61, 0) == 0 and L.fe_obs_table_bytes(258048, 62, 0) == 0
    assert L.fe_obs_table_bytes(258048, 100, 0) > 0 and L.fe_obs_table_bytes(258048, 108, 0) == 0
    assert L.fe_obs_table_bytes(258048, 104, 0) > 0 and L.fe_obs_table_bytes(258048, 128, 0) > 0    # fetched in two parts
    assert L.fe_obs_table_bytes(258048, 136, 0) == 0
    assert L.fe_obs_table_bytes(258048, 50, 1) == 2 * (258048 // 2 + 25 + 8) * 80 + 4096
    assert L.fe_obs_table_bytes(258048, 51, 1) == 0 and L.fe_obs_table_bytes(258048, 54, 1) == 0
    assert L.fe_obs_table_bytes(258048, 60, 1) == 2 * (258048 // 2 + 30 + 8) * 80 + 4096            # the reference's dtype, W = 60
    assert L.fe_obs_table_bytes(0, 60, 0) == 0 and L.fe_obs_table_bytes(100, 0, 0) == 0


def test_header_is_plain_c_and_a_c_program_links_against_the_library(built, tmp_path):
    """include/finenvs_b200.h is what a non-Python embedder binds (INTEGRATION.md §3): it must compile as C99, the struct
    sizes a C compiler sees must be the ones the ctypes mirror uses, and a C program must link and call the library."""
    import shutil
    import subprocess

    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include "finenvs_b200.h"\n'
        "int main(void) {\n"
        '  printf("%d %zu %zu %zu %zu %zu\\n", fe_version(), sizeof(FeParams), sizeof(FeSeries), sizeof(FeState),\n'
        "         sizeof(FeStats), sizeof(FeEsNet));\n"
        '  printf("%s\\n", fe_error_string(FE_ECSV));\n'
        "  void *h = 0; int64_t rows = -1;\n"
        '  printf("%d\\n", fe_csv_open("/nonexistent/x.csv", 1, &h, &rows));\n'
        "  return fe_step(0, 0, 0, 0, 0, 0, 0, 0, 1, 0) == FE_EINVAL ? 0 : 1;\n}\n")
    exe = tmp_path / "abi"
    libdir = os.path.dirname(built.LIB_PATH)
    subprocess.check_call([cc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", libdir, "-l:" + os.path.basename(built.LIB_PATH), "-Wl,-rpath," + libdir])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    l1, l2, l3 = out.stdout.splitlines()
    ver, sp, ss, sst, sstat, snet = (int(x) for x in l1.split())
    assert ver == built.ABI_VERSION
    assert (sp, ss, sst) == (ctypes.sizeof(built.FeParams), ctypes.sizeof(built.FeSeries), ctypes.sizeof(built.FeState))
    assert sstat == built.STATS_BYTES and snet == ctypes.sizeof(built.FeEsNet)
    assert "CSV" in l2 and int(l3) == -4
