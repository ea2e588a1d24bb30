"""bench.py's JSON contract, checked on the arm that needs no GPU: `--impl reference` (the unmodified reference env from
baseline/_ref on the host cores, the C oracle port beside it).  The keys and their meaning are documented in bench.py's
docstring.  On a GPU: the GPU arm times exactly --steps steps and --dump-outputs writes repeatable outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
                          "--ref-widened-envs", "0", *extra], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return lines


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["ms_per_step"] > 0 and d["value"] > 0
    assert d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    assert d["config"]["envs_per_gpu"] == 1 << 20   # the arm reports the GPU arm's config; the bounded sample is in cpu_baseline
    cb = d["cpu_baseline"]
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == d["unit"] and cb["sample"]
    assert cb["cpu_port"]["kind"] == "port" and cb["cpu_port"]["value"] > 0
    if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "finenvs")):
        assert cb["kind"] == "reference" and cb["tree"] == "baseline/_ref"
        assert {(r["envs"], r["threads"]) for r in cb["runs"]} >= {(1024, cb["cores"]), (1024, 1)}
    else:
        assert cb["kind"] == "port"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert _run("--gpus", "2", env=env) == []


def test_portfolio_workload_on_the_reference_arm():
    d = json.loads(_run("--workload", "c3")[0])
    assert d["config"]["assets"] == 30 and d["config"]["window"] == 128 and d["value"] > 0
    assert "workload c3" in d["cpu_baseline"]["cpu_port"]["sample"]


def test_reference_arm_forces_the_thread_count_under_torchrun():
    # torchrun exports OMP_NUM_THREADS=1; the arm must still use the cores the box has (round-1 SCALE ratios were void)
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    d = json.loads(_run("--gpus", "2", env=env)[0])
    ncpu = len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["cores"] == ncpu and d["cpu_baseline"]["cpu_port"]["cores"] == ncpu
    assert d["config"]["total_envs"] == 2 << 20


def _run_gpu_arm(dump_dir, envs):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "7", "--warmup", "3", "--envs", str(envs),
                          "--no-also", "--no-cpu-baseline", "--dump-outputs", str(dump_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


@pytest.mark.gpu
def test_gpu_arm_times_exactly_the_requested_steps_and_dumps_repeatable_outputs(tmp_path):
    envs = 65536                      # the full observation (79 MB) exceeds its share: obs.npy is the seeded sample
    a, b = _run_gpu_arm(tmp_path / "a", envs), _run_gpu_arm(tmp_path / "b", envs)
    for d in (a, b):
        assert d["steps"] == 7 and d["timing"]["timed_steps"] == 7 and sum(d["timing"]["steps_per_block"]) == 7
        assert d["public_step"]["timing"]["timed_steps"] == 7 and d["e2e"]["timing"]["timed_steps"] == 7
        per_step = 2 if " + " in d["roofline"]["kernel"] else 1
        assert d["gpu_launches"] == 4 * 7 * per_step   # device-resident, step(), two host-buffer legs
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["dones.npy", "obs.npy", "rewards.npy"] and sorted(os.listdir(tmp_path / "b")) == names
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    arrays = {n: np.load(tmp_path / "a" / n) for n in names}
    assert all(x.dtype == np.float32 for x in arrays.values())
    assert arrays["rewards.npy"].shape == arrays["dones.npy"].shape == (envs,)
    assert set(np.unique(arrays["dones.npy"])) <= {0.0, 1.0}
    assert arrays["dones.npy"].sum() == a["episodes_finished_last_step"] > 0   # the dump holds the last timed step
    obs = arrays["obs.npy"]
    assert 0 < obs.shape[0] < envs and obs.shape[1:] == (60, 5) and np.isfinite(obs).all()
    for n in names:                   # same arguments, same inputs: the outputs repeat bit for bit
        assert np.array_equal(arrays[n], np.load(tmp_path / "b" / n)), n
