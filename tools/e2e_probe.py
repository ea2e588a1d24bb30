"""Where the host-buffer step (fe_step_host / fe_step_host_packed) spends its time on BASELINE config 2.

One process, one GPU: device-resident step, then int32-dones and bit-packed host steps alternating (so that order effects
show), each as wall time per step over blocks of 20 steps, with the share spent inside the C call itself.  Also checks
that the packed bits equal the int32 dones of the same step.
usage: python tools/e2e_probe.py [--envs N] [--rounds R]
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--window", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--workload", default="c2")
    args = ap.parse_args()
    import torch
    import bench
    from finenvs_b200.data import loader
    from finenvs_b200.environments import TimeSeriesEnv

    N, W = args.envs, args.window
    prices, seg_start, seg_len, _ = bench.make_series(args.workload, W)
    series = loader.stage_series(prices, seg_start, seg_len, W, "cuda:0", torch.float32)
    env = TimeSeriesEnv("probe", num_intervals=W, device_id=0, series=series, num_envs=N, seed=3, random_reset="all",
                        random_offset=True)
    env.reset()
    g = torch.Generator(device="cuda:0").manual_seed(5)
    ring = [torch.rand((N, 1), generator=g, device="cuda:0") * 2 - 1 for _ in range(4)]
    ring_host = [a.cpu().pin_memory() for a in ring]
    obs = torch.empty((N, W, 5), dtype=torch.float32, device="cuda:0")
    rew = torch.empty(N, dtype=torch.float32, device="cuda:0")
    dn = torch.empty(N, dtype=torch.int32, device="cuda:0")
    print(f"kernel {env.kernel_name()}")

    def dev_block():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(args.steps):
            env.step_into(ring[i % 4], obs, rew, dn)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    for _ in range(3):
        dev_block()
    print("device step ms:", " ".join(f"{dev_block():.4f}" for _ in range(5)))

    # the same kernel with its actions read from and its rewards / dones written to pinned host memory (UVA pointers passed
    # as the "device" buffers), launches back to back without a host sync: what zero-copy costs the kernel itself
    r_pin, d_pin = torch.empty(N, dtype=torch.float32).pin_memory(), torch.empty(N, dtype=torch.int32).pin_memory()

    def zc_block():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(args.steps):
            env.step_count += 1
            rc = env._L.fe_step(env._pp, env._ps, env._pst, ring_host[i % 4].data_ptr(), obs.data_ptr(), r_pin.data_ptr(), d_pin.data_ptr(),
                                None, env.step_count, env._stream())
            assert rc == 0
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    for _ in range(3):
        zc_block()
    print("zero-copy kernel ms (back to back):", " ".join(f"{zc_block():.4f}" for _ in range(5)))

    # parity of the two wire formats on the same step: snapshot, step int32, restore, step packed
    snap = env.state_snapshot()
    _, r1, d1, _ = env.step_host(ring_host[0])
    r1, d1 = r1.clone(), d1.clone()
    env.load_state_snapshot(snap)
    _, r2, d2, _ = env.step_host(ring_host[0], packed_dones=True)
    ok = bool(torch.equal(r1, r2)) and bool(torch.equal(env.unpack_dones(d2), d1))
    print(f"packed == int32 on one step: {ok}  ({int(d1.sum())} dones)")
    assert ok

    call_s = [0.0]
    fn_i32, fn_pk = env._L.fe_step_host, env._L.fe_step_host_packed

    def host_block(packed):
        chk = 0.0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(args.steps):
            _, r_h, d_h, _ = env.step_host(ring_host[i % 4], packed_dones=packed)
            chk += float(r_h[0]) + int(d_h[0])
        return (time.perf_counter() - t0) * 1e3 / args.steps

    for rnd in range(args.rounds):
        for packed in (False, True, True, False):
            for _ in range(2):
                host_block(packed)
            ms = [host_block(packed) for _ in range(args.blocks)]
            print(f"round {rnd} {'packed' if packed else 'int32 '}: median {np.median(ms):.4f}  min {min(ms):.4f}  max {max(ms):.4f} ms/step")

    # the kernel inside the host-buffer call: events recorded on the stream right before and after each (synchronous) call
    for packed in (False, True):
        ks = []
        for i in range(60):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env.step_host(ring_host[i % 4], packed_dones=packed)
            e1.record()
            e1.synchronize()
            ks.append(e0.elapsed_time(e1))
        ks = sorted(ks[10:])
        print(f"GPU time between events around one step_host call ({'packed' if packed else 'int32 '}): median {ks[len(ks) // 2]:.4f}  min {ks[0]:.4f} ms")

    # the C call alone (no Python step_host around it): arguments prepared once
    a_dev, r_dev, d_dev, rewards, dones, done_bits = env._host_bufs
    obs2 = torch.empty((N, W, 5), dtype=torch.float32, device="cuda:0")
    stream = env._stream()
    for name, fn, out in (("int32 ", fn_i32, dones), ("packed", fn_pk, done_bits)):
        ms = []
        for b in range(args.blocks + 2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.steps):
                env.step_count += 1
                rc = fn(env._pp, env._ps, env._pst, ring_host[i % 4].data_ptr(), a_dev.data_ptr(), obs2.data_ptr(), r_dev.data_ptr(),
                        d_dev.data_ptr(), rewards.data_ptr(), out.data_ptr(), None, env.step_count, stream)
                assert rc == 0
            ms.append((time.perf_counter() - t0) * 1e3 / args.steps)
        ms = ms[2:]
        print(f"C call only {name}: median {np.median(ms):.4f}  min {min(ms):.4f} ms/step")


if __name__ == "__main__":
    main()
