#!/usr/bin/env python
"""Timing of pmg_pcg on 1 .. 8 GPUs, run under torchrun (one process per GPU; --nproc-per-node 1 for one GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29571 \
        tools/pcg_dist_probe.py [--n 16385]

At N (default 16385), V(2,2), omega = 2/3, full-interior prolongation, a random right-hand side and a zero guess:
  * pmg_pcg(precond = 1) to ||r|| < 1e-8 ||r0||: steps, device ms (pmg_last_device_ms, median of 3 solves after a warm-up
    solve) and ms per step;
  * pmg_solve(V) on the same ranks and problem: cycles and device ms;
With one process it also times, at N, the fused direction-operator pass (k_pcg_direction_apply, 32 B/point) against the
pair it replaces (k_pcg_direction + k_apply_a_dot, 40 B/point), alternated, through the test hooks; each hook call ends in a
device synchronise, which both sides pay once per call.  The card name and power limit are printed first (nvidia-smi,
read-only query), with the rank count.
"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi unavailable (%s)" % e


def pass_timing(pmg, n, rounds=5, launches=20):
    """median ms of one fused direction-operator pass and of the two-kernel pair, alternated"""
    L = pmg.lib()
    L.pmg_test_layout.restype = None
    L.pmg_test_layout.argtypes = [ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 3
    L.pmg_test_pcg_direction_apply.argtypes = ([ctypes.c_void_p] * 4 + [ctypes.c_int] * 4 + [ctypes.c_double] +
                                               [ctypes.c_void_p] * 2 + [ctypes.c_int] + [ctypes.c_void_p] +
                                               [ctypes.POINTER(ctypes.c_int)])
    L.pmg_test_pcg_direction_pair.argtypes = ([ctypes.c_void_p] * 3 + [ctypes.c_int] * 2 + [ctypes.c_double] * 2 +
                                              [ctypes.c_int] + [ctypes.c_void_p] * 2)
    pitch, px, py = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    L.pmg_test_layout(n, ctypes.byref(pitch), ctypes.byref(px), ctypes.byref(py))
    pitch, px, py = pitch.value, px.value, py.value
    rows = n + 2 * py
    rng = np.random.default_rng(5)
    z = np.zeros((rows, pitch))
    z[py + 1:py + n - 1, px + 1:px + n - 1] = rng.uniform(-1, 1, (n - 2, n - 2))
    dz = pmg.DeviceArray.from_numpy(z)
    del z
    arrs = [pmg.DeviceArray.from_numpy(np.zeros((rows, pitch))) for _ in range(3)]  # p_in / p (pair), p_out, ap
    sc = pmg.DeviceArray.from_numpy(np.array([0.75, 1.0, 0.0]))
    part = pmg.DeviceArray.from_numpy(np.zeros(148 * 32))
    off = 8 * (py * pitch + px)
    h = 1.0 / (n - 1)
    k = ctypes.c_int()

    def fused():
        pmg.check(L.pmg_test_pcg_direction_apply(dz.ptr + off, arrs[0].ptr + off, arrs[1].ptr + off, arrs[2].ptr + off, n, n,
                                                 0, pitch, h, sc.ptr, sc.ptr + 8, 0, part.ptr, ctypes.byref(k)))

    def pair():
        pmg.check(L.pmg_test_pcg_direction_pair(dz.ptr + off, arrs[0].ptr + off, arrs[2].ptr + off, n, pitch, h, 0.75, 0,
                                                part.ptr, sc.ptr + 16))

    res = {"fused": [], "pair": []}
    for fn in (fused, pair):
        fn()
    for r in range(rounds):
        for name, fn in ((("fused", fused), ("pair", pair)) if r % 2 == 0 else (("pair", pair), ("fused", fused))):
            t0 = time.perf_counter()
            for _ in range(launches):
                fn()
            res[name].append((time.perf_counter() - t0) * 1e3 / launches)
    for d in [dz, part, sc] + arrs:
        d.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16385)
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    import pmg_b200 as pmg
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    dist_kw, rank, world = {}, 0, 1
    if world_env > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        rank, world, dev = pmg.init_distributed_from_torch(local)
        dist_kw = dict(device=dev, rank=rank, n_ranks=world, agglomerate_below=min(257, a.n // 4))
    n = a.n
    if rank == 0:
        print("cards (index, name, power limit, max SM clock):\n" + card(), flush=True)
        print("ranks=%d N=%d V(2,2) omega=2/3 full-interior prolongation, random f, zero guess" % (world, n), flush=True)
    y0, y1 = pmg.partition_rows(n, world, rank) if world > 1 else (0, n)
    f = np.zeros((n, n))
    f[1:-1, 1:-1] = np.random.default_rng(72).uniform(-1, 1, (n - 2, n - 2))
    s = pmg.Solver(n, omega=2.0 / 3.0, nu1=2, nu2=2, prolong_mode=pmg.PROLONG_FULL, **dist_kw)
    s.set_rhs(np.ascontiguousarray(f[y0:y1]))
    del f
    pcg, vs = [], []
    for it in range(4):
        s.zero_guess()
        k, hist = s.pcg(precond=1, rel_tol=1e-8, max_iter=100)
        if it > 0:
            pcg.append((k, s.last_ms, hist[-1] / hist[0]))
        s.zero_guess()
        kv, hv = s.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
        if it > 0:
            vs.append((kv, s.last_ms, hv[-1] / hv[0]))
    s.close()
    ms_p = statistics.median(t for _, t, _ in pcg)
    ms_v = statistics.median(t for _, t, _ in vs)
    if world > 1:  # the slowest rank
        t = torch.tensor([ms_p, ms_v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_p, ms_v = float(t[0]), float(t[1])
    if rank == 0:
        k, kv = pcg[0][0], vs[0][0]
        print("N=%d ranks=%d: PCG(V) %d steps to 1e-8 in %.3f ms = %.3f ms per step (final rel %.2e; median of 3: %s)"
              % (n, world, k, ms_p, ms_p / k, pcg[0][2], [round(t, 3) for _, t, _ in pcg]), flush=True)
        print("N=%d ranks=%d: pmg_solve(V) %d cycles to 1e-8 in %.3f ms = %.3f ms per cycle (final rel %.2e; median of 3: %s)"
              % (n, world, kv, ms_v, ms_v / kv, vs[0][2], [round(t, 3) for _, t, _ in vs]), flush=True)
    if world == 1:
        res = pass_timing(pmg, n)
        mf, mp = statistics.median(res["fused"]), statistics.median(res["pair"])
        pts = float(n) * n
        print("N=%d direction-operator pass: fused %.3f ms (%.0f GB/s at 32 B/pt) | direction + apply_a_dot %.3f ms "
              "(%.0f GB/s at 40 B/pt) | speed-up %.2fx  (medians of 5 alternated rounds of 20 calls: %s / %s)"
              % (n, mf, 32 * pts / mf / 1e6, mp, 40 * pts / mp / 1e6, mp / mf,
                 [round(t, 4) for t in res["fused"]], [round(t, 4) for t in res["pair"]]), flush=True)
    if world > 1:
        pmg.comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
