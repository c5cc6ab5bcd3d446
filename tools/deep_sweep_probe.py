#!/usr/bin/env python
"""Timing of V(2,2), V(3,3) and V(4,4) on 1 .. 8 GPUs, run under torchrun (one process per GPU; --nproc-per-node 1 for one
GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29581 \
        tools/deep_sweep_probe.py [--sizes 4097 16385] [--out profiles/deep_sweeps.log]

At each N, omega = 2/3, a random right-hand side and a zero guess: device ms per cycle (median of 5 cycles after a warm-up
cycle) and cycles and device ms to ||r|| < 1e-8 ||r0|| (pmg_last_device_ms, median of 3 solves after a warm-up solve).  On
several GPUs the V(3,3) / V(4,4) cycles run the deep-sweep slab schedule with its up-exchange, V(2,2) the schedule
without one.  The card name and power limit are printed first (nvidia-smi, read-only query), with the rank count.
"""
import argparse
import os
import statistics
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4097, 16385])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    import pmg_b200 as pmg
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        rank, world, dev = pmg.init_distributed_from_torch(local)
    else:
        rank, dev = 0, local
    lines = []

    def say(s):
        if rank == 0:
            print(s, flush=True)
            lines.append(s)

    say("card: %s" % card().replace("\n", " | "))
    say("ranks: %d" % world)
    for n in a.sizes:
        y0, y1 = pmg.partition_rows(n, world, rank) if world > 1 else (0, n)
        f = np.zeros((n, n))
        f[1:-1, 1:-1] = np.random.default_rng(7).uniform(-1, 1, (n - 2, n - 2))
        for nu in (2, 3, 4):
            kw = dict(rank=rank, n_ranks=world) if world > 1 else {}
            s = pmg.Solver(n, device=dev, omega=2.0 / 3.0, nu1=nu, nu2=nu, **kw)
            s.set_rhs(np.ascontiguousarray(f[y0:y1]))
            s.zero_guess()
            s.cycle(pmg.V, want_norm=True)
            per = []
            for _ in range(5):
                s.cycle(pmg.V, want_norm=True)
                per.append(s.last_ms)
            solves, k = [], 0
            for i in range(4):
                s.zero_guess()
                k, _ = s.solve(pmg.V, rel_tol=1e-8, max_cycles=200)
                if i:
                    solves.append(s.last_ms)
            s.close()
            say("N=%d V(%d,%d): %.3f ms per cycle (median of 5), %d cycles to 1e-8 in %.3f ms (median of 3)"
                % (n, nu, nu, statistics.median(per), k, statistics.median(solves)))
    if world == 1:
        say("several GPUs: not measured in this run (one process); the up-exchange costs nothing on one GPU")
    if rank == 0 and a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    if world > 1:
        pmg.comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
