#!/usr/bin/env python
"""Timing of PMG_CYCLE_FMG on 1 .. 8 GPUs, run under torchrun (one process per GPU; --nproc-per-node 1 for one GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29561 \
        tools/fmg_dist_probe.py [--sizes 4097,16385] [--parent-lib PATH]

Per size, with V(2,2), omega = 2/3, reference prolongation:
  * one FMG pass: median of 7 device times (pmg_last_device_ms) after 2 warm-up passes;
  * cycles and device ms to ||r|| < 1e-8 ||r0|| for FMG-then-V (pmg_solve(FMG), the FMG pass counted as a cycle) and for
    V-cycles from zero, with the sine and a random right-hand side (median of 3 solves).
With one process it also times, at the largest size, the fused residual-restriction of the FMG set-up (pmg_bench_pass
form 7, 18 B per fine point) against the residual + restriction pair it replaced (form 8, 34 B per fine point),
alternated, and reports GB/s from those byte counts.  --parent-lib PATH (one process) alternates the one-GPU FMG pass
between that build of libpmg.so and this tree's, one child process per measurement, and checks that both give the same
iterate.  The card name and power limit are printed first (nvidia-smi, read-only query).
"""
import hashlib
import json
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


def rhs(n, kind):
    if kind == "random":
        f = np.zeros((n, n))
        f[1:-1, 1:-1] = np.random.default_rng(72).uniform(-1, 1, (n - 2, n - 2))
        return f
    x = np.sin(np.pi * np.arange(n) / (n - 1))
    return 2 * np.pi ** 2 * np.outer(x, x)


CHILD = r"""
import hashlib, json, statistics, sys
import numpy as np
sys.path.insert(0, %(root)r)
import pmg_b200 as pmg
sys.modules["_pmg_b200_pkg"].LIB_PATH = %(lib)r  # before the first call loads the library
out = {}
for n in %(sizes)r:
    f = np.zeros((n, n))
    f[1:-1, 1:-1] = np.random.default_rng(72).uniform(-1, 1, (n - 2, n - 2))
    s = pmg.Solver(n, omega=2.0 / 3.0)
    s.set_rhs(f)
    ts = []
    for it in range(9):
        s.zero_guess()
        s.cycle(pmg.FMG, want_norm=False)
        if it >= 2:
            ts.append(s.last_ms)
    out[str(n)] = {"median_ms": statistics.median(ts), "min_ms": min(ts),
                   "iterate_sha1": hashlib.sha1(s.get_solution().tobytes()).hexdigest()}
    s.close()
print("RESULT " + json.dumps(out))
"""


def parent_ab(parent, sizes, rounds=3):
    libs = {"parent": os.path.abspath(parent),
            "this": os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200", "libpmg.so")}
    res = {k: {str(n): [] for n in sizes} for k in libs}
    sha = {k: {} for k in libs}
    for r in range(rounds):
        for name in (("parent", "this") if r % 2 == 0 else ("this", "parent")):
            p = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT, "lib": libs[name], "sizes": sizes}],
                               capture_output=True, text=True, timeout=900)
            line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
            if p.returncode != 0 or not line:
                print("A/B child (%s) failed: %s" % (name, (p.stdout + p.stderr)[-2000:]), flush=True)
                return
            for n, v in json.loads(line[0][7:]).items():
                res[name][n].append(v["median_ms"])
                sha[name][n] = v["iterate_sha1"]
    for n in sizes:
        a, b = res["parent"][str(n)], res["this"][str(n)]
        print("FMG pass A/B one GPU N=%d: parent median %.3f ms %s | this %.3f ms %s | ratio this/parent %.3f | "
              "same iterate: %s" % (n, statistics.median(a), [round(v, 3) for v in a], statistics.median(b),
                                    [round(v, 3) for v in b], statistics.median(b) / statistics.median(a),
                                    sha["parent"][str(n)] == sha["this"][str(n)]), flush=True)


def main():
    import torch
    import torch.distributed as dist
    import pmg_b200 as pmg
    args = sys.argv[1:]
    sizes, parent = [4097, 16385], None
    if "--sizes" in args:
        i = args.index("--sizes")
        sizes = [int(v) for v in args[i + 1].split(",")]
    if "--parent-lib" in args:
        parent = args[args.index("--parent-lib") + 1]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world = dist.get_world_size()
    if world > 1:
        rank, world, dev = pmg.init_distributed_from_torch(local)
    else:
        rank, dev = 0, local
    if rank == 0:
        print("cards (index, name, power limit, max SM clock):\n" + card(), flush=True)
    for n in sizes:
        y0, y1 = pmg.partition_rows(n, world, rank) if world > 1 else (0, n)
        dcfg = dict(rank=rank, n_ranks=world, agglomerate_below=min(257, n // 4)) if world > 1 else {}
        s = pmg.Solver(n, omega=2.0 / 3.0, device=dev, **dcfg)
        f = rhs(n, "random")
        s.set_rhs(np.ascontiguousarray(f[y0:y1]))
        ts = []
        for it in range(9):
            s.zero_guess()
            if world > 1:
                dist.barrier()
            s.cycle(pmg.FMG, want_norm=False)
            if it >= 2:
                ts.append(s.last_ms)
        t = torch.tensor([statistics.median(ts)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            print("N=%d ranks=%d: one FMG pass median %.3f ms (max over ranks; 7 passes after 2 warm-up: %s)"
                  % (n, world, float(t.item()), [round(v, 3) for v in ts]), flush=True)
        for rk in ("sine", "random"):
            f = rhs(n, rk)
            s.set_rhs(np.ascontiguousarray(f[y0:y1]))
            line = []
            for kind, name in ((pmg.FMG, "FMG+V"), (pmg.V, "V")):
                ms, k = [], 0
                for _ in range(3):
                    s.zero_guess()
                    if world > 1:
                        dist.barrier()
                    k, hist = s.solve(kind, rel_tol=1e-8, max_cycles=100)
                    ms.append(s.last_ms)
                line.append("%s %d cycles %.3f ms (final rel %.2e)" % (name, k, statistics.median(ms), hist[-1] / hist[0]))
            if rank == 0:
                print("N=%d ranks=%d rhs=%s: %s" % (n, world, rk, " | ".join(line)), flush=True)
        if world == 1 and n == max(sizes):
            ga, gb = [], []
            for r in range(5):  # alternated: the fused pass (form 7) and the pair it replaced (form 8)
                for form in ((7, 8) if r % 2 == 0 else (8, 7)):
                    (ga if form == 7 else gb).append(s.bench_pass(form, 0, 20))
            pts = float(n) * n
            ma, mb = statistics.median(ga), statistics.median(gb)
            print("N=%d FMG set-up, level 0 -> 1: fused residual-restriction %.3f ms (%.0f GB/s at 18 B/pt) | residual + "
                  "restriction %.3f ms (%.0f GB/s at 34 B/pt) | speed-up %.2fx  (medians of 5 alternated rounds of 20 "
                  "launches: %s / %s)" % (n, ma, 18 * pts / ma / 1e6, mb, 34 * pts / mb / 1e6, mb / ma,
                                          [round(v, 4) for v in ga], [round(v, 4) for v in gb]), flush=True)
        s.close()
    if world > 1:
        pmg.comm_finalize()
    dist.destroy_process_group()
    if parent and world == 1:
        parent_ab(parent, sizes)


if __name__ == "__main__":
    main()
