#!/usr/bin/env python
"""Multi-GPU equivalence check of pmg_pcg on row slabs, run under torchrun on a box with >= 2 B200s:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29561 tests/dist_check_pcg.py [N ...]

Every rank solves its row slab; rank 0 also solves the same problem on its own GPU alone.  For N (default 1025 4097), sine
and random f, precond 1 (one V(2,2) cycle, omega = 2/3, full-interior prolongation) and 0 (plain CG), from a random guess
with a non-zero ring:
  * pmg_pcg: the same step count as one GPU, history within 1e-10 relative, iterate within 1e-9 of its largest entry (the
    rank-ordered sums group the dot products differently from one GPU's tree sums);
  * afterwards one V-cycle from the same guess on every rank: iterate bit-identical to one GPU.
Rank 0 prints a digest of each gathered PCG iterate, so that runs with and without the NVLink exchanges (PMG_P2P=0) can be
compared bit for bit.
"""
import hashlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pmg_b200 as pmg  # noqa: E402


def gather_rows(mine, n, world):
    parts = [torch.empty((pmg.partition_rows(n, world, r)[1] - pmg.partition_rows(n, world, r)[0], n),
                         dtype=torch.float64, device="cuda") for r in range(world)]
    dist.all_gather(parts, torch.from_numpy(mine).cuda())
    return torch.cat(parts).cpu().numpy()


def rhs(n, kind):
    if kind == "random":
        f = np.zeros((n, n))
        f[1:-1, 1:-1] = np.random.default_rng(7).uniform(-1, 1, (n - 2, n - 2))
        return f
    x = np.sin(np.pi * np.arange(n) / (n - 1))
    return 2 * np.pi ** 2 * np.outer(x, x)


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [1025, 4097]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world, dev = pmg.init_distributed_from_torch(local)
    ok = True
    cfg = dict(omega=2.0 / 3.0, nu1=2, nu2=2, prolong_mode=pmg.PROLONG_FULL)
    for n in sizes:
        y0, y1 = pmg.partition_rows(n, world, rank)
        phi0 = np.random.default_rng(3).standard_normal((n, n))  # non-zero ring, garbage interior
        for rk in ("sine", "random"):
            f = rhs(n, rk)
            for precond in (1, 0):
                max_iter = 60 if precond else 40
                s = pmg.Solver(n, device=dev, rank=rank, n_ranks=world, agglomerate_below=min(257, n // 4), **cfg)
                s.set_rhs(np.ascontiguousarray(f[y0:y1]))
                s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
                k, hist = s.pcg(precond=precond, rel_tol=1e-8, max_iter=max_iter)
                ms = s.last_ms
                x = gather_rows(s.get_solution(), n, world)
                s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
                s.cycle(pmg.V, want_norm=False)
                xv = gather_rows(s.get_solution(), n, world)
                s.close()
                if rank == 0:
                    one = pmg.Solver(n, device=dev, **cfg)
                    one.set_rhs(f)
                    one.set_guess(phi0)
                    k1, h1 = one.pcg(precond=precond, rel_tol=1e-8, max_iter=max_iter)
                    ms1 = one.last_ms
                    x1 = one.get_solution()
                    one.set_guess(phi0)
                    one.cycle(pmg.V, want_norm=False)
                    xv1 = one.get_solution()
                    one.close()
                    rel_hist = float(np.max(np.abs(hist - h1) / h1)) if k == k1 else float("inf")
                    x_dev = float(np.max(np.abs(x - x1)) / np.max(np.abs(x1)))
                    same_v = np.array_equal(xv, xv1)
                    good = k == k1 and rel_hist <= 1e-10 and x_dev <= 1e-9 and same_v and not np.isnan(x).any()
                    ok &= good
                    print("N=%d rhs=%s precond=%d ranks=%d: steps %d/%d max_rel_hist_dev=%.2e iterate_dev=%.2e "
                          "digest=%s | V-cycle after pcg bit_identical=%s | ms dist=%.3f single=%.3f %s"
                          % (n, rk, precond, world, k, k1, rel_hist, x_dev, hashlib.sha1(x.tobytes()).hexdigest()[:16],
                             same_v, ms, ms1, "OK" if good else "FAIL"), flush=True)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, src=0)
    pmg.comm_finalize()
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
