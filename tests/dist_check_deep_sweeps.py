#!/usr/bin/env python
"""Multi-GPU equivalence check of the deep-sweep slab schedule (3 or 4 pre/post-smoothing sweeps), run under torchrun on
a box with >= 2 B200s:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29571 tests/dist_check_deep_sweeps.py [N ...]

Every rank runs its row slab; rank 0 also runs the same problem on its own GPU alone.  For N (default 1025 4097), sine and
random f, from a random guess with a non-zero ring:
  * V(3,3), V(4,4), V(1,4), V(4,1), W(3,3) with gamma = 2 and an F pass: three cycles, iterate bit-identical to one GPU,
    norms within 1e-12 relative;
  * a V(3,3) solve to 1e-8: the same cycle count, iterate bit-identical;
  * FMG-then-V(3,3) (power-of-two rank counts; otherwise PMG_ERR_UNSUPPORTED on every rank);
  * pmg_pcg(precond = 1) with V(3,3): the same step count, history within 1e-10 relative, iterate within 1e-9;
  * pmg_create with nu1 or nu2 = 0 or 5: PMG_ERR_UNSUPPORTED on every rank, before any collective;
  * a rank count whose row partition does not nest across levels (3 ranks, at every N): pmg_create refuses it on every
    rank; the F-cycle runs at power-of-two rank counts only.
Rank 0 prints a digest of each gathered iterate, so that runs with and without the NVLink exchanges (PMG_P2P=0) can be
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
from dist_check_pcg import gather_rows, rhs  # noqa: E402

UNSUPPORTED = 6

CYCLES = [("V(3,3)", pmg.V, 3, 3, 1), ("V(4,4)", pmg.V, 4, 4, 1), ("V(1,4)", pmg.V, 1, 4, 1), ("V(4,1)", pmg.V, 4, 1, 1),
          ("W(3,3)", pmg.W, 3, 3, 2), ("F(3,3)", pmg.F, 3, 3, 1)]


def partition_nests(n, world):
    """the rule pmg_create applies between level 0 and level 1: coarse row jc lives with fine row 2 jc"""
    nc = (n - 1) // 2 + 1
    return all(pmg.partition_rows(n, world, r)[0] == 2 * pmg.partition_rows(nc, world, r)[0] for r in range(world))


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [1025, 4097]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world, dev = pmg.init_distributed_from_torch(local)
    ok = True

    def report(label, good, x, extra=""):
        nonlocal ok
        if rank == 0:
            ok &= bool(good)
            print("%s ranks=%d: %s digest=%s %s" % (label, world, extra, hashlib.sha1(x.tobytes()).hexdigest()[:16],
                                                     "OK" if good else "FAIL"), flush=True)

    # refusals: every rank returns before any collective (a hang here would be a failure of the test)
    for nu1, nu2 in ((0, 2), (2, 0), (5, 2), (2, 5)):
        try:
            pmg.Solver(257, device=dev, rank=rank, n_ranks=world, nu1=nu1, nu2=nu2).close()
            refused = False
        except pmg.PmgError as e:
            refused = e.status == UNSUPPORTED
        flag = torch.tensor([1 if refused else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        report("create nu=(%d,%d)" % (nu1, nu2), int(flag.item()) == 1, np.zeros(1), "refused on every rank")

    for n in sizes:
        y0, y1 = pmg.partition_rows(n, world, rank)
        phi0 = np.random.default_rng(3).standard_normal((n, n))
        agg = min(257, n // 4)
        if not partition_nests(n, world):
            # e.g. 3 ranks: pmg_create refuses a row partition that does not nest across levels, at every n -- on every
            # rank, before any collective
            try:
                pmg.Solver(n, device=dev, rank=rank, n_ranks=world, agglomerate_below=agg, nu1=3, nu2=3).close()
                status = 0
            except pmg.PmgError as e:
                status = e.status
            flag = torch.tensor([1 if status == UNSUPPORTED else 0], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            report("N=%d partition does not nest" % n, int(flag.item()) == 1, np.zeros(1), "refused on every rank")
            continue
        for rk in ("sine", "random"):
            f = rhs(n, rk)
            for label, kind, nu1, nu2, gamma in CYCLES:
                if kind == pmg.F and world & (world - 1):
                    continue  # the F-cycle needs equally sized slabs (a power-of-two rank count)
                cfg = dict(omega=2.0 / 3.0, nu1=nu1, nu2=nu2, gamma=gamma)
                s = pmg.Solver(n, device=dev, rank=rank, n_ranks=world, agglomerate_below=agg, **cfg)
                s.set_rhs(np.ascontiguousarray(f[y0:y1]))
                s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
                try:
                    norms = [s.cycle(kind, want_norm=True) for _ in range(3)]
                except pmg.PmgError as e:
                    s.close()
                    report("N=%d rhs=%s %s" % (n, rk, label), False, np.zeros(1), str(e))
                    continue
                x = gather_rows(s.get_solution(), n, world)
                s.close()
                if rank == 0:
                    one = pmg.Solver(n, device=dev, **cfg)
                    one.set_rhs(f)
                    one.set_guess(phi0)
                    norms1 = [one.cycle(kind, want_norm=True) for _ in range(3)]
                    x1 = one.get_solution()
                    one.close()
                    dev_n = max(abs(a - b) / b for a, b in zip(norms, norms1))
                    report("N=%d rhs=%s %s" % (n, rk, label), np.array_equal(x, x1) and dev_n <= 1e-12, x,
                           "bit_identical=%s max_rel_norm_dev=%.2e" % (np.array_equal(x, x1), dev_n))
            # a V(3,3) solve, FMG-then-V(3,3), PCG(V(3,3))
            cfg = dict(omega=2.0 / 3.0, nu1=3, nu2=3)
            s = pmg.Solver(n, device=dev, rank=rank, n_ranks=world, agglomerate_below=agg, **cfg)
            s.set_rhs(np.ascontiguousarray(f[y0:y1]))
            s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
            k, hist = s.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
            xs = gather_rows(s.get_solution(), n, world)
            s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
            fmg_status = 0
            try:
                s.cycle(pmg.FMG, want_norm=False)
                kf, _ = s.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
            except pmg.PmgError as e:
                fmg_status, kf = e.status, -1
            xf = gather_rows(s.get_solution(), n, world)
            s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
            kp, hp = s.pcg(precond=1, rel_tol=1e-8, max_iter=60)
            xp = gather_rows(s.get_solution(), n, world)
            s.close()
            if rank == 0:
                one = pmg.Solver(n, device=dev, **cfg)
                one.set_rhs(f)
                one.set_guess(phi0)
                k1, h1 = one.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
                xs1 = one.get_solution()
                one.set_guess(phi0)
                one.cycle(pmg.FMG, want_norm=False)
                kf1, _ = one.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
                xf1 = one.get_solution()
                one.set_guess(phi0)
                kp1, hp1 = one.pcg(precond=1, rel_tol=1e-8, max_iter=60)
                xp1 = one.get_solution()
                one.close()
                rel = float(np.max(np.abs(hist - h1) / h1)) if k == k1 else float("inf")
                report("N=%d rhs=%s solve V(3,3)" % (n, rk), k == k1 and np.array_equal(xs, xs1) and rel <= 1e-12, xs,
                       "cycles %d/%d max_rel_hist_dev=%.2e" % (k, k1, rel))
                if world & (world - 1) == 0:
                    report("N=%d rhs=%s FMG+V(3,3)" % (n, rk), fmg_status == 0 and kf == kf1 and np.array_equal(xf, xf1),
                           xf, "cycles %d/%d" % (kf, kf1))
                else:
                    report("N=%d rhs=%s FMG refused" % (n, rk), fmg_status == UNSUPPORTED, np.zeros(1), "status %d" % fmg_status)
                relp = float(np.max(np.abs(hp - hp1) / hp1)) if kp == kp1 else float("inf")
                xdev = float(np.max(np.abs(xp - xp1)) / np.max(np.abs(xp1)))
                report("N=%d rhs=%s pcg V(3,3)" % (n, rk), kp == kp1 and relp <= 1e-10 and xdev <= 1e-9, xp,
                       "steps %d/%d max_rel_hist_dev=%.2e iterate_dev=%.2e" % (kp, kp1, relp, xdev))
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, src=0)
    pmg.comm_finalize()
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
