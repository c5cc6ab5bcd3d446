#!/usr/bin/env python
"""Multi-GPU equivalence check of PMG_CYCLE_FMG (the general-RHS full-multigrid pass on row slabs), run under torchrun on
a box with >= 2 B200s:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29551 tests/dist_check_fmg.py [N ...]

Every rank solves its row slab; rank 0 also solves the same problem on its own GPU alone.  For N (default 1025 4097), sine
and random f, both prolongations, V(2,2) and V(1,2), omega = 2/3 and 1, from a random guess with a non-zero ring:
  * pmg_cycle(FMG): iterate bit-identical to one GPU, residual norm within 1e-12 relative;
  * pmg_solve(FMG): same cycle count, history within 1e-12 relative, iterate bit-identical.

    ... tests/dist_check_fmg.py --expect-unsupported

instead checks the refusal where the slabs of the first agglomerated level are not all equal (a rank count that is not a
power of two, or PMG_COARSE_GATHER=1): every rank gets PMG_ERR_UNSUPPORTED -- from pmg_create, or from pmg_cycle(FMG)
before any collective, after which a V-cycle still runs on every rank -- and exits cleanly.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pmg_b200 as pmg  # noqa: E402

UNSUPPORTED = 6


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


def check_unsupported(rank, world, dev):
    """every rank must see PMG_ERR_UNSUPPORTED (at pmg_create or at the FMG pass) and stay usable"""
    n = 1025
    y0, y1 = pmg.partition_rows(n, world, rank)
    f = rhs(n, "random")
    where, ok = "create", False
    try:
        s = pmg.Solver(n, omega=2.0 / 3.0, device=dev, rank=rank, n_ranks=world, agglomerate_below=min(257, n // 4))
    except pmg.PmgError as e:
        ok = e.status == UNSUPPORTED
        print("rank %d: pmg_create refused: %s" % (rank, e), flush=True)
    else:
        s.set_rhs(np.ascontiguousarray(f[y0:y1]))
        s.zero_guess()
        where = "cycle"
        try:
            s.cycle(pmg.FMG)
            print("rank %d: PMG_CYCLE_FMG ran where it must be refused" % rank, flush=True)
        except pmg.PmgError as e:
            ok = e.status == UNSUPPORTED
            print("rank %d: pmg_cycle(FMG) refused: %s" % (rank, e), flush=True)
        s.cycle(pmg.V)  # no rank was left inside a collective: the next cycle runs everywhere
        s.close()
    flags = [None] * world
    dist.all_gather_object(flags, (ok, where))
    good = all(o for o, _ in flags) and len({w for _, w in flags}) == 1
    if rank == 0:
        print("unsupported ranks=%d refused at %s on every rank: %s" % (world, flags[0][1], "OK" if good else "FAIL"),
              flush=True)
    return good


def main():
    args = sys.argv[1:]
    expect_unsupported = "--expect-unsupported" in args
    if expect_unsupported:
        args.remove("--expect-unsupported")
    sizes = [int(a) for a in args] or [1025, 4097]
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world, dev = pmg.init_distributed_from_torch(local)
    if expect_unsupported:
        ok = check_unsupported(rank, world, dev)
    else:
        ok = True
        for n in sizes:
            y0, y1 = pmg.partition_rows(n, world, rank)
            phi0 = np.random.default_rng(3).standard_normal((n, n))  # non-zero ring, garbage interior
            for rk in ("sine", "random"):
                f = rhs(n, rk)
                for prolong in (pmg.PROLONG_REFERENCE, pmg.PROLONG_FULL):
                    for nu1, omega in ((2, 2.0 / 3.0), (1, 2.0 / 3.0), (2, 1.0), (1, 1.0)):
                        cfg = dict(omega=omega, nu1=nu1, nu2=2, prolong_mode=prolong)
                        s = pmg.Solver(n, device=dev, rank=rank, n_ranks=world, agglomerate_below=min(257, n // 4), **cfg)
                        s.set_rhs(np.ascontiguousarray(f[y0:y1]))
                        s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
                        norm = s.cycle(pmg.FMG)
                        ms_pass = s.last_ms
                        one_pass = s.get_solution()
                        s.set_guess(np.ascontiguousarray(phi0[y0:y1]))
                        k, hist = s.solve(pmg.FMG, rel_tol=1e-8, max_cycles=60)
                        ms_solve = s.last_ms
                        solved = s.get_solution()
                        s.close()
                        full_pass = gather_rows(one_pass, n, world)
                        full_solved = gather_rows(solved, n, world)
                        if rank == 0:
                            one = pmg.Solver(n, device=dev, **cfg)
                            one.set_rhs(f)
                            one.set_guess(phi0)
                            norm1 = one.cycle(pmg.FMG)
                            ref_pass = one.get_solution()
                            one.set_guess(phi0)
                            k1, h1 = one.solve(pmg.FMG, rel_tol=1e-8, max_cycles=60)
                            ms1 = one.last_ms
                            ref_solved = one.get_solution()
                            one.close()
                            same_pass = np.array_equal(full_pass, ref_pass)
                            same_solved = np.array_equal(full_solved, ref_solved)
                            rel_norm = abs(norm - norm1) / norm1
                            rel_hist = float(np.max(np.abs(hist - h1) / h1)) if k == k1 else float("inf")
                            good = same_pass and same_solved and k == k1 and rel_norm <= 1e-12 and rel_hist <= 1e-12
                            ok &= good
                            print("N=%d rhs=%s prolong=%d V(%d,2) omega=%.3f ranks=%d: pass iterate_bit_identical=%s "
                                  "rel_norm_dev=%.2e | solve cycles %d/%d iterate_bit_identical=%s max_rel_hist_dev=%.2e "
                                  "| ms pass=%.3f solve dist=%.3f single=%.3f %s"
                                  % (n, rk, prolong, nu1, omega, world, same_pass, rel_norm, k, k1, same_solved, rel_hist,
                                     ms_pass, ms_solve, ms1, "OK" if good else "FAIL"), flush=True)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, src=0)
    pmg.comm_finalize()
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
