"""World-size-2 / 4 CPU test over gloo of preconditioned conjugate gradients on row slabs (`pcg_dist` in csrc/solver.cu,
pmg_pcg with n_ranks > 1), executed with the CPU oracle's operators on each rank's window:

  start:   halo rows of x exchanged, r = f - A x on the owned interior rows, ||r|| summed in rank order;
  step:    precond = 1: PADY halo rows of r exchanged, z = one `cycle_dist` V-cycle from zero on (z, r) -- level 0 does no
           exchange of its own and reads r's halo as its f halo; its last Pass B finishes the owned rows only;
           precond = 0: z = r;
           one row of z beyond the slab from each neighbour;
           rz = r.z; p = z + beta p (p = z on the first step) on the owned rows AND the interior row beyond each slab edge,
           recomputed there from z and the previous p, so p is never exchanged; Ap and p.Ap on the owned interior rows;
           x += alpha p, r -= alpha Ap, r.r -- every sum over the owned interior rows, all-gathered and added in rank order.

Every row a step neither computes nor receives is NaN: z beyond the one row the direction pass reads, r beyond its PADY
halo (and r, x beyond the owned rows after each update, where they are stale), p beyond its one extra row.  The result must
match the oracle's orc_pcg (the specification of pmg_pcg): the same step count, the history within 1e-10 relative, the
iterate within 1e-9 of its largest entry, and no NaN in an owned row.  The only source of difference is the grouping of
the sums.
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from test_dist_gloo import PADY, Slab, cycle_dist, halo_exchange  # noqa: E402


def halo_rows(slab, arr, rank, world, depth):
    """`depth` owned rows to each neighbour's halo (comm_halo_exchange with a depth below PADY)"""
    reqs = []
    up_recv = torch.zeros((depth, slab.n), dtype=torch.float64)
    dn_recv = torch.zeros((depth, slab.n), dtype=torch.float64)
    if rank > 0:
        reqs.append(dist.isend(torch.from_numpy(slab.rows(arr, slab.y0, slab.y0 + depth).copy()), rank - 1))
        reqs.append(dist.irecv(up_recv, rank - 1))
    if rank < world - 1:
        reqs.append(dist.isend(torch.from_numpy(slab.rows(arr, slab.y1 - depth, slab.y1).copy()), rank + 1))
        reqs.append(dist.irecv(dn_recv, rank + 1))
    for q in reqs:
        q.wait()
    if rank > 0:
        slab.rows(arr, slab.y0 - depth, slab.y0)[:] = up_recv.numpy()
    if rank < world - 1:
        slab.rows(arr, slab.y1, slab.y1 + depth)[:] = dn_recv.numpy()


def only_rows(slab, arr, a, b):
    """a copy of a window with every row outside global rows [a, b) NaN"""
    out = arr.copy()
    for g in range(slab.w0, slab.w1):
        if g < a or g >= b:
            out[g - slab.w0] = np.nan
    return out


def global_sum(v, world):
    """this rank's partial sum all-gathered and added in rank order: the same bits on every rank"""
    allp = [torch.zeros(1, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(allp, torch.tensor([v], dtype=torch.float64))
    s = 0.0
    for t in allp:
        s += float(t)
    return s


def pcg_dist(orc, slabs, la, rank, world, omega, lo, precond, rel_tol, max_iter):
    top = slabs[0]
    n, h = top.n, 1.0 / (top.n - 1)
    ga, gb = max(top.y0, 1), min(top.y1, n - 1)  # owned interior rows
    own = slice(ga - top.w0, gb - top.w0)
    halo_exchange(top, top.x, rank, world)
    r = np.full_like(top.x, np.nan)
    r[own] = orc.residual(top.x, top.f, h)[own]
    for g in (0, n - 1):  # the ring rows of r are zero, never NaN
        if top.w0 <= g < top.w1:
            r[g - top.w0] = 0.0
    r0 = np.sqrt(global_sum(float(np.sum(r[own] ** 2)), world))
    hist = [r0]
    p = np.full_like(top.x, np.nan)
    rz = 0.0
    k = 0
    while k < max_iter and not (hist[k] < rel_tol * hist[0]) and hist[0] > 0.0:
        if precond:
            halo_exchange(top, r, rank, world)
            sx, sf = top.x, top.f
            top.x, top.f = np.full_like(sx, np.nan), r
            cycle_dist(orc, slabs, 0, la, rank, world, omega, 1, False, True, lo)
            z = only_rows(top, top.x, top.y0, top.y1)
            top.x, top.f = sx, sf
        else:
            z = only_rows(top, r, top.y0, top.y1)
        halo_rows(top, z, rank, world, 1)
        z = only_rows(top, z, top.y0 - 1, top.y1 + 1)
        rz_new = global_sum(float(np.sum(r[own] * z[own])), world)
        # the direction on the owned rows and one interior row beyond each slab edge; zero on the Dirichlet ring
        pa, pb = max(top.y0 - 1, 1), min(top.y1 + 1, n - 1)
        rows = slice(pa - top.w0, pb - top.w0)
        pn = np.full_like(p, np.nan)
        pn[rows] = z[rows] if k == 0 else z[rows] + (rz_new / rz) * p[rows]
        pn[rows, 0] = pn[rows, n - 1] = 0.0
        for g in (0, n - 1):
            if top.w0 <= g < top.w1:
                pn[g - top.w0] = 0.0
        p = pn
        rz = rz_new
        ap = np.full_like(p, np.nan)
        a, b = ga - top.w0, gb - top.w0
        c = p[a:b, 1:n - 1]
        ap[a:b, 1:n - 1] = ((((4 * c - p[a:b, :n - 2]) - p[a:b, 2:]) - p[a - 1:b - 1, 1:n - 1]) - p[a + 1:b + 1, 1:n - 1]) / (h * h)
        ap[a:b, 0] = ap[a:b, n - 1] = 0.0
        pap = global_sum(float(np.sum(p[own] * ap[own])), world)
        alpha = rz / pap
        top.x[own] = top.x[own] + alpha * p[own]
        r[own] = r[own] - alpha * ap[own]
        r = only_rows(top, r, top.y0, top.y1)  # the rest of r (and x) is stale now
        top.x[:] = only_rows(top, top.x, top.y0, top.y1)
        k += 1
        hist.append(np.sqrt(global_sum(float(np.sum(r[own] ** 2)), world)))
    return k, np.array(hist)


def _worker(rank, world, port, n, agg_below, lo, precond, ring, q):
    import cpu_checkers as cc
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    orc = cc.load("orc")
    omega = 2.0 / 3.0
    sizes = [n]
    while sizes[-1] > 5:
        sizes.append((sizes[-1] - 1) // 2 + 1)
    la = 0
    while la < len(sizes) - 1 and sizes[la] > agg_below and ((sizes[la] - 1) // 2) // world * 2 >= 4 * PADY:
        la += 1
    assert la >= 1
    slabs = [Slab(m, rank, world) for m in sizes[:la + 1]]
    f = cc.random_rhs(n, seed=31)
    rng = np.random.default_rng(32)
    phi = rng.standard_normal((n, n)) if ring else np.zeros((n, n))
    if not ring:
        phi[1:-1, 1:-1] = rng.standard_normal((n - 2, n - 2))
    top = slabs[0]
    top.x[:] = np.nan  # only my rows are set (pmg_set_guess); f's halo rows as pmg_set_rhs exchanges them
    top.rows(top.x, top.y0, top.y1)[:] = phi[top.y0:top.y1]
    top.f[:] = f[top.w0:top.w1]
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    rel_tol, max_iter = 1e-8, 60
    k, hist = pcg_dist(orc, slabs, la, rank, world, omega, lo, precond, rel_tol, max_iter)
    want = phi.copy()
    wk, whist = orc.pcg(want, f, precond=precond, omega=omega, prolong=mode, rel_tol=rel_tol, max_iter=max_iter)
    owned = top.rows(top.x, top.y0, top.y1)
    nans = int(np.isnan(owned).sum())
    same_k = k == wk
    hist_rel = float(np.max(np.abs(hist - whist) / whist)) if same_k else float("inf")
    x_dev = float(np.max(np.abs(np.nan_to_num(owned, nan=1e300) - want[top.y0:top.y1]))) / float(np.max(np.abs(want)))
    q.put((rank, nans, same_k, k, wk, hist_rel, x_dev))
    dist.barrier()
    dist.destroy_process_group()


def _run(world, n, agg_below, lo, precond, ring, port):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, agg_below, lo, precond, ring, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    return sorted(res)


@pytest.mark.parametrize("world,n,agg_below,lo,precond,ring", [
    (2, 65, 17, 1, 1, True),     # smallest: two slab levels (65, 33), a guess with a non-zero Dirichlet ring
    (2, 257, 33, 1, 1, False),   # three slab levels (257, 129, 65)
    (2, 257, 33, 1, 0, True),    # plain CG
    (4, 257, 65, 1, 1, True),    # four ranks: middle ranks with two neighbours
    (4, 129, 17, 1, 0, False),   # four ranks, plain CG
])
def test_pcg_slab_schedule_matches_oracle(world, n, agg_below, lo, precond, ring):
    res = _run(world, n, agg_below, lo, precond, ring, port=30131 + 7 * world + n % 89 + 3 * precond + int(ring))
    assert len(res) == world
    for rank, nans, same_k, k, wk, hist_rel, x_dev in res:
        assert nans == 0, "rank %d: a halo is too shallow (poison reached an owned row)" % rank
        assert same_k, "rank %d: %d steps, the oracle took %d" % (rank, k, wk)
        assert hist_rel <= 1e-10, (rank, hist_rel)
        assert x_dev <= 1e-9, (rank, x_dev)
