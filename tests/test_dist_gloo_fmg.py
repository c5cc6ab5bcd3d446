"""World-size-2 / 4 CPU test over gloo of the multi-GPU general-RHS full-multigrid pass (`cycle_fmg_dist` in
csrc/solver.cu, PMG_CYCLE_FMG on row slabs):

  (1) the interior of x zeroed on the owned rows (ring kept), halo rows of x and f exchanged;
  (2) f_1 = R(f - A x) on the owned coarse rows from a window that holds only 2 x rows and 1 f row beyond the slab (the
      depth of the fused residual-restriction kernel);
  (3) f_{l+1} = R f_l on the slab levels after an exchange of f_l, all-gathered at the first agglomerated level, then
      restricted redundantly down to 5 x 5;
  (4) 11 sweeps from zero on the coarsest level;
  (5) upwards: whole levels redundantly (prolongation into zeros, one V-cycle); slab levels: zeroed slab, the slab
      prolongation reading the child's rows (its last Pass B finished 4 rows beyond its slab) or the whole agglomerated
      level, and the V-cycle of `cycle_dist` started at that level, whose Pass A reads the f halo rows exchanged in (3);
  (6) level 0: x += P e_1 and the V-cycle of `cycle_dist` on the caller's f.

Executed with the CPU oracle's operators on each rank's window; rows a step does not compute or receive are NaN.  The
gathered result must be BIT-IDENTICAL to the oracle's orc_fmg_general (the specification of PMG_CYCLE_FMG), with no NaN in
an owned row, for both prolongations, a random guess with a non-zero ring and two passes in a row.
"""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from test_dist_gloo import PADY, Slab, cycle_dist, halo_exchange, prolong_rows, restrict_rows  # noqa: E402

X_DEPTH, F_DEPTH = 2, 1  # rows beyond the slab the fused residual-restriction reads (csrc/kernel_residual_restrict.cuh)
COARSE_SWEEPS = 11


def only_depth(slab, arr, depth):
    """a copy of a window with every row more than `depth` rows beyond the owned rows NaN"""
    out = arr.copy()
    lo, hi = slab.y0 - depth, slab.y1 + depth
    for g in range(slab.w0, slab.w1):
        if g < lo or g >= hi:
            out[g - slab.w0] = np.nan
    return out


def fmg_dist(orc, slabs, wholes, la, rank, world, omega, lo):
    """slabs[l] for l < la (+ slabs[la] = the slab-shaped window of level la), wholes[l - la] = (x, f) for l >= la"""
    import cpu_checkers as cc
    sizes = [s.n for s in slabs[:la]] + [w[0].shape[0] for w in wholes]
    lc = len(sizes) - 1
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    top = slabs[0]
    n = top.n
    # (1) interior of x zeroed on my rows; halo rows of x and f exchanged
    ga, gb = max(top.y0, 1), min(top.y1, n - 1)
    top.rows(top.x, ga, gb)[:, 1:n - 1] = 0.0
    halo_exchange(top, top.x, rank, world)
    halo_exchange(top, top.f, rank, world)
    # (2), (3) the chain of right-hand sides
    for l in range(lc):
        if l < la:
            L, K = slabs[l], slabs[l + 1]
            if l == 0:
                xw = only_depth(L, L.x, X_DEPTH)
                fw = only_depth(L, L.f, F_DEPTH)
                out = restrict_rows(orc.residual(xw, fw, 1.0 / (n - 1)), L.w0, n, K.y0, K.y1)
            else:
                halo_exchange(L, L.f, rank, world)
                out = restrict_rows(L.f, L.w0, L.n, K.y0, K.y1)
            K.f[:] = np.nan
            K.rows(K.f, K.y0, K.y1)[:] = out
            if l + 1 == la:
                parts = [None] * world
                rows0 = (K.n - 1) // world  # equally sized slabs; the last rank's extra row is the ring
                dist.all_gather_object(parts, out[:rows0].copy())
                full = np.zeros((K.n, K.n))
                full[: K.n - 1] = np.concatenate(parts)
                wholes[0][1][:] = full
        else:
            wholes[l + 1 - la][1][:] = orc.restrict_fw(wholes[l - la][1])
    # (4) coarsest level from zero
    xc, fc = wholes[-1]
    xc[:] = 0.0
    orc.jacobi(xc, fc, 1.0 / (sizes[lc] - 1), omega=omega, num_iter=COARSE_SWEEPS - 1)
    # (5), (6) upwards
    for l in range(lc - 1, -1, -1):
        if l >= la:
            xL, fL = wholes[l - la]
            xL[:] = 0.0
            orc.prolong_add(xL, wholes[l + 1 - la][0], mode)
            orc.cycle(xL, fL, kind=cc.V, omega=omega, eps=0.0, prolong=mode)
            continue
        L = slabs[l]
        if l > 0:
            L.x[:] = 0.0
        if l + 1 == la:
            W = slabs[la]
            W.x[:] = np.nan
            a, b = max(0, W.y0 - 4), min(W.n, W.y1 + 4)
            W.rows(W.x, a, b)[:] = wholes[0][0][a:b]
            e, c0 = W.x, W.w0
        else:
            e, c0 = slabs[l + 1].x, slabs[l + 1].w0
        own = L.rows(L.x, L.y0, L.y1)
        prolong_rows(own, L.y0, e, c0, L.n, lo)
        cycle_dist(orc, slabs, l, la, rank, world, omega, 1, False, False, lo)


def _worker(rank, world, port, n, agg_below, lo, q):
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
    wholes = [(np.zeros((m, m)), np.zeros((m, m))) for m in sizes[la:]]
    f = cc.random_rhs(n, seed=72)
    phi = np.random.default_rng(71).standard_normal((n, n))  # non-zero ring, garbage interior
    top = slabs[0]
    # only my rows are set (pmg_set_rhs / pmg_set_guess); the halo rows are the pass's business
    top.x[:] = np.nan
    top.f[:] = np.nan
    top.rows(top.x, top.y0, top.y1)[:] = phi[top.y0:top.y1]
    top.rows(top.f, top.y0, top.y1)[:] = f[top.y0:top.y1]
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    want = phi.copy()
    ok_bits, nans = True, 0
    for _ in range(2):  # the second pass starts from the first one's result
        fmg_dist(orc, slabs, wholes, la, rank, world, omega, lo)
        orc.fmg_general(want, f, omega=omega, prolong=mode)
        owned = top.rows(top.x, top.y0, top.y1)
        ok_bits = ok_bits and bool(np.array_equal(owned, want[top.y0:top.y1]))
        nans += int(np.isnan(owned).sum())
    q.put((rank, ok_bits, nans, la))
    dist.barrier()
    dist.destroy_process_group()


def _run(world, n, agg_below, lo, port):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, agg_below, lo, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    return sorted(res)


@pytest.mark.parametrize("world,n,agg_below,lo", [
    (2, 257, 33, 2),   # three slab levels (257, 129, 65), reference prolongation
    (2, 129, 33, 1),   # full-interior prolongation
    (4, 513, 129, 2),  # four ranks: middle ranks with two neighbours
    (4, 257, 129, 1),  # four ranks, full-interior prolongation, level 1 already agglomerated (la = 1)
])
def test_fmg_slab_schedule_is_bit_identical(world, n, agg_below, lo):
    res = _run(world, n, agg_below, lo, port=29831 + 7 * world + n % 83 + lo)
    assert len(res) == world
    for rank, ok_bits, nans, la in res:
        assert nans == 0, "rank %d: a halo is too shallow (poison reached an owned row)" % rank
        assert ok_bits, "rank %d: FMG result differs from the single-process oracle" % rank
        assert la >= 1
