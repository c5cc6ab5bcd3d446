"""CPU tests over gloo of the DEEP-SWEEP slab schedule (`cycle_dist` in csrc/solver.cu with max(nu1, nu2) >= 3):

  * Pass A finishes xb on pass_a_depth = (8 - nu1) rounded down to even rows beyond the slab;
  * Pass B of a level l > 0 finishes x on pass_b_ext = (pass_a_depth - nu2) rounded down to even rows, level 0 on its own;
  * before Pass B of level l, the child slab's rows pass_b_ext(l + 1) + 1 .. pass_b_coarse_rows(l) beyond its slab come
    from the neighbours (the up-exchange); the agglomerated level is whole on every rank and read in place.

Executed with the CPU oracle's operators on each rank's window at 2, 3 and 4 ranks, for every (nu1, nu2) in 1..4 x 1..4,
V- and W-cycles, both prolongations, omega in {2/3, 1} and a random guess with a non-zero Dirichlet ring.  Rows a pass
neither computes nor receives are NaN; rows a window's edge leaves stale stay finite but wrong.  The gathered iterate after
several cycles must be BIT-IDENTICAL to the single-process oracle.  The F-cycle and the FMG pass (power-of-two rank
counts) run the existing gloo models with this cycle_dist.
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

from test_dist_gloo import PADY, Slab, halo_exchange, prolong_rows, restrict_rows  # noqa: E402

PAIRS = [(a, b) for a in range(1, 5) for b in range(1, 5)]


# ---- depths of the schedule (csrc/solver.cu: pass_a_depth, pass_b_ext, pass_b_coarse_rows, up_exchange_rows) ----
def deep(nu1, nu2):
    return max(nu1, nu2) >= 3


def pass_a_depth(nu1, nu2):
    return (PADY - nu1) & ~1 if deep(nu1, nu2) else 6


def pass_b_ext(nu1, nu2, l):
    if l == 0:
        return 0
    return max(0, (pass_a_depth(nu1, nu2) - nu2) & ~1) if deep(nu1, nu2) else 4


def up_exchange_rows(nu1, nu2, l):
    if not deep(nu1, nu2):
        return 0
    read = (pass_b_ext(nu1, nu2, l) + nu2 + (1 if l == 0 else 0)) // 2 + 1
    return max(0, read - pass_b_ext(nu1, nu2, l + 1))


def test_depths_fit_the_halo():
    """every pass reads only rows that exist: x / f within PADY, the up-exchange within MAX_UP_ROWS = 4"""
    for nu1, nu2 in PAIRS:
        da = pass_a_depth(nu1, nu2)
        assert da + nu1 <= PADY and da % 2 == 0
        for l in range(3):
            e = pass_b_ext(nu1, nu2, l)
            assert e % 2 == 0 and e + nu2 <= da
            assert 0 <= up_exchange_rows(nu1, nu2, l) <= 4
    # nu <= 2: today's schedule, no up-exchange
    assert all(up_exchange_rows(a, b, l) == 0 for a in (1, 2) for b in (1, 2) for l in range(3))


def poison_outside(slab, arr, ext, rank, world):
    lo = slab.y0 - (ext if rank > 0 else 0)
    hi = slab.y1 + (ext if rank < world - 1 else 0)
    for g in range(slab.w0, slab.w1):
        if g < lo or g >= hi:
            arr[g - slab.w0] = np.nan


def exchange_rows(slab, arr, rank, world, d0, d1):
    """rows at depth d0 + 1 .. d1 beyond my slab from the neighbours' owned rows (the up-exchange)"""
    import torch
    reqs, up_recv, dn_recv = [], None, None
    if rank > 0:
        reqs.append(dist.isend(torch.from_numpy(slab.rows(arr, slab.y0 + d0, slab.y0 + d1).copy()), rank - 1))
        up_recv = torch.zeros((d1 - d0, slab.n), dtype=torch.float64)
        reqs.append(dist.irecv(up_recv, rank - 1))
    if rank < world - 1:
        reqs.append(dist.isend(torch.from_numpy(slab.rows(arr, slab.y1 - d1, slab.y1 - d0).copy()), rank + 1))
        dn_recv = torch.zeros((d1 - d0, slab.n), dtype=torch.float64)
        reqs.append(dist.irecv(dn_recv, rank + 1))
    for q in reqs:
        q.wait()
    if up_recv is not None:
        slab.rows(arr, slab.y0 - d1, slab.y0 - d0)[:] = up_recv.numpy()
    if dn_recv is not None:
        slab.rows(arr, slab.y1 + d0, slab.y1 + d1)[:] = dn_recv.numpy()


def sweeps(orc, x, f, h, omega, k):
    """k Jacobi sweeps on a window; NaN poison travels as 1e300 through the oracle and back"""
    xs = np.nan_to_num(x, nan=1e300)
    orc.jacobi(xs, f, h, omega=omega, num_iter=k - 1)
    xs[np.abs(xs) > 1e200] = np.nan
    return xs


def make_cycle_dist(nu1, nu2):
    """the deep-sweep cycle_dist with the call signature of test_dist_gloo.cycle_dist"""

    def cycle_dist(orc, slabs, l, la, rank, world, omega, gamma, w_form, x_is_zero, lo):
        import cpu_checkers as cc
        L, K = slabs[l], slabs[l + 1]
        n, h = L.n, 1.0 / (L.n - 1)
        if not x_is_zero:
            halo_exchange(L, L.x, rank, world)
        if l > 0 and x_is_zero:
            halo_exchange(L, L.f, rank, world)
        # Pass A: xb = S^nu1 x, kept on pass_a_depth rows beyond the slab; the coarse RHS of the owned coarse rows
        xb = sweeps(orc, np.zeros_like(L.x) if x_is_zero else L.x, L.f, h, omega, nu1)
        r = orc.residual(np.nan_to_num(xb), np.nan_to_num(L.f), h)
        K.f[:] = np.nan
        K.rows(K.f, K.y0, K.y1)[:] = restrict_rows(r, L.w0, n, K.y0, K.y1)
        poison_outside(L, xb, pass_a_depth(nu1, nu2), rank, world)
        L.xb[:] = xb
        reps = gamma if w_form else 1
        if l + 1 < la:
            for k in range(reps):
                cycle_dist(orc, slabs, l + 1, la, rank, world, omega, gamma, w_form, k == 0, lo)
            m = up_exchange_rows(nu1, nu2, l)
            if m > 0:
                e0 = pass_b_ext(nu1, nu2, l + 1)
                exchange_rows(K, K.x, rank, world, e0, e0 + m)
        else:
            # every rank gathers the first agglomerated level and solves it; Pass B reads it in place
            nc = K.n
            parts = [None] * world
            dist.all_gather_object(parts, K.rows(K.f, K.y0, K.y1).copy())
            f_full = np.concatenate(parts)
            e = np.zeros((nc, nc))
            for _ in range(reps):
                orc.cycle(e, f_full, kind=cc.W if w_form else cc.V, omega=omega, eps=0.0, alpha=gamma, v1=nu1 - 1,
                          v2=nu2 - 1, prolong=cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE)
            K.x[:] = e[K.w0:K.w1]
        # Pass B: x = S^nu2 (xb + P e), kept on pass_b_ext rows beyond the slab
        x = L.xb.copy()
        prolong_rows(x, L.w0, K.x, K.w0, n, lo)
        x = sweeps(orc, x, L.f, h, omega, nu2)
        poison_outside(L, x, pass_b_ext(nu1, nu2, l), rank, world)
        L.x[:] = x

    return cycle_dist


class NuOracle:
    """the oracle with (v1, v2) = (nu1 - 1, nu2 - 1) as the default of every multigrid entry point"""

    def __init__(self, orc, nu1, nu2):
        self._orc, self._v = orc, dict(v1=nu1 - 1, v2=nu2 - 1)

    def __getattr__(self, name):
        return getattr(self._orc, name)

    def cycle(self, phi, f, **kw):
        return self._orc.cycle(phi, f, **{**self._v, **kw})

    def fmg_general(self, phi, f, **kw):
        return self._orc.fmg_general(phi, f, **{**self._v, **kw})


def levels(n, world, agg_below):
    sizes = [n]
    while sizes[-1] > 5:
        sizes.append((sizes[-1] - 1) // 2 + 1)
    la = 0
    while la < len(sizes) - 1 and sizes[la] > agg_below and ((sizes[la] - 1) // 2) // world * 2 >= 4 * PADY:
        la += 1
    return sizes, la


def run_cycles(orc, rank, world, case):
    """case = (kind, n, agg_below, nu1, nu2, gamma, lo, omega): 3 cycles from a random guess with a non-zero ring"""
    import cpu_checkers as cc
    kind, n, agg_below, nu1, nu2, gamma, lo, omega = case
    sizes, la = levels(n, world, agg_below)
    slabs = [Slab(m, rank, world) for m in sizes[:la + 1]]
    top = slabs[0]
    f = cc.random_rhs(n, seed=5 + n)
    phi = np.random.default_rng(n + 10 * nu1 + nu2).uniform(-1.0, 1.0, (n, n))
    top.f[:] = f[top.w0:top.w1]  # pmg_set_rhs + its halo exchange
    top.x[:] = np.nan
    top.rows(top.x, top.y0, top.y1)[:] = phi[top.y0:top.y1]  # pmg_set_guess: owned rows only
    want = phi.copy()
    w_form = kind == "W"
    cyc = make_cycle_dist(nu1, nu2)
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    for _ in range(3):
        cyc(orc, slabs, 0, la, rank, world, omega, gamma, w_form, False, lo)
        orc.cycle(want, f, kind=cc.W if w_form else cc.V, omega=omega, eps=0.0, alpha=gamma, v1=nu1 - 1, v2=nu2 - 1,
                  prolong=mode)
    owned = top.rows(top.x, top.y0, top.y1)
    return bool(np.array_equal(owned, want[top.y0:top.y1])), int(np.isnan(owned).sum()), la


def run_fcycle(orc, rank, world, case):
    """the F-cycle model of test_dist_gloo_fcycle with the deep-sweep cycle_dist"""
    import cpu_checkers as cc
    import test_dist_gloo_fcycle as fc
    _, n, agg_below, nu1, nu2, _, lo, omega = case
    norc = NuOracle(orc, nu1, nu2)
    fc.cycle_dist = make_cycle_dist(nu1, nu2)
    sizes, la = levels(n, world, agg_below)
    slabs = [Slab(m, rank, world) for m in sizes[:la + 1]]
    wholes = [(np.zeros((m, m)), np.zeros((m, m)), np.zeros((m, m))) for m in sizes[la:]]
    phi = np.random.default_rng(11).standard_normal((n, n))
    f = orc.rhs(n)
    top = slabs[0]
    top.x[:] = phi[top.w0:top.w1]
    top.f[:] = f[top.w0:top.w1]
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    fc.fcycle_dist(norc, slabs, wholes, la, rank, world, omega, lo)
    want = phi.copy()
    norc.cycle(want, f, kind=cc.F, omega=omega, eps=0.0, prolong=mode)
    owned = top.rows(top.x, top.y0, top.y1)
    return bool(np.array_equal(owned, want[top.y0:top.y1])), int(np.isnan(owned).sum()), la


def run_fmg(orc, rank, world, case):
    """the FMG model of test_dist_gloo_fmg with the deep-sweep cycle_dist; the slab prolongation P e_{l+1} reads the
    child slab after an exchange of its halo rows (cycle_fmg_dist)"""
    import cpu_checkers as cc
    import test_dist_gloo_fmg as fm
    _, n, agg_below, nu1, nu2, _, lo, omega = case
    norc = NuOracle(orc, nu1, nu2)
    fm.cycle_dist = make_cycle_dist(nu1, nu2)
    sizes, la = levels(n, world, agg_below)
    slabs = [Slab(m, rank, world) for m in sizes[:la + 1]]

    def prolong_after_exchange(own, y0, e, c0, nn, lo_):
        for s in slabs[1:la]:
            if e is s.x:
                halo_exchange(s, s.x, rank, world)
        prolong_rows(own, y0, e, c0, nn, lo_)

    fm.prolong_rows = prolong_after_exchange
    wholes = [(np.zeros((m, m)), np.zeros((m, m))) for m in sizes[la:]]
    f = cc.random_rhs(n, seed=72)
    phi = np.random.default_rng(71).standard_normal((n, n))
    top = slabs[0]
    top.x[:] = np.nan
    top.f[:] = np.nan
    top.rows(top.x, top.y0, top.y1)[:] = phi[top.y0:top.y1]
    top.rows(top.f, top.y0, top.y1)[:] = f[top.y0:top.y1]
    mode = cc.PROLONG_FULL if lo == 1 else cc.PROLONG_REFERENCE
    fm.fmg_dist(norc, slabs, wholes, la, rank, world, omega, lo)
    want = phi.copy()
    norc.fmg_general(want, f, omega=omega, prolong=mode)
    owned = top.rows(top.x, top.y0, top.y1)
    return bool(np.array_equal(owned, want[top.y0:top.y1])), int(np.isnan(owned).sum()), la


def _worker(rank, world, port, cases, q):
    import cpu_checkers as cc
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    orc = cc.load("orc")
    out = []
    for case in cases:
        fn = {"F": run_fcycle, "FMG": run_fmg}.get(case[0], run_cycles)
        out.append((case,) + fn(orc, rank, world, case))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def _run(world, cases, port):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cases, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=900) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    return sorted(res)


def _check(world, cases, port, min_la):
    res = _run(world, cases, port)
    assert len(res) == world
    bad = []
    for rank, out in res:
        for case, ok_bits, nans, la in out:
            assert la >= min_la, case
            if nans or not ok_bits:
                bad.append((rank, case, "%d NaN in owned rows" % nans if nans else "differs from the oracle"))
    assert not bad, bad


OMEGAS = (2.0 / 3.0, 1.0)


@pytest.mark.parametrize("world,n,agg_below", [
    (2, 257, 33),   # slab levels 257, 129, 65
    (3, 129, 65),   # a middle rank with two neighbours, uneven slabs; one slab level (a partition over 3 ranks does
                    # not nest across levels, which pmg_create refuses, so the agglomerated level comes next)
    (4, 257, 33),   # slab levels 257, 129
])
def test_every_sweep_pair_is_bit_identical(world, n, agg_below):
    """all 16 (nu1, nu2) pairs, V-cycles, both prolongations and both omegas in turn"""
    cases = [("V", n if i % 3 or world != 2 else 129, agg_below, a, b, 1, 1 + i % 2, OMEGAS[(i // 2) % 2])
             for i, (a, b) in enumerate(PAIRS)]
    _check(world, cases, 29931 + 11 * world, 1 if world == 3 else 2)


def test_large_grids_with_many_slab_levels():
    """n = 513 / 1025 with a small agglomeration threshold: 4-5 slab levels, so up-exchanges chain"""
    cases = [("V", 1025, 33, 3, 3, 1, 2, 2.0 / 3.0), ("V", 1025, 33, 4, 4, 1, 1, 1.0), ("V", 513, 17, 1, 4, 1, 2, 1.0),
             ("V", 513, 17, 4, 1, 1, 1, 2.0 / 3.0), ("V", 513, 17, 2, 4, 1, 2, 2.0 / 3.0), ("V", 513, 17, 3, 4, 1, 1, 2.0 / 3.0)]
    _check(2, cases, 29991, 4)


@pytest.mark.parametrize("world", [2, 4])
def test_w_cycles_are_bit_identical(world):
    """W-cycles (gamma = 2, 3): repeated visits re-exchange the iterate, each parent Pass B up-exchanges once"""
    n = 257
    cases = [("W", n, 33, 3, 3, 2, 2, 2.0 / 3.0), ("W", n, 33, 4, 4, 2, 1, 1.0), ("W", n, 33, 1, 4, 3, 2, 1.0),
             ("W", n, 33, 4, 2, 3, 1, 2.0 / 3.0)]
    _check(world, cases, 30011 + world, 2)


@pytest.mark.parametrize("world,n,agg_below", [(2, 257, 33), (4, 513, 129)])
def test_fcycle_and_fmg_are_bit_identical(world, n, agg_below):
    """the F-cycle and the FMG pass over the deep-sweep V-cycles (power-of-two rank counts)"""
    cases = [("F", n, agg_below, 3, 3, 1, 2, 2.0 / 3.0), ("F", n, agg_below, 4, 4, 1, 1, 1.0),
             ("FMG", n, agg_below, 3, 3, 1, 2, 2.0 / 3.0), ("FMG", n, agg_below, 1, 4, 1, 1, 1.0),
             ("FMG", n, agg_below, 4, 3, 1, 2, 2.0 / 3.0)]
    _check(world, cases, 30031 + world, 2)
