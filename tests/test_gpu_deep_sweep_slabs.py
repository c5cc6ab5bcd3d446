"""The deep-sweep slab schedule's passes on ONE GPU (3 or 4 pre/post-smoothing sweeps on row slabs).

Row slabs of 2-4 "ranks" live side by side in device memory, as in tests/test_gpu_slab_kernels.py:
  * Pass A with the deep spans [-pass_a_depth, ny + pass_a_depth), streaming the neighbours' halo rows in place;
  * Pass B with the coarse up-exchange prologue: the coarse iterate holds its owned rows and the pass_b_ext rows the
    child's Pass B finished, NaN beyond; the prologue waits for the (pre-set) flags, copies the next rows from the
    neighbours' coarse arrays and publishes its own epoch.
Every output is compared BIT FOR BIT with the oracle's operator sequence on the whole level, padding must stay all-zero
bits, and the time-out of the new wait is checked once against a neighbour that never publishes.
"""
import ctypes

import numpy as np
import pytest

import pmg_b200 as pmg
from test_dist_gloo_deep_sweeps import PAIRS, pass_a_depth, pass_b_ext, up_exchange_rows
from test_gpu_slab_kernels import EPOCH, PADX, PADY, DevInts, Padded, TestSlab, _lib, partition

pytestmark = pytest.mark.gpu

OMEGA = 2.0 / 3.0


def _lib_up():
    L = _lib()
    L.pmg_test_fused_up_exchange.argtypes = [ctypes.POINTER(TestSlab), ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_double, ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int),
                                             ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    L.pmg_set_p2p_timeout_ms.restype = None
    L.pmg_set_p2p_timeout_ms.argtypes = [ctypes.c_double]
    return L


def _problem(orc, n, nu1, nu2, prolong, first_visit, level0, seed):
    nc, h = (n - 1) // 2 + 1, 1.0 / (n - 1)
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, (n, n))
    if not level0:
        x[0, :] = x[-1, :] = x[:, 0] = x[:, -1] = 0.0
    f = np.zeros((n, n))
    f[1:-1, 1:-1] = rng.uniform(-1, 1, (n - 2, n - 2))
    e = np.zeros((nc, nc))
    e[1:-1, 1:-1] = rng.uniform(-1, 1, (nc - 2, nc - 2))
    xb = np.zeros_like(x) if first_visit else x.copy()
    orc.jacobi(xb, f, h, omega=OMEGA, num_iter=nu1 - 1)
    cf = orc.restrict_fw(orc.residual(xb, f, h))
    xn = xb.copy()
    orc.prolong_add(xn, e, prolong)
    orc.jacobi(xn, f, h, omega=OMEGA, num_iter=nu2 - 1)
    return dict(x=x, f=f, e=e, xb=xb, cf=cf, xn=xn, norm2=orc.norm(orc.residual(xn, f, h)) ** 2, nc=nc, h=h)


def _ranks(P, n, ranks, nu1, nu2, level, first_visit):
    """per-rank padded arrays; the coarse iterate holds what the child finished: owned rows + pass_b_ext(level + 1)"""
    nc, e_child = P["nc"], pass_b_ext(nu1, nu2, level + 1)
    R = []
    for r in range(ranks):
        y0, y1 = partition(n, ranks, r)
        c0, c1 = y0 // 2, (nc if y1 == n else y1 // 2)
        ny, nyc = y1 - y0, c1 - c0
        up, dn = r > 0, r < ranks - 1
        K = dict(y0=y0, ny=ny, c0=c0, nyc=nyc, up=up, dn=dn)
        px, pxb, pf, pcf, pe, pxn = Padded(n, ny), Padded(n, ny), Padded(n, ny), Padded(nc, nyc), Padded(nc, nyc), Padded(n, ny)
        px.view(0, ny)[:] = np.nan if first_visit else P["x"][y0:y1]
        pf.view(0, ny)[:] = P["f"][y0:y1]
        for arr in (px, pf) if level > 0 else (px,):
            if up:
                arr.view(-PADY, 0)[:] = np.nan
            if dn:
                arr.view(ny, ny + PADY)[:] = np.nan
        if level == 0:  # the finest level's f halo is local
            a, b = max(0, y0 - PADY), min(n, y1 + PADY)
            pf.view(a - y0, b - y0)[:] = P["f"][a:b]
        pe.view(0, nyc)[:] = P["e"][c0:c1]
        if up:
            pe.view(-PADY, 0)[:] = np.nan
            pe.view(-e_child, 0)[:] = P["e"][c0 - e_child:c0]
        if dn:
            pe.view(nyc, nyc + PADY)[:] = np.nan
            pe.view(nyc, nyc + e_child)[:] = P["e"][c1:c1 + e_child]
        for p in (px, pxb, pf, pcf, pe, pxn):
            p.upload()
        K.update(x=px, xb=pxb, f=pf, cf=pcf, e=pe, xn=pxn, inbox=DevInts([EPOCH, EPOCH]), outbox=DevInts([0, 0]),
                 up_in=DevInts([EPOCH, EPOCH]), up_out=DevInts([0, 0]), err=DevInts([0]), abort=DevInts([0]))
        R.append(K)
    return R


def _pass_b_slab(R, r, n, h):
    K = R[r]
    t = TestSlab()
    t.x, t.xb, t.f = K["xn"].ptr(), K["xb"].ptr(), K["f"].ptr()
    t.n, t.pitch, t.h, t.ny, t.yoff = n, K["x"].pitch, h, K["ny"], K["y0"]
    t.x_up = R[r - 1]["e"].ptr(R[r - 1]["nyc"]) if K["up"] else None
    t.x_dn = R[r + 1]["e"].ptr() if K["dn"] else None
    t.flag_up = K["up_in"].at(0) if K["up"] else None
    t.flag_dn = K["up_in"].at(1) if K["dn"] else None
    t.pub_up = K["up_out"].at(0) if K["up"] else None
    t.pub_dn = K["up_out"].at(1) if K["dn"] else None
    t.epoch, t.err = EPOCH, K["err"].ptr
    return t


CASES = [(nu1, nu2, n, ranks, level, first, split, prolong)
         for i, (nu1, nu2) in enumerate(PAIRS) if max(nu1, nu2) >= 3
         for (n, ranks, level, first, split, prolong) in [
             ((257, 2, 0, False, False, pmg.PROLONG_REFERENCE), (513, 4, 1, True, True, pmg.PROLONG_FULL),
              (1025, 3, 1, False, False, pmg.PROLONG_REFERENCE), (4097, 2, 1, False, True, pmg.PROLONG_FULL))[i % 4],
             (257, 4, 1, i % 2 == 0, False, pmg.PROLONG_REFERENCE)]]


@pytest.mark.parametrize("nu1,nu2,n,ranks,level,first_visit,split,prolong", CASES)
def test_deep_sweep_passes_match_oracle_on_one_gpu(orc, nu1, nu2, n, ranks, level, first_visit, split, prolong):
    L = _lib_up()
    P = _problem(orc, n, nu1, nu2, prolong, first_visit, level == 0, 500 + n + 7 * nu1 + nu2)
    R = _ranks(P, n, ranks, nu1, nu2, level, first_visit)
    da = pass_a_depth(nu1, nu2)
    # ---- Pass A on the deep spans ----
    for r, K in enumerate(R):
        up, dn, ny = K["up"], K["dn"], K["ny"]
        t = TestSlab()
        t.x, t.xb, t.f = K["x"].ptr(), K["xb"].ptr(), K["f"].ptr()
        t.n, t.pitch, t.h, t.ny, t.yoff = n, K["x"].pitch, P["h"], ny, K["y0"]
        peers = dict(epoch=EPOCH, err=K["err"].ptr)
        if not first_visit:
            peers.update(x_up=R[r - 1]["x"].ptr(R[r - 1]["ny"]) if up else None, x_dn=R[r + 1]["x"].ptr() if dn else None,
                         x_keep=K["x"].ptr())
        if level > 0:
            peers.update(f_up=R[r - 1]["f"].ptr(R[r - 1]["ny"]) if up else None, f_dn=R[r + 1]["f"].ptr() if dn else None,
                         f_keep=K["f"].ptr())
        peers.update(flag_up=K["inbox"].at(0) if up else None, flag_dn=K["inbox"].at(1) if dn else None,
                     pub_up=K["outbox"].at(0) if up else None, pub_dn=K["outbox"].at(1) if dn else None)

        def launch(with_peers, lo, hi, publish=True):
            for k in ("x_up", "x_dn", "f_up", "f_dn", "f_keep", "x_keep", "flag_up", "flag_dn", "pub_up", "pub_dn", "err"):
                setattr(t, k, None)
            t.epoch = 0
            if with_peers:
                for k, v in peers.items():
                    if not (k.startswith("pub_") and not publish):
                        setattr(t, k, v)
            t.span_lo, t.span_hi = lo, hi
            pmg.check(L.pmg_test_fused_down(ctypes.byref(t), K["cf"].ptr(), K["cf"].pitch, nu1, OMEGA,
                                            1 if first_visit else 0, 0))

        if split:  # cycle_dist: boundary strips [-da, 8), [ny - 8, ny + da) with the peers, interior without
            if up:
                launch(True, -da, PADY)
            if dn:
                launch(True, ny - PADY, ny + da, publish=not up)
            launch(False, PADY if up else 0, ny - PADY if dn else ny)
        else:
            launch(True, -da if up else 0, ny + da if dn else ny)
        assert K["err"].get()[0] == 0
        a, b = (-da if up else 0), (ny + da if dn else ny)
        got = K["xb"].download()
        assert np.array_equal(got.view(a, b), P["xb"][K["y0"] + a:K["y0"] + b]), "rank %d: xb" % r
        outside = got.h.copy()
        outside[PADY + a:PADY + b, PADX:PADX + n] = 0.0
        assert not outside.any(), "rank %d: Pass A wrote xb outside [-%d, ny + %d)" % (r, da, da)
        gcf = K["cf"].download()
        assert np.array_equal(gcf.view(0, K["nyc"]), P["cf"][K["c0"]:K["c0"] + K["nyc"]]), "rank %d: coarse f" % r
        # Pass B may read xb only where Pass A finished it
        if up:
            got.view(-PADY, a)[:] = np.nan
        if dn:
            got.view(b, ny + PADY)[:] = np.nan
        K["xb"].h = got.h
        K["xb"].upload()
    # ---- Pass B with the up-exchange ----
    e_child, m = pass_b_ext(nu1, nu2, level + 1), up_exchange_rows(nu1, nu2, level)
    if m == 0:  # this pair needs no exchange on this level: the prologue still runs with one row (a superset)
        m = 1
    ext = pass_b_ext(nu1, nu2, level)
    norm = level == 0 and nu2 + 1 <= da
    maxp = L.pmg_test_fused_max_partials(n)
    total = 0.0
    for r, K in enumerate(R):
        up, dn, ny = K["up"], K["dn"], K["ny"]
        t = _pass_b_slab(R, r, n, P["h"])
        t.ext_lo, t.ext_hi = (ext if up else 0), (ext if dn else 0)
        partials = pmg.DeviceArray.from_numpy(np.zeros(maxp))
        np_out = ctypes.c_int()
        pmg.check(L.pmg_test_fused_up_exchange(ctypes.byref(t), K["e"].ptr(), K["e"].pitch, nu2, OMEGA, prolong,
                                               partials.ptr if norm else None, ctypes.byref(np_out), e_child, m,
                                               K["abort"].ptr))
        assert K["err"].get()[0] == 0 and K["abort"].get()[0] == 0
        out = K["up_out"].get()
        assert (not up or out[0] == EPOCH) and (not dn or out[1] == EPOCH), "epoch not published"
        a, b = -t.ext_lo, ny + t.ext_hi
        got = K["xn"].download()
        assert np.array_equal(got.view(a, b), P["xn"][K["y0"] + a:K["y0"] + b]), "rank %d: x after Pass B" % r
        outside = got.h.copy()
        outside[PADY + a:PADY + b, PADX:PADX + n] = 0.0
        assert not outside.any(), "rank %d: Pass B wrote x outside its rows" % r
        ge = K["e"].download()
        nyc, c0 = K["nyc"], K["c0"]
        # the owned and child-finished rows keep their values; the next m rows hold the neighbour's row where a warp read
        # it and are still NaN where none did (the prolongation reads one coarse row fewer above the slab than below);
        # the rows beyond are untouched
        fa, fb = (-e_child if up else 0), (nyc + e_child if dn else nyc)
        assert np.array_equal(ge.view(fa, fb), P["e"][c0 + fa:c0 + fb]), "rank %d: coarse rows changed" % r
        ea, eb = (-(e_child + m) if up else 0), (nyc + e_child + m if dn else nyc)
        for lo_, hi_ in ((ea, fa), (fb, eb)):
            g_, w_ = ge.view(lo_, hi_), P["e"][c0 + lo_:c0 + hi_]
            assert np.all((g_ == w_) | np.isnan(g_)), "rank %d: a copied coarse row differs from the neighbour's" % r
        for lo_, hi_ in (((-PADY, ea) if up else (0, 0)), ((eb, nyc + PADY) if dn else (0, 0))):
            assert np.isnan(ge.view(lo_, hi_)).all(), "rank %d: the prologue wrote beyond its rows" % r
        pad = ge.h.copy()
        pad[:, PADX:PADX + P["nc"]] = 0.0
        assert not pad.view(np.uint64).any(), "rank %d: the prologue wrote into the coarse padding columns" % r
        total += float(partials.numpy()[:np_out.value].sum())
    if norm and not first_visit:
        assert abs(total - P["norm2"]) <= 1e-12 * P["norm2"]


def test_up_exchange_wait_times_out_and_reports(orc):
    """A neighbour that never publishes its epoch: the prologue's wait gives up after the 50 ms limit, raises the error
    word and the solve's done flag, and the kernel returns normally -- the path pmg_solve turns into PMG_ERR_COMM"""
    import time
    L = _lib_up()
    n, ranks, nu1, nu2 = 257, 2, 3, 3
    P = _problem(orc, n, nu1, nu2, pmg.PROLONG_REFERENCE, False, False, 91)
    R = _ranks(P, n, ranks, nu1, nu2, 1, False)
    K = R[1]
    K["up_in"] = DevInts([EPOCH - 1, EPOCH - 1])  # the upper neighbour is one epoch behind
    t = _pass_b_slab(R, 1, n, P["h"])
    e_child = pass_b_ext(nu1, nu2, 2)
    L.pmg_set_p2p_timeout_ms(50.0)
    try:
        t0 = time.perf_counter()
        pmg.check(L.pmg_test_fused_up_exchange(ctypes.byref(t), K["e"].ptr(), K["e"].pitch, nu2, OMEGA,
                                               pmg.PROLONG_REFERENCE, None, None, e_child, 1, K["abort"].ptr))
        dt = time.perf_counter() - t0
    finally:
        L.pmg_set_p2p_timeout_ms(0.0)  # back to the default
    assert K["err"].get()[0] != 0, "the time-out did not raise the error word"
    assert K["abort"].get()[0] != 0, "the time-out did not raise the solve's done flag"
    assert 0.04 <= dt < 5.0, "waited %.3f s for a 50 ms limit" % dt
