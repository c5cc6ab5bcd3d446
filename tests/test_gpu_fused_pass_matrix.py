"""Every whole-level form of the fused streaming passes on the B200, pass by pass, against the oracle's operator sequence.

Each case runs ONE pass through pmg_test_fused_pass on padded arrays built here -- Pass A (smoothing only, with the
restriction, from x == 0 with and without the xb store, prolong-in), Pass B (reading xb with and without the norm
partials, rebuilding xb for nu1 = 1..4) and the cross-cycle pass (every shape, stored and generated f) -- at the
B200's own strip / chunk geometry (148 SMs), and checks:
  * every array the pass writes is bit-identical to the oracle (float64 bits, so -0.0 != +0.0);
  * every padding element of every array is still all-zero bits, and the inputs keep their bits;
  * an array the pass must not read is filled with NaN (the iterate of the x == 0 forms, xb of the rebuilding Pass B,
    f of the generated-f cross pass), every output's domain starts as NaN, and unused norm partials too;
  * f and the iterate hold -0.0 and +-1e100 entries, level-0 forms a non-zero Dirichlet ring;
  * norm partials, summed exactly (math.fsum), are within 1e-14 of the exactly rounded sum of the oracle residual's
    squares.
The second half runs whole cycles with the streaming passes down to level 65 against orc.cycle, and the operator-level
entry points (pmg_restrict_to_level, pmg_norm2, pmg_diff_norm2, pmg_jacobi, pmg_release_scratch) against the oracle.
"""
import ctypes
import math

import numpy as np
import pytest

import cpu_checkers as cc
import pmg_b200 as pmg
from test_gpu_slab_kernels import PADX, PADY, Padded

pytestmark = pytest.mark.gpu

SMOOTH, PASS_A, ZERO, ZERO_NO_XB, PROLONG_IN, PASS_B, REBUILD, CROSS = range(8)
FORM_NAME = ["smooth", "passA", "zero", "zero_noxb", "prolong_in", "passB", "rebuild", "cross"]
OMEGAS = [1.0, 2.0 / 3.0, 0.8, 1.2]
SIZES = [65, 129, 513, 1025]
REF, FULL = pmg.PROLONG_REFERENCE, pmg.PROLONG_FULL
NORM_RTOL = 1e-14


class TestPass(ctypes.Structure):
    __test__ = False
    _fields_ = [("form", ctypes.c_int), ("x", ctypes.c_void_p), ("xb", ctypes.c_void_p), ("f", ctypes.c_void_p),
                ("n", ctypes.c_int), ("pitch", ctypes.c_int), ("h", ctypes.c_double), ("coarse_x", ctypes.c_void_p),
                ("coarse_f", ctypes.c_void_p), ("pitch_c", ctypes.c_int), ("nu", ctypes.c_int), ("nu_pre", ctypes.c_int),
                ("omega", ctypes.c_double), ("prolong_mode", ctypes.c_int), ("partials", ctypes.c_void_p),
                ("n_partials", ctypes.c_int), ("xb_out", ctypes.c_void_p), ("rhs_fx", ctypes.c_void_p),
                ("rhs_sy", ctypes.c_void_p), ("variant", ctypes.c_int), ("cross_shape", ctypes.c_int),
                ("min_chunk_rows", ctypes.c_int), ("deep_prefetch_below", ctypes.c_int)]


def _lib():
    L = pmg.lib()
    L.pmg_test_fused_pass.argtypes = [ctypes.POINTER(TestPass)]
    L.pmg_test_fused_max_partials.argtypes = [ctypes.c_int]
    L.pmg_restrict_to_level.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                        ctypes.c_int]
    L.pmg_diff_norm2.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_double),
                                 ctypes.POINTER(ctypes.c_double), ctypes.c_void_p]
    return L


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def special_field(rng, n, ring=True):
    """U(-1, 1) with -0.0, +0.0 and +-1e100 at an eighth of the points each (ring included unless ring=False)"""
    a = rng.uniform(-1.0, 1.0, (n, n))
    k = rng.integers(0, 8, (n, n))
    a[k == 0] = -0.0
    a[k == 1] = np.where(a[k == 1] < 0, -1e100, 1e100)
    a[k == 2] = 0.0
    if not ring:
        a[0, :] = a[-1, :] = a[:, 0] = a[:, -1] = 0.0
    return a


def padded(n, dom=None, fill=None):
    """padded level array (zero padding); domain = `dom`, or all `fill`"""
    p = Padded(n, n)
    if dom is not None:
        p.view(0, n)[:] = dom
    if fill is not None:
        p.view(0, n)[:] = fill
    return p.upload()


def all_nan(n):
    p = Padded(n, n)
    p.h[:] = np.nan
    return p.upload()


def check_out(p, want, what, lo=0, hi=None):
    """domain rows [lo, hi) bit-identical to `want`, every other element of the allocation all-zero bits"""
    n = p.n
    hi = n if hi is None else hi
    got = p.download()
    assert same_bits(got.view(lo, hi), want[lo:hi]), "%s differs from the oracle (%d of %d points)" % (
        what, int(np.count_nonzero(bits(got.view(lo, hi)) != bits(want[lo:hi]))), want[lo:hi].size)
    rest = got.h.copy()
    rest[PADY + lo:PADY + hi, PADX:PADX + n] = 0.0
    assert not bits(rest).any(), "%s: a padding element is not +0.0" % what


def check_unchanged(p, what):
    before = p.h.copy()
    assert same_bits(p.download().h, before), "%s was written" % what


def check_norm(partials, n_partials, r):
    got = partials.numpy()
    assert n_partials > 0 and np.isfinite(got[:n_partials]).all(), "a norm partial was not written"
    want = math.fsum((r * r).ravel())
    s = math.fsum(got[:n_partials])
    assert abs(s - want) <= NORM_RTOL * want, "norm partials: %.17g vs exactly rounded %.17g" % (s, want)


def run_pass(form, n, **kw):
    t = TestPass()
    t.form, t.n, t.h = form, n, 1.0 / (n - 1)
    t.variant, t.cross_shape, t.min_chunk_rows, t.deep_prefetch_below = -1, 0, 4, 0
    for k, v in kw.items():
        setattr(t, k, v)
    pmg.check(_lib().pmg_test_fused_pass(ctypes.byref(t)))
    return t


def pass_case(orc, form, n, nu, omega, prolong=REF, nu_pre=0, norm=False, with_e=True, seed=0, **tuning):
    """one Pass A / Pass B form on an n-level: build, run, compare"""
    rng = np.random.default_rng(1000 * n + 100 * form + 10 * nu + nu_pre + seed)
    h, nc = 1.0 / (n - 1), (n - 1) // 2 + 1
    f = special_field(rng, n)
    x = special_field(rng, n)  # level-0 style iterate: non-zero Dirichlet ring
    e = special_field(rng, nc, ring=False)
    pf, pe = padded(n, f), padded(nc, e)
    common = dict(f=pf.ptr(), pitch=pf.pitch, nu=nu, nu_pre=nu_pre, omega=omega, prolong_mode=prolong, pitch_c=pe.pitch,
                  **tuning)
    untouched = [(pf, "f"), (pe, "coarse x")]
    if form in (SMOOTH, PASS_A, ZERO, ZERO_NO_XB, PROLONG_IN):
        if form in (SMOOTH, PASS_A):
            want_xb = x.copy()
        else:
            want_xb = np.zeros((n, n))
            if form == PROLONG_IN:
                orc.prolong_add(want_xb, e, prolong)
        orc.jacobi(want_xb, f, h, omega=omega, num_iter=nu - 1)
        px = padded(n, x) if form in (SMOOTH, PASS_A) else all_nan(n)  # x == 0 forms: the iterate is not read
        pxb = all_nan(n) if form == ZERO_NO_XB else padded(n, fill=np.nan)
        pcf = padded(nc)
        pcf.view(1, nc - 1)[:, 1:nc - 1] = np.nan  # the ring of the coarse f is not written: zero, as in the solver
        pcf.upload()
        run_pass(form, n, x=px.ptr(), xb=pxb.ptr(), coarse_x=pe.ptr(), coarse_f=pcf.ptr(), **common)
        untouched.append((px, "the iterate"))
        if form == ZERO_NO_XB:
            untouched.append((pxb, "xb (not stored)"))
        else:
            check_out(pxb, want_xb, "xb")
        if form != SMOOTH:
            check_out(pcf, orc.restrict_fw(orc.residual(want_xb, f, h)), "coarse f")
        else:
            check_unchanged(pcf, "coarse f (smoothing only)")
    else:
        if form == REBUILD:
            xb = np.zeros((n, n))
            orc.jacobi(xb, f, h, omega=omega, num_iter=nu_pre - 1)
            pxb = all_nan(n)  # rebuilt from f, not read
        else:
            xb = x
            pxb = padded(n, xb)
        want = xb.copy()
        if with_e:
            orc.prolong_add(want, e, prolong)
        orc.jacobi(want, f, h, omega=omega, num_iter=nu - 1)
        px = padded(n, fill=np.nan)
        maxp = _lib().pmg_test_fused_max_partials(n)
        partials = pmg.DeviceArray.from_numpy(np.full(maxp, np.nan)) if norm else None
        t = run_pass(form, n, x=px.ptr(), xb=pxb.ptr(), coarse_x=pe.ptr() if with_e else None,
                     partials=partials.ptr if norm else None, **common)
        untouched.append((pxb, "xb"))
        check_out(px, want, "x")
        if norm:
            assert t.n_partials <= maxp
            check_norm(partials, t.n_partials, orc.residual(want, f, h))
        else:
            assert t.n_partials == 0
    for p, what in untouched:
        check_unchanged(p, what)


# ---- Pass A: every form, nu1 = 1..4, every omega; the sizes rotate so that every form meets every size ----
PASS_A_CASES = [(form, nu, w, SIZES[(nu + i) % 4]) for form in (SMOOTH, PASS_A, ZERO, ZERO_NO_XB) for nu in (1, 2, 3, 4)
                for i, w in enumerate(OMEGAS)]
PASS_A_CASES += [(PASS_A, 2, 2.0 / 3.0, 4097), (ZERO, 4, 0.8, 2049), (ZERO_NO_XB, 2, 1.2, 4097), (SMOOTH, 3, 1.0, 2049)]


@pytest.mark.parametrize("form,nu,omega,n", PASS_A_CASES,
                         ids=["%s-nu%d-w%.3g-n%d" % (FORM_NAME[c[0]], c[1], c[2], c[3]) for c in PASS_A_CASES])
def test_pass_a(orc, form, nu, omega, n):
    pass_case(orc, form, n, nu, omega)


PROLONG_IN_CASES = [(w, p, SIZES[(i + p) % 4]) for i, w in enumerate(OMEGAS) for p in (REF, FULL)] + [(2.0 / 3.0, REF, 2049)]


@pytest.mark.parametrize("omega,prolong,n", PROLONG_IN_CASES)
def test_pass_a_prolong_in(orc, omega, prolong, n):
    pass_case(orc, PROLONG_IN, n, 2, omega, prolong)


# ---- Pass B reading xb: nu2 = 1..4, with and without the norm partials, both prolongations, every omega ----
PASS_B_CASES = [(nu, norm, p, OMEGAS[(nu + p + norm) % 4], SIZES[(nu + 2 * p + norm) % 4]) for nu in (1, 2, 3, 4)
                for norm in (False, True) for p in (REF, FULL)]
PASS_B_CASES += [(2, True, REF, 2.0 / 3.0, 4097), (3, False, FULL, 1.2, 2049), (4, True, FULL, 0.8, 2049)]


@pytest.mark.parametrize("nu,norm,prolong,omega,n", PASS_B_CASES)
def test_pass_b(orc, nu, norm, prolong, omega, n):
    pass_case(orc, PASS_B, n, nu, omega, prolong, norm=norm)


@pytest.mark.parametrize("nu,omega,n", [(1, 1.0, 129), (2, 2.0 / 3.0, 1025), (3, 1.2, 513), (4, 0.8, 65)])
def test_pass_b_smoothing_only_with_norm(orc, nu, omega, n):
    """Pass B without a coarse correction (PROLONG = false): x = S^nu(xb) and its residual norm"""
    pass_case(orc, PASS_B, n, nu, omega, norm=True, with_e=False)


# ---- Pass B rebuilding xb = S^nu1(0; f): every (nu1, nu2) in {1..4}^2 and every omega ----
REBUILD_CASES = [(nu1, nu2, w, SIZES[(nu1 + nu2 + i) % 4], (nu1 + i) % 2) for nu1 in (1, 2, 3, 4) for nu2 in (1, 2, 3, 4)
                 for i, w in enumerate(OMEGAS)]
REBUILD_CASES += [(2, 2, 2.0 / 3.0, 4097, REF), (4, 4, 1.2, 2049, FULL), (3, 3, 0.8, 2049, REF)]


@pytest.mark.parametrize("nu1,nu2,omega,n,prolong", REBUILD_CASES)
def test_pass_b_rebuild(orc, nu1, nu2, omega, n, prolong):
    pass_case(orc, REBUILD, n, nu2, omega, prolong, nu_pre=nu1)


# ---- nu = 2: every tuning variant and the deep-prefetch path, for each form the variants serve ----
V2_FORMS = [(PASS_A, False), (ZERO, False), (ZERO_NO_XB, False), (PASS_B, False), (PASS_B, True)]


@pytest.mark.parametrize("variant", range(5))
@pytest.mark.parametrize("form,norm", V2_FORMS, ids=["passA", "zero", "zero_noxb", "passB", "passB_norm"])
def test_nu2_tuning_variants(orc, variant, form, norm):
    assert pmg.num_fused_variants() == 5
    n = (513, 1025, 2049)[variant % 3]
    pass_case(orc, form, n, 2, OMEGAS[variant % 4], FULL if variant % 2 else REF, norm=norm, variant=variant)


@pytest.mark.parametrize("form,norm", V2_FORMS, ids=["passA", "zero", "zero_noxb", "passB", "passB_norm"])
@pytest.mark.parametrize("n", [65, 513])
def test_nu2_deep_prefetch(orc, form, norm, n):
    pass_case(orc, form, n, 2, 2.0 / 3.0, norm=norm, deep_prefetch_below=n)


# ---- chunking: the default 4 rows and a minimum that forces a few tall chunks (the last one partial) ----
CHUNK_CASES = [(PASS_A, 3, 0, False), (ZERO, 1, 0, False), (ZERO_NO_XB, 2, 0, False), (PASS_B, 4, 0, True),
               (PASS_B, 2, 0, True), (REBUILD, 2, 3, False), (REBUILD, 4, 4, False)]


@pytest.mark.parametrize("min_rows", [4, 200])
@pytest.mark.parametrize("form,nu,nu_pre,norm", CHUNK_CASES)
def test_chunk_rows(orc, form, nu, nu_pre, norm, min_rows):
    pass_case(orc, form, 1025, nu, 1.2, FULL, nu_pre=nu_pre, norm=norm, min_chunk_rows=min_rows)


# ---- cross-cycle pass ----
def sine_tables(n):
    """the separable analytic right-hand side pmg_set_rhs_sine feeds the pass: f = fx[x] * sy[y], no sign bits"""
    sn = np.sin(np.pi * np.arange(n) / (n - 1))
    sn[0] = 0.0
    assert not np.signbit(sn).any()
    return 2.0 * np.pi ** 2 * sn, sn


def cross_case(orc, n, shape, gen_f, omega, prolong, store_xk, min_rows=4, seed=0):
    rng = np.random.default_rng(7 * n + shape + 100 * gen_f + seed)
    h, nc = 1.0 / (n - 1), (n - 1) // 2 + 1
    xb = special_field(rng, n)
    e = special_field(rng, nc, ring=False)
    if gen_f:
        fxv, syv = sine_tables(n)
        f = fxv[None, :] * syv[:, None]
    else:
        f = special_field(rng, n)
    xk = xb.copy()
    orc.prolong_add(xk, e, prolong)
    orc.jacobi(xk, f, h, omega=omega, num_iter=1)
    xb2 = xk.copy()
    orc.jacobi(xb2, f, h, omega=omega, num_iter=1)
    cf = orc.restrict_fw(orc.residual(xb2, f, h))

    pxb, pe = padded(n, xb), padded(nc, e)
    # the default shape forms f from the tables and must not read it; the others read it
    pf = all_nan(n) if (gen_f and shape in (0, 2)) else padded(n, f)
    pxk, pout = padded(n, fill=np.nan), padded(n, fill=np.nan)
    pcf = padded(nc)
    pcf.view(1, nc - 1)[:, 1:nc - 1] = np.nan
    pcf.upload()
    tabs = {}
    if gen_f:
        fx = np.zeros(pxb.pitch)
        fx[PADX:PADX + n] = fxv
        sy = np.zeros(n + 2 * PADY)
        sy[PADY:PADY + n] = syv
        tabs = dict(fx=pmg.DeviceArray.from_numpy(fx), sy=pmg.DeviceArray.from_numpy(sy))
    maxp = _lib().pmg_test_fused_max_partials(n)
    partials = pmg.DeviceArray.from_numpy(np.full(maxp, np.nan))
    t = run_pass(CROSS, n, x=pxk.ptr() if store_xk else None, xb=pxb.ptr(), f=pf.ptr(), pitch=pxb.pitch,
                 coarse_x=pe.ptr(), coarse_f=pcf.ptr(), pitch_c=pe.pitch, nu=2, nu_pre=2, omega=omega,
                 prolong_mode=prolong, partials=partials.ptr, xb_out=pout.ptr(),
                 rhs_fx=tabs["fx"].ptr + 8 * PADX if gen_f else None, rhs_sy=tabs["sy"].ptr + 8 * PADY if gen_f else None,
                 cross_shape=shape, min_chunk_rows=min_rows)
    assert t.n_partials <= maxp
    check_out(pout, xb2, "xb_out")
    check_out(pcf, cf, "coarse f")
    if store_xk:
        check_out(pxk, xk, "x_k")
    else:
        check_unchanged(pxk, "x_k (not stored)")
    check_norm(partials, t.n_partials, orc.residual(xk, f, h))
    for p, what in ((pxb, "xb"), (pf, "f"), (pe, "coarse x")):
        check_unchanged(p, what)


CROSS_SHAPES = [2, 3, 4, 5, 6, 7]
CROSS_CASES = [(shape, gen_f, SIZES[(shape + gen_f) % 4] if shape != 2 else (1025, 2049)[gen_f]) for shape in CROSS_SHAPES
               for gen_f in (False, True)]


@pytest.mark.parametrize("shape,gen_f,n", CROSS_CASES)
def test_cross_pass_shapes(orc, shape, gen_f, n):
    cross_case(orc, n, shape, gen_f, OMEGAS[shape % 4], FULL if shape % 2 else REF, store_xk=bool(shape % 2))


@pytest.mark.parametrize("omega", OMEGAS)
@pytest.mark.parametrize("prolong", [REF, FULL])
def test_cross_pass_default_shape(orc, omega, prolong):
    cross_case(orc, 513, 0, True, omega, prolong, store_xk=False)
    cross_case(orc, 129, 0, False, omega, prolong, store_xk=True)


@pytest.mark.parametrize("n,shape,gen_f", [(4097, 2, True), (2049, 4, False), (4097, 7, False)])
def test_cross_pass_large(orc, n, shape, gen_f):
    cross_case(orc, n, shape, gen_f, 2.0 / 3.0, REF, store_xk=False)


@pytest.mark.parametrize("shape", [2, 4])
def test_cross_pass_tall_chunks(orc, shape):
    cross_case(orc, 1025, shape, False, 1.2, FULL, store_xk=True, min_rows=200)


def test_unsupported_forms_fail_loudly():
    """A form no launcher serves launches nothing and reports it (fused_take_bad_nu) instead of skipping the pass"""
    n = 65
    px, pf = padded(n, fill=0.0), padded(n, fill=0.0)
    pe = padded(33)
    base = dict(x=px.ptr(), xb=px.ptr(), f=pf.ptr(), pitch=px.pitch, coarse_x=pe.ptr(), coarse_f=pe.ptr(), pitch_c=pe.pitch,
                omega=1.0)
    bad = [dict(form=PASS_A, nu=5), dict(form=ZERO, nu=0), dict(form=PASS_B, nu=0),
           dict(form=REBUILD, nu=2, nu_pre=5), dict(form=PROLONG_IN, nu=3), dict(form=CROSS, nu=3, nu_pre=2)]
    for kw in bad:
        k = dict(base, **kw)
        form = k.pop("form")
        with pytest.raises(pmg.PmgError) as ei:
            run_pass(form, n, **k)
        assert ei.value.status == 6, kw  # PMG_ERR_UNSUPPORTED
    # REBUILD with the norm: the rebuilding pass has no norm flavour
    partials = pmg.DeviceArray.from_numpy(np.zeros(_lib().pmg_test_fused_max_partials(n)))
    with pytest.raises(pmg.PmgError):
        run_pass(REBUILD, n, **dict(base, nu=2, nu_pre=2, partials=partials.ptr))
    with pytest.raises(pmg.PmgError) as ei:  # a rebuilding Pass B needs the sweep count of the xb it rebuilds
        run_pass(REBUILD, n, **dict(base, nu=2, nu_pre=0))
    assert ei.value.status == 1  # PMG_ERR_INVALID
    # the next good pass is not blamed for the refused ones
    run_pass(PASS_A, n, **dict(base, xb=padded(n).ptr(), nu=2))


# ---------------------------------------------------------------------------------------------------
# whole cycles: the streaming passes on every level down to 65 (no cluster kernel), against orc.cycle
# ---------------------------------------------------------------------------------------------------
def f_with_negative_zeros(n, seed):
    f = cc.random_rhs(n, seed=seed)
    rng = np.random.default_rng(seed + 1)
    k = rng.integers(0, 8, (n - 2, n - 2))
    f[1:-1, 1:-1][k == 0] = -0.0
    return f


@pytest.mark.parametrize("rebuild", [0, 1])
@pytest.mark.parametrize("omega", [1.0, 1.2])
@pytest.mark.parametrize("nu", [(1, 1), (3, 3), (4, 4), (1, 4), (4, 1)], ids=lambda nu: "nu%d%d" % nu)
@pytest.mark.parametrize("kind", [pmg.V, pmg.W], ids=["V", "W"])
def test_cycles_on_streaming_levels_match_oracle(orc, kind, nu, omega, rebuild):
    n = 513
    gamma = 2 if kind == pmg.W else 1
    f = f_with_negative_zeros(n, 500 + nu[0] * 10 + nu[1])
    phi0 = np.random.default_rng(77).uniform(-1, 1, (n, n))
    want = phi0.copy()
    L = pmg.lib()
    pmg.set_cluster_top(0)
    L.pmg_fused_set_rebuild_xb(ctypes.c_int(rebuild))
    try:
        with pmg.Solver(n, omega=omega, gamma=gamma, nu1=nu[0], nu2=nu[1]) as s:
            assert s.cluster_top == 0
            s.set_rhs(f)
            s.set_guess(phi0)
            for _ in range(2):
                orc.cycle(want, f, kind=cc.W if kind == pmg.W else cc.V, omega=omega, eps=0.0, alpha=gamma,
                          v1=nu[0] - 1, v2=nu[1] - 1)
                rn = s.cycle(kind)
                assert same_bits(s.get_solution(), want)
                r = orc.norm(orc.residual(want, f, 1.0 / (n - 1)))
                assert abs(rn - r) <= 1e-10 * r
    finally:
        L.pmg_fused_set_rebuild_xb(ctypes.c_int(-1))
        pmg.set_cluster_top(-1)


def test_large_solve_nu33_matches_operator_engine():
    """N = 8193, V(3,3): the fused engine with the xb rebuild chosen by level size (levels above the L2 size rebuild)
    against the one-kernel-per-operator engine"""
    n = 8193
    out = {}
    for engine in (pmg.ENGINE_FUSED, pmg.ENGINE_OPERATOR):
        with pmg.Solver(n, omega=2.0 / 3.0, nu1=3, nu2=3, engine=engine) as s:
            s.set_rhs_sine()
            s.zero_guess()
            k, hist = s.solve(pmg.V, 1e-8, 60)
            out[engine] = (k, hist, s.get_solution())
    (k0, h0, x0), (k1, h1, x1) = out[pmg.ENGINE_FUSED], out[pmg.ENGINE_OPERATOR]
    assert k0 == k1 and k0 < 60
    assert np.max(np.abs(h0 - h1) / np.abs(h1)) <= 1e-10
    assert same_bits(x0, x1)


# ---------------------------------------------------------------------------------------------------
# operator-level entry points
# ---------------------------------------------------------------------------------------------------
def _restrict_to_level(s, fine, n_out, out):
    pi, mi = (fine.ctypes.data, pmg.MEM_HOST) if isinstance(fine, np.ndarray) else (fine.ptr, pmg.MEM_DEVICE)
    po, mo = (out.ctypes.data, pmg.MEM_HOST) if isinstance(out, np.ndarray) else (out.ptr, pmg.MEM_DEVICE)
    return _lib().pmg_restrict_to_level(s._h, pi, mi, n_out, po, mo)


@pytest.mark.parametrize("n", [257, 1025])
def test_restrict_to_level(orc, n):
    rng = np.random.default_rng(n)
    fine = special_field(rng, n)
    f = cc.random_rhs(n, seed=n + 1)
    phi0 = rng.uniform(-1, 1, (n, n))
    levels, m = [n], n
    while m > 5:  # default n_coarse = 5
        m = (m - 1) // 2 + 1
        levels.append(m)
    with pmg.Solver(n, omega=2.0 / 3.0) as s:
        s.set_rhs(f)
        s.set_guess(phi0)
        want = fine.copy()
        dfine = pmg.DeviceArray.from_numpy(fine)
        for i, m in enumerate(levels):
            if m != n:
                want = orc.restrict_fw(want)
            for src_dev in (False, True):
                for dst_dev in (False, True):
                    out = pmg.DeviceArray((m, m)) if dst_dev else np.full((m, m), np.nan)
                    pmg.check(_restrict_to_level(s, dfine if src_dev else fine, m, out))
                    got = out.numpy() if dst_dev else out
                    assert same_bits(got, want), (m, src_dev, dst_dev)
                    if m != n:  # the restriction leaves the ring at +0.0
                        assert not bits(got[[0, -1], :]).any() and not bits(got[:, [0, -1]]).any()
        for bad in (3, 2 * n - 1, n + 2, 100):
            out = np.zeros((3, 3))
            assert _restrict_to_level(s, fine, bad, out) == 1  # PMG_ERR_INVALID
        assert same_bits(s.get_solution(), phi0), "pmg_restrict_to_level changed the iterate"
        k, hist = s.solve(pmg.V, 1e-8, 40)
        x = s.get_solution()
    with pmg.Solver(n, omega=2.0 / 3.0) as s:
        s.set_rhs(f)
        s.set_guess(phi0)
        k2, hist2 = s.solve(pmg.V, 1e-8, 40)
        assert k == k2 and same_bits(hist, hist2) and same_bits(s.get_solution(), x)


RED = 148 * 8 * 256  # reduction partials x block size of the operator-level reductions


@pytest.mark.parametrize("length", [0, 1, 31, 32, 33, 1000003, 4 * RED + 17])
def test_norm2_and_diff_norm2(length):
    rng = np.random.default_rng(length)
    a = rng.standard_normal(length) * np.exp(rng.uniform(-20, 20, length))
    b = rng.standard_normal(length)
    if length:
        b[rng.integers(0, length, max(1, length // 8))] = -0.0
    da, db = pmg.DeviceArray.from_numpy(a), pmg.DeviceArray.from_numpy(b)

    def close(got, want):
        assert (got == 0.0) if want == 0.0 else abs(got - want) <= 1e-14 * want, (got, want)

    close(pmg.norm2(da), math.fsum((a * a).tolist()))
    d2, b2 = ctypes.c_double(-1.0), ctypes.c_double(-1.0)
    pmg.check(_lib().pmg_diff_norm2(da.ptr, db.ptr, length, ctypes.byref(d2), ctypes.byref(b2), None))
    d = a - b
    close(d2.value, math.fsum((d * d).tolist()))
    close(b2.value, math.fsum((b * b).tolist()))


def _jacobi_case(orc, width, height, sweeps, omega, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, (height, width))
    f = rng.uniform(-1, 1, (height, width))
    k = rng.integers(0, 8, (height, width))
    f[k == 0] = -0.0
    f[k == 1] = 1e100
    x[k == 2] = -0.0
    h = 1.0 / (width - 1)
    want = x.copy()
    orc.jacobi(want, f, h, omega=omega, num_iter=sweeps - 1)
    dx, df = pmg.DeviceArray.from_numpy(x), pmg.DeviceArray.from_numpy(f)
    pmg.jacobi(dx, df, h, omega=omega, sweeps=sweeps)
    assert same_bits(dx.numpy(), want), (width, height, sweeps, omega)


JACOBI_SHAPES = [(256, 256), (257, 257), (258, 258), (300, 300), (333, 333), (257, 300), (300, 257)]


@pytest.mark.parametrize("omega", [1.0, 2.0 / 3.0])
@pytest.mark.parametrize("shape", JACOBI_SHAPES, ids=["%dx%d" % s for s in JACOBI_SHAPES])
def test_jacobi_blocked_threshold(orc, shape, omega):
    """Square fields >= 257 wide with >= 8 sweeps take the blocked streaming smoother (4 sweeps per pass + the rest),
    everything else the sweep-by-sweep kernel: both sides of both thresholds, widths that are not 2^k + 1"""
    for sweeps in (7, 8, 9, 10, 11, 12, 17):
        _jacobi_case(orc, shape[1], shape[0], sweeps, omega, shape[0] * 100 + sweeps)


def test_release_scratch_between_calls(orc):
    for n in (300, 257, 300):
        _jacobi_case(orc, n, n, 9, 2.0 / 3.0, n)
        pmg.check(pmg.lib().pmg_release_scratch())
        _jacobi_case(orc, n, n, 9, 2.0 / 3.0, n)
    v = np.random.default_rng(5).standard_normal(1000003)
    dv = pmg.DeviceArray.from_numpy(v)
    first = pmg.norm2(dv)
    pmg.check(pmg.lib().pmg_release_scratch())
    assert pmg.norm2(dv) == first
    pmg.check(pmg.lib().pmg_release_scratch())
    pmg.check(pmg.lib().pmg_release_scratch())  # nothing held: still fine
    r = pmg.DeviceArray.from_numpy(np.zeros((257, 257)))
    x, f = np.random.default_rng(6).standard_normal((2, 257, 257))
    n2 = pmg.residual(r, pmg.DeviceArray.from_numpy(x), pmg.DeviceArray.from_numpy(f), 1.0 / 256, want_norm2=True)
    want = orc.residual(x, f, 1.0 / 256)
    assert same_bits(r.numpy(), want)
    assert abs(n2 - math.fsum((want * want).ravel())) <= 1e-14 * n2
