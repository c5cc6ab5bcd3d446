"""The cross-cycle pass with its right-hand side generated in the pass (one GPU, f written by pmg_set_rhs_sine): the pass
forms f = (2 pi^2 sin_x) sin_y from two small tables instead of reading it from HBM.

  * Against the classic two passes per cycle reading the stored f: same cycle count, bit-identical iterate, norms equal to
    the last bits (the tree sum runs over another strip geometry), a max_cycles cut-off included.
  * Switching the right-hand side on one handle (sine -> user f, user f -> sine, sine -> stage / commit): every result is
    bit-identical to a fresh handle given only the second right-hand side.  The captured cross-cycle graphs must follow
    the switch -- a graph captured after pmg_set_rhs_sine would otherwise keep generating the sine.
"""
import ctypes

import numpy as np
import pytest

import cpu_checkers as cc
import pmg_b200 as pmg

pytestmark = pytest.mark.gpu

OMEGA = 2.0 / 3.0


def _sine_solves(n, cross):
    pmg.set_cross_cycle(cross, 0)
    try:
        with pmg.Solver(n, omega=OMEGA) as s:
            assert s.cross_cycle == bool(cross)
            s.set_rhs_sine()
            s.zero_guess()
            k, hist = s.solve(pmg.V, rel_tol=1e-8, max_cycles=100)
            x = s.get_solution()
            s.zero_guess()
            k3, hist3 = s.solve(pmg.V, rel_tol=0.0, max_cycles=3)
            x3 = s.get_solution()
    finally:
        pmg.set_cross_cycle(-1, 0)
    return k, hist, x, k3, hist3, x3


@pytest.mark.parametrize("n", [257, 4097, 16385])
def test_generated_rhs_cross_pass_matches_two_passes(n):
    two = _sine_solves(n, 0)    # two passes per cycle on level 0, f read from HBM
    gen = _sine_solves(n, 2)    # the cross-cycle pass (forced where it would not fill the machine), f generated
    assert two[0] == gen[0] and two[3] == gen[3] == 3
    if n == 16385:
        assert gen[0] == 39
    assert np.array_equal(two[2], gen[2]), "iterate differs"
    assert np.array_equal(two[5], gen[5]), "iterate after 3 cycles differs"
    for a, b in ((two[1], gen[1]), (two[4], gen[4])):
        assert np.max(np.abs(a - b) / a) <= 1e-13


def _pinned(shape):
    nbytes = int(np.prod(shape)) * 8
    p = ctypes.c_void_p()
    pmg.check(pmg.lib().pmg_host_alloc_pinned(ctypes.byref(p), nbytes))
    buf = (ctypes.c_double * (nbytes // 8)).from_address(p.value)
    return np.frombuffer(buf, dtype=np.float64).reshape(shape), p


def _solve(s):
    s.zero_guess()
    k, hist = s.solve(pmg.V, rel_tol=1e-8, max_cycles=60)
    return k, hist, s.get_solution()


def _same(a, b, what):
    assert a[0] == b[0], (what, a[0], b[0])
    assert np.array_equal(a[1], b[1]), what
    assert np.array_equal(a[2], b[2]), what


def test_rhs_switch_on_one_handle_matches_fresh_handle():
    n = 4097  # the cross-cycle pass fills the machine here: pmg_solve uses it (and its graphs) by default
    pmg.set_cross_cycle(-1, 0)
    f = cc.random_rhs(n, seed=131)
    with pmg.Solver(n, omega=OMEGA) as s:
        assert s.cross_cycle
        s.set_rhs(f)
        fresh_user = _solve(s)
    with pmg.Solver(n, omega=OMEGA) as s:
        s.set_rhs_sine()
        fresh_sine = _solve(s)
    assert fresh_user[0] != fresh_sine[0] or not np.array_equal(fresh_user[2], fresh_sine[2])

    with pmg.Solver(n, omega=OMEGA) as s:  # sine -> user f
        s.set_rhs_sine()
        _same(_solve(s), fresh_sine, "sine on a fresh handle")
        s.set_rhs(f)
        _same(_solve(s), fresh_user, "set_rhs after set_rhs_sine")
    with pmg.Solver(n, omega=OMEGA) as s:  # user f -> sine
        s.set_rhs(f)
        _same(_solve(s), fresh_user, "user f on a fresh handle")
        s.set_rhs_sine()
        _same(_solve(s), fresh_sine, "set_rhs_sine after set_rhs")
    f_pin, p = _pinned((n, n))
    try:
        f_pin[:] = f
        with pmg.Solver(n, omega=OMEGA) as s:  # sine -> stage / commit
            s.set_rhs_sine()
            _solve(s)
            s.stage_rhs(f_pin)
            s.commit_rhs()
            _same(_solve(s), fresh_user, "stage_rhs / commit_rhs after set_rhs_sine")
    finally:
        pmg.lib().pmg_host_free_pinned(p)
