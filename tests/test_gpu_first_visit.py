"""First visits of the coarse levels on the B200: a solve whose large first visits skip the xb store and rebuild xb in
Pass B (pmg_fused_set_rebuild_xb(1): every whole level) must give the same cycle count, the same residual history and
the same iterate, bit for bit, as the solve that stores xb on every level (0) and as the default (-1: by level size),
for V-, W- and F-cycles."""
import ctypes

import numpy as np
import pytest

import pmg_b200 as pmg

pytestmark = pytest.mark.gpu


def _solve(n, kind, mode, omega):
    pmg.lib().pmg_fused_set_rebuild_xb(ctypes.c_int(mode))
    try:
        with pmg.Solver(n, omega=omega) as s:
            s.set_rhs_sine()
            s.zero_guess()
            k, hist = s.solve(kind, 1e-8, 60)
            return k, hist, s.get_solution()
    finally:
        pmg.lib().pmg_fused_set_rebuild_xb(ctypes.c_int(-1))


@pytest.mark.parametrize("n,kind,omega", [(4097, pmg.V, 2.0 / 3.0), (4097, pmg.W, 1.0), (2049, pmg.F, 2.0 / 3.0),
                                          (8193, pmg.V, 0.8)])
def test_rebuilt_xb_matches_stored_xb(n, kind, omega):
    k0, h0, x0 = _solve(n, kind, 0, omega)
    k1, h1, x1 = _solve(n, kind, 1, omega)
    ka, ha, xa = _solve(n, kind, -1, omega)
    assert k0 == k1 == ka
    assert np.array_equal(h0, h1) and np.array_equal(h0, ha)
    assert np.array_equal(x0, x1) and np.array_equal(x0, xa)
