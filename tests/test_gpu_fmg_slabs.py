"""The fused residual-restriction of the FMG set-up (csrc/kernel_residual_restrict.cuh) on ONE GPU, through the test hook
pmg_test_residual_restrict: whole levels, and the row-slab windows of 2, 4 and 8 "ranks" side by side in one device buffer
with every x row more than 2 rows and every f row more than 1 row beyond the slab NaN (the depth cycle_fmg_dist relies on).
The coarse right-hand side is compared BIT FOR BIT with the oracle's residual followed by its restriction; every other
element of the coarse arrays (ring, other ranks' rows, padding) must stay all-zero bits and the inputs keep their bits.
This is the GPU twin of tests/cpp/test_residual_restrict_emu.cpp and gives the slab path hardware coverage on a one-GPU box,
where tests/test_gpu_dist_fmg.py has to skip."""
import ctypes

import numpy as np
import pytest

import cpu_checkers as cc
import pmg_b200 as pmg

pytestmark = pytest.mark.gpu

PADX, PADY = 16, 8


def _lib():
    L = pmg.lib()
    L.pmg_test_layout.restype = None
    L.pmg_test_layout.argtypes = [ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 3
    L.pmg_test_residual_restrict.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 7 + [ctypes.c_double]
    return L


def level_pitch(n):
    p, px, py = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib().pmg_test_layout(n, ctypes.byref(p), ctypes.byref(px), ctypes.byref(py))
    assert (px.value, py.value) == (PADX, PADY)
    return p.value


def partition(n, ranks, r):
    return pmg.partition_rows(n, ranks, r)


def make_case(n, seed):
    """x with a non-zero ring and zero patches, f with -0.0 / +-1e100 entries there; the oracle's R(f - A x)"""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, (n, n))
    f = rng.uniform(-1, 1, (n, n))
    yy, xx = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    patch = ((yy // 6) + (xx // 6)) % 5 == 0
    x[patch] = 0.0
    k = rng.integers(0, 97, (n, n))
    f[k == 0] = 1e100
    f[k == 1] = -1e100
    f[(k < 12) & patch] = -0.0
    orc = cc.load("orc")
    want = orc.restrict_fw(orc.residual(x, f, 1.0 / (n - 1)))
    return x, f, want


def windows(d, n, spans, depth):
    """the windows [y0 - PADY, y1 + PADY) of the dense field d stacked in one padded host array; rows more than `depth`
    beyond the owned rows (and outside the grid) NaN from end to end.  Returns (array, row offset of each window's row 0)"""
    pitch = level_pitch(n)
    heights = [y1 - y0 + 2 * PADY for y0, y1 in spans]
    a = np.full((sum(heights), pitch), np.nan)
    offs, o = [], 0
    for (y0, y1), hgt in zip(spans, heights):
        offs.append(o + PADY)
        for lr in range(-PADY, y1 - y0 + PADY):
            g = y0 + lr
            if y0 - depth <= g < y1 + depth and 0 <= g < n:
                a[o + PADY + lr] = 0.0
                a[o + PADY + lr, PADX:PADX + n] = d[g]
        o += hgt
    return a, offs


def run(n, ranks, seed):
    nc = (n - 1) // 2 + 1
    x, f, want = make_case(n, seed)
    fine = [partition(n, ranks, r) for r in range(ranks)]
    coarse = [partition(nc, ranks, r) for r in range(ranks)] if ranks > 1 else [(0, nc)]
    if ranks > 1:
        assert all(c0 * 2 == y0 for (y0, _), (c0, _) in zip(fine, coarse))
    depth_x, depth_f = (2, 1) if ranks > 1 else (0, 0)
    hx, ox = windows(x, n, fine, depth_x)
    hf, of = windows(f, n, fine, depth_f)
    pc, pf = level_pitch(nc), level_pitch(n)
    hc = np.zeros((sum(c1 - c0 + 2 * PADY for c0, c1 in coarse), pc))
    dx, df, dc = pmg.DeviceArray.from_numpy(hx), pmg.DeviceArray.from_numpy(hf), pmg.DeviceArray.from_numpy(hc)
    oc, o = [], 0
    for c0, c1 in coarse:
        oc.append(o + PADY)
        o += c1 - c0 + 2 * PADY
    for r in range(ranks):
        (c0, c1) = coarse[r]
        pmg.check(_lib().pmg_test_residual_restrict(dx.ptr + 8 * (ox[r] * pf + PADX), df.ptr + 8 * (of[r] * pf + PADX),
                                                    dc.ptr + 8 * (oc[r] * pc + PADX), n, nc, c1 - c0, c0, pf, pf, pc,
                                                    1.0 / (n - 1)))
    got = dc.numpy()
    assert dx.numpy().tobytes() == hx.tobytes() and df.numpy().tobytes() == hf.tobytes(), "an input was written"
    expect = np.zeros_like(hc)
    for r, (c0, c1) in enumerate(coarse):
        for lr in range(c1 - c0):
            g = c0 + lr
            if 1 <= g <= nc - 2:
                expect[oc[r] + lr, PADX + 1:PADX + nc - 1] = want[g, 1:nc - 1]
    bad = np.argwhere(got.view(np.uint64) != expect.view(np.uint64))
    assert bad.size == 0, "%d elements differ, first at %s: got %r want %r" % (
        len(bad), tuple(bad[0]), got[tuple(bad[0])], expect[tuple(bad[0])])


@pytest.mark.parametrize("n", [5, 9, 33, 129, 1025, 4097])
def test_whole_level_is_bit_identical(n):
    run(n, 1, seed=n)


@pytest.mark.parametrize("n,ranks", [(257, 2), (257, 4), (1025, 2), (1025, 8), (4097, 4), (4097, 8)])
def test_slab_windows_are_bit_identical(n, ranks):
    run(n, ranks, seed=n + ranks)


def test_fmg_pass_and_solve_match_oracle_at_4097():
    """the one-GPU FMG pass with the fused set-up at a size with several strips and row chunks per level"""
    n = 4097
    orc = cc.load("orc")
    f = cc.random_rhs(n, seed=72)
    phi0 = np.random.default_rng(71).standard_normal((n, n))
    want = phi0.copy()
    orc.fmg_general(want, f, prolong=cc.PROLONG_FULL)
    with pmg.Solver(n, omega=2.0 / 3.0, prolong_mode=pmg.PROLONG_FULL) as s:
        s.set_rhs(f)
        s.set_guess(phi0)
        s.cycle(pmg.FMG)
        assert np.array_equal(s.get_solution(), want)
