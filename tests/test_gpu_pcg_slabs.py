"""The fused direction-operator pass of pmg_pcg on row slabs (csrc/kernel_pcg.cuh) on ONE GPU, through the test hook
pmg_test_pcg_direction_apply: whole levels, and the row-slab windows of 2, 4 and 8 "ranks" side by side in one device
buffer with every z and p row more than 1 row beyond the slab NaN and their Dirichlet ring NaN, for the first step (p = z)
and a later one (p = z + beta p).  p and A p are compared BIT FOR BIT with the oracle's direction update followed by its
apply_laplacian expression; every other element of the output arrays (ring, other rows, padding) must stay all-zero bits,
the inputs keep their bits and the partial sums add up to p . A p within 1e-14 relative.  This is the GPU twin of
tests/cpp/test_pcg_emu.cpp and gives the slab path hardware coverage on a one-GPU box, where tests/test_gpu_dist_pcg.py has
to skip."""
import ctypes
import math

import numpy as np
import pytest

import pmg_b200 as pmg

pytestmark = pytest.mark.gpu

PADX, PADY = 16, 8
MAX_PARTIALS = 148 * 32


def _lib():
    L = pmg.lib()
    L.pmg_test_layout.restype = None
    L.pmg_test_layout.argtypes = [ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 3
    L.pmg_test_pcg_direction_apply.argtypes = ([ctypes.c_void_p] * 4 + [ctypes.c_int] * 4 + [ctypes.c_double] +
                                               [ctypes.c_void_p] * 2 + [ctypes.c_int] + [ctypes.c_void_p] +
                                               [ctypes.POINTER(ctypes.c_int)])
    return L


def level_pitch(n):
    p, px, py = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib().pmg_test_layout(n, ctypes.byref(p), ctypes.byref(px), ctypes.byref(py))
    assert (px.value, py.value) == (PADX, PADY)
    return p.value


def make_case(n, first, seed):
    """z, p_old random with a zero ring; the oracle's direction update (orc_pcg) and apply_a (pmg_oracle_smoothers.c)"""
    rng = np.random.default_rng(seed)
    z = np.zeros((n, n))
    p_old = np.zeros((n, n))
    z[1:-1, 1:-1] = rng.uniform(-1, 1, (n - 2, n - 2))
    p_old[1:-1, 1:-1] = rng.uniform(-1, 1, (n - 2, n - 2))
    num, den = rng.uniform(0.5, 1.0, 2)
    p = z.copy() if first else z + (num / den) * p_old  # numpy: one rounding per operation, as the oracle
    p[0, :] = p[-1, :] = p[:, 0] = p[:, -1] = 0.0
    h = 1.0 / (n - 1)
    ap = np.zeros((n, n))
    c = p[1:-1, 1:-1]
    ap[1:-1, 1:-1] = ((((4 * c - p[1:-1, :-2]) - p[1:-1, 2:]) - p[:-2, 1:-1]) - p[2:, 1:-1]) / (h * h)
    dot = math.fsum((p * ap).ravel())
    return z, p_old, p, ap, num, den, dot


def windows(d, n, spans, depth):
    """the windows [y0 - PADY, y1 + PADY) of d stacked in one padded host array; rows more than `depth` beyond the owned
    rows (and outside the grid) NaN from end to end, the Dirichlet ring NaN.  Returns (array, row offset of each row 0)"""
    pitch = level_pitch(n)
    a = np.full((sum(y1 - y0 + 2 * PADY for y0, y1 in spans), pitch), np.nan)
    offs, o = [], 0
    for y0, y1 in spans:
        offs.append(o + PADY)
        for lr in range(-PADY, y1 - y0 + PADY):
            g = y0 + lr
            if y0 - depth <= g < y1 + depth and 0 <= g < n:
                row = a[o + PADY + lr]
                row[:] = 0.0
                row[PADX:PADX + n] = d[g]
                row[PADX] = row[PADX + n - 1] = np.nan
                if g in (0, n - 1):
                    row[PADX:PADX + n] = np.nan
        o += y1 - y0 + 2 * PADY
    return a, offs


def run(n, ranks, first, seed):
    z, p_old, p, ap, num, den, dot = make_case(n, first, seed)
    spans = [pmg.partition_rows(n, ranks, r) for r in range(ranks)] if ranks > 1 else [(0, n)]
    depth = 1 if ranks > 1 else 0
    hz, offs = windows(z, n, spans, depth)
    hp, _ = windows(p_old, n, spans, depth)
    pitch = level_pitch(n)
    dz, dp = pmg.DeviceArray.from_numpy(hz), pmg.DeviceArray.from_numpy(hp)
    dpo, dap = pmg.DeviceArray.from_numpy(np.zeros_like(hz)), pmg.DeviceArray.from_numpy(np.zeros_like(hz))
    dsc = pmg.DeviceArray.from_numpy(np.array([num, den]))
    dpart = pmg.DeviceArray.from_numpy(np.zeros(MAX_PARTIALS))
    total = []
    for r, (y0, y1) in enumerate(spans):
        off = 8 * (offs[r] * pitch + PADX)
        k = ctypes.c_int()
        pmg.check(_lib().pmg_test_pcg_direction_apply(dz.ptr + off, dp.ptr + off, dpo.ptr + off, dap.ptr + off, n, y1 - y0,
                                                      y0, pitch, 1.0 / (n - 1), dsc.ptr, dsc.ptr + 8, int(first),
                                                      dpart.ptr, ctypes.byref(k)))
        total.extend(dpart.numpy()[:k.value].tolist())
    assert dz.numpy().tobytes() == hz.tobytes() and dp.numpy().tobytes() == hp.tobytes(), "an input was written"
    want_p, want_ap = np.zeros_like(hz), np.zeros_like(hz)
    for r, (y0, y1) in enumerate(spans):
        lo = -1 if r > 0 else 0
        hi = y1 - y0 + (1 if r < len(spans) - 1 else 0)
        for lr in range(lo, hi):
            g = y0 + lr
            if 1 <= g <= n - 2:
                want_p[offs[r] + lr, PADX + 1:PADX + n - 1] = p[g, 1:n - 1]
                if 0 <= lr < y1 - y0:
                    want_ap[offs[r] + lr, PADX + 1:PADX + n - 1] = ap[g, 1:n - 1]
    for name, got, want in (("p", dpo.numpy(), want_p), ("ap", dap.numpy(), want_ap)):
        bad = np.argwhere(got.view(np.uint64) != want.view(np.uint64))
        assert bad.size == 0, "%s: %d elements differ, first at %s: got %r want %r" % (
            name, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])
    assert abs(math.fsum(total) - dot) <= 1e-14 * abs(dot), (math.fsum(total), dot)


@pytest.mark.parametrize("first", [1, 0])
@pytest.mark.parametrize("n", [5, 9, 33, 129, 1025, 4097])
def test_whole_level_is_bit_identical(n, first):
    run(n, 1, first, seed=n + first)


@pytest.mark.parametrize("first", [1, 0])
@pytest.mark.parametrize("n,ranks", [(129, 2), (257, 4), (513, 8), (1025, 2), (1025, 8), (4097, 4)])
def test_slab_windows_are_bit_identical(n, ranks, first):
    run(n, ranks, first, seed=n + ranks + first)
