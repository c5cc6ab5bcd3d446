// kernel_residual_restrict.cuh -- coarse f = R(f - A x) in one pass over x and f (the set-up of PMG_CYCLE_FMG).
// Included by kernels_basic.cu (which owns the launcher) and, under PMG_HOST_EMULATION, by
// tests/cpp/test_residual_restrict_emu.cpp, which runs this source on the CPU against the oracle.
#pragma once
#include "pmg_internal.h"

namespace pmg {

constexpr int RR_WARPS = 8;        // warps per CTA
constexpr int RR_COLS = 31;        // coarse columns a warp writes: lane 0 only feeds lane 1 its odd residual column
constexpr int RR_TARGET_WARPS = 148 * 32;  // shorter row chunks until the grid has about this many warps (4 CTAs per SM)

struct RRGeom {
    int jc_lo, jc_hi;  // local coarse rows written: the global interior rows [1, nc - 2] of the window
    int strips, chunk, blocks;
};

// rows_c local coarse rows whose global index is local + yoff_c (whole level: rows_c = nc, yoff_c = 0)
inline RRGeom residual_restrict_geom(int nc, int rows_c, int yoff_c)
{
    RRGeom g{};
    g.jc_lo = 1 - yoff_c > 0 ? 1 - yoff_c : 0;
    g.jc_hi = nc - 1 - yoff_c < rows_c ? nc - 1 - yoff_c : rows_c;
    const int rows = g.jc_hi - g.jc_lo;
    if (rows < 1 || nc < 3) return g;
    g.strips = (nc - 2 + RR_COLS - 1) / RR_COLS;
    g.chunk = 64;
    while (g.chunk > 8 && (long)g.strips * ((rows + g.chunk - 1) / g.chunk) < RR_TARGET_WARPS) g.chunk /= 2;
    const long warps = (long)g.strips * ((rows + g.chunk - 1) / g.chunk);
    g.blocks = (int)((warps + RR_WARPS - 1) / RR_WARPS);
    return g;
}

// Fused residual + full-weighting restriction, bit-identical to k_residual followed by k_restrict: every fine residual is
// residual_point(...) and every coarse value restrict_point(...) with the same arguments in the same order.
//
// Scheme: a row-streaming warp.  Warp w owns a strip of 32 fine column PAIRS (2ic, 2ic + 1), ic = 31 * strip + lane, and
// a chunk of coarse rows; it walks down the chunk two fine rows per coarse row, keeping three x rows, the east neighbour
// of lane 31 and the previous odd residual row in registers.  The residuals of a row pair are formed once per lane; the
// west column 2ic - 1 a coarse point needs is lane - 1's odd column, and the x neighbours 2ic - 1 / 2ic + 2 come from the
// adjacent lanes, all by shuffle.  So inside a strip every x and f element is loaded once and every residual computed
// once.  Lane 0 writes nothing (its pair is the previous strip's lane 31), and a chunk re-reads the 2 x rows and 1 f row
// above it; with 64-row chunks on large levels that is 1/32 of the columns and ~2 % of the rows, read by neighbouring
// warps of the same CTA or chunk moments apart (L1 / L2), so HBM sees x and f once: 16 B read + 2 B written per fine
// point (the residual array plus a separate restriction move 24 + 10 B).  A shared-memory tile would need the same
// column and row overlap plus a barrier per row.
//
// Reads, relative to the coarse rows written (local jc in [jc_lo, jc_hi)): x rows [2 jc_lo - 2, 2 jc_hi], f rows
// [2 jc_lo - 1, 2 jc_hi - 1].  On a row slab (rows_c coarse rows over 2 rows_c or 2 rows_c - 1 fine rows) that is at
// most 2 rows of x and 1 row of f beyond the owned fine rows on each side, within PADY.  Columns: x up to 2ic + 2 with
// ic < 31 * strips + 32, i.e. at most nf + 61, inside the right padding; only coarse interior points are written.
// x, f: logical (0,0) of the solver's padded layout (logical column 0 16-byte aligned, even pitches).
__global__ void __launch_bounds__(RR_WARPS * 32)
    k_residual_restrict(const double *__restrict__ x, const double *__restrict__ f, double *__restrict__ coarse, int nc,
                        RRGeom g, int pitch_x, int pitch_f, int pitch_c, double inv_h2)
{
    const int lane = threadIdx.x & 31;
    const long w = (long)blockIdx.x * RR_WARPS + (threadIdx.x >> 5);
    const int strip = (int)(w % g.strips);
    const int j0 = g.jc_lo + (int)(w / g.strips) * g.chunk;
    if (j0 >= g.jc_hi) return;  // warp-uniform
    const int j1 = min(j0 + g.chunk, g.jc_hi);
    const int ic = RR_COLS * strip + lane;
    const int cx = 2 * ic;
    const bool writes = lane > 0 && ic <= nc - 2;
    const unsigned FULL = 0xffffffffu;
    auto ldx = [&](int y) { return *reinterpret_cast<const double2 *>(x + (ptrdiff_t)y * pitch_x + cx); };
    auto ldf = [&](int y) { return *reinterpret_cast<const double2 *>(f + (ptrdiff_t)y * pitch_f + cx); };
    auto east = [&](int y) { return lane == 31 ? x[(ptrdiff_t)y * pitch_x + cx + 2] : 0.0; };
    // residuals of one fine row at columns cx (r0) and cx + 1 (r1); xs / xc / xn = rows y - 1, y, y + 1
    auto resid = [&](const double2 &xs, const double2 &xc, const double2 &xn, double xe31, const double2 &fr, double &r0,
                     double &r1) {
        const double xw = __shfl_up_sync(FULL, xc.y, 1);  // x(y, cx - 1)
        double xe = __shfl_down_sync(FULL, xc.x, 1);      // x(y, cx + 2)
        if (lane == 31) xe = xe31;
        r0 = residual_point(inv_h2, fr.x, xc.x, xw, xc.y, xs.x, xn.x);
        r1 = residual_point(inv_h2, fr.y, xc.y, xc.x, xe, xs.y, xn.y);
    };
    // warm-up: residual row 2 j0 - 1 (the south row of the first coarse row)
    double2 xa = ldx(2 * j0 - 2), xb = ldx(2 * j0 - 1), xc = ldx(2 * j0);
    double eb = east(2 * j0 - 1), ec = east(2 * j0);
    double rs0, rs1;
    resid(xa, xb, xc, eb, ldf(2 * j0 - 1), rs0, rs1);
#pragma unroll 2
    for (int jc = j0; jc < j1; ++jc) {
        const int y = 2 * jc;
        const double2 xd = ldx(y + 1), xe = ldx(y + 2), f0 = ldf(y), f1 = ldf(y + 1);
        const double ed = east(y + 1), ee = east(y + 2);
        double rc0, rc1, rn0, rn1;
        resid(xb, xc, xd, ec, f0, rc0, rc1);  // row 2jc
        resid(xc, xd, xe, ed, f1, rn0, rn1);  // row 2jc + 1
        const double sw = __shfl_up_sync(FULL, rs1, 1), wv = __shfl_up_sync(FULL, rc1, 1), nw = __shfl_up_sync(FULL, rn1, 1);
        if (writes)
            coarse[(ptrdiff_t)jc * pitch_c + ic] = restrict_point(rc0, rc1, wv, rn0, rs0, sw, rs1, nw, rn1);
        rs0 = rn0;
        rs1 = rn1;
        xb = xd;
        xc = xe;
        ec = ee;
    }
}

}  // namespace pmg
