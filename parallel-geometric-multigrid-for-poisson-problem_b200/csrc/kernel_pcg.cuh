// kernel_pcg.cuh -- the level-0 vector passes of pmg_pcg on row slabs: the fused direction-operator pass and the update,
// both reading their CG scalars from device memory.  Included by kernels_basic.cu (which owns the launchers) and, under
// PMG_HOST_EMULATION, by tests/cpp/test_pcg_emu.cpp, which runs this source on the CPU against the oracle.
#pragma once
#include "pmg_internal.h"

#ifdef PMG_HOST_EMULATION
inline double __ddiv_rn(double a, double b) { return a / b; }
#endif

namespace pmg {

constexpr int PD_WARPS = 8;              // warps per CTA
constexpr int PD_MAX_WARPS = 148 * 32;   // at most 4 CTAs per SM; every warp grid-strides over its work items
static_assert(PD_MAX_WARPS == PCG_MAX_PARTIALS, "the partial buffer pmg_internal.h promises");

struct PDGeom {
    int a_lo, a_hi;  // local rows of A p: the global interior rows [1, n - 2] among the window's owned rows [0, rows)
    int strips, chunk, items, blocks;
};

// rows owned local rows whose global index is local + yoff (whole level: rows = n, yoff = 0)
inline PDGeom pcg_geom(int n, int rows, int yoff)
{
    PDGeom g{};
    g.a_lo = 1 - yoff > 0 ? 1 - yoff : 0;
    g.a_hi = n - 1 - yoff < rows ? n - 1 - yoff : rows;
    const int r = g.a_hi - g.a_lo;
    if (r < 1 || n < 3) return g;
    g.strips = (n - 2 + 31) / 32;
    g.chunk = 64;
    while (g.chunk > 8 && (long)g.strips * ((r + g.chunk - 1) / g.chunk) < PD_MAX_WARPS) g.chunk /= 2;
    g.items = g.strips * ((r + g.chunk - 1) / g.chunk);
    const int warps = g.items < PD_MAX_WARPS ? g.items : PD_MAX_WARPS;
    g.blocks = (warps + PD_WARPS - 1) / PD_WARPS;
    return g;
}

// partial sums written by a launch of geometry g (warps without a work item write 0)
inline int pcg_partials(const PDGeom &g) { return g.blocks * PD_WARPS; }

__device__ __forceinline__ double pcg_warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = dadd(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// The direction-operator pass of one CG step, in one sweep over a window (or a whole level):
//   p_out = z + beta p_in  (first: p_out = z), beta = *beta_num / *beta_den
//   ap    = (4 p - W - E - S - N) / h^2       (DynamicGridUtils::apply_laplacian: un-fused dsub, then a division, as
//                                              k_apply_a_dot)
//   partials[warp] = sum of p . ap over the warp's points
// p_out, ap and the sums cover the owned interior rows [a_lo, a_hi); p_out is ALSO written on the interior rows a_lo - 1
// and a_hi next to a neighbour's slab.  Those two rows are recomputed here from z and p_in rather than exchanged, so p
// needs no halo exchange: the next step's pass reads p_in exactly on the rows this one wrote.  The pass reads z and p_in
// on rows [a_lo - 1, a_hi] (one row beyond each slab edge) and nothing on the ring or in the padding; it writes p_out
// and ap on interior points only, so their Dirichlet ring and padding keep whatever they hold (zero).  p_in and p_out
// are different arrays: a neighbouring warp may still read p_in at the points this one writes.
// Traffic: z, p_in read, p_out, ap written -- 32 B/point, against 40 for k_pcg_direction followed by k_apply_a_dot.
//
// Scheme: warp = a strip of 32 interior columns x a chunk of rows, walked downwards with the rows y - 1, y, y + 1 of the
// new direction in registers; the west / east neighbours come from the adjacent lanes by shuffle, lanes 0 and 31
// recompute their outer neighbour.  A chunk recomputes the direction on the one row above and below it (L1 / L2).
__global__ void __launch_bounds__(PD_WARPS * 32)
    k_pcg_direction_apply(const double *__restrict__ z, const double *__restrict__ p_in, double *__restrict__ p_out,
                          double *__restrict__ ap, int n, int yoff, PDGeom g, int pitch, double h2,
                          const double *__restrict__ beta_num, const double *__restrict__ beta_den, int first,
                          double *__restrict__ partials)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * PD_WARPS + (threadIdx.x >> 5);
    const int nw = gridDim.x * PD_WARPS;
    const double beta = first ? 0.0 : __ddiv_rn(*beta_num, *beta_den);
    // the new direction at local (y, x); zero on the Dirichlet ring and outside the grid (never loaded there)
    auto pnew = [&](int y, int x) -> double {
        const int gy = y + yoff;
        if (gy < 1 || gy > n - 2 || x < 1 || x > n - 2) return 0.0;
        const ptrdiff_t i = (ptrdiff_t)y * pitch + x;
        return first ? z[i] : dadd(z[i], dmul(beta, p_in[i]));
    };
    const bool write_lo = g.a_lo - 1 + yoff >= 1, write_hi = g.a_hi + yoff <= n - 2;  // the rows next to a neighbour
    double acc = 0.0;
    for (int it = wid; it < g.items; it += nw) {  // warp-uniform
        const int x = 1 + 32 * (it % g.strips) + lane;
        const int y0 = g.a_lo + (it / g.strips) * g.chunk;
        const int y1 = min(y0 + g.chunk, g.a_hi);
        const bool col = x <= n - 2;
        double ps = pnew(y0 - 1, x), pc = pnew(y0, x);
        if (col && y0 == g.a_lo && write_lo) p_out[(ptrdiff_t)(y0 - 1) * pitch + x] = ps;
        for (int y = y0; y < y1; ++y) {
            const double pn = pnew(y + 1, x);
            double w = __shfl_up_sync(FULL, pc, 1), e = __shfl_down_sync(FULL, pc, 1);
            if (lane == 0) w = pnew(y, x - 1);
            if (lane == 31) e = pnew(y, x + 1);
            if (col) {
                const ptrdiff_t i = (ptrdiff_t)y * pitch + x;
                const double v = __ddiv_rn(dsub(dsub(dsub(dsub(dmul(4.0, pc), w), e), ps), pn), h2);
                p_out[i] = pc;
                ap[i] = v;
                acc = dadd(acc, dmul(pc, v));
            }
            ps = pc;
            pc = pn;
        }
        if (col && y1 == g.a_hi && write_hi) p_out[(ptrdiff_t)y1 * pitch + x] = pc;
    }
    acc = pcg_warp_sum(acc);
    if (lane == 0) partials[wid] = acc;
}

// x += alpha p ; r -= alpha ap ; partials[warp] = sum of r . r -- k_pcg_update's arithmetic on the owned interior rows,
// with alpha = *alpha_num / *alpha_den read from device memory
__global__ void __launch_bounds__(PD_WARPS * 32)
    k_pcg_update_dev(double *__restrict__ x, double *__restrict__ r, const double *__restrict__ p,
                     const double *__restrict__ ap, int n, PDGeom g, int pitch, const double *__restrict__ alpha_num,
                     const double *__restrict__ alpha_den, double *__restrict__ partials)
{
    const int lane = threadIdx.x & 31;
    const int wid = blockIdx.x * PD_WARPS + (threadIdx.x >> 5);
    const int nw = gridDim.x * PD_WARPS;
    const double alpha = __ddiv_rn(*alpha_num, *alpha_den);
    double acc = 0.0;
    for (int it = wid; it < g.items; it += nw) {
        const int xx = 1 + 32 * (it % g.strips) + lane;
        const int y0 = g.a_lo + (it / g.strips) * g.chunk;
        const int y1 = min(y0 + g.chunk, g.a_hi);
        if (xx > n - 2) continue;
        for (int y = y0; y < y1; ++y) {
            const ptrdiff_t i = (ptrdiff_t)y * pitch + xx;
            x[i] = dadd(x[i], dmul(alpha, p[i]));
            const double rv = dsub(r[i], dmul(alpha, ap[i]));
            r[i] = rv;
            acc = dadd(acc, dmul(rv, rv));
        }
    }
    acc = pcg_warp_sum(acc);
    if (lane == 0) partials[wid] = acc;
}

}  // namespace pmg
