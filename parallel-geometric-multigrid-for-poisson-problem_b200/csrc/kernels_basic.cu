// kernels_basic.cu -- one kernel per reference operator (the PMG_ENGINE_OPERATOR engine and the
// operator-level C ABI that replaces class Parallel, 3_part_parallel/Parallel_Method.cu:144-199).
//
// Every kernel takes pointers to logical (0,0) plus a row pitch, so the same code serves the dense
// reference layout (pitch = width) and the solver's padded hierarchy.  Arithmetic follows the
// reference's evaluation order with explicit round-to-nearest adds/multiplies (no FMA contraction):
// outputs are bit-identical to the CPU path.  All are HBM-bound: 24 B/pt (Jacobi, residual),
// 10 B/fine-pt (restriction), 18 B/fine-pt (prolongation) -- see DESIGN.md section 4.
#include <atomic>
#include <cstdlib>

#define PMG_NEEDS_PEER_WAIT
#include "pmg_internal.h"
#include "kernel_residual_restrict.cuh"
#include "kernel_pcg.cuh"

namespace pmg {

static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
unsigned long long launches_so_far() { return g_launches.load(std::memory_order_relaxed); }

namespace {

constexpr int BX = 64, BY = 4;  // 256 threads; a warp covers 32 consecutive columns of one row

inline dim3 grid2d(int nx, int ny) { return dim3((nx + BX - 1) / BX, (ny + BY - 1) / BY); }

// ---- weighted Jacobi sweep: Smoother.hpp:61-70 (replaces jacobi_kernel, Parallel_Method.cu:6-24,
//      which updates in place and races) -------------------------------------------------------------
__global__ void __launch_bounds__(BX *BY)
    k_jacobi_sweep(double *__restrict__ out, const double *__restrict__ in, const double *__restrict__ f,
                   int nx, int ny, int pitch_x, int pitch_f, JacobiCoef c)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x >= nx || y >= ny) return;
    size_t i = (size_t)y * pitch_x + x;
    double v = in[i];
    if (x > 0 && x < nx - 1 && y > 0 && y < ny - 1)
        v = jacobi_point(c, f[(size_t)y * pitch_f + x], v, in[i - 1], in[i + 1], in[i - pitch_x],
                         in[i + pitch_x]);
    out[i] = v;
}

// ---- all sweeps of a small level inside one CTA (coarsest-grid solve, MultiGrid.hpp:59-63) ---------
__global__ void __launch_bounds__(1024)
    k_jacobi_small(double *__restrict__ xg, const double *__restrict__ fg, int nx, int ny, int pitch_x,
                   int pitch_f, JacobiCoef c, int sweeps, int x_is_zero, const int *__restrict__ done)
{
    pdl_prologue();
    __shared__ double a[SMALL_MAX_POINTS], b[SMALL_MAX_POINTS], fs[SMALL_MAX_POINTS];
    if (done != nullptr && *done) return;
    int l = nx * ny;
    for (int i = threadIdx.x; i < l; i += blockDim.x) {
        int y = i / nx, x = i - y * nx;
        double v = x_is_zero ? 0.0 : xg[(size_t)y * pitch_x + x];
        a[i] = v;
        b[i] = v;
        fs[i] = fg[(size_t)y * pitch_f + x];
    }
    __syncthreads();
    double *src = a, *dst = b;
    for (int s = 0; s < sweeps; ++s) {
        for (int i = threadIdx.x; i < l; i += blockDim.x) {
            int y = i / nx, x = i - y * nx;
            if (x > 0 && x < nx - 1 && y > 0 && y < ny - 1)
                dst[i] = jacobi_point(c, fs[i], src[i], src[i - 1], src[i + 1], src[i - nx], src[i + nx]);
        }
        __syncthreads();
        double *t = src;
        src = dst;
        dst = t;
    }
    for (int i = threadIdx.x; i < l; i += blockDim.x) {
        int y = i / nx, x = i - y * nx;
        xg[(size_t)y * pitch_x + x] = src[i];
    }
}

// ---- a whole V-cycle of the small levels inside ONE CTA ------------------------------------------------------
// Levels n0 (<= VSMALL_TOP) -> ... -> n_coarse live in shared memory (x, scratch, f per level); every operator is
// the reference's, point for point (pmg_internal.h), separated by block barriers.  Replaces 2 launches per
// level (each ~5 us of pure latency at these sizes) by one.  MultiGrid.hpp:57-94 restricted to small N.
extern __shared__ __align__(16) double g_vs_smem[];

__device__ __forceinline__ void vs_sweeps(double *&cur, double *&oth, const double *f, int n, const JacobiCoef &c,
                                          int sweeps)
{
    // 2-D thread decomposition (64 columns x blockDim/64 rows): no integer divisions in the point loops
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6, nty = blockDim.x >> 6;
    for (int s = 0; s < sweeps; ++s) {
        for (int y = ty; y < n; y += nty)
            for (int x = tx; x < n; x += 64) {
                const int i = y * n + x;
                double v = cur[i];
                if (x > 0 && x < n - 1 && y > 0 && y < n - 1)
                    v = jacobi_point(c, f[i], v, cur[i - 1], cur[i + 1], cur[i - n], cur[i + n]);
                oth[i] = v;
            }
        __syncthreads();
        double *t = cur;
        cur = oth;
        oth = t;
    }
}

__global__ void __launch_bounds__(1024)
    k_vcycle_small(double *__restrict__ xg, const double *__restrict__ fg, int n0, int pitch_x, int pitch_f,
                   int n_coarse, double h0, double omega, int nu1, int nu2, int coarse_sweeps, int lo,
                   int x_is_zero, int gamma, const int *__restrict__ done)
{
    pdl_prologue();
    if (done != nullptr && *done) return;
    constexpr int MAXL = 8;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6, nty = blockDim.x >> 6;
    double *cur[MAXL], *oth[MAXL], *f[MAXL];
    int n[MAXL];
    double h[MAXL];
    int nl = 0;
    {
        double *p = g_vs_smem;
        int m = n0;
        double hh = h0;
        for (;;) {
            n[nl] = m;
            h[nl] = hh;
            cur[nl] = p;
            oth[nl] = p + m * m;
            f[nl] = p + 2 * m * m;
            p += 3 * m * m;
            ++nl;
            if (m <= n_coarse || m <= 3 || nl == MAXL) break;
            m = (m - 1) / 2 + 1;
            hh = 2 * hh;  // MultiGrid.hpp:83
        }
    }
    // level 0: right-hand side from global memory, iterate zero (first visit of a coarse level) or loaded
    for (int i = threadIdx.x; i < n0 * n0; i += blockDim.x) {
        int y = i / n0, x = i - y * n0;
        f[0][i] = fg[(size_t)y * pitch_f + x];
        cur[0][i] = x_is_zero ? 0.0 : xg[(size_t)y * pitch_x + x];
    }
    __syncthreads();
    auto coef_of = [&](int k) {
        JacobiCoef c;
        c.h2 = h[k] * h[k];
        c.omega = omega;
        c.om1 = 1.0 - omega;
        c.w4 = 0.25 * omega;
        c.weighted = (omega != 1.0);
        return c;
    };
    // pre-smooth, residual, restriction into level k+1, whose iterate is zeroed (MultiGrid.hpp:66-82)
    auto descend = [&](int k) {
        vs_sweeps(cur[k], oth[k], f[k], n[k], coef_of(k), nu1);
        const double inv_h2 = 1.0 / (h[k] * h[k]);
        const int m = n[k];
        double *r = oth[k];
        for (int y = 1 + ty; y < m - 1; y += nty)
            for (int x = 1 + tx; x < m - 1; x += 64) {
                const int i = y * m + x;
                r[i] = residual_point(inv_h2, f[k][i], cur[k][i], cur[k][i - 1], cur[k][i + 1], cur[k][i - m],
                                      cur[k][i + m]);
            }
        __syncthreads();
        const int mc = n[k + 1];
        for (int jc = ty; jc < mc; jc += nty)
            for (int ic = tx; ic < mc; ic += 64) {
                double v = 0.0;
                if (ic > 0 && ic < mc - 1 && jc > 0 && jc < mc - 1) {
                    const double *q = r + (2 * jc) * m + 2 * ic;
                    v = restrict_point(q[0], q[1], q[-1], q[m], q[-m], q[-m - 1], q[-m + 1], q[m - 1], q[m + 1]);
                }
                f[k + 1][jc * mc + ic] = v;
                cur[k + 1][jc * mc + ic] = 0.0;
            }
        __syncthreads();
    };
    // prolongation-and-add from level k+1, post-smooth (MultiGrid.hpp:86-89)
    auto ascend = [&](int k) {
        const int m = n[k], mc = n[k + 1];
        const double *e = cur[k + 1];
        for (int y = lo + ty; y <= m - 2; y += nty)
            for (int x = lo + tx; x <= m - 2; x += 64) {
                const int i = y * m + x;
                const double *q = e + (y >> 1) * mc + (x >> 1);
                double v;
                if ((y & 1) == 0)
                    v = ((x & 1) == 0) ? q[0] : dmul(0.5, dadd(q[0], q[1]));
                else
                    v = ((x & 1) == 0) ? dmul(0.5, dadd(q[0], q[mc]))
                                       : dmul(0.25, dadd(dadd(dadd(q[0], q[1]), q[mc]), q[mc + 1]));
                cur[k][i] = dadd(cur[k][i], v);
            }
        __syncthreads();
        vs_sweeps(cur[k], oth[k], f[k], n[k], coef_of(k), nu2);
    };
    // the recursion of v_cycle (gamma = 1) / w_cycle (gamma visits of every coarser level, MultiGrid.hpp:124-125)
    // unrolled into a loop; every thread follows the same path
    if (nl == 1) {
        vs_sweeps(cur[0], oth[0], f[0], n[0], coef_of(0), coarse_sweeps);
    } else {
        int visits[MAXL];
        int k = 0;
        bool down = true;
        for (;;) {
            if (down) {
                if (k == nl - 1) {  // coarsest level (MultiGrid.hpp:59-63)
                    vs_sweeps(cur[k], oth[k], f[k], n[k], coef_of(k), coarse_sweeps);
                    down = false;
                    --k;
                } else {
                    descend(k);
                    visits[k] = 0;
                    ++k;
                }
            } else {  // one visit of level k+1 has finished
                if (++visits[k] < gamma) {
                    ++k;
                    down = true;
                } else {
                    ascend(k);
                    if (k == 0) break;
                    --k;
                }
            }
        }
    }
    for (int i = threadIdx.x; i < n0 * n0; i += blockDim.x) {
        int y = i / n0, x = i - y * n0;
        xg[(size_t)y * pitch_x + x] = cur[0][i];
    }
}

// ---- residual: DynamicGridUtils.hpp:59-69 (replaces device_compute_residual, Parallel_Method.cu:26-46)
__global__ void __launch_bounds__(BX *BY)
    k_residual(double *__restrict__ r, const double *__restrict__ xg, const double *__restrict__ f, int nx,
               int ny, int pitch_r, int pitch_x, int pitch_f, double inv_h2)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x < 1 || y < 1 || x >= nx - 1 || y >= ny - 1) return;
    size_t i = (size_t)y * pitch_x + x;
    r[(size_t)y * pitch_r + x] = residual_point(inv_h2, f[(size_t)y * pitch_f + x], xg[i], xg[i - 1],
                                                xg[i + 1], xg[i - pitch_x], xg[i + pitch_x]);
}

// ---- deterministic sum reductions -------------------------------------------------------------------
constexpr int RED_THREADS = 256;
constexpr int RED_BLOCKS = 148 * 8;

__device__ __forceinline__ double block_sum(double v)
{
    __shared__ double warp_part[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = dadd(v, __shfl_xor_sync(0xffffffffu, v, o));
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) warp_part[w] = v;
    __syncthreads();
    int nw = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nw) ? warp_part[threadIdx.x] : 0.0;
    if (w == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = dadd(v, __shfl_xor_sync(0xffffffffu, v, o));
    }
    return v;  // valid in thread 0
}

// sum over the interior of (f - A x)^2 without materialising r (16 B/pt)
__global__ void __launch_bounds__(RED_THREADS)
    k_residual_norm2(const double *__restrict__ xg, const double *__restrict__ f, int nx, int ny,
                     int pitch_x, int pitch_f, double inv_h2, double *__restrict__ partials)
{
    double acc = 0.0;
    int chunks_x = (nx + RED_THREADS - 1) / RED_THREADS;
    long total = (long)chunks_x * ny;
    for (long t = blockIdx.x; t < total; t += gridDim.x) {
        int y = (int)(t / chunks_x);
        int x = (int)(t - (long)y * chunks_x) * RED_THREADS + threadIdx.x;
        if (x >= 1 && y >= 1 && x < nx - 1 && y < ny - 1) {
            size_t i = (size_t)y * pitch_x + x;
            double r = residual_point(inv_h2, f[(size_t)y * pitch_f + x], xg[i], xg[i - 1], xg[i + 1],
                                      xg[i - pitch_x], xg[i + pitch_x]);
            acc = dadd(acc, dmul(r, r));
        }
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// The reference's summation ORDER (DynamicGridUtils.hpp:21-27: sum += r[i]*r[i], i ascending over the
// row-major array; ring entries are zero and leave the running sum unchanged).  All threads of one CTA
// compute the squares of the next 2048 interior points into shared memory while thread 0 adds the
// previous 2048 one at a time -- the result is bit-identical to the CPU loop.  Validation only.
constexpr int SEQ_CHUNK = 2048;
__global__ void __launch_bounds__(1024)
    k_residual_norm2_seq(const double *__restrict__ xg, const double *__restrict__ f, int nx, int ny,
                         int pitch_x, int pitch_f, double inv_h2, double *__restrict__ out)
{
    __shared__ double buf[2][SEQ_CHUNK];
    const int per_row = (nx - 2 + SEQ_CHUNK - 1) / SEQ_CHUNK;
    const long chunks = (long)per_row * (ny - 2);
    double acc = 0.0;
    for (long c = 0; c <= chunks; ++c) {
        if (c < chunks) {
            int y = 1 + (int)(c / per_row);
            int x0 = 1 + (int)(c - (long)(y - 1) * per_row) * SEQ_CHUNK;
            double *dst = buf[c & 1];
            for (int k = threadIdx.x; k < SEQ_CHUNK; k += blockDim.x) {
                int x = x0 + k;
                double sq = 0.0;
                if (x < nx - 1) {
                    size_t i = (size_t)y * pitch_x + x;
                    double r = residual_point(inv_h2, f[(size_t)y * pitch_f + x], xg[i], xg[i - 1], xg[i + 1],
                                              xg[i - pitch_x], xg[i + pitch_x]);
                    sq = dmul(r, r);
                }
                dst[k] = sq;
            }
        }
        if (threadIdx.x == 0 && c > 0) {
            long p = c - 1;
            int y = 1 + (int)(p / per_row);
            int x0 = 1 + (int)(p - (long)(y - 1) * per_row) * SEQ_CHUNK;
            int cnt = min(SEQ_CHUNK, nx - 1 - x0);
            const double *src = buf[p & 1];
#pragma unroll 8
            for (int k = 0; k < cnt; ++k) acc = dadd(acc, src[k]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = acc;
}

__global__ void __launch_bounds__(RED_THREADS)
    k_norm2(const double *__restrict__ v, size_t l, double *__restrict__ partials)
{
    double acc = 0.0;
    for (size_t i = (size_t)blockIdx.x * RED_THREADS + threadIdx.x; i < l;
         i += (size_t)gridDim.x * RED_THREADS) {
        double t = v[i];
        acc = dadd(acc, dmul(t, t));
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

__global__ void __launch_bounds__(1024) k_final_sum(const double *__restrict__ partials, int count,
                                                    double *__restrict__ out)
{
    pdl_prologue();
    double acc = 0.0;
    for (int i = threadIdx.x; i < count; i += blockDim.x) acc = dadd(acc, partials[i]);
    acc = block_sum(acc);
    if (threadIdx.x == 0) *out = acc;
}

__global__ void k_solve_begin(const double *__restrict__ norm2, SolveCtrl *ctrl, double *__restrict__ hist2,
                              double rel_tol, int max_cycles)
{
    hist2[0] = *norm2;
    ctrl->r0 = sqrt(*norm2);
    ctrl->rel_tol = rel_tol;
    ctrl->cycles = 0;
    ctrl->max_cycles = max_cycles;
    ctrl->done = (max_cycles <= 0) ? 1 : 0;
}

// The solve's control block (and, at the end, its history) written into MAPPED PINNED host memory by a kernel instead
// of a cudaMemcpyAsync: a device-to-host copy would queue on the DMA engine behind whatever bulk transfer another stream
// has in flight (pmg_fetch_solution_begin: 2 GB, ~36 ms), and the host would learn that the solve has converged that
// much later.  A store from a kernel does not pass through the copy engines.
__global__ void __launch_bounds__(1024)
    k_ctrl_to_host(const SolveCtrl *__restrict__ ctrl, SolveCtrl *host_ctrl, const double *__restrict__ hist2,
                   double *host_hist, int hist_cap)
{
    pdl_prologue();
    if (host_hist != nullptr) {
        const int k = ctrl->cycles;
        for (int i = threadIdx.x; i <= k && i < hist_cap; i += blockDim.x) host_hist[i] = hist2[i];
    }
    if (threadIdx.x == 0) *host_ctrl = *ctrl;
    __threadfence_system();
}

// Last kernel of a cycle (MultiGridTestRunner.hpp:210-211 + the relative stopping test the reference lacks)
__global__ void __launch_bounds__(1024)
    k_cycle_finish(const double *__restrict__ partials, int count, SolveCtrl *ctrl, double *__restrict__ hist2)
{
    pdl_prologue();
    if (ctrl->done) return;
    double acc = 0.0;
    for (int i = threadIdx.x; i < count; i += blockDim.x) acc = dadd(acc, partials[i]);
    acc = block_sum(acc);
    if (threadIdx.x == 0) {
        int c = ctrl->cycles + 1;
        ctrl->cycles = c;
        hist2[c] = acc;
        if (sqrt(acc) < dmul(ctrl->rel_tol, ctrl->r0) || c >= ctrl->max_cycles) ctrl->done = 1;
    }
}

// ---- full-weighting restriction: MultiGrid.hpp:187-205 (replaces restriction_kernel_full_weighting,
//      Parallel_Method.cu:48-78) ---------------------------------------------------------------------
//      Row slabs: `rows` local coarse rows, local row 0 = global coarse row `yoff` (local fine row = 2 * local
//      coarse row because slabs start on even fine rows); whole level: rows = nc, yoff = 0.
__global__ void __launch_bounds__(BX *BY)
    k_restrict(const double *__restrict__ fine, double *__restrict__ coarse, int nc, int rows, int yoff, int pitch_f,
               int pitch_c)
{
    int ic = blockIdx.x * BX + threadIdx.x;
    int jc = blockIdx.y * BY + threadIdx.y;
    if (ic < 1 || ic >= nc - 1 || jc >= rows || jc + yoff < 1 || jc + yoff >= nc - 1) return;
    const double *c = fine + (size_t)(2 * jc) * pitch_f + 2 * ic;
    coarse[(size_t)jc * pitch_c + ic] =
        restrict_point(c[0], c[1], c[-1], c[pitch_f], c[-pitch_f], c[-pitch_f - 1], c[-pitch_f + 1],
                       c[pitch_f - 1], c[pitch_f + 1]);
}

// ---- bilinear prolongation-and-add: MultiGrid.hpp:208-226.  One thread per FINE point; the parity of
//      (x, y) selects the same expression the reference's coarse-point loop evaluates for that point.
//      lo = 2 (REFERENCE: fine row/col 1 skipped) or 1 (FULL). ---------------------------------------
//      Row slabs: `rows` local fine rows, local row 0 = global fine row `yoff` (even), coarse local row 0 =
//      global coarse row yoff / 2; whole level: rows = nf, yoff = 0.
__global__ void __launch_bounds__(BX *BY)
    k_prolong_add(const double *__restrict__ coarse, double *__restrict__ fine, int nf, int rows, int yoff,
                  int pitch_c, int pitch_f, int lo)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x < lo || x > nf - 2 || y >= rows || y + yoff < lo || y + yoff > nf - 2) return;
    int ic = x >> 1, jc = y >> 1;
    const double *c = coarse + (size_t)jc * pitch_c + ic;
    double v;
    if ((y & 1) == 0)
        v = ((x & 1) == 0) ? c[0] : dmul(0.5, dadd(c[0], c[1]));
    else
        v = ((x & 1) == 0) ? dmul(0.5, dadd(c[0], c[pitch_c]))
                           : dmul(0.25, dadd(dadd(dadd(c[0], c[1]), c[pitch_c]), c[pitch_c + 1]));
    size_t i = (size_t)y * pitch_f + x;
    fine[i] = dadd(fine[i], v);
}

__global__ void __launch_bounds__(BX *BY)
    k_copy2d(double *__restrict__ dst, int pitch_d, const double *__restrict__ src, int pitch_s, int nx, int ny)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x < nx && y < ny) dst[(size_t)y * pitch_d + x] = src[(size_t)y * pitch_s + x];
}

__global__ void __launch_bounds__(BX *BY) k_fill2d(double *__restrict__ dst, int pitch_d, int nx, int ny, double v)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x < nx && y < ny) dst[(size_t)y * pitch_d + x] = v;
}

__global__ void __launch_bounds__(BX *BY)
    k_rhs_separable(double *__restrict__ f, int pitch, int nx, int ny, double factor,
                    const double *__restrict__ sx, const double *__restrict__ sy)
{
    int x = blockIdx.x * BX + threadIdx.x;
    int y = blockIdx.y * BY + threadIdx.y;
    if (x < nx && y < ny) f[(size_t)y * pitch + x] = dmul(dmul(factor, sx[x]), sy[y]);
}

// ---- smoothers beyond weighted Jacobi (SURVEY.md 8f-3) ----------------------------------------------------------
// GaussSeidelSmoother's update (Smoother.hpp:141-143): x = 0.25 * (x[i-1] + x[i+1] + x[i-width] + x[i+width] + h*h*f)
__device__ __forceinline__ double gs_point(double h2, double f, double xw, double xe, double xs, double xn)
{
    return dmul(0.25, dadd(dadd(dadd(dadd(xw, xe), xs), xn), dmul(h2, f)));
}

// one colour of a red-black Gauss-Seidel sweep, in place: the points with (x + y) & 1 == colour read only points of the
// other colour, so every point of a colour can be updated at once -- the parallel form of the reference's smoother
__global__ void __launch_bounds__(BX *BY)
    k_rbgs_half(double *__restrict__ x, const double *__restrict__ f, int nx, int ny, int pitch_x, int pitch_f, double h2,
                int colour)
{
    const int y = blockIdx.y * BY + threadIdx.y;
    const int xx = 2 * (blockIdx.x * BX + threadIdx.x) + ((y + colour) & 1);
    if (xx < 1 || xx > nx - 2 || y < 1 || y > ny - 2) return;
    double *c = x + (size_t)y * pitch_x + xx;
    *c = gs_point(h2, f[(size_t)y * pitch_f + xx], c[-1], c[1], c[-pitch_x], c[pitch_x]);
}

// GaussSeidelSmoother::smooth (Smoother.hpp:134-145) EXACTLY, lexicographic order included: the points of one
// anti-diagonal x + y = d depend only on diagonal d-1 (new west and south values) and d+1 (old east and north values), so
// a sweep is 2n-5 dependent steps, each parallel along its diagonal.  One CTA walks the diagonals with a barrier in
// between -- a validation path for the reference's part-1 smoother (its sizes are N <= 129), not a fast smoother:
// use the red-black ordering for that.
__global__ void __launch_bounds__(1024)
    k_gs_lex(double *__restrict__ x, const double *__restrict__ f, int nx, int ny, int pitch_x, int pitch_f, double h2,
             int sweeps)
{
    for (int s = 0; s < sweeps; ++s)
        for (int d = 2; d <= (nx - 2) + (ny - 2); ++d) {
            const int ylo = max(1, d - (nx - 2)), yhi = min(ny - 2, d - 1);
            for (int y = ylo + (int)threadIdx.x; y <= yhi; y += (int)blockDim.x) {
                double *c = x + (size_t)y * pitch_x + (d - y);
                *c = gs_point(h2, f[(size_t)y * pitch_f + (d - y)], c[-1], c[1], c[-pitch_x], c[pitch_x]);
            }
            __syncthreads();
        }
}

// Mixed-precision EXPERIMENT (SURVEY.md 8f-4): the weighted-Jacobi sweep evaluated in fp32 -- operands rounded to float,
// the reference's expression order kept, result widened again -- while the fields stay fp64 in HBM and the residual and
// the grid transfers stay fp64.  It answers "what would fp32 smoothing do to the convergence history" without an fp32
// copy of the hierarchy; it does not save bandwidth (an fp32 hierarchy would halve the 24 B/point of a sweep).
__global__ void __launch_bounds__(BX *BY)
    k_jacobi_sweep_f32(double *__restrict__ out, const double *__restrict__ in, const double *__restrict__ f, int nx, int ny,
                       int pitch_x, int pitch_f, float h2, float omega, float om1, int weighted)
{
    const int x = blockIdx.x * BX + threadIdx.x, y = blockIdx.y * BY + threadIdx.y;
    if (x >= nx || y >= ny) return;
    const size_t i = (size_t)y * pitch_x + x;
    if (x == 0 || y == 0 || x == nx - 1 || y == ny - 1) {
        out[i] = in[i];
        return;
    }
    const float xc = (float)in[i], xw = (float)in[i - 1], xe = (float)in[i + 1], xs = (float)in[i - pitch_x],
                xn = (float)in[i + pitch_x], ff = (float)f[(size_t)y * pitch_f + x];
    const float acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(h2, ff), xw), xe), xs), xn);
    const float jac = __fmul_rn(0.25f, acc);
    out[i] = (double)(weighted ? __fadd_rn(__fmul_rn(om1, xc), __fmul_rn(omega, jac)) : jac);
}

// sum over l entries of (a[i] - b[i])^2 and of b[i]^2: the relative error norm of Smoother::smooth's `errors` output
// (Smoother.hpp:92-98: ||x - x_true|| / ||x_true||, DynamicGridUtils::compute_error + norm)
__global__ void __launch_bounds__(RED_THREADS)
    k_diff_norm2(const double *__restrict__ a, const double *__restrict__ b, size_t l, double *__restrict__ partials_d,
                 double *__restrict__ partials_b)
{
    double accd = 0.0, accb = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < l; i += (size_t)gridDim.x * blockDim.x) {
        const double d = dsub(a[i], b[i]);
        accd = dadd(accd, dmul(d, d));
        accb = dadd(accb, dmul(b[i], b[i]));
    }
    accd = block_sum(accd);
    accb = block_sum(accb);
    if (threadIdx.x == 0) {
        partials_d[blockIdx.x] = accd;
        partials_b[blockIdx.x] = accb;
    }
}

// ---- vector kernels of the preconditioned conjugate gradient wrapper (pmg_pcg); padded 2-D arrays, interior only ----
// ap = A p = (4p - W - E - S - N) / (h*h)  (DynamicGridUtils::apply_laplacian, DynamicGridUtils.hpp:46-56: a DIVISION),
// and the partial sums of p . ap
__global__ void __launch_bounds__(RED_THREADS)
    k_apply_a_dot(const double *__restrict__ p, double *__restrict__ ap, int nx, int ny, int pitch, double h2,
                  double *__restrict__ partials)
{
    double acc = 0.0;
    const int chunks_x = (nx + RED_THREADS - 1) / RED_THREADS;
    for (long c = blockIdx.x; c < (long)chunks_x * ny; c += gridDim.x) {
        const int y = (int)(c / chunks_x), xx = (int)(c % chunks_x) * RED_THREADS + threadIdx.x;
        if (xx >= 1 && xx <= nx - 2 && y >= 1 && y <= ny - 2) {
            const double *q = p + (size_t)y * pitch + xx;
            const double t = dsub(dsub(dsub(dsub(dmul(4.0, q[0]), q[-1]), q[1]), q[-pitch]), q[pitch]);
            const double v = __ddiv_rn(t, h2);
            ap[(size_t)y * pitch + xx] = v;
            acc = dadd(acc, dmul(q[0], v));
        }
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// partial sums of a . b over the interior
__global__ void __launch_bounds__(RED_THREADS)
    k_dot_interior(const double *__restrict__ a, const double *__restrict__ b, int nx, int ny, int pitch,
                   double *__restrict__ partials)
{
    double acc = 0.0;
    const int chunks_x = (nx + RED_THREADS - 1) / RED_THREADS;
    for (long c = blockIdx.x; c < (long)chunks_x * ny; c += gridDim.x) {
        const int y = (int)(c / chunks_x), xx = (int)(c % chunks_x) * RED_THREADS + threadIdx.x;
        if (xx >= 1 && xx <= nx - 2 && y >= 1 && y <= ny - 2)
            acc = dadd(acc, dmul(a[(size_t)y * pitch + xx], b[(size_t)y * pitch + xx]));
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// x += alpha p ; r -= alpha ap ; partial sums of r . r
__global__ void __launch_bounds__(RED_THREADS)
    k_pcg_update(double *__restrict__ x, double *__restrict__ r, const double *__restrict__ p, const double *__restrict__ ap,
                 int nx, int ny, int pitch, double alpha, double *__restrict__ partials)
{
    double acc = 0.0;
    const int chunks_x = (nx + RED_THREADS - 1) / RED_THREADS;
    for (long c = blockIdx.x; c < (long)chunks_x * ny; c += gridDim.x) {
        const int y = (int)(c / chunks_x), xx = (int)(c % chunks_x) * RED_THREADS + threadIdx.x;
        if (xx >= 1 && xx <= nx - 2 && y >= 1 && y <= ny - 2) {
            const size_t i = (size_t)y * pitch + xx;
            x[i] = dadd(x[i], dmul(alpha, p[i]));
            const double rv = dsub(r[i], dmul(alpha, ap[i]));
            r[i] = rv;
            acc = dadd(acc, dmul(rv, rv));
        }
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// p = z + beta p  (beta == 0 with first == 1: p = z)
__global__ void __launch_bounds__(BX *BY)
    k_pcg_direction(double *__restrict__ p, const double *__restrict__ z, int nx, int ny, int pitch, double beta, int first)
{
    const int xx = blockIdx.x * BX + threadIdx.x, y = blockIdx.y * BY + threadIdx.y;
    if (xx < 1 || xx > nx - 2 || y < 1 || y > ny - 2) return;
    const size_t i = (size_t)y * pitch + xx;
    p[i] = first ? z[i] : dadd(z[i], dmul(beta, p[i]));
}

// ---- NVLink peer-to-peer halo exchange ----------------------------------------------------------------------
__global__ void k_halo_signal(int *up_flag, int *dn_flag, int epoch)
{
    // everything this stream ran before is complete; make it visible system-wide, then publish
    __threadfence_system();
    if (up_flag) asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(up_flag), "r"(epoch) : "memory");
    if (dn_flag) asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(dn_flag), "r"(epoch) : "memory");
}

// blockIdx.y: 0 = rows from the upper neighbour into my rows [-depth, 0), 1 = from the lower into [ny, ny+depth)
__global__ void __launch_bounds__(256)
    k_halo_pull(double *__restrict__ mine, int ny, int pitch, int depth, const double *__restrict__ up_src,
                const double *__restrict__ dn_src, const int *flag_from_up, const int *flag_from_dn, int epoch,
                int *err, int *abort)
{
    const bool from_up = blockIdx.y == 0;
    const double *src = from_up ? up_src : dn_src;
    if (src == nullptr) return;
    __shared__ int ok;
    if (threadIdx.x == 0) ok = wait_flag(from_up ? flag_from_up : flag_from_dn, epoch) ? 1 : 0;
    __syncthreads();
    if (!ok) {
        if (threadIdx.x == 0) {
            *err = 1;
            if (abort != nullptr) *abort = 1;
        }
        return;
    }
    // whole padded rows, 16 bytes per thread per step (row starts are 128-byte aligned)
    double *dst = mine - PADX + (ptrdiff_t)(from_up ? -depth : ny) * pitch;
    const double2 *s2 = reinterpret_cast<const double2 *>(src - PADX);
    double2 *d2 = reinterpret_cast<double2 *>(dst);
    const size_t n2 = (size_t)depth * pitch / 2;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) {
        double2 v;
        asm volatile("ld.global.cv.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(s2 + i));
        d2[i] = v;
    }
}

__global__ void k_signal_all(int *const *slots, int n_ranks, int my_rank, int epoch)
{
    __threadfence_system();
    int r = threadIdx.x;
    if (r < n_ranks && r != my_rank)
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(slots[r]), "r"(epoch) : "memory");
}

constexpr int GATHER_ILP = 4;
// blockIdx.y = source rank
__global__ void __launch_bounds__(256)
    k_gather_pull(double *__restrict__ full, int pitch, int rows, const double *const *__restrict__ srcs,
                  const int *inbox, int my_rank, int epoch, int *err, int *const *slots, int n_ranks,
                  const int *__restrict__ epoch_base, int *abort)
{
    pdl_prologue();
    const int r = blockIdx.y;
    if (epoch_base != nullptr) epoch += *epoch_base;
    // "my slab is final" (everything this stream ran before this launch is complete): published by the first block
    if (slots != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && (int)threadIdx.x < n_ranks &&
        (int)threadIdx.x != my_rank) {
        __threadfence_system();
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(slots[threadIdx.x]), "r"(epoch) : "memory");
    }
    __shared__ int ok;
    if (threadIdx.x == 0) ok = (r == my_rank) ? 1 : (wait_flag(inbox + r, epoch) ? 1 : 0);
    __syncthreads();
    if (!ok) {
        if (threadIdx.x == 0) {
            *err = 1;
            if (abort != nullptr) *abort = 1;
        }
        return;
    }
    // a remote load costs an NVLink round trip (~2-3 us): keep GATHER_ILP independent loads in flight per thread
    // and enough blocks (launch_gather_pull) that every thread makes one or two trips, not twenty
    const size_t n2 = (size_t)rows * pitch / 2;
    const double2 *s2 = reinterpret_cast<const double2 *>(srcs[r]);
    double2 *d2 = reinterpret_cast<double2 *>(full - PADX + (size_t)r * rows * pitch);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += GATHER_ILP * stride) {
        double2 v[GATHER_ILP];
#pragma unroll
        for (int u = 0; u < GATHER_ILP; ++u)
            if (i + u * stride < n2)
                asm volatile("ld.global.cv.v2.f64 {%0, %1}, [%2];" : "=d"(v[u].x), "=d"(v[u].y) : "l"(s2 + i + u * stride));
#pragma unroll
        for (int u = 0; u < GATHER_ILP; ++u)
            if (i + u * stride < n2) d2[i + u * stride] = v[u];
    }
}

inline JacobiCoef make_coef(double h, double omega)
{
    JacobiCoef c;
    c.h2 = h * h;
    c.omega = omega;
    c.om1 = 1.0 - omega;
    c.w4 = 0.25 * omega;
    c.weighted = (omega != 1.0);
    return c;
}

}  // namespace

JacobiCoef jacobi_coef(double h, double omega) { return make_coef(h, omega); }

void launch_jacobi_sweep(double *out, const double *in, const double *f, int nx, int ny, int pitch_x,
                         int pitch_f, double h, double omega, cudaStream_t st)
{
    k_jacobi_sweep<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(out, in, f, nx, ny, pitch_x, pitch_f,
                                                            make_coef(h, omega));
    count_launch();
}

void launch_jacobi_small(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                         double omega, int sweeps, bool x_is_zero, cudaStream_t st, const int *done)
{
    int l = nx * ny;
    int threads = l >= 1024 ? 1024 : ((l + 31) / 32) * 32;
    launch_pdl(k_jacobi_small, dim3(1), dim3(threads), 0, st, x, f, nx, ny, pitch_x, pitch_f, make_coef(h, omega), sweeps, x_is_zero ? 1 : 0, done);
    count_launch();
}

size_t vcycle_small_smem(int n0, int n_coarse)
{
    size_t d = 0;
    for (int m = n0, k = 0; k < 8; ++k) {
        d += 3 * (size_t)m * m;
        if (m <= n_coarse || m <= 3) break;
        m = (m - 1) / 2 + 1;
    }
    return d * sizeof(double);
}

// which generation of the single-CTA small-level kernel runs: 1 = k_vcycle_small (this file), 2 = k_vcycle_small2
// (kernels_small.cu: per-level thread groups on named barriers), 3 = k_coarse_local (kernels_coarse.cu: level sizes
// as template parameters, one-warp deep levels; the default).  PMG_SMALL_VERSION=1/2/3 overrides the default
// (PMG_SMALL_V2=0/1 is the round-1 spelling of 1/2).
static int g_small_version = 0;
int vcycle_small_version()
{
    if (g_small_version == 0) {
        g_small_version = PMG_SMALL_DEFAULT_VERSION;
        if (const char *e = getenv("PMG_SMALL_V2")) g_small_version = (e[0] == '1') ? 2 : ((e[0] == '0') ? 1 : g_small_version);
        if (const char *e = getenv("PMG_SMALL_VERSION"))
            if (e[0] >= '1' && e[0] <= '3') g_small_version = e[0] - '0';
    }
    return g_small_version;
}
void vcycle_small_set_version(int v) { g_small_version = (v >= 1 && v <= 3) ? v : 0; }

void launch_vcycle_small(double *x, const double *f, int n0, int pitch_x, int pitch_f, int n_coarse, double h0,
                         double omega, int nu1, int nu2, int coarse_sweeps, int prolong_mode, bool x_is_zero,
                         int gamma, cudaStream_t st, const int *done)
{
    if (vcycle_small_version() == 3 && coarse_local_supported(n0, gamma)) {
        launch_coarse_local(x, f, n0, pitch_x, pitch_f, n_coarse, h0, omega, nu1, nu2, coarse_sweeps, prolong_mode, x_is_zero,
                            gamma, st, done);
        return;
    }
    if (vcycle_small_version() >= 2 && vcycle_small_v2_supported(gamma)) {
        launch_vcycle_small_v2(x, f, n0, pitch_x, pitch_f, n_coarse, h0, omega, nu1, nu2, coarse_sweeps, prolong_mode,
                               x_is_zero, gamma, st, done);
        return;
    }
    size_t smem = vcycle_small_smem(n0, n_coarse);
    static unsigned long long smem_mask = 0;  // per-device attribute: once per device ordinal
    {
        int dev = 0;
        cudaGetDevice(&dev);
        if (!((smem_mask >> (dev & 63)) & 1ull)) {
            cudaFuncSetAttribute(k_vcycle_small, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            smem_mask |= 1ull << (dev & 63);
        }
    }
    const int threads = n0 > 33 ? 1024 : (n0 > 17 ? 512 : 256);
    launch_pdl(k_vcycle_small, dim3(1), dim3(threads), smem, st, x, f, n0, pitch_x, pitch_f, n_coarse, h0, omega, nu1, nu2, coarse_sweeps,
                                            prolong_mode == PMG_PROLONG_FULL ? 1 : 2, x_is_zero ? 1 : 0, gamma < 1 ? 1 : gamma, done);
    count_launch();
}

void launch_residual(double *r, const double *x, const double *f, int nx, int ny, int pitch_r, int pitch_x,
                     int pitch_f, double h, cudaStream_t st)
{
    k_residual<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(r, x, f, nx, ny, pitch_r, pitch_x, pitch_f,
                                                        1.0 / (h * h));
    count_launch();
}

int reduce_partials() { return RED_BLOCKS; }

void launch_final_sum(const double *d_partials, int count, double *d_out, cudaStream_t st)
{
    launch_pdl(k_final_sum, dim3(1), dim3(1024), 0, st, d_partials, count, d_out);
    count_launch();
}

void launch_solve_begin(const double *d_norm2, SolveCtrl *ctrl, double *hist2, double rel_tol, int max_cycles,
                        cudaStream_t st)
{
    k_solve_begin<<<1, 1, 0, st>>>(d_norm2, ctrl, hist2, rel_tol, max_cycles);
    count_launch();
}

void launch_ctrl_to_host(const SolveCtrl *ctrl, SolveCtrl *host_ctrl, const double *hist2, double *host_hist, int hist_cap,
                         cudaStream_t st)
{
    launch_pdl(k_ctrl_to_host, dim3(1), dim3(host_hist ? 1024 : 32), 0, st, ctrl, host_ctrl, hist2, host_hist, hist_cap);
    count_launch();
}

void launch_cycle_finish(const double *d_partials, int count, SolveCtrl *ctrl, double *hist2, cudaStream_t st)
{
    launch_pdl(k_cycle_finish, dim3(1), dim3(1024), 0, st, d_partials, count, ctrl, hist2);
    count_launch();
}

int launch_residual_partials(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                             double *d_partials, cudaStream_t st)
{
    long chunks = (long)((nx + RED_THREADS - 1) / RED_THREADS) * ny;
    int blocks = (int)(chunks < RED_BLOCKS ? chunks : RED_BLOCKS);
    if (blocks < 1) blocks = 1;
    k_residual_norm2<<<blocks, RED_THREADS, 0, st>>>(x, f, nx, ny, pitch_x, pitch_f, 1.0 / (h * h), d_partials);
    count_launch();
    return blocks;
}

void launch_residual_norm2(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f,
                           double h, double *d_partials, double *d_out, cudaStream_t st)
{
    const int blocks = launch_residual_partials(x, f, nx, ny, pitch_x, pitch_f, h, d_partials, st);
    launch_final_sum(d_partials, blocks, d_out, st);
}

void launch_halo_signal(int *up_flag, int *dn_flag, int epoch, cudaStream_t st)
{
    k_halo_signal<<<1, 1, 0, st>>>(up_flag, dn_flag, epoch);
    count_launch();
}

void launch_halo_pull(double *mine, int ny, int pitch, int depth, const double *up_src, const double *dn_src,
                      const int *flag_from_up, const int *flag_from_dn, int epoch, int *err, cudaStream_t st, int *abort)
{
    size_t n2 = (size_t)depth * pitch / 2;
    int bx = (int)((n2 + 255) / 256);
    if (bx > 64) bx = 64;
    if (bx < 1) bx = 1;
    k_halo_pull<<<dim3(bx, 2), 256, 0, st>>>(mine, ny, pitch, depth, up_src, dn_src, flag_from_up, flag_from_dn, epoch, err, abort);
    count_launch();
}

__global__ void k_set_ints(int *dst, IntPack16 vals, int count)
{
    pdl_prologue();
    if ((int)threadIdx.x < count) dst[threadIdx.x] = vals.v[threadIdx.x];
}

void launch_set_ints(int *dst, const IntPack16 &vals, int count, cudaStream_t st)
{
    launch_pdl(k_set_ints, dim3(1), dim3(32), 0, st, dst, vals, count < 16 ? count : 16);
    count_launch();
}

void launch_signal_all(int *const *slots, int n_ranks, int my_rank, int epoch, cudaStream_t st)
{
    k_signal_all<<<1, 32, 0, st>>>(slots, n_ranks, my_rank, epoch);
    count_launch();
}

void launch_gather_pull(double *full, int pitch, int rows, const double *const *srcs, const int *inbox, int n_ranks,
                        int my_rank, int epoch, int *err, cudaStream_t st, int *const *slots, const int *epoch_base,
                        int *abort)
{
    size_t n2 = (size_t)rows * pitch / 2;
    int bx = (int)((n2 + 256 * GATHER_ILP - 1) / (256 * GATHER_ILP));  // one trip per thread ...
    int cap = (148 * 4) / (n_ranks > 0 ? n_ranks : 1);                   // ... within about one wave of CTAs
    if (cap < 16) cap = 16;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    launch_pdl(k_gather_pull, dim3(bx, n_ranks), dim3(256), 0, st, full, pitch, rows, srcs, inbox, my_rank, epoch, err, slots, n_ranks,
                                                     epoch_base, abort);
    count_launch();
}

static int g_pdl = -1;
bool pdl_enabled()
{
    if (g_pdl < 0) {
        const char *e = getenv("PMG_PDL");
        g_pdl = (e && e[0] == '0') ? 0 : 1;
    }
    return g_pdl == 1;
}
void pdl_set_enabled(int on) { g_pdl = on ? 1 : 0; }

void basic_set_wait_timeout_ns(unsigned long long ns) { cudaMemcpyToSymbol(g_wait_timeout_ns, &ns, sizeof(ns)); }

void launch_residual_norm2_sequential(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f,
                                      double h, double *d_out, cudaStream_t st)
{
    k_residual_norm2_seq<<<1, 1024, 0, st>>>(x, f, nx, ny, pitch_x, pitch_f, 1.0 / (h * h), d_out);
    count_launch();
}

void launch_norm2(const double *v, size_t l, double *d_partials, double *d_out, cudaStream_t st)
{
    size_t want = (l + RED_THREADS - 1) / RED_THREADS;
    int blocks = (int)(want < (size_t)RED_BLOCKS ? want : (size_t)RED_BLOCKS);
    if (blocks < 1) blocks = 1;
    k_norm2<<<blocks, RED_THREADS, 0, st>>>(v, l, d_partials);
    count_launch();
    launch_final_sum(d_partials, blocks, d_out, st);
}

void launch_jacobi_sweep_f32(double *out, const double *in, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                             double omega, cudaStream_t st)
{
    k_jacobi_sweep_f32<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(out, in, f, nx, ny, pitch_x, pitch_f, (float)(h * h),
                                                                  (float)omega, (float)(1.0 - omega), omega != 1.0 ? 1 : 0);
    count_launch();
}

// d_out[0] = sum (a - b)^2, d_out[1] = sum b^2 ; d_partials: 2 * reduce_partials() doubles
void launch_diff_norm2(const double *a, const double *b, size_t l, double *d_partials, double *d_out, cudaStream_t st)
{
    size_t want = (l + RED_THREADS - 1) / RED_THREADS;
    int blocks = (int)(want < (size_t)RED_BLOCKS ? want : (size_t)RED_BLOCKS);
    if (blocks < 1) blocks = 1;
    k_diff_norm2<<<blocks, RED_THREADS, 0, st>>>(a, b, l, d_partials, d_partials + RED_BLOCKS);
    count_launch();
    launch_final_sum(d_partials, blocks, d_out, st);
    launch_final_sum(d_partials + RED_BLOCKS, blocks, d_out + 1, st);
}

void launch_rbgs_half(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h, int colour,
                      cudaStream_t st)
{
    k_rbgs_half<<<grid2d((nx + 1) / 2 + 1, ny), dim3(BX, BY), 0, st>>>(x, f, nx, ny, pitch_x, pitch_f, h * h, colour);
    count_launch();
}

void launch_gs_lex(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h, int sweeps, cudaStream_t st)
{
    if (sweeps <= 0) return;
    int threads = ((min(nx, ny) + 31) / 32) * 32;
    threads = threads < 32 ? 32 : (threads > 1024 ? 1024 : threads);
    k_gs_lex<<<1, threads, 0, st>>>(x, f, nx, ny, pitch_x, pitch_f, h * h, sweeps);
    count_launch();
}

static int red_blocks_for(int nx, int ny)
{
    long chunks = (long)((nx + RED_THREADS - 1) / RED_THREADS) * ny;
    int blocks = (int)(chunks < RED_BLOCKS ? chunks : RED_BLOCKS);
    return blocks < 1 ? 1 : blocks;
}

void launch_apply_a_dot(const double *p, double *ap, int nx, int ny, int pitch, double h, double *d_partials, double *d_out,
                        cudaStream_t st)
{
    const int blocks = red_blocks_for(nx, ny);
    k_apply_a_dot<<<blocks, RED_THREADS, 0, st>>>(p, ap, nx, ny, pitch, h * h, d_partials);
    count_launch();
    launch_final_sum(d_partials, blocks, d_out, st);
}

void launch_dot_interior(const double *a, const double *b, int nx, int ny, int pitch, double *d_partials, double *d_out,
                         cudaStream_t st)
{
    const int blocks = red_blocks_for(nx, ny);
    k_dot_interior<<<blocks, RED_THREADS, 0, st>>>(a, b, nx, ny, pitch, d_partials);
    count_launch();
    launch_final_sum(d_partials, blocks, d_out, st);
}

void launch_pcg_update(double *x, double *r, const double *p, const double *ap, int nx, int ny, int pitch, double alpha,
                       double *d_partials, double *d_out, cudaStream_t st)
{
    const int blocks = red_blocks_for(nx, ny);
    k_pcg_update<<<blocks, RED_THREADS, 0, st>>>(x, r, p, ap, nx, ny, pitch, alpha, d_partials);
    count_launch();
    launch_final_sum(d_partials, blocks, d_out, st);
}

void launch_pcg_direction(double *p, const double *z, int nx, int ny, int pitch, double beta, bool first, cudaStream_t st)
{
    k_pcg_direction<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(p, z, nx, ny, pitch, beta, first ? 1 : 0);
    count_launch();
}

int launch_pcg_direction_apply(const double *z, const double *p_in, double *p_out, double *ap, int n, int rows, int yoff, int pitch,
                               double h, const double *beta_num, const double *beta_den, bool first, double *d_partials,
                               cudaStream_t st)
{
    const PDGeom g = pcg_geom(n, rows, yoff);
    if (g.blocks < 1) return 0;
    k_pcg_direction_apply<<<g.blocks, PD_WARPS * 32, 0, st>>>(z, p_in, p_out, ap, n, yoff, g, pitch, h * h, beta_num, beta_den,
                                                             first ? 1 : 0, d_partials);
    count_launch();
    return pcg_partials(g);
}

int launch_pcg_update_dev(double *x, double *r, const double *p, const double *ap, int n, int rows, int yoff, int pitch,
                          const double *alpha_num, const double *alpha_den, double *d_partials, cudaStream_t st)
{
    const PDGeom g = pcg_geom(n, rows, yoff);
    if (g.blocks < 1) return 0;
    k_pcg_update_dev<<<g.blocks, PD_WARPS * 32, 0, st>>>(x, r, p, ap, n, g, pitch, alpha_num, alpha_den, d_partials);
    count_launch();
    return pcg_partials(g);
}

void launch_restrict(const double *fine, double *coarse, int nf, int nc, int pitch_f, int pitch_c, cudaStream_t st)
{
    (void)nf;
    k_restrict<<<grid2d(nc, nc), dim3(BX, BY), 0, st>>>(fine, coarse, nc, nc, 0, pitch_f, pitch_c);
    count_launch();
}

void launch_residual_restrict(const double *x, const double *f, double *coarse, int nf, int nc, int rows_c, int yoff_c,
                              int pitch_x, int pitch_f, int pitch_c, double h, cudaStream_t st)
{
    (void)nf;
    const RRGeom g = residual_restrict_geom(nc, rows_c, yoff_c);
    if (g.blocks < 1) return;
    k_residual_restrict<<<g.blocks, RR_WARPS * 32, 0, st>>>(x, f, coarse, nc, g, pitch_x, pitch_f, pitch_c, 1.0 / (h * h));
    count_launch();
}

void launch_restrict_rows(const double *fine, double *coarse, int nc, int rows_c, int yoff_c, int pitch_f,
                          int pitch_c, cudaStream_t st)
{
    if (rows_c < 1) return;
    k_restrict<<<grid2d(nc, rows_c), dim3(BX, BY), 0, st>>>(fine, coarse, nc, rows_c, yoff_c, pitch_f, pitch_c);
    count_launch();
}

void launch_prolong_add(const double *coarse, double *fine, int nc, int nf, int pitch_c, int pitch_f, int mode,
                        cudaStream_t st)
{
    (void)nc;
    k_prolong_add<<<grid2d(nf, nf), dim3(BX, BY), 0, st>>>(coarse, fine, nf, nf, 0, pitch_c, pitch_f,
                                                           mode == PMG_PROLONG_FULL ? 1 : 2);
    count_launch();
}

void launch_prolong_add_rows(const double *coarse, double *fine, int nf, int rows_f, int yoff_f, int pitch_c,
                             int pitch_f, int mode, cudaStream_t st)
{
    if (rows_f < 1) return;
    k_prolong_add<<<grid2d(nf, rows_f), dim3(BX, BY), 0, st>>>(coarse, fine, nf, rows_f, yoff_f, pitch_c, pitch_f,
                                                               mode == PMG_PROLONG_FULL ? 1 : 2);
    count_launch();
}

void launch_copy2d(double *dst, int pitch_d, const double *src, int pitch_s, int nx, int ny, cudaStream_t st)
{
    k_copy2d<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(dst, pitch_d, src, pitch_s, nx, ny);
    count_launch();
}

void launch_fill2d(double *dst, int pitch_d, int nx, int ny, double v, cudaStream_t st)
{
    k_fill2d<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(dst, pitch_d, nx, ny, v);
    count_launch();
}

void launch_rhs_separable(double *f, int pitch, int nx, int ny, double factor, const double *sx,
                          const double *sy, cudaStream_t st)
{
    k_rhs_separable<<<grid2d(nx, ny), dim3(BX, BY), 0, st>>>(f, pitch, nx, ny, factor, sx, sy);
    count_launch();
}

}  // namespace pmg
