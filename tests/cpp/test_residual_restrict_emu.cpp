// test_residual_restrict_emu.cpp -- the fused residual-restriction of the FMG set-up (k_residual_restrict,
// csrc/kernel_residual_restrict.cuh) run from the kernel source on the CPU (tests/cpp/emu/host_emulation.h) and compared BIT
// FOR BIT with the CPU oracle's residual followed by its full-weighting restriction:
//   * whole levels n = 5 .. 1025;
//   * row-slab windows of 2, 4 and 8 ranks (pmg_partition_rows), every x row more than 2 rows and every f row more than 1
//     row beyond the owned rows NaN -- a deeper read shows up as a NaN in the output;
//   * an f with -0.0 and +-1e100 entries over patches of zero iterate (signed zeros reach the restriction).
// Every element of the coarse array other than the interior points of the window -- the ring, rows of other ranks and the
// padding -- must stay all-zero bits, and the inputs must keep their bits.
#include <cmath>
#include <cstring>
#include <random>
#include <vector>

#include "../../parallel-geometric-multigrid-for-poisson-problem_b200/csrc/kernel_residual_restrict.cuh"
#include "../../oracle/oracle.h"

using namespace pmg;

static int g_bad = 0;
static std::mt19937_64 g_rng(4711);
static double rnd() { return std::uniform_real_distribution<double>(-1.0, 1.0)(g_rng); }
static bool same_bits(double a, double b) { return std::memcmp(&a, &b, 8) == 0; }

// a window of rows [-PADY, rows + PADY) in the solver's padded layout; local row 0 = global row y0
struct Window {
    int n, rows, y0, pitch;
    std::vector<double> base;
    Window(int n_, int rows_, int y0_, double fill)
        : n(n_), rows(rows_), y0(y0_), pitch(level_pitch(n_)), base((size_t)level_pitch(n_) * (rows_ + 2 * PADY), fill) {}
    double *p() { return base.data() + (size_t)PADY * pitch + PADX; }
    double *row(int local) { return p() + (ptrdiff_t)local * pitch; }
};

static void partition(int n, int ranks, int r, int &y0, int &y1)  // pmg_partition_rows
{
    long pairs = (n - 1) / 2;
    long a = pairs * r / ranks, b = pairs * (r + 1) / ranks;
    y0 = (int)(2 * a);
    y1 = (r == ranks - 1) ? n : (int)(2 * b);
}

// the window of a dense n x n field: global rows [y0 - depth, y1 + depth) within the grid copied (padding columns zero),
// every other row of the window NaN from end to end
static Window cut(const std::vector<double> &d, int n, int y0, int y1, int depth)
{
    Window w(n, y1 - y0, y0, std::nan(""));
    for (int lr = -PADY; lr < (y1 - y0) + PADY; ++lr) {
        const int g = y0 + lr;
        if (g < y0 - depth || g >= y1 + depth || g < 0 || g >= n) continue;
        double *q = w.row(lr);
        for (int x = -PADX; x < w.pitch - PADX; ++x) q[x] = 0.0;
        std::memcpy(q, d.data() + (size_t)g * n, (size_t)n * 8);
    }
    return w;
}

static void run_kernel(Window &x, Window &f, Window &c, int nf, int nc, int rows_c, int yoff_c)
{
    const RRGeom g = residual_restrict_geom(nc, rows_c, yoff_c);
    if (g.blocks < 1) return;
    const double inv_h2 = 1.0 / ((1.0 / (nf - 1)) * (1.0 / (nf - 1)));
    emu_launch_warps(dim3(g.blocks), dim3(RR_WARPS * 32), [&] {
        k_residual_restrict(x.p(), f.p(), c.p(), nc, g, x.pitch, f.pitch, c.pitch, inv_h2);
    });
}

// x with a non-zero ring and zero patches, f with -0.0 / +-1e100 entries; the oracle's R(f - A x)
static void make_case(int n, std::vector<double> &x, std::vector<double> &f, std::vector<double> &want)
{
    const int nc = (n - 1) / 2 + 1;
    x.assign((size_t)n * n, 0.0);
    f.assign((size_t)n * n, 0.0);
    for (int y = 0; y < n; ++y)
        for (int i = 0; i < n; ++i) {
            const bool patch = ((y / 6) + (i / 6)) % 5 == 0;  // x == +0 around these points: residuals of +-0
            x[(size_t)y * n + i] = patch ? 0.0 : rnd();
            double v = rnd();
            const unsigned k = (unsigned)(g_rng() % 97);
            if (k == 0) v = 1e100;
            if (k == 1) v = -1e100;
            if (k < 12 && patch) v = -0.0;
            f[(size_t)y * n + i] = v;
        }
    std::vector<double> r((size_t)n * n, 0.0);
    want.assign((size_t)nc * nc, 0.0);
    orc_residual(r.data(), x.data(), f.data(), n, n, 1.0 / (n - 1));
    orc_restrict_fw(r.data(), want.data(), n, nc);
}

// coarse window: interior points of global rows [1, nc - 2] inside the window equal `want`, everything else zero bits
static bool check_coarse(Window &c, int nc, const std::vector<double> &want)
{
    bool ok = true;
    for (int lr = -PADY; lr < c.rows + PADY; ++lr) {
        const int g = c.y0 + lr;
        const double *q = c.row(lr);
        for (int x = -PADX; x < c.pitch - PADX; ++x) {
            const bool owned = lr >= 0 && lr < c.rows && g >= 1 && g <= nc - 2 && x >= 1 && x <= nc - 2;
            ok = ok && same_bits(q[x], owned ? want[(size_t)g * nc + x] : 0.0);
        }
    }
    return ok;
}

static void whole_level(int n)
{
    const int nc = (n - 1) / 2 + 1;
    std::vector<double> x, f, want;
    make_case(n, x, f, want);
    Window px = cut(x, n, 0, n, 0), pf = cut(f, n, 0, n, 0), pc(nc, nc, 0, 0.0);
    const std::vector<double> x0 = px.base, f0 = pf.base;
    run_kernel(px, pf, pc, n, nc, nc, 0);
    const bool ok = check_coarse(pc, nc, want) && std::memcmp(px.base.data(), x0.data(), x0.size() * 8) == 0 &&
                    std::memcmp(pf.base.data(), f0.data(), f0.size() * 8) == 0;
    if (!ok) ++g_bad;
    std::printf("whole level n=%d: %s\n", n, ok ? "ok" : "MISMATCH");
    std::fflush(stdout);
}

static void slabs(int n, int ranks)
{
    const int nc = (n - 1) / 2 + 1;
    std::vector<double> x, f, want;
    make_case(n, x, f, want);
    bool ok = true;
    for (int r = 0; r < ranks; ++r) {
        int y0, y1, c0, c1;
        partition(n, ranks, r, y0, y1);
        partition(nc, ranks, r, c0, c1);
        if (c0 * 2 != y0) {
            std::printf("  partition does not nest (n=%d, ranks=%d)\n", n, ranks);
            ++g_bad;
            return;
        }
        Window px = cut(x, n, y0, y1, 2), pf = cut(f, n, y0, y1, 1), pc(nc, c1 - c0, c0, 0.0);
        const std::vector<double> x0 = px.base, f0 = pf.base;
        run_kernel(px, pf, pc, n, nc, c1 - c0, c0);
        const bool good = check_coarse(pc, nc, want) && std::memcmp(px.base.data(), x0.data(), x0.size() * 8) == 0 &&
                          std::memcmp(pf.base.data(), f0.data(), f0.size() * 8) == 0;
        if (!good) std::printf("  MISMATCH: rank %d of %d (n=%d, rows %d..%d)\n", r, ranks, n, y0, y1);
        ok = ok && good;
    }
    if (!ok) ++g_bad;
    std::printf("slabs n=%d ranks=%d: %s\n", n, ranks, ok ? "ok" : "MISMATCH");
    std::fflush(stdout);
}

int main()
{
    int runs = 0;
    for (int n : {5, 9, 17, 33, 65, 129, 257, 513, 1025}) {
        whole_level(n);
        ++runs;
    }
    for (int ranks : {2, 4, 8})  // (3 ranks: the partition of a 2^k + 1 grid does not nest across levels)
        for (int n : {129, 257, 513}) {
            slabs(n, ranks);
            ++runs;
        }
    std::printf(g_bad ? "FAILED (%d)\n" : "all bit-identical (%d runs)\n", g_bad ? g_bad : runs);
    return g_bad ? 1 : 0;
}
