// test_pcg_emu.cpp -- the fused direction-operator pass of pmg_pcg on row slabs (k_pcg_direction_apply,
// csrc/kernel_pcg.cuh) run from the kernel source on the CPU (tests/cpp/emu/host_emulation.h) and compared with the direction
// update of the oracle's orc_pcg (p = z + beta p, or p = z on the first step) followed by its apply_laplacian expression
// (oracle/pmg_oracle_smoothers.c: apply_a):
//   * whole levels n = 5 .. 1025;
//   * row-slab windows of 2, 4 and 8 ranks (pmg_partition_rows), every z and p row more than 1 row beyond the owned rows
//     NaN, and the Dirichlet ring of z and p NaN -- a deeper read or a read of the ring shows up as a NaN in the output;
//   * first = 0 and 1.
// p and A p must be bit-identical to the oracle's on every point the pass owns (the owned interior rows, plus the interior
// rows next to a neighbour's slab for p), every other element of the output arrays -- ring, padding, other rows -- must
// keep all-zero bits, the inputs must keep their bits, and the partial sums must add up to p . A p (compensated sum of the
// rounded products) within 1e-14 relative.
#include <cmath>
#include <cstring>
#include <random>
#include <vector>

#include "../../parallel-geometric-multigrid-for-poisson-problem_b200/csrc/kernel_pcg.cuh"

using namespace pmg;

static int g_bad = 0;
static std::mt19937_64 g_rng(90210);
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

// the window of a dense n x n field: global rows [y0 - depth, y1 + depth) within the grid copied (padding columns zero,
// Dirichlet ring NaN), every other row of the window NaN from end to end
static Window cut(const std::vector<double> &d, int n, int y0, int y1, int depth)
{
    Window w(n, y1 - y0, y0, std::nan(""));
    for (int lr = -PADY; lr < (y1 - y0) + PADY; ++lr) {
        const int g = y0 + lr;
        if (g < y0 - depth || g >= y1 + depth || g < 0 || g >= n) continue;
        double *q = w.row(lr);
        for (int x = -PADX; x < w.pitch - PADX; ++x) q[x] = 0.0;
        std::memcpy(q, d.data() + (size_t)g * n, (size_t)n * 8);
        if (g == 0 || g == n - 1)
            for (int x = 0; x < n; ++x) q[x] = std::nan("");
        q[0] = q[n - 1] = std::nan("");
    }
    return w;
}

struct Case {
    std::vector<double> z, p_old, p, ap;
    double num, den, dot;
};

// z, p_old random with a zero ring; the oracle's direction update and A p, and p . A p
static Case make_case(int n, bool first)
{
    Case c;
    c.z.assign((size_t)n * n, 0.0);
    c.p_old.assign((size_t)n * n, 0.0);
    for (int y = 1; y < n - 1; ++y)
        for (int i = 1; i < n - 1; ++i) {
            c.z[(size_t)y * n + i] = rnd();
            c.p_old[(size_t)y * n + i] = rnd();
        }
    c.num = 0.5 + 0.5 * std::fabs(rnd());
    c.den = 0.5 + 0.5 * std::fabs(rnd());
    const double beta = c.num / c.den;
    c.p.assign((size_t)n * n, 0.0);
    c.ap.assign((size_t)n * n, 0.0);
    for (int y = 1; y < n - 1; ++y)  // orc_pcg: memcpy(p, z) on the first step, else p[i] = z[i] + beta * p[i]
        for (int i = 1; i < n - 1; ++i) {
            const size_t k = (size_t)y * n + i;
            c.p[k] = first ? c.z[k] : c.z[k] + beta * c.p_old[k];
        }
    const double h = 1.0 / (n - 1);
    const int width = n;
    const double *p = c.p.data();
    for (int y = 1; y < n - 1; ++y)  // apply_a, statement for statement
        for (int xp = 1; xp < width - 1; ++xp) {
            long i = (long)y * width + xp;
            c.ap[i] = (4 * p[i] - p[i - 1] - p[i + 1] - p[i - width] - p[i + width]) / (h * h);
        }
    // the sum of the rounded products p[i] * ap[i], compensated (Neumaier): the exactly rounded total to well below 1e-14
    double s = 0.0, comp = 0.0;
    for (size_t i = 0; i < c.p.size(); ++i) {
        const double t = c.p[i] * c.ap[i], u = s + t;
        comp += std::fabs(s) >= std::fabs(t) ? (s - u) + t : (t - u) + s;
        s = u;
    }
    c.dot = s + comp;
    return c;
}

// runs the kernel on one window; returns the sum of its partials
static double run_kernel(Window &z, Window &pin, Window &pout, Window &ap, int n, bool first, double num, double den)
{
    const PDGeom g = pcg_geom(n, z.rows, z.y0);
    if (g.blocks < 1) return 0.0;
    std::vector<double> part(PD_MAX_WARPS, std::nan(""));
    const double h = 1.0 / (n - 1);
    emu_launch_warps(dim3(g.blocks), dim3(PD_WARPS * 32), [&] {
        k_pcg_direction_apply(z.p(), pin.p(), pout.p(), ap.p(), n, z.y0, g, z.pitch, h * h, &num, &den, first ? 1 : 0,
                              part.data());
    });
    double s = 0.0;
    for (int i = 0; i < pcg_partials(g); ++i) s += part[i];
    return s;
}

// p_out: interior points of the owned rows and of the interior rows next to a neighbour (lo / hi) equal `want`;
// ap: interior points of the owned rows; everything else zero bits
static bool check_out(Window &w, int n, const std::vector<double> &want, bool lo, bool hi)
{
    bool ok = true;
    for (int lr = -PADY; lr < w.rows + PADY; ++lr) {
        const int g = w.y0 + lr;
        const double *q = w.row(lr);
        const bool row = (lr >= 0 && lr < w.rows) || (lo && lr == -1) || (hi && lr == w.rows);
        for (int x = -PADX; x < w.pitch - PADX; ++x) {
            const bool owned = row && g >= 1 && g <= n - 2 && x >= 1 && x <= n - 2;
            ok = ok && same_bits(q[x], owned ? want[(size_t)g * n + x] : 0.0);
        }
    }
    return ok;
}

static bool run_windows(int n, int ranks, bool first, int depth)
{
    const Case c = make_case(n, first);
    bool ok = true;
    double total = 0.0;
    for (int r = 0; r < ranks; ++r) {
        int y0, y1;
        if (ranks == 1) {
            y0 = 0;
            y1 = n;
        } else {
            partition(n, ranks, r, y0, y1);
        }
        const int d = ranks == 1 ? 0 : depth;
        Window z = cut(c.z, n, y0, y1, d), pin = cut(c.p_old, n, y0, y1, d);
        Window pout(n, y1 - y0, y0, 0.0), ap(n, y1 - y0, y0, 0.0);
        const std::vector<double> z0 = z.base, p0 = pin.base;
        total += run_kernel(z, pin, pout, ap, n, first, c.num, c.den);
        const bool good = check_out(pout, n, c.p, r > 0, r < ranks - 1) && check_out(ap, n, c.ap, false, false) &&
                          std::memcmp(z.base.data(), z0.data(), z0.size() * 8) == 0 &&
                          std::memcmp(pin.base.data(), p0.data(), p0.size() * 8) == 0;
        if (!good) std::printf("  MISMATCH: rank %d of %d (n=%d, rows %d..%d)\n", r, ranks, n, y0, y1);
        ok = ok && good;
    }
    const double rel = std::fabs(total - c.dot) / std::fabs(c.dot);
    if (!(rel <= 1e-14)) {
        std::printf("  MISMATCH: partial sums %.17g vs %.17g (rel %.2e)\n", total, c.dot, rel);
        ok = false;
    }
    return ok;
}

static void report(const char *what, int n, int ranks, bool first, bool ok)
{
    if (!ok) ++g_bad;
    std::printf("%s n=%d ranks=%d first=%d: %s\n", what, n, ranks, first ? 1 : 0, ok ? "ok" : "MISMATCH");
    std::fflush(stdout);
}

int main()
{
    int runs = 0;
    for (int first : {1, 0}) {
        for (int n : {5, 9, 17, 33, 65, 129, 257, 513, 1025}) {
            report("whole level", n, 1, first, run_windows(n, 1, first, 0));
            ++runs;
        }
        for (int ranks : {2, 4, 8})
            for (int n : {129, 257, 513}) {
                report("slabs", n, ranks, first, run_windows(n, ranks, first, 1));
                ++runs;
            }
    }
    std::printf(g_bad ? "FAILED (%d)\n" : "all bit-identical (%d runs)\n", g_bad ? g_bad : runs);
    return g_bad ? 1 : 0;
}
