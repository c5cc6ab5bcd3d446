// test_up_exchange_emu.cpp -- Pass B with the coarse up-exchange prologue of the deep-sweep slab schedule (k_up with UPX,
// csrc/kernels_fused.cu, launched by launch_fused_up with lv.hp.x_keep set) run from the kernel source on the CPU
// (tests/cpp/emu/host_emulation.h: warps one after another in index order) on 2-4 row slabs side by side:
//   * xb holds the rows Pass A finished (pass_a_depth beyond the slab), NaN beyond;
//   * the coarse iterate holds its owned rows and the rows_from rows the child's Pass B finished, NaN beyond (zero padding
//     beyond the grid); the prologue must copy rows rows_from + 1 .. rows_from + rows_count from the neighbours' arrays
//     (flags pre-set) before any warp reads them -- a warp that reads a copied row without waiting and copying it itself
//     reads NaN here, because it runs before the warp that copies;
//   * every (nu1, nu2) with a 3 or 4, level 0 (own rows, fused norm where it fits) and coarser levels (pass_b_ext rows),
//     both prolongations, omega 2/3 and 1, 148 SMs (chunks of 4 rows: some chunk ends at ny - nu2 - norm) and 2 SMs.
// x must be bit-identical to the oracle's S^nu2(xb + P e) on the rows the pass finishes, nothing else of x may change,
// the coarse array must hold the exact rows the prologue copies and keep every other bit (padding included), the epoch
// must be published and no wait may fail.
#include <cmath>
#include <cstring>
#include <random>
#include <vector>

#include "../../parallel-geometric-multigrid-for-poisson-problem_b200/csrc/kernels_fused.cu"
#include "../../oracle/oracle.h"

namespace pmg {
void count_launch(int) {}
unsigned long long launches_so_far() { return 0; }
JacobiCoef jacobi_coef(double h, double omega)
{
    JacobiCoef c;
    c.h2 = h * h;
    c.omega = omega;
    c.om1 = 1.0 - omega;
    c.w4 = 0.25 * omega;
    c.weighted = (omega != 1.0);
    return c;
}
}  // namespace pmg

using namespace pmg;

static int g_bad = 0;
static int g_runs = 0;
static std::mt19937_64 g_rng(4242);
static double rnd() { return std::uniform_real_distribution<double>(-1.0, 1.0)(g_rng); }
static bool same_bits(double a, double b) { return std::memcmp(&a, &b, 8) == 0; }

static void check(bool ok, const char *what, int n, int a = 0, int b = 0)
{
    if (!ok) {
        std::printf("  MISMATCH: %s (n=%d, %d, %d)\n", what, n, a, b);
        ++g_bad;
    }
}

// the slab schedule's depths (csrc/solver.cu: pass_a_depth, pass_b_ext, pass_b_coarse_rows, up_exchange_rows)
static int pass_a_depth(int nu1) { return (PADY - nu1) & ~1; }
static int pass_b_ext(int nu1, int nu2, int l) { return l == 0 ? 0 : std::max(0, (pass_a_depth(nu1) - nu2) & ~1); }
static int coarse_rows_read(int nu1, int nu2, int l) { return (pass_b_ext(nu1, nu2, l) + nu2 + (l == 0 ? 1 : 0)) / 2 + 1; }

struct Dense {
    int n;
    std::vector<double> v;
    explicit Dense(int n_) : n(n_), v((size_t)n_ * n_, 0.0) {}
    double &at(int y, int x) { return v[(size_t)y * n + x]; }
    void randomize(bool ring)
    {
        for (int y = 0; y < n; ++y)
            for (int x = 0; x < n; ++x) at(y, x) = (ring || (y > 0 && y < n - 1 && x > 0 && x < n - 1)) ? rnd() : 0.0;
    }
};

// `rows` rows of an n-column level in the solver's padded layout: logical (0,0) at base[PADY * pitch + PADX]
struct Padded {
    int n, rows, pitch;
    std::vector<double> base;
    Padded(int n_, int rows_) : n(n_), rows(rows_), pitch(level_pitch(n_)), base((size_t)level_pitch(n_) * (rows_ + 2 * PADY), 0.0) {}
    double *p() { return base.data() + (size_t)PADY * pitch + PADX; }
    double &at(int y, int x) { return p()[(ptrdiff_t)y * pitch + x]; }
    // local rows [a, b): global rows of d where they exist, zero beyond the grid, `beyond` outside [lo, hi) (local)
    void fill(Dense &d, int y0, int lo, int hi, double beyond)
    {
        for (int y = -PADY; y < rows + PADY; ++y)
            for (int x = 0; x < n; ++x) {
                const int g = y + y0;
                at(y, x) = (g < 0 || g >= d.n) ? 0.0 : (y >= lo && y < hi ? d.at(g, x) : beyond);
            }
    }
    bool untouched_outside(const Padded &other, int a, int b) const
    {
        for (int r = -PADY; r < rows + PADY; ++r)
            for (int c = -PADX; c < pitch - PADX; ++c) {
                if (r >= a && r < b && c >= 0 && c < n) continue;
                size_t i = (size_t)(r + PADY) * pitch + PADX + c;
                if (std::memcmp(&base[i], &other.base[i], 8) != 0) return false;
            }
        return true;
    }
};

static void partition(int n, int ranks, int r, int &y0, int &y1)  // pmg_partition_rows
{
    long pairs = (n - 1) / 2;
    long a = pairs * r / ranks, b = pairs * (r + 1) / ranks;
    y0 = (int)(2 * a);
    y1 = (r == ranks - 1) ? n : (int)(2 * b);
}

struct Rank {
    int y0, y1, ny, yc0, yc1, nyc;
    Padded xb, f, e, x;
    int inbox[2];
    Rank(int n, int nc, int y0_, int y1_, int yc0_, int yc1_)
        : y0(y0_), y1(y1_), ny(y1_ - y0_), yc0(yc0_), yc1(yc1_), nyc(yc1_ - yc0_), xb(n, y1_ - y0_), f(n, y1_ - y0_),
          e(nc, yc1_ - yc0_), x(n, y1_ - y0_), inbox{0, 0} {}
};

static void up_exchange_pass(int n, int ranks, int nu1, int nu2, int level, int prolong, double omega, int sms)
{
    emu_num_sms = sms;
    fused_set_variant(-1);
    const int nc = (n - 1) / 2 + 1, epoch = 9;
    const double h = 1.0 / (n - 1);
    const double poison = std::nan("");
    const int da = pass_a_depth(nu1), ext = pass_b_ext(nu1, nu2, level), from = pass_b_ext(nu1, nu2, level + 1);
    const int count = std::max(1, coarse_rows_read(nu1, nu2, level) - from);
    const bool norm = level == 0 && nu2 + 1 <= da;
    Dense xb(n), f(n), e(nc);
    xb.randomize(level == 0);
    f.randomize(false);
    e.randomize(false);
    Dense want = xb;  // x = S^nu2(xb + P e) and its residual norm
    orc_prolong_add(want.v.data(), e.v.data(), n, nc, prolong);
    orc_jacobi(want.v.data(), f.v.data(), n, n, h, omega, nu2 - 1, 0.0, nullptr);
    Dense r2(n);
    orc_residual(r2.v.data(), want.v.data(), f.v.data(), n, n, h);
    const double nn = orc_norm(r2.v.data(), (long)n * n), norm2 = nn * nn;
    std::vector<Rank> R;
    for (int r = 0; r < ranks; ++r) {
        int y0, y1;
        partition(n, ranks, r, y0, y1);
        R.emplace_back(n, nc, y0, y1, y0 / 2, y1 == n ? nc : y1 / 2);
    }
    for (int r = 0; r < ranks; ++r) {
        Rank &K = R[r];
        const bool up = r > 0, dn = r < ranks - 1;
        K.xb.fill(xb, K.y0, up ? -da : 0, dn ? K.ny + da : K.ny, poison);  // what Pass A finished
        K.f.fill(f, K.y0, -PADY, K.ny + PADY, poison);                      // f halo local (level 0) or kept by Pass A
        K.e.fill(e, K.yc0, up ? -from : 0, dn ? K.nyc + from : K.nyc, poison);  // what the child's Pass B finished
        K.inbox[0] = K.inbox[1] = epoch;
    }
    std::vector<int> outbox(2 * ranks, 0);
    double s2 = 0.0;
    for (int r = 0; r < ranks; ++r) {
        Rank &K = R[r];
        const bool up = r > 0, dn = r < ranks - 1;
        Padded x0 = K.x, e0 = K.e;
        FusedLevel lv{};
        lv.x = K.x.p();
        lv.xb = K.xb.p();
        lv.f = K.f.p();
        lv.n = n;
        lv.pitch = K.x.pitch;
        lv.h = h;
        lv.ny = K.ny;
        lv.yoff = K.y0;
        lv.ext_lo = up ? ext : 0;
        lv.ext_hi = dn ? ext : 0;
        int err = 0, abort = 0;
        HaloPeers hp{};
        hp.x_up = up ? R[r - 1].e.p() + (ptrdiff_t)R[r - 1].nyc * K.e.pitch : nullptr;  // coarse row -1 == its last row
        hp.x_dn = dn ? R[r + 1].e.p() : nullptr;
        hp.x_keep = K.e.p();
        hp.flag_up = up ? &K.inbox[0] : nullptr;
        hp.flag_dn = dn ? &K.inbox[1] : nullptr;
        hp.pub_up = up ? &outbox[2 * r] : nullptr;
        hp.pub_dn = dn ? &outbox[2 * r + 1] : nullptr;
        hp.epoch = epoch;
        hp.err = &err;
        hp.abort = &abort;
        hp.rows_from = from;
        hp.rows_count = count;
        lv.hp = hp;
        std::vector<double> partials((size_t)fused_max_partials(n), 0.0);
        int np = 0;
        launch_fused_up(lv, K.e.p(), K.e.pitch, nu2, omega, prolong, norm ? partials.data() : nullptr, &np, nullptr);
        check(fused_take_bad_nu() == 0, "launch_fused_up refused the pass", n, r);
        check(err == 0 && abort == 0, "flag wait failed", n, r);
        check((!up || outbox[2 * r] == epoch) && (!dn || outbox[2 * r + 1] == epoch), "epoch not published", n, r);
        const int a = -lv.ext_lo, b = K.ny + lv.ext_hi;
        bool ok = true;
        int nan_rows = 0;
        for (int y = a; y < b; ++y) {
            bool row_ok = true;
            for (int xx = 0; xx < n; ++xx) row_ok = row_ok && same_bits(K.x.at(y, xx), want.at(y + K.y0, xx));
            ok = ok && row_ok;
            nan_rows += row_ok ? 0 : 1;
        }
        if (!ok) std::printf("  rank %d: %d rows of x differ\n", r, nan_rows);
        check(ok, "Pass B with up-exchange: x", n, r, ranks);
        check(K.x.untouched_outside(x0, a, b), "Pass B wrote x outside its rows", n, r);
        // the coarse array: a row up to rows_from + count beyond the slab either kept its bits (no warp reads it: the rows
        // above the slab that the prolongation reads are one fewer than below) or holds the neighbour's row; the rows the
        // prolongation does read were checked through x above; nothing else changed
        const int ea = up ? -(from + count) : 0, eb = dn ? K.nyc + from + count : K.nyc;
        ok = true;
        for (int y = ea; y < eb; ++y)
            for (int xx = 0; xx < nc; ++xx)
                ok = ok && (same_bits(K.e.at(y, xx), e.at(y + K.yc0, xx)) || same_bits(K.e.at(y, xx), e0.at(y, xx)));
        check(ok, "coarse rows after the prologue", n, r, ranks);
        check(K.e.untouched_outside(e0, ea, eb), "the prologue wrote the coarse array outside its rows (padding included)", n, r);
        for (int i = 0; i < np; ++i) s2 += partials[i];
    }
    if (norm) check(std::fabs(s2 - norm2) <= 1e-12 * norm2, "rank-summed residual norm", n, ranks);
    ++g_runs;
    std::printf("up-exchange n=%d ranks=%d nu=(%d,%d) level=%d prolong=%d omega=%g sms=%d rows_from=%d rows_count=%d: %s\n", n,
                ranks, nu1, nu2, level, prolong, omega, sms, from, count, g_bad ? "see above" : "ok");
    std::fflush(stdout);
}

int main()
{
    int i = 0;
    for (int nu1 = 1; nu1 <= 4; ++nu1)
        for (int nu2 = 1; nu2 <= 4; ++nu2) {
            if (std::max(nu1, nu2) < 3) continue;
            const int prolong = (i & 1) ? ORC_PROLONG_FULL : ORC_PROLONG_REFERENCE;
            const double omega = (i & 2) ? 1.0 : 2.0 / 3.0;
            up_exchange_pass(257, 2, nu1, nu2, 0, prolong, omega, 148);   // finest level: own rows, fused norm where it fits
            up_exchange_pass(257, 2, nu1, nu2, 1, prolong, omega, 148);   // coarser level: pass_b_ext rows
            up_exchange_pass(513, 4, nu1, nu2, 1, prolong, omega, 148);   // middle ranks with two neighbours
            up_exchange_pass(257, 3, nu1, nu2, i % 2, prolong, omega, 2);  // tall chunks, uneven slabs
            ++i;
        }
    std::printf("%s (%d runs)\n", g_bad ? "MISMATCHES" : "all bit-identical", g_runs);
    return g_bad ? 1 : 0;
}
