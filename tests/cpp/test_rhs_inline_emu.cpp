// test_rhs_inline_emu.cpp -- the cross-cycle pass (k_cross, default wide shape) with its right-hand side GENERATED in the
// row feed from the two tables pmg_set_rhs_sine builds (FusedLevel::rhs_fx / rhs_sy), run from the kernel source on the CPU
// (tests/cpp/emu/host_emulation.h) and compared BIT FOR BIT with
//   * the same pass reading the stored f (the array k_rhs_separable writes, built here with the same multiplications), and
//   * the CPU oracle's operator sequence (Pass B of cycle k, then Pass A of cycle k+1).
// The generated run gets an f array full of NaN, so any read of f would show.  Sizes and SM counts are chosen so that strips
// reach the right-hand padding and chunks reach the padding rows above and below.
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
static std::mt19937_64 g_rng(4242);
static double rnd() { return std::uniform_real_distribution<double>(-1.0, 1.0)(g_rng); }
static bool same_bits(double a, double b) { return std::memcmp(&a, &b, 8) == 0; }

static void check(bool ok, const char *what, int n, int sms)
{
    if (!ok) {
        std::printf("  MISMATCH: %s (n=%d, sms=%d)\n", what, n, sms);
        ++g_bad;
    }
}

struct Dense {
    int n;
    std::vector<double> v;
    explicit Dense(int n_) : n(n_), v((size_t)n_ * n_, 0.0) {}
    double &at(int y, int x) { return v[(size_t)y * n + x]; }
};

// the solver's padded layout of an n x n level: logical (0,0) at base[PADY * pitch + PADX]
struct Padded {
    int n, pitch;
    std::vector<double> base;
    Padded(int n_, double fill = 0.0) : n(n_), pitch(level_pitch(n_)), base((size_t)level_pitch(n_) * (n_ + 2 * PADY), fill) {}
    double *p() { return base.data() + (size_t)PADY * pitch + PADX; }
    double &at(int y, int x) { return p()[(ptrdiff_t)y * pitch + x]; }
    void load(Dense &d)
    {
        for (int y = 0; y < n; ++y)
            for (int x = 0; x < n; ++x) at(y, x) = d.at(y, x);
    }
};

struct Result {
    std::vector<double> out, cf, partials;
};

static Result run_pass(Padded &pin, Padded &pf, Padded &pe, const double *fx, const double *sy, int n, double omega, int prolong)
{
    const int nc = (n - 1) / 2 + 1;
    Padded pout(n, std::nan("")), pcf(nc);
    FusedLevel lv{};
    lv.x = nullptr;  // one-GPU solve: x_k is not written
    lv.xb = pin.p();
    lv.f = pf.p();
    lv.n = n;
    lv.pitch = pin.pitch;
    lv.h = 1.0 / (n - 1);
    lv.rhs_fx = fx;
    lv.rhs_sy = sy;
    Result r;
    r.partials.assign((size_t)fused_max_partials(n), 0.0);
    int np = 0;
    launch_fused_cross(lv, pout.p(), pe.p(), pcf.p(), pe.pitch, omega, prolong, r.partials.data(), &np, nullptr, nullptr);
    r.partials.resize((size_t)np);
    r.out = pout.base;
    r.cf = pcf.base;
    return r;
}

static bool same_vec(const std::vector<double> &a, const std::vector<double> &b)
{
    return a.size() == b.size() && std::memcmp(a.data(), b.data(), a.size() * 8) == 0;
}

static void generated_cross(int n, double omega, int prolong, int sms)
{
    emu_num_sms = sms;
    fused_set_cross_minb(2);  // the default shape: the only one with the generated feed
    const int nc = (n - 1) / 2 + 1;
    const double h = 1.0 / (n - 1);
    // the tables as pmg_set_rhs_sine builds them (ensure_fmg's sine table, analytic_rhs's factor)
    std::vector<double> sn(n);
    for (int i = 0; i < n; ++i) sn[i] = std::sin(1.0 * M_PI * (i * h) / 1.0);
    bool no_sign = true;
    for (double v : sn) no_sign = no_sign && !std::signbit(v);
    check(no_sign, "a sine value carries a sign bit: zero padding would not reproduce the array's +0", n, sms);
    const double factor = (M_PI * M_PI / (1.0 * 1.0)) * (1.0 * 1.0 + 1.0 * 1.0);
    const int pitch = level_pitch(n);
    std::vector<double> fx(pitch, 0.0), sy(n + 2 * PADY, 0.0);
    for (int i = 0; i < n; ++i) {
        fx[PADX + i] = factor * sn[i];
        sy[PADY + i] = sn[i];
    }
    // f as k_rhs_separable writes it: (factor * sin_x) * sin_y on the n x n level, zero padding
    Dense f(n);
    for (int y = 0; y < n; ++y)
        for (int x = 0; x < n; ++x) f.at(y, x) = (factor * sn[x]) * sn[y];
    Padded pf(n);
    pf.load(f);
    // every position the pass can read -- padding rows and columns included -- is the table product, bit for bit
    bool tables_ok = true;
    for (int r = -PADY; r < n + PADY; ++r)
        for (int c = -PADX; c < pitch - PADX; ++c) tables_ok = tables_ok && same_bits(fx[PADX + c] * sy[PADY + r], pf.at(r, c));
    check(tables_ok, "fx[x] * sy[y] differs from the stored f somewhere in the padded array", n, sms);

    Dense xb(n), e(nc);
    for (auto &v : xb.v) v = rnd();
    for (int y = 1; y < nc - 1; ++y)
        for (int x = 1; x < nc - 1; ++x) e.at(y, x) = rnd();
    // the oracle: x_k = S^2(xb + P e), its residual norm, xb' = S^2(x_k), coarse f = R(f - A xb')
    Dense xk = xb;
    orc_prolong_add(xk.v.data(), e.v.data(), n, nc, prolong);
    orc_jacobi(xk.v.data(), f.v.data(), n, n, h, omega, 1, 0.0, nullptr);
    Dense r(n);
    orc_residual(r.v.data(), xk.v.data(), f.v.data(), n, n, h);
    const double nn = orc_norm(r.v.data(), (long)n * n);
    Dense xb2 = xk;
    orc_jacobi(xb2.v.data(), f.v.data(), n, n, h, omega, 1, 0.0, nullptr);
    Dense r2(n), cf(nc);
    orc_residual(r2.v.data(), xb2.v.data(), f.v.data(), n, n, h);
    orc_restrict_fw(r2.v.data(), cf.v.data(), n, nc);

    Padded pin(n), pe(nc), pnan(n, std::nan(""));
    pin.load(xb);
    pe.load(e);
    const Result stored = run_pass(pin, pf, pe, nullptr, nullptr, n, omega, prolong);
    const Result gen = run_pass(pin, pnan, pe, fx.data() + PADX, sy.data() + PADY, n, omega, prolong);

    check(same_vec(gen.out, stored.out), "generated f: xb' differs from the stored-f pass", n, sms);
    check(same_vec(gen.cf, stored.cf), "generated f: coarse f differs from the stored-f pass", n, sms);
    check(same_vec(gen.partials, stored.partials), "generated f: norm partials differ from the stored-f pass", n, sms);
    Padded gout(n), gcf(nc);
    gout.base = gen.out;
    gcf.base = gen.cf;
    bool ok_x = true, ok_c = true;
    for (int y = 0; y < n; ++y)
        for (int x = 0; x < n; ++x) ok_x = ok_x && same_bits(gout.at(y, x), xb2.at(y, x));
    for (int y = 0; y < nc; ++y)
        for (int x = 0; x < nc; ++x) ok_c = ok_c && same_bits(gcf.at(y, x), cf.at(y, x));
    check(ok_x, "generated f: xb' = S^2(S^2(xb + P e)) against the oracle", n, sms);
    check(ok_c, "generated f: coarse f = R(f - A xb') against the oracle", n, sms);
    double sum = 0.0;
    for (double v : gen.partials) sum += v;
    check(std::fabs(sum - nn * nn) <= 1e-12 * nn * nn, "generated f: residual norm of x_k", n, sms);
    std::printf("generated-f cross pass n=%d omega=%.3f prolong=%d sms=%d: %s\n", n, omega, prolong, sms,
                g_bad ? "see above" : "ok");
}

int main()
{
    const double w = 2.0 / 3.0;
    generated_cross(129, w, ORC_PROLONG_REFERENCE, 148);  // 2 strips: the second one reaches the right-hand padding
    generated_cross(129, 1.0, ORC_PROLONG_FULL, 2);       // few SMs: tall chunks, chunk overlap
    generated_cross(257, w, ORC_PROLONG_REFERENCE, 1);    // one chunk from the top padding rows to the bottom ones
    generated_cross(257, w, ORC_PROLONG_FULL, 148);
    generated_cross(257, w, ORC_PROLONG_REFERENCE, 5);
    generated_cross(1025, w, ORC_PROLONG_REFERENCE, 148);  // ten strips, the B200's wave
    generated_cross(1025, 1.0, ORC_PROLONG_REFERENCE, 7);
    std::printf(g_bad ? "FAILED (%d)\n" : "all bit-identical\n", g_bad);
    return g_bad ? 1 : 0;
}
