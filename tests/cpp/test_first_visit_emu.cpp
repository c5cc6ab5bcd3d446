// test_first_visit_emu.cpp -- the first visit of a coarse level (x == 0 on entry) on the fused engine, run from the kernel
// source on the CPU (tests/cpp/emu/host_emulation.h) and compared BIT FOR BIT with the CPU oracle:
//   * Pass A (k_down, ZEROX) with its pointwise first sweep: xb and the coarse f, with an all-NaN iterate array (not read);
//     and the large-level form that does not store xb: the skipped xb array (all NaN) keeps every bit, the same coarse f;
//   * Pass B (k_up) from that xb, and rebuilding xb = S^nu1(0; f) from f (REBUILD) with an all-NaN xb array: the same new
//     iterate as the reading pass and as the oracle;
//   * f with -0.0 and +-1e100 entries (in the interior and on the ring); omega = 1, 2/3, 0.8 and 1.2, so that a pointwise
//     sweep without its +0 normalisation (h^2 * -0 + 0 = +0) gives -0.0 where the reference gives +0.0;
//   * the padding of every output array stays all-zero bits; the inputs keep their bits.
#define main fused_kernel_emu_main
#include "test_fused_kernel_emu.cpp"
#undef main

static std::mt19937_64 g_fv_rng(4242);

// f: random, with -0.0 and +-1e100 at some points (ring included)
static void fill_f(Dense &f)
{
    for (int y = 0; y < f.n; ++y)
        for (int x = 0; x < f.n; ++x) {
            const double u = std::uniform_real_distribution<double>(-1.0, 1.0)(g_fv_rng);
            switch (g_fv_rng() % 8) {
            case 0: f.at(y, x) = -0.0; break;
            case 1: f.at(y, x) = u < 0 ? -1e100 : 1e100; break;
            case 2: f.at(y, x) = 0.0; break;
            default: f.at(y, x) = u;
            }
        }
}

static bool padding_zero(const Padded &a, int rows, int cols)
{
    for (int r = -PADY; r < a.rows + PADY; ++r)
        for (int c = -PADX; c < a.pitch - PADX; ++c) {
            if (r >= 0 && r < rows && c >= 0 && c < cols) continue;
            uint64_t bits;
            std::memcpy(&bits, &a.base[(size_t)(r + PADY) * a.pitch + PADX + c], 8);
            if (bits != 0) return false;
        }
    return true;
}

static bool equal_to(Padded &p, Dense &d)
{
    for (int y = 0; y < d.n; ++y)
        for (int x = 0; x < d.n; ++x)
            if (!same_bits(p.at(y, x), d.at(y, x))) return false;
    return true;
}

static void all_nan(Padded &p) { std::fill(p.base.begin(), p.base.end(), std::nan("")); }

static void first_visit(int n, int nu1, int nu2, double omega, int prolong, int sms)
{
    emu_num_sms = sms;
    fused_set_variant(-1);
    const int nc = (n - 1) / 2 + 1;
    const double h = 1.0 / (n - 1);
    Dense x(n), f(n), e(nc);  // x: zero, ring included (first visit)
    fill_f(f);
    e.randomize(true);
    Expected E = expected_visit(x, f, e, h, omega, nu1, nu2, prolong, true);

    Padded px(n, n), pxb(n, n), pf(n, n), pe(nc, nc), pcf(nc, nc);
    all_nan(px);  // x == 0 is known: the iterate array is not read
    pf.load(f, 0, 0, n);
    pe.load(e, 0, 0, nc);
    const Padded px0 = px, pf0 = pf, pe0 = pe;
    FusedLevel lv{};
    lv.x = px.p();
    lv.xb = pxb.p();
    lv.f = pf.p();
    lv.n = n;
    lv.pitch = px.pitch;
    lv.h = h;

    launch_fused_down(lv, pcf.p(), pcf.pitch, nu1, omega, true, nullptr, nullptr, true);
    const bool ok_a = equal_to(pxb, E.xb) && padding_zero(pxb, n, n);
    const bool ok_c = equal_to(pcf, E.cf) && padding_zero(pcf, nc, nc);
    check(ok_a, "first-visit Pass A: xb = S^nu1(0)", n, nu1, (int)(omega * 100));
    check(ok_c, "first-visit Pass A: coarse f = R(f - A xb)", n, nu1, (int)(omega * 100));

    // Pass A without the xb store: the same coarse f, the xb array untouched
    Padded pskip(n, n), pcf2(nc, nc);
    all_nan(pskip);
    const Padded pskip0 = pskip;
    lv.xb = pskip.p();
    launch_fused_down(lv, pcf2.p(), pcf2.pitch, nu1, omega, true, nullptr, nullptr, false);
    const bool ok_a2 = std::memcmp(pskip.base.data(), pskip0.base.data(), pskip.base.size() * 8) == 0 &&
                       std::memcmp(pcf2.base.data(), pcf.base.data(), pcf.base.size() * 8) == 0;
    check(ok_a2, "first-visit Pass A without xb: xb untouched, same coarse f", n, nu1, (int)(omega * 100));

    // Pass B from the stored xb
    Padded pxn(n, n);
    lv.xb = pxb.p();
    lv.x = pxn.p();
    launch_fused_up(lv, pe.p(), pe.pitch, nu2, omega, prolong, nullptr, nullptr, nullptr, nullptr, 0);
    const bool ok_b = equal_to(pxn, E.xnew) && padding_zero(pxn, n, n);
    check(ok_b, "first-visit Pass B: x = S^nu2(xb + P e)", n, nu2, (int)(omega * 100));

    // Pass B rebuilding xb from f: an all-NaN xb array, the same bits as the reading pass
    Padded pxr(n, n), pnan(n, n);
    all_nan(pnan);
    const Padded pnan0 = pnan;
    lv.xb = pnan.p();
    lv.x = pxr.p();
    launch_fused_up(lv, pe.p(), pe.pitch, nu2, omega, prolong, nullptr, nullptr, nullptr, nullptr, nu1);
    const bool ok_r = pxr.base == pxn.base && equal_to(pxr, E.xnew) && padding_zero(pxr, n, n) &&
                      std::memcmp(pnan.base.data(), pnan0.base.data(), pnan.base.size() * 8) == 0;
    check(ok_r, "first-visit Pass B rebuilding xb", n, nu2, nu1);

    check(fused_take_bad_nu() == 0, "a launcher refused the pass", n, nu1, nu2);
    check(std::memcmp(px.base.data(), px0.base.data(), px.base.size() * 8) == 0 && pf.base == pf0.base && pe.base == pe0.base,
          "first visit: inputs untouched", n, nu1, nu2);
    std::printf("first visit n=%d nu=(%d,%d) omega=%.3f prolong=%d sms=%d: %s\n", n, nu1, nu2, omega, prolong, sms,
                (ok_a && ok_c && ok_a2 && ok_b && ok_r) ? "ok" : "MISMATCH");
    std::fflush(stdout);
}

int main()
{
    const double W[4] = {1.0, 2.0 / 3.0, 0.8, 1.2};
    const int P[2] = {ORC_PROLONG_REFERENCE, ORC_PROLONG_FULL};
    int runs = 0;
    // every sweep-count pair 1..3, every omega, both prolongations on the small levels
    for (int n : {5, 9, 129})
        for (int nu1 = 1; nu1 <= 3; ++nu1)
            for (int nu2 = 1; nu2 <= 3; ++nu2)
                for (double w : W) {
                    first_visit(n, nu1, nu2, w, P[(nu1 + nu2 + n) & 1], n == 129 ? 3 : 148);
                    ++runs;
                }
    for (double w : W)
        for (int prolong : P) {
            first_visit(257, 2, 2, w, prolong, 148);  // the headline V(2,2)
            first_visit(129, 4, 4, w, prolong, 148);
            runs += 2;
        }
    first_visit(257, 1, 3, 1.2, ORC_PROLONG_FULL, 7);
    first_visit(257, 3, 1, 1.0, ORC_PROLONG_REFERENCE, 148);
    first_visit(1025, 2, 2, 2.0 / 3.0, ORC_PROLONG_REFERENCE, 148);  // several strips and chunks, the B200's wave
    first_visit(1025, 3, 2, 1.2, ORC_PROLONG_FULL, 20);
    runs += 4;
    std::printf(g_bad ? "FAILED (%d)\n" : "all bit-identical (%d runs)\n", g_bad ? g_bad : runs);
    return g_bad ? 1 : 0;
}
