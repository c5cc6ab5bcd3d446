// test_cross_edges_emu.cpp -- the cross-cycle pass (k_cross) at the edges of the level, run from the kernel source on the CPU
// (tests/cpp/emu/host_emulation.h) and compared BIT FOR BIT with the CPU oracle.  The wide shape freezes the Dirichlet
// columns in slot 0 only and lets padding columns and odd padding rows compute values no domain point reads; these cases pin
// what that must not change:
//   * a Dirichlet ring that is not zero: random values, -0.0 and values of magnitude 1e100, in the iterate, in f and in the
//     coarse correction e;
//   * the padding of every output array (xb', x_k, coarse f) is still all-zero bits after the pass;
//   * both prolongations; wide (4 columns per lane, stored and generated f, prefetch 2 and 3) and narrow shapes;
//   * row slabs on 2-4 ranks with the wide shapes (the slab test of test_fused_kernel_emu.cpp, which also requires every
//     position outside the owned rows -- padding columns included -- to keep its bits).
#define main fused_kernel_emu_main
#include "test_fused_kernel_emu.cpp"
#undef main

static std::mt19937_64 g_edge_rng(97);

// a value for a Dirichlet ring point: ordinary, signed zero, or huge
static double ring_value()
{
    const double u = std::uniform_real_distribution<double>(-1.0, 1.0)(g_edge_rng);
    switch (g_edge_rng() % 5) {
    case 0: return -0.0;
    case 1: return u < 0 ? -1e100 : 1e100;
    case 2: return 0.0;
    default: return u;
    }
}

static void fill_ring(Dense &d)
{
    const int n = d.n;
    for (int y = 0; y < n; ++y)
        for (int x = 0; x < n; ++x)
            if (y == 0 || y == n - 1 || x == 0 || x == n - 1) d.at(y, x) = ring_value();
}

// every position of a padded array outside rows [0, rows) x columns [0, cols) is +0.0, bit for bit
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

static void edge_cross(int n, int prolong, int sms, int minb, bool gen_f, bool write_xk)
{
    emu_num_sms = sms;
    fused_set_cross_minb(minb);
    const double omega = 2.0 / 3.0;
    const int nc = (n - 1) / 2 + 1;
    const double h = 1.0 / (n - 1);
    Dense xb(n), f(n), e(nc);
    xb.randomize(true);
    fill_ring(xb);
    e.randomize(true);
    fill_ring(e);
    std::vector<double> fx, sy;
    if (gen_f) {
        // the tables pmg_set_rhs_sine builds; f is their product (the ring of f is then the sine's, zero or tiny)
        std::vector<double> sn(n);
        for (int i = 0; i < n; ++i) sn[i] = std::sin(1.0 * M_PI * (i * h) / 1.0);
        const double factor = (M_PI * M_PI / (1.0 * 1.0)) * (1.0 * 1.0 + 1.0 * 1.0);
        fx.assign((size_t)level_pitch(n), 0.0);
        sy.assign((size_t)n + 2 * PADY, 0.0);
        for (int i = 0; i < n; ++i) {
            fx[PADX + i] = factor * sn[i];
            sy[PADY + i] = sn[i];
        }
        for (int y = 0; y < n; ++y)
            for (int x = 0; x < n; ++x) f.at(y, x) = (factor * sn[x]) * sn[y];
    } else {
        f.randomize(true);
        fill_ring(f);
    }
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

    Padded pin(n, n), pout(n, n), pxk(n, n), pf(n, n), pe(nc, nc), pcf(nc, nc);
    pin.load(xb, 0, 0, n);
    pe.load(e, 0, 0, nc);
    if (gen_f)
        pf.fill_rows(0, n, std::nan(""));  // the generated flavour must not read f
    else
        pf.load(f, 0, 0, n);
    pout.fill_rows(0, n, std::nan(""));
    pxk.fill_rows(0, n, std::nan(""));
    pcf.fill_rows(0, nc, std::nan(""));
    Padded pin0 = pin, pf0 = pf, pe0 = pe;
    FusedLevel lv{};
    lv.x = write_xk ? pxk.p() : nullptr;
    lv.xb = pin.p();
    lv.f = pf.p();
    lv.n = n;
    lv.pitch = pin.pitch;
    lv.h = h;
    if (gen_f) {
        lv.rhs_fx = fx.data() + PADX;
        lv.rhs_sy = sy.data() + PADY;
    }
    std::vector<double> partials((size_t)fused_max_partials(n), 0.0);
    int np = 0;
    launch_fused_cross(lv, pout.p(), pe.p(), pcf.p(), pe.pitch, omega, prolong, partials.data(), &np, nullptr, nullptr);
    bool ok_x = true, ok_k = true, ok_c = true;
    for (int y = 0; y < n; ++y)
        for (int x = 0; x < n; ++x) {
            ok_x = ok_x && same_bits(pout.at(y, x), xb2.at(y, x));
            ok_k = ok_k && (write_xk ? same_bits(pxk.at(y, x), xk.at(y, x)) : std::isnan(pxk.at(y, x)));
        }
    for (int y = 0; y < nc; ++y)
        for (int x = 0; x < nc; ++x) {
            // the pass writes the coarse rows 1 .. nc - 2 (zero in the ring columns); rows 0 and nc - 1 keep what they held
            const bool ring_row = y == 0 || y == nc - 1;
            ok_c = ok_c && (ring_row ? std::isnan(pcf.at(y, x)) : same_bits(pcf.at(y, x), cf.at(y, x)));
        }
    double sum = 0.0;
    for (int i = 0; i < np; ++i) sum += partials[(size_t)i];
    const char *shape = minb == 2 || minb == 7 ? "wide" : "narrow";
    check(ok_x, "edges: xb' = S^2(S^2(xb + P e))", n, minb, gen_f);
    check(ok_k, "edges: x_k", n, minb, gen_f);
    check(ok_c, "edges: coarse f = R(f - A xb')", n, minb, gen_f);
    check(std::fabs(sum - nn * nn) <= 1e-12 * nn * nn, "edges: residual norm of x_k", n, minb, gen_f);
    check(padding_zero(pout, n, n), "edges: padding of xb' not all-zero", n, minb, gen_f);
    check(padding_zero(pxk, n, n), "edges: padding of x_k not all-zero", n, minb, gen_f);
    check(padding_zero(pcf, nc, nc), "edges: padding of coarse f not all-zero", n, minb, gen_f);
    check(pin.untouched_outside(pin0, 0, 0) && pf.untouched_outside(pf0, 0, 0) && pe.untouched_outside(pe0, 0, 0),
          "edges: inputs untouched", n, minb, gen_f);
    std::printf("edge cross pass n=%d prolong=%d sms=%d %s minb=%d f=%s x_k=%s: %s\n", n, prolong, sms, shape, minb,
                gen_f ? "generated" : "stored", write_xk ? "written" : "kept", (ok_x && ok_k && ok_c) ? "ok" : "MISMATCH");
}

int main(int argc, char **argv)
{
    const bool full = argc > 1 && std::strcmp(argv[1], "full") == 0;
    const int P[2] = {ORC_PROLONG_REFERENCE, ORC_PROLONG_FULL};
    for (int prolong : P) {
        edge_cross(129, prolong, 148, 2, false, false);  // wide, stored f: 2 strips, the second reaches the right-hand padding
        edge_cross(129, prolong, 148, 2, true, false);   // wide, generated f (the solve's flavour)
        edge_cross(257, prolong, 3, 2, true, true);      // tall chunks through the padding rows; x_k written
        edge_cross(257, prolong, 148, 7, false, true);   // wide, one more row of prefetch
        edge_cross(257, prolong, 148, 4, false, true);   // narrow
        edge_cross(129, prolong, 2, 3, false, false);    // narrow, few SMs
        edge_cross(1025, prolong, 148, 2, true, false);  // ten strips, the B200's wave
    }
    edge_cross(1025, ORC_PROLONG_REFERENCE, 7, 2, false, true);
    if (full) edge_cross(4097, ORC_PROLONG_REFERENCE, 148, 2, true, false);
    // row slabs on 2-4 ranks, wide shapes
    slab_cross(129, 2, ORC_PROLONG_REFERENCE, 148, 2);
    slab_cross(257, 3, ORC_PROLONG_FULL, 148, 2);
    slab_cross(257, 4, ORC_PROLONG_REFERENCE, 2, 2);
    slab_cross(257, 4, ORC_PROLONG_FULL, 148, 7);
    std::printf(g_bad ? "FAILED (%d)\n" : "all bit-identical\n", g_bad);
    return g_bad ? 1 : 0;
}
