// solver.cu -- host side of libpmg.so: the level hierarchy in HBM, the V/W/F cycle drivers and the C ABI
// of include/pmg.h.  It mirrors the control flow of MultigridSolver (2_part_MG/MultiGrid.hpp:57-183) and
// of the runner's outer loop (2_part_MG/MultiGridTestRunner.hpp:190-212), but every buffer is allocated
// once at pmg_create (the reference allocates three arrays per level per call, MultiGrid.hpp:70-82, and
// its GPU twin leaks them, Parallel_Mg.cu:38-54) and no stage ever runs on the CPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "pmg_internal.h"

#include <execinfo.h>
#include <fcntl.h>
#include <signal.h>
#include <unistd.h>

namespace pmg {

// PMG_DEBUG_SIGNALS=<file>: append a native backtrace to <file> on SIGSEGV / SIGABRT (debug aid; off by default)
static int g_debug_fd = -1;
static void pmg_signal_handler(int sig)
{
    void *frames[64];
    int n = backtrace(frames, 64);
    const char msg[] = "\n[libpmg] fatal signal, native backtrace:\n";
    (void)!write(g_debug_fd, msg, sizeof(msg) - 1);
    backtrace_symbols_fd(frames, n, g_debug_fd);
    signal(sig, SIG_DFL);
    raise(sig);
}
static int install_debug_signals()
{
    const char *e = getenv("PMG_DEBUG_SIGNALS");
    if (e && e[0]) {
        g_debug_fd = open(e, O_WRONLY | O_CREAT | O_APPEND, 0644);
        if (g_debug_fd >= 0) {
            signal(SIGSEGV, pmg_signal_handler);
            signal(SIGABRT, pmg_signal_handler);
        }
    }
    return 0;
}
static int g_debug_signals = install_debug_signals();

thread_local std::string g_last_error;
static int g_cluster_override = -1;  // pmg_set_cluster_top: -1 = PMG_CLUSTER / the default
static int g_cross_override = -1;    // pmg_set_cross_cycle: -1 = PMG_CROSS / the default

static pmg_status fail(pmg_status s, const std::string &msg)
{
    g_last_error = msg;
    return s;
}

#define PMG_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(PMG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " (" +  \
                                          __FILE__ + ":" + std::to_string(__LINE__) + ")");         \
    } while (0)

static bool is_pow2_plus_1(int n) { return n >= 3 && ((n - 1) & (n - 2)) == 0; }

struct Level {
    int n = 0, pitch = 0;
    int ny = 0, y0 = 0;  // row slab [y0, y0 + ny) of a level partitioned over ranks; ny == 0: whole level
    double h = 0.0;
    size_t elems = 0;
    double *base_x = nullptr, *base_xb = nullptr, *base_f = nullptr, *base_r = nullptr;
    double *x = nullptr, *xb = nullptr, *f = nullptr, *r = nullptr;  // logical (0,0)
    double *d_sin = nullptr;  // sin(pi * i * h), i < n  (F-cycle analytic RHS; lazily built)
    // NVLink peer-to-peer halo exchange: the neighbours' boundary rows of x and f as seen from this process
    // (upper neighbour's row ny_up - PADY, lower neighbour's row 0) and the raw IPC mappings to close
    const double *up_x = nullptr, *dn_x = nullptr, *up_f = nullptr, *dn_f = nullptr;
    // (level 0 only) the same for the two arrays the cross-cycle pass alternates between: [0] = xb, [1] = xc
    const double *up_xb[2] = {nullptr, nullptr}, *dn_xb[2] = {nullptr, nullptr};
    int halo_epoch = 0;
    int up_epoch = 0;  // deep-sweep schedule: up-exchanges of this level's iterate (one per Pass B of the parent)
};

// ---- slab schedule depths (DESIGN.md section 6) -------------------------------------------------------------------
// With nu <= 2 the slab cycle recomputes every halo row the way up needs: Pass A finishes xb on 6 rows beyond the slab,
// Pass B on levels l > 0 finishes x on 4, exactly the coarse rows the parent's prolongation reads.  With 3 or 4 sweeps
// no such choice exists for an 8-row halo, so the deep-sweep schedule derives the depths from the sweep counts and
// exchanges the rest of the child's rows on the way up (cycle_dist, k_up's coarse prologue).
static bool deep_sweeps(const pmg_config &c) { return std::max(c.nu1, c.nu2) >= 3; }

// rows beyond the slab on which Pass A finishes xb: nu1 sweeps eat one of the PADY exchanged rows each (even: the
// fused passes start their row chunks on even rows)
static int pass_a_depth(const pmg_config &c) { return deep_sweeps(c) ? (PADY - c.nu1) & ~1 : 6; }

// rows beyond the slab on which Pass B of level l finishes x: the finest level's own rows only; below it as many as
// the xb depth allows (nu2 sweeps eat one row each; even)
static int pass_b_ext(const pmg_config &c, int l)
{
    if (l == 0) return 0;
    return deep_sweeps(c) ? std::max(0, (pass_a_depth(c) - c.nu2) & ~1) : 4;
}

// coarse rows beyond the slab that Pass B of level l reads: it needs xb + P e on ext + nu2 (+1 for the finest level's
// residual norm) fine rows beyond, and fine row ny + q - 1 (odd) interpolates coarse rows up to depth q / 2 + 1
static int pass_b_coarse_rows(const pmg_config &c, int l) { return (pass_b_ext(c, l) + c.nu2 + (l == 0 ? 1 : 0)) / 2 + 1; }

// rows of level l + 1's iterate that the deep-sweep schedule exchanges before Pass B of level l (beyond the
// pass_b_ext(c, l + 1) rows the child finished itself); 0 with nu <= 2.  At most 3 <= MAX_UP_ROWS.
static int up_exchange_rows(const pmg_config &c, int l)
{
    return deep_sweeps(c) ? std::max(0, pass_b_coarse_rows(c, l) - pass_b_ext(c, l + 1)) : 0;
}

// the finest level's Pass B sums the residual norm itself when xb reaches one row further than its sweeps eat
static bool pass_b_norm_fits(const pmg_config &c) { return c.nu2 + 1 <= pass_a_depth(c); }

// d_flags inbox (FLAG_SLOTS ints): [2l], [2l+1] = down exchange of level l from the upper / lower neighbour (l < 16),
// [32 + rank] = gather inbox (n_ranks <= 32), [UP_FLAG_SLOT + 2k], [+1] = up-exchange of level k's iterate (k < 16).
// The largest grid, N = 32769, has at most 10 slab levels (2 ranks), so every slot is far from its limit.
constexpr int UP_FLAG_SLOT = 64, FLAG_SLOTS = 96;

}  // namespace pmg

using namespace pmg;

struct pmg_solver {
    pmg_config cfg;
    int device = 0;
    cudaStream_t stream = nullptr;
    std::vector<Level> lv;
    double *d_partials = nullptr;
    int partials_cap = 0;
    double *d_scalar = nullptr;  // device double (sum of squares)
    double *h_scalar = nullptr;  // pinned host mirror
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double last_ms = 0.0;
    // F-cycle: level-0 analytic RHS lives in its own array so the caller's f survives
    double *base_f_fmg0 = nullptr, *f_fmg0 = nullptr;
    bool fmg_ready = false;
    bool rhs_is_analytic = false;  // level 0's f was written by pmg_set_rhs_sine and by nothing since (one GPU); change it
                                   // with set_rhs_analytic (the cross-cycle graphs depend on it)
    // level 0's analytic right-hand side as f(y, x) = fx[x] * sy[y] (FusedLevel::rhs_fx / rhs_sy), built by pmg_set_rhs_sine:
    // the cross-cycle pass forms f from these instead of reading it while rhs_is_analytic holds for the array rhs_tab_f
    double *base_rhs_fx = nullptr, *base_rhs_sy = nullptr;
    const double *rhs_fx = nullptr, *rhs_sy = nullptr, *rhs_tab_f = nullptr;
    bool fmg0_rhs_cached = false;  // f_fmg0 holds the analytic right-hand side of level 0 (a constant of the hierarchy)
    // CUDA graphs of one fused cycle, keyed by [kind V/W][0: no norm, 1: norm -> d_scalar,
    // 2: norm -> device-side solve control (asynchronous solve)]
    cudaGraphExec_t graph[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    int graph_kernels[2][3] = {{0, 0, 0}, {0, 0, 0}};  // kernel nodes per replay (launch bookkeeping)
    bool fused = false;
    bool small_vcycle = true;  // PMG_SMALL_VCYCLE=0 disables the single-CTA kernel for the levels <= 65
    // overlapped host transfers (pmg_stage_rhs / pmg_fetch_solution_begin): a staging copy of f, a snapshot of x, one
    // copy stream per direction so that both DMA directions run beside the solver stream
    double *base_f_stage = nullptr, *base_x_snap = nullptr;
    cudaStream_t copy_in_stream = nullptr, copy_out_stream = nullptr;
    cudaEvent_t ev_staged = nullptr, ev_snap = nullptr, ev_fetched = nullptr, ev_consumed = nullptr;
    bool staged = false, fetching = false;
    double *pcg_base[4] = {nullptr, nullptr, nullptr, nullptr};  // r, z, p, A p of pmg_pcg (level-0 layout; lazily allocated)
    // pmg_pcg on row slabs (pcg_dist; lazily allocated): the second direction array (the fused direction-operator pass reads
    // one and writes the other) and [0, 1] r.z of alternate steps, [2] p.Ap, [4 ...] per-warp partial sums
    double *base_pcg_p2 = nullptr, *d_pcg_sc = nullptr;
    // cross-cycle solve (one GPU, V-cycles): per cycle ONE graph = coarse part from level 1 + the cross-cycle pass on level 0
    // + the convergence kernel; [parity]: which of the two level-0 arrays is the pass's input
    cudaGraphExec_t cross_graph[2] = {nullptr, nullptr};
    int cross_graph_kernels[2] = {0, 0};
    bool cross_on = true;      // PMG_CROSS=0: the classic two passes per cycle on level 0
    bool cross_forced = false; // PMG_CROSS=2 / pmg_set_cross_cycle(2): also where the pass does not fill the machine
    double *base_xc = nullptr, *xc = nullptr;  // third level-0 array: xb and xc alternate as the cross pass's input / output
    bool cross_active = false; // (row slabs) cycle_dist runs the cross pass instead of Pass B(0) / Pass A(0) of the next cycle
    int cross_count = 0;       // cross passes queued in the current solve
    int cluster_top = 0;       // level size from which ONE 16-CTA cluster launch runs the rest of the cycle (257 / 129;
                               // 0: off -- PMG_CLUSTER=0, an unsuitable configuration, or a device that cannot co-schedule
                               // the cluster)
    // asynchronous solve: device control block + history of squared norms, pinned mirrors, batch events
    SolveCtrl *d_ctrl = nullptr;
    double *d_hist2 = nullptr;
    int hist_cap = 0;
    SolveCtrl *h_ctrl = nullptr;  // 2 slots in MAPPED pinned memory (written by k_ctrl_to_host, no copy engine)
    double *h_hist = nullptr;     // hist_cap doubles, mapped pinned: the history of the last solve
    cudaEvent_t ev_batch[2] = {nullptr, nullptr};
    // ---- row-slab decomposition over ranks (one process per GPU) ----
    // lv[l] for l < agg_level are SLABS (ny > 0); lv[l] for l >= agg_level are whole levels that only rank 0
    // works on ("agglomerated"); `aslab` is the slab-shaped window of level agg_level the finest
    // agglomerated level is gathered from / scattered to.
    bool dist = false;
    int rank = 0, n_ranks = 1, agg_level = 0;
    Level aslab;
    std::vector<std::vector<int>> y0s, y1s;  // [level <= agg_level][rank]
    double *d_gather = nullptr;              // one double per rank (norm all-gather)
    cudaStream_t comm_stream = nullptr;      // halo exchanges and the norm all-gather run here, beside compute
    cudaEvent_t ev_ready = nullptr, ev_halo = nullptr, ev_passb = nullptr, ev_norm = nullptr;
    bool norm_pending = false;               // an ev_norm has been recorded that the next Pass B(0) must wait for
    bool coarse_redundant = false;           // every rank solves the agglomerated levels (all-gather, no scatter)
    int split_min_rows = 2048;               // slabs at least this tall overlap the exchange with interior rows (only
                                             // without the halo prologue, which makes the split unnecessary)
    bool split_from_env = false;
    bool p2p = false;                        // halo rows are pulled from the neighbours' memory over NVLink
    bool p2p_fused = true;                   // ... by Pass A itself (no pull kernel, no local copy of the x halo)
    int *d_flags = nullptr;                  // my inbox: epochs published by neighbours (layout: UP_FLAG_SLOT)
    int *up_flags = nullptr, *dn_flags = nullptr;  // the neighbours' inboxes (peer mappings)
    int *d_comm_err = nullptr;               // raised by a pull whose wait timed out
    // peer-to-peer all-gather of the first agglomerated level's right-hand side (V-cycles): double-buffered slab
    double *agg_f[2] = {nullptr, nullptr};   // bases of the two slab buffers (agg_f[0] == aslab.base_f)
    int **d_agg_slots = nullptr;             // [rank] -> that rank's inbox slot for me (peer pointers)
    const double **d_agg_srcs[2] = {nullptr, nullptr};  // per buffer: [rank] -> that rank's slab row 0 (padded start)
    std::vector<void *> agg_maps;            // IPC mappings to close
    int agg_epoch = 0;
    bool p2p_gather = false, cycle_has_collective = false;
    bool p2p_gather_w = true;                // W-cycles use the NVLink all-gather too (see cycle_dist)
    // the redundant solve of the agglomerated levels (fixed pointers, no communication) replayed as a CUDA graph
    cudaGraphExec_t coarse_graph[2] = {nullptr, nullptr};  // [V, W]
    int coarse_graph_kernels[2] = {0, 0};
    bool coarse_graph_on = true;  // PMG_COARSE_GRAPH=0 launches the kernels one by one
    // The latency-bound MIDDLE of a distributed V-cycle -- Pass A of the short-slab levels, the all-gather, the redundant
    // coarse solve and Pass B back up: ~16 launches on one stream, no host-visible events -- replayed as ONE CUDA graph
    // per all-gather buffer parity.  A captured launch keeps its arguments, so the epochs of the visit are written to
    // `d_epochs` ([l] = halo epoch of slab level l, [15] = all-gather epoch) by a tiny kernel ahead of each replay and
    // the kernels add them in (HaloPeers::epoch_base).  Default since round 2 (PMG_MID_GRAPH=0 switches it off).
    int *d_epochs = nullptr;
    cudaGraphExec_t mid_graph[2] = {nullptr, nullptr};
    int mid_graph_kernels[2] = {0, 0};
    bool mid_graph_on = true;
    bool capturing_mid = false;
};

namespace pmg {

static void drop_cross_graphs(pmg_solver *s)
{
    for (auto &g : s->cross_graph)
        if (g) {
            cudaGraphExecDestroy(g);
            g = nullptr;
        }
}

static void drop_graphs(pmg_solver *s)
{
    for (auto &row : s->graph)
        for (auto &g : row)
            if (g) {
                cudaGraphExecDestroy(g);
                g = nullptr;
            }
    for (auto &g : s->coarse_graph)
        if (g) {
            cudaGraphExecDestroy(g);
            g = nullptr;
        }
    for (auto &g : s->mid_graph)
        if (g) {
            cudaGraphExecDestroy(g);
            g = nullptr;
        }
    drop_cross_graphs(s);
}

// A captured cross-cycle graph keeps the f feed it was captured with (generated from the tables or read from HBM): a graph
// captured after pmg_set_rhs_sine must not outlive a user right-hand side, so the graphs go whenever the flag changes.
static void set_rhs_analytic(pmg_solver *s, bool on)
{
    if (s->rhs_is_analytic != on) drop_cross_graphs(s);
    s->rhs_is_analytic = on;
}

static FusedLevel fused_view(const Level &L)
{
    FusedLevel v;
    v.x = L.x;
    v.xb = L.xb;
    v.f = L.f;
    v.n = L.n;
    v.pitch = L.pitch;
    v.h = L.h;
    v.ny = L.ny;
    v.yoff = L.y0;
    v.ext_lo = v.ext_hi = 0;
    v.span_lo = v.span_hi = 0;
    v.hp = HaloPeers{};
    v.rhs_fx = v.rhs_sy = nullptr;
    return v;
}

// The cross-cycle pass on level 0 with f generated from the tables -- only if v.f is the array pmg_set_rhs_sine wrote and
// nothing has written since (PCG and the F-cycle point level 0 at other arrays for a while)
static void use_rhs_tables(const pmg_solver *s, FusedLevel &v)
{
    if (s->rhs_is_analytic && s->rhs_fx != nullptr && v.f == s->rhs_tab_f) {
        v.rhs_fx = s->rhs_fx;
        v.rhs_sy = s->rhs_sy;
    }
}

static pmg_status alloc_zero(double **p, size_t elems)
{
    if (cudaMalloc((void **)p, elems * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        return fail(PMG_ERR_ALLOC, "cudaMalloc of " + std::to_string(elems * sizeof(double)) + " bytes failed");
    }
    PMG_CUDA(cudaMemset(*p, 0, elems * sizeof(double)));
    return PMG_OK;
}

// ---- smoothing on one level (Smoother::smooth, Smoother.hpp:38-116) -----------------------------------
// Operator-granular: ping-pong sweeps; with smoother_eps > 0 the reference's per-sweep absolute-norm exit.
// Chebyshev-Jacobi weights for `n` sweeps on the eigenvalue range [1/2, 2] of D^-1 A (pmg.h); the expression is the CPU
// checker's (orc_chebyshev_weights), evaluated by the same libm
static void chebyshev_weights(int n, double *w)
{
    const double lo = 0.5, hi = 2.0;
    const double d = 0.5 * (hi + lo), c = 0.5 * (hi - lo);
    for (int k = 0; k < n; ++k) w[k] = 1.0 / (d - c * std::cos(M_PI * (2 * k + 1) / (2.0 * n)));
}

// the smoothers beyond weighted Jacobi (operator-granular; pmg.h: pmg_smoother)
static pmg_status smooth_other(pmg_solver *s, int l, int sweeps, bool x_is_zero)
{
    Level &L = s->lv[l];
    const pmg_config &c = s->cfg;
    if (sweeps <= 0) return PMG_OK;
    if (x_is_zero) launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
    if (c.smoother == PMG_SMOOTHER_RBGS) {
        for (int it = 0; it < sweeps; ++it) {
            launch_rbgs_half(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, 0, s->stream);
            launch_rbgs_half(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, 1, s->stream);
        }
    } else if (c.smoother == PMG_SMOOTHER_GS_LEX) {
        if (c.smoother_eps > 0.0) {  // GaussSeidelSmoother's absolute-norm exit (Smoother.hpp:147-159), tested per sweep
            for (int it = 0; it < sweeps; ++it) {
                launch_gs_lex(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, 1, s->stream);
                launch_residual_norm2(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, s->d_partials, s->d_scalar, s->stream);
                PMG_CUDA(cudaMemcpyAsync(s->h_scalar, s->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
                PMG_CUDA(cudaStreamSynchronize(s->stream));
                if (std::sqrt(*s->h_scalar) < c.smoother_eps) break;
            }
        } else {
            launch_gs_lex(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, sweeps, s->stream);
        }
    } else {  // PMG_SMOOTHER_CHEBYSHEV
        if (sweeps > 64) return fail(PMG_ERR_UNSUPPORTED, "Chebyshev-Jacobi: at most 64 sweeps per smoothing step");
        double w[64];
        chebyshev_weights(sweeps, w);
        for (int it = 0; it < sweeps; ++it) {
            launch_jacobi_sweep(L.xb, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, w[it], s->stream);
            std::swap(L.x, L.xb);
            std::swap(L.base_x, L.base_xb);
        }
    }
    return PMG_OK;
}

static pmg_status smooth_operator(pmg_solver *s, int l, int sweeps, bool x_is_zero, const int *done = nullptr)
{
    Level &L = s->lv[l];
    const pmg_config &c = s->cfg;
    if (c.smoother != PMG_SMOOTHER_JACOBI) return smooth_other(s, l, sweeps, x_is_zero);
    if (x_is_zero && !(c.smoother_eps <= 0.0 && L.n * L.n <= SMALL_MAX_POINTS))
        launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
    if (c.smoother_eps > 0.0) {
        for (int it = 0; it < sweeps; ++it) {
            launch_jacobi_sweep(L.xb, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, c.omega, s->stream);
            std::swap(L.x, L.xb);
            std::swap(L.base_x, L.base_xb);
            launch_residual_norm2(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, s->d_partials, s->d_scalar, s->stream);
            PMG_CUDA(cudaMemcpyAsync(s->h_scalar, s->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
            PMG_CUDA(cudaStreamSynchronize(s->stream));
            if (std::sqrt(*s->h_scalar) < c.smoother_eps) break;  // Smoother.hpp:84-88
        }
        return PMG_OK;
    }
    if (L.n * L.n <= SMALL_MAX_POINTS && !c.smoother_fp32) {
        launch_jacobi_small(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, c.omega, sweeps, x_is_zero, s->stream, done);
        return PMG_OK;
    }
    if (x_is_zero && c.smoother_fp32 && L.n * L.n <= SMALL_MAX_POINTS) launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
    for (int it = 0; it < sweeps; ++it) {
        if (c.smoother_fp32)
            launch_jacobi_sweep_f32(L.xb, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, c.omega, s->stream);
        else
            launch_jacobi_sweep(L.xb, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, c.omega, s->stream);
        std::swap(L.x, L.xb);
        std::swap(L.base_x, L.base_xb);
    }
    return PMG_OK;
}

// MultigridSolver::v_cycle / w_cycle (MultiGrid.hpp:57-94 / 96-136), one kernel per reference operator
static pmg_status cycle_operator(pmg_solver *s, int l, bool w_form, bool x_is_zero)
{
    const pmg_config &c = s->cfg;
    Level &L = s->lv[l];
    if (L.n <= c.n_coarse || l + 1 == (int)s->lv.size())
        return smooth_operator(s, l, c.coarse_sweeps, x_is_zero);  // :59-63
    pmg_status rc = smooth_operator(s, l, c.nu1, x_is_zero);       // :66
    if (rc != PMG_OK) return rc;
    Level &K = s->lv[l + 1];
    launch_residual(L.r, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.pitch, L.h, s->stream);  // :69-71
    launch_restrict(L.r, K.f, L.n, K.n, L.pitch, K.pitch, s->stream);                     // :74-78
    int reps = w_form ? c.gamma : 1;
    for (int k = 0; k < reps; ++k) {  // :81-83 / :121-125 (e_coarse = 0 before the first visit)
        rc = cycle_operator(s, l + 1, w_form, k == 0);
        if (rc != PMG_OK) return rc;
    }
    launch_prolong_add(K.x, L.x, K.n, L.n, K.pitch, L.pitch, c.prolong_mode, s->stream);  // :86
    return smooth_operator(s, l, c.nu2, false);                                          // :89
}

// The same cycle on the fused engine: two streaming passes per level visit.
// prolong_in (nested iteration, streaming levels only): the iterate of level l on entry is P (prolong_in->x) into a zeroed
// grid; it is formed inside Pass A and never written (fmg_up_from)
static pmg_status cycle_fused(pmg_solver *s, int l, bool w_form, bool x_is_zero, bool want_norm, int *n_partials,
                              const int *done = nullptr, const Level *prolong_in = nullptr)
{
    const pmg_config &c = s->cfg;
    Level &L = s->lv[l];
    if (L.n <= c.n_coarse || l + 1 == (int)s->lv.size())
        return smooth_operator(s, l, c.coarse_sweeps, x_is_zero, done);
    // from level 257 (or 129) down: ONE launch of a 16-CTA cluster, levels distributed over the CTAs' shared memories
    if (l > 0 && L.n == s->cluster_top &&
        launch_coarse_cluster(L.x, L.f, L.n, L.pitch, L.pitch, c.n_coarse, L.h, c.omega, c.nu1, c.nu2, c.coarse_sweeps,
                              c.prolong_mode, x_is_zero, w_form ? c.gamma : 1, s->stream, done))
        return PMG_OK;
    // the small levels (V or W recursion alike) run as ONE single-CTA kernel in shared memory
    if (l > 0 && L.n <= VSMALL_TOP && s->small_vcycle && (int)s->lv.size() - l <= 8 &&
        s->lv.back().n * s->lv.back().n <= SMALL_MAX_POINTS) {
        launch_vcycle_small(L.x, L.f, L.n, L.pitch, L.pitch, c.n_coarse, L.h, c.omega, c.nu1, c.nu2, c.coarse_sweeps,
                            c.prolong_mode, x_is_zero, w_form ? c.gamma : 1, s->stream, done);
        return PMG_OK;
    }
    Level &K = s->lv[l + 1];
    // a large first visit does not store xb: Pass B rebuilds it from f (which no coarser visit changes)
    const bool rebuild = prolong_in == nullptr && x_is_zero && !want_norm && fused_rebuild_xb(fused_view(L), c.nu1);
    if (prolong_in != nullptr)
        launch_fused_down_prolong(fused_view(L), prolong_in->x, prolong_in->pitch, K.f, K.pitch, c.omega, c.prolong_mode,
                                  s->stream, done);
    else
        launch_fused_down(fused_view(L), K.f, K.pitch, c.nu1, c.omega, x_is_zero, s->stream, done, !rebuild);
    int reps = w_form ? c.gamma : 1;
    for (int k = 0; k < reps; ++k) {
        pmg_status rc = cycle_fused(s, l + 1, w_form, k == 0, false, nullptr, done);
        if (rc != PMG_OK) return rc;
    }
    launch_fused_up(fused_view(L), K.x, K.pitch, c.nu2, c.omega, c.prolong_mode,
                    want_norm ? s->d_partials : nullptr, n_partials, s->stream, done, rebuild ? c.nu1 : 0);
    return PMG_OK;
}

static bool fused_graph_ok(const pmg_solver *s);

// Multi-GPU: every rank solves the agglomerated levels [agg_level, coarsest] itself.  The launch sequence has fixed
// arguments and no communication, so it is captured once and replayed (7+ launches -> one graph launch).
static pmg_status coarse_solve_redundant(pmg_solver *s, bool w_form, int reps)
{
    auto direct = [&]() -> pmg_status {
        for (int k = 0; k < reps; ++k) {
            pmg_status rc = cycle_fused(s, s->agg_level, w_form, k == 0, false, nullptr, nullptr);
            if (rc != PMG_OK) return rc;
        }
        return PMG_OK;
    };
    if (!s->coarse_graph_on || !fused_graph_ok(s) || s->capturing_mid) return direct();
    cudaGraphExec_t &ge = s->coarse_graph[w_form ? 1 : 0];
    int &gk = s->coarse_graph_kernels[w_form ? 1 : 0];
    if (ge == nullptr) {
        const unsigned long long before = launches_so_far();
        PMG_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
        pmg_status rc = direct();
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamEndCapture(s->stream, &g);
        if (e != cudaSuccess) return fail(PMG_ERR_CUDA, std::string("cudaStreamEndCapture (coarse solve): ") + cudaGetErrorString(e));
        if (rc != PMG_OK) {
            cudaGraphDestroy(g);
            return rc;
        }
        gk = (int)(launches_so_far() - before);  // counted during capture; the replay below executes them
        e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(PMG_ERR_CUDA, std::string("cudaGraphInstantiate (coarse solve): ") + cudaGetErrorString(e));
        PMG_CUDA(cudaGraphLaunch(ge, s->stream));
        return PMG_OK;
    }
    PMG_CUDA(cudaGraphLaunch(ge, s->stream));
    count_launch(gk);
    return PMG_OK;
}

// ---- optional phase trace of the distributed cycle (PMG_DIST_TRACE=1): CUDA events between the phases ----
struct TraceMark {
    const char *label;
    int level;
    cudaEvent_t ev;
};
static std::vector<TraceMark> g_trace;
static int g_trace_on = -1;
static void trace_mark(pmg_solver *s, const char *label, int level)
{
    if (g_trace_on < 0) {
        const char *e = getenv("PMG_DIST_TRACE");
        g_trace_on = (e && e[0] == '1') ? 1 : 0;
    }
    if (!g_trace_on) return;
    TraceMark m{label, level, nullptr};
    cudaEventCreate(&m.ev);
    cudaEventRecord(m.ev, s->stream);
    g_trace.push_back(m);
}

// The fused cycle on row slabs (DESIGN.md section 6).  Per level visit: ONE halo exchange of PADY rows on
// the way down (the iterate on the finest level / on repeated W visits, the restricted right-hand side on a
// first visit) and none on the way up -- Pass A also finishes 6 halo rows of xb, Pass B 4 halo rows of x,
// which is exactly what the parent's prolongation and this level's second pass read.
// The exchange runs on `comm_stream` WHILE Pass A works on the interior rows [8, ny-8), which need no halo;
// the two boundary strips [-6, 8) and [ny-8, ny+6) follow once the halo has landed.
// Deep-sweep schedule (max(nu1, nu2) >= 3): Pass A finishes pass_a_depth rows, Pass B pass_b_ext rows, and before Pass B
// of level l the up_exchange_rows(l) coarse rows beyond what the child finished come from the neighbours.
static pmg_status cycle_dist(pmg_solver *s, int l, bool w_form, bool x_is_zero, bool want_norm, int *n_partials,
                             const int *done);
static pmg_status up_exchange(pmg_solver *s, int k, int m, FusedLevel &v);

// First level of the middle graph: the smallest lg >= 1 such that the slab levels lg .. agg_level-1 all run on the
// compute stream alone (no interior / boundary split, hence no cross-stream events); 0 = no graph.
static int mid_graph_first_level(const pmg_solver *s, bool w_form)
{
    // (not with the deep-sweep schedule: d_epochs holds one halo epoch per level, and its up-exchange would need a
    // second one; the graph only trims launch latency on short slab levels, measured for nu = 2)
    if (!s->mid_graph_on || w_form || !s->p2p || !s->p2p_fused || !s->p2p_gather || !s->coarse_redundant ||
        !s->cycle_has_collective || s->d_epochs == nullptr || g_trace_on == 1 || !s->cfg.use_graph || deep_sweeps(s->cfg))
        return 0;
    int lg = s->agg_level;
    while (lg > 1 && s->lv[lg - 1].ny < s->split_min_rows) --lg;
    return lg < s->agg_level ? lg : 0;
}

// levels lg .. coarsest and back: epochs to device memory, then the graph of this all-gather parity
static pmg_status run_mid_graph(pmg_solver *s, int lg)
{
    IntPack16 vals{};
    for (int l = lg; l < s->agg_level; ++l) vals.v[l] = ++s->lv[l].halo_epoch;
    vals.v[15] = ++s->agg_epoch;
    const int parity = s->agg_epoch & 1;
    s->aslab.f = s->agg_f[parity] + level_origin(s->aslab.n);
    launch_set_ints(s->d_epochs, vals, 16, s->stream);
    cudaGraphExec_t &ge = s->mid_graph[parity];
    int &gk = s->mid_graph_kernels[parity];
    if (ge == nullptr) {
        const unsigned long long before = launches_so_far();
        PMG_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
        s->capturing_mid = true;  // cycle_dist: no epoch increments, epochs through d_epochs, plain coarse launches
        pmg_status rc = cycle_dist(s, lg, false, true, false, nullptr, nullptr);
        s->capturing_mid = false;
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamEndCapture(s->stream, &g);
        // nothing ran: take back the epochs this visit had claimed, or the next visit would wait for one too many
        auto roll_back = [&]() {
            for (int l = lg; l < s->agg_level; ++l) --s->lv[l].halo_epoch;
            --s->agg_epoch;
        };
        if (e != cudaSuccess) {
            roll_back();
            return fail(PMG_ERR_CUDA, std::string("cudaStreamEndCapture (middle graph): ") + cudaGetErrorString(e));
        }
        if (rc != PMG_OK) {
            cudaGraphDestroy(g);
            roll_back();
            return rc;
        }
        gk = (int)(launches_so_far() - before);
        e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) {
            roll_back();
            return fail(PMG_ERR_CUDA, std::string("cudaGraphInstantiate (middle graph): ") + cudaGetErrorString(e));
        }
        PMG_CUDA(cudaGraphLaunch(ge, s->stream));
        return PMG_OK;
    }
    PMG_CUDA(cudaGraphLaunch(ge, s->stream));
    count_launch(gk);
    return PMG_OK;
}

static pmg_status cycle_dist(pmg_solver *s, int l, bool w_form, bool x_is_zero, bool want_norm, int *n_partials,
                             const int *done)
{
    const pmg_config &c = s->cfg;
    Level &L = s->lv[l];
    const bool last_slab = (l + 1 == s->agg_level);
    Level &K = last_slab ? s->aslab : s->lv[l + 1];
    const bool up_nb = s->rank > 0, dn_nb = s->rank < s->n_ranks - 1;
    const int da = pass_a_depth(c);
    pmg_status rc;
    trace_mark(s, "begin", l);
    // NVLink all-gather of the agglomerated level into the double-buffered slab.  Two buffers are enough for ANY
    // number of gathers per cycle (W form: gamma^l of them): gather k+2 re-uses the buffer of gather k, and a rank
    // re-writes that buffer (Pass A of the last slab level) only after ITS gather k+1 returned, i.e. after every
    // rank published epoch k+1, which each rank does from its gather-(k+1) launch -- stream-ordered after its
    // gather-k launch finished reading.  PMG_P2P_GATHER_W=0 sends W-cycles back to the NCCL all-gather.
    const bool pull_gather = last_slab && s->p2p_gather && s->coarse_redundant && s->cycle_has_collective &&
                             (!w_form || c.gamma == 1 || s->p2p_gather_w);
    if (pull_gather) {
        if (!s->capturing_mid) ++s->agg_epoch;  // (run_mid_graph advanced it before the capture / replay)
        s->aslab.f = s->agg_f[s->agg_epoch & 1] + level_origin(s->aslab.n);
    } else if (last_slab) {
        s->aslab.f = s->agg_f[0] ? s->agg_f[0] + level_origin(s->aslab.n) : s->aslab.f;
    }
    // (1)+(2) halo exchange and Pass A.  Large slabs: the exchange AND the two boundary strips
    // [-6, 8), [ny-8, ny+6) run on the communication stream while the compute stream works on the interior
    // rows [8, ny-8), which need no halo; the streams join before the next level.  Small slabs (the interior
    // is shorter than an exchange): exchange, then one launch.
    // cross-cycle solve (level 0): from the second cycle on there is no Pass A -- the previous cycle's cross pass did its work
    const bool cross = (l == 0) && s->cross_active;
    const bool skip_pass_a = cross && s->cross_count > 0;
    double *halo_field = skip_pass_a ? nullptr : (!x_is_zero ? L.x : (l > 0 ? L.f : nullptr));
    const bool split = halo_field && !cross && L.ny >= s->split_min_rows && (up_nb || dn_nb);
    FusedLevel v = fused_view(L);
    HaloPeers halo_peers{};
    if (halo_field) {
        int epoch = 0;
        if (s->p2p) {  // publish "my boundary rows of this level are final" in the neighbours' inboxes
            epoch = s->capturing_mid ? 0 : ++L.halo_epoch;  // captured launches take the epoch from d_epochs[l]
            if (!s->p2p_fused)  // (the fused exchange publishes from inside Pass A, see hp.pub_up / pub_dn below)
                launch_halo_signal(up_nb ? s->up_flags + 2 * l + 1 : nullptr, dn_nb ? s->dn_flags + 2 * l : nullptr, epoch,
                                   s->stream);
        }
        // tall slabs: exchange + boundary strips on the communication stream beside the interior pass;
        // short slabs: everything in order on the compute stream (no cross-stream hops)
        cudaStream_t xs = split ? s->comm_stream : s->stream;
        if (split || !s->p2p) {
            xs = s->comm_stream;
            PMG_CUDA(cudaEventRecord(s->ev_ready, s->stream));
            PMG_CUDA(cudaStreamWaitEvent(s->comm_stream, s->ev_ready, 0));
        }
        HaloPeers hp{};
        if (s->p2p && s->p2p_fused) {
            // FUSED: Pass A waits for the neighbours' epoch itself and reads their boundary rows in place over
            // NVLink; the f rows it fetches are kept in the local halo rows for Pass B.  Level 0 keeps reading
            // its static local f halo (exchanged once in pmg_set_rhs).
            if (!x_is_zero) {
                hp.x_up = up_nb ? L.up_x + (ptrdiff_t)PADY * L.pitch : nullptr;
                hp.x_dn = dn_nb ? L.dn_x : nullptr;
                hp.x_keep = L.x;
            }
            if (l > 0) {
                hp.f_up = up_nb ? L.up_f + (ptrdiff_t)PADY * L.pitch : nullptr;
                hp.f_dn = dn_nb ? L.dn_f : nullptr;
                hp.f_keep = L.f;
            }
            hp.flag_up = up_nb ? s->d_flags + 2 * l : nullptr;
            hp.flag_dn = dn_nb ? s->d_flags + 2 * l + 1 : nullptr;
            hp.pub_up = up_nb ? s->up_flags + 2 * l + 1 : nullptr;  // published by the FIRST launch that carries hp
            hp.pub_dn = dn_nb ? s->dn_flags + 2 * l : nullptr;
            hp.epoch = epoch;
            hp.epoch_base = s->capturing_mid ? s->d_epochs + l : nullptr;
            hp.err = s->d_comm_err;
            hp.abort = &s->d_ctrl->done;  // a timed-out wait also stops Pass B(0) from committing (see below)
        } else if (s->p2p) {  // separate pull kernel: neighbours' rows are copied into the local halo rows
            const bool is_x = (halo_field == L.x);
            launch_halo_pull(halo_field, L.ny, L.pitch, PADY, is_x ? L.up_x : L.up_f, is_x ? L.dn_x : L.dn_f,
                             s->d_flags + 2 * l, s->d_flags + 2 * l + 1, epoch, s->d_comm_err, xs, &s->d_ctrl->done);
        } else if ((rc = comm_halo_exchange(halo_field, L.ny, L.pitch, PADY, xs)) != PMG_OK) {
            return rc;
        }
        halo_peers = hp;
        if (split) {
            v.hp = hp;
            if (up_nb) {
                v.span_lo = -da;
                v.span_hi = PADY;
                launch_fused_down(v, K.f, K.pitch, c.nu1, c.omega, x_is_zero, s->comm_stream, nullptr);
                v.hp.pub_up = v.hp.pub_dn = nullptr;  // published once
            }
            if (dn_nb) {
                v.span_lo = L.ny - PADY;
                v.span_hi = L.ny + da;
                launch_fused_down(v, K.f, K.pitch, c.nu1, c.omega, x_is_zero, s->comm_stream, nullptr);
            }
            v.hp = HaloPeers{};
        }
        if (xs == s->comm_stream) PMG_CUDA(cudaEventRecord(s->ev_halo, s->comm_stream));
    }
    const bool halo_on_comm = halo_field && (split || !s->p2p);
    if (split) {
        v.span_lo = up_nb ? PADY : 0;
        v.span_hi = dn_nb ? L.ny - PADY : L.ny;
        launch_fused_down(v, K.f, K.pitch, c.nu1, c.omega, x_is_zero, s->stream, nullptr);
        trace_mark(s, "passA_in", l);
        PMG_CUDA(cudaStreamWaitEvent(s->stream, s->ev_halo, 0));
        trace_mark(s, "passA_bd", l);
    } else if (!skip_pass_a) {
        if (halo_on_comm) PMG_CUDA(cudaStreamWaitEvent(s->stream, s->ev_halo, 0));
        trace_mark(s, "halo", l);
        v.span_lo = up_nb ? -da : 0;
        v.span_hi = dn_nb ? L.ny + da : L.ny;
        v.hp = halo_peers;  // fused exchange (null when the halo rows were copied in)
        launch_fused_down(v, K.f, K.pitch, c.nu1, c.omega, x_is_zero, s->stream, nullptr);
        trace_mark(s, "passA", l);
    }
    int reps = w_form ? c.gamma : 1;
    if (!last_slab && !s->capturing_mid && mid_graph_first_level(s, w_form) == l + 1) {
        if ((rc = run_mid_graph(s, l + 1)) != PMG_OK) return rc;  // everything below this level: one graph launch
    } else if (!last_slab) {
        for (int k = 0; k < reps; ++k)
            if ((rc = cycle_dist(s, l + 1, w_form, k == 0, false, nullptr, done)) != PMG_OK) return rc;
    } else {
        Level &A = s->lv[s->agg_level];
        const int *y0 = s->y0s[s->agg_level].data(), *y1 = s->y1s[s->agg_level].data();
        if (s->coarse_redundant) {
            // every rank receives the whole first agglomerated level and solves it: no scatter, no idle ranks
            if (pull_gather) {
                // publishes "my slab is final" to every rank, then pulls theirs (one launch)
                launch_gather_pull(A.f, A.pitch, y1[0] - y0[0], s->d_agg_srcs[s->agg_epoch & 1], s->d_flags + 32,
                                   s->n_ranks, s->rank, s->capturing_mid ? 0 : s->agg_epoch, s->d_comm_err, s->stream,
                                   s->d_agg_slots, s->capturing_mid ? s->d_epochs + 15 : nullptr, &s->d_ctrl->done);
            } else if ((rc = comm_allgather_rows(K.f, A.f, y1[0] - y0[0], A.pitch, s->stream)) != PMG_OK) {
                return rc;
            }
            trace_mark(s, "allgather", l + 1);
            if ((rc = coarse_solve_redundant(s, w_form, reps)) != PMG_OK) return rc;
            trace_mark(s, "coarse", l + 1);
            // no scatter: Pass B below reads its coarse rows straight out of the whole level (coarse_x)
        } else {
            if ((rc = comm_gather_rows(K.f, A.f, A.pitch, y0, y1, s->stream)) != PMG_OK) return rc;
            trace_mark(s, "gather", l + 1);
            if (s->rank == 0)
                for (int k = 0; k < reps; ++k)
                    if ((rc = cycle_fused(s, s->agg_level, w_form, k == 0, false, nullptr, nullptr)) != PMG_OK) return rc;
            trace_mark(s, "coarse", l + 1);
            if ((rc = comm_scatter_rows(A.x, K.x, A.n, A.pitch, y0, y1, 4, s->stream)) != PMG_OK) return rc;
        }
        trace_mark(s, "scatter", l + 1);
    }
    trace_mark(s, "child", l);
    // (3) Pass B.  Only the finest level's Pass B changes state that outlives the cycle (x_0), so it alone
    // honours the device-side `done` flag -- after waiting for the previous cycle's norm, which was combined
    // on the communication stream while this cycle was already running.
    if (l == 0 && s->norm_pending) {
        PMG_CUDA(cudaStreamWaitEvent(s->stream, s->ev_norm, 0));
        s->norm_pending = false;
    }
    {
        FusedLevel v = fused_view(L);
        const int e = pass_b_ext(c, l);
        v.ext_lo = up_nb ? e : 0;
        v.ext_hi = dn_nb ? e : 0;
        // coarse correction: the child slab's iterate, or -- below the last slab level, where every rank holds the
        // whole agglomerated level -- that level's rows around my slab, read in place (same pitch; the rows beyond
        // the grid are the level's zero padding, exactly what a slab's halo rows hold there)
        const double *coarse_x = K.x;
        if (last_slab && s->coarse_redundant) {
            const Level &A = s->lv[s->agg_level];
            coarse_x = A.x + (ptrdiff_t)s->y0s[s->agg_level][s->rank] * A.pitch;
        }
        // with peer-memory exchanges the finest level's last pass ALWAYS looks at the control block's flag: a wait
        // that timed out raises it (HaloPeers::abort), so an iterate built on stale halo rows is never committed
        const int *guard = done ? done : (s->p2p ? &s->d_ctrl->done : nullptr);
        if (cross) {
            // Pass B of this cycle and Pass A of the next one in one sweep: reads xb_k (buffer `in`, whose halo rows the
            // first cycle's Pass A computed and every later cycle pulls from the neighbours in the halo prologue), writes
            // x_k into the iterate's array, xb_{k+1} into the other buffer and the next cycle's coarse right-hand side
            const int par = s->cross_count & 1;
            v.ext_lo = v.ext_hi = 0;
            v.xb = par ? s->xc : L.xb;
            double *out = par ? L.xb : s->xc;
            if (s->cross_count > 0) {
                HaloPeers hp{};
                hp.x_up = up_nb ? L.up_xb[par] + (ptrdiff_t)PADY * L.pitch : nullptr;
                hp.x_dn = dn_nb ? L.dn_xb[par] : nullptr;
                hp.x_keep = v.xb;
                hp.flag_up = up_nb ? s->d_flags + 0 : nullptr;
                hp.flag_dn = dn_nb ? s->d_flags + 1 : nullptr;
                hp.pub_up = up_nb ? s->up_flags + 1 : nullptr;
                hp.pub_dn = dn_nb ? s->dn_flags + 0 : nullptr;
                hp.epoch = ++L.halo_epoch;
                hp.err = s->d_comm_err;
                hp.abort = &s->d_ctrl->done;
                v.hp = hp;
            }
            launch_fused_cross(v, out, coarse_x, K.f, K.pitch, c.omega, c.prolong_mode, s->d_partials, n_partials, s->stream,
                               guard);
            ++s->cross_count;
        } else {
            // deep-sweep schedule: the child slab's rows beyond those its Pass B finished (the whole agglomerated level
            // is read in place and needs none)
            const int m = last_slab ? 0 : up_exchange_rows(c, l);
            if (m > 0 && (rc = up_exchange(s, l + 1, m, v)) != PMG_OK) return rc;
            const bool fused_norm = want_norm && pass_b_norm_fits(c);
            launch_fused_up(v, coarse_x, K.pitch, c.nu2, c.omega, c.prolong_mode, fused_norm ? s->d_partials : nullptr,
                            n_partials, s->stream, l == 0 ? guard : nullptr);
            if (want_norm && !fused_norm) {
                // xb does not reach the extra row the fused norm reads (nu1 + nu2 = 7, 8): sum (f - A x)^2 over the owned
                // rows in a pass of its own, after an exchange of one row of the new iterate
                if ((rc = comm_halo_exchange(L.x, L.ny, L.pitch, 1, s->stream)) != PMG_OK) return rc;
                const int ga = std::max(L.y0, 1), gb = std::min(L.y0 + L.ny, L.n - 1);  // owned interior rows
                const int a = ga - L.y0, b = gb - L.y0;
                const int np = launch_residual_partials(L.x + (ptrdiff_t)(a - 1) * L.pitch, L.f + (ptrdiff_t)(a - 1) * L.pitch,
                                                        L.n, b - a + 2, L.pitch, L.pitch, L.h, s->d_partials, s->stream);
                if (n_partials) *n_partials = np;
            }
        }
    }
    trace_mark(s, "passB", l);
    return PMG_OK;
}

// Deep-sweep schedule: rows pass_b_ext(k) + 1 .. + m beyond the slab of level k's iterate from the neighbours, before
// Pass B of level k - 1 (v: that pass) reads them.  Over NVLink with PMG_P2P_FUSED on (default) in Pass B's coarse
// prologue; with a pull kernel ahead of it otherwise; by NCCL without peer access.  The last two move all
// pass_b_ext(k) + m rows, each side one contiguous block.  Every rank runs the same sequence of cycles, so the epochs
// agree; a neighbour re-writes its rows only after its next Pass A of level k waited for this rank's epoch of that
// level, which this rank publishes after the pass below.
static pmg_status up_exchange(pmg_solver *s, int k, int m, FusedLevel &v)
{
    Level &K = s->lv[k];
    const bool up_nb = s->rank > 0, dn_nb = s->rank < s->n_ranks - 1;
    const int from = pass_b_ext(s->cfg, k);
    if (!s->p2p) return comm_halo_exchange(K.x, K.ny, K.pitch, from + m, s->stream);
    const int epoch = ++K.up_epoch;
    const int slot = UP_FLAG_SLOT + 2 * k;
    if (!s->p2p_fused) {
        launch_halo_signal(up_nb ? s->up_flags + slot + 1 : nullptr, dn_nb ? s->dn_flags + slot : nullptr, epoch, s->stream);
        launch_halo_pull(K.x, K.ny, K.pitch, from + m, up_nb ? K.up_x + (ptrdiff_t)(PADY - from - m) * K.pitch : nullptr,
                         dn_nb ? K.dn_x : nullptr, s->d_flags + slot, s->d_flags + slot + 1, epoch, s->d_comm_err, s->stream,
                         &s->d_ctrl->done);
        return PMG_OK;
    }
    HaloPeers hp{};
    hp.x_up = up_nb ? K.up_x + (ptrdiff_t)PADY * K.pitch : nullptr;
    hp.x_dn = dn_nb ? K.dn_x : nullptr;
    hp.x_keep = K.x;
    hp.flag_up = up_nb ? s->d_flags + slot : nullptr;
    hp.flag_dn = dn_nb ? s->d_flags + slot + 1 : nullptr;
    hp.pub_up = up_nb ? s->up_flags + slot + 1 : nullptr;
    hp.pub_dn = dn_nb ? s->dn_flags + slot : nullptr;
    hp.epoch = epoch;
    hp.err = s->d_comm_err;
    hp.abort = &s->d_ctrl->done;  // a timed-out wait also stops the finest level's Pass B from committing
    hp.rows_from = from;
    hp.rows_count = m;
    v.hp = hp;
    return PMG_OK;
}

// sum over this rank's owned interior rows of (f - A x)^2 -> d_scalar[0], then the rank-ordered global sum
static pmg_status dist_residual_norm2(pmg_solver *s)
{
    Level &L = s->lv[0];
    pmg_status rc = comm_halo_exchange(L.x, L.ny, L.pitch, PADY, s->stream);
    if (rc != PMG_OK) return rc;
    int ga = std::max(L.y0, 1), gb = std::min(L.y0 + L.ny, L.n - 1);  // owned interior rows [ga, gb)
    int a = ga - L.y0, b = gb - L.y0;
    // a window whose own "ring" rows are local rows a-1 and b
    launch_residual_norm2(L.x + (ptrdiff_t)(a - 1) * L.pitch, L.f + (ptrdiff_t)(a - 1) * L.pitch, L.n, b - a + 2,
                          L.pitch, L.pitch, L.h, s->d_partials, s->d_scalar, s->stream);
    if ((rc = comm_allgather_double(s->d_scalar, s->d_gather, s->stream)) != PMG_OK) return rc;
    launch_final_sum(s->d_gather, s->n_ranks, s->d_scalar, s->stream);
    return PMG_OK;
}

static pmg_status residual_norm2_async(pmg_solver *s)
{
    if (s->dist) return dist_residual_norm2(s);
    Level &L = s->lv[0];
    if (s->cfg.norm_mode == PMG_NORM_SEQUENTIAL)
        launch_residual_norm2_sequential(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, s->d_scalar, s->stream);
    else
        launch_residual_norm2(L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.h, s->d_partials, s->d_scalar, s->stream);
    return PMG_OK;
}

static pmg_status read_scalar(pmg_solver *s, double *out)
{
    PMG_CUDA(cudaMemcpyAsync(s->h_scalar, s->d_scalar, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    PMG_CUDA(cudaGetLastError());
    *out = *s->h_scalar;
    return PMG_OK;
}

// ---- F-cycle -------------------------------------------------------------------------------------------
static pmg_status ensure_fmg(pmg_solver *s)
{
    if (s->fmg_ready) return PMG_OK;
    for (Level &L : s->lv) {
        // DynamicGridUtils.hpp:120-122 with globals a = p = q = 1: sin(p * M_PI * x / a), x = i*h
        std::vector<double> tab(L.n);
        const double a = 1.0, p = 1.0;
        for (int i = 0; i < L.n; ++i) {
            double x = i * L.h;
            tab[i] = std::sin(p * M_PI * x / a);
        }
        PMG_CUDA(cudaMalloc((void **)&L.d_sin, L.n * sizeof(double)));
        PMG_CUDA(cudaMemcpy(L.d_sin, tab.data(), L.n * sizeof(double), cudaMemcpyHostToDevice));
    }
    pmg_status rc = alloc_zero(&s->base_f_fmg0, s->lv[0].elems);
    if (rc != PMG_OK) return rc;
    s->f_fmg0 = s->base_f_fmg0 + level_origin(s->lv[0].n);
    s->fmg_ready = true;
    return PMG_OK;
}

static void analytic_rhs(pmg_solver *s, const Level &L, double *f)
{
    const double a = 1.0, p = 1.0, q = 1.0;
    double factor = (M_PI * M_PI / (a * a)) * (p * p + q * q);  // DynamicGridUtils.hpp:113
    launch_rhs_separable(f, L.pitch, L.n, L.n, factor, L.d_sin, L.d_sin, s->stream);
}

// MultigridSolver::f_cycle (MultiGrid.hpp:138-183): nested iteration from level l_init -- whose x / f arrays hold the
// starting iterate and right-hand side -- up to the finest level, with the ANALYTIC right-hand side on every finer
// level (:162); the result is the finest level's iterate.
// norm_np (nullable): if the last V-cycle can deliver the residual norm of the result (its Pass B on level 0 sums
// (f - A x)^2 against the analytic right-hand side), *norm_np receives the number of partial sums in s->d_partials; -1 if not
static pmg_status fmg_up_from(pmg_solver *s, int l_init, int *norm_np = nullptr)
{
    if (norm_np) *norm_np = -1;
    const pmg_config &c = s->cfg;
    pmg_status rc = PMG_OK;
    double *user_f = s->lv[0].f;
    for (int l = l_init - 1; l >= 0; --l) {
        Level &K = s->lv[l + 1];
        Level &L = s->lv[l];
        // smoother->smooth(phi_current, f_current, N, N, h, 3)  (:153)
        if (s->fused && fused_supported(c.fmg_sweeps) && K.n * K.n > SMALL_MAX_POINTS) {
            launch_fused_down(fused_view(K), nullptr, 0, c.fmg_sweeps, c.omega, false, s->stream);
            std::swap(K.x, K.xb);
            std::swap(K.base_x, K.base_xb);
        } else {
            rc = smooth_operator(s, l + 1, c.fmg_sweeps, false);
            if (rc != PMG_OK) break;
        }
        double *f_l = (l == 0) ? s->f_fmg0 : L.f;
        if (l != 0 || !s->fmg0_rhs_cached) analytic_rhs(s, L, f_l);                          // :162
        if (l == 0) s->fmg0_rhs_cached = true;  // level 0's copy is a dedicated array: written once per hierarchy
        // On the levels the V-cycle streams (n >= 513: never the cluster / single-CTA kernels), "zero the fine grid, add
        // P phi_coarse" (:161, :164) is folded into Pass A of the V-cycle (:167): the prolonged iterate is never written.
        const bool fold = s->fused && L.n >= 513 && L.n > c.n_coarse && fused_down_prolong_supported(c.nu1) &&
                          !c.smoother_fp32 && c.smoother == PMG_SMOOTHER_JACOBI;
        if (!fold) {
            launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);                               // :161
            launch_prolong_add(K.x, L.x, K.n, L.n, K.pitch, L.pitch, c.prolong_mode, s->stream);  // :164
        }
        if (l == 0) L.f = s->f_fmg0;
        // the runner's residual after the pass (MultiGridTestRunner.hpp:210-211) is taken against the caller's f: the
        // last Pass B can deliver it only if that f IS the analytic right-hand side (pmg_set_rhs_sine, untouched since)
        const bool fold_norm = norm_np != nullptr && l == 0 && s->fused && s->rhs_is_analytic &&
                               c.norm_mode != PMG_NORM_SEQUENTIAL && L.n >= 513 && L.n > c.n_coarse;
        int np = 0;
        rc = s->fused ? cycle_fused(s, l, false, false, fold_norm, fold_norm ? &np : nullptr, nullptr, fold ? &K : nullptr)
                      : cycle_operator(s, l, false, false);  // :167
        if (fold_norm && rc == PMG_OK) *norm_np = np;
        if (l == 0) L.f = user_f;
        if (rc != PMG_OK) break;
    }
    s->lv[0].f = user_f;
    return rc;
}

// MultigridSolver::compute_coarsest_grid (MultiGrid.hpp:28-55): repeated full weighting from level 0 down to level
// l_out.  Level 0's input is `src0`; the scratch of every coarser level is its xb array (ring == 0).
static void restrict_chain(pmg_solver *s, const double *src0, int l_out)
{
    for (int l = 0; l < l_out; ++l) {
        const Level &L = s->lv[l];
        Level &K = s->lv[l + 1];
        launch_restrict(l == 0 ? src0 : L.xb, K.xb, L.n, K.n, L.pitch, K.pitch, s->stream);
    }
}

// The runner's F-cycle wrapper (MultiGridTestRunner.hpp:192-205) = compute_coarsest_grid + f_cycle from the
// coarsest level with the analytic coarse right-hand side (:142).
static pmg_status cycle_f(pmg_solver *s, int *norm_np = nullptr)
{
    if (norm_np) *norm_np = -1;
    pmg_status rc = ensure_fmg(s);
    if (rc != PMG_OK) return rc;
    const int nl = (int)s->lv.size();
    int lc = nl - 1;  // index of the coarsest level (n == n_coarse, or the 3x3 grid)
    if (lc == 0) return PMG_OK;  // N <= N_coarse: f_cycle's while loop never runs (MultiGrid.hpp:150)
    drop_graphs(s);              // the pass below may swap x/xb roles on levels >= 1
    // (1) phi restricted down to the coarsest grid
    restrict_chain(s, s->lv[0].x, lc);
    launch_copy2d(s->lv[lc].x, s->lv[lc].pitch, s->lv[lc].xb, s->lv[lc].pitch, s->lv[lc].n, s->lv[lc].n, s->stream);
    // (2) nested iteration upwards
    analytic_rhs(s, s->lv[lc], s->lv[lc].f);  // MultiGridTestRunner.hpp:142
    return fmg_up_from(s, lc, norm_np);
}

// PMG_CYCLE_FMG: one full-multigrid pass for an arbitrary right-hand side and Dirichlet ring (pmg.h; not a
// reference function -- SURVEY.md 8f-2; specification: the CPU checker's orc_fmg_general).  The coarse right-hand
// sides are the levels' own f arrays; r0 = f - A x is never stored (launch_residual_restrict forms R r0 directly).
static pmg_status cycle_fmg_general(pmg_solver *s)
{
    const pmg_config &c = s->cfg;
    const int lc = (int)s->lv.size() - 1;
    Level &L0 = s->lv[0];
    drop_graphs(s);  // the coarsest solve may swap x / xb roles
    // x = (ring kept, interior 0)
    if (L0.n > 2) launch_fill2d(L0.x + L0.pitch + 1, L0.pitch, L0.n - 2, L0.n - 2, 0.0, s->stream);
    if (lc == 0 || L0.n <= c.n_coarse) return smooth_operator(s, 0, c.coarse_sweeps, false);
    // f_1 = R(f - A x), then the chain of restrictions
    Level &L1 = s->lv[1];
    launch_residual_restrict(L0.x, L0.f, L1.f, L0.n, L1.n, L1.n, 0, L0.pitch, L0.pitch, L1.pitch, L0.h, s->stream);
    for (int l = 1; l < lc; ++l) {
        const Level &L = s->lv[l];
        Level &K = s->lv[l + 1];
        launch_restrict(L.f, K.f, L.n, K.n, L.pitch, K.pitch, s->stream);
    }
    // coarsest level: coarse_sweeps sweeps from zero
    pmg_status rc = smooth_operator(s, lc, c.coarse_sweeps, true);
    if (rc != PMG_OK) return rc;
    // upwards: prolongation into a zeroed level, one V-cycle there; on the finest level the true problem (x, f)
    for (int l = lc - 1; l >= 0; --l) {
        Level &K = s->lv[l + 1];
        Level &L = s->lv[l];
        if (l > 0) launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
        launch_prolong_add(K.x, L.x, K.n, L.n, K.pitch, L.pitch, c.prolong_mode, s->stream);
        rc = s->fused ? cycle_fused(s, l, false, false, false, nullptr) : cycle_operator(s, l, false, false);
        if (rc != PMG_OK) return rc;
    }
    return PMG_OK;
}

// PMG_CYCLE_FMG on row slabs: the operator sequence of cycle_fmg_general, level by level, under the rules of cycle_f_dist
// (below): slab levels (l < agg_level) on slabs with an NCCL halo exchange ahead of every slab operator that reads a
// neighbour row, whole levels redundantly on every rank, the V-cycle of a slab level = cycle_dist started there.  Halo
// depths: the fused residual-restriction reads 2 x rows and 1 f row beyond the slab, the slab restriction 1 f row, the
// slab prolongation 1 coarse row below the slab -- which the child's last Pass B (4 finished rows beyond its slab, see
// cycle_dist; with the deep-sweep schedule an exchange of the child's halo) or the whole agglomerated level read in
// place already holds.  The f halo rows every later cycle_dist(l)
// reads are the ones exchanged in the chain; nothing rewrites f_l before that cycle.  Every rewrite of an array a
// neighbour may still read over NVLink (x_l, f_l) has an NCCL collective in between: the exchanges here and the
// all-gather of the agglomerated level inside each cycle_dist.
static pmg_status cycle_fmg_dist(pmg_solver *s)
{
    if (!s->coarse_redundant)
        return fail(PMG_ERR_UNSUPPORTED, "multi-GPU FMG pass needs equally sized slabs on the first agglomerated level");
    const pmg_config &c = s->cfg;
    const int nl = (int)s->lv.size(), lc = nl - 1, la = s->agg_level;
    const int *ay0 = s->y0s[la].data(), *ay1 = s->y1s[la].data();
    Level &A = s->lv[la];
    Level &L0 = s->lv[0];
    pmg_status rc;
    s->cycle_has_collective = false;  // the agglomerated level travels by NCCL all-gather inside these V-cycles
    drop_graphs(s);                   // the coarsest solve may swap the x / xb roles of a whole level
    if (s->agg_f[0]) s->aslab.f = s->agg_f[0] + level_origin(s->aslab.n);  // the buffer the NCCL all-gather sends from
    // (1) x = (ring kept, interior 0) on my rows; halo rows of x and f for the residual
    {
        const int ga = std::max(L0.y0, 1), gb = std::min(L0.y0 + L0.ny, L0.n - 1);
        if (gb > ga) launch_fill2d(L0.x + (ptrdiff_t)(ga - L0.y0) * L0.pitch + 1, L0.pitch, L0.n - 2, gb - ga, 0.0, s->stream);
        if ((rc = comm_halo_exchange(L0.x, L0.ny, L0.pitch, PADY, s->stream)) != PMG_OK) return rc;
        if ((rc = comm_halo_exchange(L0.f, L0.ny, L0.pitch, PADY, s->stream)) != PMG_OK) return rc;
    }
    // (2) f_1 = R(f - A x) on my coarse rows; (3) f_{l+1} = R f_l down the slab levels, all-gathered into the whole level
    // the redundant V-cycles read, then restricted redundantly
    for (int l = 0; l < lc; ++l) {
        Level &L = s->lv[l];
        if (l < la) {
            Level &K = (l + 1 == la) ? s->aslab : s->lv[l + 1];
            if (l == 0) {
                launch_residual_restrict(L.x, L.f, K.f, L.n, K.n, K.ny, K.y0, L.pitch, L.pitch, K.pitch, L.h, s->stream);
            } else {
                if ((rc = comm_halo_exchange(L.f, L.ny, L.pitch, PADY, s->stream)) != PMG_OK) return rc;
                launch_restrict_rows(L.f, K.f, K.n, K.ny, K.y0, L.pitch, K.pitch, s->stream);
            }
            if (l + 1 == la && (rc = comm_allgather_rows(K.f, A.f, ay1[0] - ay0[0], A.pitch, s->stream)) != PMG_OK) return rc;
        } else {
            Level &K = s->lv[l + 1];
            launch_restrict(L.f, K.f, L.n, K.n, L.pitch, K.pitch, s->stream);
        }
    }
    // (4) coarsest level: coarse_sweeps sweeps from zero, on every rank
    if ((rc = smooth_operator(s, lc, c.coarse_sweeps, true)) != PMG_OK) return rc;
    // (5) upwards: e_l = P e_{l+1} into zeros, one V-cycle on (e_l, f_l); (6) level 0: x += P e_1, one V-cycle on (x, f)
    for (int l = lc - 1; l >= 0; --l) {
        Level &K = s->lv[l + 1];
        Level &L = s->lv[l];
        if (l >= la) {
            launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
            launch_prolong_add(K.x, L.x, K.n, L.n, K.pitch, L.pitch, c.prolong_mode, s->stream);
            rc = cycle_fused(s, l, false, false, false, nullptr);
        } else {
            if (l > 0) PMG_CUDA(cudaMemsetAsync(L.base_x, 0, L.elems * sizeof(double), s->stream));
            // the coarse iterate: the child slab, or my rows of the whole agglomerated level read in place.  The
            // deep-sweep schedule's Pass B may finish no row beyond the child slab: its halo rows are exchanged.
            if (l + 1 < la && deep_sweeps(c) && (rc = comm_halo_exchange(K.x, K.ny, K.pitch, PADY, s->stream)) != PMG_OK)
                return rc;
            const double *e = (l + 1 == la) ? A.x + (ptrdiff_t)ay0[s->rank] * A.pitch : K.x;
            launch_prolong_add_rows(e, L.x, L.n, L.ny, L.y0, K.pitch, L.pitch, c.prolong_mode, s->stream);
            rc = cycle_dist(s, l, false, false, false, nullptr, nullptr);
        }
        if (rc != PMG_OK) return rc;
    }
    drop_graphs(s);  // a coarse solve captured above holds x / xb roles the coarsest smoothing may have swapped
    return PMG_OK;
}

// The F-cycle on row slabs.  Same operator sequence as cycle_f, level by level:
//   * levels l < agg_level are slabs: every slab operator that reads a neighbour row is preceded by an NCCL halo
//     exchange of PADY rows (set-up work -- a handful of exchanges per level, not on the V-cycle's critical path);
//     the FMG smoothing runs as passes of <= 2 sweeps (8 halo rows in, >= 6 valid rows out), x -> xb -> x, so the
//     x / f pointers the neighbours have mapped over NVLink never change roles;
//   * levels l >= agg_level are whole on every rank and processed redundantly, exactly as on one GPU (every rank
//     computes bit-identical copies);
//   * the V-cycle of level l is cycle_dist started at level l (cycle_fused for the whole levels).
// Every phase boundary that re-writes an array a neighbour may still be reading over NVLink (x, f of a slab level)
// has an NCCL exchange with that neighbour in between, which orders the write after the neighbour's reads.
static pmg_status cycle_f_dist(pmg_solver *s)
{
    if (!s->coarse_redundant)
        return fail(PMG_ERR_UNSUPPORTED, "multi-GPU F-cycle needs equally sized slabs on the first agglomerated level");
    pmg_status rc = ensure_fmg(s);
    if (rc != PMG_OK) return rc;
    const pmg_config &c = s->cfg;
    const int nl = (int)s->lv.size(), lc = nl - 1, la = s->agg_level;
    const bool up_nb = s->rank > 0, dn_nb = s->rank < s->n_ranks - 1;
    const int *ay0 = s->y0s[la].data(), *ay1 = s->y1s[la].data();
    Level &A = s->lv[la];
    s->cycle_has_collective = false;  // the agglomerated level travels by NCCL all-gather inside these V-cycles
    drop_graphs(s);                   // the smoothing of the whole levels below swaps their x / xb roles
    // (1) phi restricted down to the coarsest grid (MultiGridTestRunner.hpp:192-200); scratch = the xb arrays
    for (int l = 0; l < lc; ++l) {
        Level &L = s->lv[l];
        if (l < la) {
            double *fine = (l == 0) ? L.x : L.xb;
            if ((rc = comm_halo_exchange(fine, L.ny, L.pitch, PADY, s->stream)) != PMG_OK) return rc;
            Level &K = (l + 1 == la) ? s->aslab : s->lv[l + 1];
            double *coarse = (l + 1 == la) ? K.x : K.xb;
            launch_restrict_rows(fine, coarse, K.n, K.ny, K.y0, L.pitch, K.pitch, s->stream);
            if (l + 1 == la && (rc = comm_allgather_rows(K.x, A.xb, ay1[0] - ay0[0], A.pitch, s->stream)) != PMG_OK)
                return rc;
        } else {
            Level &K = s->lv[l + 1];
            launch_restrict(L.xb, K.xb, L.n, K.n, L.pitch, K.pitch, s->stream);
        }
    }
    launch_copy2d(s->lv[lc].x, s->lv[lc].pitch, s->lv[lc].xb, s->lv[lc].pitch, s->lv[lc].n, s->lv[lc].n, s->stream);
    // (2) nested iteration upwards with the ANALYTIC right-hand side on every level (MultiGrid.hpp:150-170)
    const double factor = (M_PI * M_PI / (1.0 * 1.0)) * (1.0 * 1.0 + 1.0 * 1.0);  // DynamicGridUtils.hpp:113, a = p = q = 1
    double *user_f = s->lv[0].f;
    analytic_rhs(s, s->lv[lc], s->lv[lc].f);
    for (int l = lc - 1; l >= 0; --l) {
        Level &K = s->lv[l + 1];
        Level &L = s->lv[l];
        // smoother->smooth(phi_current, f_current, N, N, h, 3)  (:153)
        if (l + 1 >= la) {
            if (fused_supported(c.fmg_sweeps) && K.n * K.n > SMALL_MAX_POINTS) {
                launch_fused_down(fused_view(K), nullptr, 0, c.fmg_sweeps, c.omega, false, s->stream);
                std::swap(K.x, K.xb);
                std::swap(K.base_x, K.base_xb);
            } else if ((rc = smooth_operator(s, l + 1, c.fmg_sweeps, false)) != PMG_OK) {
                break;
            }
        } else {
            double *cur = K.x, *oth = K.xb;
            int left = c.fmg_sweeps;
            do {
                if ((rc = comm_halo_exchange(cur, K.ny, K.pitch, PADY, s->stream)) != PMG_OK) return rc;
                const int b = std::min(2, left);
                if (b > 0) {
                    FusedLevel v = fused_view(K);
                    v.x = cur;
                    v.xb = oth;
                    v.ext_lo = up_nb ? 2 : 0;  // one coarse row beyond the slab feeds the prolongation below
                    v.ext_hi = dn_nb ? 2 : 0;
                    launch_fused_down(v, nullptr, 0, b, c.omega, false, s->stream);
                    std::swap(cur, oth);
                }
                left -= b;
            } while (left > 0);
            if (cur != K.x) {  // odd number of passes: bring rows [-2, ny + 2) back into the x array
                const int a = up_nb ? -2 : 0, b = K.ny + (dn_nb ? 2 : 0);
                PMG_CUDA(cudaMemcpyAsync(K.x - PADX + (ptrdiff_t)a * K.pitch, K.xb - PADX + (ptrdiff_t)a * K.pitch,
                                         (size_t)(b - a) * K.pitch * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
            }
        }
        if (l < la) {
            // analytic RHS of my rows, halo rows included (:162); zeroed iterate (:161); prolongation (:164)
            double *f_l = (l == 0) ? s->f_fmg0 : L.f;
            const int ga = std::max(L.y0 - PADY, 0), gb = std::min(L.y0 + L.ny + PADY, L.n);
            launch_rhs_separable(f_l + (ptrdiff_t)(ga - L.y0) * L.pitch, L.pitch, L.n, gb - ga, factor, L.d_sin,
                                 L.d_sin + ga, s->stream);
            PMG_CUDA(cudaMemsetAsync(L.base_x, 0, L.elems * sizeof(double), s->stream));
            // the coarse iterate: the child slab, or my rows of the whole agglomerated level read in place
            const double *e = (l + 1 == la) ? A.x + (ptrdiff_t)ay0[s->rank] * A.pitch : K.x;
            launch_prolong_add_rows(e, L.x, L.n, L.ny, L.y0, K.pitch, L.pitch, c.prolong_mode, s->stream);
            if (l == 0) L.f = s->f_fmg0;
            rc = cycle_dist(s, l, false, false, false, nullptr, nullptr);  // :167
            if (l == 0) L.f = user_f;
        } else {
            analytic_rhs(s, L, L.f);
            launch_fill2d(L.x, L.pitch, L.n, L.n, 0.0, s->stream);
            launch_prolong_add(K.x, L.x, K.n, L.n, K.pitch, L.pitch, c.prolong_mode, s->stream);
            rc = cycle_fused(s, l, false, false, false, nullptr);
        }
        if (rc != PMG_OK) break;
    }
    s->lv[0].f = user_f;
    drop_graphs(s);  // the smoothing of the whole levels swapped x / xb roles: a captured coarse solve is stale
    return rc;
}

// One fused V/W cycle, replayed from a CUDA graph when allowed.  mode 0: no norm, 1: norm -> d_scalar,
// 2: norm -> device-side solve control (k_cycle_finish) with every kernel honouring ctrl->done.
static bool fused_graph_ok(const pmg_solver *s)
{
    // pointer roles are stable across a fused cycle unless the coarsest solve ping-pongs an odd count
    const Level &Lc = s->lv.back();
    return s->cfg.use_graph && (Lc.n * Lc.n <= SMALL_MAX_POINTS || (s->cfg.coarse_sweeps % 2) == 0);
}

static pmg_status run_fused_graph(pmg_solver *s, bool w, int mode)
{
    if (s->dist) {
        // direct launches (NCCL calls sit between the kernels); norms are combined in rank order
        int np = 0;
        const int *done = (mode == 2) ? &s->d_ctrl->done : nullptr;
        s->cycle_has_collective = (mode != 0);  // the norm all-gather: every rank passes it once per cycle
        pmg_status rc = cycle_dist(s, 0, w, false, mode != 0, &np, done);
        if (rc != PMG_OK || mode == 0) return rc;
        // the norm is combined on the communication stream; only the NEXT cycle's last pass waits for it
        cudaStream_t ns = (mode == 2) ? s->comm_stream : s->stream;
        if (mode == 2) {
            PMG_CUDA(cudaEventRecord(s->ev_passb, s->stream));
            PMG_CUDA(cudaStreamWaitEvent(ns, s->ev_passb, 0));
        }
        launch_final_sum(s->d_partials, np, s->d_scalar, ns);
        if ((rc = comm_allgather_double(s->d_scalar, s->d_gather, ns)) != PMG_OK) return rc;
        if (mode == 1) {
            launch_final_sum(s->d_gather, s->n_ranks, s->d_scalar, ns);
        } else {
            launch_cycle_finish(s->d_gather, s->n_ranks, s->d_ctrl, s->d_hist2, ns);
            PMG_CUDA(cudaEventRecord(s->ev_norm, ns));
            s->norm_pending = true;
        }
        trace_mark(s, "norm", 0);
        return PMG_OK;
    }
    bool graph_ok = fused_graph_ok(s);
    cudaGraphExec_t &ge = s->graph[w ? 1 : 0][mode];
    int &gk = s->graph_kernels[w ? 1 : 0][mode];
    if (graph_ok && ge != nullptr) {
        PMG_CUDA(cudaGraphLaunch(ge, s->stream));
        count_launch(gk);
        return PMG_OK;
    }
    unsigned long long before = launches_so_far();
    if (graph_ok) PMG_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
    int n_partials = 0;
    const int *done = (mode == 2) ? &s->d_ctrl->done : nullptr;
    pmg_status rc = cycle_fused(s, 0, w, false, mode != 0, &n_partials, done);
    if (rc == PMG_OK && mode == 1) launch_final_sum(s->d_partials, n_partials, s->d_scalar, s->stream);
    if (rc == PMG_OK && mode == 2) launch_cycle_finish(s->d_partials, n_partials, s->d_ctrl, s->d_hist2, s->stream);
    if (graph_ok) {
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamEndCapture(s->stream, &g);
        if (e != cudaSuccess) return fail(PMG_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
        if (rc != PMG_OK) {
            cudaGraphDestroy(g);
            return rc;
        }
        // the launches counted during capture are the ones the first replay below executes
        gk = (int)(launches_so_far() - before);
        PMG_CUDA(cudaGraphInstantiate(&ge, g, 0));
        cudaGraphDestroy(g);
        PMG_CUDA(cudaGraphLaunch(ge, s->stream));
    }
    return rc;
}

static pmg_status run_cycle_inner(pmg_solver *s, pmg_cycle_kind kind, bool want_norm);

static pmg_status run_cycle(pmg_solver *s, pmg_cycle_kind kind, bool want_norm)
{
    pmg_status rc = run_cycle_inner(s, kind, want_norm);
    if (const int bad = fused_take_bad_nu())  // a fused launcher was asked for a sweep count it has no instantiation of
        return fail(PMG_ERR_UNSUPPORTED, "fused engine: no kernel for " + std::to_string(bad) + " sweeps per pass");
    return rc;
}

static pmg_status run_cycle_inner(pmg_solver *s, pmg_cycle_kind kind, bool want_norm)
{
    pmg_status rc;
    if (kind == PMG_CYCLE_FMG) {
        rc = s->dist ? cycle_fmg_dist(s) : cycle_fmg_general(s);
        if (rc == PMG_OK && want_norm) rc = residual_norm2_async(s);
        return rc;
    }
    if (kind == PMG_CYCLE_F) {
        int np = -1;
        rc = s->dist ? cycle_f_dist(s) : cycle_f(s, want_norm ? &np : nullptr);
        if (rc == PMG_OK && want_norm) {
            if (np >= 0)
                launch_final_sum(s->d_partials, np, s->d_scalar, s->stream);  // the last Pass B summed (f - A x)^2
            else
                rc = residual_norm2_async(s);
        }
        return rc;
    }
    if (kind != PMG_CYCLE_V && kind != PMG_CYCLE_W) return fail(PMG_ERR_INVALID, "unknown cycle kind");
    bool w = (kind == PMG_CYCLE_W);
    if (s->fused && want_norm && s->cfg.norm_mode == PMG_NORM_SEQUENTIAL) {
        rc = run_cycle_inner(s, kind, false);
        if (rc == PMG_OK) rc = residual_norm2_async(s);
        return rc;
    }
    if (!s->fused) {
        rc = cycle_operator(s, 0, w, false);
        if (rc == PMG_OK && want_norm) rc = residual_norm2_async(s);
        return rc;
    }
    if (!s->dist && ((int)s->lv.size() == 1 || s->lv[0].n <= s->cfg.n_coarse)) {
        rc = cycle_fused(s, 0, w, false, false, nullptr);
        if (rc == PMG_OK && want_norm) rc = residual_norm2_async(s);
        return rc;
    }
    return run_fused_graph(s, w, want_norm ? 1 : 0);
}

}  // namespace pmg

// =========================================================================================================
//                                                C ABI
// =========================================================================================================
extern "C" {

const char *pmg_version(void) { return "pmg-b200 0.1 (sm_100a)"; }

const char *pmg_last_error(void) { return g_last_error.c_str(); }

const char *pmg_status_string(pmg_status s)
{
    switch (s) {
        case PMG_OK: return "ok";
        case PMG_ERR_INVALID: return "invalid argument";
        case PMG_ERR_CUDA: return "CUDA error";
        case PMG_ERR_NO_DEVICE: return "no sm_100 CUDA device (there is no CPU fallback)";
        case PMG_ERR_ALLOC: return "allocation failed";
        case PMG_ERR_COMM: return "communication error";
        case PMG_ERR_UNSUPPORTED: return "unsupported";
    }
    return "unknown";
}

void pmg_config_default(pmg_config *cfg, int n)
{
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->n = n;
    cfg->nu1 = 2;   // reference v1 = 1 -> 2 sweeps (MultiGrid.hpp:15, Smoother.hpp:59)
    cfg->nu2 = 2;
    cfg->omega = 1.0;
    cfg->gamma = 3;  // 2_part_MG/main.cpp:15 alpha = 3
    cfg->n_coarse = 5;
    cfg->coarse_sweeps = 11;
    cfg->fmg_sweeps = 4;
    cfg->prolong_mode = PMG_PROLONG_REFERENCE;
    cfg->engine = PMG_ENGINE_FUSED;
    cfg->smoother_eps = 0.0;
    cfg->device = -1;
    cfg->use_graph = 1;
    cfg->rank = 0;
    cfg->n_ranks = 1;
    cfg->agglomerate_below = 513;
    cfg->norm_mode = PMG_NORM_TREE;
}

unsigned long long pmg_kernel_launches(void) { return launches_so_far(); }

int pmg_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

pmg_status pmg_create(const pmg_config *cfg, pmg_solver **out)
{
    if (!cfg || !out) return fail(PMG_ERR_INVALID, "null argument");
    *out = nullptr;
    if (!is_pow2_plus_1(cfg->n)) return fail(PMG_ERR_INVALID, "n must be 2^k + 1 (k >= 1)");
    if (cfg->n > 46340) return fail(PMG_ERR_INVALID, "n too large");
    if (cfg->nu1 < 0 || cfg->nu2 < 0 || cfg->coarse_sweeps < 0 || cfg->fmg_sweeps < 0 || cfg->gamma < 1)
        return fail(PMG_ERR_INVALID, "negative sweep count or gamma < 1");
    if (!is_pow2_plus_1(cfg->n_coarse)) return fail(PMG_ERR_INVALID, "n_coarse must be 2^k + 1");
    if (!(cfg->omega > 0.0)) return fail(PMG_ERR_INVALID, "omega must be positive");
    if (cfg->norm_mode != PMG_NORM_TREE && cfg->norm_mode != PMG_NORM_SEQUENTIAL)
        return fail(PMG_ERR_INVALID, "bad norm_mode");
    if (cfg->smoother < PMG_SMOOTHER_JACOBI || cfg->smoother > PMG_SMOOTHER_CHEBYSHEV)
        return fail(PMG_ERR_INVALID, "bad smoother");
    if (cfg->smoother_fp32 && (cfg->smoother != PMG_SMOOTHER_JACOBI || cfg->n_ranks > 1 || cfg->smoother_eps > 0.0))
        return fail(PMG_ERR_UNSUPPORTED, "smoother_fp32: weighted Jacobi without the eps exit, one GPU (an experiment)");
    if (cfg->smoother != PMG_SMOOTHER_JACOBI && cfg->n_ranks > 1)
        return fail(PMG_ERR_UNSUPPORTED, "multi-GPU: weighted Jacobi only (the other smoothers run on the operator engine)");
    if (cfg->smoother_eps > 0.0 && (cfg->smoother == PMG_SMOOTHER_RBGS || cfg->smoother == PMG_SMOOTHER_CHEBYSHEV))
        return fail(PMG_ERR_UNSUPPORTED, "smoother_eps: the reference's early exit exists for its Jacobi and Gauss-Seidel smoothers only");
    const bool dist = cfg->n_ranks > 1;
    if (dist) {
        if (!comm_ready() || comm_size() != cfg->n_ranks || comm_rank() != cfg->rank)
            return fail(PMG_ERR_INVALID, "n_ranks > 1 needs pmg_comm_init with the same rank / n_ranks first");
        if (cfg->engine != PMG_ENGINE_FUSED || !(cfg->nu1 >= 1 && cfg->nu1 <= 4 && cfg->nu2 >= 1 && cfg->nu2 <= 4) ||
            cfg->smoother_eps > 0.0 || cfg->norm_mode != PMG_NORM_TREE)
            return fail(PMG_ERR_UNSUPPORTED,
                        "multi-GPU: fused engine, 1-4 pre/post sweeps, smoother_eps = 0 and the tree norm only");
    }
    int ndev = pmg_device_count();
    if (ndev <= 0) return fail(PMG_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    int dev = cfg->device;
    if (dev < 0) PMG_CUDA(cudaGetDevice(&dev));
    if (dev >= ndev) return fail(PMG_ERR_INVALID, "device ordinal out of range");
    PMG_CUDA(cudaSetDevice(dev));
    int major = 0;
    PMG_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10)
        return fail(PMG_ERR_NO_DEVICE, "device is not sm_100 (kernels are built for sm_100a only)");

    pmg_solver *s = new (std::nothrow) pmg_solver();
    if (!s) return fail(PMG_ERR_ALLOC, "host allocation failed");
    s->cfg = *cfg;
    s->device = dev;
    s->fused = (cfg->engine == PMG_ENGINE_FUSED) && fused_supported(cfg->nu1) && fused_supported(cfg->nu2) &&
               !(cfg->smoother_eps > 0.0) && cfg->smoother == PMG_SMOOTHER_JACOBI && !cfg->smoother_fp32;
    pmg_status rc = PMG_OK;
    pmg_status local_fail = PMG_OK;  // (several ranks) first rank-local failure of the set-up, agreed upon collectively
    auto bail = [&](pmg_status st) {
        pmg_destroy(s);
        return st;
    };
    (void)fused_max_partials(3);  // warms the cached SM count outside any stream capture
    if (const char *e = getenv("PMG_SMALL_VCYCLE")) s->small_vcycle = !(e[0] == '0');
    if (const char *e = getenv("PMG_CROSS")) {
        s->cross_on = !(e[0] == '0');
        s->cross_forced = (e[0] == '2');
    }
    if (g_cross_override >= 0) {
        s->cross_on = g_cross_override != 0;
        s->cross_forced = g_cross_override == 2;
    }
    {
        // cluster kernel: needs the default coarse end of the hierarchy (coarsest level <= 17, reached by halving) and
        // the fused engine; PMG_CLUSTER=0 switches it off, PMG_CLUSTER=257 makes 257 the top instead of 129 (measured:
        // 129 is the faster split -- the level-257 visit costs 18 000 cycles in the cluster, about what its two
        // streaming passes take; profiles/r2_small_kernel_probe.log)
        int want = 129;
        if (const char *e = getenv("PMG_CLUSTER")) want = (e[0] == '0') ? 0 : (atoi(e) == 257 ? 257 : 129);
        if (g_cluster_override >= 0) want = g_cluster_override;
        if (want && s->fused && s->small_vcycle && cfg->n_coarse <= 17 && vcycle_small_version() == 3) {
            if (cfg->n > want && coarse_cluster_available(want))
                s->cluster_top = want;
            else if (cfg->n > 129 && coarse_cluster_available(129))
                s->cluster_top = 129;
        }
    }
    if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(PMG_ERR_CUDA, "cudaStreamCreate failed"));
    cudaEventCreate(&s->ev0);
    cudaEventCreate(&s->ev1);
    // level chain N -> (N-1)/2+1 -> ... -> n_coarse (MultiGrid.hpp:74)
    for (int n = cfg->n;; n = (n - 1) / 2 + 1) {
        Level L;
        L.n = n;
        L.pitch = level_pitch(n);
        L.h = 1.0 / (n - 1);  // MultiGridTestRunner.hpp:131 with a = 1; coarse levels: 2h (MultiGrid.hpp:83)
        L.elems = level_elems(n);
        s->lv.push_back(L);
        if (n <= cfg->n_coarse || n <= 3) break;
    }
    if (dist) {
        s->dist = true;
        s->rank = cfg->rank;
        s->n_ranks = cfg->n_ranks;
        // levels stay partitioned while every rank keeps >= 4*PADY rows and the level is above the threshold
        int la = 0;
        const int nl = (int)s->lv.size();
        while (la < nl - 1 && s->lv[la].n > cfg->agglomerate_below && ((s->lv[la].n - 1) / 2) / cfg->n_ranks * 2 >= 4 * PADY)
            ++la;
        if (la == 0) return bail(fail(PMG_ERR_UNSUPPORTED, "grid too small to partition over n_ranks (or agglomerate_below >= n)"));
        s->agg_level = la;
        s->y0s.resize(la + 1);
        s->y1s.resize(la + 1);
        for (int l = 0; l <= la; ++l) {
            s->y0s[l].resize(cfg->n_ranks);
            s->y1s[l].resize(cfg->n_ranks);
            for (int r = 0; r < cfg->n_ranks; ++r) pmg_partition_rows(s->lv[l].n, cfg->n_ranks, r, &s->y0s[l][r], &s->y1s[l][r]);
            if (l > 0)  // the coarse partition must be the fine one halved (coarse row jc lives with fine row 2jc)
                for (int r = 0; r < cfg->n_ranks; ++r)
                    if (s->y0s[l][r] * 2 != s->y0s[l - 1][r])
                        return bail(fail(PMG_ERR_UNSUPPORTED, "row partition does not nest across levels for this n / n_ranks"));
        }
        auto slab_shape = [&](Level &L, int l) {
            L.y0 = s->y0s[l][cfg->rank];
            L.ny = s->y1s[l][cfg->rank] - L.y0;
            L.elems = (size_t)L.pitch * (size_t)(L.ny + 2 * PADY);
        };
        for (int l = 0; l < la; ++l) slab_shape(s->lv[l], l);
        s->aslab = s->lv[la];
        slab_shape(s->aslab, la);
        Level &A = s->aslab;
        if ((rc = alloc_zero(&A.base_x, A.elems)) != PMG_OK) local_fail = rc;
        if ((rc = alloc_zero(&A.base_f, A.elems)) != PMG_OK) local_fail = rc;
        A.x = A.base_x + level_origin(A.n);
        A.f = A.base_f + level_origin(A.n);
        if ((rc = alloc_zero(&s->d_gather, (size_t)cfg->n_ranks)) != PMG_OK) local_fail = rc;
        // highest priority: its small latency-bound kernels (NCCL, boundary strips) are scheduled ahead of the
        // bandwidth-bound interior pass they run beside
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        if (cudaStreamCreateWithPriority(&s->comm_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess)
            local_fail = fail(PMG_ERR_CUDA, "cudaStreamCreate failed");
        cudaEventCreateWithFlags(&s->ev_ready, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&s->ev_halo, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&s->ev_passb, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&s->ev_norm, cudaEventDisableTiming);
        // all-gather + redundant coarse solve needs equally sized slabs (the last rank's extra row is the ring)
        bool equal = true;
        for (int r = 0; r + 1 < cfg->n_ranks; ++r)
            equal = equal && (s->y1s[la][r] - s->y0s[la][r] == s->y1s[la][0] - s->y0s[la][0]);
        equal = equal && (s->y1s[la][cfg->n_ranks - 1] - s->y0s[la][cfg->n_ranks - 1] == s->y1s[la][0] - s->y0s[la][0] + 1);
        const char *env = getenv("PMG_COARSE_GATHER");
        s->coarse_redundant = equal && !(env && env[0] == '1');
        if (const char *e2 = getenv("PMG_SPLIT_MIN_ROWS")) {
            s->split_min_rows = atoi(e2);
            s->split_from_env = true;
        }
        if (const char *e3 = getenv("PMG_P2P_FUSED")) s->p2p_fused = !(e3[0] == '0');
        if (const char *e4 = getenv("PMG_COARSE_GRAPH")) s->coarse_graph_on = !(e4[0] == '0');
        if (const char *e5 = getenv("PMG_HALO_PROLOGUE")) fused_set_halo_prologue(e5[0] == '1');
        if (const char *e6 = getenv("PMG_MID_GRAPH")) s->mid_graph_on = (e6[0] == '1');
        {  // wall-time limit of a peer-flag wait (pmg_internal.h: wait_flag); generous by default, see ADVICE r1
            double secs = 30.0;
            if (const char *e7 = getenv("PMG_P2P_TIMEOUT_S")) secs = atof(e7);
            if (!(secs > 0.0)) secs = 30.0;
            const unsigned long long ns = (unsigned long long)(secs * 1e9);
            fused_set_wait_timeout_ns(ns);
            basic_set_wait_timeout_ns(ns);
        }
    }
    for (size_t l = 0; l < s->lv.size(); ++l) {
        Level &L = s->lv[l];
        // (several ranks: a failure here must not leave the OTHER ranks waiting in the IPC collectives below -- it is
        // recorded and every rank leaves together after comm_all_agree)
        if ((rc = alloc_zero(&L.base_x, L.elems)) != PMG_OK) { if (!dist) return bail(rc); local_fail = rc; }
        if ((rc = alloc_zero(&L.base_xb, L.elems)) != PMG_OK) { if (!dist) return bail(rc); local_fail = rc; }
        if ((rc = alloc_zero(&L.base_f, L.elems)) != PMG_OK) { if (!dist) return bail(rc); local_fail = rc; }
        size_t o = level_origin(L.n);
        L.x = L.base_x + o;
        L.xb = L.base_xb + o;
        L.f = L.base_f + o;
        if (!s->fused) {
            if ((rc = alloc_zero(&L.base_r, L.elems)) != PMG_OK) return bail(rc);
            L.r = L.base_r + o;
        }
    }
    if (dist) {
        // every rank-local allocation is behind us: agree on the outcome before the first collective of the set-up
        if (!comm_all_agree(local_fail == PMG_OK, nullptr, s->stream)) {
            if (local_fail == PMG_OK) fail(PMG_ERR_ALLOC, "set-up failed on another rank (allocation); all ranks leave pmg_create together");
            return bail(local_fail == PMG_OK ? PMG_ERR_ALLOC : local_fail);
        }
        const char *env = getenv("PMG_P2P");
        bool want = !(env && env[0] == '0');
        if (want) {
            // Everything the neighbours (halo pulls) or all ranks (agglomerated-level all-gather) read over NVLink
            // is exported with CUDA IPC: the inbox flags, the x / f slab arrays of every partitioned level and the
            // two buffers of the first agglomerated level's right-hand side.
            const int R = cfg->n_ranks, me = cfg->rank;
            bool ok = cudaMalloc((void **)&s->d_flags, FLAG_SLOTS * sizeof(int)) == cudaSuccess &&
                      cudaMemset(s->d_flags, 0, FLAG_SLOTS * sizeof(int)) == cudaSuccess &&
                      cudaMalloc((void **)&s->d_epochs, 16 * sizeof(int)) == cudaSuccess &&
                      cudaMemset(s->d_epochs, 0, 16 * sizeof(int)) == cudaSuccess &&
                      // mapped pinned HOST memory: kernels store to it only when a peer wait times out, the host
                      // reads it after every solve without a device-to-host copy (which would queue behind bulk DMA)
                      cudaHostAlloc((void **)&s->d_comm_err, sizeof(int), cudaHostAllocMapped) == cudaSuccess;
            if (s->d_comm_err) *s->d_comm_err = 0;
            const bool want_gather = s->coarse_redundant && R <= 32;
            if (want_gather) {
                s->agg_f[0] = s->aslab.base_f;
                ok = ok && alloc_zero(&s->agg_f[1], s->aslab.elems) == PMG_OK;
            }
            // the two arrays the cross-cycle pass alternates between on level 0 (neighbours pull their boundary rows)
            ok = ok && alloc_zero(&s->base_xc, s->lv[0].elems) == PMG_OK;
            if (s->base_xc) s->xc = s->base_xc + level_origin(s->lv[0].n);
            // (1) handle exchange: the same list on every rank, whatever happened locally so far
            std::vector<void *> bases;
            bases.push_back(s->d_flags);
            for (int l = 0; l < s->agg_level; ++l) {
                bases.push_back(s->lv[l].base_x);
                bases.push_back(s->lv[l].base_f);
            }
            if (want_gather) {
                bases.push_back(s->agg_f[0]);
                bases.push_back(s->agg_f[1]);
            }
            const size_t cross_base_index = bases.size();
            bases.push_back(s->lv[0].base_xb);
            bases.push_back(s->base_xc);
            std::vector<std::vector<unsigned char>> hs(bases.size(), std::vector<unsigned char>((size_t)R * IPC_HANDLE_BYTES));
            for (size_t i = 0; i < bases.size(); ++i)
                ok = (comm_ipc_exchange(bases[i], hs[i].data(), s->stream) == PMG_OK) && ok;
            if (const char *ef = getenv("PMG_P2P_FAIL_RANK"))  // test hook: pretend this rank cannot map its peers
                if (atoi(ef) == me) ok = false;
            // (2) local mappings
            auto open_peer = [&](size_t i, int r) -> void * {
                if (!ok) return nullptr;
                void *p = comm_ipc_open(hs[i].data() + (size_t)r * IPC_HANDLE_BYTES);
                if (!p) {
                    ok = false;
                    return nullptr;
                }
                s->agg_maps.push_back(p);
                return p;
            };
            std::vector<void *> flag_peers((size_t)R, nullptr);
            for (int r = 0; r < R; ++r)
                if (r != me && (want_gather || r == me - 1 || r == me + 1)) flag_peers[r] = open_peer(0, r);
            if (ok) {
                if (me > 0) s->up_flags = (int *)flag_peers[me - 1];
                if (me < R - 1) s->dn_flags = (int *)flag_peers[me + 1];
            }
            size_t bi = 1;
            for (int l = 0; l < s->agg_level; ++l) {
                Level &L = s->lv[l];
                const size_t o = level_origin(L.n);
                for (int which = 0; which < 2; ++which, ++bi) {
                    if (me > 0) {
                        int ny_up = s->y1s[l][me - 1] - s->y0s[l][me - 1];
                        const double *p = (const double *)open_peer(bi, me - 1);
                        if (p) (which == 0 ? L.up_x : L.up_f) = p + o + (ptrdiff_t)(ny_up - PADY) * L.pitch;
                    }
                    if (me < R - 1) {
                        const double *p = (const double *)open_peer(bi, me + 1);
                        if (p) (which == 0 ? L.dn_x : L.dn_f) = p + o;
                    }
                }
            }
            if (want_gather) {
                std::vector<int *> slots((size_t)R, nullptr);
                for (int r = 0; ok && r < R; ++r) slots[r] = (r == me ? s->d_flags : (int *)flag_peers[r]) + 32 + me;
                ok = ok && cudaMalloc((void **)&s->d_agg_slots, sizeof(int *) * R) == cudaSuccess &&
                     cudaMemcpy(s->d_agg_slots, slots.data(), sizeof(int *) * R, cudaMemcpyHostToDevice) == cudaSuccess;
                for (int b = 0; b < 2; ++b, ++bi) {
                    std::vector<const double *> srcs((size_t)R, nullptr);
                    for (int r = 0; r < R; ++r) {
                        const double *p = (r == me) ? s->agg_f[b] : (const double *)open_peer(bi, r);
                        srcs[r] = p ? p + level_origin(s->aslab.n) - PADX : nullptr;  // padded start of local row 0
                    }
                    ok = ok && cudaMalloc((void **)&s->d_agg_srcs[b], sizeof(double *) * R) == cudaSuccess &&
                         cudaMemcpy(s->d_agg_srcs[b], srcs.data(), sizeof(double *) * R, cudaMemcpyHostToDevice) == cudaSuccess;
                }
            }
            {   // level 0: the neighbours' xb and xc arrays (cross-cycle pass)
                Level &L = s->lv[0];
                const size_t o = level_origin(L.n);
                for (int which = 0; which < 2; ++which) {
                    if (me > 0) {
                        int ny_up = s->y1s[0][me - 1] - s->y0s[0][me - 1];
                        const double *p = (const double *)open_peer(cross_base_index + which, me - 1);
                        if (p) L.up_xb[which] = p + o + (ptrdiff_t)(ny_up - PADY) * L.pitch;
                    }
                    if (me < R - 1) {
                        const double *p = (const double *)open_peer(cross_base_index + which, me + 1);
                        if (p) L.dn_xb[which] = p + o;
                    }
                }
            }
            // (3) every rank takes the same path: NVLink pulls if all mappings exist everywhere, NCCL otherwise
            double *d_agree = nullptr;
            bool all_ok = cudaMalloc((void **)&d_agree, sizeof(double) * (R + 1)) == cudaSuccess &&
                          comm_all_agree(ok, d_agree, s->stream);
            cudaFree(d_agree);
            if (!all_ok) {
                for (void *m : s->agg_maps) comm_ipc_close(m);
                s->agg_maps.clear();
                s->up_flags = s->dn_flags = nullptr;
                for (int l = 0; l < s->agg_level; ++l) s->lv[l].up_x = s->lv[l].dn_x = s->lv[l].up_f = s->lv[l].dn_f = nullptr;
                for (int w = 0; w < 2; ++w) s->lv[0].up_xb[w] = s->lv[0].dn_xb[w] = nullptr;
                s->p2p = s->p2p_gather = false;
            } else {
                const char *eg = getenv("PMG_P2P_GATHER");
                s->p2p_gather = want_gather && !(eg && eg[0] == '0');
                if (const char *ew = getenv("PMG_P2P_GATHER_W")) s->p2p_gather_w = !(ew[0] == '0');
                s->p2p = true;
                // With the halo prologue only the boundary warps of Pass A wait for the neighbours and the interior warps
                // start at once, i.e. the overlap happens INSIDE one launch: the interior / boundary split (three launches
                // on two streams joined by events) only adds latency.  Measured on 8 GPUs: 623 -> 566 us per cycle.
                if (!s->split_from_env && s->p2p_fused && fused_halo_prologue()) s->split_min_rows = 1 << 30;
            }
        }
    }
    s->partials_cap = std::max(reduce_partials(), fused_max_partials(cfg->n));
    if ((rc = alloc_zero(&s->d_partials, (size_t)s->partials_cap)) != PMG_OK) return bail(rc);
    if ((rc = alloc_zero(&s->d_scalar, 2)) != PMG_OK) return bail(rc);
    if (cudaMallocHost((void **)&s->h_scalar, 2 * sizeof(double)) != cudaSuccess)
        return bail(fail(PMG_ERR_ALLOC, "cudaMallocHost failed"));
    s->hist_cap = 256;
    if (cudaMalloc((void **)&s->d_ctrl, sizeof(SolveCtrl)) != cudaSuccess ||
        cudaMemset(s->d_ctrl, 0, sizeof(SolveCtrl)) != cudaSuccess ||
        cudaHostAlloc((void **)&s->h_ctrl, 2 * sizeof(SolveCtrl), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostAlloc((void **)&s->h_hist, (size_t)s->hist_cap * sizeof(double), cudaHostAllocMapped) != cudaSuccess)
        return bail(fail(PMG_ERR_ALLOC, "solve-control allocation failed"));
    std::memset(s->h_ctrl, 0, 2 * sizeof(SolveCtrl));
    if ((rc = alloc_zero(&s->d_hist2, (size_t)s->hist_cap)) != PMG_OK) return bail(rc);
    cudaEventCreateWithFlags(&s->ev_batch[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&s->ev_batch[1], cudaEventDisableTiming);
    if (cudaDeviceSynchronize() != cudaSuccess) return bail(fail(PMG_ERR_CUDA, "device synchronize failed"));
    *out = s;
    return PMG_OK;
}

void pmg_destroy(pmg_solver *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    drop_graphs(s);
    for (Level &L : s->lv) {
        cudaFree(L.base_x);
        cudaFree(L.base_xb);
        cudaFree(L.base_f);
        cudaFree(L.base_r);
        cudaFree(L.d_sin);
    }
    cudaFree(s->base_rhs_fx);
    cudaFree(s->base_rhs_sy);
    cudaFree(s->base_f_fmg0);
    for (double *b : s->pcg_base) cudaFree(b);
    cudaFree(s->base_pcg_p2);
    cudaFree(s->d_pcg_sc);
    cudaFree(s->base_xc);
    cudaFree(s->base_f_stage);
    cudaFree(s->base_x_snap);
    for (cudaStream_t st : {s->copy_in_stream, s->copy_out_stream})
        if (st) {
            cudaStreamSynchronize(st);
            cudaStreamDestroy(st);
        }
    for (cudaEvent_t e : {s->ev_staged, s->ev_snap, s->ev_fetched, s->ev_consumed})
        if (e) cudaEventDestroy(e);
    cudaFree(s->aslab.base_x);
    cudaFree(s->aslab.base_f);
    cudaFree(s->d_gather);
    for (void *m : s->agg_maps) comm_ipc_close(m);  // includes the neighbours' flag mappings
    cudaFree(s->agg_f[1]);
    cudaFree(s->d_agg_slots);
    cudaFree((void *)s->d_agg_srcs[0]);
    cudaFree((void *)s->d_agg_srcs[1]);
    cudaFree(s->d_flags);
    cudaFree(s->d_epochs);
    if (s->d_comm_err) cudaFreeHost(s->d_comm_err);
    if (s->comm_stream) {
        cudaStreamSynchronize(s->comm_stream);
        cudaStreamDestroy(s->comm_stream);
    }
    for (cudaEvent_t e : {s->ev_ready, s->ev_halo, s->ev_passb, s->ev_norm})
        if (e) cudaEventDestroy(e);
    cudaFree(s->d_partials);
    cudaFree(s->d_scalar);
    if (s->h_scalar) cudaFreeHost(s->h_scalar);
    cudaFree(s->d_ctrl);
    cudaFree(s->d_hist2);
    if (s->h_ctrl) cudaFreeHost(s->h_ctrl);
    if (s->h_hist) cudaFreeHost(s->h_hist);
    for (auto &e : s->ev_batch)
        if (e) cudaEventDestroy(e);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// With n_ranks > 1 every rank passes ITS OWN ROWS [y0, y1) of the field (ny x n doubles, dense).
static pmg_status copy_in(pmg_solver *s, double *dst_logical, const double *src, pmg_mem where)
{
    if (!s || !src) return fail(PMG_ERR_INVALID, "null argument");
    const Level &L = s->lv[0];
    const int rows = s->dist ? L.ny : L.n;
    PMG_CUDA(cudaSetDevice(s->device));
    PMG_CUDA(cudaMemcpy2DAsync(dst_logical, (size_t)L.pitch * sizeof(double), src, (size_t)L.n * sizeof(double),
                               (size_t)L.n * sizeof(double), (size_t)rows,
                               where == PMG_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s->stream));
    if (s->dist) {
        pmg_status rc = comm_halo_exchange(dst_logical, L.ny, L.pitch, PADY, s->stream);
        if (rc != PMG_OK) return rc;
    }
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    return PMG_OK;
}

pmg_status pmg_set_rhs(pmg_solver *s, const double *f, pmg_mem where)
{
    if (s) set_rhs_analytic(s, false);
    return copy_in(s, s ? s->lv[0].f : nullptr, f, where);
}

pmg_status pmg_set_guess(pmg_solver *s, const double *phi, pmg_mem where)
{
    if (s && !phi) return pmg_zero_guess(s);  // NULL = the zero start (no 8 N^2 bytes of zeros over PCIe)
    return copy_in(s, s ? s->lv[0].x : nullptr, phi, where);
}

pmg_status pmg_get_solution(pmg_solver *s, double *phi, pmg_mem where)
{
    if (!s || !phi) return fail(PMG_ERR_INVALID, "null argument");
    const Level &L = s->lv[0];
    PMG_CUDA(cudaSetDevice(s->device));
    PMG_CUDA(cudaMemcpy2DAsync(phi, (size_t)L.n * sizeof(double), L.x, (size_t)L.pitch * sizeof(double),
                               (size_t)L.n * sizeof(double), (size_t)(s->dist ? L.ny : L.n),
                               where == PMG_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s->stream));
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    return PMG_OK;
}

pmg_status pmg_zero_guess(pmg_solver *s)
{
    if (!s) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaSetDevice(s->device));
    PMG_CUDA(cudaMemsetAsync(s->lv[0].base_x, 0, s->lv[0].elems * sizeof(double), s->stream));
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    return PMG_OK;
}

// ---- overlapped host transfers ---------------------------------------------------------------------------------
static pmg_status ensure_transfer(pmg_solver *s)
{
    if (s->copy_in_stream) return PMG_OK;
    pmg_status rc = alloc_zero(&s->base_f_stage, s->lv[0].elems);
    if (rc == PMG_OK) rc = alloc_zero(&s->base_x_snap, s->lv[0].elems);
    if (rc != PMG_OK) return rc;
    PMG_CUDA(cudaStreamCreateWithFlags(&s->copy_in_stream, cudaStreamNonBlocking));
    PMG_CUDA(cudaStreamCreateWithFlags(&s->copy_out_stream, cudaStreamNonBlocking));
    for (cudaEvent_t *e : {&s->ev_staged, &s->ev_snap, &s->ev_fetched, &s->ev_consumed})
        PMG_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return PMG_OK;
}

pmg_status pmg_stage_rhs(pmg_solver *s, const double *f_host)
{
    if (!s || !f_host) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaSetDevice(s->device));
    pmg_status rc = ensure_transfer(s);
    if (rc != PMG_OK) return rc;
    const Level &L = s->lv[0];
    const int rows = s->dist ? L.ny : L.n;
    // the staging array is free again once the previous commit's device copy has read it
    if (s->ev_consumed) PMG_CUDA(cudaStreamWaitEvent(s->copy_in_stream, s->ev_consumed, 0));
    PMG_CUDA(cudaMemcpy2DAsync(s->base_f_stage + level_origin(L.n), (size_t)L.pitch * sizeof(double), f_host,
                               (size_t)L.n * sizeof(double), (size_t)L.n * sizeof(double), (size_t)rows,
                               cudaMemcpyHostToDevice, s->copy_in_stream));
    PMG_CUDA(cudaEventRecord(s->ev_staged, s->copy_in_stream));
    s->staged = true;
    return PMG_OK;
}

pmg_status pmg_commit_rhs(pmg_solver *s)
{
    if (!s) return fail(PMG_ERR_INVALID, "null argument");
    if (!s->staged) return fail(PMG_ERR_INVALID, "pmg_commit_rhs without a pmg_stage_rhs before it");
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L = s->lv[0];
    PMG_CUDA(cudaStreamWaitEvent(s->stream, s->ev_staged, 0));
    // a device copy (1.4 ms at N = 16385) rather than a pointer swap: the captured cycle graphs and, on several GPUs,
    // the neighbours' peer mappings keep addressing the same f array
    set_rhs_analytic(s, false);
    PMG_CUDA(cudaMemcpyAsync(L.base_f, s->base_f_stage, L.elems * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
    PMG_CUDA(cudaEventRecord(s->ev_consumed, s->stream));
    s->staged = false;
    if (s->dist) {
        pmg_status rc = comm_halo_exchange(L.f, L.ny, L.pitch, PADY, s->stream);
        if (rc != PMG_OK) return rc;
    }
    return PMG_OK;
}

pmg_status pmg_fetch_solution_begin(pmg_solver *s, double *phi_host)
{
    if (!s || !phi_host) return fail(PMG_ERR_INVALID, "null argument");
    if (s->fetching) return fail(PMG_ERR_INVALID, "pmg_fetch_solution_begin while a fetch is in flight (call pmg_fetch_solution_wait)");
    PMG_CUDA(cudaSetDevice(s->device));
    pmg_status rc = ensure_transfer(s);
    if (rc != PMG_OK) return rc;
    const Level &L = s->lv[0];
    PMG_CUDA(cudaMemcpyAsync(s->base_x_snap, L.base_x, L.elems * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
    PMG_CUDA(cudaEventRecord(s->ev_snap, s->stream));
    PMG_CUDA(cudaStreamWaitEvent(s->copy_out_stream, s->ev_snap, 0));
    PMG_CUDA(cudaMemcpy2DAsync(phi_host, (size_t)L.n * sizeof(double), s->base_x_snap + level_origin(L.n),
                               (size_t)L.pitch * sizeof(double), (size_t)L.n * sizeof(double), (size_t)(s->dist ? L.ny : L.n),
                               cudaMemcpyDeviceToHost, s->copy_out_stream));
    PMG_CUDA(cudaEventRecord(s->ev_fetched, s->copy_out_stream));
    s->fetching = true;
    return PMG_OK;
}

pmg_status pmg_fetch_solution_wait(pmg_solver *s)
{
    if (!s) return fail(PMG_ERR_INVALID, "null argument");
    if (!s->fetching) return PMG_OK;
    PMG_CUDA(cudaSetDevice(s->device));
    PMG_CUDA(cudaEventSynchronize(s->ev_fetched));
    s->fetching = false;
    return PMG_OK;
}

// fx = factor * sin in the padded column layout of level 0, sy = sin with PADY zero rows above and below: dmul(fx[x], sy[y])
// is the dmul(dmul(factor, sin_x), sin_y) k_rhs_separable writes, and +0 wherever the array holds its zero padding -- as long
// as no sine value carries a sign bit (-0 * +0 would give -0).  If one does, no tables are built and the pass reads f.
static pmg_status ensure_rhs_tables(pmg_solver *s)
{
    if (s->base_rhs_fx != nullptr) return PMG_OK;
    const Level &L = s->lv[0];
    std::vector<double> sn(L.n);
    PMG_CUDA(cudaMemcpy(sn.data(), L.d_sin, L.n * sizeof(double), cudaMemcpyDeviceToHost));
    for (double v : sn)
        if (std::signbit(v)) return PMG_OK;
    const double a = 1.0, p = 1.0, q = 1.0;
    const double factor = (M_PI * M_PI / (a * a)) * (p * p + q * q);  // as analytic_rhs
    std::vector<double> fx(L.pitch, 0.0), sy(L.n + 2 * PADY, 0.0);
    for (int i = 0; i < L.n; ++i) {
        fx[PADX + i] = factor * sn[i];
        sy[PADY + i] = sn[i];
    }
    pmg_status rc = alloc_zero(&s->base_rhs_fx, fx.size());
    if (rc == PMG_OK) rc = alloc_zero(&s->base_rhs_sy, sy.size());
    if (rc != PMG_OK) return rc;
    PMG_CUDA(cudaMemcpy(s->base_rhs_fx, fx.data(), fx.size() * sizeof(double), cudaMemcpyHostToDevice));
    PMG_CUDA(cudaMemcpy(s->base_rhs_sy, sy.data(), sy.size() * sizeof(double), cudaMemcpyHostToDevice));
    s->rhs_fx = s->base_rhs_fx + PADX;
    s->rhs_sy = s->base_rhs_sy + PADY;
    return PMG_OK;
}

pmg_status pmg_set_rhs_sine(pmg_solver *s)
{
    if (!s) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaSetDevice(s->device));
    pmg_status rc = ensure_fmg(s);
    if (rc != PMG_OK) return rc;
    if (s->dist) {
        const Level &L = s->lv[0];
        int ga = std::max(L.y0 - PADY, 0), gb = std::min(L.y0 + L.ny + PADY, L.n);  // rows incl. halo
        const double a = 1.0, p = 1.0, q = 1.0;
        double factor = (M_PI * M_PI / (a * a)) * (p * p + q * q);
        launch_rhs_separable(L.f + (ptrdiff_t)(ga - L.y0) * L.pitch, L.pitch, L.n, gb - ga, factor, L.d_sin,
                             L.d_sin + ga, s->stream);
    } else {
        analytic_rhs(s, s->lv[0], s->lv[0].f);
        if ((rc = ensure_rhs_tables(s)) != PMG_OK) return rc;
        s->rhs_tab_f = s->lv[0].f;
        set_rhs_analytic(s, true);
    }
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_residual_norm(pmg_solver *s, double *norm_out)
{
    if (!s || !norm_out) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaSetDevice(s->device));
    pmg_status rc = residual_norm2_async(s);
    if (rc != PMG_OK) return rc;
    double v = 0.0;
    rc = read_scalar(s, &v);
    if (rc != PMG_OK) return rc;
    *norm_out = std::sqrt(v);
    return PMG_OK;
}

// a peer-to-peer wait that timed out raised the device flag (bounded spins never hang the GPU)
static pmg_status check_comm_err(pmg_solver *s)
{
    if (!s->p2p) return PMG_OK;
    const int err = *(volatile int *)s->d_comm_err;  // mapped host memory; the callers have synchronised the stream
    // sticky on purpose: after a timeout the ranks' epochs no longer agree, so this solver (and its peers') must be
    // destroyed and re-created; every later call reports the same error (pmg.h, multi-GPU section)
    if (err) return fail(PMG_ERR_COMM, "peer-to-peer halo exchange timed out waiting for a neighbour (PMG_P2P_TIMEOUT_S); "
                                       "the solver is unusable, destroy it on every rank");
    return PMG_OK;
}

pmg_status pmg_cycle(pmg_solver *s, pmg_cycle_kind kind, double *res_norm_out)
{
    if (!s) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaSetDevice(s->device));
    if (s->p2p)  // Pass B(0) honours the control block's flag (timed-out peer wait); a finished pmg_solve left it raised
        PMG_CUDA(cudaMemsetAsync(&s->d_ctrl->done, 0, sizeof(int), s->stream));
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    pmg_status rc = run_cycle(s, kind, res_norm_out != nullptr);
    if (rc != PMG_OK) return rc;
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    if (res_norm_out) {
        double v = 0.0;
        rc = read_scalar(s, &v);
        if (rc != PMG_OK) return rc;
        *res_norm_out = std::sqrt(v);
    } else {
        PMG_CUDA(cudaStreamSynchronize(s->stream));
        PMG_CUDA(cudaGetLastError());
    }
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    return check_comm_err(s);
}

static int level_of_size(const pmg_solver *s, int n)
{
    for (size_t l = 0; l < s->lv.size(); ++l)
        if (s->lv[l].n == n) return (int)l;
    return -1;
}

pmg_status pmg_restrict_to_level(pmg_solver *s, const double *fine, pmg_mem where_in, int n_out, double *out,
                                 pmg_mem where_out)
{
    if (!s || !fine || !out) return fail(PMG_ERR_INVALID, "null argument");
    if (s->dist) return fail(PMG_ERR_UNSUPPORTED, "pmg_restrict_to_level is single-GPU only");
    const int lo = level_of_size(s, n_out);
    if (lo < 0) return fail(PMG_ERR_INVALID, "n_out is not a level of this solver's hierarchy");
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L0 = s->lv[0];
    const cudaMemcpyKind kin = where_in == PMG_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const cudaMemcpyKind kout = where_out == PMG_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    // stage the input in the finest level's ping-pong partner (scratch: every pass re-writes it before reading it)
    PMG_CUDA(cudaMemcpy2DAsync(L0.xb, (size_t)L0.pitch * sizeof(double), fine, (size_t)L0.n * sizeof(double),
                               (size_t)L0.n * sizeof(double), (size_t)L0.n, kin, s->stream));
    restrict_chain(s, L0.xb, lo);
    const Level &K = s->lv[lo];
    PMG_CUDA(cudaMemcpy2DAsync(out, (size_t)K.n * sizeof(double), K.xb, (size_t)K.pitch * sizeof(double),
                               (size_t)K.n * sizeof(double), (size_t)K.n, kout, s->stream));
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_f_cycle_from(pmg_solver *s, const double *phi_init, const double *f_init, int n_init, pmg_mem where,
                            double *res_norm_out)
{
    if (!s || !phi_init || !f_init) return fail(PMG_ERR_INVALID, "null argument");
    if (s->dist) return fail(PMG_ERR_UNSUPPORTED, "pmg_f_cycle_from is single-GPU only (pmg_cycle(PMG_CYCLE_F) shards)");
    const int li = level_of_size(s, n_init);
    if (li < 0) return fail(PMG_ERR_INVALID, "n_init is not a level of this solver's hierarchy");
    PMG_CUDA(cudaSetDevice(s->device));
    pmg_status rc = ensure_fmg(s);
    if (rc != PMG_OK) return rc;
    drop_graphs(s);  // the smoothing below may swap x / xb roles on levels >= 1
    Level &L = s->lv[li];
    const cudaMemcpyKind k = where == PMG_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    PMG_CUDA(cudaMemcpy2DAsync(L.x, (size_t)L.pitch * sizeof(double), phi_init, (size_t)L.n * sizeof(double),
                               (size_t)L.n * sizeof(double), (size_t)L.n, k, s->stream));
    if (li > 0)  // on the finest level the loop body never runs and f is not used (MultiGrid.hpp:150)
        PMG_CUDA(cudaMemcpy2DAsync(L.f, (size_t)L.pitch * sizeof(double), f_init, (size_t)L.n * sizeof(double),
                                   (size_t)L.n * sizeof(double), (size_t)L.n, k, s->stream));
    if ((rc = fmg_up_from(s, li)) != PMG_OK) return rc;
    if (const int bad = fused_take_bad_nu())
        return fail(PMG_ERR_UNSUPPORTED, "fused engine: no kernel for " + std::to_string(bad) + " sweeps per pass");
    if (res_norm_out && (rc = residual_norm2_async(s)) != PMG_OK) return rc;
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    if (res_norm_out) {
        double v = 0.0;
        if ((rc = read_scalar(s, &v)) != PMG_OK) return rc;
        *res_norm_out = std::sqrt(v);
    } else {
        PMG_CUDA(cudaStreamSynchronize(s->stream));
        PMG_CUDA(cudaGetLastError());
    }
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    return PMG_OK;
}

// cross-cycle pass on row slabs: needs the halo prologue over NVLink peer memory and at least two slab levels (the next
// cycle's coarse right-hand side is written at the END of a cycle: with one slab level it would land in the all-gather's
// double buffer of the wrong parity)
static bool cross_ok_dist(const pmg_solver *s, bool w)
{
    return s->cross_on && !w && s->dist && s->p2p && s->p2p_fused && fused_halo_prologue() && s->agg_level >= 2 &&
           s->xc != nullptr && fused_cross_supported(s->cfg.nu1, s->cfg.nu2) && s->cfg.norm_mode == PMG_NORM_TREE &&
           g_trace_on != 1 && (s->cross_forced || fused_cross_utilisation(s->lv[0].n, s->lv[0].ny) >= 0.9) &&
           (s->rank == 0 || (s->lv[0].up_xb[0] && s->lv[0].up_xb[1])) &&
           (s->rank == s->n_ranks - 1 || (s->lv[0].dn_xb[0] && s->lv[0].dn_xb[1]));
}

/* Fused V/W solve with device-side convergence control: cycles are queued one batch ahead of the host's
 * knowledge of the residual, the last kernel of each cycle records ||r||^2 and raises `done`, and every
 * kernel queued after that returns at once.  The GPU never waits for the host between cycles. */
static pmg_status solve_fused_async(pmg_solver *s, bool w, double rel_tol, int max_cycles, double *res_history,
                                    int *n_cycles_out)
{
    if (max_cycles + 1 > s->hist_cap) {
        if (s->d_hist2) cudaFree(s->d_hist2);
        s->d_hist2 = nullptr;
        if (s->h_hist) cudaFreeHost(s->h_hist);
        s->h_hist = nullptr;
        s->hist_cap = max_cycles + 1 + 64;
        pmg_status rc = alloc_zero(&s->d_hist2, (size_t)s->hist_cap);
        if (rc != PMG_OK) return rc;
        if (cudaHostAlloc((void **)&s->h_hist, (size_t)s->hist_cap * sizeof(double), cudaHostAllocMapped) != cudaSuccess)
            return fail(PMG_ERR_ALLOC, "history mirror allocation failed");
        drop_graphs(s);  // the captured graphs hold the old history pointer
    }
    Level &L = s->lv[0];
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    {
        pmg_status rc0 = residual_norm2_async(s);
        if (rc0 != PMG_OK) return rc0;
    }
    launch_solve_begin(s->d_scalar, s->d_ctrl, s->d_hist2, rel_tol, max_cycles, s->stream);
    // row slabs: the cross-cycle pass replaces Pass B(0) of a cycle and Pass A(0) of the next one (cycle_dist)
    s->cross_active = s->dist && cross_ok_dist(s, w);
    s->cross_count = 0;
    struct CrossOff {
        pmg_solver *s;
        ~CrossOff() { s->cross_active = false; }
    } cross_off{s};
    // enough queued work to cover a host round trip: one cycle on big grids, a few on small ones
    const int batch = L.n >= 2049 ? 1 : (L.n >= 513 ? 2 : 4);
    int queued = 0, slot = 0;
    bool pending[2] = {false, false};
    bool finished = false;
    while (!finished) {
        int b = std::min(batch, max_cycles - queued);
        for (int i = 0; i < b; ++i) {
            pmg_status rc = run_fused_graph(s, w, 2);
            if (rc != PMG_OK) return rc;
        }
        queued += b;
        cudaStream_t cs = s->dist ? s->comm_stream : s->stream;  // the stream whose last kernel wrote the control block
        launch_ctrl_to_host(s->d_ctrl, &s->h_ctrl[slot], nullptr, nullptr, 0, cs);  // (a kernel: no copy engine)
        PMG_CUDA(cudaEventRecord(s->ev_batch[slot], cs));
        pending[slot] = true;
        int prev = slot ^ 1;
        if (pending[prev]) {  // look at the batch before this one while this one runs
            PMG_CUDA(cudaEventSynchronize(s->ev_batch[prev]));
            pending[prev] = false;
            if (((volatile SolveCtrl *)s->h_ctrl)[prev].done) finished = true;
        }
        if (queued >= max_cycles || b == 0) finished = true;
        slot ^= 1;
    }
    if (s->dist) {  // join the communication stream (last norm) before the end-of-solve timestamp
        PMG_CUDA(cudaEventRecord(s->ev_halo, s->comm_stream));
        PMG_CUDA(cudaStreamWaitEvent(s->stream, s->ev_halo, 0));
        s->norm_pending = false;
    }
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    launch_ctrl_to_host(s->d_ctrl, &s->h_ctrl[0], s->d_hist2, s->h_hist, s->hist_cap, s->stream);
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    PMG_CUDA(cudaGetLastError());
    {
        pmg_status rce = check_comm_err(s);
        if (rce != PMG_OK) return rce;
    }
    int k = ((volatile SolveCtrl *)s->h_ctrl)[0].cycles;
    if (k < 0 || k > max_cycles)
        return fail(PMG_ERR_CUDA, "solve control block corrupted (cycles = " + std::to_string(k) + ")");
    if (res_history) {
        const volatile double *h2 = s->h_hist;
        for (int i = 0; i <= k; ++i) res_history[i] = std::sqrt(h2[i]);
    }
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    if (n_cycles_out) *n_cycles_out = k;
    return PMG_OK;
}

// ---- cross-cycle solve (one GPU, V-cycles, nu1 = nu2 = 2) -------------------------------------------------------------
// On level 0 the last pass of cycle k (prolongation, post-smoothing, norm) and the first pass of cycle k+1 (pre-smoothing,
// residual, restriction) are back-to-back sweeps over the same array.  k_cross does both in one sweep: x_k lives only in
// the register pipeline, and level 0 moves 28 B/point per cycle instead of 52.  xb and a third array xc alternate as the
// pass's input and output; when the device-side control reports convergence after cycle k, the input array of that pass
// (xb_k) and the coarse correction e_k are still intact, and ONE ordinary Pass B produces the iterate the reference
// returns.  (Row slabs write x_k every cycle instead, see k_cross.)  Iterates are bit-identical to the two-pass path; the
// norms differ in the last bits only (another grouping of the tree sum).
static bool cross_ok(const pmg_solver *s, bool w)
{
    return s->cross_on && !w && !s->dist && s->fused && fused_cross_supported(s->cfg.nu1, s->cfg.nu2) &&
           s->cfg.norm_mode == PMG_NORM_TREE && s->lv.size() > 2 && s->lv[1].n > s->cfg.n_coarse && fused_graph_ok(s) &&
           (s->cross_forced || fused_cross_utilisation(s->lv[0].n, s->lv[0].n) >= 0.9);
}

static pmg_status ensure_xc(pmg_solver *s)
{
    if (s->base_xc) return PMG_OK;
    pmg_status rc = alloc_zero(&s->base_xc, s->lv[0].elems);
    if (rc != PMG_OK) return rc;
    s->xc = s->base_xc + level_origin(s->lv[0].n);
    return PMG_OK;
}

// one cycle's worth of work after the level-0 pre-smoothing: coarse part from level 1, cross pass, convergence kernel
static pmg_status run_cross_cycle(pmg_solver *s, int parity)
{
    cudaGraphExec_t &ge = s->cross_graph[parity];
    int &gk = s->cross_graph_kernels[parity];
    if (ge != nullptr) {
        PMG_CUDA(cudaGraphLaunch(ge, s->stream));
        count_launch(gk);
        return PMG_OK;
    }
    const pmg_config &c = s->cfg;
    Level &L = s->lv[0];
    Level &K = s->lv[1];
    const int *done = &s->d_ctrl->done;
    const unsigned long long before = launches_so_far();
    PMG_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
    pmg_status rc = cycle_fused(s, 1, false, true, false, nullptr, done);
    int np = 0;
    if (rc == PMG_OK) {
        FusedLevel v = fused_view(L);
        v.x = nullptr;                            // x_k is not written (solve_cross produces it once, at the end)
        v.xb = parity ? s->xc : L.xb;             // input: xb_k
        use_rhs_tables(s, v);                     // f generated in the pass (set_rhs_analytic drops this graph when that changes)
        double *out = parity ? L.xb : s->xc;      // output: xb_{k+1}
        launch_fused_cross(v, out, K.x, K.f, K.pitch, c.omega, c.prolong_mode, s->d_partials, &np, s->stream, done);
        launch_cycle_finish(s->d_partials, np, s->d_ctrl, s->d_hist2, s->stream);
    }
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(s->stream, &g);
    if (e != cudaSuccess) return fail(PMG_ERR_CUDA, std::string("cudaStreamEndCapture (cross cycle): ") + cudaGetErrorString(e));
    if (rc != PMG_OK) {
        cudaGraphDestroy(g);
        return rc;
    }
    gk = (int)(launches_so_far() - before);
    e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return fail(PMG_ERR_CUDA, std::string("cudaGraphInstantiate (cross cycle): ") + cudaGetErrorString(e));
    PMG_CUDA(cudaGraphLaunch(ge, s->stream));
    return PMG_OK;
}

static pmg_status solve_cross(pmg_solver *s, double rel_tol, int max_cycles, double *res_history, int *n_cycles_out)
{
    const pmg_config &c = s->cfg;
    Level &L = s->lv[0];
    Level &K = s->lv[1];
    pmg_status rc = ensure_xc(s);
    if (rc != PMG_OK) return rc;
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    if ((rc = residual_norm2_async(s)) != PMG_OK) return rc;
    launch_solve_begin(s->d_scalar, s->d_ctrl, s->d_hist2, rel_tol, max_cycles, s->stream);
    const int *done = &s->d_ctrl->done;
    // first half of cycle 1: xb = S^nu1(x), coarse f = R(f - A xb)
    launch_fused_down(fused_view(L), K.f, K.pitch, c.nu1, c.omega, false, s->stream, done);
    const int batch = L.n >= 2049 ? 1 : (L.n >= 513 ? 2 : 4);
    int queued = 0, slot = 0;
    bool pending[2] = {false, false};
    bool finished = max_cycles <= 0;
    while (!finished) {
        const int b = std::min(batch, max_cycles - queued);
        for (int i = 0; i < b; ++i) {
            if ((rc = run_cross_cycle(s, queued & 1)) != PMG_OK) return rc;
            ++queued;
        }
        launch_ctrl_to_host(s->d_ctrl, &s->h_ctrl[slot], nullptr, nullptr, 0, s->stream);
        PMG_CUDA(cudaEventRecord(s->ev_batch[slot], s->stream));
        pending[slot] = true;
        const int prev = slot ^ 1;
        if (pending[prev]) {
            PMG_CUDA(cudaEventSynchronize(s->ev_batch[prev]));
            pending[prev] = false;
            if (((volatile SolveCtrl *)s->h_ctrl)[prev].done) finished = true;
        }
        if (queued >= max_cycles || b == 0) finished = true;
        slot ^= 1;
    }
    launch_ctrl_to_host(s->d_ctrl, &s->h_ctrl[0], s->d_hist2, s->h_hist, s->hist_cap, s->stream);
    PMG_CUDA(cudaStreamSynchronize(s->stream));
    PMG_CUDA(cudaGetLastError());
    const int k = ((volatile SolveCtrl *)s->h_ctrl)[0].cycles;
    if (k < 0 || k > max_cycles)
        return fail(PMG_ERR_CUDA, "solve control block corrupted (cycles = " + std::to_string(k) + ")");
    if (k > 0) {
        // x_k = S^nu2(xb_k + P e_k): xb_k is the input array of the k-th cross pass; e_k is still level 1's iterate, because
        // every kernel queued after the pass that raised `done` returned at once
        FusedLevel v = fused_view(L);
        v.xb = ((k - 1) & 1) ? s->xc : L.xb;
        launch_fused_up(v, K.x, K.pitch, c.nu2, c.omega, c.prolong_mode, nullptr, nullptr, s->stream, nullptr);
    }
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    PMG_CUDA(cudaGetLastError());
    if (const int bad = fused_take_bad_nu())
        return fail(PMG_ERR_UNSUPPORTED, "fused engine: no kernel for " + std::to_string(bad) + " sweeps per pass");
    if (res_history) {
        const volatile double *h2 = s->h_hist;
        for (int i = 0; i <= k; ++i) res_history[i] = std::sqrt(h2[i]);
    }
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    if (n_cycles_out) *n_cycles_out = k;
    return PMG_OK;
}

static pmg_status solve_impl(pmg_solver *s, pmg_cycle_kind kind, double rel_tol, int max_cycles, double *res_history,
                             int *n_cycles_out);

pmg_status pmg_solve(pmg_solver *s, pmg_cycle_kind kind, double rel_tol, int max_cycles, double *res_history,
                     int *n_cycles_out)
{
    try {  // no C++ exception may cross the C ABI
        return solve_impl(s, kind, rel_tol, max_cycles, res_history, n_cycles_out);
    } catch (const std::exception &e) {
        return fail(PMG_ERR_ALLOC, std::string("exception in pmg_solve: ") + e.what());
    }
}

static pmg_status solve_impl(pmg_solver *s, pmg_cycle_kind kind, double rel_tol, int max_cycles, double *res_history,
                             int *n_cycles_out)
{
    if (!s || max_cycles < 0) return fail(PMG_ERR_INVALID, "bad argument");
    PMG_CUDA(cudaSetDevice(s->device));
    if (s->fused && (kind == PMG_CYCLE_V || kind == PMG_CYCLE_W) && s->cfg.norm_mode == PMG_NORM_TREE &&
        s->lv.size() > 1 && s->lv[0].n > s->cfg.n_coarse && (s->dist || fused_graph_ok(s))) {
        if (max_cycles + 1 > s->hist_cap || !cross_ok(s, kind == PMG_CYCLE_W))
            return solve_fused_async(s, kind == PMG_CYCLE_W, rel_tol, max_cycles, res_history, n_cycles_out);
        return solve_cross(s, rel_tol, max_cycles, res_history, n_cycles_out);
    }
    if (s->p2p) PMG_CUDA(cudaMemsetAsync(&s->d_ctrl->done, 0, sizeof(int), s->stream));  // see pmg_cycle
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    pmg_status rc = residual_norm2_async(s);
    if (rc != PMG_OK) return rc;
    double v = 0.0;
    rc = read_scalar(s, &v);
    if (rc != PMG_OK) return rc;
    double r0 = std::sqrt(v);
    if (res_history) res_history[0] = r0;
    int k = 0;
    while (k < max_cycles) {
        // PMG_CYCLE_FMG: one full-multigrid pass, then V-cycles
        rc = run_cycle(s, (kind == PMG_CYCLE_FMG && k > 0) ? PMG_CYCLE_V : kind, true);
        if (rc != PMG_OK) return rc;
        rc = read_scalar(s, &v);
        if (rc != PMG_OK) return rc;
        ++k;
        double rn = std::sqrt(v);
        if (res_history) res_history[k] = rn;
        if (rn < rel_tol * r0) break;
    }
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    if (n_cycles_out) *n_cycles_out = k;
    return check_comm_err(s);
}

// ---- preconditioned conjugate gradients (pmg.h; specification: the CPU checker's orc_pcg) -----------------------------
static pmg_status pcg_dist(pmg_solver *s, int precond, double rel_tol, int max_iter, double *res_history, int *n_iter_out);

static pmg_status pcg_impl(pmg_solver *s, int precond, double rel_tol, int max_iter, double *res_history, int *n_iter_out)
{
    if (!s || max_iter < 0 || (precond != 0 && precond != 1)) return fail(PMG_ERR_INVALID, "bad argument");
    if (s->dist) return pcg_dist(s, precond, rel_tol, max_iter, res_history, n_iter_out);
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L = s->lv[0];
    for (double *&b : s->pcg_base)
        if (!b) {
            pmg_status rc = alloc_zero(&b, L.elems);
            if (rc != PMG_OK) return rc;
        }
    const size_t o = level_origin(L.n);
    double *r = s->pcg_base[0] + o, *z_arr = s->pcg_base[1] + o, *p = s->pcg_base[2] + o, *ap = s->pcg_base[3] + o;
    auto scalar = [&](double *out) -> pmg_status { return read_scalar(s, out); };
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    // r = f - A x on the interior (the padding and the ring of r stay zero)
    launch_residual(r, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.pitch, L.h, s->stream);
    launch_dot_interior(r, r, L.n, L.n, L.pitch, s->d_partials, s->d_scalar, s->stream);
    double rr = 0.0;
    pmg_status rc = scalar(&rr);
    if (rc != PMG_OK) return rc;
    const double r0 = std::sqrt(rr);
    if (res_history) res_history[0] = r0;
    int k = 0;
    double rz = 0.0, rnorm = r0;
    while (k < max_iter && !(rnorm < rel_tol * r0) && r0 > 0.0) {
        const double *z = r;
        if (precond) {
            // z = M r: one cycle on (z, r) from z = 0 -- the finest level temporarily works on the PCG arrays
            double *sx = L.x, *sxb = L.xb, *sbx = L.base_x, *sbxb = L.base_xb;
            double *sf = L.f, *sbf = L.base_f;
            PMG_CUDA(cudaMemsetAsync(s->pcg_base[1], 0, L.elems * sizeof(double), s->stream));
            L.x = z_arr;
            L.base_x = s->pcg_base[1];
            L.f = r;
            L.base_f = s->pcg_base[0];
            rc = s->fused ? cycle_fused(s, 0, false, false, false, nullptr) : cycle_operator(s, 0, false, false);
            z = L.x;  // (the operator engine may have left the result in the ping-pong partner)
            L.x = sx;
            L.xb = sxb;
            L.base_x = sbx;
            L.base_xb = sbxb;
            L.f = sf;
            L.base_f = sbf;
            if (rc != PMG_OK) return rc;
            if (const int bad = fused_take_bad_nu())
                return fail(PMG_ERR_UNSUPPORTED, "fused engine: no kernel for " + std::to_string(bad) + " sweeps per pass");
        }
        double rz_new = 0.0;
        launch_dot_interior(r, z, L.n, L.n, L.pitch, s->d_partials, s->d_scalar, s->stream);
        if ((rc = scalar(&rz_new)) != PMG_OK) return rc;
        launch_pcg_direction(p, z, L.n, L.n, L.pitch, k == 0 ? 0.0 : rz_new / rz, k == 0, s->stream);
        rz = rz_new;
        double pap = 0.0;
        launch_apply_a_dot(p, ap, L.n, L.n, L.pitch, L.h, s->d_partials, s->d_scalar, s->stream);
        if ((rc = scalar(&pap)) != PMG_OK) return rc;
        const double alpha = rz / pap;
        launch_pcg_update(L.x, r, p, ap, L.n, L.n, L.pitch, alpha, s->d_partials, s->d_scalar, s->stream);
        if ((rc = scalar(&rr)) != PMG_OK) return rc;
        ++k;
        rnorm = std::sqrt(rr);
        if (res_history) res_history[k] = rnorm;
    }
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    if (n_iter_out) *n_iter_out = k;
    if (precond) drop_graphs(s);  // the operator engine's coarse solves may have swapped x / xb roles below level 0
    return PMG_OK;
}

// pmg_pcg on row slabs: orc_pcg's step on this rank's owned rows of level 0.  Per step:
//   precond: exchange PADY halo rows of r, then z = one cycle_dist(0) from zero on (z, r).  With x_is_zero, level 0 does
//     no halo exchange and its Pass A reads the LOCAL f halo rows, so pointing level 0 at the PCG arrays touches no array
//     a neighbour maps over NVLink; it also means r's halo must be fresh before every preconditioner cycle;
//   one row of z beyond the slab from the neighbours (level 0's last Pass B finishes the owned rows only -- cycle_dist:
//     ext 0 on level 0), which the direction-operator pass reads;
//   rz = r.z, p = z + beta p with Ap and p.Ap (one fused pass, launch_pcg_direction_apply), x += alpha p and r -= alpha Ap
//     with r.r.  Every dot product is summed per rank, all-gathered and summed in rank order (launch_final_sum).
// alpha and beta never leave the GPU: the kernels divide the device-side sums themselves, so a step has ONE device-to-host
// read, ||r||.  The sums differ from one GPU's only in their grouping, hence the tolerance (not bit identity) in pmg.h.
static pmg_status pcg_dist(pmg_solver *s, int precond, double rel_tol, int max_iter, double *res_history, int *n_iter_out)
{
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L = s->lv[0];
    for (double *&b : s->pcg_base)
        if (!b) {
            pmg_status rc = alloc_zero(&b, L.elems);
            if (rc != PMG_OK) return rc;
        }
    if (!s->base_pcg_p2) {
        pmg_status rc = alloc_zero(&s->base_pcg_p2, L.elems);
        if (rc != PMG_OK) return rc;
    }
    if (!s->d_pcg_sc) {
        pmg_status rc = alloc_zero(&s->d_pcg_sc, 4 + (size_t)PCG_MAX_PARTIALS);
        if (rc != PMG_OK) return rc;
    }
    const size_t o = level_origin(L.n);
    double *r = s->pcg_base[0] + o, *z_arr = s->pcg_base[1] + o, *ap = s->pcg_base[3] + o;
    double *pp[2] = {s->pcg_base[2] + o, s->base_pcg_p2 + o};
    double *sc = s->d_pcg_sc, *part = s->d_pcg_sc + 4;
    cudaStream_t st = s->stream;
    // the window whose own "ring" rows are local rows a-1 and b: whole-level interior kernels on the owned interior rows
    const int ga = std::max(L.y0, 1), gb = std::min(L.y0 + L.ny, L.n - 1), a = ga - L.y0, b = gb - L.y0;
    const ptrdiff_t wo = (ptrdiff_t)(a - 1) * L.pitch;
    const int wrows = b - a + 2;
    // this rank's sum in d_scalar -> the rank-ordered global sum in *dst, the same bits on every rank
    auto global_sum = [&](double *dst) -> pmg_status {
        pmg_status rc = comm_allgather_double(s->d_scalar, s->d_gather, st);
        if (rc == PMG_OK) launch_final_sum(s->d_gather, s->n_ranks, dst, st);
        return rc;
    };
    if (s->p2p)  // Pass B(0) of the preconditioner honours the control block's flag; a finished pmg_solve left it raised
        PMG_CUDA(cudaMemsetAsync(&s->d_ctrl->done, 0, sizeof(int), st));
    s->cycle_has_collective = false;  // the agglomerated level travels by NCCL all-gather inside the preconditioner
    drop_graphs(s);
    PMG_CUDA(cudaEventRecord(s->ev0, st));
    pmg_status rc = comm_halo_exchange(L.x, L.ny, L.pitch, PADY, st);
    if (rc != PMG_OK) return rc;
    launch_residual(r + wo, L.x + wo, L.f + wo, L.n, wrows, L.pitch, L.pitch, L.pitch, L.h, st);
    launch_dot_interior(r + wo, r + wo, L.n, wrows, L.pitch, s->d_partials, s->d_scalar, st);
    if ((rc = global_sum(s->d_scalar)) != PMG_OK) return rc;
    double rr = 0.0;
    if ((rc = read_scalar(s, &rr)) != PMG_OK) return rc;
    const double r0 = std::sqrt(rr);
    if (res_history) res_history[0] = r0;
    int k = 0;
    double rnorm = r0;
    // every rank reads the same bits of ||r|| (rank-ordered sums), so all take the same branch here and run the same
    // collectives inside cycle_dist
    while (k < max_iter && !(rnorm < rel_tol * r0) && r0 > 0.0) {
        double *z = r;
        if (precond) {
            if ((rc = comm_halo_exchange(r, L.ny, L.pitch, PADY, st)) != PMG_OK) return rc;
            double *sx = L.x, *sbx = L.base_x, *sf = L.f, *sbf = L.base_f;
            L.x = z_arr;
            L.base_x = s->pcg_base[1];
            L.f = r;
            L.base_f = s->pcg_base[0];
            rc = cycle_dist(s, 0, false, true, false, nullptr, nullptr);
            z = L.x;
            L.x = sx;
            L.base_x = sbx;
            L.f = sf;
            L.base_f = sbf;
            if (rc != PMG_OK) return rc;
            if (const int bad = fused_take_bad_nu())
                return fail(PMG_ERR_UNSUPPORTED, "fused engine: no kernel for " + std::to_string(bad) + " sweeps per pass");
        }
        if ((rc = comm_halo_exchange(z, L.ny, L.pitch, 1, st)) != PMG_OK) return rc;
        double *rz = sc + (k & 1), *rz_prev = sc + ((k & 1) ^ 1), *pap = sc + 2;
        launch_dot_interior(r + wo, z + wo, L.n, wrows, L.pitch, s->d_partials, s->d_scalar, st);
        if ((rc = global_sum(rz)) != PMG_OK) return rc;
        double *p = pp[k & 1];
        int np = launch_pcg_direction_apply(z, pp[(k & 1) ^ 1], p, ap, L.n, L.ny, L.y0, L.pitch, L.h, rz, rz_prev, k == 0, part,
                                            st);
        launch_final_sum(part, np, s->d_scalar, st);
        if ((rc = global_sum(pap)) != PMG_OK) return rc;
        np = launch_pcg_update_dev(L.x, r, p, ap, L.n, L.ny, L.y0, L.pitch, rz, pap, part, st);
        launch_final_sum(part, np, s->d_scalar, st);
        if ((rc = global_sum(s->d_scalar)) != PMG_OK) return rc;
        if ((rc = read_scalar(s, &rr)) != PMG_OK) return rc;
        if ((rc = check_comm_err(s)) != PMG_OK) return rc;  // a timed-out peer wait in the preconditioner
        ++k;
        rnorm = std::sqrt(rr);
        if (res_history) res_history[k] = rnorm;
    }
    PMG_CUDA(cudaEventRecord(s->ev1, st));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    if (n_iter_out) *n_iter_out = k;
    drop_graphs(s);  // the coarse solves may have swapped x / xb roles of the whole levels
    return check_comm_err(s);
}

pmg_status pmg_pcg(pmg_solver *s, int precond, double rel_tol, int max_iter, double *res_history, int *n_iter_out)
{
    try {
        return pcg_impl(s, precond, rel_tol, max_iter, res_history, n_iter_out);
    } catch (const std::exception &e) {
        return fail(PMG_ERR_ALLOC, std::string("exception in pmg_pcg: ") + e.what());
    }
}

pmg_status pmg_last_device_ms(pmg_solver *s, double *ms_out)
{
    if (!s || !ms_out) return fail(PMG_ERR_INVALID, "null argument");
    *ms_out = s->last_ms;
    return PMG_OK;
}

void *pmg_stream(pmg_solver *s) { return s ? (void *)s->stream : nullptr; }

/* ---- tuning / benchmarking hooks (not part of the reference surface) ---------------------------------- */
/* run-time switch for the phase trace (same effect as PMG_DIST_TRACE=1 / 0) */
void pmg_dist_trace_enable(int on) { g_trace_on = on ? 1 : 0; }

/* PMG_DIST_TRACE=1: prints, per phase label and level, the average device time between consecutive marks of
 * the distributed cycle recorded since the last dump (the stream must be idle). */
void pmg_dist_trace_dump(int rank_to_print)
{
    if (g_trace.empty()) return;
    cudaDeviceSynchronize();
    struct Acc { double ms = 0; int n = 0; };
    std::vector<std::pair<std::string, Acc>> acc;
    for (size_t i = 1; i < g_trace.size(); ++i) {
        if (std::strcmp(g_trace[i].label, "begin") == 0 && g_trace[i].level == 0) continue;  // gap between cycles
        float ms = 0.f;
        cudaEventElapsedTime(&ms, g_trace[i - 1].ev, g_trace[i].ev);
        std::string key = std::string(g_trace[i].label) + "@" + std::to_string(g_trace[i].level);
        size_t k = 0;
        for (; k < acc.size(); ++k) if (acc[k].first == key) break;
        if (k == acc.size()) acc.push_back({key, Acc()});
        acc[k].second.ms += ms;
        acc[k].second.n += 1;
    }
    if (comm_rank() == rank_to_print) {
        double tot = 0;
        for (auto &a : acc) tot += a.second.ms / a.second.n;
        std::printf("[pmg trace rank %d] per-cycle phase times (us), total %.1f\n", comm_rank(), tot * 1e3);
        for (auto &a : acc) std::printf("   %-12s %8.1f  (x%d)\n", a.first.c_str(), 1e3 * a.second.ms / a.second.n, a.second.n);
        std::fflush(stdout);
    }
    for (auto &m : g_trace) cudaEventDestroy(m.ev);
    g_trace.clear();
}

/* generation of the single-CTA kernel for the levels <= 65 (1 or 2; 0 = default / PMG_SMALL_V2); graphs captured
 * with the other generation are dropped by the caller re-creating the solver */
void pmg_small_vcycle_set_version(int v) { vcycle_small_set_version(v); }
int pmg_small_vcycle_version(void) { return vcycle_small_version(); }

/* programmatic dependent launch of the cycle kernels (pmg_internal.h); takes effect for solvers created afterwards
 * (captured graphs keep the edges they were captured with) */
void pmg_set_pdl(int on) { pdl_set_enabled(on); }

/* cross-cycle solve (level 0: Pass B of cycle k and Pass A of cycle k+1 fused) for solvers created afterwards: 1, 0, or
 * -1 = PMG_CROSS / the default (on) */
void pmg_set_cross_cycle(int on) { g_cross_override = on < 0 ? -1 : (on >= 2 ? 2 : (on ? 1 : 0)); }
/* 1 if the last / next pmg_solve(PMG_CYCLE_V) on this handle takes the cross-cycle path */
int pmg_cross_cycle_active(const pmg_solver *s)
{
    if (!s) return 0;
    return s->dist ? (cross_ok_dist(s, false) ? 1 : 0) : (cross_ok(s, false) ? 1 : 0);
}
void pmg_fused_set_cross_minb(int m) { fused_set_cross_minb(m); }

/* top level of the 16-CTA cluster kernel for solvers created afterwards: 257, 129, 0 = off, -1 = PMG_CLUSTER / default */
void pmg_set_cluster_top(int n) { g_cluster_override = (n == 257 || n == 129 || n == 0) ? n : -1; }
int pmg_cluster_top(const pmg_solver *s) { return s ? s->cluster_top : 0; }

int pmg_fused_num_variants(void) { return fused_num_variants(); }
void pmg_fused_set_variant(int v) { fused_set_variant(v); }
void pmg_fused_set_min_chunk_rows(int r) { fused_set_min_chunk_rows(r); }
/* first visits of whole levels: skip the xb store and rebuild xb in Pass B -- -1 by size (default), 0 never, 1 always;
 * read when a cycle is recorded, so set it before the solver's first cycle */
void pmg_fused_set_rebuild_xb(int mode) { fused_set_rebuild_xb(mode); }
void pmg_fused_set_deep_prefetch_below(int n) { fused_set_deep_prefetch_below(n); }
void pmg_fused_set_halo_prologue(int on) { fused_set_halo_prologue(on); }

/* Times the single-CTA small-level kernel alone (benchmark hook): `reps` launches of one V- (gamma = 1) or W-visit of
 * the levels n0 (<= 65) ... 5 on scratch arrays, generation `version` (1, 2, 3); *us_avg = average microseconds per
 * launch, CUDA events on a private stream.  From T(n0, gamma) = own(n0) + gamma * T((n0-1)/2+1, gamma) the cost of one
 * visit of every level follows (tools/small_kernel_probe.py). */
pmg_status pmg_bench_small(int n0, int gamma, int reps, int version, double *us_avg)
{
    const bool cluster = coarse_cluster_top(n0);  // 129 / 257: the 16-CTA cluster kernel instead
    if (!us_avg || reps < 1 || gamma < 1 || n0 < 3 || (n0 > VSMALL_TOP && !cluster) || ((n0 - 1) & (n0 - 2)) != 0)
        return fail(PMG_ERR_INVALID, "bad argument");
    if (pmg_device_count() <= 0) return fail(PMG_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    const int pitch = level_pitch(n0);
    double *x = nullptr, *f = nullptr;
    pmg_status rc = alloc_zero(&x, level_elems(n0));
    if (rc == PMG_OK) rc = alloc_zero(&f, level_elems(n0));
    if (rc != PMG_OK) {
        cudaFree(x);
        return rc;
    }
    launch_fill2d(f + level_origin(n0) + pitch + 1, pitch, n0 - 2, n0 - 2, 1.0, nullptr);
    const int before = vcycle_small_version();
    vcycle_small_set_version(version);
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaStreamCreate(&st);
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    if (cluster && !coarse_cluster_available(n0)) {
        cudaFree(x);
        cudaFree(f);
        return fail(PMG_ERR_UNSUPPORTED, "a 16-CTA cluster cannot be scheduled on this device");
    }
    auto one = [&]() {
        if (cluster)
            launch_coarse_cluster(x + level_origin(n0), f + level_origin(n0), n0, pitch, pitch, 5, 1.0 / 1024.0, 2.0 / 3.0, 2, 2,
                                  11, PMG_PROLONG_REFERENCE, true, gamma, st, nullptr);
        else
            launch_vcycle_small(x + level_origin(n0), f + level_origin(n0), n0, pitch, pitch, 5, 1.0 / 1024.0, 2.0 / 3.0, 2, 2,
                                11, PMG_PROLONG_REFERENCE, true, gamma, st, nullptr);
    };
    cudaDeviceSynchronize();
    one();
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps; ++i) one();
    cudaEventRecord(e1, st);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    vcycle_small_set_version(before);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaStreamDestroy(st);
    cudaFree(x);
    cudaFree(f);
    if (e != cudaSuccess) return fail(PMG_ERR_CUDA, cudaGetErrorString(e));
    *us_avg = 1e3 * ms / reps;
    return PMG_OK;
}

/* cycles per level of the most recent coarse-kernel launch (k_coarse_local / k_coarse_cluster): slot k = own cycles of all
 * visits of level 2^k + 1 as seen by thread 0 (of CTA 0), slot 0 = the whole kernel body */
pmg_status pmg_coarse_profile(long long out[16])
{
    if (!out) return fail(PMG_ERR_INVALID, "null argument");
    PMG_CUDA(cudaDeviceSynchronize());
    coarse_profile_read(out);
    return PMG_OK;
}

/* `sweeps` weighted-Jacobi sweeps on the solver's finest level, `block` sweeps per streaming pass
 * (block = 1: one HBM pass per sweep, 24 B/point -- the "Jacobi sweep GB/s" sub-metric). */
pmg_status pmg_smooth(pmg_solver *s, int sweeps, int block)
{
    if (!s || sweeps < 0 || !fused_supported(block)) return fail(PMG_ERR_INVALID, "bad argument");
    if (s->dist) return fail(PMG_ERR_UNSUPPORTED, "pmg_smooth is single-GPU only");
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L = s->lv[0];
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    int left = sweeps;
    while (left > 0) {
        int b = left < block ? left : block;
        launch_fused_down(fused_view(L), nullptr, 0, b, s->cfg.omega, false, s->stream);
        std::swap(L.x, L.xb);
        std::swap(L.base_x, L.base_xb);
        left -= b;
    }
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    PMG_CUDA(cudaGetLastError());
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->last_ms = ms;
    drop_graphs(s);  // graphs captured earlier hold the old x/xb roles
    return PMG_OK;
}

/* Times one fused pass of level `level` in isolation: which = 0 Pass A (sweeps+residual+restriction),
 * 1 Pass B with the residual norm, 2 Pass B without, 3 Pass A with x == 0 (coarse-level form), 4 the cross-cycle pass
 * (Pass B of one cycle + Pass A of the next; level 0, one GPU, x_k not written as in pmg_solve), 5 Pass A with x == 0
 * without the xb store, 6 Pass B rebuilding xb from f (the pair a large first visit runs instead of 3 and 2), 7 the fused
 * residual-restriction R(f - A x) of the FMG set-up (one GPU), 8 the residual + restriction pair it replaces (the residual
 * stored in the level's xb array).  `reps`
 * launches between two CUDA events on the solver stream; *ms_avg = average per launch.  Clobbers the
 * iterate (benchmark use only). */
pmg_status pmg_bench_pass(pmg_solver *s, int which, int level, int reps, double *ms_avg)
{
    if (!s || !ms_avg || reps < 1 || level < 0 || level + 1 >= (int)s->lv.size() || !s->fused)
        return fail(PMG_ERR_INVALID, "bad argument (needs the fused engine and a non-coarsest level)");
    PMG_CUDA(cudaSetDevice(s->device));
    Level &L = s->lv[level];
    Level &K = s->lv[level + 1];
    const pmg_config &c = s->cfg;
    int np = 0;
    if (which == 4) {
        if (level != 0 || s->dist || !fused_cross_supported(c.nu1, c.nu2))
            return fail(PMG_ERR_UNSUPPORTED, "cross-cycle pass: level 0, one GPU, nu1 = nu2 = 2");
        pmg_status rcx = ensure_xc(s);
        if (rcx != PMG_OK) return rcx;
    }
    if ((which == 7 || which == 8) && s->dist) return fail(PMG_ERR_UNSUPPORTED, "forms 7 and 8 time a whole level (one GPU)");
    auto one = [&]() {
        if (which == 7) {
            launch_residual_restrict(L.x, L.f, K.f, L.n, K.n, K.n, 0, L.pitch, L.pitch, K.pitch, L.h, s->stream);
        } else if (which == 8) {
            launch_residual(L.xb, L.x, L.f, L.n, L.n, L.pitch, L.pitch, L.pitch, L.h, s->stream);
            launch_restrict(L.xb, K.f, L.n, K.n, L.pitch, K.pitch, s->stream);
        } else if (which == 4) {
            FusedLevel v = fused_view(L);
            v.x = nullptr;
            use_rhs_tables(s, v);  // the flavour pmg_solve runs
            launch_fused_cross(v, s->xc, K.x, K.f, K.pitch, c.omega, c.prolong_mode, s->d_partials, &np, s->stream);
        } else if (which == 0 || which == 3 || which == 5)
            launch_fused_down(fused_view(L), K.f, K.pitch, c.nu1, c.omega, which != 0, s->stream, nullptr, which != 5);
        else
            launch_fused_up(fused_view(L), K.x, K.pitch, c.nu2, c.omega, c.prolong_mode,
                            which == 1 ? s->d_partials : nullptr, &np, s->stream, nullptr, which == 6 ? c.nu1 : 0);
    };
    one();  // warm-up
    PMG_CUDA(cudaEventRecord(s->ev0, s->stream));
    for (int i = 0; i < reps; ++i) one();
    PMG_CUDA(cudaEventRecord(s->ev1, s->stream));
    PMG_CUDA(cudaEventSynchronize(s->ev1));
    PMG_CUDA(cudaGetLastError());
    float ms = 0.f;
    PMG_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    if (fused_take_bad_nu()) return fail(PMG_ERR_UNSUPPORTED, "this pass form needs a whole level (one GPU)");
    *ms_avg = ms / reps;
    return PMG_OK;
}

/* ---- test hooks: one fused pass on caller-built padded arrays (not part of the reference surface) ----------
 * tests/test_gpu_slab_kernels.py runs the multi-GPU flavours of Pass A / Pass B -- row slabs, halo rows read from a
 * "neighbour" through HaloPeers (in place or with the halo prologue), interior / boundary spans, rows finished beyond
 * the slab -- on ONE GPU, with every rank's arrays in the same device memory, and compares them with the oracle.
 * All pointers are device pointers to logical (0,0) of arrays in the solver's padded layout (pmg_test_layout). */
static pmg_status require_device();

typedef struct {
    double *x, *xb;
    const double *f;
    int n, pitch;
    double h;
    int ny, yoff, ext_lo, ext_hi, span_lo, span_hi;
    const double *x_up, *x_dn, *f_up, *f_dn;
    double *f_keep, *x_keep;
    int *flag_up, *flag_dn, *pub_up, *pub_dn;
    int epoch;
    int *err;
} pmg_test_slab;

void pmg_test_layout(int n, int *pitch, int *padx, int *pady)
{
    if (pitch) *pitch = level_pitch(n);
    if (padx) *padx = PADX;
    if (pady) *pady = PADY;
}

static FusedLevel test_view(const pmg_test_slab *t)
{
    FusedLevel v{};
    v.x = t->x;
    v.xb = t->xb;
    v.f = t->f;
    v.n = t->n;
    v.pitch = t->pitch;
    v.h = t->h;
    v.ny = t->ny;
    v.yoff = t->yoff;
    v.ext_lo = t->ext_lo;
    v.ext_hi = t->ext_hi;
    v.span_lo = t->span_lo;
    v.span_hi = t->span_hi;
    v.hp.x_up = t->x_up;
    v.hp.x_dn = t->x_dn;
    v.hp.f_up = t->f_up;
    v.hp.f_dn = t->f_dn;
    v.hp.f_keep = t->f_keep;
    v.hp.x_keep = t->x_keep;
    v.hp.flag_up = t->flag_up;
    v.hp.flag_dn = t->flag_dn;
    v.hp.pub_up = t->pub_up;
    v.hp.pub_dn = t->pub_dn;
    v.hp.epoch = t->epoch;
    v.hp.err = t->err;
    return v;
}

pmg_status pmg_test_fused_down(const pmg_test_slab *t, double *coarse_f, int pitch_c, int nu1, double omega, int x_is_zero,
                               int halo_prologue)
{
    if (!t || !fused_supported(nu1)) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    const int before = fused_halo_prologue();
    fused_set_halo_prologue(halo_prologue);
    launch_fused_down(test_view(t), coarse_f, pitch_c, nu1, omega, x_is_zero != 0, nullptr);
    fused_set_halo_prologue(before);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_test_fused_up(const pmg_test_slab *t, const double *coarse_x, int pitch_c, int nu2, double omega,
                             int prolong_mode, double *d_partials, int *n_partials)
{
    if (!t || !fused_supported(nu2)) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    FusedLevel v = test_view(t);
    v.hp = HaloPeers{};
    launch_fused_up(v, coarse_x, pitch_c, nu2, omega, prolong_mode, d_partials, n_partials, nullptr);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* Pass B with the deep-sweep schedule's coarse up-exchange on a caller-built slab: t->x / xb / f / ext as for
 * pmg_test_fused_up; t->x_up / x_dn / flags / pubs / epoch / err describe the COARSE iterate coarse_x (its neighbours'
 * copies, as cycle_dist passes them: x_up = the upper neighbour's coarse row ny_up), whose rows rows_from + 1 ..
 * rows_from + rows_count beyond the slab the prologue copies in.  abort (nullable): raised with err on a time-out. */
pmg_status pmg_test_fused_up_exchange(const pmg_test_slab *t, double *coarse_x, int pitch_c, int nu2, double omega,
                                      int prolong_mode, double *d_partials, int *n_partials, int rows_from, int rows_count,
                                      int *abort)
{
    if (!t || !coarse_x || !fused_supported(nu2) || rows_from < 0 || rows_count < 1 || rows_count > MAX_UP_ROWS || t->ny <= 0)
        return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    FusedLevel v = test_view(t);
    v.hp.f_up = v.hp.f_dn = nullptr;
    v.hp.f_keep = nullptr;
    v.hp.x_keep = coarse_x;
    v.hp.abort = abort;
    v.hp.rows_from = rows_from;
    v.hp.rows_count = rows_count;
    launch_fused_up(v, coarse_x, pitch_c, nu2, omega, prolong_mode, d_partials, n_partials, nullptr);
    if (fused_take_bad_nu()) return fail(PMG_ERR_UNSUPPORTED, "Pass B with the up-exchange refused these arguments");
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* the cross-cycle pass on a caller-built slab: t->xb = input (xb_k), t->x = where x_k goes (nullable), t->x_up / x_dn /
 * x_keep / flags = the neighbours' copies of the INPUT array (halo prologue) */
pmg_status pmg_test_fused_cross(const pmg_test_slab *t, double *xb_out, const double *coarse_x, double *coarse_f, int pitch_c,
                                double omega, int prolong_mode, double *d_partials, int *n_partials)
{
    if (!t || !xb_out || !coarse_x || !coarse_f || !d_partials) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    launch_fused_cross(test_view(t), xb_out, coarse_x, coarse_f, pitch_c, omega, prolong_mode, d_partials, n_partials, nullptr);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* the fused residual-restriction of the FMG set-up on caller-built arrays (launch_residual_restrict's arguments): a whole
 * level (rows_c = nc, yoff_c = 0) or one rank's row-slab window, so that tests/test_gpu_fmg_slabs.py covers the slab path on
 * one GPU */
pmg_status pmg_test_residual_restrict(const double *x, const double *f, double *coarse, int nf, int nc, int rows_c, int yoff_c,
                                      int pitch_x, int pitch_f, int pitch_c, double h)
{
    if (!x || !f || !coarse || nf < 3 || nc != (nf - 1) / 2 + 1 || rows_c < 0 || yoff_c < 0 || yoff_c + rows_c > nc)
        return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    launch_residual_restrict(x, f, coarse, nf, nc, rows_c, yoff_c, pitch_x, pitch_f, pitch_c, h, nullptr);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* the fused direction-operator pass of pmg_pcg on row slabs (launch_pcg_direction_apply's arguments) on caller-built arrays:
 * a whole level (rows = n, yoff = 0) or one rank's window, so that tests/test_gpu_pcg_slabs.py covers the slab path on one
 * GPU.  beta = *beta_num / *beta_den (device pointers); d_partials: PCG_MAX_PARTIALS doubles; *n_partials = count written */
pmg_status pmg_test_pcg_direction_apply(const double *z, const double *p_in, double *p_out, double *ap, int n, int rows, int yoff,
                                        int pitch, double h, const double *beta_num, const double *beta_den, int first,
                                        double *d_partials, int *n_partials)
{
    if (!z || !p_in || !p_out || !ap || !beta_num || !beta_den || !d_partials || !n_partials || n < 3 || rows < 1 ||
        yoff < 0 || yoff + rows > n)
        return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    *n_partials = launch_pcg_direction_apply(z, p_in, p_out, ap, n, rows, yoff, pitch, h, beta_num, beta_den, first != 0,
                                             d_partials, nullptr);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* the one-GPU pair the fused pass replaces, k_pcg_direction followed by k_apply_a_dot (and its final sum into *d_out), on a
 * whole level: the baseline tools/pcg_dist_probe.py times the fused pass against */
pmg_status pmg_test_pcg_direction_pair(const double *z, double *p, double *ap, int n, int pitch, double h, double beta, int first,
                                       double *d_partials, double *d_out)
{
    if (!z || !p || !ap || !d_partials || !d_out || n < 3) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    launch_pcg_direction(p, z, n, n, pitch, beta, first != 0, nullptr);
    launch_apply_a_dot(p, ap, n, n, pitch, h, d_partials, d_out, nullptr);
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* wall-time limit of the peer-flag waits (PMG_P2P_TIMEOUT_S), in milliseconds: lets a test provoke the time-out path */
void pmg_set_p2p_timeout_ms(double ms)
{
    const unsigned long long ns = (unsigned long long)((ms > 0.0 ? ms : 30000.0) * 1e6);
    fused_set_wait_timeout_ns(ns);
    basic_set_wait_timeout_ns(ns);
}

int pmg_test_fused_max_partials(int n) { return fused_max_partials(n); }

/* One fused pass over a WHOLE level (one GPU) on caller-built padded arrays, in each form the single-GPU solve launches,
 * for the pass-by-pass comparison with the oracle (tests/test_gpu_fused_pass_matrix.py).  `form`:
 *   0 Pass A smoothing only           xb = S^nu(x)
 *   1 Pass A                          xb = S^nu(x),      coarse_f = R(f - A xb)
 *   2 Pass A from x == 0              xb = S^nu(0),      coarse_f            (x not read)
 *   3 Pass A from x == 0, no xb store                    coarse_f            (x not read, xb not written)
 *   4 Pass A prolong-in (nu = 2)      xb = S^2(P coarse_x), coarse_f         (x not read)
 *   5 Pass B                          x = S^nu(xb + P coarse_x) (coarse_x nullable: no prolongation), norm partials if
 *                                     partials != null
 *   6 Pass B rebuilding xb            x = S^nu(S^nu_pre(0) + P coarse_x)     (xb not read)
 *   7 cross-cycle pass (nu = nu_pre = 2): x = S^2(xb + P coarse_x) (x nullable: not stored), its norm partials,
 *                                     xb_out = S^2 x, coarse_f = R(f - A xb_out); f generated from rhs_fx / rhs_sy when
 *                                     both are set (FusedLevel::rhs_fx)
 * The pass runs under the given tuning (the setters' arguments: pmg_fused_set_variant, _cross_minb, _min_chunk_rows,
 * _deep_prefetch_below); every tuning switch is put back afterwards.  A form no launcher serves is PMG_ERR_UNSUPPORTED. */
typedef struct {
    int form;
    double *x, *xb;
    const double *f;
    int n, pitch;
    double h;
    const double *coarse_x;
    double *coarse_f;
    int pitch_c;
    int nu, nu_pre;
    double omega;
    int prolong_mode;
    double *partials;
    int n_partials;  // out
    double *xb_out;
    const double *rhs_fx, *rhs_sy;
    int variant, cross_shape, min_chunk_rows, deep_prefetch_below;
} pmg_test_pass;

pmg_status pmg_test_fused_pass(pmg_test_pass *t)
{
    if (!t || t->form < 0 || t->form > 7 || !is_pow2_plus_1(t->n) || (t->form == 6 && t->nu_pre == 0))
        return fail(PMG_ERR_INVALID, "bad argument");
    if ((t->form == 4 && !fused_down_prolong_supported(t->nu)) ||
        (t->form == 7 && !fused_cross_supported(t->nu_pre, t->nu)))
        return fail(PMG_ERR_UNSUPPORTED, "no kernel for this sweep count in this pass form");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    FusedLevel v{};
    v.x = t->x;
    v.xb = t->xb;
    v.f = t->f;
    v.n = t->n;
    v.pitch = t->pitch;
    v.h = t->h;
    const FusedTuning saved = fused_get_tuning();
    fused_set_variant(t->variant);
    fused_set_cross_minb(t->cross_shape);
    fused_set_min_chunk_rows(t->min_chunk_rows);
    fused_set_deep_prefetch_below(t->deep_prefetch_below);
    t->n_partials = 0;
    switch (t->form) {
        case 0: launch_fused_down(v, nullptr, 0, t->nu, t->omega, false, nullptr); break;
        case 1:
        case 2:
        case 3:
            launch_fused_down(v, t->coarse_f, t->pitch_c, t->nu, t->omega, t->form != 1, nullptr, nullptr, t->form != 3);
            break;
        case 4:
            launch_fused_down_prolong(v, t->coarse_x, t->pitch_c, t->coarse_f, t->pitch_c, t->omega, t->prolong_mode, nullptr);
            break;
        case 5:
        case 6:
            launch_fused_up(v, t->coarse_x, t->pitch_c, t->nu, t->omega, t->prolong_mode, t->partials, &t->n_partials,
                            nullptr, nullptr, t->form == 6 ? t->nu_pre : 0);
            break;
        default:
            v.rhs_fx = t->rhs_fx;
            v.rhs_sy = t->rhs_sy;
            launch_fused_cross(v, t->xb_out, t->coarse_x, t->coarse_f, t->pitch_c, t->omega, t->prolong_mode, t->partials,
                               &t->n_partials, nullptr);
            break;
    }
    fused_set_tuning(saved);
    if (const int bad = fused_take_bad_nu())
        return fail(PMG_ERR_UNSUPPORTED,
                    "pass form " + std::to_string(t->form) + " launched nothing (" + std::to_string(bad) + ")");
    PMG_CUDA(cudaDeviceSynchronize());
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* ---- operator level (dense reference layout, device pointers) ------------------------------------------ */
// Scratch of the operator-level calls, one set PER DEVICE ordinal: reduction partials and the padded buffers of the
// blocked smoother.  The calls are synchronous, and they hold g_scratch_mu from launch to completion, so concurrent
// callers (any streams) never share a live scratch.  pmg_release_scratch() frees everything.
static std::mutex g_scratch_mu;
struct OpScratch {
    double *partials = nullptr;  // reduce_partials() + 2 doubles
    int jac_n = 0;
    double *jac[3] = {nullptr, nullptr, nullptr};
};
static OpScratch g_scratch[64];

static OpScratch &scratch_of_current_device()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return g_scratch[dev & 63];
}

// caller holds g_scratch_mu
static pmg_status op_scratch(double **partials)
{
    OpScratch &sc = scratch_of_current_device();
    if (!sc.partials) {
        if (cudaMalloc((void **)&sc.partials, (reduce_partials() + 2) * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            return fail(PMG_ERR_ALLOC, "cudaMalloc failed");
        }
    }
    *partials = sc.partials;
    return PMG_OK;
}

static pmg_status require_device()
{
    if (pmg_device_count() <= 0) return fail(PMG_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    return PMG_OK;
}

/* Long smoothing runs on a square dense field (the reference's "Jacobi, 100 iterations" micro-benchmark,
 * ParallelTestRunner.cu:275-284) go through the temporally blocked streaming kernel: the field is re-laid out on
 * the padded layout once, smoothed 4 sweeps per HBM pass, and copied back -- bit-identical to sweep-by-sweep. */
static pmg_status jacobi_blocked(double *x, const double *f, int n, double h, double omega, int sweeps, cudaStream_t st)
{
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    OpScratch &sc = scratch_of_current_device();
    double *(&buf)[3] = sc.jac;
    const size_t elems = level_elems(n), o = level_origin(n);
    if (sc.jac_n != n) {  // one size cached per device (the benchmark sweeps over sizes); pmg_release_scratch frees it
        for (double *&b : buf) {
            cudaFree(b);
            b = nullptr;
        }
        sc.jac_n = 0;
        for (double *&b : buf) {
            pmg_status rc = alloc_zero(&b, elems);
            if (rc != PMG_OK) {
                for (double *&c : buf) {
                    cudaFree(c);
                    c = nullptr;
                }
                return rc;
            }
        }
        sc.jac_n = n;
    }
    const int pitch = level_pitch(n);
    FusedLevel v{};
    v.x = buf[0] + o;
    v.xb = buf[1] + o;
    v.f = buf[2] + o;
    v.n = n;
    v.pitch = pitch;
    v.h = h;
    launch_copy2d(v.x, pitch, x, n, n, n, st);
    launch_copy2d(buf[2] + o, pitch, f, n, n, n, st);
    int left = sweeps;
    while (left > 0) {
        int b = left < 4 ? left : 4;
        launch_fused_down(v, nullptr, 0, b, omega, false, st);
        std::swap(v.x, v.xb);
        left -= b;
    }
    launch_copy2d(x, n, v.x, pitch, n, n, st);
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_jacobi(double *x, const double *f, int width, int height, double h, double omega, int sweeps,
                      double *scratch, void *stream)
{
    if (!x || !f || width < 3 || height < 3 || sweeps < 0) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (width == height && width >= 257 && sweeps >= 8) return jacobi_blocked(x, f, width, h, omega, sweeps, st);
    double *tmp = scratch;
    size_t bytes = (size_t)width * height * sizeof(double);
    if (!tmp && cudaMalloc((void **)&tmp, bytes) != cudaSuccess) {
        cudaGetLastError();
        return fail(PMG_ERR_ALLOC, "cudaMalloc failed");
    }
    double *a = x, *b = tmp;
    for (int it = 0; it < sweeps; ++it) {
        launch_jacobi_sweep(b, a, f, width, height, width, width, h, omega, st);
        std::swap(a, b);
    }
    cudaError_t e = cudaSuccess;
    if (a != x) e = cudaMemcpyAsync(x, a, bytes, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (!scratch) cudaFree(tmp);
    if (e != cudaSuccess) return fail(PMG_ERR_CUDA, cudaGetErrorString(e));
    return PMG_OK;
}

pmg_status pmg_gauss_seidel(double *x, const double *f, int width, int height, double h, int sweeps, int ordering,
                            void *stream)
{
    if (!x || !f || width < 3 || height < 3 || sweeps < 0 || (ordering != 0 && ordering != 1))
        return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (ordering == 0) {
        launch_gs_lex(x, f, width, height, width, width, h, sweeps, st);
    } else {
        for (int it = 0; it < sweeps; ++it) {
            launch_rbgs_half(x, f, width, height, width, width, h, 0, st);
            launch_rbgs_half(x, f, width, height, width, width, h, 1, st);
        }
    }
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_residual(double *r, const double *x, const double *f, int width, int height, double h,
                        double *norm2_out, void *stream)
{
    if (!x || !f || (!r && !norm2_out) || width < 3 || height < 3) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (r) launch_residual(r, x, f, width, height, width, width, width, h, st);
    std::unique_lock<std::mutex> lk(g_scratch_mu, std::defer_lock);
    if (norm2_out) {
        lk.lock();  // held until the result has been read back (below)
        double *part = nullptr;
        if ((rc = op_scratch(&part)) != PMG_OK) return rc;
        launch_residual_norm2(x, f, width, height, width, width, h, part, part + reduce_partials(), st);
        PMG_CUDA(cudaMemcpyAsync(norm2_out, part + reduce_partials(), sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_restrict_fw(const double *fine, double *coarse, int nf, int nc, void *stream)
{
    if (!fine || !coarse || nf < 3 || nc != (nf - 1) / 2 + 1) return fail(PMG_ERR_INVALID, "bad argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    launch_restrict(fine, coarse, nf, nc, nf, nc, st);
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_prolong_add(const double *coarse, double *fine, int nc, int nf, int mode, void *stream)
{
    if (!fine || !coarse || nf < 3 || nc != (nf - 1) / 2 + 1) return fail(PMG_ERR_INVALID, "bad argument");
    if (mode != PMG_PROLONG_REFERENCE && mode != PMG_PROLONG_FULL) return fail(PMG_ERR_INVALID, "bad prolong mode");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    launch_prolong_add(coarse, fine, nc, nf, nc, nf, mode, st);
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

pmg_status pmg_diff_norm2(const double *a, const double *b, size_t l, double *diff2_out, double *b2_out, void *stream)
{
    if (!a || !b || !diff2_out || !b2_out) return fail(PMG_ERR_INVALID, "null argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double *part = nullptr, *out = nullptr;
    if (cudaMalloc((void **)&part, (2 * reduce_partials() + 2) * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        return fail(PMG_ERR_ALLOC, "cudaMalloc failed");
    }
    out = part + 2 * reduce_partials();
    launch_diff_norm2(a, b, l, part, out, st);
    double h[2] = {0.0, 0.0};
    cudaError_t e = cudaMemcpyAsync(h, out, 2 * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFree(part);
    if (e != cudaSuccess) return fail(PMG_ERR_CUDA, cudaGetErrorString(e));
    *diff2_out = h[0];
    *b2_out = h[1];
    return PMG_OK;
}

pmg_status pmg_norm2(const double *v, size_t l, double *norm2_out, void *stream)
{
    if (!v || !norm2_out) return fail(PMG_ERR_INVALID, "null argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    double *part = nullptr;
    if ((rc = op_scratch(&part)) != PMG_OK) return rc;
    launch_norm2(v, l, part, part + reduce_partials(), st);
    PMG_CUDA(cudaMemcpyAsync(norm2_out, part + reduce_partials(), sizeof(double), cudaMemcpyDeviceToHost, st));
    PMG_CUDA(cudaStreamSynchronize(st));
    PMG_CUDA(cudaGetLastError());
    return PMG_OK;
}

/* frees the per-device scratch the operator-level calls keep between calls (reduction partials, the padded buffers of
 * the blocked smoother behind pmg_jacobi); safe at any time, the next call re-allocates */
pmg_status pmg_release_scratch(void)
{
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    int ndev = pmg_device_count(), cur = 0;
    if (ndev <= 0) return PMG_OK;
    cudaGetDevice(&cur);
    for (int d = 0; d < ndev && d < 64; ++d) {
        OpScratch &sc = g_scratch[d];
        if (!sc.partials && !sc.jac[0]) continue;
        cudaSetDevice(d);
        cudaFree(sc.partials);
        for (double *&b : sc.jac) {
            cudaFree(b);
            b = nullptr;
        }
        sc = OpScratch();
    }
    cudaSetDevice(cur);
    return PMG_OK;
}

/* ---- memory helpers ------------------------------------------------------------------------------------- */
pmg_status pmg_device_alloc(void **p, size_t bytes)
{
    if (!p) return fail(PMG_ERR_INVALID, "null argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    if (cudaMalloc(p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return fail(PMG_ERR_ALLOC, "cudaMalloc failed");
    }
    return PMG_OK;
}

pmg_status pmg_device_free(void *p)
{
    PMG_CUDA(cudaFree(p));
    return PMG_OK;
}

pmg_status pmg_host_alloc_pinned(void **p, size_t bytes)
{
    if (!p) return fail(PMG_ERR_INVALID, "null argument");
    pmg_status rc = require_device();
    if (rc != PMG_OK) return rc;
    if (cudaMallocHost(p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return fail(PMG_ERR_ALLOC, "cudaMallocHost failed");
    }
    return PMG_OK;
}

pmg_status pmg_host_free_pinned(void *p)
{
    PMG_CUDA(cudaFreeHost(p));
    return PMG_OK;
}

pmg_status pmg_memcpy(void *dst, const void *src, size_t bytes, int dst_is_device, int src_is_device)
{
    cudaMemcpyKind k = dst_is_device ? (src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice)
                                     : (src_is_device ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost);
    PMG_CUDA(cudaMemcpy(dst, src, bytes, k));
    return PMG_OK;
}

pmg_status pmg_device_synchronize(void)
{
    PMG_CUDA(cudaDeviceSynchronize());
    return PMG_OK;
}

/* rows [y0, y1) of an n-row level owned by `rank`: even-aligned splits so that coarse row jc lives where
 * fine row 2jc lives; the last rank also takes the odd final row. */
pmg_status pmg_partition_rows(int n, int n_ranks, int rank, int *y0, int *y1)
{
    if (n < 3 || n_ranks < 1 || rank < 0 || rank >= n_ranks || !y0 || !y1) return fail(PMG_ERR_INVALID, "bad argument");
    long pairs = (n - 1) / 2;  // fine row pairs (2j, 2j+1); the final row n-1 is appended to the last rank
    long a = pairs * rank / n_ranks, b = pairs * (rank + 1) / n_ranks;
    *y0 = (int)(2 * a);
    *y1 = (rank == n_ranks - 1) ? n : (int)(2 * b);
    return PMG_OK;
}

}  // extern "C"
