// pmg_internal.h -- declarations shared by the CUDA translation units of libpmg.so.
// Nothing here is part of the public ABI (that is include/pmg.h).
#pragma once
#if defined(PMG_HOST_EMULATION) && defined(__CUDACC__)
#error "PMG_HOST_EMULATION is for the g++-compiled kernel tests under tests/cpp only; libpmg.so is never built with it"
#endif
#ifdef PMG_HOST_EMULATION
// tests/cpp/emu/host_emulation.h: runs a single-CTA kernel's source on CPU threads (barrier logic and arithmetic
// checked against the oracle without a GPU); test infrastructure only, never part of libpmg.so
#include "host_emulation.h"
#else
#include <cuda_runtime.h>
#endif

#include <cstddef>
#include <cstdint>

#include "pmg.h"

namespace pmg {

// ---- HBM layout of one level (DESIGN.md section 3) -------------------------------------------------
// A level with n x n logical points (ring included) is stored as (n + 2*PADY) rows of `pitch`
// doubles.  Logical (row y, col x) lives at base[(y + PADY) * pitch + PADX + x].  PADX doubles on the
// left make logical column -PADX 128-byte aligned (base comes from cudaMalloc, pitch % 16 == 0), which
// is what the streaming kernels' 32-byte vector accesses need; the right padding lets every warp strip
// load its full 128 columns without a bounds test; PADY zero rows above and below do the same for the
// row pipeline warm-up/drain.  Padding is zero-filled once and never becomes non-zero.
constexpr int PADX = 16;
constexpr int PADY = 8;

inline int level_pitch(int n) { return ((PADX + n + 144) + 15) / 16 * 16; }
inline size_t level_elems(int n) { return (size_t)level_pitch(n) * (size_t)(n + 2 * PADY); }
inline size_t level_origin(int n) { return (size_t)PADY * level_pitch(n) + PADX; }

// un-fused arithmetic in the reference's evaluation order (no FMA contraction, whatever -fmad says)
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
// a*b + c in ONE instruction, used only where a is a power of two: the product is then exact, so the result is bit for
// bit that of dadd(dmul(a, b), c) (barring results below 2^-1022, which no grid function here reaches).  Likewise
// w*(0.25*s) == (0.25*w)*s: JacobiCoef::w4.  These save ~13 % of the fp64 instructions of a cycle.
__device__ __forceinline__ double dfma_pow2(double a, double b, double c) { return __fma_rn(a, b, c); }

struct JacobiCoef {
    double h2;      // h*h
    double omega;   // w
    double om1;     // 1.0 - w
    double w4;      // 0.25 * w (exact)
    int weighted;   // w != 1.0
};

// Smoother.hpp:66-68 + the omega form of SURVEY.md 8c:
//   jac = 0.25*((h*h*f) + W + E + S + N);  out = (w == 1) ? jac : (1-w)*x + w*jac
// `s` = up (row y-1, "idx - width"), `n` = down (row y+1, "idx + width")
__device__ __forceinline__ double jacobi_point(const JacobiCoef &c, double f, double xc, double xw,
                                               double xe, double xs, double xn)
{
    double acc = dadd(dadd(dadd(dadd(dmul(c.h2, f), xw), xe), xs), xn);
    return c.weighted ? dadd(dmul(c.om1, xc), dmul(c.w4, acc)) : dmul(0.25, acc);
}

// DynamicGridUtils.hpp:66:  f - (1.0/(h*h)) * (4*x - W - E - S - N)
__device__ __forceinline__ double residual_point(double inv_h2, double f, double xc, double xw,
                                                 double xe, double xs, double xn)
{
    double t = dsub(dsub(dsub(dfma_pow2(4.0, xc, -xw), xe), xs), xn);
    return dsub(f, dmul(inv_h2, t));
}

// MultiGrid.hpp:199-202:  0.25*c + 0.125*(E + W + N + S) + 0.0625*(SW + SE + NW + NE)
// (s* = row 2jc-1, n* = row 2jc+1; the reference adds "+1, -1, +Nf, -Nf" then "-Nf-1, -Nf+1, +Nf-1, +Nf+1")
__device__ __forceinline__ double restrict_point(double c, double e, double w, double n, double s,
                                                 double sw, double se, double nw, double ne)
{
    double edge = dadd(dadd(dadd(e, w), n), s);
    double corner = dadd(dadd(dadd(sw, se), nw), ne);
    return dfma_pow2(0.0625, corner, dfma_pow2(0.125, edge, dmul(0.25, c)));
}

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------
// The kernels of a cycle are short (5-30 us below level 2) and strictly dependent, so the ~2 us between the end of
// one and the start of the next is a visible part of a cycle (16-30 launches per V-cycle, thousands per W-cycle).  Every
// kernel on the cycle path is launched with cudaLaunchAttributeProgrammaticStreamSerialization and begins with
// pdl_prologue(): `griddepcontrol.wait` blocks until the preceding kernel has COMPLETED and its writes are visible
// (so nothing below it can observe a half-finished predecessor), `griddepcontrol.launch_dependents` then lets the
// NEXT kernel's CTAs be scheduled as this one's drain, where they park on their own wait.  Correctness never depends
// on it (without the attribute both instructions are no-ops); PMG_PDL=0 launches the classic way.
// Measured (profiles/r2_pdl_probe.log): 53.3 -> 49.6 us per V-cycle at N = 257, 305 -> 300 us at 4097 -- but a level-0
// pass at N = 16385 got 5 % SLOWER when its successor's CTAs were made resident early (they take shared memory and
// slots away from a kernel sized as exactly one resident wave).  So the big streaming passes release their
// dependents only when a warp has finished its rows (pdl_wait at the top, pdl_trigger at the end); the small
// kernels do both at the top.
#ifdef PMG_HOST_EMULATION
__device__ __forceinline__ void pdl_prologue() {}
__device__ __forceinline__ void pdl_wait() {}
__device__ __forceinline__ void pdl_trigger() {}
#else
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue()
{
    pdl_wait();
    pdl_trigger();
}
bool pdl_enabled();
void pdl_set_enabled(int on);
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- launch bookkeeping ---------------------------------------------------------------------------
void count_launch(int n = 1);
unsigned long long launches_so_far();
JacobiCoef jacobi_coef(double h, double omega);

// ---- operator-granular kernels (kernels_basic.cu); all pointers address logical (0,0) ------------
// out = one weighted-Jacobi sweep of in (interior); ring and nothing else copied from in
void launch_jacobi_sweep(double *out, const double *in, const double *f, int nx, int ny, int pitch_x,
                         int pitch_f, double h, double omega, cudaStream_t st);
// whole `sweeps` on a level that fits one CTA's shared memory (nx*ny <= SMALL_MAX_POINTS); in place
constexpr int SMALL_MAX_POINTS = 33 * 33;
// x_is_zero: start from x == 0 without reading x (first visit of a coarse level)
void launch_jacobi_small(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                         double omega, int sweeps, bool x_is_zero, cudaStream_t st, const int *done = nullptr);
// one V- (gamma = 1) or W-cycle (gamma visits of every coarser level) of the levels n0 (<= VSMALL_TOP) ... n_coarse
// in a single CTA's shared memory; x receives the result on the n0 level (whole array incl. ring);
// x_is_zero: start from 0 instead of reading x
constexpr int VSMALL_TOP = 65;
void launch_vcycle_small(double *x, const double *f, int n0, int pitch_x, int pitch_f, int n_coarse, double h0,
                         double omega, int nu1, int nu2, int coarse_sweeps, int prolong_mode, bool x_is_zero,
                         int gamma, cudaStream_t st, const int *done = nullptr);
// second generation of the same kernel (kernels_small.cu); launch_vcycle_small dispatches on vcycle_small_version()
constexpr int PMG_SMALL_DEFAULT_VERSION = 3;
int vcycle_small_version();
void vcycle_small_set_version(int v);  // 1, 2, 3, or 0 = re-read PMG_SMALL_VERSION / the default
// third generation (kernels_coarse.cu, k_coarse_local): level sizes are template parameters
bool coarse_local_supported(int n0, int gamma);
void launch_coarse_local(double *x, const double *f, int n0, int pitch_x, int pitch_f, int n_coarse, double h0, double omega,
                         int nu1, int nu2, int coarse_sweeps, int prolong_mode, bool x_is_zero, int gamma, cudaStream_t st,
                         const int *done = nullptr);
bool vcycle_small_v2_supported(int gamma);
void launch_vcycle_small_v2(double *x, const double *f, int n0, int pitch_x, int pitch_f, int n_coarse, double h0,
                            double omega, int nu1, int nu2, int coarse_sweeps, int prolong_mode, bool x_is_zero,
                            int gamma, cudaStream_t st, const int *done = nullptr);
void launch_residual(double *r, const double *x, const double *f, int nx, int ny, int pitch_r,
                     int pitch_x, int pitch_f, double h, cudaStream_t st);
// sum over the interior of (f - A x)^2 -> *d_out (device double); `d_partials` >= reduce_partials() doubles
int reduce_partials();
void launch_residual_norm2(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f,
                           double h, double *d_partials, double *d_out, cudaStream_t st);
// its first half: the partial sums only; returns how many (<= reduce_partials()) -- reduce with launch_final_sum
int launch_residual_partials(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                             double *d_partials, cudaStream_t st);
// same quantity summed in the reference's left-to-right order (bit-identical to the CPU loop; slow)
void launch_residual_norm2_sequential(const double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f,
                                      double h, double *d_out, cudaStream_t st);
void launch_norm2(const double *v, size_t l, double *d_partials, double *d_out, cudaStream_t st);
// fixed-order sum of `count` partials -> *d_out
void launch_final_sum(const double *d_partials, int count, double *d_out, cudaStream_t st);

// Device-side control block of an asynchronous solve: the last kernel of every cycle appends the residual
// norm to the history and raises `done` when ||r|| < rel_tol * ||r0|| or the cycle budget is used up; all
// later kernels see `done` and return immediately, so the host can queue cycles ahead without waiting.
struct SolveCtrl {
    double r0;        // ||r0||
    double rel_tol;
    int done;
    int cycles;       // cycles completed
    int max_cycles;
    int pad;
};
// hist2[0] = *d_norm2 ; ctrl initialised
void launch_solve_begin(const double *d_norm2, SolveCtrl *ctrl, double *hist2, double rel_tol, int max_cycles,
                        cudaStream_t st);
// hist2[++cycles] = fixed-order sum of the partials; convergence test (skipped when already done)
void launch_cycle_finish(const double *d_partials, int count, SolveCtrl *ctrl, double *hist2, cudaStream_t st);
// ---- smoothers beyond weighted Jacobi and the vector kernels of pmg_pcg (SURVEY.md 8f-3; kernels_basic.cu) ----
// mixed-precision experiment: one weighted-Jacobi sweep with fp32 arithmetic on the fp64 fields (SURVEY.md 8f-4)
void launch_jacobi_sweep_f32(double *out, const double *in, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h,
                             double omega, cudaStream_t st);
// d_out[0] = sum (a - b)^2, d_out[1] = sum b^2 over l entries; d_partials: 2 * reduce_partials() doubles
void launch_diff_norm2(const double *a, const double *b, size_t l, double *d_partials, double *d_out, cudaStream_t st);
// one colour ((x + y) & 1 == colour) of a red-black Gauss-Seidel sweep, in place; GaussSeidelSmoother's expression
void launch_rbgs_half(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h, int colour,
                      cudaStream_t st);
// `sweeps` lexicographic Gauss-Seidel sweeps exactly as Smoother.hpp:134-145 (anti-diagonal wavefront, one CTA)
void launch_gs_lex(double *x, const double *f, int nx, int ny, int pitch_x, int pitch_f, double h, int sweeps, cudaStream_t st);
// ap = A p (interior) and *d_out = p . ap ; *d_out = a . b ; x += alpha p, r -= alpha ap, *d_out = r . r ; p = z + beta p
void launch_apply_a_dot(const double *p, double *ap, int nx, int ny, int pitch, double h, double *d_partials, double *d_out,
                        cudaStream_t st);
void launch_dot_interior(const double *a, const double *b, int nx, int ny, int pitch, double *d_partials, double *d_out,
                         cudaStream_t st);
void launch_pcg_update(double *x, double *r, const double *p, const double *ap, int nx, int ny, int pitch, double alpha,
                       double *d_partials, double *d_out, cudaStream_t st);
void launch_pcg_direction(double *p, const double *z, int nx, int ny, int pitch, double beta, bool first, cudaStream_t st);
// row slabs (kernel_pcg.cuh): the fused direction-operator pass and the update with device-side scalars, on the owned
// rows [0, rows) of a window whose local row 0 is global row yoff (whole level: rows = n, yoff = 0).  Each writes one
// partial sum per warp to d_partials (at most PCG_MAX_PARTIALS) and returns their count (0: nothing to do)
constexpr int PCG_MAX_PARTIALS = 148 * 32;
int launch_pcg_direction_apply(const double *z, const double *p_in, double *p_out, double *ap, int n, int rows, int yoff, int pitch,
                               double h, const double *beta_num, const double *beta_den, bool first, double *d_partials,
                               cudaStream_t st);
int launch_pcg_update_dev(double *x, double *r, const double *p, const double *ap, int n, int rows, int yoff, int pitch,
                          const double *alpha_num, const double *alpha_den, double *d_partials, cudaStream_t st);

// *host_ctrl = *ctrl and (host_hist != nullptr) host_hist[0..cycles] = hist2[...], both in mapped pinned host memory,
// written by a kernel: no copy engine involved (see k_ctrl_to_host)
void launch_ctrl_to_host(const SolveCtrl *ctrl, SolveCtrl *host_ctrl, const double *hist2, double *host_hist, int hist_cap,
                         cudaStream_t st);
void launch_restrict(const double *fine, double *coarse, int nf, int nc, int pitch_f, int pitch_c,
                     cudaStream_t st);
void launch_prolong_add(const double *coarse, double *fine, int nc, int nf, int pitch_c, int pitch_f,
                        int mode, cudaStream_t st);
// the same two operators on ROW SLABS (pointers address each slab's local row 0, column 0): rows_c / rows_f local
// rows whose global index is local + yoff_c / yoff_f; yoff_f is even and the coarse slab starts at yoff_f / 2, so
// local fine row 2j sits under local coarse row j.  Restriction reads fine rows [-1, 2*rows_c); prolongation
// reads coarse rows [0, rows_f / 2 + 1].
void launch_restrict_rows(const double *fine, double *coarse, int nc, int rows_c, int yoff_c, int pitch_f,
                          int pitch_c, cudaStream_t st);
void launch_prolong_add_rows(const double *coarse, double *fine, int nf, int rows_f, int yoff_f, int pitch_c,
                             int pitch_f, int mode, cudaStream_t st);
// coarse(interior) = R(f - A x) in one pass (kernel_residual_restrict.cuh), bit-identical to launch_residual into a scratch
// array followed by launch_restrict; 18 B per fine point instead of 34.  Same slab convention as launch_restrict_rows
// (whole level: rows_c = nc, yoff_c = 0); reads x rows [-2, 2 rows_c] and f rows [-1, 2 rows_c - 1] of the fine window.
void launch_residual_restrict(const double *x, const double *f, double *coarse, int nf, int nc, int rows_c, int yoff_c,
                              int pitch_x, int pitch_f, int pitch_c, double h, cudaStream_t st);
// dst(y,x) = src(y,x) for a ny x nx window, arbitrary pitches (layout conversion at the ABI)
void launch_copy2d(double *dst, int pitch_d, const double *src, int pitch_s, int nx, int ny,
                   cudaStream_t st);
void launch_fill2d(double *dst, int pitch_d, int nx, int ny, double v, cudaStream_t st);
// f(y,x) = (factor * sx[x]) * sy[y]   (DynamicGridUtils.hpp:113-122 with 1-D sine tables)
void launch_rhs_separable(double *f, int pitch, int nx, int ny, double factor, const double *sx,
                          const double *sy, cudaStream_t st);

// The cluster kernel (kernels_coarse.cu, k_coarse_cluster): the levels n0 (257 or 129) ... n_coarse of one V- or W-cycle
// in ONE launch of a 16-CTA thread-block cluster, levels >= 33 distributed over the CTAs' shared memories (DSMEM).
// Returns false -- and launches nothing -- when the configuration or the device cannot run it (the caller then takes
// the streaming passes + the single-CTA kernel).
bool coarse_cluster_top(int n);
bool coarse_cluster_available(int n0);
// per-level cycle profile of the last coarse-kernel launch on the current device (slot k: level 2^k + 1, slot 0: all)
void coarse_profile_read(long long out[16]);
bool launch_coarse_cluster(double *x, const double *f, int n0, int pitch_x, int pitch_f, int n_coarse, double h0, double omega,
                           int nu1, int nu2, int coarse_sweeps, int prolong_mode, bool x_is_zero, int gamma, cudaStream_t st,
                           const int *done = nullptr);

// ---- fused streaming kernels (kernels_fused.cu) ---------------------------------------------------
// Halo rows read straight out of the neighbours' HBM over NVLink (all null on one GPU / when the halo rows are
// local).  Local row r < 0 lives at up + r*pitch, local row r >= ny at dn + (r - ny)*pitch (pointers to logical
// column 0).  f halo rows fetched this way are also written to `f_keep` so that the later Pass B reads them locally.
struct HaloPeers {
    const double *x_up, *x_dn, *f_up, *f_dn;
    double *f_keep;                // local f (writable): halo rows fetched from a peer are kept for Pass B
    const int *flag_up, *flag_dn;  // inbox flags that must reach `epoch` before the first peer access
    int *pub_up, *pub_dn;          // the neighbours' inbox slots for ME (peer pointers): thread 0 of the launch
                                   // publishes `epoch` there first -- everything this stream ran before the launch
                                   // is complete, so "my boundary rows are final" needs no kernel of its own
    int epoch;
    int *err;                      // raised if that wait times out
    double *x_keep;                // local x (writable): where the halo prologue stores the neighbours' x rows
    const int *epoch_base;         // (nullable) device int added to `epoch`: a captured launch keeps its arguments, so
                                   // the host writes the visit's epoch to device memory before each graph replay
    int *abort;                    // (nullable) the solve's device-side `done` flag: raised together with *err so that
                                   // the finest level's last pass does not commit an iterate built on stale halo rows
    // Pass B's up-exchange (deep-sweep slab schedule, x_keep != nullptr in launch_fused_up): x_up / x_dn / x_keep / flags
    // describe the COARSE iterate, and the prologue copies its rows at depth rows_from + 1 .. rows_from + rows_count
    // beyond the slab (rows_count <= MAX_UP_ROWS) -- the ones the child's own Pass B did not finish
    int rows_from, rows_count;
};
constexpr int MAX_UP_ROWS = 4;

#if !defined(PMG_HOST_EMULATION) && defined(PMG_NEEDS_PEER_WAIT)
// Bounded acquire spin on a flag another GPU publishes with st.release.sys.  The bound is WALL time on the device
// (%globaltimer), 30 s unless PMG_P2P_TIMEOUT_S says otherwise (pmg_create): ordinary rank skew -- a rank doing host I/O
// between cycles, first-use graph instantiation, lazy module load -- must never trip it; it exists so that a DEAD
// neighbour turns into PMG_ERR_COMM instead of a hung GPU.  One copy of the limit per translation unit that waits on
// peers (the library is built without relocatable device code); each TU exports a setter (…_set_wait_timeout_ns).
static __device__ unsigned long long g_wait_timeout_ns = 30ull * 1000ull * 1000ull * 1000ull;
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ bool wait_flag(const int *flag, int epoch)
{
    unsigned long long t0 = 0;
    unsigned ns = 32;
    for (unsigned it = 0;; ++it) {
        int v;
        asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v >= epoch) return true;
        __nanosleep(ns);
        if (ns < 1000) ns *= 2;  // short polls first (the usual wait is a few microseconds), then back off
        if ((it & 255u) == 255u) {
            const unsigned long long now = global_timer_ns();
            if (t0 == 0)
                t0 = now;
            else if (now - t0 > g_wait_timeout_ns)
                return false;
        }
    }
}
#endif

struct FusedLevel {
    double *x;    // logical (0,0) of the level's current iterate
    double *xb;   // ping-pong partner
    const double *f;
    int n, pitch;
    double h;
    // row slab of a level partitioned over ranks (all zero on one GPU): the arrays hold local rows
    // [-PADY, ny + PADY); local row 0 is global row yoff.  ext_lo/ext_hi: see StripGeom.
    int ny, yoff, ext_lo, ext_hi;
    int span_lo, span_hi;  // if span_hi > span_lo: write only local rows [span_lo, span_hi) (span_lo even)
    HaloPeers hp;          // Pass A: fused halo exchange (wait for the neighbours, read their rows in place);
                           // Pass B: the coarse iterate's up-exchange when hp.x_keep != nullptr (see HaloPeers)
    // (nullable; cross-cycle pass, one GPU) f is separable and bit for bit f(y, x) = fx[x] * sy[y] with zeros in the padding:
    // fx addresses logical column 0 of one padded row (pitch doubles), sy logical row 0 of n + 2*PADY entries.  The
    // default shape then forms f in the pass instead of reading it (20 B/point instead of 28).
    const double *rhs_fx, *rhs_sy;
};
// Pass A (down): xb = S^nu1(x);  coarse_f(interior) = R(f - A xb).  x_is_zero: the iterate is known to
// be identically zero on entry (coarse levels of a V-cycle) so x is not read.
bool fused_supported(int nu);
// Pass A with the iterate on entry given as P e_in (prolongation of a coarse iterate into zero), never materialised
bool fused_down_prolong_supported(int nu1);
void launch_fused_down_prolong(const FusedLevel &lv, const double *e_in, int pitch_e, double *coarse_f, int pitch_c, double omega,
                               int prolong_mode, cudaStream_t st, const int *done = nullptr);
// a launcher called with an unsupported sweep count launches nothing and records the count; returns and clears it
// (0 = none; -1 = a store_xb / rebuild_nu1 request outside a first visit of a whole level, or a sweep count of 0): the
// cycle drivers turn it into PMG_ERR_UNSUPPORTED instead of a silently skipped pass
int fused_take_bad_nu();
// `done` (nullable): device flag; when set the kernel returns at once (device-side convergence control)
// store_xb = false (x_is_zero, coarse_f, whole level only): xb is not written; Pass B must then rebuild it (rebuild_nu1)
void launch_fused_down(const FusedLevel &lv, double *coarse_f, int pitch_c, int nu1, double omega,
                       bool x_is_zero, cudaStream_t st, const int *done = nullptr, bool store_xb = true);
// Pass B (up): x = S^nu2(xb + P coarse_x); optionally sum (f - A x)^2 over the interior into partials
// (count returned through *n_partials; reduce with launch_final_sum)
// rebuild_nu1 > 0 (whole level, coarse_x, no norm): xb is not read but rebuilt as S^nu1(0; f) -- after a Pass A with
// x_is_zero and store_xb = false
// lv.hp.x_keep != nullptr (row slabs, deep-sweep schedule): before the prolongation, the coarse prologue publishes
// lv.hp.epoch, the warps whose rows reach beyond the slab wait for the neighbours' epoch and copy the coarse rows
// lv.hp.rows_from + 1 .. + rows_count beyond the slab from lv.hp.x_up / x_dn into lv.hp.x_keep (== coarse_x)
void launch_fused_up(const FusedLevel &lv, const double *coarse_x, int pitch_c, int nu2, double omega,
                     int prolong_mode, double *d_partials, int *n_partials, cudaStream_t st,
                     const int *done = nullptr, int rebuild_nu1 = 0);
// Whether a first visit (x == 0) of this level skips the xb store and rebuilds xb in Pass B: whole levels whose three
// arrays (x, xb, f) exceed the L2 cache.  Below that the xb store and read stay in L2 and cost less than the extra sweep.
bool fused_rebuild_xb(const FusedLevel &lv, int nu1);
// -1: by size (default; PMG_REBUILD_XB=0/1 in the environment overrides it), 0: never, 1: on every whole level
void fused_set_rebuild_xb(int mode);
int fused_max_partials(int n);
// Cross-cycle pass (level 0 of a V-cycle solve, one GPU): Pass B of cycle k and Pass A of cycle k+1 in one sweep over
// HBM -- reads lv.xb (xb_k), coarse_x (e_k), lv.f; writes lv.x (x_k), xb_out (xb_{k+1}, NOT lv.xb), coarse_f and the partial
// sums of the residual norm of x_k.  36 B/point instead of 52 (28 without x_k; 20 when f comes from lv.rhs_fx / rhs_sy).  Row slabs: lv.hp = the neighbours' copies of the INPUT array
// (x_up / x_dn / x_keep / flags / epoch as for Pass A); rows [0, ny) are written, 6 halo rows above and 4 below are read.
bool fused_cross_supported(int nu1, int nu2);
double fused_cross_utilisation(int n, int rows);  // resident warp slots the pass fills (the solve wants >= 0.9)
void launch_fused_cross(const FusedLevel &lv, double *xb_out, const double *coarse_x, double *coarse_f, int pitch_c, double omega,
                        int prolong_mode, double *d_partials, int *n_partials, cudaStream_t st, const int *done = nullptr);
void fused_set_cross_minb(int m);  // CTAs per SM promised to the compiler for the cross-cycle pass (2, 3, 4)
// tuning: which (columns per lane, prefetch depth, CTAs per SM) instantiation the nu == 2 passes use
int fused_num_variants();
void fused_set_variant(int v);
int fused_get_variant();
void fused_set_min_chunk_rows(int r);
// levels with n <= this run the nu == 2 passes with the deep-prefetch variant (7 rows in flight per warp);
// n < 0: back to PMG_DEEP_PREFETCH_BELOW / the default
constexpr int PMG_DEEP_PREFETCH_DEFAULT = 0;
void fused_set_deep_prefetch_below(int n);
// Pass A's fused halo exchange copies the neighbours' halo rows in a prologue (all loads in flight, only the
// boundary warps wait for the flags) instead of streaming them in place.  Default since round 2: bit-identical on
// 2 and 8 GPUs and, together with the middle graph and no interior/boundary split, 657 -> 566 us per V-cycle at
// N = 16385 on 8 GPUs (profiles/r2_dist8_latency_options.log).  PMG_HALO_PROLOGUE=0 restores in-place streaming.
constexpr int PMG_HALO_PROLOGUE_DEFAULT = 1;
void fused_set_halo_prologue(int on);
int fused_halo_prologue();
// every tuning switch of the fused passes above (variants, cross-pass shape, chunk rows, deep prefetch, xb rebuild, halo
// prologue), read and written as a whole so that a caller can run one pass under other settings and put them back
struct FusedTuning {
    int variant_down, variant_down_zero, variant_up, variant_up_norm, cross_minb, min_chunk_rows, deep_prefetch_below,
        rebuild_xb, halo_prologue;
};
FusedTuning fused_get_tuning();
void fused_set_tuning(const FusedTuning &t);
// limit of the peer-flag waits (wait_flag above), per translation unit that waits
void fused_set_wait_timeout_ns(unsigned long long ns);
void basic_set_wait_timeout_ns(unsigned long long ns);

// ---- multi-GPU plumbing (comm.cu): no-ops returning PMG_OK while no communicator exists ---------------
bool comm_ready();
int comm_rank();
int comm_size();
pmg_status comm_halo_exchange(double *p, int ny, int pitch, int depth, cudaStream_t st);
pmg_status comm_gather_rows(const double *slab, double *full, int pitch, const int *y0s, const int *y1s,
                            cudaStream_t st);
pmg_status comm_scatter_rows(const double *full, double *slab, int n_rows, int pitch, const int *y0s,
                             const int *y1s, int halo, cudaStream_t st);
pmg_status comm_allgather_double(const double *d_mine, double *d_all, cudaStream_t st);
// CUDA IPC in three phases so that no rank can leave a collective half way: (1) exchange handles (collective),
// (2) open the mappings needed (local), (3) agree that everybody succeeded (collective).
constexpr int IPC_HANDLE_BYTES = 64;
pmg_status comm_ipc_exchange(void *base, unsigned char *handles /* n_ranks * IPC_HANDLE_BYTES */, cudaStream_t st);
void *comm_ipc_open(const unsigned char *handle);
bool comm_all_agree(bool ok, double *d_scratch /* 1 + n_ranks doubles; nullptr: the communicator's own */, cudaStream_t st);
void comm_ipc_close(void *peer);

// ---- NVLink peer-to-peer halo exchange (kernels_basic.cu) -------------------------------------------------
// Producer side: after the kernel that finished this rank's boundary rows, publish `epoch` in the neighbours'
// inbox flags (system-scope release).  up_flag / dn_flag: peer pointers, null where there is no neighbour.
void launch_halo_signal(int *up_flag, int *dn_flag, int epoch, cudaStream_t st);
// Consumer side: wait (bounded spin, acquire) until both neighbours have published `epoch` in MY inbox flags,
// then copy their `depth` boundary rows straight out of their arrays over NVLink into my halo rows.
//   mine: logical origin of my slab array, ny owned rows; up_src: peer pointer to the upper neighbour's row
//   (its ny - depth), dn_src: peer pointer to the lower neighbour's row 0; flags: my inbox {from_up, from_dn};
//   err: device int raised if the spin times out.
void launch_halo_pull(double *mine, int ny, int pitch, int depth, const double *up_src, const double *dn_src,
                      const int *flag_from_up, const int *flag_from_dn, int epoch, int *err, cudaStream_t st,
                      int *abort = nullptr);
// All-gather of a slab-partitioned level over NVLink: `slots[r]` = rank r's inbox slot for THIS rank (peer
// pointers, device array); every rank publishes `epoch` there, then pulls the other ranks' `rows` slab rows
// (`srcs[r]` = peer pointer to rank r's padded row 0, device array; srcs[my_rank] is local) into `full`.
void launch_signal_all(int *const *slots, int n_ranks, int my_rank, int epoch, cudaStream_t st);
// slots != nullptr: the pull kernel publishes `epoch` itself (no launch_signal_all needed before it)
// epoch_base (nullable): device int added to `epoch` (graph replay, see HaloPeers)
void launch_gather_pull(double *full, int pitch, int rows, const double *const *srcs, const int *inbox, int n_ranks,
                        int my_rank, int epoch, int *err, cudaStream_t st, int *const *slots = nullptr,
                        const int *epoch_base = nullptr, int *abort = nullptr);
// dst[i] = vals[i], i < count <= 16 (the epochs of one cycle, written ahead of a graph replay)
struct IntPack16 {
    int v[16];
};
void launch_set_ints(int *dst, const IntPack16 &vals, int count, cudaStream_t st);
// every rank contributes `rows` owned rows of its slab; all ranks receive the whole level (rank r's block at
// row r*rows of `full`).  Needs equally sized slabs (the extra last row of the last rank is the zero ring).
pmg_status comm_allgather_rows(const double *slab, double *full, int rows, int pitch, cudaStream_t st);

}  // namespace pmg
