/*
 * pmg.h -- C ABI of the B200-native geometric multigrid solver for the 2-D Poisson problem.
 *
 * This is the drop-in boundary for the reference's multigrid hot path.  The reference
 * (FraVirgu/Parallel-Geometric-Multigrid-for-Poisson-problem) has no FFI layer: its boundary is the
 * C++ class surface
 *     Smoother::smooth                                   Smoother.hpp:23-28
 *     MultigridSolver::{v_cycle,w_cycle,f_cycle}         2_part_MG/MultiGrid.hpp:57,96,138
 *     Parallel::{ComputeJacobi,ComputeResidual,ComputeRestriction,ComputeProlungator}
 *                                                        3_part_parallel/Parallel_Method.cu:144-199
 *     ParallelMultiGridSolver::{v_cycle,w_cycle}         3_part_parallel/Parallel_Mg.cu:21,62
 * include/pmg.hpp re-creates those class shapes on top of the functions below, so a reference
 * runner is re-pointed at this library by changing an #include (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, `pmg_status` return codes (the reference has no error
 *     reporting at all; here every CUDA/NCCL failure is surfaced, nothing falls back to the CPU).
 *   - Field layout at the ABI = the reference's: row-major N x N doubles INCLUDING the Dirichlet
 *     ring, idx = y*width + x (Smoother.hpp:65), N = 2^k + 1, h = 1/(N-1).  Internally the solver
 *     re-lays fields out on a padded, 128-byte-pitched hierarchy in HBM (DESIGN.md section 3).
 *   - Sweep counts are TRUE sweep counts.  The reference's `num_iter` means num_iter+1 sweeps
 *     (Smoother.hpp:59); the C++ shims in pmg.hpp do the +1.
 *   - fp64 throughout.  The stencil arithmetic reproduces the reference's expression order without
 *     FMA contraction, so operator outputs are bit-identical to the CPU path; only the residual
 *     NORM (a parallel tree sum instead of a left-to-right sum) differs, by ~1e-15 relative.
 *   - One solver handle is used by one host thread at a time; different handles are independent.
 */
#ifndef PMG_H
#define PMG_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMG_VERSION_MAJOR 0
#define PMG_VERSION_MINOR 1

typedef enum pmg_status {
    PMG_OK = 0,
    PMG_ERR_INVALID = 1,     /* bad argument (size not 2^k+1, null pointer, bad enum ...)          */
    PMG_ERR_CUDA = 2,        /* a CUDA runtime call or kernel failed; see pmg_last_error()         */
    PMG_ERR_NO_DEVICE = 3,   /* no sm_100 device visible: there is NO CPU fallback                 */
    PMG_ERR_ALLOC = 4,       /* device or pinned-host allocation failed                            */
    PMG_ERR_COMM = 5,        /* NCCL / peer-access failure in the multi-GPU path                   */
    PMG_ERR_UNSUPPORTED = 6  /* valid request this build cannot serve (documented at the function) */
} pmg_status;

/* MultigridSolver::v_cycle / w_cycle / f_cycle (MultiGrid.hpp:57 / :96 / :138) */
typedef enum pmg_cycle_kind {
    PMG_CYCLE_V = 0,
    PMG_CYCLE_W = 1,
    PMG_CYCLE_F = 2,
    /* NOT in the reference: one full-multigrid pass for an ARBITRARY right-hand side and Dirichlet ring (the
     * reference's F-cycle regenerates the analytic RHS on every level, MultiGrid.hpp:162, and zeroes the ring).
     * The iterate's ring is kept, its interior restarted from 0: r0 = f - A x; f_1 = R r0, f_{l+1} = R f_l; coarsest
     * level: coarse_sweeps sweeps from 0; upwards e_l = P e_{l+1} and one V-cycle on (e_l, f_l); finest level
     * x += P e_1 and one V-cycle on (x, f).  pmg_solve with this kind = one such pass, then V-cycles.  One GPU, and
     * row slabs too (n_ranks a power of two; otherwise PMG_ERR_UNSUPPORTED on every rank).
     * Specification: the CPU checker's orc_fmg_general, which the GPU result equals bit for bit. */
    PMG_CYCLE_FMG = 3
} pmg_cycle_kind;

/* PMG_PROLONG_REFERENCE reproduces MultigridSolver::prolongation (MultiGrid.hpp:208-226): fine row 1
 * and fine column 1 receive no correction.  PMG_PROLONG_FULL corrects every interior fine point
 * (what the reference's GPU kernel does, Parallel_Method.cu:79-138) -- not parity with the CPU path,
 * 3x fewer cycles. */
typedef enum pmg_prolong_mode { PMG_PROLONG_REFERENCE = 0, PMG_PROLONG_FULL = 1 } pmg_prolong_mode;

typedef enum pmg_mem { PMG_MEM_HOST = 0, PMG_MEM_DEVICE = 1 } pmg_mem;

/* DynamicGridUtils::norm (DynamicGridUtils.hpp:21-27) adds the squares left to right.  On smooth fields
 * that running sum drifts: at N = 16385 it differs from the exactly rounded sum by up to ~1e-9 relative.
 * PMG_NORM_TREE (default) is a deterministic parallel tree sum fused into the last pass (accurate to
 * ~1e-15, agrees with the reference to <= 1e-10 up to N = 4097 and to 2e-9 at N = 16385).
 * PMG_NORM_SEQUENTIAL reproduces the reference's summation order on the device, one element at a time,
 * so every per-cycle norm is BIT-IDENTICAL to the CPU path at any size; it costs ~4 ns per grid point
 * per norm and exists for validation. */
typedef enum pmg_norm_mode { PMG_NORM_TREE = 0, PMG_NORM_SEQUENTIAL = 1 } pmg_norm_mode;

/* Smoothers behind the reference's `Smoother` interface (Smoother.hpp:8-31), injected into the cycles like
 * MultigridSolver's Smoother* (MultiGrid.hpp:12,22):
 *   JACOBI     weighted Jacobi (omega = 1: JacobiSmoother, Smoother.hpp:33-117) -- the only one the fused engine runs;
 *   RBGS       Gauss-Seidel in red-black order, the parallel form of GaussSeidelSmoother: same update expression
 *              (Smoother.hpp:141-143), points with (x + y) even first, then the odd ones;
 *   GS_LEX     GaussSeidelSmoother EXACTLY, lexicographic order included (anti-diagonal wavefront on one CTA): bit-identical
 *              to the reference, a validation path -- ~2n dependent steps per sweep;
 *   CHEBYSHEV  Chebyshev-Jacobi: the Jacobi sweep with per-sweep weights w_k = 1 / (d - c cos(pi (2k+1) / (2 nu))) for the
 *              eigenvalue range [1/2, 2] of D^-1 A (d = 5/4, c = 3/4); omega is ignored.
 * All but JACOBI run on the operator engine (one kernel per sweep / half sweep), single GPU.  Sweep counts are TRUE counts
 * for every smoother (the reference's GaussSeidelSmoother loops `iter < num_iter`, its Jacobi `<=`; the C++ shims do the
 * mapping). */
typedef enum pmg_smoother {
    PMG_SMOOTHER_JACOBI = 0,
    PMG_SMOOTHER_RBGS = 1,
    PMG_SMOOTHER_GS_LEX = 2,
    PMG_SMOOTHER_CHEBYSHEV = 3
} pmg_smoother;

typedef enum pmg_engine {
    PMG_ENGINE_FUSED = 0,   /* temporally blocked streaming kernels (2 HBM passes per level visit)  */
    PMG_ENGINE_OPERATOR = 1 /* one kernel per reference operator (Parallel::Compute* granularity)  */
} pmg_engine;

typedef struct pmg_config {
    int n;               /* grid points per side, 2^k + 1, k >= 1                                   */
    int nu1, nu2;        /* pre / post smoothing sweeps (reference v1+1 / v2+1 = 2 / 2)             */
    double omega;        /* Jacobi weight; 1.0 = the reference's undamped smoother bit for bit      */
    int gamma;           /* W-cycle recursion count (reference `alpha`, MultiGrid.hpp:13,124)       */
    int n_coarse;        /* coarsest level size (MultiGrid.hpp:19: 5)                               */
    int coarse_sweeps;   /* sweeps on the coarsest level (MultiGrid.hpp:61: 10+1)                   */
    int fmg_sweeps;      /* sweeps per level on the way up in the F-cycle (MultiGrid.hpp:153: 3+1)  */
    int prolong_mode;    /* pmg_prolong_mode                                                        */
    int engine;          /* pmg_engine                                                              */
    double smoother_eps; /* Smoother::epsilon (Smoother.hpp:11,84): absolute ||r|| early exit tested */
                         /* after every sweep.  0 disables it (parity runs, SURVEY 8c).  > 0 forces  */
                         /* the OPERATOR engine with a host readback per sweep.                      */
    int device;          /* CUDA ordinal, -1 = current device                                       */
    int use_graph;       /* 1: replay each cycle as a CUDA graph                                    */
    /* ---- multi-GPU (row-slab decomposition, one process per GPU); leave zeroed for 1 GPU ---- */
    int rank, n_ranks;
    int agglomerate_below; /* levels with n <= this are all-gathered and solved redundantly by every rank (513) */
    int norm_mode;       /* pmg_norm_mode: how the per-cycle residual norm is summed                */
    int smoother;        /* pmg_smoother (0 = weighted Jacobi)                                       */
    int smoother_fp32;   /* EXPERIMENT (SURVEY 8f-4): 1 = the Jacobi smoother computes in fp32 (fields, residual */
                         /* and grid transfers stay fp64; operator engine, one GPU).  Not parity: it shows  */
                         /* where an fp32 smoother stops converging.  0 = fp64 (default)                    */
    int reserved[5];
} pmg_config;

typedef struct pmg_solver pmg_solver; /* opaque */

/* ---- library ---------------------------------------------------------------------------------- */
const char *pmg_version(void);
/* message of the most recent failure on the calling thread ("" if none) */
const char *pmg_last_error(void);
const char *pmg_status_string(pmg_status s);
/* reference defaults: V(2,2), omega = 2/3 is NOT the reference default -- it has no omega; the
 * struct is filled with nu1=nu2=2, omega=1, gamma=3, n_coarse=5, coarse_sweeps=11, fmg_sweeps=4,
 * REFERENCE prolongation, FUSED engine, smoother_eps=0. */
void pmg_config_default(pmg_config *cfg, int n);
/* number of this library's kernels launched by the calling process so far (bench gpu_launches) */
unsigned long long pmg_kernel_launches(void);

/* ---- solver handle (replaces MultigridSolver / ParallelMultiGridSolver objects) ---------------- */
pmg_status pmg_create(const pmg_config *cfg, pmg_solver **out);
void pmg_destroy(pmg_solver *s);
/* f / phi: n*n doubles in the reference layout, in host or device memory */
pmg_status pmg_set_rhs(pmg_solver *s, const double *f, pmg_mem where);
/* phi == NULL: the zero start, same as pmg_zero_guess (nothing crosses PCIe) */
pmg_status pmg_set_guess(pmg_solver *s, const double *phi, pmg_mem where);
pmg_status pmg_get_solution(pmg_solver *s, double *phi, pmg_mem where);
/* Overlapped host transfers for a STREAM of problems on one hierarchy (the reference's runners solve one problem after
 * the other, MultiGridTestRunner.hpp:66-109): both PCIe directions run on copy streams of their own beside the solver.
 *   pmg_stage_rhs            starts copying the NEXT right-hand side (PINNED host memory, n x n or this rank's rows)
 *                            into a staging array and returns at once;
 *   pmg_commit_rhs           makes the staged array the solver's right-hand side (device-side wait + device copy;
 *                            with n_ranks > 1 also the halo exchange) -- call it before the solve that uses it;
 *   pmg_fetch_solution_begin snapshots the iterate on the device (so the next solve may overwrite it) and starts
 *                            copying the snapshot to PINNED host memory; returns at once;
 *   pmg_fetch_solution_wait  blocks until that copy has arrived (call it before the next _begin and before reading).
 * Typical loop:  stage(f0); for k: { commit(); stage(f_{k+1}); set_guess(NULL); solve(); fetch_wait(); fetch_begin(out_k); }
 * Costs two extra level-0 arrays and two device copies (1.4 ms each at N = 16385) per problem. */
pmg_status pmg_stage_rhs(pmg_solver *s, const double *f_host);
pmg_status pmg_commit_rhs(pmg_solver *s);
pmg_status pmg_fetch_solution_begin(pmg_solver *s, double *phi_host);
pmg_status pmg_fetch_solution_wait(pmg_solver *s);
/* phi = 0 (DynamicGridUtils::initialize_zeros, DynamicGridUtils.hpp:14-18) */
pmg_status pmg_zero_guess(pmg_solver *s);
/* f = 2 pi^2 sin(pi x) sin(pi y) generated on the device (DynamicGridUtils::compute_rhs, :111-124,
 * globals a=p=q=1); bit-identical to the host function */
pmg_status pmg_set_rhs_sine(pmg_solver *s);
/* ||f - A phi||_2, un-scaled, as MultiGridTestRunner.hpp:210-211 */
pmg_status pmg_residual_norm(pmg_solver *s, double *norm_out);
/* one cycle in place (MultiGridTestRunner.hpp:190-209; F = the runner's wrapper :192-205);
 * res_norm_out (nullable) receives ||f - A phi|| after the cycle */
pmg_status pmg_cycle(pmg_solver *s, pmg_cycle_kind kind, double *res_norm_out);
/* MultigridSolver::compute_coarsest_grid (MultiGrid.hpp:28-55): `fine` (n x n, the solver's size) restricted by repeated
 * full weighting down to the n_out x n_out level of the hierarchy (rings stay zero); the solver's iterate is untouched.
 * Single GPU. */
pmg_status pmg_restrict_to_level(pmg_solver *s, const double *fine, pmg_mem where_in, int n_out, double *out,
                                 pmg_mem where_out);
/* MultigridSolver::f_cycle(phi, f, N_init, h_init) (MultiGrid.hpp:138-183): nested iteration from the n_init x n_init
 * level -- starting iterate phi_init and right-hand side f_init, both n_init x n_init -- up to the solver's n: per level
 * fmg_sweeps sweeps, prolongation into a zeroed finer grid, the ANALYTIC right-hand side there (:162) and one V-cycle.
 * The result is the solver's iterate (the reference's `final_solution`: pmg_get_solution); the solver's own right-hand
 * side is untouched.  n_init == n copies phi_init (the while loop never runs).  res_norm_out nullable.  Single GPU. */
pmg_status pmg_f_cycle_from(pmg_solver *s, const double *phi_init, const double *f_init, int n_init, pmg_mem where,
                            double *res_norm_out);
/* cycles until ||r|| < rel_tol*||r0|| or max_cycles; res_history (nullable, max_cycles+1 doubles):
 * [0] = ||r0||, [k] = after cycle k; n_cycles_out (nullable) = cycles done.  The "residual-history
 * output" the reference computes and discards (MultiGridTestRunner.hpp:210-212). */
pmg_status pmg_solve(pmg_solver *s, pmg_cycle_kind kind, double rel_tol, int max_cycles,
                     double *res_history, int *n_cycles_out);
/* Conjugate gradients on A x = f from the current iterate, preconditioned by ONE multigrid cycle of this solver from a
 * zero start (precond = 1: the solver's V-cycle -- smoother, sweep counts, prolongation as configured; use
 * PMG_PROLONG_FULL, the reference prolongation is not the transpose of the restriction) or not at all (precond = 0: the
 * iteration of ConjugateGradientSmoother, Smoother.hpp:170-256, from the given start).  res_history (nullable,
 * max_iter + 1 doubles): [0] = ||r0||, [k] = ||r_k|| (recurrence residual); stops when ||r_k|| < rel_tol ||r0||.
 * On row slabs (n_ranks > 1, any rank count and any sweep counts nu1, nu2 = 1..4 the V-cycle accepts; with 3 or 4 sweeps
 * the preconditioner uses the deep-sweep slab schedule) every rank calls it with the same arguments and works on
 * its own rows: the iterate it updates and f are this rank's slab, and every rank receives the same history and step
 * count (the dot products are summed per rank and then in rank order, so every rank stops at the same step).  Against
 * one GPU, whose sums are grouped differently, the step count is the same in the tested cases, the history agrees to
 * about 1e-10 relative and the iterate to about 1e-9 of its largest entry -- NOT bit for bit.  A peer-wait time-out
 * inside the preconditioner is PMG_ERR_COMM, as for the cycles.
 * SURVEY.md 8f-3: "CG as an outer Krylov wrapper preconditioned by one V-cycle". */
pmg_status pmg_pcg(pmg_solver *s, int precond, double rel_tol, int max_iter, double *res_history, int *n_iter_out);
/* device time of the last pmg_solve / pmg_cycle in milliseconds (CUDA events on the solver stream) */
pmg_status pmg_last_device_ms(pmg_solver *s, double *ms_out);
/* the CUDA stream (cudaStream_t) the solver launches on, for callers that time with their own events */
void *pmg_stream(pmg_solver *s);

/* ---- operator level (replaces class Parallel, Parallel_Method.cu:144-199, and the DynamicGridUtils
 *      helpers); DEVICE pointers, dense reference layout (pitch = width), synchronous on return like
 *      the reference wrappers.  `stream` is a cudaStream_t (NULL = default stream). ------------------ */
/* `sweeps` weighted-Jacobi sweeps in place on x; scratch: width*height doubles (nullable: allocated
 * and freed inside).  Parallel::ComputeJacobi(d_x,d_f,height,width,h,v) == sweeps = v+1, omega = 1,
 * but race-free (double buffered) unlike jacobi_kernel (Parallel_Method.cu:6-24). */
pmg_status pmg_jacobi(double *x, const double *f, int width, int height, double h, double omega,
                      int sweeps, double *scratch, void *stream);
/* `sweeps` Gauss-Seidel sweeps in place, GaussSeidelSmoother's update (Smoother.hpp:134-145): ordering 0 = lexicographic
 * (the reference's, bit-identical; one CTA walks the anti-diagonals), 1 = red-black (parallel) */
pmg_status pmg_gauss_seidel(double *x, const double *f, int width, int height, double h, int sweeps, int ordering,
                            void *stream);
/* r = f - A x on the interior (ring of r untouched); norm2_out (nullable, HOST pointer) = sum r^2 */
pmg_status pmg_residual(double *r, const double *x, const double *f, int width, int height, double h,
                        double *norm2_out, void *stream);
/* coarse interior = full weighting of fine (MultiGrid.hpp:187-205); coarse ring untouched */
pmg_status pmg_restrict_fw(const double *fine, double *coarse, int nf, int nc, void *stream);
/* fine += P coarse (MultiGrid.hpp:208-226) */
pmg_status pmg_prolong_add(const double *coarse, double *fine, int nc, int nf, int mode, void *stream);
/* sum (a[i] - b[i])^2 and sum b[i]^2 over l entries -> HOST doubles: the pieces of Smoother::smooth's `errors` output,
 * ||x - x_true|| / ||x_true|| (Smoother.hpp:92-98; DynamicGridUtils::compute_error + norm) */
pmg_status pmg_diff_norm2(const double *a, const double *b, size_t l, double *diff2_out, double *b2_out, void *stream);
/* sum v[i]^2 over l entries -> HOST double (DynamicGridUtils::norm squared, :21-27) */
pmg_status pmg_norm2(const double *v, size_t l, double *norm2_out, void *stream);

/* The operator-level calls keep a little per-device scratch between calls (reduction partials; for long pmg_jacobi
 * runs three padded copies of the field).  This frees it; the next call re-allocates. */
pmg_status pmg_release_scratch(void);

/* ---- memory helpers for callers without a CUDA toolchain ------------------------------------- */
pmg_status pmg_device_alloc(void **p, size_t bytes);
pmg_status pmg_device_free(void *p);
pmg_status pmg_host_alloc_pinned(void **p, size_t bytes);
pmg_status pmg_host_free_pinned(void *p);
pmg_status pmg_memcpy(void *dst, const void *src, size_t bytes, int dst_is_device, int src_is_device);
pmg_status pmg_device_synchronize(void);
int pmg_device_count(void);

/* ---- multi-GPU bootstrap (one process per GPU; ids travel over the caller's own channel, e.g.
 *      torch.distributed).  With n_ranks > 1 the solver partitions every fine level into row slabs; pmg_set_rhs /
 *      pmg_set_guess / pmg_get_solution then move THIS RANK'S rows [y0, y1) (pmg_partition_rows), (y1-y0) x n
 *      doubles.  Halo rows travel over NVLink peer memory (CUDA IPC) when every rank can map its neighbours,
 *      over NCCL send/recv otherwise (PMG_P2P=0 forces the latter).  V-, W-, F-cycles and the general-RHS FMG pass
 *      (PMG_CYCLE_FMG, also as the start of pmg_solve), 1 <= nu1, nu2 <= 4 (3 and 4 sweeps add a halo exchange of the
 *      coarse iterate on the way up, DESIGN.md section 6a -- checked on CPU models and by its kernels on one GPU, not yet
 *      run on several GPUs); results are bit-identical to one GPU (the F-cycle and
 *      the FMG pass need equally sized slabs: n_ranks a power of two).  pmg_pcg runs on slabs too, to a tolerance
 *      against one GPU (see there).
 *      Failure semantics: a rank that waits longer than PMG_P2P_TIMEOUT_S (environment, default 30 s of device wall time)
 *      for a neighbour's rows gives up, the finest level's iterate of that cycle is NOT committed, and the call -- and
 *      every later call on that handle -- returns PMG_ERR_COMM: the ranks' exchange epochs no longer agree, so the
 *      solver must be destroyed and re-created on every rank. ------------ */
#define PMG_COMM_ID_BYTES 128
pmg_status pmg_comm_unique_id(unsigned char id[PMG_COMM_ID_BYTES]);
/* must be called (collectively) before pmg_create with cfg.n_ranks > 1 */
pmg_status pmg_comm_init(const unsigned char id[PMG_COMM_ID_BYTES], int rank, int n_ranks, int device);
pmg_status pmg_comm_finalize(void);
/* rows [*y0, *y1) of an n-row level owned by `rank` (even-aligned splits); pure host arithmetic */
pmg_status pmg_partition_rows(int n, int n_ranks, int rank, int *y0, int *y1);

#ifdef __cplusplus
}
#endif
#endif /* PMG_H */
