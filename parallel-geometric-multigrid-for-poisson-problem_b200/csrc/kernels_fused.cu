// kernels_fused.cu -- temporally blocked, warp-streaming kernels: the PMG_ENGINE_FUSED engine.
//
// One multigrid level visit costs two passes over HBM instead of the reference's eight-plus:
//
//   Pass A  (k_down)  xb = S^nu1(x);  f_coarse = R(f - A xb)        reads x,f   writes xb, f_coarse
//                     = Smoother::smooth + compute_residual + restrict_full_weighting
//                       (MultiGrid.hpp:66-78)                         26 B / point  (18 if x == 0)
//   Pass B  (k_up)    x  = S^nu2(xb + P e_coarse) [, sum (f - A x)^2] reads xb,e,f  writes x
//                     = prolongation + Smoother::smooth (+ the runner's residual norm)
//                       (MultiGrid.hpp:86-89, MultiGridTestRunner.hpp:210-211)   26 B / point
//
// First visit of a coarse level (x == 0 on entry): Pass A's first sweep is pointwise in f (sweep_row_from_zero: no
// neighbours, no row of delay).  On whole levels larger than the L2 cache (fused_rebuild_xb) Pass A does not store xb
// (10 B / point) and Pass B rebuilds xb = S^nu1(0; f) from the f rows it reads anyway (18 B / point): 28 B instead of 44.
//
// Execution model (DESIGN.md section 4).  No shared memory, no block barriers: every WARP owns a
// strip of 128 columns (32 lanes x 4 consecutive columns, two 128-bit loads per lane per row per
// array) and streams down a chunk of rows.  All stages of the pass are pipelined over the rows in
// registers: sweep k finalises row j-k when input row j arrives, the residual follows one row behind
// the last sweep and the full-weighting stencil one row behind that.  Horizontal neighbours come from
// two warp shuffles per stage per row; vertical neighbours are the register window.  Strips overlap
// by HALO columns on each side (the temporally blocked stages eat one column per stage), chunks
// overlap by the pipeline depth in rows; overlapped data is re-read from L2, not HBM.  Rows are
// prefetched PF rows ahead, either into registers (RegFeed) or -- the default -- with cp.async into a
// per-warp shared-memory ring (SmemFeed: each lane's 16-byte pieces land in its own slots, so the ring
// is a private FIFO that needs no barrier; it also holds the delay line of f rows the later stages
// read, which is what frees enough registers for 4 CTAs per SM with nothing spilled).
//
// Arithmetic is the reference's, operation for operation and in its order (pmg_internal.h), with no
// FMA contraction: every value written is bit-identical to the CPU path.  Partial sums
// ((h^2 f + W) + E) + S are formed when a row arrives and completed with + N one row later, which is
// exactly the reference's left-to-right evaluation.
#include <cstdlib>
#include <cstring>

#define PMG_NEEDS_PEER_WAIT
#include "pmg_internal.h"

namespace pmg {

namespace {

// Tunables (template parameters of the kernels; `Variant` picks a combination at run time):
//   C     columns per lane (4: two 128-bit accesses per row per array, strip = 128; 2: one, strip = 64)
//   PF    rows prefetched ahead
//   MINB  CTAs per SM promised to the compiler (register budget = 65536 / (128*MINB))
//   SM    stage rows through shared memory with cp.async (true) or through registers (false)
constexpr int WARPS_PER_CTA = 4;

__host__ __device__ constexpr int halo_for(int stages) { return stages <= 4 ? 4 : 8; }

struct StripGeom {
    int n;           // GLOBAL points per side (columns of this slab; rows of the whole level)
    int ny;          // rows of this slab that the rank owns (== n on one GPU)
    int yoff;        // global row index of local row 0 (even; 0 on one GPU)
    int row_lo;      // the pass writes the iterate for local rows [row_lo, row_hi) (row_lo even).  One GPU:
    int row_hi;      //   [0, n).  Slabs: up to [-6, ny + 6) -- halo rows recomputed instead of exchanged -- or a
                     //   sub-range when interior and boundary rows are launched separately (comm overlap)
    int pitch;       // row pitch of x / xb / f (doubles)
    int n_strips;    // strips across
    int n_chunks;    // row chunks
    int chunk_rows;  // rows per chunk (even)
    int halo;        // strip overlap per side (multiple of 4)
    int stride;      // STRIP - 2*halo: columns owned per strip
};

template <int C>
struct Row {
    double v[C];
};

template <int C>
__device__ __forceinline__ Row<C> load_row(const double *__restrict__ p)
{
    // 128-bit read-only loads; p is 16*C/2-byte aligned by construction of the layout
    Row<C> r;
#pragma unroll
    for (int k = 0; k < C / 2; ++k) {
        const double2 a = __ldg(reinterpret_cast<const double2 *>(p) + k);
        r.v[2 * k] = a.x;
        r.v[2 * k + 1] = a.y;
    }
    return r;
}

template <int C>
__device__ __forceinline__ void store_row(double *__restrict__ p, const Row<C> &r)
{
#ifndef PMG_HOST_EMULATION
    if constexpr (C == 4) {
        // one 256-bit store per lane (sm_100: STG.E.ENL2.256): a warp writes 1 KB of a row with one instruction instead
        // of two half-sector ones; p is 32-byte aligned (columns per lane = 4, PADX and the pitch multiples of 4)
        asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(r.v[0]), "d"(r.v[1]), "d"(r.v[2]), "d"(r.v[3])
                     : "memory");
    } else
#endif
    {
#pragma unroll
        for (int k = 0; k < C / 2; ++k)
            reinterpret_cast<double2 *>(p)[k] = make_double2(r.v[2 * k], r.v[2 * k + 1]);
    }
}

// an owner lane's row: all C columns, or (the lane whose slot 0 is the last column, wide cross pass) the first one only.
// Both as predicated stores: a branch around each would cost more instructions in the row loop than the stores themselves.
template <int C>
__device__ __forceinline__ void store_owned(double *__restrict__ p, const Row<C> &r, bool all, bool first_only)
{
#ifndef PMG_HOST_EMULATION
    if constexpr (C == 4) {
        asm volatile("{\n\t.reg .pred pa, po;\n\tsetp.ne.b32 pa, %5, 0;\n\tsetp.ne.b32 po, %6, 0;\n\t"
                     "@pa st.global.v4.f64 [%0], {%1, %2, %3, %4};\n\t@po st.global.f64 [%0], %1;\n\t}"
                     ::"l"(p), "d"(r.v[0]), "d"(r.v[1]), "d"(r.v[2]), "d"(r.v[3]), "r"((int)all), "r"((int)first_only)
                     : "memory");
        return;
    }
#endif
    if (all)
        store_row<C>(p, r);
    else if (first_only)
        *p = r.v[0];
}

// coarse points of a lane (C / 2 of them): all, or the first one only
template <int NP>
__device__ __forceinline__ void store_coarse_owned(double *__restrict__ p, const double (&o)[NP], bool all, bool first_only)
{
#ifndef PMG_HOST_EMULATION
    if constexpr (NP == 2) {
        asm volatile("{\n\t.reg .pred pa, po;\n\tsetp.ne.b32 pa, %3, 0;\n\tsetp.ne.b32 po, %4, 0;\n\t"
                     "@pa st.global.v2.f64 [%0], {%1, %2};\n\t@po st.global.f64 [%0], %1;\n\t}"
                     ::"l"(p), "d"(o[0]), "d"(o[1]), "r"((int)all), "r"((int)first_only)
                     : "memory");
        return;
    }
#endif
    if (NP == 2 && all)
        *reinterpret_cast<double2 *>(p) = make_double2(o[0], o[NP - 1]);
    else if (NP == 1 ? all : first_only)
        *p = o[0];
}

template <int C>
__device__ __forceinline__ Row<C> zero_row()
{
    Row<C> r;
#pragma unroll
    for (int k = 0; k < C; ++k) r.v[k] = 0.0;
    return r;
}

// west / east neighbours of a lane's C columns
template <int C>
__device__ __forceinline__ void neighbours(const Row<C> &c, Row<C> &w, Row<C> &e)
{
    double from_left = __shfl_up_sync(0xffffffffu, c.v[C - 1], 1);
    double from_right = __shfl_down_sync(0xffffffffu, c.v[0], 1);
#pragma unroll
    for (int k = 0; k < C; ++k) {
        w.v[k] = (k == 0) ? from_left : c.v[k == 0 ? 0 : k - 1];
        e.v[k] = (k == C - 1) ? from_right : c.v[k == C - 1 ? k : k + 1];
    }
}

// fine += P e for one point: `sum` = the coarse values the point interpolates, unscaled (1, 2 or 4 of them); the weight
// 1 / 0.5 / 0.25 follows from the parities of the fine row and column and is applied inside the addition (exact)
__device__ __forceinline__ double add_correction(double fine, double sum, int odd_row, int odd_col)
{
    if (!odd_row && !odd_col) return dadd(fine, sum);
    return dfma_pow2((odd_row && odd_col) ? 0.25 : 0.5, sum, fine);
}

// One weighted-Jacobi stage of the row pipeline.  `cen[p]` = input row i-1 (p = parity of the step; the two
// slots ping-pong so that no register has to be copied at the loop back-edge), `part` = the partial sum
// ((h^2 f + W) + E) + S of row i-1.  Given input row i (`in`) and f of row i it returns the finished output
// row i-1 and advances the state to row i.
template <int C>
struct SweepStage {
    Row<C> cen[2], part;
    __device__ __forceinline__ void init()
    {
        cen[0] = zero_row<C>();
        cen[1] = zero_row<C>();
        part = zero_row<C>();
    }
    template <bool WEIGHTED>
    __device__ __forceinline__ Row<C> step(const int p, const Row<C> &in, const Row<C> &f_row, const JacobiCoef &c,
                                           bool out_row_interior, const bool (&col_interior)[C])
    {
        Row<C> out, w, e;
        const Row<C> &prev = cen[p];
#pragma unroll
        for (int k = 0; k < C; ++k) {
            const double sum = dadd(part.v[k], in.v[k]);
            double val = WEIGHTED ? dadd(dmul(c.om1, prev.v[k]), dmul(c.w4, sum)) : dmul(0.25, sum);
            out.v[k] = (out_row_interior && col_interior[k]) ? val : prev.v[k];
        }
        neighbours<C>(in, w, e);
#pragma unroll
        for (int k = 0; k < C; ++k)
            part.v[k] = dadd(dadd(dadd(dmul(c.h2, f_row.v[k]), w.v[k]), e.v[k]), prev.v[k]);
        cen[p ^ 1] = in;
        return out;
    }
    // The same stage on the wide cross-pass geometry (k_cross, 4 columns per lane): `h2f` = h^2 f of row i, formed once by
    // the feed.  Only slot 0 can hold a Dirichlet column, so slots 1-3 are frozen only with the whole row: keep0 = slot 0
    // keeps its value, keep_row = the whole output row does (a constant false where the row's parity rules it out).
    template <bool WEIGHTED>
    __device__ __forceinline__ Row<C> step_wide(const int p, const Row<C> &in, const Row<C> &h2f, const JacobiCoef &c,
                                                bool keep0, bool keep_row)
    {
        static_assert(C == 4, "wide geometry: 4 columns per lane");
        Row<C> out, w, e;
        const Row<C> &prev = cen[p];
#pragma unroll
        for (int k = 0; k < C; ++k) {
            const double sum = dadd(part.v[k], in.v[k]);
            double val = WEIGHTED ? dadd(dmul(c.om1, prev.v[k]), dmul(c.w4, sum)) : dmul(0.25, sum);
            out.v[k] = ((k == 0) ? keep0 : keep_row) ? prev.v[k] : val;
        }
        neighbours<C>(in, w, e);
#pragma unroll
        for (int k = 0; k < C; ++k) part.v[k] = dadd(dadd(dadd(h2f.v[k], w.v[k]), e.v[k]), prev.v[k]);
        cen[p ^ 1] = in;
        return out;
    }
};

// The first sweep from x == 0 (first visit of a coarse level), as a per-point expression of f: no shuffles, no state, no
// row of delay.  SweepStage::step with every input +0 evaluates, in the reference's order,
//   sum = ((((h^2 f + W) + E) + S) + N) with W = E = S = N = +0,   val = om1 * x + w4 * sum  (x = +0)  or  0.25 * sum.
// Adding +0 is exact and idempotent except that it turns -0 into +0, so the four additions are one: dadd(h^2 f, +0)
// (f = -0, or h^2 f underflowing to -0, must give +0 as in the reference).  dmul(om1, +0) is -0 when omega > 1 (om1 < 0)
// and +0 otherwise; it is kept because it decides the sign of a zero result: -0 + (w4 * sum) is -0 when w4 * sum
// underflows to -0, +0 + (-0) is +0.  omega = 1 is the unweighted 0.25 * sum.  Frozen points keep their input, +0.
template <bool WEIGHTED>
__device__ __forceinline__ double sweep_from_zero(double f, const JacobiCoef &c)
{
    const double sum = dadd(dmul(c.h2, f), 0.0);
    return WEIGHTED ? dadd(dmul(c.om1, 0.0), dmul(c.w4, sum)) : dmul(0.25, sum);
}

template <int C, bool WEIGHTED>
__device__ __forceinline__ Row<C> sweep_row_from_zero(const Row<C> &f_row, const JacobiCoef &c, bool row_interior,
                                                      const bool (&col_interior)[C])
{
    Row<C> out;
#pragma unroll
    for (int k = 0; k < C; ++k) out.v[k] = (row_interior && col_interior[k]) ? sweep_from_zero<WEIGHTED>(f_row.v[k], c) : 0.0;
    return out;
}

// Residual stage: same pipeline shape; returns r of row i-1 given x row i.
template <int C>
struct ResidualStage {
    Row<C> part;    // ((4x - W) - E) - S of row i-1
    Row<C> cen[2];  // x row i-1 (ping-pong on the step parity)
    __device__ __forceinline__ void init()
    {
        cen[0] = zero_row<C>();
        cen[1] = zero_row<C>();
        part = zero_row<C>();
    }
    __device__ __forceinline__ Row<C> step(const int p, const Row<C> &in, const Row<C> &f_prev, double inv_h2)
    {
        Row<C> r, w, e;
#pragma unroll
        for (int k = 0; k < C; ++k)
            r.v[k] = dsub(f_prev.v[k], dmul(inv_h2, dsub(part.v[k], in.v[k])));
        neighbours<C>(in, w, e);
#pragma unroll
        for (int k = 0; k < C; ++k)
            part.v[k] = dsub(dsub(dfma_pow2(4.0, in.v[k], -w.v[k]), e.v[k]), cen[p].v[k]);
        cen[p ^ 1] = in;
        return r;
    }
};

template <int C>
__device__ __forceinline__ void strip_setup(const StripGeom &g, int wid, int lane, int &col, int &r0, int &r1,
                                            bool &owner, bool (&col_interior)[C])
{
    int chunk = wid / g.n_strips;
    int strip = wid - chunk * g.n_strips;
    col = -g.halo + strip * g.stride + C * lane;
    r0 = g.row_lo + chunk * g.chunk_rows;
    r1 = min(r0 + g.chunk_rows, g.row_hi);
    int first_owner = g.halo / C;
    owner = (lane >= first_owner) && (lane < first_owner + g.stride / C);
#pragma unroll
    for (int k = 0; k < C; ++k) col_interior[k] = (col + k > 0) && (col + k < g.n - 1);
}

// ---------------------------------------------------------------------------------------------------
// Row feeds: how rows of x and f travel from HBM to the pipeline, and where the delay line of f rows
// (f of row j-d, needed by stage d) lives.
// ---------------------------------------------------------------------------------------------------
// Where a row comes from: this rank's slab, or -- for halo rows of a fused halo exchange -- the neighbour's HBM.
struct RowSource {
    const double *x_up, *x_dn, *f_up, *f_dn;  // already offset by this lane's column
    double *f_keep;
    int ny, pitch;
    __device__ __forceinline__ void init(const HaloPeers &hp, int col, int ny_, int pitch_)
    {
        x_up = hp.x_up ? hp.x_up + col : nullptr;
        x_dn = hp.x_dn ? hp.x_dn + col : nullptr;
        f_up = hp.f_up ? hp.f_up + col : nullptr;
        f_dn = hp.f_dn ? hp.f_dn + col : nullptr;
        f_keep = hp.f_keep ? hp.f_keep + col : nullptr;
        ny = ny_;
        pitch = pitch_;
    }
    __device__ __forceinline__ const double *x_row(const double *local, int row) const
    {
        if (row < 0 && x_up) return x_up + (ptrdiff_t)row * pitch;
        if (row >= ny && x_dn) return x_dn + (ptrdiff_t)(row - ny) * pitch;
        return local + (ptrdiff_t)row * pitch;
    }
    __device__ __forceinline__ const double *f_row(const double *local, int row) const
    {
        if (row < 0 && f_up) return f_up + (ptrdiff_t)row * pitch;
        if (row >= ny && f_dn) return f_dn + (ptrdiff_t)(row - ny) * pitch;
        return local + (ptrdiff_t)row * pitch;
    }
    // f halo rows fetched from a peer are kept locally for the later Pass B
    __device__ __forceinline__ bool keeps(int row) const
    {
        return f_keep != nullptr && ((row < 0 && f_up) || (row >= ny && f_dn));
    }
};

// PADY rows x C columns of this lane, peer memory -> local halo rows: all loads first (L1-bypassing), then the stores
template <int C>
__device__ __forceinline__ void copy_halo_rows(const double *__restrict__ src, double *__restrict__ dst, int pitch)
{
    double2 v[PADY][C / 2];
#pragma unroll
    for (int r = 0; r < PADY; ++r)
#pragma unroll
        for (int p = 0; p < C / 2; ++p) v[r][p] = __ldcg(reinterpret_cast<const double2 *>(src + (ptrdiff_t)r * pitch) + p);
#pragma unroll
    for (int r = 0; r < PADY; ++r)
#pragma unroll
        for (int p = 0; p < C / 2; ++p) reinterpret_cast<double2 *>(dst + (ptrdiff_t)r * pitch)[p] = v[r][p];
}

template <int C, int PF, int S, bool USE_X>
struct RegFeed {
    static constexpr int UNROLL = PF;  // slot index must be static: the row loop is unrolled by PF
    static constexpr int SMEM_PER_WARP = 0;
    Row<C> xbuf[PF], fbuf[PF], fq[S + 2];
    const double *x, *f;
    RowSource src;
    int pitch, last_row;
    __device__ __forceinline__ void init(const double *x_, const double *f_, int pitch_, int col, int j_start,
                                         int last_row_, int /*lane*/, int /*warp_in_cta*/, const HaloPeers &hp, int ny)
    {
        x = x_ + col;
        f = f_ + col;
        pitch = pitch_;
        last_row = last_row_;
        src.init(hp, col, ny, pitch_);
#pragma unroll
        for (int d = 0; d < PF; ++d) {
            xbuf[d] = USE_X ? load_row<C>(src.x_row(x, j_start + d)) : zero_row<C>();
            fbuf[d] = load_row<C>(src.f_row(f, j_start + d));
        }
#pragma unroll
        for (int d = 0; d < S + 2; ++d) fq[d] = zero_row<C>();
    }
    // start of the step whose input row is jj (u = unrolled slot index); returns x row jj
    __device__ __forceinline__ Row<C> begin(int u, int jj)
    {
        Row<C> cur = xbuf[u];
#pragma unroll
        for (int d = S + 1; d > 0; --d) fq[d] = fq[d - 1];
        fq[0] = fbuf[u];
        if (src.keeps(jj)) store_row<C>(src.f_keep + (ptrdiff_t)jj * pitch, fq[0]);
        int nr = min(jj + PF, last_row);
        if (USE_X) xbuf[u] = load_row<C>(src.x_row(x, nr));
        fbuf[u] = load_row<C>(src.f_row(f, nr));
        return cur;
    }
    __device__ __forceinline__ Row<C> f_row(int d) const { return fq[d]; }  // f of row jj - d
    __device__ __forceinline__ void end() {}
};

// The few PTX primitives the kernels use.  Under PMG_HOST_EMULATION (tests/cpp/emu/host_emulation.h: the kernel source
// run lane by lane on the CPU, test infrastructure only) they act on the emulated shared-memory array instead.
#ifdef PMG_HOST_EMULATION
#define g_dyn_smem emu_smem
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void *gptr) { std::memcpy(emu_smem + saddr, gptr, 16); }
__device__ __forceinline__ void cp_async_commit() {}
template <int N>
__device__ __forceinline__ void cp_async_wait() {}
__device__ __forceinline__ void lds_v2(uint32_t a, double &v0, double &v1)
{
    std::memcpy(&v0, emu_smem + a, 8);
    std::memcpy(&v1, emu_smem + a + 8, 8);
}
__device__ __forceinline__ void sts_zero_v2(uint32_t a) { std::memset(emu_smem + a, 0, 16); }
__device__ __forceinline__ void sts_v2(uint32_t a, double v0, double v1)
{
    std::memcpy(emu_smem + a, &v0, 8);
    std::memcpy(emu_smem + a + 8, &v1, 8);
}
__device__ __forceinline__ void publish_epoch(int *flag, int epoch) { *(volatile int *)flag = epoch; }
__device__ __forceinline__ void __threadfence_system() {}
__device__ __forceinline__ bool wait_flag(const int *flag, int epoch) { return *(const volatile int *)flag >= epoch; }
#else
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void *gptr)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(saddr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ void lds_v2(uint32_t a, double &v0, double &v1)
{
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];\n" : "=d"(v0), "=d"(v1) : "r"(a));
}
__device__ __forceinline__ void sts_zero_v2(uint32_t a)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %1};\n" ::"r"(a), "d"(0.0) : "memory");
}
__device__ __forceinline__ void sts_v2(uint32_t a, double v0, double v1)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};\n" ::"r"(a), "d"(v0), "d"(v1) : "memory");
}
__device__ __forceinline__ void publish_epoch(int *flag, int epoch)
{
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
}

extern __shared__ __align__(16) unsigned char g_dyn_smem[];
#endif

// GEN_F (cross-cycle pass on one GPU, analytic right-hand side): f(row, col) = fx[col] * sy[row] is not streamed from HBM
// but formed when the row is issued -- the same dmul(dmul(factor, sin_x), sin_y) k_rhs_separable wrote, so the same
// bits -- and stored into the same ring slot with st.shared.  The ring is lane-private: program order is enough.
// H2F: a second ring of NF slots, parallel to the f ring, holds h^2 f of the same rows, formed once per point (with GEN_F
// when the row is generated, otherwise when its cp.async has landed) instead of once per sweep stage that reads it.
template <int C, int PF, int S, bool USE_X, bool GEN_F = false, bool H2F = false>
struct SmemFeed {
    static constexpr int UNROLL = 2;
    static constexpr int NF = (PF + S + 2 <= 8) ? 8 : 16;            // f ring slots  (power of two >= PF + S + 2)
    static constexpr int NXR = (PF + 1 <= 4) ? 4 : 8;                // x ring slots  (power of two >= PF + 1)
    static constexpr int NX = USE_X ? NXR : 0;
    static constexpr int NH = H2F ? NF : 0;                          // h^2 f ring slots (slot i holds the row of f slot i)
    static constexpr int PLANES = C / 2;               // 16-byte pieces per lane per row
    static constexpr int ROW_BYTES = PLANES * 512;     // plane p of a row: 32 lanes x 16 B, conflict free
    static constexpr int SMEM_PER_WARP = (NF + NH + NX) * ROW_BYTES;
    static_assert(PF + S + 2 <= NF && PF + 1 <= NXR, "ring too small");
    uint32_t fbase, xbase;  // shared-window addresses of this lane's first piece in slot 0 (h^2 f ring: fbase + NF rows)
    const double *x, *f;
    RowSource src;
    int pitch, last_row, t;
    double h2;              // H2F
    double fx[C];           // GEN_F: fx of this lane's columns
    const double *sy;       // GEN_F: sy[row], rows [-PADY, ny + PADY)
    double sy_next;         // GEN_F: sy of the row the next issue() fills (rows are issued in order)
    // GEN_F: call before init().  fx addresses logical column 0 of a padded row, sy logical row 0.
    __device__ __forceinline__ void set_rhs_tables(const double *fx_, const double *sy_, int col)
    {
#pragma unroll
        for (int p = 0; p < PLANES; ++p) {
            const double2 a = __ldg(reinterpret_cast<const double2 *>(fx_ + col) + p);
            fx[2 * p] = a.x;
            fx[2 * p + 1] = a.y;
        }
        sy = sy_;
    }
    __device__ __forceinline__ void issue(int row, int slot_t)
    {
        uint32_t fa = fbase + (uint32_t)(slot_t & (NF - 1)) * ROW_BYTES;
        if constexpr (GEN_F) {
            // issued rows are consecutive (clamped at last_row): fetch sy one row ahead so no store waits for a load
            const double syr = sy_next;
            sy_next = __ldg(sy + min(row + 1, last_row));
#pragma unroll
            for (int p = 0; p < PLANES; ++p) {
                const double f0 = dmul(fx[2 * p], syr), f1 = dmul(fx[2 * p + 1], syr);
                sts_v2(fa + p * 512, f0, f1);
                if constexpr (H2F) sts_v2(fa + NF * ROW_BYTES + p * 512, dmul(h2, f0), dmul(h2, f1));
            }
        } else {
            const double *fr = src.f_row(f, row);
#pragma unroll
            for (int p = 0; p < PLANES; ++p) cp_async16(fa + p * 512, fr + 2 * p);
        }
        if (USE_X) {
            const double *xr = src.x_row(x, row);
            uint32_t xa = xbase + (uint32_t)(slot_t & (NXR - 1)) * ROW_BYTES;
#pragma unroll
            for (int p = 0; p < PLANES; ++p) cp_async16(xa + p * 512, xr + 2 * p);
        }
        cp_async_commit();
    }
    __device__ __forceinline__ static Row<C> lds_row(uint32_t a)
    {
        Row<C> r;
#pragma unroll
        for (int p = 0; p < PLANES; ++p) lds_v2(a + p * 512, r.v[2 * p], r.v[2 * p + 1]);
        return r;
    }
    __device__ __forceinline__ void init(const double *x_, const double *f_, int pitch_, int col, int j_start,
                                         int last_row_, int lane, int warp_in_cta, const HaloPeers &hp, int ny)
    {
        x = x_ + col;
        f = f_ + col;
        pitch = pitch_;
        last_row = last_row_;
        t = 0;
        src.init(hp, col, ny, pitch_);
        uint32_t base = (uint32_t)__cvta_generic_to_shared(g_dyn_smem) + warp_in_cta * SMEM_PER_WARP;
        // zero this lane's pieces (warm-up steps read slots that were never filled)
#pragma unroll
        for (int sl = 0; sl < NF + NH + NX; ++sl)
#pragma unroll
            for (int p = 0; p < PLANES; ++p) sts_zero_v2(base + sl * ROW_BYTES + p * 512 + lane * 16);
        fbase = base + lane * 16;
        xbase = base + (NF + NH) * ROW_BYTES + lane * 16;
        if constexpr (GEN_F) sy_next = __ldg(sy + j_start);
#pragma unroll
        for (int d = 0; d < PF; ++d) issue(j_start + d, d);
    }
    __device__ __forceinline__ Row<C> begin(int /*u*/, int jj)
    {
        cp_async_wait<PF - 1>();  // all but the newest PF-1 groups have landed => row jj is in its slot
        if (src.keeps(jj)) store_row<C>(src.f_keep + (ptrdiff_t)jj * pitch, lds_row(fbase + (uint32_t)(t & (NF - 1)) * ROW_BYTES));
        if constexpr (H2F && !GEN_F) {
            const uint32_t fa = fbase + (uint32_t)(t & (NF - 1)) * ROW_BYTES;
            const Row<C> fr = lds_row(fa);
#pragma unroll
            for (int p = 0; p < PLANES; ++p) sts_v2(fa + NF * ROW_BYTES + p * 512, dmul(h2, fr.v[2 * p]), dmul(h2, fr.v[2 * p + 1]));
        }
        Row<C> cur = USE_X ? lds_row(xbase + (uint32_t)(t & (NXR - 1)) * ROW_BYTES) : zero_row<C>();
        issue(min(jj + PF, last_row), t + PF);
        return cur;
    }
    __device__ __forceinline__ Row<C> f_row(int d) const
    {
        return lds_row(fbase + (uint32_t)((t - d) & (NF - 1)) * ROW_BYTES);
    }
    __device__ __forceinline__ Row<C> h2f_row(int d) const  // H2F: h^2 f of row jj - d
    {
        return lds_row(fbase + (uint32_t)(NF + ((t - d) & (NF - 1))) * ROW_BYTES);
    }
    __device__ __forceinline__ void end() { ++t; }
};

template <int C, int PF, int S, bool USE_X, bool SM>
struct FeedSelect {
    using type = RegFeed<C, PF, S, USE_X>;
};
template <int C, int PF, int S, bool USE_X>
struct FeedSelect<C, PF, S, USE_X, true> {
    using type = SmemFeed<C, PF, S, USE_X>;
};

// coarse rows of the prolongation (Pass B, the cross-cycle pass and Pass A's prolong-in form)
template <int C>
struct CoarseRow {
    double v[C / 2 + 1];  // coarse columns cc .. cc + C/2
};

template <int C>
__device__ __forceinline__ CoarseRow<C> load_coarse(const double *__restrict__ p)
{
    CoarseRow<C> r;
    if (C == 4) {
        const double2 t = __ldg(reinterpret_cast<const double2 *>(p));
        r.v[0] = t.x;
        r.v[1] = t.y;
    } else {
        r.v[0] = __ldg(p);
    }
    return r;
}

// ---------------------------------------------------------------------------------------------------
// Pass A.  S sweeps; RESID adds residual + full weighting into the coarse RHS; ZEROX: x == 0 on entry.
// ---------------------------------------------------------------------------------------------------
// PIN ("prolong in", one GPU, with ZEROX): the iterate on entry is P e_in -- the bilinear prolongation of a coarse iterate
// into a zeroed grid (nested iteration, MultiGrid.hpp:161-164) -- formed on the fly from the coarse rows instead of being
// written by a fill + a prolongation kernel and read back (8 + 18 + 8 B per point less).
// ZEROX without PIN: the first sweep is pointwise (sweep_row_from_zero) on the arriving f row, so the pipeline has S - 1
// stages of row delay instead of S and the chunk bounds shrink by one row at each end.
// NO_XB (one GPU, ZEROX): xb is not stored -- Pass B rebuilds it from f (k_up with REBUILD) -- and the pass only reads f
// and writes the coarse f.
template <int C, int PF, int MINB, bool SM, int S, bool ZEROX, bool RESID, bool WEIGHTED, bool PROLOGUE = false, bool PIN = false,
          bool NO_XB = false>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, MINB)
    k_down(const double *__restrict__ x, double *__restrict__ xo, const double *__restrict__ f,
           double *__restrict__ cf, StripGeom g, int pitch_c, int nc, JacobiCoef coef, double inv_h2,
           const int *__restrict__ done, HaloPeers hp, const double *__restrict__ e_in, int pitch_e, int lo)
{
    static_assert(!PIN || (ZEROX && SM), "prolong-in: the iterate is not read, shared-memory feed (row pairs)");
    static_assert(!NO_XB || (ZEROX && RESID && !PIN), "xb is rebuilt by Pass B only on a first visit");
    constexpr bool PW = ZEROX && !PIN;  // pointwise first sweep
    constexpr int SD = PW ? S - 1 : S;  // sweep stages with a row of delay
    using Feed = typename FeedSelect<C, PF, S, !ZEROX, SM>::type;
    pdl_wait();
    const bool pdl_early = gridDim.x <= 296u;  // at most two CTAs per SM: a latency-bound level (pmg_internal.h)
    if (pdl_early) pdl_trigger();
    if (done != nullptr && *done) return;  // device-side convergence control: the solve already stopped
    constexpr int NP = C / 2;  // coarse points per lane (fine columns v0, v2, ...)
    // broadcast from lane 0 so the compiler KNOWS the warp index (hence every loop bound below) is warp-uniform:
    // the row loop then needs no divergence guards around its shuffles
    const int wid = __shfl_sync(0xffffffffu, (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (wid >= g.n_strips * g.n_chunks) return;
    int col, r0, r1;
    bool owner, cin[C];
    strip_setup<C>(g, wid, lane, col, r0, r1, owner, cin);

    // Rows this chunk must finish: x_S on [r0, r1) and, for the coarse rows it owns (fine row 2jc inside
    // the chunk AND inside the slab), r on [2jc-1, 2jc+1], i.e. x_S two rows earlier and one row later.
    // (The pointwise first sweep needs no rows around the one it finishes: x_S row i depends on f rows i - SD .. i + SD.)
    const int lead = RESID ? 2 : 0;
    int j_start_ = min(r0, max(r0, 0) - lead) - SD;
    if (PIN) j_start_ -= (j_start_ & 1);  // even: the row parity of the prolongation is static in the unrolled body
    const int j_start = j_start_;
    const int j_end = max(r1 - 1, min(r1, g.ny) - 1 + (RESID ? 1 : 0)) + SD;  // inclusive

    SweepStage<C> st[S];
    ResidualStage<C> rs;
#pragma unroll
    for (int k = 0; k < S; ++k) st[k].init();
    rs.init();
    // full-weighting state per coarse point of this lane:
    //   south row 2jc-1: s_mid (centre value), s_cor = SW + SE;  centre row 2jc: c_mid, c_ew = E + W
    double s_mid[NP], s_cor[NP], c_mid[NP], c_ew[NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) s_mid[q] = s_cor[q] = c_mid[q] = c_ew[q] = 0.0;

    // fused halo exchange.  First, one thread of the launch tells the neighbours that MY boundary rows are final
    // (the kernels that produced them ran earlier on this stream) ...
    const int epoch = hp.epoch + (hp.epoch_base != nullptr ? *hp.epoch_base : 0);
    if ((hp.pub_up != nullptr || hp.pub_dn != nullptr) && blockIdx.x == 0 && threadIdx.x == 0) {
        __threadfence_system();
        if (hp.pub_up != nullptr) publish_epoch(hp.pub_up, epoch);
        if (hp.pub_dn != nullptr) publish_epoch(hp.pub_dn, epoch);
    }
    // ... then, before the first access to a neighbour's rows, wait until it has published them.
    HaloPeers feed_peers = hp;  // what the row feed sees
    if constexpr (!PROLOGUE) {
        // every warp waits; halo rows are streamed from the neighbour's memory in place by the row feed
        if (hp.flag_up != nullptr || hp.flag_dn != nullptr) {
            int ok = 1;
            if (lane == 0) {
                if (hp.flag_up != nullptr) ok = wait_flag(hp.flag_up, epoch) ? ok : 0;
                if (hp.flag_dn != nullptr) ok = wait_flag(hp.flag_dn, epoch) ? ok : 0;
            }
            ok = __shfl_sync(0xffffffffu, ok, 0);
            if (!ok) {
                if (lane == 0) {
                    *hp.err = 1;
                    if (hp.abort != nullptr) *hp.abort = 1;
                }
                return;
            }
        }
    } else {
        // HALO PROLOGUE (shared-memory feed only; opt-in, PMG_HALO_PROLOGUE=1).  Only the warps whose rows reach into
        // a neighbour's slab wait for its flag -- the others start at once and hide the flag latency -- and they copy
        // the PADY remote rows of their strip into the local halo rows with every load in flight at once (one NVLink
        // round trip instead of one per pipelined row step), then stream from local memory.  Each lane later reads
        // back exactly the 16-byte pieces it wrote itself (cp.async.cg, L2), so no barrier is needed.
        static_assert(!PROLOGUE || SM, "the register feed reads through the non-coherent path: no prologue");
        if (hp.flag_up != nullptr || hp.flag_dn != nullptr) {
            const bool need_up = hp.flag_up != nullptr && j_start < 0;
            const bool need_dn = hp.flag_dn != nullptr && j_end >= g.ny;
            if (need_up || need_dn) {
                int ok = 1;
                if (lane == 0) {
                    if (need_up) ok = wait_flag(hp.flag_up, epoch) ? ok : 0;
                    if (need_dn) ok = wait_flag(hp.flag_dn, epoch) ? ok : 0;
                }
                ok = __shfl_sync(0xffffffffu, ok, 0);
                if (!ok) {
                    if (lane == 0) {
                        *hp.err = 1;
                        if (hp.abort != nullptr) *hp.abort = 1;
                    }
                    return;
                }
                const ptrdiff_t up_off = (ptrdiff_t)col - (ptrdiff_t)PADY * g.pitch, dn_off = (ptrdiff_t)col + (ptrdiff_t)g.ny * g.pitch;
                if (need_up) {
                    if (!ZEROX && hp.x_up != nullptr) copy_halo_rows<C>(hp.x_up + up_off, hp.x_keep + up_off, g.pitch);
                    if (hp.f_up != nullptr) copy_halo_rows<C>(hp.f_up + up_off, hp.f_keep + up_off, g.pitch);
                }
                if (need_dn) {
                    if (!ZEROX && hp.x_dn != nullptr) copy_halo_rows<C>(hp.x_dn + col, hp.x_keep + dn_off, g.pitch);
                    if (hp.f_dn != nullptr) copy_halo_rows<C>(hp.f_dn + col, hp.f_keep + dn_off, g.pitch);
                }
            }
            feed_peers = HaloPeers{};
        }
    }
    Feed feed;
    feed.init(x, f, g.pitch, col, j_start, g.ny + PADY - 1, lane, threadIdx.x >> 5, feed_peers, g.ny);
    const int ycoarse = g.yoff >> 1;  // global coarse row of local coarse row 0

    // prolong-in: coarse rows ec = row jc, en = row jc+1, eb = prefetch of row jc+2 (as in Pass B)
    static_assert(!PIN || Feed::UNROLL % 2 == 0, "rows are processed in (even, odd) pairs");
    const int cc = col >> 1;
    const int nc_last_row = ((g.ny - 1) >> 1) + PADY;
    CoarseRow<C> ec, en, eb;
    bool cprol[C];
    if (PIN) {
#pragma unroll
        for (int k = 0; k < C; ++k) cprol[k] = (col + k >= lo) && (col + k <= g.n - 2);
        const int jc0 = j_start >> 1;
        ec = load_coarse<C>(e_in + (ptrdiff_t)jc0 * pitch_e + cc);
        ec.v[NP] = __shfl_down_sync(0xffffffffu, ec.v[0], 1);
        eb = load_coarse<C>(e_in + (ptrdiff_t)(jc0 + 1) * pitch_e + cc);
        en = ec;
    }

    for (int j = j_start; j <= j_end; j += Feed::UNROLL) {
#pragma unroll
        for (int u = 0; u < Feed::UNROLL; ++u) {
            const int jj = j + u;  // input row of this step (steps past j_end are harmless: stores are masked)
            Row<C> cur = feed.begin(u, jj);
            if (PIN) {  // cur (zero) += P e_in: row jj of the iterate the sweeps start from
                const bool rowp = (jj + g.yoff >= lo) && (jj + g.yoff <= g.n - 2);
                double corr[C];  // the coarse values each point interpolates, summed but not yet weighted
                if ((u & 1) == 0) {
                    en = eb;
                    en.v[NP] = __shfl_down_sync(0xffffffffu, eb.v[0], 1);
                    const int nr = min((jj >> 1) + 2, nc_last_row);
                    eb = load_coarse<C>(e_in + (ptrdiff_t)nr * pitch_e + cc);
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = ec.v[q];
                        corr[2 * q + 1] = dadd(ec.v[q], ec.v[q + 1]);
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = dadd(ec.v[q], en.v[q]);
                        corr[2 * q + 1] = dadd(dadd(dadd(ec.v[q], ec.v[q + 1]), en.v[q]), en.v[q + 1]);
                    }
                    ec = en;
                }
#pragma unroll
                for (int k = 0; k < C; ++k)
                    if (rowp && cprol[k]) cur.v[k] = add_correction(cur.v[k], corr[k], u & 1, k & 1);
            }
            // PW: cur = x_1 row jj, formed from f row jj alone
            if (PW)
                cur = sweep_row_from_zero<C, WEIGHTED>(feed.f_row(0), coef, jj + g.yoff > 0 && jj + g.yoff < g.n - 1, cin);
            // sweeps: stage k consumes row jj-k of its input and finishes row jj-k-1 of its output
#pragma unroll
            for (int k = 0; k < SD; ++k) {
                const int out_row = jj - k - 1 + g.yoff;  // global row
                cur = st[k].template step<WEIGHTED>(u & 1, cur, feed.f_row(k), coef, out_row > 0 && out_row < g.n - 1, cin);
            }
            // cur = x_S row jj - SD
            const int xrow = jj - SD;
            if (!NO_XB && owner && xrow >= r0 && xrow < r1) store_row<C>(xo + (ptrdiff_t)xrow * g.pitch + col, cur);
            if (RESID) {
                Row<C> r = rs.step(u & 1, cur, feed.f_row(SD + 1), inv_h2);  // r of row jj - SD - 1
                const int rrow = jj - SD - 1;
                double left = __shfl_up_sync(0xffffffffu, r.v[C - 1], 1);
                if (rrow & 1) {
                    // north row 2jc+1 of coarse row jc: finish the stencil
                    const int jc = (rrow - 1) >> 1;
                    const int ic = col >> 1;  // col is a multiple of C => exact
                    double o[NP];
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        double west = (q == 0) ? left : r.v[q == 0 ? 0 : 2 * q - 1];
                        double edge = dadd(dadd(c_ew[q], r.v[2 * q]), s_mid[q]);
                        double corner = dadd(dadd(s_cor[q], west), r.v[2 * q + 1]);
                        double val = dfma_pow2(0.0625, corner, dfma_pow2(0.125, edge, dmul(0.25, c_mid[q])));
                        o[q] = (ic + q >= 1 && ic + q < nc - 1) ? val : 0.0;
                        // this row is also the south row of coarse row jc+1
                        s_mid[q] = r.v[2 * q];
                        s_cor[q] = dadd(west, r.v[2 * q + 1]);
                    }
                    // stored by the chunk and the rank that own fine row 2jc; coarse ring rows stay zero
                    if (owner && jc + ycoarse >= 1 && jc + ycoarse < nc - 1 && 2 * jc >= r0 && 2 * jc < r1 &&
                        jc >= 0 && 2 * jc < g.ny) {
                        double *dst = cf + (ptrdiff_t)jc * pitch_c + ic;
                        if (NP == 2)
                            *reinterpret_cast<double2 *>(dst) = make_double2(o[0], o[NP - 1]);
                        else
                            *dst = o[0];
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        double west = (q == 0) ? left : r.v[q == 0 ? 0 : 2 * q - 1];
                        c_mid[q] = r.v[2 * q];
                        c_ew[q] = dadd(r.v[2 * q + 1], west);  // E + W (MultiGrid.hpp:200: idx+1 first, then idx-1)
                    }
                }
            }
            feed.end();
        }
    }
    if (!pdl_early) pdl_trigger();
    cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------
// Pass B.  x = S^nu2(xb + P e) ; NORM adds sum over the interior of (f - A x)^2 (one partial per warp).
// PROLONG = false makes it a plain smoothing (+norm) pass.
// REBUILD = nu1 > 0 (one GPU, first visit, Pass A ran with NO_XB): xb = S^nu1(0; f) is not read but rebuilt from f ahead of
// the prolongation -- a pointwise sweep (sweep_row_from_zero) and nu1 - 1 sweep stages -- so the pass reads f and e and
// writes x: 18 B/point, and Pass A drops its 8 B/point xb store.
// ---------------------------------------------------------------------------------------------------
template <int C, int PF, int MINB, bool SM, int S, bool PROLONG, bool NORM, bool WEIGHTED, int REBUILD = 0>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, MINB)
    k_up(const double *__restrict__ xb, double *__restrict__ xo, const double *__restrict__ f,
         const double *__restrict__ e, StripGeom g, int pitch_c, int lo, JacobiCoef coef, double inv_h2,
         double *__restrict__ partials, const int *__restrict__ done)
{
    constexpr int D1 = REBUILD > 0 ? REBUILD - 1 : 0;  // rebuild sweep stages with a row of delay
    using Feed = typename FeedSelect<C, PF, S + D1, REBUILD == 0, SM>::type;
    pdl_wait();
    const bool pdl_early = gridDim.x <= 296u;  // at most two CTAs per SM: a latency-bound level (pmg_internal.h)
    if (pdl_early) pdl_trigger();
    if (done != nullptr && *done) return;
    static_assert(Feed::UNROLL % 2 == 0, "rows are processed in (even, odd) pairs");
    constexpr int NP = C / 2;
    // broadcast from lane 0 so the compiler KNOWS the warp index (hence every loop bound below) is warp-uniform:
    // the row loop then needs no divergence guards around its shuffles
    const int wid = __shfl_sync(0xffffffffu, (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (wid >= g.n_strips * g.n_chunks) return;
    int col, r0, r1;
    bool owner, cin[C];
    strip_setup<C>(g, wid, lane, col, r0, r1, owner, cin);

    // r0 is even; start on an even row so that row parity is static inside the unrolled body.  jj (below) is the row of xb
    // that enters the prolongation; with REBUILD the feed delivers f row jj + D1 and xb row jj leaves the rebuild stages.
    // xb row i is exact once the feed started at row i - D1 or earlier, or at a row <= 1: rows <= 0 are Dirichlet or padding
    // rows, zero in every sweep, so the zeroed stage state is then exact.  (Hence the clamp, which keeps the feed inside
    // the PADY padding rows: the rebuild runs on whole levels only.)
    int j_start = r0 - S - (NORM ? 1 : 0) - 2 * D1;
    if (REBUILD > 0) j_start = max(j_start, -PADY - D1);
    j_start -= (j_start & 1);
    if (REBUILD > 0 && j_start + D1 < -PADY) j_start += 2;  // a clamped start: the feed's first row is still <= 1
    const int j_end = r1 - 1 + S + (NORM ? 1 : 0);

    SweepStage<C> pre[D1 > 0 ? D1 : 1];
#pragma unroll
    for (int k = 0; k < D1; ++k) pre[k].init();
    SweepStage<C> st[S];
    ResidualStage<C> rs;
#pragma unroll
    for (int k = 0; k < S; ++k) st[k].init();
    rs.init();
    double acc = 0.0;

    bool cprol[C];  // columns that receive a correction
#pragma unroll
    for (int k = 0; k < C; ++k) cprol[k] = (col + k >= lo) && (col + k <= g.n - 2);

    Feed feed;
    feed.init(xb, f, g.pitch, col, j_start + D1, g.ny + PADY - 1, lane, threadIdx.x >> 5, HaloPeers{}, g.ny);

    // coarse rows: ec = row jc, en = row jc+1, eb = prefetch of row jc+2 (raw, before the shuffle)
    const int cc = col >> 1;
    const int nc_last_row = ((g.ny - 1) >> 1) + PADY;  // last local coarse row in the allocation
    CoarseRow<C> ec, en, eb;
#pragma unroll
    for (int q = 0; q <= NP; ++q) ec.v[q] = en.v[q] = eb.v[q] = 0.0;
    if (PROLONG) {
        const int jc0 = j_start >> 1;  // j_start even (possibly negative: arithmetic shift == floor)
        ec = load_coarse<C>(e + (ptrdiff_t)jc0 * pitch_c + cc);
        ec.v[NP] = __shfl_down_sync(0xffffffffu, ec.v[0], 1);
        eb = load_coarse<C>(e + (ptrdiff_t)(jc0 + 1) * pitch_c + cc);
    }

    for (int j = j_start; j <= j_end; j += Feed::UNROLL) {
#pragma unroll
        for (int u = 0; u < Feed::UNROLL; ++u) {
            const int jj = j + u;  // u even: fine row 2jc, u odd: fine row 2jc+1
            Row<C> cur = feed.begin(u, jj + D1);
            if (REBUILD > 0) {  // cur = xb row jj: the pointwise first sweep on f row jj + D1, then D1 sweep stages
                cur = sweep_row_from_zero<C, WEIGHTED>(feed.f_row(0), coef, jj + D1 + g.yoff > 0 && jj + D1 + g.yoff < g.n - 1, cin);
#pragma unroll
                for (int k = 0; k < D1; ++k) {
                    const int out_row = jj + D1 - k - 1 + g.yoff;
                    cur = pre[k].template step<WEIGHTED>(u & 1, cur, feed.f_row(k), coef, out_row > 0 && out_row < g.n - 1, cin);
                }
            }
            if (PROLONG) {
                const bool rowp = (jj + g.yoff >= lo) && (jj + g.yoff <= g.n - 2);
                double corr[C];  // the coarse values each point interpolates, summed but not yet weighted
                if ((u & 1) == 0) {
                    // coarse row jc+1 arrives (loaded one pair ago); fetch jc+2 for the next pair
                    en = eb;
                    en.v[NP] = __shfl_down_sync(0xffffffffu, eb.v[0], 1);
                    int nr = min((jj >> 1) + 2, nc_last_row);
                    eb = load_coarse<C>(e + (ptrdiff_t)nr * pitch_c + cc);
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = ec.v[q];
                        corr[2 * q + 1] = dadd(ec.v[q], ec.v[q + 1]);
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = dadd(ec.v[q], en.v[q]);
                        corr[2 * q + 1] = dadd(dadd(dadd(ec.v[q], ec.v[q + 1]), en.v[q]), en.v[q + 1]);
                    }
                    ec = en;
                }
#pragma unroll
                for (int k = 0; k < C; ++k)
                    if (rowp && cprol[k]) cur.v[k] = add_correction(cur.v[k], corr[k], u & 1, k & 1);
            }
#pragma unroll
            for (int k = 0; k < S; ++k) {
                const int out_row = jj - k - 1 + g.yoff;
                cur = st[k].template step<WEIGHTED>(u & 1, cur, feed.f_row(D1 + k), coef, out_row > 0 && out_row < g.n - 1, cin);
            }
            const int xrow = jj - S;
            if (owner && xrow >= r0 && xrow < r1) store_row<C>(xo + (ptrdiff_t)xrow * g.pitch + col, cur);
            if (NORM) {
                Row<C> r = rs.step(u & 1, cur, feed.f_row(D1 + S + 1), inv_h2);
                const int rrow = jj - S - 1;
                if (owner && rrow >= r0 && rrow < r1 && rrow >= 0 && rrow < g.ny && rrow + g.yoff > 0 &&
                    rrow + g.yoff < g.n - 1) {
#pragma unroll
                    for (int k = 0; k < C; ++k)
                        if (cin[k]) acc = dadd(acc, dmul(r.v[k], r.v[k]));
                }
            }
            feed.end();
        }
    }
    if (!pdl_early) pdl_trigger();
    cp_async_wait<0>();
    if (NORM) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc = dadd(acc, __shfl_xor_sync(0xffffffffu, acc, o));
        if (lane == 0) partials[wid] = acc;
    }
}

// ---------------------------------------------------------------------------------------------------
// Cross-cycle pass (level 0 of a V-cycle solve): Pass B of cycle k and Pass A of cycle k+1 in ONE sweep over HBM.
//   x_k      = S^nu2(xb_k + P e_k)                            -> xk   (write-only: the pipeline keeps using its registers)
//   norm_k   = sum over the interior of (f - A x_k)^2        -> partials (the history entry of cycle k)
//   xb_{k+1} = S^nu1(x_k)                                    -> xo   (an array other than xb)
//   f_coarse = R(f - A xb_{k+1})                             -> cf
// Two back-to-back passes over the same array read xb, e, f and write x, then read x, f and write xb, cf: 52 B/point.
// Fused, x_k is never read back: 8 (xb) + 8 (f) + 2 (e) + 8 (xb') + 2 (cf) = 28 B/point, plus 8 when x_k is written.
//   * xk == nullptr (one GPU): x_k stays in the registers.  The solve keeps the INPUT array of the last pass that ran, and
//     when the device-side control reports "cycle k converged", xb_k and e_k are both intact (everything queued after
//     `done` returns at once): one ordinary Pass B produces the iterate.  A B200 under its 1 kW cap is ENERGY-bound in
//     this solve, so the 8 B/point matter: 3.31 -> 3.04 ms per cycle at N = 16385 without the store, 3.31 with it.
//   * xk != nullptr (row slabs): the coarse levels of the next cycle run before the norm of this one is known, so e_k does
//     not survive; x_k is written every cycle instead (the pass of the next cycle honours `done` and leaves it alone).
// Same arithmetic, same order as the two passes: every value is bit-identical.  On row slabs (several GPUs) the input's halo rows -- 6 above, 4 below -- are copied from the
// neighbours' arrays in the halo prologue, exactly as Pass A does for the iterate.
//   * GEN_F (one GPU, f written by pmg_set_rhs_sine): f is not read; the row feed forms f = fx[col] * sy[row] from two
//     padded tables (SmemFeed), 20 B/point instead of 28.  Every stage of the row pipeline is the same code.
// ---------------------------------------------------------------------------------------------------
template <int C, int PF, int MINB, int S2, int S1, bool WEIGHTED, bool GEN_F = false>
__global__ void __launch_bounds__(32 * WARPS_PER_CTA, MINB)
    k_cross(const double *__restrict__ xb, double *__restrict__ xo, double *__restrict__ xk, const double *__restrict__ f,
            const double *__restrict__ e, double *__restrict__ cf, StripGeom g, int pitch_c, int lo, int nc, JacobiCoef coef,
            double inv_h2, double *__restrict__ partials, const int *__restrict__ done, HaloPeers hp,
            const double *__restrict__ rhs_fx, const double *__restrict__ rhs_sy)
{
    constexpr int S = S2 + S1;
    // WIDE: 4 columns per lane on strips of 128 columns that own 112 (halo 8), so col = -8 + 112 strip + 4 lane = 0 (mod 4);
    // every level has n = 2^k + 1 with n - 1 = 0 (mod 4) (launch_fused_cross takes a narrow shape for n = 3).  Hence the
    // Dirichlet columns 0 and n - 1 can only sit in slot 0 of a lane; slots 1-3 hold interior columns or padding.  The
    // wide pass freezes slot 0 only and lets the padding columns (and the padding rows of odd parity) compute values that
    // are never read by a domain point:
    //  * a sweep stage's output at a point depends on the input at that point and at its 4 neighbours, unless the point is
    //    frozen -- then it is its input.  Columns 0 and n - 1 are frozen in every stage, rows 0 and n - 1 (both even) in
    //    every stage whose output row is even.  A padding column's only domain neighbours are column 0 or n - 1, a padding
    //    row's only domain neighbours are row 0 or n - 1; by induction over the stages every domain value of every stage
    //    equals the value with zero padding.  The prolongation's corrections in padding slots are input to such columns.
    //  * residual: r at an interior point reads x at domain points only.  r at a boundary or padding point is read by the
    //    norm, which masks it per lane (nmask) and per row, and by the restriction only for coarse boundary or padding
    //    columns (coarse point ic reads fine columns 2ic - 1 .. 2ic + 1; for 1 <= ic <= nc - 2, including the west value
    //    shuffled from the lane to the left, that is [1, n - 2]; likewise rows).  Coarse columns 0 and nc - 1 = (n - 1) / 2
    //    are even, i.e. q = 0, and are still set to 0.
    //  * stores: owner lanes start at column 0; a lane beyond column n - 1 stores nothing, the lane at column n - 1 only
    //    slot 0 (coarse: q = 0).  So the padding of every output array stays zero in HBM (DESIGN section 3).
    constexpr bool WIDE = (C == 4);
    using Feed = SmemFeed<C, PF, S, true, GEN_F, WIDE>;
    pdl_wait();
    if (done != nullptr && *done) return;
    static_assert(Feed::UNROLL % 2 == 0, "rows are processed in (even, odd) pairs");
    constexpr int NP = C / 2;
    const int wid = __shfl_sync(0xffffffffu, (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (wid >= g.n_strips * g.n_chunks) return;
    int col, r0, r1;
    bool owner, cin[C];
    strip_setup<C>(g, wid, lane, col, r0, r1, owner, cin);
    const bool keep_c0 = !cin[0];                                 // WIDE: slot 0 is column 0, n - 1 or padding
    const bool st_all = owner && (!WIDE || col + C - 1 <= g.n - 1);  // the lane stores all its columns
    const bool st_one = WIDE && owner && col == g.n - 1;          // ... or only slot 0 (coarse: q = 0)
    bool nmask[C];                                                // the norm's columns
#pragma unroll
    for (int k = 0; k < C; ++k) nmask[k] = owner && cin[k];

    // rows this chunk must finish: xb' on [r0, r1) and, for the coarse rows it owns, r' on [2jc-1, 2jc+1]
    int j_start = min(r0, max(r0, 0) - 2) - S;
    j_start -= (j_start & 1);  // even, so that the row parity of the prolongation is static in the unrolled body
    const int j_end = max(r1 - 1, min(r1, g.ny)) + S;  // inclusive

    SweepStage<C> st[S];
    ResidualStage<C> rs_norm, rs;
#pragma unroll
    for (int k = 0; k < S; ++k) st[k].init();
    rs_norm.init();
    rs.init();
    double acc = 0.0;
    double s_mid[NP], s_cor[NP], c_mid[NP], c_ew[NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) s_mid[q] = s_cor[q] = c_mid[q] = c_ew[q] = 0.0;
    // columns that receive a correction.  WIDE: slot 2 holds columns 2 .. n - 3 or padding, slot 3 columns 3 .. n - 2 or
    // padding, so only slots 0 (columns 0, n - 1) and 1 (column 1, skipped by the reference prolongation) need the test
    bool cprol[C];
#pragma unroll
    for (int k = 0; k < C; ++k) cprol[k] = (WIDE && k >= 2) || ((col + k >= lo) && (col + k <= g.n - 2));

    // row slabs: tell the neighbours that my rows of the input array are final, then copy their boundary rows into my
    // halo rows (halo prologue: only the warps whose rows reach into a neighbour's slab wait for its flag)
    if (hp.flag_up != nullptr || hp.flag_dn != nullptr || hp.pub_up != nullptr || hp.pub_dn != nullptr) {
        const int epoch = hp.epoch + (hp.epoch_base != nullptr ? *hp.epoch_base : 0);
        if ((hp.pub_up != nullptr || hp.pub_dn != nullptr) && blockIdx.x == 0 && threadIdx.x == 0) {
            __threadfence_system();
            if (hp.pub_up != nullptr) publish_epoch(hp.pub_up, epoch);
            if (hp.pub_dn != nullptr) publish_epoch(hp.pub_dn, epoch);
        }
        const bool need_up = hp.flag_up != nullptr && j_start < 0;
        const bool need_dn = hp.flag_dn != nullptr && j_end >= g.ny;
        if (need_up || need_dn) {
            int ok = 1;
            if (lane == 0) {
                if (need_up) ok = wait_flag(hp.flag_up, epoch) ? ok : 0;
                if (need_dn) ok = wait_flag(hp.flag_dn, epoch) ? ok : 0;
            }
            ok = __shfl_sync(0xffffffffu, ok, 0);
            if (!ok) {
                if (lane == 0) {
                    *hp.err = 1;
                    if (hp.abort != nullptr) *hp.abort = 1;
                }
                return;
            }
            const ptrdiff_t up_off = (ptrdiff_t)col - (ptrdiff_t)PADY * g.pitch, dn_off = (ptrdiff_t)col + (ptrdiff_t)g.ny * g.pitch;
            if (need_up && hp.x_up != nullptr) copy_halo_rows<C>(hp.x_up + up_off, hp.x_keep + up_off, g.pitch);
            if (need_dn && hp.x_dn != nullptr) copy_halo_rows<C>(hp.x_dn + col, hp.x_keep + dn_off, g.pitch);
        }
    }
    Feed feed;
    feed.h2 = coef.h2;
    if constexpr (GEN_F) feed.set_rhs_tables(rhs_fx, rhs_sy, col);
    feed.init(xb, f, g.pitch, col, j_start, g.ny + PADY - 1, lane, threadIdx.x >> 5, HaloPeers{}, g.ny);

    const int cc = col >> 1;
    const int nc_last_row = ((g.ny - 1) >> 1) + PADY;
    // Coarse rows: ec = row jc, en = row jc+1, eq[i] = row jc+1+i on its way from HBM (raw, before the shuffle).  With the
    // wide strips only 2 warps per scheduler are resident and one row pair (~0.9 us of work) does not cover a loaded-DRAM
    // round trip: with a single row in flight 23 % of all warp samples sat on the shuffle that consumes it (ncu source
    // page), so the wide shape keeps three rows in flight.
    constexpr int CPF = (C == 4) ? 3 : 1;
    CoarseRow<C> ec, en, eq[CPF];
#pragma unroll
    for (int q = 0; q <= NP; ++q) ec.v[q] = en.v[q] = 0.0;
    {
        const int jc0 = j_start >> 1;
        ec = load_coarse<C>(e + (ptrdiff_t)jc0 * pitch_c + cc);
        ec.v[NP] = __shfl_down_sync(0xffffffffu, ec.v[0], 1);
#pragma unroll
        for (int i = 0; i < CPF; ++i) {
            eq[i].v[NP] = 0.0;
            eq[i] = load_coarse<C>(e + (ptrdiff_t)min(jc0 + 1 + i, nc_last_row) * pitch_c + cc);
        }
    }
    const int ycoarse = g.yoff >> 1;

    for (int j = j_start; j <= j_end; j += Feed::UNROLL) {
#pragma unroll
        for (int u = 0; u < Feed::UNROLL; ++u) {
            const int jj = j + u;  // u even: fine row 2jc, u odd: 2jc+1
            Row<C> cur = feed.begin(u, jj);
            {   // prolongation-and-add (MultiGrid.hpp:86)
                // an odd row below n - 1 is at most n - 2 (n is odd): odd rows need the lower bound only
                const bool rowp = (jj + g.yoff >= lo) && ((u & 1) != 0 || jj + g.yoff <= g.n - 2);
                double corr[C];  // the coarse values each point interpolates, summed but not yet weighted
                if ((u & 1) == 0) {
                    en = eq[0];
                    en.v[NP] = __shfl_down_sync(0xffffffffu, eq[0].v[0], 1);
#pragma unroll
                    for (int i = 0; i + 1 < CPF; ++i) eq[i] = eq[i + 1];
                    int nr = min((jj >> 1) + 1 + CPF, nc_last_row);
                    eq[CPF - 1] = load_coarse<C>(e + (ptrdiff_t)nr * pitch_c + cc);
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = ec.v[q];
                        corr[2 * q + 1] = dadd(ec.v[q], ec.v[q + 1]);
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        corr[2 * q] = dadd(ec.v[q], en.v[q]);
                        corr[2 * q + 1] = dadd(dadd(dadd(ec.v[q], ec.v[q + 1]), en.v[q]), en.v[q + 1]);
                    }
                    ec = en;
                }
#pragma unroll
                for (int k = 0; k < C; ++k)
                    if (rowp && cprol[k]) cur.v[k] = add_correction(cur.v[k], corr[k], u & 1, k & 1);
            }
            // stage k finishes x row jj-k-1
            auto sweep = [&](const int k, const Row<C> &in) -> Row<C> {
                const int out_row = jj - k - 1 + g.yoff;
                const bool interior_row = out_row > 0 && out_row < g.n - 1;
                if constexpr (WIDE) {
                    // rows 0 and n - 1 are even (yoff is even): only the stages whose output row is even can meet one
                    const bool keep_row = ((u + k + 1) & 1) == 0 && !interior_row;
                    return st[k].template step_wide<WEIGHTED>(u & 1, in, feed.h2f_row(k), coef, keep_c0 || keep_row, keep_row);
                } else {
                    return st[k].template step<WEIGHTED>(u & 1, in, feed.f_row(k), coef, interior_row, cin);
                }
            };
            // post-smoothing of cycle k (:89)
#pragma unroll
            for (int k = 0; k < S2; ++k) cur = sweep(k, cur);
            {   // cur = x_k row jj - S2: the iterate of cycle k, written for the case that cycle k is the last one
                const int krow = jj - S2;
                if (xk != nullptr) {
                    const bool row_ok = krow >= r0 && krow < r1;
                    store_owned<C>(xk + (ptrdiff_t)krow * g.pitch + col, cur, row_ok && st_all, row_ok && st_one);
                }
                // the runner's residual norm of cycle k (MultiGridTestRunner.hpp:210-211): r of x row jj - S2 - 1
                Row<C> r = rs_norm.step(u & 1, cur, feed.f_row(S2 + 1), inv_h2);
                const int rrow = jj - S2 - 1;
                // rows 0 and n - 1 are even: an odd row in [r0, r1) is an interior row
                if (rrow >= r0 && rrow < r1 && rrow >= 0 && rrow < g.ny &&
                    (((u + S2 + 1) & 1) != 0 || (rrow + g.yoff > 0 && rrow + g.yoff < g.n - 1))) {
#pragma unroll
                    for (int k = 0; k < C; ++k)
                        if (nmask[k]) acc = dadd(acc, dmul(r.v[k], r.v[k]));
                }
            }
            // pre-smoothing of cycle k+1 (:66)
#pragma unroll
            for (int k = S2; k < S; ++k) cur = sweep(k, cur);
            const int xrow = jj - S;
            const bool xrow_ok = xrow >= r0 && xrow < r1;
            store_owned<C>(xo + (ptrdiff_t)xrow * g.pitch + col, cur, xrow_ok && st_all, xrow_ok && st_one);
            {   // residual + full weighting of cycle k+1 (:69-78), as in k_down
                Row<C> r = rs.step(u & 1, cur, feed.f_row(S + 1), inv_h2);
                const int rrow = jj - S - 1;
                double left = __shfl_up_sync(0xffffffffu, r.v[C - 1], 1);
                if (((u + S + 1) & 1) != 0) {  // rrow odd (j is even)
                    const int jc = (rrow - 1) >> 1;
                    const int ic = col >> 1;
                    double o[NP];
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        double west = (q == 0) ? left : r.v[q == 0 ? 0 : 2 * q - 1];
                        double edge = dadd(dadd(c_ew[q], r.v[2 * q]), s_mid[q]);
                        double corner = dadd(dadd(s_cor[q], west), r.v[2 * q + 1]);
                        double val = dfma_pow2(0.0625, corner, dfma_pow2(0.125, edge, dmul(0.25, c_mid[q])));
                        // WIDE: q = 1 is an interior coarse column or padding that is not stored
                        o[q] = ((WIDE && q == 1) || (ic + q >= 1 && ic + q < nc - 1)) ? val : 0.0;
                        s_mid[q] = r.v[2 * q];
                        s_cor[q] = dadd(west, r.v[2 * q + 1]);
                    }
                    const bool jc_ok =
                        jc + ycoarse >= 1 && jc + ycoarse < nc - 1 && 2 * jc >= r0 && 2 * jc < r1 && jc >= 0 && 2 * jc < g.ny;
                    store_coarse_owned<NP>(cf + (ptrdiff_t)jc * pitch_c + ic, o, jc_ok && st_all, jc_ok && st_one);
                } else {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        double west = (q == 0) ? left : r.v[q == 0 ? 0 : 2 * q - 1];
                        c_mid[q] = r.v[2 * q];
                        c_ew[q] = dadd(r.v[2 * q + 1], west);
                    }
                }
            }
            feed.end();
        }
    }
    pdl_trigger();
    cp_async_wait<0>();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc = dadd(acc, __shfl_xor_sync(0xffffffffu, acc, o));
    if (lane == 0) partials[wid] = acc;
}

// ---- run-time variant table ---------------------------------------------------------------------
struct VariantDesc {
    int c, pf, minb, sm;
};
constexpr int NUM_VARIANTS = 5;
constexpr VariantDesc VARIANTS[NUM_VARIANTS] = {
    {2, 3, 4, 1},  // 0: shared-memory staged, 2 columns per lane, 16 warps/SM   (default for Pass A)
    {2, 3, 5, 1},  // 1: same, 20 warps/SM                                       (default for Pass B)
    {2, 4, 4, 0},  // 2: register staged, 2 columns per lane
    {2, 3, 6, 1},  // 3: shared-memory staged, 24 warps/SM
    {2, 7, 4, 1},  // 4: 7 rows in flight per warp (16 + 8 ring slots): for the LATENCY-bound small levels, where a
                   //    warp's whole chunk is a dozen rows and the pass time is (rows x load latency / depth)
};
// fused halo exchange with the halo prologue (see k_down); PMG_HALO_PROLOGUE=1, or fused_set_halo_prologue
int g_halo_prologue = PMG_HALO_PROLOGUE_DEFAULT;
// levels with n <= this use variant 4 (0 = never).  PMG_DEEP_PREFETCH_BELOW overrides.
int g_deep_prefetch_below = -1;
int deep_prefetch_below()
{
    if (g_deep_prefetch_below < 0) {
        const char *e = getenv("PMG_DEEP_PREFETCH_BELOW");
        g_deep_prefetch_below = e ? atoi(e) : PMG_DEEP_PREFETCH_DEFAULT;
        if (g_deep_prefetch_below < 0) g_deep_prefetch_below = 0;
    }
    return g_deep_prefetch_below;
}
// measured best per kernel flavour on B200 (tools/tune_fused.py): Pass A, Pass A from x == 0, Pass B, Pass B + norm
int g_variant_down = 0, g_variant_down_zero = 3, g_variant_up = 1, g_variant_up_norm = 3;

int g_fused_bad_nu = 0;  // last sweep count a launcher was asked for and could not serve (fused_take_bad_nu)

int g_min_chunk_rows = 4;  // even; the pipeline warm-up (4..8 rows) is paid once per chunk

int g_num_sms[64] = {0};  // per device ordinal
int num_sms()
{
#ifdef PMG_HOST_EMULATION
    return emu_num_sms;
#else
    int dev = 0;
    cudaGetDevice(&dev);
    int &v = g_num_sms[dev & 63];
    if (v == 0) {
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        if (v <= 0) v = 148;
    }
    return v;
#endif
}

StripGeom make_geom(const FusedLevel &lv, int stages, const VariantDesc &v, int ext_lo, int ext_hi, int halo = -1)
{
    const int n = lv.n;
    StripGeom g;
    g.n = n;
    g.ny = lv.ny > 0 ? lv.ny : n;
    g.yoff = lv.ny > 0 ? lv.yoff : 0;
    g.row_lo = -ext_lo;
    g.row_hi = g.ny + ext_hi;
    if (lv.span_hi > lv.span_lo) {  // explicit row range (interior / boundary split)
        g.row_lo = lv.span_lo;
        g.row_hi = lv.span_hi;
    }
    g.pitch = lv.pitch;
    g.halo = halo >= 0 ? halo : halo_for(stages);  // (an explicit halo must be a multiple of the columns per lane)
    g.stride = 32 * v.c - 2 * g.halo;
    g.n_strips = (n + g.stride - 1) / g.stride;
    // one resident wave: every warp of the grid is on an SM for the whole pass (no tail wave)
    int resident = num_sms() * v.minb * WARPS_PER_CTA;
    int chunks = resident / g.n_strips;
    if (chunks < 1) chunks = 1;
    const int span = g.row_hi - g.row_lo;  // rows the pass writes
    int rows = (span + chunks - 1) / chunks;
    rows += rows & 1;
    if (rows < g_min_chunk_rows) rows = g_min_chunk_rows;
    g.chunk_rows = rows;
    g.n_chunks = (span + rows - 1) / rows;
    return g;
}

inline int grid_for(const StripGeom &g)
{
    int warps = g.n_strips * g.n_chunks;
    return (warps + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
}

#ifdef PMG_HOST_EMULATION
template <typename K>
void set_smem(K, int) {}
#define PMG_LAUNCH(kernel, grid, block, smem, stream, ...) \
    emu_launch_warps((grid), (block), [&] { kernel(__VA_ARGS__); })
#else
template <typename K>
void set_smem(K kernel, int bytes)
{
    if (bytes > 0) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
#define PMG_LAUNCH(kernel, grid, block, smem, stream, ...) launch_pdl(kernel, (grid), (block), (smem), (stream), __VA_ARGS__)
#endif

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: set it once per (kernel, device ordinal),
// not once per process, so that a second solver on another GPU of the same process launches correctly
inline int current_device()
{
#ifdef PMG_HOST_EMULATION
    return 0;
#else
    int d = 0;
    cudaGetDevice(&d);
    return d & 63;
#endif
}
#define PMG_SMEM_ONCE(k, sm)                         \
    do {                                             \
        static unsigned long long mask_ = 0;         \
        const int d_ = current_device();             \
        if (!((mask_ >> d_) & 1ull)) {               \
            set_smem(k, sm);                         \
            mask_ |= 1ull << d_;                     \
        }                                            \
    } while (0)

template <int C, int PF, int MINB, bool SM, int S, bool WEIGHTED>
void down_launch_w(const FusedLevel &lv, double *cf, int pitch_c, bool x_is_zero, bool resid, bool store_xb, const StripGeom &g,
                   int nc, const JacobiCoef &c, double inv, dim3 grid, dim3 block, const int *done, cudaStream_t st)
{
    // the halo-prologue flavour exists for the headline sweep count on the shared-memory feed only
    constexpr bool CAN_PROLOGUE = SM && S == 2;
    const bool prologue = CAN_PROLOGUE && g_halo_prologue && (lv.hp.flag_up != nullptr || lv.hp.flag_dn != nullptr);
    if (resid && x_is_zero && prologue) {
        auto k = k_down<C, PF, MINB, SM, S, true, true, WEIGHTED, CAN_PROLOGUE>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, false, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    } else if (resid && prologue) {
        auto k = k_down<C, PF, MINB, SM, S, false, true, WEIGHTED, CAN_PROLOGUE>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, true, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    } else if (resid && x_is_zero && !store_xb) {
        auto k = k_down<C, PF, MINB, SM, S, true, true, WEIGHTED, false, false, true>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, false, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    } else if (resid && x_is_zero) {
        auto k = k_down<C, PF, MINB, SM, S, true, true, WEIGHTED>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, false, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    } else if (resid) {
        auto k = k_down<C, PF, MINB, SM, S, false, true, WEIGHTED>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, true, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    } else {
        auto k = k_down<C, PF, MINB, SM, S, false, false, WEIGHTED>;
        int sm = WARPS_PER_CTA * FeedSelect<C, PF, S, true, SM>::type::SMEM_PER_WARP;
        PMG_SMEM_ONCE(k, sm);
        PMG_LAUNCH(k, grid, block, sm, st, lv.x, lv.xb, lv.f, (double *)nullptr, g, 0, nc, c, inv, done, lv.hp, (const double *)nullptr, 0, 0);
    }
}

template <int C, int PF, int MINB, bool SM, int S>
void down_launch(const FusedLevel &lv, double *cf, int pitch_c, double omega, bool x_is_zero, bool resid, bool store_xb,
                 const int *done, cudaStream_t st)
{
    StripGeom g = make_geom(lv, S + (resid ? 2 : 0), VariantDesc{C, PF, MINB, SM}, lv.ext_lo, lv.ext_hi);
    JacobiCoef c = jacobi_coef(lv.h, omega);
    double inv = 1.0 / (lv.h * lv.h);
    int nc = (lv.n - 1) / 2 + 1;
    dim3 grid(grid_for(g)), block(32 * WARPS_PER_CTA);
    if (c.weighted) {
        down_launch_w<C, PF, MINB, SM, S, true>(lv, cf, pitch_c, x_is_zero, resid, store_xb, g, nc, c, inv, grid, block, done, st);
    } else {
        down_launch_w<C, PF, MINB, SM, S, false>(lv, cf, pitch_c, x_is_zero, resid, store_xb, g, nc, c, inv, grid, block, done, st);
    }
    count_launch();
}

// Pass A whose iterate on entry is P e_in (prolong-in form of k_down): headline sweep count, the x == 0 variant's shape
template <bool WEIGHTED>
void down_prolong_launch_w(const FusedLevel &lv, const double *e_in, int pitch_e, int lo, double *cf, int pitch_c,
                           const JacobiCoef &c, const int *done, cudaStream_t st)
{
    constexpr int C = 2, PF = 3, MINB = 5, S = 2;
    StripGeom g = make_geom(lv, S + 2, VariantDesc{C, PF, MINB, 1}, lv.ext_lo, lv.ext_hi);
    const double inv = 1.0 / (lv.h * lv.h);
    const int nc = (lv.n - 1) / 2 + 1;
    auto k = k_down<C, PF, MINB, true, S, true, true, WEIGHTED, false, true>;
    int sm = WARPS_PER_CTA * SmemFeed<C, PF, S, false>::SMEM_PER_WARP;
    PMG_SMEM_ONCE(k, sm);
    PMG_LAUNCH(k, dim3(grid_for(g)), dim3(32 * WARPS_PER_CTA), sm, st, lv.x, lv.xb, lv.f, cf, g, pitch_c, nc, c, inv, done,
               HaloPeers{}, e_in, pitch_e, lo);
}

template <int C, int PF, int MINB, bool SM, int S, bool PROLONG, bool NORM, bool WEIGHTED, int REBUILD = 0>
void up_launch_k(const FusedLevel &lv, const double *e, int pitch_c, const StripGeom &g, int lo,
                 const JacobiCoef &c, double inv, double *d_partials, const int *done, cudaStream_t st)
{
    auto k = k_up<C, PF, MINB, SM, S, PROLONG, NORM, WEIGHTED, REBUILD>;
    int sm = WARPS_PER_CTA * FeedSelect<C, PF, S + (REBUILD > 0 ? REBUILD - 1 : 0), REBUILD == 0, SM>::type::SMEM_PER_WARP;
    PMG_SMEM_ONCE(k, sm);
    PMG_LAUNCH(k, dim3(grid_for(g)), dim3(32 * WARPS_PER_CTA), sm, st, lv.xb, lv.x, lv.f, e, g, pitch_c, lo, c, inv, d_partials, done);
}

template <int C, int PF, int MINB, bool SM, int S, bool PROLONG, bool NORM>
void up_launch_one(const FusedLevel &lv, const double *e, int pitch_c, const StripGeom &g, int lo,
                   const JacobiCoef &c, double inv, double *d_partials, const int *done, cudaStream_t st)
{
    if (c.weighted)
        up_launch_k<C, PF, MINB, SM, S, PROLONG, NORM, true>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
    else
        up_launch_k<C, PF, MINB, SM, S, PROLONG, NORM, false>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
}

template <int C, int PF, int MINB, bool SM, int S>
void up_launch(const FusedLevel &lv, const double *e, int pitch_c, double omega, int lo, bool norm,
               double *d_partials, int *n_partials, const int *done, cudaStream_t st)
{
    StripGeom g = make_geom(lv, S + (norm ? 2 : 1), VariantDesc{C, PF, MINB, SM}, lv.ext_lo, lv.ext_hi);
    JacobiCoef c = jacobi_coef(lv.h, omega);
    double inv = 1.0 / (lv.h * lv.h);
    if (e != nullptr) {
        if (norm)
            up_launch_one<C, PF, MINB, SM, S, true, true>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
        else
            up_launch_one<C, PF, MINB, SM, S, true, false>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
    } else {
        if (norm)
            up_launch_one<C, PF, MINB, SM, S, false, true>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
        else
            up_launch_one<C, PF, MINB, SM, S, false, false>(lv, e, pitch_c, g, lo, c, inv, d_partials, done, st);
    }
    count_launch();
    if (n_partials) *n_partials = norm ? g.n_strips * g.n_chunks : 0;
}

// Pass B of a first visit that rebuilds xb = S^nu1(0; f) (k_up with REBUILD = nu1): prolongation, no norm, whole level.
// One shape per sweep count: the Pass B variant the solve uses by default.
template <int C, int PF, int MINB, bool SM, int S, int NU1>
void up_rebuild_launch(const FusedLevel &lv, const double *e, int pitch_c, double omega, int lo, const int *done, cudaStream_t st)
{
    StripGeom g = make_geom(lv, (NU1 - 1) + S + 1, VariantDesc{C, PF, MINB, SM}, lv.ext_lo, lv.ext_hi);
    JacobiCoef c = jacobi_coef(lv.h, omega);
    double inv = 1.0 / (lv.h * lv.h);
    if (c.weighted)
        up_launch_k<C, PF, MINB, SM, S, true, false, true, NU1>(lv, e, pitch_c, g, lo, c, inv, nullptr, done, st);
    else
        up_launch_k<C, PF, MINB, SM, S, true, false, false, NU1>(lv, e, pitch_c, g, lo, c, inv, nullptr, done, st);
    count_launch();
}

template <int C, int PF, int MINB, bool SM, int S>
void up_rebuild_dispatch(const FusedLevel &lv, const double *e, int pitch_c, double omega, int lo, int nu1, const int *done,
                         cudaStream_t st)
{
    switch (nu1) {
        case 1: up_rebuild_launch<C, PF, MINB, SM, S, 1>(lv, e, pitch_c, omega, lo, done, st); break;
        case 2: up_rebuild_launch<C, PF, MINB, SM, S, 2>(lv, e, pitch_c, omega, lo, done, st); break;
        case 3: up_rebuild_launch<C, PF, MINB, SM, S, 3>(lv, e, pitch_c, omega, lo, done, st); break;
        case 4: up_rebuild_launch<C, PF, MINB, SM, S, 4>(lv, e, pitch_c, omega, lo, done, st); break;
        default: break;
    }
}

// geometry of the cross-cycle pass: 4 sweeps + residual + restriction eat 6 columns per side
template <int C, int PF, int MINB, bool WEIGHTED, bool GEN_F = false>
void cross_launch_w(const FusedLevel &lv_in, double *xb_out, const double *e, int pitch_c, double *cf, int lo, double *d_partials,
                    int *n_partials, const JacobiCoef &c, const int *done, cudaStream_t st)
{
    // lv_in.xb = input (xb_k), lv_in.x = where x_k goes, lv_in.hp = the neighbours' copies of the input array (row slabs)
    VariantDesc v{C, PF, MINB, 1};
    // strips of 64 columns own 52 (19 % overlap instead of 25 % with a halo of 8); 4 columns per lane: 128 own 112
    StripGeom g = make_geom(lv_in, 6, v, 0, 0, C == 2 ? 6 : 8);
    double inv = 1.0 / (lv_in.h * lv_in.h);
    int nc = (lv_in.n - 1) / 2 + 1;
    auto k = k_cross<C, PF, MINB, 2, 2, WEIGHTED, GEN_F>;
    int sm = WARPS_PER_CTA * SmemFeed<C, PF, 4, true, GEN_F, C == 4>::SMEM_PER_WARP;
    PMG_SMEM_ONCE(k, sm);
    PMG_LAUNCH(k, dim3(grid_for(g)), dim3(32 * WARPS_PER_CTA), sm, st, lv_in.xb, xb_out, lv_in.x, lv_in.f, e, cf, g, pitch_c, lo, nc, c,
               inv, d_partials, done, lv_in.hp, lv_in.rhs_fx, lv_in.rhs_sy);
    if (n_partials) *n_partials = g.n_strips * g.n_chunks;
}

}  // namespace

bool fused_supported(int nu) { return nu >= 1 && nu <= 4; }
int fused_take_bad_nu()
{
    int v = g_fused_bad_nu;
    g_fused_bad_nu = 0;
    return v;
}

// Cross-cycle pass on a level or a row slab of it: reads lv.xb (= xb_k), coarse_x (= e_k), lv.f; writes lv.x (= x_k), xb_out
// (= xb_{k+1}, an array other than lv.xb), coarse_f and the norm partials of x_k.  nu1 = nu2 = 2 only.
// Shape of the cross-cycle pass.  2 (default): 4 columns per lane -- strips of 128 columns own 112 --, 2 CTAs of 4 warps
// per SM with up to 255 registers: a quarter fewer instructions per point than the narrow shape (half the shuffles and
// row bookkeeping per point, 12.5 % instead of 19 % halo columns) and 11 % faster at N = 16385 although only 8 warps per SM
// are resident.  3 .. 6: 2 columns per lane with that many CTAs per SM (4 was the default before; 5 and 6 spill).
// 7: the wide shape with one more row of prefetch.  (12 wide warps per SM -- 168 registers -- spill and are 1.5x slower;
// the two-pass kernels, which are bandwidth- and not instruction-bound, are SLOWER with wide strips: 3.2-3.9 TB/s.)
constexpr int PMG_CROSS_SHAPE_DEFAULT = 2;
int g_cross_minb = PMG_CROSS_SHAPE_DEFAULT;
bool fused_cross_supported(int nu1, int nu2) { return nu1 == 2 && nu2 == 2; }
// Fraction of the resident warp slots the cross-cycle pass fills on an n-column level of `rows` rows.  The grid is one
// resident wave of (strips x chunks) warps with chunks = floor(slots / strips): at n = 32769 the 631 strips of 52 columns
// leave 3 chunks = 80 % of the slots (the two-pass kernels' 586 strips of 56 columns give 4 chunks = 99 %), and the pass
// is then SLOWER than the two passes it replaces (8 GPUs, N = 32769: 1.81 -> 1.86 ms per cycle).  The solve uses it only
// above 0.9.
double fused_cross_utilisation(int n, int rows)
{
    FusedLevel lv{};
    lv.n = n;
    lv.ny = rows;
    lv.pitch = level_pitch(n);
    const bool wide = g_cross_minb == 2 || g_cross_minb == 7;
    VariantDesc v{wide ? 4 : 2, 2, wide ? 2 : g_cross_minb, 1};
    StripGeom g = make_geom(lv, 6, v, 0, 0, wide ? 8 : 6);
    return (double)(g.n_strips * g.n_chunks) / (double)(num_sms() * v.minb * WARPS_PER_CTA);
}
void fused_set_cross_minb(int m) { g_cross_minb = (m >= 2 && m <= 7) ? m : PMG_CROSS_SHAPE_DEFAULT; }
void launch_fused_cross(const FusedLevel &lv, double *xb_out, const double *coarse_x, double *coarse_f, int pitch_c, double omega,
                        int prolong_mode, double *d_partials, int *n_partials, cudaStream_t st, const int *done)
{
    const int lo = prolong_mode == PMG_PROLONG_FULL ? 1 : 2;
    JacobiCoef c = jacobi_coef(lv.h, omega);
    // f from the tables: one GPU only (a slab's halo rows of f are not generated), and only when the caller passed them
    const bool gen_f = lv.rhs_fx != nullptr && lv.rhs_sy != nullptr && lv.ny == 0;
#define PMG_CROSS(MINB)                                                                                                        \
    do {                                                                                                                       \
        if (c.weighted)                                                                                                        \
            cross_launch_w<2, 2, MINB, true>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st);  \
        else                                                                                                                   \
            cross_launch_w<2, 2, MINB, false>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st); \
    } while (0)
    if (g_cross_minb == 4)
        PMG_CROSS(4);
    else if ((g_cross_minb == 2 || g_cross_minb == 7) && (lv.n - 1) % 4 == 0) {
        // 4 columns per lane, 8 warps per SM; 7 = one more row of prefetch.  The wide kernel freezes the Dirichlet columns in
        // slot 0 only, which needs n - 1 = 0 (mod 4): every level but n = 3, which takes the narrow shape below
#define PMG_CROSS4(PF)                                                                                                         \
    do {                                                                                                                       \
        if (c.weighted)                                                                                                        \
            cross_launch_w<4, PF, 2, true>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st);   \
        else                                                                                                                   \
            cross_launch_w<4, PF, 2, false>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st);  \
    } while (0)
        if (g_cross_minb == 2 && gen_f) {  // the default shape alone has the generated-f flavour
            if (c.weighted)
                cross_launch_w<4, 2, 2, true, true>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st);
            else
                cross_launch_w<4, 2, 2, false, true>(lv, xb_out, coarse_x, pitch_c, coarse_f, lo, d_partials, n_partials, c, done, st);
        } else if (g_cross_minb == 2)
            PMG_CROSS4(2);
        else
            PMG_CROSS4(3);
#undef PMG_CROSS4
    }
    else if (g_cross_minb == 5)
        PMG_CROSS(5);
    else if (g_cross_minb == 6)
        PMG_CROSS(6);
    else
        PMG_CROSS(3);
#undef PMG_CROSS
    count_launch();
}

int fused_num_variants() { return NUM_VARIANTS; }
void fused_set_variant(int v)
{
    // bit 16 clear: one variant for both passes; set: low byte = Pass A variant, next byte = Pass B variant
    int d = v & 0xff, u = (v >> 8) & 0xff;
    if (!(v & 0x10000)) u = d;
    g_variant_down = g_variant_down_zero = (d >= 0 && d < NUM_VARIANTS) ? d : 0;
    g_variant_up = g_variant_up_norm = (u >= 0 && u < NUM_VARIANTS) ? u : 0;
    if (v < 0) {  // restore the per-kernel defaults
        g_variant_down = 0;
        g_variant_down_zero = 3;
        g_variant_up = 1;
        g_variant_up_norm = 3;
    }
}
int fused_get_variant() { return g_variant_down | (g_variant_up << 8); }
void fused_set_min_chunk_rows(int r) { g_min_chunk_rows = (r >= 2) ? (r + (r & 1)) : 2; }

int g_rebuild_xb = -2;  // -2: not yet read from PMG_REBUILD_XB
void fused_set_rebuild_xb(int mode) { g_rebuild_xb = (mode == 0 || mode == 1) ? mode : -1; }
static size_t l2_bytes()
{
#ifdef PMG_HOST_EMULATION
    return (size_t)126 << 20;
#else
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    static int cached[64] = {};
    int &c = cached[dev & 63];
    if (c == 0) c = (cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev) == cudaSuccess && v > 0) ? v : -1;
    return c > 0 ? (size_t)c : 0;
#endif
}
bool fused_rebuild_xb(const FusedLevel &lv, int nu1)
{
    if (g_rebuild_xb == -2) {
        const char *e = getenv("PMG_REBUILD_XB");
        g_rebuild_xb = (e && (e[0] == '0' || e[0] == '1')) ? e[0] - '0' : -1;
    }
    if (lv.ny != 0 || !fused_supported(nu1) || g_rebuild_xb == 0) return false;
    if (g_rebuild_xb == 1) return true;
    const size_t l2 = l2_bytes();
    return l2 > 0 && 3 * level_elems(lv.n) * sizeof(double) > l2;
}
void fused_set_deep_prefetch_below(int n) { g_deep_prefetch_below = n; }
void fused_set_halo_prologue(int on) { g_halo_prologue = on ? 1 : 0; }
void fused_set_wait_timeout_ns(unsigned long long ns)
{
#ifndef PMG_HOST_EMULATION
    cudaMemcpyToSymbol(g_wait_timeout_ns, &ns, sizeof(ns));
#else
    (void)ns;
#endif
}
int fused_halo_prologue() { return g_halo_prologue; }

int fused_max_partials(int n)
{
    int best = 0;
    FusedLevel lv{};
    lv.n = n;
    lv.pitch = level_pitch(n);
    for (int v = 0; v < NUM_VARIANTS; ++v) {
        StripGeom g = make_geom(lv, 8, VARIANTS[v], 8, 8);
        int c = g.n_strips * g.n_chunks;
        g = make_geom(lv, 4, VARIANTS[v], 8, 8);
        if (g.n_strips * g.n_chunks > c) c = g.n_strips * g.n_chunks;
        if (c > best) best = c;
    }
    return best + 64;
}

// The tuning variants exist for the headline V(2,2) configuration only; other sweep counts use variant 0.
#define PMG_DISPATCH_S2(VAR, FN, ...)                                       \
    switch (VAR) {                                                          \
        case 1: FN<2, 3, 5, true, 2>(__VA_ARGS__); break;                   \
        case 2: FN<2, 4, 4, false, 2>(__VA_ARGS__); break;                  \
        case 3: FN<2, 3, 6, true, 2>(__VA_ARGS__); break;                   \
        case 4: FN<2, 7, 4, true, 2>(__VA_ARGS__); break;                   \
        default: FN<2, 3, 4, true, 2>(__VA_ARGS__); break;                  \
    }

void launch_fused_down(const FusedLevel &lv, double *coarse_f, int pitch_c, int nu1, double omega,
                       bool x_is_zero, cudaStream_t st, const int *done, bool store_xb)
{
    bool resid = coarse_f != nullptr;
    // the xb store is skipped only where Pass B can rebuild xb: a first visit of a whole level
    if (!fused_supported(nu1) || (!store_xb && !(x_is_zero && resid && lv.ny == 0))) {  // never skip a pass silently
        g_fused_bad_nu = fused_supported(nu1) ? -1 : nu1;
        return;
    }
    switch (nu1) {
        case 1: down_launch<2, 3, 4, true, 1>(lv, coarse_f, pitch_c, omega, x_is_zero, resid, store_xb, done, st); break;
        case 2: PMG_DISPATCH_S2(lv.n <= deep_prefetch_below() ? 4 : ((x_is_zero && resid) ? g_variant_down_zero : g_variant_down), down_launch, lv, coarse_f, pitch_c, omega, x_is_zero, resid, store_xb, done, st); break;
        case 3: down_launch<2, 3, 4, true, 3>(lv, coarse_f, pitch_c, omega, x_is_zero, resid, store_xb, done, st); break;
        case 4: down_launch<2, 2, 4, true, 4>(lv, coarse_f, pitch_c, omega, x_is_zero, resid, store_xb, done, st); break;
        default: break;
    }
}

bool fused_down_prolong_supported(int nu1) { return nu1 == 2; }
// xb = S^2(P e_in), coarse_f = R(f - A xb): Pass A of the first cycle on a level that nested iteration has just reached
// (MultiGrid.hpp:161-167) without materialising P e_in.  One GPU, nu1 = 2.
void launch_fused_down_prolong(const FusedLevel &lv, const double *e_in, int pitch_e, double *coarse_f, int pitch_c, double omega,
                               int prolong_mode, cudaStream_t st, const int *done)
{
    const int lo = prolong_mode == PMG_PROLONG_FULL ? 1 : 2;
    JacobiCoef c = jacobi_coef(lv.h, omega);
    if (c.weighted)
        down_prolong_launch_w<true>(lv, e_in, pitch_e, lo, coarse_f, pitch_c, c, done, st);
    else
        down_prolong_launch_w<false>(lv, e_in, pitch_e, lo, coarse_f, pitch_c, c, done, st);
    count_launch();
}

void launch_fused_up(const FusedLevel &lv, const double *coarse_x, int pitch_c, int nu2, double omega,
                     int prolong_mode, double *d_partials, int *n_partials, cudaStream_t st, const int *done, int rebuild_nu1)
{
    bool norm = d_partials != nullptr;
    int lo = prolong_mode == PMG_PROLONG_FULL ? 1 : 2;
    if (!fused_supported(nu2)) {
        g_fused_bad_nu = nu2;
        if (n_partials) *n_partials = 0;
        return;
    }
    if (rebuild_nu1 != 0) {  // xb rebuilt from f: whole level, with a prolongation, without the norm
        if (n_partials) *n_partials = 0;
        if (!fused_supported(rebuild_nu1) || norm || coarse_x == nullptr || lv.ny != 0) {
            g_fused_bad_nu = fused_supported(rebuild_nu1) ? -1 : rebuild_nu1;
            return;
        }
        switch (nu2) {
            case 1: up_rebuild_dispatch<2, 3, 4, true, 1>(lv, coarse_x, pitch_c, omega, lo, rebuild_nu1, done, st); break;
            case 2: up_rebuild_dispatch<2, 3, 5, true, 2>(lv, coarse_x, pitch_c, omega, lo, rebuild_nu1, done, st); break;
            case 3: up_rebuild_dispatch<2, 3, 4, true, 3>(lv, coarse_x, pitch_c, omega, lo, rebuild_nu1, done, st); break;
            case 4: up_rebuild_dispatch<2, 2, 4, true, 4>(lv, coarse_x, pitch_c, omega, lo, rebuild_nu1, done, st); break;
            default: break;
        }
        return;
    }
    switch (nu2) {
        case 1: up_launch<2, 3, 4, true, 1>(lv, coarse_x, pitch_c, omega, lo, norm, d_partials, n_partials, done, st); break;
        case 2: PMG_DISPATCH_S2(lv.n <= deep_prefetch_below() ? 4 : (norm ? g_variant_up_norm : g_variant_up), up_launch, lv, coarse_x, pitch_c, omega, lo, norm, d_partials, n_partials, done, st); break;
        case 3: up_launch<2, 3, 4, true, 3>(lv, coarse_x, pitch_c, omega, lo, norm, d_partials, n_partials, done, st); break;
        case 4: up_launch<2, 2, 4, true, 4>(lv, coarse_x, pitch_c, omega, lo, norm, d_partials, n_partials, done, st); break;
        default: break;
    }
}

}  // namespace pmg
