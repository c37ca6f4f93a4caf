// Tensor-core version of the on-chip sweep for 32 < d <= 64: block Gauss-Jordan with
// 8 x 8 pivot blocks whose rank-8 updates are pairs of DMMA.8x8x4 (mma.sync.m8n8k4.f64).
//
// Why.  The scalar rank-1 sweep (small_gj.cuh) is bound by shared->register bandwidth
// (16 doubles/clk/SM; a 4 x 2 register tile gets 1.2 FMA per loaded double, the FP64 pipe
// needs 4) and by one barrier per pivot.  A 16 x 32 warp tile updated by DMMA gets
// 10.7 FMA per loaded double and needs ONE barrier per 8 pivots.  The remaining serial
// chain (publish -> barrier -> 8 x 8 pivot-block inverse) is hidden by running TWO
// independent problems (CTAs) per SM: 256 threads and <= 128 registers each, with the
// Adam moments parked in tensor memory (TMEM) -- the 256 KB per SM that tcgen05 kernels
// use for accumulators and that is otherwise idle here (FP64 has no tcgen05 kind).
//
// Layout.  256 threads = 8 warps in a 4 (wr) x 2 (wc) grid (wr = warp / 2); warp (wr, wc) owns rows
// 16wr.., columns 32wc.. of the 64 x 64 padded matrix as 2 x 4 DMMA accumulator tiles:
//   a[ti][tj][e] = A[16wr + 8ti + lane/4][32wc + 8tj + 2(lane%4) + e].
// The score accumulator g and the Adam moments use the same ownership.  A pivot block is exactly
// ONE accumulator tile: block b (pivots K = 8b..8b+7) is tile (ti, tj) = (b & 1, b & 3) of warp
// (wr, wc) = (b >> 1, b >> 2), the "diagonal warp" of the step.
//
// Block step b -- block form of the publish identity of small_gj.cuh:
//   publish  Rpub = A[K, :] + [I at the K block],  Cpub = A[:, K] - [I at the K block];
//            -Q = -(A[K,K])^{-1} was computed one step EARLY by the diagonal warp,
//   barrier, then every warp:  CS = Cpub (-Q)      (two DMMA per 8 rows, see dmma_block_step),
//            A += CS Rpub  (16 DMMA).
// With the two I's the same product turns the pivot block into Q, the pivot rows into
// Q A[K,:] and the pivot columns into -A[:,K] Q: no tile is special and nothing is zeroed.
// The 8 x 8 pivot blocks are themselves inverted by scalar Gauss-Jordan in natural order,
// so the sweep yields the same d scalar pivots as small_gj.cuh: log|det| = sum log|pivot|,
// and "M-matrix" = all pivots > 0.
#pragma once
#include "small_gj.cuh"

namespace dagma {

constexpr int DM_DP = 64;          // padded dimension
constexpr int DM_NT = 256;         // threads per CTA
constexpr int DM_LD = 68;          // row stride (doubles) of the padded smem matrices / row lines
constexpr int DM_PB = 8;           // pivot block
constexpr int DM_TMEM_COLS = 128;  // 32-bit TMEM columns per CTA: 2 warps per lane quarter x 64

struct DmmaSmem {                  // offsets in doubles
    static constexpr int ncov = 0;                         // -cov, [64][68]
    static constexpr int W = ncov + DM_DP * DM_LD;         // W,    [64][68]
    static constexpr int rbuf = W + DM_DP * DM_LD;         // 2 x [8][68]      published pivot rows
    static constexpr int cbuf = rbuf + 2 * DM_PB * DM_LD;  // 2 x 2 x [64][4]  published pivot columns (two 4-column planes)
    static constexpr int qbuf = cbuf + 2 * DM_DP * DM_PB;  // 2 x 64           -Q in B-fragment order
    static constexpr int pinfo = qbuf + 2 * 64;            // 64               fraction-free pivots in natural order
    static constexpr int red = pinfo + 64;                 // 96
    static constexpr int mbar = red + 96;                  // 1 (the step barrier, 8 bytes)
    static constexpr int total = mbar + 2;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(DmmaSmem::rbuf % 2 == 0 && DmmaSmem::cbuf % 2 == 0 && DmmaSmem::qbuf % 2 == 0 &&
              DmmaSmem::pinfo % 2 == 0 && DmmaSmem::W % 2 == 0, "16-byte alignment of vector accesses");

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

struct DmmaPos {
    int warp, lane, wr, wc, qr, qc;
    __device__ __forceinline__ explicit DmmaPos(int tid) {
        warp = tid >> 5; lane = tid & 31; wr = warp >> 1; wc = warp & 1; qr = lane >> 2; qc = lane & 3;
    }
    __device__ __forceinline__ int row(int ti) const { return 16 * wr + 8 * ti + qr; }
    __device__ __forceinline__ int col(int tj) const { return 32 * wc + 8 * tj + 2 * qc; }   // + e
};

// ---------------------------------------------------------------- mbarrier (split arrive / wait)
__device__ __forceinline__ void mbar_init(uint32_t addr, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t addr) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t addr, uint32_t parity) {
    // one cheap test first (the last arriver of a phase is usually the warp on the serial chain),
    // then try_wait, which suspends the warp in hardware
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\t"
                 "WAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@!p bra WAIT_%=;\n\tDONE_%=:\n\t}"
                 ::"r"(addr), "r"(parity) : "memory");
}

__device__ __forceinline__ bool mbar_test(uint32_t addr, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    return ok != 0;
}

// Work a warp can do while it waits for the step barrier of the sweep (see dmma_block_step): `more()` -- is there a
// unit left, `unit()` -- do one.  The default has none.
struct NoFill {
    __device__ __forceinline__ bool more() const { return false; }
    __device__ __forceinline__ void unit() {}
};

// The diagonal warp of block `b` inverts the pivot block P = A[K,K] = its accumulator tile (TI, TJ):
// lane (qr, qc) holds P[qr][2qc], P[qr][2qc+1].  Two phases of four pivots, each a FRACTION-FREE
// Gauss-Jordan in natural pivot order over all 8 rows: rows i != k become p_k row_i - x_ik row_k, so no
// reciprocal sits between two pivots; the row scales (D_i = prod_{m>=i} p_m for the rows of the phase,
// the product of its four pivots for the other rows) are divided out once per phase.  Four pivots per
// phase keep the scale products inside 8th powers of the true pivots.  Broadcasts are warp shuffles.
// For the Z-matrices of DAGMA the off-diagonal updates still add numbers of one sign, exactly as in the
// scaled elimination.
// Writes -Q (in the order the B fragments of the next block step read it) and the eight fraction-free
// pivots p_k (all > 0 <=> all scalar pivots > 0; log|det P| = sum_k ((k & 3) - 2) log|p_k|).
// `extra(k)` is issued right after the shuffles of pivot k: independent tensor work of the same warp that
// fits in the shuffle latency (the chain is latency bound, the warp's issue slots are mostly free).
template <int TI, int TJ, class Extra>
__device__ __forceinline__ void stage_pivot_block(const double (&a)[2][4][2], const DmmaPos& ps, double* sm, int b,
                                                  int qslot, Extra&& extra) {
    constexpr unsigned FULL = 0xffffffffu;
    const int i = ps.qr, jq = ps.qc;
    double x0 = a[TI][TJ][0], x1 = a[TI][TJ][1];
    double* pi = sm + DmmaSmem::pinfo + b * DM_PB;
#pragma unroll
    for (int ph = 0; ph < 2; ++ph) {
        double D = 1.0, E = 1.0;                  // E = prod of the phase's earlier pivots: scale of its rows not yet pivoted
        const int irel = i - 4 * ph;              // rows outside the phase collect all four pivots
        const int ie = (irel > 3) ? -1 : irel;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const int k = 4 * ph + kk, kl = k >> 1;
            const double xs = (k & 1) ? x1 : x0;  // column k, in the lanes qc == kl
            const double p = __shfl_sync(FULL, xs, 4 * k + kl);
            const double c = __shfl_sync(FULL, xs, 4 * i + kl);
            const double r0 = __shfl_sync(FULL, x0, 4 * k + jq), r1 = __shfl_sync(FULL, x1, 4 * k + jq);
            extra(k);
            if (ps.lane == 0) pi[k] = p;
            const bool ik = (i == k), j0k = (2 * jq == k), j1k = (2 * jq + 1 == k);
            // off the chain: what the pivot row / pivot column lanes become
            const double nce = -c * E;
            const double alt0 = ik ? (j0k ? E : x0) : nce, alt1 = ik ? (j1k ? E : x1) : nce;
            const double Dp = D * p;
            D = (kk >= ie) ? Dp : D;
            E *= p;
            // on the chain: one multiply, one fma, one select per element.  (A variant with five instead of seven
            // FP64 instructions per pivot -- the pivot-column lanes fed through the same fma by operand selects, the row
            // scales rebuilt after the phase -- was measured 16 % SLOWER, 1.55 k against 1.34 k clk per block
            // inversion inside the sweep: the selects and the late row scale sit on the dependency chain, and the chain
            // is bound by latency, not by issue slots.)
            const double t0 = fma(-c, r0, p * x0), t1 = fma(-c, r1, p * x1);
            x0 = (ik || j0k) ? alt0 : t0;
            x1 = (ik || j1k) ? alt1 : t1;
        }
        const double rd = fast_rcp(D);
        x0 *= rd;
        x1 *= rd;
    }
    // -Q[k][n] goes where lane (qr, qc) of k-slab kk = k / 4 finds its B fragment:
    //   B[qc][qr] = -Q[4kk + qc][(qr >> 1) + 4 (qr & 1)]   <=>   index 32 (k / 4) + 4 (2 (n & 3) + n / 4) + (k & 3)
    double* qd = sm + DmmaSmem::qbuf + qslot * 64 + 32 * (i >> 2) + (i & 3);
    const int n0 = 2 * jq, n1 = 2 * jq + 1;
    qd[4 * (2 * (n0 & 3) + (n0 >> 2))] = -x0;
    qd[4 * (2 * (n1 & 3) + (n1 >> 2))] = -x1;
}

// publish the pivot rows (+I) / pivot columns (-I) of block B into line buffer B & 1;
// the +-I touches only the pivot block itself, i.e. tile (TI, TJ) of the diagonal warp
template <int B>
__device__ __forceinline__ void publish_block(const double (&a)[2][4][2], const DmmaPos& ps, double* sm) {
    constexpr int TI = B & 1, TJ = B & 3, CUR = B & 1;
    double* rb = sm + DmmaSmem::rbuf + CUR * DM_PB * DM_LD;
    double* cb = sm + DmmaSmem::cbuf + CUR * DM_DP * DM_PB;
    const bool rown = ps.wr == (B >> 1), cown = ps.wc == (B >> 2);
    double p0 = a[TI][TJ][0], p1 = a[TI][TJ][1], m0 = p0, m1 = p1;      // pivot-block tile: row / column copy
    if (rown && cown) {
        const int dlt = ps.qr - 2 * ps.qc;
        const double i0 = (dlt == 0) ? 1.0 : 0.0, i1 = (dlt == 1) ? 1.0 : 0.0;
        p0 += i0; p1 += i1; m0 -= i0; m1 -= i1;
    }
    if (rown) {
        double* dst = rb + ps.qr * DM_LD + ps.col(0);
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
            *reinterpret_cast<double2*>(dst + 8 * tj) = (tj == TJ) ? make_double2(p0, p1) : make_double2(a[TI][tj][0], a[TI][tj][1]);
    }
    if (cown) {
        double* dst = cb + (ps.qc >> 1) * (DM_DP * 4) + ps.row(0) * 4 + 2 * (ps.qc & 1);
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)
            *reinterpret_cast<double2*>(dst + 32 * ti) = (ti == TI) ? make_double2(m0, m1) : make_double2(a[ti][TJ][0], a[ti][TJ][1]);
    }
}

// G += (-cov)[:, K] W[K, :] for the k-block kb of 4 (8 DMMA); independent of the elimination
__device__ __forceinline__ void gemm_chunk(double (&g)[2][4][2], const DmmaPos& ps, const double* sm, int kb) {
    const double* nc = sm + DmmaSmem::ncov;
    const double* Ws = sm + DmmaSmem::W;
    const int k0 = 4 * kb;
    double an[2], bw[4];
#pragma unroll
    for (int ti = 0; ti < 2; ++ti) an[ti] = nc[ps.row(ti) * DM_LD + k0 + ps.qc];
#pragma unroll
    for (int tj = 0; tj < 4; ++tj) bw[tj] = Ws[(k0 + ps.qc) * DM_LD + 32 * ps.wc + 8 * tj + ps.qr];
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) dmma(g[ti][tj][0], g[ti][tj][1], an[ti], bw[tj]);
}

#ifdef DAGMA_SWEEP_TRACE
// debug build only: cycle stamps of the serial chain (CTA 0, the block steps of one sweep)
__device__ long long g_sweep_trace[64 * 8];
#define SWEEP_STAMP(slot, cond) do { if (blockIdx.x == 0 && (cond) && ps.lane == 0 && sy.trace >= 0 && sy.trace < 64) g_sweep_trace[sy.trace * 8 + (slot)] = clock64(); } while (0)
#else
#define SWEEP_STAMP(slot, cond) do { } while (0)
#endif

#ifndef DAGMA_SWEEP_JIT_ROWS
#define DAGMA_SWEEP_JIT_ROWS 0       // 1: pivot-row fragments loaded tile by tile inside the block step
#endif

#ifndef DAGMA_FILL_MATE_SKIP
#define DAGMA_FILL_MATE_SKIP 0       // 1: the warp that shares the sub-partition (FP64 pipe) with the next diagonal warp does no filler work during that block step
#endif

#ifndef DAGMA_STAGE_INTERLEAVE
#define DAGMA_STAGE_INTERLEAVE 1     // diagonal warp: its publish-critical DMMAs 1 inside / 0 after / 2 before the pivot-block chain
#endif

struct SweepSync {        // per-thread view of the step barrier
    uint32_t bar;         // shared address of the mbarrier (count = warps)
    uint32_t phase;       // parity to wait for next
#ifdef DAGMA_SWEEP_TRACE
    int trace = -1;
#endif
};

// One block step, B compile time.  On entry the lines of block B are published and every warp has
// arrived on the step barrier; the step
//   waits for it,
//   forms CS, updates FIRST the five tiles that hold the pivot rows / columns of block B + 1,
//   lets the diagonal warp invert the next pivot block, publishes the lines of block B + 1 and
//   arrives -- and only then updates its remaining three tiles, off the serial chain.
// CS = Cpub (-Q) for 8 rows is ONE accumulator tile: the B fragments carry -Q[:, n/2] in the even and
// -Q[:, 4 + n/2] in the odd columns n, so that c0 / c1 of lane (qr, qc) are CS[qr][qc] / CS[qr][4 + qc]
// = exactly its A fragments for the two k-slabs of the rank-8 update.
template <int B, class Fill>
__device__ __forceinline__ void dmma_block_step(double (&a)[2][4][2], const DmmaPos& ps, double* sm, int nb,
                                                SweepSync& sy, Fill& fill) {
    constexpr int CUR = B & 1;
    constexpr int BN = (B + 1) & 7;                                   // next block
    constexpr int TIN = BN & 1, TJN = BN & 3;
    const double* rb = sm + DmmaSmem::rbuf + CUR * DM_PB * DM_LD;
    const double* cb = sm + DmmaSmem::cbuf + CUR * DM_DP * DM_PB;
    const double* qb = sm + DmmaSmem::qbuf + CUR * 64;
    const bool has_next = B + 1 < nb;
    const bool diag_next = has_next && (ps.wr == (BN >> 1)) && (ps.wc == (BN >> 2));
#ifdef DAGMA_SWEEP_TRACE
    const bool trc_diag = diag_next;
    const bool trc_other = (ps.warp == ((((BN >> 1) + 2) & 3) * 2 + (1 - (BN >> 2))));   // a warp far from the diagonal
#endif
    SWEEP_STAMP(0, trc_diag);
    SWEEP_STAMP(5, trc_other);
    // Every warp but the one that is about to run the pivot chain of this step spends the wait on independent work
    // (the fit kernel: k-blocks of the score GEMM) -- one unit at a time, polling the barrier in between, so the step
    // starts at most one unit late for warps that are off the critical path and not at all late for the chain.
#if DAGMA_FILL_MATE_SKIP
    // warps w and w ^ 4 issue to the same sub-partition: the filler DMMAs of the mate (16 clk of the FP64 pipe each) would
    // sit in front of the dependent FP64 instructions of the pivot chain
    const bool mate_next = has_next && (ps.warp == ((2 * (BN >> 1) + (BN >> 2)) ^ 4));
    if (!diag_next && !mate_next)
#else
    if (!diag_next)
#endif
        while (fill.more() && !mbar_test(sy.bar, sy.phase)) fill.unit();
    mbar_wait(sy.bar, sy.phase);
    sy.phase ^= 1u;
    SWEEP_STAMP(1, trc_diag);
    SWEEP_STAMP(6, trc_other);
    double bq[2], ac[2][2], acs[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) bq[kk] = qb[32 * kk + ps.lane];
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) ac[ti][kk] = cb[kk * (DM_DP * 4) + ps.row(ti) * 4 + ps.qc];
#if DAGMA_SWEEP_JIT_ROWS
    // the pivot-row fragments are fetched tile by tile (two 8-byte loads in front of the two DMMAs that use them)
    // instead of all eight up front: 12 registers fewer are live across the step -- room for the accumulators of
    // the filler work (the score GEMM of the fit kernel)
    const double* rbl = rb + ps.qc * DM_LD + 32 * ps.wc + ps.qr;
    auto upd = [&](int ti, int tj) {
        const double b0 = rbl[8 * tj], b1 = rbl[4 * DM_LD + 8 * tj];
        dmma(a[ti][tj][0], a[ti][tj][1], acs[ti][0], b0);
        dmma(a[ti][tj][0], a[ti][tj][1], acs[ti][1], b1);
    };
#else
    double br[2][4];
#pragma unroll
    for (int kk = 0; kk < 2; ++kk)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) br[kk][tj] = rb[(4 * kk + ps.qc) * DM_LD + 32 * ps.wc + 8 * tj + ps.qr];
    auto upd = [&](int ti, int tj) {
        dmma(a[ti][tj][0], a[ti][tj][1], acs[ti][0], br[0][tj]);
        dmma(a[ti][tj][0], a[ti][tj][1], acs[ti][1], br[1][tj]);
    };
#endif
    auto cs1 = [&](int ti) { dmma(acs[ti][0], acs[ti][1], ac[ti][0], bq[0]); };
    auto cs2 = [&](int ti) { dmma(acs[ti][0], acs[ti][1], ac[ti][1], bq[1]); };
    // ---- the serial chain first: CS of the next pivot rows, the next pivot block itself
    cs1(TIN);
    cs2(TIN);
    upd(TIN, TJN);
    SWEEP_STAMP(2, trc_diag);
    // the rest of the next pivot rows / columns (what the publish needs)
    constexpr int O0 = (TJN == 0) ? 1 : 0, O1 = (TJN <= 1) ? 2 : 1, O2 = (TJN <= 2) ? 3 : 2;   // tj != TJN
    auto portion = [&](int k) {
        if (k == 0) cs1(TIN ^ 1);
        else if (k == 1) cs2(TIN ^ 1);
        else if (k == 2) upd(TIN, O0);
        else if (k == 3) upd(TIN, O1);
        else if (k == 4) upd(TIN, O2);
        else if (k == 5) upd(TIN ^ 1, TJN);
    };
    if (diag_next) {
#if DAGMA_STAGE_INTERLEAVE == 1
        stage_pivot_block<TIN, TJN>(a, ps, sm, B + 1, CUR ^ 1, portion);
#elif DAGMA_STAGE_INTERLEAVE == 2
#pragma unroll
        for (int k = 0; k < 6; ++k) portion(k);          // the other publish-critical tiles first, then a clean chain
        stage_pivot_block<TIN, TJN>(a, ps, sm, B + 1, CUR ^ 1, [](int) {});
#else
        stage_pivot_block<TIN, TJN>(a, ps, sm, B + 1, CUR ^ 1, [](int) {});
#pragma unroll
        for (int k = 0; k < 6; ++k) portion(k);
#endif
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) portion(k);
    }
    SWEEP_STAMP(3, trc_diag);
    if (has_next) {
        publish_block<BN>(a, ps, sm);
        __syncwarp();
        if (ps.lane == 0) mbar_arrive(sy.bar);
    }
    SWEEP_STAMP(4, trc_diag);
    // ---- the three tiles nobody is waiting for
#pragma unroll
    for (int tj = 0; tj < 4; ++tj)
        if (tj != TJN) upd(TIN ^ 1, tj);
    SWEEP_STAMP(7, trc_other);
#ifdef DAGMA_SWEEP_TRACE
    if (sy.trace >= 0) ++sy.trace;
#endif
}

// a := a^{-1} on the leading 8*ceil(d/8) block (padding inside the last pivot block must
// carry a unit diagonal).  pinfo[k] = fraction-free pivots (see stage_pivot_block), k < 8*ceil(d/8).
// All warps must have passed a __syncthreads since the last use of the line buffers.
template <class Fill>
__device__ __forceinline__ void dmma_sweep(double (&a)[2][4][2], const DmmaPos& ps, double* sm, int d, SweepSync& sy,
                                           Fill& fill) {
    const int nb = (d + DM_PB - 1) / DM_PB;
    if (ps.wr == 0 && ps.wc == 0) stage_pivot_block<0, 0>(a, ps, sm, 0, 0, [](int) {});
    publish_block<0>(a, ps, sm);
    __syncwarp();
    if (ps.lane == 0) mbar_arrive(sy.bar);
    dmma_block_step<0>(a, ps, sm, nb, sy, fill);
    if (nb > 1) dmma_block_step<1>(a, ps, sm, nb, sy, fill);
    if (nb > 2) dmma_block_step<2>(a, ps, sm, nb, sy, fill);
    if (nb > 3) dmma_block_step<3>(a, ps, sm, nb, sy, fill);
    if (nb > 4) dmma_block_step<4>(a, ps, sm, nb, sy, fill);
    if (nb > 5) dmma_block_step<5>(a, ps, sm, nb, sy, fill);
    if (nb > 6) dmma_block_step<6>(a, ps, sm, nb, sy, fill);
    if (nb > 7) dmma_block_step<7>(a, ps, sm, nb, sy, fill);
    __syncthreads();
}
__device__ __forceinline__ void dmma_sweep(double (&a)[2][4][2], const DmmaPos& ps, double* sm, int d, SweepSync& sy) {
    NoFill none;
    dmma_sweep(a, ps, sm, d, sy, none);
}

// g += (-cov) W over the k range 4*ceil(d/4): 16 independent DMMA per k-block and warp, no serial chain --
// the phase that keeps the FP64 pipe busy while the other CTA of the SM is inside its sweep.  Kept apart
// from the sweep so that g is not live (32 registers) while the sweep holds its line fragments.
__device__ __forceinline__ void dmma_score_gemm(double (&g)[2][4][2], const DmmaPos& ps, const double* sm, int d) {
    const int nk = (d + 3) >> 2;
#pragma unroll 1
    for (int kb = 0; kb < nk; ++kb) gemm_chunk(g, ps, sm, kb);
}

// The score GEMM as filler work of the sweep: one k-block (8 DMMA) per unit; what the waits did not absorb is finished
// after the sweep.
struct ScoreFill {
    double (&g)[2][4][2];
    const DmmaPos& ps;
    const double* sm;
    int kb, nk;
    __device__ __forceinline__ bool more() const { return kb < nk; }
    __device__ __forceinline__ void unit() { gemm_chunk(g, ps, sm, kb++); }
};

// ---------------------------------------------------------------- tensor memory (TMEM) scratch
// Thread-private spill space: warp w owns TMEM lanes 32(w%4)..+31 (hardware rule for
// tcgen05.ld/st), thread = lane; the two warps of a lane quarter use disjoint column ranges.
template <int COLS = DM_TMEM_COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_slot_addr) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot_addr),
                 "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS = DM_TMEM_COLS>
__device__ __forceinline__ void tmem_free(uint32_t taddr) {             // one full warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tmem_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 8 doubles <-> 16 consecutive 32-bit columns of the thread's own TMEM lane
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const double (&x)[8]) {
    uint32_t r[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        r[2 * i] = (uint32_t)__double2loint(x[i]);
        r[2 * i + 1] = (uint32_t)__double2hiint(x[i]);
    }
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
struct TmemLoad8 {   // issue now, finish() later (after which get() is valid)
    uint32_t r[16];
    __device__ __forceinline__ void issue(uint32_t taddr) {
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr)
            : "memory");
    }
    // the wait names the registers so no use of them can be scheduled above it
    __device__ __forceinline__ void finish() {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                       "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                       "+r"(r[15])
                     :
                     : "memory");
    }
    __device__ __forceinline__ double get(int i) const { return __hiloint2double((int)r[2 * i + 1], (int)r[2 * i]); }
};

}  // namespace dagma
