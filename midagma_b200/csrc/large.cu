// Multi-CTA path for d > 64 and for the logistic loss (SURVEY.md 8a rows a1-a5 at
// C2 / C5 sizes): FP64 DMMA GEMM, blocked Gauss-Jordan inverse, score reductions and
// the fused Adam / feasibility update, all driven by a small device-resident state
// block so that a whole inner iteration is a fixed launch sequence (CUDA-graph
// replayable, no host synchronisation until the next convergence checkpoint).
//
// Blocked inverse (d > 128), in place, no pivoting (M-matrix).  Single level (d <= 256), block 64:
//   step kb:  P = A[K,K];  Q = P^{-1} (tensor-core sweep of small_dmma.cuh, redundantly in every
//             panel CTA);  CS = -Cpub Q (d x 64) with Cpub = A[:,K] and its K block replaced by P - I;
//             Rpub = A[K,:]           with its K block replaced by I + P;
//             A += CS * Rpub          (one d x d x 64 DMMA GEMM, no special tiles).
// The two replacements make the single GEMM produce Q in the pivot block, Q A[K,:] in
// the pivot rows and -A[:,K] Q in the pivot columns (block form of the identity used
// by the on-chip sweep, see small_gj.cuh).  Two levels (d > 256): the same step with 256-wide
// blocks whose pivot block is inverted by the single-level sweep, so that the d x d updates are
// rank-256 GEMMs.  log|det| comes from the pivots of all 4 x 4 pivot blocks.
#include "common.cuh"
#include "gemm_f64.cuh"
#include "gemm_tma.cuh"
#include "small_gj.cuh"
#include "small_dmma.cuh"
#include "lin_state.h"
#include <cstdlib>
#include "../../include/dagma_b200.h"

namespace dagma {

int logdet_inv_small(cudaStream_t, int, int, double, const double*, int, int, double*, double*,
                     double*, double*, int, double*, int*);

// ------------------------------------------------------------------ GEMM host side
template <int BM, int BN, int WM, int WN>
static int gemm_launch_tile(cudaStream_t stream, int transA, int M, int N, int K, double alpha, const double* A,
                            int lda, const double* B, int ldb, double beta, double* C, int ldc, int epi, double* ws,
                            size_t ws_bytes) {
    using T = GemmTile<BM, BN, WM, WN>;
    constexpr int GTHREADS = T::THREADS;
    static bool attr_done = false;
    if (!attr_done) {
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_f64_kernel<false, EPI_NONE, BM, BN, WM, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM_BYTES));
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_f64_kernel<false, EPI_SIGMOID, BM, BN, WM, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM_BYTES));
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_f64_kernel<true, EPI_NONE, BM, BN, WM, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM_BYTES));
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_f64_kernel<true, EPI_SIGMOID, BM, BN, WM, WN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM_BYTES));
        attr_done = true;
    }
    const int tm = (M + BM - 1) / BM, tn = (N + BN - 1) / BN;
    const int ktiles = (K + GBK - 1) / GBK;
    // split K when the output grid cannot fill the machine and K is long
    int splits = 1;
    const int slots = 148 * T::MINB * BM * BN / (128 * 64);   // in units that keep the old heuristic
    if (tm * tn < slots / 2 && ktiles >= 8 && ws != nullptr) {
        splits = slots / (tm * tn);
        if (splits > ktiles / 4) splits = ktiles / 4;
        while (splits > 1 && (size_t)splits * M * N * sizeof(double) > ws_bytes) --splits;
        if (splits < 1) splits = 1;
    }
    // K = 0: one pass with an empty k range, so the kernel's epilogue leaves beta * C (and the sigmoid), as BLAS does
    const int kchunk_tiles = ktiles > 0 ? (ktiles + splits - 1) / splits : 1;
    splits = ktiles > 0 ? (ktiles + kchunk_tiles - 1) / kchunk_tiles : 1;
    GemmArgs P{M, N, K, A, lda, B, ldb, C, ldc, alpha, beta, kchunk_tiles * GBK, splits > 1 ? ws : nullptr};
    dim3 grid(tn, tm, splits);
    const size_t sm = T::SMEM_BYTES;
    if (splits > 1) {   // epilogue is applied by the reduce kernel
        if (transA) gemm_f64_kernel<true, EPI_NONE, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
        else gemm_f64_kernel<false, EPI_NONE, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
        DAGMA_CUDA_OK(cudaGetLastError());
        const int blocks = (int)(((size_t)M * N + 255) / 256);
        if (epi == EPI_SIGMOID)
            splitk_reduce_kernel<EPI_SIGMOID><<<blocks < 1184 ? blocks : 1184, 256, 0, stream>>>(ws, splits, M, N, C, ldc, alpha, beta);
        else
            splitk_reduce_kernel<EPI_NONE><<<blocks < 1184 ? blocks : 1184, 256, 0, stream>>>(ws, splits, M, N, C, ldc, alpha, beta);
    } else if (epi == EPI_SIGMOID) {
        if (transA) gemm_f64_kernel<true, EPI_SIGMOID, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
        else gemm_f64_kernel<false, EPI_SIGMOID, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
    } else {
        if (transA) gemm_f64_kernel<true, EPI_NONE, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
        else gemm_f64_kernel<false, EPI_NONE, BM, BN, WM, WN><<<grid, GTHREADS, sm, stream>>>(P);
    }
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

// DAGMA_GEMM_TILE (debug / A-B timing): 0 = 64 x 64 tile, 128 threads, four CTAs per SM (default: the finest
// granularity wins at the 2000-wide outputs of this path); 1 = 128 x 128, one CTA; 2 = 128 x 64, two CTAs
static int gemm_tile_variant() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_GEMM_TILE");
        v = e ? atoi(e) : 0;
    }
    return v;
}

static unsigned* tma_queue(cudaStream_t stream);
static int tma_mode();
static bool gemm_tma_ok(int transA, int M, int N, int K, const double* A, int lda, const double* B, int ldb);
static int gemm_tma_launch(cudaStream_t stream, int M, int N, int K, double alpha, const double* A, int lda,
                           const double* B, int ldb, double beta, double* C, int ldc, int epi, unsigned* queue,
                           int mode);
static int gemm_tma_sched(int M, int N, int K, double beta, int epi);

static int gemm_launch(cudaStream_t stream, int transA, int M, int N, int K, double alpha, const double* A, int lda,
                       const double* B, int ldb, double beta, double* C, int ldc, int epi, double* ws,
                       size_t ws_bytes) {
    if (M <= 0 || N <= 0) return 0;
    if (gemm_tma_ok(transA, M, N, K, A, lda, B, ldb)) {
        const int sched = gemm_tma_sched(M, N, K, beta, epi);
        if (sched >= 0)
            return gemm_tma_launch(stream, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi,
                                   (sched & 1) ? tma_queue(stream) : nullptr, sched);
    }
    if (gemm_tile_variant() == 1)
        return gemm_launch_tile<128, 128, 4, 2>(stream, transA, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi, ws, ws_bytes);
    if (gemm_tile_variant() == 2)
        return gemm_launch_tile<128, 64, 4, 2>(stream, transA, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi, ws, ws_bytes);
    return gemm_launch_tile<64, 64, 2, 2>(stream, transA, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi, ws, ws_bytes);
}

// ------------------------------------------------------------------ blocked inverse
constexpr int NB = 64;
#ifndef DAGMA_PDL_DEFAULT
#define DAGMA_PDL_DEFAULT 0
#endif
#ifndef DAGMA_TMA_DEFAULT
#define DAGMA_TMA_DEFAULT 5      // outer-step update tiles + long stand-alone GEMMs (see tma_mode)
#endif

// build M = s I - (square ? A o A : A), scaled by inv_scale, into out (d x d, ld = d)
__global__ void build_m_kernel(const double* __restrict__ A, int lda, double* __restrict__ out, int d, double s,
                               double inv_scale, int square) {
    const size_t total = (size_t)d * d;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / d), c = (int)(e - (size_t)r * d);
        double x = A[(size_t)r * lda + c];
        if (square) x *= x;
        out[e] = (((r == c) ? s : 0.0) - x) * inv_scale;
    }
}

struct TileStepArgs {
    const double* Ain;   // n x n (ld = n), state before block step kb
    double* Aout;        // n x n (ld = n), state after it (a different buffer: tiles are owned, not synchronised)
    int n, kb;
    double* pivots;      // fraction-free pivots (see stage_pivot_block), 4*ceil(n/4) entries
#ifdef DAGMA_OUTER_TRACE
    int trace_kb = -1;
#endif
};

// One block step (block 64) of the single-level Gauss-Jordan as ONE launch without any inter-CTA
// synchronisation: CTA (bi, bj) owns the 64 x 64 tile (bi, bj) and recomputes what it needs --
//   Q = P^{-1} by the tensor-core sweep of small_dmma.cuh (P = A[K,K], 32 KB, L2 resident),
//   CS_i = -(A[I,K] - [bi == kb] I) Q,   R_j = A[K,J] + [bj == kb] I,
//   tile_out = tile_in + CS_i R_j        (two 64^3 DMMA products).
// Reading the old state from Ain (through L2) and writing the new one to Aout (ping-pong) removes every hazard;
// the redundancy (nblk^2 sweeps, nblk CS products) runs in parallel on otherwise idle SMs.


__device__ __forceinline__ double ldcg(const double* p) { return __ldcg(p); }   // L2: written by other CTAs

#ifdef DAGMA_OUTER_TRACE
// debug build only: %globaltimer stamps (ns) of one two-level inversion, [outer step][slot]
//   0 first CTA in   1 server 0: pivot tile updated   2 server 0: past the first barrier
//   3..6 server 0: tile step kb done   7 last server done   8 last update item done   9 first CS' item starts
//   10 last CS' item done   11 last CTA out   12 first update item starts   13 last R' item done
//   16 + 5 kb + {0 loads, 1 sweep, 2 CS product, 3 R loaded, 4 tile written}: inside tile step kb of server 0
__device__ unsigned long long g_outer_trace[16 * 40];
__device__ int g_outer_step;
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define OT_SET(slot) do { if (threadIdx.x == 0) g_outer_trace[g_outer_step * 40 + (slot)] = gtime(); } while (0)
#define OT_MAX(slot) do { if ((threadIdx.x & 127) == 0) atomicMax(&g_outer_trace[g_outer_step * 40 + (slot)], gtime()); } while (0)
#define OT_MIN(slot) do { if ((threadIdx.x & 127) == 0) atomicMin(&g_outer_trace[g_outer_step * 40 + (slot)], gtime()); } while (0)
#define OT_TILE(slot) do { if (P.trace_kb >= 0) OT_SET(16 + 5 * P.trace_kb + (slot)); } while (0)
#define FT_SET(k, slot) do { if (threadIdx.x == 0 && blockIdx.x == 0) g_outer_trace[(k) * 40 + (slot)] = gtime(); } while (0)
#define FT_MAX(k, slot) do { if ((threadIdx.x & 127) == 0) atomicMax(&g_outer_trace[(k) * 40 + (slot)], gtime()); } while (0)
#define FT_MIN(k, slot) do { if ((threadIdx.x & 127) == 0) atomicMin(&g_outer_trace[(k) * 40 + (slot)], gtime()); } while (0)
__global__ void flow_trace_begin_kernel() {
    for (int q = 0; q < 16 * 40; ++q) g_outer_trace[q] = (q % 40 == 12) ? ~0ull : 0ull;
}
__global__ void outer_trace_begin_kernel(int step) {
    g_outer_step = step;
    for (int q = 0; q < 40; ++q) g_outer_trace[step * 40 + q] = (q == 0 || q == 9 || q == 12) ? ~0ull : 0ull;
}
#else
#define OT_SET(slot) do { } while (0)
#define OT_MAX(slot) do { } while (0)
#define OT_MIN(slot) do { } while (0)
#define OT_TILE(slot) do { } while (0)
#define FT_SET(k, slot) do { } while (0)
#define FT_MAX(k, slot) do { } while (0)
#define FT_MIN(k, slot) do { } while (0)
#endif

#ifndef DAGMA_TILE_STEP_PREFETCH
#define DAGMA_TILE_STEP_PREFETCH 1   // 1: A[I,K] / A[K,J] land in shared memory by cp.async WHILE the sweep runs; 0: loads between the phases
#endif
// shared memory of a tile step (doubles): the two operand tiles sit where the fit kernel keeps -cov and W, which the
// sweep does not touch; Q goes on top of the sweep's line buffers once the sweep is over; the step barrier of the
// sweep lives behind it (it must survive from one tile step to the next)
constexpr int TS_CS = DmmaSmem::ncov, TS_R = DmmaSmem::W, TS_Q = DmmaSmem::rbuf;
constexpr int TS_MBAR = TS_Q + DM_DP * DM_LD;
constexpr int TS_TOTAL = TS_MBAR + 2;
static_assert(TS_MBAR >= DmmaSmem::total && TS_MBAR % 2 == 0, "the barrier is outside everything the sweep writes");

__device__ __forceinline__ void tile_step(const TileStepArgs& P, int bi, int bj, double* psm, SweepSync& sy) {
    using S = DmmaSmem;
    constexpr int LD = DM_LD;
    double* Cs = psm + TS_CS;       // [64][68]  A[I,K] - [bi == kb] I, later CS
    double* Rs = psm + TS_R;        // [64][68]  A[K,J] + [bj == kb] I
    double* Qs = psm + TS_Q;        // [64][68]  Q (after the sweep)
    const int tid = threadIdx.x;
    const DmmaPos ps(tid);
    const int n = P.n, k0 = P.kb * NB;
    const int kn = min(NB, n - k0);
    const int r0 = bi * NB, c0 = bj * NB;
    const bool vec = ((n & 1) == 0) && ((reinterpret_cast<uintptr_t>(P.Ain) & 15) == 0);

#if DAGMA_TILE_STEP_PREFETCH
    // ---- both operand tiles are requested now and land during the sweep (zero fill outside the matrix / the block)
    load_slab<NB, NB, DM_NT>(smem_u32(Cs), LD, P.Ain, n, r0, k0, n, k0 + kn, vec, tid);
    load_slab<NB, NB, DM_NT>(smem_u32(Rs), LD, P.Ain, n, k0, c0, k0 + kn, n, vec, tid);
    cp_async_commit();
#endif
    // ---- P into the accumulator layout (identity padding)
    double a[2][4][2], acc[2][4][2];
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int r = ps.row(ti), c = ps.col(tj);
            if (vec) {                                  // n even: c and c + 1 are inside or outside together
                double2 v = make_double2((r == c) ? 1.0 : 0.0, (r == c + 1) ? 1.0 : 0.0);
                if (r < kn && c < kn) v = __ldcg(reinterpret_cast<const double2*>(&P.Ain[(size_t)(k0 + r) * n + k0 + c]));
                a[ti][tj][0] = v.x;
                a[ti][tj][1] = v.y;
            } else {
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    a[ti][tj][e] = (r < kn && c + e < kn) ? ldcg(&P.Ain[(size_t)(k0 + r) * n + k0 + c + e]) : ((r == c + e) ? 1.0 : 0.0);
            }
        }
#if !DAGMA_TILE_STEP_PREFETCH
    {   // all 16 loads of a thread in flight before the first use
        double v[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = tid + q * DM_NT, r = e >> 6, c = e & 63;
            v[q] = (r0 + r < n && c < kn) ? ldcg(&P.Ain[(size_t)(r0 + r) * n + k0 + c]) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = tid + q * DM_NT, r = e >> 6, c = e & 63;
            Cs[r * LD + c] = v[q];
        }
    }
#endif
    __syncthreads();
    OT_TILE(0);
    dmma_sweep(a, ps, psm, kn, sy);
    OT_TILE(1);
    const bool piv_out = (bi == 0 && bj == 0 && tid < 4 * ((kn + 3) >> 2));
    const double piv = piv_out ? psm[S::pinfo + tid] : 0.0;          // Q is about to overwrite the line buffers
#if DAGMA_TILE_STEP_PREFETCH
    cp_async_wait<0>();
#else
    {
        double w[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = tid + q * DM_NT, r = e >> 6, c = e & 63;
            w[q] = (r < kn && c0 + c < n) ? ldcg(&P.Ain[(size_t)(k0 + r) * n + c0 + c]) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = tid + q * DM_NT, r = e >> 6, c = e & 63;
            Rs[r * LD + c] = w[q];
        }
    }
#endif
    __syncthreads();                 // the copies of every thread have landed; the pivots are in registers
    if (piv_out) P.pivots[k0 + tid] = piv;
    if (tid < kn) {                  // the two identities of the publish trick
        if (bi == P.kb) Cs[tid * LD + tid] -= 1.0;
        if (bj == P.kb) Rs[tid * LD + tid] += 1.0;
    }
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int r = ps.row(ti), c = ps.col(tj);
            const bool in0 = (r < kn && c < kn), in1 = (r < kn && c + 1 < kn);
            *reinterpret_cast<double2*>(Qs + r * LD + c) = make_double2(in0 ? a[ti][tj][0] : 0.0, in1 ? a[ti][tj][1] : 0.0);
        }
    __syncthreads();
    // the old tile travels while the first product runs
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int r = r0 + ps.row(ti), c = c0 + ps.col(tj);
            if (vec) {
                double2 v = make_double2(0.0, 0.0);
                if (r < n && c < n) v = __ldcg(reinterpret_cast<const double2*>(&P.Ain[(size_t)r * n + c]));
                a[ti][tj][0] = v.x;
                a[ti][tj][1] = v.y;
            } else {
                a[ti][tj][0] = (r < n && c < n) ? ldcg(&P.Ain[(size_t)r * n + c]) : 0.0;
                a[ti][tj][1] = (r < n && c + 1 < n) ? ldcg(&P.Ain[(size_t)r * n + c + 1]) : 0.0;
            }
        }
    // ---- CS = -((A[I,K] - dI) Q)   (warp tile 16 x 32, 16 k-blocks of 4; the sign costs nothing: rounding is symmetric)
    auto product = [&](const double* Am, const double* Bm) {
#pragma unroll 4
        for (int kk = 0; kk < NB; kk += 4) {
            double an[2], bw[4];
#pragma unroll
            for (int ti = 0; ti < 2; ++ti) an[ti] = Am[ps.row(ti) * LD + kk + ps.qc];
#pragma unroll
            for (int tj = 0; tj < 4; ++tj) bw[tj] = Bm[(kk + ps.qc) * LD + 32 * ps.wc + 8 * tj + ps.qr];
#pragma unroll
            for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                for (int tj = 0; tj < 4; ++tj) dmma(acc[ti][tj][0], acc[ti][tj][1], an[ti], bw[tj]);
        }
    };
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) acc[ti][tj][0] = acc[ti][tj][1] = 0.0;
    product(Cs, Qs);
    __syncthreads();                 // every warp is done reading A[I,K] and Q
    OT_TILE(2);
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            *reinterpret_cast<double2*>(Cs + ps.row(ti) * LD + ps.col(tj)) = make_double2(-acc[ti][tj][0], -acc[ti][tj][1]);
            acc[ti][tj][0] = a[ti][tj][0];                              // accumulators restart from the old tile
            acc[ti][tj][1] = a[ti][tj][1];
        }
    __syncthreads();
    OT_TILE(3);
    // ---- tile_out = tile_in + CS R
    product(Cs, Rs);
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int r = r0 + ps.row(ti), c = c0 + ps.col(tj);
            if (vec) {
                if (r < n && c < n) *reinterpret_cast<double2*>(&P.Aout[(size_t)r * n + c]) = make_double2(acc[ti][tj][0], acc[ti][tj][1]);
            } else {
                if (r < n && c < n) P.Aout[(size_t)r * n + c] = acc[ti][tj][0];
                if (r < n && c + 1 < n) P.Aout[(size_t)r * n + c + 1] = acc[ti][tj][1];
            }
        }
    OT_TILE(4);
}


__global__ void __launch_bounds__(DM_NT, 1) inv_tile_step_kernel(const TileStepArgs P) {
    extern __shared__ __align__(16) double psm[];
    SweepSync sy{smem_u32(psm + TS_MBAR), 0u};
    if (threadIdx.x == 0) mbar_init(sy.bar, DM_NT / 32);
    tile_step(P, blockIdx.y, blockIdx.x, psm, sy);
}

// ---- look-ahead "panel server": the whole inversion of the NEXT 256-wide pivot block as one kernel that
// runs beside the d x d update.  One CTA per 64 x 64 tile of the block (<= 16 CTAs); each asks for the
// whole shared memory of an SM, so it shares its SM with nobody and the update kernel simply runs on the
// remaining SMs.  Phase 0: tile of P' = A[K',K'] + CS[K',:] R[:,K'] (the update restricted to the pivot
// block); then nblk tile steps, separated by a counter barrier in global memory.  The CTAs of ONE launch
// wait for each other, never for another kernel: if some are scheduled late the early ones spin, nothing
// else is blocked, and the spin is bounded (err flag) -- progress never depends on co-residency.
struct ServerArgs {
    double *buf0, *buf1;     // ping-pong n x n (ld = n)
    int n, nblk;
    double* pivots;
    unsigned* counter;       // zeroed before the launch
    int* err;
};
__device__ __forceinline__ void server_barrier(unsigned* counter, unsigned target, int* err) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        unsigned spins = 0;
        while (*((volatile unsigned*)counter) < target) {
            if (*(volatile int*)err) break;
            if (++spins > (1u << 26)) { *err = 1; break; }
        }
        __threadfence();
    }
    __syncthreads();
}

// server CTA `rank` of `nctas`: owns tile (rank / nblk, rank % nblk) of the next pivot block, whose
// current value the CTAs have just written to buf0
__device__ __forceinline__ void server_role(const ServerArgs& P, int rank, unsigned nctas, double* psm) {
    using S = DmmaSmem;
    const int tid = threadIdx.x;
    const int bi = rank / P.nblk, bj = rank % P.nblk;
    const int n = P.n;
    SweepSync sy{smem_u32(psm + TS_MBAR), 0u};
    if (tid == 0) mbar_init(sy.bar, DM_NT / 32);

    server_barrier(P.counter, nctas, P.err);
    if (rank == 0) OT_SET(2);

    // ---- the block steps
    double *in = P.buf0, *out = P.buf1;
    for (int kb = 0; kb < P.nblk; ++kb) {
        TileStepArgs T{in, out, n, kb, P.pivots};
#ifdef DAGMA_OUTER_TRACE
        T.trace_kb = (rank == 0) ? kb : -1;
#endif
        tile_step(T, bi, bj, psm, sy);
        if (rank == 0) OT_SET(3 + kb);
        if (kb + 1 < P.nblk) server_barrier(P.counter, nctas * (unsigned)(kb + 2), P.err);
        double* t = in;
        in = out;
        out = t;
    }
    __syncthreads();
}

// ---- one outer step of the two-level algorithm as ONE persistent kernel (two CTAs per SM).
// Work items are pulled from an atomic queue, in this order (K = current 256-block, K' = next one):
//   [server CTAs only]  tile (i, j) of the pivot block: A[K'_i,K'_j] += CS[K'_i,:] R[:,K'_j], then the
//                       inversion of that block (tile steps + counter barrier)  -> Q'
//   update tiles         A[I,J] += CS[I,:] R[:,J]: column strip K' first, then row strip K', then the rest
//   CS' tiles            CS'[I,:] = -(A[I,K'] - [I in K'] I) Q'    -- wait for: column strip done, Q' done
//   R' tiles             R'[:,J]  =   A[K',J] + [J in K'] I        -- wait for: row strip done
// so the next outer step needs no other kernel: CS / R are double buffered across steps.  Waiting items sit
// at the end of the queue behind items that never wait, every wait is bounded, and the CTAs of the serial
// look-ahead chain get their SM to themselves (the co-resident worker CTA sleeps meanwhile).
struct OuterArgs {
    double* A; int d;                       // d x d in place (ld = d, d even)
    const double* CS; const double* R;      // current: d x kn (ld = kn), kn x d (ld = d)
    int kn;
    double* CSn; double* Rn;                // next:    d x kn1 (ld = kn1), kn1 x d (ld = d)
    int k1, kn1;                            // first column and width of the next block (kn1 = 0: last step)
    const double* Qn;                       // where the server leaves Q' (kn1 x kn1, ld = kn1)
    unsigned* sync;                         // [0] server barrier [1] queue [2] err [3] col strip [4] row strip [5] server done [6] CS' / CS queue [7] CS tiles done
    int* sm_busy;                           // [SM id] 1 while a server CTA runs there; [SM_SLOTS + SM id] CS' role claimed
    int nserver;
    ServerArgs srv;
    int use_tma;                            // update tiles fed by TMA (gemm_tma.cuh) instead of cp.async
    int sleep;                              // 1: a worker CTA that shares its SM with a look-ahead CTA sleeps meanwhile
    // cs_head = 1: the step forms ITS OWN CS = -(A[:,K] - E) Q at its start (Q = Qc, left behind by the look-ahead of
    // the previous step) instead of the previous step forming it as its tail: only the look-ahead CTAs wait for the
    // row blocks of CS they need (rows K', first in the queue), so the product overlaps the serial chain instead of
    // preceding it.  CSw = CS (writable), k0 = first column of K.
    int cs_head;
    double* CSw; const double* Qc; int k0;
    unsigned* cs_rows;                      // [row block] CS tiles finished (cs_head)
};
constexpr int SM_SLOTS = 256;
constexpr int CS_ROW_SLOTS = 256;           // row blocks of 64: d <= 16384
constexpr int SYNC_STRIDE = 8 + 2 * SM_SLOTS + CS_ROW_SLOTS;    // unsigned words of one outer step's sync block
// Worker side: a 256-thread CTA is TWO independent 128-thread tile engines (half = tid / 128), each the
// main loop of gemm_f64_kernel<64, 64, 2, 2> (64 x 64 x 16 slabs, warp tile 32 x 32, 3-stage cp.async
// pipeline, one barrier per k-slab -- a named barrier of the half).  Four engines per SM cover each
// other's barrier / copy waits exactly as four CTAs of the stand-alone GEMM do.
using EngT = GemmTile<64, 64, 2, 2>;
constexpr int EN_NT = 128;
constexpr int EN_STG = EngT::A_STAGE + EngT::B_STAGE;                   // doubles per pipeline stage
constexpr int EN_SMEM = GSTAGES * EN_STG;                               // doubles per engine
constexpr size_t OUTER_SMEM_BYTES = (2 * (size_t)EN_SMEM > (size_t)DmmaSmem::total ? 2 * (size_t)EN_SMEM : (size_t)DmmaSmem::total) * sizeof(double);
static_assert(NB * NB <= EN_SMEM, "the split-K partial of a server tile is parked in the engine's stages");
static_assert((size_t)TS_TOTAL * sizeof(double) <= OUTER_SMEM_BYTES, "a tile step fits in the shared memory of an outer-step CTA");
constexpr size_t TILE_STEP_SMEM_BYTES = (size_t)TS_TOTAL * sizeof(double);

__device__ __forceinline__ unsigned smid() {
    unsigned r;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(r));
    return r;
}
__device__ __forceinline__ bool wait_count(volatile unsigned* c, unsigned target, int* err, unsigned ns = 500) {
    unsigned spins = 0;
    while (*c < target) {
        __nanosleep(ns);
        if (++spins > (1u << 22)) { *err = 2; return false; }
    }
    __threadfence();
    return true;
}
__device__ __forceinline__ bool spin_count(volatile unsigned* c, unsigned target, int* err) {   // the serial chain: no sleep
    unsigned spins = 0;
    while (*c < target) {
        if (++spins > (1u << 26)) { *err = 3; return false; }
    }
    __threadfence();
    return true;
}
#ifndef DAGMA_HALF_SYNC_IMM
#define DAGMA_HALF_SYNC_IMM 1
#endif
__device__ __forceinline__ void half_sync(int half) {            // barrier of one 128-thread engine
#if DAGMA_HALF_SYNC_IMM
    if (half) asm volatile("bar.sync 2, %0;" ::"n"(EN_NT) : "memory");
    else asm volatile("bar.sync 1, %0;" ::"n"(EN_NT) : "memory");
#else
    asm volatile("bar.sync %0, %1;" ::"r"(half + 1), "n"(EN_NT) : "memory");
#endif
}

struct EnginePos {          // thread of an engine: warp (wm, wn) of a 2 x 2 grid owns a 32 x 32 tile
    int htid, lane, wm, wn, qr, qc;
    __device__ __forceinline__ explicit EnginePos(int tid) {
        htid = tid & (EN_NT - 1);
        lane = htid & 31;
        const int w = htid >> 5;
        wm = w >> 1; wn = w & 1; qr = lane >> 2; qc = lane & 3;
    }
    __device__ __forceinline__ int row(int i) const { return 32 * wm + 8 * i + qr; }
    __device__ __forceinline__ int col(int j) const { return 32 * wn + 8 * j + 2 * qc; }   // + e
};

// acc += Am[r0.., kbeg..kend) * Bm[kbeg..kend, c0..)  for one 64 x 64 tile; operands come through L2
// (cp.async.cg).  rmax / cmax: valid rows of Am / columns of Bm.  lda, ldb even, bases 16-byte aligned.
// engine_prefetch requests the first two slabs (two commit groups, stages 0 and 1); engine_gemm with
// prefetched = true continues from there, so the requests can be made before the previous tile's epilogue.
__device__ __forceinline__ void engine_issue(const double* Am, int lda, const double* Bm, int ldb, int r0, int c0,
                                             int rmax, int cmax, int kbeg, int kend, int kt, uint32_t ebase, int htid) {
    const int nk = (kend - kbeg + GBK - 1) / GBK;
    if (kt < nk) {
        const int st = kt % GSTAGES;
        const uint32_t sa = ebase + (uint32_t)(st * EN_STG) * 8, sb = sa + (uint32_t)EngT::A_STAGE * 8;
        const int k0 = kbeg + kt * GBK;
        load_slab<NB, GBK, EN_NT>(sa, EngT::LDA_N, Am, lda, r0, k0, rmax, kend, true, htid);
        load_slab<GBK, NB, EN_NT>(sb, EngT::LDB_S, Bm, ldb, k0, c0, kend, cmax, true, htid);
    }
    cp_async_commit();
}
__device__ __forceinline__ void engine_prefetch(const double* Am, int lda, const double* Bm, int ldb, int r0, int c0,
                                                int rmax, int cmax, int kbeg, int kend, double* esm, int htid) {
    const uint32_t ebase = smem_u32(esm);
#pragma unroll
    for (int st = 0; st < GSTAGES - 1; ++st) engine_issue(Am, lda, Bm, ldb, r0, c0, rmax, cmax, kbeg, kend, st, ebase, htid);
}
__device__ __forceinline__ void engine_gemm(double (&acc)[4][4][2], const double* Am, int lda, const double* Bm, int ldb,
                                            int r0, int c0, int rmax, int cmax, int kbeg, int kend, double* esm,
                                            const EnginePos& ep, int half, bool prefetched = false) {
    const uint32_t ebase = smem_u32(esm);
    const int nk = (kend - kbeg + GBK - 1) / GBK;
    if (!prefetched) {
        half_sync(half);                       // the stages may still be read by the previous item
        engine_prefetch(Am, lda, Bm, ldb, r0, c0, rmax, cmax, kbeg, kend, esm, ep.htid);
    }
    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<GSTAGES - 2>();
        half_sync(half);                       // slab kt landed; slab kt-1 is free for reuse
        engine_issue(Am, lda, Bm, ldb, r0, c0, rmax, cmax, kbeg, kend, kt + GSTAGES - 1, ebase, ep.htid);
        const double* As = esm + (kt % GSTAGES) * EN_STG;
        const double* Bs = As + EngT::A_STAGE;
#pragma unroll
        for (int kk = 0; kk < GBK; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[ep.row(i) * EngT::LDA_N + kk + ep.qc];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[(kk + ep.qc) * EngT::LDB_S + 32 * ep.wn + 8 * j + ep.qr];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    cp_async_wait<0>();
}

__global__ void __launch_bounds__(DM_NT, 2) outer_step_kernel(const OuterArgs P,
                                                              const __grid_constant__ CUtensorMap mapCS,
                                                              const __grid_constant__ CUtensorMap mapR) {
    extern __shared__ __align__(16) double psm[];
    __shared__ unsigned s_tile[2];
    __shared__ __align__(8) unsigned long long s_tbars[2][2 * TM_STAGES];
    const int tid = threadIdx.x;
    const int half = tid >> 7;
    const EnginePos ep(tid);
    double* esm = psm + half * EN_SMEM;
    TmaPipe<Tm64> pipe;
    tm_pipe_init(pipe, smem_u32(esm), smem_u32(s_tbars[half]), P.use_tma && ep.htid == 0);
    if (P.use_tma && ep.htid == 0) {
        tm_prefetch_map(&mapCS);
        tm_prefetch_map(&mapR);
    }
    __syncthreads();
    // Programmatic dependent launch (DAGMA_PDL): everything above -- pipeline barriers, tensor-map prefetch -- may run
    // while the previous outer step is still draining (its CTAs leave one by one during the CS' tail); from here on the
    // step reads what that kernel wrote.  The trigger right behind the wait lets the NEXT step's CTAs take the slots
    // this step's CTAs free up; they block in their own wait until this grid has completed and flushed.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int d = P.d, kn = P.kn, k1 = P.k1, kn1 = P.kn1;
    int* err = reinterpret_cast<int*>(P.sync + 2);
    volatile int* busy = P.sm_busy + (smid() % SM_SLOTS);
    double acc[4][4][2];
    OT_MIN(0);

    auto load_acc = [&](const double* M, int ld, int r0, int c0, int rmax, int cmax) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                double2 v = make_double2(0.0, 0.0);
                if (r < rmax && c < cmax) v = __ldcg(reinterpret_cast<const double2*>(M + (size_t)r * ld + c));
                acc[i][j][0] = v.x;
                acc[i][j][1] = v.y;
            }
    };
    auto zero_acc = [&]() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    };

    // ================= look-ahead: the CTAs of the next pivot block =================
    if ((int)blockIdx.x < P.nserver) {
        if (tid == 0) *busy = 1;
        const int nb1 = P.srv.nblk, bi = blockIdx.x / nb1, bj = blockIdx.x % nb1;
        const int r0 = k1 + bi * NB, c0 = k1 + bj * NB;
        // the pivot-block tile of the update itself (its result is both the new A tile and the server's input),
        // split over k between the two engines of the CTA: this product sits on the serial chain
        const int kmid = min(kn, ((kn / 2 + GBK - 1) / GBK) * GBK);
        if (half == 0) load_acc(P.A, d, r0, c0, d, d);
        else zero_acc();
        if (P.cs_head && kn > 0) {                // the rows of CS this tile needs: formed by the worker CTAs, first in their queue
            if (tid == 0) (void)spin_count(P.cs_rows + r0 / NB, (unsigned)((kn + NB - 1) / NB), err);
            __syncthreads();
        }
        engine_gemm(acc, P.CS, kn, P.R, d, r0, c0, d, d, half ? kmid : 0, half ? kn : kmid, esm, ep, half);
        half_sync(half);
        if (half == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<double2*>(esm + ep.row(i) * NB + ep.col(j)) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
        __syncthreads();
        if (half == 0) {
            const double* part = psm + EN_SMEM;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                    if (r < d && c < d) {
                        const double2 q = *reinterpret_cast<const double2*>(part + ep.row(i) * NB + ep.col(j));
                        const double2 v = make_double2(acc[i][j][0] + q.x, acc[i][j][1] + q.y);
                        *reinterpret_cast<double2*>(P.A + (size_t)r * d + c) = v;
                        *reinterpret_cast<double2*>(P.srv.buf0 + (size_t)(r - k1) * kn1 + (c - k1)) = v;
                    }
                }
        }
        __syncthreads();
        if (blockIdx.x == 0) OT_SET(1);
        if (tid == 0) {                           // this tile belongs to the column strip and to the row strip
            __threadfence();
            atomicAdd(P.sync + 3, 1u);
            atomicAdd(P.sync + 4, 1u);
        }
        server_role(P.srv, blockIdx.x, (unsigned)P.nserver, psm);
        OT_MAX(7);
        if (tid == 0) {
            __threadfence();
            atomicAdd(P.sync + 5, 1u);
            *busy = 0;
        }
        __syncthreads();
    }

    const int tn = (d + NB - 1) / NB;
    const int cb1 = k1 / NB, nk1 = (kn1 + NB - 1) / NB;          // block-column range of K'
    // ================= CS = -(A[:,K] - E) Q of THIS step (cs_head) =================
    // One 64 x 64 tile per CTA and item, split over k between the CTA's two engines; the row blocks of K' come first
    // (the look-ahead CTAs are waiting for exactly those), every finished tile is counted per row block and in total.
    // Nothing writes A[:,K] before all tiles are done: the update tiles below wait for the total.
    const int nkc = (kn + NB - 1) / NB;
    const int n_csh = (P.cs_head && kn > 0) ? tn * nkc : 0;
    bool cs_worker = false;
    if (n_csh > 0 && (int)blockIdx.x >= P.nserver) {      // ONE CTA per SM: a tile alone on its SM takes half the time
        if (tid == 0) s_tile[0] = (atomicExch(reinterpret_cast<int*>(P.sm_busy) + SM_SLOTS + (smid() % SM_SLOTS), 1) == 0) ? 1u : 0u;
        __syncthreads();
        cs_worker = s_tile[0] != 0u;
        __syncthreads();
    }
    if (cs_worker) {
        const int kmid = min(kn, ((kn / 2 + GBK - 1) / GBK) * GBK);
        const int cb0 = P.k0 / NB;
        for (;;) {
            if (tid == 0) s_tile[0] = atomicAdd(P.sync + 6, 1u);
            __syncthreads();
            const int u = (int)s_tile[0];
            __syncthreads();
            if (u >= n_csh) break;
            OT_MIN(9);
            const int rb = u / nkc, jb = u % nkc;
            const int bi = (rb < nk1) ? cb1 + rb : ((rb - nk1) < cb1 ? rb - nk1 : rb);     // rows K' first, then the others in order
            const int r0 = bi * NB, c0 = jb * NB;
            zero_acc();
            engine_gemm(acc, P.A + P.k0, d, P.Qc, kn, r0, c0, d, kn, half ? kmid : 0, half ? kn : kmid, esm, ep, half);
            half_sync(half);
            if (half == 1) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<double2*>(esm + ep.row(i) * NB + ep.col(j)) = make_double2(acc[i][j][0], acc[i][j][1]);
            }
            __syncthreads();
            if (half == 0) {
                const double* part = psm + EN_SMEM;
                const bool inK = (bi >= cb0) && (bi < cb0 + nkc);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                        if (r < d && c < kn) {
                            const double2 q2 = *reinterpret_cast<const double2*>(part + ep.row(i) * NB + ep.col(j));
                            double2 v = make_double2(-(acc[i][j][0] + q2.x), -(acc[i][j][1] + q2.y));
                            if (inK) {
                                const double2 q = __ldcg(reinterpret_cast<const double2*>(P.Qc + (size_t)(r - P.k0) * kn + c));
                                v.x += q.x;
                                v.y += q.y;
                            }
                            *reinterpret_cast<double2*>(P.CSw + (size_t)r * kn + c) = v;
                        }
                    }
            }
            __syncthreads();
            if (tid == 0) {
                __threadfence();
                atomicAdd(P.cs_rows + bi, 1u);
                atomicAdd(P.sync + 7, 1u);
            }
            OT_MAX(10);
        }
    }

    // ================= the queue (each engine pulls its own items) =================
    const int n_cs = tn * nk1 - nk1 * nk1;                       // column strip without the pivot block
    const int n_rs = nk1 * (tn - nk1);                           // row strip without the pivot block
    const int n_rest = (tn - nk1) * (tn - nk1);
    const int n_upd = (kn > 0) ? n_cs + n_rs + n_rest : 0;       // kn = 0: the step in front of the first block (nothing to apply)
    const int n_csn = tn * nk1, n_rn = nk1 * tn;
    const int n_items = n_upd + n_rn;
    auto outside = [&](int u) { return u < cb1 ? u : u + nk1; };  // u-th block index not in K'
    auto upd_tile = [&](int t, int& bi, int& bj, int& strip) {
        strip = 0;
        if (t < n_cs) { bi = outside(t / nk1); bj = cb1 + t % nk1; strip = 1; }
        else if (t < n_cs + n_rs) { const int u = t - n_cs; bi = cb1 + u / (tn - nk1); bj = outside(u % (tn - nk1)); strip = 2; }
        else { const int u = t - n_cs - n_rs; bi = outside(u / (tn - nk1)); bj = outside(u % (tn - nk1)); }
    };
    if (P.use_tma) {
        // ---- TMA-fed engines: one continuous slab stream per engine.  The index of the NEXT item is pulled when
        // an update tile starts (the atomic's latency hides behind the tile) and its first slabs are requested
        // during the tile's last slabs; accumulators start at zero and are added to A by red.global.add.f64.
        const TmaFrag<Tm64> fr(ep.wm, ep.wn, ep.qr, ep.qc);
        const bool elected = (ep.htid == 0);
        const int nkt = (kn + TM_BK - 1) / TM_BK;
        constexpr unsigned T_NONE = 0xffffffffu;
        tm_fence_proxy();                        // the stages may have been written through the generic proxy
        half_sync(half);
        if (elected) {
            while (P.sleep && *busy) __nanosleep(2000);
            if (n_csh > 0) {                     // CS of this step is complete (and, being read by TMA: ordered before the async proxy)
                (void)wait_count(P.sync + 7, (unsigned)n_csh, err, 200);
                asm volatile("fence.proxy.async;" ::: "memory");
            }
            s_tile[half] = atomicAdd(P.sync + 1, 1u);
        }
        half_sync(half);
        int t = (int)s_tile[half];
        int primed = 0;
        while (t < n_items) {
            unsigned tnx = T_NONE;
            if (t < n_upd) {
                OT_MIN(12);
                int bi, bj, strip;
                upd_tile(t, bi, bj, strip);
                const TmaTile cur{bi * NB, bj * NB, 0, nkt};
                TmaTile nxt{0, 0, 0, 0};
                if (elected && !(P.sleep && *busy)) {
                    tnx = atomicAdd(P.sync + 1, 1u);
                    if ((int)tnx < n_upd) {
                        int bi2, bj2, st2;
                        upd_tile((int)tnx, bi2, bj2, st2);
                        nxt = TmaTile{bi2 * NB, bj2 * NB, 0, nkt};
                    }
                }
                zero_acc();
                primed = tm_tile_gemm(pipe, fr, acc, &mapCS, &mapR, cur, primed, nxt, elected, ep.lane);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = cur.r0 + ep.row(i), c = cur.c0 + ep.col(j);
                        if (r < d && c < d) {
                            double* q = P.A + (size_t)r * d + c;
                            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(q)), "d"(acc[i][j][0]) : "memory");
                            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(q + 1)), "d"(acc[i][j][1]) : "memory");
                        }
                    }
                if (strip) {
                    half_sync(half);
                    if (elected) {
                        __threadfence();
                        atomicAdd(P.sync + 2 + strip, 1u);
                    }
                }
                OT_MAX(8);
            } else {
                // ---- R' tile: rows 64 ib.. of the next row strip, columns of block bj
                const int u = t - n_upd, ib = u / tn, bj = u % tn;
                if (elected && kn > 0) (void)wait_count(P.sync + 4, (unsigned)(tn * nk1), err);
                half_sync(half);
                const int c0 = bj * NB;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int rr = ib * NB + ep.row(i), c = c0 + ep.col(j);     // rr: row inside the strip
                        if (rr < kn1 && c < d) {
                            double2 v = __ldcg(reinterpret_cast<const double2*>(P.A + (size_t)(k1 + rr) * d + c));
                            if (c == k1 + rr) v.x += 1.0;
                            if (c + 1 == k1 + rr) v.y += 1.0;
                            *reinterpret_cast<double2*>(P.Rn + (size_t)rr * d + c) = v;
                        }
                    }
                OT_MAX(13);
            }
            if (elected) {
                if (tnx == T_NONE) {
                    while (P.sleep && *busy) __nanosleep(2000);
                    tnx = atomicAdd(P.sync + 1, 1u);
                }
                s_tile[half] = tnx;
            }
            half_sync(half);
            t = (int)s_tile[half];
        }
        half_sync(half);
    } else
    for (;;) {
        half_sync(half);
        if (ep.htid == 0) {
            while (P.sleep && *busy) __nanosleep(2000);
            if (n_csh > 0) (void)wait_count(P.sync + 7, (unsigned)n_csh, err, 200);
            s_tile[half] = atomicAdd(P.sync + 1, 1u);
        }
        half_sync(half);
        int t = (int)s_tile[half];
        if (t >= n_items) break;
        if (t < n_upd) {
            OT_MIN(12);
            // ---- update tile
            int bi, bj, strip = 0;
            if (t < n_cs) { bi = outside(t / nk1); bj = cb1 + t % nk1; strip = 1; }
            else if (t < n_cs + n_rs) { const int u = t - n_cs; bi = cb1 + u / (tn - nk1); bj = outside(u % (tn - nk1)); strip = 2; }
            else { const int u = t - n_cs - n_rs; bi = outside(u / (tn - nk1)); bj = outside(u % (tn - nk1)); }
            const int r0 = bi * NB, c0 = bj * NB;
            load_acc(P.A, d, r0, c0, d, d);
            engine_gemm(acc, P.CS, kn, P.R, d, r0, c0, d, d, 0, kn, esm, ep, half);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                    if (r < d && c < d) *reinterpret_cast<double2*>(P.A + (size_t)r * d + c) = make_double2(acc[i][j][0], acc[i][j][1]);
                }
            if (strip) {
                half_sync(half);
                if (ep.htid == 0) {
                    __threadfence();
                    atomicAdd(P.sync + 2 + strip, 1u);
                }
            }
            OT_MAX(8);
        } else {
            // ---- R' tile: rows 64 ib.. of the next row strip, columns of block bj
            const int u = t - n_upd, ib = u / tn, bj = u % tn;
            if (ep.htid == 0 && kn > 0) (void)wait_count(P.sync + 4, (unsigned)(tn * nk1), err);
            half_sync(half);
            const int c0 = bj * NB;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = ib * NB + ep.row(i), c = c0 + ep.col(j);     // rr: row inside the strip
                    if (rr < kn1 && c < d) {
                        double2 v = __ldcg(reinterpret_cast<const double2*>(P.A + (size_t)(k1 + rr) * d + c));
                        if (c == k1 + rr) v.x += 1.0;
                        if (c + 1 == k1 + rr) v.y += 1.0;
                        *reinterpret_cast<double2*>(P.Rn + (size_t)rr * d + c) = v;
                    }
                }
            OT_MAX(13);
        }
    }

    // ================= CS' = -(A[:,K'] - E) Q' : the tail of the step, on the serial chain =================
    // These tiles can only start when the look-ahead is done, i.e. when most engines have run out of work:
    // ONE CTA per SM (the first to get here) takes them from a second queue and computes each with both of
    // its engines (split over k), so the 64 nk1-by-tn tiles spread over all SMs instead of piling up on the
    // SMs whose engines happened to finish first.
    __syncthreads();
    if (kn1 > 0 && !P.cs_head) {
        if (tid == 0) s_tile[0] = (atomicExch(reinterpret_cast<int*>(P.sm_busy) + SM_SLOTS + (smid() % SM_SLOTS), 1) == 0) ? 1u : 0u;
        __syncthreads();
        const bool claimed = s_tile[0] != 0u;
        __syncthreads();
        const int kmid = min(kn1, ((kn1 / 2 + GBK - 1) / GBK) * GBK);
        while (claimed) {
            if (tid == 0) s_tile[0] = atomicAdd(P.sync + 6, 1u);
            __syncthreads();
            const int u = (int)s_tile[0];
            __syncthreads();
            if (u >= n_csn) break;
            const int bi = u / nk1, jb = u % nk1;
            if (tid == 0) (void)((kn == 0 || wait_count(P.sync + 3, (unsigned)(tn * nk1), err)) && wait_count(P.sync + 5, (unsigned)P.nserver, err));
            __syncthreads();
            OT_MIN(9);
            const int r0 = bi * NB, c0 = jb * NB;
            zero_acc();
            engine_gemm(acc, P.A + k1, d, P.Qn, kn1, r0, c0, d, kn1, half ? kmid : 0, half ? kn1 : kmid, esm, ep, half);
            half_sync(half);
            if (half == 1) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<double2*>(esm + ep.row(i) * NB + ep.col(j)) = make_double2(acc[i][j][0], acc[i][j][1]);
            }
            __syncthreads();
            if (half == 0) {
                const double* part = psm + EN_SMEM;
                const bool inK = (bi >= cb1) && (bi < cb1 + nk1);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                        if (r < d && c < kn1) {
                            const double2 q2 = *reinterpret_cast<const double2*>(part + ep.row(i) * NB + ep.col(j));
                            double2 v = make_double2(-(acc[i][j][0] + q2.x), -(acc[i][j][1] + q2.y));
                            if (inK) {
                                const double2 q = __ldcg(reinterpret_cast<const double2*>(P.Qn + (size_t)(r - k1) * kn1 + c));
                                v.x += q.x;
                                v.y += q.y;
                            }
                            *reinterpret_cast<double2*>(P.CSn + (size_t)r * kn1 + c) = v;
                        }
                    }
            }
            __syncthreads();
            OT_MAX(10);
        }
    }
    OT_MAX(11);
}

// ---- timing experiment: the stand-alone GEMM's tiles computed by engine pairs (256-thread CTAs, two per SM,
// named barriers) -- isolates the engine structure from the queue / dependency logic of the persistent kernels
__global__ void __launch_bounds__(DM_NT, 2) engine_pair_gemm_kernel(const double* A, const double* B, double* C, int d,
                                                                    int persistent, unsigned* queue) {
    extern __shared__ __align__(16) double psm[];
    __shared__ unsigned s_t[2];
    const int tid = threadIdx.x, half = tid >> 7;
    const EnginePos ep(tid);
    double* esm = psm + half * EN_SMEM;
    const int tn = (d + NB - 1) / NB, ntiles = tn * tn;
    double acc[4][4][2];
    int t = 2 * blockIdx.x + half;
    for (;;) {
        if (persistent) {
            half_sync(half);
            if (ep.htid == 0) s_t[half] = atomicAdd(queue, 1u);
            half_sync(half);
            t = (int)s_t[half];
        }
        if (t >= ntiles) break;
        const int r0 = (t / tn) * NB, c0 = (t % tn) * NB;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        engine_gemm(acc, A, d, B, d, r0, c0, d, d, 0, d, esm, ep, half);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                if (r < d && c < d) *reinterpret_cast<double2*>(C + (size_t)r * d + c) = make_double2(acc[i][j][0], acc[i][j][1]);
            }
        if (!persistent) break;
    }
}

// ---- TMA-fed GEMM (gemm_tma.cuh): C = alpha A B + beta C, A row-major M x K, B row-major K x N, persistent CTAs.
// Two tile configurations: 64 x 64 (128 threads, four CTAs per SM, 3 stages) and 128 x 128 (512 threads, ONE CTA
// per SM, 6 stages of 32 KB: half the L2 -> SM operand traffic per flop -- at 64 x 64 the slab stream is 8 flop per
// byte, about 4 TB/s at the FP64 peak).  Three schedules:
//   static   tile t, t + grid, ...                                   (queue == nullptr, balanced == 0)
//   queue    tiles pulled from an atomic counter
//   balanced every CTA gets the same number of 16-wide k-slabs: the (tile, slab) sequence is cut into grid equal
//            ranges ("stream-K").  A tile that straddles a cut is shared by exactly two CTAs (a range is at least one
//            tile long); both add their partial product to the zero-initialised tile with red.global.add.f64, and
//            0 + a + b = 0 + b + a exactly, so the result does not depend on the order.  Needs beta = 0, no epilogue.
// The first slabs of the next tile are requested during the last slabs of the current one, so the slab stream never
// drains between tiles.
struct TmaGemmArgs {
    int M, N, K;
    double* C; int ldc;
    double alpha, beta;
    int epi;
    unsigned* queue;            // zeroed before the launch (queue schedule)
    int balanced;
};
template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, 512 / Cfg::THREADS) gemm_tma_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                                   const __grid_constant__ CUtensorMap mapB,
                                                                                   const TmaGemmArgs P) {
    extern __shared__ __align__(1024) unsigned char tsm[];
    __shared__ __align__(8) unsigned long long bars[2 * Cfg::STAGES];
    __shared__ unsigned s_next;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / Cfg::WN, wn = warp % Cfg::WN, qr = lane >> 2, qc = lane & 3;
    const bool elected = (tid == 0);
    TmaPipe<Cfg> pipe;
    tm_pipe_init(pipe, smem_u32(tsm), smem_u32(bars), elected);
    if (elected) {
        tm_prefetch_map(&mapA);
        tm_prefetch_map(&mapB);
    }
    __syncthreads();
    const TmaFrag<Cfg> fr(wm, wn, qr, qc);
    const int tn = (P.N + Cfg::BN - 1) / Cfg::BN, tmr = (P.M + Cfg::BM - 1) / Cfg::BM, ntiles = tn * tmr;
    const int nk = (P.K + TM_BK - 1) / TM_BK;
    const bool vecC = ((P.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(P.C) & 15) == 0);
    // the work of this CTA as a range [u, hi) of (tile, slab) units; tile schedules: whole tiles only
    long long u = 0, hi = 0;
    if (P.balanced) {
        const long long U = (long long)ntiles * nk;
        u = U * blockIdx.x / gridDim.x;
        hi = U * (blockIdx.x + 1) / gridDim.x;
    }
    auto segment = [&](long long v, long long lim, int t) {      // balanced: the piece of a tile that starts at unit v
        if (P.balanced) {
            if (v >= lim) return TmaTile{0, 0, 0, 0};
            const int tile = (int)(v / nk), kb = (int)(v - (long long)tile * nk);
            const int len = (int)((lim - v) < (long long)(nk - kb) ? (lim - v) : (long long)(nk - kb));
            return TmaTile{(tile / tn) * Cfg::BM, (tile % tn) * Cfg::BN, kb * TM_BK, len};
        }
        if (t >= ntiles) return TmaTile{0, 0, 0, 0};
        return TmaTile{(t / tn) * Cfg::BM, (t % tn) * Cfg::BN, 0, nk};
    };
    int t = blockIdx.x, primed = 0;
    TmaTile cur = segment(u, hi, t);
    while (cur.nk > 0) {
        unsigned t_next = (unsigned)t + gridDim.x;           // static striding unless a queue is given
        if (P.queue && elected) t_next = atomicAdd(P.queue, 1u) + gridDim.x;
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        TmaTile nxt{0, 0, 0, 0};
        if (elected) {
            if (P.queue) s_next = t_next;
            nxt = segment(u + cur.nk, hi, (int)t_next);
        }
        primed = tm_tile_gemm(pipe, fr, acc, &mapA, &mapB, cur, primed, nxt, elected, lane);
        const bool partial = P.balanced && cur.nk < nk;       // a piece of a shared tile: add to the zeroed tile
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = cur.r0 + 32 * wm + 8 * i + qr;
            if (r >= P.M) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = cur.c0 + 32 * wn + 8 * j + 2 * qc;
                if (c >= P.N) continue;
                double* p = P.C + (size_t)r * P.ldc + c;
                const bool two = (c + 1 < P.N);
                double v0 = P.alpha * acc[i][j][0], v1 = P.alpha * acc[i][j][1];
                if (partial) {
                    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "d"(v0) : "memory");
                    if (two) asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p + 1)), "d"(v1) : "memory");
                    continue;
                }
                if (P.beta != 0.0) {
                    v0 = fma(P.beta, p[0], v0);
                    if (two) v1 = fma(P.beta, p[1], v1);
                }
                if (P.epi == EPI_SIGMOID) {
                    v0 = 1.0 / (1.0 + exp(-v0));
                    v1 = 1.0 / (1.0 + exp(-v1));
                }
                if (two && vecC) *reinterpret_cast<double2*>(p) = make_double2(v0, v1);
                else {
                    p[0] = v0;
                    if (two) p[1] = v1;
                }
            }
        }
        if (P.queue) {
            __syncthreads();
            t_next = s_next;
            __syncthreads();
        }
        t = (int)t_next;
        u += cur.nk;
        cur = segment(u, hi, t);
    }
}
// balanced schedule: zero the tiles that straddle a cut (CTA b looks at the start of its own range)
template <class Cfg>
__global__ void __launch_bounds__(256) gemm_tma_zero_shared_kernel(double* C, int ldc, int M, int N, int K, int grid_main) {
    const int tn = (N + Cfg::BN - 1) / Cfg::BN, tmr = (M + Cfg::BM - 1) / Cfg::BM;
    const int nk = (K + TM_BK - 1) / TM_BK;
    const long long U = (long long)tn * tmr * nk;
    const long long lo = U * blockIdx.x / grid_main;
    if (lo % nk == 0) return;
    const int tile = (int)(lo / nk), r0 = (tile / tn) * Cfg::BM, c0 = (tile % tn) * Cfg::BN;
    for (int e = threadIdx.x; e < Cfg::BM * Cfg::BN; e += 256) {
        const int r = r0 + e / Cfg::BN, c = c0 + e % Cfg::BN;
        if (r < M && c < N) C[(size_t)r * ldc + c] = 0.0;
    }
}

template <class Cfg>
static int gemm_tma_launch_cfg(cudaStream_t stream, int M, int N, int K, double alpha, const double* A, int lda,
                               const double* B, int ldb, double beta, double* C, int ldc, int epi, unsigned* queue,
                               int balanced) {
    constexpr size_t SMEM = Cfg::PIPE_BYTES + 1024;
    static bool attr = false;
    if (!attr) {
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_tma_kernel<Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        DAGMA_CUDA_OK(cudaFuncSetAttribute(gemm_tma_kernel<Cfg>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr = true;
    }
    CUtensorMap mapA, mapB;
    int rc = tm_make_a_map(&mapA, A, M, K, lda, Cfg::BM);
    if (rc) return rc;
    rc = tm_make_b_map(&mapB, B, K, N, ldb, Cfg::BN);
    if (rc) return rc;
    int sms = 0, dev = 0;
    DAGMA_CUDA_OK(cudaGetDevice(&dev));
    DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int ntiles = ((M + Cfg::BM - 1) / Cfg::BM) * ((N + Cfg::BN - 1) / Cfg::BN);
    const int nk = (K + TM_BK - 1) / TM_BK;
    const int slots = (512 / Cfg::THREADS) * sms;
    const int grid = ntiles < slots ? ntiles : slots;
    // balanced needs: no epilogue on shared tiles, every range at least one tile long
    if (balanced && !(beta == 0.0 && epi == EPI_NONE && (long long)ntiles * nk / grid >= nk)) balanced = 0;
    if (balanced) {
        queue = nullptr;
        gemm_tma_zero_shared_kernel<Cfg><<<grid, 256, 0, stream>>>(C, ldc, M, N, K, grid);
        DAGMA_CUDA_OK(cudaGetLastError());
    }
    if (queue) DAGMA_CUDA_OK(cudaMemsetAsync(queue, 0, sizeof(unsigned), stream));
    TmaGemmArgs P{M, N, K, C, ldc, alpha, beta, epi, queue, balanced};
    gemm_tma_kernel<Cfg><<<grid, Cfg::THREADS, SMEM, stream>>>(mapA, mapB, P);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}
// mode: bit 0 = atomic tile queue, bit 1 = balanced k-slab ranges, bit 2 = 128 x 128 tiles (else 64 x 64)
static int gemm_tma_launch(cudaStream_t stream, int M, int N, int K, double alpha, const double* A, int lda,
                           const double* B, int ldb, double beta, double* C, int ldc, int epi, unsigned* queue,
                           int mode) {
    if (!(mode & 1)) queue = nullptr;
    if (mode & 4)
        return gemm_tma_launch_cfg<Tm128>(stream, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi, queue, (mode >> 1) & 1);
    return gemm_tma_launch_cfg<Tm64>(stream, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, epi, queue, (mode >> 1) & 1);
}
// tile-queue words of the stand-alone TMA GEMM: a small ring in device memory, allocated once per process
// (outside stream capture: the first GEMM of a process is never captured -- engines warm up before they record
// a graph); nullptr (static tile striding) if that first call happens during a capture
static unsigned* tma_queue(cudaStream_t stream) {
    static unsigned* ring = nullptr;
    static unsigned next = 0;
    if (!ring) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return nullptr;
        if (cudaMalloc((void**)&ring, 64 * sizeof(unsigned)) != cudaSuccess) {
            ring = nullptr;
            (void)cudaGetLastError();
            return nullptr;
        }
    }
    return ring + (next++ % 64);
}
// can the TMA GEMM take this problem?  (16-byte aligned operands, even leading dimensions, enough tiles to
// fill the machine without split-K)
static bool gemm_tma_ok(int transA, int M, int N, int K, const double* A, int lda, const double* B, int ldb) {
    return !transA && M > 0 && N > 0 && K > 0 && (lda % 2 == 0) && (ldb % 2 == 0) &&
           (reinterpret_cast<uintptr_t>(A) % 16 == 0) && (reinterpret_cast<uintptr_t>(B) % 16 == 0) &&
           ((M + 63) / 64) * ((N + 63) / 64) >= 296;
}
// =====================================================================================================
// Two-level inverse as ONE dependency-driven persistent kernel ("flow" kernel).
//
// The multi-kernel version above ends every outer step with a tail that nothing overlaps (CS' of the next
// step can only start when the look-ahead inversion is done; then kernel exit, launch gap, first slabs of
// the next kernel).  Here the whole inversion is one launch:
//   * the chain team (the 16 lowest CTAs, an SM each) runs the serial chain for ALL pivot blocks:
//       CS_k rows of K_{k+1}  ->  pivot block P_{k+1} = A[K',K'] + CS_k[K',:] A[K_k,K']  ->  4 tile steps -> Q_{k+1}
//     waiting only for the three groups of tiles it reads;
//   * every other engine (two per CTA, four per SM) pulls items from one queue that lists, step by step,
//       R_k tiles (row copies + E^T), the remaining CS_k tiles, the update tiles A[I,J] += CS_k[I,:] R_k[:,J]
//     (column strip and row strip of K_{k+1} first), and waits for exactly what the item reads:
//     Q_k, per-tile version counters, per-block-row / per-block-column "CS / R ready" counters.
// Dependencies always point to earlier queue items or to the chain, and the chain's own dependencies are earlier
// queue items, so an item that is being waited for is always held by a running engine: progress does not need
// all CTAs to be co-resident (the chain team is: lowest block indices).  Every wait is bounded.
constexpr int FL_MAX_OB = 32, FL_MAX_TN = 64, FL_NSRV = (256 / NB) * (256 / NB);
struct FlowCtr {            // word offsets into the counter block (unsigned)
    static constexpr int queue = 0, err = 1, bar = 2;
    static constexpr int q_done = 8;                                   // [k]  servers that left block k's inversion
    static constexpr int upd_done = q_done + FL_MAX_OB;                // [k]
    static constexpr int cs_done = upd_done + FL_MAX_OB;               // [k]
    static constexpr int cs_rows = 128;                                // [k][bi]  CS_k tiles ready in block row bi
    static constexpr int r_cols = cs_rows + FL_MAX_OB * FL_MAX_TN;     // [k][bj]  R_k tiles ready in block column bj
    static constexpr int tile_ver = r_cols + FL_MAX_OB * FL_MAX_TN;    // [bi][bj] outer steps applied to the tile
    static constexpr int fill_ver = tile_ver + FL_MAX_TN * FL_MAX_TN;  // [bi][bj] k-chunks of the rider GEMM applied to the tile
    static constexpr int busy = fill_ver + FL_MAX_TN * FL_MAX_TN;      // [SM id]
    static constexpr int total = busy + SM_SLOTS;
};
struct FlowArgs {
    double* A; int d, nob, tn;
    double* CS[2]; double* R[2];            // per step parity: d x kn (ld = kn), kn x d (ld = d)
    double* X[2]; double* Y[2];             // per block parity: pivot block ping-pong (ld = kn)
    double* pivots;
    unsigned* ctr;
    // optional rider: gC = gA gB (all d x d, ld = d), an independent GEMM cut into the same 64 x 64 x 256 items
    // and queued ahead of each outer step's own items, so that it fills the time the engines would otherwise
    // spend waiting for the serial chain (the score GEMM cov @ W of the same iteration)
    const double* gA; const double* gB; double* gC;
    int sleep_coresident;                   // 1: the CTA that shares an SM with a chain-team CTA sleeps while the chain runs
    int rider_only;                         // debug / timing: skip the inversion, run only the rider's items
    int fill_k;                             // k extent of a rider item (256 = the outer block; rider_only timing: any multiple of 16)
    int item_base[FL_MAX_OB + 1];           // first queue index of step k
};

__device__ __forceinline__ bool flow_wait_ge(volatile unsigned* c, unsigned target, unsigned* err, unsigned code) {
    unsigned spins = 0;
    while (*c < target) {
        __nanosleep(200);
        if (*(volatile unsigned*)err) return false;              // somebody gave up: drain without waiting
        if (++spins > (1u << 23)) { *err = code; return false; }
    }
    return true;
}

__global__ void __launch_bounds__(DM_NT, 2) flow_inverse_kernel(const FlowArgs P) {
    extern __shared__ __align__(16) double psm[];
    const int tid = threadIdx.x;
    const int half = tid >> 7;
    const EnginePos ep(tid);
    double* esm = psm + half * EN_SMEM;
    const int d = P.d, tn = P.tn, nob = P.nob;
    constexpr int OB = 256, NKB = OB / NB;
    unsigned* ctr = P.ctr;
    unsigned* err = ctr + FlowCtr::err;
    volatile unsigned* vctr = ctr;
    volatile unsigned* busy = ctr + FlowCtr::busy + (smid() % SM_SLOTS);
    double acc[4][4][2];
    auto kn_of = [&](int k) { return min(OB, d - k * OB); };
    auto nk_of = [&](int k) { return (kn_of(k) + NB - 1) / NB; };
    auto n_upd_of = [&](int k) { const int n1 = (k + 1 < nob) ? nk_of(k + 1) : 0; return (unsigned)(tn * tn - n1 * n1); };
    auto zero_acc = [&]() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    };
    auto load_acc = [&](const double* M, int ld, int r0, int c0, int rmax, int cmax) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                double2 v = make_double2(0.0, 0.0);
                if (r < rmax && c < cmax) v = __ldcg(reinterpret_cast<const double2*>(M + (size_t)r * ld + c));
                acc[i][j][0] = v.x;
                acc[i][j][1] = v.y;
            }
    };
    // both engines of the CTA: acc(half 0) += partial(half 1) through the shared memory of engine 1
    auto combine_halves = [&]() {
        half_sync(half);
        if (half == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<double2*>(esm + ep.row(i) * NB + ep.col(j)) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
        __syncthreads();
        if (half == 0) {
            const double* part = psm + EN_SMEM;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double2 q = *reinterpret_cast<const double2*>(part + ep.row(i) * NB + ep.col(j));
                    acc[i][j][0] += q.x;
                    acc[i][j][1] += q.y;
                }
        }
    };

    // ================= the chain team =================
    if ((int)blockIdx.x < FL_NSRV && !P.rider_only) {
        const int rank = blockIdx.x;
        if (tid == 0 && P.sleep_coresident) *busy = 1;
        unsigned bar_target = 0;
        auto team_barrier = [&]() {
            bar_target += FL_NSRV;
            server_barrier(ctr + FlowCtr::bar, bar_target, reinterpret_cast<int*>(err));
        };
        SweepSync sy{smem_u32(psm + TS_MBAR), 0u};
        for (int kk = 0; kk < nob; ++kk) {                 // block kk is inverted here
            const int knk = kn_of(kk), nkk = nk_of(kk), cbk = kk * NKB, k1 = kk * OB;
            double* X = P.X[kk & 1];
            double* Y = P.Y[kk & 1];
            if (kk == 0) {
                // P_0: plain copy of the leading tiles
                for (int u = rank; u < nkk * nkk; u += FL_NSRV) {
                    const int bi = u / nkk, bj = u % nkk;
                    if (half == 0) {
                        load_acc(P.A, d, bi * NB, bj * NB, d, d);
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int r = bi * NB + ep.row(i), c = bj * NB + ep.col(j);
                                if (r < knk && c < knk) *reinterpret_cast<double2*>(X + (size_t)r * knk + c) = make_double2(acc[i][j][0], acc[i][j][1]);
                            }
                    }
                }
            } else {
                const int k = kk - 1, kn = kn_of(k), nk = nk_of(k), cb = k * NKB, k0 = k * OB;
                double* CSk = P.CS[k & 1];
                // ---- wait for what the chain reads: Q_k, tiles (K', K_k), (K_k, K'), (K', K') at version k,
                //      and the previous users of the buffers
                {   // one wait per thread: the counters are almost always there already, and a poll is an L2 round trip
                    const int n1 = nkk * nk, n2 = n1 + nkk, n3 = n2 + nkk * nkk;
                    if (tid == 0) flow_wait_ge(vctr + FlowCtr::q_done + k, FL_NSRV, err, 10);
                    else if (tid == 1 && k >= 2) flow_wait_ge(vctr + FlowCtr::upd_done + (k - 2), n_upd_of(k - 2), err, 11);
                    else if (tid == 2 && k >= 1) flow_wait_ge(vctr + FlowCtr::cs_done + (k - 1), (unsigned)(tn * nk_of(k - 1)), err, 12);
                    else if (tid >= 32 && tid < 32 + n3) {
                        const int q = tid - 32;
                        if (q < n1) flow_wait_ge(vctr + FlowCtr::tile_ver + (cbk + q / nk) * FL_MAX_TN + cb + q % nk, (unsigned)k, err, 13);
                        else if (q < n2) flow_wait_ge(vctr + FlowCtr::r_cols + k * FL_MAX_TN + cbk + (q - n1), (unsigned)nk, err, 14);
                        else flow_wait_ge(vctr + FlowCtr::tile_ver + (cbk + (q - n2) / nkk) * FL_MAX_TN + cbk + (q - n2) % nkk, (unsigned)k, err, 15);
                    }
                    __threadfence();
                }
                __syncthreads();
                FT_SET(kk, 0);
                const double* Qk = (nk & 1) ? P.Y[k & 1] : P.X[k & 1];
                const int kmid = min(kn, ((kn / 2 + GBK - 1) / GBK) * GBK);
                // ---- CS_k rows of K': tile (bi, jb) = -A[K'_bi, K_k] Q_k[:, jb]
                for (int u = rank; u < nkk * nk; u += FL_NSRV) {
                    const int bi = u / nk, jb = u % nk;
                    const int r0 = k1 + bi * NB, c0 = jb * NB;
                    zero_acc();
                    engine_gemm(acc, P.A + k0, d, Qk, kn, r0, c0, d, kn, half ? kmid : 0, half ? kn : kmid, esm, ep, half);
                    combine_halves();
                    if (half == 0) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                                if (r < d && c < kn) *reinterpret_cast<double2*>(CSk + (size_t)r * kn + c) = make_double2(-acc[i][j][0], -acc[i][j][1]);
                            }
                    }
                    __syncthreads();
                    if (tid == 0) {
                        __threadfence();
                        atomicAdd(ctr + FlowCtr::cs_rows + k * FL_MAX_TN + cbk + bi, 1u);
                        atomicAdd(ctr + FlowCtr::cs_done + k, 1u);
                    }
                }
                team_barrier();
                FT_SET(kk, 1);
                // ---- P_{kk} tile (bi, bj) = A[K'_bi, K'_bj] + CS_k[K'_bi, :] R_k[:, K'_bj]   (R_k: A[K_k, K'] is overwritten by step k)
                for (int u = rank; u < nkk * nkk; u += FL_NSRV) {
                    const int bi = u / nkk, bj = u % nkk;
                    const int r0 = k1 + bi * NB, c0 = k1 + bj * NB;
                    if (half == 0) load_acc(P.A, d, r0, c0, d, d);
                    else zero_acc();
                    engine_gemm(acc, CSk, kn, P.R[k & 1], d, r0, c0, d, d, half ? kmid : 0, half ? kn : kmid, esm, ep, half);
                    combine_halves();
                    if (half == 0) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int r = r0 + ep.row(i), c = c0 + ep.col(j);
                                if (r < d && c < d) {
                                    const double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
                                    *reinterpret_cast<double2*>(P.A + (size_t)r * d + c) = v;
                                    *reinterpret_cast<double2*>(X + (size_t)(r - k1) * knk + (c - k1)) = v;
                                }
                            }
                    }
                    __syncthreads();
                    if (tid == 0) {
                        __threadfence();
                        atomicAdd(ctr + FlowCtr::tile_ver + (cbk + bi) * FL_MAX_TN + cbk + bj, 1u);
                    }
                }
            }
            team_barrier();
            // ---- the inversion of block kk: nkk tile steps, ping-pong X -> Y -> X ...
            if (tid == 0) mbar_init(sy.bar, DM_NT / 32);      // the engines' slabs overwrite it between blocks
            sy.phase = 0u;
            __syncthreads();
            FT_SET(kk, 2);
            double *in = X, *out = Y;
            for (int kb = 0; kb < nkk; ++kb) {
                if (rank < nkk * nkk) {
                    TileStepArgs T{in, out, knk, kb, P.pivots + k1};
                    tile_step(T, rank / nkk, rank % nkk, psm, sy);
                }
                if (kb + 1 < nkk) team_barrier();
                double* t = in;
                in = out;
                out = t;
            }
            __syncthreads();
            FT_SET(kk, 3);
            if (tid == 0) {
                __threadfence();
                atomicAdd(ctr + FlowCtr::q_done + kk, 1u);
            }
            if (tid == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sy.bar) : "memory");
            __syncthreads();
        }
        if (tid == 0) {
            __threadfence();
            *busy = 0;
        }
        __syncthreads();
    }

    // ================= the queue (each engine pulls its own items) =================
    // Every engine runs ONE continuous stream of 64 x 16 / 16 x 64 operand slabs through its 3-stage cp.async
    // pipeline: while the last slabs of an item are multiplied, the next item has already been pulled from the
    // queue, its dependencies polled and its first two slabs requested, so that an item boundary costs the
    // epilogue only (accumulators start at zero and are added to the tile by red.global.add.f64: no load).
    const int n_total = P.item_base[nob];
    enum { IT_NONE = 0, IT_FILL = 1, IT_R = 2, IT_CS = 3, IT_UPD = 4 };
    struct Item {
        int type, k, bi, bj;               // CS: bj = column tile jb of the strip; R: bi = row tile ib of the strip
        const double* Am; const double* Bm;
        int lda, ldb, r0, c0, rmax, cmax, kbeg, kend;
    };
    int kstep = 0;
    auto decode = [&](int t) {
        Item it{};
        if (t >= n_total) return it;
        while (t >= P.item_base[kstep + 1]) ++kstep;
        const int k = kstep;
        int u0 = t - P.item_base[k];
        const int kn = kn_of(k), nk = nk_of(k), k0 = k * OB;
        const bool more = k + 1 < nob;
        const int nk1 = more ? nk_of(k + 1) : 0, cb1 = (k + 1) * NKB;
        const int n_fill = (P.gC != nullptr) ? tn * tn : 0;
        const int n_r = P.rider_only ? 0 : nk * tn, n_cs = P.rider_only ? 0 : (tn - nk1) * nk;
        auto outside = [&](int v) { return v < cb1 ? v : v + nk1; };   // v-th block index not in K'
        it.k = k;
        if (u0 < n_r) {                 // R_k tile: rows 64 ib.. of the row strip K_k, columns of block bj (+ E^T)
            it.type = IT_R; it.bi = u0 / tn; it.bj = u0 % tn;
            return it;
        }
        u0 -= n_r;
        if (u0 < n_fill) {              // rider tile: gC[I,J] (+)= gA[I, Kc] gB[Kc, J], k-chunk c = k
            it.type = IT_FILL; it.bi = u0 / tn; it.bj = u0 % tn;
            it.Am = P.gA; it.lda = d; it.Bm = P.gB; it.ldb = d;
            it.r0 = it.bi * NB; it.c0 = it.bj * NB; it.rmax = d; it.cmax = d;
            it.kbeg = k * P.fill_k; it.kend = min(d, (k + 1) * P.fill_k);
            return it;
        }
        u0 -= n_fill;
        if (u0 < n_cs) {                // CS_k tile outside the rows of K': -(A[I, K_k] - [I in K_k] I) Q_k
            it.type = IT_CS; it.bi = more ? outside(u0 / nk) : u0 / nk; it.bj = u0 % nk;
            it.Am = P.A + k0; it.lda = d; it.Bm = (nk & 1) ? P.Y[k & 1] : P.X[k & 1]; it.ldb = kn;
            it.r0 = it.bi * NB; it.c0 = it.bj * NB; it.rmax = d; it.cmax = kn; it.kbeg = 0; it.kend = kn;
            return it;
        }
        u0 -= n_cs;                     // update tile: column strip of K' first, then its row strip, then the rest
        it.type = IT_UPD;
        if (!more) { it.bi = u0 / tn; it.bj = u0 % tn; }
        else {
            const int n_c = (tn - nk1) * nk1, n_rw = nk1 * (tn - nk1);
            if (u0 < n_c) { it.bi = outside(u0 / nk1); it.bj = cb1 + u0 % nk1; }
            else if (u0 < n_c + n_rw) { const int v = u0 - n_c; it.bi = cb1 + v / (tn - nk1); it.bj = outside(v % (tn - nk1)); }
            else { const int v = u0 - n_c - n_rw; it.bi = outside(v / (tn - nk1)); it.bj = outside(v % (tn - nk1)); }
        }
        it.Am = P.CS[k & 1]; it.lda = kn; it.Bm = P.R[k & 1]; it.ldb = d;
        it.r0 = it.bi * NB; it.c0 = it.bj * NB; it.rmax = d; it.cmax = d; it.kbeg = 0; it.kend = kn;
        return it;
    };
    // dependency q (q < 8) of an item: counter and the value it must have reached; false: no such dependency
    auto dep_of = [&](const Item& it, int q, volatile unsigned*& c, unsigned& target) {
        const int k = it.k;
        switch (it.type) {
        case IT_FILL:
            if (q == 0 && k > 0) { c = vctr + FlowCtr::fill_ver + it.bi * FL_MAX_TN + it.bj; target = (unsigned)k; return true; }
            return false;
        case IT_R:
            if (q == 0) { c = vctr + FlowCtr::tile_ver + (k * NKB + it.bi) * FL_MAX_TN + it.bj; target = (unsigned)k; return true; }
            if (q == 1 && k >= 2) { c = vctr + FlowCtr::upd_done + (k - 2); target = n_upd_of(k - 2); return true; }
            return false;
        case IT_CS:
            if (q == 0) { c = vctr + FlowCtr::q_done + k; target = FL_NSRV; return true; }
            if (q == 1 && k >= 2) { c = vctr + FlowCtr::upd_done + (k - 2); target = n_upd_of(k - 2); return true; }
            if (q >= 2 && q - 2 < nk_of(k)) { c = vctr + FlowCtr::tile_ver + it.bi * FL_MAX_TN + k * NKB + (q - 2); target = (unsigned)k; return true; }
            return false;
        case IT_UPD:
            if (q == 0) { c = vctr + FlowCtr::cs_rows + k * FL_MAX_TN + it.bi; target = (unsigned)nk_of(k); return true; }
            if (q == 1) { c = vctr + FlowCtr::r_cols + k * FL_MAX_TN + it.bj; target = (unsigned)nk_of(k); return true; }
            if (q == 2) { c = vctr + FlowCtr::tile_ver + it.bi * FL_MAX_TN + it.bj; target = (unsigned)k; return true; }
            return false;
        }
        return false;
    };
    auto wait_deps = [&](const Item& it) {                 // blocking; lanes 0..7 of the engine's first warp
        if (ep.htid < 8) {
            volatile unsigned* c; unsigned target;
            if (dep_of(it, ep.htid, c, target)) flow_wait_ge(c, target, err, 30 + it.type);
            __threadfence();
        }
        half_sync(half);
    };
    auto deps_ready = [&](const Item& it) -> bool {        // non-blocking; called by the engine's first warp
        volatile unsigned* c; unsigned target;
        bool ok = true;
        if (ep.lane < 8 && dep_of(it, ep.lane, c, target)) ok = (*c >= target);
        ok = __all_sync(0xffffffffu, ok);
        if (ok) __threadfence();
        return ok;
    };
    auto pull = [&]() -> unsigned {                        // engine leader only
        unsigned spins = 0;
        while (P.sleep_coresident && *busy) {
            __nanosleep(2000);
            if (++spins > (1u << 22)) { *err = 20; break; }
        }
        return atomicAdd(ctr + FlowCtr::queue, 1u);
    };
    auto signal_done = [&](const Item& it) {               // all threads of the engine; their stores are issued
        half_sync(half);
        if (ep.htid == 0) {
            __threadfence();
            const int k = it.k;
            if (it.type == IT_FILL) atomicAdd(ctr + FlowCtr::fill_ver + it.bi * FL_MAX_TN + it.bj, 1u);
            else if (it.type == IT_R) atomicAdd(ctr + FlowCtr::r_cols + k * FL_MAX_TN + it.bj, 1u);
            else if (it.type == IT_CS) {
                atomicAdd(ctr + FlowCtr::cs_rows + k * FL_MAX_TN + it.bi, 1u);
                atomicAdd(ctr + FlowCtr::cs_done + k, 1u);
            } else {
                atomicAdd(ctr + FlowCtr::tile_ver + it.bi * FL_MAX_TN + it.bj, 1u);
                atomicAdd(ctr + FlowCtr::upd_done + k, 1u);
            }
        }
    };
#ifndef DAGMA_FLOW_RED
#define DAGMA_FLOW_RED 1      // 1: add the accumulators to the tile with red.global.add.f64 (measured faster), 0: load / add / store
#endif
    auto add2 = [](double* p, double v0, double v1) {      // the tile has one writer at a time (version counters)
#if DAGMA_FLOW_RED
        asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "d"(v0) : "memory");
        asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p + 1)), "d"(v1) : "memory");
#else
        double2 o = __ldcg(reinterpret_cast<const double2*>(p));
        o.x += v0;
        o.y += v1;
        *reinterpret_cast<double2*>(p) = o;
#endif
    };
    auto epilogue = [&](const Item& it) {
        const int k = it.k;
        if (it.type == IT_FILL) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = it.r0 + ep.row(i), c = it.c0 + ep.col(j);
                    if (r < d && c < d) {
                        double* p = P.gC + (size_t)r * d + c;
                        if (k == 0) *reinterpret_cast<double2*>(p) = make_double2(acc[i][j][0], acc[i][j][1]);
                        else add2(p, acc[i][j][0], acc[i][j][1]);
                    }
                }
        } else if (it.type == IT_UPD) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = it.r0 + ep.row(i), c = it.c0 + ep.col(j);
                    if (r < d && c < d) {
                        double* p = P.A + (size_t)r * d + c;
                        add2(p, acc[i][j][0], acc[i][j][1]);
                    }
                }
            FT_MAX(k, 8);
        } else if (it.type == IT_CS) {
            const int kn = kn_of(k), k0 = k * OB, cb = k * NKB;
            const bool inK = (it.bi >= cb) && (it.bi < cb + nk_of(k));
            double* CSk = P.CS[k & 1];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = it.r0 + ep.row(i), c = it.c0 + ep.col(j);
                    if (r < d && c < kn) {
                        double2 v = make_double2(-acc[i][j][0], -acc[i][j][1]);
                        if (inK) {
                            const double2 q = __ldcg(reinterpret_cast<const double2*>(it.Bm + (size_t)(r - k0) * kn + c));
                            v.x += q.x;
                            v.y += q.y;
                        }
                        *reinterpret_cast<double2*>(CSk + (size_t)r * kn + c) = v;
                    }
                }
        }
    };
    auto copy_r = [&](const Item& it) {
        const int k = it.k, kn = kn_of(k), k0 = k * OB, c0 = it.bj * NB;
        double* Rk = P.R[k & 1];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int rr = it.bi * NB + ep.row(i), c = c0 + ep.col(j);     // rr: row inside the strip
                if (rr < kn && c < d) {
                    double2 v = __ldcg(reinterpret_cast<const double2*>(P.A + (size_t)(k0 + rr) * d + c));
                    if (c == k0 + rr) v.x += 1.0;
                    if (c + 1 == k0 + rr) v.y += 1.0;
                    *reinterpret_cast<double2*>(Rk + (size_t)rr * d + c) = v;
                }
            }
    };
    __shared__ unsigned s_next[2], s_ready[2];
    half_sync(half);
    if (ep.htid == 0) s_next[half] = pull();
    half_sync(half);
    int t_cur = (int)s_next[half];
    Item cur = decode(t_cur);
    bool cur_ready = false, prefetched = false;
    while (cur.type != IT_NONE) {
        if (!cur_ready) wait_deps(cur);
        if (cur.type == IT_R) {
            copy_r(cur);
            signal_done(cur);
            half_sync(half);
            if (ep.htid == 0) s_next[half] = pull();
            half_sync(half);
            cur = decode((int)s_next[half]);
            cur_ready = prefetched = false;
            continue;
        }
        if (cur.type == IT_UPD) FT_MIN(cur.k, 12);
        // ---- a GEMM item.  Request its first slabs (unless the previous item already did), then look ahead while
        //      they are in flight: pull the next item, poll its dependencies once, remember only the index.
        half_sync(half);
        if (!prefetched)
            engine_prefetch(cur.Am, cur.lda, cur.Bm, cur.ldb, cur.r0, cur.c0, cur.rmax, cur.cmax, cur.kbeg, cur.kend, esm, ep.htid);
        if (ep.htid == 0) s_next[half] = pull();
        half_sync(half);
        const int t_nxt = (int)s_next[half];
        if (ep.htid < 32) {
            const Item peek = decode(t_nxt);
            const bool ok = (peek.type == IT_FILL || peek.type == IT_CS || peek.type == IT_UPD) && deps_ready(peek);
            if (ep.htid == 0) s_ready[half] = ok ? 1u : 0u;
        }
        zero_acc();
        engine_gemm(acc, cur.Am, cur.lda, cur.Bm, cur.ldb, cur.r0, cur.c0, cur.rmax, cur.cmax, cur.kbeg, cur.kend, esm, ep,
                    half, true);
        half_sync(half);                                   // every warp is done with the stages (and s_ready is visible)
        const Item nxt = decode(t_nxt);
        const bool nxt_ready = (s_ready[half] != 0u);
        if (nxt_ready)                                     // its first slabs fly during this item's epilogue
            engine_prefetch(nxt.Am, nxt.lda, nxt.Bm, nxt.ldb, nxt.r0, nxt.c0, nxt.rmax, nxt.cmax, nxt.kbeg, nxt.kend, esm, ep.htid);
        epilogue(cur);
        signal_done(cur);
        cur = nxt;
        cur_ready = prefetched = nxt_ready;
    }
    cp_async_wait<0>();
}

#ifdef DAGMA_OUTER_TRACE
}  // namespace dagma
extern "C" int dagma_debug_outer_trace(unsigned long long* out_host) {
    return (int)cudaMemcpyFromSymbol(out_host, dagma::g_outer_trace, sizeof(unsigned long long) * 16 * 40);
}
namespace dagma {
#endif

// per-block partial minima of the inverse (grid-stride; finished by inv_finish_kernel)
__global__ void __launch_bounds__(256) min_partial_kernel(const double* __restrict__ Minv, size_t total,
                                                          double* __restrict__ partial) {
    __shared__ double red[32];
    double mn = INFINITY;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x)
        mn = fmin(mn, Minv[e]);
    mn = block_min<256>(mn, red, threadIdx.x);
    if (threadIdx.x == 0) partial[blockIdx.x] = mn;
}

// after the sweep: log|det| from the fraction-free pivots (weights k mod 4 - 2, see stage_pivot_block),
// min entry from the per-block partial minima, info; optional outputs (scaled back)
constexpr int MIN_PARTIALS = 592;
__global__ void inv_finish_kernel(const double* __restrict__ partial_min, const double* __restrict__ pivots, int d,
                                  double s, double inv_scale, double log_scale, double* logabsdet, double* h,
                                  double* min_entry, int* info) {
    __shared__ double red[96];
    const int tid = threadIdx.x;
    double ld = 0.0, z1 = 0.0, z2 = 0.0;
    bool bad = false;
    const int np = (d + 3) & ~3;
    for (int k = tid; k < np; k += blockDim.x) {
        const double p = pivots[k];
        ld += (double)((k & 3) - 2) * log(fabs(p));
        bad |= !(p > 0.0);
    }
    double mn = INFINITY;
    for (int e = tid; e < MIN_PARTIALS; e += blockDim.x) mn = fmin(mn, partial_min[e]);
    block_sum3<1024>(ld, z1, z2, red, tid);
    mn = block_min<1024>(mn, red, tid) * inv_scale;
    const int anybad = __syncthreads_or(bad);
    if (tid == 0) {
        const double lad = ld + (double)d * log_scale;
        if (logabsdet) *logabsdet = lad;
        if (h) *h = -lad + (double)d * log(s);
        if (min_entry) *min_entry = mn;
        if (info) *info = anybad ? 1 : ((mn + 1e-16 < 0.0) ? 2 : 0);
    }
}

// out = scale * Minv  and/or  grad = (square ? 2 A^T-indexed : 1) * Minv^T
__global__ void inv_outputs_kernel(const double* __restrict__ Minv, const double* __restrict__ A, int lda, int d,
                                   double inv_scale, int square, double* minv_out, double* grad_out, int ldo) {
    __shared__ double tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    const int x = threadIdx.x, y0 = threadIdx.y;     // 32 x 8
    for (int y = y0; y < 32; y += 8) {
        const int r = by + y, c = bx + x;
        double v = (r < d && c < d) ? Minv[(size_t)r * d + c] * inv_scale : 0.0;
        tile[y][x] = v;
        if (minv_out && r < d && c < d) minv_out[(size_t)r * ldo + c] = v;
    }
    __syncthreads();
    if (grad_out) {
        for (int y = y0; y < 32; y += 8) {
            const int r = bx + y, c = by + x;       // transposed position
            if (r < d && c < d) {
                const double f = square ? 2.0 * A[(size_t)r * lda + c] : 1.0;
                grad_out[(size_t)r * ldo + c] = f * tile[x][y];
            }
        }
    }
}

// outer block of the two-level blocked inverse (d > OB); DAGMA_OUTER_BLOCK = 256 | 512 for A-B timing
static int outer_block() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_OUTER_BLOCK");
        v = e ? atoi(e) : 256;
        if (v != 256 && v != 512) v = 256;
    }
    return v;
}

struct LargeWs {                   // offsets in doubles into the caller's workspace
    size_t M, CS, Rbuf, CS2, Rbuf2, piv, Pbuf, Pbuf2, Pbuf3, Pbuf4, pmin, sync, flow, total;
    explicit LargeWs(int d) {
        const int OB = outer_block();
        const size_t dd = ((size_t)d * d + 1) & ~(size_t)1;        // keep every buffer 16-byte aligned
        const size_t strip = ((size_t)d * OB + 1) & ~(size_t)1;
        M = 0;
        CS = M + dd;
        Rbuf = CS + strip;
        CS2 = Rbuf + strip;                      // second set: the fused outer step writes the next CS / R
        Rbuf2 = CS2 + strip;
        piv = Rbuf2 + strip;
        Pbuf = piv + (((size_t)d + 64 + 1) & ~(size_t)1);
        Pbuf2 = Pbuf + (size_t)OB * OB;
        Pbuf3 = Pbuf2 + (size_t)OB * OB;
        Pbuf4 = Pbuf3 + (size_t)OB * OB;
        pmin = Pbuf4 + (size_t)OB * OB;
        sync = pmin + MIN_PARTIALS + 8;          // barrier counter, tile queue, error flag, per-SM busy flags
        flow = sync + (SYNC_STRIDE + 1) / 2 + 8;
        total = flow + (FlowCtr::total + 1) / 2;
    }
};
static size_t large_ws_bytes(int d) { return LargeWs(d).total * sizeof(double); }

// ---- small helpers of the two-level algorithm
// dst (rows x cols, ld = ldd) = src (ld = lds) [+ identity on the diagonal starting at column diag_col]
__global__ void copy_block_kernel(const double* __restrict__ src, int lds, double* __restrict__ dst, int ldd,
                                  int rows, int cols, int diag_col, double diag_add) {
    const size_t total = (size_t)rows * cols;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols), c = (int)(e - (size_t)r * cols);
        double v = src[(size_t)r * lds + c];
        if (c - diag_col == r) v += diag_add;
        dst[(size_t)r * ldd + c] = v;
    }
}
// one launch for the two small fix-ups of an outer step:  CS[K,:] += Q  and  R = A[K,:] + E_K^T
__global__ void outer_prep_kernel(const double* __restrict__ Q, double* __restrict__ CSk, int kn,
                                  const double* __restrict__ Arows, int d, int k0, double* __restrict__ R) {
    const size_t nq = (Q != nullptr) ? (size_t)kn * kn : 0, total = nq + (size_t)kn * d;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        if (e < nq) {
            CSk[e] += Q[e];
        } else {
            const size_t f = e - nq;
            const int r = (int)(f / d), c = (int)(f - (size_t)r * d);
            double v = Arows[f];
            if (c - k0 == r) v += 1.0;
            R[f] = v;
        }
    }
}

// single-level block Gauss-Jordan (block 64) of the dense n x n matrix in `buf0` (ld = n); `buf1` is the
// ping-pong partner.  Returns (through *result) the buffer that holds the inverse; piv: n (+3) pivots.
static int gj_nb64(cudaStream_t stream, double* buf0, double* buf1, int n, double* piv, double** result) {
    static bool attr = false;
    if (!attr) {
        DAGMA_CUDA_OK(cudaFuncSetAttribute(inv_tile_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)TILE_STEP_SMEM_BYTES));
        attr = true;
    }
    const int nblk = (n + NB - 1) / NB;
    double *in = buf0, *out = buf1;
    for (int kb = 0; kb < nblk; ++kb) {
        TileStepArgs P{in, out, n, kb, piv};
        inv_tile_step_kernel<<<dim3(nblk, nblk), DM_NT, TILE_STEP_SMEM_BYTES, stream>>>(P);
        DAGMA_CUDA_OK(cudaGetLastError());
        double* t = in;
        in = out;
        out = t;
    }
    *result = in;
    return 0;
}

// side stream + events for the look-ahead of the two-level algorithm (one set per process: the library
// drives one GPU stream per process, SURVEY 8b3; capturable -- the fork / join pattern below is what
// CUDA-graph stream capture records as parallel branches)
struct LookAhead {
    cudaStream_t side = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static int lookahead_get(LookAhead** out) {
    static LookAhead la;
    if (!la.side) {
        // highest priority: the panel chain is short and serial, the d x d update it overlaps is wide
        int lo = 0, hi = 0;
        DAGMA_CUDA_OK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        DAGMA_CUDA_OK(cudaStreamCreateWithPriority(&la.side, cudaStreamNonBlocking, hi));
        DAGMA_CUDA_OK(cudaEventCreateWithFlags(&la.fork, cudaEventDisableTiming));
        DAGMA_CUDA_OK(cudaEventCreateWithFlags(&la.join, cudaEventDisableTiming));
    }
    *out = &la;
    return 0;
}

// DAGMA_OUTER_SLEEP (A-B timing): 1 (default) = the worker CTA that shares an SM with a CTA of the look-ahead chain
// sleeps while the chain runs (the chain has its SMs to itself), 0 = it keeps pulling update tiles
static int outer_sleep() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_OUTER_SLEEP");
        v = e ? atoi(e) : 1;
    }
    return v;
}

// DAGMA_FIRST_BLOCK (A-B timing): 1 = the first pivot block is inverted and its CS / R strips are formed by a step of
// outer_step_kernel with nothing to apply (one launch), 0 (default) = by copy + 4 tile-step launches + a GEMM + a prep
// kernel (seven launches).  Measured equal at d = 2000 (inverse 0.960 vs 0.957 ms): the first block is bound by its
// own serial pivot chain either way, so the proven sequence stays the default.
static bool first_block_fused() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_FIRST_BLOCK");
        v = e ? atoi(e) : 0;
    }
    return v != 0;
}

// DAGMA_LOOKAHEAD (A-B timing): 1 = one persistent kernel per outer step with the look-ahead inside (default, even d),
// 2 = the whole inversion as ONE dependency-driven kernel (flow_inverse_kernel; can carry a rider GEMM) -- measured
//     on par for the inverse alone (1.01 vs 0.97 ms at d = 2000) and for inverse + cov@W (1.58 vs 1.52 ms): its
//     engines reach the same ~65 % of the DMMA pipe as the per-step kernels, so it stays opt-in,
// 0 = plain GEMM update + chain of small kernels on a high-priority side stream
// DAGMA_CS_HEAD (A-B timing): 0 (default) = the previous step forms the CS strip as its tail (on the serial chain);
// 1 = every outer step forms its own CS strip at its start, rows K' first (the look-ahead chain waits only for those),
// one CTA per SM.  Measured at d = 2000 (B200, round 2): 0.896 ms against 0.871 ms -- a 64 x 64 x 256 item of two
// engines is bound by its 8 dependent slab round trips (17 us alone on an SM, as in the tail), so the chain starts
// 17 us late and the overlap it buys (the tail leaves the critical path) does not pay for it.
// DAGMA_PDL (A-B timing): 1 = consecutive outer steps are launched with programmatic stream serialization (the next
// step's prologue overlaps the tail of the current one), 0 = plain stream order
static int pdl_mode() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_PDL");
        v = e ? atoi(e) : DAGMA_PDL_DEFAULT;
    }
    return v;
}

static int cs_head_mode() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_CS_HEAD");
        v = e ? atoi(e) : 0;
    }
    return v != 0 ? 1 : 0;
}
static int lookahead_mode() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_LOOKAHEAD");
        v = e ? atoi(e) : 1;
    }
    return v;
}

// DAGMA_TMA: which slab pipelines are fed by TMA (cp.async.bulk.tensor + mbarrier pipeline, gemm_tma.cuh) instead
// of per-thread cp.async.  Bit 0: the update tiles of the outer step of the two-level inverse; bit 1: the
// stand-alone GEMM whenever its operands qualify; bit 2: the stand-alone GEMM where it was measured to win
// (scripts/perf_tma.py on B200, TFLOP/s):            2000^3    4096^3    2000 x 2000 x 256 (+= C)
//     cp.async 64 x 64, four CTAs per SM               28.9      32.2        25.9
//     TMA 128 x 128, balanced k-slab ranges            32.4      35.5         --      (cuBLAS: 32.7 / 35.4)
//     TMA 128 x 128, tile queue                        28.8      35.2        22.4
// i.e. the balanced schedule once the output has a 128 x 128 tile per SM and K is long, the queue only for
// large outputs; short-K updates stay on cp.async.  Unset = bits 0 and 2.  0 = cp.async everywhere.
static int tma_mode() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_TMA");
        v = e ? atoi(e) : DAGMA_TMA_DEFAULT;
        if (v && !tm_encode_fn()) v = 0;
    }
    return v;
}
// schedule / tile of the stand-alone TMA GEMM (bits as in gemm_tma_launch: 1 queue, 2 balanced, 4 = 128 x 128
// tiles), or -1: stay on the cp.async kernel.  DAGMA_TMA_GEMM_MODE forces a mode.
static int gemm_tma_sched(int M, int N, int K, double beta, int epi) {
    static int forced = -2;
    if (forced == -2) {
        const char* e = getenv("DAGMA_TMA_GEMM_MODE");
        forced = e ? atoi(e) : -1;
    }
    const int m = tma_mode();
    if (!(m & 6)) return -1;
    if (forced >= 0) return forced;
    const long long t128 = (long long)((M + 127) / 128) * ((N + 127) / 128);
    const bool plain = (beta == 0.0 && epi == EPI_NONE);
    if (m & 2) return plain ? (4 | 2) : (4 | 1);
    if (plain && t128 >= 148 && K >= 512) return 4 | 2;
    if (t128 >= 4 * 148 && K >= 1024) return 4 | 1;
    return -1;
}

// two-level block Gauss-Jordan, outer block OB = 256: per outer block K
//   Q  = P^{-1}, P = A[K,K]          (single-level sweep on a copy of the 256 x 256 block)
//   CS = -A[:,K] Q, CS[K,:] += Q      (= -(A[:,K] - E_K) Q : the "- I" of the publish identity)
//   R  = A[K,:] + E_K^T               (row copy: the GEMM below overwrites those rows)
//   A += CS R                         (one d x d x 256 DMMA GEMM, accumulators initialised from A)
// Look-ahead: the next pivot block P' = A[K',K'] + CS[K',:] R[:,K'] is formed first (a 256^3 GEMM) and
// inverted on a side stream while the main stream runs the d x d update, so the serial panel chain
// (4 sweeps + 4 small GEMMs) is off the critical path.
struct RiderGemm {        // C = A B (all d x d, ld = d) carried out by the flow kernel beside the inversion; C == nullptr: none
    const double* A = nullptr;
    const double* B = nullptr;
    double* C = nullptr;
};
// can the rider of this size be carried by the flow kernel?  (otherwise the caller runs a plain GEMM)
static bool flow_supported(int d) {
    const int OB = outer_block();
    return lookahead_mode() == 2 && (d % 2 == 0) && OB == 256 && d > OB && (d + OB - 1) / OB <= FL_MAX_OB &&
           (d + NB - 1) / NB <= FL_MAX_TN;
}
static int flow_sleep_mode(bool rider) {     // DAGMA_FLOW_SLEEP (A-B timing): default 1 without a rider, 0 with one
    static int v = -2;
    if (v == -2) {
        const char* e = getenv("DAGMA_FLOW_SLEEP");
        v = e ? atoi(e) : -1;
    }
    return v >= 0 ? v : (rider ? 0 : 1);
}

static int gj_inplace_two_level(cudaStream_t stream, double* Mw, int d, double* ws, const RiderGemm& rider) {
    const int OB = outer_block();
    const LargeWs L(d);
    double *CS = ws + L.CS, *Rbuf = ws + L.Rbuf, *piv = ws + L.piv, *Pbuf = ws + L.Pbuf, *Pbuf2 = ws + L.Pbuf2;
    double* Q = nullptr;             // where the inverse of the current pivot block lives (Pbuf or Pbuf2)
    LookAhead* la = nullptr;
    int rc = lookahead_get(&la);
    if (rc) return rc;
    const int nob = (d + OB - 1) / OB;
    if (flow_supported(d)) {
        // the whole inversion as one dependency-driven kernel
        static bool attr = false;
        if (!attr) {
            DAGMA_CUDA_OK(cudaFuncSetAttribute(flow_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)OUTER_SMEM_BYTES));
            DAGMA_CUDA_OK(cudaFuncSetAttribute(flow_inverse_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                               cudaSharedmemCarveoutMaxShared));
            attr = true;
        }
        int sms = 0, dev = 0;
        DAGMA_CUDA_OK(cudaGetDevice(&dev));
        DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        unsigned* ctr = reinterpret_cast<unsigned*>(ws + L.flow);
        DAGMA_CUDA_OK(cudaMemsetAsync(ctr, 0, FlowCtr::total * sizeof(unsigned), stream));
        FlowArgs FA{};
        FA.A = Mw; FA.d = d; FA.nob = nob; FA.tn = (d + NB - 1) / NB;
        FA.CS[0] = CS; FA.CS[1] = ws + L.CS2; FA.R[0] = Rbuf; FA.R[1] = ws + L.Rbuf2;
        FA.X[0] = Pbuf; FA.Y[0] = Pbuf2; FA.X[1] = ws + L.Pbuf3; FA.Y[1] = ws + L.Pbuf4;
        FA.pivots = piv; FA.ctr = ctr;
        FA.gA = rider.A; FA.gB = rider.B; FA.gC = rider.C;
        FA.sleep_coresident = flow_sleep_mode(rider.C != nullptr);
        FA.rider_only = (rider.C != nullptr && getenv("DAGMA_FLOW_RIDER_ONLY") != nullptr) ? 1 : 0;
        FA.fill_k = OB;
        if (FA.rider_only && getenv("DAGMA_FLOW_FILL_K")) {          // timing experiment: longer rider items
            FA.fill_k = atoi(getenv("DAGMA_FLOW_FILL_K"));
            FA.nob = (d + FA.fill_k - 1) / FA.fill_k;
        }
        const int n_fill = rider.C ? FA.tn * FA.tn : 0;
        FA.item_base[0] = 0;
        for (int k = 0; k < FA.nob; ++k) {
            const int kn = (d - k * OB) < OB ? (d - k * OB) : OB, nk = (kn + NB - 1) / NB;
            const int kn1 = (k + 1 < nob) ? ((d - (k + 1) * OB) < OB ? (d - (k + 1) * OB) : OB) : 0, nk1 = (kn1 + NB - 1) / NB;
            FA.item_base[k + 1] = FA.item_base[k] + n_fill + (FA.rider_only ? 0 : nk * FA.tn + (FA.tn - nk1) * nk + (FA.tn * FA.tn - nk1 * nk1));
        }
#ifdef DAGMA_OUTER_TRACE
        flow_trace_begin_kernel<<<1, 1, 0, stream>>>();
#endif
        const int grid = 2 * sms > FL_NSRV ? 2 * sms : FL_NSRV;
        flow_inverse_kernel<<<grid, DM_NT, OUTER_SMEM_BYTES, stream>>>(FA);
        DAGMA_CUDA_OK(cudaGetLastError());
        return 0;
    }
    const bool fused_first = (lookahead_mode() >= 1) && (d % 2 == 0) && first_block_fused();
    if (!fused_first) {   // first pivot block by the plain kernels
        const int kn = d < OB ? d : OB;
        copy_block_kernel<<<64, 256, 0, stream>>>(Mw, d, Pbuf, kn, kn, kn, 0, 0.0);
        DAGMA_CUDA_OK(cudaGetLastError());
        rc = gj_nb64(stream, Pbuf, Pbuf2, kn, piv, &Q);
        if (rc) return rc;
    }
    const bool fused = (lookahead_mode() >= 1) && (d % 2 == 0);
    unsigned* sync_base = reinterpret_cast<unsigned*>(ws + L.sync);
    unsigned* flow_words = reinterpret_cast<unsigned*>(ws + L.flow);
    if (fused) {
        static bool attr = false;
        if (!attr) {
            DAGMA_CUDA_OK(cudaFuncSetAttribute(outer_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)OUTER_SMEM_BYTES));
            DAGMA_CUDA_OK(cudaFuncSetAttribute(outer_step_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                               cudaSharedmemCarveoutMaxShared));
            attr = true;
        }
        int sms = 0, dev = 0;
        DAGMA_CUDA_OK(cudaGetDevice(&dev));
        DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        // CS / R of the first block: by the plain kernels (default), or by a step "-1" of the same persistent kernel
        // with nothing to apply (kn = 0) -- its look-ahead CTAs invert A[K0,K0] in place of the 4 tile-step launches,
        // its CS' / R' items replace the first CS GEMM and the prep kernel; every later pair is produced by the
        // previous step
        double *CSa = CS, *Ra = Rbuf, *CSb = ws + L.CS2, *Rb = ws + L.Rbuf2;
        const int cs_head = cs_head_mode();
        if (!fused_first) {
            const int kn = d < OB ? d : OB;
            if (!cs_head) {
                rc = gemm_launch(stream, 0, d, kn, kn, -1.0, Mw, d, Q, kn, 0.0, CSa, kn, EPI_NONE, nullptr, 0);
                if (rc) return rc;
            }
            outer_prep_kernel<<<296, 256, 0, stream>>>(cs_head ? nullptr : Q, CSa, kn, Mw, d, 0, Ra);
            DAGMA_CUDA_OK(cudaGetLastError());
        }
        const double* Qc = Q;                              // inverse of the current pivot block (cs_head)
        for (int ob = fused_first ? -1 : 0; ob < nob; ++ob) {
            const bool pre = ob < 0;                       // the step in front of the first block
            const int k0 = pre ? 0 : ob * OB, kn = pre ? 0 : ((d - k0) < OB ? (d - k0) : OB);
            const bool more = ob + 1 < nob;
            const int k1 = pre ? 0 : k0 + OB, kn1 = more ? ((d - k1) < OB ? (d - k1) : OB) : 0;
            const int nblk1 = (kn1 + NB - 1) / NB;
            // cs_head: the step reads Qc while its look-ahead CTAs ping-pong the next block: two buffer pairs, in turn
            const bool pair1 = cs_head && (((ob + 1) & 1) != 0);
            double *bufA = pair1 ? ws + L.Pbuf3 : Pbuf, *bufB = pair1 ? ws + L.Pbuf4 : Pbuf2;
            double* Qn = (nblk1 & 1) ? bufB : bufA;
            // every outer step has its own zeroed sync block (one memset for all of them: no memset node
            // between two step kernels); beyond the space of the flow counters: one memset per step
            unsigned* sync_words = sync_base;
            const int slot = ob + 1;                       // slot 0: the step in front of the first block
            if ((slot + 1) * SYNC_STRIDE <= FlowCtr::total) {
                if (ob == (fused_first ? -1 : 0)) {
                    const int nfit = FlowCtr::total / SYNC_STRIDE < nob + 1 ? FlowCtr::total / SYNC_STRIDE : nob + 1;
                    DAGMA_CUDA_OK(cudaMemsetAsync(flow_words, 0, (size_t)nfit * SYNC_STRIDE * sizeof(unsigned), stream));
                }
                sync_words = flow_words + slot * SYNC_STRIDE;
            } else {
                DAGMA_CUDA_OK(cudaMemsetAsync(sync_words, 0, SYNC_STRIDE * sizeof(unsigned), stream));
            }
#ifdef DAGMA_OUTER_TRACE
            outer_trace_begin_kernel<<<1, 1, 0, stream>>>(ob < 0 ? 15 : ob);
#endif
            OuterArgs OA{Mw, d, CSa, Ra, kn, CSb, Rb, k1, kn1, Qn, sync_words, reinterpret_cast<int*>(sync_words + 8),
                         nblk1 * nblk1,
                         ServerArgs{bufA, bufB, kn1, nblk1, piv + k1, sync_words, reinterpret_cast<int*>(sync_words + 2)},
                         pre ? 0 : (tma_mode() & 1), outer_sleep(),
                         cs_head, CSa, Qc, k0, sync_words + 8 + 2 * SM_SLOTS};
            Qc = Qn;
            CUtensorMap mapCS, mapR;
            memset(&mapCS, 0, sizeof(mapCS));
            memset(&mapR, 0, sizeof(mapR));
            if (OA.use_tma) {
                rc = tm_make_a_map(&mapCS, CSa, d, kn, kn);
                if (rc) return rc;
                rc = tm_make_b_map(&mapR, Ra, kn, d, d);
                if (rc) return rc;
            }
            if (pdl_mode()) {
                cudaLaunchConfig_t cfg{};
                cfg.gridDim = dim3(2 * sms);
                cfg.blockDim = dim3(DM_NT);
                cfg.dynamicSmemBytes = OUTER_SMEM_BYTES;
                cfg.stream = stream;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                at[0].val.programmaticStreamSerializationAllowed = 1;
                cfg.attrs = at;
                cfg.numAttrs = 1;
                DAGMA_CUDA_OK(cudaLaunchKernelEx(&cfg, outer_step_kernel, OA, mapCS, mapR));
            } else {
                outer_step_kernel<<<2 * sms, DM_NT, OUTER_SMEM_BYTES, stream>>>(OA, mapCS, mapR);
                DAGMA_CUDA_OK(cudaGetLastError());
            }
            double* t = CSa; CSa = CSb; CSb = t;
            t = Ra; Ra = Rb; Rb = t;
        }
        return 0;
    }
    for (int ob = 0; ob < nob; ++ob) {
        const int k0 = ob * OB, kn = (d - k0) < OB ? (d - k0) : OB;
        rc = gemm_launch(stream, 0, d, kn, kn, -1.0, Mw + k0, d, Q, kn, 0.0, CS, kn, EPI_NONE, nullptr, 0);
        if (rc) return rc;
        outer_prep_kernel<<<296, 256, 0, stream>>>(Q, CS + (size_t)k0 * kn, kn, Mw + (size_t)k0 * d, d, k0, Rbuf);
        DAGMA_CUDA_OK(cudaGetLastError());
        const bool more = ob + 1 < nob;
        const int k1 = k0 + OB, kn1 = more ? ((d - k1) < OB ? (d - k1) : OB) : 0;
        if (more) {   // copy of the next pivot block: the d x d update below overwrites A[K',K'] in place
            copy_block_kernel<<<64, 256, 0, stream>>>(Mw + (size_t)k1 * d + k1, d, Pbuf, kn1, kn1, kn1, 0, 0.0);
            DAGMA_CUDA_OK(cudaGetLastError());
        }
        if (more) {   // side stream: next pivot block P' = A[K',K'] + CS[K',:] R[:,K'], then its inversion
            DAGMA_CUDA_OK(cudaEventRecord(la->fork, stream));
            DAGMA_CUDA_OK(cudaStreamWaitEvent(la->side, la->fork, 0));
            rc = gemm_launch(la->side, 0, kn1, kn1, kn, 1.0, CS + (size_t)k1 * kn, kn, Rbuf + k1, d, 1.0, Pbuf, kn1,
                             EPI_NONE, nullptr, 0);
            if (rc) return rc;
            rc = gj_nb64(la->side, Pbuf, Pbuf2, kn1, piv + k1, &Q);
            if (rc) return rc;
            DAGMA_CUDA_OK(cudaEventRecord(la->join, la->side));
        }
        rc = gemm_launch(stream, 0, d, d, kn, 1.0, CS, kn, Rbuf, d, 1.0, Mw, d, EPI_NONE, nullptr, 0);
        if (rc) return rc;
        if (more) DAGMA_CUDA_OK(cudaStreamWaitEvent(stream, la->join, 0));
    }
    return 0;
}

// one problem; ws layout: see large_ws_bytes
static int logdet_inv_blocked(cudaStream_t stream, int d, double s, const double* a_dev, int lda, int square,
                              double* logabsdet, double* h, double* minv, double* grad, int ldo,
                              double* min_entry, int* info, double* ws, const RiderGemm& rider = RiderGemm()) {
    double scale = 1.0;
    if (s > 0.0 && isfinite(s)) {
        int e = 0;
        const double f = frexp(s, &e);
        if (f == 0.5) --e;
        scale = ldexp(1.0, e);
    }
    const double inv_scale = 1.0 / scale;
    // work in place in the caller's minv buffer when it is dense (ldo == d), else in ws
    const LargeWs L(d);
    double* Mw = (minv != nullptr && ldo == d) ? minv : ws + L.M;
    double* piv = ws + L.piv;
    build_m_kernel<<<592, 256, 0, stream>>>(a_dev, lda, Mw, d, s, inv_scale, square);
    DAGMA_CUDA_OK(cudaGetLastError());
    int rc = 0;
    if (d > outer_block()) {
        rc = gj_inplace_two_level(stream, Mw, d, ws, rider);
    } else {                                   // ping-pong between Mw and the CS strip (d * OB >= d * d here)
        double* res = nullptr;
        rc = gj_nb64(stream, Mw, ws + L.CS, d, piv, &res);
        if (rc == 0 && res != Mw)
            DAGMA_CUDA_OK(cudaMemcpyAsync(Mw, res, (size_t)d * d * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    }
    if (rc) return rc;
    min_partial_kernel<<<MIN_PARTIALS, 256, 0, stream>>>(Mw, (size_t)d * d, ws + L.pmin);
    DAGMA_CUDA_OK(cudaGetLastError());
    inv_finish_kernel<<<1, 1024, 0, stream>>>(ws + L.pmin, piv, d, s, inv_scale, log(scale), logabsdet, h, min_entry, info);
    DAGMA_CUDA_OK(cudaGetLastError());
    if (grad != nullptr || (minv != nullptr && (minv != Mw || inv_scale != 1.0))) {
        dim3 grid((d + 31) / 32, (d + 31) / 32);
        // note: when minv == Mw and a rescale is needed the tile kernel rewrites it in place
        inv_outputs_kernel<<<grid, dim3(32, 8), 0, stream>>>(Mw, a_dev, lda, d, inv_scale, square,
                                                             (minv == Mw && inv_scale == 1.0) ? nullptr : minv, grad, ldo);
        DAGMA_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

int logdet_inv_large(cudaStream_t stream, int batch, int d, double s, const double* a_dev, int lda, int square,
                     double* logabsdet, double* h, double* minv, double* grad, int ldo, double* min_entry,
                     int* info) {
    double* ws = nullptr;
    DAGMA_CUDA_OK(cudaMallocAsync((void**)&ws, large_ws_bytes(d), stream));
    int rc = 0;
    for (int b = 0; b < batch && rc == 0; ++b) {
        rc = logdet_inv_blocked(stream, d, s, a_dev + (size_t)b * d * lda, lda, square,
                                logabsdet ? logabsdet + b : nullptr, h ? h + b : nullptr,
                                minv ? minv + (size_t)b * d * ldo : nullptr, grad ? grad + (size_t)b * d * ldo : nullptr,
                                ldo, min_entry ? min_entry + b : nullptr, info ? info + b : nullptr, ws);
    }
    cudaFreeAsync(ws, stream);
    return rc;
}

// ------------------------------------------------------------------ iteration state (LinState: lin_state.h)
// end of an inner iteration: latch `halted` when the inverse was infeasible, else advance beta^it and the counter
__device__ __forceinline__ void linear_advance(LinState* st) {
    if (st->halted != 0) return;
    if (st->info != 0) {
        st->halted = 1;
        return;
    }
    double p1h = st->p1_hi, p1l = st->p1_lo, p2h = st->p2_hi, p2l = st->p2_lo;
    dd_mul(p1h, p1l, st->beta1);
    dd_mul(p2h, p2l, st->beta2);
    st->p1_hi = p1h; st->p1_lo = p1l; st->p2_hi = p2h; st->p2_lo = p2l;
    st->it += 1;
}
// called by thread 0 of every block when the block is done with the state block: the LAST block to get here has seen
// every other block finish (so nobody reads the state any more) and advances it -- no separate 1-thread launch
__device__ __forceinline__ void linear_advance_by_last_block(LinState* st, int blocks) {
    __threadfence();
    if (atomicAdd(&st->pad, 1) == blocks - 1) {
        st->pad = 0;
        linear_advance(st);
    }
}

// Gobj, Adam, step, masks for one inner iteration (linear.py:248, 158-162, 275-276).
// No-op (and latches `halted`) when the inverse of this iteration was infeasible.
__global__ void __launch_bounds__(256) linear_update_kernel(LinState* st, int d, double* __restrict__ W,
                                                             const double* __restrict__ Minv,
                                                             const double* __restrict__ T,
                                                             const double* __restrict__ cov, double* __restrict__ m,
                                                             double* __restrict__ v, const uint8_t* mask_exc,
                                                             const uint8_t* mask_inc, const double* __restrict__ extraT,
                                                             double extra_scale) {
    __shared__ double tile[32][33];
    __shared__ double tile2[32][33];
    const bool stop = (st->halted != 0) || (st->info != 0);
    const bool leader = (threadIdx.x == 0 && threadIdx.y == 0);
    const int nblocks = gridDim.x * gridDim.y;
    if (stop) {                              // uniform over the grid: only the latch / advance remains
        if (leader) linear_advance_by_last_block(st, nblocks);
        return;
    }
    const double mu = st->mu, lr = st->lr, lambda1 = st->lambda1, b1 = st->beta1, b2 = st->beta2;
    double p1h = st->p1_hi, p1l = st->p1_lo, p2h = st->p2_hi, p2l = st->p2_lo;
    dd_mul(p1h, p1l, b1);
    dd_mul(p2h, p2l, b2);
    const double c1 = 1.0 / ((1.0 - p1h) - p1l), c2 = 1.0 / ((1.0 - p2h) - p2l);
    const double gscale = st->gscale;
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    const int x = threadIdx.x, y0 = threadIdx.y;
    // tile of Minv at the transposed block position
    for (int y = y0; y < 32; y += 8) {
        const int r = bx + y, c = by + x;
        tile[y][x] = (r < d && c < d) ? Minv[(size_t)r * d + c] : 0.0;
        if (extraT) tile2[y][x] = (r < d && c < d) ? extraT[(size_t)r * d + c] : 0.0;
    }
    __syncthreads();
    for (int y = y0; y < 32; y += 8) {
        const int r = by + y, c = bx + x;
        if (r >= d || c >= d) continue;
        const size_t e = (size_t)r * d + c;
        const double w = W[e];
        const double minvT = tile[x][y];
        const double sg = (w > 0.0) ? 1.0 : ((w < 0.0) ? -1.0 : 0.0);
        const double gsc = fma(gscale, T[e], -cov[e]);          // l2: cov W - cov ; logistic: X^T sigma / n - cov
        double go = fma(mu, gsc, mu * lambda1 * sg);
        go = fma(2.0 * w, minvT + 1e-16, go);
        if (mask_inc && mask_inc[e]) go = fma(-2.0 * mu * lambda1, sg, go);
        if (extraT) go = fma(extra_scale * (2.0 * w), tile2[x][y], go);      // + weight * 2 W o G^T (trek regulariser)
        const double mn = fma(m[e], b1, (1.0 - b1) * go);
        const double vn = fma(v[e], b2, (1.0 - b2) * (go * go));
        m[e] = mn;
        v[e] = vn;
        const double dir = fast_div(mn * c1, fast_sqrt_nonneg(vn * c2) + 1e-8);
        double wn = w - lr * dir;
        if (mask_exc && mask_exc[e]) wn = 0.0;
        W[e] = wn;
    }
    __syncthreads();                                         // no thread of this block uses the state block any more
    if (leader) linear_advance_by_last_block(st, nblocks);
}


// W += sign * lr * dir(m, v, it)   (back-tracking, linear.py:235, 239)
__global__ void linear_apply_dir_kernel(const LinState* st, int d, double* __restrict__ W,
                                        const double* __restrict__ m, const double* __restrict__ v, double sign) {
    const double c1 = 1.0 / ((1.0 - st->p1_hi) - st->p1_lo), c2 = 1.0 / ((1.0 - st->p2_hi) - st->p2_lo);
    const double scale = sign * st->lr;
    const size_t total = (size_t)d * d;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const double dir = fast_div(m[e] * c1, fast_sqrt_nonneg(v[e] * c2) + 1e-8);
        W[e] = __dadd_rn(W[e], __dmul_rn(scale, dir));
    }
}

// l2: score_acc = 1/2 sum (I - W) o (cov - T), l1_acc = sum |W|   (T = cov W)
// logistic: only l1_acc (the loss comes from logistic_loss_kernel)
__global__ void __launch_bounds__(1024) linear_objective_kernel(LinState* st, int d, const double* __restrict__ W,
                                                                 const double* __restrict__ T,
                                                                 const double* __restrict__ cov, int l2) {
    __shared__ double red[96];
    const int tid = threadIdx.x;
    double sc = 0.0, l1 = 0.0, z = 0.0;
    const size_t total = (size_t)d * d;
    for (size_t e = tid; e < total; e += blockDim.x) {
        const int r = (int)(e / d), c = (int)(e - (size_t)r * d);
        const double w = W[e];
        l1 += fabs(w);
        if (l2) sc = fma(((r == c) ? 1.0 : 0.0) - w, cov[e] - T[e], sc);
    }
    block_sum3<1024>(sc, l1, z, red, tid);
    if (tid == 0) {
        st->score_acc = 0.5 * sc;
        st->l1_acc = l1;
    }
}

// The same reductions over row blocks on many CTAs (a 32 MB pass at d = 2000: 2.6 ms on one CTA, HBM-bound on a grid):
// CTA b sums the rows b, b + grid, ... (no 64-bit divide), writes its pair of partial sums, and the CTA that takes the
// last ticket adds the partials in CTA order -- fixed order, so the result does not depend on the schedule.
// ws: [0] ticket (unsigned, zero on entry, re-armed on exit), [1 + 2 b], [2 + 2 b] partials.
__global__ void __launch_bounds__(256) linear_objective_mb_kernel(LinState* st, int d, const double* __restrict__ W,
                                                                  const double* __restrict__ T,
                                                                  const double* __restrict__ cov, int l2,
                                                                  double* __restrict__ ws) {
    __shared__ double red[96];
    __shared__ unsigned s_last;
    const int tid = threadIdx.x;
    double sc = 0.0, l1 = 0.0, z = 0.0;
    for (int r = blockIdx.x; r < d; r += gridDim.x) {
        const size_t row = (size_t)r * d;
        for (int c = tid; c < d; c += 256) {
            const double w = W[row + c];
            l1 += fabs(w);
            if (l2) sc = fma(((r == c) ? 1.0 : 0.0) - w, cov[row + c] - T[row + c], sc);
        }
    }
    block_sum3<256>(sc, l1, z, red, tid);
    if (tid == 0) {
        ws[1 + 2 * blockIdx.x] = sc;
        ws[2 + 2 * blockIdx.x] = l1;
        __threadfence();
        s_last = (atomicAdd(reinterpret_cast<unsigned*>(ws), 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (tid == 0) {
        double a = 0.0, b = 0.0;
        for (unsigned k = 0; k < gridDim.x; ++k) {
            a += __ldcg(ws + 1 + 2 * k);
            b += __ldcg(ws + 2 + 2 * k);
        }
        st->score_acc = 0.5 * a;
        st->l1_acc = b;
        *reinterpret_cast<unsigned*>(ws) = 0u;
    }
}

// partial[b] = sum over a slice of (logaddexp(0, R) - X o R)   (linear.py:91); finished by a 1-block pass
__global__ void __launch_bounds__(256) logistic_loss_kernel(const double* __restrict__ X, const double* __restrict__ R,
                                                             size_t total, double* partial) {
    __shared__ double red[96];
    double acc = 0.0, z1 = 0.0, z2 = 0.0;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const double r = R[e];
        const double sp = fmax(r, 0.0) + log1p(exp(-fabs(r)));
        acc += sp - X[e] * r;
    }
    block_sum3<256>(acc, z1, z2, red, threadIdx.x);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
__global__ void sum_partials_kernel(const double* partial, int n, double scale, double* out) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += partial[i];
    *out = s * scale;
}

// the reference's stand-alone Adam step (linear.py:158-163): updates m, v, writes the direction
__global__ void adam_direction_kernel(size_t n, const double* __restrict__ g, double* __restrict__ m,
                                      double* __restrict__ v, double b1, double b2, double bc1, double bc2,
                                      double* __restrict__ out) {
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        const double go = g[e];
        const double mn = m[e] * b1 + (1.0 - b1) * go;
        const double vn = v[e] * b2 + (1.0 - b2) * (go * go);
        m[e] = mn;
        v[e] = vn;
        out[e] = (mn / bc1) / (sqrt(vn / bc2) + 1e-8);
    }
}

}  // namespace dagma

using namespace dagma;

// =============================================================================== C ABI
extern "C" int dagma_adam_direction_f64(dagma_stream_t stream, size_t n, const double* grad_dev, double* m_dev,
                                        double* v_dev, double beta1, double beta2, double bias1, double bias2,
                                        double* out_dev) {
    DAGMA_REQUIRE(grad_dev && m_dev && v_dev && out_dev, "null pointer");
    const int blocks = (int)((n + 255) / 256);
    adam_direction_kernel<<<blocks < 1184 ? blocks : 1184, 256, 0, (cudaStream_t)stream>>>(n, grad_dev, m_dev, v_dev, beta1,
                                                                                         beta2, bias1, bias2, out_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" size_t dagma_large_workspace_bytes(int d) { return large_ws_bytes(d); }

extern "C" int dagma_gemm_f64(dagma_stream_t stream, int trans_a, int M, int N, int K, double alpha,
                              const double* a_dev, int lda, const double* b_dev, int ldb, double beta,
                              double* c_dev, int ldc, int epilogue, double* ws_dev, size_t ws_bytes) {
    DAGMA_REQUIRE(a_dev && b_dev && c_dev, "null pointer");
    DAGMA_REQUIRE(K >= 0 && lda >= 1 && lda >= (trans_a ? M : K) && ldb >= N && ldc >= N, "bad leading dimension");
    // K = 0: C = beta C (then the epilogue) whatever alpha is -- alpha times the empty sum would be NaN for alpha = inf
    return gemm_launch((cudaStream_t)stream, trans_a, M, N, K, K > 0 ? alpha : 0.0, a_dev, lda, b_dev, ldb, beta, c_dev,
                       ldc, epilogue, ws_dev, ws_bytes);
}

extern "C" int dagma_logdet_inv_ws_f64(dagma_stream_t stream, int d, double s, const double* a_dev, int lda,
                                       int square_input, double* logabsdet_dev, double* h_dev, double* minv_dev,
                                       double* grad_dev, int ldo, double* min_entry_dev, int* info_dev,
                                       double* ws_dev, size_t ws_bytes) {
    DAGMA_REQUIRE(d >= 1 && a_dev, "bad arguments");
    if (d <= DAGMA_ONCHIP_INV_MAX_D)
        return logdet_inv_small((cudaStream_t)stream, 1, d, s, a_dev, lda, square_input, logabsdet_dev, h_dev,
                                minv_dev, grad_dev, ldo, min_entry_dev, info_dev);
    DAGMA_REQUIRE(ws_dev && ws_bytes >= large_ws_bytes(d), "workspace too small (dagma_large_workspace_bytes)");
    return logdet_inv_blocked((cudaStream_t)stream, d, s, a_dev, lda, square_input, logabsdet_dev, h_dev, minv_dev,
                              grad_dev, ldo, min_entry_dev, info_dev, ws_dev);
}

extern "C" int dagma_logdet_inv_gemm_ws_f64(dagma_stream_t stream, int d, double s, const double* a_dev, int lda,
                                            int square_input, double* logabsdet_dev, double* h_dev, double* minv_dev,
                                            double* grad_dev, int ldo, double* min_entry_dev, int* info_dev,
                                            double* ws_dev, size_t ws_bytes, const double* ga_dev,
                                            const double* gb_dev, double* gc_dev) {
    DAGMA_REQUIRE(d >= 1 && a_dev && ga_dev && gb_dev && gc_dev, "bad arguments");
    if (d > DAGMA_ONCHIP_INV_MAX_D && flow_supported(d)) {
        DAGMA_REQUIRE(ws_dev && ws_bytes >= large_ws_bytes(d), "workspace too small (dagma_large_workspace_bytes)");
        RiderGemm rider;
        rider.A = ga_dev; rider.B = gb_dev; rider.C = gc_dev;
        return logdet_inv_blocked((cudaStream_t)stream, d, s, a_dev, lda, square_input, logabsdet_dev, h_dev, minv_dev,
                                  grad_dev, ldo, min_entry_dev, info_dev, ws_dev, rider);
    }
    int rc = dagma_logdet_inv_ws_f64(stream, d, s, a_dev, lda, square_input, logabsdet_dev, h_dev, minv_dev, grad_dev, ldo,
                                     min_entry_dev, info_dev, ws_dev, ws_bytes);
    if (rc) return rc;
    return gemm_launch((cudaStream_t)stream, 0, d, d, d, 1.0, ga_dev, d, gb_dev, d, 0.0, gc_dev, d, EPI_NONE, nullptr, 0);
}

extern "C" int dagma_bench_engine_gemm(dagma_stream_t stream, int d, const double* a_dev, const double* b_dev,
                                       double* c_dev, int persistent, unsigned* queue_dev) {
    DAGMA_REQUIRE(d % 2 == 0 && a_dev && b_dev && c_dev, "bad arguments");
    DAGMA_CUDA_OK(cudaFuncSetAttribute(engine_pair_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)OUTER_SMEM_BYTES));
    const int tn = (d + NB - 1) / NB, ntiles = tn * tn;
    if (persistent) DAGMA_CUDA_OK(cudaMemsetAsync(queue_dev, 0, sizeof(unsigned), (cudaStream_t)stream));
    engine_pair_gemm_kernel<<<persistent ? 296 : (ntiles + 1) / 2, DM_NT, OUTER_SMEM_BYTES, (cudaStream_t)stream>>>(
        a_dev, b_dev, c_dev, d, persistent, queue_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

// timing experiment: C = A B by the TMA-fed GEMM; mode 0 = static tile striding, 1 = atomic tile queue
extern "C" int dagma_bench_tma_gemm(dagma_stream_t stream, int M, int N, int K, const double* a_dev, int lda,
                                    const double* b_dev, int ldb, double* c_dev, int ldc, double alpha, double beta,
                                    int mode, unsigned* queue_dev) {
    DAGMA_REQUIRE(a_dev && b_dev && c_dev, "bad arguments");
    return gemm_tma_launch((cudaStream_t)stream, M, N, K, alpha, a_dev, lda, b_dev, ldb, beta, c_dev, ldc, EPI_NONE,
                           queue_dev, mode);
}

extern "C" int dagma_linear_update_ex_f64(dagma_stream_t stream, int d, void* state_dev, double* w_dev,
                                          const double* minv_dev, const double* t_dev, const double* cov_dev,
                                          double* m_dev, double* v_dev, const uint8_t* mask_exc_dev,
                                          const uint8_t* mask_inc_dev, const double* extra_t_dev, double extra_scale) {
    DAGMA_REQUIRE(state_dev && w_dev && minv_dev && t_dev && cov_dev && m_dev && v_dev, "null pointer");
    dim3 grid((d + 31) / 32, (d + 31) / 32);
    linear_update_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>((LinState*)state_dev, d, w_dev, minv_dev, t_dev,
                                                                        cov_dev, m_dev, v_dev, mask_exc_dev, mask_inc_dev,
                                                                        extra_t_dev, extra_scale);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int dagma_linear_update_f64(dagma_stream_t stream, int d, void* state_dev, double* w_dev,
                                       const double* minv_dev, const double* t_dev, const double* cov_dev,
                                       double* m_dev, double* v_dev, const uint8_t* mask_exc_dev,
                                       const uint8_t* mask_inc_dev) {
    return dagma_linear_update_ex_f64(stream, d, state_dev, w_dev, minv_dev, t_dev, cov_dev, m_dev, v_dev, mask_exc_dev,
                                      mask_inc_dev, nullptr, 0.0);
}

extern "C" int dagma_linear_apply_dir_f64(dagma_stream_t stream, int d, const void* state_dev, double* w_dev,
                                          const double* m_dev, const double* v_dev, double sign) {
    DAGMA_REQUIRE(state_dev && w_dev && m_dev && v_dev, "null pointer");
    linear_apply_dir_kernel<<<592, 256, 0, (cudaStream_t)stream>>>((const LinState*)state_dev, d, w_dev, m_dev, v_dev, sign);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int dagma_linear_objective_f64(dagma_stream_t stream, int d, void* state_dev, const double* w_dev,
                                          const double* t_dev, const double* cov_dev, int l2) {
    DAGMA_REQUIRE(state_dev && w_dev, "null pointer");
    linear_objective_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>((LinState*)state_dev, d, w_dev, t_dev, cov_dev, l2);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" size_t dagma_linear_objective_workspace_bytes(void) { return (size_t)(2 * 592 + 2) * sizeof(double); }

// multi-CTA form of dagma_linear_objective_f64; ws_dev: dagma_linear_objective_workspace_bytes() bytes whose first
// 8 bytes are zero at the first call (the kernel leaves them zero)
extern "C" int dagma_linear_objective_ws_f64(dagma_stream_t stream, int d, void* state_dev, const double* w_dev,
                                             const double* t_dev, const double* cov_dev, int l2, double* ws_dev,
                                             size_t ws_bytes) {
    DAGMA_REQUIRE(state_dev && w_dev && ws_dev, "null pointer");
    DAGMA_REQUIRE(ws_bytes >= dagma_linear_objective_workspace_bytes(), "workspace too small");
    const int grid = d < 592 ? d : 592;
    linear_objective_mb_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((LinState*)state_dev, d, w_dev, t_dev, cov_dev, l2,
                                                                       ws_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int dagma_logistic_loss_f64(dagma_stream_t stream, int n, int d, const double* x_dev, const double* r_dev,
                                       double scale, double* partial_dev, int n_partial, double* out_dev) {
    DAGMA_REQUIRE(x_dev && r_dev && partial_dev && out_dev && n_partial >= 1, "bad arguments");
    const int blocks = n_partial < 592 ? n_partial : 592;
    logistic_loss_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x_dev, r_dev, (size_t)n * d, partial_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    sum_partials_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(partial_dev, blocks, scale, out_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}
