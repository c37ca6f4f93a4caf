// DagmaLinear.minimize for d <= 128 (l2 beyond the on-chip fit kernel's d <= 64, logistic at any such d): the WHOLE
// inner iteration -- fused slogdet + inverse of sI - W o W, the score products, Gobj, Adam, step, masks, feasibility
// latch (reference: src/dagma/linear.py:70-116, 138-163, 224-276) -- and any number of consecutive iterations as ONE
// persistent kernel.
//
// Why.  The launch sequence of _large.py is ~6 dependent graph nodes per iteration around a single-CTA inverse:
// C2 (logistic, d = 100, n = 10 000) took 61 us per iteration for 4e8 flop of work, launch / drain latency and the
// un-overlapped tail of the inverse, not throughput.  Here (one CTA per SM, co-resident grid, bounded spins on counters
// in L2):
//
//   inverse CTA   builds M = (sI - W o W) / 2^e on chip, inverts it with the tensor-core sweep (d <= 64) or the
//   (the last)    two-by-two block Gauss-Jordan of small_inv2.cuh (d <= 128), leaves M^{-1}, log|det|, h, the smallest
//                 entry and the feasibility code of the reference's test `any(inv + 1e-16 < 0)`.
//   workers       logistic: worker c keeps ITS rows of X (<= 72, 9 DMMA m-tiles) in shared memory for the whole launch;
//                 per iteration it stages W once, R = sigmoid(Xc W) (DMMA, the accumulators are the epilogue's input),
//                 writes R over the staged W, and Gc = Xc^T R goes to row c of `part`.  After a barrier among the
//                 workers only, every worker adds the rows of `part` for its share of the entries in a FIXED order
//                 (four lanes per entry, a fixed tree) into T -- while the inverse CTA is still on its serial chain.
//                 l2: worker c owns rows 8c .. 8c + 7 of T = cov W; its cov fragments stay in registers for the
//                 whole launch.
//   barrier, then every CTA takes the Adam step of linear_update_kernel for its share of the entries (same arithmetic,
//   same order), CTA 0 advances the state block (beta powers as double-double, iteration counter) or latches `halted`
//   when the inverse was infeasible, barrier.
//
// Rows of X sharded over the GPUs of one box (one process per GPU): the SAME kernel runs on every GPU on its rows, and
// the one exchange step of the path -- the sum of the d x d partial products over the GPUs -- happens INSIDE it over
// NVLink peer memory (csrc/peer.cu), no collective library call: after the fixed-order sum of its workers' partials a
// GPU stores the d x d result into slot `rank` of EVERY GPU's exchange buffer (plain peer stores), fences at system
// scope, and one thread raises its sequence number in every GPU's flag array; after the grid barrier each CTA waits
// (bounded) for the sequence numbers of all peers in its LOCAL flag array and adds the slots in rank order -- the same
// order on every GPU, so the replicas stay bit-identical without a broadcast.  The buffers alternate by the parity of
// the sequence number: a GPU cannot be more than one exchange ahead of a peer, because it needs that peer's flag.
//
// The state block, the buffers and the results are those of the launch sequence (LargeLinearEngine), so back-tracking,
// objective checkpoints and telemetry are unchanged.  Trek regularisers and n beyond 72 rows x (SMs - 1) workers per GPU
// stay on the launch sequence.
#include "common.cuh"
#include "small_dmma.cuh"
#include "fit_step.cuh"
#include "small_inv2.cuh"
#include "gemm_f64.cuh"
#include "lin_state.h"
#include <cstdlib>
#include "../../include/dagma_b200.h"

namespace dagma {

constexpr int LI_NT = 256;
constexpr int LI_MT1 = 9;                 // m-tiles of X rows per worker (72 rows)
constexpr int LI_RB = 8 * LI_MT1;
constexpr unsigned LI_SPIN_MAX = 1u << 22;
constexpr int LI_MAX_D = 128;
constexpr int LI_MAX_RANKS = 8;           // GPUs of one box that may share the rows of X

struct LiPlan {
    int G, NW, NR;                        // CTAs, workers, rows of X per worker (logistic; multiple of 8)
    int SB, nsub;                         // streaming (NR > 72): rows per sub-block, sub-blocks per worker; else SB = NR, nsub = 1
    int ldx, kd;                          // row stride of the staged operands (= 4 mod 16), d rounded up to 4
    int o_w, o_x, o_r, total;             // shared-memory offsets / size of a worker (doubles)
    int smem_doubles;                     // dynamic shared memory of the launch
    bool stream;                          // the worker's rows do not fit: X is streamed through shared memory every iteration
    bool ok;
};
constexpr int LI_SMEM_CAP = 29000;        // doubles of shared memory a worker may plan with (227 KB = 29 056)
constexpr int LI_MAX_ROWS = 4096;         // rows per worker in streaming mode
__host__ __device__ inline LiPlan li_plan(int logistic, int n, int d, int sms, int allow_stream) {
    LiPlan L{};
    L.ok = false;
    if (d < 1 || d > LI_MAX_D || sms < 3) return L;
    L.ldx = 16 * ((d + 15) / 16) + 4;
    L.kd = 4 * ((d + 3) / 4);
    L.stream = false;
    if (logistic) {
        if (n < 1) return L;
        const int per = (n + (sms - 1) - 1) / (sms - 1);
        L.NR = 8 * ((per + 7) / 8);
        L.SB = L.NR;
        L.nsub = 1;
        if (L.NR > LI_RB) {
            // streaming: W, one sub-block of X and its R side by side (R cannot take the place of W, which every
            // sub-block needs); 16-byte cp.async of the rows of X wants an even d
            L.stream = true;
            if (!allow_stream || (d & 1) != 0 || L.NR > LI_MAX_ROWS) return L;
            L.SB = 8 * (((LI_SMEM_CAP - L.kd * L.ldx) / (2 * L.ldx)) / 8);
            if (L.SB > LI_RB) L.SB = LI_RB;
            if (L.SB < 16) return L;
            L.nsub = (L.NR + L.SB - 1) / L.SB;
        }
        L.NW = (n + L.NR - 1) / L.NR;
    } else {
        L.NR = L.SB = 0;
        L.nsub = 1;
        L.NW = (d + 7) / 8;
        if (L.NW > sms - 1) return L;
    }
    L.G = L.NW + 1;
    L.o_w = 0;
    if (L.stream) {
        L.o_x = L.kd * L.ldx;
        L.o_r = L.o_x + L.SB * L.ldx;
        L.total = L.o_r + L.SB * L.ldx + 2;
    } else {
        const int wrows = L.kd > L.NR ? L.kd : L.NR;      // R (NR rows) is written over the staged W (kd rows)
        L.o_x = wrows * L.ldx;
        L.o_r = L.o_w;
        L.total = L.o_x + L.NR * L.ldx + 2;
    }
    const int inv = d <= DM_DP ? DmmaSmem::total : Inv2Smem::total;
    L.smem_doubles = L.total > inv ? L.total : inv;
    L.ok = (size_t)L.smem_doubles * sizeof(double) <= 227 * 1024;
    return L;
}

struct LinIterArgs {
    LinState* st;
    double *W, *m, *v, *Minv, *T;
    const double *cov, *X;
    const uint8_t *mask_exc, *mask_inc;
    double* part;                         // logistic: [NW][d * d] un-scaled partial products
    unsigned* sync;                       // [0] grid barrier arrivals [1] worker barrier arrivals [2] error (zeroed per launch)
    int logistic, n, d, iters, sms, allow_stream;
    // rows of X sharded over `nranks` GPUs of one box (logistic only; nranks = 1: none of this is touched).
    // xchg[r]: rank r's exchange buffer as mapped into THIS process, [2 (parity)][nranks (writer)][d * d] doubles;
    // flags[r]: rank r's [nranks] sequence numbers (writer q's partial sums of iteration `seq` have landed in rank r's
    // buffer); seq: this rank's count of exchanged iterations (lives as long as the buffers, never reset).
    int rank, nranks;
    double* xchg[LI_MAX_RANKS];
    unsigned* flags[LI_MAX_RANKS];
    unsigned* seq;
};

#ifdef DAGMA_LIN_TRACE
// debug build only: %globaltimer stamps (ns) of the LAST iteration of a launch.  worker 0: [0] iteration starts
// [1] W staged  [2] Z done  [3] R written  [4] partial product written  [5] past the workers' barrier  [6] T reduced
// [7] past barrier 1  [8] step taken  [9] past barrier 2;  inverse CTA: [10] starts  [11] M built  [12] inverted
// [13] outputs written
__device__ unsigned long long g_lin_trace[16];
__device__ __forceinline__ unsigned long long li_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define LI_STAMP(slot, cond) do { if ((cond) && threadIdx.x == 0) g_lin_trace[slot] = li_gtime(); } while (0)
#else
#define LI_STAMP(slot, cond) do { } while (0)
#endif

// barrier number `k` (0, 1, ...) of this launch among `cnt` CTAs: one atomic per CTA, no reset; bounded
__device__ __forceinline__ void li_barrier(unsigned* ctr, unsigned* err, unsigned cnt, unsigned& k) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned target = cnt * (k + 1);
        __threadfence();
        atomicAdd(ctr, 1u);
        unsigned spins = 0;
        while (*(volatile unsigned*)ctr < target) {
            if ((++spins & 63u) == 0u) {
                if (*(volatile unsigned*)err) break;
                if (spins > LI_SPIN_MAX) { atomicExch(err, 1u); break; }
            }
        }
        __threadfence();
    }
    ++k;
    __syncthreads();
}

// ---------------------------------------------------------------- the CTA that owns the inverse
// Before the grid barrier: M^{-1}, its smallest entry and the feasibility code (what the step needs); the CTA's partial
// sums of log|det| come back in `ld` and are finished by li_inverse_logdet AFTER the step, off the critical path.
struct LiInvScale {
    double s, scale, inv_scale;
};
__device__ __forceinline__ LiInvScale li_inv_scale(const LinIterArgs& P) {
    LiInvScale q;
    q.s = *(volatile double*)&P.st->s;
    q.scale = 1.0;
    if (q.s > 0.0 && isfinite(q.s)) {          // s / 2^e in (0.5, 1]: exact (logdet_inv_small)
        int e = 0;
        const double f = frexp(q.s, &e);
        if (f == 0.5) --e;
        q.scale = ldexp(1.0, e);
    }
    q.inv_scale = 1.0 / q.scale;
    return q;
}
// once per launch (d > 64): the identity padding of the four tiles -- the elimination leaves it exactly as it is
__device__ __forceinline__ void li_inverse_init(const LinIterArgs& P, double* psm) {
    if (P.d <= DM_DP) return;
    for (int r = threadIdx.x >> 5; r < 2 * DM_DP; r += LI_NT / 32)
        for (int c = threadIdx.x & 31; c < 2 * DM_DP; c += 32)
            psm[Inv2Smem::at(r >> 6, c >> 6) + (r & 63) * DM_LD + (c & 63)] = (r == c) ? 1.0 : 0.0;
}
__device__ __forceinline__ void li_inverse_role(const LinIterArgs& P, double* psm, SweepSync& sy, const LiInvScale& q,
                                                double& ld) {
    using S = DmmaSmem;
    constexpr int LD = DM_LD;
    const int tid = threadIdx.x, d = P.d;
    const DmmaPos ps(tid);
    double* red = psm + S::red;
    const double s = q.s, inv_scale = q.inv_scale;
    double mn = INFINITY;
    bool badpiv = false;
    ld = 0.0;
    LI_STAMP(10, true);
    if (d <= DM_DP) {
        double a[2][4][2];
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)                           // all sixteen loads of a thread in flight
#pragma unroll
            for (int tj = 0; tj < 4; ++tj)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = ps.row(ti), c = ps.col(tj) + e;
                    a[ti][tj][e] = (r < d && c < d) ? __ldcg(P.W + (size_t)r * d + c) : 0.0;
                }
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)
#pragma unroll
            for (int tj = 0; tj < 4; ++tj)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = ps.row(ti), c = ps.col(tj) + e;
                    const double x = a[ti][tj][e];
                    a[ti][tj][e] = (r < d && c < d) ? (((r == c) ? s : 0.0) - x * x) * inv_scale : ((r == c) ? 1.0 : 0.0);
                }
        LI_STAMP(11, true);
        dmma_sweep(a, ps, psm, d, sy);
        LI_STAMP(12, true);
        if (tid < ((d + 3) & ~3)) {
            const double p = psm[S::pinfo + tid];
            ld = (double)((tid & 3) - 2) * log(fabs(p));
            badpiv = !(p > 0.0);
        }
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)
#pragma unroll
            for (int tj = 0; tj < 4; ++tj)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int r = ps.row(ti), c = ps.col(tj) + e;
                    if (r < d && c < d) {
                        const double mi = a[ti][tj][e] * inv_scale;
                        mn = fmin(mn, mi);
                        P.Minv[(size_t)r * d + c] = mi;
                    }
                }
    } else {
        // M = (s I - W o W) / 2^e into the tiles: thread (warp, lane) owns the rows warp + 8 i and the columns lane + 32 j;
        // all of its loads (L2: W changes every iteration) are in flight before the first use.  The padding keeps the
        // identity of li_inverse_init.
        {
            const int lane = tid & 31, w8 = tid >> 5;
#pragma unroll
            for (int ih = 0; ih < 2; ++ih) {                     // rows of the upper / lower tiles: 32 loads per batch
                double t[8][4];
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = w8 + 8 * i + DM_DP * ih, c = lane + 32 * j;
                        t[i][j] = (r < d && c < d) ? __ldcg(P.W + (size_t)r * d + c) : 0.0;
                    }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int r = w8 + 8 * i + DM_DP * ih, c = lane + 32 * j;
                        if (r < d && c < d)
                            psm[Inv2Smem::at(ih, j >> 1) + (r & 63) * LD + (c & 63)] = (((r == c) ? s : 0.0) - t[i][j] * t[i][j]) * inv_scale;
                    }
            }
        }
        // the padding INSIDE the last pivot block comes back from the fraction-free elimination as p / p (one ulp from
        // 1): reset it, everything else of the padding is reproduced exactly
        if (tid < DM_PB && d + tid < 8 * ((d + 7) / 8)) {
            const int r = d + tid;
            psm[Inv2Smem::at(r >> 6, r >> 6) + (r & 63) * LD + (r & 63)] = 1.0;
        }
        __syncthreads();
        LI_STAMP(11, true);
        // the tiles of the inverse leave for global memory (and enter the minimum) straight from the accumulators of
        // the last block step
        inv2_block_gj(psm, ps, sy, d, [&](int bi, int bj, const double (&acc)[2][4][2], double sign) {
            const double f = sign * inv_scale;
#pragma unroll
            for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                for (int tj = 0; tj < 4; ++tj) {
                    const int r = DM_DP * bi + ps.row(ti), c = DM_DP * bj + ps.col(tj);
                    const double m0 = f * acc[ti][tj][0], m1 = f * acc[ti][tj][1];
                    if (r < d && c < d) {
                        mn = fmin(mn, m0);
                        P.Minv[(size_t)r * d + c] = m0;
                        if (c + 1 < d) {
                            mn = fmin(mn, m1);
                            P.Minv[(size_t)r * d + c + 1] = m1;
                        }
                    }
                }
        });
        LI_STAMP(12, true);
        const double* pv = psm + Inv2Smem::piv;
        if (tid < 2 * DM_DP) {
            const double p = pv[tid];
            ld = (double)((tid & 3) - 2) * log(fabs(p));
            badpiv = !(p > 0.0);
        }
    }
    mn = block_min<LI_NT>(mn, red, tid);
    const int anybad = __syncthreads_or(badpiv);
    if (tid == 0) {
        volatile LinState* st = P.st;
        st->min_entry = mn;
        st->info = anybad ? 1 : ((mn + 1e-16 < 0.0) ? 2 : 0);
    }
    LI_STAMP(13, true);
}
__device__ __forceinline__ void li_inverse_logdet(const LinIterArgs& P, double* psm, const LiInvScale& q, double ld) {
    double zero1 = 0.0, zero2 = 0.0;
    block_sum3<LI_NT>(ld, zero1, zero2, psm + DmmaSmem::red, threadIdx.x);
    if (threadIdx.x == 0) {
        volatile LinState* st = P.st;
        const double lad = ld + (double)P.d * log(q.scale);
        st->logabsdet = lad;
        st->h = -lad + (double)P.d * log(q.s);
    }
}

// This iteration's W into the leading d x d of Ws [kd][ldx].  W changes between iterations, so it must come from L2:
// cp.async.cg in 16-byte pieces when d is even (every piece in flight at once), else L2 loads in batches of sixteen.
// The padding of Ws is not written here: it was zeroed at the start of the launch and only ever holds finite numbers
// (zeros, or values of R), which the zero padding of the other operand annihilates.
__device__ __forceinline__ void li_stage_w(const LinIterArgs& P, const LiPlan& L, double* Ws) {
    const int d = P.d, tid = threadIdx.x;
    if ((d & 1) == 0) {
        const int hc = d >> 1;
        for (int r = tid >> 5; r < d; r += LI_NT / 32)
            for (int c2 = tid & 31; c2 < hc; c2 += 32)
                cp_async16(smem_u32(Ws + r * L.ldx + 2 * c2), P.W + (size_t)r * d + 2 * c2, true);
        cp_async_commit();
        cp_async_wait<0>();
    } else {
        const int dd = d * d;
        for (int e0 = tid; e0 < dd; e0 += 16 * LI_NT) {
            double t[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) t[u] = (e0 + u * LI_NT < dd) ? __ldcg(P.W + e0 + u * LI_NT) : 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int e = e0 + u * LI_NT;
                if (e < dd) Ws[(e / d) * L.ldx + (e % d)] = t[u];
            }
        }
    }
}

// ---------------------------------------------------------------- logistic worker: rows [c NR, (c + 1) NR) of X
__device__ __forceinline__ void li_logistic_role(const LinIterArgs& P, const LiPlan& L, double* sm, int cta) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, qr = lane >> 2, qc = lane & 3;
    const int d = P.d, ldx = L.ldx, MT = L.NR / 8, NT = (d + 7) / 8, KT = L.kd / 4;
    double* Ws = sm + L.o_w;
    double* Rs = sm + L.o_w;                  // R takes the place of W once every warp is done with it
    const double* Xs = sm + L.o_x;
    const int nt[2] = {warp, warp + 8};
    const bool nv[2] = {nt[0] < NT, nt[1] < NT};

    li_stage_w(P, L, Ws);
    __syncthreads();
    LI_STAMP(1, cta == 0);
    // ---- Z = Xc W (K = d): all m-tiles of the worker x the warp's two n-tiles
    double z[LI_MT1][2][2];
#pragma unroll
    for (int i = 0; i < LI_MT1; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) z[i][j][0] = z[i][j][1] = 0.0;
    if (nv[0]) {
        const double* ap = Xs + qr * ldx + qc;
        const double* bp = Ws + qc * ldx + qr;
#pragma unroll 2
        for (int ks = 0; ks < KT; ++ks) {
            double a[LI_MT1], b[2];
#pragma unroll
            for (int i = 0; i < LI_MT1; ++i) a[i] = (i < MT) ? ap[8 * i * ldx + 4 * ks] : 0.0;
            b[0] = bp[4 * ks * ldx + 8 * nt[0]];
            b[1] = nv[1] ? bp[4 * ks * ldx + 8 * nt[1]] : 0.0;
#pragma unroll
            for (int i = 0; i < LI_MT1; ++i)
                if (i < MT) {
                    dmma(z[i][0][0], z[i][0][1], a[i], b[0]);
                    dmma(z[i][1][0], z[i][1][1], a[i], b[1]);
                }
        }
    }
    __syncthreads();                          // every warp is done reading W
    LI_STAMP(2, cta == 0);
    // ---- R = sigmoid(Z)
#pragma unroll
    for (int j = 0; j < 2; ++j)
        if (nv[j]) {
#pragma unroll
            for (int i = 0; i < LI_MT1; ++i)
                if (i < MT)
                    *reinterpret_cast<double2*>(Rs + (8 * i + qr) * ldx + 8 * nt[j] + 2 * qc) =
                        make_double2(li_sigmoid(z[i][j][0]), li_sigmoid(z[i][j][1]));
        }
    __syncthreads();
    LI_STAMP(3, cta == 0);
    // ---- Gc = Xc^T R (K = rows of the worker): m-tiles in two passes of eight, the warp's two n-tiles
    double* prow = P.part + (size_t)cta * d * d;
    const int MTd = (d + 7) / 8, KR = L.NR / 4;
    const bool vec = (d & 1) == 0;
    if (nv[0]) {
#pragma unroll 1
        for (int mp = 0; mp < MTd; mp += 8) {
            const int mc = min(8, MTd - mp);
            double g[8][2][2];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) g[i][j][0] = g[i][j][1] = 0.0;
            const double* ap = Xs + qc * ldx + 8 * mp + qr;
            const double* bp = Rs + qc * ldx + qr;
#pragma unroll 2
            for (int ks = 0; ks < KR; ++ks) {
                double a[8], b[2];
#pragma unroll
                for (int i = 0; i < 8; ++i) a[i] = (i < mc) ? ap[4 * ks * ldx + 8 * i] : 0.0;
                b[0] = bp[4 * ks * ldx + 8 * nt[0]];
                b[1] = nv[1] ? bp[4 * ks * ldx + 8 * nt[1]] : 0.0;
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (i < mc) {
                        dmma(g[i][0][0], g[i][0][1], a[i], b[0]);
                        dmma(g[i][1][0], g[i][1][1], a[i], b[1]);
                    }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int r = 8 * (mp + i) + qr, c = 8 * nt[j] + 2 * qc;
                    if (i < mc && nv[j] && r < d && c < d) {
                        double* q = prow + (size_t)r * d + c;
                        if (vec) *reinterpret_cast<double2*>(q) = make_double2(g[i][j][0], g[i][j][1]);
                        else {
                            q[0] = g[i][j][0];
                            if (c + 1 < d) q[1] = g[i][j][1];
                        }
                    }
                }
        }
    }
}

// ---------------------------------------------------------------- logistic worker, rows streamed (NR > 72)
// The worker's NR rows pass through shared memory in sub-blocks of SB rows every iteration (X is constant and stays in
// L2); W is staged once per iteration, R has its own buffer, and the warp's tiles of Gc -- all 16 m-tiles x its two
// n-tiles -- live in registers across the sub-blocks; Z is formed four m-tiles at a time.
__device__ __forceinline__ void li_logistic_stream_role(const LinIterArgs& P, const LiPlan& L, double* sm, int cta) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, qr = lane >> 2, qc = lane & 3;
    const int d = P.d, ldx = L.ldx, NT = (d + 7) / 8, KT = L.kd / 4, MTd = (d + 7) / 8, hc = d >> 1;
    double* Ws = sm + L.o_w;
    double* Xs = sm + L.o_x;
    double* Rs = sm + L.o_r;
    const int nt[2] = {warp, warp + 8};
    const bool nv[2] = {nt[0] < NT, nt[1] < NT};
    li_stage_w(P, L, Ws);
    double g[16][2][2];
#pragma unroll
    for (int i = 0; i < 16; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) g[i][j][0] = g[i][j][1] = 0.0;
#pragma unroll 1
    for (int sb = 0; sb < L.nsub; ++sb) {
        const int r0 = cta * L.NR + sb * L.SB, cnt = min(L.SB, L.NR - sb * L.SB);
        __syncthreads();                      // the previous sub-block is done with Xs / Rs
        for (int r = warp; r < cnt; r += LI_NT / 32)
            for (int c2 = lane; c2 < hc; c2 += 32)
                cp_async16(smem_u32(Xs + r * ldx + 2 * c2), P.X + (size_t)(r0 + r) * d + 2 * c2, r0 + r < P.n);
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();                      // the rows (and, the first time, W) have landed for every thread
        if (nv[0]) {
            const int MT = cnt / 8;
#pragma unroll 1
            for (int mc = 0; mc < MT; mc += 4) {
                const int mcnt = min(4, MT - mc);
                double z[4][2][2];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 2; ++j) z[i][j][0] = z[i][j][1] = 0.0;
                const double* ap = Xs + (8 * mc + qr) * ldx + qc;
                const double* bp = Ws + qc * ldx + qr;
#pragma unroll 2
                for (int ks = 0; ks < KT; ++ks) {
                    double a[4], b[2];
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[i] = (i < mcnt) ? ap[8 * i * ldx + 4 * ks] : 0.0;
                    b[0] = bp[4 * ks * ldx + 8 * nt[0]];
                    b[1] = nv[1] ? bp[4 * ks * ldx + 8 * nt[1]] : 0.0;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (i < mcnt) {
                            dmma(z[i][0][0], z[i][0][1], a[i], b[0]);
                            dmma(z[i][1][0], z[i][1][1], a[i], b[1]);
                        }
                }
#pragma unroll
                for (int j = 0; j < 2; ++j)
                    if (nv[j]) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (i < mcnt)
                                *reinterpret_cast<double2*>(Rs + (8 * (mc + i) + qr) * ldx + 8 * nt[j] + 2 * qc) =
                                    make_double2(li_sigmoid(z[i][j][0]), li_sigmoid(z[i][j][1]));
                    }
            }
        }
        __syncthreads();
        if (nv[0]) {
            const double* ap = Xs + qc * ldx + qr;
            const double* bp = Rs + qc * ldx + qr;
            const int KR = cnt / 4;
#pragma unroll 2
            for (int ks = 0; ks < KR; ++ks) {
                double a[16], b[2];
#pragma unroll
                for (int i = 0; i < 16; ++i) a[i] = (i < MTd) ? ap[4 * ks * ldx + 8 * i] : 0.0;
                b[0] = bp[4 * ks * ldx + 8 * nt[0]];
                b[1] = nv[1] ? bp[4 * ks * ldx + 8 * nt[1]] : 0.0;
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (i < MTd) {
                        dmma(g[i][0][0], g[i][0][1], a[i], b[0]);
                        dmma(g[i][1][0], g[i][1][1], a[i], b[1]);
                    }
            }
        }
    }
    double* prow = P.part + (size_t)cta * d * d;
    if (nv[0]) {
#pragma unroll
        for (int i = 0; i < 16; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int r = 8 * i + qr, c = 8 * nt[j] + 2 * qc;                 // d is even: c + 1 < d with c
                if (i < MTd && nv[j] && r < d && c < d)
                    *reinterpret_cast<double2*>(prow + (size_t)r * d + c) = make_double2(g[i][j][0], g[i][j][1]);
            }
    }
}

// T = sum over the workers' rows of `part`, fixed order: four lanes per entry (lane q adds the rows q, q + 4, ... --
// all of its loads in flight at once), then (s0 + s1) + (s2 + s3)
constexpr int LI_RED = 40;                    // rows per lane and pass: 4 x 40 >= the 147 workers of a B200
__device__ __forceinline__ void li_reduce_partials(const LinIterArgs& P, const LiPlan& L, int cta, unsigned seq) {
    const int dd = P.d * P.d, NW = L.NW;
    const size_t slot = ((size_t)(seq & 1u) * P.nranks + P.rank) * dd;        // sharded rows: where this GPU's sums go
    const int q = threadIdx.x & 3;
    const int rounds = (dd + NW * (LI_NT / 4) - 1) / (NW * (LI_NT / 4));       // uniform trip count: the shuffles need all lanes
    for (int rd = 0; rd < rounds; ++rd) {
        const int e = rd * NW * (LI_NT / 4) + cta * (LI_NT / 4) + (threadIdx.x >> 2);
        const bool in = e < dd;
        const double* src = P.part + (in ? e : 0);
        double acc = 0.0;
        for (int c0 = q; c0 < NW; c0 += 4 * LI_RED) {
            double t[LI_RED];
#pragma unroll
            for (int u = 0; u < LI_RED; ++u) t[u] = (in && c0 + 4 * u < NW) ? __ldcg(src + (size_t)(c0 + 4 * u) * dd) : 0.0;
#pragma unroll
            for (int u = 0; u < LI_RED; ++u)
                if (c0 + 4 * u < NW) acc += t[u];
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (P.nranks == 1) {
            if (in && q == 0) P.T[e] = acc;
        } else if (in) {
            // every lane of the four holds the sum: lane q serves the GPUs q, q + 4 (peer stores over NVLink; the own
            // buffer is one of them)
            for (int r = q; r < P.nranks; r += 4) P.xchg[r][slot + e] = acc;
        }
    }
    if (P.nranks > 1) __threadfence_system();
}

// ---------------------------------------------------------------- l2 worker: rows 8 cta .. 8 cta + 7 of T = cov W
struct LiCovFrag {
    double a[LI_MAX_D / 4];                   // A fragments of the worker's eight rows of cov, all k-steps
};
__device__ __forceinline__ void li_l2_load(const LinIterArgs& P, const LiPlan& L, int cta, LiCovFrag& f) {
    const int lane = threadIdx.x & 31, qr = lane >> 2, qc = lane & 3, d = P.d;
    const int r = 8 * cta + qr;
#pragma unroll
    for (int ks = 0; ks < LI_MAX_D / 4; ++ks) {
        const int k = 4 * ks + qc;
        f.a[ks] = (ks < L.kd / 4 && r < d && k < d) ? __ldg(P.cov + (size_t)r * d + k) : 0.0;
    }
}
__device__ __forceinline__ void li_l2_role(const LinIterArgs& P, const LiPlan& L, double* sm, int cta, const LiCovFrag& f) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, qr = lane >> 2, qc = lane & 3;
    const int d = P.d, ldx = L.ldx, NT = (d + 7) / 8, KT = L.kd / 4;
    double* Ws = sm + L.o_w;
    li_stage_w(P, L, Ws);
    __syncthreads();
    const int nt0 = warp, nt1 = warp + 8;
    if (nt0 < NT) {
        const bool v1 = nt1 < NT;
        double t[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
        const double* bp = Ws + qc * ldx + qr;
#pragma unroll
        for (int ks = 0; ks < LI_MAX_D / 4; ++ks)
            if (ks < KT) {
                const double b0 = bp[4 * ks * ldx + 8 * nt0], b1 = v1 ? bp[4 * ks * ldx + 8 * nt1] : 0.0;
                dmma(t[0][0], t[0][1], f.a[ks], b0);
                dmma(t[1][0], t[1][1], f.a[ks], b1);
            }
        const int r = 8 * cta + qr;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int c = 8 * (j ? nt1 : nt0) + 2 * qc;
            if ((j == 0 || v1) && r < d && c < d) {
                P.T[(size_t)r * d + c] = t[j][0];
                if (c + 1 < d) P.T[(size_t)r * d + c + 1] = t[j][1];
            }
        }
    }
}

// the scalars of the state block as every CTA reads them at the START of an iteration (CTA 0 advances the block after
// the first grid barrier)
struct LiScalars {
    double mu, lr, lambda1, b1, b2, gscale, c1, c2, p1h, p1l, p2h, p2l;
};

// ---------------------------------------------------------------- the step: linear_update_kernel, entry by entry
__device__ __forceinline__ void li_update(const LinIterArgs& P, int cta, int G, const LiScalars& sc, unsigned seq) {
    const int d = P.d, dd = d * d;
    const double* xs = (P.nranks > 1) ? P.xchg[P.rank] + (size_t)(seq & 1u) * P.nranks * dd : nullptr;
    for (int e = cta * LI_NT + threadIdx.x; e < dd; e += G * LI_NT) {
        const int r = e / d, c = e - r * d;
        const double w = __ldcg(P.W + e);
        const double minvT = __ldcg(P.Minv + (size_t)c * d + r);
        double tt;
        if (P.nranks == 1) tt = __ldcg(P.T + e);
        else {                                                  // the GPUs' sums in rank order: the same on every GPU
            tt = 0.0;
            for (int q = 0; q < P.nranks; ++q) tt += __ldcg(xs + (size_t)q * dd + e);
        }
        const double sg = (w > 0.0) ? 1.0 : ((w < 0.0) ? -1.0 : 0.0);
        const double gsc = fma(sc.gscale, tt, -__ldg(P.cov + e));
        double go = fma(sc.mu, gsc, sc.mu * sc.lambda1 * sg);
        go = fma(2.0 * w, minvT + 1e-16, go);
        if (P.mask_inc && P.mask_inc[e]) go = fma(-2.0 * sc.mu * sc.lambda1, sg, go);
        const double mn = fma(P.m[e], sc.b1, (1.0 - sc.b1) * go);
        const double vn = fma(P.v[e], sc.b2, (1.0 - sc.b2) * (go * go));
        P.m[e] = mn;
        P.v[e] = vn;
        const double dir = fast_div(mn * sc.c1, fast_sqrt_nonneg(vn * sc.c2) + 1e-8);
        double wn = w - sc.lr * dir;
        if (P.mask_exc && P.mask_exc[e]) wn = 0.0;
        P.W[e] = wn;
    }
}

// MODE (0 l2, 1 logistic with resident rows, 2 logistic with streamed rows) is a template parameter so that each variant
// carries only its own live state (the l2 workers keep 64 registers of cov fragments across the whole launch, the
// streaming workers 128 registers of accumulators across their sub-blocks)
template <int MODE>
__global__ void __launch_bounds__(LI_NT, 1) linear_iter_kernel(const LinIterArgs P) {
    constexpr bool LOGISTIC = MODE != 0;
    extern __shared__ __align__(16) double sm[];
    __shared__ LiScalars s_sc;
    __shared__ unsigned s_seq;
    const int tid = threadIdx.x, cta = blockIdx.x, G = gridDim.x;
    const LiPlan L = li_plan(LOGISTIC ? 1 : 0, P.n, P.d, P.sms, P.allow_stream);
    const bool icta = (cta == G - 1);
    unsigned* err = P.sync + 2;
    SweepSync sy{smem_u32(sm + DmmaSmem::mbar), 0u};
    LiCovFrag cf;
    LiInvScale isc{};
    double ild = 0.0;
    if (icta) {
        if (tid == 0) mbar_init(sy.bar, DM_NT / 32);
        li_inverse_init(P, sm);
        isc = li_inv_scale(P);
    } else {
        // the staging area of W: finite everywhere before the first product (see li_stage_w)
        const int wrows = (MODE == 1 && L.NR > L.kd) ? L.NR : L.kd;
        for (int e = tid; e < wrows * L.ldx; e += LI_NT) sm[L.o_w + e] = 0.0;
    }
    if (!icta && MODE == 2) {
        for (int e = tid; e < 2 * L.SB * L.ldx; e += LI_NT) sm[L.o_x + e] = 0.0;     // the padding columns of Xs / Rs
    } else if (!icta && MODE == 1) {
        // this worker's rows of X, once per launch, zero padded to [NR][ldx]
        double* Xs = sm + L.o_x;
        const int r0 = cta * L.NR;
        for (int r = tid >> 5; r < L.NR; r += LI_NT / 32)
            for (int c = tid & 31; c < L.ldx; c += 32)
                Xs[r * L.ldx + c] = (r0 + r < P.n && c < P.d) ? __ldg(P.X + (size_t)(r0 + r) * P.d + c) : 0.0;
    } else if (!icta) {
        if constexpr (!LOGISTIC) li_l2_load(P, L, cta, cf);
    }
    __syncthreads();
    unsigned bar_all = 0, bar_w = 0;
    for (int it = 0; it < P.iters; ++it) {
        if (*(volatile int32_t*)&P.st->halted != 0 || *(volatile unsigned*)err != 0u) break;     // uniform over the grid
        LI_STAMP(0, cta == 0);
        if (tid == 0) {
            const volatile LinState* st = P.st;
            LiScalars sc;
            sc.mu = st->mu; sc.lr = st->lr; sc.lambda1 = st->lambda1; sc.b1 = st->beta1; sc.b2 = st->beta2;
            sc.gscale = st->gscale;
            sc.p1h = st->p1_hi; sc.p1l = st->p1_lo; sc.p2h = st->p2_hi; sc.p2l = st->p2_lo;
            dd_mul(sc.p1h, sc.p1l, sc.b1);
            dd_mul(sc.p2h, sc.p2l, sc.b2);
            sc.c1 = 1.0 / ((1.0 - sc.p1h) - sc.p1l);
            sc.c2 = 1.0 / ((1.0 - sc.p2h) - sc.p2l);
            s_sc = sc;
            s_seq = (P.nranks > 1) ? *(volatile unsigned*)P.seq + 1u : 0u;       // CTA 0 stores it back after the barrier
        }
        if (icta) li_inverse_role(P, sm, sy, isc, ild);
        else if constexpr (LOGISTIC) {
            if constexpr (MODE == 2) li_logistic_stream_role(P, L, sm, cta);
            else li_logistic_role(P, L, sm, cta);
            LI_STAMP(4, cta == 0);
#ifdef DAGMA_LIN_TRACE
            if (tid == 0) {                                  // [14] last / [15] first arrival at the workers' barrier
                const unsigned long long t = li_gtime();
                if (cta == 0) { g_lin_trace[14] = 0ull; g_lin_trace[15] = ~0ull; }
                atomicMax(&g_lin_trace[14], t);
                atomicMin(&g_lin_trace[15], t);
            }
#endif
            li_barrier(P.sync + 1, err, (unsigned)L.NW, bar_w);      // (publishes s_seq to the CTA as well)
            LI_STAMP(5, cta == 0);
            li_reduce_partials(P, L, cta, s_seq);
            if (P.nranks > 1) {
                // every worker's peer stores are fenced: raise this GPU's sequence number on every peer
                li_barrier(P.sync + 1, err, (unsigned)L.NW, bar_w);
                if (cta == 0 && tid < P.nranks && tid != P.rank) {
                    __threadfence_system();                      // release: everything the barrier made visible to this thread
                    *(volatile unsigned*)(P.flags[tid] + P.rank) = s_seq;
                }
            }
            LI_STAMP(6, cta == 0);
        } else {
            li_l2_role(P, L, sm, cta, cf);
        }
        li_barrier(P.sync, err, (unsigned)G, bar_all);
        LI_STAMP(7, cta == 0);
        const LiScalars sc = s_sc;
        const unsigned seq = s_seq;
        if (P.nranks > 1) {
            // the partial sums of every peer for this iteration have landed in the LOCAL buffer (bounded wait)
            if (tid < P.nranks && tid != P.rank) {
                unsigned spins = 0;
                while ((int)(*(volatile unsigned*)(P.flags[P.rank] + tid) - seq) < 0) {
                    if ((++spins & 63u) == 0u) {
                        if (*(volatile unsigned*)err) break;
                        if (spins > LI_SPIN_MAX) { atomicExch(err, 2u); break; }
                    }
                }
                __threadfence_system();
            }
            __syncthreads();
        }
        const bool stop = *(volatile int32_t*)&P.st->info != 0;
        if (cta == 0 && tid == 0) {                      // linear_advance: everybody has read the scalars of this iteration
            volatile LinState* st = P.st;
            if (P.nranks > 1) *(volatile unsigned*)P.seq = seq;
            if (stop) st->halted = 1;
            else {
                st->p1_hi = sc.p1h; st->p1_lo = sc.p1l; st->p2_hi = sc.p2h; st->p2_lo = sc.p2l;
                st->it = st->it + 1;
            }
        }
        if (!stop) li_update(P, cta, G, sc, seq);
        if (icta) li_inverse_logdet(P, sm, isc, ild);        // h / log|det| of this iteration: nobody on the device waits for them
        LI_STAMP(8, cta == 0);
        li_barrier(P.sync, err, (unsigned)G, bar_all);
        LI_STAMP(9, cta == 0);
    }
    if (tid == 0 && cta == 0 && *(volatile unsigned*)err != 0u) P.st->info = 99;      // a barrier timed out
}

}  // namespace dagma

using namespace dagma;

static int li_sms() {
    static int sms = -1;
    if (sms < 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess)
            sms = v;
        else
            return 0;
    }
    return sms;
}

// DAGMA_LIN_STREAM (A-B timing): 1 = logistic problems whose rows do not fit the workers' shared memory stream them
// through it every iteration (li_logistic_stream_role); 0 (default) = such problems are reported as unsupported and keep
// the launch sequence, whose large GEMMs are the faster route there (n = 20 000 ... 160 000 at d = 100: 88 ... 472 us per
// iteration against 103 ... 695 streamed)
static int li_allow_stream() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DAGMA_LIN_STREAM");
        v = e ? atoi(e) : 0;
    }
    return v;
}

extern "C" int dagma_linear_iter_supported(int logistic, int n, int d) {
    return li_plan(logistic, n, d, li_sms(), li_allow_stream()).ok ? 1 : 0;
}

extern "C" size_t dagma_linear_iter_workspace_doubles(int logistic, int n, int d) {
    const LiPlan L = li_plan(logistic, n, d, li_sms(), li_allow_stream());
    if (!L.ok) return 0;
    return (logistic ? (size_t)L.NW * d * d : 0) + 8;
}

static int linear_iter_launch(cudaStream_t stream, int logistic, int n, int d, int iters, void* state_dev, double* w_dev,
                              double* m_dev, double* v_dev, double* minv_dev, double* t_dev, const double* cov_dev,
                              const double* x_dev, const uint8_t* mask_exc_dev, const uint8_t* mask_inc_dev,
                              double* part_dev, unsigned* sync_dev, int rank, int nranks, void* const* xchg_ptrs,
                              void* const* flag_ptrs, unsigned* seq_dev) {
    DAGMA_REQUIRE(state_dev && w_dev && m_dev && v_dev && minv_dev && t_dev && cov_dev && part_dev && sync_dev, "null pointer");
    DAGMA_REQUIRE(!logistic || x_dev, "the logistic loss needs X");
    const LiPlan L = li_plan(logistic, n, d, li_sms(), li_allow_stream());
    DAGMA_REQUIRE(iters >= 0 && L.ok, "shape not supported by the fused iteration (dagma_linear_iter_supported)");
    const size_t smem = (size_t)L.smem_doubles * sizeof(double);
    const int mode = logistic ? (L.stream ? 2 : 1) : 0;
    static size_t attr[3] = {0, 0, 0};
    if (smem > attr[mode]) {
        const void* fn = mode == 0 ? (const void*)linear_iter_kernel<0>
                       : mode == 1 ? (const void*)linear_iter_kernel<1> : (const void*)linear_iter_kernel<2>;
        DAGMA_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr[mode] = smem;
    }
    DAGMA_REQUIRE((double)L.G * 3.0 * (double)iters < 4.0e9, "too many iterations for one launch");
    LinIterArgs A{};
    A.st = (LinState*)state_dev;
    A.W = w_dev; A.m = m_dev; A.v = v_dev; A.Minv = minv_dev; A.T = t_dev;
    A.cov = cov_dev; A.X = x_dev;
    A.mask_exc = mask_exc_dev; A.mask_inc = mask_inc_dev;
    A.part = part_dev; A.sync = sync_dev;
    A.logistic = logistic; A.n = n; A.d = d; A.iters = iters; A.sms = li_sms(); A.allow_stream = li_allow_stream();
    A.rank = rank; A.nranks = nranks; A.seq = seq_dev;
    for (int r = 0; r < nranks && nranks > 1; ++r) {
        A.xchg[r] = (double*)xchg_ptrs[r];
        A.flags[r] = (unsigned*)flag_ptrs[r];
    }
    DAGMA_CUDA_OK(cudaMemsetAsync(sync_dev, 0, 4 * sizeof(unsigned), stream));
    if (mode == 2) linear_iter_kernel<2><<<L.G, LI_NT, smem, stream>>>(A);
    else if (mode == 1) linear_iter_kernel<1><<<L.G, LI_NT, smem, stream>>>(A);
    else linear_iter_kernel<0><<<L.G, LI_NT, smem, stream>>>(A);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int dagma_linear_iter_f64(dagma_stream_t stream, int logistic, int n, int d, int iters, void* state_dev,
                                     double* w_dev, double* m_dev, double* v_dev, double* minv_dev, double* t_dev,
                                     const double* cov_dev, const double* x_dev, const uint8_t* mask_exc_dev,
                                     const uint8_t* mask_inc_dev, double* part_dev, unsigned* sync_dev) {
    return linear_iter_launch((cudaStream_t)stream, logistic, n, d, iters, state_dev, w_dev, m_dev, v_dev, minv_dev, t_dev,
                              cov_dev, x_dev, mask_exc_dev, mask_inc_dev, part_dev, sync_dev, 0, 1, nullptr, nullptr, nullptr);
}

extern "C" size_t dagma_linear_iter_exchange_bytes(int d, int nranks) {
    if (d < 1 || d > LI_MAX_D || nranks < 2 || nranks > LI_MAX_RANKS) return 0;
    return (size_t)2 * nranks * d * d * sizeof(double) + 256;
}

extern "C" int dagma_linear_iter_sharded_f64(dagma_stream_t stream, int n_local, int d, int iters, void* state_dev,
                                             double* w_dev, double* m_dev, double* v_dev, double* minv_dev, double* t_dev,
                                             const double* cov_dev, const double* x_dev, const uint8_t* mask_exc_dev,
                                             const uint8_t* mask_inc_dev, double* part_dev, unsigned* sync_dev, int rank,
                                             int nranks, void* const* exchange_ptrs) {
    DAGMA_REQUIRE(nranks >= 2 && nranks <= LI_MAX_RANKS && rank >= 0 && rank < nranks && exchange_ptrs, "bad rank arguments");
    // layout of a GPU's exchange allocation (dagma_linear_iter_exchange_bytes): [2][nranks][d * d] doubles, then
    // [nranks] flags, then this GPU's own sequence counter
    void* xp[LI_MAX_RANKS];
    void* fp[LI_MAX_RANKS];
    const size_t data = (size_t)2 * nranks * d * d * sizeof(double);
    for (int r = 0; r < nranks; ++r) {
        DAGMA_REQUIRE(exchange_ptrs[r], "null exchange pointer");
        xp[r] = exchange_ptrs[r];
        fp[r] = (char*)exchange_ptrs[r] + data;
    }
    unsigned* seq = (unsigned*)((char*)exchange_ptrs[rank] + data) + 32;
    return linear_iter_launch((cudaStream_t)stream, 1, n_local, d, iters, state_dev, w_dev, m_dev, v_dev, minv_dev, t_dev,
                              cov_dev, x_dev, mask_exc_dev, mask_inc_dev, part_dev, sync_dev, rank, nranks, xp, fp, seq);
}

#ifdef DAGMA_LIN_TRACE
extern "C" int dagma_debug_lin_trace(unsigned long long* out_host) {
    DAGMA_CUDA_OK(cudaDeviceSynchronize());
    DAGMA_CUDA_OK(cudaMemcpyFromSymbol(out_host, g_lin_trace, sizeof(unsigned long long) * 16));
    return 0;
}
#endif
