// Batched DagmaLinear('l2', trek_reg=PST(seq="inv" | "exp", mode="opt") or TCC(cycle_penalty="spectral", mode="opt"))
// .minimize / fit for 1 <= d <= 64: one CTA per
// problem runs the whole schedule (stages, retries, back-tracking, checkpoints) -- the trek-regularised sibling of
// fit_small_dmma_kernel (small_fit_dmma.cu) and fit_small_logistic_kernel (small_fit_logistic.cu), with the same
// contract (dagma_small_fit_args) and the same reference semantics (src/dagma/linear.py:165-333 inner loop, :441-457
// stage loop; quirks Q1-Q7 of SURVEY.md 8), plus the PST term of src/dagma/linear.py:224-276 and
// src/notreks/notreks.py:496-507, 599-619 with the closed-form adjoints of _pst.py.  The kernel is a template on the
// series; everything but the trek block is shared.
//
// seq = "inv":
//   X   = ((1 + eps) I - W o W)^{-1}                (a second block Gauss-Jordan sweep, no domain check)
//   v_p = H[i_p, j_p],  H = X^T X                   (only the m pair values, each a dot product of two columns of X)
//   G_S = G_H + G_H^T                               (pair weights: mean 1/m, sum 1, max ties share, lse softmax(v))
//   GT^T = X^T (X G_S) X^T                          (= (X Gt X)^T with Gt = G_F^T, G_F = X G_S: three DMMA products)
//   Gobj += weight * 2 W o GT^T;  obj += weight * pst(W) at the checkpoints
//
// seq = "exp" (the arithmetic of _pst.PstEngine and oracle/notreks_ref.py, degree-18 Taylor on M = W o W / 2^12 by
// Horner, then 12 squarings):
//   F   = expm(W o W):  R1 = I + M / 18;  R1 <- I + (M R1) / j, j = 17..1;  R1 <- R1 R1 (12 times)      (29 products)
//         (1 / 18 and 1 / j scale as products with the reciprocal, as in _pst.PstEngine)
//   v_p = H[i_p, j_p],  H = F^T F;  G_S as above;  E = (F G_S)^T / 2^12                                  (1 product)
//   GT  = top-right block of expm([[W o W, Gt], [0, W o W]]), Gt = (F G_S)^T, without forming the 2d x 2d matrix:
//         every iterate of the block algorithm is [[R1, R2], [0, R1]], so with R2 = E / 18 at the start
//         Horner   R1 <- I + (M R1) / j,   R2 <- (M R2 + E R1) / j                                       (51 products)
//         squaring R1 <- R1 R1,            R2 <- R1 R2 + R2 R1                                           (36 products)
//         and R2 ends as GT (R1 ends as F again, bit for bit).
//
// Mapping (256 threads, ONE CTA per SM -- the trek buffers take 102 KB (inv: X, G_S, a product buffer) or 136 KB (exp:
// M, R1, G_S / R2, E) of shared memory next to the 87 KB of the l2 sweep; problems pulled from an atomic work queue,
// no grid barriers):
//   * sweep 1 inverts M^T = sI - (W o W)^T with the score GEMM cov (I - W) as filler work, as in the l2 kernel; the
//     gradient without the trek term and the feasibility flag are formed right after it, the former parked in tensor
//     memory next to the Adam moments, so the registers are free for the trek block;
//   * every product accumulates in DMMA registers, then a barrier, then the result is stored in place;
//   * pair weights are scattered into G_S with shared-memory atomics.  Every contribution to one entry comes from pairs
//     with the same unordered key {i, j}, whose values are bit-identical (each computed in the order of (min, max)),
//     so all addends of one entry are equal and their sum does not depend on the order the atomics land in.  The
//     normalisation (1/m, 1/ties, 1/sum exp) is applied to GT^T as one scalar.  inv, mean / sum: G_S is built once
//     per problem and the pair values are only needed at the checkpoints.  exp: G_S shares its buffer with R2, so it
//     is rebuilt every iteration (O(m) atomics next to 117 products).
//
// TCC (the arithmetic of _tcc.SpectralTcc / PerronSolver, src/notreks/notreks.py:156-239, 340-378): the Perron pair of
// A = [[W2, w S], [I, W2^T]], W2 = W o W, by power steps that never form A:
//     v1' = W2 v1 + w S v2,  v2' = v1 + W2^T v2,  u1' = W2^T u1 + u2,  u2' = w S^T u1 + W2 u2,  x <- x' / (||x'|| + eps)
//   from the all-ones vectors at every evaluation, with the schedule of PerronSolver (power: n_iter steps; eig: 8 steps,
//   then chunks of 64 steps on A + rho0 / 4 I until v stops moving, unless rho0 = 0).  Thread t < 128 owns row t of the
//   v chain, thread 128 + t row t of the u chain; each row is a dot product of length d over W2 or W2^T (both kept in
//   shared memory, column access) plus the S part, a walk over the set bits of a 64-bit row / column word of S held in
//   a register.  The squared norms are warp partials summed in warp order: one barrier per step, and every sum has a
//   fixed order and owner, so a problem gives the same bits alone or anywhere in a batch.  The gradient is the rank-2
//   fold 2 W o (u1 v1^T + v2 u2^T) / (m (u.v + eps)) (minus the approx_trek_graph baseline), formed entry by entry in
//   the Adam epilogue; no d x d product.  One solve serves the checkpoint value and the step that follows it.
#include "common.cuh"
#define DAGMA_SWEEP_JIT_ROWS 1        // the score filler's accumulators need the registers of the row fragments
#include "small_dmma.cuh"
#include "fit_step.cuh"
#include "../../include/dagma_b200.h"

namespace dagma {

constexpr int PS_TMEM_COLS = 256;         // per thread: m, v (64 columns) and the gradient without the trek term (32)
constexpr int PST_INV = 0, PST_EXP = 1, TREK_TCC = 2;   // the trek term of a kernel instantiation

struct PstSmem {                          // offsets in doubles; the sweep's buffers keep the offsets of DmmaSmem
    static constexpr int X = DmmaSmem::total;                 // [64][68] X = ((1 + eps) I - W o W)^{-1}
    static constexpr int GS = X + DM_DP * DM_LD;              // [64][68] G_H + G_H^T, un-normalised
    static constexpr int P = GS + DM_DP * DM_LD;              // [64][68] G_F, then G_F X^T
    static constexpr int total = P + DM_DP * DM_LD;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(PstSmem::X % 2 == 0, "16-byte alignment of vector accesses");

struct PstExpSmem {                       // seq = "exp": offsets in doubles after the sweep's buffers
    static constexpr int M = DmmaSmem::total;                 // [64][68] W o W / 2^12
    static constexpr int R1 = M + DM_DP * DM_LD;              // [64][68] Horner / squaring iterate; F after the forward chain
    static constexpr int GS = R1 + DM_DP * DM_LD;             // [64][68] G_H + G_H^T, un-normalised; then R2 (-> GT)
    static constexpr int E = GS + DM_DP * DM_LD;              // [64][68] (F G_S)^T / 2^12
    static constexpr int total = E + DM_DP * DM_LD;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(PstExpSmem::M % 2 == 0, "16-byte alignment of vector accesses");
static_assert(PstExpSmem::bytes + 1024 <= 232448, "one CTA per SM must fit the opt-in shared memory of a block");

struct TccSmem {                          // TCC: offsets in doubles after the sweep's buffers
    static constexpr int W2 = DmmaSmem::total;                // [64][68] W o W
    static constexpr int W2T = W2 + DM_DP * DM_LD;            // [64][68] (W o W)^T
    static constexpr int X = W2T + DM_DP * DM_LD;             // 2 x [256] iterates: v at 0, u at 128 (rows < 2d used)
    static constexpr int VP = X + 2 * 256;                    // [128] v before a chunk
    static constexpr int NRED = VP + 128;                     // 2 x [8] warp partials of the squared norms
    static constexpr int SRED = NRED + 16;                    // [8][3] warp partials of the Perron scalars
    static constexpr int DRED = SRED + 24;                    // [8] warp partials of ||v - v_prev||^2
    static constexpr int SBITS = DRED + 8;                    // [2][64] uint64: rows of S, columns of S
    static constexpr int total = SBITS + 128;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(TccSmem::W2 % 2 == 0 && TccSmem::bytes + 1024 <= 232448, "TCC shared memory layout");

// per-problem parameters of the TCC instantiation (the PST ones ignore them)
struct TccArgs {
    const double* w;                      // [batch] weight of the S block
    const double* eps;                    // [batch] eps of the normalisation and the denominators
    const int32_t* n_iter;                // [batch] steps of method "power"
    const int32_t* flags;                 // [batch] DAGMA_TCC_* bits
    long long* perron_steps;              // [batch] power steps of all solves (may be NULL)
};

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

// Row rr (< 2d) of A x (form 0) or A^T x (form 1) for a 2d-vector x, A = [[W2, w S], [I, W2^T]].  The rows with an S
// part (form 0 top: S row i, form 1 bottom: S column i) walk the set bits of sb in increasing order.  B x is form 0
// with sb = 0.
__device__ __forceinline__ double tcc_row(int form, int rr, int d, const double* W2, const double* W2T,
                                          const double* x, unsigned long long sb, double w) {
    const bool top = rr < d;
    const int i = top ? rr : rr - d;
    const bool srow = (form == 0) == top;
    const double* M = srow ? W2T : W2;                       // M[k][i]: (W2)_{ik} for srow, (W2)_{ki} otherwise
    const double* xh = x + (top ? 0 : d);
    const double* xo = x + (top ? d : 0);
    double acc = 0.0;
#pragma unroll 4
    for (int k = 0; k < d; ++k) acc = fma(M[k * DM_LD + i], xh[k], acc);
    if (!srow) return acc + xo[i];
    double sacc = 0.0;
    while (sb) {
        sacc += xo[__ffsll((long long)sb) - 1];
        sb &= sb - 1;
    }
    return fma(w, sacc, acc);
}

struct TccResult {
    double tval;                          // penalty / m
    double g1, g2;                        // 1 / (m (u.v + eps)), 1 / (m (u.u + eps)) (0 for DAG_learning)
    const double* V;                      // [256] normalised v (0..2d), u (128..128 + 2d)
    int steps;
    bool cap;
};

// The Perron solve of one evaluation at Ws (PerronSolver.power / .converged, then SpectralTcc.compute / .value).
// Uniform control flow: every decision reads values all threads computed in the same order.
__device__ TccResult tcc_perron(double* smem, const double* Ws, int d, int m, double w, double eps, int n_iter,
                                int flags, unsigned long long sb, int tid) {
    constexpr int LD = DM_LD;
    double* W2 = smem + TccSmem::W2;
    double* W2T = smem + TccSmem::W2T;
    double* X = smem + TccSmem::X;
    double* VP = smem + TccSmem::VP;
    double* nred = smem + TccSmem::NRED;
    double* sred = smem + TccSmem::SRED;
    double* dred = smem + TccSmem::DRED;
    const int chain = tid >> 7, rr = tid & 127, warp = tid >> 5, lane = tid & 31;
    const bool active = rr < 2 * d;
    for (int idx = tid; idx < d * d; idx += DM_NT) {
        const int r = idx / d, c = idx - r * d;
        const double x = Ws[r * LD + c];
        W2[r * LD + c] = x * x;
        W2T[c * LD + r] = x * x;
    }
    if (active) X[128 * chain + rr] = 1.0;
    __syncthreads();
    int cur = 0;
    bool unit = true;                     // X[cur] is used as it stands (ones, or normalised vectors)
    auto inv_norm = [&]() -> double {
        if (unit) return 1.0;
        const double* q = nred + 8 * cur + 4 * chain;
        return 1.0 / (sqrt(((q[0] + q[1]) + q[2]) + q[3]) + eps);
    };
    // n steps x <- (A x + shift x) / (||.|| + eps) of both chains (the division deferred to the next reader)
    auto steps = [&](int n, double shift) {
#pragma unroll 1
        for (int k = 0; k < n; ++k) {
            const double sc = inv_norm();
            const double* x = X + 256 * cur + 128 * chain;
            double y = 0.0;
            if (active) {
                double acc = tcc_row(chain, rr, d, W2, W2T, x, sb, w);
                if (shift != 0.0) acc = fma(shift, x[rr], acc);
                y = acc * sc;
                X[256 * (cur ^ 1) + 128 * chain + rr] = y;
            }
            const double q = warp_sum(y * y);
            if (lane == 0) nred[8 * (cur ^ 1) + warp] = q;
            __syncthreads();
            cur ^= 1;
            unit = false;
        }
    };
    auto finish = [&]() {                 // normalise in place: X[cur] = v, u
        const double sc = inv_norm();
        if (active) X[256 * cur + 128 * chain + rr] *= sc;
        __syncthreads();
        unit = true;
    };
    double vav = 0.0, vv = 0.0, uv = 0.0, ubu = 0.0, uu = 0.0;
    auto scalars = [&]() {                // v.Av, v.v, u.v (v chain); u.Bu, u.u (u chain)
        const double* V = X + 256 * cur;
        double p0 = 0.0, p1 = 0.0, p2 = 0.0;
        if (active) {
            if (chain == 0) {
                const double vr = V[rr];
                p0 = vr * tcc_row(0, rr, d, W2, W2T, V, sb, w);
                p1 = vr * vr;
                p2 = V[128 + rr] * vr;
            } else {
                const double ur = V[128 + rr];
                p0 = ur * tcc_row(0, rr, d, W2, W2T, V + 128, 0ull, w);
                p1 = ur * ur;
            }
        }
        p0 = warp_sum(p0);
        p1 = warp_sum(p1);
        p2 = warp_sum(p2);
        if (lane == 0) { sred[3 * warp] = p0; sred[3 * warp + 1] = p1; sred[3 * warp + 2] = p2; }
        __syncthreads();
        vav = ((sred[0] + sred[3]) + sred[6]) + sred[9];
        vv = ((sred[1] + sred[4]) + sred[7]) + sred[10];
        uv = ((sred[2] + sred[5]) + sred[8]) + sred[11];
        ubu = ((sred[12] + sred[15]) + sred[18]) + sred[21];
        uu = ((sred[13] + sred[16]) + sred[19]) + sred[22];
        __syncthreads();                  // sred is free again
    };
    TccResult res;
    res.cap = false;
    if (flags & DAGMA_TCC_POWER) {
        const int n = n_iter > 0 ? n_iter : 0;
        steps(n, 0.0);
        finish();
        scalars();
        res.steps = n;
    } else {
        steps(DAGMA_TCC_EIG_WARMUP, 0.0);
        finish();
        scalars();
        res.steps = DAGMA_TCC_EIG_WARMUP;
        const double rho0 = fabs(vav / (vv + eps));
        if (rho0 > DAGMA_TCC_EIG_NILPOTENT) {   // else nilpotent: the warm-up vectors stand (PerronSolver.converged)
            const double shift = DAGMA_TCC_EIG_SHIFT * rho0;
            bool conv = false;
#pragma unroll 1
            for (int c = 0; c < DAGMA_TCC_EIG_MAX_CHUNKS && !conv; ++c) {
                if (chain == 0 && active) VP[rr] = X[256 * cur + rr];
                steps(DAGMA_TCC_EIG_CHUNK, shift);   // (its first barrier orders VP before the reads below)
                finish();
                res.steps += DAGMA_TCC_EIG_CHUNK;
                double df = 0.0;
                if (chain == 0 && active) {
                    const double e = X[256 * cur + rr] - VP[rr];
                    df = e * e;
                }
                df = warp_sum(df);
                if (lane == 0) dred[warp] = df;
                __syncthreads();
                const double dn = ((dred[0] + dred[1]) + dred[2]) + dred[3];
                conv = dn <= DAGMA_TCC_EIG_TOL * DAGMA_TCC_EIG_TOL;
                __syncthreads();              // dred is free again
            }
            res.cap = !conv;
            scalars();
        }
    }
    const double rm = 1.0 / (double)m;
    const bool approx = !(flags & DAGMA_TCC_DAG_LEARNING);
    const double rho = vav / (vv + eps);
    res.tval = (approx ? rho - ubu / (uu + eps) : rho) * rm;
    res.g1 = rm / (uv + eps);
    res.g2 = approx ? rm / (uu + eps) : 0.0;
    res.V = X + 256 * cur;
    return res;
}

// acc = A B over k < 4 nk on DMMA.8x8x4, accumulator ownership of DmmaPos; A(r, k) = TA ? A[k][r] : A[r][k] and
// B(k, c) = TB ? B[c][k] : B[k][c], both [64][DM_LD].  Warps whose tiles lie outside d x d get zeros.
template <bool TA, bool TB>
__device__ __forceinline__ void pst_product(double (&acc)[2][4][2], const DmmaPos& ps, const double* A, const double* B,
                                            int d) {
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) acc[ti][tj][0] = acc[ti][tj][1] = 0.0;
    if (16 * ps.wr >= d || 32 * ps.wc >= d) return;
    const int nk = (d + 3) >> 2;
#pragma unroll 2
    for (int kb = 0; kb < nk; ++kb) {
        const int k = 4 * kb + ps.qc;
        double a[2], b[4];
#pragma unroll
        for (int ti = 0; ti < 2; ++ti) {
            const int r = ps.row(ti);
            a[ti] = TA ? A[k * DM_LD + r] : A[r * DM_LD + k];
        }
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int c = 32 * ps.wc + 8 * tj + ps.qr;
            b[tj] = TB ? B[c * DM_LD + k] : B[k * DM_LD + c];
        }
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)
#pragma unroll
            for (int tj = 0; tj < 4; ++tj) dmma(acc[ti][tj][0], acc[ti][tj][1], a[ti], b[tj]);
    }
}

__device__ __forceinline__ void store_tiles(double* dst, const double (&acc)[2][4][2], const DmmaPos& ps) {
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
            *reinterpret_cast<double2*>(dst + ps.row(ti) * DM_LD + ps.col(tj)) = make_double2(acc[ti][tj][0], acc[ti][tj][1]);
}

// H[i][j] = sum_k X[k][i] X[k][j] in the order of the unordered pair: (i, j) and (j, i) give the same bits
__device__ __forceinline__ double pair_value(const double* Xs, int d, int i, int j) {
    const int lo = min(i, j), hi = max(i, j);
    double v = 0.0;
#pragma unroll 4
    for (int k = 0; k < d; ++k) v = fma(Xs[k * DM_LD + lo], Xs[k * DM_LD + hi], v);
    return v;
}

__device__ __forceinline__ void scatter_pair(double* GS, int i, int j, double g) {
    atomicAdd(GS + i * DM_LD + j, g);       // G_H
    atomicAdd(GS + j * DM_LD + i, g);       // G_H^T
}

// u = A1 B1 and t = A1 B2 + A2 B1 in one pass over k (operands as pst_product with TA = TB = false): a step of the
// coupled exp chain -- Horner (A1, A2, B1, B2) = (M, E, R1, R2), squaring (R1, R2, R1, R2)
__device__ __forceinline__ void pst_coupled_product(double (&u)[2][4][2], double (&t)[2][4][2], const DmmaPos& ps,
                                                    const double* A1, const double* A2, const double* B1,
                                                    const double* B2, int d) {
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) u[ti][tj][0] = u[ti][tj][1] = t[ti][tj][0] = t[ti][tj][1] = 0.0;
    if (16 * ps.wr >= d || 32 * ps.wc >= d) return;
    const int nk = (d + 3) >> 2;
#pragma unroll 1
    for (int kb = 0; kb < nk; ++kb) {
        const int k = 4 * kb + ps.qc;
        double a1[2], a2[2], b1[4], b2[4];
#pragma unroll
        for (int ti = 0; ti < 2; ++ti) {
            a1[ti] = A1[ps.row(ti) * DM_LD + k];
            a2[ti] = A2[ps.row(ti) * DM_LD + k];
        }
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int c = 32 * ps.wc + 8 * tj + ps.qr;
            b1[tj] = B1[k * DM_LD + c];
            b2[tj] = B2[k * DM_LD + c];
        }
#pragma unroll
        for (int ti = 0; ti < 2; ++ti)
#pragma unroll
            for (int tj = 0; tj < 4; ++tj) {
                dmma(u[ti][tj][0], u[ti][tj][1], a1[ti], b1[tj]);
                dmma(t[ti][tj][0], t[ti][tj][1], a1[ti], b2[tj]);
                dmma(t[ti][tj][0], t[ti][tj][1], a2[ti], b1[tj]);
            }
    }
}

// dst = I_d + acc * (1 / j)  (a Horner step of the Taylor polynomial, scaled as _pst.PstEngine scales it: by the
// reciprocal -- a division sends the many exact zeros of the padded tiles down its slow path; the identity only
// inside d x d, so the padding stays 0)
__device__ __forceinline__ void store_horner(double* dst, const double (&acc)[2][4][2], const DmmaPos& ps, int d,
                                             double rj) {
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) {
            const int r = ps.row(ti), c = ps.col(tj);
            const double i0 = (r == c && r < d) ? 1.0 : 0.0, i1 = (r == c + 1 && r < d) ? 1.0 : 0.0;
            *reinterpret_cast<double2*>(dst + r * DM_LD + c) = make_double2(i0 + acc[ti][tj][0] * rj,
                                                                              i1 + acc[ti][tj][1] * rj);
        }
}

__device__ __forceinline__ void store_scaled(double* dst, const double (&acc)[2][4][2], const DmmaPos& ps, double rj) {
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
            *reinterpret_cast<double2*>(dst + ps.row(ti) * DM_LD + ps.col(tj)) =
                make_double2(acc[ti][tj][0] * rj, acc[ti][tj][1] * rj);
}

// R1 = I_d + M * (1 / 18) (both [64][DM_LD], whole padded square); the start of both Horner chains
__device__ __forceinline__ void exp_horner_start(double* R1, const double* M, int d, int tid) {
    constexpr double RDEG = 1.0 / (double)DAGMA_PST_EXP_DEGREE;
    for (int idx = tid; idx < DM_DP * DM_DP; idx += DM_NT) {
        const int r = idx >> 6, c = idx & 63;
        R1[r * DM_LD + c] = ((r == c && r < d) ? 1.0 : 0.0) + M[r * DM_LD + c] * RDEG;
    }
}

template <int SEQ>
__global__ void __launch_bounds__(DM_NT, 1) fit_small_pst_kernel(const dagma_small_fit_args P,
                                                                  const int32_t* __restrict__ pair_off,
                                                                  const int32_t* __restrict__ pairs,
                                                                  const double* __restrict__ trek_weight, int agg,
                                                                  double eps_inv, const TccArgs tcc) {
    using S = DmmaSmem;
    constexpr bool EXP = SEQ == PST_EXP;
    constexpr bool TCC = SEQ == TREK_TCC;
    constexpr int NT = DM_NT, LD = DM_LD;
    extern __shared__ __align__(16) double smem[];
    double* ncov = smem + S::ncov;
    double* Ws = smem + S::W;
    double* pinfo = smem + S::pinfo;
    double* red = smem + S::red;
    double* Xs = smem + PstSmem::X;
    double* GS = smem + (EXP ? PstExpSmem::GS : PstSmem::GS);
    double* Ps = smem + PstSmem::P;
    double* Ms = smem + PstExpSmem::M;                       // exp only
    double* R1s = smem + PstExpSmem::R1;
    double* Es = smem + PstExpSmem::E;
    const double* Fs = EXP ? R1s : Xs;                       // the columns the pair values are dot products of
    __shared__ unsigned s_prob;
    __shared__ uint32_t s_tmem;
    // Adam bias correction, kept by one lane (see fit_small_dmma_kernel)
    __shared__ double s_pow[4];
    __shared__ double s_pow_next[4];
    __shared__ double s_bias[2][2];

    const int tid = threadIdx.x;
    const DmmaPos ps(tid);
    const int d = P.d;
    const int np = 4 * ((d + 3) >> 2);
    const size_t dd = (size_t)d * d;
    const bool pair_agg = !TCC && (agg == DAGMA_PST_MAX || agg == DAGMA_PST_LSE);   // G_S depends on the pair values
    unsigned long long* sbits = reinterpret_cast<unsigned long long*>(smem + TccSmem::SBITS);   // TCC only

    SweepSync sy{smem_u32(smem + S::mbar), 0u};
    if (tid == 0) mbar_init(sy.bar, NT / 32);

    if (ps.warp == 0) tmem_alloc<PS_TMEM_COLS>(smem_u32(&s_tmem));
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    const uint32_t tmem_base = s_tmem;
    // columns of a thread: [m(ti=0) 16 | v(ti=0) 16 | m(ti=1) 16 | v(ti=1) 16 | Gobj0(ti=0) 16 | Gobj0(ti=1) 16]
    const uint32_t tm = tmem_base + ((uint32_t)(32 * (ps.warp & 3)) << 16) + (uint32_t)((ps.warp >> 2) * 96);
    const uint32_t tg = tm + 64;

    unsigned excbits = 0, incbits = 0;
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = ps.row(ti), c = ps.col(tj) + e;
                if (r < d && c < d) {
                    if (P.mask_exc_dev && P.mask_exc_dev[r * d + c]) excbits |= 1u << (ti * 8 + tj * 2 + e);
                    if (P.mask_inc_dev && P.mask_inc_dev[r * d + c]) incbits |= 1u << (ti * 8 + tj * 2 + e);
                }
            }

    for (;;) {
        if (tid == 0) s_prob = atomicAdd(P.work_counter_dev, 1u);
        __syncthreads();
        const unsigned b = s_prob;
        __syncthreads();
        if (b >= (unsigned)P.batch) break;

        const double* cov_g = P.cov_dev + (size_t)b * dd;
        double* W_g = P.w_dev + (size_t)b * dd;
        const double lambda1 = P.lambda1_dev[b];
        const int p0 = pair_off[b];
        const int m = pair_off[b + 1] - p0;
        const int2* pr = reinterpret_cast<const int2*>(pairs) + p0;
        const double weight = trek_weight[b];

        for (int idx = tid; idx < DM_DP * DM_DP; idx += NT) {
            const int r = idx >> 6, c = idx & 63;
            const bool in = (r < d) && (c < d);
            ncov[r * LD + c] = in ? -cov_g[r * d + c] : 0.0;
            Ws[r * LD + c] = in ? W_g[r * d + c] : 0.0;
        }
        double tcc_w = 0.0, tcc_eps = 0.0;
        int tcc_n_iter = 0, tcc_flags = 0;
        long long perron_steps = 0;
        unsigned long long sb = 0;
        if constexpr (TCC) {
            tcc_w = tcc.w[b];
            tcc_eps = tcc.eps[b];
            tcc_n_iter = tcc.n_iter[b];
            tcc_flags = tcc.flags[b];
            if (tid < 128) sbits[tid] = 0ull;
            __syncthreads();
            for (int p = tid; p < m; p += NT) {      // S[i][j] = 1 (duplicates set the same bit)
                const int2 ij = pr[p];
                atomicOr(sbits + ij.x, 1ull << ij.y);          // row i of S
                atomicOr(sbits + 64 + ij.y, 1ull << ij.x);     // column j of S
            }
            __syncthreads();
            const int rr = tid & 127;
            if (tid < 128 && rr < d) sb = sbits[rr];                         // v chain, top rows: S rows
            if (tid >= 128 && rr >= d && rr < 2 * d) sb = sbits[64 + rr - d];   // u chain, bottom rows: S columns
        } else {
            for (int e = tid; e < DM_DP * LD; e += NT) GS[e] = 0.0;
        }
        __syncthreads();
        if (!EXP && !TCC && m > 0 && !pair_agg) {               // inv, mean / sum: G_S counts the pairs, fixed for the problem
            for (int p = tid; p < m; p += NT) {
                const int2 ij = pr[p];
                scatter_pair(GS, ij.x, ij.y, 1.0);
            }
        }
        __syncthreads();

        double a[2][4][2], g[2][4][2];
        int status = 0;
        int n_ckpt = 0;

        int stage = 0;
        bool final_phase = (P.n_stages == 0);
        double mu = 0, s_cur = 1, lr = 0, lr_adam = P.lr, obj_prev = 1e16;
        double last_obj = 0, last_score = 0, last_h = 0;
        int iters_max = 0, it = 0, retries = 0, backtracks = 0;
        bool in_backtrack = false;

        auto start_attempt = [&]() {
            it = 0;
            lr = lr_adam;
            obj_prev = 1e16;
            in_backtrack = false;
            backtracks = 0;
            if (tid == DM_NT - 32) { s_pow[0] = 1.0; s_pow[1] = 0.0; s_pow[2] = 1.0; s_pow[3] = 0.0; }
            const double z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int q = 0; q < 4; ++q) tmem_st8(tm + 16 * q, z);
            tmem_wait_st();
        };
        auto start_stage = [&]() {
            mu = P.mu[stage];
            s_cur = P.s[stage];
            iters_max = P.iters[stage];
            lr_adam = P.lr;
            retries = 0;
            start_attempt();
        };
        auto write_W = [&]() {
            __syncthreads();
            for (int idx = tid; idx < d * d; idx += NT) {
                const int r = idx / d, c = idx - r * d;
                W_g[idx] = Ws[r * LD + c];
            }
        };
        auto read_W = [&]() {
            __syncthreads();
            for (int idx = tid; idx < d * d; idx += NT) {
                const int r = idx / d, c = idx - r * d;
                Ws[r * LD + c] = W_g[idx];
            }
            __syncthreads();
        };
        auto write_stage_stats = [&]() {
            if (tid == 0 && P.stage_stats_dev) {
                double* st = P.stage_stats_dev + ((size_t)b * P.n_stages + stage) * 8;
                st[0] = (double)it;
                st[1] = lr;
                st[2] = s_cur;
                st[3] = last_obj;
                st[4] = last_score;
                st[5] = last_h;
                st[6] = (double)retries;
                st[7] = (double)backtracks;
            }
        };
        // Ws += scale * dir(m, v, it): the previous Adam direction rebuilt from the moments
        auto apply_dir = [&](double scale) {
            const double c1 = s_bias[it & 1][0] * (1.0 - P.beta1), c2 = s_bias[it & 1][1] * (1.0 - P.beta2);
#pragma unroll
            for (int ti = 0; ti < 2; ++ti) {
                TmemLoad8 lm, lv;
                lm.issue(tm + 32 * ti);
                lv.issue(tm + 32 * ti + 16);
                lm.finish();
                lv.finish();
                double* wp = Ws + ps.row(ti) * LD;
#pragma unroll
                for (int tj = 0; tj < 4; ++tj) {
                    double2 w = *reinterpret_cast<double2*>(wp + ps.col(tj));
                    const double d0 = fast_div(lm.get(2 * tj) * c1, fast_sqrt_nonneg(lv.get(2 * tj) * c2) + 1e-8);
                    const double d1 = fast_div(lm.get(2 * tj + 1) * c1, fast_sqrt_nonneg(lv.get(2 * tj + 1) * c2) + 1e-8);
                    w.x = __dadd_rn(w.x, __dmul_rn(scale, d0));
                    w.y = __dadd_rn(w.y, __dmul_rn(scale, d1));
                    *reinterpret_cast<double2*>(wp + ps.col(tj)) = w;
                }
            }
            __syncthreads();
        };

        if (!final_phase) start_stage();

        for (;;) {
            const double s_use = final_phase ? 1.0 : s_cur;
            const bool at_ckpt = !final_phase && !in_backtrack && it >= 1 &&
                                 (it % P.checkpoint == 0 || it == iters_max);
            // ================= sweep 1: M^{-T}, with g = cov (I - W) as filler work =================
#pragma unroll
            for (int ti = 0; ti < 2; ++ti) {
                const int r = ps.row(ti);
#pragma unroll
                for (int tj = 0; tj < 4; ++tj) {
                    const int c = ps.col(tj);
                    const double w0 = Ws[c * LD + r], w1 = Ws[(c + 1) * LD + r];     // W^T
                    const double dg = (r < d) ? s_use : 1.0;
                    a[ti][tj][0] = ((r == c) ? dg : 0.0) - w0 * w0;
                    a[ti][tj][1] = ((r == c + 1) ? dg : 0.0) - w1 * w1;
                    const double2 nc = *reinterpret_cast<const double2*>(ncov + r * LD + c);
                    g[ti][tj][0] = -nc.x;
                    g[ti][tj][1] = -nc.y;
                }
            }
            if (tid == DM_NT - 32 && !final_phase) {      // bias factors of iteration it + 1
                DD q1{s_pow[0], s_pow[1]}, q2{s_pow[2], s_pow[3]};
                q1.mul(P.beta1);
                q2.mul(P.beta2);
                s_pow_next[0] = q1.hi; s_pow_next[1] = q1.lo; s_pow_next[2] = q2.hi; s_pow_next[3] = q2.lo;
                s_bias[(it + 1) & 1][0] = fast_rcp(q1.one_minus());
                s_bias[(it + 1) & 1][1] = fast_rcp(q2.one_minus());
            }
            {
                ScoreFill fill{g, ps, smem, 0, (d + 3) >> 2};
                dmma_sweep(a, ps, smem, d, sy, fill);
#pragma unroll 1
                while (fill.more()) fill.unit();
            }
            // now: a = M^{-T},  g = cov (I - W),  pinfo[0..np) = pivots

            // ================= objective without the trek term (checkpoint / final) =================
            double score = 0.0, h = 0.0, l1 = 0.0;
            if (at_ckpt || final_phase) {
                double sc = 0.0, ld = 0.0;
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) {
                    const int r = ps.row(ti);
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        const int c = ps.col(tj);
                        const double2 w = *reinterpret_cast<const double2*>(Ws + r * LD + c);
                        const double dif0 = ((r == c && r < d) ? 1.0 : 0.0) - w.x;
                        const double dif1 = ((r == c + 1 && r < d) ? 1.0 : 0.0) - w.y;
                        sc = fma(dif0, g[ti][tj][0], sc);
                        sc = fma(dif1, g[ti][tj][1], sc);
                        l1 += fabs(w.x) + fabs(w.y);
                    }
                }
                if (tid < np) ld = (double)((tid & 3) - 2) * log(fabs(pinfo[tid]));
                block_sum3<NT>(sc, l1, ld, red, tid);
                score = 0.5 * sc;
                h = -ld + (double)d * log(s_use);
                if (final_phase) {
                    if (tid == 0 && P.final_dev) {
                        P.final_dev[2 * (size_t)b] = h;
                        P.final_dev[2 * (size_t)b + 1] = score;
                    }
                    break;
                }
            }

            // ================= feasibility of iteration it + 1 (sweep 2 overwrites pinfo) =================
            bool bad = false;
            if (tid < np) bad = !(pinfo[tid] > 0.0);
#pragma unroll
            for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                for (int tj = 0; tj < 4; ++tj)
                    bad |= below_minus_1e16(a[ti][tj][0]) | below_minus_1e16(a[ti][tj][1]);
            bad = __syncthreads_or(bad);

            if (!bad) {
                // Gobj without the trek term = -mu cov (I - W) + mu l1 sign(W) + 2 W o (M^{-T} + 1e-16) (+ include
                // mask), linear.py:248, parked in tensor memory while sweep 2 needs the registers
                const double l1c = mu * lambda1, incc = -2.0 * mu * lambda1, nmu = -mu;
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) {
                    const double* wp = Ws + ps.row(ti) * LD;
                    double go[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const double w = wp[ps.col(q >> 1) + (q & 1)];
                        go[q] = fma(nmu, g[ti][q >> 1][q & 1], signed_const(w, l1c));
                        go[q] = fma(twice(w), a[ti][q >> 1][q & 1] + 1e-16, go[q]);
                        if (incbits >> (ti * 8 + q) & 1u) go[q] += signed_const(w, incc);
                    }
                    tmem_st8(tg + 16 * ti, go);
                }
                tmem_wait_st();
            }

            // ================= PST (inv / exp) or TCC at the current W =================
            double tval = 0.0, tscale = 0.0;
            double t[2][4][2];
            TccResult tr;
            const bool trek = m > 0 && (at_ckpt || !bad);
            if (TCC && trek) {
                tr = tcc_perron(smem, Ws, d, m, tcc_w, tcc_eps, tcc_n_iter, tcc_flags, sb, tid);
                perron_steps += tr.steps;
                if (tr.cap) status |= DAGMA_ST_PERRON_CAP;
                tval = tr.tval;
            } else if (trek) {
                if constexpr (!EXP) {
                    const double dgx = 1.0 + eps_inv;
#pragma unroll
                    for (int ti = 0; ti < 2; ++ti) {
                        const int r = ps.row(ti);
#pragma unroll
                        for (int tj = 0; tj < 4; ++tj) {
                            const int c = ps.col(tj);
                            const double2 w = *reinterpret_cast<const double2*>(Ws + r * LD + c);
                            const double dg = (r < d) ? dgx : 1.0;
                            a[ti][tj][0] = ((r == c) ? dg : 0.0) - w.x * w.x;
                            a[ti][tj][1] = ((r == c + 1) ? dg : 0.0) - w.y * w.y;
                        }
                    }
                    dmma_sweep(a, ps, smem, d, sy);
                    store_tiles(Xs, a, ps);
                    if (pair_agg)
                        for (int idx = tid; idx < d * d; idx += NT) GS[(idx / d) * LD + idx % d] = 0.0;
                    __syncthreads();
                } else {
                    // F = expm(W o W): M = W o W / 2^12, R1 = I + M / 18, Horner j = 17..1, 12 squarings.  G_S is
                    // cleared meanwhile: its buffer held R2 of the previous iteration (the padding stays 0).
                    constexpr double SC = 1.0 / (double)(1 << DAGMA_PST_EXP_SQUARINGS);
                    for (int idx = tid; idx < DM_DP * DM_DP; idx += NT) {
                        const double w = Ws[(idx >> 6) * LD + (idx & 63)];
                        Ms[(idx >> 6) * LD + (idx & 63)] = (w * w) * SC;
                    }
                    for (int idx = tid; idx < d * d; idx += NT) GS[(idx / d) * LD + idx % d] = 0.0;
                    __syncthreads();
                    exp_horner_start(R1s, Ms, d, tid);
                    __syncthreads();
#pragma unroll 1
                    for (int j = DAGMA_PST_EXP_DEGREE - 1; j >= 1; --j) {
                        pst_product<false, false>(t, ps, Ms, R1s, d);
                        __syncthreads();
                        store_horner(R1s, t, ps, d, 1.0 / (double)j);
                        __syncthreads();
                    }
#pragma unroll 1
                    for (int q = 0; q < DAGMA_PST_EXP_SQUARINGS; ++q) {
                        pst_product<false, false>(t, ps, R1s, R1s, d);
                        __syncthreads();
                        store_tiles(R1s, t, ps);
                        __syncthreads();
                    }
                    if (!pair_agg) {                        // mean / sum: G_S counts the pairs
                        for (int p = tid; p < m; p += NT) {
                            const int2 ij = pr[p];
                            scatter_pair(GS, ij.x, ij.y, 1.0);
                        }
                        __syncthreads();
                    }
                }
                // pair values -> value and the un-normalised pair weights; tscale = weight x normalisation
                if (!pair_agg) {
                    if (at_ckpt) {
                        double sv = 0.0, z1 = 0.0, z2 = 0.0;
                        for (int p = tid; p < m; p += NT) {
                            const int2 ij = pr[p];
                            sv += pair_value(Fs, d, ij.x, ij.y);
                        }
                        block_sum3<NT>(sv, z1, z2, red, tid);
                        tval = (agg == DAGMA_PST_MEAN) ? sv / (double)m : sv;
                    }
                    tscale = (agg == DAGMA_PST_MEAN) ? weight / (double)m : weight;
                } else {
                    double mx = -INFINITY;
                    for (int p = tid; p < m; p += NT) {
                        const int2 ij = pr[p];
                        mx = fmax(mx, pair_value(Fs, d, ij.x, ij.y));
                    }
                    mx = block_max<NT>(mx, red, tid);
                    double se = 0.0, z1 = 0.0, z2 = 0.0;
                    for (int p = tid; p < m; p += NT) {
                        const int2 ij = pr[p];
                        const double v = pair_value(Fs, d, ij.x, ij.y);
                        if (agg == DAGMA_PST_MAX) {
                            if (v == mx) {                  // torch shares the gradient of max() between ties
                                se += 1.0;
                                scatter_pair(GS, ij.x, ij.y, 1.0);
                            }
                        } else {
                            const double e = exp(v - mx);
                            se += e;
                            scatter_pair(GS, ij.x, ij.y, e);
                        }
                    }
                    block_sum3<NT>(se, z1, z2, red, tid);   // (its barriers also publish the scatter)
                    tval = (agg == DAGMA_PST_MAX) ? mx : mx + log(se);
                    tscale = weight / se;
                }
                if constexpr (!EXP) {
                    // GT^T = X^T (X G_S) X^T
                    pst_product<false, false>(t, ps, Xs, GS, d);       // G_F = X G_S
                    store_tiles(Ps, t, ps);
                    __syncthreads();
                    pst_product<false, true>(t, ps, Ps, Xs, d);        // U = G_F X^T
                    __syncthreads();
                    store_tiles(Ps, t, ps);
                    __syncthreads();
                    pst_product<true, false>(t, ps, Xs, Ps, d);        // GT^T = X^T U
                } else if (!bad) {                          // (an infeasible iterate only needs the value)
                    constexpr double SC = 1.0 / (double)(1 << DAGMA_PST_EXP_SQUARINGS);
                    constexpr double RDEG = 1.0 / (double)DAGMA_PST_EXP_DEGREE;
                    pst_product<false, false>(t, ps, R1s, GS, d);      // G_F = F G_S
                    __syncthreads();
                    // E = G_F^T / 2^12 and R2 = E * (1 / 18) (over G_S, dead now); R1 restarts at I + M * (1 / 18)
#pragma unroll
                    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int at = (ps.col(tj) + e) * LD + ps.row(ti);
                                const double ev = t[ti][tj][e] * SC;
                                Es[at] = ev;
                                GS[at] = ev * RDEG;
                            }
                    exp_horner_start(R1s, Ms, d, tid);
                    __syncthreads();
                    double u[2][4][2];
#pragma unroll 1
                    for (int j = DAGMA_PST_EXP_DEGREE - 1; j >= 1; --j) {
                        pst_coupled_product(u, t, ps, Ms, Es, R1s, GS, d);    // M R1,  M R2 + E R1
                        __syncthreads();
                        const double rj = 1.0 / (double)j;
                        store_horner(R1s, u, ps, d, rj);
                        store_scaled(GS, t, ps, rj);
                        __syncthreads();
                    }
#pragma unroll 1
                    for (int q = 0; q < DAGMA_PST_EXP_SQUARINGS; ++q) {
                        pst_coupled_product(u, t, ps, R1s, GS, R1s, GS, d);   // R1 R1,  R1 R2 + R2 R1
                        __syncthreads();
                        store_tiles(R1s, u, ps);
                        store_tiles(GS, t, ps);
                        __syncthreads();
                    }
                    // GT^T fragments for the Adam epilogue
#pragma unroll
                    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
                            for (int e = 0; e < 2; ++e) t[ti][tj][e] = GS[(ps.col(tj) + e) * LD + ps.row(ti)];
                }
            }

            if (at_ckpt) {
                const double obj = mu * (score + lambda1 * l1) + h + weight * tval;
                last_obj = obj;
                last_score = score;
                last_h = h;
                if (tid == 0 && P.ckpt_log_dev && n_ckpt < P.ckpt_log_cap) {
                    double* row = P.ckpt_log_dev + ((size_t)b * P.ckpt_log_cap + n_ckpt) * 6;
                    row[0] = stage; row[1] = it; row[2] = obj; row[3] = score; row[4] = h; row[5] = lr;
                }
                ++n_ckpt;
                const bool converged = fabs((obj_prev - obj) / obj_prev) <= P.tol;
                obj_prev = obj;
                if (converged || it == iters_max) goto stage_done;
            } else if (!in_backtrack && it == iters_max) {
                goto stage_done;   // only reachable for iters_max == 0
            }

            if (bad) {
                if (it == 0 || s_cur <= 0.9) {            // linear.py:231-233
                    if (P.retry_on_fail) {
                        if (++retries > 64) {
                            status |= DAGMA_ST_RETRY_LIMIT;
                            --retries;
                            read_W();
                            write_stage_stats();
                            if (!P.final_dev) goto problem_done;
                            final_phase = true;
                            continue;
                        }
                        lr_adam *= 0.5;                    // linear.py:450-451
                        s_cur += 0.1;
                        read_W();
                        start_attempt();
                        continue;
                    }
                    status |= DAGMA_ST_OUT_OF_DOMAIN;
                    write_W();
                    write_stage_stats();
                    goto problem_done;
                }
                apply_dir(lr);                             // W += lr * grad   :235
                lr *= 0.5;                                 //                  :236
                if (lr <= 1e-16) {                         //                  :237-238
                    status |= DAGMA_ST_LR_UNDERFLOW;
                    goto stage_done;
                }
                apply_dir(-lr);                            // W -= lr * grad   :239
                ++backtracks;
                in_backtrack = true;
                continue;                                  // re-invert        :240
            }
            in_backtrack = false;

            {
                // ================= Adam step (iteration it + 1) =================
                ++it;
                const double k1 = s_bias[it & 1][0] * (1.0 - P.beta1), k2 = s_bias[it & 1][1] * (1.0 - P.beta2);
                if (tid == DM_NT - 32) {
                    s_pow[0] = s_pow_next[0]; s_pow[1] = s_pow_next[1]; s_pow[2] = s_pow_next[2]; s_pow[3] = s_pow_next[3];
                }
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) {
                    TmemLoad8 lm, lv, lg;
                    lg.issue(tg + 16 * ti);
                    lm.issue(tm + 32 * ti);
                    lv.issue(tm + 32 * ti + 16);
                    double* wp = Ws + ps.row(ti) * LD;
                    double w[8], go[8], mn[8], vn[8];
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        const double2 v2 = *reinterpret_cast<const double2*>(wp + ps.col(tj));
                        w[2 * tj] = v2.x;
                        w[2 * tj + 1] = v2.y;
                    }
                    lg.finish();
#pragma unroll
                    for (int q = 0; q < 8; ++q) go[q] = lg.get(q);
                    if (TCC && trek) {                     // + weight * 2 W o (rank-2 fold)   (_tcc.SpectralTcc.compute)
                        const double* v = tr.V;
                        const double* u = tr.V + 128;
                        const int r = ps.row(ti);
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const int c = ps.col(q >> 1) + (q & 1);
                            if (r < d && c < d) {
                                const double g = tr.g1 * fma(u[r], v[c], v[d + r] * u[d + c]) -
                                                 tr.g2 * fma(u[r], u[c], u[d + r] * u[d + c]);
                                go[q] = fma(twice(w[q]), weight * g, go[q]);
                            }
                        }
                    } else if (trek) {                     // + weight * 2 W o GT^T   (linear.py:251-258)
#pragma unroll
                        for (int q = 0; q < 8; ++q) go[q] = fma(twice(w[q]), tscale * t[ti][q >> 1][q & 1], go[q]);
                    }
                    lm.finish();
                    lv.finish();
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        mn[q] = lm.get(q);
                        vn[q] = lv.get(q);
                    }
#pragma unroll
                    for (int q0 = 0; q0 < 8; q0 += DAGMA_ADAM_GROUP)
                        adam_entries<DAGMA_ADAM_GROUP>(w + q0, go + q0, mn + q0, vn + q0, P.beta1, P.beta2, k1, k2, lr);
                    tmem_st8(tm + 32 * ti, mn);
                    tmem_st8(tm + 32 * ti + 16, vn);
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        double2 v2 = make_double2(w[2 * tj], w[2 * tj + 1]);
                        if (excbits >> (ti * 8 + 2 * tj) & 1u) v2.x = 0.0;
                        if (excbits >> (ti * 8 + 2 * tj + 1) & 1u) v2.y = 0.0;
                        *reinterpret_cast<double2*>(wp + ps.col(tj)) = v2;
                    }
                }
                tmem_wait_st();
                __syncthreads();
                continue;
            }

        stage_done:
            write_stage_stats();
            write_W();
            ++stage;
            if (stage < P.n_stages) {
                start_stage();
                __syncthreads();
                continue;
            }
            if (!P.final_dev) goto problem_done;
            final_phase = true;
            __syncthreads();
        }
    problem_done:
        if (tid == 0) {
            if (P.status_dev) P.status_dev[b] = status;
            if (P.ckpt_count_dev) P.ckpt_count_dev[b] = n_ckpt < P.ckpt_log_cap ? n_ckpt : P.ckpt_log_cap;
            if (TCC && tcc.perron_steps) tcc.perron_steps[b] = perron_steps;
        }
        __syncthreads();
    }

    tmem_fence_before();
    __syncthreads();
    if (ps.warp == 0) tmem_free<PS_TMEM_COLS>(tmem_base);
}

}  // namespace dagma

using namespace dagma;

namespace {

int check_pst_args(const dagma_small_fit_args* args, const int32_t* pair_off_dev, const int32_t* pairs_dev,
                   const double* trek_weight_dev, int agg) {
    DAGMA_REQUIRE(args != nullptr, "null args");
    const dagma_small_fit_args& a = *args;
    DAGMA_REQUIRE(a.batch >= 1, "batch must be positive");
    DAGMA_REQUIRE(a.d >= 1 && a.d <= DAGMA_SMALL_MAX_D, "d out of range for the on-chip PST fit");
    DAGMA_REQUIRE(a.n_stages >= 0 && a.n_stages <= DAGMA_MAX_STAGES, "too many stages");
    DAGMA_REQUIRE(a.checkpoint >= 1, "checkpoint must be >= 1");
    DAGMA_REQUIRE(a.cov_dev && a.w_dev && a.lambda1_dev && a.work_counter_dev, "null device pointer");
    DAGMA_REQUIRE(pair_off_dev && pairs_dev && trek_weight_dev, "null pair / weight pointer");
    DAGMA_REQUIRE(agg >= DAGMA_PST_MEAN && agg <= DAGMA_PST_LSE, "agg must be one of DAGMA_PST_MEAN .. DAGMA_PST_LSE");
    return 0;
}

// one CTA per SM: 189 KB (inv), 223 KB (exp) or 157 KB (tcc) of shared memory; 256 TMEM columns of the 512 of an SM
template <int SEQ>
int launch_pst(dagma_stream_t stream_, const dagma_small_fit_args& a, const int32_t* pair_off_dev,
               const int32_t* pairs_dev, const double* trek_weight_dev, int agg, double eps_inv,
               const TccArgs& tcc = TccArgs{}) {
    DAGMA_REQUIRE(a.ckpt_diag_dev == nullptr, "the PST fit writes no telemetry rows (ckpt_diag_dev must be NULL)");
    DAGMA_REQUIRE(((uintptr_t)pairs_dev & 7u) == 0, "pairs_dev must be 8-byte aligned");
    const size_t smem = SEQ == PST_EXP ? PstExpSmem::bytes : SEQ == TREK_TCC ? TccSmem::bytes : PstSmem::bytes;
    cudaStream_t stream = (cudaStream_t)stream_;
    int dev = 0, sms = 0;
    DAGMA_CUDA_OK(cudaGetDevice(&dev));
    DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_pst_kernel<SEQ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_pst_kernel<SEQ>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    long ctas = sms;
    if (ctas > a.batch) ctas = a.batch;
    DAGMA_CUDA_OK(cudaMemsetAsync(a.work_counter_dev, 0, sizeof(uint32_t), stream));
    fit_small_pst_kernel<SEQ><<<(int)ctas, DM_NT, smem, stream>>>(a, pair_off_dev, pairs_dev, trek_weight_dev, agg,
                                                                   eps_inv, tcc);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" int dagma_linear_fit_small_pst_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                              const int32_t* pair_off_dev, const int32_t* pairs_dev,
                                              const double* trek_weight_dev, int agg, double eps_inv) {
    if (const int rc = check_pst_args(args, pair_off_dev, pairs_dev, trek_weight_dev, agg)) return rc;
    DAGMA_REQUIRE(eps_inv >= 0.0 && eps_inv < 1e300, "eps_inv must be finite and >= 0");
    return launch_pst<PST_INV>(stream, *args, pair_off_dev, pairs_dev, trek_weight_dev, agg, eps_inv);
}

extern "C" int dagma_linear_fit_small_pst_exp_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                                  const int32_t* pair_off_dev, const int32_t* pairs_dev,
                                                  const double* trek_weight_dev, int agg) {
    if (const int rc = check_pst_args(args, pair_off_dev, pairs_dev, trek_weight_dev, agg)) return rc;
    return launch_pst<PST_EXP>(stream, *args, pair_off_dev, pairs_dev, trek_weight_dev, agg, 0.0);
}

extern "C" int dagma_linear_fit_small_tcc_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                              const int32_t* pair_off_dev, const int32_t* pairs_dev,
                                              const double* weight_dev, const double* w_dev, const double* eps_dev,
                                              const int32_t* n_iter_dev, const int32_t* flags_dev,
                                              int64_t* perron_steps_dev) {
    if (const int rc = check_pst_args(args, pair_off_dev, pairs_dev, weight_dev, DAGMA_PST_MEAN)) return rc;
    DAGMA_REQUIRE(w_dev && eps_dev && n_iter_dev && flags_dev, "null TCC parameter pointer");
    const TccArgs tcc{w_dev, eps_dev, n_iter_dev, flags_dev, reinterpret_cast<long long*>(perron_steps_dev)};
    return launch_pst<TREK_TCC>(stream, *args, pair_off_dev, pairs_dev, weight_dev, DAGMA_PST_MEAN, 0.0, tcc);
}
