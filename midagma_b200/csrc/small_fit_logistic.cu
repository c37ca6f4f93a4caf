// Batched DagmaLinear('logistic').minimize / fit for 1 <= d <= 64: one CTA per problem runs the whole schedule
// (stages, retries, back-tracking, checkpoints) -- the logistic counterpart of fit_small_dmma_kernel
// (small_fit_dmma.cu), with the same contract (dagma_small_fit_args) and the same reference semantics
// (src/dagma/linear.py:90-92 score, :165-333 inner loop, :441-457 stage loop; quirks Q1-Q7 of SURVEY.md 8).
//
// Mapping (256 threads, TWO CTAs per SM, problems pulled from an atomic work queue; no grid barriers):
//   * score products: the problem's X [n][d] streams through shared memory in tiles of LG_TR rows, double-buffered by
//     cp.async (X does not stay on chip: 512 KB at d = 64, n = 1000).  Per tile, on DMMA.8x8x4:
//       Z_t = X_t W         warp w owns columns 8w .. 8w + 7 of Z_t (all LG_TR rows);
//       R_t = sigmoid(Z_t)  written to shared memory (0 in the padding columns);
//       T  += X_t^T R_t     into the accumulators of the sweep's ownership ([2][4] tiles per warp),
//     tiles in a fixed order, so every problem's sums are the same wherever and whenever it runs.  The 1/n is
//     applied afterwards (G_loss = fma(1/n, T, -cov), as linear_update_kernel and lin_iter.cu do): with binary X at
//     W = 0 the exact ties of DESIGN 2 (C2) come out as an exact 0.
//     On checkpoint iterations the same pass sums softplus(Z) - X o Z (the loss at the current W, linear.py:91).
//   * G_loss waits in tensor memory next to the Adam moments while the sweep holds M^{-T} in registers.
//   * inverse of M^T = sI - (W o W)^T: the block Gauss-Jordan of small_dmma.cuh, as in the l2 kernel (same
//     feasibility predicate, same log|det|); then the Adam step of the l2 kernel (fit_step.cuh).
#include "common.cuh"
#define DAGMA_SWEEP_JIT_ROWS 1        // pivot-row fragments loaded tile by tile: the loop state stays in registers
#include "small_dmma.cuh"
#include "gemm_f64.cuh"
#include "fit_step.cuh"
#include "../../include/dagma_b200.h"

namespace dagma {

constexpr int LG_TR = 32;                 // rows of X per tile
constexpr int LG_TMEM_COLS = 256;         // per thread: m, v (64 columns) and G_loss (32), two warps per lane quarter

struct LogiSmem {                         // offsets in doubles; the sweep's buffers keep the offsets of DmmaSmem
    static constexpr int X = DmmaSmem::ncov;                   // 2 x [LG_TR][68] X tiles (the sweep leaves this area alone)
    static constexpr int R = DmmaSmem::total;                  // [LG_TR][68] sigmoid(X_t W)
    static constexpr int total = R + LG_TR * DM_LD;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(2 * LG_TR * DM_LD <= DmmaSmem::W - DmmaSmem::ncov, "the X tiles fit the area of -cov");
static_assert(LogiSmem::R % 2 == 0, "16-byte alignment of vector accesses");

__device__ __forceinline__ double softplus(double z) { return fmax(z, 0.0) + log1p(exp(-fabs(z))); }

// T = X^T sigmoid(X W) over all n rows into g (accumulator ownership of DmmaPos); with `want_loss`, `loss` gets this
// thread's share of sum (softplus(X W) - X o X W).  Ws: W zero padded to [64][68].  The padding columns of the X tiles
// and of R are zero on entry and stay zero.
__device__ __forceinline__ void logistic_products(const double* __restrict__ xb, int n, int d, double* sm,
                                                  const DmmaPos& ps, double (&g)[2][4][2], bool want_grad,
                                                  bool want_loss, double& loss) {
    constexpr int NT = DM_NT, LD = DM_LD;
    const int tid = threadIdx.x;
    const double* Ws = sm + DmmaSmem::W;
    double* Rs = sm + LogiSmem::R;
    const int ntile = (n + LG_TR - 1) / LG_TR, KT = (d + 3) >> 2;
    auto load_tile = [&](int t) {
        double* dst = sm + LogiSmem::X + (t & 1) * LG_TR * LD;
        const int r0 = t * LG_TR;
        if ((d & 1) == 0) {                   // rows start on 16 bytes: X of a problem is n * d doubles, d even
            const int hc = d >> 1;
            for (int idx = tid; idx < LG_TR * hc; idx += NT) {
                const int r = idx / hc, c2 = idx - r * hc;
                const bool ok = r0 + r < n;
                cp_async16(smem_u32(dst + r * LD + 2 * c2), ok ? xb + (size_t)(r0 + r) * d + 2 * c2 : xb, ok);
            }
        } else {
            for (int idx = tid; idx < LG_TR * d; idx += NT) {
                const int r = idx / d, c = idx - r * d;
                const bool ok = r0 + r < n;
                cp_async8(smem_u32(dst + r * LD + c), ok ? xb + (size_t)(r0 + r) * d + c : xb, ok);
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj) g[ti][tj][0] = g[ti][tj][1] = 0.0;
    const int w = ps.warp, qr = ps.qr, qc = ps.qc;
    const bool zwarp = 8 * w < d;                                  // owns a column block of Z
    const bool twarp = 16 * ps.wr < d && 32 * ps.wc < d;           // owns tiles of T inside d x d
    load_tile(0);
#pragma unroll 1
    for (int t = 0; t < ntile; ++t) {
        cp_async_wait<0>();
        __syncthreads();                      // tile t has landed; every warp is done with tile t - 1 and with R
        if (t + 1 < ntile) load_tile(t + 1);
        const double* Xt = sm + LogiSmem::X + (t & 1) * LG_TR * LD;
        if (zwarp) {
            double z[4][2];
#pragma unroll
            for (int i = 0; i < 4; ++i) z[i][0] = z[i][1] = 0.0;
            const double* ap = Xt + qr * LD + qc;
            const double* bp = Ws + qc * LD + 8 * w + qr;
#pragma unroll 4
            for (int ks = 0; ks < KT; ++ks) {
                const double b = bp[4 * ks * LD];
#pragma unroll
                for (int i = 0; i < 4; ++i) dmma(z[i][0], z[i][1], ap[8 * i * LD + 4 * ks], b);
            }
            const int c = 8 * w + 2 * qc;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = 8 * i + qr;
                if (want_grad)
                    *reinterpret_cast<double2*>(Rs + r * LD + c) =
                        make_double2(c < d ? li_sigmoid(z[i][0]) : 0.0, c + 1 < d ? li_sigmoid(z[i][1]) : 0.0);
                if (want_loss && t * LG_TR + r < n) {
                    if (c < d) loss += softplus(z[i][0]) - Xt[r * LD + c] * z[i][0];
                    if (c + 1 < d) loss += softplus(z[i][1]) - Xt[r * LD + c + 1] * z[i][1];
                }
            }
        }
        if (!want_grad) continue;
        __syncthreads();                      // R_t complete
        if (twarp) {
            const double* ap = Xt + qc * LD + 16 * ps.wr + qr;
            const double* bp = Rs + qc * LD + 32 * ps.wc + qr;
#pragma unroll 2
            for (int ks = 0; ks < LG_TR / 4; ++ks) {
                double a[2], b[4];
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) a[ti] = ap[4 * ks * LD + 8 * ti];
#pragma unroll
                for (int tj = 0; tj < 4; ++tj) b[tj] = bp[4 * ks * LD + 8 * tj];
#pragma unroll
                for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) dmma(g[ti][tj][0], g[ti][tj][1], a[ti], b[tj]);
            }
        }
    }
    __syncthreads();                          // the tiles and R are free again
}

__global__ void __launch_bounds__(DM_NT, 2) fit_small_logistic_kernel(const dagma_small_fit_args P, int n,
                                                                       const double* __restrict__ X) {
    constexpr int NT = DM_NT, LD = DM_LD;
    extern __shared__ __align__(16) double smem[];
    double* Ws = smem + DmmaSmem::W;
    double* pinfo = smem + DmmaSmem::pinfo;
    double* red = smem + DmmaSmem::red;
    __shared__ unsigned s_prob;
    __shared__ uint32_t s_tmem;
    // Adam bias correction, kept by one lane (see fit_small_dmma_kernel)
    __shared__ double s_pow[4];
    __shared__ double s_pow_next[4];
    __shared__ double s_bias[2][2];
    __shared__ unsigned s_excbits[DM_NT], s_incbits[DM_NT];   // edge masks of a thread's 16 entries (registers are full)

    const int tid = threadIdx.x;
    const DmmaPos ps(tid);
    const int d = P.d;
    const int np = 4 * ((d + 3) >> 2);
    const size_t dd = (size_t)d * d;
    const double inv_n = 1.0 / (double)n;

    SweepSync sy{smem_u32(smem + DmmaSmem::mbar), 0u};
    if (tid == 0) mbar_init(sy.bar, NT / 32);
    // the padding of the X tiles and of R must be zero (finite, annihilated by the other operand)
    for (int e = tid; e < 2 * LG_TR * LD; e += NT) smem[LogiSmem::X + e] = 0.0;
    for (int e = tid; e < LG_TR * LD; e += NT) smem[LogiSmem::R + e] = 0.0;

    if (ps.warp == 0) tmem_alloc<LG_TMEM_COLS>(smem_u32(&s_tmem));
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    const uint32_t tmem_base = s_tmem;
    // columns of a thread: [m(ti=0) 16 | v(ti=0) 16 | m(ti=1) 16 | v(ti=1) 16 | G_loss(ti=0) 16 | G_loss(ti=1) 16]
    const uint32_t tm = tmem_base + ((uint32_t)(32 * (ps.warp & 3)) << 16) + (uint32_t)((ps.warp >> 2) * 96);
    const uint32_t tg = tm + 64;

    unsigned exc = 0, inc = 0;
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = ps.row(ti), c = ps.col(tj) + e;
                if (r < d && c < d) {
                    if (P.mask_exc_dev && P.mask_exc_dev[r * d + c]) exc |= 1u << (ti * 8 + tj * 2 + e);
                    if (P.mask_inc_dev && P.mask_inc_dev[r * d + c]) inc |= 1u << (ti * 8 + tj * 2 + e);
                }
            }
    s_excbits[tid] = exc;
    s_incbits[tid] = inc;

    for (;;) {
        if (tid == 0) s_prob = atomicAdd(P.work_counter_dev, 1u);
        __syncthreads();
        const unsigned b = s_prob;
        __syncthreads();
        if (b >= (unsigned)P.batch) break;

        const double* cov_g = P.cov_dev + (size_t)b * dd;
        const double* x_g = X + (size_t)b * n * d;
        double* W_g = P.w_dev + (size_t)b * dd;
        const double lambda1 = P.lambda1_dev[b];

        for (int idx = tid; idx < DM_DP * DM_DP; idx += NT) {
            const int r = idx >> 6, c = idx & 63;
            Ws[r * LD + c] = (r < d && c < d) ? W_g[r * d + c] : 0.0;
        }
        __syncthreads();

        double a[2][4][2];
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
            // ================= score products at the current W =================
            double loss = 0.0;
            {
                double g[2][4][2];
                logistic_products(x_g, n, d, smem, ps, g, !final_phase, at_ckpt || final_phase, loss);
                if (!final_phase) {
                    // G_loss = X^T sigmoid(X W) / n - cov   (linear.py:92), parked in tensor memory for the step
#pragma unroll
                    for (int ti = 0; ti < 2; ++ti) {
                        double gl[8];
                        const int r = ps.row(ti);
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const int c = ps.col(q >> 1) + (q & 1);
                            const double cv = (r < d && c < d) ? __ldg(cov_g + r * d + c) : 0.0;
                            gl[q] = fma(inv_n, g[ti][q >> 1][q & 1], -cv);
                        }
                        tmem_st8(tg + 16 * ti, gl);
                    }
                    tmem_wait_st();
                }
            }

            // ================= build M^T and run the sweep =================
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
            dmma_sweep(a, ps, smem, d, sy);
            // now: a = M^{-T}, pinfo[0..np) = pivots

            // ================= objective (checkpoint / final) =================
            if (at_ckpt || final_phase) {
                double sc = loss, l1 = 0.0, ld = 0.0;
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) {
                    const int r = ps.row(ti);
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        const double2 w = *reinterpret_cast<const double2*>(Ws + r * LD + ps.col(tj));
                        l1 += fabs(w.x) + fabs(w.y);
                    }
                }
                if (tid < np) ld = (double)((tid & 3) - 2) * log(fabs(pinfo[tid]));
                block_sum3<NT>(sc, l1, ld, red, tid);
                const double score = sc * inv_n;
                const double h = -ld + (double)d * log(s_use);
                if (final_phase) {
                    if (tid == 0 && P.final_dev) {
                        P.final_dev[2 * (size_t)b] = h;
                        P.final_dev[2 * (size_t)b + 1] = score;
                    }
                    break;
                }
                const double obj = mu * (score + lambda1 * l1) + h;
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
            } else if (!final_phase && !in_backtrack && it == iters_max) {
                goto stage_done;   // only reachable for iters_max == 0
            }

            {
                // ================= feasibility of iteration it + 1 =================
                bool bad = false;
                if (tid < np) bad = !(pinfo[tid] > 0.0);
#pragma unroll
                for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj)
                        bad |= below_minus_1e16(a[ti][tj][0]) | below_minus_1e16(a[ti][tj][1]);
                bad = __syncthreads_or(bad);
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
            }

            {
                // ================= gradient, Adam, step (iteration it + 1) =================
                ++it;
                const double k1 = s_bias[it & 1][0] * (1.0 - P.beta1), k2 = s_bias[it & 1][1] * (1.0 - P.beta2);
                if (tid == DM_NT - 32) {
                    s_pow[0] = s_pow_next[0]; s_pow[1] = s_pow_next[1]; s_pow[2] = s_pow_next[2]; s_pow[3] = s_pow_next[3];
                }
                const double l1c = mu * lambda1, incc = -2.0 * mu * lambda1;
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
                        const double2 t = *reinterpret_cast<const double2*>(wp + ps.col(tj));
                        w[2 * tj] = t.x;
                        w[2 * tj + 1] = t.y;
                    }
                    lg.finish();
                    // Gobj = mu G_loss + mu l1 sign(W) + 2 W o (M^{-T} + 1e-16)   linear.py:248
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        go[q] = fma(mu, lg.get(q), signed_const(w[q], l1c));
                        go[q] = fma(twice(w[q]), a[ti][q >> 1][q & 1] + 1e-16, go[q]);
                    }
                    if (P.mask_inc_dev) {
                        const unsigned incbits = s_incbits[tid];
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            if (incbits >> (ti * 8 + q) & 1u) go[q] += signed_const(w[q], incc);
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
                    const unsigned excbits = P.mask_exc_dev ? s_excbits[tid] : 0u;
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        double2 t = make_double2(w[2 * tj], w[2 * tj + 1]);
                        if (excbits >> (ti * 8 + 2 * tj) & 1u) t.x = 0.0;
                        if (excbits >> (ti * 8 + 2 * tj + 1) & 1u) t.y = 0.0;
                        *reinterpret_cast<double2*>(wp + ps.col(tj)) = t;
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
        }
        __syncthreads();
    }

    tmem_fence_before();
    __syncthreads();
    if (ps.warp == 0) tmem_free<LG_TMEM_COLS>(tmem_base);
}

}  // namespace dagma

using namespace dagma;

extern "C" int dagma_linear_fit_small_logistic_f64(dagma_stream_t stream_, const dagma_small_fit_args* args, int n,
                                                   const double* x_dev) {
    DAGMA_REQUIRE(args != nullptr, "null args");
    const dagma_small_fit_args& a = *args;
    DAGMA_REQUIRE(a.batch >= 1, "batch must be positive");
    DAGMA_REQUIRE(a.d >= 1 && a.d <= DAGMA_SMALL_MAX_D, "d out of range for the on-chip logistic fit");
    DAGMA_REQUIRE(n >= 1, "n must be positive");
    DAGMA_REQUIRE(a.n_stages >= 0 && a.n_stages <= DAGMA_MAX_STAGES, "too many stages");
    DAGMA_REQUIRE(a.checkpoint >= 1, "checkpoint must be >= 1");
    DAGMA_REQUIRE(a.cov_dev && a.w_dev && a.lambda1_dev && a.work_counter_dev && x_dev, "null device pointer");
    DAGMA_REQUIRE(a.ckpt_diag_dev == nullptr, "the logistic fit writes no telemetry rows (ckpt_diag_dev must be NULL)");
    cudaStream_t stream = (cudaStream_t)stream_;
    int dev = 0, sms = 0;
    DAGMA_CUDA_OK(cudaGetDevice(&dev));
    DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_logistic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)LogiSmem::bytes));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_logistic_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    // two CTAs per SM: __launch_bounds__(256, 2) caps registers at 128, 2 x 98 KB of shared memory fit the carve-out
    // and 2 x 256 TMEM columns are the 512 of an SM
    long ctas = 2L * sms;
    if (ctas > a.batch) ctas = a.batch;
    DAGMA_CUDA_OK(cudaMemsetAsync(a.work_counter_dev, 0, sizeof(uint32_t), stream));
    fit_small_logistic_kernel<<<(int)ctas, DM_NT, LogiSmem::bytes, stream>>>(a, n, x_dev);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}
