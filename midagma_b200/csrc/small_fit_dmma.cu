// Tensor-core (DMMA) variant of the on-chip batched DAGMA-linear fit for 32 < d <= 64.
//
// Same contract and reference semantics as fit_small_kernel (small_fit.cu; quirks Q1-Q7 of
// SURVEY.md 8, src/dagma/linear.py:165-333 and :441-457); what changes is the machine mapping:
//   * one 256-thread CTA per problem, TWO CTAs per SM, so the serial publish / barrier /
//     pivot-block chain of one problem is hidden behind the DMMA work of the other;
//   * the sweep is the block-4 Gauss-Jordan of small_dmma.cuh: inverse and cov @ W both run
//     on the FP64 tensor pipe (DMMA.8x8x4);
//   * the kernel inverts M^T = sI - (W o W)^T, so the accumulator tile already holds the
//     entries of M^{-T} that the gradient 2 W o M^{-T} needs (linear.py:248) -- no transpose;
//   * Adam moments live in tensor memory (tcgen05.ld/st), W and -cov in shared memory,
//     M^{-T} and cov (I - W) in registers.
#include "common.cuh"
#ifndef DAGMA_FIT_GEMM_IN_SWEEP
#define DAGMA_FIT_GEMM_IN_SWEEP 1     // 1: the score GEMM fills the waits of the sweep; 0: a separate phase after it
#endif
#ifndef DAGMA_SWEEP_JIT_ROWS
#define DAGMA_SWEEP_JIT_ROWS DAGMA_FIT_GEMM_IN_SWEEP   // the filler's accumulators need the registers of the row fragments
#endif
#include "small_dmma.cuh"
#include "small_fit_internal.h"
#include "fit_step.cuh"

#ifndef DAGMA_FIT_GEMM_IN_SWEEP
#define DAGMA_FIT_GEMM_IN_SWEEP 1     // 1: the score GEMM fills the waits of the sweep; 0: a separate phase after it
#endif
#include "../../include/dagma_b200.h"

namespace dagma {

#ifdef DAGMA_SWEEP_TRACE
// debug build only: phase stamps of iteration 51 of CTA 0 -> rows 16.. of g_sweep_trace
// [0] iteration start, [1] M built, [2] sweep done, [3] score GEMM done, [4] feasibility known, [5] Adam pass done
#define PHASE_STAMP(slot) do { if (blockIdx.x == 0 && tid == 0 && it == 50) g_sweep_trace[16 * 8 + (slot)] = clock64(); } while (0)
#define PHASE_STAMP_END(slot) do { if (blockIdx.x == 0 && tid == 0 && it == 51) g_sweep_trace[16 * 8 + (slot)] = clock64(); } while (0)
#else
#define PHASE_STAMP(slot) do { } while (0)
#define PHASE_STAMP_END(slot) do { } while (0)
#endif

// Residency probe: how many CTAs of the fit kernel are on one SM at the same time (max over SMs, over the last launch).
// The launch geometry assumes two (registers, shared memory and tensor memory are sized for exactly that), the occupancy
// API of driver 580 answers 1 for this kernel, so the kernel counts for itself and dagma_fit_dmma_residency() reports it
// (tests/test_dmma_cold_gpu.py asserts 2).  Two atomics per CTA lifetime.
__device__ int g_fit_resident[512];
__device__ int g_fit_max_resident;

// DIAG: the instantiation that also writes the telemetry rows (ckpt_diag_dev); the plain one carries none of that code,
// so switching logging on costs the logged run a few registers and the unlogged run nothing.
template <bool DIAG>
__global__ void __launch_bounds__(DM_NT, 2) fit_small_dmma_kernel(const dagma_small_fit_args P) {
    using S = DmmaSmem;
    constexpr int NT = DM_NT, LD = DM_LD;
    extern __shared__ __align__(16) double smem[];
    double* ncov = smem + S::ncov;
    double* Ws = smem + S::W;
    double* pinfo = smem + S::pinfo;
    double* red = smem + S::red;
    __shared__ unsigned s_prob;
    __shared__ uint32_t s_tmem;
    // Adam bias correction, kept by ONE lane instead of by every thread: the running powers beta^it (double-double) and
    // the reciprocals c = 1 / (1 - beta^it) of the iteration that is about to run, slot it & 1 (the other slot still
    // holds the factors of the last executed step, which back-tracking needs to rebuild its direction)
    __shared__ double s_pow[4];          // committed p1.hi, p1.lo, p2.hi, p2.lo  (= beta^it)
    __shared__ double s_pow_next[4];     // beta^(it + 1), computed ahead
    __shared__ double s_bias[2][2];      // [slot][c1, c2]

    const int tid = threadIdx.x;
    const DmmaPos ps(tid);
    const int d = P.d;
    const int np = 4 * ((d + 3) >> 2);          // pivots swept (d rounded up to the block size)
    unsigned my_sm = 0;
    if (tid == 0) {
        asm volatile("mov.u32 %0, %%smid;" : "=r"(my_sm));
        atomicMax(&g_fit_max_resident, atomicAdd(&g_fit_resident[my_sm & 511u], 1) + 1);
    }
    const size_t dd = (size_t)d * d;

    // ---- step barrier of the sweep: one arrival per warp
    SweepSync sy{smem_u32(smem + S::mbar), 0u};
    if (tid == 0) mbar_init(sy.bar, NT / 32);

    // ---- tensor-memory scratch for the Adam moments (thread-private, 64 columns per thread)
    if (ps.warp == 0) tmem_alloc(smem_u32(&s_tmem));
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    const uint32_t tmem_base = s_tmem;
    const uint32_t tm = tmem_base + ((uint32_t)(32 * (ps.warp & 3)) << 16) + (uint32_t)((ps.warp >> 2) * 64);
    // columns: [m(ti=0) 16 | v(ti=0) 16 | m(ti=1) 16 | v(ti=1) 16]

    // exclusion / inclusion bit masks of this thread's 16 entries (shared by the batch)
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

        for (int idx = tid; idx < DM_DP * DM_DP; idx += NT) {
            const int r = idx >> 6, c = idx & 63;
            const bool in = (r < d) && (c < d);
            ncov[r * LD + c] = in ? -cov_g[r * d + c] : 0.0;
            Ws[r * LD + c] = in ? W_g[r * d + c] : 0.0;
        }
        __syncthreads();

        double a[2][4][2], g[2][4][2];
        int status = 0;
        int n_ckpt = 0;

        // ---- state of the path-following loop ----
        int stage = 0;
        bool final_phase = (P.n_stages == 0);
        double mu = 0, s_cur = 1, lr = 0, lr_adam = P.lr, obj_prev = 1e16;
        double last_obj = 0, last_score = 0, last_h = 0;
        int iters_max = 0, it = 0, retries = 0, backtracks = 0;
        bool in_backtrack = false;

        unsigned long long t_attempt = 0;        // %globaltimer at the start of the minimize call (telemetry)
        auto start_attempt = [&]() {
            it = 0;
            t_attempt = global_ns();
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
        auto write_W = [&]() {   // Ws -> global (stage result / restart point)
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
            // ================= build M^T and run the fused sweep =================
            const double s_use = final_phase ? 1.0 : s_cur;
            PHASE_STAMP(0);
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
#ifdef DAGMA_SWEEP_TRACE
            sy.trace = (it == 50) ? 0 : -1;          // trace the sweep of iteration 51
#endif
            PHASE_STAMP(1);
            // bias factors of iteration it + 1, by lane 0 of the last warp: at the start of the sweep that warp only
            // waits for the first pivot block, so this costs nothing on the critical path; the sweep's barriers make
            // the values visible to everybody before the Adam pass reads them
            if (tid == DM_NT - 32 && !final_phase) {
                DD q1{s_pow[0], s_pow[1]}, q2{s_pow[2], s_pow[3]};
                q1.mul(P.beta1);
                q2.mul(P.beta2);
                s_pow_next[0] = q1.hi; s_pow_next[1] = q1.lo; s_pow_next[2] = q2.hi; s_pow_next[3] = q2.lo;
                s_bias[(it + 1) & 1][0] = fast_rcp(q1.one_minus());
                s_bias[(it + 1) & 1][1] = fast_rcp(q2.one_minus());
            }
            auto init_g = [&]() {
#pragma unroll
                for (int ti = 0; ti < 2; ++ti)
#pragma unroll
                    for (int tj = 0; tj < 4; ++tj) {
                        const double2 nc = *reinterpret_cast<const double2*>(ncov + ps.row(ti) * LD + ps.col(tj));
                        g[ti][tj][0] = __hiloint2double(__double2hiint(nc.x) ^ (int)0x80000000, __double2loint(nc.x));   // -nc: sign
                        g[ti][tj][1] = __hiloint2double(__double2hiint(nc.y) ^ (int)0x80000000, __double2loint(nc.y));   // bit, not FP64
                    }
            };
#if DAGMA_FIT_GEMM_IN_SWEEP
            // g = cov - cov W rides inside the sweep: the warps that wait for the pivot chain of a block step work on
            // k-blocks of the score GEMM instead (it needs only W and cov), so the GEMM is off the critical path
            init_g();
            ScoreFill fill{g, ps, smem, 0, (d + 3) >> 2};
            dmma_sweep(a, ps, smem, d, sy, fill);
            PHASE_STAMP(2);
#pragma unroll 1
            while (fill.more()) fill.unit();
#else
            dmma_sweep(a, ps, smem, d, sy);
            PHASE_STAMP(2);
            init_g();
            dmma_score_gemm(g, ps, smem, d);
#endif
            PHASE_STAMP(3);
            // now: a = M^{-T},  g = cov - cov W = cov (I - W),  pinfo[0..np) = pivots

            // ================= objective pieces (checkpoint / final) =================
            const bool at_ckpt = !final_phase && !in_backtrack && it >= 1 &&
                                 (it % P.checkpoint == 0 || it == iters_max);
            if (at_ckpt || final_phase) {
                double sc = 0.0, l1 = 0.0, ld = 0.0;
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
                if (tid < np) ld = (double)((tid & 3) - 2) * log(fabs(pinfo[tid]));   // fraction-free pivots
                block_sum3<NT>(sc, l1, ld, red, tid);
                const double score = 0.5 * sc;
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
                PHASE_STAMP(4);
                if (bad) {
                    if (it == 0 || s_cur <= 0.9) {            // linear.py:231-233
                        if (P.retry_on_fail) {
                            if (++retries > 64) {
                                // the reference would keep retrying; give up on the stage's restart point, but
                                // leave complete outputs: stage stats, status, and the final h / score of that W
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
                if (tid == DM_NT - 32) {                       // commit beta^it (nobody else reads s_pow)
                    s_pow[0] = s_pow_next[0]; s_pow[1] = s_pow_next[1]; s_pow[2] = s_pow_next[2]; s_pow[3] = s_pow_next[3];
                }
                const double l1c = mu * lambda1, incc = -2.0 * mu * lambda1, nmu = -mu;
                if (DIAG && P.ckpt_diag_dev != nullptr && (it % P.checkpoint == 0 || it == iters_max)) {
                    // Telemetry row of this checkpoint iteration (cold: once per `checkpoint` iterations): read-only
                    // passes that repeat the arithmetic of the step on the side, three sums per pass so that the
                    // accumulators do not add to the register pressure of the hot loop below.
                    double acc[10];
#pragma unroll
                    for (int pass = 0; pass < 4; ++pass) {
                        double x = 0.0, y = 0.0, z = (pass == 3) ? 1.7976931348623157e308 : 0.0;
#pragma unroll
                        for (int ti = 0; ti < 2; ++ti) {             // (static indices: a and g stay in registers)
                            TmemLoad8 lm, lv;
                            lm.issue(tm + 32 * ti);
                            lv.issue(tm + 32 * ti + 16);
                            lm.finish();
                            lv.finish();
                            const double* wp = Ws + ps.row(ti) * LD;
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                const double w = wp[ps.col(q >> 1) + (q & 1)];
                                const double gs = nmu * g[ti][q >> 1][q & 1];
                                const double gh = twice(w) * (a[ti][q >> 1][q & 1] + 1e-16);
                                const bool inc = (incbits >> (ti * 8 + q) & 1u) != 0u;
                                const double go = gs + signed_const(w, l1c) + gh + (inc ? signed_const(w, incc) : 0.0);
                                if (pass == 0) {
                                    x = fma(go, go, x); y = fma(gs, gs, y); z = fma(gh, gh, z);
                                } else {
                                    const double Mn = fma(lm.get(q), P.beta1, go), Un = fma(lv.get(q), P.beta2, go * go);
                                    const double dir = fast_div(Mn * k1, fast_sqrt_nonneg(Un * k2) + 1e-8);
                                    const bool exc = (excbits >> (ti * 8 + q) & 1u) != 0u;
                                    const double aw = fabs(exc ? 0.0 : fma(-lr, dir, w));
                                    if (pass == 1) {
                                        x += (w != 0.0) ? 1.0 : 0.0; y += (w != 0.0 && inc) ? 1.0 : 0.0; z = fma(dir, dir, z);
                                    } else if (pass == 2) {
                                        x = fma(aw, aw, x); y += aw;
                                    } else {
                                        x = fmax(x, aw); if (aw > 0.0) z = fmin(z, aw);
                                    }
                                }
                            }
                        }
                        if (pass < 3) {
                            block_sum3<NT>(x, y, z, red, tid);
                            acc[3 * pass] = x; acc[3 * pass + 1] = y; acc[3 * pass + 2] = z;
                        } else {
                            acc[8] = block_max<NT>(x, red, tid);
                            acc[9] = block_min<NT>(z, red, tid);
                        }
                    }
                    if (tid == 0 && n_ckpt < P.ckpt_log_cap) {
                        double* row = P.ckpt_diag_dev + ((size_t)b * P.ckpt_log_cap + n_ckpt) * DAGMA_DIAG_COLS;
                        row[0] = sqrt(acc[0]); row[1] = sqrt(acc[1]); row[2] = sqrt(acc[2]);
                        row[3] = fabs(l1c) * sqrt(acc[3]); row[4] = fabs(incc) * sqrt(acc[4]); row[5] = sqrt(acc[5]);
                        row[6] = sqrt(acc[6]); row[7] = acc[7]; row[8] = acc[8]; row[9] = (acc[8] > 0.0) ? acc[9] : 0.0;
                        row[10] = 1e-9 * (double)(global_ns() - t_attempt);
                    }
                }
#pragma unroll
                for (int ti = 0; ti < 2; ++ti) {
                    TmemLoad8 lm, lv;
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
                    // Gobj = -mu cov (I - W) + mu l1 sign(W) + 2 W o (M^{-T} + 1e-16)   linear.py:248
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        go[q] = fma(nmu, g[ti][q >> 1][q & 1], signed_const(w[q], l1c));
                        go[q] = fma(twice(w[q]), a[ti][q >> 1][q & 1] + 1e-16, go[q]);
                    }
                    if (P.mask_inc_dev) {            // uniform branch: no predicated FP64 issue slots without include edges
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
                    for (int q0 = 0; q0 < 8; q0 += DAGMA_ADAM_GROUP)     // Newton chains of a group interleave
                        adam_entries<DAGMA_ADAM_GROUP>(w + q0, go + q0, mn + q0, vn + q0, P.beta1, P.beta2, k1, k2, lr);
                    tmem_st8(tm + 32 * ti, mn);
                    tmem_st8(tm + 32 * ti + 16, vn);
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
                PHASE_STAMP_END(5);
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
    if (ps.warp == 0) tmem_free(tmem_base);
    if (tid == 0) atomicSub(&g_fit_resident[my_sm & 511u], 1);
}

#ifdef DAGMA_SWEEP_TRACE
}  // namespace dagma

extern "C" int dagma_debug_sweep_trace(long long* out_host) {
    return (int)cudaMemcpyFromSymbol(out_host, dagma::g_sweep_trace, sizeof(long long) * 64 * 8);
}
namespace dagma {
#endif

int fit_dmma_geometry(int batch, int sms, int* ctas, int* threads, size_t* smem_bytes) {
    constexpr size_t bytes = DmmaSmem::bytes;
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_dmma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_dmma_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_dmma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(fit_small_dmma_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    // Two CTAs per SM by construction: __launch_bounds__(256, 2) caps registers at 128 (2 x 256 x 128
    // = the whole file), 2 x 80.8 KB of shared memory fit the 228 KB carve-out and 2 x 128 TMEM columns
    // fit the 512 of an SM.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor reports 1 for this kernel on
    // driver 580 although two are resident -- ncu: sm__warps_active 25 % = 16 warps; if only one fitted,
    // the work-queue loop would still be correct, the surplus CTAs just start late.)
    int per_sm = 0;
    DAGMA_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fit_small_dmma_kernel<false>, DM_NT, bytes));
    if (per_sm < 1) return set_error(-5, "DMMA fit kernel does not fit on an SM");
    per_sm = 2;
    long n = (long)sms * per_sm;
    if (n > batch) n = batch;
    if (ctas) *ctas = (int)n;
    if (threads) *threads = DM_NT;
    if (smem_bytes) *smem_bytes = bytes;
    return 0;
}

int launch_fit_dmma(cudaStream_t stream, const dagma_small_fit_args& a, int sms) {
    int ctas = 0;
    int rc = fit_dmma_geometry(a.batch, sms, &ctas, nullptr, nullptr);
    if (rc) return rc;
    void* maxp = nullptr;
    DAGMA_CUDA_OK(cudaGetSymbolAddress(&maxp, g_fit_max_resident));
    DAGMA_CUDA_OK(cudaMemsetAsync(maxp, 0, sizeof(int), stream));
    if (a.ckpt_diag_dev)
        fit_small_dmma_kernel<true><<<ctas, DM_NT, DmmaSmem::bytes, stream>>>(a);
    else
        fit_small_dmma_kernel<false><<<ctas, DM_NT, DmmaSmem::bytes, stream>>>(a);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace dagma

// max number of CTAs of the last 32 < d <= 64 fit launch that shared an SM (synchronises with the device)
extern "C" int dagma_fit_dmma_residency(int* out_host) {
    DAGMA_REQUIRE(out_host != nullptr, "null pointer");
    DAGMA_CUDA_OK(cudaDeviceSynchronize());
    DAGMA_CUDA_OK(cudaMemcpyFromSymbol(out_host, dagma::g_fit_max_resident, sizeof(int)));
    return 0;
}
