/*
 * dagma_b200.h -- C ABI of libdagma_b200.so: the B200 (sm_100a) implementation of
 * DAGMA's inner-optimisation hot path.
 *
 * The reference (fbleile/midagma) has no FFI: its boundary is the Python method
 * surface of DagmaLinear / DagmaMLP / DagmaNonlinear / notreks (SURVEY.md 8b).  Each
 * entry point below names the reference code it replaces (paths relative to the
 * reference root, file:line).  All matrices are FP64, row-major, caller-owned.
 * Pointers named *_dev are device pointers; everything else is host data.
 * Every function returns 0 on success, <0 on API misuse / CUDA error (the text is
 * available from dagma_last_error()); numerical failure is reported through
 * per-problem status words, never through the return code -- mirroring the
 * reference, where leaving the M-matrix domain is a return flag, not an exception
 * (src/dagma/linear.py:230-233).  Nothing here has a CPU fallback.
 */
#ifndef DAGMA_B200_H
#define DAGMA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dagma_stream_t;            /* a cudaStream_t (0 = default stream) */

#define DAGMA_SMALL_MAX_D   64           /* fused on-chip fit path: d <= 64      */
#define DAGMA_ONCHIP_INV_MAX_D 128       /* on-chip logdet+inverse: d <= 128     */
#define DAGMA_MAX_STAGES    16
#define DAGMA_DIAG_COLS     11           /* columns of a checkpoint telemetry row (ckpt_diag_dev)        */

/* per-problem status bits written by the fit / minimize kernels */
#define DAGMA_ST_OK            0
#define DAGMA_ST_OUT_OF_DOMAIN 1         /* minimize returned (W, False)  linear.py:231-233 */
#define DAGMA_ST_LR_UNDERFLOW  2         /* lr <= 1e-16 exit              linear.py:237-238 */
#define DAGMA_ST_RETRY_LIMIT   4         /* more than 64 stage retries (reference would spin) */

/* ---- library / device ---------------------------------------------------------- */
int         dagma_version(void);
const char* dagma_last_error(void);
/* 0 iff the current device is compute capability 10.x; anything else is an error
 * (there is no other code path).  Optionally returns the SM count. */
int         dagma_device_check(int* sm_count);

/* ---- (i) fused slogdet + inverse ------------------------------------------------
 * Replaces: DagmaLinear._h            src/dagma/linear.py:113-115  (square_input=1)
 *           DagmaMLP.h_func           src/dagma/nonlinear.py:82-85 (A built by caller)
 *           logdet_acyc_value_gradA   src/notreks/notreks.py:263-274 (square_input=0)
 * For each problem b:  M = s*I - (square_input ? A*A (Hadamard) : A);
 *   logabsdet[b] = log|det M|,  h[b] = -logabsdet + d*log(s),
 *   minv_dev  (optional) = M^{-1},
 *   grad_dev  (optional) = square_input ? 2*A o M^{-T} : M^{-T},
 *   min_entry[b] = min(M^{-1}),  info[b] = 0 ok | 1 non-positive pivot (not an M-matrix)
 *                                          | 2 negative entry: min(M^{-1}) + 1e-16 < 0.
 * d <= 128 runs one persistent CTA per problem (Gauss-Jordan in registers);
 * larger d runs the blocked multi-CTA path (batch is then looped).               */
int dagma_logdet_inv_f64(dagma_stream_t stream, int batch, int d, double s,
                         const double* a_dev, int lda, int square_input,
                         double* logabsdet_dev, double* h_dev,
                         double* minv_dev, double* grad_dev, int ldo,
                         double* min_entry_dev, int* info_dev);

/* ---- (iii) the inner loop / whole path-following fit, small d, batched -----------
 * Replaces: DagmaLinear.minimize  src/dagma/linear.py:165-333 (l2 loss, trek_reg None)
 *           DagmaLinear.fit       src/dagma/linear.py:441-457 (the stage loop + retries)
 * One persistent CTA per problem runs `n_stages` calls of minimize back to back
 * without leaving the SM: W, the Adam moments, cov and M^{-1} stay in registers /
 * shared memory.  Problems are pulled from an atomic work queue.                 */
typedef struct dagma_small_fit_args {
    int32_t batch;            /* number of independent problems                          */
    int32_t d;                /* nodes, 1..DAGMA_SMALL_MAX_D                              */
    int32_t n_stages;         /* T (fit) or 1 (minimize)                                  */
    int32_t checkpoint;       /* convergence-check interval          linear.py:279        */
    int32_t retry_on_fail;    /* 1: fit semantics (lr/2, s+0.1, redo) linear.py:446-451
                                 0: minimize semantics (stop, status OUT_OF_DOMAIN)       */
    int32_t ckpt_log_cap;     /* rows available per problem in ckpt_log_dev (0 = none)    */
    double  lr;               /* initial Adam step of every stage    linear.py:444        */
    double  tol;              /* relative objective tolerance        linear.py:328        */
    double  beta1, beta2;     /* Adam                                linear.py:158-162    */
    double  mu[DAGMA_MAX_STAGES];      /* mu_t (already multiplied out, Q7)               */
    double  s[DAGMA_MAX_STAGES];       /* s_t                                             */
    int32_t iters[DAGMA_MAX_STAGES];   /* max inner iterations of stage t                 */
    const double*  cov_dev;       /* [batch][d][d]  X^T X / n          linear.py:428      */
    const double*  lambda1_dev;   /* [batch]                                              */
    double*        w_dev;         /* [batch][d][d]  in: start point, out: raw W           */
    const uint8_t* mask_exc_dev;  /* [d][d] 1 = excluded edge, shared by the batch, or 0  */
    const uint8_t* mask_inc_dev;  /* [d][d] 1 = included edge, shared by the batch, or 0  */
    /* outputs */
    int32_t* status_dev;          /* [batch] DAGMA_ST_* bits                              */
    double*  stage_stats_dev;     /* [batch][n_stages][8]: iters done, final lr, final s,
                                     obj, score, h, retries, back-tracks                  */
    double*  final_dev;           /* [batch][2]: h(W, s=1) and score(W)  linear.py:456-457 */
    double*  ckpt_log_dev;        /* [batch][cap][6]: stage, iter, obj, score, h, lr       */
    int32_t* ckpt_count_dev;      /* [batch]                                               */
    uint32_t* work_counter_dev;   /* one zero-initialised uint32 (work queue head)         */
    /* optional telemetry of the checkpoint iterations (the fork's `minimize.checkpoint` event,
       src/dagma/linear.py:262-273, 307-324), one row per ckpt_log row, or NULL:
       [batch][cap][DAGMA_DIAG_COLS] = ||Gobj||, ||G_score||, ||G_h||, ||G_l1||, ||G_inc||, ||Adam direction||,
       ||W||, sum|W|, max|W|, min nonzero |W| (after the step), seconds since the minimize call started   */
    double*  ckpt_diag_dev;
} dagma_small_fit_args;

int dagma_linear_fit_small_f64(dagma_stream_t stream, const dagma_small_fit_args* args);
/* DagmaLinear('logistic').minimize / fit for a batch of problems; src/dagma/linear.py:90-92, 165-333, 441-457.
 * args->cov_dev = X^T X / n of the UN-centred X; x_dev [batch][n][d] row-major; 1 <= d <= DAGMA_SMALL_MAX_D;
 * args->ckpt_diag_dev must be NULL (no telemetry rows on this path).  One CTA per problem (two per SM), pulled
 * from the work queue; X streams through shared memory every iteration.                                       */
int dagma_linear_fit_small_logistic_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                        int n, const double* x_dev);
/* DagmaLinear('l2', trek_reg=PST(seq="inv", mode="opt")).minimize / fit for a batch of problems;
 * src/dagma/linear.py:165-333, 441-457 with the trek term of :224-276, src/notreks/notreks.py:500-507, 599-619:
 *   Gobj += w_b * 2 W o GT^T,  GT = X Gt X,  X = ((1 + eps_inv) I - W o W)^{-1},  obj += w_b * pst(W).
 * Pairs of problem b: pairs_dev[pair_off_dev[b] .. pair_off_dev[b + 1]) as (i, j) int32 pairs, 0 <= i, j < d, duplicates
 * accumulate; pair_off_dev [batch + 1] with pair_off_dev[0] = 0; pairs_dev 8-byte aligned and non-NULL (also when
 * there are no pairs).  trek_weight_dev [batch] = w_b.  A problem without pairs has no trek term.  agg (DAGMA_PST_*)
 * and eps_inv are shared by the batch.  1 <= d <= DAGMA_SMALL_MAX_D; args->ckpt_diag_dev must be NULL.  One CTA per
 * problem (one per SM), pulled from the work queue.                                                              */
#define DAGMA_PST_MEAN 0
#define DAGMA_PST_SUM 1
#define DAGMA_PST_MAX 2
#define DAGMA_PST_LSE 3
int dagma_linear_fit_small_pst_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                   const int32_t* pair_off_dev, const int32_t* pairs_dev,
                                   const double* trek_weight_dev, int agg, double eps_inv);
/* The same for PST(seq="exp", mode="opt") (src/notreks/notreks.py:496-498): F = expm(W o W) by the degree-
 * DAGMA_PST_EXP_DEGREE Taylor polynomial (Horner) of W o W / 2^DAGMA_PST_EXP_SQUARINGS followed by that many squarings,
 * H = F^T F, and GT = the top-right block of expm([[W o W, Gt], [0, W o W]]) with Gt = (F (G_H + G_H^T))^T, by the same
 * algorithm on the two blocks of the block upper-triangular iterates.  Same contract and checks as above; the series
 * has no eps_inv.  One CTA per problem (one per SM).                                                              */
#define DAGMA_PST_EXP_DEGREE 18
#define DAGMA_PST_EXP_SQUARINGS 12
int dagma_linear_fit_small_pst_exp_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                       const int32_t* pair_off_dev, const int32_t* pairs_dev,
                                       const double* trek_weight_dev, int agg);
/* The same for TCC(cycle_penalty="spectral", mode="opt") (src/notreks/notreks.py:156-239, 340-378), version
 * approx_trek_graph or DAG_learning: the Perron pair (rho, u, v) of A = [[W o W, w S], [I, (W o W)^T]] (S the 0/1
 * indicator of the pairs, duplicates set the same entry) by power steps x <- x' / (||x'|| + eps) from the all-ones
 * vectors at every evaluation, A never formed:
 *   Gobj += weight_b * 2 W o [(u1 v1^T + v2 u2^T) / (m (u.v + eps)) - (u1 u1^T + u2 u2^T) / (m (u.u + eps))],
 *   obj  += weight_b * (rho - u.Bu / (u.u + eps)) / m,   B = [[W o W, 0], [I, (W o W)^T]],
 * the baseline terms for approx_trek_graph only; m = pair_off_dev[b + 1] - pair_off_dev[b] (duplicates counted).
 * Per problem: w_dev, eps_dev, n_iter_dev, flags_dev (DAGMA_TCC_* bits).  DAGMA_TCC_POWER: n_iter_dev[b] unshifted
 * steps.  Otherwise (eig_*): DAGMA_TCC_EIG_WARMUP unshifted steps, rho0 = |v.Av / (v.v + eps)|; if rho0 >
 * DAGMA_TCC_EIG_NILPOTENT, chunks of DAGMA_TCC_EIG_CHUNK steps on A + DAGMA_TCC_EIG_SHIFT rho0 I until
 * ||v - v_prev||^2 <= DAGMA_TCC_EIG_TOL^2 or DAGMA_TCC_EIG_MAX_CHUNKS chunks (then status gains DAGMA_ST_PERRON_CAP).
 * perron_steps_dev [batch] (NULL allowed): power steps of all evaluations of the problem.  Pairs, pair_off_dev,
 * weight_dev and the other arguments as in dagma_linear_fit_small_pst_f64.  One CTA per problem (one per SM).     */
#define DAGMA_ST_PERRON_CAP 8            /* some Perron solve hit DAGMA_TCC_EIG_MAX_CHUNKS (not converged) */
#define DAGMA_TCC_POWER 1                /* flags: method "power" (else eig_numpy / eig_torch)              */
#define DAGMA_TCC_DAG_LEARNING 2         /* flags: version DAG_learning (else approx_trek_graph)            */
#define DAGMA_TCC_EIG_WARMUP 8
#define DAGMA_TCC_EIG_CHUNK 64
#define DAGMA_TCC_EIG_MAX_CHUNKS 600
#define DAGMA_TCC_EIG_TOL 1e-13
#define DAGMA_TCC_EIG_SHIFT 0.25
#define DAGMA_TCC_EIG_NILPOTENT 1e-200
int dagma_linear_fit_small_tcc_f64(dagma_stream_t stream, const dagma_small_fit_args* args,
                                   const int32_t* pair_off_dev, const int32_t* pairs_dev, const double* weight_dev,
                                   const double* w_dev, const double* eps_dev, const int32_t* n_iter_dev,
                                   const int32_t* flags_dev, int64_t* perron_steps_dev);
/* launch geometry chosen for (d): CTAs, threads, dynamic shared memory bytes */
int dagma_linear_fit_small_geometry(int d, int batch, int* ctas, int* threads, size_t* smem_bytes);

/* max number of CTAs of the last 32 < d <= DAGMA_SMALL_MAX_D fit launch that shared one SM, counted by the kernel
 * itself (the geometry above assumes 2 for that path); synchronises with the device                          */
int dagma_fit_dmma_residency(int* out_host);

/* ---- host-buffer convenience: the call a reference user makes --------------------
 * Replaces: DagmaLinear.fit for a batch of problems given host covariances; does
 * H2D, the fit and D2H on `stream`, then synchronises.  w_host in/out [batch][d][d].  */
int dagma_linear_fit_small_host_f64(dagma_stream_t stream, const dagma_small_fit_args* args_host_ptrs);

/* ---- large-d / logistic building blocks (one inner iteration = a fixed launch sequence) ---
 * FP64 tensor-core (DMMA) GEMM, row-major:  C = alpha * op(A) * B + beta * C, optional
 * sigmoid epilogue (epilogue = 1).  Replaces the BLAS calls of the score:
 *   cov @ (I - W)                       src/dagma/linear.py:86, 244
 *   X @ W, (X^T / n) @ sigmoid(X @ W)   src/dagma/linear.py:90-92, 246
 * ws_dev: optional split-K workspace (deterministic two-pass reduction).
 * lda >= K (trans_a: lda >= M), ldb >= N, ldc >= N; K = 0 gives C = beta * C (then the
 * epilogue), as BLAS does.                                                            */
int dagma_gemm_f64(dagma_stream_t stream, int trans_a, int M, int N, int K, double alpha,
                   const double* a_dev, int lda, const double* b_dev, int ldb, double beta,
                   double* c_dev, int ldc, int epilogue, double* ws_dev, size_t ws_bytes);

/* single-problem fused slogdet+inverse with caller-provided workspace (graph capturable);
 * d <= 128 on chip, larger d blocked Gauss-Jordan with DMMA trailing updates.           */
size_t dagma_large_workspace_bytes(int d);
int dagma_logdet_inv_ws_f64(dagma_stream_t stream, int d, double s, const double* a_dev, int lda,
                            int square_input, double* logabsdet_dev, double* h_dev, double* minv_dev,
                            double* grad_dev, int ldo, double* min_entry_dev, int* info_dev,
                            double* ws_dev, size_t ws_bytes);

/* the same inverse with a "rider": gc = ga @ gb (all d x d, row-major, ld = d), an independent GEMM of the same
 * iteration (cov @ W of the l2 score, src/dagma/linear.py:86, 244).  For d > 256 both are ONE dependency-driven
 * persistent kernel: the rider's 64 x 64 x 256 tiles fill the time the engines would otherwise spend waiting for
 * the serial pivot chain of the blocked inverse.  Smaller d: the two run back to back.                       */
int dagma_logdet_inv_gemm_ws_f64(dagma_stream_t stream, int d, double s, const double* a_dev, int lda,
                                 int square_input, double* logabsdet_dev, double* h_dev, double* minv_dev,
                                 double* grad_dev, int ldo, double* min_entry_dev, int* info_dev,
                                 double* ws_dev, size_t ws_bytes, const double* ga_dev, const double* gb_dev,
                                 double* gc_dev);

/* device-resident iteration state (19 doubles): mu, s, lr, lambda1, beta1, beta2,
 * beta1^it (hi, lo), beta2^it (hi, lo), logabsdet, h, min_entry, score_acc, l1_acc,
 * loss_acc, gscale, then int32 it, halted, info, pad.                                   */
#define DAGMA_LIN_STATE_DOUBLES 19
/* Gobj + Adam + step + masks + iteration counter; no-op (latching `halted`) if the
 * inverse of this iteration was infeasible.   src/dagma/linear.py:248, 158-162, 275-276  */
int dagma_linear_update_f64(dagma_stream_t stream, int d, void* state_dev, double* w_dev,
                            const double* minv_dev, const double* t_dev, const double* cov_dev,
                            double* m_dev, double* v_dev, const uint8_t* mask_exc_dev,
                            const uint8_t* mask_inc_dev);
/* the same update with one more gradient term  extra_scale * 2 W o extra_t^T  (extra_t_dev row-major d x d or NULL):
 * the trek regulariser in mode "opt", weight * d pst / d W  (src/dagma/linear.py:251-258, src/notreks/notreks.py:
 * 454-619; for PST seq="inv" extra_t = X M_s H with X = (I - W o W)^{-1}, H = X^T X, M_s the symmetrised pair mask) */
int dagma_linear_update_ex_f64(dagma_stream_t stream, int d, void* state_dev, double* w_dev,
                               const double* minv_dev, const double* t_dev, const double* cov_dev,
                               double* m_dev, double* v_dev, const uint8_t* mask_exc_dev,
                               const uint8_t* mask_inc_dev, const double* extra_t_dev, double extra_scale);
/* W += sign * lr * (previous Adam direction)     src/dagma/linear.py:235, 239           */
int dagma_linear_apply_dir_f64(dagma_stream_t stream, int d, const void* state_dev, double* w_dev,
                               const double* m_dev, const double* v_dev, double sign);
/* The WHOLE inner iteration -- fused inverse, score product(s), the update above -- and `iters` consecutive ones as
 * ONE persistent kernel (csrc/lin_iter.cu) for d <= 128, l2 or logistic, un-sharded rows, no trek regulariser: one CTA
 * inverts sI - W o W on chip while the worker CTAs form T (logistic: every worker keeps <= 72 rows of X in shared
 * memory for the whole launch, partial X^T sigmoid(XW) per worker summed in a fixed order; l2: cov W), then every CTA
 * updates its share of the entries; CTA 0 advances the state block.  Replaces the loop body of DagmaLinear.minimize
 * (src/dagma/linear.py:224-276) between two checkpoints; state block, buffers and results are those of the launch
 * sequence (inverse -> dagma_gemm_f64 -> dagma_linear_update_f64).
 *   supported          : 1 when the shape is covered on this device (logistic: n <= 72 (SMs - 1), the rows stay resident
 *                        in shared memory; DAGMA_LIN_STREAM=1 opts in to streaming more rows through it every iteration,
 *                        measured slower than the launch sequence)
 *   workspace_doubles  : size of part_dev
 *   x_dev [n][d] row-major (logistic only, else NULL / n = 0); sync_dev: 4 uint32 that live as long as the state
 *   block; info = 99 in the state block: a grid barrier timed out (the grid was not co-resident).                  */
int dagma_linear_iter_supported(int logistic, int n, int d);
size_t dagma_linear_iter_workspace_doubles(int logistic, int n, int d);
int dagma_linear_iter_f64(dagma_stream_t stream, int logistic, int n, int d, int iters, void* state_dev,
                          double* w_dev, double* m_dev, double* v_dev, double* minv_dev, double* t_dev,
                          const double* cov_dev, const double* x_dev, const uint8_t* mask_exc_dev,
                          const uint8_t* mask_inc_dev, double* part_dev, unsigned* sync_dev);
/* Rows of X sharded over the GPUs of ONE box, one process per GPU (SURVEY.md 8e2; the reference has no multi-device
 * path: this replaces the all-reduce a torch.distributed port of linear.py:246 would issue every iteration).  The same
 * persistent kernel runs on every GPU on its n_local rows; the sum of the d x d partial products over the GPUs happens
 * inside it by plain stores / loads over NVLink peer memory, in rank order on every GPU (bit-identical replicas).
 *   exchange_bytes : size of one GPU's exchange allocation (dagma_peer_alloc), zero on entry of the first launch
 *   exchange_ptrs  : [nranks] host array, entry r = rank r's allocation as mapped into THIS process (entry `rank`: the
 *                    own allocation; the others: dagma_peer_import of the handles the peers exported)
 * All ranks must launch the same sequence of calls (same iters); a peer that does not show up ends the launch with
 * info = 99 after a bounded wait.                                                                                  */
size_t dagma_linear_iter_exchange_bytes(int d, int nranks);
int dagma_linear_iter_sharded_f64(dagma_stream_t stream, int n_local, int d, int iters, void* state_dev,
                                  double* w_dev, double* m_dev, double* v_dev, double* minv_dev, double* t_dev,
                                  const double* cov_dev, const double* x_dev, const uint8_t* mask_exc_dev,
                                  const uint8_t* mask_inc_dev, double* part_dev, unsigned* sync_dev, int rank,
                                  int nranks, void* const* exchange_ptrs);
/* Batched graph evaluation (csrc/graph_metrics.cu): the counts behind utils.count_accuracy and the test utils.is_dag
 * (src/dagma/utils.py:245-310, 13-18; no igraph) for `batch` estimates in one launch.
 *   est_dev  [batch][d][d] int8 in {0, 1, -1} (-1: undirected edge of a CPDAG, once per pair)
 *   true_dev [batch][d][d] uint8 (or ONE [d][d] matrix for all problems when true_shared = 1)
 *   counts_dev [batch][8] int32: nnz, condition positive, true positive, false positive, reverse, extra (lower
 *   triangle of the skeleton), missing (lower), is_dag (directed support of the estimate)                            */
int dagma_graph_metrics(dagma_stream_t stream, int batch, int d, const int8_t* est_dev, const uint8_t* true_dev,
                        int true_shared, int* counts_dev);
/* Peer-visible device memory (csrc/peer.cu): an allocation of its own (zeroed), its 64-byte inter-process handle, the
 * import of a peer's handle into this process (peer access enabled on demand) and the matching release / free.       */
#define DAGMA_PEER_HANDLE_BYTES 64
int dagma_peer_alloc(size_t bytes, void** out_dev);
int dagma_peer_free(void* dev);
int dagma_peer_export(void* dev, unsigned char* handle_out);
int dagma_peer_import(const unsigned char* handle, void** out_dev);
int dagma_peer_release(void* imported_dev);
/* a non-blocking stream of its own for one lane of a mid-d batch (midagma_b200.linear._run_lanes)                     */
int dagma_stream_create(void** out_stream);
int dagma_stream_destroy(void* stream);
/* checkpoint reductions: l2 score 1/2 tr((I-W)^T cov (I-W)) and sum|W|   linear.py:85-87, 129 */
int dagma_linear_objective_f64(dagma_stream_t stream, int d, void* state_dev, const double* w_dev,
                               const double* t_dev, const double* cov_dev, int l2);
/* the same on a grid of CTAs (fixed-order two-level sum); ws_dev: dagma_linear_objective_workspace_bytes() bytes, the
 * first 8 zero before the first call                                                        */
size_t dagma_linear_objective_workspace_bytes(void);
int dagma_linear_objective_ws_f64(dagma_stream_t stream, int d, void* state_dev, const double* w_dev,
                                  const double* t_dev, const double* cov_dev, int l2, double* ws_dev, size_t ws_bytes);
/* out = scale * sum(logaddexp(0, R) - X o R)      src/dagma/linear.py:91                 */
int dagma_logistic_loss_f64(dagma_stream_t stream, int n, int d, const double* x_dev, const double* r_dev,
                            double scale, double* partial_dev, int n_partial, double* out_dev);

/* Replaces: DagmaLinear._adam_update   src/dagma/linear.py:158-163 (bias1 = 1 - beta1^iter) */
int dagma_adam_direction_f64(dagma_stream_t stream, size_t n, const double* grad_dev, double* m_dev,
                             double* v_dev, double beta1, double beta2, double bias1, double bias2,
                             double* out_dev);

/* ---- (iv) DagmaMLP / DagmaNonlinear, dims = [d, m1, 1] --------------------------------------
 * theta = [W1 (P x d) | b1 (P) | W2 (P) | b2 (d)], P = d*m1 (fc1.weight, fc1.bias, fc2.0.weight,
 * fc2.0.bias of the reference state_dict, src/dagma/nonlinear.py:36-43).  Activations are
 * [P][n] (transposed).  Device state block (17 doubles): mu, s, lr, lambda1, lambda2, beta1,
 * beta2, logabsdet, h, min_entry, S, l1, obj, score, lr_gamma, then int32 step, halted, info.
 * One iteration of DagmaNonlinear.minimize (nonlinear.py:212-225) is:
 *   dagma_mlp_adj  -> dagma_logdet_inv_ws (square_input = 0)  -> dagma_gemm (Zt = W1 Xt)
 *   -> dagma_mlp_forward -> [all-reduce S] -> dagma_mlp_objective -> dagma_mlp_backward
 *   -> dagma_gemm (gW1 = dZt X) -> [all-reduce grads] -> dagma_mlp_adam                        */
#define DAGMA_MLP_STATE_DOUBLES 17
/* A[i][j] = sum_k fc1[j,k,i]^2 and partial sums of |fc1|        nonlinear.py:82-84, 97          */
int dagma_mlp_adj_f64(dagma_stream_t stream, int d, int m1, const double* theta_dev, double* a_dev,
                      double* l1_partial_dev);
/* sigmoid + locally-connected layer + residual + partial sum of squares   nonlinear.py:60-65,
 * locally_connected.py:70-74; writes S and l1 into the state block                              */
int dagma_mlp_forward_f64(dagma_stream_t stream, int n, int d, int m1, double* zt_dev,
                          const double* theta_dev, const double* xt_dev, double* res_dev,
                          double* out_opt_dev, double* s_partial_dev, const double* l1_partial_dev,
                          void* state_dev);
/* score = d/2 log(S / n), obj = mu (score + lambda1 l1) + h; latches halted if h < 0
 *                                                               nonlinear.py:158, 215-221        */
int dagma_mlp_objective_f64(dagma_stream_t stream, void* state_dev, int n_total, int d);
/* closed-form backward of the two-layer MLP (un-scaled sums)     autograd of nonlinear.py:218-222 */
int dagma_mlp_backward_f64(dagma_stream_t stream, int n, int d, int m1, double* ht_dev,
                           const double* theta_dev, const double* res_dev, double* part_dev,
                           double* grads_tail_dev);
/* torch.optim.Adam(betas, weight_decay = mu lambda2) over theta + ExponentialLR   nonlinear.py:208-225 */
int dagma_mlp_adam_f64(dagma_stream_t stream, int d, int m1, void* state_dev, double* theta_dev,
                       const double* grads_dev, double* m_dev, double* v_dev, const double* minv_dev);
/* same step over a flat theta of `total` doubles whose first d*m1*d entries are fc1.weight (any stack) */
int dagma_mlp_adam_ex_f64(dagma_stream_t stream, int d, int m1, size_t total, void* state_dev, double* theta_dev,
                          const double* grads_dev, double* m_dev, double* v_dev, const double* minv_dev);
/* The WHOLE iteration above -- and `iters` consecutive ones -- as ONE persistent kernel (csrc/mlp_iter.cu) for
 * dims = [d, m1, 1], d <= 64, m1 <= 40, un-sharded rows: worker CTAs own (node slice, sample group) pairs and keep
 * their samples in shared memory, one CTA inverts sI - A on chip, two grid barriers per iteration, every sum in a
 * fixed order.  Replaces the loop body of DagmaNonlinear.minimize (nonlinear.py:212-225) between two checkpoints.
 *   supported          : 1 when the shape is covered on this device (otherwise use the sequence above)
 *   workspace_doubles  : size of part_dev
 *   x_dev [n][d] row-major (this process's rows, n_total = n); sync_dev: 4 zeroed uint32 that live as long as the
 *   state block; info = 99 in the state block: a grid barrier timed out (the grid was not co-resident).          */
int dagma_mlp_iter_supported(int n, int d, int m1);
size_t dagma_mlp_iter_workspace_doubles(int n, int d, int m1);
int dagma_mlp_iter_f64(dagma_stream_t stream, int n, int n_total, int d, int m1, int iters, void* state_dev,
                       double* theta_dev, double* m_dev, double* v_dev, const double* x_dev, double* part_dev,
                       double* minv_dev, unsigned* sync_dev);
/* The same with the rows of X sharded over the GPUs of ONE box, one process per GPU (SURVEY.md 8e2): the sums of the
 * un-scaled gradients and of S over the GPUs happen inside the kernel over NVLink peer memory, in rank order on every
 * GPU (bit-identical replicas, no collective call in the loop).  exchange_ptrs: as for dagma_linear_iter_sharded_f64,
 * allocations of dagma_mlp_iter_exchange_bytes(d, m1, nranks) bytes.                                              */
size_t dagma_mlp_iter_exchange_bytes(int d, int m1, int nranks);
int dagma_mlp_iter_sharded_f64(dagma_stream_t stream, int n_local, int n_total, int d, int m1, int iters,
                               void* state_dev, double* theta_dev, double* m_dev, double* v_dev, const double* x_dev,
                               double* part_dev, double* minv_dev, unsigned* sync_dev, int rank, int nranks,
                               void* const* exchange_ptrs);
/* Batched DagmaNonlinear.minimize (nonlinear.py:161-236, one call per problem) for many independent dims = [d, m1, 1]
 * problems of the same shape, ONE CTA per problem from a work queue (csrc/mlp_batch.cu).  Problem b runs up to
 * max_iter iterations from states_dev[b] (MlpState: mu, s, lr, lambda1, lambda2, beta1, beta2, lr_gamma, step and
 * halted are read; lr, logabsdet, h, S, l1, obj, score, step and halted are written), theta/m/v [batch][W] with
 * W = d*m1*d + 2*d*m1 + d (the layout above) and x_dev [batch][n][d]; it stops at h < 0 (halted = 1: the reference
 * returns False, nonlinear.py:215-217) or when the objective meets tol at a checkpoint iteration
 * (i % checkpoint == 0 or i == max_iter - 1, nonlinear.py:226-231).  idx_dev (optional): the n_idx problems to
 * run; NULL runs all of them.  grad_dev [batch][W]: scratch; iters_dev[b]: the iterations run;
 * work_counter_dev: one uint32.
 *   supported : 1 when 1 <= d <= 64, 1 <= m1 <= 40 and n >= 1                                               */
int dagma_mlp_batch_supported(int n, int d, int m1);
int dagma_mlp_minimize_batch_f64(dagma_stream_t stream, int batch, int n, int d, int m1, int max_iter, int checkpoint,
                                 double tol, const int* idx_dev, int n_idx, void* states_dev, double* theta_dev,
                                 double* m_dev, double* v_dev, const double* x_dev, double* grad_dev, int* iters_dev,
                                 unsigned* work_counter_dev);
/* General LocallyConnected stacks dims = [d, m_1, ..., 1] (nonlinear.py:39-43, 60-65), transposed activations
 * [d * width][n], one call per layer.
 *   lc_forward : in ([d*mi][n]; + bias_in for the first layer) is replaced by H = sigmoid(in);
 *                out[(j*mo+o)][s] = b[j][o] + sum_k H[j*mi+k][s] w[j][k][o]          locally_connected.py:70-74
 *   residual   : res = out (+ bias) - xt, S = sum res^2 and l1 -> state (the tail of nonlinear.py:60-66, 158)
 *   lc_backward: H is replaced by dZ = (sum_o w[j][k][o] dzn[j*mo+o]) H (1 - H); grads = [gW (d*mi*mo) | gb (d*mo)]
 *                un-scaled sums over the samples (part_dev: ceil(n/256) rows of that width)
 *   row_sums   : out[r] = sum_s a[r][s]  (fc1.bias gradient)                                              */
int dagma_lc_forward_f64(dagma_stream_t stream, int n, int d, int mi, int mo, double* in_dev,
                         const double* bias_in_dev, const double* w_dev, const double* b_dev, double* out_dev);
int dagma_mlp_residual_f64(dagma_stream_t stream, int n, int d, const double* out_dev, const double* bias_dev,
                           const double* xt_dev, double* res_dev, double* out_opt_dev, double* s_partial_dev,
                           const double* l1_partial_dev, void* state_dev);
int dagma_lc_backward_f64(dagma_stream_t stream, int n, int d, int mi, int mo, double* h_dev, const double* dzn_dev,
                          const double* w_dev, double* part_dev, double* grads_dev);
int dagma_row_sums_f64(dagma_stream_t stream, int rows, int n, const double* a_dev, double* out_dev);
/* LocallyConnected.forward                                       locally_connected.py:55-75     */
int dagma_locally_connected_f64(dagma_stream_t stream, int n, int d, int m1, int m2, const double* in_dev,
                                const double* w_dev, const double* b_dev, double* out_dev);
/* out = sum (a - b)^2  (log_mse_loss, nonlinear.py:158)                                           */
int dagma_sumsq_diff_f64(dagma_stream_t stream, size_t total, const double* a_dev, const double* b_dev,
                         double* partial_dev, int n_partial, double* out_dev);

/* ---- the fork's log-det trek-cycle-coupling constraint -----------------------------------
 * A = [[W o W, w S], [I, (W o W)^T]] (2d x 2d; with_s = 0: baseline B)   src/notreks/notreks.py:319-337
 * fold: out (+)= sign * 2 W o (G11 + G22^T)                              src/notreks/notreks.py:285-287, 384
 * The value/gradient themselves come from dagma_logdet_inv_f64(square_input = 0).             */
int dagma_tcc_assemble_f64(dagma_stream_t stream, int d, const double* w_dev, const double* s_dev,
                           double w, int with_s, double* a_dev);
int dagma_tcc_fold_f64(dagma_stream_t stream, int d, const double* w_dev, const double* g_dev, double sign,
                       int accumulate, double* out_dev);

/* ---- the fork's spectral trek-cycle-coupling penalty (SURVEY.md 8f3) ---------------------------
 * Replaces: perron_eig_with_gradA(method="power")           src/notreks/notreks.py:178-194
 *           and, iterated to convergence on A + shift I, the Perron pair the eig methods return (:196-231)
 * n_iter steps of v <- A v / (||A v|| + eps), u <- A^T u / (||A^T u|| + eps) from the all-ones vectors (start = 0)
 * or from the given unit vectors (start = 1); one pass over A per step serves both chains.  square != 0: the
 * matrix is a_dev o a_dev.  scal_dev[0..3] = rho = v.(A v) / (v.v + eps), u.v, u.u, v.v.                        */
size_t dagma_power_workspace_bytes(int n);
int dagma_perron_power_f64(dagma_stream_t stream, int n, const double* a_dev, int lda, int square, double shift,
                           int n_iter, double eps, int start, double* v_dev, double* u_dev, double* scal_dev,
                           double* ws_dev, size_t ws_bytes);
/* y = A x (or (A o A) x): the Rayleigh baseline u.(B u) of the "approx_trek_graph" version   notreks.py:365   */
int dagma_matvec_f64(dagma_stream_t stream, int n, const double* a_dev, int lda, int square, const double* x_dev,
                     double* y_dev);
/* out4 = [x.y, x.x, y.y, |x - y|^2] (fixed-order sums)                                                        */
int dagma_vec_dots_f64(dagma_stream_t stream, int n, const double* x_dev, const double* y_dev, double* out4_dev);
/* out (+)= num / (den_dev[0] + eps) * 2 W o (a1 b1^T + a2 b2^T): d rho / dA = u v^T / (u.v) folded onto W through
 * A11 = W o W, A22 = (W o W)^T without forming the 2d x 2d outer product     notreks.py:236, 278-287, 343-371
 * (w_dev = NULL: the factor 2 W is left out -- the d / d(W o W) form the fused update kernel consumes)          */
int dagma_rank2_fold_f64(dagma_stream_t stream, int d, const double* w_dev, const double* a1_dev,
                         const double* b1_dev, const double* a2_dev, const double* b2_dev, double num,
                         const double* den_dev, double eps, int accumulate, double* out_dev);

/* ---- data staging in front of the path ---------------------------------------------
 * Replaces: X -= X.mean(0) (in place) and cov = X^T X / n   src/dagma/linear.py:410-411, 428
 * x_dev [batch][n][d] (centred in place when center != 0), cov_dev [batch][d][d].     */
int dagma_center_cov_f64(dagma_stream_t stream, int batch, int n, int d, double* x_dev,
                         int center, double* cov_dev);

/* ---- pairwise independence tests in front of the path (SURVEY.md 8f4) ----------------
 * Replaces: hsic_stat / dcor_stat / permutation_pvalue      src/notreks/mi_tests.py:19-135
 * Every variable's double-centred Gram matrix (RBF kernel: kind 0, sigma2_dev[v]; absolute distance: kind 1)
 * is built once, g_dev [nvars][n][n]; a permuted statistic is the gathered dot product
 * out[q * nperm + p] = scale * sum_ab G[vi[q]][a][b] * G[vj[q]][pi(a)][pi(b)], pi = perms_dev[q][p][0..n).
 * dagma_mi_upper_d2_f64 writes the n (n - 1) / 2 squared distances of one column (input of the median
 * heuristic, mi_tests.py:41-46).                                                                        */
int dagma_mi_upper_d2_f64(dagma_stream_t stream, int n, int d, int col, const double* x_dev, double* out_dev);
int dagma_mi_centered_gram_f64(dagma_stream_t stream, int n, int d, int nvars, const int* cols_dev,
                               const double* x_dev, const double* sigma2_dev, int kind, double* g_dev,
                               double* rowmean_dev, double* allmean_dev);
size_t dagma_mi_perm_workspace_bytes(int n, int npairs, int nperm);
int dagma_mi_perm_dots_f64(dagma_stream_t stream, int n, const double* g_dev, int npairs, const int* vi_dev,
                           const int* vj_dev, const int* perms_dev, int nperm, double scale, double* ws_dev,
                           size_t ws_bytes, double* out_dev);

/* ---- FP64 pipe yardsticks used by bench.py for the roofline denominator ---------- */
int dagma_bench_fp64_fma(dagma_stream_t stream, int ctas, int threads, int iters, double* sink_dev);
int dagma_bench_fp64_dmma(dagma_stream_t stream, int ctas, int threads, int iters, double* sink_dev);
/* 4 x 4 accumulator tiles from 4 A / 4 B fragments (mode 1: fragments reloaded from shared memory) */
int dagma_bench_fp64_dmma_tiles(dagma_stream_t stream, int ctas, int threads, int iters, int mode,
                                double* sink_dev);
/* dependent-issue latencies (cycles / op, one warp): out_dev[0..8] = DFMA, DMMA via C, DMMA via A,
 * 64-bit SHFL, MUFU.RCP64H + DFMA, LDS chase, STS/sync/LDS round trip, DADD, DMUL (16 doubles) */
int dagma_bench_latency(dagma_stream_t stream, double* out_dev);
/* serial chain of the on-chip sweep in isolation: out[0] clk per 8 x 8 pivot-block inversion, out[1] with the
   diagonal warp's DMMAs interleaved, out[2] max |P - inv(inv(P))| */
int dagma_bench_stage(dagma_stream_t stream, double* out_dev);
/* timing experiment: c = a @ b (d x d, d even) by the engine pairs of the persistent inverse kernels, one 64 x 64 tile
   per engine (persistent = 0) or from an atomic queue (persistent = 1; queue_dev: one unsigned) */
int dagma_bench_engine_gemm(dagma_stream_t stream, int d, const double* a_dev, const double* b_dev, double* c_dev,
                            int persistent, unsigned* queue_dev);
/* timing experiment: c = alpha a @ b + beta c by the TMA-fed GEMM (cp.async.bulk.tensor slabs + mbarrier pipeline;
   a: M x K, b: K x N, row-major, even leading dimensions, 16-byte aligned); mode 0 = static tile striding,
   1 = tiles from an atomic queue (queue_dev: one unsigned) */
int dagma_bench_tma_gemm(dagma_stream_t stream, int M, int N, int K, const double* a_dev, int lda,
                         const double* b_dev, int ldb, double* c_dev, int ldc, double alpha, double beta, int mode,
                         unsigned* queue_dev);

#ifdef __cplusplus
}
#endif
#endif /* DAGMA_B200_H */
