// Batched DagmaNonlinear.minimize for many independent DagmaMLP [d, m1, 1] problems, d <= 64, m1 <= 40: ONE CTA per
// problem runs up to max_iter iterations of the inner loop (reference: src/dagma/nonlinear.py:161-236; the iteration
// of _MlpEngine / mlp_iter_kernel).  The path-following and retry policy of fit (nonlinear.py:509-527) stays on the
// host; a retry relaunches only the failed problems through the index list.
//
// Mapping (256 threads, TWO CTAs per SM, problems pulled from an atomic work queue; no grid barriers, no host round
// trips).  Per iteration:
//   h        A(W1)[i][j] = sum_k W1[j m1 + k][i]^2 into shared memory, M = (sI - A) / 2^e in the accumulator layout,
//            inverted by the tensor-core sweep of small_dmma.cuh (as mlp_iter's h CTA does): h, log|det|, and
//            M^{-1} kept in shared memory for the step.  h < 0: the problem halts before the step
//            (nonlinear.py:215-217).
//   data     node slice by node slice (<= 40 rows of fc1.weight, the MiPlan slicing of mlp_iter.cu), the problem's X
//            streams through shared memory in tiles of MB_TR rows, double-buffered by cp.async.  Per tile:
//              Z = W1_slice X_t^T      DMMA.8x8x4, one warp per m-tile (two n-tiles = the tile's rows)
//              H = sigmoid(Z + b1), out, res, S += res^2, gb2 += res      four threads per node
//              dZ = res W2 H (1 - H) over H, gb1 += dZ, gW2 += res H      four threads per hidden unit
//              gW1_slice += dZ X_t     DMMA, warp w owns the accumulator tiles w, w + 8, ... in registers
//            every sum un-scaled and in a fixed order (tiles in order, fixed thread ownership): a problem's result
//            does not depend on which CTA runs it, or when.  The slice's sums go to the problem's row of `grad`.
//   step     objective at the pre-step parameters, then the torch-Adam step over all parameters exactly as
//            mlp_iter's phase B (d / S, l1 sub-gradient, dh/dW1 = 2 W1 M^{-T}, weight decay mu lambda2,
//            ExponentialLR every 1000 steps); at checkpoint iterations (i % checkpoint == 0 or i == max_iter - 1)
//            |(obj_prev - obj) / obj_prev| <= tol ends the call (nonlinear.py:226-231).
// Parameters, Adam moments and the gradient sums live in global memory (the resident problems' working set stays
// mostly in L2).
#include "common.cuh"
#include "small_dmma.cuh"
#include "gemm_f64.cuh"
#include "mlp_state.h"
#include "../../include/dagma_b200.h"

namespace dagma {

constexpr int MB_NT = 256;        // threads per CTA
constexpr int MB_TR = 16;         // rows of X per tile (two DMMA n-tiles)
constexpr int MB_PR = 40;         // rows of fc1.weight per node slice: <= 5 m-tiles
constexpr int MB_SEG = 4;         // threads per node / hidden unit in the element-wise passes
constexpr int MB_LDH = MB_TR + 4; // row stride of H (= 4 mod 16: conflict-free fragments)
constexpr int MB_ACC = 5;         // gW1 accumulator tiles per warp: 5 m-tiles x 8 n-tiles / 8 warps

struct MbSmem {                   // offsets in doubles; the sweep's buffers keep the offsets of DmmaSmem
    static constexpr int A = DmmaSmem::ncov;                   // A, then M^{-1}, [64][68] (the sweep leaves it alone)
    static constexpr int W1 = DmmaSmem::W;                     // [40][68] fc1.weight rows of the slice (zero padded)
    static constexpr int H = W1 + MB_PR * DM_LD;               // [40][MB_LDH] H, then dZ
    static constexpr int R = H + MB_PR * MB_LDH;               // [40][MB_TR] residuals; at a slice's end, the segment sums
    static constexpr int b1 = R + MB_PR * MB_TR;               // [40]
    static constexpr int W2 = b1 + MB_PR;                      // [40]
    static constexpr int b2 = W2 + MB_PR;                      // [40]
    static constexpr int X = (DmmaSmem::total + 1) & ~1;       // 2 x [MB_TR][68] X tiles
    static constexpr int total = X + 2 * MB_TR * DM_LD;
    static constexpr size_t bytes = (size_t)total * sizeof(double);
};
static_assert(MbSmem::b2 + MB_PR <= DmmaSmem::rbuf, "the slice buffers fit the area of W");
static_assert(MbSmem::H % 2 == 0 && MbSmem::X % 2 == 0, "16-byte alignment of vector accesses");
static_assert(3 * MB_PR * MB_SEG <= MB_PR * MB_TR, "the segment sums fit the residual buffer");

struct MbArgs {
    int batch, n, d, m1, max_iter, checkpoint;
    double tol;
    const int* idx;              // [n_run] problems to run (null: 0 .. n_run - 1)
    int n_run;
    MlpState* st;                // [batch]
    double *theta, *m, *v, *grad;// [batch][W]
    const double* X;             // [batch][n][d]
    int* iters;                  // [batch]
    unsigned* counter;
};

// 1 / (1 + exp(-z)) as mlp_iter.cu computes it
__device__ __forceinline__ double mb_sigmoid(double z) { return fast_rcp(1.0 + exp(fmin(-z, 700.0))); }

// h at the current fc1.weight: M^{-1} -> sm[A] ([d][68]); returns h, writes log|det| and sum |W1| (all threads)
__device__ __forceinline__ double mb_h(const double* W1, int d, int m1, double s, double* sm, const DmmaPos& ps,
                                      SweepSync& sy, double& lad_out, double& l1_out) {
    const int tid = threadIdx.x;
    double* As = sm + MbSmem::A;
    double l1 = 0.0;
    for (int e = tid; e < d * d; e += MB_NT) {
        const int j = e / d, i = e - j * d;
        double x = 0.0;
        for (int k = 0; k < m1; ++k) {
            const double w = __ldcg(W1 + (size_t)(j * m1 + k) * d + i);
            x = fma(w, w, x);
            l1 += fabs(w);
        }
        As[i * DM_LD + j] = x;
    }
    double scale = 1.0;
    if (s > 0.0 && isfinite(s)) {              // s / 2^e in (0.5, 1]: exact, keeps the publish identity in its accurate range
        int e = 0;
        const double f = frexp(s, &e);
        if (f == 0.5) --e;
        scale = ldexp(1.0, e);
    }
    const double inv_scale = 1.0 / scale;
    __syncthreads();
    double a[2][4][2];
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = ps.row(ti), c = ps.col(tj) + e;
                double v = (r == c) ? 1.0 : 0.0;
                if (r < d && c < d) v = (((r == c) ? s : 0.0) - As[r * DM_LD + c]) * inv_scale;
                a[ti][tj][e] = v;
            }
    dmma_sweep(a, ps, sm, d, sy);              // ends with a barrier: every read of A is done
    double ld = 0.0, zero = 0.0;
    if (tid < ((d + 3) & ~3)) ld = (double)((tid & 3) - 2) * log(fabs(sm[DmmaSmem::pinfo + tid]));
#pragma unroll
    for (int ti = 0; ti < 2; ++ti)
#pragma unroll
        for (int tj = 0; tj < 4; ++tj)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = ps.row(ti), c = ps.col(tj) + e;
                if (r < d && c < d) As[r * DM_LD + c] = a[ti][tj][e] * inv_scale;
            }
    block_sum3<MB_NT>(ld, l1, zero, sm + DmmaSmem::red, tid);     // (its barriers publish M^{-1})
    lad_out = ld + (double)d * log(scale);
    l1_out = l1;
    return -lad_out + (double)d * log(s);
}

// one node slice (nodes j0 .. j0 + jn - 1): forward, residuals, backward over all n rows; the slice's un-scaled sums
// -> grad; sq accumulates this thread's share of S (fixed ownership across slices and tiles)
__device__ __forceinline__ void mb_slice(const MbArgs& P, const double* theta, const double* xb, double* grad, double* sm,
                                         int j0, int jn, double& sq) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, qr = lane >> 2, qc = lane & 3;
    const int n = P.n, d = P.d, m1 = P.m1, PP = d * m1, p0 = j0 * m1, PR = jn * m1;
    const int MT = (PR + 7) >> 3, NT = (d + 7) >> 3, KT = (d + 3) >> 2, ntile = (n + MB_TR - 1) / MB_TR;
    double *W1s = sm + MbSmem::W1, *Hs = sm + MbSmem::H, *Rs = sm + MbSmem::R;
    double *b1s = sm + MbSmem::b1, *W2s = sm + MbSmem::W2, *b2s = sm + MbSmem::b2;

    auto load_tile = [&](int t) {
        double* dst = sm + MbSmem::X + (t & 1) * MB_TR * DM_LD;
        const int r0 = t * MB_TR;
        if ((d & 1) == 0) {                   // rows start on 16 bytes: X of a problem is n * d doubles, d even
            const int hc = d >> 1;
            for (int e = tid; e < MB_TR * hc; e += MB_NT) {
                const int r = e / hc, c2 = e - r * hc;
                const bool ok = r0 + r < n;
                cp_async16(smem_u32(dst + r * DM_LD + 2 * c2), ok ? xb + (size_t)(r0 + r) * d + 2 * c2 : xb, ok);
            }
        } else {
            for (int e = tid; e < MB_TR * d; e += MB_NT) {
                const int r = e / d, c = e - r * d;
                const bool ok = r0 + r < n;
                cp_async8(smem_u32(dst + r * DM_LD + c), ok ? xb + (size_t)(r0 + r) * d + c : xb, ok);
            }
        }
        cp_async_commit();
    };
    load_tile(0);
    // this iteration's parameters of the slice, zero padded to whole m-tiles / k-steps
    for (int e = tid; e < 8 * MT * DM_LD; e += MB_NT) {
        const int r = e / DM_LD, c = e - r * DM_LD;
        W1s[e] = (r < PR && c < d) ? __ldcg(theta + (size_t)(p0 + r) * d + c) : 0.0;
    }
    for (int e = tid; e < PR; e += MB_NT) {
        b1s[e] = __ldcg(theta + (size_t)PP * d + p0 + e);
        W2s[e] = __ldcg(theta + (size_t)PP * d + PP + p0 + e);
    }
    for (int e = tid; e < jn; e += MB_NT) b2s[e] = __ldcg(theta + (size_t)PP * d + 2 * PP + j0 + e);

    double g[MB_ACC][2];
#pragma unroll
    for (int i = 0; i < MB_ACC; ++i) g[i][0] = g[i][1] = 0.0;
    double gb1 = 0.0, gw2 = 0.0, gb2 = 0.0;
    const int sgm = tid & (MB_SEG - 1), own = tid / MB_SEG;        // node (res pass) / hidden unit (dZ pass) of the thread

#pragma unroll 1
    for (int t = 0; t < ntile; ++t) {
        cp_async_wait<0>();
        __syncthreads();                      // tile t has landed; everybody is done with tile t - 1, H and R
        if (t + 1 < ntile) load_tile(t + 1);
        const double* Xt = sm + MbSmem::X + (t & 1) * MB_TR * DM_LD;
        // ---- Z = W1 X_t^T, H = sigmoid(Z + b1): warp = m-tile, both n-tiles
        if (warp < MT) {
            const double* ap = W1s + (8 * warp + qr) * DM_LD + qc;
            const double* bp = Xt + qr * DM_LD + qc;
            double z[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 4
            for (int ks = 0; ks < KT; ++ks) {
                const double a = ap[4 * ks];
                dmma(z[0], z[1], a, bp[4 * ks]);
                dmma(z[2], z[3], a, bp[8 * DM_LD + 4 * ks]);
            }
            const int p = 8 * warp + qr;
            if (p < PR) {
                const double bb = b1s[p];
                double* hp = Hs + p * MB_LDH + 2 * qc;
                *reinterpret_cast<double2*>(hp) = make_double2(mb_sigmoid(z[0] + bb), mb_sigmoid(z[1] + bb));
                *reinterpret_cast<double2*>(hp + 8) = make_double2(mb_sigmoid(z[2] + bb), mb_sigmoid(z[3] + bb));
            }
        }
        __syncthreads();
        // ---- out, res (0 past the last row), S, gb2: four threads per node, every fourth row each
        if (own < jn) {
            const int jl = own;
#pragma unroll
            for (int s = sgm; s < MB_TR; s += MB_SEG) {
                double o = b2s[jl];
                for (int k = 0; k < m1; ++k) o = fma(Hs[(jl * m1 + k) * MB_LDH + s], W2s[jl * m1 + k], o);
                const double r = (t * MB_TR + s < n) ? o - Xt[s * DM_LD + j0 + jl] : 0.0;
                Rs[jl * MB_TR + s] = r;
                sq = fma(r, r, sq);
                gb2 += r;
            }
        }
        __syncthreads();
        // ---- dZ over H, gb1, gW2: four threads per hidden unit
        if (own < PR) {
            const int p = own, jl = p / m1;
            const double w2 = W2s[p];
            double* hrow = Hs + p * MB_LDH;
            const double* rrow = Rs + jl * MB_TR;
#pragma unroll
            for (int s = sgm; s < MB_TR; s += MB_SEG) {
                const double hh = hrow[s], r = rrow[s];
                const double dz = r * w2 * hh * (1.0 - hh);
                hrow[s] = dz;
                gw2 = fma(r, hh, gw2);
                gb1 += dz;
            }
        }
        __syncthreads();
        // ---- gW1 += dZ X_t (K = the tile's rows): warp w owns the accumulator tiles w, w + 8, ...
#pragma unroll
        for (int i = 0; i < MB_ACC; ++i) {
            const int q = warp + 8 * i;
            if (q < MT * NT) {
                const int mt = q / NT, nt = q - mt * NT;
                const double* ap = Hs + (8 * mt + qr) * MB_LDH + qc;
                const double* bp = Xt + qc * DM_LD + 8 * nt + qr;
#pragma unroll
                for (int ks = 0; ks < MB_TR / 4; ++ks) dmma(g[i][0], g[i][1], ap[4 * ks], bp[4 * ks * DM_LD]);
            }
        }
    }
    // ---- the slice's sums -> grad: gW1 from the accumulators, the segment sums in a fixed order
#pragma unroll
    for (int i = 0; i < MB_ACC; ++i) {
        const int q = warp + 8 * i;
        if (q < MT * NT) {
            const int mt = q / NT, nt = q - mt * NT, p = 8 * mt + qr, c = 8 * nt + 2 * qc;
            if (p < PR) {
                if (c < d) grad[(size_t)(p0 + p) * d + c] = g[i][0];
                if (c + 1 < d) grad[(size_t)(p0 + p) * d + c + 1] = g[i][1];
            }
        }
    }
    __syncthreads();                          // R is free
    double* seg = Rs;                         // [3][40][MB_SEG]: gb1, gW2, gb2
    if (own < PR) {
        seg[own * MB_SEG + sgm] = gb1;
        seg[(MB_PR + own) * MB_SEG + sgm] = gw2;
    }
    if (own < jn) seg[(2 * MB_PR + own) * MB_SEG + sgm] = gb2;
    __syncthreads();
    if (tid < PR) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int q = 0; q < MB_SEG; ++q) {
            a += seg[tid * MB_SEG + q];
            b += seg[(MB_PR + tid) * MB_SEG + q];
        }
        grad[(size_t)PP * d + p0 + tid] = a;
        grad[(size_t)PP * d + PP + p0 + tid] = b;
    }
    if (tid < jn) {
        double a = 0.0;
#pragma unroll
        for (int q = 0; q < MB_SEG; ++q) a += seg[(2 * MB_PR + tid) * MB_SEG + q];
        grad[(size_t)PP * d + 2 * PP + j0 + tid] = a;
    }
    __syncthreads();                          // the next slice overwrites the slice buffers
}

__global__ void __launch_bounds__(MB_NT, 2) mlp_batch_kernel(const MbArgs P) {
    extern __shared__ __align__(16) double sm[];
    __shared__ unsigned s_prob;
    const int tid = threadIdx.x;
    const DmmaPos ps(tid);
    const int d = P.d, m1 = P.m1, PP = d * m1, W = PP * d + 2 * PP + d, nW1 = PP * d;
    const int JN = MB_PR / m1 < d ? MB_PR / m1 : d;

    SweepSync sy{smem_u32(sm + DmmaSmem::mbar), 0u};
    if (tid == 0) mbar_init(sy.bar, MB_NT / 32);
    // padding columns of the X tiles (never written by the copies) and rows of H past the slice: zero, finite
    for (int e = tid; e < 2 * MB_TR * DM_LD; e += MB_NT) sm[MbSmem::X + e] = 0.0;
    for (int e = tid; e < MB_PR * MB_LDH; e += MB_NT) sm[MbSmem::H + e] = 0.0;
    __syncthreads();

    for (;;) {
        if (tid == 0) s_prob = atomicAdd(P.counter, 1u);
        __syncthreads();
        const unsigned q = s_prob;
        __syncthreads();
        if (q >= (unsigned)P.n_run) break;
        const int b = P.idx ? P.idx[q] : (int)q;
        MlpState* st = P.st + b;
        double* theta = P.theta + (size_t)b * W;
        double* mm = P.m + (size_t)b * W;
        double* vv = P.v + (size_t)b * W;
        double* grad = P.grad + (size_t)b * W;
        const double* xb = P.X + (size_t)b * P.n * d;
        const double mu = st->mu, s = st->s, lambda1 = st->lambda1, lambda2 = st->lambda2;
        const double beta1 = st->beta1, beta2 = st->beta2, gamma = st->lr_gamma;
        double lr = st->lr;
        int step = st->step, halted = st->halted, it = 0;
        double h = st->h, lad = st->logabsdet, l1 = st->l1, S = st->S, score = st->score, obj = st->obj;
        double obj_prev = 1e16;
        const double wd = mu * lambda2, l1c = mu * lambda1;

#pragma unroll 1
        for (int i = 0; i < P.max_iter && !halted; ++i) {
            // ---- h at the pre-step parameters; h < 0: no step (nonlinear.py:215-217)
            h = mb_h(theta, d, m1, s, sm, ps, sy, lad, l1);
            if (h < 0.0) {
                halted = 1;
                break;
            }
            // ---- forward / backward, slice by slice
            double sq = 0.0;
#pragma unroll 1
            for (int j0 = 0; j0 < d; j0 += JN) mb_slice(P, theta, xb, grad, sm, j0, min(JN, d - j0), sq);
            double z1 = 0.0, z2 = 0.0;
            block_sum3<MB_NT>(sq, z1, z2, sm + DmmaSmem::red, tid);
            S = sq;
            score = 0.5 * (double)d * log(S / (double)P.n);
            obj = mu * (score + lambda1 * l1) + h;
            // ---- the Adam step (mi_update of mlp_iter.cu)
            const double bc1 = -expm1((double)(step + 1) * log(beta1)), bc2 = -expm1((double)(step + 1) * log(beta2));
            const double gs = mu * (double)d / S;
            const double step_size = lr / bc1, bc2s = sqrt(bc2);
            const double* Minv = sm + MbSmem::A;
            for (int e = tid; e < W; e += MB_NT) {
                const double p = theta[e], mo = mm[e], vo = vv[e];
                double gr = gs * __ldcg(grad + e);
                if (e < nW1) {
                    const int row = e / d, ii = e - row * d, j = row / m1;
                    const double sg = (p > 0.0) ? 1.0 : ((p < 0.0) ? -1.0 : 0.0);
                    gr = fma(l1c, sg, gr);
                    gr = fma(2.0 * p, Minv[j * DM_LD + ii], gr);
                }
                gr = fma(wd, p, gr);
                const double mn = mo + (gr - mo) * (1.0 - beta1);      // exp_avg.lerp_(grad, 1 - beta1)
                const double vn = fma(vo, beta2, (1.0 - beta2) * gr * gr);
                mm[e] = mn;
                vv[e] = vn;
                const double denom = sqrt(vn) / bc2s + 1e-8;
                theta[e] = p - step_size * (mn / denom);
            }
            __syncthreads();                  // theta is re-read (from L2) by the next iteration
            ++step;
            ++it;
            if (gamma != 1.0 && step % 1000 == 0) lr *= gamma;                  // ExponentialLR (nonlinear.py:224-225)
            if (i % P.checkpoint == 0 || i == P.max_iter - 1) {                 // nonlinear.py:226-231
                if (fabs((obj_prev - obj) / obj_prev) <= P.tol) break;
                obj_prev = obj;
            }
        }
        if (tid == 0) {
            st->lr = lr;
            st->logabsdet = lad;
            st->h = h;
            st->S = S;
            st->l1 = l1;
            st->obj = obj;
            st->score = score;
            st->step = step;
            st->halted = halted;
            P.iters[b] = it;
        }
        __syncthreads();
    }
}

}  // namespace dagma

using namespace dagma;

extern "C" int dagma_mlp_batch_supported(int n, int d, int m1) {
    return (n >= 1 && d >= 1 && d <= DAGMA_SMALL_MAX_D && m1 >= 1 && m1 <= MB_PR) ? 1 : 0;
}

extern "C" int dagma_mlp_minimize_batch_f64(dagma_stream_t stream_, int batch, int n, int d, int m1, int max_iter,
                                            int checkpoint, double tol, const int* idx_dev, int n_idx, void* states_dev,
                                            double* theta_dev, double* m_dev, double* v_dev, const double* x_dev,
                                            double* grad_dev, int* iters_dev, unsigned* work_counter_dev) {
    DAGMA_REQUIRE(batch >= 1, "batch must be positive");
    DAGMA_REQUIRE(dagma_mlp_batch_supported(n, d, m1), "shape not supported (dagma_mlp_batch_supported)");
    DAGMA_REQUIRE(max_iter >= 0 && checkpoint >= 1, "max_iter must be >= 0 and checkpoint >= 1");
    DAGMA_REQUIRE(idx_dev == nullptr || (n_idx >= 0 && n_idx <= batch), "n_idx out of range");
    DAGMA_REQUIRE(states_dev && theta_dev && m_dev && v_dev && x_dev && grad_dev && iters_dev && work_counter_dev,
                  "null device pointer");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int n_run = idx_dev ? n_idx : batch;
    if (n_run == 0) return 0;
    int dev = 0, sms = 0;
    DAGMA_CUDA_OK(cudaGetDevice(&dev));
    DAGMA_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(mlp_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MbSmem::bytes));
    DAGMA_CUDA_OK(cudaFuncSetAttribute(mlp_batch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
    MbArgs A{};
    A.batch = batch; A.n = n; A.d = d; A.m1 = m1; A.max_iter = max_iter; A.checkpoint = checkpoint; A.tol = tol;
    A.idx = idx_dev; A.n_run = n_run;
    A.st = (MlpState*)states_dev;
    A.theta = theta_dev; A.m = m_dev; A.v = v_dev; A.grad = grad_dev; A.X = x_dev;
    A.iters = iters_dev; A.counter = work_counter_dev;
    // two CTAs per SM: __launch_bounds__(256, 2) caps registers at 128, 2 x 106 KB of shared memory fit the carve-out
    long ctas = 2L * sms;
    if (ctas > n_run) ctas = n_run;
    DAGMA_CUDA_OK(cudaMemsetAsync(work_counter_dev, 0, sizeof(unsigned), stream));
    mlp_batch_kernel<<<(int)ctas, MB_NT, MbSmem::bytes, stream>>>(A);
    DAGMA_CUDA_OK(cudaGetLastError());
    return 0;
}
