// Data staging in front of the hot path: in-place column centring of X and
// cov = X^T X / n  (reference: src/dagma/linear.py:410-411, 428), batched.
// Runs once per fit; written as a plain tiled FP64 kernel (32 x 32 output tile per
// CTA, 2 x 2 per thread, X streamed through shared memory in 32-row slabs).
#include "common.cuh"
#include "../../include/dagma_b200.h"

namespace dagma {

__global__ void center_columns_kernel(double* x, int n, int d) {
    // grid: (ceil(d/32), batch); block: 32 x 8
    double* X = x + (size_t)blockIdx.y * n * d;
    const int c = blockIdx.x * 32 + threadIdx.x;
    __shared__ double part[8][33];
    double s = 0.0;
    if (c < d)
        for (int r = threadIdx.y; r < n; r += 8) s += X[(size_t)r * d + c];
    part[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += part[i][threadIdx.x];
    const double mean = tot / (double)n;
    if (c < d)
        for (int r = threadIdx.y; r < n; r += 8) X[(size_t)r * d + c] -= mean;
}

__global__ void __launch_bounds__(256) cov_kernel(const double* __restrict__ x, double* __restrict__ cov,
                                                   int n, int d, int row0, int rows) {
    // grid: (ceil(d/32), ceil(d/32), batch); block 16 x 16; thread -> 2 x 2 outputs.
    // Uses rows [row0, row0 + rows) of X (row sharding for the multi-GPU score path).
    const double* X = x + (size_t)blockIdx.z * n * d;
    double* Cv = cov + (size_t)blockIdx.z * d * d;
    __shared__ double A[32][33], B[32][33];
    const int ti = threadIdx.y, tj = threadIdx.x, tid = ti * 16 + tj;
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    double acc[2][2] = {{0, 0}, {0, 0}};
    for (int r0 = row0; r0 < row0 + rows; r0 += 32) {
        for (int e = tid; e < 32 * 32; e += 256) {
            const int rr = e >> 5, cc = e & 31;
            const int r = r0 + rr;
            const bool ok = r < row0 + rows;
            A[rr][cc] = (ok && i0 + cc < d) ? X[(size_t)r * d + i0 + cc] : 0.0;
            B[rr][cc] = (ok && j0 + cc < d) ? X[(size_t)r * d + j0 + cc] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int rr = 0; rr < 32; ++rr) {
            const double a0 = A[rr][ti], a1 = A[rr][ti + 16], b0 = B[rr][tj], b1 = B[rr][tj + 16];
            acc[0][0] = fma(a0, b0, acc[0][0]);
            acc[0][1] = fma(a0, b1, acc[0][1]);
            acc[1][0] = fma(a1, b0, acc[1][0]);
            acc[1][1] = fma(a1, b1, acc[1][1]);
        }
        __syncthreads();
    }
    const double inv_n = 1.0 / (double)n;
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int w = 0; w < 2; ++w) {
            const int i = i0 + ti + 16 * u, j = j0 + tj + 16 * w;
            if (i < d && j < d) Cv[(size_t)i * d + j] = acc[u][w] * inv_n;
        }
}

}  // namespace dagma

using namespace dagma;

extern "C" int dagma_center_cov_f64(dagma_stream_t stream_, int batch, int n, int d, double* x_dev,
                                    int center, double* cov_dev) {
    DAGMA_REQUIRE(batch >= 1 && n >= 1 && d >= 1, "bad shape");
    DAGMA_REQUIRE(x_dev && cov_dev, "null pointer");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int tiles = (d + 31) / 32;
    // the problems sit on gridDim.y / gridDim.z, which CUDA caps at 65 535: larger batches go in slices
    constexpr int kMaxGridYZ = 65535;
    for (int b0 = 0; b0 < batch; b0 += kMaxGridYZ) {
        const int nb = batch - b0 < kMaxGridYZ ? batch - b0 : kMaxGridYZ;
        double* x = x_dev + (size_t)b0 * n * d;
        if (center) {
            center_columns_kernel<<<dim3(tiles, nb), dim3(32, 8), 0, stream>>>(x, n, d);
            DAGMA_CUDA_OK(cudaGetLastError());
        }
        cov_kernel<<<dim3(tiles, tiles, nb), dim3(16, 16), 0, stream>>>(x, cov_dev + (size_t)b0 * d * d, n, d, 0, n);
        DAGMA_CUDA_OK(cudaGetLastError());
    }
    return 0;
}
