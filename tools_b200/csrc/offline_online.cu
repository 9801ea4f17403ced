// Online half of samp_p from a pool entry (qf_samp_p_online, DESIGN 4.12).
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int TPB = 256;

inline int grid_for(long long work, int per_block, int max_blocks = 148 * 16) {
    long long g = (work + per_block - 1) / per_block;
    if (g < 1) g = 1;
    if (g > max_blocks) g = max_blocks;
    return (int)g;
}

// Row b: out[b][0:M] = x[b][0:M] as fp64, v[b][0:N] = (u[b] + a[b]) mod q.  u and a are residues in [0, q), q < 2^62, so
// the sum needs one conditional subtraction.
__global__ void pool_expand_kernel(const int32_t* __restrict__ x, long ldx, double* __restrict__ out, long ldo, int M,
                                   const int64_t* __restrict__ u, long ldu, const int64_t* __restrict__ a, long lda,
                                   int64_t* __restrict__ v, long ldv, int N, int B, unsigned long long q) {
    const long W = (long)M + N, total = (long)B * W;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / W;
        const int j = (int)(i - b * W);
        if (j < M) {
            out[b * ldo + j] = (double)x[b * ldx + j];
        } else {
            const int c = j - M;
            unsigned long long s = (unsigned long long)u[b * ldu + c] + (unsigned long long)a[b * lda + c];
            if (s >= q) s -= q;
            v[b * ldv + c] = (int64_t)s;
        }
    }
}

// T[b][n] -= dv * (scale[n] * mul) for the contraction value dv of row b, column n, given as X = -dv * mul (the store-only
// epilogue with a unit scale vector: a power-of-two scaling of dv, exact).  X / mul = -dv exactly, and the fma is the one
// the update epilogues of gemm_i8.cu contract to, so T ends as if the contraction had accumulated onto it.
__global__ void pool_centre_kernel(const double* __restrict__ X, long ldx, double* __restrict__ T, long ldt,
                                   const double* __restrict__ scale, double mul, int N, int B) {
    const long total = (long)B * N;
    const double inv = 1.0 / mul;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / N;
        const int n = (int)(i - b * N);
        double* t = T + b * ldt + n;
        *t = fma(X[b * ldx + n] * inv, scale[n] * mul, *t);
    }
}

}  // namespace

cudaError_t qf_launch_pool_expand(const int32_t* x, long ldx, double* out, long ldo, int M, const int64_t* u, long ldu,
                                  const int64_t* a, long lda, int64_t* v, long ldv, int N, int B, unsigned long long q,
                                  cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    pool_expand_kernel<<<grid_for((long long)B * (M + N), TPB), TPB, 0, stream>>>(x, ldx, out, ldo, M, u, ldu, a, lda, v, ldv,
                                                                                  N, B, q);
    return cudaGetLastError();
}

cudaError_t qf_launch_pool_centre(const double* X, long ldx, double* T, long ldt, const double* scale, double mul, int N, int B,
                                  cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    pool_centre_kernel<<<grid_for((long long)B * N, TPB), TPB, 0, stream>>>(X, ldx, T, ldt, scale, mul, N, B);
    return cudaGetLastError();
}
