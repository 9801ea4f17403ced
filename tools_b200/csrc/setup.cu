// One-off key-setup kernels for the nearest-plane engine (per key, not per target):
// from the short basis S (columns b_j) and its GSO S~ (columns b~_i) derive
//   d_i   = ||b~_i||^2
//   Mt    = rows b~_i / d_i                 (centre -> GSO coordinates)
//   St    = S^t                              (rows b_j)
//   U     = Mt * S  (mu-coefficients, upper unitriangular)   -- via gemm_f64
// which turn GPV08 SampleD (MatZ::sample_d_precomputed_gso, gpv.rs:160) into
// "one GEMM + triangular back-substitution with randomized rounding".
#include "common.cuh"
#include "kernels.h"

namespace {

__global__ void colnorm2_kernel(const double* __restrict__ G, long ld, int rows, int cols, double* __restrict__ d) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    double acc = 0;
    for (int r = 0; r < rows; ++r) {
        double v = G[(long)r * ld + c];
        acc += v * v;
    }
    d[c] = acc;
}

// out[c][r] = in[r][c] * (scale ? 1/scale[c] : 1)
__global__ void transpose_scale_kernel(const double* __restrict__ in, long ldin, double* __restrict__ out, long ldout,
                                       int rows, int cols, const double* __restrict__ scale) {
    __shared__ double tile[32][33];
    int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int r = r0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < rows && c < cols) ? in[(long)r * ldin + c] : 0.0;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int c = c0 + i, r = r0 + threadIdx.x;
        if (c < cols && r < rows) {
            double v = tile[threadIdx.x][i];
            if (scale) v /= scale[c];
            out[(long)c * ldout + r] = v;
        }
    }
}

__global__ void gather_cols_kernel(const double* __restrict__ in, long ldin, const int* __restrict__ cols, int ncols,
                                   double* __restrict__ out, long ldout, int rows) {
    long total = (long)rows * ncols;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long r = i / ncols;
        int j = (int)(i - r * ncols);
        out[r * ldout + j] = in[r * ldin + cols[j]];
    }
}

__global__ void make_dg_kernel(const double* __restrict__ d, int count, double s, DGaussParams* __restrict__ dg) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dg[i] = make_dgauss(s / sqrt(d[i]));
}

}  // namespace

cudaError_t qf_launch_colnorm2(const double* G, long ld, int rows, int cols, double* d, cudaStream_t stream) {
    colnorm2_kernel<<<(cols + 127) / 128, 128, 0, stream>>>(G, ld, rows, cols, d);
    return cudaGetLastError();
}
cudaError_t qf_launch_transpose_scale(const double* in, long ldin, double* out, long ldout, int rows, int cols,
                                      const double* scale, cudaStream_t stream) {
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
    transpose_scale_kernel<<<grid, block, 0, stream>>>(in, ldin, out, ldout, rows, cols, scale);
    return cudaGetLastError();
}
cudaError_t qf_launch_gather_cols(const double* in, long ldin, const int* cols, int ncols, double* out, long ldout,
                                  int rows, cudaStream_t stream) {
    long long total = (long long)rows * ncols;
    long long g = (total + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    gather_cols_kernel<<<(int)g, 256, 0, stream>>>(in, ldin, cols, ncols, out, ldout, rows);
    return cudaGetLastError();
}
cudaError_t qf_launch_make_dg(const double* d, int count, double s, DGaussParams* dg, cudaStream_t stream) {
    make_dg_kernel<<<(count + 127) / 128, 128, 0, stream>>>(d, count, s, dg);
    return cudaGetLastError();
}

// ---- fixed-point digit planes of the mu-coefficients for the tensor-core nearest-plane updates ----
// The big off-diagonal updates use the entries U[i][j] with row i above the `blk`-column block of j (i < (j / blk) blk).
// They are scaled per row and per `sblk`-column block c (sblk a multiple of blk: one launch may contract several
// adjacent blk-blocks and applies one scale per row): U[i][j] * 2^e(i,c) rounded to an integer of L balanced base-256
// digits, scale[c*D + i] = 2^-e(i,c).  Entries at or below their block keep zero digits.  The last block of either kind may be
// wider than its step (a thin ragged top joins the block below it): it starts at fs_last / ss_last.
namespace {

__global__ void ozaki_scale_kernel(const double* __restrict__ U, long ld, int D, int blk, int sblk, int fs_last, int ss_last,
                                   int L, double* __restrict__ scale, int split) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int nblk = ss_last / sblk + 1;
    const long total = (long)D * nblk;
    for (long w = (long)blockIdx.x * wpb + (threadIdx.x >> 5); w < total; w += (long)gridDim.x * wpb) {
        const int c = (int)(w / D), i = (int)(w - (long)c * D);
        double mx = 0.0;
        int j1 = (c == nblk - 1) ? D : (c + 1) * sblk;
        if (i < split) j1 = min(j1, split);  // two-phase recursion: rows below the split never meet columns above it
        // first column whose blk-block starts above row i (none if row i lies in the last block)
        const int j0 = i >= fs_last ? D : max(c * sblk, (i / blk + 1) * blk);
        for (int j = j0 + lane; j < j1; j += 32) mx = fmax(mx, fabs(U[(long)i * ld + j]));
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) {
            // |U| 2^e < 2^(8L-2)  (capacity of L balanced digits is ~0.498 * 256^L)
            int e = (mx > 0.0) ? (8 * L - 2) - (ilogb(mx) + 1) : 0;
            scale[(long)c * D + i] = ldexp(1.0, -e);
        }
    }
}

__global__ void ozaki_digits_kernel(const double* __restrict__ U, long ld, int D, int blk, int sblk, int fs_last, int ss_last,
                                    int L, const double* __restrict__ scale, int8_t* __restrict__ planes, long plane_stride,
                                    long ldk, int split) {
    const long total = (long)D * D;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int i = (int)(t / D), j = (int)(t - (long)i * D);
        const int c = min(j, ss_last) / sblk;
        long long v = 0;
        if (i < min((j / blk) * blk, fs_last) && !(i < split && j >= split))
            v = __double2ll_rn(U[(long)i * ld + j] / scale[(long)c * D + i]);
        for (int l = 0; l < L; ++l) {
            long long lo = ((v + 128) & 255) - 128;
            if (l == L - 1) lo = v;
            planes[l * plane_stride + (long)i * ldk + j] = (int8_t)lo;
            v = (v - lo) >> 8;
        }
    }
}

}  // namespace

cudaError_t qf_launch_ozaki_prepare(const double* U, long ld, int D, int blk, int sblk, int fs_last, int ss_last, int L,
                                    double* scale, int8_t* planes, long plane_stride, long ldk, cudaStream_t stream, int split) {
    if (blk <= 0 || sblk % blk != 0 || fs_last % blk != 0 || ss_last % sblk != 0) return cudaErrorInvalidValue;
    const int nblk = ss_last / sblk + 1;
    long long warps = (long long)D * nblk;
    long long g = (warps + 7) / 8;
    if (g > 148 * 32) g = 148 * 32;
    ozaki_scale_kernel<<<(int)g, 256, 0, stream>>>(U, ld, D, blk, sblk, fs_last, ss_last, L, scale, split);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ozaki_digits_kernel<<<148 * 16, 256, 0, stream>>>(U, ld, D, blk, sblk, fs_last, ss_last, L, scale, planes, plane_stride, ldk,
                                                      split);
    return cudaGetLastError();
}

namespace {
__global__ void gadget_to_gso_kernel(const double* __restrict__ U, long ldu, int nk, int k, int rev,
                                     const double* __restrict__ skinv, double* __restrict__ out, long ldo) {
    const long total = (long)nk * nk;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / nk), c = (int)(idx - (long)i * nk);
        const int bc = c / k, t = c - bc * k;
        double acc = 0.0;
        for (int tp = 0; tp < k; ++tp) {
            const int cc = bc * k + tp, col = rev ? nk - 1 - cc : cc;
            if (col < i) continue;  // U is upper unitriangular (the computed lower part is rounding noise)
            const double u = col == i ? 1.0 : U[(long)i * ldu + col];
            acc = fma(u, skinv[tp * k + t], acc);
        }
        out[(long)i * ldo + c] = acc;
    }
}
}  // namespace
cudaError_t qf_launch_gadget_to_gso(const double* U, long ldu, int nk, int k, int rev, const double* skinv, double* out,
                                    long ldo, cudaStream_t stream) {
    gadget_to_gso_kernel<<<148 * 16, 256, 0, stream>>>(U, ldu, nk, k, rev, skinv, out, ldo);
    return cudaGetLastError();
}

// ---- blocked Cholesky (per key): compute_sqrt_sigma_2, mp_perturbation.rs:111-139 --------------------
// One diagonal block (nb <= 64) in shared memory: A_jj = L L^t in place (strict upper part zeroed) and
// Linv = L^-1 (row-major nb x 64, lower triangular) for the panel solve  L_ij = A_ij L_jj^-t  as a GEMM.
namespace {

constexpr int POTRF_NB = 64;

__global__ void __launch_bounds__(256, 1)
potrf_diag_kernel(double* A, long ld, int nb, double* Linv, int* info) {
    __shared__ double L[POTRF_NB][POTRF_NB + 1];
    __shared__ int bad;
    const int tid = threadIdx.x;
    if (tid == 0) bad = 0;
    for (int t = tid; t < POTRF_NB * POTRF_NB; t += blockDim.x) {
        const int i = t / POTRF_NB, j = t % POTRF_NB;
        L[i][j] = (i < nb && j <= i) ? A[(long)i * ld + j] : 0.0;
        Linv[i * POTRF_NB + j] = 0.0;
    }
    __syncthreads();
    for (int j = 0; j < nb; ++j) {
        if (tid == 0) {
            const double d = L[j][j];
            if (!(d > 0.0)) { bad = 1; L[j][j] = 1.0; } else L[j][j] = sqrt(d);
        }
        __syncthreads();
        const double inv = 1.0 / L[j][j];
        for (int i = j + 1 + tid; i < nb; i += blockDim.x) L[i][j] *= inv;
        __syncthreads();
        // trailing update of the lower triangle: L[i][k] -= L[i][j] L[k][j],  j < k <= i
        const int r = nb - j - 1;
        for (int t = tid; t < r * r; t += blockDim.x) {
            const int i = j + 1 + t / r, k = j + 1 + t % r;
            if (k <= i) L[i][k] -= L[i][j] * L[k][j];
        }
        __syncthreads();
    }
    // Linv = L^-1 by forward substitution, one column per thread (a thread only re-reads its own writes)
    if (tid < nb) {
        const int c = tid;
        Linv[c * POTRF_NB + c] = 1.0 / L[c][c];
        for (int i = c + 1; i < nb; ++i) {
            double acc = 0.0;
            for (int k = c; k < i; ++k) acc += L[i][k] * Linv[k * POTRF_NB + c];
            Linv[i * POTRF_NB + c] = -acc / L[i][i];
        }
    }
    for (int t = tid; t < POTRF_NB * POTRF_NB; t += blockDim.x) {
        const int i = t / POTRF_NB, j = t % POTRF_NB;
        if (i < nb && j < nb) A[(long)i * ld + j] = (j <= i) ? L[i][j] : 0.0;
    }
    if (tid == 0 && bad) atomicOr(info, 1);
}

// out[i][j] = in[i][j] for a rows x cols block (strided copy)
__global__ void copy_block_kernel(const double* __restrict__ in, long ldin, double* __restrict__ out, long ldout, long rows,
                                  int cols) {
    const long total = rows * cols;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long i = t / cols;
        const int j = (int)(t - i * cols);
        out[i * ldout + j] = in[i * ldin + j];
    }
}

// C (n x n, holds G = R R^t on entry for the top-left mb x mb block when full == 0):
//   full == 0:  C[i][j] = coef * (diag * [i==j] - gcoef * C[i][j])                      (Schur complement, n = m_bar)
//   full == 1:  C = coef * (Sigma - gcoef * [[G, R],[R^t, I]] - I) on n = m_bar + nk, G read from Gin (m_bar x m_bar),
//               Sigma == nullptr means diag * I                                         (mp_perturbation.rs:125-135)
__global__ void sigma2_assemble_kernel(double* __restrict__ C, long ldc, long n, int full, const double* __restrict__ Gin,
                                       long ldg, const double* __restrict__ R, long ldr, long mb, const double* __restrict__ Sigma,
                                       long lds, double diag, double gcoef, double coef) {
    const long total = n * n;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long i = t / n, j = t - i * n;
        double v;
        if (!full) {
            v = coef * ((i == j ? diag : 0.0) - gcoef * C[i * ldc + j]);
        } else {
            double tt;
            if (i < mb && j < mb) tt = Gin[i * ldg + j];
            else if (i < mb) tt = R[i * ldr + (j - mb)];
            else if (j < mb) tt = R[j * ldr + (i - mb)];
            else tt = (i == j) ? 1.0 : 0.0;
            const double sg = Sigma ? Sigma[i * lds + j] : (i == j ? diag : 0.0);
            v = coef * (sg - gcoef * tt - (i == j ? 1.0 : 0.0));
        }
        C[i * ldc + j] = v;
    }
}

// zero the strict upper triangle of an n x n matrix
__global__ void tril_kernel(double* __restrict__ A, long ld, long n) {
    const long total = n * n;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long i = t / n, j = t - i * n;
        if (j > i) A[i * ld + j] = 0.0;
    }
}

}  // namespace

cudaError_t qf_launch_tril(double* A, long ld, long n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    tril_kernel<<<148 * 8, 256, 0, stream>>>(A, ld, n);
    return cudaGetLastError();
}
cudaError_t qf_launch_potrf_diag(double* A, long ld, int nb, double* Linv, int* info, cudaStream_t stream) {
    if (nb < 1 || nb > POTRF_NB) return cudaErrorInvalidValue;
    potrf_diag_kernel<<<1, 256, 0, stream>>>(A, ld, nb, Linv, info);
    return cudaGetLastError();
}
cudaError_t qf_launch_copy_block(const double* in, long ldin, double* out, long ldout, long rows, int cols, cudaStream_t stream) {
    if (rows <= 0 || cols <= 0) return cudaSuccess;
    long long g = ((long long)rows * cols + 255) / 256;
    if (g > 148 * 8) g = 148 * 8;
    copy_block_kernel<<<(int)g, 256, 0, stream>>>(in, ldin, out, ldout, rows, cols);
    return cudaGetLastError();
}
cudaError_t qf_launch_sigma2_assemble(double* C, long ldc, long n, int full, const double* Gin, long ldg, const double* R,
                                      long ldr, long mb, const double* Sigma, long lds, double diag, double gcoef, double coef,
                                      cudaStream_t stream) {
    sigma2_assemble_kernel<<<148 * 8, 256, 0, stream>>>(C, ldc, n, full, Gin, ldg, R, ldr, mb, Sigma, lds, diag, gcoef, coef);
    return cudaGetLastError();
}

// ---- fixed-point digit planes of a dense real key matrix, one scale per row -------------------------
// (sqrt(Sigma_2) or its Schur factor for the perturbation contraction x_2 = L g on the tensor cores)
// planes[l][i][j] = digit l of rint(L[i][j] * 2^e_i), 2^e_i chosen so that the row fits Ldig balanced digits;
// scale[i] = mult * 2^-e_i  (the tensor-core epilogue computes out -= V * scale; mult carries the sign and the
// fixed-point scale of the other operand).
namespace {

__global__ void scale_vec_kernel(double* __restrict__ v, int n, double mult) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] *= mult;
}

__global__ void fixed_rows_scale_kernel(const double* __restrict__ L, long ld, int rows, int cols, int Ldig,
                                        double* __restrict__ scale) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (long i = (long)blockIdx.x * wpb + (threadIdx.x >> 5); i < rows; i += (long)gridDim.x * wpb) {
        double mx = 0.0;
        for (int j = lane; j < cols; j += 32) mx = fmax(mx, fabs(L[i * ld + j]));
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) {
            const int e = (mx > 0.0) ? (8 * Ldig - 2) - (ilogb(mx) + 1) : 0;
            scale[i] = ldexp(1.0, -e);
        }
    }
}

__global__ void fixed_rows_digits_kernel(const double* __restrict__ L, long ld, int rows, int cols, int Ldig,
                                         const double* __restrict__ scale, int8_t* __restrict__ planes, long plane_stride,
                                         long ldk) {
    const long total = (long)rows * cols;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long i = t / cols;
        const int j = (int)(t - i * cols);
        long long v = __double2ll_rn(L[i * ld + j] / scale[i]);
        for (int l = 0; l < Ldig; ++l) {
            long long lo = ((v + 128) & 255) - 128;
            if (l == Ldig - 1) lo = v;
            planes[l * plane_stride + i * ldk + j] = (int8_t)lo;
            v = (v - lo) >> 8;
        }
    }
}

}  // namespace

cudaError_t qf_launch_fixed_rows_prepare(const double* L, long ld, int rows, int cols, int Ldig, double mult, double* scale,
                                         int8_t* planes, long plane_stride, long ldk, cudaStream_t stream) {
    int g = (rows + 7) / 8;
    if (g > 148 * 32) g = 148 * 32;
    fixed_rows_scale_kernel<<<g, 256, 0, stream>>>(L, ld, rows, cols, Ldig, scale);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    fixed_rows_digits_kernel<<<148 * 16, 256, 0, stream>>>(L, ld, rows, cols, Ldig, scale, planes, plane_stride, ldk);
    scale_vec_kernel<<<(rows + 255) / 256, 256, 0, stream>>>(scale, rows, mult);
    return cudaGetLastError();
}

// ---- GSO building blocks (MatQ::gso, gpv.rs:91) ------------------------------------------------------------
namespace {
// rdiag[i] = (first ? 1 : rdiag[i]) * L[i][i] for the nb diagonal entries of a 64-wide Cholesky block
__global__ void gso_rdiag_kernel(double* __restrict__ rdiag, const double* __restrict__ L, long ldl, int nb, int first) {
    const int i = threadIdx.x;
    if (i < nb) rdiag[i] = (first ? 1.0 : rdiag[i]) * L[(long)i * ldl + i];
}
// out[t][j] = in[t][j] * colscale[j]
__global__ void scale_cols_kernel(const double* __restrict__ in, long ldin, double* __restrict__ out, long ldout, long rows,
                                  long cols, const double* __restrict__ colscale) {
    const long total = rows * cols;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long i = t / cols, j = t - i * cols;
        out[i * ldout + j] = in[i * ldin + j] * colscale[j];
    }
}
}  // namespace

cudaError_t qf_launch_gso_rdiag(double* rdiag, const double* L, long ldl, int nb, int first, cudaStream_t stream) {
    gso_rdiag_kernel<<<1, 64, 0, stream>>>(rdiag, L, ldl, nb, first);
    return cudaGetLastError();
}
cudaError_t qf_launch_scale_cols(const double* in, long ldin, double* out, long ldout, long rows, long cols,
                                 const double* colscale, cudaStream_t stream) {
    if (rows <= 0 || cols <= 0) return cudaSuccess;
    scale_cols_kernel<<<148 * 8, 256, 0, stream>>>(in, ldin, out, ldout, rows, cols, colscale);
    return cudaGetLastError();
}

// ---- ring short basis (short_basis_ring.rs:64-166): the polynomial arithmetic of gen_short_basis_for_trapdoor_ring ----
// P[c][h] = sum_j x^h_j * w_cj mod (X^n + 1)  (c = 0, 1: the digit polynomials of -a_c; h = 0: x = e, h = 1: x = r) and
// Q[c'][h] = sum_j S_k[j][c'] x^h_j  (c' < k).  One CTA per output polynomial, one thread per coefficient.
namespace {
__global__ void ring_basis_polys_kernel(const int32_t* __restrict__ e, const int32_t* __restrict__ r,
                                        const int32_t* __restrict__ w, const int64_t* __restrict__ sk, int n, int k,
                                        int64_t* __restrict__ P, int64_t* __restrict__ Q) {
    const int o = blockIdx.x;  // 0..3: P[c][h]; 4..: Q[c'][h]
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        long long acc = 0;
        if (o < 4) {
            const int c = o >> 1, h = o & 1;
            const int32_t* x = h ? r : e;
            for (int j = 0; j < k; ++j) {
                const int32_t* xj = x + (long)j * n;
                const int32_t* wj = w + ((long)c * k + j) * n;
                for (int i = 0; i < n; ++i) {  // coefficient t of x_j * w_cj: x_j[i] w_cj[t - i], sign flips on wrap-around
                    const int d = t - i;
                    acc += d >= 0 ? (long long)xj[i] * wj[d] : -(long long)xj[i] * wj[d + n];
                }
            }
            P[(long)o * n + t] = acc;
        } else {
            const int cc = (o - 4) >> 1, h = (o - 4) & 1;
            const int32_t* x = h ? r : e;
            for (int j = 0; j < k; ++j) acc += sk[(long)j * k + cc] * (long long)x[(long)j * n + t];
            Q[(long)(o - 4) * n + t] = acc;
        }
    }
}
}  // namespace

cudaError_t qf_launch_ring_basis_polys(const int32_t* e, const int32_t* r, const int32_t* w, const int64_t* sk, int n, int k,
                                       int64_t* P, int64_t* Q, cudaStream_t stream) {
    ring_basis_polys_kernel<<<4 + 2 * k, 256, 0, stream>>>(e, r, w, sk, n, k, P, Q);
    return cudaGetLastError();
}

// ---- tag inverse (short_basis_classical.rs:106, MatZq::inverse): Gauss-Jordan over Z_q on M = [H | I] (n x 2n residues,
// row-major, q < 2^62, 128-bit products).  Column c takes as pivot the first row r >= c whose entry is a unit mod q -- the
// rule of the host restatement gadget._inverse_mod, so both fail on the same tags.  On success the right half of M is H^-1 and *fail = 0;
// without a unit pivot *fail = c + 1 and M is left part-reduced.  One CTA per matrix (blockIdx.x selects one of `count`
// matrices M_t = M + t n 2n with its own f and fail slot): n pivot steps separated by block barriers; per step the factors
// of column c are saved in f (n words) before the rows are updated.
namespace {
__device__ __forceinline__ uint64_t gcd_dev(uint64_t a, uint64_t b) {
    while (b) { const uint64_t t = a % b; a = b; b = t; }
    return a;
}
// a^-1 mod q for gcd(a, q) = 1 (extended Euclid; the coefficients stay below q < 2^62 in magnitude)
__device__ __forceinline__ uint64_t inv_mod_dev(uint64_t a, uint64_t q) {
    long long t = 0, nt = 1;
    uint64_t r = q, nr = a % q;
    while (nr) {
        const uint64_t qu = r / nr;
        const long long tt = t - (long long)qu * nt; t = nt; nt = tt;
        const uint64_t rr = r - qu * nr; r = nr; nr = rr;
    }
    return t < 0 ? (uint64_t)(t + (long long)q) : (uint64_t)t;
}

__global__ void __launch_bounds__(1024) mat_inverse_mod_kernel(uint64_t* __restrict__ M, uint64_t* __restrict__ f, int n,
                                                               uint64_t q, int* __restrict__ fail) {
    __shared__ int piv;
    __shared__ uint64_t inv;
    const long w = 2L * n;
    M += (long)blockIdx.x * n * w;
    f += (long)blockIdx.x * n;
    fail += blockIdx.x;
    const int tid = threadIdx.x, nth = blockDim.x;
    for (int c = 0; c < n; ++c) {
        if (tid == 0) piv = n;
        __syncthreads();
        for (int r = c + tid; r < n; r += nth)
            if (gcd_dev(M[(long)r * w + c], q) == 1) atomicMin(&piv, r);
        __syncthreads();
        const int p = piv;
        if (p == n) {
            if (tid == 0) *fail = c + 1;
            return;
        }
        if (tid == 0) inv = inv_mod_dev(M[(long)p * w + c], q);
        if (p != c)
            for (long j = c + tid; j < w; j += nth) {
                const uint64_t t = M[(long)p * w + j];
                M[(long)p * w + j] = M[(long)c * w + j];
                M[(long)c * w + j] = t;
            }
        __syncthreads();
        for (long j = c + tid; j < w; j += nth) M[(long)c * w + j] = mulmod_u64(M[(long)c * w + j], inv, q);
        for (int r = tid; r < n; r += nth) f[r] = r == c ? 0 : M[(long)r * w + c];
        __syncthreads();
        // rows r != c: M[r][j] -= f[r] M[c][j] for j >= c (columns left of c are already zero in row c)
        const long cols = w - c, total = (long)n * cols;
        for (long t = tid; t < total; t += nth) {
            const int r = (int)(t / cols);
            const uint64_t fr = f[r];
            if (!fr) continue;
            const long j = c + (t - (long)r * cols);
            const uint64_t sub = mulmod_u64(fr, M[(long)c * w + j], q);
            const uint64_t v = M[(long)r * w + j];
            M[(long)r * w + j] = v >= sub ? v - sub : v + (q - sub);
        }
        __syncthreads();
    }
    if (tid == 0) *fail = 0;
}
}  // namespace

cudaError_t qf_launch_mat_inverse_mod(uint64_t* M, uint64_t* f, int n, unsigned long long q, int* fail, cudaStream_t stream) {
    if (n < 1 || q < 2 || q >= (1ull << 62)) return cudaErrorInvalidValue;
    return qf_launch_mat_inverse_mod_batched(M, f, n, q, fail, 1, stream);
}

cudaError_t qf_launch_mat_inverse_mod_batched(uint64_t* M, uint64_t* f, int n, unsigned long long q, int* fail, int count,
                                              cudaStream_t stream) {
    if (n < 1 || q < 2 || q >= (1ull << 62) || count < 1) return cudaErrorInvalidValue;
    mat_inverse_mod_kernel<<<count, 1024, 0, stream>>>(M, f, n, (uint64_t)q, fail);
    return cudaGetLastError();
}

// ---- tag table (qf_set_tag_table): [H_t | I] from caller tags, and H_t^-1 column-major per tag for the per-target kernel
namespace {
__global__ void tag_build_kernel(const int64_t* __restrict__ tags, int count, int n, uint64_t q, uint64_t* __restrict__ M) {
    const long nn = (long)n * n, total = (long)count * n * 2 * n;
    for (long x = blockIdx.x * (long)blockDim.x + threadIdx.x; x < total; x += (long)gridDim.x * blockDim.x) {
        const long t = x / (2 * nn), rem = x - t * 2 * nn, i = rem / (2 * n), j = rem - i * 2 * n;
        uint64_t v;
        if (j < n) {
            const long long h = tags[t * nn + i * n + j] % (long long)q;
            v = (uint64_t)(h < 0 ? h + (long long)q : h);
        } else {
            v = (j - n == i) ? 1 : 0;
        }
        M[x] = v;
    }
}

// tab[t][j][i] = (H_t^-1)[i][j] = M_t[i][n + j] (32- or 64-bit words): thread i of the per-target kernel reads row i
template <typename W>
__global__ void tag_pack_kernel(const uint64_t* __restrict__ M, int count, int n, W* __restrict__ tab) {
    const long nn = (long)n * n, total = (long)count * nn;
    for (long x = blockIdx.x * (long)blockDim.x + threadIdx.x; x < total; x += (long)gridDim.x * blockDim.x) {
        const long t = x / nn, rem = x - t * nn, j = rem / n, i = rem - j * n;
        tab[x] = (W)M[t * 2 * nn + i * 2 * n + n + j];
    }
}
inline int tag_grid(long long work) { return (int)std::min<long long>((work + 255) / 256, 148LL * 16); }

// f_a tag table (qf_set_f_a_tags): tab[t][j][i] = (tags[t][i][j] - H_0[i][j]) mod q
template <typename W>
__global__ void tag_diff_pack_kernel(const int64_t* __restrict__ tags, int count, int n, uint64_t q, const uint64_t* __restrict__ h0,
                                     W* __restrict__ tab) {
    const long nn = (long)n * n, total = (long)count * nn;
    for (long x = blockIdx.x * (long)blockDim.x + threadIdx.x; x < total; x += (long)gridDim.x * blockDim.x) {
        const long t = x / nn, rem = x - t * nn, j = rem / n, i = rem - j * n;
        const long long h = tags[t * nn + i * n + j] % (long long)q;
        const uint64_t v = (uint64_t)(h < 0 ? h + (long long)q : h), z = h0 ? h0[i * n + j] : (i == j ? 1 : 0);
        tab[x] = (W)(v >= z ? v - z : v + (q - z));
    }
}
}  // namespace

cudaError_t qf_launch_tag_diff_pack(const int64_t* tags, int count, int n, unsigned long long q, const uint64_t* h0,
                                    int word_bytes, void* tab, cudaStream_t stream) {
    if (n < 1 || count < 1 || q < 2 || (word_bytes != 4 && word_bytes != 8)) return cudaErrorInvalidValue;
    const int grid = tag_grid((long long)count * n * n);
    if (word_bytes == 4) tag_diff_pack_kernel<uint32_t><<<grid, 256, 0, stream>>>(tags, count, n, (uint64_t)q, h0, (uint32_t*)tab);
    else tag_diff_pack_kernel<uint64_t><<<grid, 256, 0, stream>>>(tags, count, n, (uint64_t)q, h0, (uint64_t*)tab);
    return cudaGetLastError();
}

cudaError_t qf_launch_tag_build(const int64_t* tags, int count, int n, unsigned long long q, uint64_t* M, cudaStream_t stream) {
    if (n < 1 || count < 1 || q < 2) return cudaErrorInvalidValue;
    tag_build_kernel<<<tag_grid((long long)count * n * 2 * n), 256, 0, stream>>>(tags, count, n, (uint64_t)q, M);
    return cudaGetLastError();
}

cudaError_t qf_launch_tag_pack(const uint64_t* M, int count, int n, int word_bytes, void* tab, cudaStream_t stream) {
    if (n < 1 || count < 1 || (word_bytes != 4 && word_bytes != 8)) return cudaErrorInvalidValue;
    const int grid = tag_grid((long long)count * n * n);
    if (word_bytes == 4) tag_pack_kernel<uint32_t><<<grid, 256, 0, stream>>>(M, count, n, (uint32_t*)tab);
    else tag_pack_kernel<uint64_t><<<grid, 256, 0, stream>>>(M, count, n, (uint64_t*)tab);
    return cudaGetLastError();
}
