// Conversion, recombination and elementwise sampler kernels.
// All are HBM-streaming: flat grid-stride loops, lanes on the contiguous
// (coordinate) dimension, one warp per target row where a row reduction is needed.
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

// ---- conversions -----------------------------------------------------------
__global__ void i32_to_f64_kernel(const int32_t* __restrict__ in, long ldin, double* __restrict__ out, long ldout,
                                  int B, int M, unsigned long long* __restrict__ norm2) {
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (long b = (long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); b < B;
         b += (long)gridDim.x * warps_per_block) {
        const int32_t* src = in + b * ldin;
        double* dst = out + b * ldout;
        NormAcc acc;
        acc.clear();
        for (int j = lane; j < M; j += 32) {
            int32_t v = src[j];
            dst[j] = (double)v;
            acc.add_sq(v);
        }
        if (norm2) {
            acc.warp_reduce();
            if (lane == 0) norm2[b] = acc.value();
        }
    }
}

__global__ void i64_to_f64_kernel(const int64_t* __restrict__ in, long ldin, double* __restrict__ out, long ldout,
                                  int B, int M, double scale) {
    long total = (long)B * M;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / M;
        int j = (int)(i - b * M);
        out[b * ldout + j] = scale * (double)in[b * ldin + j];
    }
}

__global__ void f64_to_i32_kernel(const double* __restrict__ in, long ldin, int32_t* __restrict__ out, long ldout,
                                  int B, int M, int* flag) {
    long total = (long)B * M;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / M;
        int j = (int)(i - b * M);
        double v = in[b * ldin + j];
        double r = rint(v);
        if (r != v || fabs(r) > 2147483647.0) {
            if (flag) atomicOr(flag, 1);
            r = fmax(fmin(r, 2147483647.0), -2147483647.0);
        }
        out[b * ldout + j] = (int32_t)r;
    }
}

__global__ void domain_flags_kernel(const unsigned long long* __restrict__ norm2, unsigned long long bound,
                                    uint8_t* __restrict__ flags, int B) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
        flags[b] = norm2[b] <= bound ? 1 : 0;
}

// ---- recombination of exact fp64 partial products --------------------------
template <typename OutT>
__global__ void combine_kernel(CombineArgs a, OutT* __restrict__ out, long ldout, int B, int N) {
    long total = (long)B * N;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / N;
        int n = (int)(i - b * N);
        __int128 v = 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (c < a.nacc) {
                long long t = __double2ll_rn(a.acc[c][b * a.ldacc + n]);
                v += ((__int128)t) << a.shift[c];
            }
        }
        if (a.acc_sign < 0) v = -v;
        if (a.base) v += (__int128)a.base[b * a.ldbase + n];
        if (a.q) {
            out[b * ldout + n] = (OutT)mod_i128(v, a.q);
        } else {
            out[b * ldout + n] = (OutT)(long long)v;
        }
    }
}

__global__ void combine_i32_kernel(CombineArgs a, int32_t* __restrict__ out, long ldout, int B, int N, int* flag) {
    long total = (long)B * N;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / N;
        int n = (int)(i - b * N);
        __int128 v = 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (c < a.nacc) {
                long long t = __double2ll_rn(a.acc[c][b * a.ldacc + n]);
                v += ((__int128)t) << a.shift[c];
            }
        }
        if (a.acc_sign < 0) v = -v;
        if (a.base) v += (__int128)a.base[b * a.ldbase + n];
        if (v > 2147483647 || v < -2147483647) {
            if (flag) atomicOr(flag, 1);
            v = 0;
        }
        out[b * ldout + n] = (int32_t)(long long)v;
    }
}

__global__ void finalize_pert_kernel(const double* __restrict__ P, long ldp, const double* __restrict__ Zb, long ldz,
                                     int32_t* __restrict__ out, long ldo, int B, int M, int split, int* flag) {
    long total = (long)B * M;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / M;
        int j = (int)(i - b * M);
        double v = P[b * ldp + j];
        if (j >= split) v += Zb[b * ldz + (j - split)];
        double r = rint(v);
        if (r != v || fabs(r) > 2147483647.0) {
            if (flag) atomicOr(flag, 1);
            r = 0;
        }
        out[b * ldo + j] = (int32_t)r;
    }
}

__global__ void split_chunks_kernel(const double* __restrict__ in, long ldin, double* o0, double* o1, double* o2,
                                    double* o3, int nchunks, int bits, long ldout, int B, int M) {
    long total = (long)B * M;
    const double scale = ldexp(1.0, bits), inv = ldexp(1.0, -bits);
    double* outs[4] = {o0, o1, o2, o3};
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / M;
        int j = (int)(i - b * M);
        double rem = in[b * ldin + j];
        for (int c = 0; c < nchunks; ++c) {
            if (c == nchunks - 1) {
                outs[c][b * ldout + j] = rem;
            } else {
                double hi = rint(rem * inv);
                outs[c][b * ldout + j] = rem - hi * scale;
                rem = hi;
            }
        }
    }
}

__global__ void scatter_cols_kernel(const double* __restrict__ src, long ldsrc, const int* __restrict__ cols,
                                    int ncols, double* __restrict__ dst, long lddst, int B, double scale) {
    long total = (long)B * ncols;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / ncols;
        int j = (int)(i - b * ncols);
        dst[b * lddst + cols[j]] = scale * src[b * ldsrc + j];
    }
}

// ---- samplers --------------------------------------------------------------
__global__ void normal_fill_kernel(double* __restrict__ out, long ld, int B, int M, uint64_t seed,
                                   uint64_t first_target, uint32_t tag) {
    const int half = (M + 1) >> 1;
    long total = (long)B * half;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / half;
        int p = (int)(i - b * half);
        Philox rng;
        rng.init(seed, (first_target + (uint64_t)b) * (uint64_t)half + (uint64_t)p, tag);
        float n0, n1;
        rng.normal2(n0, n1);
        double* row = out + b * ld;
        row[2 * p] = (double)n0;
        if (2 * p + 1 < M) row[2 * p + 1] = (double)n1;
    }
}

__global__ void dgauss_kernel(const double* __restrict__ center, long ldc, double* __restrict__ out_f64, long ldo,
                              int32_t* __restrict__ out_i32, long ldoi, int B, int M, DGaussParams dg,
                              uint64_t seed, uint64_t first_target, uint32_t tag, int* flag) {
    long total = (long)B * M;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / M;
        int j = (int)(i - b * M);
        Philox rng;
        rng.init(seed, (first_target + (uint64_t)b) * (uint64_t)M + (uint64_t)j, tag);
        double c = center ? center[b * ldc + j] : 0.0;
        double z = sample_dgauss(dg, c, rng, flag);
        if (out_f64) out_f64[b * ldo + j] = z;
        if (out_i32) out_i32[b * ldoi + j] = (int32_t)z;
    }
}

__global__ void uniform_modq_kernel(int64_t* __restrict__ out, long count, unsigned long long q, uint64_t seed,
                                    uint64_t first_index) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long)gridDim.x * blockDim.x) {
        Philox rng;
        rng.init(seed, first_index + (uint64_t)i, QF_STREAM_UNIFORM);
        uint64_t rh = ((uint64_t)rng.next() << 32) | rng.next();
        uint64_t rl = ((uint64_t)rng.next() << 32) | rng.next();
        // floor((rh*2^64 + rl) * q / 2^128): bias < q / 2^128
        uint64_t hi = __umul64hi(rh, q);
        uint64_t lo = rh * q;
        uint64_t carry = __umul64hi(rl, q);
        uint64_t s = lo + carry;
        if (s < lo) hi += 1;
        out[i] = (int64_t)hi;
    }
}

// R = U{0,1} - U{0,1} entrywise (trapdoor_distribution.rs:82-86): P(-1)=P(1)=1/4, P(0)=1/2.
// 16 entries per thread (one 128-bit Philox block gives 2 bits per entry for 64 entries;
// we use one block per 16 entries to keep the counter <-> entry map trivial).
__global__ void ternary_kernel(int8_t* __restrict__ out, long count, uint64_t seed) {
    long groups = (count + 15) / 16;
    for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long)gridDim.x * blockDim.x) {
        Philox rng;
        rng.init(seed, (uint64_t)g, QF_STREAM_TERNARY);
        uint32_t bits = rng.next();
        long base = g * 16;
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            if (base + t < count) {
                int a = (bits >> (2 * t)) & 1, b = (bits >> (2 * t + 1)) & 1;
                out[base + t] = (int8_t)(a - b);
            }
        }
    }
}

}  // namespace

cudaError_t qf_launch_i32_to_f64(const int32_t* in, long ldin, double* out, long ldout, int B, int M,
                                 unsigned long long* norm2, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    i32_to_f64_kernel<<<grid_for(B, TPB / 32), TPB, 0, stream>>>(in, ldin, out, ldout, B, M, norm2);
    return cudaGetLastError();
}
cudaError_t qf_launch_i64_to_f64(const int64_t* in, long ldin, double* out, long ldout, int B, int M, double scale,
                                 cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    i64_to_f64_kernel<<<grid_for((long long)B * M, TPB), TPB, 0, stream>>>(in, ldin, out, ldout, B, M, scale);
    return cudaGetLastError();
}
cudaError_t qf_launch_f64_to_i32(const double* in, long ldin, int32_t* out, long ldout, int B, int M, int* flag,
                                 cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    f64_to_i32_kernel<<<grid_for((long long)B * M, TPB), TPB, 0, stream>>>(in, ldin, out, ldout, B, M, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_domain_flags(const unsigned long long* norm2, unsigned long long bound, uint8_t* flags, int B,
                                   cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    domain_flags_kernel<<<grid_for(B, TPB), TPB, 0, stream>>>(norm2, bound, flags, B);
    return cudaGetLastError();
}
cudaError_t qf_launch_combine_i64(const CombineArgs& a, int64_t* out, long ldout, int B, int N, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    combine_kernel<int64_t><<<grid_for((long long)B * N, TPB), TPB, 0, stream>>>(a, out, ldout, B, N);
    return cudaGetLastError();
}
cudaError_t qf_launch_combine_f64(const CombineArgs& a, double* out, long ldout, int B, int N, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    combine_kernel<double><<<grid_for((long long)B * N, TPB), TPB, 0, stream>>>(a, out, ldout, B, N);
    return cudaGetLastError();
}
cudaError_t qf_launch_combine_i32(const CombineArgs& a, int32_t* out, long ldout, int B, int N, int* flag,
                                  cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    combine_i32_kernel<<<grid_for((long long)B * N, TPB), TPB, 0, stream>>>(a, out, ldout, B, N, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_finalize_pert(const double* P, long ldp, const double* Zb, long ldz, int32_t* out, long ldo,
                                    int B, int M, int split, int* flag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    finalize_pert_kernel<<<grid_for((long long)B * M, TPB), TPB, 0, stream>>>(P, ldp, Zb, ldz, out, ldo, B, M, split,
                                                                            flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_split_chunks(const double* in, long ldin, double* const* out, int nchunks, int bits, long ldout,
                                   int B, int M, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    double* o[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int c = 0; c < nchunks && c < 4; ++c) o[c] = out[c];
    split_chunks_kernel<<<grid_for((long long)B * M, TPB), TPB, 0, stream>>>(in, ldin, o[0], o[1], o[2], o[3], nchunks,
                                                                              bits, ldout, B, M);
    return cudaGetLastError();
}
cudaError_t qf_launch_scatter_cols_f64(const double* src, long ldsrc, const int* cols, int ncols, double* dst,
                                       long lddst, int B, double scale, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    scatter_cols_kernel<<<grid_for((long long)B * ncols, TPB), TPB, 0, stream>>>(src, ldsrc, cols, ncols, dst, lddst, B,
                                                                                scale);
    return cudaGetLastError();
}
cudaError_t qf_launch_normal_fill(double* out, long ld, int B, int M, uint64_t seed, uint64_t first_target,
                                  uint32_t tag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    normal_fill_kernel<<<grid_for((long long)B * ((M + 1) / 2), TPB), TPB, 0, stream>>>(out, ld, B, M, seed,
                                                                                       first_target, tag);
    return cudaGetLastError();
}
cudaError_t qf_launch_dgauss(const double* center, long ldc, double* out_f64, long ldo, int32_t* out_i32, long ldoi,
                             int B, int M, double s, uint64_t seed, uint64_t first_target, uint32_t tag, int* flag,
                             cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    DGaussParams dg = make_dgauss(s);
    dgauss_kernel<<<grid_for((long long)B * M, TPB), TPB, 0, stream>>>(center, ldc, out_f64, ldo, out_i32, ldoi, B, M,
                                                                      dg, seed, first_target, tag, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_uniform_modq(int64_t* out, long count, unsigned long long q, uint64_t seed,
                                   uint64_t first_index, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    uniform_modq_kernel<<<grid_for(count, TPB), TPB, 0, stream>>>(out, count, q, seed, first_index);
    return cudaGetLastError();
}
cudaError_t qf_launch_ternary(int8_t* out, long count, uint64_t seed, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    ternary_kernel<<<grid_for((count + 15) / 16, TPB), TPB, 0, stream>>>(out, count, seed);
    return cudaGetLastError();
}

// ---- limb splitting for the tcgen05 int8 contraction ---------------------------------------
// value = sum_l 256^l d_l with balanced digits d_l in [-128,127]; L digits cover
// [-128 S, 127 S], S = (256^L - 1)/255.  planes: L matrices of B x ldk bytes.
namespace {

// nz (optional): zero-tile map, nz[l * nz_plane + nz_idx] = 1 when digit l is non-zero (benign race: all writers store 1)
__device__ __forceinline__ void split_digits(long long v, int L, int8_t* planes, long plane_stride, long off, int* flag,
                                             uint8_t* nz = nullptr, long nz_plane = 0, long nz_idx = 0) {
    for (int l = 0; l < L - 1; ++l) {
        long long lo = ((v + 128) & 255) - 128;
        planes[l * plane_stride + off] = (int8_t)lo;
        if (nz && lo != 0 && !nz[l * nz_plane + nz_idx]) nz[l * nz_plane + nz_idx] = 1;
        v = (v - lo) >> 8;
    }
    if ((v > 127 || v < -128) && flag) atomicOr(flag, 8);
    planes[(L - 1) * plane_stride + off] = (int8_t)v;
    if (nz && v != 0 && !nz[(L - 1) * nz_plane + nz_idx]) nz[(L - 1) * nz_plane + nz_idx] = 1;
}

// One warp per target row, 128 columns (= one zero-tile) per warp iteration, 4 consecutive columns per lane:
// one vector load, one char4 store per digit plane, and one warp vote per digit for the zero-tile map
// (no global reads on the flag path).  col0 and ldk are multiples of 128 / 4 for every caller.
// returns (warp-uniform, when nz is given) the index of the highest digit plane this warp found non-zero, -1 if none
__device__ __forceinline__ int split4(const long long v[4], int L, int8_t* planes, long plane_stride, long off, int* flag,
                                      uint8_t* nz, long nz_plane, long nz_idx, int valid, int lane) {
    long long w[4] = {v[0], v[1], v[2], v[3]};
    int top = -1;
    for (int l = 0; l < L; ++l) {
        int8_t dd[4];
        bool any = false;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            long long lo = ((w[t] + 128) & 255) - 128;
            if (l == L - 1) {
                lo = w[t];
                if ((lo > 127 || lo < -128) && flag && t < valid) atomicOr(flag, 8);
            }
            dd[t] = (int8_t)lo;
            any |= (t < valid) && (dd[t] != 0);
            w[t] = (w[t] - lo) >> 8;
        }
        if (valid == 4) {
            char4 d;
            d.x = dd[0]; d.y = dd[1]; d.z = dd[2]; d.w = dd[3];
            *reinterpret_cast<char4*>(planes + l * plane_stride + off) = d;
        } else {
            for (int t = 0; t < valid; ++t) planes[l * plane_stride + off + t] = dd[t];
        }
        if (nz) {
            const bool warp_any = __any_sync(0xffffffffu, any);
            if (warp_any && lane == 0) nz[l * nz_plane + nz_idx] = 1;
            if (warp_any) top = l;
        }
    }
    return top;
}

// gate0..2 (optional device ints): raised (atomicMax) to the index of the highest non-zero digit plane written by this
// launch -- the contractions that consume these planes pick, on the device, the variant compiled for that many digits
__global__ void split_f64_limbs_kernel(const double* __restrict__ in, long ldin, int8_t* __restrict__ planes,
                                       long plane_stride, long ldk, int B, int M, int L, int* flag, uint8_t* nz,
                                       int nz_m_tiles, int nz_kb_total, int col0, int* gate0, int* gate1, int* gate2, int* gate3) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const int iters = (M + 127) >> 7;
    const long total = (long)B * iters;  // (row, 128-column tile) pairs, one per warp iteration
    for (long w = (long)blockIdx.x * wpb + (threadIdx.x >> 5); w < total; w += (long)gridDim.x * wpb) {
        const long b = w / iters;
        const int j = ((int)(w - b * iters) << 7) + lane * 4;
        const int valid = max(0, min(4, M - j));
        long long v[4] = {0, 0, 0, 0};
        const double* src = in + b * ldin + j;
        if (valid == 4 && ((((uintptr_t)src) & 15) == 0)) {
            const double2 a0 = *reinterpret_cast<const double2*>(src), a1 = *reinterpret_cast<const double2*>(src + 2);
            const double x[4] = {a0.x, a0.y, a1.x, a1.y};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                double xx = x[t];
                if (!(fabs(xx) < 9.0e18)) { if (flag) atomicOr(flag, 8); xx = 0; }
                v[t] = __double2ll_rn(xx);
            }
        } else {
            for (int t = 0; t < valid; ++t) {
                double xx = src[t];
                if (!(fabs(xx) < 9.0e18)) { if (flag) atomicOr(flag, 8); xx = 0; }
                v[t] = __double2ll_rn(xx);
            }
        }
        const int top = split4(v, L, planes, plane_stride, b * ldk + j, flag, nz, (long)nz_m_tiles * nz_kb_total,
                               (b >> 7) * nz_kb_total + ((col0 + j) >> 7), valid, lane);
        if (lane == 0 && top > 0) {  // plain read first: almost every warp finds the gate already high enough
            if (gate0 && *(volatile int*)gate0 < top) atomicMax(gate0, top);
            if (gate1 && *(volatile int*)gate1 < top) atomicMax(gate1, top);
            if (gate2 && *(volatile int*)gate2 < top) atomicMax(gate2, top);
            if (gate3 && *(volatile int*)gate3 < top) atomicMax(gate3, top);
        }
    }
}

// 32-bit variant of split4 for int32 inputs (values beyond +-2^30 belong to out-of-domain targets: clamped)
__device__ __forceinline__ void split4_i32(const int v[4], int L, int8_t* planes, long plane_stride, long off,
                                           uint8_t* nz, long nz_plane, long nz_idx, int valid, int lane) {
    int w[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) w[t] = max(-(1 << 30), min(1 << 30, v[t]));
    for (int l = 0; l < L; ++l) {
        int dd[4];
        int any = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            int lo = ((w[t] + 128) & 255) - 128;
            if (l == L - 1) lo = w[t];
            dd[t] = lo;
            any |= (t < valid) ? (lo & 255) : 0;
            w[t] = (w[t] - lo) >> 8;
        }
        if (valid == 4) {
            const unsigned pk = (dd[0] & 255) | ((dd[1] & 255) << 8) | ((dd[2] & 255) << 16) | ((unsigned)(dd[3] & 255) << 24);
            *reinterpret_cast<unsigned*>(planes + l * plane_stride + off) = pk;
        } else {
            for (int t = 0; t < valid; ++t) planes[l * plane_stride + off + t] = (int8_t)dd[t];
        }
        if (nz) {
            const bool warp_any = __any_sync(0xffffffffu, any != 0);
            if (warp_any && lane == 0) nz[l * nz_plane + nz_idx] = 1;
        }
    }
}

__global__ void __launch_bounds__(256)
split_i32_limbs_kernel(const int32_t* __restrict__ in, long ldin, int8_t* __restrict__ planes,
                       long plane_stride, long ldk, int B, int M, int L,
                       unsigned long long* __restrict__ norm2, uint8_t* nz, int nz_m_tiles,
                       int nz_kb_total) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const bool vec = ((ldin & 3) == 0) && ((((uintptr_t)in) & 15) == 0);
    const int iters = (M + 127) >> 7;
    for (long b = (long)blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += (long)gridDim.x * wpb) {
        const int32_t* src = in + b * ldin;
        NormAcc acc;
        acc.clear();
        const long nz_plane = (long)nz_m_tiles * nz_kb_total, nz_row = (b >> 7) * nz_kb_total;
        int it = 0;
        // two 128-column tiles per trip: both vector loads are issued before either is consumed
        for (; it + 1 < iters && vec && ((it + 2) << 7) <= M; it += 2) {
            const int j0 = (it << 7) + lane * 4, j1 = j0 + 128;
            const int4 q0 = __ldcs(reinterpret_cast<const int4*>(src + j0));
            const int4 q1 = __ldcs(reinterpret_cast<const int4*>(src + j1));
            const int v0[4] = {q0.x, q0.y, q0.z, q0.w}, v1[4] = {q1.x, q1.y, q1.z, q1.w};
            acc.add_sq4(v0[0], v0[1], v0[2], v0[3]);
            acc.add_sq4(v1[0], v1[1], v1[2], v1[3]);
            split4_i32(v0, L, planes, plane_stride, b * ldk + j0, nz, nz_plane, nz_row + (j0 >> 7), 4, lane);
            split4_i32(v1, L, planes, plane_stride, b * ldk + j1, nz, nz_plane, nz_row + (j1 >> 7), 4, lane);
        }
        for (; it < iters; ++it) {
            const int j = (it << 7) + lane * 4;
            const int valid = max(0, min(4, M - j));
            int v[4] = {0, 0, 0, 0};
            for (int t = 0; t < valid; ++t) v[t] = src[j + t];
            acc.add_sq4(v[0], v[1], v[2], v[3]);
            split4_i32(v, L, planes, plane_stride, b * ldk + j, nz, nz_plane, nz_row + (j >> 7), valid, lane);
        }
        if (norm2) {
            acc.warp_reduce();
            if (lane == 0) norm2[b] = acc.value();
        }
    }
}

__global__ void add_cols_i32_kernel(int32_t* __restrict__ e, long lde, const double* __restrict__ sol, long ldsol,
                                    const int* __restrict__ cols, int ncols, int B) {
    long total = (long)B * ncols;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        long b = i / ncols;
        int j = (int)(i - b * ncols);
        e[b * lde + cols[j]] += (int32_t)__double2ll_rn(sol[b * ldsol + j]);
    }
}

}  // namespace

namespace {
__global__ void pert_xb_kernel(const double* __restrict__ G, long ldg, double* __restrict__ X2, long ldx,
                               int8_t* __restrict__ planes, long plane_stride, long ldk, int B, int mb, int nk,
                               double sqrt_beta, double fscale, int L, int* flag) {
    const long total = (long)B * nk;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / nk;
        const int j = (int)(i - b * nk);
        const double xb = sqrt_beta * G[b * ldg + mb + j];
        X2[b * ldx + mb + j] = xb;
        split_digits(__double2ll_rn(xb * fscale), L, planes, plane_stride, b * ldk + j, flag);
    }
}
}  // namespace
namespace {
__global__ void pert_normal_digits_kernel(int B, int M, int split, uint64_t seed, uint64_t first_target,
                                          int8_t* __restrict__ gplanes, long gplane_stride, long ldkg, int LG, double gscale,
                                          double* __restrict__ X2, long ldx, int8_t* __restrict__ bplanes, long bplane_stride,
                                          long ldkb, int LB, double sqrt_beta, double bscale, int* flag) {
    const int half = (M + 1) >> 1;
    const long total = (long)B * half;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / half;
        const int p = (int)(i - b * half);
        Philox rng;
        rng.init(seed, (first_target + (uint64_t)b) * (uint64_t)half + (uint64_t)p, QF_STREAM_PERT_NORMAL);
        float nn[2];
        rng.normal2(nn[0], nn[1]);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int j = 2 * p + t;
            if (j >= M) break;
            if (j < split) {
                split_digits(__double2ll_rn((double)nn[t] * gscale), LG, gplanes, gplane_stride, b * ldkg + j, flag);
            } else {
                const double xb = sqrt_beta * (double)nn[t];
                X2[b * ldx + j] = xb;
                split_digits(__double2ll_rn(xb * bscale), LB, bplanes, bplane_stride, b * ldkb + (j - split), flag);
            }
        }
    }
}
}  // namespace
cudaError_t qf_launch_pert_normal_digits(int B, int M, int split, uint64_t seed, uint64_t first_target, int8_t* gplanes,
                                         long gplane_stride, long ldkg, int LG, double gscale, double* X2, long ldx,
                                         int8_t* bplanes, long bplane_stride, long ldkb, int LB, double sqrt_beta, double bscale,
                                         int* flag, cudaStream_t stream) {
    if (B <= 0 || M <= 0) return cudaSuccess;
    pert_normal_digits_kernel<<<grid_for((long long)B * ((M + 1) / 2), TPB), TPB, 0, stream>>>(
        B, M, split, seed, first_target, gplanes, gplane_stride, ldkg, LG, gscale, X2, ldx, bplanes, bplane_stride, ldkb, LB,
        sqrt_beta, bscale, flag);
    return cudaGetLastError();
}
namespace {
// I2[b][row] += sum_c S'[row][c] z1[b][c] for the block-diagonal gadget basis S' = (I_n (x) S_k), columns reversed
// when `reversed` (short_basis_classical.rs:80-82): only the k columns of the row's own block contribute.
__global__ void sprime_apply_kernel(const double* __restrict__ Z, long ldz, double* __restrict__ I2, long ldi, int B, int nk,
                                    int k, const double* __restrict__ sk, int reversed) {
    const long total = (long)B * nk;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / nk;
        const int row = (int)(i - b * nk);
        const int blk = row / k, t = row - blk * k;
        const double* zr = Z + b * ldz;
        // row t of S_k has at most three non-zeros: the diagonal, the sub-diagonal -1 and (q not a power of the base)
        // the digit of q in the last column
        double acc = 0.0;
        const int cand[3] = {t - 1, t, k - 1};
#pragma unroll
        for (int e = 0; e < 3; ++e) {
            const int c = cand[e];
            if (c < 0 || (e == 2 && (c == t || c == t - 1))) continue;
            const double sv = sk[t * k + c];
            if (sv == 0.0) continue;
            const int cc = blk * k + c;                      // column of I_n (x) S_k
            const int col = reversed ? nk - 1 - cc : cc;     // where that column sits in S'
            acc = fma(sv, zr[col], acc);
        }
        I2[b * ldi + row] += acc;
    }
}
// e[b][i] += z2[b][i] (i < mb),  e[b][mb + row] = I2[b][row] (+ g3[b][row], two-phase form): the structured form of e = S z
__global__ void gpv_struct_finalize_kernel(int32_t* __restrict__ e, long lde, const double* __restrict__ Z2, long ldz,
                                           const double* __restrict__ I2, long ldi, int B, int mb, int nk, int* flag,
                                           const int8_t* __restrict__ g3, long ldg) {
    const int m = mb + nk;
    const long total = (long)B * m;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / m;
        const int j = (int)(i - b * m);
        double v = j < mb ? (double)e[b * lde + j] + Z2[b * ldz + j]
                          : I2[b * ldi + (j - mb)] + (g3 ? (double)g3[b * ldg + (j - mb)] : 0.0);
        if (!(fabs(v) < 2147483647.0)) { if (flag) atomicOr(flag, 4); v = 0.0; }
        e[b * lde + j] = (int32_t)__double2ll_rn(v);
    }
}
}  // namespace
namespace {
// e_bot = g3 + S' z1 in one pass (two-phase form, api.cu samp_p_np2_chunk): four consecutive gadget rows per thread;
// writes the int32 values into e[b][mb + row] and their balanced base-256 digit planes (the x operand of R e_bot).
__global__ void gpv_ebot_kernel(const double* __restrict__ Z, long ldz, const int8_t* __restrict__ g3, long ldg,
                                int32_t* __restrict__ e, long lde, int mb, int8_t* __restrict__ planes, long plane_stride,
                                long ldk, int L, int B, int nk, int k, const double* __restrict__ sk, int reversed, int* flag) {
    const int nq = nk >> 2;
    const long total = (long)B * nq;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / nq;
        const int r0 = (int)(i - b * nq) << 2;
        const double* zr = Z + b * ldz;
        const unsigned gw = *reinterpret_cast<const unsigned*>(g3 + b * ldg + r0);
        long long v[4];
#pragma unroll
        for (int t4 = 0; t4 < 4; ++t4) {
            const int row = r0 + t4, blk = row / k, t = row - blk * k;
            double acc = (double)(int8_t)((gw >> (8 * t4)) & 255);
            const int cand[3] = {t - 1, t, k - 1};
#pragma unroll
            for (int c3 = 0; c3 < 3; ++c3) {
                const int c = cand[c3];
                if (c < 0 || (c3 == 2 && (c == t || c == t - 1))) continue;
                const double sv = sk[t * k + c];
                if (sv == 0.0) continue;
                const int cc = blk * k + c;
                acc = fma(sv, zr[reversed ? nk - 1 - cc : cc], acc);
            }
            if (!(fabs(acc) < 2147483647.0)) { if (flag) atomicOr(flag, 4); acc = 0.0; }
            v[t4] = __double2ll_rn(acc);
        }
        *reinterpret_cast<int4*>(e + b * lde + mb + r0) = make_int4((int)v[0], (int)v[1], (int)v[2], (int)v[3]);
        for (int l = 0; l < L; ++l) {
            unsigned pk = 0;
#pragma unroll
            for (int t4 = 0; t4 < 4; ++t4) {
                long long d = ((v[t4] + 128) & 255) - 128;
                if (l == L - 1) {
                    d = v[t4];
                    if (d > 127 || d < -128) { if (flag) atomicOr(flag, 8); d = 0; }
                }
                v[t4] = (v[t4] - d) >> 8;
                pk |= (unsigned)(d & 255) << (8 * t4);
            }
            *reinterpret_cast<unsigned*>(planes + (long)l * plane_stride + b * ldk + r0) = pk;
        }
    }
}
}  // namespace
cudaError_t qf_launch_gpv_ebot(const double* Z, long ldz, const int8_t* g3, long ldg, int32_t* e, long lde, int mb,
                               int8_t* planes, long plane_stride, long ldk, int L, int B, int nk, int k, const double* sk,
                               int reversed, int* flag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    // four rows per thread, 16-byte int32 stores, 4-byte digit stores
    if ((nk & 3) || (ldg & 3) || (ldk & 3) || (plane_stride & 3) || (lde & 3) || (mb & 3) || (((uintptr_t)e) & 15) ||
        (((uintptr_t)g3) & 3) || (((uintptr_t)planes) & 3))
        return cudaErrorInvalidValue;
    gpv_ebot_kernel<<<grid_for((long long)B * (nk / 4), TPB), TPB, 0, stream>>>(Z, ldz, g3, ldg, e, lde, mb, planes, plane_stride,
                                                                               ldk, L, B, nk, k, sk, reversed, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_sprime_apply(const double* Z, long ldz, double* I2, long ldi, int B, int nk, int k, const double* sk,
                                   int reversed, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    sprime_apply_kernel<<<grid_for((long long)B * nk, TPB), TPB, 0, stream>>>(Z, ldz, I2, ldi, B, nk, k, sk, reversed);
    return cudaGetLastError();
}
cudaError_t qf_launch_gpv_struct_finalize(int32_t* e, long lde, const double* Z2, long ldz, const double* I2, long ldi, int B,
                                          int mb, int nk, int* flag, cudaStream_t stream, const int8_t* g3, long ldg) {
    if (B <= 0) return cudaSuccess;
    gpv_struct_finalize_kernel<<<grid_for((long long)B * (mb + nk), TPB), TPB, 0, stream>>>(e, lde, Z2, ldz, I2, ldi, B, mb, nk,
                                                                                           flag, g3, ldg);
    return cudaGetLastError();
}
namespace {
// g3[b][blk * k + t] = digit t (base `base`) of h[b][blk]: the gadget-lattice coset representative with G g3 = h
// (gadget_classical.rs:169-182, find_solution_gadget_vec), one thread per (target, syndrome entry)
__global__ void gadget_digits_kernel(const int64_t* __restrict__ h, long ldh, int8_t* __restrict__ plane, long ldk, int B,
                                     int n, int k, unsigned base, uint8_t* __restrict__ nz, int nz_kb_total,
                                     double* __restrict__ I2, long ldi) {
    // one thread per four consecutive output digits (coalesced 4-byte / 32-byte stores); nk = n k is a multiple of 4 for
    // every caller (the structured path needs nk % 128 == 0), ragged tails take the scalar branch
    const int nk = n * k, nq = (nk + 3) >> 2;
    const long total = (long)B * nq;
    const bool pow2 = (base & (base - 1)) == 0;
    const int sh = 31 - __clz(base);
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / nq;
        const int c0 = (int)(i - b * nq) << 2;
        unsigned d[4] = {0, 0, 0, 0};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int c = c0 + e;
            if (c >= nk) break;
            const int blk = c / k, t = c - blk * k;
            unsigned long long v = (unsigned long long)h[b * ldh + blk];
            if (pow2) {
                d[e] = (t * sh < 64) ? (unsigned)((v >> (t * sh)) & (base - 1)) : 0u;
            } else {
                for (int r = 0; r < t; ++r) v /= base;
                d[e] = (unsigned)(v % base);
            }
        }
        if (c0 + 3 < nk && ((ldk & 3) == 0)) {
            *reinterpret_cast<unsigned*>(plane + b * ldk + c0) = d[0] | (d[1] << 8) | (d[2] << 16) | (d[3] << 24);
            if (I2) {
                double* o = I2 + b * ldi + c0;
                if (((ldi & 1) == 0) && ((((uintptr_t)I2) & 15) == 0)) {
                    reinterpret_cast<double2*>(o)[0] = make_double2((double)d[0], (double)d[1]);
                    reinterpret_cast<double2*>(o)[1] = make_double2((double)d[2], (double)d[3]);
                } else {
                    for (int e = 0; e < 4; ++e) o[e] = (double)d[e];
                }
            }
        } else {
            for (int e = 0; e < 4 && c0 + e < nk; ++e) {
                plane[b * ldk + c0 + e] = (int8_t)d[e];
                if (I2) I2[b * ldi + c0 + e] = (double)d[e];
            }
        }
    }
    if (nz) {  // plane 0 of the zero-tile map: every (128-target, 128-column) tile of the digit block is live
        const int kbn = (nk + 127) >> 7, mt = (B + 127) >> 7;
        for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)mt * kbn; i += (long)gridDim.x * blockDim.x)
            nz[(i / kbn) * nz_kb_total + (i % kbn)] = 1;
    }
}
}  // namespace
cudaError_t qf_launch_gadget_digits(const int64_t* h, long ldh, int8_t* plane, long ldk, int B, int n, int k, unsigned base,
                                    uint8_t* nz, int nz_kb_total, cudaStream_t stream, double* I2, long ldi) {
    if (B <= 0) return cudaSuccess;
    if (base < 2 || base > 128) return cudaErrorInvalidValue;
    gadget_digits_kernel<<<grid_for((long long)B * ((n * k + 3) / 4), TPB), TPB, 0, stream>>>(h, ldh, plane, ldk, B, n, k, base, nz,
                                                                                          nz_kb_total, I2, ldi);
    return cudaGetLastError();
}
cudaError_t qf_launch_pert_xb(const double* G, long ldg, double* X2, long ldx, int8_t* planes, long plane_stride, long ldk,
                              int B, int mb, int nk, double sqrt_beta, double fscale, int L, int* flag, cudaStream_t stream) {
    if (B <= 0 || nk <= 0) return cudaSuccess;
    pert_xb_kernel<<<grid_for((long long)B * nk, TPB), TPB, 0, stream>>>(G, ldg, X2, ldx, planes, plane_stride, ldk, B, mb, nk,
                                                                        sqrt_beta, fscale, L, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_split_f64_limbs(const double* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B,
                                      int M, int L, int* flag, uint8_t* nz, int nz_m_tiles, int nz_kb_total, int col0,
                                      cudaStream_t stream, int* gate0, int* gate1, int* gate2, int* gate3) {
    if (B <= 0) return cudaSuccess;
    // char4 stores need 4-byte aligned plane addresses: planes pointer, ldk and col0 multiples of 4 (true for all callers)
    if ((((uintptr_t)planes) & 3) || (ldk & 3) || (col0 & 3)) return cudaErrorMisalignedAddress;
    if (nz && (col0 & 127)) return cudaErrorInvalidValue;
    split_f64_limbs_kernel<<<grid_for((long long)B * ((M + 127) / 128), TPB / 32), TPB, 0, stream>>>(
        in, ldin, planes, plane_stride, ldk, B, M, L, flag, nz, nz_m_tiles, nz_kb_total, col0, gate0, gate1, gate2, gate3);
    return cudaGetLastError();
}
cudaError_t qf_launch_split_i32_limbs(const int32_t* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B,
                                      int M, int L, unsigned long long* norm2, uint8_t* nz, int nz_m_tiles,
                                      int nz_kb_total, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    split_i32_limbs_kernel<<<grid_for(B, TPB / 32), TPB, 0, stream>>>(in, ldin, planes, plane_stride, ldk, B, M, L, norm2,
                                                                      nz, nz_m_tiles, nz_kb_total);
    return cudaGetLastError();
}
cudaError_t qf_launch_add_cols_i32(int32_t* e, long lde, const double* sol, long ldsol, const int* cols, int ncols,
                                   int B, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    add_cols_i32_kernel<<<grid_for((long long)B * ncols, TPB), TPB, 0, stream>>>(e, lde, sol, ldsol, cols, ncols, B);
    return cudaGetLastError();
}

// ---- narrow boundary types: int16 Domain values (|entry| <= 6 s r < 2^15 at C2 / C3) and the device-side range check of
// the targets ------------------------------------------------------------------------------------------------------------
namespace {
// 8 values per thread: two 128-bit loads, one 128-bit store; *flag |= 64 when a value does not fit int16
__global__ void __launch_bounds__(256) narrow_i32_i16_kernel(const int32_t* __restrict__ in, int16_t* __restrict__ out, size_t count,
                                                             int* flag) {
    const size_t groups = count >> 3;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    bool bad = false;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
        const int4 a = __ldcs(reinterpret_cast<const int4*>(in) + 2 * g), b = __ldcs(reinterpret_cast<const int4*>(in) + 2 * g + 1);
        const int v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        unsigned pk[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            bad |= (v[2 * t] != (int)(short)v[2 * t]) | (v[2 * t + 1] != (int)(short)v[2 * t + 1]);
            pk[t] = ((unsigned)v[2 * t] & 0xFFFFu) | ((unsigned)v[2 * t + 1] << 16);
        }
        __stcs(reinterpret_cast<uint4*>(out) + g, make_uint4(pk[0], pk[1], pk[2], pk[3]));
    }
    if (blockIdx.x == 0 && threadIdx.x < (count & 7)) {
        const size_t i = (groups << 3) + threadIdx.x;
        const int v = in[i];
        bad |= v != (int)(short)v;
        out[i] = (int16_t)v;
    }
    if (bad && flag) atomicOr(flag, 64);
}
__global__ void __launch_bounds__(256) widen_i16_i32_kernel(const int16_t* __restrict__ in, int32_t* __restrict__ out, size_t count) {
    const size_t groups = count >> 3;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
        const uint4 a = __ldcs(reinterpret_cast<const uint4*>(in) + g);
        const unsigned w[4] = {a.x, a.y, a.z, a.w};
        int v[8];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            v[2 * t] = (int)(short)(w[t] & 0xFFFFu);
            v[2 * t + 1] = (int)(short)(w[t] >> 16);
        }
        __stcs(reinterpret_cast<int4*>(out) + 2 * g, make_int4(v[0], v[1], v[2], v[3]));
        __stcs(reinterpret_cast<int4*>(out) + 2 * g + 1, make_int4(v[4], v[5], v[6], v[7]));
    }
    if (blockIdx.x == 0 && threadIdx.x < (count & 7)) {
        const size_t i = (groups << 3) + threadIdx.x;
        out[i] = (int32_t)in[i];
    }
}
// *flag |= 32 when some residue lies outside [0, q)
__global__ void __launch_bounds__(256) range_check_i64_kernel(const int64_t* __restrict__ v, size_t count, unsigned long long q, int* flag) {
    bool bad = false;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        bad |= (unsigned long long)v[i] >= q;  // negative values are huge as unsigned
    if (bad) atomicOr(flag, 32);
}
// balanced base-256 digits of int64 values (|v| < 2^63): planes[l][b][j] = digit l of in[b][j] for j < M, zero for
// M <= j < ldk; *flag |= 8 when a value does not fit L digits.  One thread per (row, column).
__global__ void __launch_bounds__(256) split_i64_limbs_kernel(const int64_t* __restrict__ in, long ldin, int8_t* __restrict__ planes,
                                                              long plane_stride, long ldk, int B, int M, int L, int* flag) {
    const long total = (long)B * ldk;
    bool bad = false;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long b = t / ldk, j = t - b * ldk;
        long long v = j < M ? in[b * ldin + j] : 0;
        for (int l = 0; l < L; ++l) {
            long long lo = ((v + 128) & 255) - 128;
            if (l == L - 1) {
                bad |= v != lo;
                lo = v;
            }
            v = (v - lo) >> 8;
            planes[l * plane_stride + b * ldk + j] = (int8_t)lo;
        }
    }
    if (bad && flag) atomicOr(flag, 8);
}
}  // namespace
cudaError_t qf_launch_narrow_i32_i16(const int32_t* in, int16_t* out, size_t count, int* flag, cudaStream_t stream) {
    if (count == 0) return cudaSuccess;
    if ((((uintptr_t)in) & 15) || (((uintptr_t)out) & 15)) return cudaErrorMisalignedAddress;
    narrow_i32_i16_kernel<<<grid_for((long long)((count >> 3) + 1), 256, 148 * 8), 256, 0, stream>>>(in, out, count, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_widen_i16_i32(const int16_t* in, int32_t* out, size_t count, cudaStream_t stream) {
    if (count == 0) return cudaSuccess;
    if ((((uintptr_t)in) & 15) || (((uintptr_t)out) & 15)) return cudaErrorMisalignedAddress;
    widen_i16_i32_kernel<<<grid_for((long long)((count >> 3) + 1), 256, 148 * 8), 256, 0, stream>>>(in, out, count);
    return cudaGetLastError();
}
cudaError_t qf_launch_range_check_i64(const int64_t* v, size_t count, unsigned long long q, int* flag, cudaStream_t stream) {
    if (count == 0) return cudaSuccess;
    range_check_i64_kernel<<<grid_for((long long)count, 256, 148 * 4), 256, 0, stream>>>(v, count, q, flag);
    return cudaGetLastError();
}
cudaError_t qf_launch_split_i64_limbs(const int64_t* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B, int M,
                                      int L, int* flag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (M > ldk || L < 1 || L > 8) return cudaErrorInvalidValue;
    split_i64_limbs_kernel<<<grid_for((long long)B * ldk, 256, 148 * 8), 256, 0, stream>>>(in, ldin, planes, plane_stride, ldk, B, M,
                                                                                         L, flag);
    return cudaGetLastError();
}

// ---- per-target tag (qf_samp_p_tagged): v'_b = H_t^-1 (v_b + H_0 y_b) - y_b mod q with y_b = G p_bot_b, t = tidx[b] ----------
// PSFPerturbation passes p; PSFGPV's two-phase recursion passes P == nullptr (y = 0, h0 == nullptr): h_t = H_t^-1 w.
// One CTA per target; thread i owns rows i, i + blockDim, ... .  The tables hold each n x n matrix column-major (word
// [j][i] = M[i][j]), so at a fixed column the threads of a warp read consecutive words; y and w live in shared memory.
// Exact for every q < 2^62 and n:
//  - W = uint32_t (q <= 2^32): the shared vectors are held as 16-bit halves, so a table word times a half is < 2^48 and a
//    row of n <= 2^14 such products stays below 2^62 in a plain 64-bit register (two IMAD.WIDE per entry, no carries);
//    one Barrett step per half reduces the sums (mod_halves needs a0, a1 < 2^62).
//  - W = uint64_t: a product of residues is < 2^124 and a row sum runs in three words (192 bits) before one reduction,
//    so (q - 1)^2 n >= 2^128 cannot wrap.
namespace {
struct ModAcc {
    unsigned long long lo = 0, mid = 0;
    unsigned int hi = 0;
    __device__ __forceinline__ void mac(uint64_t a, uint64_t b) {
        const unsigned long long pl = a * b, ph = __umul64hi(a, b);
        asm("add.cc.u64 %0, %0, %3;\n\taddc.cc.u64 %1, %1, %4;\n\taddc.u32 %2, %2, 0;" : "+l"(lo), "+l"(mid), "+r"(hi) : "l"(pl), "l"(ph));
    }
    __device__ __forceinline__ uint64_t reduce(uint64_t q) const {
        typedef unsigned __int128 u128;
        const uint64_t top = (uint64_t)((((u128)hi) << 64 | mid) % q);
        return (uint64_t)((((u128)top) << 64 | lo) % q);
    }
};

// (a1 2^16 + a0) mod q for a0, a1 < 2^62, q <= 2^32 (magic = floor(2^64 / q))
__device__ __forceinline__ uint64_t mod_halves(uint64_t a0, uint64_t a1, uint64_t q, uint64_t magic) {
    const uint64_t h = mod_i64_barrett((long long)a1, q, magic);
    return mod_i64_barrett((long long)(a0 + (h << 16)), q, magic);
}
__device__ __forceinline__ uint2 halves(uint64_t x) { return make_uint2((unsigned)(x & 0xFFFF), (unsigned)(x >> 16)); }

// A residue as the shared vectors of the two regimes hold it: 16-bit halves for W = uint32_t, one word for W = uint64_t.
template <typename W> struct PolySV;
template <> struct PolySV<uint32_t> {
    typedef uint2 T;
    static __device__ __forceinline__ uint2 put(uint64_t x) { return halves(x); }
    static __device__ __forceinline__ uint64_t get(uint2 h) { return h.x + ((uint64_t)h.y << 16); }
};
template <> struct PolySV<uint64_t> {
    typedef uint64_t T;
    static __device__ __forceinline__ uint64_t put(uint64_t x) { return x; }
    static __device__ __forceinline__ uint64_t get(uint64_t x) { return x; }
};

// ---- product of tags in polynomial form (DESIGN 4.10): r = a * b mod (f, q), f = X^n + sum_{i<n} f_i X^i monic --------
// The one product of the inverse (poly_tag_inverse_kernel), the samp_p syndrome and the f_a correction.  a: n residues in
// any memory; b: n residues in shared memory (PolySV<W>); c: 2n - 1 PolySV<W> of shared scratch; xr: rows X^{n+j} mod f
// for j < n - 1, n words each (qf_launch_poly_xpow; n^2 words shared by every CTA, so L2-resident).  Schoolbook
// c_l = sum_{i+j=l} a_i b_j for l < 2n - 1, then r_i = c_i + sum_{j < n-1} c_{n+j} xr[j][i]: no sequential chain, and one
// code path for every f.  Exact for every q < 2^62 in the regimes of tag_syndrome_kernel: for W = uint32_t (q <= 2^32) a
// sum of at most n <= 2^14 products word x half stays below 2^62 (mod_halves), for W = uint64_t it runs in 192 bits.
// Every thread of the CTA calls it.  emit(i, r_i) runs after a barrier that follows the last read of a and b (so it may
// overwrite them); c may be rewritten only after the next barrier.
template <typename W, typename A, typename Emit>
__device__ __forceinline__ void poly_mulmod(const A* a, const typename PolySV<W>::T* b, typename PolySV<W>::T* c,
                                            const W* __restrict__ xr, uint64_t q, uint64_t magic, int n, Emit emit) {
    for (int l = threadIdx.x; l < 2 * n - 1; l += blockDim.x) {
        const int i0 = max(0, l - n + 1), i1 = min(l, n - 1);
        if constexpr (sizeof(W) == 4) {
            uint64_t a0 = 0, a1 = 0;
#pragma unroll 4
            for (int i = i0; i <= i1; ++i) {
                const uint64_t x = a[i];
                const uint2 y = b[l - i];
                a0 += x * y.x;
                a1 += x * y.y;
            }
            c[l] = halves(mod_halves(a0, a1, q, magic));
        } else {
            ModAcc s;
#pragma unroll 2
            for (int i = i0; i <= i1; ++i) s.mac(a[i], b[l - i]);
            c[l] = s.reduce(q);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if constexpr (sizeof(W) == 4) {
            const uint2 ci = c[i];
            uint64_t a0 = ci.x, a1 = ci.y;
#pragma unroll 4
            for (int j = 0; j < n - 1; ++j) {
                const uint64_t x = xr[(long)j * n + i];
                const uint2 y = c[n + j];
                a0 += x * y.x;
                a1 += x * y.y;
            }
            emit(i, mod_halves(a0, a1, q, magic));
        } else {
            ModAcc s;
            s.mac(c[i], 1);
#pragma unroll 2
            for (int j = 0; j < n - 1; ++j) s.mac(xr[(long)j * n + i], c[n + j]);
            emit(i, s.reduce(q));
        }
    }
}

// y_i = sum_{s<k} sb[s] base^s mod q for one row of int32 entries (G sigma_bot), as fa_tag_correct_kernel forms it: (sb mod
// q) times the halves of base^s mod q for W = uint32_t (k <= 64 terms < 2^48), 192-bit sums otherwise
template <typename W>
__device__ __forceinline__ uint64_t gadget_row_mod(const int32_t* sb, const uint64_t* __restrict__ gpow, uint64_t q,
                                                   uint64_t magic, int k) {
    if constexpr (sizeof(W) == 4) {
        uint64_t a0 = 0, a1 = 0;
        for (int s = 0; s < k; ++s) {
            const uint64_t sm = mod_i64_barrett((long long)sb[s], q, magic), gs = gpow[s];
            a0 += sm * (gs & 0xFFFF);
            a1 += sm * (gs >> 16);
        }
        return mod_halves(a0, a1, q, magic);
    } else {
        ModAcc a;
        for (int s = 0; s < k; ++s) a.mac(sb[s] < 0 ? (uint64_t)((long long)sb[s] + (long long)q) : (uint64_t)sb[s], gpow[s]);
        return a.reduce(q);
    }
}

// POLY: the table holds s_t = h_t^-1 as n words per tag and the last step is v' = s_t * w mod (f, q) - y (xr: the rows of
// poly_mulmod); otherwise H_t^-1 as n x n words and v' = H_t^-1 w - y.  y and w are formed the same way in both.
template <typename W, bool POLY>
__global__ void __launch_bounds__(512) tag_syndrome_kernel(const int64_t* __restrict__ V, long ldv, const double* __restrict__ P,
                                                           long ldp, int m_bar, const int32_t* __restrict__ tidx, int ntags,
                                                           const W* __restrict__ tab, const W* __restrict__ h0,
                                                           const uint64_t* __restrict__ gpow, uint64_t q, uint64_t magic, int n,
                                                           int k, int64_t* __restrict__ out, long ldout, int* flag,
                                                           const W* __restrict__ xr) {
    extern __shared__ uint64_t tag_sh[];
    const long b = blockIdx.x;
    const int t = tidx[b];
    if (t < 0 || t >= ntags) {  // the table is not read; the gadget sampler gets a valid residue
        for (int i = threadIdx.x; i < n; i += blockDim.x) out[b * ldout + i] = 0;
        if (threadIdx.x == 0 && flag) atomicOr(flag, QF_FLAG_TAG_INDEX);
        return;
    }
    const double* pb = P ? P + b * ldp + m_bar : nullptr;
    const W* hi = tab + (long)t * n * (POLY ? 1 : n);
    if constexpr (sizeof(W) == 4) {
        uint2* ys = reinterpret_cast<uint2*>(tag_sh);  // 16-bit halves of y and w
        uint2* ws = ys + n;
        // y_i = sum_s base^s p[m_bar + i k + s] mod q: (p mod q) times the halves of base^s mod q, k <= 64 terms < 2^48
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            uint64_t a0 = 0, a1 = 0;
            for (int s = 0; s < (P ? k : 0); ++s) {
                const uint64_t pm = mod_i64_barrett((long long)pb[(long)i * k + s], q, magic), g = gpow[s];
                a0 += pm * (g & 0xFFFF);
                a1 += pm * (g >> 16);
            }
            ys[i] = halves(mod_halves(a0, a1, q, magic));
        }
        __syncthreads();
        // w = v + H_0 y (v + y for H_0 = I)
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint2 yi = ys[i];
            uint64_t hy = yi.x + ((uint64_t)yi.y << 16);
            if (h0) {
                uint64_t a0 = 0, a1 = 0;
#pragma unroll 8
                for (int j = 0; j < n; ++j) {
                    const uint64_t h = h0[(long)j * n + i];
                    const uint2 yj = ys[j];
                    a0 += h * yj.x;
                    a1 += h * yj.y;
                }
                hy = mod_halves(a0, a1, q, magic);
            }
            const uint64_t sum = (uint64_t)V[b * ldv + i] + hy;
            ws[i] = halves(sum >= q ? sum - q : sum);
        }
        __syncthreads();
        // v' = H_t^-1 w - y
        if constexpr (POLY) {
            poly_mulmod<W>(hi, ws, ws + n, xr, q, magic, n, [&](int i, uint64_t x) {
                const uint64_t yi = PolySV<W>::get(ys[i]);
                out[b * ldout + i] = (int64_t)(x >= yi ? x - yi : x + (q - yi));
            });
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                uint64_t a0 = 0, a1 = 0;
#pragma unroll 8
                for (int j = 0; j < n; ++j) {
                    const uint64_t h = hi[(long)j * n + i];
                    const uint2 wj = ws[j];
                    a0 += h * wj.x;
                    a1 += h * wj.y;
                }
                const uint64_t x = mod_halves(a0, a1, q, magic);
                const uint2 yh = ys[i];
                const uint64_t yi = yh.x + ((uint64_t)yh.y << 16);
                out[b * ldout + i] = (int64_t)(x >= yi ? x - yi : x + (q - yi));
            }
        }
    } else {
        typedef __int128 i128;
        uint64_t* y = tag_sh;
        uint64_t* w = tag_sh + n;
        // |p| < 2^53, base^s mod q < 2^62, k <= 64 terms fit 128 bits
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            i128 acc = 0;
            for (int s = 0; s < (P ? k : 0); ++s) acc += (i128)(long long)pb[(long)i * k + s] * (i128)gpow[s];
            const i128 r = acc % (i128)q;
            y[i] = (uint64_t)(r < 0 ? r + (i128)q : r);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            uint64_t hy = y[i];
            if (h0) {
                ModAcc a;
#pragma unroll 4
                for (int j = 0; j < n; ++j) a.mac(h0[(long)j * n + i], y[j]);
                hy = a.reduce(q);
            }
            const uint64_t sum = (uint64_t)V[b * ldv + i] + hy;
            w[i] = sum >= q ? sum - q : sum;
        }
        __syncthreads();
        if constexpr (POLY) {
            poly_mulmod<W>(hi, w, w + n, xr, q, magic, n, [&](int i, uint64_t x) {
                const uint64_t yi = y[i];
                out[b * ldout + i] = (int64_t)(x >= yi ? x - yi : x + (q - yi));
            });
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                ModAcc a;
#pragma unroll 4
                for (int j = 0; j < n; ++j) a.mac(hi[(long)j * n + i], w[j]);
                const uint64_t x = a.reduce(q), yi = y[i];
                out[b * ldout + i] = (int64_t)(x >= yi ? x - yi : x + (q - yi));
            }
        }
    }
}

template <typename W, bool POLY>
cudaError_t launch_tag_syndrome(const int64_t* V, long ldv, const double* P, long ldp, int m_bar, const int32_t* tidx,
                                int ntags, const void* tab, const void* h0, const uint64_t* gpow, uint64_t q, int n, int k,
                                int B, int64_t* out, long ldout, int* flag, const void* xr, cudaStream_t stream) {
    const int threads = n >= 512 ? 512 : (n + 31) / 32 * 32;
    // y and w; the polynomial form adds the 2n - 1 words of the product's scratch
    const size_t smem = (size_t)(POLY ? 4 : 2) * n * sizeof(uint64_t);
    cudaError_t e;
    if (smem > 48 * 1024 &&
        (e = cudaFuncSetAttribute(tag_syndrome_kernel<W, POLY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return e;
    tag_syndrome_kernel<W, POLY><<<B, threads, smem, stream>>>(V, ldv, P, ldp, m_bar, tidx, ntags, (const W*)tab,
                                                                         (const W*)h0, gpow, q, qf_barrett_magic(q), n, k, out,
                                                                         ldout, flag, (const W*)xr);
    return cudaGetLastError();
}
}  // namespace

cudaError_t qf_launch_tag_syndrome(const int64_t* V, long ldv, const double* P, long ldp, int m_bar, const int32_t* tidx,
                                   int ntags, const void* tab, const void* h0, int word_bytes, const uint64_t* gpow,
                                   unsigned long long q, int n, int k, int B, int64_t* out, long ldout, int* flag,
                                   cudaStream_t stream, const void* xr) {
    if (B <= 0) return cudaSuccess;
    if (n < 1 || k < 1 || k > 64 || q < 2 || q >= (1ull << 62) || (word_bytes != 4 && word_bytes != 8) ||
        (word_bytes == 4 && (q > (1ull << 32) || n > (1 << 14))))
        return cudaErrorInvalidValue;
    if (word_bytes == 4)
        return xr ? launch_tag_syndrome<uint32_t, true>(V, ldv, P, ldp, m_bar, tidx, ntags, tab, h0, gpow, q, n, k, B, out, ldout, flag, xr, stream)
                  : launch_tag_syndrome<uint32_t, false>(V, ldv, P, ldp, m_bar, tidx, ntags, tab, h0, gpow, q, n, k, B, out, ldout, flag, xr, stream);
    return xr ? launch_tag_syndrome<uint64_t, true>(V, ldv, P, ldp, m_bar, tidx, ntags, tab, h0, gpow, q, n, k, B, out, ldout, flag, xr, stream)
              : launch_tag_syndrome<uint64_t, false>(V, ldv, P, ldp, m_bar, tidx, ntags, tab, h0, gpow, q, n, k, B, out, ldout, flag, xr, stream);
}

// ---- per-target tag of f_a (qf_f_a_tagged): u_b += D_t y_b mod q with y_b = G sigma_bot_b, D_t = H_t - H_0, t = tidx[b] -------
// The table D (T x n x n words, column-major as the samp_p table) is n^2 words per tag, far more than the n outputs of a
// target, so the targets are grouped by tag first: a counting sort of the chunk's tag indices (histogram over T + 1 bins,
// the last one for indices outside the table; exclusive scan; scatter into a permutation), each tag's run cut into groups of
// at most QF_F_A_TAG_GROUP targets, one CTA per group.  Every table word a CTA loads serves all targets of its group.
namespace {
constexpr int FA_G = QF_F_A_TAG_GROUP;

// lanes of a warp with the same bin: one atomic per distinct bin; returns the lane's rank among its peers
__device__ __forceinline__ int fa_warp_add(int* ctr, int bin, bool active, int* base) {
    const unsigned act = __ballot_sync(0xFFFFFFFFu, active);
    if (!active) return 0;
    const unsigned peers = __match_any_sync(act, bin);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int b0 = 0;
    if (lane == leader) b0 = atomicAdd(ctr + bin, __popc(peers));
    *base = __shfl_sync(peers, b0, leader);
    return __popc(peers & ((1u << lane) - 1));
}

__global__ void fa_tag_hist_kernel(const int32_t* __restrict__ tidx, int B, int ntags, int* __restrict__ hist, int* flag) {
    for (int b0 = blockIdx.x * blockDim.x; b0 < B; b0 += gridDim.x * blockDim.x) {
        const int b = b0 + threadIdx.x;
        int bin = ntags;
        if (b < B) {
            const int t = tidx[b];
            if (t >= 0 && t < ntags) bin = t;
            else if (flag) atomicOr(flag, QF_FLAG_TAG_INDEX);
        }
        int base;
        fa_warp_add(hist, bin, b < B, &base);
    }
}

// one CTA: off[t] = sum_{t' < t} hist[t'] (hist becomes the scatter cursor), gstart[t] = sum_{t' < t} ceil(hist[t'] / G) over
// the valid bins, gstart[ntags] = number of groups
__global__ void __launch_bounds__(1024) fa_tag_scan_kernel(int* __restrict__ hist, int ntags, int* __restrict__ off,
                                                           int* __restrict__ gstart) {
    __shared__ int wc[32], wg[32];
    const int nb = ntags + 1, per = (nb + blockDim.x - 1) / blockDim.x;
    const int t0 = min(nb, (int)threadIdx.x * per), t1 = min(nb, t0 + per);
    int c = 0, g = 0;
    for (int t = t0; t < t1; ++t) {
        const int h = hist[t];
        c += h;
        if (t < ntags) g += (h + FA_G - 1) / FA_G;
    }
    // block-wide exclusive scan of (c, g)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ic = c, ig = g;
    for (int d = 1; d < 32; d <<= 1) {
        const int xc = __shfl_up_sync(0xFFFFFFFFu, ic, d), xg = __shfl_up_sync(0xFFFFFFFFu, ig, d);
        if (lane >= d) { ic += xc; ig += xg; }
    }
    if (lane == 31) { wc[warp] = ic; wg[warp] = ig; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        int vc = lane < nw ? wc[lane] : 0, vg = lane < nw ? wg[lane] : 0;
        for (int d = 1; d < 32; d <<= 1) {
            const int xc = __shfl_up_sync(0xFFFFFFFFu, vc, d), xg = __shfl_up_sync(0xFFFFFFFFu, vg, d);
            if (lane >= d) { vc += xc; vg += xg; }
        }
        if (lane < nw) { wc[lane] = vc; wg[lane] = vg; }
    }
    __syncthreads();
    int rc = ic - c + (warp ? wc[warp - 1] : 0), rg = ig - g + (warp ? wg[warp - 1] : 0);
    for (int t = t0; t < t1; ++t) {
        const int h = hist[t];
        hist[t] = rc;
        off[t] = rc;
        if (t < ntags) gstart[t] = rg;
        rc += h;
        if (t < ntags) rg += (h + FA_G - 1) / FA_G;
    }
    if (threadIdx.x == blockDim.x - 1) gstart[ntags] = rg;
}

__global__ void fa_tag_scatter_kernel(const int32_t* __restrict__ tidx, int B, int ntags, int* __restrict__ cur,
                                      int* __restrict__ perm) {
    for (int b0 = blockIdx.x * blockDim.x; b0 < B; b0 += gridDim.x * blockDim.x) {
        const int b = b0 + threadIdx.x;
        int bin = ntags;
        if (b < B) {
            const int t = tidx[b];
            if (t >= 0 && t < ntags) bin = t;
        }
        int base = 0;
        const int r = fa_warp_add(cur, bin, b < B, &base);
        if (b < B) perm[base + r] = b;
    }
}

// One CTA per group of at most FA_G targets of one tag t.  FA_G = 1 (CTA b is target b, no sort) is not built by the
// library: scripts/bench_f_a_tagged.py builds it to measure what the grouping gains (DESIGN 4.9).  y_g = G sigma_bot of the
// group's targets sits in shared memory as [j][g]; thread i owns rows i, i + blockDim, ... and loads each word D_t[i][j] once
// for all targets.  Exact for every q < 2^62 and int32 sigma (sigma is reduced mod q first):
//  - W = uint32_t (q <= 2^32, n <= 2^14): y as 16-bit halves, a row sum of n products word x half < 2^48 stays below 2^62
//    (mod_halves), as in tag_syndrome_kernel;
//  - W = uint64_t: 192-bit row sums (ModAcc).
// Unused slots of a partial group hold y = 0 and are not written.
template <typename W>
__global__ void __launch_bounds__(512) fa_tag_correct_kernel(const int32_t* __restrict__ sigma, long lds, int m_bar,
                                                             const int32_t* __restrict__ tidx, int ntags,
                                                             const int* __restrict__ perm, const int* __restrict__ off,
                                                             const int* __restrict__ gstart, const W* __restrict__ tab,
                                                             const uint64_t* __restrict__ gpow, uint64_t q, uint64_t magic,
                                                             int n, int k, int64_t* __restrict__ u, long ldu, int* flag) {
    extern __shared__ uint64_t fa_sh[];
    __shared__ int s_t, s_cnt, s_row[FA_G];
    if (threadIdx.x == 0) {
        int cnt = 0, t = 0;
        if constexpr (FA_G == 1) {
            t = tidx[blockIdx.x];
            if (t >= 0 && t < ntags) {
                cnt = 1;
                s_row[0] = blockIdx.x;
            } else if (flag) {
                atomicOr(flag, QF_FLAG_TAG_INDEX);
            }
        } else {
            const int g = blockIdx.x;
            if (g < gstart[ntags]) {  // the grid is an upper bound on the groups the sort made
                int lo = 0, hi = ntags - 1;  // last t with gstart[t] <= g
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (gstart[mid] <= g) lo = mid;
                    else hi = mid - 1;
                }
                t = lo;
                const int first = off[t] + (g - gstart[t]) * FA_G;
                cnt = min(FA_G, off[t + 1] - first);
                for (int c = 0; c < cnt; ++c) s_row[c] = perm[first + c];
            }
        }
        s_t = t;
        s_cnt = cnt;
    }
    __syncthreads();
    const int cnt = s_cnt;
    if (!cnt) return;
    const W* d = tab + (long)s_t * n * n;
    if constexpr (sizeof(W) == 4) {
        uint2* ys = reinterpret_cast<uint2*>(fa_sh);
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            for (int c = 0; c < FA_G; ++c) {
                uint2 v = make_uint2(0, 0);
                if (c < cnt) {
                    const int32_t* sb = sigma + (long)s_row[c] * lds + m_bar + (long)i * k;
                    uint64_t a0 = 0, a1 = 0;
                    for (int s = 0; s < k; ++s) {
                        const uint64_t sm = mod_i64_barrett((long long)sb[s], q, magic), gs = gpow[s];
                        a0 += sm * (gs & 0xFFFF);
                        a1 += sm * (gs >> 16);
                    }
                    v = halves(mod_halves(a0, a1, q, magic));
                }
                ys[i * FA_G + c] = v;
            }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            uint64_t a0[FA_G], a1[FA_G];
#pragma unroll
            for (int c = 0; c < FA_G; ++c) a0[c] = a1[c] = 0;
#pragma unroll 4
            for (int j = 0; j < n; ++j) {
                const uint64_t h = d[(long)j * n + i];
#pragma unroll
                for (int c = 0; c < FA_G; ++c) {
                    const uint2 yj = ys[j * FA_G + c];
                    a0[c] += h * yj.x;
                    a1[c] += h * yj.y;
                }
            }
#pragma unroll
            for (int c = 0; c < FA_G; ++c)
                if (c < cnt) {
                    int64_t* ub = u + (long)s_row[c] * ldu + i;
                    const uint64_t sum = (uint64_t)*ub + mod_halves(a0[c], a1[c], q, magic);
                    *ub = (int64_t)(sum >= q ? sum - q : sum);
                }
        }
    } else {
        uint64_t* ys = fa_sh;
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            for (int c = 0; c < FA_G; ++c) {
                uint64_t v = 0;
                if (c < cnt) {
                    const int32_t* sb = sigma + (long)s_row[c] * lds + m_bar + (long)i * k;
                    ModAcc a;
                    for (int s = 0; s < k; ++s) a.mac(sb[s] < 0 ? (uint64_t)((long long)sb[s] + (long long)q) : (uint64_t)sb[s], gpow[s]);
                    v = a.reduce(q);
                }
                ys[i * FA_G + c] = v;
            }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            ModAcc a[FA_G];
#pragma unroll 2
            for (int j = 0; j < n; ++j) {
                const uint64_t h = d[(long)j * n + i];
#pragma unroll
                for (int c = 0; c < FA_G; ++c) a[c].mac(h, ys[j * FA_G + c]);
            }
#pragma unroll
            for (int c = 0; c < FA_G; ++c)
                if (c < cnt) {
                    int64_t* ub = u + (long)s_row[c] * ldu + i;
                    const uint64_t sum = (uint64_t)*ub + a[c].reduce(q);
                    *ub = (int64_t)(sum >= q ? sum - q : sum);
                }
        }
    }
}

inline int fa_sort_grid(int B) { return std::max(1, std::min((B + 255) / 256, 148 * 8)); }

// the y of a group (8 n bytes per target) plus the kernel's static shared memory fit what one block may opt into
cudaError_t fa_smem_fits(int n, bool* fits) {
    cudaFuncAttributes a4, a8;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a4, fa_tag_correct_kernel<uint32_t>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a8, fa_tag_correct_kernel<uint64_t>)) != cudaSuccess) return e;
    int dev = 0, optin = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    *fits = (size_t)n * FA_G * sizeof(uint64_t) + std::max(a4.sharedSizeBytes, a8.sharedSizeBytes) <= (size_t)optin;
    return cudaSuccess;
}
}  // namespace

cudaError_t qf_f_a_tag_supported(int n, int k, int* ok) {
    bool fits = false;
    cudaError_t e = fa_smem_fits(n, &fits);
    if (e != cudaSuccess) return e;
    *ok = n >= 1 && k >= 1 && k <= 64 && n <= (1 << 14) && fits;
    return cudaSuccess;
}

cudaError_t qf_launch_f_a_tag_sort(const int32_t* tidx, int B, int ntags, int* hist, int* off, int* gstart, int* perm,
                                   int* flag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (ntags < 1 || ntags == INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(hist, 0, (size_t)(ntags + 1) * sizeof(int), stream);
    if (e != cudaSuccess) return e;
    fa_tag_hist_kernel<<<fa_sort_grid(B), 256, 0, stream>>>(tidx, B, ntags, hist, flag);
    fa_tag_scan_kernel<<<1, 1024, 0, stream>>>(hist, ntags, off, gstart);
    fa_tag_scatter_kernel<<<fa_sort_grid(B), 256, 0, stream>>>(tidx, B, ntags, hist, perm);
    return cudaGetLastError();
}

cudaError_t qf_launch_f_a_tag_correct(const int32_t* sigma, long lds, int m_bar, const int32_t* tidx, int ntags,
                                      const int* perm, const int* off, const int* gstart, const void* tab, int word_bytes,
                                      const uint64_t* gpow, unsigned long long q, int n, int k, int B, int64_t* u, long ldu,
                                      int* flag, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (n < 1 || k < 1 || k > 64 || q < 2 || q >= (1ull << 62) || (word_bytes != 4 && word_bytes != 8) ||
        (word_bytes == 4 && (q > (1ull << 32) || n > (1 << 14))))
        return cudaErrorInvalidValue;
    bool fits = false;
    cudaError_t e = fa_smem_fits(n, &fits);
    if (e != cudaSuccess) return e;
    if (!fits) return cudaErrorInvalidValue;
    const int threads = n >= 512 ? 512 : (n + 31) / 32 * 32;
    const size_t smem = (size_t)n * FA_G * sizeof(uint64_t);
    const uint64_t magic = qf_barrett_magic(q);
    // groups: sum_t ceil(c_t / G) <= ceil(B / G) + (tags present) -- CTAs past the count the sort wrote exit at once
    const long grid = FA_G == 1 ? (long)B : (long)(B + FA_G - 1) / FA_G + std::min(ntags, B);
    if (word_bytes == 4) {
        if (smem > 48 * 1024 &&
            (e = cudaFuncSetAttribute(fa_tag_correct_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return e;
        fa_tag_correct_kernel<uint32_t><<<(unsigned)grid, threads, smem, stream>>>(sigma, lds, m_bar, tidx, ntags, perm, off, gstart,
                                                                        (const uint32_t*)tab, gpow, (uint64_t)q, magic, n, k,
                                                                        u, ldu, flag);
    } else {
        if (smem > 48 * 1024 &&
            (e = cudaFuncSetAttribute(fa_tag_correct_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return e;
        fa_tag_correct_kernel<uint64_t><<<(unsigned)grid, threads, smem, stream>>>(sigma, lds, m_bar, tidx, ntags, perm, off, gstart,
                                                                        (const uint64_t*)tab, gpow, (uint64_t)q, magic, n, k,
                                                                        u, ldu, flag);
    }
    return cudaGetLastError();
}

// ---- tags in polynomial form (qf_set_tag_table_poly, qf_set_f_a_tags_poly; DESIGN 4.10) ---------------------------------
// H_t = rot_f(h_t), column c = coeffs(h_t X^c mod f).  rot_f(a) b = a * b mod f and rot_f(h)^-1 = rot_f(h^-1), so a tag is
// n words, inverting it costs O(n^2) and applying it is one poly_mulmod.
namespace {
typedef unsigned __int128 u128;

__device__ __forceinline__ uint64_t mulmod_p(uint64_t a, uint64_t b, uint64_t p) {
    return p <= (1ull << 32) ? (a * b) % p : (uint64_t)((u128)a * b % p);
}
// a^-1 mod p for a unit a (extended Euclid on integers; |t| <= p < 2^62)
__device__ uint64_t inv_mod_p(uint64_t a, uint64_t p) {
    long long t = 0, nt = 1;
    uint64_t r = p, nr = a;
    while (nr) {
        const uint64_t qq = r / nr;
        const long long tt = t - (long long)qq * nt;
        t = nt;
        nt = tt;
        const uint64_t rr = r - qq * nr;
        r = nr;
        nr = rr;
    }
    return t < 0 ? (uint64_t)(t + (long long)p) : (uint64_t)t;
}

// rows X^{n+j} mod (f, q), j < n - 1: row 0 = -f, row j+1 = X row j mod f = (row j shifted up) - row_j[n-1] f.  One CTA; the
// rows are built in place in the table (a barrier per row makes row j visible to the block).
template <typename W>
__global__ void __launch_bounds__(512) poly_xpow_kernel(const uint64_t* __restrict__ fq, int n, uint64_t q, W* xr) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) xr[i] = (W)(fq[i] ? q - fq[i] : 0);
    for (int j = 0; j + 1 < n - 1; ++j) {
        __syncthreads();
        const W* row = xr + (long)j * n;
        const uint64_t top = row[n - 1];
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint64_t lo = i ? (uint64_t)row[i - 1] : 0, d = (uint64_t)((u128)top * fq[i] % q);
            xr[(long)(j + 1) * n + i] = (W)(lo >= d ? lo - d : lo + (q - d));
        }
    }
}

// tab[x] = tags[x] mod q in words of W (count words, any sign)
template <typename W>
__global__ void poly_tag_pack_kernel(const int64_t* __restrict__ tags, long count, uint64_t q, W* __restrict__ tab) {
    for (long x = (long)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (long)gridDim.x * blockDim.x) {
        const long long v = tags[x] % (long long)q;
        tab[x] = (W)(v < 0 ? v + (long long)q : v);
    }
}

// One CTA per tag h (count tags of n int64 coefficients, any sign), q = p^e:
//  1. h mod q, and extended Euclid in F_p[X] against f mod p, one elimination step A -= c X^(dA - dB) B per iteration
//     (at most 2n; thread 0 keeps the degrees and the one scalar inverse per remainder, the threads the O(n) update), with
//     the cofactors tA, tB: tA h = A, tB h = B mod (f, p).  B a non-zero constant: s = tB / B mod p; B = 0: not a unit.
//  2. Newton s <- s (2 - h s) mod (f, q), `lifts` = ceil(log2 e) times (the error 1 - h s squares each time).
//  3. h s = 1 mod (f, q) is checked exactly before s is stored (n words of W per tag).
// fail[t] = 0 on success, 1 when h is not a unit (the tag's words are then left unwritten).
template <typename W>
__global__ void __launch_bounds__(256) poly_tag_inverse_kernel(const int64_t* __restrict__ tags, int n,
                                                               const uint64_t* __restrict__ fq, const W* __restrict__ xr,
                                                               uint64_t q, uint64_t magic, uint64_t p, int lifts,
                                                               W* __restrict__ tab, int* __restrict__ fail) {
    typedef typename PolySV<W>::T SV;
    extern __shared__ uint64_t pi_sh[];
    // Euclid: two remainders and two cofactors of n + 1 coefficients; Newton: h, s (words), s and u (PolySV), product scratch
    uint64_t* rem[2] = {pi_sh, pi_sh + (n + 1)};
    uint64_t* cof[2] = {pi_sh + 2 * (n + 1), pi_sh + 3 * (n + 1)};
    uint64_t* h = pi_sh + 4 * (n + 1);
    uint64_t* s = h + n;
    SV* s_sv = reinterpret_cast<SV*>(s + n);
    SV* u_sv = s_sv + n;
    SV* c = u_sv + n;
    __shared__ int s_op, s_which, s_da, s_db, s_sh;
    __shared__ uint64_t s_cc, s_ilc;
    const long t = blockIdx.x;
    const int64_t* ht = tags + t * n;
    for (int i = threadIdx.x; i <= n; i += blockDim.x) {
        uint64_t hv = 0;
        if (i < n) {
            const long long v = ht[i] % (long long)q;
            hv = (uint64_t)(v < 0 ? v + (long long)q : v);
            h[i] = hv;
        }
        rem[0][i] = i < n ? fq[i] % p : 1 % p;
        rem[1][i] = hv % p;
        cof[0][i] = 0;
        cof[1][i] = i == 0;
    }
    __syncthreads();
    // control (thread 0): op 0 = eliminate rem[which] -= cc X^sh rem[1 - which]; 1 = rem[1 - which] is a unit; 2 = not a unit
    auto plan = [&](int da, int db, int which, bool fresh_b) {
        const uint64_t* A = rem[which];
        const uint64_t* B = rem[which ^ 1];
        if (da < db) {  // the remainder fell below the divisor: swap roles
            which ^= 1;
            const int x = da;
            da = db;
            db = x;
            A = rem[which];
            B = rem[which ^ 1];
            fresh_b = true;
        }
        s_which = which;
        s_da = da;
        s_db = db;
        if (db <= 0) {
            s_op = db == 0 ? 1 : 2;
            return;
        }
        if (fresh_b) s_ilc = inv_mod_p(B[db], p);
        s_cc = mulmod_p(A[da], s_ilc, p);
        s_sh = da - db;
        s_op = 0;
    };
    if (threadIdx.x == 0) {
        int db = n - 1;
        while (db >= 0 && rem[1][db] == 0) --db;
        plan(n, db, 0, true);
    }
    for (;;) {
        __syncthreads();
        const int op = s_op;
        if (op) break;
        const int which = s_which, db = s_db, sh = s_sh;
        const uint64_t cc = s_cc;
        uint64_t *A = rem[which], *tA = cof[which];
        const uint64_t *B = rem[which ^ 1], *tB = cof[which ^ 1];
        for (int i = threadIdx.x; i + sh <= n; i += blockDim.x) {
            if (i <= db) {
                const uint64_t d = mulmod_p(cc, B[i], p), a = A[i + sh];
                A[i + sh] = a >= d ? a - d : a + (p - d);
            }
            const uint64_t d = mulmod_p(cc, tB[i], p), a = tA[i + sh];
            tA[i + sh] = a >= d ? a - d : a + (p - d);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int da = s_da - 1;  // A[s_da] is now 0
            while (da >= 0 && A[da] == 0) --da;
            plan(da, db, which, false);
        }
    }
    const bool unit = s_op == 1;
    if (!unit) {
        if (threadIdx.x == 0) fail[t] = 1;
        return;
    }
    {
        const int wb = s_which ^ 1;
        const uint64_t ib = inv_mod_p(rem[wb][0], p);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint64_t v = mulmod_p(cof[wb][i], ib, p);
            s[i] = v;
            s_sv[i] = PolySV<W>::put(v);
        }
    }
    __syncthreads();
    const uint64_t two = 2 % q;
    for (int it = 0; it < lifts; ++it) {
        poly_mulmod<W>(h, s_sv, c, xr, q, magic, n, [&](int i, uint64_t r) {  // u = 2 - h s
            const uint64_t w = i == 0 ? two : 0;
            u_sv[i] = PolySV<W>::put(w >= r ? w - r : w + (q - r));
        });
        __syncthreads();
        poly_mulmod<W>(s, u_sv, c, xr, q, magic, n, [&](int i, uint64_t r) {  // s <- s u
            s[i] = r;
            s_sv[i] = PolySV<W>::put(r);
        });
        __syncthreads();
    }
    bool ok = true;
    poly_mulmod<W>(h, s_sv, c, xr, q, magic, n, [&](int i, uint64_t r) { ok = ok && r == (i == 0 ? 1 % q : 0); });
    ok = __syncthreads_and(ok);
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (ok) tab[t * n + i] = (W)s[i];
    if (threadIdx.x == 0) fail[t] = ok ? 0 : 1;
}

// f_a in polynomial form, one CTA per target b (t = tidx[b]): u_b += h_t * y_b mod (f, q) - H_0 y_b, y_b = G sigma_bot_b.
// n words per tag need no grouping by tag.  h0_kind: 0 H_0 = 0, 1 H_0 = I, 2 dense H_0 (n x n column-major words of W, the
// same for every target, L2-resident).  An index outside the table never addresses it: the row keeps A sigma and the flag
// bit is set.
template <typename W>
__global__ void __launch_bounds__(512) fa_tag_poly_kernel(const int32_t* __restrict__ sigma, long lds, int m_bar,
                                                          const int32_t* __restrict__ tidx, int ntags, const W* __restrict__ tab,
                                                          const W* __restrict__ xr, const W* __restrict__ h0, int h0_kind,
                                                          const uint64_t* __restrict__ gpow, uint64_t q, uint64_t magic, int n,
                                                          int k, int64_t* __restrict__ u, long ldu, int* flag) {
    typedef typename PolySV<W>::T SV;
    extern __shared__ uint64_t fp_sh[];
    const long b = blockIdx.x;
    const int t = tidx[b];
    if (t < 0 || t >= ntags) {
        if (threadIdx.x == 0 && flag) atomicOr(flag, QF_FLAG_TAG_INDEX);
        return;
    }
    SV* ys = reinterpret_cast<SV*>(fp_sh);
    SV* c = ys + n;
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        ys[i] = PolySV<W>::put(gadget_row_mod<W>(sigma + b * lds + m_bar + (long)i * k, gpow, q, magic, k));
    __syncthreads();
    poly_mulmod<W>(tab + (long)t * n, ys, c, xr, q, magic, n, [&](int i, uint64_t r) {
        uint64_t hy = 0;
        if (h0_kind == 1) {
            hy = PolySV<W>::get(ys[i]);
        } else if (h0_kind == 2) {
            if constexpr (sizeof(W) == 4) {
                uint64_t a0 = 0, a1 = 0;
#pragma unroll 4
                for (int j = 0; j < n; ++j) {
                    const uint64_t x = h0[(long)j * n + i];
                    const uint2 yj = ys[j];
                    a0 += x * yj.x;
                    a1 += x * yj.y;
                }
                hy = mod_halves(a0, a1, q, magic);
            } else {
                ModAcc a;
#pragma unroll 2
                for (int j = 0; j < n; ++j) a.mac(h0[(long)j * n + i], ys[j]);
                hy = a.reduce(q);
            }
        }
        int64_t* ub = u + b * ldu + i;
        uint64_t v = (uint64_t)*ub + r;
        v = v >= q ? v - q : v;
        *ub = (int64_t)(v >= hy ? v - hy : v + (q - hy));
    });
}

constexpr size_t poly_inverse_smem(int n) { return ((size_t)4 * (n + 1) + (size_t)6 * n) * sizeof(uint64_t); }
constexpr size_t poly_syndrome_smem(int n) { return (size_t)4 * n * sizeof(uint64_t); }
constexpr size_t poly_fa_smem(int n) { return (size_t)3 * n * sizeof(uint64_t); }

cudaError_t smem_optin(int* optin) {
    int dev = 0;
    cudaError_t e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    return cudaDeviceGetAttribute(optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
}

// static + dynamic shared memory of the kernel within one block's opt-in limit
template <typename K>
cudaError_t smem_fits(K kernel, size_t dyn, int optin, bool* fits) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kernel);
    if (e != cudaSuccess) return e;
    *fits = *fits && dyn + a.sharedSizeBytes <= (size_t)optin;
    return cudaSuccess;
}

template <typename K>
cudaError_t set_smem(K kernel, size_t dyn) {
    return dyn > 48 * 1024 ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn) : cudaSuccess;
}
}  // namespace

cudaError_t qf_poly_tag_supported(int n, int k, int samp_p, int* ok) {
    int optin = 0;
    cudaError_t e = smem_optin(&optin);
    if (e != cudaSuccess) return e;
    bool fits = n >= 1 && k >= 1 && k <= 64 && n <= (1 << 14);
    if (samp_p) {
        if ((e = smem_fits(poly_tag_inverse_kernel<uint32_t>, poly_inverse_smem(n), optin, &fits)) != cudaSuccess) return e;
        if ((e = smem_fits(poly_tag_inverse_kernel<uint64_t>, poly_inverse_smem(n), optin, &fits)) != cudaSuccess) return e;
        if ((e = smem_fits(tag_syndrome_kernel<uint32_t, true>, poly_syndrome_smem(n), optin, &fits)) != cudaSuccess) return e;
        if ((e = smem_fits(tag_syndrome_kernel<uint64_t, true>, poly_syndrome_smem(n), optin, &fits)) != cudaSuccess) return e;
    } else {
        if ((e = smem_fits(fa_tag_poly_kernel<uint32_t>, poly_fa_smem(n), optin, &fits)) != cudaSuccess) return e;
        if ((e = smem_fits(fa_tag_poly_kernel<uint64_t>, poly_fa_smem(n), optin, &fits)) != cudaSuccess) return e;
    }
    *ok = fits;
    return cudaSuccess;
}

cudaError_t qf_launch_poly_xpow(const uint64_t* fq, int n, unsigned long long q, int word_bytes, void* xr, cudaStream_t stream) {
    if (n < 2) return cudaSuccess;  // no row: a product of constants needs no reduction
    const int threads = n >= 512 ? 512 : (n + 31) / 32 * 32;
    if (word_bytes == 4) poly_xpow_kernel<uint32_t><<<1, threads, 0, stream>>>(fq, n, (uint64_t)q, (uint32_t*)xr);
    else poly_xpow_kernel<uint64_t><<<1, threads, 0, stream>>>(fq, n, (uint64_t)q, (uint64_t*)xr);
    return cudaGetLastError();
}

cudaError_t qf_launch_poly_tag_pack(const int64_t* tags, long count, unsigned long long q, int word_bytes, void* tab,
                                    cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    const int grid = grid_for(count, 256, 148 * 8);
    if (word_bytes == 4) poly_tag_pack_kernel<uint32_t><<<grid, 256, 0, stream>>>(tags, count, (uint64_t)q, (uint32_t*)tab);
    else poly_tag_pack_kernel<uint64_t><<<grid, 256, 0, stream>>>(tags, count, (uint64_t)q, (uint64_t*)tab);
    return cudaGetLastError();
}

cudaError_t qf_launch_poly_tag_inverse(const int64_t* tags, int count, int n, const uint64_t* fq, const void* xr,
                                       int word_bytes, unsigned long long q, unsigned long long p, int lifts, void* tab,
                                       int* fail, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    if (n < 1 || q < 2 || q >= (1ull << 62) || p < 2 || q % p || (word_bytes != 4 && word_bytes != 8) ||
        (word_bytes == 4 && (q > (1ull << 32) || n > (1 << 14))))
        return cudaErrorInvalidValue;
    const int threads = n >= 256 ? 256 : (n + 31) / 32 * 32;
    const size_t smem = poly_inverse_smem(n);
    const uint64_t magic = qf_barrett_magic(q);
    cudaError_t e;
    if (word_bytes == 4) {
        if ((e = set_smem(poly_tag_inverse_kernel<uint32_t>, smem)) != cudaSuccess) return e;
        poly_tag_inverse_kernel<uint32_t><<<count, threads, smem, stream>>>(tags, n, fq, (const uint32_t*)xr, (uint64_t)q, magic,
                                                                            (uint64_t)p, lifts, (uint32_t*)tab, fail);
    } else {
        if ((e = set_smem(poly_tag_inverse_kernel<uint64_t>, smem)) != cudaSuccess) return e;
        poly_tag_inverse_kernel<uint64_t><<<count, threads, smem, stream>>>(tags, n, fq, (const uint64_t*)xr, (uint64_t)q, magic,
                                                                            (uint64_t)p, lifts, (uint64_t*)tab, fail);
    }
    return cudaGetLastError();
}

cudaError_t qf_launch_f_a_tag_poly(const int32_t* sigma, long lds, int m_bar, const int32_t* tidx, int ntags, const void* tab,
                                   const void* xr, const void* h0, int h0_kind, int word_bytes, const uint64_t* gpow,
                                   unsigned long long q, int n, int k, int B, int64_t* u, long ldu, int* flag,
                                   cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (n < 1 || k < 1 || k > 64 || q < 2 || q >= (1ull << 62) || (word_bytes != 4 && word_bytes != 8) ||
        (word_bytes == 4 && (q > (1ull << 32) || n > (1 << 14))) || h0_kind < 0 || h0_kind > 2 || (h0_kind == 2 && !h0))
        return cudaErrorInvalidValue;
    const int threads = n >= 512 ? 512 : (n + 31) / 32 * 32;
    const size_t smem = poly_fa_smem(n);
    const uint64_t magic = qf_barrett_magic(q);
    cudaError_t e;
    if (word_bytes == 4) {
        if ((e = set_smem(fa_tag_poly_kernel<uint32_t>, smem)) != cudaSuccess) return e;
        fa_tag_poly_kernel<uint32_t><<<B, threads, smem, stream>>>(sigma, lds, m_bar, tidx, ntags, (const uint32_t*)tab,
                                                                   (const uint32_t*)xr, (const uint32_t*)h0, h0_kind, gpow,
                                                                   (uint64_t)q, magic, n, k, u, ldu, flag);
    } else {
        if ((e = set_smem(fa_tag_poly_kernel<uint64_t>, smem)) != cudaSuccess) return e;
        fa_tag_poly_kernel<uint64_t><<<B, threads, smem, stream>>>(sigma, lds, m_bar, tidx, ntags, (const uint64_t*)tab,
                                                                   (const uint64_t*)xr, (const uint64_t*)h0, h0_kind, gpow,
                                                                   (uint64_t)q, magic, n, k, u, ldu, flag);
    }
    return cudaGetLastError();
}
