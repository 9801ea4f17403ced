// Ring f_a:  u = sum_j a_j * sigma_j  in  Z_q[X]/(X^n + 1)   (gpv_ring.rs:243-247;
// the product is the one rot^-(.) defines, rotation_matrix.rs:41-63).
//
// The product is computed EXACTLY over the integers with a shared-memory
// negacyclic NTT over the Goldilocks prime p = 2^64 - 2^32 + 1 (2^32-th roots of
// unity, reduction by shifts/adds only) and reduced mod q at the very end, so one
// kernel serves every modulus (3329, 7681, 12289, 2^k, 2^31-1 ...) for which
//     npoly * n * (q/2) * max|sigma|  <  2^63
// (the host checks this).  One CTA per target; the key transforms a_hat_j are
// precomputed once; per target: npoly forward NTTs, a pointwise multiply-accumulate
// in the transform domain and ONE inverse NTT.  ||sigma||^2 for check_domain
// (gpv_ring.rs:274-283) is reduced in the same pass.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr uint64_t GP = 0xFFFFFFFF00000001ull;
constexpr uint64_t GEPS = 0xFFFFFFFFull;

__host__ __device__ __forceinline__ uint64_t gl_add(uint64_t a, uint64_t b) {
    uint64_t s = a + b;
    if (s < a) s += GEPS;
    if (s >= GP) s -= GP;
    return s;
}
__host__ __device__ __forceinline__ uint64_t gl_sub(uint64_t a, uint64_t b) {
    uint64_t d = a - b;
    if (a < b) d -= GEPS;
    return d;
}
__device__ __forceinline__ uint64_t gl_mul(uint64_t a, uint64_t b) {
    uint64_t lo = a * b, hi = __umul64hi(a, b);
    uint64_t hh = hi >> 32, hl = hi & GEPS;
    uint64_t t0 = lo - hh;
    if (lo < hh) t0 -= GEPS;
    uint64_t t1 = hl * GEPS;
    uint64_t r = t0 + t1;
    if (r < t1) r += GEPS;
    if (r >= GP) r -= GP;
    return r;
}
inline uint64_t gl_mul_host(uint64_t a, uint64_t b) {
    return (uint64_t)(((unsigned __int128)a * b) % GP);
}
inline uint64_t gl_pow_host(uint64_t a, uint64_t e) {
    uint64_t r = 1;
    while (e) {
        if (e & 1) r = gl_mul_host(r, a);
        a = gl_mul_host(a, a);
        e >>= 1;
    }
    return r;
}

__device__ __forceinline__ uint64_t gl_from_i64(long long v) {
    return v >= 0 ? (uint64_t)v : GP - (uint64_t)(-v);
}

// forward negacyclic NTT (Cooley-Tukey, natural in -> bit-reversed out); nh = n/2 threads
__device__ __forceinline__ void ntt_forward(uint64_t* a, const uint64_t* __restrict__ psi_rev, int n, int t_id,
                                            bool active) {
    int t = n;
    for (int m = 1; m < n; m <<= 1) {
        t >>= 1;
        if (active) {
            int i = t_id / t, r = t_id - i * t;
            int j = 2 * i * t + r;
            uint64_t s = psi_rev[m + i];
            uint64_t u = a[j], v = gl_mul(a[j + t], s);
            a[j] = gl_add(u, v);
            a[j + t] = gl_sub(u, v);
        }
        __syncthreads();
    }
}
// inverse (Gentleman-Sande, bit-reversed in -> natural out), without the 1/n scaling
__device__ __forceinline__ void ntt_inverse(uint64_t* a, const uint64_t* __restrict__ psi_inv_rev, int n, int t_id,
                                            bool active) {
    int t = 1;
    for (int m = n; m > 1; m >>= 1) {
        int h = m >> 1;
        if (active) {
            int i = t_id / t, r = t_id - i * t;
            int j = 2 * i * t + r;
            uint64_t s = psi_inv_rev[h + i];
            uint64_t u = a[j], v = a[j + t];
            a[j] = gl_add(u, v);
            a[j + t] = gl_mul(gl_sub(u, v), s);
        }
        __syncthreads();
        t <<= 1;
    }
}

__global__ void ring_prepare_kernel(const int64_t* __restrict__ a, uint64_t* __restrict__ a_hat, int n,
                                    unsigned long long q, const uint64_t* __restrict__ tw) {
    extern __shared__ uint64_t sm[];
    const int poly = blockIdx.x, t_id = threadIdx.x, nh = n >> 1;
    for (int i = t_id; i < n; i += nh) {
        long long v = (long long)((unsigned long long)a[(long)poly * n + i] % q);
        if ((unsigned long long)v > q / 2) v -= (long long)q;  // centred lift
        sm[i] = gl_from_i64(v);
    }
    __syncthreads();
    ntt_forward(sm, tw, n, t_id, true);
    for (int i = t_id; i < n; i += nh) a_hat[(long)poly * n + i] = sm[i];
}

// KEYED: target b reads the key at a_hat + key_idx[b] npoly n (a table of nkeys keys); an index outside [0, nkeys) sets
// *flag |= QF_FLAG_KEY_INDEX and gives a zero row that is not in the domain, without reading the table.
template <bool KEYED>
__global__ void ring_f_a_kernel(const int32_t* __restrict__ sigma, const uint64_t* __restrict__ a_hat,
                                int64_t* __restrict__ out, unsigned long long* __restrict__ norm2, int B, int npoly,
                                int n, unsigned long long q, const uint64_t* __restrict__ tw,
                                const int32_t* __restrict__ key_idx, int nkeys, int* flag) {
    extern __shared__ uint64_t sm[];
    const int PP = blockDim.y, nh = n >> 1;
    const int t_id = threadIdx.x, y = threadIdx.y;
    uint64_t* work = sm + (size_t)y * n;           // PP x n
    uint64_t* acc = sm + (size_t)PP * n + (size_t)y * n;  // PP x n
    __shared__ unsigned long long nrm_s;
    __shared__ unsigned int nrm_ovf;
    const uint64_t* psi_rev = tw;
    const uint64_t* psi_inv_rev = tw + n;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const uint64_t* key = a_hat;
        if (KEYED) {  // block-uniform branch
            const int t = key_idx[b];
            if (t < 0 || t >= nkeys) {
                if (y == 0) {
                    for (int i = t_id; i < n; i += nh) out[(long)b * n + i] = 0;
                    if (t_id == 0) {
                        if (flag) atomicOr(flag, QF_FLAG_KEY_INDEX);
                        if (norm2) norm2[b] = ~0ull;
                    }
                }
                continue;
            }
            key = a_hat + (long)t * npoly * n;
        }
        if (t_id == 0 && y == 0) { nrm_s = 0; nrm_ovf = 0; }
        for (int i = t_id; i < n; i += nh) acc[i] = 0;
        NormAcc nrm;  // saturating squared norm (common.cuh)
        nrm.clear();
        const int rounds = (npoly + PP - 1) / PP;
        for (int rd = 0; rd < rounds; ++rd) {
            const int j = rd * PP + y;
            const bool active = j < npoly;
            __syncthreads();
            if (active) {
                const int32_t* src = sigma + ((long)b * npoly + j) * n;
                for (int i = t_id; i < n; i += nh) {
                    long long v = src[i];
                    nrm.add_sq(src[i]);
                    work[i] = gl_from_i64(v);
                }
            }
            __syncthreads();
            ntt_forward(work, psi_rev, n, t_id, active);
            if (active) {
                const uint64_t* ah = key + (long)j * n;
                for (int i = t_id; i < n; i += nh) acc[i] = gl_add(acc[i], gl_mul(work[i], ah[i]));
            }
        }
        __syncthreads();
        // reduce the PP partial accumulators into slice 0's work buffer
        uint64_t* res = sm;
        if (y == 0) {
            for (int i = t_id; i < n; i += nh) {
                uint64_t s = 0;
                for (int yy = 0; yy < PP; ++yy) s = gl_add(s, sm[(size_t)PP * n + (size_t)yy * n + i]);
                res[i] = s;
            }
        }
        if (norm2) {
            nrm.warp_reduce();
            if (((t_id + y * nh) & 31) == 0) {
                const unsigned long long old = atomicAdd(&nrm_s, nrm.lo);
                if (nrm.hi || old + nrm.lo < old) atomicOr(&nrm_ovf, 1u);
            }
        }
        __syncthreads();
        ntt_inverse(res, psi_inv_rev, n, t_id, y == 0);
        if (y == 0) {
            const uint64_t n_inv = tw[2 * n];
            for (int i = t_id; i < n; i += nh) {
                uint64_t r = gl_mul(res[i], n_inv);
                unsigned long long m;
                if (r > GP / 2) {  // negative: value = -(p - r)
                    unsigned long long neg = (GP - r) % q;
                    m = neg ? q - neg : 0;
                } else {
                    m = r % q;
                }
                out[(long)b * n + i] = (int64_t)m;
            }
            if (t_id == 0 && norm2) norm2[b] = nrm_ovf ? ~0ull : nrm_s;
        }
        __syncthreads();
    }
}

// O(n^2) fallback: thread per (target, output coefficient), 128-bit accumulation.
// KEYED: as ring_f_a_kernel, with the raw keys at a + key_idx[b] npoly n.
template <bool KEYED>
__global__ void ring_schoolbook_kernel(const int32_t* __restrict__ sigma, const int64_t* __restrict__ a,
                                       int64_t* __restrict__ out, unsigned long long* __restrict__ norm2, int B,
                                       int npoly, int n, unsigned long long q, const int32_t* __restrict__ key_idx,
                                       int nkeys, int* flag) {
    long total = (long)B * n;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        long b = idx / n;
        int i = (int)(idx - b * n);
        const int64_t* key = a;
        if (KEYED) {
            const int t = key_idx[b];
            if (t < 0 || t >= nkeys) {
                out[b * n + i] = 0;
                if (i == 0) {
                    if (flag) atomicOr(flag, QF_FLAG_KEY_INDEX);
                    if (norm2) norm2[b] = ~0ull;
                }
                continue;
            }
            key = a + (long)t * npoly * n;
        }
        __int128 acc = 0;
        NormAcc nrm;
        nrm.clear();
        for (int j = 0; j < npoly; ++j) {
            const int32_t* s = sigma + ((long)b * npoly + j) * n;
            const int64_t* aj = key + (long)j * n;
            for (int t = 0; t < n; ++t) {
                // coefficient i gets a[t] * s[i-t] (t <= i) and -a[t] * s[n+i-t] (t > i)
                long long sv = (t <= i) ? (long long)s[i - t] : -(long long)s[n + i - t];
                acc += (__int128)aj[t] * sv;
            }
            if (i == 0 && norm2)
                for (int t = 0; t < n; ++t) nrm.add_sq(s[t]);
        }
        out[b * n + i] = (int64_t)mod_i128(acc, q);
        if (i == 0 && norm2) norm2[b] = nrm.value();
    }
}

// Keys of ring TrapGen (gadget_ring.rs:74-78), count at once: A_t = [1 | a_bar_t | g^t - (a_bar_t r_t + e_t)] with
// ar = a_bar_t r_{t,j} mod q (count x k x n), e (count x k x n), gpow[j] = base^j mod q; out count x (k+2) x n.
__global__ void ring_trap_assemble_kernel(const int64_t* __restrict__ a_bar, const int64_t* __restrict__ ar,
                                          const int32_t* __restrict__ e, const uint64_t* __restrict__ gpow,
                                          int64_t* __restrict__ out, long count, int k, int n, unsigned long long q) {
    const long per = (long)(k + 2) * n, total = count * per;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long t = idx / per;
        const long rem = idx - t * per;
        const int row = (int)(rem / n), i = (int)(rem - (long)row * n);
        unsigned long long v;
        if (row == 0) {
            v = (i == 0) ? 1 % q : 0;
        } else if (row == 1) {
            v = (unsigned long long)a_bar[t * n + i] % q;
        } else {
            const long src = (t * k + (row - 2)) * n + i;
            // g_j - ar - e with ar in [0, q), |e| < 2^31: |value| < 2^63
            long long x = (i == 0 ? (long long)gpow[row - 2] : 0) - ar[src] - (long long)e[src];
            long long m = x % (long long)q;
            v = (unsigned long long)(m < 0 ? m + (long long)q : m);
        }
        out[idx] = (int64_t)v;
    }
}

}  // namespace

cudaError_t qf_launch_ring_f_a_schoolbook(const int32_t* sigma, const int64_t* a, int64_t* out,
                                          unsigned long long* norm2, int B, int npoly, int n, unsigned long long q,
                                          cudaStream_t stream, const int32_t* key_idx, int nkeys, int* flag) {
    if (B <= 0) return cudaSuccess;
    long long total = (long long)B * n;
    long long g = (total + 127) / 128;
    if (g > 148 * 16) g = 148 * 16;
    if (key_idx)
        ring_schoolbook_kernel<true><<<(int)g, 128, 0, stream>>>(sigma, a, out, norm2, B, npoly, n, q, key_idx, nkeys, flag);
    else
        ring_schoolbook_kernel<false><<<(int)g, 128, 0, stream>>>(sigma, a, out, norm2, B, npoly, n, q, nullptr, 0, nullptr);
    return cudaGetLastError();
}

cudaError_t qf_launch_ring_trap_assemble(const int64_t* a_bar, const int64_t* ar, const int32_t* e, const uint64_t* gpow,
                                         int64_t* out, long count, int k, int n, unsigned long long q, cudaStream_t stream) {
    if (count <= 0) return cudaSuccess;
    long long total = (long long)count * (k + 2) * n;
    long long g = (total + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    ring_trap_assemble_kernel<<<(int)g, 256, 0, stream>>>(a_bar, ar, e, gpow, out, count, k, n, q);
    return cudaGetLastError();
}

void qf_ring_make_tables(int n, uint64_t* host_out) {
    int logn = 0;
    while ((1 << logn) < n) ++logn;
    const uint64_t psi = gl_pow_host(7, (GP - 1) / (2ull * (uint64_t)n));
    const uint64_t psi_inv = gl_pow_host(psi, GP - 2);
    for (int k = 0; k < n; ++k) {
        int r = 0;
        for (int bit = 0; bit < logn; ++bit)
            if (k & (1 << bit)) r |= 1 << (logn - 1 - bit);
        host_out[k] = gl_pow_host(psi, (uint64_t)r);
        host_out[n + k] = gl_pow_host(psi_inv, (uint64_t)r);
    }
    host_out[2 * n] = gl_pow_host((uint64_t)n, GP - 2);
}

cudaError_t qf_launch_ring_prepare(const int64_t* a, uint64_t* a_hat, long npoly, int n, unsigned long long q,
                                   const uint64_t* tw, cudaStream_t stream) {
    if (npoly <= 0) return cudaSuccess;
    if (n < 2 || n > 2048 || (n & (n - 1))) return cudaErrorInvalidValue;
    if (npoly > 0x7fffffffL) return cudaErrorInvalidValue;
    ring_prepare_kernel<<<(unsigned)npoly, n / 2, (size_t)n * 8, stream>>>(a, a_hat, n, q, tw);
    return cudaGetLastError();
}

cudaError_t qf_launch_ring_f_a(const int32_t* sigma, const uint64_t* a_hat, int64_t* out, unsigned long long* norm2,
                               int B, int npoly, int n, unsigned long long q, const uint64_t* tw,
                               cudaStream_t stream, const int32_t* key_idx, int nkeys, int* flag) {
    if (B <= 0) return cudaSuccess;
    if (n < 2 || n > 2048 || (n & (n - 1))) return cudaErrorInvalidValue;
    int nh = n / 2;
    int pp = 256 / nh;
    if (pp < 1) pp = 1;
    if (pp > npoly) pp = npoly;
    if (pp > 8) pp = 8;
    dim3 block(nh, pp);
    size_t smem = (size_t)2 * pp * n * 8;
    static size_t configured_dev[QF_MAX_DEVICES][2] = {};
    size_t& configured = configured_dev[qf_device_slot()][key_idx ? 1 : 0];
    if (smem > 48 * 1024 && smem > configured) {
        cudaError_t e = key_idx ? cudaFuncSetAttribute(ring_f_a_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                : cudaFuncSetAttribute(ring_f_a_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = smem;
    }
    int grid = B < 148 * 8 ? B : 148 * 8;
    if (key_idx)
        ring_f_a_kernel<true><<<grid, block, smem, stream>>>(sigma, a_hat, out, norm2, B, npoly, n, q, tw, key_idx, nkeys, flag);
    else
        ring_f_a_kernel<false><<<grid, block, smem, stream>>>(sigma, a_hat, out, norm2, B, npoly, n, q, tw, nullptr, 0, nullptr);
    return cudaGetLastError();
}
