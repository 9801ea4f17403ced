// Ring f_a for NTT-friendly word-size moduli (q prime < 2^16), e.g. q = 3329, 7681, 12289:
//   u = sum_j a_j * sigma_j  in  Z_q[X]/(X^n + 1)     (gpv_ring.rs:243-247, rotation_matrix.rs:41-63)
// computed directly mod q with a register/shuffle NTT -- one WARP per target, no shared-memory
// traffic for the data and no block barriers:
//   * 2n | q-1 (7681, 12289 at n = 256): complete negacyclic NTT, pointwise products;
//   * only n | q-1 (3329 at n = 256, the FIPS 203 modulus): X^n + 1 splits into n/2 quadratics
//     X^2 - zeta_i; the transform is two interleaved size-n/2 negacyclic NTTs on the even / odd
//     coefficients and products are degree-1 "base multiplications" mod X^2 - zeta_i.
// Both are exact ring arithmetic mod q, hence bit-exact against the reference product.
// Element e of a size-N' sequence lives in register r = e / 32 of lane e % 32: butterflies with stride
// >= 32 are register-to-register, strides 16..1 use one __shfl_xor each.
#include <vector>

#include "common.cuh"
#include "domain_code.cuh"
#include "kernels.h"

namespace {

struct SmallRing {
    uint32_t q, barrett;  // barrett = floor(2^32 / q)
    int n, d, np;         // d = 1 (complete) or 2 (quadratic factors); np = n / d = NTT length
    uint32_t np_inv;      // np^-1 mod q
};

__device__ __forceinline__ uint32_t red(uint32_t x, const SmallRing& R) {  // x < 2^32 -> [0, q)
    uint32_t t = __umulhi(x, R.barrett);
    uint32_t r = x - t * R.q;
    return r >= R.q ? r - R.q : r;
}
__device__ __forceinline__ uint32_t mulq(uint32_t a, uint32_t b, const SmallRing& R) { return red(a * b, R); }
__device__ __forceinline__ uint32_t addq(uint32_t a, uint32_t b, const SmallRing& R) {
    uint32_t s = a + b;
    return s >= R.q ? s - R.q : s;
}
__device__ __forceinline__ uint32_t subq(uint32_t a, uint32_t b, const SmallRing& R) { return a >= b ? a - b : a + R.q - b; }

// tables (global, L1-resident): [0, np) psi_rev, [np, 2np) psi_inv_rev, [2np, 3np) zeta of factor p (d = 2)
template <int EPL>
__device__ __forceinline__ void ntt_fwd(uint32_t (&v)[EPL], const uint32_t* __restrict__ tw, int lane, const SmallRing& R) {
    constexpr int NP = EPL * 32;
    // strides >= 32: pairs live in the same lane
#pragma unroll
    for (int t = NP / 2; t >= 32; t >>= 1) {
        const int m = NP / (2 * t), tr = t / 32;
#pragma unroll
        for (int r = 0; r < EPL; ++r) {
            if ((r / tr) & 1) continue;  // r is the lower element of its pair
            const uint32_t s = tw[m + r / (2 * tr)];
            const uint32_t u = v[r], w = mulq(v[r + tr], s, R);
            v[r] = addq(u, w, R);
            v[r + tr] = subq(u, w, R);
        }
    }
#pragma unroll
    for (int t = 16; t >= 1; t >>= 1) {
        const int m = NP / (2 * t);
        const bool upper = lane & t;
#pragma unroll
        for (int r = 0; r < EPL; ++r) {
            const int e = r * 32 + lane;
            const uint32_t s = tw[m + e / (2 * t)];
            const uint32_t other = __shfl_xor_sync(0xffffffffu, v[r], t);
            const uint32_t w = mulq(upper ? v[r] : other, s, R);
            v[r] = upper ? subq(other, w, R) : addq(v[r], w, R);
        }
    }
}

template <int EPL>
__device__ __forceinline__ void ntt_inv(uint32_t (&v)[EPL], const uint32_t* __restrict__ twi, int lane, const SmallRing& R) {
    constexpr int NP = EPL * 32;
#pragma unroll
    for (int t = 1; t <= 16; t <<= 1) {
        const int h = NP / (2 * t);
        const bool upper = lane & t;
#pragma unroll
        for (int r = 0; r < EPL; ++r) {
            const int e = r * 32 + lane;
            const uint32_t s = twi[h + e / (2 * t)];
            const uint32_t other = __shfl_xor_sync(0xffffffffu, v[r], t);
            v[r] = upper ? mulq(subq(other, v[r], R), s, R) : addq(v[r], other, R);
        }
    }
#pragma unroll
    for (int t = 32; t <= NP / 2; t <<= 1) {
        const int h = NP / (2 * t), tr = t / 32;
#pragma unroll
        for (int r = 0; r < EPL; ++r) {
            if ((r / tr) & 1) continue;
            const uint32_t s = twi[h + r / (2 * tr)];
            const uint32_t u = v[r], w = v[r + tr];
            v[r] = addq(u, w, R);
            v[r + tr] = mulq(subq(u, w, R), s, R);
        }
    }
}

// KEYED: row b reads the key at a_hat + key_idx[b] npoly n (a table of nkeys keys); an index outside [0, nkeys) sets
// *flag |= QF_FLAG_KEY_INDEX and gives a zero row that is not in the domain, without reading the table.  The keyed form
// asks for 4 blocks per SM at 128-point tiles (the 3329 / n = 256 case): without that bound ptxas spills a register.
// PACKED (keyed only): sigma is unused and row b is the slot b of pk (DESIGN 4.11).  The warp reads the high parts of one
// polynomial into its tile of n words of dynamic shared memory (packed_high, in entry order across the row; the cursor sits
// after the tile), then each lane joins the entries it owns with their fixed fields; pk.ok[b] = 1 when the slot is
// canonical (0 for a bad index).  The packed complete 256-point tile (D = 1) asks for 3 blocks per SM: at 4 it spills.
template <int EPL, int D, bool KEYED = false, bool PACKED = false>
__global__ void __launch_bounds__(128, (KEYED && EPL * D == 8) ? ((PACKED && D == 1) ? 3 : 4) : 0)
ring_small_kernel(const int32_t* __restrict__ sigma, const uint32_t* __restrict__ a_hat, int64_t* __restrict__ out,
                  unsigned long long* __restrict__ norm2, int B, int npoly, SmallRing R, const uint32_t* __restrict__ tw,
                  const int32_t* __restrict__ key_idx = nullptr, int nkeys = 0, int* flag = nullptr, PackedRows pk = {}) {
    static_assert(!PACKED || KEYED, "the packed form is keyed");
    extern __shared__ uint32_t rs_tiles[];
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    constexpr int NP = EPL * 32;
    const int n = NP * D;
    uint32_t* tile = rs_tiles + (threadIdx.x >> 5) * (n + 4);
    PackedCursor* cur = reinterpret_cast<PackedCursor*>(tile + n);
    for (long b = (long)blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += (long)gridDim.x * wpb) {
        int t = 0;
        if (KEYED) {
            t = key_idx[b];
            if (t < 0 || t >= nkeys) {
                for (int i = lane; i < n; i += 32) out[b * n + i] = 0;
                if (lane == 0) {
                    if (flag) atomicOr(flag, QF_FLAG_KEY_INDEX);
                    if (norm2) norm2[b] = ~0ull;
                    if (PACKED) pk.ok[b] = 0;
                }
                continue;
            }
        }
        if (PACKED) packed_begin(cur, lane);
        uint32_t acc[D][EPL];
#pragma unroll
        for (int c = 0; c < D; ++c)
#pragma unroll
            for (int r = 0; r < EPL; ++r) acc[c][r] = 0;
        NormAcc nrm;  // saturating squared norm (common.cuh)
        nrm.clear();
        for (int j = 0; j < npoly; ++j) {
            const int32_t* src = sigma + ((long)b * npoly + j) * n;
            if (PACKED) packed_high(pk, b, cur, tile, n, lane);
            bool bad = false;
            uint32_t v[D][EPL];
#pragma unroll
            for (int r = 0; r < EPL; ++r) {
                const int e = r * 32 + lane;
                int32_t x[D];
                if (PACKED) {
#pragma unroll
                    for (int c = 0; c < D; ++c) x[c] = packed_value(pk, b, (long long)j * n + D * e + c, tile[D * e + c], bad);
                } else if (D == 2) {
                    const int2 t = *reinterpret_cast<const int2*>(src + 2 * e);
                    x[0] = t.x;
                    x[D - 1] = t.y;
                } else {
                    x[0] = src[e];
                }
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    nrm.add_sq(x[c]);
                    int32_t m = x[c] % (int32_t)R.q;
                    v[c][r] = (uint32_t)(m < 0 ? m + (int32_t)R.q : m);
                }
            }
            if (PACKED && bad) cur->bad = 1;
#pragma unroll
            for (int c = 0; c < D; ++c) ntt_fwd<EPL>(v[c], tw, lane, R);
            // (the largest tile re-reads its index from L1 instead of keeping it live: no spill at 255 registers)
            const int kt = (KEYED && EPL * D == 32) ? __ldg(key_idx + b) : t;
            const uint32_t* ah = a_hat + ((long)kt * npoly + j) * n;
#pragma unroll
            for (int r = 0; r < EPL; ++r) {
                const int e = r * 32 + lane;
                if (D == 1) {
                    acc[0][r] = addq(acc[0][r], mulq(v[0][r], ah[e], R), R);
                } else {
                    // (s0 + s1 X)(a0 + a1 X) mod X^2 - zeta
                    const uint2 av = *reinterpret_cast<const uint2*>(ah + 2 * e);
                    const uint32_t zeta = tw[2 * NP + e];
                    const uint32_t s0 = v[0][r], s1 = v[D - 1][r];
                    const uint32_t c0 = addq(mulq(s0, av.x, R), mulq(mulq(s1, av.y, R), zeta, R), R);
                    const uint32_t c1 = addq(mulq(s0, av.y, R), mulq(s1, av.x, R), R);
                    acc[0][r] = addq(acc[0][r], c0, R);
                    acc[D - 1][r] = addq(acc[D - 1][r], c1, R);
                }
            }
        }
#pragma unroll
        for (int c = 0; c < D; ++c) ntt_inv<EPL>(acc[c], tw + NP, lane, R);
        int64_t* dst = out + (long)b * n;
#pragma unroll
        for (int r = 0; r < EPL; ++r) {
            const int e = r * 32 + lane;
            if (D == 2) {
                longlong2 o;
                o.x = (long long)mulq(acc[0][r], R.np_inv, R);
                o.y = (long long)mulq(acc[D - 1][r], R.np_inv, R);
                *reinterpret_cast<longlong2*>(dst + 2 * e) = o;
            } else {
                dst[e] = (long long)mulq(acc[0][r], R.np_inv, R);
            }
        }
        if (norm2) {
            nrm.warp_reduce();
            if (lane == 0) norm2[b] = nrm.value();
        }
        if (PACKED) {
            const bool canon = packed_finish(pk, b, cur, lane);
            if (lane == 0) pk.ok[b] = canon ? 1 : 0;
        }
    }
}

// Forward transform of npolys key polynomials on the device, one warp per polynomial: the words qf_ring_small_key writes
// (same butterflies, exact mod q), for a table of many keys.
template <int EPL, int D>
__global__ void __launch_bounds__(128)
ring_small_key_kernel(const int64_t* __restrict__ a, uint32_t* __restrict__ a_hat, long npolys, SmallRing R,
                      const uint32_t* __restrict__ tw) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    constexpr int NP = EPL * 32;
    const int n = NP * D;
    const uint32_t p32 = (uint32_t)((1ull << 32) - (unsigned long long)R.barrett * R.q);  // 2^32 mod q (q odd)
    for (long p = (long)blockIdx.x * wpb + (threadIdx.x >> 5); p < npolys; p += (long)gridDim.x * wpb) {
        const int64_t* src = a + p * n;
        uint32_t v[D][EPL];
#pragma unroll
        for (int r = 0; r < EPL; ++r)
#pragma unroll
            for (int c = 0; c < D; ++c) {
                // x mod q in 32-bit arithmetic: (hi mod q) (2^32 mod q) + (lo mod q) < q^2 <= 2^32
                const unsigned long long x = (unsigned long long)src[D * (r * 32 + lane) + c];
                v[c][r] = ((uint32_t)(x >> 32) % R.q * p32 + (uint32_t)x % R.q) % R.q;
            }
#pragma unroll
        for (int c = 0; c < D; ++c) ntt_fwd<EPL>(v[c], tw, lane, R);
        uint32_t* dst = a_hat + p * n;
#pragma unroll
        for (int r = 0; r < EPL; ++r)
#pragma unroll
            for (int c = 0; c < D; ++c) dst[D * (r * 32 + lane) + c] = v[c][r];
    }
}

// ---- host side: roots and key transforms ------------------------------------------------------
uint64_t powmod(uint64_t a, uint64_t e, uint64_t q) {
    uint64_t r = 1;
    a %= q;
    while (e) {
        if (e & 1) r = r * a % q;
        a = a * a % q;
        e >>= 1;
    }
    return r;
}
bool is_prime(uint64_t q) {
    if (q < 2) return false;
    for (uint64_t p = 2; p * p <= q; ++p)
        if (q % p == 0) return false;
    return true;
}
int bitrev(int x, int bits) {
    int r = 0;
    for (int i = 0; i < bits; ++i)
        if (x & (1 << i)) r |= 1 << (bits - 1 - i);
    return r;
}

}  // namespace

// Returns 0 if (q, n) is not served by this path.  Otherwise fills the plan: d, np, tables (3*np words) and np_inv.
int qf_ring_small_plan(unsigned long long q, int n, int* d_out, std::vector<uint32_t>* tables, uint32_t* np_inv) {
    if (q >= 65536 || q < 3 || !is_prime(q) || n < 64 || (n & (n - 1))) return 0;
    int d;
    if ((q - 1) % (2ull * n) == 0) d = 1;
    else if ((q - 1) % (unsigned long long)n == 0) d = 2;
    else return 0;
    const int np = n / d;
    if (np < 32 || np > 1024) return 0;
    int logn = 0;
    while ((1 << logn) < np) ++logn;
    // primitive root of unity of order 2*np: g^((q-1)/(2 np)) for a generator g
    uint64_t omega = 0;
    for (uint64_t g = 2; g < q && !omega; ++g) {
        uint64_t w = powmod(g, (q - 1) / (2ull * np), q);
        if (powmod(w, np, q) == q - 1) omega = w;  // w^np = -1  <=> order exactly 2 np
    }
    if (!omega) return 0;
    const uint64_t omega_inv = powmod(omega, q - 2, q);
    tables->assign(3 * (size_t)np, 0);
    for (int k = 0; k < np; ++k) {
        const int r = bitrev(k, logn);
        (*tables)[k] = (uint32_t)powmod(omega, r, q);
        (*tables)[np + k] = (uint32_t)powmod(omega_inv, r, q);
        (*tables)[2 * np + k] = (uint32_t)powmod(omega, 2ull * r + 1, q);  // zeta of output slot k
    }
    *np_inv = (uint32_t)powmod(np, q - 2, q);
    *d_out = d;
    return 1;
}

// Forward transform of the key polynomials on the host (same butterflies as the kernel), npoly x n.
void qf_ring_small_key(const int64_t* a, int npoly, int n, int d, unsigned long long q, const uint32_t* tables,
                       uint32_t* a_hat) {
    const int np = n / d;
    std::vector<uint64_t> v(np);
    for (int j = 0; j < npoly; ++j)
        for (int c = 0; c < d; ++c) {
            for (int e = 0; e < np; ++e) v[e] = (uint64_t)a[(long)j * n + d * e + c] % q;
            int t = np;
            for (int m = 1; m < np; m <<= 1) {
                t >>= 1;
                for (int i = 0; i < m; ++i) {
                    const uint64_t s = tables[m + i];
                    for (int k = 2 * i * t; k < 2 * i * t + t; ++k) {
                        const uint64_t u = v[k], w = v[k + t] * s % q;
                        v[k] = (u + w) % q;
                        v[k + t] = (u + q - w) % q;
                    }
                }
            }
            for (int e = 0; e < np; ++e) a_hat[(long)j * n + d * e + c] = (uint32_t)v[e];
        }
}

namespace {
SmallRing small_ring(int n, int d, unsigned long long q, uint32_t np_inv) {
    SmallRing R;
    R.q = (uint32_t)q;
    R.barrett = (uint32_t)((1ull << 32) / q);
    R.n = n; R.d = d; R.np = n / d; R.np_inv = np_inv;
    return R;
}
}  // namespace

cudaError_t qf_launch_ring_small(const int32_t* sigma, const uint32_t* a_hat, int64_t* out, unsigned long long* norm2,
                                 int B, int npoly, int n, int d, unsigned long long q, uint32_t np_inv,
                                 const uint32_t* tw, cudaStream_t stream, const int32_t* key_idx, int nkeys, int* flag,
                                 const PackedRows* packed) {
    if (B <= 0) return cudaSuccess;
    if (packed && (!key_idx || !qf_ring_small_packed_fused(n))) return cudaErrorInvalidValue;
    const SmallRing R = small_ring(n, d, q, np_inv);
    const int wpb = 4;
    long long g = ((long long)B + wpb - 1) / wpb;
    if (g > 148 * 16) g = 148 * 16;
    const int epl = R.np / 32;
    const size_t tiles = packed ? (size_t)wpb * (n + 4) * 4 : 0;  // a tile and a cursor per warp: at most 8.06 KB (n <= 512)
#define QF_RS_I32(E, DD)                                                                                                \
    (key_idx ? ring_small_kernel<E, DD, true><<<(int)g, 32 * wpb, 0, stream>>>(sigma, a_hat, out, norm2, B, npoly, R, tw, \
                                                                                key_idx, nkeys, flag)                  \
             : ring_small_kernel<E, DD><<<(int)g, 32 * wpb, 0, stream>>>(sigma, a_hat, out, norm2, B, npoly, R, tw))
#define QF_RS(E, DD)                                                                                                    \
    (packed ? ring_small_kernel<E, DD, true, true><<<(int)g, 32 * wpb, tiles, stream>>>(nullptr, a_hat, out, norm2, B,  \
                                                                                        npoly, R, tw, key_idx, nkeys,   \
                                                                                        flag, *packed)                  \
            : QF_RS_I32(E, DD))
    if (d == 1) {
        switch (epl) {
            case 2: QF_RS(2, 1); break;
            case 4: QF_RS(4, 1); break;
            case 8: QF_RS(8, 1); break;
            case 16: QF_RS(16, 1); break;
            case 32: QF_RS_I32(32, 1); break;
            default: return cudaErrorInvalidValue;
        }
    } else {
        switch (epl) {
            case 1: QF_RS(1, 2); break;
            case 2: QF_RS(2, 2); break;
            case 4: QF_RS(4, 2); break;
            case 8: QF_RS(8, 2); break;
            case 16: QF_RS_I32(16, 2); break;
            default: return cudaErrorInvalidValue;
        }
    }
#undef QF_RS
#undef QF_RS_I32
    return cudaGetLastError();
}

// The packed form spills at n = 1024 (255 registers hold the int32 tile with nothing to spare), so there the caller
// decodes into an int32 staging buffer and launches the int32 keyed form.
bool qf_ring_small_packed_fused(int n) { return n <= 512; }

cudaError_t qf_launch_ring_small_key(const int64_t* a, uint32_t* a_hat, long npolys, int n, int d, unsigned long long q,
                                     const uint32_t* tw, cudaStream_t stream) {
    if (npolys <= 0) return cudaSuccess;
    const SmallRing R = small_ring(n, d, q, 0);
    const int wpb = 4;
    long long g = ((long long)npolys + wpb - 1) / wpb;
    if (g > 148 * 16) g = 148 * 16;
    const int epl = R.np / 32;
#define QF_RK(E, DD) ring_small_key_kernel<E, DD><<<(int)g, 32 * wpb, 0, stream>>>(a, a_hat, npolys, R, tw)
    if (d == 1) {
        switch (epl) {
            case 2: QF_RK(2, 1); break;
            case 4: QF_RK(4, 1); break;
            case 8: QF_RK(8, 1); break;
            case 16: QF_RK(16, 1); break;
            case 32: QF_RK(32, 1); break;
            default: return cudaErrorInvalidValue;
        }
    } else {
        switch (epl) {
            case 1: QF_RK(1, 2); break;
            case 2: QF_RK(2, 2); break;
            case 4: QF_RK(4, 2); break;
            case 8: QF_RK(8, 2); break;
            case 16: QF_RK(16, 2); break;
            default: return cudaErrorInvalidValue;
        }
    }
#undef QF_RK
    return cudaGetLastError();
}
