// Shared device helpers for the qfall B200 backend (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#define QF_SM_COUNT_DEFAULT 148

// ---------------------------------------------------------------------------
// Philox4x32-10 counter RNG.  key = 64-bit seed, counter = 128 bits.
// Counter layout used everywhere in this library:
//   c0,c1 = 64-bit global element index (target_index * dim + coordinate)
//   c2    = stream tag (which sampling site draws; see QF_STREAM_*)
//   c3    = block counter within the element's private stream
// so every (seed, site, element) owns an independent stream and results do not
// depend on launch geometry, chunking or the number of GPUs.
// ---------------------------------------------------------------------------
#define QF_STREAM_SAMP_D 1u
#define QF_STREAM_PERT_NORMAL 2u
#define QF_STREAM_PERT_ROUND 3u
#define QF_STREAM_GADGET 4u
#define QF_STREAM_NP 5u
#define QF_STREAM_UNIFORM 6u
#define QF_STREAM_TERNARY 7u
#define QF_STREAM_RING_TD 8u
#define QF_STREAM_SAMPLE_Z 9u
// bits of the per-context numeric flag (qf_synchronize / qf_samp_p report QF_ERR_NUMERIC when any is set)
#define QF_FLAG_DGAUSS_BAILOUT 16
// a tag index of qf_samp_p_tagged_dev outside the installed tag table (reported by check_flag as QF_ERR_INVALID)
#define QF_FLAG_TAG_INDEX 128
// a key index of qf_ring_f_a_keyed_dev outside the installed ring key table (reported by check_flag as QF_ERR_INVALID)
#define QF_FLAG_KEY_INDEX 256

struct Philox {
    uint32_t k0, k1;
    uint32_t c0, c1, c2, c3;
    uint32_t out[4];
    int have;  // number of unread 32-bit words in out (read from the top)

    __device__ __forceinline__ void init(uint64_t seed, uint64_t index, uint32_t stream) {
        k0 = (uint32_t)seed;
        k1 = (uint32_t)(seed >> 32);
        c0 = (uint32_t)index;
        c1 = (uint32_t)(index >> 32);
        c2 = stream;
        c3 = 0;
        have = 0;
    }
    __device__ __forceinline__ void block() {
        uint32_t a0 = c0, a1 = c1, a2 = c2, a3 = c3, x0 = k0, x1 = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0 = __umulhi(0xD2511F53u, a0), lo0 = 0xD2511F53u * a0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, a2), lo1 = 0xCD9E8D57u * a2;
            uint32_t n0 = hi1 ^ a1 ^ x0, n2 = hi0 ^ a3 ^ x1;
            a0 = n0; a1 = lo1; a2 = n2; a3 = lo0;
            x0 += 0x9E3779B9u; x1 += 0xBB67AE85u;
        }
        out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3;
        c3 += 1;
        have = 4;
    }
    __device__ __forceinline__ uint32_t next() {
        if (have == 0) block();
        return out[--have];
    }
    // uniform in (0,1), 24 bits
    __device__ __forceinline__ float uniform24() {
        return ((float)(next() >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
    }
    // two independent N(0,1) (Box-Muller), consumes 2 words
    __device__ __forceinline__ void normal2(float& n0, float& n1) {
        uint32_t b0 = next(), b1 = next();
        // u in (0,1]: 40 bits = b0 and the low byte of b1 (the angle below keeps 24 bits of b1 after rounding, so that
        // byte is otherwise unused): u >= 2^-41, i.e. |n| reaches sqrt(82 ln 2) = 7.54 (a 32-bit u stops at 6.76).
        // The reference's support is 6 s = 15 sigma; the mass this proposal cannot reach is 4.7e-14 per draw.
        float u = fmaf(__uint2float_rn(b0), 2.3283064365386963e-10f, ((float)(b1 & 255u) + 0.5f) * 9.094947017729282e-13f);
        float rad = sqrtf(-2.0f * logf(u));
        float ang = __uint2float_rn(b1) * 4.6566128730773926e-10f;  // [0,2) in units of pi
        float s, c;
        sincospif(ang, &s, &c);
        n0 = rad * c;
        n1 = rad * s;
    }
};

// ---------------------------------------------------------------------------
// Exact 1-D discrete Gaussian D_{Z, s, c},  rho(x) = exp(-pi (x-c)^2 / s^2)
// (qfall-math convention, CONTRIBUTING.md:35-45; s = sigma * sqrt(2 pi)).
//
// Rounded-normal proposal with exact rejection correction:
//   y ~ N(c, sigma'^2), sigma'^2 = sigma^2 (1+eps);  x = round(y);
//   accept with probability exp(E - Emax),
//   E = -(x-c)^2/(2 sigma^2) + (y-c)^2/(2 sigma'^2),  Emax = 1/(8 sigma^2 eps) >= sup E.
// The accepted x has pmf  int_{x-1/2}^{x+1/2} phi_{sigma'}(y-c) exp(E-Emax) dy
//   = const * exp(-(x-c)^2/(2 sigma^2)),  i.e. exactly D_{Z,s,c}.
// eps minimises sqrt(1+eps) exp(Emax): eps = (1 + sqrt(1+16 sigma^2)) / (8 sigma^2).
// Acceptance is 0.69 at sigma = 1.2 and -> 1 as sigma grows, with one exp per
// trial (the reference's uniform-proposal SampleZ accepts ~1/12).
// Support is additionally cut to |x - c| <= 6 s like the reference.
// ---------------------------------------------------------------------------
struct DGaussParams {
    float sigma_p;   // proposal std-dev sigma'
    float inv2s2;    // 1 / (2 sigma^2)
    float emax;      // 1 / (8 sigma^2 eps)
    float tail;      // 6 s
};

__host__ __device__ inline DGaussParams make_dgauss(double s) {
    DGaussParams p;
    double sigma = s * 0.3989422804014327;  // 1/sqrt(2 pi)
    double s2 = sigma * sigma;
    double eps = (1.0 + sqrt(1.0 + 16.0 * s2)) / (8.0 * s2);
    p.sigma_p = (float)(sigma * sqrt(1.0 + eps));
    p.inv2s2 = (float)(0.5 / s2);
    p.emax = (float)(1.0 / (8.0 * s2 * eps));
    p.tail = (float)(6.0 * s);
    return p;
}

// Returns the sample as a double (exact integer value; centers may exceed 2^31).
// flag (optional): device int, QF_FLAG_DGAUSS_BAILOUT is ORed in if 4096 rounds (8192 proposals) were all rejected --
// probability < 0.4^8192 for valid parameters, so in practice it signals corrupt parameters (NaN centre / width).
__device__ __forceinline__ double sample_dgauss(const DGaussParams& p, double center, Philox& rng, int* flag = nullptr) {
    double c_int = rint(center);
    float c_frac = (float)(center - c_int);
    for (int it = 0; it < 4096; ++it) {
        float n0, n1;
        rng.normal2(n0, n1);
        float u0 = rng.uniform24(), u1 = rng.uniform24();
        {
            float x = rintf(fmaf(p.sigma_p, n0, c_frac));
            float d = x - c_frac;
            float e = fmaf(-d * d, p.inv2s2, fmaf(0.5f * n0, n0, -p.emax));
            if (fabsf(d) <= p.tail && __logf(u0) < e) return c_int + (double)x;
        }
        {
            float x = rintf(fmaf(p.sigma_p, n1, c_frac));
            float d = x - c_frac;
            float e = fmaf(-d * d, p.inv2s2, fmaf(0.5f * n1, n1, -p.emax));
            if (fabsf(d) <= p.tail && __logf(u1) < e) return c_int + (double)x;
        }
    }
    if (flag) atomicOr(flag, QF_FLAG_DGAUSS_BAILOUT);
    return c_int;
}

// ---------------------------------------------------------------------------
// Squared Euclidean norm of int32 entries for check_domain (gpv.rs:219-224), exact and SATURATING: a square is
// at most 2^62, so a plain u64 sum wraps after four such entries (16 entries of 2^30 sum to 2^64 = 0, which would
// pass every bound).  96-bit accumulator (64-bit sum + carry count); value() is the exact sum, or 2^64 - 1 when it
// does not fit 64 bits (above every admissible bound, which is < 2^62).
// ---------------------------------------------------------------------------
struct NormAcc {
    unsigned long long lo;
    unsigned int hi;
    __device__ __forceinline__ void clear() { lo = 0; hi = 0; }
    __device__ __forceinline__ void add(unsigned long long x) {
        asm("{\n\t.reg .u32 l0, l1, x0, x1;\n\t"
            "mov.b64 {l0, l1}, %0;\n\tmov.b64 {x0, x1}, %2;\n\t"
            "add.cc.u32 l0, l0, x0;\n\taddc.cc.u32 l1, l1, x1;\n\taddc.u32 %1, %1, 0;\n\t"
            "mov.b64 %0, {l0, l1};\n\t}"
            : "+l"(lo), "+r"(hi) : "l"(x));
    }
    __device__ __forceinline__ void add_sq(int v) { const long long w = v; add((unsigned long long)(w * w)); }
    // squares of four int32 values: the two pair sums are <= 2^63 each and cannot wrap
    __device__ __forceinline__ void add_sq4(int a, int b, int c, int d) {
        const long long la = a, lb = b, lc = c, ld = d;
        add((unsigned long long)(la * la) + (unsigned long long)(lb * lb));
        add((unsigned long long)(lc * lc) + (unsigned long long)(ld * ld));
    }
    __device__ __forceinline__ void merge(const NormAcc& o) { add(o.lo); hi += o.hi; }
    __device__ __forceinline__ void warp_reduce() {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            NormAcc t;
            t.lo = __shfl_xor_sync(0xffffffffu, lo, o);
            t.hi = __shfl_xor_sync(0xffffffffu, hi, o);
            merge(t);
        }
    }
    __device__ __forceinline__ unsigned long long value() const { return hi ? ~0ull : lo; }
};

// ---------------------------------------------------------------------------
// modular arithmetic helpers, q < 2^62
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mulmod_u64(uint64_t a, uint64_t b, uint64_t q) {
    // a, b < q < 2^62.  128-bit product reduced with a floating estimate + fixup.
    unsigned __int128 p = (unsigned __int128)a * b;
    return (uint64_t)(p % q);
}

__device__ __forceinline__ uint64_t mod_i128(__int128 v, uint64_t q) {
    __int128 r = v % (__int128)q;
    if (r < 0) r += q;
    return (uint64_t)r;
}

// v mod q in [0, q) for |v| < 2^63, q < 2^63, with magic = floor(2^64 / q): the quotient estimate
// umul64hi(|v|, magic) is at most 2 below the true one (|v| / 2^64 < 1), so two conditional subtractions finish it.
// (A 128-bit `%` is a library call of a few hundred instructions; the contraction epilogues reduce 16 K values per tile.)
__device__ __forceinline__ uint64_t mod_i64_barrett(long long v, uint64_t q, uint64_t magic) {
    const uint64_t a = v < 0 ? (uint64_t)(-v) : (uint64_t)v;
    uint64_t r = a - __umul64hi(a, magic) * q;
    if (r >= q) r -= q;
    if (r >= q) r -= q;
    return (v < 0 && r) ? q - r : r;
}
static inline uint64_t qf_barrett_magic(uint64_t q) { return q ? (uint64_t)((((unsigned __int128)1) << 64) / q) : 0; }

static inline int qf_ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Launcher-side caches (largest dynamic shared memory configured for a kernel, SM count) are kept PER DEVICE: function
// attributes belong to the device context the launch runs in.
#define QF_MAX_DEVICES 64
static inline int qf_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= QF_MAX_DEVICES) dev = 0;
    return dev;
}
