// Packed Domain values: a lossless Golomb-Rice code of int32 preimage rows (DESIGN 4.11, include/qfall_b200.h).
//
// A row of dim entries x_i is stored in a slot of slot_bytes bytes (a multiple of 16), streams LSB-first.  With a = |x_i|,
// h_i = a >> k and sign = (x_i < 0):
//   fixed part   entry i is the (k+1)-bit field (a mod 2^k) | sign << k at bit i (k+1); it ends at byte
//                H0 = 16 ceil(dim (k+1) / 128), padding bits zero;
//   high stream  from byte H0: h_i zero bits then one 1 bit, for i = 0 .. dim-1 in order; zero up to the end of the slot;
//   length       nbytes = H0 + ceil(sum (h_i + 1) / 8).
// The two parts are apart so that neither direction parses sequentially: the fixed part is a bit-field array, and the
// high part of entry i ends at the i-th 1 bit of the high stream (ballot / popc and a warp prefix sum).
// One warp per row in both kernels.
#include <cmath>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int kMaxWarps = 8;

template <typename T>
__device__ __forceinline__ T warp_incl_sum(T v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// Encoder.  Lane l takes entries i0 + 4 l .. i0 + 4 l + 3 of each block of 128 (a block's fixed fields are 4 (k+1) whole
// words); an exclusive warp scan of the per-lane sums of h_i + 1 places the terminators.  The slot is assembled in a zeroed
// buffer with atomicOr -- shared memory (SMEM) and then copied out with 16-byte stores, or the output slot itself when
// slot_bytes exceeds what shared memory holds.  A row that does not fit or holds INT32_MIN gets nbytes = -1, zero slot.
template <bool SMEM>
__global__ void __launch_bounds__(kMaxWarps * 32) domain_encode_kernel(const int32_t* __restrict__ in, long long rows, int dim,
                                                                       int k, long long slot_bytes, long long h0,
                                                                       uint8_t* __restrict__ out, int32_t* __restrict__ nbytes) {
    extern __shared__ uint4 smem_slots[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= rows) return;
    const long long nvec = slot_bytes / 16;
    uint4* gslot = reinterpret_cast<uint4*>(out + row * slot_bytes);
    uint4* bufv = SMEM ? smem_slots + (size_t)warp * nvec : gslot;
    uint32_t* buf = reinterpret_cast<uint32_t*>(bufv);
    for (long long v = lane; v < nvec; v += 32) bufv[v] = make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();

    const int32_t* x = in + row * (long long)dim;
    const uint32_t kmask = (1u << k) - 1u;
    const int fb = k + 1;
    const unsigned long long hcap = (unsigned long long)(slot_bytes - h0) * 8ull;  // bits of the high stream
    const unsigned long long hstart = (unsigned long long)h0 * 8ull;
    unsigned long long base = 0;  // high-stream bits of the blocks before this one
    bool bad = false;
    for (int i0 = 0; i0 < dim; i0 += 128) {
        const int ib = i0 + 4 * lane;
        int32_t v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = ib + j < dim ? __ldg(x + ib + j) : 0;
        unsigned long long len[4], sum = 0;  // h + 1 (0 past the row), up to 2^31 each
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool present = ib + j < dim;
            bad |= v[j] == INT32_MIN;
            const uint32_t a = v[j] < 0 ? 0u - (uint32_t)v[j] : (uint32_t)v[j];
            len[j] = present ? (unsigned long long)(a >> k) + 1ull : 0ull;
            sum += len[j];
            if (present) {
                const uint32_t f = (a & kmask) | ((uint32_t)(v[j] < 0) << k);
                const unsigned long long p = (unsigned long long)(ib + j) * fb;
                const int sh = (int)(p & 31);
                atomicOr(buf + (p >> 5), f << sh);
                if (sh + fb > 32) atomicOr(buf + (p >> 5) + 1, f >> (32 - sh));
            }
        }
        const unsigned long long incl = warp_incl_sum(sum, lane);
        const unsigned long long total = __shfl_sync(0xffffffffu, incl, 31);
        unsigned long long pos = base + (incl - sum);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (len[j]) {
                const unsigned long long t = pos + len[j] - 1;  // terminator of entry ib + j
                if (t < hcap) {
                    const unsigned long long b = hstart + t;
                    atomicOr(buf + (b >> 5), 1u << (b & 31));
                } else {
                    bad = true;
                }
                pos += len[j];
            }
        }
        base += total;
        if (__any_sync(0xffffffffu, bad)) break;
    }
    bad = __any_sync(0xffffffffu, bad);
    __syncwarp();
    if (bad) {
        for (long long v = lane; v < nvec; v += 32) gslot[v] = make_uint4(0u, 0u, 0u, 0u);
        if (lane == 0) nbytes[row] = -1;
        return;
    }
    if (SMEM)
        for (long long v = lane; v < nvec; v += 32) gslot[v] = bufv[v];
    if (lane == 0) nbytes[row] = (int32_t)(h0 + (long long)((base + 7) / 8));
}

// Decoder.  Fixed fields are read in place; the high stream is read 128 bits per lane, and the rank of each 1 bit (its
// entry) and the position of the 1 bit before it come from a warp prefix sum of popc and a prefix max of the last 1 bit.
// Every canonical check of the format runs; ok[row] = 0 on any failure (the row's values are then unspecified).
__global__ void __launch_bounds__(kMaxWarps * 32) domain_decode_kernel(const uint8_t* __restrict__ in, long long rows, int dim,
                                                                       int k, long long slot_bytes, long long h0,
                                                                       int32_t* __restrict__ out, uint8_t* __restrict__ ok) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (row >= rows) return;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(in + row * slot_bytes);
    const int fb = k + 1;
    const uint32_t kmask = (1u << k) - 1u, fmask = (2u << k) - 1u;
    const unsigned long long fbits = (unsigned long long)dim * fb;
    bool bad = false;
    // padding of the fixed part: bits [dim (k+1), 8 H0)
    for (long long wi = (long long)(fbits >> 5) + lane; wi < h0 / 4; wi += 32) {
        uint32_t x = __ldg(w + wi);
        if (wi == (long long)(fbits >> 5)) x &= ~((1u << (fbits & 31)) - 1u);
        bad |= x != 0;
    }
    const uint4* hs = reinterpret_cast<const uint4*>(in + row * slot_bytes + h0);
    const long long nv = (slot_bytes - h0) / 16;
    int32_t* o = out + row * (long long)dim;
    long long ones = 0;   // terminators before this round (warp uniform)
    long long prev = -1;  // bit position of the last terminator before this round
    for (long long v0 = 0; v0 < nv; v0 += 32) {
        const long long vi = v0 + lane;
        const uint4 q = vi < nv ? __ldg(hs + vi) : make_uint4(0u, 0u, 0u, 0u);
        const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
        const uint32_t c = __popc(wd[0]) + __popc(wd[1]) + __popc(wd[2]) + __popc(wd[3]);
        const uint32_t incl = warp_incl_sum(c, lane);
        const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
        long long last = -1;
#pragma unroll
        for (int j = 3; j >= 0; --j)
            if (last < 0 && wd[j]) last = vi * 128 + j * 32 + 31 - __clz(wd[j]);
        long long mx = last;  // inclusive prefix max over the lanes
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, mx, d);
            if (lane >= d) mx = t > mx ? t : mx;
        }
        long long before = __shfl_up_sync(0xffffffffu, mx, 1);
        before = lane == 0 ? prev : (before > prev ? before : prev);
        long long r = ones + (long long)(incl - c);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t bits = wd[j];
            while (bits) {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                const long long t = vi * 128 + j * 32 + b;
                const unsigned long long h = (unsigned long long)(t - before - 1);
                before = t;
                if (r < dim) {
                    const unsigned long long p = (unsigned long long)r * fb;
                    const unsigned long long two = ((unsigned long long)__ldg(w + (p >> 5) + 1) << 32) | __ldg(w + (p >> 5));
                    const uint32_t f = (uint32_t)(two >> (p & 31)) & fmask;
                    const uint32_t sign = f >> k;
                    if (h > (0x7fffffffull >> k)) {
                        bad = true;
                    } else {
                        const uint32_t mag = (uint32_t)(h << k) | (f & kmask);
                        bad |= mag > 0x7fffffffu || (sign && mag == 0);
                        o[r] = sign ? -(int32_t)mag : (int32_t)mag;
                    }
                } else {
                    bad = true;  // a 1 bit after the dim-th
                }
                ++r;
            }
        }
        ones += tot;
        const long long lastw = __shfl_sync(0xffffffffu, mx, 31);
        prev = lastw > prev ? lastw : prev;
    }
    bad |= ones < dim;
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) ok[row] = bad ? 0 : 1;
}

}  // namespace

long long qf_domain_h0(long long dim, int k) { return 16 * ((dim * (k + 1) + 127) / 128); }

cudaError_t qf_launch_domain_encode(const int32_t* in, long long rows, int dim, int k, long long slot_bytes, uint8_t* out,
                                    int32_t* nbytes, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    if ((((uintptr_t)out) & 15) || (((uintptr_t)in) & 3)) return cudaErrorMisalignedAddress;
    const long long h0 = qf_domain_h0(dim, k);
    int dev = 0, smem_block = 0, smem_sm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_block, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    if (e != cudaSuccess) return e;
    if (slot_bytes <= smem_block) {
        // warps (= rows) per CTA: the most resident warps per SM, shared memory being the limit (1 KB reserved per CTA)
        int best_w = 1, best_res = 0;
        for (int wpc = 1; wpc <= kMaxWarps; ++wpc) {
            const long long bytes = wpc * slot_bytes;
            if (bytes > smem_block) break;
            const int res = (int)(smem_sm / (bytes + 1024)) * wpc;
            if (res >= best_res) best_res = res, best_w = wpc;
        }
        const size_t bytes = (size_t)best_w * slot_bytes;
        e = cudaFuncSetAttribute(domain_encode_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        const long long grid = (rows + best_w - 1) / best_w;
        domain_encode_kernel<true><<<(unsigned)grid, best_w * 32, bytes, stream>>>(in, rows, dim, k, slot_bytes, h0, out, nbytes);
    } else {
        const long long grid = (rows + kMaxWarps - 1) / kMaxWarps;
        domain_encode_kernel<false><<<(unsigned)grid, kMaxWarps * 32, 0, stream>>>(in, rows, dim, k, slot_bytes, h0, out, nbytes);
    }
    return cudaGetLastError();
}

cudaError_t qf_launch_domain_decode(const uint8_t* in, long long rows, int dim, int k, long long slot_bytes, int32_t* out,
                                    uint8_t* ok, cudaStream_t stream) {
    if (rows <= 0) return cudaSuccess;
    if ((((uintptr_t)in) & 15) || (((uintptr_t)out) & 3)) return cudaErrorMisalignedAddress;
    const long long grid = (rows + kMaxWarps - 1) / kMaxWarps;
    domain_decode_kernel<<<(unsigned)grid, kMaxWarps * 32, 0, stream>>>(in, rows, dim, k, slot_bytes, qf_domain_h0(dim, k), out,
                                                                       ok);
    return cudaGetLastError();
}

// k minimising E[k + 2 + h] for X ~ D_{Z,w} (rho(x) = exp(-pi x^2 / w^2), summed over |x| <= 20 w), and
// slot = H0 + ceil((dim E[h+1] + 12 sqrt(dim Var[h+1])) / 8) rounded up to 16
void qf_domain_code_recommend(double w, long long dim, int* k_out, long long* slot_out) {
    const long long X = (long long)std::floor(20.0 * w);
    std::vector<double> p((size_t)X + 1);
    double z = 0;
    for (long long a = 0; a <= X; ++a) {
        const double t = (double)a / w;
        p[a] = std::exp(-M_PI * t * t) * (a ? 2.0 : 1.0);
        z += p[a];
    }
    double eh[31] = {0}, eh2[31] = {0};
    for (long long a = 0; a <= X; ++a) {
        const double pa = p[a] / z;
        for (int k = 0; k < 31; ++k) {
            const double h = (double)(a >> k);
            eh[k] += pa * h;
            eh2[k] += pa * h * h;
        }
    }
    int best = 0;
    for (int k = 1; k < 31; ++k)
        if (k + eh[k] < best + eh[best]) best = k;
    const double var = std::max(0.0, eh2[best] - eh[best] * eh[best]);
    const double bits = (double)dim * (eh[best] + 1.0) + 12.0 * std::sqrt((double)dim * var);
    long long slot = qf_domain_h0(dim, best) + (long long)std::ceil(bits / 8.0);
    *k_out = best;
    *slot_out = (slot + 15) / 16 * 16;
}
