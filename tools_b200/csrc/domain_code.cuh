// Decoding packed Domain values inside a kernel that consumes them (DESIGN 4.11, 4.13): the format of domain_code.cu read
// one run of entries at a time, so that a warp can hand one polynomial of a row to its NTT without writing the int32 row
// to memory.  Every canonical check of domain_decode_kernel runs here as well; a failure sets the row's bad flag (its
// values are then unspecified, as with qf_domain_decode_dev).
//
// The cursor of a row lives in shared memory, not in registers: the consuming kernels run register-bound transforms between
// two reads of the same row, and nothing of the decoder stays live across them.
#pragma once

#include <cstdint>

// The packed rows of a batch: row b is the slot at p + b slot_bytes; ok[b] receives 1 when the slot is canonical.
struct PackedRows {
    const uint8_t* p;
    long long slot_bytes, h0;  // h0 = qf_domain_h0(dim, k)
    int dim, k;
    uint8_t* ok;
};

// Where one row's walk stands (shared memory, one per row being decoded)
struct PackedCursor {
    long long prev;  // bit of the last terminator read (relative to the high stream), -1 before the first
    int ones;        // entries whose high part has been read
    int bad;         // a canonical check failed
};

__device__ __forceinline__ const uint32_t* packed_words(const PackedRows& pk, long long row) {
    return reinterpret_cast<const uint32_t*>(pk.p + row * pk.slot_bytes);
}

// Start a row (lane 0 writes; the next packed_high of the warp reads)
__device__ __forceinline__ void packed_begin(PackedCursor* cur, int lane) {
    if (lane == 0) {
        cur->prev = -1;
        cur->ones = 0;
        cur->bad = 0;
    }
    __syncwarp();
}

// Warp-collective: the high parts h_i of the row's next cnt entries into tile[0 .. cnt), in entry order.  32 words of the
// stream per round, from the word that holds the bit after the last terminator (a round shared with the previous call is
// read again, from L1).  The rank of a 1 bit is its entry; the 1 bit before it comes from a ballot over the lanes whose word
// is not zero.  A high part above INT32_MAX >> k, or a stream that ends early, marks the row bad.
template <typename T>
__device__ __forceinline__ void packed_high(const PackedRows& pk, long long row, PackedCursor* cur, T* tile, int cnt,
                                            int lane) {
    const uint32_t* hw = packed_words(pk, row) + pk.h0 / 4;
    const long long nhw = (pk.slot_bytes - pk.h0) / 4;
    const uint32_t hmax = 0x7fffffffu >> pk.k;
    long long prev = cur->prev;
    const long long e0 = cur->ones, target = e0 + cnt;
    long long ones = e0;
    long long w0 = (prev + 1) >> 5;
    bool bad = false;
    __syncwarp();
    while (ones < target) {
        if (w0 >= nhw) {  // the stream ended before the target-th terminator: fewer than dim entries
            bad = true;
            break;
        }
        const long long wi = w0 + lane;
        uint32_t wd = wi < nhw ? __ldg(hw + wi) : 0u;
        if (wi == ((prev + 1) >> 5)) wd &= ~0u << ((prev + 1) & 31);  // terminators of earlier entries
        const uint32_t c = __popc(wd);
        uint32_t incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t nz = __ballot_sync(0xffffffffu, wd != 0);
        const uint32_t lower = nz & ((1u << lane) - 1u);
        const int lastb = wd ? 31 - __clz(wd) : 0;
        const int src = lower ? 31 - __clz(lower) : 0;
        const int lb = __shfl_sync(0xffffffffu, lastb, src);
        long long before = lower ? (w0 + src) * 32 + lb : prev;
        long long r = ones + (long long)(incl - c);
        long long mine = -1;  // the bit of terminator target - 1, in the lane that holds it
        uint32_t bits = wd;
        while (bits && r < target) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            const long long t = wi * 32 + b;
            const unsigned long long h = (unsigned long long)(t - before - 1);
            before = t;
            bad |= h > hmax;
            tile[r - e0] = (T)(h > hmax ? 0u : (uint32_t)h);
            if (r == target - 1) mine = t;
            ++r;
        }
        const uint32_t has = __ballot_sync(0xffffffffu, mine >= 0);
        if (has) {
            prev = __shfl_sync(0xffffffffu, mine, __ffs(has) - 1);
            ones = target;
        } else {
            ones += tot;
            if (nz) prev = (w0 + 31 - __clz(nz)) * 32 + __shfl_sync(0xffffffffu, lastb, 31 - __clz(nz));
            w0 += 32;
        }
    }
    bad = __any_sync(0xffffffffu, bad);
    __syncwarp();
    if (lane == 0) {
        cur->prev = prev;
        cur->ones = (int)ones;
        if (bad) cur->bad = 1;
    }
    __syncwarp();
}

// Entry e of the row from its high part h: the fixed field at bit e (k+1) holds a mod 2^k and the sign.  A sign on a zero
// magnitude sets *bad (any thread may call this; h <= INT32_MAX >> k keeps the magnitude at most INT32_MAX).
__device__ __forceinline__ int32_t packed_value(const PackedRows& pk, long long row, long long e, uint32_t h, bool& bad) {
    const uint32_t* w = packed_words(pk, row);
    const int k = pk.k;
    const unsigned long long p = (unsigned long long)e * (k + 1);
    const unsigned long long two = ((unsigned long long)__ldg(w + (p >> 5) + 1) << 32) | __ldg(w + (p >> 5));
    const uint32_t f = (uint32_t)(two >> (p & 31)) & ((2u << k) - 1u);
    const uint32_t mag = (h << k) | (f & ((1u << k) - 1u)), sign = f >> k;
    bad |= sign && mag == 0;
    return sign ? -(int32_t)mag : (int32_t)mag;
}

// Warp-collective, after the dim-th entry and after every packed_value of the row is visible in cur->bad: no 1 bit after
// the dim-th terminator up to the end of the slot, and zero padding after the fixed fields.  Returns whether the row is a
// canonical code (warp-uniform).
__device__ __forceinline__ bool packed_finish(const PackedRows& pk, long long row, const PackedCursor* cur, int lane) {
    const uint32_t* w = packed_words(pk, row);
    const int h0w = (int)(pk.h0 / 4);
    const long long nhw = (pk.slot_bytes - pk.h0) / 4;
    __syncwarp();
    const long long prev = cur->prev;
    bool bad = cur->bad || cur->ones < pk.dim;
    for (long long wi = ((prev + 1) >> 5) + lane; wi < nhw; wi += 32) {
        uint32_t x = __ldg(w + h0w + wi);
        if (wi == ((prev + 1) >> 5)) x &= ~0u << ((prev + 1) & 31);
        bad |= x != 0;
    }
    const unsigned long long fbits = (unsigned long long)pk.dim * (pk.k + 1);
    for (long long wi = (long long)(fbits >> 5) + lane; wi < h0w; wi += 32) {
        uint32_t x = __ldg(w + wi);
        if (wi == (long long)(fbits >> 5)) x &= ~((1u << (fbits & 31)) - 1u);
        bad |= x != 0;
    }
    return !__any_sync(0xffffffffu, bad);
}
