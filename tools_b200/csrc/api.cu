// C ABI (include/qfall_b200.h) and the host-side pipelines that compose the kernels.
//
// Data layout in HBM (everything "one row per target", row length padded to 16 elements):
//   Domain batch   int32  B x dim          (sigma, e, samp_d)           -- caller visible
//   Range batch    int64  B x n            (u, f_a output)              -- caller visible
//   work matrices  fp64   Bc x ld          (exact integers or reals)    -- per chunk of Bc targets
//   key matrices   fp64   rows x ld        W[coord][k], K-major         -- A chunks, sqrt(Sigma_2), R, S, U, Mt_P
// A batch is processed in chunks of `chunk` targets so that the workspace is bounded;
// the key material is resident for the lifetime of the context.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/qfall_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace {

typedef unsigned __int128 u128;
typedef __int128 i128;

struct Dev {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void swap(Dev& o) {
        std::swap(p, o.p);
        std::swap(cap, o.cap);
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    ~Dev() { release(); }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

inline long pad16(long x) { return (x + 15) / 16 * 16; }
inline int bitlen_u64(unsigned long long v) {
    int b = 0;
    while (v) { ++b; v >>= 1; }
    return b;
}

uint64_t inv_mod(uint64_t a, uint64_t q) {  // a^{-1} mod q, gcd(a,q)=1
    i128 t = 0, nt = 1, r = q, nr = a % q;
    while (nr != 0) {
        i128 qu = r / nr;
        i128 tmp = t - qu * nt; t = nt; nt = tmp;
        tmp = r - qu * nr; r = nr; nr = tmp;
    }
    if (t < 0) t += q;
    return (uint64_t)t;
}
uint64_t gcd_u64(uint64_t a, uint64_t b) {
    while (b) { uint64_t t = a % b; a = b; b = t; }
    return a;
}
inline uint64_t mulmod_h(uint64_t a, uint64_t b, uint64_t q) { return (uint64_t)((u128)a * b % q); }

}  // namespace

struct qf_ctx {
    qf_params prm{};
    int device = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    long n = 0, k = 0, m_bar = 0, nk = 0, m = 0;
    long dim = 0;        // Domain length: m (classical) or n*(k+2) (ring)
    long ld_dim = 0, ld_n = 0, ld_nk = 0;
    unsigned long long bound = 0;
    double s_samp_d = 0;
    long chunk = 0;

    // classical key
    bool has_a = false;
    int a_nchunks = 0, a_bits = 0;
    Dev dA[4];
    std::vector<int64_t> hA;
    // perturbation trapdoor
    bool has_pert = false;
    Dev dR, dL, dSk, dSkGso;
    // structured sqrt(Sigma_2) (qf_set_trapdoor_perturbation with sqrt_sigma_2 == NULL): x_b ~ N(0, beta I) on the
    // gadget block, x_t = L_s g_t - kappa R x_b with L_s the m_bar x m_bar Cholesky factor of the Schur complement
    bool pert_structured = false;
    int l_tri = 1;   // supplied sqrt(Sigma_2) is lower triangular (the Cholesky factor): skip the zero half
    Dev dLs, dXbScale;
    // x_2 = L g on the tensor cores: fixed-point digit planes of L (one scale per row) times fixed-point normals
    bool pert_i8 = false;
    Dev dLl, dLlScale;
    long ldk_l = 0, l_dim = 0;
    int lg_limbs = 3, ll_limbs = 4;
    double g_fscale = 0;
    long ld_mb = 0;
    double sqrt_beta = 0, xb_fscale = 0;
    int xb_limbs = 3;
    // the installed key is A = [A_bar | H G - A_bar R] for the installed R (recognised by qf_set_trapdoor_perturbation and,
    // on the two-phase recursion, qf_set_trapdoor_gpv; replaced by qf_set_tag / qf_gpv_set_tag): key_tag = H mod q (n x n).
    // For H != I, key_tagged is set and v = u - A p becomes v' = H^-1 v before the gadget sampler (digit planes of H^-1 in
    // dHinvl).
    bool pert_gadget_key = false;
    std::vector<uint64_t> key_tag;
    // nearest-plane engine (GPV, ring)
    bool has_np = false;
    int npiv = 0;
    bool ainv_identity = false;
    long ld_piv = 0;
    int ainv_nchunks = 0, ainv_bits = 0;
    Dev dPiv, dAinv[4], dMtP, dU, dS, dDg;
    int z_nchunks = 1, z_bits = 0;
    double zlimit = 0;
    // ring key
    bool has_ring = false, ring_ntt = false, ring_small = false;
    int ring_d = 1;
    uint32_t ring_np_inv = 0;
    Dev dAhat, dTw, dAraw, dAhat32, dTw32;
    // dense negacyclic matrix [rot^-(a_0) | ... | rot^-(a_{k+1})] mod q as u8 digit planes (n x n(k+2)): ring f_a
    // as one tensor-core contraction with the digit split of sigma fused in (rotation_matrix.rs:41-96)
    bool ring_dense = false;
    int ring_limbs = 0;
    Dev dRotl;
    std::vector<int64_t> hAring;
    // ring key table (qf_ring_set_key_table, DESIGN 4.13): key_count keys of (k+2) polynomials, independent of the installed
    // key.  key_family 2: ring_small transforms (uint32, d = key_d, np^-1 = key_np_inv, tables in dKeyTw); 1: Goldilocks
    // transforms (uint64, tables in dKeyTw); 0: the raw residues (int64, schoolbook).  dKeyIdx: key indices of the host
    // path's chunks.
    int64_t key_count = 0;
    int key_family = 0, key_d = 1;
    uint32_t key_np_inv = 0;
    Dev dKeyTab, dKeyTw, dKeyIdx;
    // workspace
    Dev w[12];  // (w[10]: digit planes of the particular solution)
    Dev dNorm, dFlag, dRetry, io_a, io_b, io_b2, io_c, io_a2, io_h[2];
    Dev io_p[2], io_n[2];  // packed Domain rows and their lengths (qf_samp_p_packed, qf_f_a_packed)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    cudaEvent_t ev_u_in[2] = {nullptr, nullptr}, ev_u_used[2] = {nullptr, nullptr};
    // tcgen05 int8 path for the exact integer contractions
    bool use_i8 = true;
    bool fused_fa = true;  // f_a: digit split fused into the contraction (gemm_i8_fused.cu)
    long ldk_dim = 0, ldk_nk = 0;
    int x_limbs = 0;       // digits for Domain-sized values (|.| <= sqrt(bound))
    int a_limbs = 0;       // u8 digits of a residue
    Dev dAl;               // A as a_limbs planes of n x ldk_dim
    Dev dRl;               // R as one s8 plane m_bar x ldk_nk
    Dev dSl;               // S as s_limbs planes of dim x ldk_dim
    int s_limbs = 0, z_limbs = 0;
    // G-trapdoor structure of the short basis, S = [[R S', I + R W],[S', W]] (short_basis_classical.rs:54-110),
    // recovered and verified exactly when the trapdoor is installed: e = S z then costs two thin contractions
    // (W z2 and R (S' z1 + W z2)) instead of the dense m x m one
    bool gpv_struct = false;
    int gpv_rev = 0, i2_limbs = 2;
    Dev dWl, dSkf;         // W as nk x ldk_mb u8 plane; S_k (k x k, fp64)
    long ldk_mb = 0;
    // tensor-core nearest-plane updates: fixed-point digit planes of U per 1024-column block
    bool use_ozaki = false;
    int u_limbs = 7;
    // centre -> GSO coordinates T = -Mt_P sol_P on tcgen05: fixed-point digit planes of Mt_P (one scale per row)
    bool mtp_i8 = false;
    Dev dMtPl, dMtPscale;
    long ldk_piv = 0;
    int sol_limbs = 0;
    bool np_fuse_split = true;  // the diagonal-block kernel writes the digit planes of z itself (no split pass over Z)
    bool np_fuse64 = true; // the rank-64 updates inside a 256-block run in the tail of the diagonal-block kernel
    int np_dlo = 2;        // digit sums below 256^np_dlo are dropped from the fixed-point updates (error budget: np_block)
    Dev dUl, dUscale, dNz, dMma;
    // highest non-zero digit plane of z per 256-block [0, n256), per 1024-block [n256, n256 + n1024), per 4096-block
    // [.., + n4096) and over the gadget-free block z2 [last]: written by the digit split, read by the conditional
    // contraction launches
    Dev dGate;
    int gate_n256 = 0, gate_n1024 = 0, gate_n4096 = 0;
    // Two-phase nearest plane for the G-trapdoor basis (samp_p_np2_chunk): the key is A = [A_bar | G - A_bar R] with the R
    // recovered from S (verified when the trapdoor is installed).  Fixed-point digit planes (one scale per row) of
    // Mt_1 = rows [0, nk) x columns [0, m_bar) of D^-1 B~^t (GSO coordinates of a centre -[z; 0]) and of
    // M' = Mt_1 [R; I] = U_11 S'^-1 (GSO coordinates of a centre -[R; I] g, g in gadget coordinates: block triangular);
    // digit counts / windows of the contractions (U_22 updates, the two centre maps, U_11 updates).
    bool gadget_key_ok = false, two_phase = false;
    Dev dMt1l, dMt1scale, dMpl, dMpscale;
    // Tagged G-trapdoor key A = [A_bar | H G - A_bar R], H invertible mod q (gadget_classical.rs:56-68): the recursion runs on
    // H^-1 A = [A_bar' | G - A_bar' R], A_bar' = H^-1 A_bar, which has the same lattice and the same short basis; a target u
    // becomes u' = H^-1 u.  u8 digit planes of H^-1 (n x ldk_n, one set per digit group of modq_contract) and of A_bar'
    // (n x ldk_mb); tag_ulimbs balanced digits of a residue (the split of u).  Set by detect_gpv_structure (PSFPerturbation:
    // key_tagged, dHinvl and tag_ulimbs by qf_set_trapdoor_perturbation / qf_set_tag), dropped with the key.
    bool key_tagged = false;
    int tag_ulimbs = 0;
    long ldk_n = 0;
    Dev dHinvl, dAbpl, dTagU, dTagUl, dTagTmp;
    // Tag table of samp_p (qf_set_tag_table; PSFPerturbation, and PSFGPV on the two-phase recursion): H_t^-1 mod q for
    // tag_count tags, each n x n column-major in words of tag_word bytes (4 when q <= 2^32), relative to the installed
    // (A_bar, R) and dropped with the key or trapdoor.
    // dTagH0: the installed key's tag H_0 in the same layout while the key is tagged; dTagGpow: base^s mod q, s < k;
    // io_t: tag indices of the host path's chunks (two slots, as io_b / io_b2).
    int64_t tag_count = 0;
    int tag_word = 8;
    Dev dTagTab, dTagH0, dTagGpow, io_t[2];
    // tag_poly: dTagTab holds the tags in polynomial form instead (qf_set_tag_table_poly, DESIGN 4.10): h_t^-1 mod (f, q)
    // as n words per tag, and dTagXr the rows X^{n+j} mod (f, q), j < n - 1, of the product.
    bool tag_poly = false;
    Dev dTagXr;
    // Tag table of f_a (qf_set_f_a_tags, PSFGPV and PSFPerturbation): D_t = H_t - H_0 mod q for fa_tag_count tags, in the
    // layout of dTagTab, relative to the installed A and dropped whenever A changes.  dFaSort: hist / off / gstart of the
    // counting sort by tag (3 (T + 1) ints); dFaPerm: the sorted targets of a chunk.
    int64_t fa_tag_count = 0;
    int fa_tag_word = 8;
    Dev dFaTab, dFaGpow, dFaSort, dFaPerm;
    // fa_poly: dFaTab holds h_t mod q as n words per tag instead (qf_set_f_a_tags_poly), dFaXr the rows of the product mod
    // (f, q) and dFaH0 H_0 column-major when fa_h0_kind = 2 (0: H_0 = 0, 1: H_0 = I).
    bool fa_poly = false;
    int fa_h0_kind = 1;
    Dev dFaXr, dFaH0;
    // Pool of the target-independent half of samp_p (qf_samp_p_offline, DESIGN 4.12): entries pool_first ..
    // pool_first + pool_count - 1 under pool_seed, entry j in slot j - pool_first; pool_next slots are consumed.
    // PSFPerturbation: dPoolX = p (m int32), dPoolAx = -A p mod q (n words).  PSFGPV two-phase: dPoolX = z2 (m_bar int32),
    // dPoolAx = -A_bar z2 mod q, dPoolT = -V 256^mt1_dlo of the Mt_1 z2 contraction (nk fp64, unit scale: dOnes).
    // Dropped whenever A or the trapdoor changes (drop_pool).
    bool pool = false;
    int64_t pool_count = 0, pool_next = 0;
    uint64_t pool_seed = 0, pool_first = 0;
    Dev dPoolX, dPoolAx, dPoolT, dOnes;
    // Defaults from the error budget of DESIGN 4.2, checked at the full C2 key (scripts/ab_c2_precision.py, profiles/README_r2.md):
    // four digits everywhere; the lowest digit sum is dropped where the operand has three digits (z2), not for the
    // two-digit z1 (dropping it there moves 14 % of the preimages, keeping it 0.3 %).
    int mt1_limbs = 4, mt1_dlo = 1, u22_limbs = 4, u22_dlo = 1, u11_limbs = 4, u11_dlo = 0, mt1g_limbs = 4;
    // digits / window / smallest compiled digit count of z for the update launches of the phase that is running
    int np_wdrop_cur = 0, np_dlo_cur = 2, np_lx_min = 3;
    int np_diag_variant = 0;
    long chunk_env = 0;
    // optional per-launch timing of the contraction kernels, CUDA events on ctx->stream
    bool prof = false;
    struct ProfRec { cudaEvent_t a, b; double flops; int kind; double issued; };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> ev_pool;

    qf_status fail(qf_status st, const std::string& msg) {
        err = msg;
        return st;
    }
    void drop_pool() {
        pool = false;
        pool_count = pool_next = 0;
        dPoolX.release(); dPoolAx.release(); dPoolT.release();
    }
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char buf__[256];                                                                       \
            snprintf(buf__, sizeof buf__, "CUDA error %s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
            return ctx->fail(QF_ERR_CUDA, buf__);                                                  \
        }                                                                                          \
    } while (0)
#define LAUNCH(call)          \
    do {                      \
        CK(call);             \
        ctx->launches += 1;   \
    } while (0)
#define QF_TRY(call)                     \
    do {                                 \
        qf_status s__ = (call);          \
        if (s__ != QF_OK) return s__;    \
    } while (0)

namespace {

// largest chunk width wb such that sum_k x_k w_k stays an exact fp64 integer:
// |partial sums| <= ||x|| * 2^wb * sqrt(K) < 2^53   (Cauchy-Schwarz)
int exact_bits(double x_norm, long K) {
    double b = 52.9 - std::log2(std::max(1.0, x_norm)) - 0.5 * std::log2((double)std::max(1L, K));
    return (int)std::floor(b);
}

// Upload a non-negative integer matrix (host int64, rows x cols) as `nchunks` fp64 matrices of
// `bits`-bit digits, each rows x ld.
qf_status upload_chunks(qf_ctx* ctx, const int64_t* h, long rows, long cols, long ld, int nchunks, int bits, Dev* dst) {
    std::vector<double> tmp((size_t)rows * ld, 0.0);
    for (int c = 0; c < nchunks; ++c) {
        const unsigned long long mask = (bits >= 64) ? ~0ull : ((1ull << bits) - 1);
        for (long i = 0; i < rows; ++i)
            for (long j = 0; j < cols; ++j) {
                unsigned long long v = (unsigned long long)h[i * cols + j];
                tmp[(size_t)i * ld + j] = (double)((v >> (c * bits)) & mask);
            }
        CK(dst[c].ensure(tmp.size() * sizeof(double)));
        CK(cudaMemcpyAsync(dst[c].p, tmp.data(), tmp.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return QF_OK;
}

template <typename T>
qf_status upload_as_f64(qf_ctx* ctx, const T* h, long rows, long cols, long ld, Dev& dst) {
    CK(dst.ensure((size_t)rows * ld * sizeof(double)));
    const long rows_per = std::max(1L, (long)((64L << 20) / (ld * (long)sizeof(double))));
    std::vector<double> tmp((size_t)rows_per * ld, 0.0);
    for (long r0 = 0; r0 < rows; r0 += rows_per) {
        long rr = std::min(rows_per, rows - r0);
        for (long i = 0; i < rr; ++i)
            for (long j = 0; j < cols; ++j) tmp[(size_t)i * ld + j] = (double)h[(r0 + i) * cols + j];
        CK(cudaMemcpyAsync(dst.as<double>() + (size_t)r0 * ld, tmp.data(), (size_t)rr * ld * sizeof(double),
                           cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return QF_OK;
}

qf_status check_flag(qf_ctx* ctx) {
    int h = 0;
    CK(cudaMemcpyAsync(&h, ctx->dFlag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (h) {
        CK(cudaMemsetAsync(ctx->dFlag.p, 0, sizeof(int), ctx->stream));
        if (h & 32) return ctx->fail(QF_ERR_INVALID, "target entry outside [0,q)");
        if (h & 64) return ctx->fail(QF_ERR_NUMERIC, "a Domain entry does not fit int16: use the int32 entry point");
        if (h & QF_FLAG_TAG_INDEX) return ctx->fail(QF_ERR_INVALID, "tag index outside the installed tag table");
        if (h & QF_FLAG_KEY_INDEX) return ctx->fail(QF_ERR_INVALID, "key index outside the installed ring key table");
        char buf[128];
        snprintf(buf, sizeof buf, "internal range check tripped (flag=%d): a value left its exact-integer range", h);
        return ctx->fail(QF_ERR_NUMERIC, buf);
    }
    return QF_OK;
}

// gemm_f64 launch with optional event timing (algorithmic flops: 2 B N K, triangular: B N (N+1))
cudaError_t ctx_gemm(qf_ctx* ctx, const double* X, long ldx, const double* W, long ldw, double* C, long ldc, int B, int N,
                     int K, double alpha, double beta, int tri) {
    qf_ctx::ProfRec rec{};
    if (ctx->prof) {
        for (cudaEvent_t* e : {&rec.a, &rec.b}) {
            if (!ctx->ev_pool.empty()) { *e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
            else if (cudaEventCreate(e) != cudaSuccess) return cudaErrorUnknown;
        }
        rec.flops = tri ? (double)B * N * (double)(std::min(N, K) + 1) : 2.0 * B * (double)N * K;
        cudaEventRecord(rec.a, ctx->stream);
    }
    cudaError_t e = qf_launch_gemm_f64(X, ldx, W, ldw, C, ldc, B, N, K, alpha, beta, tri, ctx->stream);
    if (ctx->prof) {
        cudaEventRecord(rec.b, ctx->stream);
        ctx->prof_recs.push_back(rec);
    }
    return e;
}

// smallest number of balanced base-256 digits that hold |v| <= maxabs
int limbs_for(double maxabs) {
    double cap = 127.0, pw = 1.0;
    int L = 1;
    while (cap < maxabs && L < 9) { pw *= 256.0; cap += 127.0 * pw; ++L; }
    return L;
}
double limb_capacity(int L) {
    double cap = 0, pw = 1.0;
    for (int l = 0; l < L; ++l) { cap += 127.0 * pw; pw *= 256.0; }
    return cap;
}

// integer matrix (host int64, rows x cols) -> L planes of rows x ldk bytes on the device
qf_status upload_limbs(qf_ctx* ctx, const int64_t* h, long rows, long cols, long ldk, int L, bool is_signed, Dev& dst) {
    std::vector<uint8_t> tmp((size_t)L * rows * ldk, 0);
    for (long i = 0; i < rows; ++i)
        for (long j = 0; j < cols; ++j) {
            long long v = h[i * cols + j];
            for (int l = 0; l < L; ++l) {
                long long lo;
                if (is_signed) {
                    lo = ((v + 128) & 255) - 128;
                    if (l == L - 1) lo = v;
                    v = (v - lo) >> 8;
                } else {
                    lo = v & 255;
                    v >>= 8;
                }
                tmp[((size_t)l * rows + i) * ldk + j] = (uint8_t)(lo & 255);
            }
        }
    CK(dst.ensure(tmp.size()));
    CK(cudaMemcpyAsync(dst.p, tmp.data(), tmp.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

// tcgen05 int8 contraction with optional event timing
cudaError_t ctx_gemm_i8(qf_ctx* ctx, const I8GemmArgs& a, bool count_ops = true) {
    qf_ctx::ProfRec rec{};
    if (ctx->prof) {
        for (cudaEvent_t* e : {&rec.a, &rec.b}) {
            if (!ctx->ev_pool.empty()) { *e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
            else if (cudaEventCreate(e) != cudaSuccess) return cudaErrorUnknown;
        }
        rec.kind = 1;
        // of the conditional launches of one contraction (gemm_i8_gated) exactly one runs: its work is counted once
        rec.flops = count_ops ? 2.0 * a.B * (double)a.N * a.K : 0.0;
        rec.issued = rec.flops * a.LX * a.LW;
        cudaEventRecord(rec.a, ctx->stream);
    }
    I8GemmArgs aa = a;
    aa.mma_units = (ctx->prof && ctx->dMma.p) ? ctx->dMma.as<unsigned long long>() : nullptr;
    static const bool trace = getenv("QF_TRACE") && getenv("QF_TRACE")[0] == '1';
    if (trace) {  // diagnostics only: per-launch time and executed digit pairs (synchronises)
        Dev cnt;
        cudaEvent_t t0, t1;
        if (cnt.ensure(40) != cudaSuccess) return cudaErrorMemoryAllocation;
        cudaMemsetAsync(cnt.p, 0, 40, ctx->stream);
        aa.mma_units = cnt.as<unsigned long long>();
        aa.tim = cnt.as<unsigned long long>() + 1;
        cudaEventCreate(&t0); cudaEventCreate(&t1);
        cudaEventRecord(t0, ctx->stream);
        cudaError_t e2 = qf_launch_gemm_i8(aa, ctx->stream);
        cudaEventRecord(t1, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        unsigned long long hh[5] = {0, 0, 0, 0, 0};
        cudaMemcpy(hh, cnt.p, 40, cudaMemcpyDeviceToHost);
        const unsigned long long h = hh[0];
        fprintf(stderr, "     per-CTA Mclk: mma-wait-tmem_empty %.2f  mma-wait-full %.2f  epi-wait-tmem_full %.2f  epi-body %.2f\n",
                hh[1] / 148e6, hh[2] / 148e6, hh[3] / 148e6, hh[4] / 148e6);
        const double nominal = 2.0 * a.B * (double)a.N * a.K;
        fprintf(stderr, "[i8] B=%d N=%d K=%d LX=%d LW=%d kind=%d  %.3f ms  pairs/mac=%.2f of %d  %.0f TOP/s executed\n", a.B, a.N,
                a.K, a.LX, a.LW, a.out_kind, ms, (double)h / nominal, a.LX * a.LW, (double)h / (ms * 1e-3) / 1e12);
        cudaEventDestroy(t0); cudaEventDestroy(t1);
        return e2;
    }
    cudaError_t e = qf_launch_gemm_i8(aa, ctx->stream);
    if (ctx->prof) {
        cudaEventRecord(rec.b, ctx->stream);
        ctx->prof_recs.push_back(rec);
    }
    return e;
}

// out = X W^t mod q (B x N, int64, ld N) for X = lx balanced s8 digit planes of B x K (row stride ldx, plane stride xp) and a
// key matrix W of residues in u8 digit planes (LW = ctx->a_limbs, N x K, row stride ldw).  Two pipeline stages of the
// contraction must hold all x planes in shared memory, which allows at most MODQ_MAX_LX of them (residues up to ~2^47).
// Wider x is taken in two digit groups, [0, MODQ_GROUP) and [MODQ_GROUP, lx): the second group multiplies the planes of
// 256^MODQ_GROUP W mod q (wg1) and starts from the first group's result (base), so the sum is reduced mod q exactly.
constexpr int MODQ_MAX_LX = 6, MODQ_GROUP = 4;
inline int modq_groups(int lx) { return lx > MODQ_MAX_LX ? 2 : 1; }

qf_status modq_contract(qf_ctx* ctx, const int8_t* x, long ldx, long xp, int lx, const void* wg0, const void* wg1, long ldw,
                        int B, int N, int K, int64_t* tmp, int64_t* out) {
    const int groups = modq_groups(lx);
    for (int gi = 0; gi < groups; ++gi) {
        const int l0 = gi ? MODQ_GROUP : 0, l1 = groups == 1 ? lx : (gi ? lx : MODQ_GROUP);
        I8GemmArgs g{};
        g.x = x + l0 * xp; g.ldx = ldx; g.x_plane = xp;
        g.w = gi ? wg1 : wg0; g.ldw = ldw; g.w_plane = N * ldw;
        g.LX = l1 - l0; g.LW = ctx->a_limbs; g.w_signed = 0;
        g.B = B; g.N = N; g.K = K;
        g.out_kind = 0; g.sign = 1; g.q = ctx->prm.q;
        g.base = gi ? tmp : nullptr; g.ldbase = N;
        g.out = (gi + 1 == groups) ? out : tmp; g.ldout = N;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    }
    return QF_OK;
}

// Tagged key: v' = H^-1 v mod q for Bc residue vectors v (row stride n) -- tag_ulimbs balanced digits of v against the digit
// planes of H^-1 (dHinvl).  *out = the device buffer holding v' (row stride n).
qf_status tag_targets(qf_ctx* ctx, const int64_t* dV, int Bc, const int64_t** out) {
    const long n = ctx->n, C = ctx->chunk, ldkn = ctx->ldk_n, tplane = C * ldkn;
    CK(ctx->dTagUl.ensure((size_t)ctx->tag_ulimbs * tplane));
    CK(ctx->dTagU.ensure((size_t)C * n * 8));
    if (modq_groups(ctx->tag_ulimbs) > 1) CK(ctx->dTagTmp.ensure((size_t)C * n * 8));
    LAUNCH(qf_launch_split_i64_limbs(dV, n, ctx->dTagUl.as<int8_t>(), tplane, ldkn, Bc, (int)n, ctx->tag_ulimbs,
                                     ctx->dFlag.as<int>(), ctx->stream));
    const uint8_t* hl = ctx->dHinvl.as<uint8_t>();
    QF_TRY(modq_contract(ctx, ctx->dTagUl.as<int8_t>(), ldkn, tplane, ctx->tag_ulimbs, hl, hl + (size_t)ctx->a_limbs * n * ldkn,
                         ldkn, Bc, (int)n, (int)n, ctx->dTagTmp.as<int64_t>(), ctx->dTagU.as<int64_t>()));
    *out = ctx->dTagU.as<int64_t>();
    return QF_OK;
}

// ---------------------------------------------------------------------------
// exact  out = X * W^t  with W given as non-negative fp64 digit matrices
// ---------------------------------------------------------------------------
qf_status gemm_chunks(qf_ctx* ctx, const double* X, long ldx, Dev* W, int nchunks, long ldw, double** acc, long ldacc,
                      int B, int N, int K) {
    for (int c = 0; c < nchunks; ++c)
        LAUNCH(ctx_gemm(ctx, X, ldx, W[c].as<double>(), ldw, acc[c], ldacc, B, N, K, 1.0, 0.0, 0));
    return QF_OK;
}

// ---------------------------------------------------------------------------
// f_a / check_domain on one chunk (classical)
// ---------------------------------------------------------------------------
qf_status f_a_chunk(qf_ctx* ctx, const int32_t* dSigma, int Bc, int64_t* dU, uint8_t* dFlags) {
    const long ldm = ctx->ld_dim, ldn = ctx->ld_n;
    if (ctx->use_i8 && ctx->fused_fa && ctx->x_limbs <= 4) {
        // one kernel: sigma (int32) -> digits in shared memory -> tcgen05, norms on the way
        CK(ctx->dNorm.ensure((size_t)std::max<int64_t>(ctx->chunk, Bc) * 8));
        int64_t* out = dU;
        if (!out) {  // check_domain only: the contraction still runs (cheap), into scratch
            CK(ctx->w[1].ensure((size_t)std::max<int64_t>(ctx->chunk, Bc) * ctx->n * 8));
            out = ctx->w[1].as<int64_t>();
        }
        FaFusedArgs g{};
        g.x = dSigma; g.ldx = ctx->dim;
        g.w = ctx->dAl.p; g.ldw = ctx->ldk_dim; g.w_plane = (long)ctx->n * ctx->ldk_dim;
        g.LX = ctx->x_limbs; g.LW = ctx->a_limbs; g.w_signed = 0;
        g.LX_typical = limbs_for(6.0 * ctx->s_samp_d + 1.0);
        g.B = Bc; g.N = (int)ctx->n; g.K = (int)ctx->m;
        g.q = ctx->prm.q; g.out = out; g.ldout = ctx->n;
        g.norm2 = ctx->dNorm.as<unsigned long long>();
        CK(ctx->dRetry.ensure(sizeof(int)));
        g.retry_flag = ctx->dRetry.as<int>();
        qf_ctx::ProfRec rec{};
        if (ctx->prof) {
            for (cudaEvent_t* e : {&rec.a, &rec.b}) {
                if (!ctx->ev_pool.empty()) { *e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
                else CK(cudaEventCreate(e));
            }
            rec.kind = 1;
            rec.flops = 2.0 * Bc * (double)ctx->n * ctx->m;
            rec.issued = rec.flops * g.LX * g.LW;
            CK(cudaEventRecord(rec.a, ctx->stream));
            g.mma_units = ctx->dMma.p ? ctx->dMma.as<unsigned long long>() : nullptr;
        }
        static const bool trace = getenv("QF_TRACE") && getenv("QF_TRACE")[0] == '1';
        Dev cnt;
        if (trace) {  // diagnostics only (synchronises): where the CTAs of the fused kernel spend their cycles
            CK(cnt.ensure(48));
            CK(cudaMemsetAsync(cnt.p, 0, 48, ctx->stream));
            g.tim = cnt.as<unsigned long long>();
        }
        LAUNCH(qf_launch_f_a_fused(g, ctx->stream));
        if (trace) {
            unsigned long long hh[6];
            CK(cudaStreamSynchronize(ctx->stream));
            CK(cudaMemcpy(hh, cnt.p, 48, cudaMemcpyDeviceToHost));
            const double ctas = (double)((Bc + 127) / 128) * ((ctx->n + 127) / 128), kbs = (double)((ctx->m + 127) / 128);
            fprintf(stderr, "[f_a fused] B=%d: per CTA kclk: whole %.1f  mma loop %.1f (waiting for operands %.1f)  converter loop %.1f "
                    "(waiting for free stages %.1f)  epilogue %.1f   per k block: %.0f clk\n", Bc, hh[5] / ctas / 1e3, hh[1] / ctas / 1e3,
                    hh[0] / ctas / 1e3, hh[3] / ctas / 1e3, hh[2] / ctas / 1e3, hh[4] / ctas / 1e3, hh[1] / ctas / kbs);
        }
        if (ctx->prof) {
            CK(cudaEventRecord(rec.b, ctx->stream));
            ctx->prof_recs.push_back(rec);
        }
        if (dFlags)
            LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, dFlags, Bc, ctx->stream));
        return QF_OK;
    }
    if (ctx->use_i8) {
        const long ldk = ctx->ldk_dim, plane = (long)ctx->chunk * ldk;
        CK(ctx->w[0].ensure((size_t)ctx->x_limbs * plane));
        CK(ctx->dNorm.ensure((size_t)ctx->chunk * 8));
        const int nz_m = (int)((ctx->chunk + 127) / 128), nz_kb = (int)(ldk / 128);
        const size_t nzb = (size_t)ctx->x_limbs * nz_m * nz_kb;
        CK(ctx->dNz.ensure(nzb));
        CK(cudaMemsetAsync(ctx->dNz.p, 0, nzb, ctx->stream));
        LAUNCH(qf_launch_split_i32_limbs(dSigma, ctx->dim, ctx->w[0].as<int8_t>(), plane, ldk, Bc, (int)ctx->dim,
                                         ctx->x_limbs, ctx->dNorm.as<unsigned long long>(), ctx->dNz.as<uint8_t>(), nz_m,
                                         nz_kb, ctx->stream));
        if (dFlags)
            LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, dFlags, Bc, ctx->stream));
        if (dU) {
            I8GemmArgs g{};
            g.x = ctx->w[0].as<int8_t>(); g.ldx = ldk; g.x_plane = plane;
            g.w = ctx->dAl.p; g.ldw = ldk; g.w_plane = (long)ctx->n * ldk;
            g.LX = ctx->x_limbs; g.LW = ctx->a_limbs; g.w_signed = 0;
            g.B = Bc; g.N = (int)ctx->n; g.K = (int)ctx->m;
            g.out_kind = 0; g.sign = 1; g.q = ctx->prm.q; g.base = nullptr; g.ldbase = 0; g.out = dU; g.ldout = ctx->n;
            g.flag = ctx->dFlag.as<int>();
            g.x_nz = ctx->dNz.as<uint8_t>(); g.nz_m_tiles = nz_m; g.nz_kb_total = nz_kb;
            LAUNCH(ctx_gemm_i8(ctx, g));
        }
        return QF_OK;
    }
    CK(ctx->w[0].ensure((size_t)ctx->chunk * ldm * 8));
    CK(ctx->dNorm.ensure((size_t)ctx->chunk * 8));
    double* X = ctx->w[0].as<double>();
    LAUNCH(qf_launch_i32_to_f64(dSigma, ctx->dim, X, ldm, Bc, (int)ctx->dim, ctx->dNorm.as<unsigned long long>(),
                                ctx->stream));
    if (dFlags)
        LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, dFlags, Bc, ctx->stream));
    if (dU) {
        double* acc[4] = {nullptr, nullptr, nullptr, nullptr};
        CombineArgs ca{};
        for (int c = 0; c < ctx->a_nchunks; ++c) {
            CK(ctx->w[1 + c].ensure((size_t)ctx->chunk * ldn * 8));
            acc[c] = ctx->w[1 + c].as<double>();
            ca.acc[c] = acc[c];
            ca.shift[c] = c * ctx->a_bits;
        }
        QF_TRY(gemm_chunks(ctx, X, ldm, ctx->dA, ctx->a_nchunks, ldm, acc, ldn, Bc, (int)ctx->n, (int)ctx->m));
        ca.nacc = ctx->a_nchunks; ca.acc_sign = 1; ca.ldacc = ldn; ca.base = nullptr; ca.ldbase = 0; ca.q = ctx->prm.q;
        LAUNCH(qf_launch_combine_i64(ca, dU, ctx->n, Bc, (int)ctx->n, ctx->stream));
    }
    return QF_OK;
}

qf_status ring_f_a_chunk(qf_ctx* ctx, const int32_t* dSigma, int Bc, int64_t* dU, uint8_t* dFlags) {
    CK(ctx->dNorm.ensure((size_t)std::max<int64_t>(ctx->chunk, Bc) * 8));
    const int npoly = (int)(ctx->k + 2);
    int64_t* out = dU;
    if (!out) {
        CK(ctx->w[1].ensure((size_t)std::max<int64_t>(ctx->chunk, Bc) * ctx->n * 8));
        out = ctx->w[1].as<int64_t>();
    }
    if (ctx->ring_dense && ctx->x_limbs <= 4) {
        FaFusedArgs g{};
        g.x = dSigma; g.ldx = ctx->dim;
        g.w = ctx->dRotl.p; g.ldw = ctx->ldk_dim; g.w_plane = (long)ctx->n * ctx->ldk_dim;
        g.LX = ctx->x_limbs; g.LW = ctx->ring_limbs; g.w_signed = 0;
        g.LX_typical = limbs_for(6.0 * ctx->s_samp_d + 1.0);
        g.B = Bc; g.N = (int)ctx->n; g.K = (int)ctx->dim;
        g.q = ctx->prm.q; g.out = out; g.ldout = ctx->n;
        g.norm2 = ctx->dNorm.as<unsigned long long>();
        CK(ctx->dRetry.ensure(sizeof(int)));
        g.retry_flag = ctx->dRetry.as<int>();
        LAUNCH(qf_launch_f_a_fused(g, ctx->stream));
    } else if (ctx->ring_small)
        LAUNCH(qf_launch_ring_small(dSigma, ctx->dAhat32.as<uint32_t>(), out, ctx->dNorm.as<unsigned long long>(), Bc, npoly,
                                    (int)ctx->n, ctx->ring_d, ctx->prm.q, ctx->ring_np_inv, ctx->dTw32.as<uint32_t>(),
                                    ctx->stream));
    else if (ctx->ring_ntt)
        LAUNCH(qf_launch_ring_f_a(dSigma, ctx->dAhat.as<uint64_t>(), out, ctx->dNorm.as<unsigned long long>(), Bc, npoly,
                                  (int)ctx->n, ctx->prm.q, ctx->dTw.as<uint64_t>(), ctx->stream));
    else
        LAUNCH(qf_launch_ring_f_a_schoolbook(dSigma, ctx->dAraw.as<int64_t>(), out, ctx->dNorm.as<unsigned long long>(),
                                             Bc, npoly, (int)ctx->n, ctx->prm.q, ctx->stream));
    if (dFlags)
        LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, dFlags, Bc, ctx->stream));
    return QF_OK;
}

// Family of the NTT kernels for a ring key table (qf_ring_set_key_table) or a batch of ring TrapGen products, by the rules
// of qf_ring_set_a: ring_small (2) for word-size NTT-friendly primes unless QF_DISABLE_SMALL_NTT=1, else Goldilocks (1)
// when n is a power of two in [64, 2048] and npoly n (q/2) max|sigma| < 2^63, else schoolbook (0).  Never the dense path.
int ring_key_family(unsigned long long q, long n, long npoly, double max_abs, int* d, std::vector<uint32_t>* tables,
                    uint32_t* np_inv) {
    const char* env = getenv("QF_DISABLE_SMALL_NTT");
    if (!(env && env[0] == '1') && qf_ring_small_plan(q, (int)n, d, tables, np_inv) != 0) return 2;
    if (n >= 64 && (n & (n - 1)) == 0 && n <= 2048 && (double)npoly * (double)n * ((double)q / 2) * max_abs < 9.0e18) return 1;
    return 0;
}

// Build the transforms of npolys key polynomials (raw residues, host) into tab (device) for a family, in slices of at
// most 2^16 polynomials through the staging buffer stage.  Family 0 copies the residues.  Enqueued on ctx->stream.
qf_status ring_key_transform(qf_ctx* ctx, const int64_t* keys, long npolys, int family, int d, const Dev& tw, Dev& tab,
                             Dev& stage) {
    const long n = ctx->n;
    const unsigned long long q = ctx->prm.q;
    if (family == 0) {
        CK(cudaMemcpyAsync(tab.p, keys, (size_t)npolys * n * 8, cudaMemcpyHostToDevice, ctx->stream));
        return QF_OK;
    }
    const long slice = std::min<long>(npolys, 1L << 16);
    CK(stage.ensure((size_t)slice * n * 8));
    for (long p0 = 0; p0 < npolys; p0 += slice) {
        const long np = std::min(slice, npolys - p0);
        CK(cudaMemcpyAsync(stage.p, keys + p0 * n, (size_t)np * n * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (family == 2)
            LAUNCH(qf_launch_ring_small_key(stage.as<int64_t>(), tab.as<uint32_t>() + p0 * n, np, (int)n, d, q,
                                            tw.as<uint32_t>(), ctx->stream));
        else
            LAUNCH(qf_launch_ring_prepare(stage.as<int64_t>(), tab.as<uint64_t>() + p0 * n, np, (int)n, q, tw.as<uint64_t>(),
                                          ctx->stream));
    }
    return QF_OK;
}

// Tables of a family (device): ring_small 3 np words, Goldilocks 2n + 1 words
qf_status ring_key_tables(qf_ctx* ctx, int family, const std::vector<uint32_t>& small, Dev& tw) {
    if (family == 2) {
        CK(tw.ensure(small.size() * 4));
        CK(cudaMemcpy(tw.p, small.data(), small.size() * 4, cudaMemcpyHostToDevice));
    } else if (family == 1) {
        std::vector<uint64_t> t(2 * ctx->n + 1);
        qf_ring_make_tables((int)ctx->n, t.data());
        CK(tw.ensure(t.size() * 8));
        CK(cudaMemcpy(tw.p, t.data(), t.size() * 8, cudaMemcpyHostToDevice));
    }
    return QF_OK;
}

// Keyed ring product: out[b] = sum_j a^(t)_j sigma[b][j] mod (X^n + 1, q) for t = dKidx[b], keys of npoly polynomials
// in tab (family, d, np_inv, tw as built by ring_key_transform); norm2 optional.
qf_status ring_keyed_launch(qf_ctx* ctx, int family, int d, uint32_t np_inv, const Dev& tw, const Dev& tab, int64_t nkeys,
                            const int32_t* dSigma, const int32_t* dKidx, int Bc, int npoly, int64_t* dU,
                            unsigned long long* norm2) {
    const int n = (int)ctx->n;
    const unsigned long long q = ctx->prm.q;
    int* flag = ctx->dFlag.as<int>();
    if (family == 2)
        LAUNCH(qf_launch_ring_small(dSigma, tab.as<uint32_t>(), dU, norm2, Bc, npoly, n, d, q, np_inv, tw.as<uint32_t>(),
                                    ctx->stream, dKidx, (int)nkeys, flag));
    else if (family == 1)
        LAUNCH(qf_launch_ring_f_a(dSigma, tab.as<uint64_t>(), dU, norm2, Bc, npoly, n, q, tw.as<uint64_t>(), ctx->stream, dKidx,
                                  (int)nkeys, flag));
    else
        LAUNCH(qf_launch_ring_f_a_schoolbook(dSigma, tab.as<int64_t>(), dU, norm2, Bc, npoly, n, q, ctx->stream, dKidx,
                                             (int)nkeys, flag));
    return QF_OK;
}

// ring f_a with a key per target (qf_ring_f_a_keyed): one keyed NTT-family launch, then the domain flags
qf_status ring_f_a_keyed_chunk(qf_ctx* ctx, const int32_t* dSigma, const int32_t* dKidx, int Bc, int64_t* dU, uint8_t* dFlags) {
    CK(ctx->dNorm.ensure((size_t)std::max<int64_t>(ctx->chunk, Bc) * 8));
    QF_TRY(ring_keyed_launch(ctx, ctx->key_family, ctx->key_d, ctx->key_np_inv, ctx->dKeyTw, ctx->dKeyTab, ctx->key_count,
                             dSigma, dKidx, Bc, (int)(ctx->k + 2), dU, ctx->dNorm.as<unsigned long long>()));
    LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, dFlags, Bc, ctx->stream));
    return QF_OK;
}

// ---------------------------------------------------------------------------
// PSFPerturbation::samp_p on one chunk (mp_perturbation.rs:304-336)
// ---------------------------------------------------------------------------
qf_status pert_lg_i8(qf_ctx* ctx, const int8_t* gp, long gplane, int Bc, double* X2, long ldx, bool tri);

// The chunk is split at the first read of the target (DESIGN 4.12): pert_perturbation and pert_ap (p and A p) are the
// offline half, pert_finish (from v = u - A p on) the online half.
qf_status pert_workspace(qf_ctx* ctx) {
    const long ldm = ctx->ld_dim, C = ctx->chunk;
    CK(ctx->w[0].ensure((size_t)C * ldm * 8));   // g, later reused
    CK(ctx->w[1].ensure((size_t)C * ldm * 8));   // x2 = sqrt(Sigma2) g
    CK(ctx->w[2].ensure((size_t)C * ldm * 8));   // p
    CK(ctx->w[3].ensure((size_t)C * ctx->ld_nk * 8));  // z
    CK(ctx->w[4].ensure((size_t)C * ctx->n * 8));  // v (int64)
    return QF_OK;
}

// p <- D_{Z^m, r sqrt(Sigma_2)} into P (w[2])
qf_status pert_perturbation(qf_ctx* ctx, int Bc, uint64_t seed, uint64_t first) {
    const long ldm = ctx->ld_dim;
    const long C = ctx->chunk;
    QF_TRY(pert_workspace(ctx));
    double* G = ctx->w[0].as<double>();
    double* X2 = ctx->w[1].as<double>();
    double* P = ctx->w[2].as<double>();
    // p <- D_{Z^m, r sqrt(Sigma_2)} : x2 = sqrt(Sigma_2) * N(0,I), p_i <- D_{Z, r, x2_i}   (:315)
    const bool st = ctx->pert_structured;
    if (st) CK(ctx->w[5].ensure((size_t)ctx->xb_limbs * C * ctx->ldk_nk));
    if (ctx->pert_i8) {
        // normals straight to fixed-point digits (no fp64 copy of g), x_2 = L g on tcgen05
        const long gplane = C * ctx->ldk_l;
        LAUNCH(qf_launch_pert_normal_digits(Bc, (int)ctx->m, st ? (int)ctx->m_bar : (int)ctx->m, seed, first,
                                            ctx->w[0].as<int8_t>(), gplane, ctx->ldk_l, ctx->lg_limbs, ctx->g_fscale, X2, ldm,
                                            st ? ctx->w[5].as<int8_t>() : nullptr, C * ctx->ldk_nk, ctx->ldk_nk, ctx->xb_limbs,
                                            ctx->sqrt_beta, ctx->xb_fscale, ctx->dFlag.as<int>(), ctx->stream));
        QF_TRY(pert_lg_i8(ctx, ctx->w[0].as<int8_t>(), gplane, Bc, X2, ldm, st ? true : ctx->l_tri != 0));
    } else {
        LAUNCH(qf_launch_normal_fill(G, ldm, Bc, (int)ctx->m, seed, first, QF_STREAM_PERT_NORMAL, ctx->stream));
        if (st) {
            // x_b = sqrt(beta) g_b (kept exact in x2, fixed-point digits for the tensor cores); x_t = L_s g_t
            LAUNCH(qf_launch_pert_xb(G, ldm, X2, ldm, ctx->w[5].as<int8_t>(), C * ctx->ldk_nk, ctx->ldk_nk, Bc, (int)ctx->m_bar,
                                     (int)ctx->nk, ctx->sqrt_beta, ctx->xb_fscale, ctx->xb_limbs, ctx->dFlag.as<int>(), ctx->stream));
            LAUNCH(ctx_gemm(ctx, G, ldm, ctx->dLs.as<double>(), ctx->ld_mb, X2, ldm, Bc, (int)ctx->m_bar, (int)ctx->m_bar, 1.0, 0.0, 1));
        } else {
            LAUNCH(ctx_gemm(ctx, G, ldm, ctx->dL.as<double>(), ldm, X2, ldm, Bc, (int)ctx->m, (int)ctx->m, 1.0, 0.0, ctx->l_tri));
        }
    }
    if (st) {
        // x_t -= kappa R x_b  (ternary R, fixed-point x_b) on tcgen05
        const long ldk = ctx->ldk_nk, plane = C * ldk;
        I8GemmArgs g{};
        g.x = ctx->w[5].as<int8_t>(); g.ldx = ldk; g.x_plane = plane;
        g.w = ctx->dRl.p; g.ldw = ldk; g.w_plane = (long)ctx->m_bar * ldk;
        g.LX = ctx->xb_limbs; g.LW = 1; g.w_signed = 1;
        g.B = Bc; g.N = (int)ctx->m_bar; g.K = (int)ctx->nk;
        g.out_kind = 3; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = X2; g.ldout = ldm;
        g.flag = ctx->dFlag.as<int>();
        g.scale = ctx->dXbScale.as<double>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    }
    LAUNCH(qf_launch_dgauss(X2, ldm, P, ldm, nullptr, 0, Bc, (int)ctx->m, ctx->prm.r, seed, first, QF_STREAM_PERT_ROUND,
                            ctx->dFlag.as<int>(), ctx->stream));
    return QF_OK;
}

// V = (base - A p) mod q for the p in P (base == nullptr: -A p mod q)   (:318)
qf_status pert_ap(qf_ctx* ctx, const int64_t* dUin, int Bc, int64_t* V) {
    const long ldm = ctx->ld_dim, ldn = ctx->ld_n, C = ctx->chunk;
    double* P = ctx->w[2].as<double>();
    if (ctx->use_i8) {
        const long ldk = ctx->ldk_dim, plane = C * ldk;
        CK(ctx->w[0].ensure((size_t)ctx->x_limbs * plane));  // g is dead: reuse as digit planes of p
        LAUNCH(qf_launch_split_f64_limbs(P, ldm, ctx->w[0].as<int8_t>(), plane, ldk, Bc, (int)ctx->m, ctx->x_limbs,
                                         ctx->dFlag.as<int>(), nullptr, 0, 0, 0, ctx->stream));
        I8GemmArgs g{};
        g.x = ctx->w[0].as<int8_t>(); g.ldx = ldk; g.x_plane = plane;
        g.w = ctx->dAl.p; g.ldw = ldk; g.w_plane = (long)ctx->n * ldk;
        g.LX = ctx->x_limbs; g.LW = ctx->a_limbs; g.w_signed = 0;
        g.B = Bc; g.N = (int)ctx->n; g.K = (int)ctx->m;
        g.out_kind = 0; g.sign = -1; g.q = ctx->prm.q; g.base = dUin; g.ldbase = ctx->n; g.out = V; g.ldout = ctx->n;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    } else {
        double* acc[4] = {nullptr, nullptr, nullptr, nullptr};
        CombineArgs ca{};
        for (int c = 0; c < ctx->a_nchunks; ++c) {
            CK(ctx->w[5 + c].ensure((size_t)C * ldn * 8));
            acc[c] = ctx->w[5 + c].as<double>();
            ca.acc[c] = acc[c];
            ca.shift[c] = c * ctx->a_bits;
        }
        QF_TRY(gemm_chunks(ctx, P, ldm, ctx->dA, ctx->a_nchunks, ldm, acc, ldn, Bc, (int)ctx->n, (int)ctx->m));
        ca.nacc = ctx->a_nchunks; ca.acc_sign = -1; ca.ldacc = ldn; ca.base = dUin; ca.ldbase = ctx->n; ca.q = ctx->prm.q;
        LAUNCH(qf_launch_combine_i64(ca, V, ctx->n, Bc, (int)ctx->n, ctx->stream));
    }
    return QF_OK;
}

// from v = u - A p (V, w[4]) and p (P, w[2]) on: the gadget preimage z and e = p + [R; I] z
// dTidx (optional, device): the tag index of every target of the chunk in the installed tag table (qf_samp_p_tagged)
qf_status pert_finish(qf_ctx* ctx, int Bc, uint64_t seed, uint64_t first, int32_t* dE, const int32_t* dTidx) {
    const long ldm = ctx->ld_dim, ldnk = ctx->ld_nk, C = ctx->chunk;
    double* P = ctx->w[2].as<double>();
    double* Z = ctx->w[3].as<double>();
    const int64_t* V = ctx->w[4].as<int64_t>();
    // tagged key A = [A_bar | H G - A_bar R]: A [R; I] = H G, so z solves G z = v' = H^-1 v
    const int64_t* Vg = V;
    if (dTidx) {
        // per-target tag H_t: A_t = A + [0 | (H_t - H_0) G], so v'_t = H_t^-1 (u - A_t p) = H_t^-1 (v + H_0 y) - y with
        // y = G p_bot (DESIGN 4.4): the same v' as after qf_set_tag(H_t)
        CK(ctx->dTagU.ensure((size_t)C * ctx->n * 8));
        LAUNCH(qf_launch_tag_syndrome(V, ctx->n, P, ldm, (int)ctx->m_bar, dTidx, (int)ctx->tag_count, ctx->dTagTab.p,
                                      ctx->key_tagged ? ctx->dTagH0.p : nullptr, ctx->tag_word, ctx->dTagGpow.as<uint64_t>(),
                                      ctx->prm.q, (int)ctx->n, (int)ctx->k, Bc, ctx->dTagU.as<int64_t>(), ctx->n,
                                      ctx->dFlag.as<int>(), ctx->stream, ctx->tag_poly ? ctx->dTagXr.p : nullptr));
        Vg = ctx->dTagU.as<int64_t>();
    } else if (ctx->key_tagged) {
        QF_TRY(tag_targets(ctx, V, Bc, &Vg));
    }
    // z <- D_{Lambda_v^perp(G), r sqrt(b^2+1)}   (:321-326 -> :173-191)
    const double s_g = ctx->prm.r * std::sqrt((double)(ctx->prm.base * ctx->prm.base + 1));
    LAUNCH(qf_launch_gadget_sample(Vg, ctx->n, Z, ldnk, Bc, (int)ctx->n, (int)ctx->k, (int)ctx->prm.base, ctx->prm.q,
                                   ctx->dSk.as<double>(), ctx->dSkGso.as<double>(), s_g, seed, first, ctx->dFlag.as<int>(),
                                   ctx->stream));
    // e = p + [R; I] z   (:328-335): top block accumulates R z into p in place (exact small integers)
    if (ctx->use_i8) {
        const long ldk = ctx->ldk_nk, plane = C * ldk;
        const int LZ = 2;
        CK(ctx->w[1].ensure((size_t)LZ * plane));  // x2 is dead: reuse as digit planes of z
        LAUNCH(qf_launch_split_f64_limbs(Z, ldnk, ctx->w[1].as<int8_t>(), plane, ldk, Bc, (int)ctx->nk, LZ,
                                         ctx->dFlag.as<int>(), nullptr, 0, 0, 0, ctx->stream));
        I8GemmArgs g{};
        g.x = ctx->w[1].as<int8_t>(); g.ldx = ldk; g.x_plane = plane;
        g.w = ctx->dRl.p; g.ldw = ldk; g.w_plane = (long)ctx->m_bar * ldk;
        g.LX = LZ; g.LW = 1; g.w_signed = 1;
        g.B = Bc; g.N = (int)ctx->m_bar; g.K = (int)ctx->nk;
        g.out_kind = 2; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = P; g.ldout = ldm;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    } else {
        LAUNCH(ctx_gemm(ctx, Z, ldnk, ctx->dR.as<double>(), ldnk, P, ldm, Bc, (int)ctx->m_bar, (int)ctx->nk, 1.0, 1.0, 0));
    }
    LAUNCH(qf_launch_finalize_pert(P, ldm, Z, ldnk, dE, ctx->m, Bc, (int)ctx->m, (int)ctx->m_bar, ctx->dFlag.as<int>(),
                                   ctx->stream));
    return QF_OK;
}

qf_status samp_p_pert_chunk(qf_ctx* ctx, const int64_t* dUin, int Bc, uint64_t seed, uint64_t first, int32_t* dE,
                            const int32_t* dTidx = nullptr) {
    QF_TRY(pert_perturbation(ctx, Bc, seed, first));
    QF_TRY(pert_ap(ctx, dUin, Bc, ctx->w[4].as<int64_t>()));
    return pert_finish(ctx, Bc, seed, first, dE, dTidx);
}

// ---------------------------------------------------------------------------
// GPV / ring samp_p on one chunk: GPV08 SampleD in GSO coordinates (gpv.rs:152-161,
// gpv_ring.rs:160-212)
// ---------------------------------------------------------------------------
// Block sizes of the recursion: 64-wide diagonal blocks are sequential per target (np_diag, which also applies the rank-64
// updates inside its 256-block); the updates between 256-blocks inside a 1024-block, between 1024-blocks inside a
// 4096-block and between 4096-blocks run on tcgen05 (fixed-point digits); fp64 GEMMs (gemm_f64) remain for dimensions
// below the tensor-core threshold.  The top level contracts K = 4096 coordinates per launch: its epilogue
// (a read-modify-write of T, serialised with the MMAs because TMEM holds one tile) is paid once per 4096 instead of
// once per 1024 coordinates.
constexpr long NP_SIZES[4] = {64, 256, 1024, 4096};
constexpr int NP_TOP = 4;
constexpr long NP_SCALE_BLOCK = NP_SIZES[3];  // column block over which the digits of U share one scale per row
constexpr long NP_THIN = 512;                 // a ragged top block narrower than this is merged into the block below it
constexpr long NP_PROP_LD = NP_SIZES[2] + NP_THIN;  // proposals of one (possibly merged) 1024-block, per target

// Blocks of step S over [0, D): [b S, (b+1) S), except that a ragged remainder narrower than NP_THIN at the top joins the
// last full block (a thin block would cost a whole read-modify-write pass over T for a handful of coordinates:
// D = 12352 = 3 * 4096 + 64).  Returns the start of the last block.
static long np_last_block_start(long D, long S) {
    long top = (D - 1) / S * S;
    if (top > 0 && D - top < NP_THIN) top -= S;
    return top;
}

// One contraction with the z digit planes as x operand, launched once per digit count LXv in [3, z_limbs]: every launch is
// conditional on the device-side gate (highest non-zero digit plane of the z block it consumes), so exactly one of them
// runs -- the one compiled for the digits that are really there (fewer accumulators in TMEM = wider tiles, less operand
// traffic per MAC).  Without a gate a single launch with all z_limbs digits.
qf_status gemm_i8_gated(qf_ctx* ctx, I8GemmArgs g, const int* gate, int lx_min = 3) {
    const int Lmax = g.LX;
    if (!gate || Lmax <= lx_min) {
        LAUNCH(ctx_gemm_i8(ctx, g));
        return QF_OK;
    }
    for (int lx = lx_min; lx <= Lmax; ++lx) {
        I8GemmArgs v = g;
        v.LX = lx;
        v.gate = gate;
        v.gate_lo = lx == lx_min ? 0 : lx - 1;
        v.gate_hi = lx == Lmax ? 1 << 20 : lx - 1;
        LAUNCH(ctx_gemm_i8(ctx, v, lx == Lmax));
    }
    return QF_OK;
}

// column -> index of its block at step S (the ragged top joins the last full block, np_last_block_start)
static inline int np_block_index(long col, long D, long S) {
    return (int)(std::min(col, np_last_block_start(D, S)) / S);
}

// Process coordinates [lo, hi) in descending order.  Precondition: T[:, lo:hi] already carries the
// updates of every coordinate >= hi.  level 0 = one sequential diagonal block.  prop0 = first coordinate of the
// enclosing 1024-level block (origin of the pre-generated proposals).
qf_status np_block(qf_ctx* ctx, double* T, double* Z, int Bc, long lo, long hi, int level, long prop0, uint64_t seed,
                   uint64_t first) {
    const long D = ctx->dim, ldD = ctx->ld_dim;
    const double* U = ctx->dU.as<double>();
    if (level == 0) {
        // [lo, hi) wider than 64: a whole 256-block, the kernel walks its diagonal blocks and fuses the rank-64 updates
        NpDigitOut dig{};
        const bool fuse_digits = ctx->use_ozaki && ctx->np_fuse_split;
        if (fuse_digits && (lo & 63)) return ctx->fail(QF_ERR_NUMERIC, "internal: diagonal block not 64-aligned");
        if (fuse_digits) {  // the digit planes of this block of z, written by the kernel that produced it
            const long ldk = ctx->ldk_dim;
            int* gates = ctx->dGate.as<int>();
            dig.planes = ctx->w[8].as<int8_t>(); dig.plane_stride = (long)ctx->chunk * ldk; dig.ldk = ldk; dig.L = ctx->z_limbs;
            dig.nz = ctx->dNz.as<uint8_t>(); dig.nz_m_tiles = (int)((ctx->chunk + 127) / 128); dig.nz_kb_total = (int)(ldk / 128);
            dig.gate[0] = gates + np_block_index(lo, D, NP_SIZES[1]);
            dig.gate[1] = gates + ctx->gate_n256 + np_block_index(lo, D, NP_SIZES[2]);
            dig.gate[2] = gates + ctx->gate_n256 + ctx->gate_n1024 + np_block_index(lo, D, NP_SIZES[3]);
            dig.gate[3] = (ctx->gpv_struct && hi > ctx->nk) ? gates + ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096 : nullptr;
        }
        LAUNCH(qf_launch_np_diag(T, ldD, Z, ldD, U, ldD, ctx->dDg.as<DGaussParams>(),
                                 ctx->w[9].as<float4>(), ctx->chunk, Bc, (int)lo, (int)(hi - lo), (int)D,
                                 seed, first, ctx->zlimit, ctx->dFlag.as<int>(), ctx->stream, (int)lo, fuse_digits ? &dig : nullptr,
                                 (int)prop0, ctx->np_diag_variant));
        return QF_OK;
    }
    if (level == 1 && ctx->np_fuse64 && (lo & 63) == 0)
        // a whole 256-block in one launch: its diagonal blocks and the rank-64 updates between them (lattice.cu)
        return np_block(ctx, T, Z, Bc, lo, hi, 0, prop0, seed, first);
    const long step = NP_SIZES[level - 1];
    const bool i8_level = level >= 2 && ctx->use_ozaki;
    for (long sub_hi = hi; sub_hi > lo;) {
        long sub_lo = std::max(lo, (sub_hi - 1) / step * step);
        // tensor-core levels: the ragged top of the whole recursion joins the block below it (the digit planes of U are
        // masked and scaled for exactly this partition, see setup: np_last_block_start)
        if (i8_level && sub_hi == D && sub_lo > lo && sub_hi - sub_lo < NP_THIN) sub_lo = std::max(lo, sub_lo - step);
        if (level == 3) {
            // the rejection-sampling proposals of this 1024-block for all targets, at full occupancy
            CK(ctx->w[9].ensure((size_t)ctx->chunk * NP_PROP_LD * sizeof(float4)));
            // (coordinate-major: row i holds the proposals of all targets of the chunk for coordinate sub_lo + i)
            LAUNCH(qf_launch_np_propose(ctx->w[9].as<float4>(), ctx->chunk, Bc, (int)sub_lo, (int)(sub_hi - sub_lo), (int)D,
                                        seed, first, ctx->stream));
            prop0 = sub_lo;
        }
        QF_TRY(np_block(ctx, T, Z, Bc, sub_lo, sub_hi, level - 1, prop0, seed, first));
        if (i8_level) {
            const long ldk = ctx->ldk_dim, plane = (long)ctx->chunk * ldk;
            const int nz_m = (int)((ctx->chunk + 127) / 128), nz_kb = (int)(ldk / 128);
            int8_t* zp = ctx->w[8].as<int8_t>();
            int* gates = ctx->dGate.as<int>();
            int* gate0 = gates + np_block_index(sub_lo, D, NP_SIZES[1]);
            int* gate1 = gates + ctx->gate_n256 + np_block_index(sub_lo, D, NP_SIZES[2]);
            int* gate4 = gates + ctx->gate_n256 + ctx->gate_n1024 + np_block_index(sub_lo, D, NP_SIZES[3]);
            int* gate_z2 = gates + ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096;
            // digits of the finished 256-block of z (kept: the levels above and the final S z reuse them) -- unless the
            // diagonal-block kernels have written them already
            if (level == 2 && !ctx->np_fuse_split)
                LAUNCH(qf_launch_split_f64_limbs(Z + sub_lo, ldD, zp + sub_lo, plane, ldk, Bc, (int)(sub_hi - sub_lo), ctx->z_limbs,
                                                 ctx->dFlag.as<int>(), ctx->dNz.as<uint8_t>(), nz_m, nz_kb, (int)sub_lo,
                                                 ctx->stream, gate0, gate1, gate4,
                                                 (ctx->gpv_struct && sub_hi > ctx->nk) ? gate_z2 : nullptr));
            // the update of the rows above it (within the enclosing block) on the tensor cores:
            //   T[:, lo:sub_lo] -= (z digits) x (fixed-point digits of U) * 2^-e
            if (sub_lo > lo && sub_hi - sub_lo < NP_SIZES[1]) {
                // a thin block: per-tile overheads dominate the tensor-core path, use fp64
                LAUNCH(ctx_gemm(ctx, Z + sub_lo, ldD, U + lo * ldD + sub_lo, ldD, T + lo, ldD, Bc, (int)(sub_lo - lo),
                                (int)(sub_hi - sub_lo), -1.0, 1.0, 0));
            } else if (sub_lo > lo) {
                I8GemmArgs g{};
                g.x = zp + sub_lo; g.ldx = ldk; g.x_plane = plane;
                // (two-phase recursion: only the top planes of U that the phase's error budget needs)
                const int wdrop = ctx->np_wdrop_cur;
                g.w = ctx->dUl.as<int8_t>() + (size_t)wdrop * D * ldk + lo * ldk + sub_lo; g.ldw = ldk; g.w_plane = D * ldk;
                g.LX = ctx->z_limbs; g.LW = ctx->u_limbs - wdrop; g.w_signed = 1;
                g.scale_mul = std::ldexp(1.0, 8 * wdrop);
                g.B = Bc; g.N = (int)(sub_lo - lo); g.K = (int)(sub_hi - sub_lo);
                g.out_kind = 3; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = T + lo; g.ldout = ldD;
                g.flag = ctx->dFlag.as<int>();
                g.scale = ctx->dUscale.as<double>() + (sub_lo / NP_SCALE_BLOCK) * D + lo;
                g.x_nz = ctx->dNz.as<uint8_t>(); g.nz_m_tiles = nz_m; g.nz_kb_total = nz_kb;
                g.nz_kb_off = (int)(sub_lo / 128); g.nz_m_off = 0;
                // Dropped digit sums d < np_dlo: per launch |error| <= K 2^14 256^(d_lo - 1) d_lo scale_row (scale_row =
                // row maximum of |U| / (127 256^6)), i.e. < 2^-27 |U|max K^(1/2) typically at d_lo = 2 -- four orders
                // below the 2^-12 the centres need (the widths s / ||b~_i|| are >= 2.3), and below the fp64 rounding of T
                // at |T| ~ 2^24.
                g.d_lo = ctx->np_dlo_cur;
                QF_TRY(gemm_i8_gated(ctx, g, level == 2 ? gate0 : level == 3 ? gate1 : gate4, ctx->np_lx_min));
            }
        } else if (sub_lo > lo) {
            LAUNCH(ctx_gemm(ctx, Z + sub_lo, ldD, U + lo * ldD + sub_lo, ldD, T + lo, ldD, Bc, (int)(sub_lo - lo),
                            (int)(sub_hi - sub_lo), -1.0, 1.0, 0));
        }
        sub_hi = sub_lo;
    }
    return QF_OK;
}

qf_status samp_p_np1_chunk(qf_ctx* ctx, const int64_t* dUin, int Bc, uint64_t seed, uint64_t first, int32_t* dE) {
    const long D = ctx->dim, ldD = ctx->ld_dim, ldp = ctx->ld_piv, C = ctx->chunk;
    const int np = ctx->npiv;
    CK(ctx->w[0].ensure((size_t)C * ldp * 8));  // u as fp64
    CK(ctx->w[1].ensure((size_t)C * ldp * 8));  // sol_P
    CK(ctx->w[2].ensure((size_t)C * ldD * 8));  // T
    CK(ctx->w[3].ensure((size_t)C * ldD * 8));  // Z
    double* Uf = ctx->w[0].as<double>();
    double* Sol = ctx->w[1].as<double>();
    double* T = ctx->w[2].as<double>();
    double* Z = ctx->w[3].as<double>();
    // particular solution on the pivot columns: sol_P = A_P^{-1} u mod q   (gpv.rs:153-156)
    if (ctx->ainv_identity) {
        LAUNCH(qf_launch_i64_to_f64(dUin, ctx->n, Sol, ldp, Bc, np, 1.0, ctx->stream));
    } else {
        LAUNCH(qf_launch_i64_to_f64(dUin, ctx->n, Uf, ldp, Bc, np, 1.0, ctx->stream));
        double* acc[4] = {nullptr, nullptr, nullptr, nullptr};
        CombineArgs ca{};
        for (int c = 0; c < ctx->ainv_nchunks; ++c) {
            CK(ctx->w[4 + c].ensure((size_t)C * ldD * 8));
            acc[c] = ctx->w[4 + c].as<double>();
            ca.acc[c] = acc[c];
            ca.shift[c] = c * ctx->ainv_bits;
        }
        QF_TRY(gemm_chunks(ctx, Uf, ldp, ctx->dAinv, ctx->ainv_nchunks, ldp, acc, ldp, Bc, np, np));
        ca.nacc = ctx->ainv_nchunks; ca.acc_sign = 1; ca.ldacc = ldp; ca.base = nullptr; ca.ldbase = 0; ca.q = ctx->prm.q;
        LAUNCH(qf_launch_combine_f64(ca, Sol, ldp, Bc, np, ctx->stream));
    }
    // centre c = -sol in GSO coordinates: T = -(B~^t D^-1)[:,P] sol_P   (gpv.rs:158)
    if (ctx->mtp_i8) {
        // exact digits of sol (residues < q) times fixed-point digits of Mt_P on the tensor cores; the epilogue stores
        // T = -V * scale (no read of T)
        const long ldkp = ctx->ldk_piv, planep = C * ldkp;
        CK(ctx->w[10].ensure((size_t)ctx->sol_limbs * planep));
        if (np < ldkp) CK(cudaMemsetAsync(ctx->w[10].p, 0, (size_t)ctx->sol_limbs * planep, ctx->stream));
        LAUNCH(qf_launch_split_f64_limbs(Sol, ldp, ctx->w[10].as<int8_t>(), planep, ldkp, Bc, np, ctx->sol_limbs,
                                         ctx->dFlag.as<int>(), nullptr, 0, 0, 0, ctx->stream));
        I8GemmArgs g{};
        g.x = ctx->w[10].as<int8_t>(); g.ldx = ldkp; g.x_plane = planep;
        g.w = ctx->dMtPl.p; g.ldw = ldkp; g.w_plane = D * ldkp;
        g.LX = ctx->sol_limbs; g.LW = ctx->u_limbs; g.w_signed = 1;
        g.B = Bc; g.N = (int)D; g.K = np;
        g.out_kind = 3; g.sign = 1; g.q = 0; g.out = T; g.ldout = ldD;
        g.flag = ctx->dFlag.as<int>();
        g.scale = ctx->dMtPscale.as<double>();
        g.d_lo = ctx->np_dlo; g.overwrite = 1;
        LAUNCH(ctx_gemm_i8(ctx, g));
    } else {
        LAUNCH(ctx_gemm(ctx, Sol, ldp, ctx->dMtP.as<double>(), ldp, T, ldD, Bc, (int)D, np, -1.0, 0.0, 0));
    }
    // randomized nearest plane, i = D-1 .. 0 (gpv.rs:160), blocked on three levels: 64-wide diagonal
    // blocks are sequential per target (np_diag); everything off the diagonal is a GEMM with K = 64, 256
    // or 1024, so that most of the work runs at K = 1024.
    if (ctx->use_ozaki) {
        const long ldk = ctx->ldk_dim;
        const size_t nzb = (size_t)ctx->z_limbs * ((ctx->chunk + 127) / 128) * (ldk / 128);
        CK(ctx->w[8].ensure((size_t)ctx->z_limbs * C * ldk));
        CK(ctx->dNz.ensure(nzb));
        CK(cudaMemsetAsync(ctx->dNz.p, 0, nzb, ctx->stream));
        ctx->gate_n256 = np_block_index(D - 1, D, NP_SIZES[1]) + 1;
        ctx->gate_n1024 = np_block_index(D - 1, D, NP_SIZES[2]) + 1;
        ctx->gate_n4096 = np_block_index(D - 1, D, NP_SIZES[3]) + 1;
        const size_t gb = (size_t)(ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096 + 1) * sizeof(int);
        CK(ctx->dGate.ensure(gb));
        CK(cudaMemsetAsync(ctx->dGate.p, 0, gb, ctx->stream));
    }
    ctx->np_wdrop_cur = 0; ctx->np_dlo_cur = ctx->np_dlo; ctx->np_lx_min = 3;
    QF_TRY(np_block(ctx, T, Z, Bc, 0, D, NP_TOP, 0, seed, first));
    // e = sol + S z   (exact integers)
    if (ctx->use_i8) {
        // z -> balanced base-256 digits, S z on the tensor cores, then add sol on its pivot columns
        const long ldk = ctx->ldk_dim, plane = C * ldk;
        int8_t* zp;
        I8GemmArgs g{};
        if (ctx->use_ozaki) {
            zp = ctx->w[8].as<int8_t>();  // digits were produced block by block during the recursion
            g.x_nz = ctx->dNz.as<uint8_t>(); g.nz_m_tiles = (int)((ctx->chunk + 127) / 128); g.nz_kb_total = (int)(ldk / 128);
        } else {
            CK(ctx->w[2].ensure((size_t)std::max<long>(ctx->z_limbs * plane, C * ldD * 8)));  // T is dead: reuse
            zp = ctx->w[2].as<int8_t>();
            LAUNCH(qf_launch_split_f64_limbs(Z, ldD, zp, plane, ldk, Bc, (int)D, ctx->z_limbs, ctx->dFlag.as<int>(), nullptr, 0,
                                             0, 0, ctx->stream));
        }
        if (ctx->gpv_struct) {
            // S z = [z2 + R i2 ; i2],  i2 = S' z1 + W z2  (z1 = z[0:nk], z2 = z[nk:m])
            const long nk = ctx->nk, mb = ctx->m_bar, ldnk = ctx->ld_nk, ldk_nk = ctx->ldk_nk;
            CK(ctx->w[4].ensure((size_t)C * ldnk * 8));
            double* I2 = ctx->w[4].as<double>();
            CK(cudaMemsetAsync(I2, 0, (size_t)Bc * ldnk * 8, ctx->stream));
            g.x = zp + nk; g.ldx = ldk; g.x_plane = plane;
            g.w = ctx->dWl.p; g.ldw = ctx->ldk_mb; g.w_plane = nk * ctx->ldk_mb;
            g.LX = ctx->z_limbs; g.LW = 1; g.w_signed = 0;
            g.B = Bc; g.N = (int)nk; g.K = (int)mb;
            g.out_kind = 2; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = I2; g.ldout = ldnk;
            g.flag = ctx->dFlag.as<int>();
            if (g.x_nz) g.nz_kb_off = (int)(nk / 128);
            QF_TRY(gemm_i8_gated(ctx, g, ctx->use_ozaki ? ctx->dGate.as<int>() + ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096 : nullptr));
            LAUNCH(qf_launch_sprime_apply(Z, ldD, I2, ldnk, Bc, (int)nk, (int)ctx->k, ctx->dSkf.as<double>(), ctx->gpv_rev,
                                          ctx->stream));
            const long plane2 = C * ldk_nk;
            CK(ctx->w[2].ensure((size_t)std::max<long>(ctx->i2_limbs * plane2, C * ldD * 8)));  // T is dead: digits of i2
            int8_t* ip = ctx->w[2].as<int8_t>();
            LAUNCH(qf_launch_split_f64_limbs(I2, ldnk, ip, plane2, ldk_nk, Bc, (int)nk, ctx->i2_limbs, ctx->dFlag.as<int>(),
                                             nullptr, 0, 0, 0, ctx->stream));
            I8GemmArgs h{};
            h.x = ip; h.ldx = ldk_nk; h.x_plane = plane2;
            h.w = ctx->dRl.p; h.ldw = ldk_nk; h.w_plane = mb * ldk_nk;
            h.LX = ctx->i2_limbs; h.LW = 1; h.w_signed = 1;
            h.B = Bc; h.N = (int)mb; h.K = (int)nk;
            h.out_kind = 1; h.sign = 1; h.q = 0; h.out = dE; h.ldout = D;
            h.flag = ctx->dFlag.as<int>();
            LAUNCH(ctx_gemm_i8(ctx, h));
            LAUNCH(qf_launch_gpv_struct_finalize(dE, D, Z + nk, ldD, I2, ldnk, Bc, (int)mb, (int)nk, ctx->dFlag.as<int>(),
                                                 ctx->stream));
        } else {
            g.x = zp; g.ldx = ldk; g.x_plane = plane;
            g.w = ctx->dSl.p; g.ldw = ldk; g.w_plane = D * ldk;
            g.LX = ctx->z_limbs; g.LW = ctx->s_limbs; g.w_signed = 1;
            g.B = Bc; g.N = (int)D; g.K = (int)D;
            g.out_kind = 1; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = dE; g.ldout = D;
            g.flag = ctx->dFlag.as<int>();
            LAUNCH(ctx_gemm_i8(ctx, g));
        }
        LAUNCH(qf_launch_add_cols_i32(dE, D, Sol, ldp, ctx->dPiv.as<int>(), np, Bc, ctx->stream));
    } else {
        double* acc[4] = {nullptr, nullptr, nullptr, nullptr};
        double* zc[4] = {nullptr, nullptr, nullptr, nullptr};
        CombineArgs ca{};
        const int nc = ctx->z_nchunks;
        for (int c = 0; c < nc; ++c) {
            CK(ctx->w[4 + c].ensure((size_t)C * ldD * 8));
            acc[c] = ctx->w[4 + c].as<double>();
            ca.acc[c] = acc[c];
            ca.shift[c] = c * ctx->z_bits;
        }
        if (nc > 1) {
            zc[0] = T;  // T is dead now
            for (int c = 1; c < nc; ++c) {
                CK(ctx->w[7 + c].ensure((size_t)C * ldD * 8));
                zc[c] = ctx->w[7 + c].as<double>();
            }
            LAUNCH(qf_launch_split_chunks(Z, ldD, zc, nc, ctx->z_bits, ldD, Bc, (int)D, ctx->stream));
        } else {
            zc[0] = Z;
        }
        // acc_0 starts as the particular solution scattered to its pivot columns
        CK(cudaMemsetAsync(acc[0], 0, (size_t)Bc * ldD * 8, ctx->stream));
        LAUNCH(qf_launch_scatter_cols_f64(Sol, ldp, ctx->dPiv.as<int>(), np, acc[0], ldD, Bc, 1.0, ctx->stream));
        for (int c = 0; c < nc; ++c)
            LAUNCH(ctx_gemm(ctx, zc[c], ldD, ctx->dS.as<double>(), ldD, acc[c], ldD, Bc, (int)D, (int)D, 1.0,
                                      c == 0 ? 1.0 : 0.0, 0));
        ca.nacc = nc; ca.acc_sign = 1; ca.ldacc = ldD; ca.base = nullptr; ca.ldbase = 0; ca.q = 0;
        LAUNCH(qf_launch_combine_i32(ca, dE, D, Bc, (int)D, ctx->dFlag.as<int>(), ctx->stream));
    }
    return QF_OK;
}

// ---------------------------------------------------------------------------
// PSFGPV::samp_p for the G-trapdoor basis S = [[R S', I + R W],[S', W]] of A = [A_bar | G - A_bar R], in two phases.
//
// The reference loop (gpv.rs:152-161, MatZ::sample_d_precomputed_gso) walks i = m-1 .. 0 with centre -sol.  Its output law
// depends on the centre only modulo the lattice, and -- at step i -- only modulo the sub-lattice spanned by b_0 .. b_i
// (a shift by such a vector moves c'_i .. c'_0 by integers and z by the same integers: the same e).  So
//   phase 1 (i = m-1 .. nk): centre -x with the gadget preimage x = [R g; g], g = digits(u)  (A x = u).  x lies in the real
//            span of the first nk basis vectors [R;I] S', hence its GSO coordinates vanish for i >= nk:
//            c'_i = -sum_{j>i} U_ij z_j, block U_22 only.  z_2 = z[nk:] is large (the widths s/||b~_i|| are ~10^4-10^5).
//   between: the residual centre -x - S[:, nk:] z_2 is reduced modulo L_1 = [R;I] S' Z^nk to
//            c_1 = -[z_2; 0] - [R; I] g3,  g3 = digits((u - A_bar z_2) mod q)     (G W = -A_bar, G g = u mod q);
//   phase 2 (i = nk-1 .. 0): its GSO coordinates T_1 = -Mt_1 z_2 - M' g3 (Mt_1 = the first m_bar columns of rows [0, nk) of
//            D^-1 B~^t; M' = Mt [R; I] = U_11 S'^-1 is block triangular with entries <= 1/2), then the recursion with block
//            U_11 only; z_1 is small (|z_1| ~ s) because c_1 is reduced.
//   output:  e = [z_2 + R e_bot; e_bot],  e_bot = g3 + S' z_1        (A e = A_bar z_2 + G g3 = u).
// Against the one-pass form this never forms sol = A_P^-1 u, never multiplies the nk x m_bar block U_12 by z_2 at 45-bit
// precision against a 31-bit z_1, and replaces the nk x m_bar product W z_2 by the n x m_bar product A_bar z_2:
// 9-12 digit-pair products per useful MAC instead of 18-25.
// ---------------------------------------------------------------------------
// dTidx (optional, device): the tag index of every target of the chunk in the installed tag table (qf_samp_p_tagged).  The
// tag enters only between the phases (DESIGN 4.3): for A_t = [A_bar | H_t G - A_bar R], g3 = digits(h_t) with
// h_t = H_t^-1 (u - A_bar z2) mod q, the same integer vector as after qf_gpv_set_tag(H_t); everything else is tag-independent.
// The chunk is split at the first read of the target (DESIGN 4.12): np2_workspace + np2_phase1 and the products of z2
// (np2_abar_z2, np2_mt1_z2) are the offline half, np2_finish (from h on) the online half.
qf_status np2_workspace(qf_ctx* ctx) {
    const long D = ctx->dim, ldD = ctx->ld_dim, C = ctx->chunk, n = ctx->n;
    const long ldk = ctx->ldk_dim, plane = C * ldk;
    const int nz_m = (int)((C + 127) / 128), nz_kb = (int)(ldk / 128);
    const int L = ctx->z_limbs;
    CK(ctx->w[0].ensure((size_t)C * n * 8));     // h = u - A_bar z2 mod q
    CK(ctx->w[2].ensure((size_t)C * ldD * 8));   // T
    CK(ctx->w[3].ensure((size_t)C * ldD * 8));   // Z
    CK(ctx->w[4].ensure((size_t)C * ctx->ld_nk * 8));  // e_bot = g3 + S' z1
    CK(ctx->w[8].ensure((size_t)L * plane));     // digit planes of z
    CK(ctx->w[10].ensure((size_t)C * ctx->ldk_nk));   // g3 (one digit plane)
    const size_t nzb = (size_t)L * nz_m * nz_kb;
    CK(ctx->dNz.ensure(nzb));
    CK(cudaMemsetAsync(ctx->dNz.p, 0, nzb, ctx->stream));
    ctx->gate_n256 = np_block_index(D - 1, D, NP_SIZES[1]) + 1;
    ctx->gate_n1024 = np_block_index(D - 1, D, NP_SIZES[2]) + 1;
    ctx->gate_n4096 = np_block_index(D - 1, D, NP_SIZES[3]) + 1;
    const size_t gb = (size_t)(ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096 + 1) * sizeof(int);
    CK(ctx->dGate.ensure(gb));
    CK(cudaMemsetAsync(ctx->dGate.p, 0, gb, ctx->stream));
    return QF_OK;
}

// ---- phase 1: coordinates m-1 .. nk, centres start at 0 (never reads the target)
qf_status np2_phase1(qf_ctx* ctx, int Bc, uint64_t seed, uint64_t first) {
    const long D = ctx->dim, ldD = ctx->ld_dim, nk = ctx->nk;
    double* T = ctx->w[2].as<double>();
    CK(cudaMemset2DAsync(T + nk, (size_t)ldD * 8, 0, (size_t)ctx->m_bar * 8, (size_t)Bc, ctx->stream));
    ctx->np_wdrop_cur = ctx->u_limbs - ctx->u22_limbs; ctx->np_dlo_cur = ctx->u22_dlo; ctx->np_lx_min = 3;
    return np_block(ctx, T, ctx->w[3].as<double>(), Bc, nk, D, NP_TOP, 0, seed, first);
}

// out = (base - A_bar z2) mod q, exact (base == nullptr: -A_bar z2 mod q).  A_bar = the first m_bar columns of the installed
// digit planes of A, or (abar_tagged) the digit planes of A_bar' = H^-1 A_bar of a tagged key.
qf_status np2_abar_z2(qf_ctx* ctx, const int64_t* base, bool abar_tagged, int Bc, int64_t* out) {
    const long C = ctx->chunk, nk = ctx->nk, n = ctx->n, ldk = ctx->ldk_dim;
    const long ldw = abar_tagged ? ctx->ldk_mb : ldk;
    I8GemmArgs g{};
    g.x = ctx->w[8].as<int8_t>() + nk; g.ldx = ldk; g.x_plane = C * ldk;
    g.w = abar_tagged ? ctx->dAbpl.p : ctx->dAl.p; g.ldw = ldw; g.w_plane = n * ldw;
    g.LX = ctx->z_limbs; g.LW = ctx->a_limbs; g.w_signed = 0;
    g.B = Bc; g.N = (int)n; g.K = (int)ctx->m_bar;
    g.out_kind = 0; g.sign = -1; g.q = ctx->prm.q; g.base = base; g.ldbase = n;
    g.out = out; g.ldout = n;
    g.flag = ctx->dFlag.as<int>();
    g.x_nz = ctx->dNz.as<uint8_t>(); g.nz_m_tiles = (int)((C + 127) / 128); g.nz_kb_total = (int)(ldk / 128);
    g.nz_kb_off = (int)(nk / 128);
    return gemm_i8_gated(ctx, g, ctx->dGate.as<int>() + ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096);
}

// Mt_1 z2: the digit planes of z2 written by phase 1 against all digits of Mt_1; out -= V * scale (overwrite: out = -V * scale)
qf_status np2_mt1_z2(qf_ctx* ctx, int Bc, double* out, long ldout, const double* scale, int overwrite) {
    const long C = ctx->chunk, nk = ctx->nk, ldk = ctx->ldk_dim;
    I8GemmArgs g{};
    g.x = ctx->w[8].as<int8_t>() + nk; g.ldx = ldk; g.x_plane = C * ldk;
    g.w = ctx->dMt1l.p; g.ldw = ctx->ldk_mb; g.w_plane = nk * ctx->ldk_mb;
    g.LX = ctx->z_limbs; g.LW = ctx->mt1_limbs; g.w_signed = 1;
    g.B = Bc; g.N = (int)nk; g.K = (int)ctx->m_bar;
    g.out_kind = 3; g.sign = 1; g.q = 0; g.out = out; g.ldout = ldout;
    g.flag = ctx->dFlag.as<int>();
    g.scale = scale;
    g.d_lo = ctx->mt1_dlo; g.overwrite = overwrite;
    g.x_nz = ctx->dNz.as<uint8_t>(); g.nz_m_tiles = (int)((C + 127) / 128); g.nz_kb_total = (int)(ldk / 128);
    g.nz_kb_off = (int)(nk / 128);
    return gemm_i8_gated(ctx, g, ctx->dGate.as<int>() + ctx->gate_n256 + ctx->gate_n1024 + ctx->gate_n4096);
}

// From h = digits source (H: the residues (u - A_bar z2) mod q of the recursion's target) on: g3, the centres of phase 2,
// phase 2 and e.  z2 in Z[:, nk:].  Tpool == nullptr: Mt_1 z2 is contracted here from the digit planes of z2; otherwise
// Tpool holds its store-only unit-scale output (a pool entry, row stride nk).
qf_status np2_finish(qf_ctx* ctx, const int64_t* H, int Bc, uint64_t seed, uint64_t first, int32_t* dE, const double* Tpool) {
    const long D = ctx->dim, ldD = ctx->ld_dim, C = ctx->chunk, nk = ctx->nk, mb = ctx->m_bar, n = ctx->n;
    const long ldnk = ctx->ld_nk, ldk_nk = ctx->ldk_nk;
    double* T = ctx->w[2].as<double>();
    double* Z = ctx->w[3].as<double>();
    int8_t* gp = ctx->w[10].as<int8_t>();
    int* flag = ctx->dFlag.as<int>();
    // ---- g3 = digits(h): one s8 plane (the x operand of its centre map) and, as fp64, the start of e_bot = g3 + S' z1
    // (fused tail: e_bot is formed in one pass from z1 and the g3 plane -- needs 16-byte aligned int32 rows; otherwise e_bot is
    // accumulated in fp64 as in the one-pass form)
    const bool fused_tail = (nk & 3) == 0 && (mb & 3) == 0 && (D & 3) == 0 && (ldk_nk & 3) == 0;
    double* I2 = ctx->w[4].as<double>();
    LAUNCH(qf_launch_gadget_digits(H, n, gp, ldk_nk, Bc, (int)n, (int)ctx->k, (unsigned)ctx->prm.base, nullptr, 0, ctx->stream,
                                   fused_tail ? nullptr : I2, ldnk));
    // ---- centres of phase 2 in GSO coordinates: T[:, 0:nk] = -M' g3 - Mt_1 z2, two launches:
    // (a) M' g3 (M' = U_11 S'^-1, entries <= 1/2, block triangular: the k blocks outside the triangle are skipped
    //     in-kernel), one digit of 0 .. base-1 against four digits: store-only epilogue;
    // (b) Mt_1 z2, accumulated onto (a) (from a pool entry: the same fma, pool_centre).
    {
        I8GemmArgs g{};
        g.x = gp; g.ldx = ldk_nk; g.x_plane = C * ldk_nk;
        g.w = ctx->dMpl.p; g.ldw = ldk_nk; g.w_plane = nk * ldk_nk;
        g.LX = 1; g.LW = ctx->mt1g_limbs; g.w_signed = 1;
        g.B = Bc; g.N = (int)nk; g.K = (int)nk;
        g.out_kind = 3; g.sign = 1; g.q = 0; g.out = T; g.ldout = ldD;
        g.flag = flag;
        g.scale = ctx->dMpscale.as<double>();
        g.d_lo = 0; g.overwrite = 1;
        g.tri_mode = ctx->gpv_rev ? 3 : 4; g.tri_slack = (int)ctx->k;
        LAUNCH(ctx_gemm_i8(ctx, g));
    }
    if (Tpool)
        LAUNCH(qf_launch_pool_centre(Tpool, nk, T, ldD, ctx->dMt1scale.as<double>(), std::ldexp(1.0, 8 * ctx->mt1_dlo), (int)nk,
                                     Bc, ctx->stream));
    else
        QF_TRY(np2_mt1_z2(ctx, Bc, T, ldD, ctx->dMt1scale.as<double>(), 0));
    // ---- phase 2: coordinates nk-1 .. 0
    ctx->np_wdrop_cur = ctx->u_limbs - ctx->u11_limbs; ctx->np_dlo_cur = ctx->u11_dlo; ctx->np_lx_min = 2;
    QF_TRY(np_block(ctx, T, Z, Bc, 0, nk, NP_TOP, 0, seed, first));

    // ---- e_bot = g3 + S' z1,  e_top = z2 + R e_bot
    const long plane2 = C * ldk_nk;
    CK(ctx->w[2].ensure((size_t)std::max<long>(ctx->i2_limbs * plane2, C * ldD * 8)));  // T is dead: digits of e_bot
    int8_t* ip = ctx->w[2].as<int8_t>();
    if (fused_tail) {
        LAUNCH(qf_launch_gpv_ebot(Z, ldD, gp, ldk_nk, dE, D, (int)mb, ip, plane2, ldk_nk, ctx->i2_limbs, Bc, (int)nk, (int)ctx->k,
                                  ctx->dSkf.as<double>(), ctx->gpv_rev, flag, ctx->stream));
    } else {
        LAUNCH(qf_launch_sprime_apply(Z, ldD, I2, ldnk, Bc, (int)nk, (int)ctx->k, ctx->dSkf.as<double>(), ctx->gpv_rev,
                                      ctx->stream));
        LAUNCH(qf_launch_split_f64_limbs(I2, ldnk, ip, plane2, ldk_nk, Bc, (int)nk, ctx->i2_limbs, flag, nullptr, 0, 0, 0,
                                         ctx->stream));
    }
    {
        I8GemmArgs h{};
        h.x = ip; h.ldx = ldk_nk; h.x_plane = plane2;
        h.w = ctx->dRl.p; h.ldw = ldk_nk; h.w_plane = mb * ldk_nk;
        h.LX = ctx->i2_limbs; h.LW = 1; h.w_signed = 1;
        h.B = Bc; h.N = (int)mb; h.K = (int)nk;
        h.out_kind = 1; h.sign = 1; h.q = 0; h.out = dE; h.ldout = D;
        h.flag = flag;
        LAUNCH(ctx_gemm_i8(ctx, h));
    }
    // e_top += z2 (and, unfused, e_bot from its fp64 form)
    LAUNCH(qf_launch_gpv_struct_finalize(dE, D, Z + nk, ldD, I2, ldnk, Bc, (int)mb, fused_tail ? 0 : (int)nk, flag, ctx->stream));
    return QF_OK;
}

// Per-target tag (dTidx): h_t = H_t^-1 w for w = u - A_bar z2 in dTagU (any installed tag), written to H (w[0])
qf_status np2_tag_syndrome(qf_ctx* ctx, const int32_t* dTidx, int Bc) {
    const long n = ctx->n;
    LAUNCH(qf_launch_tag_syndrome(ctx->dTagU.as<int64_t>(), n, nullptr, 0, 0, dTidx, (int)ctx->tag_count, ctx->dTagTab.p,
                                  nullptr, ctx->tag_word, nullptr, ctx->prm.q, (int)n, (int)ctx->k, Bc, ctx->w[0].as<int64_t>(), n,
                                  ctx->dFlag.as<int>(), ctx->stream, ctx->tag_poly ? ctx->dTagXr.p : nullptr));
    return QF_OK;
}

qf_status samp_p_np2_chunk(qf_ctx* ctx, const int64_t* dUin, int Bc, uint64_t seed, uint64_t first, int32_t* dE,
                           const int32_t* dTidx = nullptr) {
    QF_TRY(np2_workspace(ctx));
    QF_TRY(np2_phase1(ctx, Bc, seed, first));
    // ---- tagged key: the recursion runs on H^-1 A, so its target is u' = H^-1 u mod q (phase 1 never reads the target)
    const bool abar_tagged = ctx->key_tagged && !dTidx;
    const int64_t* ub = dUin;
    if (abar_tagged) QF_TRY(tag_targets(ctx, dUin, Bc, &ub));
    // ---- h = (u - A_bar z2) mod q (for a tagged key u' - A_bar' z2).  With a tag per target: w = u - A_bar z2 whatever the
    // installed tag, then h_t = H_t^-1 w per target.
    int64_t* H = ctx->w[0].as<int64_t>();
    if (dTidx) CK(ctx->dTagU.ensure((size_t)ctx->chunk * ctx->n * 8));
    QF_TRY(np2_abar_z2(ctx, ub, abar_tagged, Bc, dTidx ? ctx->dTagU.as<int64_t>() : H));
    if (dTidx) QF_TRY(np2_tag_syndrome(ctx, dTidx, Bc));
    return np2_finish(ctx, H, Bc, seed, first, dE, nullptr);
}

// dTidx (tag per target) only with the two-phase recursion (samp_p_tagged_ready)
qf_status samp_p_np_chunk(qf_ctx* ctx, const int64_t* dUin, int Bc, uint64_t seed, uint64_t first, int32_t* dE,
                          const int32_t* dTidx = nullptr) {
    return ctx->two_phase ? samp_p_np2_chunk(ctx, dUin, Bc, seed, first, dE, dTidx)
                          : samp_p_np1_chunk(ctx, dUin, Bc, seed, first, dE);
}

// ---------------------------------------------------------------------------
// samp_p in two halves over the context's pool (DESIGN 4.12).  Pool slot j holds the offline state of sampler index
// pool_first + j; both halves run the launches of the composed chunk functions above, so an online row is bit-identical to
// qf_samp_p (qf_samp_p_tagged) at its index.
// ---------------------------------------------------------------------------
long pool_xdim(const qf_ctx* ctx) { return ctx->prm.kind == QF_PSF_PERTURBATION ? ctx->m : ctx->m_bar; }
long pool_tdim(const qf_ctx* ctx) { return ctx->prm.kind == QF_PSF_PERTURBATION ? 0 : ctx->nk; }

// offline half of Bc entries into slots slot0 .. slot0 + Bc - 1 (sampler indices first ..)
qf_status samp_p_offline_chunk(qf_ctx* ctx, int Bc, uint64_t seed, uint64_t first, int64_t slot0) {
    const long xd = pool_xdim(ctx), n = ctx->n;
    int32_t* X = ctx->dPoolX.as<int32_t>() + slot0 * xd;
    int64_t* Ax = ctx->dPoolAx.as<int64_t>() + slot0 * n;
    if (ctx->prm.kind == QF_PSF_PERTURBATION) {
        QF_TRY(pert_perturbation(ctx, Bc, seed, first));
        QF_TRY(pert_ap(ctx, nullptr, Bc, Ax));
        LAUNCH(qf_launch_f64_to_i32(ctx->w[2].as<double>(), ctx->ld_dim, X, xd, Bc, (int)xd, ctx->dFlag.as<int>(), ctx->stream));
        return QF_OK;
    }
    const long nk = ctx->nk;
    QF_TRY(np2_workspace(ctx));
    QF_TRY(np2_phase1(ctx, Bc, seed, first));
    // A_bar z2 on the untagged planes of A (their first m_bar columns are A_bar whatever the installed tag): the online half
    // applies H^-1 to u - A_bar z2, the same residues as u' - A_bar' z2
    QF_TRY(np2_abar_z2(ctx, nullptr, false, Bc, Ax));
    QF_TRY(np2_mt1_z2(ctx, Bc, ctx->dPoolT.as<double>() + slot0 * nk, nk, ctx->dOnes.as<double>(), 1));
    LAUNCH(qf_launch_f64_to_i32(ctx->w[3].as<double>() + nk, ctx->ld_dim, X, xd, Bc, (int)xd, ctx->dFlag.as<int>(), ctx->stream));
    return QF_OK;
}

// online half for the targets dUin of Bc entries from slot slot0 on
qf_status samp_p_online_chunk(qf_ctx* ctx, const int64_t* dUin, int Bc, int64_t slot0, int32_t* dE, const int32_t* dTidx) {
    const long xd = pool_xdim(ctx), n = ctx->n;
    const uint64_t seed = ctx->pool_seed, first = ctx->pool_first + (uint64_t)slot0;
    const int32_t* X = ctx->dPoolX.as<int32_t>() + slot0 * xd;
    const int64_t* Ax = ctx->dPoolAx.as<int64_t>() + slot0 * n;
    if (ctx->prm.kind == QF_PSF_PERTURBATION) {
        QF_TRY(pert_workspace(ctx));
        LAUNCH(qf_launch_pool_expand(X, xd, ctx->w[2].as<double>(), ctx->ld_dim, (int)xd, dUin, n, Ax, n, ctx->w[4].as<int64_t>(),
                                     n, (int)n, Bc, ctx->prm.q, ctx->stream));
        return pert_finish(ctx, Bc, seed, first, dE, dTidx);
    }
    const long nk = ctx->nk;
    QF_TRY(np2_workspace(ctx));
    int64_t* H = ctx->w[0].as<int64_t>();
    if (dTidx) CK(ctx->dTagU.ensure((size_t)ctx->chunk * n * 8));
    // z2 into Z[:, nk:], w = u - A_bar z2 mod q
    LAUNCH(qf_launch_pool_expand(X, xd, ctx->w[3].as<double>() + nk, ctx->ld_dim, (int)xd, dUin, n, Ax, n,
                                 dTidx ? ctx->dTagU.as<int64_t>() : H, n, (int)n, Bc, ctx->prm.q, ctx->stream));
    const int64_t* h = H;
    if (dTidx) QF_TRY(np2_tag_syndrome(ctx, dTidx, Bc));
    else if (ctx->key_tagged) QF_TRY(tag_targets(ctx, H, Bc, &h));
    return np2_finish(ctx, h, Bc, seed, first, dE, ctx->dPoolT.as<double>() + slot0 * nk);
}

// find n columns of A (n x m) that form a matrix invertible over Z_q by unit pivoting and return
// Ainv (row k maps u to the coefficient of pivot column k):  sol[piv[k]] = sum_j Ainv[k][j] u_j
bool find_unit_pivots(const int64_t* A, long n, long m, uint64_t q, std::vector<int>& piv, std::vector<int64_t>& Ainv) {
    std::vector<uint64_t> T((size_t)n * n, 0);
    for (long i = 0; i < n; ++i) T[i * n + i] = 1;
    std::vector<char> used(n, 0);
    std::vector<long> pivrow;
    std::vector<uint64_t> w(n);
    piv.clear();
    for (long c = 0; c < m && (long)piv.size() < n; ++c) {
        for (long i = 0; i < n; ++i) {
            u128 acc = 0;
            for (long j = 0; j < n; ++j) {
                acc += (u128)T[i * n + j] * (uint64_t)A[j * m + c];
                if ((j & 3) == 3) acc %= q;
            }
            w[i] = (uint64_t)(acc % q);
        }
        long r = -1;
        for (long i = 0; i < n; ++i)
            if (!used[i] && w[i] && gcd_u64(w[i], q) == 1) { r = i; break; }
        if (r < 0) continue;
        uint64_t inv = inv_mod(w[r], q);
        for (long j = 0; j < n; ++j) T[r * n + j] = mulmod_h(T[r * n + j], inv, q);
        for (long i = 0; i < n; ++i) {
            if (i == r || w[i] == 0) continue;
            uint64_t f = w[i];
            for (long j = 0; j < n; ++j) {
                uint64_t sub = mulmod_h(f, T[r * n + j], q);
                T[i * n + j] = (T[i * n + j] + q - sub) % q;
            }
        }
        used[r] = 1;
        piv.push_back((int)c);
        pivrow.push_back(r);
    }
    if ((long)piv.size() < n) return false;
    Ainv.assign((size_t)n * n, 0);
    for (long kk = 0; kk < n; ++kk)
        for (long j = 0; j < n; ++j) Ainv[kk * n + j] = (int64_t)T[pivrow[kk] * n + j];
    return true;
}

// ---------------------------------------------------------------------------
// Blocked right-looking Cholesky A = L L^t (lower, in place, fp64) on the device: 64-wide diagonal blocks in
// shared memory (potrf_diag), panel solve and trailing update on the DMMA GEMM.  Replaces
// MatQ::cholesky_decomposition_flint (mp_perturbation.rs:138).  The strict upper triangle is zeroed.
// ---------------------------------------------------------------------------
qf_status potrf_lower(qf_ctx* ctx, double* A, long ld, long n) {
    constexpr long NB = 64, STRIP = 1024;
    Dev dLinv, dPanel, dInfo;
    CK(dLinv.ensure(NB * NB * 8));
    CK(dPanel.ensure((size_t)std::max(1L, n) * NB * 8));
    CK(dInfo.ensure(sizeof(int)));
    CK(cudaMemsetAsync(dInfo.p, 0, sizeof(int), ctx->stream));
    double* P = dPanel.as<double>();
    for (long j = 0; j < n; j += NB) {
        const int nb = (int)std::min(NB, n - j);
        LAUNCH(qf_launch_potrf_diag(A + j * ld + j, ld, nb, dLinv.as<double>(), dInfo.as<int>(), ctx->stream));
        const long rows = n - j - nb;
        if (rows <= 0) break;
        // L_ij = A_ij L_jj^-t  (explicit inverse of the well-conditioned diagonal block)
        LAUNCH(ctx_gemm(ctx, A + (j + nb) * ld + j, ld, dLinv.as<double>(), NB, P, NB, (int)rows, nb, nb, 1.0, 0.0, 0));
        LAUNCH(qf_launch_copy_block(P, NB, A + (j + nb) * ld + j, ld, rows, nb, ctx->stream));
        // A_22 -= L_21 L_21^t, lower part only, in column strips
        for (long c0 = j + nb; c0 < n; c0 += STRIP) {
            const long c1 = std::min(n, c0 + STRIP);
            const double* Pc = P + (c0 - j - nb) * NB;
            LAUNCH(ctx_gemm(ctx, Pc, NB, Pc, NB, A + c0 * ld + c0, ld, (int)(n - c0), (int)(c1 - c0), nb, -1.0, 1.0, 0));
        }
    }
    LAUNCH(qf_launch_tril(A, ld, n, ctx->stream));
    int info = 0;
    CK(cudaMemcpyAsync(&info, dInfo.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (info) return ctx->fail(QF_ERR_INVALID, "Sigma_2 is not positive definite (s too small for this R, mp_perturbation.rs:109-110)");
    return QF_OK;
}

// G = R R^t (m_bar x m_bar, exact small integers in fp64) from the resident fp64 copy of R
qf_status gram_r(qf_ctx* ctx, const double* R, double* G, long ldg) {
    LAUNCH(ctx_gemm(ctx, R, ctx->ld_nk, R, ctx->ld_nk, G, ldg, (int)ctx->m_bar, (int)ctx->m_bar, (int)ctx->nk, 1.0, 0.0, 0));
    return QF_OK;
}

// Structured square root of the default Sigma_2 = r^2/(2 pi) ((s^2 - 1) I - (b^2+1) T T^t), T = [R; I]
// (mp_perturbation.rs:111-139 with Sigma = s^2 I).  Block form
//   Sigma_2 = coef [[alpha I - c R R^t, -c R], [-c R^t, (alpha - c) I]]
// so x_b ~ N(0, beta I), beta = coef (alpha - c), and x_t | x_b ~ N(-kappa R x_b, Schur),
// kappa = c / (alpha - c), Schur = coef (alpha I - c alpha / (alpha - c) R R^t).  Any square root of Sigma_2
// gives the same law (mp_perturbation.rs:94-104); only the m_bar x m_bar factor of Schur is dense.
qf_status setup_structured_sigma2(qf_ctx* ctx) {
    const double s = ctx->prm.s, r = ctx->prm.r, c = (double)(ctx->prm.base * ctx->prm.base + 1);
    const double alpha = s * s - 1.0, coef = r * r / (2.0 * M_PI);
    if (!(alpha - c > 0)) return ctx->fail(QF_ERR_INVALID, "Sigma_2 is not positive definite (s^2 <= b^2 + 2)");
    const double beta = coef * (alpha - c), kappa = c / (alpha - c);
    const long mb = ctx->m_bar;
    ctx->ld_mb = pad16(mb);
    CK(ctx->dLs.ensure((size_t)mb * ctx->ld_mb * 8));
    CK(cudaMemsetAsync(ctx->dLs.p, 0, (size_t)mb * ctx->ld_mb * 8, ctx->stream));
    QF_TRY(gram_r(ctx, ctx->dR.as<double>(), ctx->dLs.as<double>(), ctx->ld_mb));
    LAUNCH(qf_launch_sigma2_assemble(ctx->dLs.as<double>(), ctx->ld_mb, mb, 0, nullptr, 0, nullptr, 0, mb, nullptr, 0, alpha,
                                     c * alpha / (alpha - c), coef, ctx->stream));
    QF_TRY(potrf_lower(ctx, ctx->dLs.as<double>(), ctx->ld_mb, mb));
    // fixed-point digits of x_b for the ternary product R x_b on the tensor cores: |x_b| <= 8.7 sqrt(beta)
    ctx->sqrt_beta = std::sqrt(beta);
    ctx->xb_limbs = 3;
    int f = (int)std::floor(std::log2(limb_capacity(3) / (8.7 * ctx->sqrt_beta)));
    if (f < 8) {
        ctx->xb_limbs = 4;
        f = (int)std::floor(std::log2(limb_capacity(4) / (8.7 * ctx->sqrt_beta)));
    }
    if (f < 0) return ctx->fail(QF_ERR_UNSUPPORTED, "s * r too large for the fixed-point x_b digits");
    f = std::min(f, 30);
    ctx->xb_fscale = std::ldexp(1.0, f);
    std::vector<double> sc((size_t)mb, kappa / ctx->xb_fscale);
    CK(ctx->dXbScale.ensure(sc.size() * 8));
    CK(cudaMemcpyAsync(ctx->dXbScale.p, sc.data(), sc.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->pert_structured = true;
    return QF_OK;
}

// Fixed-point digit planes of the dense factor L (sqrt(Sigma_2), or the Schur factor of the structured form) for
// x_2 = L g on tcgen05: L rows scaled to ll_limbs balanced base-256 digits (relative resolution 2^-30 of the row
// maximum), normals g quantised to 2^-20 (their fp32 Box-Muller source carries 24 bits).  The covariance of x_2
// then differs from Sigma_2 by a relative 2^-29, far below what the rounding step D_{Z,r,x_2} can resolve.
qf_status setup_pert_i8(qf_ctx* ctx) {
    ctx->pert_i8 = false;
    const char* env = getenv("QF_DISABLE_PERT_I8");
    const long dimL = ctx->pert_structured ? ctx->m_bar : ctx->m;
    if (!ctx->use_i8 || (env && env[0] == '1') || dimL < 512) return QF_OK;
    const double* L = ctx->pert_structured ? ctx->dLs.as<double>() : ctx->dL.as<double>();
    const long ldL = ctx->pert_structured ? ctx->ld_mb : ctx->ld_dim;
    ctx->l_dim = dimL;
    ctx->ldk_l = (dimL + 127) / 128 * 128;
    const size_t bytes = (size_t)ctx->ll_limbs * dimL * ctx->ldk_l;
    CK(ctx->dLl.ensure(bytes));
    CK(ctx->dLlScale.ensure((size_t)dimL * 8));
    CK(cudaMemsetAsync(ctx->dLl.p, 0, bytes, ctx->stream));
    ctx->g_fscale = std::ldexp(1.0, (int)std::floor(std::log2(limb_capacity(ctx->lg_limbs) / 6.9)));
    LAUNCH(qf_launch_fixed_rows_prepare(L, ldL, (int)dimL, (int)dimL, ctx->ll_limbs, -1.0 / ctx->g_fscale, ctx->dLlScale.as<double>(),
                                        ctx->dLl.as<int8_t>(), dimL * ctx->ldk_l, ctx->ldk_l, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->pert_i8 = true;
    return QF_OK;
}

// X2[:, 0:l_dim] = L g from the digit planes of g (gp) and of L: one launch per 1024-row block of L, K limited to
// the block's last column when L is lower triangular; K chunked so that the s32 accumulators cannot overflow.
qf_status pert_lg_i8(qf_ctx* ctx, const int8_t* gp, long gplane, int Bc, double* X2, long ldx, bool tri) {
    const long dimL = ctx->l_dim, ldk = ctx->ldk_l;
    CK(cudaMemset2DAsync(X2, (size_t)ldx * 8, 0, (size_t)dimL * 8, (size_t)Bc, ctx->stream));
    const long kmax = (131071 / std::min(ctx->lg_limbs, ctx->ll_limbs)) / 128 * 128;
    for (long rb = 0; rb < dimL; rb += 1024) {
        const long nrows = std::min(1024L, dimL - rb);
        const long kend = tri ? std::min(dimL, rb + nrows) : dimL;
        for (long k0 = 0; k0 < kend; k0 += kmax) {
            const long kk = std::min(kmax, kend - k0);
            I8GemmArgs g{};
            g.x = gp + k0; g.ldx = ldk; g.x_plane = gplane;
            g.w = ctx->dLl.as<int8_t>() + rb * ldk + k0; g.ldw = ldk; g.w_plane = dimL * ldk;
            g.LX = ctx->lg_limbs; g.LW = ctx->ll_limbs; g.w_signed = 1;
            g.B = Bc; g.N = (int)nrows; g.K = (int)kk;
            g.out_kind = 3; g.sign = 1; g.q = 0; g.base = nullptr; g.ldbase = 0; g.out = X2 + rb; g.ldout = ldx;
            g.flag = ctx->dFlag.as<int>();
            g.scale = ctx->dLlScale.as<double>() + rb;
            LAUNCH(ctx_gemm_i8(ctx, g));
        }
    }
    return QF_OK;
}

// ---------------------------------------------------------------------------
// Unnormalised Gram-Schmidt of the columns of S (MatQ::gso, gpv.rs:91) in fp64 on the device: blocked classical
// Gram-Schmidt with re-orthogonalisation (two projection passes against the finished vectors, GEMMs on the DMMA
// path) and two Cholesky-QR passes inside each 64-vector block (Gram matrix + potrf_diag + triangular solve as a
// GEMM).  dS, dG: D x ld, S[t][j] = coordinate t of b_j, G[t][j] = coordinate t of b~_j.
// ---------------------------------------------------------------------------
qf_status gso_device(qf_ctx* ctx, const double* dS, double* dG) {
    constexpr long NB = 64;
    const long D = ctx->dim, ld = ctx->ld_dim;
    Dev dBt, dQt, dQ, dPw, dPwT, dC, dGm, dLinv, dR, dInfo;
    CK(dBt.ensure((size_t)D * ld * 8));
    CK(dQt.ensure((size_t)D * ld * 8));
    CK(dQ.ensure((size_t)D * ld * 8));
    CK(dPw.ensure((size_t)NB * ld * 8));
    CK(dPwT.ensure((size_t)D * NB * 8));
    CK(dC.ensure((size_t)NB * ld * 8));
    CK(dGm.ensure((size_t)NB * NB * 8));
    CK(dLinv.ensure((size_t)NB * NB * 8));
    CK(dR.ensure((size_t)D * 8));
    CK(dInfo.ensure(sizeof(int)));
    CK(cudaMemsetAsync(dInfo.p, 0, sizeof(int), ctx->stream));
    CK(cudaMemsetAsync(dQt.p, 0, (size_t)D * ld * 8, ctx->stream));
    CK(cudaMemsetAsync(dQ.p, 0, (size_t)D * ld * 8, ctx->stream));
    double *Bt = dBt.as<double>(), *Qt = dQt.as<double>(), *Q = dQ.as<double>(), *Pw = dPw.as<double>(),
           *PwT = dPwT.as<double>(), *C = dC.as<double>(), *Gm = dGm.as<double>(), *Linv = dLinv.as<double>(),
           *R = dR.as<double>();
    LAUNCH(qf_launch_transpose_scale(dS, ld, Bt, ld, (int)D, (int)D, nullptr, ctx->stream));  // rows = basis vectors
    for (long j0 = 0; j0 < D; j0 += NB) {
        const int nb = (int)std::min(NB, D - j0);
        LAUNCH(qf_launch_copy_block(Bt + j0 * ld, ld, Pw, ld, nb, (int)D, ctx->stream));
        if (j0 > 0)
            for (int pass = 0; pass < 2; ++pass) {  // Pw -= (Pw Q_prev) Q_prev^t, twice
                LAUNCH(ctx_gemm(ctx, Pw, ld, Qt, ld, C, ld, nb, (int)j0, (int)D, 1.0, 0.0, 0));
                LAUNCH(ctx_gemm(ctx, C, ld, Q, ld, Pw, ld, nb, (int)D, (int)j0, -1.0, 1.0, 0));
            }
        for (int pass = 0; pass < 2; ++pass) {  // Cholesky-QR of the block: Pw = L Q_block, r_jj = L_jj
            LAUNCH(ctx_gemm(ctx, Pw, ld, Pw, ld, Gm, NB, nb, nb, (int)D, 1.0, 0.0, 0));
            LAUNCH(qf_launch_potrf_diag(Gm, NB, nb, Linv, dInfo.as<int>(), ctx->stream));
            LAUNCH(qf_launch_gso_rdiag(R + j0, Gm, NB, nb, pass == 0, ctx->stream));
            LAUNCH(qf_launch_transpose_scale(Pw, ld, PwT, NB, nb, (int)D, nullptr, ctx->stream));
            LAUNCH(ctx_gemm(ctx, Linv, NB, PwT, NB, Pw, ld, nb, (int)D, nb, 1.0, 0.0, 0));
        }
        LAUNCH(qf_launch_copy_block(Pw, ld, Qt + j0 * ld, ld, nb, (int)D, ctx->stream));
        LAUNCH(qf_launch_transpose_scale(Pw, ld, Q + j0, ld, nb, (int)D, nullptr, ctx->stream));
    }
    LAUNCH(qf_launch_scale_cols(Q, ld, dG, ld, D, D, R, ctx->stream));
    int info = 0;
    CK(cudaMemcpyAsync(&info, dInfo.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (info) return ctx->fail(QF_ERR_INVALID, "gso: the basis is (numerically) rank deficient");
    return QF_OK;
}

// H^-1 mod q on the device (qf_launch_mat_inverse_mod) for the n x n residues h; *ok = false when some column has no
// unit pivot (first row at or below the diagonal whose entry is a unit mod q), and hinv is then left empty
qf_status tag_inverse(qf_ctx* ctx, const uint64_t* h, std::vector<int64_t>& hinv, bool* ok) {
    const long n = ctx->n;
    std::vector<uint64_t> mm((size_t)n * 2 * n, 0);
    for (long i = 0; i < n; ++i) {
        for (long j = 0; j < n; ++j) mm[(size_t)i * 2 * n + j] = h[i * n + j];
        mm[(size_t)i * 2 * n + n + i] = 1;
    }
    Dev dM, dF, dFail;
    CK(dM.ensure(mm.size() * 8));
    CK(dF.ensure((size_t)n * 8));
    CK(dFail.ensure(sizeof(int)));
    CK(cudaMemcpyAsync(dM.p, mm.data(), mm.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(qf_launch_mat_inverse_mod(dM.as<uint64_t>(), dF.as<uint64_t>(), (int)n, ctx->prm.q, dFail.as<int>(), ctx->stream));
    int fail = 0;
    CK(cudaMemcpyAsync(&fail, dFail.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(mm.data(), dM.p, mm.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *ok = fail == 0;
    hinv.clear();
    if (!*ok) return QF_OK;
    hinv.resize((size_t)n * n);
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) hinv[(size_t)i * n + j] = (int64_t)mm[(size_t)i * 2 * n + n + j];
    return QF_OK;
}

// u8 digit planes of H^-1 into dHl: n x ldk_n per digit group of modq_contract (H^-1, then 256^MODQ_GROUP H^-1 mod q when a
// residue needs two groups), the key operand of u' = H^-1 u
qf_status tag_planes(qf_ctx* ctx, const std::vector<int64_t>& hinv, Dev& dHl) {
    const long n = ctx->n, ldk = ctx->ldk_n;
    const uint64_t q = ctx->prm.q;
    const int groups = modq_groups(limbs_for((double)(q - 1))), L = ctx->a_limbs;
    uint64_t sh = 1;
    for (int i = 0; i < MODQ_GROUP; ++i) sh = mulmod_h(sh, 256, q);
    std::vector<uint8_t> planes((size_t)groups * L * n * ldk, 0);
    for (int gi = 0; gi < groups; ++gi)
        for (long i = 0; i < n; ++i)
            for (long j = 0; j < n; ++j) {
                const uint64_t h = (uint64_t)hinv[(size_t)i * n + j], v = gi ? mulmod_h(h, sh, q) : h;
                for (int l = 0; l < L; ++l) planes[(((size_t)gi * L + l) * n + i) * ldk + j] = (uint8_t)(v >> (8 * l));
            }
    CK(dHl.ensure(planes.size()));
    CK(cudaMemcpyAsync(dHl.p, planes.data(), planes.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

// A_bar'^t = (H^-1 A_bar)^t mod q (m_bar x n, A_bar = the first m_bar columns of the installed A) into abt, for the digit
// planes dHl of H^-1 (tag_planes): tcgen05 with the mod-q epilogue, the "targets" being the columns of A_bar as balanced digits
qf_status tag_abar(qf_ctx* ctx, const Dev& dHl, std::vector<int64_t>& abt) {
    const long n = ctx->n, mb = ctx->m_bar, m = ctx->m, ldk = ctx->ldk_n;
    const uint64_t q = ctx->prm.q;
    const int lx = limbs_for((double)(q - 1));
    const int groups = modq_groups(lx), L = ctx->a_limbs;
    std::vector<int64_t> at((size_t)mb * n);
    for (long j = 0; j < n; ++j)
        for (long c = 0; c < mb; ++c) at[(size_t)c * n + j] = ctx->hA[(size_t)j * m + c];
    Dev dX, dOut, dTmp;
    QF_TRY(upload_limbs(ctx, at.data(), mb, n, ldk, lx, true, dX));
    CK(dOut.ensure((size_t)mb * n * 8));
    if (groups > 1) CK(dTmp.ensure((size_t)mb * n * 8));
    const uint8_t* hl = dHl.as<uint8_t>();
    QF_TRY(modq_contract(ctx, dX.as<int8_t>(), ldk, mb * ldk, lx, hl, hl + (size_t)L * n * ldk, ldk, (int)mb, (int)n, (int)n,
                         dTmp.as<int64_t>(), dOut.as<int64_t>()));
    abt.resize((size_t)mb * n);
    CK(cudaMemcpyAsync(abt.data(), dOut.p, abt.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

// gadget entries base^t mod q, t < k
std::vector<uint64_t> gadget_powers(const qf_ctx* ctx) {
    std::vector<uint64_t> gpow(ctx->k);
    u128 pwt = 1;
    for (long t = 0; t < ctx->k; ++t) { gpow[t] = (uint64_t)(pwt % ctx->prm.q); pwt = pwt * (uint64_t)ctx->prm.base % ctx->prm.q; }
    return gpow;
}

// Form of the installed key A for a trapdoor R (m_bar x nk): a G-trapdoor A = [A_bar | H G - A_bar R] (gadget_classical.rs:56-68)
// with H = I, with an H invertible by unit pivoting, with an H that has no unit pivot (singular ones included), or none of these.
enum KeyForm { KEY_OTHER, KEY_IDENTITY, KEY_TAGGED, KEY_TAG_SINGULAR };
struct KeyTag {
    KeyForm form = KEY_OTHER;
    std::vector<uint64_t> h;     // H mod q, n x n (KEY_IDENTITY, KEY_TAGGED, KEY_TAG_SINGULAR)
    std::vector<int64_t> hinv;   // H^-1 mod q (KEY_TAGGED)
};

// The one place that decides how a G-trapdoor key is recognised (PSFGPV and PSFPerturbation trapdoor installs).  A_bar R on
// the tensor cores ("targets" = the columns of R, key matrix = the installed digit planes of A), compared exactly on the host:
// Y = A[:, m_bar:] + A_bar R mod q must be H G, with H read from the columns with gadget entry 1 and Y[:, j k + t] =
// base^t H[:, j] for every other column.  H = I is KEY_IDENTITY.  Otherwise, if find_tag, H^-1 is computed on the device
// (unit pivots) and, for KEY_TAGGED, its digit planes are written to dHl (tag_planes); without find_tag the key is KEY_OTHER.
qf_status match_key_tag(qf_ctx* ctx, const int8_t* R, bool find_tag, Dev& dHl, KeyTag& kt) {
    kt = KeyTag();
    const long n = ctx->n, k = ctx->k, mb = ctx->m_bar, nk = ctx->nk, m = ctx->m;
    const uint64_t q = ctx->prm.q;
    const long ldk = (mb + 127) / 128 * 128;
    Dev dRt, dAr;
    {
        // R^t as one s8 plane (nk x ldk), transposed in cache blocks
        constexpr long TB = 64;
        std::vector<uint8_t> rt((size_t)nk * ldk, 0);
        for (long i0 = 0; i0 < mb; i0 += TB)
            for (long j0 = 0; j0 < nk; j0 += TB)
                for (long i = i0; i < std::min(mb, i0 + TB); ++i)
                    for (long j = j0; j < std::min(nk, j0 + TB); ++j) rt[(size_t)j * ldk + i] = (uint8_t)R[(size_t)i * nk + j];
        CK(dRt.ensure(rt.size()));
        CK(cudaMemcpyAsync(dRt.p, rt.data(), rt.size(), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    CK(dAr.ensure((size_t)nk * n * 8));
    I8GemmArgs g{};
    g.x = dRt.as<int8_t>(); g.ldx = ldk; g.x_plane = nk * ldk;
    g.w = ctx->dAl.p; g.ldw = ctx->ldk_dim; g.w_plane = n * ctx->ldk_dim;
    g.LX = 1; g.LW = ctx->a_limbs; g.w_signed = 0;
    g.B = (int)nk; g.N = (int)n; g.K = (int)mb;
    g.out_kind = 0; g.sign = 1; g.q = q; g.out = dAr.p; g.ldout = n;
    g.flag = ctx->dFlag.as<int>();
    LAUNCH(ctx_gemm_i8(ctx, g));
    std::vector<int64_t> art((size_t)nk * n);
    CK(cudaMemcpyAsync(art.data(), dAr.p, art.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    auto Y = [&](long i, long j) -> uint64_t {
        return (uint64_t)(((u128)(uint64_t)ctx->hA[(size_t)i * m + mb + j] + (uint64_t)art[(size_t)j * n + i]) % q);
    };
    std::vector<uint64_t> h((size_t)n * n);
    bool ident = true;
    for (long i = 0; i < n; ++i)
        for (long jb = 0; jb < n; ++jb) {
            const uint64_t hij = Y(i, jb * k);
            h[(size_t)i * n + jb] = hij;
            ident = ident && hij == (i == jb ? 1u : 0u);
            for (long t = 1; t < k; ++t)
                if (Y(i, jb * k + t) != mulmod_h(hij, gpow[t], q)) return QF_OK;
        }
    if (ident) {
        kt.form = KEY_IDENTITY;
    } else {
        if (!find_tag) return QF_OK;
        bool ok = false;
        QF_TRY(tag_inverse(ctx, h.data(), kt.hinv, &ok));
        kt.form = ok ? KEY_TAGGED : KEY_TAG_SINGULAR;
        if (ok) QF_TRY(tag_planes(ctx, kt.hinv, dHl));
    }
    kt.h = std::move(h);
    return QF_OK;
}

// Recover (R, W) from a short basis of the form gen_short_basis_for_trapdoor builds (for any tag) and verify the
// factorisation exactly; on success e = S z runs in structured form.  Any mismatch leaves the dense path in place.
// Then check the key against the basis: [A_bar | G - A_bar R] (identity tag) or, if find_tag, [A_bar | H G - A_bar R].
qf_status detect_gpv_structure(qf_ctx* ctx, const int64_t* s, const std::vector<int>& piv, bool find_tag) {
    ctx->gpv_struct = false;
    ctx->key_tagged = false;
    const char* env = getenv("QF_DISABLE_GPV_STRUCT");
    if (ctx->prm.kind != QF_PSF_GPV || !ctx->use_i8 || (env && env[0] == '1')) return QF_OK;
    const long n = ctx->n, k = ctx->k, mb = ctx->m_bar, nk = ctx->nk, m = ctx->m;
    const uint64_t q = ctx->prm.q, base = (uint64_t)ctx->prm.base;
    if (nk % 128 != 0 || mb < nk || base > 256) return QF_OK;  // plane offsets / zero-tile map need 128-column alignment
    u128 pw = 1;
    for (long i = 0; i < k; ++i) pw *= base;
    if (pw < q) return QF_OK;
    const bool exact_pow = pw == (u128)q;
    std::vector<int64_t> sk((size_t)k * k, 0), qd(k, 0);
    for (long j = 0; j < k; ++j) sk[j * k + j] = (int64_t)base;
    for (long i = 0; i + 1 < k; ++i) sk[(i + 1) * k + i] = -1;
    if (!exact_pow) {
        uint64_t qq = q;
        for (long i = 0; i < k; ++i) { qd[i] = (int64_t)(qq % base); sk[i * k + (k - 1)] = qd[i]; qq /= base; }
    }
    auto colmap = [&](long cc) { return exact_pow ? nk - 1 - cc : cc; };  // column of I (x) S_k -> column of S'
    // bottom-left block must be S', bottom-right block W must hold base-b digits
    for (long row = 0; row < nk; ++row) {
        const int64_t* sr = s + (size_t)(mb + row) * m;
        const long blk = row / k, t = row % k;
        for (long cc = 0; cc < nk; ++cc) {
            const int64_t want = (cc / k == blk) ? sk[t * k + (cc % k)] : 0;
            if (sr[colmap(cc)] != want) return QF_OK;
        }
        for (long c = 0; c < mb; ++c)
            if (sr[nk + c] < 0 || (uint64_t)sr[nk + c] >= base) return QF_OK;
    }
    // R from the top-left block: Y[i][cc] = sum_t R[i][blk k + t] S_k[t][cc % k]
    std::vector<int8_t> R((size_t)mb * nk);
    std::vector<i128> x(k), P(k);
    for (long i = 0; i < mb; ++i) {
        const int64_t* sr = s + (size_t)i * m;
        for (long blk = 0; blk < n; ++blk) {
            auto Y = [&](long c) -> i128 { return (i128)sr[colmap(blk * k + c)]; };
            if (exact_pow) {
                i128 v = Y(k - 1);
                if (v % (i128)base) return QF_OK;
                x[k - 1] = v / (i128)base;
                for (long c = k - 2; c >= 0; --c) {
                    v = Y(c) + x[c + 1];
                    if (v % (i128)base) return QF_OK;
                    x[c] = v / (i128)base;
                }
            } else {
                // x_t = base^t x_0 - P_t, P_0 = 0, P_{t+1} = base P_t + Y_t;  sum_t q_t x_t = Y_{k-1}
                P[0] = 0;
                for (long t = 0; t + 1 < k; ++t) P[t + 1] = (i128)base * P[t] + Y(t);
                i128 acc = Y(k - 1);
                for (long t = 0; t < k; ++t) acc += (i128)qd[t] * P[t];
                if (acc % (i128)q) return QF_OK;
                const i128 x0 = acc / (i128)q;
                i128 pwt = 1;
                for (long t = 0; t < k; ++t) { x[t] = pwt * x0 - P[t]; pwt *= (i128)base; }
            }
            for (long t = 0; t < k; ++t) {
                if (x[t] > 127 || x[t] < -127) return QF_OK;
                R[(size_t)i * nk + blk * k + t] = (int8_t)x[t];
            }
        }
    }
    // top-right block must be I + R W: the product on the tensor cores, compared exactly
    const long ldk = ctx->ldk_nk;
    ctx->ldk_mb = (mb + 127) / 128 * 128;
    std::vector<int64_t> r64((size_t)mb * nk), wt((size_t)mb * nk), w64((size_t)nk * mb);
    for (size_t i = 0; i < r64.size(); ++i) r64[i] = R[i];
    for (long row = 0; row < nk; ++row)
        for (long c = 0; c < mb; ++c) {
            const int64_t d = s[(size_t)(mb + row) * m + nk + c];
            wt[(size_t)c * nk + row] = d;
            w64[(size_t)row * mb + c] = d;
        }
    Dev dWt, dOut;
    QF_TRY(upload_limbs(ctx, r64.data(), mb, nk, ldk, 1, true, ctx->dRl));
    QF_TRY(upload_limbs(ctx, wt.data(), mb, nk, ldk, 1, false, dWt));
    CK(dOut.ensure((size_t)mb * mb * 4));
    {
        I8GemmArgs g{};
        g.x = ctx->dRl.as<int8_t>(); g.ldx = ldk; g.x_plane = mb * ldk;
        g.w = dWt.p; g.ldw = ldk; g.w_plane = mb * ldk;
        g.LX = 1; g.LW = 1; g.w_signed = 0;
        g.B = (int)mb; g.N = (int)mb; g.K = (int)nk;
        g.out_kind = 1; g.sign = 1; g.q = 0; g.out = dOut.p; g.ldout = mb;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    }
    std::vector<int32_t> rw((size_t)mb * mb);
    CK(cudaMemcpyAsync(rw.data(), dOut.p, rw.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (long i = 0; i < mb; ++i)
        for (long c = 0; c < mb; ++c)
            if (s[(size_t)i * m + nk + c] != (int64_t)rw[(size_t)i * mb + c] + (i == c ? 1 : 0)) return QF_OK;
    // verified: install W (nk x m_bar, key of the first contraction) and S_k
    QF_TRY(upload_limbs(ctx, w64.data(), nk, mb, ctx->ldk_mb, 1, false, ctx->dWl));
    QF_TRY(upload_as_f64(ctx, sk.data(), k, k, k, ctx->dSkf));
    ctx->gpv_rev = exact_pow ? 1 : 0;
    // |S' z1 + W z2| = |e - sol| on the gadget block: 6 s tail cut, plus q if a pivot column lies there
    bool piv_low = false;
    for (int pc : piv) piv_low = piv_low || pc >= mb;
    ctx->i2_limbs = limbs_for(8.0 * ctx->prm.s + 64.0 + (piv_low ? (double)q : 0.0));
    ctx->gpv_struct = true;
    // Does the installed key have the trapdoor form A = [A_bar | H G - A_bar R] for this R (gadget_classical.rs:56-68)?  For
    // H = I, x = [R g; g] with g = digits(u) solves A x = u and the two-phase recursion applies; a tag H is looked for only if
    // find_tag.
    ctx->gadget_key_ok = false;
    if (base <= 128) {
        KeyTag kt;
        QF_TRY(match_key_tag(ctx, R.data(), find_tag, ctx->dHinvl, kt));
        ctx->gadget_key_ok = kt.form == KEY_IDENTITY;
        if (kt.form == KEY_TAGGED) {
            // A_bar' = H^-1 A_bar on the tensor cores, and G W = -A_bar' mod q exactly for the W of the installed basis: this
            // one check also rejects a wrong inverse and a basis built for another tag
            std::vector<int64_t> abt;
            QF_TRY(tag_abar(ctx, ctx->dHinvl, abt));
            const std::vector<uint64_t> gpow = gadget_powers(ctx);
            bool tag_ok = true;
            for (long i = 0; i < n && tag_ok; ++i)
                for (long c = 0; c < mb; ++c) {
                    u128 gw = (uint64_t)abt[(size_t)c * n + i];
                    for (long t = 0; t < k; ++t) gw += (u128)gpow[t] * (uint64_t)w64[(size_t)(i * k + t) * mb + c];
                    if (gw % q != 0) { tag_ok = false; break; }
                }
            if (tag_ok) {
                std::vector<int64_t> ab((size_t)n * mb);
                for (long i = 0; i < n; ++i)
                    for (long c = 0; c < mb; ++c) ab[(size_t)i * mb + c] = abt[(size_t)c * n + i];
                QF_TRY(upload_limbs(ctx, ab.data(), n, mb, ctx->ldk_mb, ctx->a_limbs, false, ctx->dAbpl));
                ctx->tag_ulimbs = limbs_for((double)(q - 1));
                ctx->key_tagged = true;
                ctx->gadget_key_ok = true;
            } else {
                ctx->dHinvl.release();
            }
        }
        if (ctx->gadget_key_ok) ctx->key_tag = std::move(kt.h);
    }
    return QF_OK;
}

template <typename F>
qf_status for_chunks(qf_ctx* ctx, int64_t batch, F&& f) {
    // balanced chunks: a batch slightly above the chunk size is split evenly instead of into a full and a tiny chunk
    const int64_t nch = std::max<int64_t>(1, (batch + ctx->chunk - 1) / ctx->chunk);
    const int64_t per = std::min<int64_t>(ctx->chunk, ((batch + nch - 1) / nch + 127) / 128 * 128);
    for (int64_t b0 = 0; b0 < batch; b0 += per) {
        int Bc = (int)std::min<int64_t>(per, batch - b0);
        QF_TRY(f(b0, Bc));
    }
    return QF_OK;
}

// Chunks of a device-resident f_a batch.  The fused kernel needs no per-chunk workspace (8 bytes of norm per target): the
// whole batch goes out as one grid, so only its last wave can be partial (chunks of 16 K targets are 1.7 waves each at
// n = 256).
template <typename F>
qf_status f_a_dev_chunks(qf_ctx* ctx, int64_t batch, F&& run) {
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    const bool fused = ctx->x_limbs <= 4 && (ring ? ctx->ring_dense : (ctx->use_i8 && ctx->fused_fa));
    if (fused) {
        constexpr int64_t kMax = 1 << 20;
        for (int64_t b0 = 0; b0 < batch; b0 += kMax) QF_TRY(run(b0, (int)std::min<int64_t>(kMax, batch - b0)));
        return QF_OK;
    }
    return for_chunks(ctx, batch, run);
}

// f_a with a tag per target (qf_f_a_tagged): A sigma from f_a_chunk, then u_b += D_t G sigma_bot_b in place, the targets
// grouped by tag on the device (no host round trip).  dTidx: device tag indices of the chunk.
qf_status f_a_tagged_chunk(qf_ctx* ctx, const int32_t* dSigma, const int32_t* dTidx, int Bc, int64_t* dU, uint8_t* dFlags) {
    QF_TRY(f_a_chunk(ctx, dSigma, Bc, dU, dFlags));
    const int T = (int)ctx->fa_tag_count;
    if (ctx->fa_poly) {  // n words per tag: one CTA per target, no grouping
        LAUNCH(qf_launch_f_a_tag_poly(dSigma, ctx->dim, (int)ctx->m_bar, dTidx, T, ctx->dFaTab.p, ctx->dFaXr.p, ctx->dFaH0.p,
                                      ctx->fa_h0_kind, ctx->fa_tag_word, ctx->dFaGpow.as<uint64_t>(), ctx->prm.q, (int)ctx->n,
                                      (int)ctx->k, Bc, dU, ctx->n, ctx->dFlag.as<int>(), ctx->stream));
        return QF_OK;
    }
    int* hist = ctx->dFaSort.as<int>();
    int *off = hist + (T + 1), *gstart = off + (T + 1), *perm = nullptr;
    if (QF_F_A_TAG_GROUP > 1) {  // always in the library; 1 only in the benchmark's comparison build (kernels.h)
        CK(ctx->dFaPerm.ensure((size_t)Bc * sizeof(int)));
        perm = ctx->dFaPerm.as<int>();
        LAUNCH(qf_launch_f_a_tag_sort(dTidx, Bc, T, hist, off, gstart, perm, ctx->dFlag.as<int>(), ctx->stream));
    }
    LAUNCH(qf_launch_f_a_tag_correct(dSigma, ctx->dim, (int)ctx->m_bar, dTidx, T, perm, off, gstart, ctx->dFaTab.p,
                                     ctx->fa_tag_word, ctx->dFaGpow.as<uint64_t>(), ctx->prm.q, (int)ctx->n, (int)ctx->k, Bc,
                                     dU, ctx->n, ctx->dFlag.as<int>(), ctx->stream));
    return QF_OK;
}

qf_status install_a(qf_ctx* ctx, const int64_t* a) {
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "qf_set_a on a ring context; use qf_ring_set_a");
    // a new key invalidates whatever trapdoor was installed for the old one: samp_p answers QF_ERR_NO_KEY until the
    // trapdoor is installed again (never a preimage of the new A computed from the old A^-1, pivots, S and R)
    ctx->has_a = false; ctx->has_np = false; ctx->has_pert = false;
    ctx->key_tagged = false; ctx->pert_gadget_key = false;
    ctx->dHinvl.release(); ctx->dAbpl.release();
    ctx->tag_count = 0; ctx->dTagTab.release(); ctx->dTagH0.release(); ctx->dTagXr.release();
    ctx->fa_tag_count = 0; ctx->dFaTab.release(); ctx->dFaXr.release(); ctx->dFaH0.release();
    ctx->drop_pool();
    const long n = ctx->n, m = ctx->m;
    for (long i = 0; i < n * m; ++i)
        if (a[i] < 0 || (uint64_t)a[i] >= ctx->prm.q) return ctx->fail(QF_ERR_INVALID, "A entry outside [0,q)");
    ctx->hA.assign(a, a + n * m);
    const int qbits = bitlen_u64(ctx->prm.q - 1);
    int wb = exact_bits(std::sqrt((double)ctx->bound), m);
    if (wb < 4) return ctx->fail(QF_ERR_UNSUPPORTED, "domain bound too large for the exact fp64 contraction");
    wb = std::min(wb, std::max(qbits, 1));
    int nch = (qbits + wb - 1) / wb;
    if (nch < 1) nch = 1;
    if (nch > 4) return ctx->fail(QF_ERR_UNSUPPORTED, "modulus needs more than 4 digit matrices at this domain bound");
    ctx->a_bits = wb;
    ctx->a_nchunks = nch;
    QF_TRY(upload_chunks(ctx, a, n, m, ctx->ld_dim, nch, wb, ctx->dA));
    ctx->a_limbs = (qbits + 7) / 8;
    QF_TRY(upload_limbs(ctx, a, n, m, ctx->ldk_dim, ctx->a_limbs, false, ctx->dAl));
    ctx->has_a = true;
    return QF_OK;
}

// Columns [c0, m) of the host copy of A into the device representations install_a built (fp64 digit matrices and u8 digit
// planes); the other columns are left as they are
qf_status upload_a_cols(qf_ctx* ctx, long c0) {
    const long n = ctx->n, m = ctx->m, w = m - c0;
    std::vector<double> f((size_t)n * w);
    const unsigned long long mask = (ctx->a_bits >= 64) ? ~0ull : ((1ull << ctx->a_bits) - 1);
    for (int c = 0; c < ctx->a_nchunks; ++c) {
        for (long i = 0; i < n; ++i)
            for (long j = 0; j < w; ++j) f[(size_t)i * w + j] = (double)(((unsigned long long)ctx->hA[(size_t)i * m + c0 + j] >> (c * ctx->a_bits)) & mask);
        CK(cudaMemcpy2DAsync(ctx->dA[c].as<double>() + c0, (size_t)ctx->ld_dim * 8, f.data(), (size_t)w * 8, (size_t)w * 8, (size_t)n,
                             cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    std::vector<uint8_t> b((size_t)n * w);
    for (int l = 0; l < ctx->a_limbs; ++l) {
        for (long i = 0; i < n; ++i)
            for (long j = 0; j < w; ++j) b[(size_t)i * w + j] = (uint8_t)((uint64_t)ctx->hA[(size_t)i * m + c0 + j] >> (8 * l));
        CK(cudaMemcpy2DAsync(ctx->dAl.as<uint8_t>() + (size_t)l * n * ctx->ldk_dim + c0, (size_t)ctx->ldk_dim, b.data(), (size_t)w, (size_t)w,
                             (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return QF_OK;
}

// PSFGPV takes a tag per target, and switches tags, only on the two-phase recursion: there the tag enters between the
// phases alone, while the one-pass recursion reads U_12, which depends on the tag (DESIGN 4.3)
qf_status gpv_tags_ready(qf_ctx* ctx) {
    if (!ctx->has_np || !ctx->two_phase)
        return ctx->fail(QF_ERR_INVALID, "PSFGPV tags need a G-trapdoor key and its basis on the two-phase recursion");
    return QF_OK;
}

// A^-1 on the unit pivots of the classical key (find_unit_pivots) as fp64 digit matrices: the particular-solution map
qf_status upload_ainv(qf_ctx* ctx, const std::vector<int64_t>& ainv) {
    ctx->npiv = (int)ctx->n;
    ctx->ainv_identity = false;
    const int qbits = bitlen_u64(ctx->prm.q - 1);
    int wb = exact_bits((double)ctx->prm.q * std::sqrt((double)ctx->n), ctx->n);
    if (wb < 2) return ctx->fail(QF_ERR_UNSUPPORTED, "modulus too large for the exact particular-solution product");
    wb = std::min(wb, qbits);
    int nch = (qbits + wb - 1) / wb;
    if (nch > 4) return ctx->fail(QF_ERR_UNSUPPORTED, "modulus needs more than 4 digit matrices (GPV)");
    ctx->ainv_bits = wb; ctx->ainv_nchunks = nch;
    ctx->ld_piv = pad16(ctx->npiv);
    return upload_chunks(ctx, ainv.data(), ctx->n, ctx->n, ctx->ld_piv, nch, wb, ctx->dAinv);
}

// the installed key's tag H_0 into dTagH0 (column-major, tag_word words) for the per-target tag kernel; none for H_0 = I
qf_status upload_tag_h0(qf_ctx* ctx) {
    if (!ctx->key_tagged) {
        ctx->dTagH0.release();
        return QF_OK;
    }
    const long n = ctx->n;
    std::vector<uint64_t> h((size_t)n * n);
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) h[(size_t)j * n + i] = ctx->key_tag[(size_t)i * n + j];
    std::vector<uint32_t> h32;
    const void* src = h.data();
    if (ctx->tag_word == 4) {
        h32.assign(h.begin(), h.end());
        src = h32.data();
    }
    CK(ctx->dTagH0.ensure((size_t)n * n * ctx->tag_word));
    CK(cudaMemcpyAsync(ctx->dTagH0.p, src, (size_t)n * n * ctx->tag_word, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

// ---- tags in polynomial form (qf_set_tag_table_poly, qf_set_f_a_tags_poly)
typedef unsigned __int128 u128h;

uint64_t powmod_u64(uint64_t a, uint64_t e, uint64_t m) {
    uint64_t r = 1 % m;
    for (a %= m; e; e >>= 1, a = (uint64_t)((u128h)a * a % m))
        if (e & 1) r = (uint64_t)((u128h)r * a % m);
    return r;
}

// deterministic for every n < 2^64 (the first twelve primes as witnesses)
bool is_prime_u64(uint64_t n) {
    if (n < 2) return false;
    static const uint64_t W[] = {2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37};
    for (uint64_t w : W)
        if (n % w == 0) return n == w;
    uint64_t d = n - 1;
    int r = 0;
    while (!(d & 1)) d >>= 1, ++r;
    for (uint64_t w : W) {
        uint64_t x = powmod_u64(w, d, n);
        if (x == 1 || x == n - 1) continue;
        bool comp = true;
        for (int i = 1; i < r && comp; ++i) {
            x = (uint64_t)((u128h)x * x % n);
            comp = x != n - 1;
        }
        if (comp) return false;
    }
    return true;
}

// r^e compared with q without overflow: -1, 0, 1
int pow_cmp(uint64_t r, int e, uint64_t q) {
    u128h x = 1;
    for (int i = 0; i < e; ++i) {
        x *= r;
        if (x > q) return 1;
    }
    return x == q ? 0 : -1;
}

// q = p^e with p prime: the largest e for which q is a perfect e-th power, and its root must be prime
bool prime_power(uint64_t q, uint64_t* p, int* e) {
    for (int ee = 63; ee >= 1; --ee) {
        uint64_t r = (uint64_t)std::llround(std::pow((double)q, 1.0 / ee));
        while (r > 1 && pow_cmp(r, ee, q) > 0) --r;
        while (pow_cmp(r + 1, ee, q) <= 0) ++r;
        if (r >= 2 && pow_cmp(r, ee, q) == 0) {
            if (!is_prime_u64(r)) return false;
            *p = r;
            *e = ee;
            return true;
        }
    }
    return false;
}

// f mod q on the device and the rows X^{n+j} mod (f, q) of the product (qf_launch_poly_xpow)
qf_status poly_modulus(qf_ctx* ctx, const int64_t* f, int word, Dev& dF, Dev& xr) {
    const long n = ctx->n;
    const uint64_t q = ctx->prm.q;
    std::vector<uint64_t> fq((size_t)n);
    for (long i = 0; i < n; ++i) {
        const int64_t v = f[i] % (int64_t)q;
        fq[i] = (uint64_t)(v < 0 ? v + (int64_t)q : v);
    }
    CK(dF.ensure((size_t)n * 8));
    CK(xr.ensure((size_t)std::max(1L, n - 1) * n * word));
    CK(cudaMemcpyAsync(dF.p, fq.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(qf_launch_poly_xpow(dF.as<uint64_t>(), (int)n, q, word, xr.p, ctx->stream));
    return QF_OK;
}
}  // namespace

extern "C" {

const char* qf_version(void) { return "qfall_b200 0.1 (sm_100a)"; }

qf_status qf_ctx_create(const qf_params* p, int device, qf_ctx** out) {
    if (!p || !out) return QF_ERR_INVALID;
    *out = nullptr;
    if (p->n < 1 || p->k < 1 || p->base < 2 || p->q < 2 || p->q >= (1ull << 62) || !(p->s > 0)) return QF_ERR_INVALID;
    if (p->kind < 0 || p->kind > 2) return QF_ERR_INVALID;
    qf_ctx* ctx = new qf_ctx();
    ctx->prm = *p;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return QF_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    ctx->n = p->n; ctx->k = p->k; ctx->m_bar = p->m_bar; ctx->nk = p->n * p->k;
    if (p->kind == QF_PSF_GPV_RING) {
        ctx->m = p->k + 2;
        ctx->dim = p->n * (p->k + 2);
    } else {
        ctx->m = p->m_bar + ctx->nk;
        ctx->dim = ctx->m;
    }
    ctx->ld_dim = pad16(ctx->dim); ctx->ld_n = pad16(ctx->n); ctx->ld_nk = pad16(ctx->nk);
    const double r = (p->kind == QF_PSF_PERTURBATION) ? p->r : 1.0;
    ctx->s_samp_d = p->s * r;
    if (p->norm_bound) {
        ctx->bound = p->norm_bound;
    } else {
        long double b = (long double)p->s * p->s * (long double)ctx->dim * (long double)r * r;
        ctx->bound = (unsigned long long)floorl(b);
    }
    ctx->ldk_dim = (ctx->dim + 127) / 128 * 128;
    ctx->ldk_nk = (ctx->nk + 127) / 128 * 128;
    ctx->ldk_n = (ctx->n + 127) / 128 * 128;
    ctx->x_limbs = limbs_for(std::sqrt((double)ctx->bound));
    {
        const char* env = getenv("QF_DISABLE_I8");
        ctx->use_i8 = !(env && env[0] == '1');
        const char* envf = getenv("QF_DISABLE_FUSED_FA");
        ctx->fused_fa = !(envf && envf[0] == '1');
        const char* envu = getenv("QF_DISABLE_NP_FUSE64");  // test switch: separate K = 64 GEMM launches as before
        ctx->np_fuse64 = !(envu && envu[0] == '1');
        const char* envs = getenv("QF_DISABLE_NP_FUSE_SPLIT");  // test switch: separate digit-split launches
        ctx->np_fuse_split = !(envs && envs[0] == '1');
        const char* envv = getenv("QF_NP_DIAG_V1");  // test switch: the quad-per-two-targets diagonal-block kernel
        ctx->np_diag_variant = (envv && envv[0] == '1') ? 1 : 0;
        if (const char* envc = getenv("QF_CHUNK")) ctx->chunk_env = atol(envc);  // experiments: targets per internal chunk
        const char* envd = getenv("QF_NP_DLO");  // test switch: 0 = every digit pair of the fixed-point updates
        if (envd) ctx->np_dlo = std::max(0, std::min(3, atoi(envd)));
    }
    // default chunk: keep ~8 fp64-sized work matrices within ~32 GB (of 180 GB); whole waves of 148 SMs x 128-target tiles.
    // Two waves (C2: 37 888 targets) give the per-target sequential kernel two CTAs per SM and halve the number of
    // latency-bound short-K launches per target: 384 k/s against 344 k/s at one wave.
    long per_target = ctx->ld_dim * 8 * 8;
    long c = (long)((32LL << 30) / std::max(1L, per_target));
    c = std::max(128L, std::min(75776L, c / 128 * 128));
    if (c >= 148 * 128) c = c / (148 * 128) * (148 * 128);
    ctx->chunk = ctx->chunk_env > 0 ? ctx->chunk_env : c;
    if (ctx->dFlag.ensure(sizeof(int)) != cudaSuccess || cudaMemset(ctx->dFlag.p, 0, sizeof(int)) != cudaSuccess) {
        delete ctx;
        return QF_ERR_CUDA;
    }
    *out = ctx;
    return QF_OK;
}

void qf_ctx_destroy(qf_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    cudaStream_t s = ctx->own_stream;
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
        if (ctx->ev_u_in[i]) cudaEventDestroy(ctx->ev_u_in[i]);
        if (ctx->ev_u_used[i]) cudaEventDestroy(ctx->ev_u_used[i]);
    }
    for (auto& r : ctx->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto& e : ctx->ev_pool) cudaEventDestroy(e);
    delete ctx;
    if (s) cudaStreamDestroy(s);
}

const char* qf_last_error(const qf_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
uint64_t qf_launch_count(const qf_ctx* ctx) { return ctx ? ctx->launches : 0; }

qf_status qf_set_stream(qf_ctx* ctx, void* s) {
    if (!ctx) return QF_ERR_INVALID;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return QF_OK;
}
qf_status qf_set_chunk(qf_ctx* ctx, int64_t c) {
    if (!ctx || c < 0) return QF_ERR_INVALID;
    if (c == 0) return QF_OK;
    ctx->chunk = std::max<int64_t>(1, c);
    return QF_OK;
}
qf_status qf_synchronize(qf_ctx* ctx) {
    if (!ctx) return QF_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    return check_flag(ctx);
}

qf_status qf_profile(qf_ctx* ctx, int enable) {
    if (!ctx) return QF_ERR_INVALID;
    ctx->prof = enable != 0;
    if (ctx->prof) {
        CK(ctx->dMma.ensure(8));
        CK(cudaMemsetAsync(ctx->dMma.p, 0, 8, ctx->stream));
    }
    return QF_OK;
}

qf_status qf_profile_read(qf_ctx* ctx, double* gemm_ms, double* gemm_flops, uint64_t* gemm_launches, double* i8_ms,
                          double* i8_ops, double* i8_issued_ops, uint64_t* i8_launches) {
    if (!ctx) return QF_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    double ms[2] = {0, 0}, fl[2] = {0, 0}, issued = 0;
    uint64_t cnt[2] = {0, 0};
    for (auto& r : ctx->prof_recs) {
        float t = 0;
        cudaEventElapsedTime(&t, r.a, r.b);
        ms[r.kind] += t;
        fl[r.kind] += r.flops;
        cnt[r.kind] += 1;
        if (r.kind == 1) issued += r.issued;
        ctx->ev_pool.push_back(r.a);
        ctx->ev_pool.push_back(r.b);
    }
    if (gemm_ms) *gemm_ms = ms[0];
    if (gemm_flops) *gemm_flops = fl[0];
    if (gemm_launches) *gemm_launches = cnt[0];
    if (i8_ms) *i8_ms = ms[1];
    if (i8_ops) *i8_ops = fl[1];
    if (ctx->dMma.p) {  // executed tensor-pipe operations counted by the kernel itself (zero digit tiles skipped)
        unsigned long long h = 0;
        CK(cudaMemcpy(&h, ctx->dMma.p, 8, cudaMemcpyDeviceToHost));
        CK(cudaMemset(ctx->dMma.p, 0, 8));
        issued = (double)h;
    }
    if (i8_issued_ops) *i8_issued_ops = issued;
    if (i8_launches) *i8_launches = cnt[1];
    ctx->prof_recs.clear();
    return QF_OK;
}

qf_status qf_set_a(qf_ctx* ctx, const int64_t* a) {
    if (!ctx || !a) return QF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    return install_a(ctx, a);
}

qf_status qf_set_trapdoor_perturbation(qf_ctx* ctx, const int8_t* r, const double* l, const int64_t* sk,
                                       const double* skg) {
    if (!ctx || !r || !sk || !skg) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a PSFPerturbation context");
    if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "install A first (qf_set_a / qf_trap_gen)");
    ctx->has_pert = false;
    ctx->key_tagged = false; ctx->pert_gadget_key = false;
    ctx->tag_count = 0; ctx->dTagTab.release(); ctx->dTagH0.release(); ctx->dTagXr.release();
    ctx->drop_pool();
    CK(cudaSetDevice(ctx->device));
    QF_TRY(upload_as_f64(ctx, r, ctx->m_bar, ctx->nk, ctx->ld_nk, ctx->dR));
    {
        std::vector<int64_t> r64((size_t)ctx->m_bar * ctx->nk);
        for (size_t i = 0; i < r64.size(); ++i) r64[i] = r[i];
        QF_TRY(upload_limbs(ctx, r64.data(), ctx->m_bar, ctx->nk, ctx->ldk_nk, 1, true, ctx->dRl));
    }
    // A = [A_bar | H G - A_bar R]: A [R; I] = H G, so samp_p samples z with G z = H^-1 (u - A p) (samp_p_pert_chunk).  A tag
    // without a unit pivot is refused, as by qf_gen_short_basis_tagged; a key of another form is installed as it is.
    {
        KeyTag kt;
        QF_TRY(match_key_tag(ctx, r, true, ctx->dHinvl, kt));
        if (kt.form == KEY_TAG_SINGULAR)
            return ctx->fail(QF_ERR_INVALID, "key is [A_bar | H G - A_bar R] with a tag H that is not invertible mod q (no unit pivot)");
        if (kt.form != KEY_TAGGED) ctx->dHinvl.release();
        ctx->pert_gadget_key = kt.form != KEY_OTHER;
        ctx->key_tagged = kt.form == KEY_TAGGED;
        ctx->tag_ulimbs = limbs_for((double)(ctx->prm.q - 1));
        ctx->key_tag = std::move(kt.h);
    }
    if (l) {
        QF_TRY(upload_as_f64(ctx, l, ctx->m, ctx->m, ctx->ld_dim, ctx->dL));
        ctx->pert_structured = false;
        ctx->l_tri = 1;
        for (long i = 0; i < ctx->m && ctx->l_tri; ++i)
            for (long j = i + 1; j < ctx->m; ++j)
                if (l[i * ctx->m + j] != 0.0) { ctx->l_tri = 0; break; }
        ctx->dLs.release();
    } else {
        if (!ctx->use_i8) return ctx->fail(QF_ERR_UNSUPPORTED, "structured sqrt(Sigma_2) needs the int8 tensor path");
        ctx->dL.release();
        QF_TRY(setup_structured_sigma2(ctx));
    }
    QF_TRY(upload_as_f64(ctx, sk, ctx->k, ctx->k, ctx->k, ctx->dSk));
    QF_TRY(upload_as_f64(ctx, skg, ctx->k, ctx->k, ctx->k, ctx->dSkGso));
    QF_TRY(setup_pert_i8(ctx));
    ctx->has_pert = true;
    return QF_OK;
}

qf_status qf_set_tag(qf_ctx* ctx, const int64_t* tag, int64_t* a_out) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a PSFPerturbation context");
    if (!ctx->has_a || !ctx->has_pert) return ctx->fail(QF_ERR_NO_KEY, "PSFPerturbation: key or trapdoor missing");
    if (!ctx->pert_gadget_key) return ctx->fail(QF_ERR_INVALID, "the installed key is not [A_bar | H G - A_bar R] for the installed R");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, k = ctx->k, mb = ctx->m_bar, m = ctx->m;
    const uint64_t q = ctx->prm.q;
    // the new tag H' as MatZq (entries reduced mod q); H'^-1 before anything changes, so that a tag without a unit pivot
    // leaves the key, its tag and the outputs as they were
    std::vector<uint64_t> h2((size_t)n * n);
    bool ident = true;
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) {
            uint64_t v = i == j ? 1 : 0;
            if (tag) {
                const int64_t t = tag[i * n + j] % (int64_t)q;
                v = (uint64_t)(t < 0 ? t + (int64_t)q : t);
            }
            h2[(size_t)i * n + j] = v;
            ident = ident && v == (i == j ? 1u : 0u);
        }
    std::vector<int64_t> hinv;
    if (!ident) {
        bool ok = false;
        QF_TRY(tag_inverse(ctx, h2.data(), hinv, &ok));
        if (!ok) return ctx->fail(QF_ERR_INVALID, "tag is not invertible mod q (no unit pivot)");
    }
    // A_2 += (H' - H) G mod q: only the last nk columns of A change, R, sqrt(Sigma_2) and the gadget basis stay.  Until the
    // device copies are consistent again the context has no key (a CUDA error on the way leaves it so).
    ctx->has_a = false;
    ctx->has_pert = false;
    // the f_a table is relative to A, which changes here
    ctx->fa_tag_count = 0; ctx->dFaTab.release(); ctx->dFaXr.release(); ctx->dFaH0.release();
    ctx->drop_pool();
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) {
            const uint64_t d = (h2[(size_t)i * n + j] + q - ctx->key_tag[(size_t)i * n + j]) % q;
            if (!d) continue;
            for (long t = 0; t < k; ++t) {
                int64_t& a = ctx->hA[(size_t)i * m + mb + j * k + t];
                a = (int64_t)(((u128)(uint64_t)a + mulmod_h(d, gpow[t], q)) % q);
            }
        }
    QF_TRY(upload_a_cols(ctx, mb));
    if (ident) ctx->dHinvl.release();
    else QF_TRY(tag_planes(ctx, hinv, ctx->dHinvl));
    ctx->key_tagged = !ident;
    ctx->key_tag = std::move(h2);
    if (ctx->tag_count) QF_TRY(upload_tag_h0(ctx));  // the tag table stays: it is relative to (A_bar, R)
    ctx->has_a = true;
    ctx->has_pert = true;
    if (a_out) memcpy(a_out, ctx->hA.data(), (size_t)n * m * sizeof(int64_t));
    return QF_OK;
}

// PSFGPV tag switch (DESIGN 4.3): for A = [A_bar | H G - A_bar R] with S_H installed on the two-phase recursion, the GSO of
// S_H' is that of S_H, so U, Mt_1, M', D and their digit planes stay; what depends on H' is rebuilt here exactly as
// qf_set_a(A') + qf_set_trapdoor_gpv(S_H') would build it: A' (host copy, the nk changed columns on the device), the key's
// tag, H'^-1 and A_bar' = H'^-1 A_bar (digit planes), W = digits(-A_bar'), and the pivots of A' when they can differ.
qf_status qf_gpv_set_tag(qf_ctx* ctx, const int64_t* tag, int64_t* a_out, int64_t* s_out) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV) return ctx->fail(QF_ERR_INVALID, "not a PSFGPV context (PSFPerturbation: qf_set_tag)");
    QF_TRY(gpv_tags_ready(ctx));
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, k = ctx->k, mb = ctx->m_bar, nk = ctx->nk, m = ctx->m;
    const uint64_t q = ctx->prm.q, base = (uint64_t)ctx->prm.base;
    // everything that can refuse runs before the context changes: H'^-1, the pivots of A', the basis for the caller
    std::vector<uint64_t> h2((size_t)n * n);
    std::vector<int64_t> h2w((size_t)n * n);
    bool ident = true;
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) {
            uint64_t v = i == j ? 1 : 0;
            if (tag) {
                const int64_t t = tag[i * n + j] % (int64_t)q;
                v = (uint64_t)(t < 0 ? t + (int64_t)q : t);
            }
            h2[(size_t)i * n + j] = v;
            h2w[(size_t)i * n + j] = (int64_t)v;
            ident = ident && v == (i == j ? 1u : 0u);
        }
    std::vector<int64_t> hinv;
    Dev dHl;
    if (!ident) {
        bool ok = false;
        QF_TRY(tag_inverse(ctx, h2.data(), hinv, &ok));
        if (!ok) return ctx->fail(QF_ERR_INVALID, "tag is not invertible mod q (no unit pivot)");
        QF_TRY(tag_planes(ctx, hinv, dHl));
    }
    // A' = A + [0 | (H' - H) G] mod q
    std::vector<int64_t> a2 = ctx->hA;
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    for (long i = 0; i < n; ++i)
        for (long j = 0; j < n; ++j) {
            const uint64_t d = (h2[(size_t)i * n + j] + q - ctx->key_tag[(size_t)i * n + j]) % q;
            if (!d) continue;
            for (long t = 0; t < k; ++t) {
                int64_t& a = a2[(size_t)i * m + mb + j * k + t];
                a = (int64_t)(((u128)(uint64_t)a + mulmod_h(d, gpow[t], q)) % q);
            }
        }
    // The pivot search walks the columns in order and stops at n pivots: when all of them lie in A_bar, which H' leaves
    // unchanged, the search over A' makes the same choices.  Otherwise it runs again.
    std::vector<int> piv((size_t)ctx->npiv);
    CK(cudaMemcpy(piv.data(), ctx->dPiv.p, piv.size() * sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<int64_t> ainv;
    const bool repivot = *std::max_element(piv.begin(), piv.end()) >= mb;
    if (repivot && !find_unit_pivots(a2.data(), n, m, q, piv, ainv))
        return ctx->fail(QF_ERR_UNSUPPORTED, "A has no n columns invertible over Z_q by unit pivoting");
    if (s_out) {
        // the basis reads A_bar only (the first m_bar columns of the installed A) and R, read back from its s8 plane
        std::vector<int8_t> r((size_t)mb * nk);
        CK(cudaMemcpy2D(r.data(), (size_t)nk, ctx->dRl.p, (size_t)ctx->ldk_nk, (size_t)nk, (size_t)mb, cudaMemcpyDeviceToHost));
        QF_TRY(qf_gen_short_basis_tagged(ctx, r.data(), ident ? nullptr : h2w.data(), s_out));
    }
    // A_bar' = H'^-1 A_bar (reads the unchanged first m_bar columns of hA) and W = digits(-A_bar'), nk x m_bar
    std::vector<int64_t> abt;
    if (!ident) QF_TRY(tag_abar(ctx, dHl, abt));
    std::vector<int64_t> w64((size_t)nk * mb), ab;
    for (long j = 0; j < n; ++j)
        for (long c = 0; c < mb; ++c) {
            uint64_t v = (q - (uint64_t)(ident ? ctx->hA[(size_t)j * m + c] : abt[(size_t)c * n + j])) % q;
            for (long t = 0; t < k; ++t) {
                w64[(size_t)(j * k + t) * mb + c] = (int64_t)(v % base);
                v /= base;
            }
        }
    // commit.  Until the device copies are consistent again the context has no trapdoor (a CUDA error on the way leaves it so).
    ctx->has_np = false;
    // the f_a table is relative to A; the samp_p table to (A_bar, R): kept
    ctx->fa_tag_count = 0; ctx->dFaTab.release(); ctx->dFaXr.release(); ctx->dFaH0.release();
    ctx->drop_pool();
    ctx->hA.swap(a2);
    QF_TRY(upload_a_cols(ctx, mb));
    if (repivot) {
        QF_TRY(upload_ainv(ctx, ainv));
        CK(cudaMemcpy(ctx->dPiv.p, piv.data(), piv.size() * sizeof(int), cudaMemcpyHostToDevice));
        bool piv_low = false;
        for (int pc : piv) piv_low = piv_low || pc >= mb;
        ctx->i2_limbs = limbs_for(8.0 * ctx->prm.s + 64.0 + (piv_low ? (double)q : 0.0));
    }
    QF_TRY(upload_limbs(ctx, w64.data(), nk, mb, ctx->ldk_mb, 1, false, ctx->dWl));
    if (ident) {
        ctx->dHinvl.release();
        ctx->dAbpl.release();
    } else {
        std::swap(ctx->dHinvl.p, dHl.p);
        std::swap(ctx->dHinvl.cap, dHl.cap);
        ab.resize((size_t)n * mb);
        for (long i = 0; i < n; ++i)
            for (long c = 0; c < mb; ++c) ab[(size_t)i * mb + c] = abt[(size_t)c * n + i];
        QF_TRY(upload_limbs(ctx, ab.data(), n, mb, ctx->ldk_mb, ctx->a_limbs, false, ctx->dAbpl));
        ctx->tag_ulimbs = limbs_for((double)(q - 1));
    }
    ctx->key_tagged = !ident;
    ctx->key_tag = std::move(h2);
    ctx->has_np = true;
    if (a_out) memcpy(a_out, ctx->hA.data(), (size_t)n * m * sizeof(int64_t));
    return QF_OK;
}

constexpr int64_t TAG_SLICE = 256;  // tags inverted per launch: 2 CTAs of 1024 threads per SM, one wave

// H_t^-1 for every tag on the device: [H_t | I] built from the caller's words (reduced mod q there), Gauss-Jordan with unit
// pivots one CTA per tag, packed column-major.  Slices of at most TAG_SLICE tags and 1 GB bound the scratch ([H | I] is
// 16 n^2 bytes per tag, 4 MB at n = 512).  The new table replaces the old one only when every tag has been inverted.
qf_status qf_set_tag_table(qf_ctx* ctx, const int64_t* tags, int64_t ntags) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV) {
        QF_TRY(gpv_tags_ready(ctx));
    } else if (ctx->prm.kind != QF_PSF_PERTURBATION) {
        return ctx->fail(QF_ERR_INVALID, "not a PSFGPV or PSFPerturbation context");
    }
    if (!tags || ntags < 1) return ctx->fail(QF_ERR_INVALID, "tag table: at least one tag needed");
    if (ctx->prm.kind == QF_PSF_PERTURBATION) {
        if (!ctx->has_a || !ctx->has_pert) return ctx->fail(QF_ERR_NO_KEY, "PSFPerturbation: key or trapdoor missing");
        if (!ctx->pert_gadget_key) return ctx->fail(QF_ERR_INVALID, "the installed key is not [A_bar | H G - A_bar R] for the installed R");
    }
    const long n = ctx->n;
    if (ctx->k > 64 || 16 * n > 227 * 1024) return ctx->fail(QF_ERR_UNSUPPORTED, "tag table: needs k <= 64 and n <= 14528");
    if (ntags > INT32_MAX) return ctx->fail(QF_ERR_INVALID, "tag table: more than 2^31 - 1 tags");
    CK(cudaSetDevice(ctx->device));
    const uint64_t q = ctx->prm.q;
    const int word = q <= (1ull << 32) ? 4 : 8;
    const size_t nn = (size_t)n * n;
    const int64_t slice = std::max<int64_t>(1, std::min<int64_t>({ntags, TAG_SLICE, (int64_t)((1ull << 30) / (16 * nn))}));
    Dev tab, dTags, dM, dF, dFail;
    CK(tab.ensure((size_t)ntags * nn * word));
    CK(dTags.ensure((size_t)slice * nn * 8));
    CK(dM.ensure((size_t)slice * nn * 16));
    CK(dF.ensure((size_t)slice * n * 8));
    CK(dFail.ensure((size_t)slice * sizeof(int)));
    std::vector<int> fail((size_t)slice);
    for (int64_t t0 = 0; t0 < ntags; t0 += slice) {
        const int cnt = (int)std::min<int64_t>(slice, ntags - t0);
        CK(cudaMemcpyAsync(dTags.p, tags + (size_t)t0 * nn, (size_t)cnt * nn * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_tag_build(dTags.as<int64_t>(), cnt, (int)n, q, dM.as<uint64_t>(), ctx->stream));
        LAUNCH(qf_launch_mat_inverse_mod_batched(dM.as<uint64_t>(), dF.as<uint64_t>(), (int)n, q, dFail.as<int>(), cnt, ctx->stream));
        LAUNCH(qf_launch_tag_pack(dM.as<uint64_t>(), cnt, (int)n, word, tab.as<char>() + (size_t)t0 * nn * word, ctx->stream));
        CK(cudaMemcpyAsync(fail.data(), dFail.p, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < cnt; ++i)
            if (fail[i]) {
                char buf[128];
                snprintf(buf, sizeof buf, "tag %lld is not invertible mod q (no unit pivot)", (long long)(t0 + i));
                return ctx->fail(QF_ERR_INVALID, buf);
            }
    }
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    CK(ctx->dTagGpow.ensure(gpow.size() * 8));
    CK(cudaMemcpyAsync(ctx->dTagGpow.p, gpow.data(), gpow.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    ctx->tag_word = word;
    if (ctx->prm.kind == QF_PSF_PERTURBATION) QF_TRY(upload_tag_h0(ctx));  // PSFGPV's h_t does not involve H_0
    std::swap(ctx->dTagTab.p, tab.p);
    std::swap(ctx->dTagTab.cap, tab.cap);
    ctx->tag_poly = false;
    ctx->dTagXr.release();
    ctx->tag_count = ntags;
    return QF_OK;
}

// D_t = H_t - H_0 mod q for every tag, built on the device from the caller's words in slices of at most 1 GB of int64 tags.
// No trapdoor is needed and no tag is inverted.  The new table replaces the old one only when it is complete.
qf_status qf_set_f_a_tags(qf_ctx* ctx, const int64_t* tags, int64_t ntags, const int64_t* h0) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "f_a tag table: not a classical context");
    if (!tags || ntags < 1) return ctx->fail(QF_ERR_INVALID, "f_a tag table: at least one tag needed");
    if (ntags >= INT32_MAX) return ctx->fail(QF_ERR_INVALID, "f_a tag table: more than 2^31 - 2 tags");
    if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    const long n = ctx->n;
    CK(cudaSetDevice(ctx->device));
    int supported = 0;
    CK(qf_f_a_tag_supported((int)std::min<long>(n, INT32_MAX), (int)ctx->k, &supported));
    if (!supported)
        return ctx->fail(QF_ERR_UNSUPPORTED, "f_a tag table: needs k <= 64 and the group's shared memory within one block's limit");
    const uint64_t q = ctx->prm.q;
    const int word = q <= (1ull << 32) ? 4 : 8;
    const size_t nn = (size_t)n * n;
    const int64_t slice = std::max<int64_t>(1, std::min<int64_t>(ntags, (int64_t)((1ull << 30) / (8 * nn))));
    Dev tab, dTags, dH0, sort;
    CK(tab.ensure((size_t)ntags * nn * word));
    CK(dTags.ensure((size_t)slice * nn * 8));
    CK(sort.ensure((size_t)3 * (ntags + 1) * sizeof(int)));
    if (h0) {
        std::vector<uint64_t> h((size_t)nn);
        for (size_t x = 0; x < nn; ++x) {
            const int64_t v = h0[x] % (int64_t)q;
            h[x] = (uint64_t)(v < 0 ? v + (int64_t)q : v);
        }
        CK(dH0.ensure(nn * 8));
        CK(cudaMemcpyAsync(dH0.p, h.data(), nn * 8, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    for (int64_t t0 = 0; t0 < ntags; t0 += slice) {
        const int cnt = (int)std::min<int64_t>(slice, ntags - t0);
        CK(cudaMemcpyAsync(dTags.p, tags + (size_t)t0 * nn, (size_t)cnt * nn * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_tag_diff_pack(dTags.as<int64_t>(), cnt, (int)n, q, dH0.as<uint64_t>(), word,
                                       tab.as<char>() + (size_t)t0 * nn * word, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));  // dTags is refilled by the next slice
    }
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    CK(ctx->dFaGpow.ensure(gpow.size() * 8));
    CK(cudaMemcpyAsync(ctx->dFaGpow.p, gpow.data(), gpow.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::swap(ctx->dFaTab.p, tab.p);
    std::swap(ctx->dFaTab.cap, tab.cap);
    std::swap(ctx->dFaSort.p, sort.p);
    std::swap(ctx->dFaSort.cap, sort.cap);
    ctx->fa_tag_word = word;
    ctx->fa_poly = false;
    ctx->dFaXr.release();
    ctx->dFaH0.release();
    ctx->fa_tag_count = ntags;
    return QF_OK;
}

// ---- tags in polynomial form: H_t = rot_f(h_t), column c = coeffs(h_t X^c mod f) (DESIGN 4.10) -------------------------

// h_t^-1 mod (f, q) for every tag on the device (qf_launch_poly_tag_inverse, one CTA per tag), for q = p^e.  Tags are
// copied in slices of at most 1 GB.  The new table replaces the old one, of either form, only when every tag is a unit.
qf_status qf_set_tag_table_poly(qf_ctx* ctx, const int64_t* f, const int64_t* tags, int64_t ntags) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV) {
        QF_TRY(gpv_tags_ready(ctx));
    } else if (ctx->prm.kind != QF_PSF_PERTURBATION) {
        return ctx->fail(QF_ERR_INVALID, "not a PSFGPV or PSFPerturbation context");
    }
    if (!f || !tags || ntags < 1) return ctx->fail(QF_ERR_INVALID, "tag table: f and at least one tag needed");
    if (ctx->prm.kind == QF_PSF_PERTURBATION) {
        if (!ctx->has_a || !ctx->has_pert) return ctx->fail(QF_ERR_NO_KEY, "PSFPerturbation: key or trapdoor missing");
        if (!ctx->pert_gadget_key) return ctx->fail(QF_ERR_INVALID, "the installed key is not [A_bar | H G - A_bar R] for the installed R");
    }
    if (ntags > INT32_MAX) return ctx->fail(QF_ERR_INVALID, "tag table: more than 2^31 - 1 tags");
    const long n = ctx->n;
    const uint64_t q = ctx->prm.q;
    uint64_t p = 0;
    int e = 0;
    if (!prime_power(q, &p, &e))
        return ctx->fail(QF_ERR_UNSUPPORTED, "tag table in polynomial form: q must be a prime power");
    CK(cudaSetDevice(ctx->device));
    int supported = 0;
    CK(qf_poly_tag_supported((int)std::min<long>(n, INT32_MAX), (int)std::min<long>(ctx->k, INT32_MAX), 1, &supported));
    if (!supported)
        return ctx->fail(QF_ERR_UNSUPPORTED, "tag table in polynomial form: needs k <= 64 and the shared memory within one block's limit");
    int lifts = 0;
    while ((1 << lifts) < e) ++lifts;
    const int word = q <= (1ull << 32) ? 4 : 8;
    const int64_t slice = std::max<int64_t>(1, std::min<int64_t>(ntags, (int64_t)((1ull << 30) / (8 * n))));
    Dev tab, xr, dF, dTags, dFail;
    QF_TRY(poly_modulus(ctx, f, word, dF, xr));
    CK(tab.ensure((size_t)ntags * n * word));
    CK(dTags.ensure((size_t)slice * n * 8));
    CK(dFail.ensure((size_t)slice * sizeof(int)));
    std::vector<int> fail((size_t)slice);
    for (int64_t t0 = 0; t0 < ntags; t0 += slice) {
        const int cnt = (int)std::min<int64_t>(slice, ntags - t0);
        CK(cudaMemcpyAsync(dTags.p, tags + (size_t)t0 * n, (size_t)cnt * n * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_poly_tag_inverse(dTags.as<int64_t>(), cnt, (int)n, dF.as<uint64_t>(), xr.p, word, q, p, lifts,
                                          tab.as<char>() + (size_t)t0 * n * word, dFail.as<int>(), ctx->stream));
        CK(cudaMemcpyAsync(fail.data(), dFail.p, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < cnt; ++i)
            if (fail[i]) {
                char buf[128];
                snprintf(buf, sizeof buf, "tag %lld is not a unit mod (f, q)", (long long)(t0 + i));
                return ctx->fail(QF_ERR_INVALID, buf);
            }
    }
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    CK(ctx->dTagGpow.ensure(gpow.size() * 8));
    CK(cudaMemcpyAsync(ctx->dTagGpow.p, gpow.data(), gpow.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    ctx->tag_word = word;
    if (ctx->prm.kind == QF_PSF_PERTURBATION) QF_TRY(upload_tag_h0(ctx));  // PSFGPV's h_t does not involve H_0
    CK(cudaStreamSynchronize(ctx->stream));
    std::swap(ctx->dTagTab.p, tab.p);
    std::swap(ctx->dTagTab.cap, tab.cap);
    std::swap(ctx->dTagXr.p, xr.p);
    std::swap(ctx->dTagXr.cap, xr.cap);
    ctx->tag_poly = true;
    ctx->tag_count = ntags;
    return QF_OK;
}

// h_t mod q as n words per tag and H_0 (NULL: I; all zero: 0; otherwise dense, column-major).  Nothing is inverted: every
// q < 2^62, singular tags and H_0 = 0 work.  The new table replaces the old one, of either form, only when it is complete.
qf_status qf_set_f_a_tags_poly(qf_ctx* ctx, const int64_t* f, const int64_t* tags, int64_t ntags, const int64_t* h0) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "f_a tag table: not a classical context");
    if (!f || !tags || ntags < 1) return ctx->fail(QF_ERR_INVALID, "f_a tag table: f and at least one tag needed");
    if (ntags >= INT32_MAX) return ctx->fail(QF_ERR_INVALID, "f_a tag table: more than 2^31 - 2 tags");
    if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    const long n = ctx->n;
    const uint64_t q = ctx->prm.q;
    CK(cudaSetDevice(ctx->device));
    int supported = 0;
    CK(qf_poly_tag_supported((int)std::min<long>(n, INT32_MAX), (int)std::min<long>(ctx->k, INT32_MAX), 0, &supported));
    if (!supported)
        return ctx->fail(QF_ERR_UNSUPPORTED, "f_a tag table in polynomial form: needs k <= 64 and the shared memory within one block's limit");
    const int word = q <= (1ull << 32) ? 4 : 8;
    const size_t nn = (size_t)n * n;
    int kind = 1;
    std::vector<uint64_t> h;
    if (h0) {
        h.resize(nn);
        bool zero = true, ident = true;
        for (long i = 0; i < n; ++i)
            for (long j = 0; j < n; ++j) {
                const int64_t v = h0[(size_t)i * n + j] % (int64_t)q;
                const uint64_t r = (uint64_t)(v < 0 ? v + (int64_t)q : v);
                h[(size_t)j * n + i] = r;
                zero = zero && r == 0;
                ident = ident && r == (i == j ? 1 % q : 0);
            }
        kind = ident ? 1 : zero ? 0 : 2;
    }
    const int64_t slice = std::max<int64_t>(1, std::min<int64_t>(ntags, (int64_t)((1ull << 30) / (8 * n))));
    Dev tab, xr, dF, dTags, dH0;
    QF_TRY(poly_modulus(ctx, f, word, dF, xr));
    CK(tab.ensure((size_t)ntags * n * word));
    CK(dTags.ensure((size_t)slice * n * 8));
    if (kind == 2) {
        std::vector<uint32_t> h32;
        const void* src = h.data();
        if (word == 4) {
            h32.assign(h.begin(), h.end());
            src = h32.data();
        }
        CK(dH0.ensure(nn * word));
        CK(cudaMemcpyAsync(dH0.p, src, nn * word, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    for (int64_t t0 = 0; t0 < ntags; t0 += slice) {
        const int cnt = (int)std::min<int64_t>(slice, ntags - t0);
        CK(cudaMemcpyAsync(dTags.p, tags + (size_t)t0 * n, (size_t)cnt * n * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_poly_tag_pack(dTags.as<int64_t>(), (long)cnt * n, q, word, tab.as<char>() + (size_t)t0 * n * word,
                                       ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));  // dTags is refilled by the next slice
    }
    const std::vector<uint64_t> gpow = gadget_powers(ctx);
    CK(ctx->dFaGpow.ensure(gpow.size() * 8));
    CK(cudaMemcpyAsync(ctx->dFaGpow.p, gpow.data(), gpow.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::swap(ctx->dFaTab.p, tab.p);
    std::swap(ctx->dFaTab.cap, tab.cap);
    std::swap(ctx->dFaXr.p, xr.p);
    std::swap(ctx->dFaXr.cap, xr.cap);
    std::swap(ctx->dFaH0.p, dH0.p);
    std::swap(ctx->dFaH0.cap, dH0.cap);
    ctx->fa_tag_word = word;
    ctx->fa_h0_kind = kind;
    ctx->fa_poly = true;
    ctx->fa_tag_count = ntags;
    return QF_OK;
}

// gen_short_basis_for_trapdoor_ring (short_basis_ring.rs:64-166) in the coefficient embedding: D x D, D = n (k + 2),
// row = polynomial row * n + coefficient, column = basis vector.  sa_l * sa_r reduced by X^n + 1:
//   column i k + c (i < n, c < k)   = X^i [ sum_j e_j s'_jc ; sum_j r_j s'_jc ; s'_0c ; ... ; s'_{k-1,c} ]
//   column n k + 2 i + c (c = 0, 1) = X^i [ sum_j e_j w_cj + (c == 0) ; sum_j r_j w_cj + (c == 1) ; w_c0 ; ... ; w_c,k-1 ]
// with w_c = base-b digit polynomials of -a_c (a_0 = 1, a_1 = a_bar) and s' = S_k (columns reversed iff base^k = q).
// The polynomial products and sums run on the device; the host only places X^i-rotations (rot^-, rotation_matrix.rs:41-63).
qf_status qf_ring_gen_short_basis(qf_ctx* ctx, const int32_t* r, const int32_t* e, int64_t* s_out) {
    if (!ctx || !r || !e || !s_out) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "not a ring context");
    if (!ctx->has_ring) return ctx->fail(QF_ERR_NO_KEY, "install the ring key first (qf_ring_set_a / qf_ring_trap_gen_from)");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, k = ctx->k, D = n * (k + 2);
    const uint64_t q = ctx->prm.q, base = (uint64_t)ctx->prm.base;
    u128 pw = 1;
    for (long i = 0; i < k; ++i) pw *= base;
    if (pw < q) return ctx->fail(QF_ERR_INVALID, "base^k < q");
    const bool exact_pow = pw == (u128)q;
    // S_k (gadget_classical.rs:248-272), columns reversed when base^k == q (short_basis_ring.rs, as the classical :80-82)
    std::vector<int64_t> sk0((size_t)k * k, 0), sk((size_t)k * k, 0);
    for (long j = 0; j < k; ++j) sk0[j * k + j] = (int64_t)base;
    for (long i = 0; i + 1 < k; ++i) sk0[(i + 1) * k + i] = -1;
    if (!exact_pow) {
        uint64_t qq = q;
        for (long i = 0; i < k; ++i) { sk0[i * k + (k - 1)] = (int64_t)(qq % base); qq /= base; }
    }
    for (long j = 0; j < k; ++j)
        for (long c = 0; c < k; ++c) sk[j * k + c] = sk0[j * k + (exact_pow ? k - 1 - c : c)];
    // w[c][j][t] = digit j of coefficient t of -a_c mod q
    std::vector<int32_t> w((size_t)2 * k * n);
    for (long c = 0; c < 2; ++c)
        for (long t = 0; t < n; ++t) {
            uint64_t v = (q - (uint64_t)ctx->hAring[(size_t)c * n + t]) % q;
            for (long j = 0; j < k; ++j) { w[((size_t)c * k + j) * n + t] = (int32_t)(v % base); v /= base; }
        }
    Dev dE, dR, dW, dSk, dP, dQ;
    CK(dE.ensure((size_t)k * n * 4)); CK(dR.ensure((size_t)k * n * 4)); CK(dW.ensure(w.size() * 4)); CK(dSk.ensure(sk.size() * 8));
    CK(dP.ensure((size_t)4 * n * 8)); CK(dQ.ensure((size_t)2 * k * n * 8));
    CK(cudaMemcpyAsync(dE.p, e, (size_t)k * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dR.p, r, (size_t)k * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dW.p, w.data(), w.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dSk.p, sk.data(), sk.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(qf_launch_ring_basis_polys(dE.as<int32_t>(), dR.as<int32_t>(), dW.as<int32_t>(), dSk.as<int64_t>(), (int)n, (int)k,
                                      dP.as<int64_t>(), dQ.as<int64_t>(), ctx->stream));
    std::vector<int64_t> P((size_t)4 * n), Q((size_t)2 * k * n);
    CK(cudaMemcpyAsync(P.data(), dP.p, P.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(Q.data(), dQ.p, Q.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // placement: entry (t, i) of rot^-(p) = coefficient t of p X^i = p[t - i] (t >= i) or -p[n + t - i]
    auto rot = [&](const int64_t* p, long t, long i) -> int64_t { return t >= i ? p[t - i] : -p[n + t - i]; };
    std::fill(s_out, s_out + (size_t)D * D, (int64_t)0);
    for (long i = 0; i < n; ++i) {
        for (long c = 0; c < k; ++c) {
            const long col = i * k + c;
            const int64_t* qe = &Q[((size_t)c * 2 + 0) * n];
            const int64_t* qr = &Q[((size_t)c * 2 + 1) * n];
            for (long t = 0; t < n; ++t) {
                s_out[(size_t)t * D + col] = rot(qe, t, i);
                s_out[(size_t)(n + t) * D + col] = rot(qr, t, i);
            }
            for (long j = 0; j < k; ++j)
                if (sk[j * k + c]) s_out[(size_t)((2 + j) * n + i) * D + col] = sk[j * k + c];
        }
        for (long c = 0; c < 2; ++c) {
            const long col = n * k + 2 * i + c;
            const int64_t* pe = &P[((size_t)c * 2 + 0) * n];
            const int64_t* pr = &P[((size_t)c * 2 + 1) * n];
            for (long t = 0; t < n; ++t) {
                s_out[(size_t)t * D + col] = rot(pe, t, i) + ((c == 0 && t == i) ? 1 : 0);
                s_out[(size_t)(n + t) * D + col] = rot(pr, t, i) + ((c == 1 && t == i) ? 1 : 0);
            }
            std::vector<int64_t> wp(n);
            for (long j = 0; j < k; ++j) {
                for (long t = 0; t < n; ++t) wp[t] = w[((size_t)c * k + j) * n + t];
                for (long t = 0; t < n; ++t) s_out[(size_t)((2 + j) * n + t) * D + col] = rot(wp.data(), t, i);
            }
        }
    }
    return QF_OK;
}

// gen_short_basis_for_trapdoor (short_basis_classical.rs:54-110) for the installed A and the tag H (NULL: identity):
// W = digits of -H^-1 A[:, :m_bar] mod q, with H^-1 (qf_launch_mat_inverse_mod) and the product (tcgen05) on the device
qf_status qf_gen_short_basis_tagged(qf_ctx* ctx, const int8_t* r, const int64_t* tag, int64_t* s_out) {
    if (!ctx || !r || !s_out) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "ring context: the ring short basis is built by the host shim");
    if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "install A first (qf_set_a / qf_trap_gen)");
    if (!ctx->use_i8) return ctx->fail(QF_ERR_UNSUPPORTED, "needs the int8 tensor path");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, k = ctx->k, mb = ctx->m_bar, nk = ctx->nk, m = ctx->m;
    const uint64_t q = ctx->prm.q, base = (uint64_t)ctx->prm.base;
    if (base > 256) return ctx->fail(QF_ERR_UNSUPPORTED, "gadget base > 256");
    // S_k (gadget_classical.rs:248-272) and whether base^k == q (then S' = S with its columns reversed, :80-82)
    u128 pw = 1;
    for (long i = 0; i < k; ++i) pw *= base;
    if (pw < q) return ctx->fail(QF_ERR_INVALID, "base^k < q");
    const bool exact_pow = pw == (u128)q;
    std::vector<int64_t> sk((size_t)k * k, 0);
    for (long j = 0; j < k; ++j) sk[j * k + j] = (int64_t)base;
    for (long i = 0; i + 1 < k; ++i) sk[(i + 1) * k + i] = -1;
    if (!exact_pow) {
        uint64_t qq = q;
        for (long i = 0; i < k; ++i) { sk[i * k + (k - 1)] = (int64_t)(qq % base); qq /= base; }
    }
    // column c of S' = column (exact_pow ? nk-1-c : c) of I_n (x) S_k
    auto sprime = [&](long row, long c) -> int64_t {
        const long cc = exact_pow ? nk - 1 - c : c;
        return (row / k == cc / k) ? sk[(row % k) * k + (cc % k)] : 0;
    };
    std::fill(s_out, s_out + (size_t)m * m, (int64_t)0);
    // bottom-left S', top-left R S' (each column of S' has at most k non-zeros, all inside one k-block)
    for (long c = 0; c < nk; ++c) {
        const long cc = exact_pow ? nk - 1 - c : c, blk = cc / k;
        for (long t = 0; t < k; ++t) {
            const long row = blk * k + t;
            const int64_t v = sprime(row, c);
            if (!v) continue;
            s_out[(size_t)(mb + row) * m + c] = v;
            for (long i = 0; i < mb; ++i) s_out[(size_t)i * m + c] += (int64_t)r[i * nk + row] * v;
        }
    }
    // A_bar' = H^-1 A[:, :m_bar] mod q (short_basis_classical.rs:106-107), transposed; the tag as MatZq: entries reduced mod q
    std::vector<int64_t> abt;
    if (tag) {
        std::vector<uint64_t> h((size_t)n * n);
        for (long i = 0; i < n * n; ++i) {
            const int64_t v = tag[i] % (int64_t)q;
            h[i] = (uint64_t)(v < 0 ? v + (int64_t)q : v);
        }
        std::vector<int64_t> hinv;
        bool ok = false;
        QF_TRY(tag_inverse(ctx, h.data(), hinv, &ok));
        if (!ok) return ctx->fail(QF_ERR_INVALID, "tag is not invertible mod q (no unit pivot)");
        Dev dHl;
        QF_TRY(tag_planes(ctx, hinv, dHl));
        QF_TRY(tag_abar(ctx, dHl, abt));
    }
    // W = base-b digits of -A_bar' mod q (short_basis_classical.rs:105-110), stored transposed for the device:
    // Wt[c][j k + t] = digit t of (q - A_bar'[j][c]) mod q
    std::vector<int64_t> wt((size_t)mb * nk);
    for (long j = 0; j < n; ++j)
        for (long c = 0; c < mb; ++c) {
            uint64_t v = (q - (uint64_t)(tag ? abt[(size_t)c * n + j] : ctx->hA[(size_t)j * m + c])) % q;
            for (long t = 0; t < k; ++t) {
                const int64_t d = (int64_t)(v % base);
                v /= base;
                wt[(size_t)c * nk + j * k + t] = d;
                s_out[(size_t)(mb + j * k + t) * m + nk + c] = d;  // bottom-right W
            }
        }
    // top-right I + R W: R (m_bar x nk, one s8 digit) times W on the tensor cores, exact int32
    {
        const long ldk = ctx->ldk_nk;
        Dev dX, dW, dOut;
        std::vector<int64_t> r64((size_t)mb * nk);
        for (size_t i = 0; i < r64.size(); ++i) r64[i] = r[i];
        QF_TRY(upload_limbs(ctx, r64.data(), mb, nk, ldk, 1, true, dX));
        QF_TRY(upload_limbs(ctx, wt.data(), mb, nk, ldk, 1, false, dW));
        CK(dOut.ensure((size_t)mb * mb * 4));
        I8GemmArgs g{};
        g.x = dX.as<int8_t>(); g.ldx = ldk; g.x_plane = mb * ldk;
        g.w = dW.p; g.ldw = ldk; g.w_plane = mb * ldk;
        g.LX = 1; g.LW = 1; g.w_signed = 0;
        g.B = (int)mb; g.N = (int)mb; g.K = (int)nk;
        g.out_kind = 1; g.sign = 1; g.q = 0; g.out = dOut.p; g.ldout = mb;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
        std::vector<int32_t> rw((size_t)mb * mb);
        CK(cudaMemcpyAsync(rw.data(), dOut.p, rw.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (long i = 0; i < mb; ++i)
            for (long c = 0; c < mb; ++c) s_out[(size_t)i * m + nk + c] = (int64_t)rw[(size_t)i * mb + c] + (i == c ? 1 : 0);
    }
    return check_flag(ctx);
}

qf_status qf_gen_short_basis(qf_ctx* ctx, const int8_t* r, int64_t* s_out) { return qf_gen_short_basis_tagged(ctx, r, nullptr, s_out); }

qf_status qf_compute_sqrt_sigma_2(qf_ctx* ctx, const int8_t* r, const double* sigma, double* out) {
    if (!ctx || !r || !out) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a PSFPerturbation context");
    CK(cudaSetDevice(ctx->device));
    const long mb = ctx->m_bar, nk = ctx->nk, m = ctx->m, ld = ctx->ld_dim, ldmb = pad16(mb);
    const double s = ctx->prm.s, rr = ctx->prm.r, c = (double)(ctx->prm.base * ctx->prm.base + 1);
    Dev dG, dC, dSig, dRf;
    QF_TRY(upload_as_f64(ctx, r, mb, nk, ctx->ld_nk, dRf));
    CK(dG.ensure((size_t)mb * ldmb * 8));
    QF_TRY(gram_r(ctx, dRf.as<double>(), dG.as<double>(), ldmb));
    CK(dC.ensure((size_t)m * ld * 8));
    if (sigma) QF_TRY(upload_as_f64(ctx, sigma, m, m, ld, dSig));
    // Sigma_2 = r^2/(2 pi) (Sigma - (b^2+1) T T^t - I)   (mp_perturbation.rs:116-135)
    LAUNCH(qf_launch_sigma2_assemble(dC.as<double>(), ld, m, 1, dG.as<double>(), ldmb, dRf.as<double>(), ctx->ld_nk, mb,
                                     sigma ? dSig.as<double>() : nullptr, ld, s * s, c, rr * rr / (2.0 * M_PI), ctx->stream));
    dSig.release();
    dG.release();
    QF_TRY(potrf_lower(ctx, dC.as<double>(), ld, m));
    CK(cudaMemcpy2DAsync(out, (size_t)m * 8, dC.p, (size_t)ld * 8, (size_t)m * 8, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

qf_status qf_gso(qf_ctx* ctx, const int64_t* s, double* gso_out) {
    if (!ctx || !s || !gso_out) return QF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const long D = ctx->dim, ld = ctx->ld_dim;
    Dev dS, dG;
    QF_TRY(upload_as_f64(ctx, s, D, D, ld, dS));
    CK(dG.ensure((size_t)D * ld * 8));
    QF_TRY(gso_device(ctx, dS.as<double>(), dG.as<double>()));
    CK(cudaMemcpy2DAsync(gso_out, (size_t)D * 8, dG.p, (size_t)ld * 8, (size_t)D * 8, (size_t)D, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

qf_status qf_set_trapdoor_gpv(qf_ctx* ctx, const int64_t* s, const double* sg) {
    if (!ctx || !s) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a GPV context");
    ctx->has_np = false;  // stays false if anything below fails half-way (pivots / A^-1 / U are overwritten in place)
    ctx->two_phase = false;
    // the tag table is relative to the old (A_bar, R)
    ctx->tag_count = 0; ctx->dTagTab.release(); ctx->dTagH0.release(); ctx->dTagXr.release();
    ctx->drop_pool();
    ctx->u_limbs = 7;
    CK(cudaSetDevice(ctx->device));
    const long D = ctx->dim, ld = ctx->ld_dim;
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    // particular-solution map
    std::vector<int> piv;
    if (ring) {
        if (!ctx->has_ring) return ctx->fail(QF_ERR_NO_KEY, "install the ring key first (qf_ring_set_a)");
        // a_0 must be the constant polynomial 1 (gadget_ring.rs:75): then x = (u, 0, ..., 0) solves a x = u
        if (ctx->hAring[0] != 1) return ctx->fail(QF_ERR_UNSUPPORTED, "ring key: a_0 != 1");
        for (long i = 1; i < ctx->n; ++i)
            if (ctx->hAring[i] != 0) return ctx->fail(QF_ERR_UNSUPPORTED, "ring key: a_0 != 1");
        ctx->npiv = (int)ctx->n;
        ctx->ainv_identity = true;
        for (int i = 0; i < ctx->npiv; ++i) piv.push_back(i);
    } else {
        if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "install A first (qf_set_a)");
        std::vector<int64_t> ainv;
        if (!find_unit_pivots(ctx->hA.data(), ctx->n, ctx->m, ctx->prm.q, piv, ainv))
            return ctx->fail(QF_ERR_UNSUPPORTED, "A has no n columns invertible over Z_q by unit pivoting");
        QF_TRY(upload_ainv(ctx, ainv));
    }
    ctx->ld_piv = pad16(ctx->npiv);
    CK(ctx->dPiv.ensure(piv.size() * sizeof(int)));
    CK(cudaMemcpy(ctx->dPiv.p, piv.data(), piv.size() * sizeof(int), cudaMemcpyHostToDevice));
    // S (row-major, S[t][j] = coordinate t of b_j) as fp64; GSO likewise
    int64_t smax = 0;
    for (long i = 0; i < D * D; ++i) smax = std::max<int64_t>(smax, s[i] < 0 ? -s[i] : s[i]);
    QF_TRY(upload_as_f64(ctx, s, D, D, ld, ctx->dS));
    Dev dG, dMt, dSt, dD;
    if (sg) {
        QF_TRY(upload_as_f64(ctx, sg, D, D, ld, dG));
    } else {  // GSO not supplied: computed here (gpv.rs:91)
        CK(dG.ensure((size_t)D * ld * 8));
        QF_TRY(gso_device(ctx, ctx->dS.as<double>(), dG.as<double>()));
    }
    CK(dD.ensure((size_t)D * 8));
    CK(dMt.ensure((size_t)D * ld * 8));
    CK(dSt.ensure((size_t)D * ld * 8));
    CK(ctx->dU.ensure((size_t)D * ld * 8));
    CK(ctx->dMtP.ensure((size_t)D * ctx->ld_piv * 8));
    CK(ctx->dDg.ensure((size_t)D * sizeof(DGaussParams)));
    LAUNCH(qf_launch_colnorm2(dG.as<double>(), ld, (int)D, (int)D, dD.as<double>(), ctx->stream));
    LAUNCH(qf_launch_transpose_scale(dG.as<double>(), ld, dMt.as<double>(), ld, (int)D, (int)D, dD.as<double>(), ctx->stream));
    LAUNCH(qf_launch_transpose_scale(ctx->dS.as<double>(), ld, dSt.as<double>(), ld, (int)D, (int)D, nullptr, ctx->stream));
    LAUNCH(ctx_gemm(ctx, dMt.as<double>(), ld, dSt.as<double>(), ld, ctx->dU.as<double>(), ld, (int)D, (int)D, (int)D,
                              1.0, 0.0, 0));
    LAUNCH(qf_launch_gather_cols(dMt.as<double>(), ld, ctx->dPiv.as<int>(), ctx->npiv, ctx->dMtP.as<double>(), ctx->ld_piv,
                                 (int)D, ctx->stream));
    LAUNCH(qf_launch_make_dg(dD.as<double>(), (int)D, ctx->prm.s, ctx->dDg.as<DGaussParams>(), ctx->stream));
    std::vector<double> hd(D);
    CK(cudaMemcpyAsync(hd.data(), dD.p, (size_t)D * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    double dmin = hd[0], dmax = hd[0];
    for (long i = 0; i < D; ++i) {
        if (!(hd[i] > 0)) return ctx->fail(QF_ERR_INVALID, "GSO has a zero / non-finite column");
        dmin = std::min(dmin, hd[i]);
        dmax = std::max(dmax, hd[i]);
    }
    if (ctx->prm.s / std::sqrt(dmin) > 2.0e6)
        return ctx->fail(QF_ERR_UNSUPPORTED, "s / min||b~_i|| exceeds the fp32 range of the integer sampler");
    // exact e = sol + S z : z digits of z_bits bits
    int zb = exact_bits(std::sqrt((double)D) * 0.5, D) - bitlen_u64((unsigned long long)smax) ;
    // (||z_c|| <= 2^(zb-1) sqrt(D); rows of S bounded entrywise by smax)
    zb = std::min(zb, 40);
    if (zb < 4) return ctx->fail(QF_ERR_UNSUPPORTED, "basis entries too large for the exact S*z product");
    const double z_est = 8.0 * ((double)ctx->prm.q * std::sqrt((double)ctx->npiv) + 8.0 * ctx->prm.s) / std::sqrt(dmin);
    int nch = 1;
    while (nch < 4 && z_est >= std::ldexp(1.0, nch * zb - 1)) ++nch;
    ctx->z_bits = zb; ctx->z_nchunks = nch;
    ctx->zlimit = std::min(std::ldexp(1.0, nch * zb - 1), std::ldexp(1.0, 52));
    ctx->s_limbs = limbs_for((double)smax);
    ctx->z_limbs = limbs_for(z_est);
    if (ctx->use_i8) {
        if (ctx->z_limbs + ctx->s_limbs - 1 > 16) return ctx->fail(QF_ERR_UNSUPPORTED, "too many digits for the int8 S*z product");
        ctx->zlimit = std::min(ctx->zlimit, limb_capacity(ctx->z_limbs));
        const char* env = getenv("QF_DISABLE_OZAKI");
        const char* envmin = getenv("QF_OZAKI_MIN_DIM");
        const long min_dim = envmin ? atol(envmin) : 2 * NP_SIZES[2];
        // two-phase recursion (samp_p_np2_chunk): G-trapdoor basis of a key of the form [A_bar | H G - A_bar R], tensor-core
        // dimensions.  z then only has to hold the phase-1 coefficients (widths s/||b~_i||, centres of the same size).
        const char* env2 = getenv("QF_DISABLE_TWO_PHASE");  // test switch: the one-pass recursion
        const bool two_phase_allowed = D > std::max(min_dim, NP_SIZES[2]) && !(env && env[0] == '1') && !(env2 && env2[0] == '1');
        // the tag of a tagged key is only looked for where two-phase can use it
        QF_TRY(detect_gpv_structure(ctx, s, piv, two_phase_allowed));
        if (ctx->gpv_struct) ctx->dSl.release();
        else QF_TRY(upload_limbs(ctx, s, D, D, ctx->ldk_dim, ctx->s_limbs, true, ctx->dSl));
        ctx->two_phase = ctx->gpv_struct && ctx->gadget_key_ok && two_phase_allowed;
        if (ctx->two_phase) {
            // the gadget digits g3 reach base - 1: one more digit of M' for bases above 4 (its error scales with |g3|)
            ctx->mt1g_limbs = ctx->prm.base > 4 ? 5 : 4;
            ctx->z_limbs = limbs_for(64.0 * ctx->prm.s / std::sqrt(dmin));
            ctx->zlimit = std::min(std::ldexp(1.0, 52), limb_capacity(ctx->z_limbs));
            if (const char* cfg = getenv("QF_NP2_CFG")) {  // experiments: "u22,dlo,u11,dlo,mt1,dlo[,mt1g]"
                int v[7] = {ctx->u22_limbs, ctx->u22_dlo, ctx->u11_limbs, ctx->u11_dlo, ctx->mt1_limbs, ctx->mt1_dlo, ctx->mt1g_limbs};
                sscanf(cfg, "%d,%d,%d,%d,%d,%d,%d", &v[0], &v[1], &v[2], &v[3], &v[4], &v[5], &v[6]);
                ctx->mt1g_limbs = std::max(1, std::min(7, v[6]));
                auto lim = [&](int x, int lo, int hi) { return std::max(lo, std::min(hi, x)); };
                ctx->u22_limbs = lim(v[0], 1, ctx->u_limbs); ctx->u22_dlo = lim(v[1], 0, ctx->u22_limbs - 1);
                ctx->u11_limbs = lim(v[2], 1, ctx->u_limbs); ctx->u11_dlo = lim(v[3], 0, ctx->u11_limbs - 1);
                ctx->mt1_limbs = lim(v[4], 1, 7); ctx->mt1_dlo = lim(v[5], 0, ctx->mt1_limbs - 1);
            }
            ctx->u_limbs = std::max(ctx->u22_limbs, ctx->u11_limbs);  // digit planes of U that are built and kept
        }
        ctx->use_ozaki = D > std::max(min_dim, NP_SIZES[2]) && ctx->z_limbs + ctx->u_limbs - 1 <= 16 && !(env && env[0] == '1');
        if (ctx->two_phase && !ctx->use_ozaki) return ctx->fail(QF_ERR_NUMERIC, "internal: two-phase recursion without the tensor-core updates");
        if (ctx->use_ozaki) {
            const long nblk = (D + NP_SCALE_BLOCK - 1) / NP_SCALE_BLOCK;
            CK(ctx->dUscale.ensure((size_t)nblk * D * 8));
            CK(ctx->dUl.ensure((size_t)ctx->u_limbs * D * ctx->ldk_dim));
            CK(cudaMemsetAsync(ctx->dUl.p, 0, (size_t)ctx->u_limbs * D * ctx->ldk_dim, ctx->stream));
            // digitised: every U[i][j] whose row lies in an earlier 256-block than its column (what the 256-, 1024- and
            // 4096-level updates read)
            LAUNCH(qf_launch_ozaki_prepare(ctx->dU.as<double>(), ld, (int)D, (int)NP_SIZES[1], (int)NP_SCALE_BLOCK,
                                           (int)np_last_block_start(D, NP_SIZES[1]), (int)np_last_block_start(D, NP_SCALE_BLOCK),
                                           ctx->u_limbs,
                                           ctx->dUscale.as<double>(), ctx->dUl.as<int8_t>(), D * ctx->ldk_dim, ctx->ldk_dim,
                                           ctx->stream, ctx->two_phase ? (int)ctx->nk : 0));
            CK(cudaStreamSynchronize(ctx->stream));
            if (ctx->two_phase) {
                const long nk = ctx->nk, mb = ctx->m_bar, k = ctx->k;
                // Mt_1 = rows [0, nk) x columns [0, m_bar) of D^-1 B~^t as fixed-point digit planes, one scale per row
                {
                    const long ldk = ctx->ldk_mb;
                    const size_t pb = (size_t)ctx->mt1_limbs * nk * ldk;
                    CK(ctx->dMt1l.ensure(pb));
                    CK(ctx->dMt1scale.ensure((size_t)nk * 8));
                    CK(cudaMemsetAsync(ctx->dMt1l.p, 0, pb, ctx->stream));
                    LAUNCH(qf_launch_fixed_rows_prepare(dMt.as<double>(), ld, (int)nk, (int)mb, ctx->mt1_limbs, 1.0,
                                                        ctx->dMt1scale.as<double>(), ctx->dMt1l.as<int8_t>(), nk * ldk, ldk,
                                                        ctx->stream));
                }
                // M' = U_11 S'^-1 (nk x nk): S_k^-1 by Gauss-Jordan on the host (k <= 64), the product on the device
                {
                    std::vector<double> a((size_t)k * 2 * k, 0.0), ski((size_t)k * k);
                    const uint64_t base = (uint64_t)ctx->prm.base, q = ctx->prm.q;
                    u128 pw = 1;
                    for (long i = 0; i < k; ++i) pw *= base;
                    for (long j = 0; j < k; ++j) { a[j * 2 * k + j] = (double)base; a[j * 2 * k + k + j] = 1.0; }
                    for (long i = 0; i + 1 < k; ++i) a[(i + 1) * 2 * k + i] = -1.0;
                    if (pw != (u128)q) {
                        uint64_t qq = q;
                        for (long i = 0; i < k; ++i) { a[i * 2 * k + (k - 1)] = (double)(qq % base); qq /= base; }
                    }
                    for (long c = 0; c < k; ++c) {
                        long pv = c;
                        for (long r = c + 1; r < k; ++r)
                            if (std::fabs(a[r * 2 * k + c]) > std::fabs(a[pv * 2 * k + c])) pv = r;
                        if (!(std::fabs(a[pv * 2 * k + c]) > 0)) return ctx->fail(QF_ERR_NUMERIC, "internal: singular gadget block");
                        if (pv != c)
                            for (long j = 0; j < 2 * k; ++j) std::swap(a[c * 2 * k + j], a[pv * 2 * k + j]);
                        const double inv = 1.0 / a[c * 2 * k + c];
                        for (long j = 0; j < 2 * k; ++j) a[c * 2 * k + j] *= inv;
                        for (long r = 0; r < k; ++r) {
                            if (r == c) continue;
                            const double f = a[r * 2 * k + c];
                            if (f != 0.0)
                                for (long j = 0; j < 2 * k; ++j) a[r * 2 * k + j] -= f * a[c * 2 * k + j];
                        }
                    }
                    for (long i = 0; i < k; ++i)
                        for (long j = 0; j < k; ++j) ski[i * k + j] = a[i * 2 * k + k + j];
                    Dev dSki;
                    CK(dSki.ensure(ski.size() * 8));
                    CK(cudaMemcpyAsync(dSki.p, ski.data(), ski.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
                    double* mp = dSt.as<double>();  // S^t is dead after the U product
                    LAUNCH(qf_launch_gadget_to_gso(ctx->dU.as<double>(), ld, (int)nk, (int)k, ctx->gpv_rev, dSki.as<double>(), mp, ld,
                                                   ctx->stream));
                    const long ldk = ctx->ldk_nk;
                    const size_t pb = (size_t)ctx->mt1g_limbs * nk * ldk;
                    CK(ctx->dMpl.ensure(pb));
                    CK(ctx->dMpscale.ensure((size_t)nk * 8));
                    CK(cudaMemsetAsync(ctx->dMpl.p, 0, pb, ctx->stream));
                    LAUNCH(qf_launch_fixed_rows_prepare(mp, ld, (int)nk, (int)nk, ctx->mt1g_limbs, 1.0, ctx->dMpscale.as<double>(),
                                                        ctx->dMpl.as<int8_t>(), nk * ldk, ldk, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                }
                ctx->dMtP.release();
                ctx->dS.release();  // read only by the one-pass fp64 form: qf_gpv_set_tag then has no copy of S to rewrite
            }
            // Mt_P as fixed-point digit planes (D rows x npiv columns, one scale per row): T = -Mt_P sol_P on tcgen05
            ctx->sol_limbs = limbs_for((double)ctx->prm.q);
            const char* envm = getenv("QF_DISABLE_MTP_I8");  // test switch: fp64 DMMA as before
            ctx->mtp_i8 = !ctx->two_phase && !(envm && envm[0] == '1') && ctx->sol_limbs + ctx->u_limbs - 1 - ctx->np_dlo <= 9;
            if (ctx->mtp_i8) {
                ctx->ldk_piv = (ctx->npiv + 127) / 128 * 128;
                const size_t pb = (size_t)ctx->u_limbs * D * ctx->ldk_piv;
                CK(ctx->dMtPl.ensure(pb));
                CK(ctx->dMtPscale.ensure((size_t)D * 8));
                CK(cudaMemsetAsync(ctx->dMtPl.p, 0, pb, ctx->stream));
                LAUNCH(qf_launch_fixed_rows_prepare(ctx->dMtP.as<double>(), ctx->ld_piv, (int)D, ctx->npiv, ctx->u_limbs, 1.0,
                                                    ctx->dMtPscale.as<double>(), ctx->dMtPl.as<int8_t>(), D * ctx->ldk_piv,
                                                    ctx->ldk_piv, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
            }
        }
    }
    ctx->has_np = true;
    return QF_OK;
}

qf_status qf_ring_set_a(qf_ctx* ctx, const int64_t* a) {
    if (!ctx || !a) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "not a ring context");
    ctx->has_ring = false; ctx->has_np = false;  // a new key invalidates the installed trapdoor
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, np = ctx->k + 2;
    for (long i = 0; i < n * np; ++i)
        if (a[i] < 0 || (uint64_t)a[i] >= ctx->prm.q) return ctx->fail(QF_ERR_INVALID, "ring key coefficient outside [0,q)");
    ctx->hAring.assign(a, a + n * np);
    CK(ctx->dAraw.ensure((size_t)n * np * 8));
    CK(cudaMemcpy(ctx->dAraw.p, a, (size_t)n * np * 8, cudaMemcpyHostToDevice));
    {
        // word-size NTT-friendly prime (3329, 7681, 12289 ...): transform directly mod q
        std::vector<uint32_t> tables;
        int d = 1;
        uint32_t np_inv = 0;
        const char* env = getenv("QF_DISABLE_SMALL_NTT");
        ctx->ring_small = !(env && env[0] == '1') && qf_ring_small_plan(ctx->prm.q, (int)n, &d, &tables, &np_inv) != 0;
        if (ctx->ring_small) {
            ctx->ring_d = d;
            ctx->ring_np_inv = np_inv;
            std::vector<uint32_t> ah((size_t)n * np);
            qf_ring_small_key(a, (int)np, (int)n, d, ctx->prm.q, tables.data(), ah.data());
            CK(ctx->dTw32.ensure(tables.size() * 4));
            CK(cudaMemcpy(ctx->dTw32.p, tables.data(), tables.size() * 4, cudaMemcpyHostToDevice));
            CK(ctx->dAhat32.ensure(ah.size() * 4));
            CK(cudaMemcpy(ctx->dAhat32.p, ah.data(), ah.size() * 4, cudaMemcpyHostToDevice));
        }
    }
    {
        // rot^-(a_j): column c holds the coefficients of a_j X^c mod X^n + 1 (rotation_matrix.rs:41-63):
        // M[i][j n + c] = a_j[i - c] for i >= c, -a_j[n + i - c] below, reduced into [0, q)
        const char* env = getenv("QF_DISABLE_RING_DENSE");
        const int qbits = bitlen_u64(ctx->prm.q - 1);
        ctx->ring_dense = ctx->use_i8 && ctx->fused_fa && !(env && env[0] == '1') && n >= 16 && n <= 512 && qbits <= 32;
        if (ctx->ring_dense) {
            std::vector<int64_t> rot((size_t)n * n * np);
            const int64_t q = (int64_t)ctx->prm.q;
            for (long j = 0; j < np; ++j)
                for (long c = 0; c < n; ++c)
                    for (long i = 0; i < n; ++i) {
                        const int64_t v = i >= c ? a[j * n + (i - c)] : (q - a[j * n + (n + i - c)]) % q;
                        rot[(size_t)i * (n * np) + j * n + c] = v;
                    }
            ctx->ring_limbs = (qbits + 7) / 8;
            QF_TRY(upload_limbs(ctx, rot.data(), n, n * np, ctx->ldk_dim, ctx->ring_limbs, false, ctx->dRotl));
        }
    }
    ctx->ring_ntt = (n >= 64) && ((n & (n - 1)) == 0) && n <= 2048;
    if (ctx->ring_ntt) {
        // exactness of the integer product: npoly * n * (q/2) * max|sigma| < 2^63
        double mag = (double)np * (double)n * ((double)ctx->prm.q / 2) * std::sqrt((double)ctx->bound);
        if (mag >= 9.0e18) ctx->ring_ntt = false;
    }
    if (ctx->ring_ntt) {
        std::vector<uint64_t> tw(2 * n + 1);
        qf_ring_make_tables((int)n, tw.data());
        CK(ctx->dTw.ensure(tw.size() * 8));
        CK(cudaMemcpy(ctx->dTw.p, tw.data(), tw.size() * 8, cudaMemcpyHostToDevice));
        CK(ctx->dAhat.ensure((size_t)n * np * 8));
        LAUNCH(qf_launch_ring_prepare(ctx->dAraw.as<int64_t>(), ctx->dAhat.as<uint64_t>(), (int)np, (int)n, ctx->prm.q,
                                      ctx->dTw.as<uint64_t>(), ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->has_ring = true;
    return QF_OK;
}

qf_status qf_trap_gen_from(qf_ctx* ctx, const int64_t* a_bar, const int8_t* r, const int64_t* tag, int64_t* a_out) {
    if (!ctx || !a_bar || !r || !a_out) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "ring context: use qf_ring_trap_gen_from");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, mb = ctx->m_bar, nk = ctx->nk, m = ctx->m, k = ctx->k;
    const uint64_t q = ctx->prm.q;
    {
        // base^k must reach q (find_solution_gadget_vec panics otherwise, gadget_classical.rs:170)
        u128 pw = 1;
        for (long i = 0; i < k && pw < q; ++i) pw *= (uint64_t)ctx->prm.base;
        if (pw < q) return ctx->fail(QF_ERR_INVALID, "base^k < q");
    }
    for (long i = 0; i < n * mb; ++i)
        if (a_bar[i] < 0 || (uint64_t)a_bar[i] >= q) return ctx->fail(QF_ERR_INVALID, "A_bar entry outside [0,q)");
    // (A_bar R)^t = R^t A_bar^t : "targets" are the nk columns of R, key matrix is A_bar (n x m_bar)
    const long ldmb = pad16(mb), ldn = ctx->ld_n;
    int rmax = 1;
    for (long i = 0; i < mb * nk; ++i) rmax = std::max(rmax, (int)std::abs((int)r[i]));
    const int qbits = bitlen_u64(q - 1);
    int wb = exact_bits((double)rmax * std::sqrt((double)mb), mb);
    if (wb < 4) return ctx->fail(QF_ERR_UNSUPPORTED, "R too large for the exact A_bar*R product");
    wb = std::min(wb, qbits);
    int nch = (qbits + wb - 1) / wb;
    if (nch > 4) return ctx->fail(QF_ERR_UNSUPPORTED, "modulus needs more than 4 digit matrices (TrapGen)");
    Dev dW[4], dX, dAcc[4], dOut, dWl, dXl;
    CK(dOut.ensure((size_t)nk * n * 8));
    if (ctx->use_i8 && rmax <= 127) {
        // tcgen05 path: "targets" = the nk columns of R (one s8 digit), key matrix = A_bar in u8 digits
        const long ldk = (mb + 127) / 128 * 128;
        const int LA = (qbits + 7) / 8;
        QF_TRY(upload_limbs(ctx, a_bar, n, mb, ldk, LA, false, dWl));
        std::vector<int64_t> rt((size_t)nk * mb);
        for (long i = 0; i < mb; ++i)
            for (long j = 0; j < nk; ++j) rt[(size_t)j * mb + i] = r[i * nk + j];
        QF_TRY(upload_limbs(ctx, rt.data(), nk, mb, ldk, 1, true, dXl));
        I8GemmArgs g{};
        g.x = dXl.as<int8_t>(); g.ldx = ldk; g.x_plane = nk * ldk;
        g.w = dWl.p; g.ldw = ldk; g.w_plane = n * ldk;
        g.LX = 1; g.LW = LA; g.w_signed = 0;
        g.B = (int)nk; g.N = (int)n; g.K = (int)mb;
        g.out_kind = 0; g.sign = 1; g.q = q; g.base = nullptr; g.ldbase = 0; g.out = dOut.p; g.ldout = n;
        g.flag = ctx->dFlag.as<int>();
        LAUNCH(ctx_gemm_i8(ctx, g));
    } else {
        QF_TRY(upload_chunks(ctx, a_bar, n, mb, ldmb, nch, wb, dW));
        {
            std::vector<double> rt((size_t)nk * ldmb, 0.0);
            for (long i = 0; i < mb; ++i)
                for (long j = 0; j < nk; ++j) rt[(size_t)j * ldmb + i] = (double)r[i * nk + j];
            CK(dX.ensure(rt.size() * 8));
            CK(cudaMemcpy(dX.p, rt.data(), rt.size() * 8, cudaMemcpyHostToDevice));
        }
        double* acc[4] = {nullptr, nullptr, nullptr, nullptr};
        CombineArgs ca{};
        for (int c = 0; c < nch; ++c) {
            CK(dAcc[c].ensure((size_t)nk * ldn * 8));
            acc[c] = dAcc[c].as<double>();
            ca.acc[c] = acc[c];
            ca.shift[c] = c * wb;
        }
        QF_TRY(gemm_chunks(ctx, dX.as<double>(), ldmb, dW, nch, ldmb, acc, ldn, (int)nk, (int)n, (int)mb));
        ca.nacc = nch; ca.acc_sign = 1; ca.ldacc = ldn; ca.base = nullptr; ca.ldbase = 0; ca.q = q;
        LAUNCH(qf_launch_combine_i64(ca, dOut.as<int64_t>(), n, (int)nk, (int)n, ctx->stream));
    }
    std::vector<int64_t> art((size_t)nk * n);
    CK(cudaMemcpyAsync(art.data(), dOut.p, art.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // A = [A_bar | tag*G - A_bar R]
    std::vector<uint64_t> gpow(k);
    {
        u128 pw = 1;
        for (long t = 0; t < k; ++t) { gpow[t] = (uint64_t)(pw % q); pw = pw * (uint64_t)ctx->prm.base; }
    }
    for (long i = 0; i < n; ++i) {
        for (long j = 0; j < mb; ++j) a_out[i * m + j] = a_bar[i * mb + j];
        for (long j = 0; j < nk; ++j) {
            long blk = j / k, t = j % k;
            uint64_t h = tag ? ((uint64_t)tag[i * n + blk] % q) : (i == blk ? 1 : 0);
            uint64_t hg = mulmod_h(h, gpow[t], q);
            uint64_t ar = (uint64_t)art[(size_t)j * n + i];
            a_out[i * m + mb + j] = (int64_t)((hg + q - ar) % q);
        }
    }
    return install_a(ctx, a_out);
}

qf_status qf_trap_gen(qf_ctx* ctx, uint64_t seed, int64_t* a_out, int8_t* r_out) {
    if (!ctx || !a_out || !r_out) return QF_ERR_INVALID;
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "ring context");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, mb = ctx->m_bar, nk = ctx->nk;
    Dev dAb, dR;
    CK(dAb.ensure((size_t)n * mb * 8));
    CK(dR.ensure((size_t)mb * nk));
    LAUNCH(qf_launch_uniform_modq(dAb.as<int64_t>(), n * mb, ctx->prm.q, seed, 0, ctx->stream));
    LAUNCH(qf_launch_ternary(dR.as<int8_t>(), mb * nk, seed, ctx->stream));
    std::vector<int64_t> ab((size_t)n * mb);
    CK(cudaMemcpyAsync(ab.data(), dAb.p, ab.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(r_out, dR.p, (size_t)mb * nk, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return qf_trap_gen_from(ctx, ab.data(), r_out, nullptr, a_out);
}

qf_status qf_ring_trap_gen_from(qf_ctx* ctx, const int64_t* a_bar, const int32_t* r, const int32_t* e, int64_t* a_out) {
    if (!ctx || !a_bar || !r || !e || !a_out) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "not a ring context");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, k = ctx->k;
    const uint64_t q = ctx->prm.q;
    // a_bar * r_j for j < k : the ring kernel with a one-polynomial "key" a_bar and k "targets" r_j
    Dev dA, dAh, dTw, dR, dOut;
    CK(dA.ensure((size_t)n * 8));
    CK(cudaMemcpy(dA.p, a_bar, (size_t)n * 8, cudaMemcpyHostToDevice));
    CK(dR.ensure((size_t)k * n * 4));
    CK(cudaMemcpy(dR.p, r, (size_t)k * n * 4, cudaMemcpyHostToDevice));
    CK(dOut.ensure((size_t)k * n * 8));
    int rmax = 1;
    for (long i = 0; i < k * n; ++i) rmax = std::max(rmax, std::abs(r[i]));
    bool ntt = (n >= 64) && ((n & (n - 1)) == 0) && n <= 2048 && ((double)n * ((double)q / 2) * rmax < 9.0e18);
    if (ntt) {
        std::vector<uint64_t> tw(2 * n + 1);
        qf_ring_make_tables((int)n, tw.data());
        CK(dTw.ensure(tw.size() * 8));
        CK(cudaMemcpy(dTw.p, tw.data(), tw.size() * 8, cudaMemcpyHostToDevice));
        CK(dAh.ensure((size_t)n * 8));
        LAUNCH(qf_launch_ring_prepare(dA.as<int64_t>(), dAh.as<uint64_t>(), 1, (int)n, q, dTw.as<uint64_t>(), ctx->stream));
        LAUNCH(qf_launch_ring_f_a(dR.as<int32_t>(), dAh.as<uint64_t>(), dOut.as<int64_t>(), nullptr, (int)k, 1, (int)n, q,
                                  dTw.as<uint64_t>(), ctx->stream));
    } else {
        LAUNCH(qf_launch_ring_f_a_schoolbook(dR.as<int32_t>(), dA.as<int64_t>(), dOut.as<int64_t>(), nullptr, (int)k, 1,
                                             (int)n, q, ctx->stream));
    }
    std::vector<int64_t> ar((size_t)k * n);
    CK(cudaMemcpyAsync(ar.data(), dOut.p, ar.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // A = [1 | a_bar | g^t - (a_bar r + e)]   (gadget_ring.rs:74-78)
    for (long t = 0; t < n; ++t) {
        a_out[t] = (t == 0) ? (int64_t)(1 % q) : 0;
        a_out[n + t] = (int64_t)((uint64_t)a_bar[t] % q);
    }
    u128 pw = 1;
    for (long j = 0; j < k; ++j) {
        for (long t = 0; t < n; ++t) {
            i128 v = -(i128)ar[j * n + t] - (i128)e[j * n + t];
            if (t == 0) v += (i128)(uint64_t)(pw % q);
            i128 mm = v % (i128)q;
            if (mm < 0) mm += q;
            a_out[(2 + j) * n + t] = (int64_t)mm;
        }
        pw = (pw * (uint64_t)ctx->prm.base) % q;
    }
    return qf_ring_set_a(ctx, a_out);
}

// ---- f_a / check_domain ------------------------------------------------------
qf_status qf_f_a_dev(qf_ctx* ctx, const int32_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !in_domain))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;  // an empty batch is valid and does nothing
    CK(cudaSetDevice(ctx->device));
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    if (ring ? !ctx->has_ring : !ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    auto run = [&](int64_t b0, int Bc) {
        const int32_t* s = sigma + b0 * ctx->dim;
        int64_t* u = u_out ? u_out + b0 * ctx->n : nullptr;
        uint8_t* f = in_domain ? in_domain + b0 : nullptr;
        return ring ? ring_f_a_chunk(ctx, s, Bc, u, f) : f_a_chunk(ctx, s, Bc, u, f);
    };
    return f_a_dev_chunks(ctx, batch, run);
}

qf_status qf_f_a(qf_ctx* ctx, const int32_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !u_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    if (ring ? !ctx->has_ring : !ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_c.ensure((size_t)C));
    std::vector<uint8_t> flags((size_t)std::max<int64_t>(batch, 1));
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_a.p, sigma + b0 * ctx->dim, (size_t)Bc * ctx->dim * 4, cudaMemcpyHostToDevice, ctx->stream));
        QF_TRY(ring ? ring_f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, ctx->io_b.as<int64_t>(), ctx->io_c.as<uint8_t>())
                    : f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, ctx->io_b.as<int64_t>(), ctx->io_c.as<uint8_t>()));
        CK(cudaMemcpyAsync(u_out + b0 * ctx->n, ctx->io_b.p, (size_t)Bc * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(flags.data() + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    bool all = true;
    for (int64_t b = 0; b < batch; ++b) all = all && flags[b];
    if (in_domain && batch) memcpy(in_domain, flags.data(), (size_t)batch);
    if (!all) return ctx->fail(QF_ERR_NOT_IN_DOMAIN, "f_a: sigma not in the domain D_n (check_domain failed)");
    return QF_OK;
}

qf_status qf_check_domain(qf_ctx* ctx, const int32_t* sigma, int64_t batch, uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !in_domain))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_c.ensure((size_t)C));
    CK(ctx->w[0].ensure((size_t)C * ctx->ld_dim * 8));
    CK(ctx->dNorm.ensure((size_t)C * 8));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_a.p, sigma + b0 * ctx->dim, (size_t)Bc * ctx->dim * 4, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_i32_to_f64(ctx->io_a.as<int32_t>(), ctx->dim, ctx->w[0].as<double>(), ctx->ld_dim, Bc, (int)ctx->dim,
                                    ctx->dNorm.as<unsigned long long>(), ctx->stream));
        LAUNCH(qf_launch_domain_flags(ctx->dNorm.as<unsigned long long>(), ctx->bound, ctx->io_c.as<uint8_t>(), Bc, ctx->stream));
        CK(cudaMemcpyAsync(in_domain + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    });
}

// ---- f_a with a tag per target (installed f_a tag table) ------------------------------------------------------------
// host tag indices of a batch against a table of ntags tags, checked before any launch
static qf_status check_tag_idx(qf_ctx* ctx, const int32_t* tag_idx, int64_t batch, int64_t ntags, const char* table) {
    for (int64_t b = 0; b < batch; ++b)
        if (tag_idx[b] < 0 || tag_idx[b] >= ntags) {
            char buf[128];
            snprintf(buf, sizeof buf, "tag index outside the installed %s (target %lld: %d)", table, (long long)b, (int)tag_idx[b]);
            return ctx->fail(QF_ERR_INVALID, buf);
        }
    return QF_OK;
}

static qf_status f_a_tagged_ready(qf_ctx* ctx) {
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "f_a tag table: not a classical context");
    if (!ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    if (!ctx->fa_tag_count) return ctx->fail(QF_ERR_NO_KEY, "no f_a tag table installed (qf_set_f_a_tags)");
    return QF_OK;
}

qf_status qf_f_a_tagged(qf_ctx* ctx, const int32_t* sigma, const int32_t* tag_idx, int64_t batch, int64_t* u_out,
                        uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !tag_idx || !u_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(f_a_tagged_ready(ctx));
    QF_TRY(check_tag_idx(ctx, tag_idx, batch, ctx->fa_tag_count, "f_a tag table"));
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_c.ensure((size_t)C));
    CK(ctx->io_t[0].ensure((size_t)C * 4));
    std::vector<uint8_t> flags((size_t)batch);
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_a.p, sigma + b0 * ctx->dim, (size_t)Bc * ctx->dim * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->io_t[0].p, tag_idx + b0, (size_t)Bc * 4, cudaMemcpyHostToDevice, ctx->stream));
        QF_TRY(f_a_tagged_chunk(ctx, ctx->io_a.as<int32_t>(), ctx->io_t[0].as<int32_t>(), Bc, ctx->io_b.as<int64_t>(),
                                ctx->io_c.as<uint8_t>()));
        CK(cudaMemcpyAsync(u_out + b0 * ctx->n, ctx->io_b.p, (size_t)Bc * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(flags.data() + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    bool all = true;
    for (int64_t b = 0; b < batch; ++b) all = all && flags[b];
    if (in_domain) memcpy(in_domain, flags.data(), (size_t)batch);
    if (!all) return ctx->fail(QF_ERR_NOT_IN_DOMAIN, "f_a: sigma not in the domain D_n (check_domain failed)");
    return QF_OK;
}

qf_status qf_f_a_tagged_dev(qf_ctx* ctx, const int32_t* sigma, const int32_t* tag_idx, int64_t batch, int64_t* u_out,
                            uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !tag_idx || !u_out || !in_domain))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(f_a_tagged_ready(ctx));
    return f_a_dev_chunks(ctx, batch, [&](int64_t b0, int Bc) {
        return f_a_tagged_chunk(ctx, sigma + b0 * ctx->dim, tag_idx + b0, Bc, u_out + b0 * ctx->n, in_domain + b0);
    });
}

// ---- ring f_a with a key per target (DESIGN 4.13) ---------------------------------------------------------------------
qf_status qf_ring_set_key_table(qf_ctx* ctx, const int64_t* keys, int64_t nkeys) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "ring key table: not a ring context");
    if (!keys || nkeys < 1 || nkeys >= 0x7fffffffLL) return ctx->fail(QF_ERR_INVALID, "ring key table: keys == NULL or nkeys outside [1, 2^31 - 1)");
    CK(cudaSetDevice(ctx->device));
    const long n = ctx->n, np = ctx->k + 2, per = n * np;
    const unsigned long long q = ctx->prm.q;
    for (int64_t t = 0; t < nkeys; ++t) {
        const int64_t* a = keys + t * per;
        bool bad = false;
        for (long i = 0; i < per; ++i) bad |= (uint64_t)a[i] >= q;  // negatives wrap to >= q
        if (bad) {
            char buf[128];
            snprintf(buf, sizeof buf, "ring key table: key %lld has a coefficient outside [0,q)", (long long)t);
            return ctx->fail(QF_ERR_INVALID, buf);
        }
    }
    std::vector<uint32_t> small;
    int d = 1;
    uint32_t np_inv = 0;
    const int family = ring_key_family(q, n, np, std::sqrt((double)ctx->bound), &d, &small, &np_inv);
    const long npolys = (long)nkeys * np;
    if (family == 1 && npolys > 0x7fffffffL) return ctx->fail(QF_ERR_UNSUPPORTED, "ring key table: more than 2^31 - 1 polynomials");
    // the new table is built beside the old one, which stays installed until the build has finished
    Dev tab, tw, stage;
    {
        cudaError_t e = tab.ensure((size_t)npolys * n * (family == 2 ? 4 : 8));
        if (e != cudaSuccess) {
            cudaGetLastError();
            return ctx->fail(QF_ERR_CUDA, std::string("ring key table does not fit in device memory: ") + cudaGetErrorString(e));
        }
    }
    QF_TRY(ring_key_tables(ctx, family, small, tw));
    QF_TRY(ring_key_transform(ctx, keys, npolys, family, d, tw, tab, stage));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->dKeyTab.swap(tab);
    ctx->dKeyTw.swap(tw);
    ctx->key_count = nkeys;
    ctx->key_family = family;
    ctx->key_d = d;
    ctx->key_np_inv = np_inv;
    return QF_OK;
}

static qf_status ring_keyed_ready(qf_ctx* ctx) {
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "ring f_a with a key per target: not a ring context");
    if (!ctx->key_count) return ctx->fail(QF_ERR_NO_KEY, "no ring key table installed (qf_ring_set_key_table)");
    return QF_OK;
}

qf_status qf_ring_f_a_keyed(qf_ctx* ctx, const int32_t* sigma, const int32_t* key_idx, int64_t batch, int64_t* u_out,
                            uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !key_idx || !u_out))) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ring_keyed_ready(ctx);
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(ring_keyed_ready(ctx));
    for (int64_t b = 0; b < batch; ++b)
        if (key_idx[b] < 0 || key_idx[b] >= ctx->key_count) {
            char buf[128];
            snprintf(buf, sizeof buf, "key index outside the installed ring key table (target %lld: %d)", (long long)b,
                     (int)key_idx[b]);
            return ctx->fail(QF_ERR_INVALID, buf);
        }
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_c.ensure((size_t)C));
    CK(ctx->dKeyIdx.ensure((size_t)C * 4));
    std::vector<uint8_t> flags((size_t)batch);
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_a.p, sigma + b0 * ctx->dim, (size_t)Bc * ctx->dim * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->dKeyIdx.p, key_idx + b0, (size_t)Bc * 4, cudaMemcpyHostToDevice, ctx->stream));
        QF_TRY(ring_f_a_keyed_chunk(ctx, ctx->io_a.as<int32_t>(), ctx->dKeyIdx.as<int32_t>(), Bc, ctx->io_b.as<int64_t>(),
                                    ctx->io_c.as<uint8_t>()));
        CK(cudaMemcpyAsync(u_out + b0 * ctx->n, ctx->io_b.p, (size_t)Bc * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(flags.data() + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    bool all = true;
    for (int64_t b = 0; b < batch; ++b) all = all && flags[b];
    if (in_domain) memcpy(in_domain, flags.data(), (size_t)batch);
    if (!all) return ctx->fail(QF_ERR_NOT_IN_DOMAIN, "f_a: sigma not in the domain D_n (check_domain failed)");
    return QF_OK;
}

qf_status qf_ring_f_a_keyed_dev(qf_ctx* ctx, const int32_t* sigma, const int32_t* key_idx, int64_t batch, int64_t* u_out,
                                uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !key_idx || !u_out || !in_domain))) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ring_keyed_ready(ctx);
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(ring_keyed_ready(ctx));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) {
        return ring_f_a_keyed_chunk(ctx, sigma + b0 * ctx->dim, key_idx + b0, Bc, u_out + b0 * ctx->n, in_domain + b0);
    });
}

qf_status qf_ring_trap_gen_batch_from(qf_ctx* ctx, int64_t count, const int64_t* a_bar, const int32_t* r, const int32_t* e,
                                      int64_t* a_out) {
    if (!ctx) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_GPV_RING) return ctx->fail(QF_ERR_INVALID, "not a ring context");
    if (count < 1 || count >= 0x7fffffffLL || !a_bar || !r || !e || !a_out)
        return ctx->fail(QF_ERR_INVALID, "ring TrapGen batch: count outside [1, 2^31 - 1) or a NULL pointer");
    const long n = ctx->n, k = ctx->k;
    const unsigned long long q = ctx->prm.q;
    if ((long long)count * k > 0x7fffffffLL) return ctx->fail(QF_ERR_INVALID, "ring TrapGen batch: count k >= 2^31");
    CK(cudaSetDevice(ctx->device));
    for (int64_t i = 0; i < count * n; ++i)
        if ((uint64_t)a_bar[i] >= q) {
            char buf[128];
            snprintf(buf, sizeof buf, "ring TrapGen batch: a_bar of key %lld has a coefficient outside [0,q)", (long long)(i / n));
            return ctx->fail(QF_ERR_INVALID, buf);
        }
    double rmax = 1;
    for (int64_t i = 0; i < count * k * n; ++i) rmax = std::max(rmax, std::fabs((double)r[i]));
    // a_bar_t r_{t,j}: a keyed ring product with one polynomial per key, B = count k rows, row t k + j -> key t
    std::vector<uint32_t> small;
    int d = 1;
    uint32_t np_inv = 0;
    const int family = ring_key_family(q, n, 1, rmax, &d, &small, &np_inv);
    const int B = (int)(count * k);
    Dev tab, tw, stage, dR, dE, dIdx, dAr, dAbar, dG, dOut;
    CK(tab.ensure((size_t)count * n * (family == 2 ? 4 : 8)));
    QF_TRY(ring_key_tables(ctx, family, small, tw));
    QF_TRY(ring_key_transform(ctx, a_bar, (long)count, family, d, tw, tab, stage));
    CK(dR.ensure((size_t)B * n * 4));
    CK(cudaMemcpyAsync(dR.p, r, (size_t)B * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    {
        std::vector<int32_t> idx((size_t)B);
        for (int b = 0; b < B; ++b) idx[b] = (int32_t)(b / k);
        CK(dIdx.ensure((size_t)B * 4));
        CK(cudaMemcpyAsync(dIdx.p, idx.data(), (size_t)B * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(dAr.ensure((size_t)B * n * 8));
        QF_TRY(ring_keyed_launch(ctx, family, d, np_inv, tw, tab, count, dR.as<int32_t>(), dIdx.as<int32_t>(), B, 1,
                                 dAr.as<int64_t>(), nullptr));
        CK(cudaStreamSynchronize(ctx->stream));  // idx leaves scope
    }
    // A_t = [1 | a_bar_t | g^t - (a_bar_t r_t + e_t)]   (gadget_ring.rs:74-78)
    std::vector<uint64_t> gpow((size_t)k);
    {
        u128 pw = 1;
        for (long j = 0; j < k; ++j) { gpow[j] = (uint64_t)(pw % q); pw = (pw * (uint64_t)ctx->prm.base) % q; }
    }
    CK(dE.ensure((size_t)B * n * 4));
    CK(cudaMemcpyAsync(dE.p, e, (size_t)B * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(dAbar.ensure((size_t)count * n * 8));
    CK(cudaMemcpyAsync(dAbar.p, a_bar, (size_t)count * n * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(dG.ensure((size_t)k * 8));
    CK(cudaMemcpyAsync(dG.p, gpow.data(), (size_t)k * 8, cudaMemcpyHostToDevice, ctx->stream));
    const size_t out_bytes = (size_t)count * (k + 2) * n * 8;
    CK(dOut.ensure(out_bytes));
    LAUNCH(qf_launch_ring_trap_assemble(dAbar.as<int64_t>(), dAr.as<int64_t>(), dE.as<int32_t>(), dG.as<uint64_t>(),
                                        dOut.as<int64_t>(), (long)count, (int)k, (int)n, q, ctx->stream));
    CK(cudaMemcpyAsync(a_out, dOut.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return QF_OK;
}

// ---- samp_d ------------------------------------------------------------------
qf_status qf_samp_d_dev(qf_ctx* ctx, int64_t batch, uint64_t seed, uint64_t first, int32_t* out) {
    if (!ctx || batch < 0 || (batch > 0 && !out)) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        LAUNCH(qf_launch_dgauss(nullptr, 0, nullptr, 0, out + b0 * ctx->dim, ctx->dim, Bc, (int)ctx->dim, ctx->s_samp_d, seed,
                                first + (uint64_t)b0, QF_STREAM_SAMP_D, ctx->dFlag.as<int>(), ctx->stream));
        return QF_OK;
    });
}

qf_status qf_samp_d(qf_ctx* ctx, int64_t batch, uint64_t seed, uint64_t first, int32_t* out) {
    if (!ctx || batch < 0 || (batch > 0 && !out)) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        LAUNCH(qf_launch_dgauss(nullptr, 0, nullptr, 0, ctx->io_a.as<int32_t>(), ctx->dim, Bc, (int)ctx->dim, ctx->s_samp_d,
                                seed, first + (uint64_t)b0, QF_STREAM_SAMP_D, ctx->dFlag.as<int>(), ctx->stream));
        CK(cudaMemcpyAsync(out + b0 * ctx->dim, ctx->io_a.p, (size_t)Bc * ctx->dim * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    });
}

// ---- samp_p ------------------------------------------------------------------
static qf_status samp_p_ready(qf_ctx* ctx) {
    if (ctx->prm.kind == QF_PSF_PERTURBATION) {
        if (!ctx->has_a || !ctx->has_pert) return ctx->fail(QF_ERR_NO_KEY, "PSFPerturbation: key or trapdoor missing");
    } else {
        if (!ctx->has_np) return ctx->fail(QF_ERR_NO_KEY, "GPV: trapdoor missing (qf_set_trapdoor_gpv)");
    }
    return QF_OK;
}

qf_status qf_samp_p_dev(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first, int32_t* e_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !e_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(samp_p_ready(ctx));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        const int64_t* uu = u + b0 * ctx->n;
        int32_t* ee = e_out + b0 * ctx->dim;
        return ctx->prm.kind == QF_PSF_PERTURBATION ? samp_p_pert_chunk(ctx, uu, Bc, seed, first + (uint64_t)b0, ee)
                                                    : samp_p_np_chunk(ctx, uu, Bc, seed, first + (uint64_t)b0, ee);
    });
}

// Output form of the host-buffer samp_p: int32, int16 (half the device->host bytes) or the packed code of DESIGN 4.11
struct SampOut {
    enum Kind { I32, I16, PACKED } kind = I32;
    int k = 0;              // PACKED: code parameter and slot size; nbytes: host, batch lengths
    int64_t slot_bytes = 0;
    int32_t* nbytes = nullptr;
    size_t row_bytes(long dim) const { return kind == I32 ? (size_t)dim * 4 : kind == I16 ? (size_t)dim * 2 : (size_t)slot_bytes; }
};

// host-buffer samp_p in one of the SampOut forms
// tidx (optional, host): tag index of every target in the installed tag table (qf_samp_p_tagged), copied with the targets
// pool_slot0 >= 0: the online half of the pool entries from that slot on (qf_samp_p_online; seed and first unused)
static qf_status samp_p_host(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first, void* e_out,
                             const SampOut& fmt, const int32_t* tidx = nullptr, int64_t pool_slot0 = -1) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !e_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(samp_p_ready(ctx));
    const long C = ctx->chunk;
    const bool i16 = fmt.kind == SampOut::I16, packed = fmt.kind == SampOut::PACKED;
    const size_t esz = fmt.row_bytes(ctx->dim);  // bytes per result row on the host
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    if (tidx) CK(ctx->io_t[0].ensure((size_t)C * 4));
    if (i16) CK(ctx->io_h[0].ensure((size_t)C * ctx->dim * 2));
    if (packed) {
        CK(ctx->io_p[0].ensure((size_t)C * esz));
        CK(ctx->io_n[0].ensure((size_t)C * 4));
    }
    // Both directions of the host traffic run on a second stream: the device->host copy of chunk i and the host->device
    // copy of the targets of chunk i+1 overlap the computation (two result buffers, two target buffers, events in both
    // directions); only the first chunk's targets and the last chunk's results are exposed.
    const bool overlap = batch > C;
    if (overlap) {
        if (i16) CK(ctx->io_h[1].ensure((size_t)C * ctx->dim * 2));
        else if (packed) {
            CK(ctx->io_p[1].ensure((size_t)C * esz));
            CK(ctx->io_n[1].ensure((size_t)C * 4));
        } else CK(ctx->io_a2.ensure((size_t)C * ctx->dim * 4));
        CK(ctx->io_b2.ensure((size_t)C * ctx->n * 8));
        if (tidx) CK(ctx->io_t[1].ensure((size_t)C * 4));
        if (!ctx->copy_stream) {
            CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
            for (int i = 0; i < 2; ++i) {
                CK(cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&ctx->ev_u_in[i], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&ctx->ev_u_used[i], cudaEventDisableTiming));
            }
        }
    }
    // chunk boundaries (the same balanced split as for_chunks)
    const int64_t nch = std::max<int64_t>(1, (batch + C - 1) / C);
    const int64_t per = std::min<int64_t>(C, ((batch + nch - 1) / nch + 127) / 128 * 128);
    auto u_buf = [&](int64_t i) { return (overlap && (i & 1)) ? ctx->io_b2.as<int64_t>() : ctx->io_b.as<int64_t>(); };
    auto t_buf = [&](int64_t i) { return ctx->io_t[(overlap && (i & 1)) ? 1 : 0].as<int32_t>(); };
    auto copy_u = [&](int64_t i, cudaStream_t st) -> qf_status {
        const int64_t b0 = i * per, Bc = std::min<int64_t>(per, batch - b0);
        CK(cudaMemcpyAsync(u_buf(i), u + b0 * ctx->n, (size_t)Bc * ctx->n * 8, cudaMemcpyHostToDevice, st));
        if (tidx) CK(cudaMemcpyAsync(t_buf(i), tidx + b0, (size_t)Bc * 4, cudaMemcpyHostToDevice, st));
        return QF_OK;
    };
    if (overlap) {
        QF_TRY(copy_u(0, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_u_in[0], ctx->copy_stream));
    }
    int64_t idx = 0;
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        const int slot = (int)(idx & 1);
        // int32 results of the chunk: with int16 or packed output they are converted into the slot's own buffer, so one
        // int32 buffer serves both slots
        int32_t* dres = (fmt.kind == SampOut::I32 && overlap && slot) ? ctx->io_a2.as<int32_t>() : ctx->io_a.as<int32_t>();
        if (overlap && idx >= 2) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[slot], 0));  // buffer free again?
        if (overlap) {
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_u_in[slot], 0));  // this chunk's targets have arrived
            if (b0 + Bc < batch) {  // the next chunk's targets, as soon as the computation that read that buffer is done
                if (idx >= 1) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_u_used[slot ^ 1], 0));
                QF_TRY(copy_u(idx + 1, ctx->copy_stream));
                CK(cudaEventRecord(ctx->ev_u_in[slot ^ 1], ctx->copy_stream));
            }
        } else {
            QF_TRY(copy_u(idx, ctx->stream));
        }
        const int64_t* du = u_buf(idx);
        // the targets must be residues in [0, q): checked on the device (a host loop over batch x n values would sit in
        // front of every call), reported by check_flag as QF_ERR_INVALID
        LAUNCH(qf_launch_range_check_i64(du, (size_t)Bc * ctx->n, ctx->prm.q, ctx->dFlag.as<int>(), ctx->stream));
        const int32_t* dt = tidx ? t_buf(idx) : nullptr;
        if (pool_slot0 >= 0) QF_TRY(samp_p_online_chunk(ctx, du, Bc, pool_slot0 + b0, dres, dt));
        else QF_TRY(ctx->prm.kind == QF_PSF_PERTURBATION ? samp_p_pert_chunk(ctx, du, Bc, seed, first + (uint64_t)b0, dres, dt)
                                                         : samp_p_np_chunk(ctx, du, Bc, seed, first + (uint64_t)b0, dres, dt));
        if (overlap) CK(cudaEventRecord(ctx->ev_u_used[slot], ctx->stream));
        const int bs = overlap ? slot : 0;
        const void* src = dres;
        if (i16) {
            int16_t* d16 = ctx->io_h[bs].as<int16_t>();
            LAUNCH(qf_launch_narrow_i32_i16(dres, d16, (size_t)Bc * ctx->dim, ctx->dFlag.as<int>(), ctx->stream));
            src = d16;
        } else if (packed) {
            LAUNCH(qf_launch_domain_encode(dres, Bc, (int)ctx->dim, fmt.k, fmt.slot_bytes, ctx->io_p[bs].as<uint8_t>(),
                                           ctx->io_n[bs].as<int32_t>(), ctx->stream));
            src = ctx->io_p[bs].p;
        }
        char* dst = (char*)e_out + (size_t)b0 * esz;
        cudaStream_t cs = overlap ? ctx->copy_stream : ctx->stream;
        if (overlap) {
            CK(cudaEventRecord(ctx->ev_done[slot], ctx->stream));
            CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done[slot], 0));
        }
        CK(cudaMemcpyAsync(dst, src, (size_t)Bc * esz, cudaMemcpyDeviceToHost, cs));
        if (packed) CK(cudaMemcpyAsync(fmt.nbytes + b0, ctx->io_n[bs].p, (size_t)Bc * 4, cudaMemcpyDeviceToHost, cs));
        if (overlap) CK(cudaEventRecord(ctx->ev_copied[slot], ctx->copy_stream));
        else CK(cudaStreamSynchronize(ctx->stream));
        ++idx;
        return QF_OK;
    }));
    if (overlap) CK(cudaStreamSynchronize(ctx->copy_stream));
    QF_TRY(check_flag(ctx));
    if (packed) {
        for (int64_t b = 0; b < batch; ++b)
            if (fmt.nbytes[b] < 0) {
                char buf[192];
                snprintf(buf, sizeof buf, "packed samp_p: the code of target %lld does not fit its slot of %lld bytes (its row is "
                         "zero, nbytes -1; qf_samp_p at first_index + %lld gives its preimage)", (long long)b,
                         (long long)fmt.slot_bytes, (long long)b);
                return ctx->fail(QF_ERR_NUMERIC, buf);
            }
    }
    return QF_OK;
}

qf_status qf_samp_p(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first, int32_t* e_out) {
    return samp_p_host(ctx, u, batch, seed, first, e_out, SampOut{});
}
qf_status qf_samp_p_i16(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first, int16_t* e_out) {
    SampOut f;
    f.kind = SampOut::I16;
    return samp_p_host(ctx, u, batch, seed, first, e_out, f);
}

// ---- samp_p with a tag per target (PSFPerturbation, PSFGPV on the two-phase recursion; installed tag table) -----------
static qf_status samp_p_tagged_ready(qf_ctx* ctx) {
    if (ctx->prm.kind == QF_PSF_GPV) QF_TRY(gpv_tags_ready(ctx));
    else if (ctx->prm.kind != QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a PSFGPV or PSFPerturbation context");
    QF_TRY(samp_p_ready(ctx));
    if (!ctx->tag_count) return ctx->fail(QF_ERR_NO_KEY, "no tag table installed (qf_set_tag_table)");
    return QF_OK;
}

qf_status qf_samp_p_tagged(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed, uint64_t first,
                           int32_t* e_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !tag_idx || !e_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    QF_TRY(samp_p_tagged_ready(ctx));
    QF_TRY(check_tag_idx(ctx, tag_idx, batch, ctx->tag_count, "tag table"));
    return samp_p_host(ctx, u, batch, seed, first, e_out, SampOut{}, tag_idx);
}

qf_status qf_samp_p_tagged_dev(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed,
                               uint64_t first, int32_t* e_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !tag_idx || !e_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    QF_TRY(samp_p_tagged_ready(ctx));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        const int64_t* uu = u + b0 * ctx->n;
        int32_t* ee = e_out + b0 * ctx->dim;
        return ctx->prm.kind == QF_PSF_PERTURBATION ? samp_p_pert_chunk(ctx, uu, Bc, seed, first + (uint64_t)b0, ee, tag_idx + b0)
                                                    : samp_p_np_chunk(ctx, uu, Bc, seed, first + (uint64_t)b0, ee, tag_idx + b0);
    });
}

// ---- offline / online samp_p (DESIGN 4.12) ---------------------------------------------------------------------------
qf_status qf_samp_p_offline(qf_ctx* ctx, int64_t count, uint64_t seed, uint64_t first) {
    if (!ctx || count < 0) return QF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (ctx->prm.kind == QF_PSF_GPV_RING) return ctx->fail(QF_ERR_UNSUPPORTED, "samp_p pool: not on a ring context");
    QF_TRY(samp_p_ready(ctx));
    if (ctx->prm.kind == QF_PSF_GPV && !ctx->two_phase)
        return ctx->fail(QF_ERR_UNSUPPORTED, "samp_p pool: PSFGPV needs the two-phase recursion (the one-pass form reads the "
                                             "target first)");
    ctx->drop_pool();
    const long xd = pool_xdim(ctx), td = pool_tdim(ctx);
    const size_t per = (size_t)xd * 4 + (size_t)ctx->n * 8 + (size_t)td * 8;
    if ((uint64_t)count > (uint64_t)(SIZE_MAX / 2) / per) return ctx->fail(QF_ERR_INVALID, "samp_p pool: count too large");
    const size_t c = (size_t)std::max<int64_t>(count, 1);
    cudaError_t e = ctx->dPoolX.ensure(c * xd * 4);
    if (e == cudaSuccess) e = ctx->dPoolAx.ensure(c * ctx->n * 8);
    if (e == cudaSuccess && td) e = ctx->dPoolT.ensure(c * td * 8);
    if (e == cudaSuccess && td && ctx->dOnes.cap < (size_t)td * 8) {
        std::vector<double> ones((size_t)td, 1.0);
        e = ctx->dOnes.ensure((size_t)td * 8);
        if (e == cudaSuccess) e = cudaMemcpy(ctx->dOnes.p, ones.data(), (size_t)td * 8, cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        ctx->drop_pool();
        char buf[192];
        snprintf(buf, sizeof buf, "samp_p pool: %lld entries of %zu bytes do not fit in device memory (%s)", (long long)count, per,
                 cudaGetErrorString(e));
        return ctx->fail(QF_ERR_CUDA, buf);
    }
    qf_status st = for_chunks(ctx, count, [&](int64_t b0, int Bc) -> qf_status {
        return samp_p_offline_chunk(ctx, Bc, seed, first + (uint64_t)b0, b0);
    });
    if (st == QF_OK) {
        CK(cudaStreamSynchronize(ctx->stream));
        st = check_flag(ctx);
    }
    if (st != QF_OK) {
        ctx->drop_pool();
        return st;
    }
    ctx->pool = true;
    ctx->pool_count = count;
    ctx->pool_next = 0;
    ctx->pool_seed = seed;
    ctx->pool_first = first;
    return QF_OK;
}

qf_status qf_samp_p_pool_info(const qf_ctx* ctx, int64_t* remaining, uint64_t* next_index) {
    if (!ctx) return QF_ERR_INVALID;
    if (remaining) *remaining = ctx->pool ? ctx->pool_count - ctx->pool_next : 0;
    if (next_index) *next_index = ctx->pool ? ctx->pool_first + (uint64_t)ctx->pool_next : 0;
    return QF_OK;
}

// checks of an online call; on success the call owns slots *slot0 .. *slot0 + batch - 1 (the cursor has moved)
static qf_status samp_p_online_accept(qf_ctx* ctx, const int32_t* tag_idx, int64_t batch, bool host_idx, int64_t* slot0,
                                      uint64_t* first_index_out) {
    CK(cudaSetDevice(ctx->device));
    if (!ctx->pool) return ctx->fail(QF_ERR_NO_KEY, "no samp_p pool installed (qf_samp_p_offline)");
    if (tag_idx) QF_TRY(samp_p_tagged_ready(ctx));
    else QF_TRY(samp_p_ready(ctx));
    if (batch > ctx->pool_count - ctx->pool_next) {
        char buf[160];
        snprintf(buf, sizeof buf, "samp_p pool: batch %lld exceeds the %lld remaining entries", (long long)batch,
                 (long long)(ctx->pool_count - ctx->pool_next));
        return ctx->fail(QF_ERR_INVALID, buf);
    }
    if (tag_idx && host_idx && batch > 0) QF_TRY(check_tag_idx(ctx, tag_idx, batch, ctx->tag_count, "tag table"));
    *slot0 = ctx->pool_next;
    if (first_index_out) *first_index_out = ctx->pool_first + (uint64_t)ctx->pool_next;
    ctx->pool_next += batch;
    return QF_OK;
}

qf_status qf_samp_p_online(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, int32_t* e_out,
                           uint64_t* first_index_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !e_out))) return QF_ERR_INVALID;
    int64_t slot0 = 0;
    QF_TRY(samp_p_online_accept(ctx, tag_idx, batch, true, &slot0, first_index_out));
    if (batch == 0) return QF_OK;
    return samp_p_host(ctx, u, batch, 0, 0, e_out, SampOut{}, tag_idx, slot0);
}

qf_status qf_samp_p_online_dev(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, int32_t* e_out,
                               uint64_t* first_index_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !e_out))) return QF_ERR_INVALID;
    int64_t slot0 = 0;
    QF_TRY(samp_p_online_accept(ctx, tag_idx, batch, false, &slot0, first_index_out));
    return for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        return samp_p_online_chunk(ctx, u + b0 * ctx->n, Bc, slot0 + b0, e_out + b0 * ctx->dim, tag_idx ? tag_idx + b0 : nullptr);
    });
}

// int16 Domain input: widened on the device (the H2D copy, which dominates the host path, is halved)
qf_status qf_f_a_i16(qf_ctx* ctx, const int16_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && (!sigma || !u_out))) return QF_ERR_INVALID;
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    if (ring ? !ctx->has_ring : !ctx->has_a) return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    const long C = ctx->chunk;
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_h[0].ensure((size_t)C * ctx->dim * 2));
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_c.ensure((size_t)C));
    std::vector<uint8_t> flags((size_t)batch);
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_h[0].p, sigma + b0 * ctx->dim, (size_t)Bc * ctx->dim * 2, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_widen_i16_i32(ctx->io_h[0].as<int16_t>(), ctx->io_a.as<int32_t>(), (size_t)Bc * ctx->dim, ctx->stream));
        QF_TRY(ring ? ring_f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, ctx->io_b.as<int64_t>(), ctx->io_c.as<uint8_t>())
                    : f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, ctx->io_b.as<int64_t>(), ctx->io_c.as<uint8_t>()));
        CK(cudaMemcpyAsync(u_out + b0 * ctx->n, ctx->io_b.p, (size_t)Bc * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(flags.data() + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    bool all = true;
    for (int64_t b = 0; b < batch; ++b) all = all && flags[b];
    if (in_domain) memcpy(in_domain, flags.data(), (size_t)batch);
    if (!all) return ctx->fail(QF_ERR_NOT_IN_DOMAIN, "f_a: sigma not in the domain D_n (check_domain failed)");
    return QF_OK;
}

// device utility for the final gather of int32 Domain results in 16 bits: *overflow (device int, caller-zeroed) |= 64
qf_status qf_narrow_i32_i16_dev(const int32_t* in, int16_t* out, size_t count, int* overflow, void* cuda_stream) {
    if ((!in || !out) && count) return QF_ERR_INVALID;
    cudaError_t e = qf_launch_narrow_i32_i16(in, out, count, overflow, (cudaStream_t)cuda_stream);
    return e == cudaSuccess ? QF_OK : (e == cudaErrorMisalignedAddress ? QF_ERR_INVALID : QF_ERR_CUDA);
}

// ---- packed Domain values (DESIGN 4.11) ---------------------------------------------------------------------------
static bool packed_args_ok(int64_t dim, int k, int64_t slot_bytes) {
    return dim > 0 && dim <= INT32_MAX && k >= 0 && k <= 30 && slot_bytes % 16 == 0 &&
           slot_bytes >= qf_domain_h0(dim, k) + (dim + 7) / 8;
}

qf_status qf_domain_code_params(qf_ctx* ctx, int* k, int64_t* slot_bytes) {
    if (!ctx || !k || !slot_bytes) return QF_ERR_INVALID;
    long long sb = 0;
    qf_domain_code_recommend(ctx->s_samp_d, ctx->dim, k, &sb);
    *slot_bytes = sb;
    return QF_OK;
}

qf_status qf_samp_p_packed(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed, uint64_t first,
                           int k, int64_t slot_bytes, uint8_t* out, int32_t* nbytes) {
    if (!ctx || batch < 0 || (batch > 0 && (!u || !out || !nbytes))) return QF_ERR_INVALID;
    if (!packed_args_ok(ctx->dim, k, slot_bytes))
        return ctx->fail(QF_ERR_INVALID, "packed Domain code: k outside [0, 30] or slot_bytes not a multiple of 16 of at least "
                                         "H0 + ceil(dim / 8)");
    if (batch == 0) return QF_OK;
    if (tag_idx) {
        QF_TRY(samp_p_tagged_ready(ctx));
        QF_TRY(check_tag_idx(ctx, tag_idx, batch, ctx->tag_count, "tag table"));
    }
    SampOut f;
    f.kind = SampOut::PACKED;
    f.k = k;
    f.slot_bytes = slot_bytes;
    f.nbytes = nbytes;
    return samp_p_host(ctx, u, batch, seed, first, out, f, tag_idx);
}

qf_status qf_f_a_packed(qf_ctx* ctx, const uint8_t* packed, const int32_t* tag_idx, int64_t batch, int k, int64_t slot_bytes,
                        int64_t* u_out, uint8_t* in_domain) {
    if (!ctx || batch < 0 || (batch > 0 && !packed)) return QF_ERR_INVALID;
    if (!packed_args_ok(ctx->dim, k, slot_bytes))
        return ctx->fail(QF_ERR_INVALID, "packed Domain code: k outside [0, 30] or slot_bytes not a multiple of 16 of at least "
                                         "H0 + ceil(dim / 8)");
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    const bool ring = ctx->prm.kind == QF_PSF_GPV_RING;
    if (tag_idx) {
        QF_TRY(f_a_tagged_ready(ctx));
        QF_TRY(check_tag_idx(ctx, tag_idx, batch, ctx->fa_tag_count, "f_a tag table"));
    } else if (ring ? !ctx->has_ring : !ctx->has_a) {
        return ctx->fail(QF_ERR_NO_KEY, "no key installed");
    }
    const long C = ctx->chunk;
    CK(ctx->io_p[0].ensure((size_t)C * slot_bytes));
    CK(ctx->io_n[0].ensure((size_t)C));
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->io_c.ensure((size_t)C));
    if (u_out) CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    if (tag_idx) CK(ctx->io_t[0].ensure((size_t)C * 4));
    std::vector<uint8_t> flags((size_t)batch), canon((size_t)batch);
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_p[0].p, packed + b0 * slot_bytes, (size_t)Bc * slot_bytes, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_domain_decode(ctx->io_p[0].as<uint8_t>(), Bc, (int)ctx->dim, k, slot_bytes, ctx->io_a.as<int32_t>(),
                                       ctx->io_n[0].as<uint8_t>(), ctx->stream));
        int64_t* du = u_out ? ctx->io_b.as<int64_t>() : nullptr;
        if (tag_idx && u_out) {  // the tag changes u only: flags alone come from the untagged f_a
            CK(cudaMemcpyAsync(ctx->io_t[0].p, tag_idx + b0, (size_t)Bc * 4, cudaMemcpyHostToDevice, ctx->stream));
            QF_TRY(f_a_tagged_chunk(ctx, ctx->io_a.as<int32_t>(), ctx->io_t[0].as<int32_t>(), Bc, du, ctx->io_c.as<uint8_t>()));
        } else {
            QF_TRY(ring ? ring_f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, du, ctx->io_c.as<uint8_t>())
                        : f_a_chunk(ctx, ctx->io_a.as<int32_t>(), Bc, du, ctx->io_c.as<uint8_t>()));
        }
        if (u_out) CK(cudaMemcpyAsync(u_out + b0 * ctx->n, du, (size_t)Bc * ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(flags.data() + b0, ctx->io_c.p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(canon.data() + b0, ctx->io_n[0].p, (size_t)Bc, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    QF_TRY(check_flag(ctx));
    bool all = true;
    for (int64_t b = 0; b < batch; ++b) {
        flags[b] = flags[b] && canon[b];
        all = all && flags[b];
    }
    if (in_domain) memcpy(in_domain, flags.data(), (size_t)batch);
    if (!all) return ctx->fail(QF_ERR_NOT_IN_DOMAIN, "f_a: a packed sigma is not canonical or not in the domain D_n");
    return QF_OK;
}

qf_status qf_domain_encode_dev(const int32_t* in, int64_t rows, int64_t dim, int k, int64_t slot_bytes, uint8_t* out,
                               int32_t* nbytes, void* cuda_stream) {
    if (rows < 0 || !packed_args_ok(dim, k, slot_bytes) || (rows > 0 && (!in || !out || !nbytes))) return QF_ERR_INVALID;
    cudaError_t e = qf_launch_domain_encode(in, rows, (int)dim, k, slot_bytes, out, nbytes, (cudaStream_t)cuda_stream);
    return e == cudaSuccess ? QF_OK : (e == cudaErrorMisalignedAddress ? QF_ERR_INVALID : QF_ERR_CUDA);
}

qf_status qf_domain_decode_dev(const uint8_t* in, int64_t rows, int64_t dim, int k, int64_t slot_bytes, int32_t* out, uint8_t* ok,
                               void* cuda_stream) {
    if (rows < 0 || !packed_args_ok(dim, k, slot_bytes) || (rows > 0 && (!in || !out || !ok))) return QF_ERR_INVALID;
    cudaError_t e = qf_launch_domain_decode(in, rows, (int)dim, k, slot_bytes, out, ok, (cudaStream_t)cuda_stream);
    return e == cudaSuccess ? QF_OK : (e == cudaErrorMisalignedAddress ? QF_ERR_INVALID : QF_ERR_CUDA);
}

// ---- PSFPerturbation::randomized_nearest_plane_gadget (mp_perturbation.rs:173-191) ----------------------------
qf_status qf_randomized_nearest_plane_gadget(qf_ctx* ctx, const int64_t* v, int64_t batch, uint64_t seed, uint64_t first,
                                             int32_t* z_out) {
    if (!ctx || batch < 0 || (batch > 0 && (!v || !z_out))) return QF_ERR_INVALID;
    if (ctx->prm.kind != QF_PSF_PERTURBATION) return ctx->fail(QF_ERR_INVALID, "not a PSFPerturbation context");
    if (!ctx->has_pert) return ctx->fail(QF_ERR_NO_KEY, "PSFPerturbation: trapdoor missing (gadget short basis)");
    if (batch == 0) return QF_OK;
    CK(cudaSetDevice(ctx->device));
    for (int64_t i = 0; i < batch * ctx->n; ++i)
        if (v[i] < 0 || (uint64_t)v[i] >= ctx->prm.q) return ctx->fail(QF_ERR_INVALID, "syndrome entry outside [0,q)");
    const long C = ctx->chunk, ldnk = ctx->ld_nk;
    CK(ctx->io_b.ensure((size_t)C * ctx->n * 8));
    CK(ctx->io_a.ensure((size_t)C * ctx->dim * 4));
    CK(ctx->w[3].ensure((size_t)C * ldnk * 8));
    const double s_g = ctx->prm.r * std::sqrt((double)(ctx->prm.base * ctx->prm.base + 1));
    QF_TRY(for_chunks(ctx, batch, [&](int64_t b0, int Bc) -> qf_status {
        CK(cudaMemcpyAsync(ctx->io_b.p, v + b0 * ctx->n, (size_t)Bc * ctx->n * 8, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(qf_launch_gadget_sample(ctx->io_b.as<int64_t>(), ctx->n, ctx->w[3].as<double>(), ldnk, Bc, (int)ctx->n, (int)ctx->k,
                                       (int)ctx->prm.base, ctx->prm.q, ctx->dSk.as<double>(), ctx->dSkGso.as<double>(), s_g, seed,
                                       first + (uint64_t)b0, ctx->dFlag.as<int>(), ctx->stream));
        LAUNCH(qf_launch_f64_to_i32(ctx->w[3].as<double>(), ldnk, ctx->io_a.as<int32_t>(), ctx->nk, Bc, (int)ctx->nk,
                                    ctx->dFlag.as<int>(), ctx->stream));
        CK(cudaMemcpyAsync(z_out + b0 * ctx->nk, ctx->io_a.p, (size_t)Bc * ctx->nk * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return QF_OK;
    }));
    return check_flag(ctx);
}

// ---- compression -----------------------------------------------------------------
static qf_status compress_any(const void* in, void* out, size_t count, uint64_t q, uint32_t d, int dev, void* stream,
                              int dec, int wide) {
    if ((!in || !out) && count) return QF_ERR_INVALID;
    if (d < 1) return QF_ERR_INVALID;  // reference: assert!(d >= 1), lossy_compression_fips203.rs:91-94
    if (count == 0) return QF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t esz = wide ? 8 : 2;
    auto run = [&](const void* di, void* dout) -> cudaError_t {
        return wide ? qf_launch_compress_i64((const int64_t*)di, (int64_t*)dout, count, q, d, dec, st)
                    : qf_launch_compress_u16((const uint16_t*)di, (uint16_t*)dout, count, (uint32_t)q, d, dec, st);
    };
    if (!wide && (q > 65535 || d > 16)) return QF_ERR_UNSUPPORTED;
    if (wide && (q >= (1ull << 62) || d > 62)) return QF_ERR_UNSUPPORTED;
    if (dev) {
        cudaError_t e = run(in, out);
        return e == cudaSuccess ? QF_OK : (e == cudaErrorInvalidValue ? QF_ERR_INVALID : QF_ERR_CUDA);
    }
    void *di = nullptr, *dout = nullptr;
    if (cudaMalloc(&di, count * esz) != cudaSuccess) return QF_ERR_CUDA;
    if (cudaMalloc(&dout, count * esz) != cudaSuccess) { cudaFree(di); return QF_ERR_CUDA; }
    qf_status rc = QF_OK;
    if (cudaMemcpyAsync(di, in, count * esz, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (rc == QF_OK) {
        cudaError_t e = run(di, dout);
        if (e != cudaSuccess) rc = (e == cudaErrorInvalidValue ? QF_ERR_INVALID : QF_ERR_CUDA);
    }
    if (rc == QF_OK && cudaMemcpyAsync(out, dout, count * esz, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == QF_OK) rc = QF_ERR_CUDA;
    cudaFree(di);
    cudaFree(dout);
    return rc;
}

qf_status qf_compress_u16(const uint16_t* in, uint16_t* out, size_t count, uint32_t q, uint32_t d, int dev, void* st) {
    return compress_any(in, out, count, q, d, dev, st, 0, 0);
}
qf_status qf_decompress_u16(const uint16_t* in, uint16_t* out, size_t count, uint32_t q, uint32_t d, int dev, void* st) {
    return compress_any(in, out, count, q, d, dev, st, 1, 0);
}
qf_status qf_compress_i64(const int64_t* in, int64_t* out, size_t count, uint64_t q, uint32_t d, int dev, void* st) {
    return compress_any(in, out, count, q, d, dev, st, 0, 1);
}
qf_status qf_decompress_i64(const int64_t* in, int64_t* out, size_t count, uint64_t q, uint32_t d, int dev, void* st) {
    return compress_any(in, out, count, q, d, dev, st, 1, 1);
}

// ---- Compress_d + ByteEncode_d / ByteDecode_d + Decompress_d (FIPS 203 Algorithms 5, 6) ------------------------------
static qf_status byte_code_any(const void* in, void* out, size_t npoly, uint32_t q, uint32_t d, int flag, int dev, void* stream,
                               int decode) {
    if ((!in || !out) && npoly) return QF_ERR_INVALID;
    if (d < 1) return QF_ERR_INVALID;  // same contract as lossy_compress (lossy_compression_fips203.rs:91-94)
    if (d > 12 || q > 65535 || q < 2) return QF_ERR_UNSUPPORTED;
    if (npoly == 0) return QF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t coeff_bytes = npoly * 512, packed_bytes = npoly * 32 * (size_t)d;
    const size_t in_bytes = decode ? packed_bytes : coeff_bytes, out_bytes = decode ? coeff_bytes : packed_bytes;
    auto run = [&](const void* di, void* dout) -> cudaError_t {
        return decode ? qf_launch_byte_decode((const uint8_t*)di, (uint16_t*)dout, npoly, q, d, flag, st)
                      : qf_launch_byte_encode((const uint16_t*)di, (uint8_t*)dout, npoly, q, d, flag, st);
    };
    auto map_err = [](cudaError_t e) { return e == cudaSuccess ? QF_OK : (e == cudaErrorInvalidValue ? QF_ERR_INVALID : QF_ERR_CUDA); };
    if (dev) return map_err(run(in, out));
    void *di = nullptr, *dout = nullptr;
    if (cudaMalloc(&di, in_bytes) != cudaSuccess) return QF_ERR_CUDA;
    if (cudaMalloc(&dout, out_bytes) != cudaSuccess) { cudaFree(di); return QF_ERR_CUDA; }
    qf_status rc = QF_OK;
    if (cudaMemcpyAsync(di, in, in_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (rc == QF_OK) rc = map_err(run(di, dout));
    if (rc == QF_OK && cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == QF_OK) rc = QF_ERR_CUDA;
    cudaFree(di);
    cudaFree(dout);
    return rc;
}

qf_status qf_compress_encode_u16(const uint16_t* in, uint8_t* out, size_t npoly, uint32_t q, uint32_t d, int compress, int dev,
                                 void* st) {
    return byte_code_any(in, out, npoly, q, d, compress, dev, st, 0);
}
qf_status qf_decode_decompress_u16(const uint8_t* in, uint16_t* out, size_t npoly, uint32_t q, uint32_t d, int decompress,
                                   int dev, void* st) {
    return byte_code_any(in, out, npoly, q, d, decompress, dev, st, 1);
}

// ---- common_encodings.rs:49-153, batched ----------------------------------------------------------------------------------
// in_bytes / out_bytes per element are fixed by the direction: digits are bytes, coefficients coeff_bytes (2 or 8) wide
static qf_status encode_any(const void* in, void* out, size_t count, size_t in_esz, size_t out_esz, int dev, cudaStream_t st,
                            cudaError_t (*run)(const void*, void*, void*), void* closure) {
    auto map_err = [](cudaError_t e) { return e == cudaSuccess ? QF_OK : (e == cudaErrorMisalignedAddress ? QF_ERR_INVALID : QF_ERR_CUDA); };
    if (dev) return map_err(run(in, out, closure));
    void *di = nullptr, *dout = nullptr;
    if (cudaMalloc(&di, count * in_esz) != cudaSuccess) return QF_ERR_CUDA;
    if (cudaMalloc(&dout, count * out_esz) != cudaSuccess) { cudaFree(di); return QF_ERR_CUDA; }
    qf_status rc = QF_OK;
    if (cudaMemcpyAsync(di, in, count * in_esz, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (rc == QF_OK) rc = map_err(run(di, dout, closure));
    if (rc == QF_OK && cudaMemcpyAsync(out, dout, count * out_esz, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QF_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == QF_OK) rc = QF_ERR_CUDA;
    cudaFree(di);
    cudaFree(dout);
    return rc;
}
struct EncClosure { size_t count; unsigned long long q; unsigned base; int coeff_bytes; cudaStream_t st; };

static qf_status encode_args_ok(const void* in, const void* out, size_t count, uint64_t q, uint32_t base, int coeff_bytes) {
    if ((!in || !out) && count) return QF_ERR_INVALID;
    if (base < 2 || q < 2) return QF_ERR_INVALID;  // MathError::InvalidIntegerInput (common_encodings.rs:133-137)
    if (base > 256 || q >= (1ull << 62)) return QF_ERR_UNSUPPORTED;
    if (coeff_bytes != 2 && coeff_bytes != 8) return QF_ERR_INVALID;
    if (coeff_bytes == 2 && q > 65535) return QF_ERR_INVALID;
    return QF_OK;
}

qf_status qf_encode_digits(const uint8_t* digits, void* coeffs, size_t count, uint64_t q, uint32_t base, int coeff_bytes,
                           int device_ptrs, void* cuda_stream) {
    qf_status st = encode_args_ok(digits, coeffs, count, q, base, coeff_bytes);
    if (st != QF_OK || count == 0) return st;
    EncClosure c{count, q, base, coeff_bytes, (cudaStream_t)cuda_stream};
    return encode_any(digits, coeffs, count, 1, (size_t)coeff_bytes, device_ptrs, c.st,
                      [](const void* i, void* o, void* cl) {
                          auto* c = (EncClosure*)cl;
                          return qf_launch_encode_digits((const uint8_t*)i, o, c->count, c->q, c->base, c->coeff_bytes, c->st);
                      }, &c);
}
qf_status qf_decode_digits(const void* coeffs, uint8_t* digits, size_t count, uint64_t q, uint32_t base, int coeff_bytes,
                           int device_ptrs, void* cuda_stream) {
    qf_status st = encode_args_ok(coeffs, digits, count, q, base, coeff_bytes);
    if (st != QF_OK || count == 0) return st;
    EncClosure c{count, q, base, coeff_bytes, (cudaStream_t)cuda_stream};
    return encode_any(coeffs, digits, count, (size_t)coeff_bytes, 1, device_ptrs, c.st,
                      [](const void* i, void* o, void* cl) {
                          auto* c = (EncClosure*)cl;
                          return qf_launch_decode_digits(i, (uint8_t*)o, c->count, c->q, c->base, c->coeff_bytes, c->st);
                      }, &c);
}
qf_status qf_encode_bits_u16(const uint8_t* msg, uint16_t* coeffs, size_t nbytes, uint32_t q, int device_ptrs, void* cuda_stream) {
    qf_status st = encode_args_ok(msg, coeffs, nbytes, q, 2, 2);
    if (st != QF_OK || nbytes == 0) return st;
    EncClosure c{nbytes, q, 2, 2, (cudaStream_t)cuda_stream};
    // count = message bytes; 16 bytes of coefficients per message byte
    return encode_any(msg, coeffs, nbytes, 1, 16, device_ptrs, c.st,
                      [](const void* i, void* o, void* cl) {
                          auto* c = (EncClosure*)cl;
                          return qf_launch_encode_bits_u16((const uint8_t*)i, (uint16_t*)o, c->count, (uint32_t)c->q, c->st);
                      }, &c);
}
qf_status qf_decode_bits_u16(const uint16_t* coeffs, uint8_t* msg, size_t nbytes, uint32_t q, int device_ptrs, void* cuda_stream) {
    qf_status st = encode_args_ok(coeffs, msg, nbytes, q, 2, 2);
    if (st != QF_OK || nbytes == 0) return st;
    EncClosure c{nbytes, q, 2, 2, (cudaStream_t)cuda_stream};
    return encode_any(coeffs, msg, nbytes, 16, 1, device_ptrs, c.st,
                      [](const void* i, void* o, void* cl) {
                          auto* c = (EncClosure*)cl;
                          return qf_launch_decode_bits_u16((const uint16_t*)i, (uint8_t*)o, c->count, (uint32_t)c->q, c->st);
                      }, &c);
}

qf_status qf_sample_z(const double* centers, size_t count, double s, uint64_t seed, int64_t* out) {
    if (!centers || !out || !(s > 0)) return QF_ERR_INVALID;
    if (!(s < 2.0e6)) return QF_ERR_UNSUPPORTED;  // proposals are rounded in fp32: 7.6 sigma' must stay below 2^24
    if (count == 0) return QF_OK;
    // one "target" per value so that every value owns its Philox stream (its own stream id: qf_samp_d with the same
    // seed draws from QF_STREAM_SAMP_D); slabs of 2^24 values bound the device buffers and the int launch arguments
    const size_t slab = (size_t)1 << 24, cap = count < slab ? count : slab;
    double *dc = nullptr, *dz = nullptr;
    int* dflag = nullptr;
    if (cudaMalloc(&dc, cap * 8) != cudaSuccess) return QF_ERR_CUDA;
    if (cudaMalloc(&dz, cap * 8) != cudaSuccess) { cudaFree(dc); return QF_ERR_CUDA; }
    if (cudaMalloc(&dflag, sizeof(int)) != cudaSuccess) { cudaFree(dc); cudaFree(dz); return QF_ERR_CUDA; }
    qf_status rc = cudaMemset(dflag, 0, sizeof(int)) == cudaSuccess ? QF_OK : QF_ERR_CUDA;
    std::vector<double> hz(cap);
    for (size_t o = 0; o < count && rc == QF_OK; o += slab) {
        const size_t cnt = count - o < slab ? count - o : slab;
        if (cudaMemcpy(dc, centers + o, cnt * 8, cudaMemcpyHostToDevice) != cudaSuccess) rc = QF_ERR_CUDA;
        if (rc == QF_OK && qf_launch_dgauss(dc, 1, dz, 1, nullptr, 0, (int)cnt, 1, s, seed, (uint64_t)o, QF_STREAM_SAMPLE_Z, dflag,
                                            nullptr) != cudaSuccess)
            rc = QF_ERR_CUDA;
        if (rc == QF_OK && cudaMemcpy(hz.data(), dz, cnt * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = QF_ERR_CUDA;
        if (rc == QF_OK)
            for (size_t i = 0; i < cnt; ++i) out[o + i] = (int64_t)hz[i];
    }
    int hflag = 0;
    if (rc == QF_OK && cudaMemcpy(&hflag, dflag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) rc = QF_ERR_CUDA;
    if (rc == QF_OK && hflag) rc = QF_ERR_NUMERIC;  // a centre was NaN / infinite: the sampler gave up (common.cuh)
    cudaFree(dc);
    cudaFree(dz);
    cudaFree(dflag);
    return rc;
}

// Debug / self-test entry: exact V = X W^t through the tcgen05 int8 path, host buffers.
// x: B x K signed (|x| < 2^(8 LX - 1)), w: N x K (residues < 2^(8 LW) if !w_signed, else |w| < 2^(8 LW - 1)).
qf_status qf_debug_gemm_i8(const int64_t* x, const int64_t* w, int w_signed, int LX, int LW, int64_t B, int64_t N,
                           int64_t K, uint64_t q, int64_t* out) {
    if (!x || !w || !out || B < 1 || N < 1 || K < 1) return QF_ERR_INVALID;
    const long ldk = (K + 127) / 128 * 128;
    std::vector<int8_t> hx((size_t)LX * B * ldk, 0);
    std::vector<uint8_t> hw((size_t)LW * N * ldk, 0);
    for (long b = 0; b < B; ++b)
        for (long kk = 0; kk < K; ++kk) {
            long long v = x[b * K + kk];
            for (int j = 0; j < LX; ++j) {
                long long lo = ((v + 128) & 255) - 128;  // balanced digit in [-128,127]
                if (j == LX - 1) lo = v;
                hx[((size_t)j * B + b) * ldk + kk] = (int8_t)lo;
                v = (v - lo) / 256;
            }
        }
    for (long nn = 0; nn < N; ++nn)
        for (long kk = 0; kk < K; ++kk) {
            long long v = w[nn * K + kk];
            for (int i = 0; i < LW; ++i) {
                long long lo;
                if (w_signed) { lo = ((v + 128) & 255) - 128; if (i == LW - 1) lo = v; v = (v - lo) / 256; }
                else { lo = v & 255; v >>= 8; }
                hw[((size_t)i * N + nn) * ldk + kk] = (uint8_t)(lo & 255);
            }
        }
    int8_t* dx = nullptr; uint8_t* dw = nullptr; int64_t* dout = nullptr;
    qf_status rc = QF_OK;
    if (cudaMalloc(&dx, hx.size()) != cudaSuccess || cudaMalloc(&dw, hw.size()) != cudaSuccess ||
        cudaMalloc(&dout, (size_t)B * N * 8) != cudaSuccess)
        rc = QF_ERR_CUDA;
    if (rc == QF_OK && (cudaMemcpy(dx, hx.data(), hx.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
                        cudaMemcpy(dw, hw.data(), hw.size(), cudaMemcpyHostToDevice) != cudaSuccess))
        rc = QF_ERR_CUDA;
    if (rc == QF_OK) {
        I8GemmArgs a{};
        a.x = dx; a.ldx = ldk; a.x_plane = (long)B * ldk;
        a.w = dw; a.ldw = ldk; a.w_plane = (long)N * ldk;
        a.LX = LX; a.LW = LW; a.w_signed = w_signed; a.B = (int)B; a.N = (int)N; a.K = (int)K;
        a.out_kind = 0; a.sign = 1; a.q = q; a.base = nullptr; a.ldbase = 0; a.out = dout; a.ldout = N; a.flag = nullptr;
        cudaError_t e = qf_launch_gemm_i8(a, nullptr);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { fprintf(stderr, "qf_debug_gemm_i8: %s\n", cudaGetErrorString(e)); rc = QF_ERR_CUDA; }
    }
    if (rc == QF_OK && cudaMemcpy(out, dout, (size_t)B * N * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = QF_ERR_CUDA;
    cudaFree(dx); cudaFree(dw); cudaFree(dout);
    return rc;
}

// Peak of the int8 tensor pipe as this library can drive it: a plain one-digit-pair contraction (LX = LW = 1: 128 x 256
// tiles, two accumulator buffers in TMEM, int32 store epilogue) on random bytes, long K.  `iters` launches timed one by one
// (best = burst figure), then launches back to back for >= sustain_ms (sustained figure, clocks settled under load).
qf_status qf_probe_i8_peak(int device, int64_t B, int64_t N, int64_t K, int iters, double sustain_ms, double* best_tops,
                           double* sustained_tops, double* pipe_tops) {
    if (B < 1 || N < 1 || K < 128 || K > 65536 || (K & 127) || iters < 1) return QF_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return QF_ERR_CUDA;
    int8_t* dx = nullptr; uint8_t* dw = nullptr; int32_t* dout = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaStream_t st = nullptr;
    qf_status rc = QF_OK;
    const size_t xb = (size_t)B * K, wb = (size_t)N * K;
    if (cudaMalloc(&dx, xb) != cudaSuccess || cudaMalloc(&dw, wb) != cudaSuccess || cudaMalloc(&dout, (size_t)B * N * 4) != cudaSuccess ||
        cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess ||
        cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
        rc = QF_ERR_CUDA;
    if (rc == QF_OK && (qf_launch_uniform_modq((int64_t*)dx, (long)(xb / 8), 1ull << 62, 11, 0, st) != cudaSuccess ||
                        qf_launch_uniform_modq((int64_t*)dw, (long)(wb / 8), 1ull << 62, 12, 0, st) != cudaSuccess))
        rc = QF_ERR_CUDA;
    I8GemmArgs a{};
    a.x = dx; a.ldx = K; a.x_plane = (long)xb;
    a.w = dw; a.ldw = K; a.w_plane = (long)wb;
    a.LX = 1; a.LW = 1; a.w_signed = 0; a.B = (int)B; a.N = (int)N; a.K = (int)K;
    a.out_kind = 1; a.sign = 1; a.q = 0; a.out = dout; a.ldout = N; a.flag = nullptr;
    const double ops = 2.0 * (double)B * (double)N * (double)K;
    double best = 0, sustained = 0;
    for (int i = 0; i < iters + 2 && rc == QF_OK; ++i) {  // two warm-ups
        cudaEventRecord(e0, st);
        if (qf_launch_gemm_i8(a, st) != cudaSuccess) { rc = QF_ERR_CUDA; break; }
        cudaEventRecord(e1, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) { rc = QF_ERR_CUDA; break; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (i >= 2 && ms > 0) best = std::max(best, ops / (ms * 1e-3) / 1e12);
    }
    if (rc == QF_OK && sustain_ms > 0 && best > 0) {
        const int reps = std::max(4, (int)(sustain_ms / (ops / (best * 1e12) * 1e3)) + 1);
        cudaEventRecord(e0, st);
        for (int i = 0; i < reps; ++i)
            if (qf_launch_gemm_i8(a, st) != cudaSuccess) { rc = QF_ERR_CUDA; break; }
        cudaEventRecord(e1, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) rc = QF_ERR_CUDA;
        float ms = 0;
        if (rc == QF_OK) cudaEventElapsedTime(&ms, e0, e1);
        if (ms > 0) sustained = ops * reps / (ms * 1e-3) / 1e12;
    }
    // the pipe itself: MMAs on resident operands, one CTA per SM (best of 3 launches of ~5 ms)
    if (rc == QF_OK && pipe_tops && B >= 1024) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        double bestp = 0;
        for (int i = 0; i < 4 && rc == QF_OK; ++i) {
            double pops = 0;
            cudaEventRecord(e0, st);
            if (qf_launch_i8_pipe_probe(dx, dw, 20000, sms, &pops, st) != cudaSuccess) { rc = QF_ERR_CUDA; break; }
            cudaEventRecord(e1, st);
            if (cudaStreamSynchronize(st) != cudaSuccess) { rc = QF_ERR_CUDA; break; }
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (i >= 1 && ms > 0) bestp = std::max(bestp, pops / (ms * 1e-3) / 1e12);
        }
        *pipe_tops = bestp;
    }
    if (best_tops) *best_tops = best;
    if (sustained_tops) *sustained_tops = sustained;
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (st) cudaStreamDestroy(st);
    cudaFree(dx); cudaFree(dw); cudaFree(dout);
    return rc;
}

qf_status qf_fill_uniform_modq_dev(int64_t* out, size_t count, uint64_t q, uint64_t seed, void* st) {
    if (!out || q < 2) return QF_ERR_INVALID;
    return qf_launch_uniform_modq(out, (long)count, q, seed, 0, (cudaStream_t)st) == cudaSuccess ? QF_OK : QF_ERR_CUDA;
}

}  // extern "C"
