// Internal launcher declarations (device pointers everywhere).  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"
#include "domain_code.cuh"

// ---- gemm_f64.cu ----------------------------------------------------------
cudaError_t qf_launch_gemm_f64(const double* X, long ldx, const double* W, long ldw, double* C, long ldc,
                               int B, int N, int K, double alpha, double beta, int tri_lower,
                               cudaStream_t stream);

// ---- elementwise.cu -------------------------------------------------------
// out[b][j] = (double) in[b][j]; optionally norm2[b] = sum_j in[b][j]^2 (exact, u64 saturating)
cudaError_t qf_launch_i32_to_f64(const int32_t* in, long ldin, double* out, long ldout, int B, int M,
                                 unsigned long long* norm2, cudaStream_t stream);
cudaError_t qf_launch_i64_to_f64(const int64_t* in, long ldin, double* out, long ldout, int B, int M,
                                 double scale, cudaStream_t stream);
// out[b][j] = (int32) in[b][j]; sets *flag if a value does not fit / is not an integer
cudaError_t qf_launch_f64_to_i32(const double* in, long ldin, int32_t* out, long ldout, int B, int M,
                                 int* flag, cudaStream_t stream);
// in_domain[b] = norm2[b] <= bound
cudaError_t qf_launch_domain_flags(const unsigned long long* norm2, unsigned long long bound, uint8_t* flags,
                                   int B, cudaStream_t stream);
// flags[b] &= norm2[b] <= bound: flags already holds a per-row ok byte (a canonical packed slot) that the domain check ANDs in
cudaError_t qf_launch_domain_flags_and(const unsigned long long* norm2, unsigned long long bound, uint8_t* flags,
                                       int B, cudaStream_t stream);

struct CombineArgs {
    const double* acc[4];   // exact-integer fp64 partial products, B x N each, leading dim ldacc
    int shift[4];           // value = sum_c acc_c * 2^shift_c
    int nacc;
    int acc_sign;           // +1 or -1
    long ldacc;
    const int64_t* base;    // optional B x N (ld ldbase): out = base + acc_sign * value
    long ldbase;
    unsigned long long q;   // 0: plain integer result, else reduce into [0,q)
};
cudaError_t qf_launch_combine_i64(const CombineArgs& a, int64_t* out, long ldout, int B, int N, cudaStream_t stream);
cudaError_t qf_launch_combine_f64(const CombineArgs& a, double* out, long ldout, int B, int N, cudaStream_t stream);
// int32 output; sets *flag when a value does not fit
cudaError_t qf_launch_combine_i32(const CombineArgs& a, int32_t* out, long ldout, int B, int N, int* flag,
                                  cudaStream_t stream);
// out[b][j] = (int32)(P[b][j] + (j >= split ? Zb[b][j-split] : 0))   (e = p + [R;I] z, lower part)
cudaError_t qf_launch_finalize_pert(const double* P, long ldp, const double* Zb, long ldz, int32_t* out, long ldo,
                                    int B, int M, int split, int* flag, cudaStream_t stream);

// split an exact-integer fp64 matrix into balanced chunks of `bits` bits: in = sum_c out_c * 2^(c*bits)
cudaError_t qf_launch_split_chunks(const double* in, long ldin, double* const* out, int nchunks, int bits,
                                   long ldout, int B, int M, cudaStream_t stream);
// dst[b][cols[j]] = src[b][j]  (dst pre-zeroed by the caller)
cudaError_t qf_launch_scatter_cols_f64(const double* src, long ldsrc, const int* cols, int ncols, double* dst,
                                       long lddst, int B, double scale, cudaStream_t stream);

// ---- samplers (elementwise.cu) -------------------------------------------
cudaError_t qf_launch_normal_fill(double* out, long ld, int B, int M, uint64_t seed, uint64_t first_target,
                                  uint32_t tag, cudaStream_t stream);
// out[b][j] <- D_{Z, s, center[b][j]} (center == nullptr: centred at 0); flag (optional): sampler bail-out bit
cudaError_t qf_launch_dgauss(const double* center, long ldc, double* out_f64, long ldo, int32_t* out_i32,
                             long ldoi, int B, int M, double s, uint64_t seed, uint64_t first_target,
                             uint32_t tag, int* flag, cudaStream_t stream);
// structured e = S z for the G-trapdoor short basis S = [[R S', I + R W],[S', W]] (api.cu detect_gpv_structure)
cudaError_t qf_launch_sprime_apply(const double* Z, long ldz, double* I2, long ldi, int B, int nk, int k, const double* sk,
                                   int reversed, cudaStream_t stream);
cudaError_t qf_launch_gpv_struct_finalize(int32_t* e, long lde, const double* Z2, long ldz, const double* I2, long ldi, int B,
                                          int mb, int nk, int* flag, cudaStream_t stream, const int8_t* g3 = nullptr,
                                          long ldg = 0);
// two-phase form: e_bot = g3 + S' z1 written as int32 into e[b][mb + row] and as L balanced digit planes (one pass over z1)
cudaError_t qf_launch_gpv_ebot(const double* Z, long ldz, const int8_t* g3, long ldg, int32_t* e, long lde, int mb,
                               int8_t* planes, long plane_stride, long ldk, int L, int B, int nk, int k, const double* sk,
                               int reversed, int* flag, cudaStream_t stream);
// two-phase nearest plane (api.cu samp_p_np2_chunk): base-b digits of the syndromes h (B x n, in [0,q)) in gadget order,
// g3[b][blk*k + t] = digit t of h[b][blk], written as ONE s8 digit plane (B x ldk, columns [0, n*k)) and marked in
// plane 0 of the zero-tile map (k blocks [0, ceil(n*k/128)) of every target tile)
cudaError_t qf_launch_gadget_digits(const int64_t* h, long ldh, int8_t* plane, long ldk, int B, int n, int k, unsigned base,
                                    uint8_t* nz, int nz_kb_total, cudaStream_t stream, double* I2 = nullptr, long ldi = 0);
// M'[i][bc k + t] = sum_t' U[i][col(bc, t')] Skinv[t'][t] over the upper unitriangular part of U (col = the basis column
// of gadget coordinate bc k + t', reversed when `rev`): the map from a gadget-coordinate vector g (centre -[R;I] g) to
// GSO coordinates of the first nk basis vectors (api.cu samp_p_np2_chunk)
cudaError_t qf_launch_gadget_to_gso(const double* U, long ldu, int nk, int k, int rev, const double* skinv, double* out,
                                    long ldo, cudaStream_t stream);
// structured perturbation (api.cu setup_structured_sigma2): X2[b][mb+j] = sqrt_beta * G[b][mb+j] and the balanced
// base-256 digits of rint(that * fscale) into L planes of B x ldk bytes
cudaError_t qf_launch_pert_xb(const double* G, long ldg, double* X2, long ldx, int8_t* planes, long plane_stride, long ldk,
                              int B, int mb, int nk, double sqrt_beta, double fscale, int L, int* flag, cudaStream_t stream);
// N(0,1) draws of the perturbation (same Philox stream as qf_launch_normal_fill) written as fixed-point digits:
// coordinates j < split: LG planes of rint(g * gscale) at gplanes[b * ldkg + j];
// coordinates j >= split (structured square root only): x_b = sqrt_beta * g into X2[b][j] and LB planes of
// rint(x_b * bscale) at bplanes[b * ldkb + (j - split)].
cudaError_t qf_launch_pert_normal_digits(int B, int M, int split, uint64_t seed, uint64_t first_target, int8_t* gplanes,
                                         long gplane_stride, long ldkg, int LG, double gscale, double* X2, long ldx,
                                         int8_t* bplanes, long bplane_stride, long ldkb, int LB, double sqrt_beta, double bscale,
                                         int* flag, cudaStream_t stream);
cudaError_t qf_launch_uniform_modq(int64_t* out, long count, unsigned long long q, uint64_t seed,
                                   uint64_t first_index, cudaStream_t stream);
cudaError_t qf_launch_ternary(int8_t* out, long count, uint64_t seed, cudaStream_t stream);

// ---- lattice.cu -------------------------------------------------------------
// Gadget-lattice preimage (mp_perturbation.rs:173-191) for every (target, row):
// V: B x n residues, Z: B x (n*k) exact-integer doubles.
// sk: k x k block basis (row-major), gso: k x k GSO (columns are b~_i), both in device memory.
cudaError_t qf_launch_gadget_sample(const int64_t* V, long ldv, double* Z, long ldz, int B, int n, int k,
                                    int base, unsigned long long q, const double* sk, const double* gso,
                                    double s_g, uint64_t seed, uint64_t first_target, int* flag, cudaStream_t stream);
// One diagonal block of the randomized nearest-plane recursion in GSO coordinates:
// for i = j0+nb-1 .. j0:  c' = T[b][i] - sum_{j>i in block} U[i][j] z_j ;  z_i <- D_{Z, s/||b~_i||, c'}
// writes Z[b][i].  dg: per-coordinate sampler parameters (length >= j0+nb).
// *flag is set when |z| >= zlimit (exact-integer range check).
// prop: this block's pre-generated proposals (np_propose), coordinate-major: prop[(i - j0) * ldprop + b]
// dig (optional): the kernel also writes the balanced base-256 digit planes of its block of z (L planes of B x ldk bytes,
// planes already offset to column 0), marks the zero-tile map and raises the digit-count gates, like qf_launch_split_f64_limbs
struct NpDigitOut {
    int8_t* planes; long plane_stride, ldk; int L;
    uint8_t* nz; int nz_m_tiles, nz_kb_total;
    int* gate[4];
};
// nb <= 64: one diagonal block [j0, j0 + nb).  nb > 64 (j0 a multiple of 64, up_lo = j0): the whole block range, its
// 64-wide diagonal blocks from the top down, each followed by the rank-64 update of the columns of the range below it,
//   T[b][j] -= sum_i Z[b][j0' + i] U[j][j0' + i]   for this CTA's own targets (no cross-CTA dependence: one launch).
// prop: proposals of coordinate prop0 onwards (prop0 = -1: j0)
cudaError_t qf_launch_np_diag(double* T, long ldt, double* Z, long ldz, const double* U, long ldu,
                              const DGaussParams* dg, const float4* prop, long ldprop, int B, int j0, int nb, int dim,
                              uint64_t seed, uint64_t first_target, double zlimit, int* flag, cudaStream_t stream, int up_lo = -1,
                              const NpDigitOut* dig = nullptr, int prop0 = -1, int variant = 0);
// two proposals per (target, coordinate) for coordinates [j_lo, j_lo + width): out[(i - j_lo) * ldo + b]
cudaError_t qf_launch_np_propose(float4* out, long ldo, int B, int j_lo, int width, int dim, uint64_t seed,
                                 uint64_t first_target, cudaStream_t stream);

// ---- compress.cu -----------------------------------------------------------
cudaError_t qf_launch_compress_u16(const uint16_t* in, uint16_t* out, size_t count, uint32_t q, uint32_t d,
                                   int decompress, cudaStream_t stream);
// Compress_d + ByteEncode_d / ByteDecode_d + Decompress_d, one warp per degree-256 polynomial (compress.cu)
cudaError_t qf_launch_byte_encode(const uint16_t* in, uint8_t* out, size_t npoly, uint32_t q, uint32_t d, int compress,
                                  cudaStream_t stream);
cudaError_t qf_launch_byte_decode(const uint8_t* in, uint16_t* out, size_t npoly, uint32_t q, uint32_t d, int decompress,
                                  cudaStream_t stream);
cudaError_t qf_launch_compress_i64(const int64_t* in, int64_t* out, size_t count, unsigned long long q,
                                   uint32_t d, int decompress, cudaStream_t stream);

// ---- encodings.cu : common_encodings.rs:49-153, batched (digits as bytes, base <= 256; bit-packed base 2) ----------
cudaError_t qf_launch_encode_digits(const uint8_t* digits, void* coeffs, size_t count, unsigned long long q, unsigned base,
                                    int coeff_bytes, cudaStream_t stream);
cudaError_t qf_launch_decode_digits(const void* coeffs, uint8_t* digits, size_t count, unsigned long long q, unsigned base,
                                    int coeff_bytes, cudaStream_t stream);
cudaError_t qf_launch_encode_bits_u16(const uint8_t* msg, uint16_t* coeffs, size_t nbytes, uint32_t q, cudaStream_t stream);
cudaError_t qf_launch_decode_bits_u16(const uint16_t* coeffs, uint8_t* msg, size_t nbytes, uint32_t q, cudaStream_t stream);

// ---- ring_ntt.cu -----------------------------------------------------------
// Negacyclic products over Z_q[X]/(X^n+1) through an exact NTT over the Goldilocks prime.
// a_hat: npoly x n precomputed transforms of the key polynomials (centred lift of a mod q).
// tw: device table of 2n+1 words (psi powers bit-reversed, inverse powers, 1/n) from qf_ring_make_tables.
void qf_ring_make_tables(int n, uint64_t* host_out);
// one CTA per polynomial: npoly may be every polynomial of a key table (< 2^31)
cudaError_t qf_launch_ring_prepare(const int64_t* a, uint64_t* a_hat, long npoly, int n, unsigned long long q,
                                   const uint64_t* tw, cudaStream_t stream);
// out[b] = sum_j a_j * sigma[b][j] mod (X^n+1, q);  sigma: B x npoly x n (int32), out: B x n
// key_idx != NULL (device, B ints): keyed form, row b uses the key a_hat + key_idx[b] npoly n of a table of nkeys keys;
// an index outside [0, nkeys) is not used to address the table, sets *flag |= QF_FLAG_KEY_INDEX, and its row gets u = 0
// and norm2 = ~0 (not in the domain).  The same holds for the keyed forms of the two launchers below.
cudaError_t qf_launch_ring_f_a(const int32_t* sigma, const uint64_t* a_hat, int64_t* out, unsigned long long* norm2,
                               int B, int npoly, int n, unsigned long long q, const uint64_t* tw,
                               cudaStream_t stream, const int32_t* key_idx = nullptr, int nkeys = 0, int* flag = nullptr,
                               const PackedRows* packed = nullptr);
// packed != NULL (keyed only, n >= 64): sigma is unused and row b is decoded from slot b of *packed inside the kernel;
// packed->ok[b] = 1 when the slot is canonical.  The same for qf_launch_ring_small.
// Schoolbook fallback for degrees that are not a power of two (or < 64): a is the raw key, npoly x n in [0,q).
cudaError_t qf_launch_ring_f_a_schoolbook(const int32_t* sigma, const int64_t* a, int64_t* out,
                                          unsigned long long* norm2, int B, int npoly, int n, unsigned long long q,
                                          cudaStream_t stream, const int32_t* key_idx = nullptr, int nkeys = 0,
                                          int* flag = nullptr);
// count ring TrapGen keys [1 | a_bar_t | g^t - (a_bar_t r_t + e_t)] mod q from ar = a_bar_t r_{t,j} mod q (count x k x n),
// e (count x k x n) and gpow[j] = base^j mod q; out: count x (k+2) x n
cudaError_t qf_launch_ring_trap_assemble(const int64_t* a_bar, const int64_t* ar, const int32_t* e, const uint64_t* gpow,
                                         int64_t* out, long count, int k, int n, unsigned long long q, cudaStream_t stream);

// ---- setup.cu (per-key, not per-target) --------------------------------------
cudaError_t qf_launch_colnorm2(const double* G, long ld, int rows, int cols, double* d, cudaStream_t stream);
cudaError_t qf_launch_transpose_scale(const double* in, long ldin, double* out, long ldout, int rows, int cols,
                                      const double* scale, cudaStream_t stream);
cudaError_t qf_launch_gather_cols(const double* in, long ldin, const int* cols, int ncols, double* out, long ldout,
                                  int rows, cudaStream_t stream);
cudaError_t qf_launch_make_dg(const double* d, int count, double s, DGaussParams* dg, cudaStream_t stream);
// blocked Cholesky building blocks (compute_sqrt_sigma_2, mp_perturbation.rs:111-139)
cudaError_t qf_launch_potrf_diag(double* A, long ld, int nb, double* Linv, int* info, cudaStream_t stream);
cudaError_t qf_launch_fixed_rows_prepare(const double* L, long ld, int rows, int cols, int Ldig, double mult, double* scale,
                                         int8_t* planes, long plane_stride, long ldk, cudaStream_t stream);
cudaError_t qf_launch_gso_rdiag(double* rdiag, const double* L, long ldl, int nb, int first, cudaStream_t stream);
cudaError_t qf_launch_scale_cols(const double* in, long ldin, double* out, long ldout, long rows, long cols,
                                 const double* colscale, cudaStream_t stream);
cudaError_t qf_launch_tril(double* A, long ld, long n, cudaStream_t stream);
cudaError_t qf_launch_copy_block(const double* in, long ldin, double* out, long ldout, long rows, int cols, cudaStream_t stream);
cudaError_t qf_launch_sigma2_assemble(double* C, long ldc, long n, int full, const double* Gin, long ldg, const double* R,
                                      long ldr, long mb, const double* Sigma, long lds, double diag, double gcoef, double coef,
                                      cudaStream_t stream);

// ---- gemm_i8.cu : exact integer contraction on tcgen05 (kind::i8) --------------------------
struct I8GemmArgs {
    const int8_t* x;    // LX planes of B x K balanced s8 limbs, row stride ldx, plane stride x_plane (bytes)
    long ldx, x_plane;
    const void* w;      // LW planes of N x K limbs (u8 residue limbs or balanced s8 limbs)
    long ldw, w_plane;
    int LX, LW, w_signed;
    int B, N, K;
    int out_kind;       // 0: int64 (base, sign, optional mod q)  1: int32 store  2: fp64 accumulate
    int sign;
    unsigned long long q;
    const int64_t* base;
    long ldbase;
    void* out;
    long ldout;
    int* flag;
    const double* scale;   // out_kind 3: out[b][n] -= V * scale[n]  (fp64)
    // optional zero-tile map of x: nz[(j * nz_m_tiles + nz_m_off + m_tile) * nz_kb_total + nz_kb_off + kb] != 0
    // iff digit plane j has a non-zero byte in that 128-target x 128-column tile (K offset must be 128-aligned)
    const uint8_t* x_nz;
    int nz_m_tiles, nz_kb_total, nz_kb_off, nz_m_off;
    // optional device counter: += int8 operations the tensor pipe actually executed (zero digit tiles are skipped)
    unsigned long long* mma_units;
    unsigned long long* tim;  // optional: 4 phase cycle counters (diagnostics)
    // out_kind 3 only: digit sums D_d with d < d_lo are not computed (their pairs lie below the error budget)
    int d_lo;
    int overwrite;  // out_kind 3 only: out = -V * scale[n] (store) instead of out -= V * scale[n]
    // optional conditional launch: the grid runs only if gate_lo <= *gate <= gate_hi (device int)
    const int* gate;
    int gate_lo, gate_hi;
    // out_kind 3 only: extra factor on scale[n] (0 = 1): the caller passes the TOP planes of a fixed-point matrix
    // (w advanced by `dropped` planes, LW reduced) and 256^dropped here
    double scale_mul;
    // structured key matrix: rows [n0, n0 + nt) are zero in the columns  1: k >= n0 + nt + tri_slack;
    // 2: k < K - (n0 + nt) - tri_slack;  3: k >= K - n0 + tri_slack;  4: k < n0 - tri_slack.  Those k blocks are skipped.
    int tri_mode, tri_slack;
};
int qf_i8_tile_n(int LX, int LW, int N, int d_lo = 0);
// gemm_i8_fused.cu: out = X W^t mod q with X read as int32 (digit split fused into the contraction) and the
// squared row norms of X accumulated on the way (norm2 optional)
struct FaFusedArgs {
    const int32_t* x; long ldx;   // B x K
    const void* w; long ldw, w_plane;  // LW planes of N x K limbs
    int LX, LW, w_signed;
    int LX_typical;   // digits covering the sampler's tail cut (0: unknown)
    int B, N, K;
    unsigned long long q;
    int64_t* out; long ldout;
    unsigned long long* norm2;
    unsigned long long* mma_units;
    int* retry_flag;   // optional device int: enables the optimistic (LX - 1 digits first) launch pair
    unsigned long long* tim;  // optional diagnostics (QF_TRACE): 6 cycle counters summed over CTAs, see gemm_i8_fused.cu
};
cudaError_t qf_launch_f_a_fused(const FaFusedArgs& a, cudaStream_t stream);
cudaError_t qf_launch_gemm_i8(const I8GemmArgs& a, cudaStream_t stream);
// tensor-pipe ceiling probe: MMAs on shared-memory-resident operands (gemm_i8.cu)
cudaError_t qf_launch_i8_pipe_probe(const int8_t* x, const uint8_t* w, int iters, int grid, double* ops_out, cudaStream_t stream);

// ---- limb splitting (elementwise.cu) ---------------------------------------------------------
// balanced s8 digits; *flag |= 8 when a value does not fit L digits
// nz (optional, pre-zeroed): zero-tile map [L][nz_m_tiles][nz_kb_total] over 128-target x 128-column tiles;
// col0 = global column of in[.][0] (the planes pointer is already offset by col0)
// gate0..2 (optional, need nz): device ints raised to the index of the highest non-zero digit plane written
cudaError_t qf_launch_split_f64_limbs(const double* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B,
                                      int M, int L, int* flag, uint8_t* nz, int nz_m_tiles, int nz_kb_total, int col0,
                                      cudaStream_t stream, int* gate0 = nullptr, int* gate1 = nullptr, int* gate2 = nullptr,
                                      int* gate3 = nullptr);
cudaError_t qf_launch_split_i32_limbs(const int32_t* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B,
                                      int M, int L, unsigned long long* norm2, uint8_t* nz, int nz_m_tiles,
                                      int nz_kb_total, cudaStream_t stream);
// e[b][cols[j]] += (int32) sol[b][j]
cudaError_t qf_launch_add_cols_i32(int32_t* e, long lde, const double* sol, long ldsol, const int* cols, int ncols,
                                   int B, cudaStream_t stream);
// fixed-point digit planes of U for the tensor-core nearest-plane updates (see setup.cu)
// split > 0: the entries U[i][j] with i < split <= j are left out (two-phase recursion: that block is never multiplied)
cudaError_t qf_launch_ozaki_prepare(const double* U, long ld, int D, int blk, int sblk, int fs_last, int ss_last, int L,
                                    double* scale, int8_t* planes, long plane_stride, long ldk, cudaStream_t stream,
                                    int split = 0);

// narrow boundary types (elementwise.cu): int16 Domain values, device-side range check of residues
// narrow: *flag |= 64 when a value does not fit int16; range check: *flag |= 32 when a residue is outside [0, q)
cudaError_t qf_launch_narrow_i32_i16(const int32_t* in, int16_t* out, size_t count, int* flag, cudaStream_t stream);
cudaError_t qf_launch_widen_i16_i32(const int16_t* in, int32_t* out, size_t count, cudaStream_t stream);
cudaError_t qf_launch_range_check_i64(const int64_t* v, size_t count, unsigned long long q, int* flag, cudaStream_t stream);

// online half of samp_p from a pool entry (offline_online.cu, DESIGN 4.12): out[b][0:M] = x[b] as fp64 and
// v[b] = (u[b] + a[b]) mod q (u, a residues); T[b][n] = fma(X[b][n] / mul, scale[n] * mul, T[b][n]) with X the store-only
// unit-scale output of the contraction (-dv mul): the same value as the accumulating epilogue of that contraction
cudaError_t qf_launch_pool_expand(const int32_t* x, long ldx, double* out, long ldo, int M, const int64_t* u, long ldu,
                                  const int64_t* a, long lda, int64_t* v, long ldv, int N, int B, unsigned long long q,
                                  cudaStream_t stream);
cudaError_t qf_launch_pool_centre(const double* X, long ldx, double* T, long ldt, const double* scale, double mul, int N, int B,
                                  cudaStream_t stream);

// packed Domain values (domain_code.cu, DESIGN 4.11): rows x dim int32 <-> rows slots of slot_bytes bytes (k in [0, 30],
// slot_bytes a multiple of 16 and at least H0 + ceil(dim / 8); checked by the callers).  Encode: nbytes[row], -1 and a zero
// slot when the code does not fit or the row holds INT32_MIN.  Decode: ok[row] = 1 iff the slot is canonical.
// out (encode) / in (decode) 16-byte aligned, else cudaErrorMisalignedAddress.
long long qf_domain_h0(long long dim, int k);
cudaError_t qf_launch_domain_encode(const int32_t* in, long long rows, int dim, int k, long long slot_bytes, uint8_t* out,
                                    int32_t* nbytes, cudaStream_t stream);
cudaError_t qf_launch_domain_decode(const uint8_t* in, long long rows, int dim, int k, long long slot_bytes, int32_t* out,
                                    uint8_t* ok, cudaStream_t stream);
// recommended (k, slot_bytes) for entries ~ D_{Z,w} (qf_domain_code_params)
void qf_domain_code_recommend(double w, long long dim, int* k, long long* slot_bytes);
// balanced s8 digit planes of int64 values (B x M, row stride ldin) into L planes of B x ldk bytes, columns [M, ldk) zeroed;
// *flag |= 8 when a value does not fit L digits (the x operand of a contraction whose "targets" are residues, e.g. u' = H^-1 u)
cudaError_t qf_launch_split_i64_limbs(const int64_t* in, long ldin, int8_t* planes, long plane_stride, long ldk, int B, int M,
                                      int L, int* flag, cudaStream_t stream);

// tag inverse of a G-trapdoor key (setup.cu): Gauss-Jordan over Z_q with unit pivots on M = [H | I] (n x 2n residues,
// q < 2^62); on return *fail = 0 and the right half of M is H^-1, or *fail = c + 1 when column c has no unit pivot.
// f: n words of device scratch.
cudaError_t qf_launch_mat_inverse_mod(uint64_t* M, uint64_t* f, int n, unsigned long long q, int* fail, cudaStream_t stream);
// the same kernel on `count` matrices at once (one CTA each): M count x n x 2n, f count x n words, fail count ints
cudaError_t qf_launch_mat_inverse_mod_batched(uint64_t* M, uint64_t* f, int n, unsigned long long q, int* fail, int count,
                                              cudaStream_t stream);
// tag table (setup.cu): M_t = [H_t mod q | I] (count x n x 2n) from int64 tags (count x n x n, any sign), and the right
// halves of inverted M_t packed column-major per tag into tab (count x n x n words of word_bytes = 4 or 8)
cudaError_t qf_launch_tag_build(const int64_t* tags, int count, int n, unsigned long long q, uint64_t* M, cudaStream_t stream);
cudaError_t qf_launch_tag_pack(const uint64_t* M, int count, int n, int word_bytes, void* tab, cudaStream_t stream);
// per-target tag of samp_p (elementwise.cu): out[b] = H_{tidx[b]}^-1 (V[b] + H_0 y) - y mod q, y = G p_bot, p_bot =
// P[b][m_bar:]; tab / h0 column-major n x n words (word_bytes 4 needs q <= 2^32 and n <= 2^14); h0 = NULL means H_0 = I; gpow: base^s mod q,
// s < k <= 64.  A tag index outside [0, ntags) sets *flag |= QF_FLAG_TAG_INDEX and gives out[b] = 0.
// xr != NULL: the table is in polynomial form (n words h_t^-1 per tag, xr from qf_launch_poly_xpow) and
// out[b] = h_t^-1 * (V[b] + H_0 y) mod (f, q) - y.
cudaError_t qf_launch_tag_syndrome(const int64_t* V, long ldv, const double* P, long ldp, int m_bar, const int32_t* tidx,
                                   int ntags, const void* tab, const void* h0, int word_bytes, const uint64_t* gpow,
                                   unsigned long long q, int n, int k, int B, int64_t* out, long ldout, int* flag,
                                   cudaStream_t stream, const void* xr = nullptr);
// f_a tag table (setup.cu): tab[t] = (tags[t] - H_0) mod q column-major (count x n x n words of word_bytes = 4 or 8) from
// int64 tags (count x n x n, any sign); h0: n x n residues row-major, NULL means H_0 = I
cudaError_t qf_launch_tag_diff_pack(const int64_t* tags, int count, int n, unsigned long long q, const uint64_t* h0,
                                    int word_bytes, void* tab, cudaStream_t stream);
// per-target tag of f_a (elementwise.cu): targets are grouped by tag into groups of at most QF_F_A_TAG_GROUP, one CTA per
// group, so that a word of the table serves every target of the group.  The library is built with 8; the value 1 (one
// target per CTA, no sort) exists for the comparison build of scripts/bench_f_a_tagged.py.
#ifndef QF_F_A_TAG_GROUP
#define QF_F_A_TAG_GROUP 8
#endif
// Counting sort of the tag indices of B targets: hist, off and gstart hold ntags + 1 ints each; afterwards perm (B ints)
// lists the targets tag by tag, off[t] is where tag t starts in perm (off[ntags]: indices outside the table) and gstart[t]
// its first group (gstart[ntags]: the number of groups).  An index outside [0, ntags) sets *flag |= QF_FLAG_TAG_INDEX.
// Not used when QF_F_A_TAG_GROUP = 1.
// *ok = 1 when the correction kernel runs for this n and k on the current device (k <= 64, n <= 2^14, and its static plus
// dynamic shared memory fit the per-block opt-in limit: n <= 3631 at QF_F_A_TAG_GROUP = 8 on sm_100a)
cudaError_t qf_f_a_tag_supported(int n, int k, int* ok);
cudaError_t qf_launch_f_a_tag_sort(const int32_t* tidx, int B, int ntags, int* hist, int* off, int* gstart, int* perm,
                                   int* flag, cudaStream_t stream);
// u[b] += D_t G sigma[b][m_bar:] mod q for t = tidx[b] (in place, u[b] = A sigma[b] from f_a); tab: the table of
// qf_launch_tag_diff_pack; gpow: base^s mod q, s < k <= 64; word_bytes 4 needs q <= 2^32.  With QF_F_A_TAG_GROUP > 1 it
// reads the output of qf_launch_f_a_tag_sort (tidx unused); with 1 it reads tidx and flags an index outside the table.
// Rows of such indices are left as A sigma.
cudaError_t qf_launch_f_a_tag_correct(const int32_t* sigma, long lds, int m_bar, const int32_t* tidx, int ntags,
                                      const int* perm, const int* off, const int* gstart, const void* tab, int word_bytes,
                                      const uint64_t* gpow, unsigned long long q, int n, int k, int B, int64_t* u, long ldu,
                                      int* flag, cudaStream_t stream);

// tags in polynomial form (elementwise.cu, DESIGN 4.10): H_t = rot_f(h_t), f = X^n + sum_{i<n} f_i X^i with fq = f_i mod q.
// *ok = 1 when the kernels of the samp_p table (samp_p != 0: inverse and syndrome) or of the f_a table run for this n and k
// on the current device: k <= 64, n <= 2^14, static plus dynamic shared memory within the per-block opt-in limit.
cudaError_t qf_poly_tag_supported(int n, int k, int samp_p, int* ok);
// xr = rows X^{n+j} mod (f, q), j < n - 1, n words of word_bytes each (nothing for n = 1)
cudaError_t qf_launch_poly_xpow(const uint64_t* fq, int n, unsigned long long q, int word_bytes, void* xr, cudaStream_t stream);
// tab[x] = tags[x] mod q, count words of word_bytes (any sign)
cudaError_t qf_launch_poly_tag_pack(const int64_t* tags, long count, unsigned long long q, int word_bytes, void* tab,
                                    cudaStream_t stream);
// tab[t] = h_t^-1 mod (f, q) for count tags of n coefficients (any sign), q = p^e, lifts = ceil(log2 e), one CTA per tag;
// fail[t] = 0 on success, 1 when h_t is not a unit (its words are then not written)
cudaError_t qf_launch_poly_tag_inverse(const int64_t* tags, int count, int n, const uint64_t* fq, const void* xr,
                                       int word_bytes, unsigned long long q, unsigned long long p, int lifts, void* tab,
                                       int* fail, cudaStream_t stream);
// u[b] += h_t * y_b mod (f, q) - H_0 y_b with y_b = G sigma[b][m_bar:], t = tidx[b], one CTA per target; h0_kind 0: H_0 = 0,
// 1: H_0 = I, 2: h0 (n x n column-major words).  An index outside [0, ntags) sets *flag |= QF_FLAG_TAG_INDEX and leaves
// the row as A sigma.
cudaError_t qf_launch_f_a_tag_poly(const int32_t* sigma, long lds, int m_bar, const int32_t* tidx, int ntags, const void* tab,
                                   const void* xr, const void* h0, int h0_kind, int word_bytes, const uint64_t* gpow,
                                   unsigned long long q, int n, int k, int B, int64_t* u, long ldu, int* flag,
                                   cudaStream_t stream);

// polynomial arithmetic of the ring short basis (setup.cu): P[2][2][n], Q[k][2][n]
cudaError_t qf_launch_ring_basis_polys(const int32_t* e, const int32_t* r, const int32_t* w, const int64_t* sk, int n, int k,
                                       int64_t* P, int64_t* Q, cudaStream_t stream);

// ---- ring_small.cu : register/shuffle NTT mod q for NTT-friendly primes q < 2^16 ----------------
#ifdef __cplusplus
#include <vector>
int qf_ring_small_plan(unsigned long long q, int n, int* d_out, std::vector<uint32_t>* tables, uint32_t* np_inv);
#endif
void qf_ring_small_key(const int64_t* a, int npoly, int n, int d, unsigned long long q, const uint32_t* tables,
                       uint32_t* a_hat);
cudaError_t qf_launch_ring_small(const int32_t* sigma, const uint32_t* a_hat, int64_t* out, unsigned long long* norm2,
                                 int B, int npoly, int n, int d, unsigned long long q, uint32_t np_inv,
                                 const uint32_t* tw, cudaStream_t stream, const int32_t* key_idx = nullptr, int nkeys = 0,
                                 int* flag = nullptr, const PackedRows* packed = nullptr);
// whether qf_launch_ring_small takes packed rows at degree n (the others decode first, qf_launch_domain_decode)
bool qf_ring_small_packed_fused(int n);
// qf_ring_small_key on the device for npolys polynomials (one warp each): bit-identical words
cudaError_t qf_launch_ring_small_key(const int64_t* a, uint32_t* a_hat, long npolys, int n, int d, unsigned long long q,
                                     const uint32_t* tw, cudaStream_t stream);
