/* qfall_b200.h -- C ABI of the B200 (sm_100a) backend for the batched PSF /
 * FIPS 203 hot path of qfall/tools.
 *
 * This is the drop-in boundary: every entry point replaces one method of the
 * reference's `PSF` trait (src/primitive/psf.rs:39-81) or of its
 * `LossyCompressionFIPS203` trait (src/compression/lossy_compression_fips203.rs:20-59)
 * for a BATCH of B targets.  A Rust shim converts qfall-math values to the
 * fixed-width buffers below (see INTEGRATION.md for the extern "C" block).
 *
 * Conventions
 *  - plain pointers and sizes only; all matrices row-major;
 *  - Range values (u, A, a_bar, tags ...) are residues in [0,q), q < 2^62, stored
 *    as int64 (the FLINT small-word form qfall-math holds them in);
 *  - Domain values (sigma, e, samp_d output) are int32 (|entry| <= s*r*sqrt(m));
 *  - a batch is "one row per target": sigma/e are B x m, u is B x n;
 *    ring values are B x (k+2) x n coefficients (coefficient embedding order,
 *    gpv_ring.rs:172-178);
 *  - every function returns a qf_status, never aborts; qf_last_error() gives text;
 *  - functions without a suffix take HOST pointers and synchronise before
 *    returning; `_dev` variants take DEVICE pointers, enqueue on the context's
 *    stream and do not synchronise;
 *  - one context per thread (or external locking): the reference types are
 *    neither Send nor Sync (gadget_parameters.rs:51).
 *  - samplers are keyed by (seed, first_index + row): a batch split across calls,
 *    chunks or GPUs yields the same preimages as one call.
 */
#ifndef QFALL_B200_H
#define QFALL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    QF_OK = 0,
    QF_ERR_INVALID = 1,       /* bad argument / shape (reference: panic or MathError) */
    QF_ERR_CUDA = 2,          /* CUDA runtime failure */
    QF_ERR_NOT_IN_DOMAIN = 3, /* f_a: some sigma fails check_domain (reference: assert!, gpv.rs:191) */
    QF_ERR_NO_KEY = 4,        /* key / trapdoor not installed */
    QF_ERR_UNSUPPORTED = 5,   /* parameter range outside this backend */
    QF_ERR_NUMERIC = 6        /* internal range check tripped (value did not fit) */
} qf_status;

typedef enum {
    QF_PSF_GPV = 0,          /* src/primitive/psf/gpv.rs */
    QF_PSF_PERTURBATION = 1, /* src/primitive/psf/mp_perturbation.rs */
    QF_PSF_GPV_RING = 2      /* src/primitive/psf/gpv_ring.rs */
} qf_psf_kind;

/* GadgetParameters / GadgetParametersRing (gadget_parameters.rs:44-52, 73-81) plus the
 * Gaussian parameters of the PSF struct (gpv.rs:54-57, mp_perturbation.rs:58-62,
 * gpv_ring.rs:63-67). */
typedef struct {
    int32_t kind;       /* qf_psf_kind */
    int64_t n;          /* security parameter / ring degree */
    int64_t k;          /* gadget length ceil(log_base q) */
    int64_t m_bar;      /* classical: columns of A_bar; ring: k + 2 */
    int64_t base;       /* gadget base */
    uint64_t q;         /* modulus, < 2^62 */
    double s;           /* Gaussian parameter s */
    double r;           /* rounding parameter r (perturbation only; 1 otherwise) */
    uint64_t norm_bound; /* floor of the check_domain bound (s^2 m [r^2]); 0 = derive from s, r */
} qf_params;

typedef struct qf_ctx qf_ctx;

/* ---- context ----------------------------------------------------------- */
qf_status qf_ctx_create(const qf_params* params, int device, qf_ctx** out);
void qf_ctx_destroy(qf_ctx* ctx);
const char* qf_last_error(const qf_ctx* ctx);
/* run on a caller-owned CUDA stream (cudaStream_t); NULL = the context's own stream */
qf_status qf_set_stream(qf_ctx* ctx, void* cuda_stream);
/* targets processed per internal chunk (bounds the workspace); 0 = default.  The default keeps the work matrices of
 * samp_p within ~32 GB of device memory (PSFGPV n = 256, q = 2^24: 37 888 targets = two waves of 148 SMs x 128 targets);
 * smaller chunks trade throughput for memory (one wave: -9 % at that size). */
qf_status qf_set_chunk(qf_ctx* ctx, int64_t targets_per_chunk);
qf_status qf_synchronize(qf_ctx* ctx);
/* number of kernels this context has launched so far */
uint64_t qf_launch_count(const qf_ctx* ctx);

/* Per-launch CUDA-event timing of the two contraction kernels on the context's stream: the fp64
 * DMMA contraction (gemm_*) and the tcgen05 int8 limb contraction (i8_*).  qf_profile_read
 * synchronises, returns the summed kernel time, the algorithmic operations (2*B*N*K per launch;
 * i8_issued_ops additionally counts every digit-pair product the tensor pipe executed) and the
 * launch counts, and resets the counters.  Any output pointer may be NULL. */
qf_status qf_profile(qf_ctx* ctx, int enable);
qf_status qf_profile_read(qf_ctx* ctx, double* gemm_ms, double* gemm_flops, uint64_t* gemm_launches, double* i8_ms,
                          double* i8_ops, double* i8_issued_ops, uint64_t* i8_launches);

/* ---- key material -------------------------------------------------------- */
/* A: n x m residues (PSFGPV / PSFPerturbation `A`, gpv.rs:60, mp_perturbation.rs:194) */
qf_status qf_set_a(qf_ctx* ctx, const int64_t* a);
/* PSFPerturbation trapdoor (mp_perturbation.rs:195): R m_bar x nk in {-1,0,1} (any small ints),
 * sqrt_sigma_2 m x m (any square root of Sigma_2; a lower-triangular one such as the Cholesky factor
 * compute_sqrt_sigma_2 returns costs half the work), and ONE k x k diagonal block of the gadget short basis
 * I_n (x) S_k with its GSO (gadget_classical.rs:248-287; the shim checks block-diagonality).
 * sqrt_sigma_2 == NULL: the backend derives its own square root of the DEFAULT covariance
 * Sigma = s^2 I (what PSFPerturbation::trap_gen builds, mp_perturbation.rs:227-231) from R, s, r on the
 * device, in block form (only an m_bar x m_bar Cholesky factor is dense) -- same law, ~4x less work per target.
 * Needs an installed A (QF_ERR_NO_KEY otherwise).  Tagged keys A = [A_bar | H G - A_bar R] (gadget_classical.rs:56-68) for
 * this R are recognised: A [R; I] = H G, so samp_p samples the gadget preimage of H^-1 (u - A p) mod q (H^-1 by
 * Gauss-Jordan with unit pivots on the device).  For H = I the sampler is the untagged one.  A key of this form whose H
 * has no unit pivot (singular H included) is QF_ERR_INVALID and no trapdoor is installed; a key of any other form is
 * installed as given. */
qf_status qf_set_trapdoor_perturbation(qf_ctx* ctx, const int8_t* r, const double* sqrt_sigma_2,
                                       const int64_t* s_block, const double* s_block_gso);
/* Switch the tag of the installed PSFPerturbation key without re-installing the trapdoor: A = [A_bar | H G - A_bar R]
 * becomes [A_bar | H' G - A_bar R], i.e. A[:, m_bar:] += (H' - H) G mod q, bit-identical to qf_trap_gen_from(A_bar, R, H').
 * tag: n x n (host), entries taken mod q; NULL means H' = I.  a_out: the new A, n x m (host), may be NULL.  R, sqrt(Sigma_2)
 * and the gadget basis stay installed; every device copy of A and H^-1 are replaced.  QF_ERR_INVALID on a context of
 * another kind, QF_ERR_NO_KEY without key and trapdoor, QF_ERR_INVALID when the installed key was not recognised as a
 * G-trapdoor for the installed R, and QF_ERR_INVALID for a tag H' without a unit pivot (the key and its tag then stay as
 * they were).  PSFGPV contexts switch tags with qf_gpv_set_tag. */
qf_status qf_set_tag(qf_ctx* ctx, const int64_t* tag, int64_t* a_out);
/* Switch the tag of the installed PSFGPV key without re-installing the trapdoor: A = [A_bar | H G - A_bar R] becomes
 * [A_bar | H' G - A_bar R] (A[:, m_bar:] += (H' - H) G mod q), bit-identical to qf_trap_gen_from(A_bar, R, H').  The GSO of
 * the short basis does not depend on the tag, so the fp64 matrices derived from it stay on the device; everything else is
 * what qf_set_a(A') + qf_set_trapdoor_gpv(S_H') builds.  tag: n x n (host), entries taken mod q; NULL means H' = I.
 * a_out: the new A, n x m (host), may be NULL.  s_out: the short basis for the installed R and H', m x m (host),
 * bit-identical to qf_gen_short_basis_tagged(R, H'), may be NULL.  Needs the two-phase recursion (a G-trapdoor key and its
 * basis from qf_gen_short_basis_tagged, dim above the tensor-core threshold): QF_ERR_INVALID otherwise, also without a key,
 * on a context of another kind, and for an H' without a unit pivot (nothing then changes).  Drops the f_a tag table and
 * keeps the samp_p tag table. */
qf_status qf_gpv_set_tag(qf_ctx* ctx, const int64_t* tag, int64_t* a_out, int64_t* s_out);
/* Tag table for samp_p with a tag per target (PSFPerturbation, and PSFGPV on the two-phase recursion): one trapdoor serves
 * the keys A_t = [A_bar | H_t G - A_bar R] of many tags in one batch (IBE key extraction, per-message tags).  tags:
 * ntags x n x n (host), entries taken mod q (negatives allowed), relative to the installed (A_bar, R); the installed key may
 * itself be tagged (any H_0).  H_t^-1 is computed on the device (Gauss-Jordan with unit pivots, as qf_set_tag).
 * QF_ERR_INVALID on a ring context, on a PSFGPV context whose key and trapdoor do not run the two-phase recursion (no key
 * included), for ntags < 1 or tags == NULL, when the installed PSFPerturbation key was not recognised as a G-trapdoor for
 * the installed R, and when a tag has no unit pivot (qf_last_error names its index; the previous table then stays);
 * QF_ERR_NO_KEY without PSFPerturbation key and trapdoor.  The table is dropped when a key or trapdoor is installed
 * (qf_set_a, qf_trap_gen, qf_trap_gen_from, qf_set_trapdoor_perturbation, qf_set_trapdoor_gpv) and kept by qf_set_tag and
 * qf_gpv_set_tag.  Device memory: ntags n^2 words of 4 bytes (q <= 2^32) or 8 bytes. */
qf_status qf_set_tag_table(qf_ctx* ctx, const int64_t* tags, int64_t ntags);
/* Tag table for f_a with a tag per target (PSFGPV and PSFPerturbation): for the installed key A = [A_bar | H_0 G - A_bar R]
 * and tags H_t, A_t := A + [0 | (H_t - H_0) G] is the key of tag t, [A_bar | H_t G - A_bar R].  tags: ntags x n x n, h0:
 * n x n (host; entries taken mod q, negatives allowed); h0 == NULL means H_0 = I, and H_0 = 0 (the base key
 * [A_bar | -A_bar R]) is allowed.  Needs no trapdoor and inverts nothing, so a verifier holding only A can install it and
 * singular tags are allowed; R is not known here, so A_t is defined by the formula and not checked against A_bar.  Stores
 * D_t = H_t - H_0 mod q on the device: ntags n^2 words of 4 bytes (q <= 2^32) or 8 bytes, plus 3 (ntags + 1) ints.
 * QF_ERR_INVALID on a ring context and for ntags < 1 or tags == NULL; QF_ERR_NO_KEY without a key.  The table is dropped
 * whenever A changes (qf_set_a, qf_trap_gen, qf_trap_gen_from, qf_set_tag, qf_gpv_set_tag) and is independent of
 * qf_set_tag_table. */
qf_status qf_set_f_a_tags(qf_ctx* ctx, const int64_t* tags, int64_t ntags, const int64_t* h0);
/* samp_p tag table in polynomial form: H_t = rot_f(h_t). f: n low coefficients of the monic modulus; tags: ntags x n.
 * f = X^n + sum_{i<n} f_i X^i, and column c of rot_f(h) holds the coefficients of h X^c mod f (for f = X^n + 1 that is
 * rot^-, rotation_matrix.rs:41-63).  Entries are taken mod q, negatives allowed.  The table then serves qf_samp_p_tagged[_dev]
 * exactly as qf_set_tag_table with the tags rot_f(h_t) would, bit for bit, but stores h_t^-1 mod (f, q) as n words per tag
 * and inverts each tag in O(n^2) on the device (extended Euclid mod p, Newton lifting to q = p^e).  It replaces the table
 * installed last, of either form; contexts, refusals and lifetime are those of qf_set_tag_table, and in addition:
 * QF_ERR_UNSUPPORTED when q is not a prime power or the kernels' shared memory exceeds one block's limit; QF_ERR_INVALID
 * when a tag is not a unit mod (f, q) (qf_last_error names its index; the previous table then stays).  For q = p^e a tag
 * is a unit exactly when rot_f(h_t) is invertible mod q, which is when qf_set_tag_table accepts it.  Device memory: ntags n
 * + n^2 words of 4 bytes (q <= 2^32) or 8 bytes. */
qf_status qf_set_tag_table_poly(qf_ctx* ctx, const int64_t* f, const int64_t* tags, int64_t ntags);
/* f_a tag table in polynomial form: A_t = A + [0 | (rot_f(h_t) - H_0) G]; h0: n x n matrix as in qf_set_f_a_tags (NULL = I).
 * f and tags as in qf_set_tag_table_poly.  qf_f_a_tagged[_dev] then give what qf_set_f_a_tags with the tags rot_f(h_t)
 * gives, bit for bit.  Inverts nothing: every q < 2^62, singular tags and H_0 = 0 work.  It replaces the f_a table
 * installed last, of either form; contexts, refusals and lifetime are those of qf_set_f_a_tags, and QF_ERR_UNSUPPORTED when
 * the kernel's shared memory exceeds one block's limit.  Device memory: ntags n + n^2 words (+ n^2 for a dense H_0). */
qf_status qf_set_f_a_tags_poly(qf_ctx* ctx, const int64_t* f, const int64_t* tags, int64_t ntags, const int64_t* h0);
/* gen_short_basis_for_trapdoor with tag = I (short_basis_classical.rs:54-110): the short basis
 * S_A = [[I,R],[0,I]] [[0,I],[S',W]] = [[R S', I + R W],[S', W]] of Lambda^perp(A) for the installed A and the
 * trapdoor R (m_bar x nk); W = digits of -A[:, :m_bar], S' column-reversed iff base^k = q.  The m_bar x nk x m_bar
 * product R W runs on the tensor cores; s_out is m x m (host), columns are the basis vectors.  Exact. */
qf_status qf_gen_short_basis(qf_ctx* ctx, const int8_t* r, int64_t* s_out);
/* gen_short_basis_for_trapdoor with a tag (short_basis_classical.rs:54-110): as qf_gen_short_basis for the installed
 * A = [A_bar | H G - A_bar R] with W = digits of -H^-1 A[:, :m_bar] mod q.  tag: n x n (host), entries taken mod q;
 * NULL means H = I (then identical to qf_gen_short_basis).  H^-1 is computed on the device by Gauss-Jordan with unit
 * pivots (first row at or below the diagonal whose entry is a unit mod q); QF_ERR_INVALID when no such pivot exists,
 * where the reference panics in MatZq::inverse.  Exact. */
qf_status qf_gen_short_basis_tagged(qf_ctx* ctx, const int8_t* r, const int64_t* tag, int64_t* s_out);
/* compute_sqrt_sigma_2 (mp_perturbation.rs:111-139) on the device: lower Cholesky factor (m x m, row-major, host)
 * of Sigma_2 = r^2/(2 pi) (Sigma - (b^2+1) [R;I][R;I]^t - I); sigma == NULL means Sigma = s^2 I.
 * QF_ERR_INVALID when Sigma_2 is not positive definite (the reference panics in the Cholesky). */
qf_status qf_compute_sqrt_sigma_2(qf_ctx* ctx, const int8_t* r, const double* sigma, double* sqrt_sigma_2_out);
/* PSFGPV trapdoor (gpv.rs:61): short basis S (dim x dim, columns are basis vectors) and its
 * GSO.  dim = m for QF_PSF_GPV, n*(k+2) (coefficient embedding) for QF_PSF_GPV_RING.
 * s_gso == NULL: the GSO is computed on the device (as qf_gso) and never leaves it.
 * G-trapdoor keys A = [A_bar | H G - A_bar R] with the basis of qf_gen_short_basis_tagged are recognised for the
 * identity tag and for any tag H invertible by unit pivoting: samp_p then runs the two-phase recursion on H^-1 A.  Drops
 * the samp_p tag table. */
qf_status qf_set_trapdoor_gpv(qf_ctx* ctx, const int64_t* s, const double* s_gso);
/* MatQ::gso as used at gpv.rs:91: unnormalised Gram-Schmidt of the columns of S (dim x dim) in fp64 on the
 * device (blocked Gram-Schmidt with re-orthogonalisation).  gso_out: dim x dim, host. */
qf_status qf_gso(qf_ctx* ctx, const int64_t* s, double* gso_out);
/* gen_short_basis_for_trapdoor_ring (short_basis_ring.rs:64-166) for the installed ring key and the trapdoor (r, e),
 * k x n small coefficients each, in the coefficient embedding: s_out is dim x dim (host), dim = n (k + 2), row =
 * polynomial row * n + coefficient, columns are the basis vectors.  Exact; feed it to qf_set_trapdoor_gpv. */
qf_status qf_ring_gen_short_basis(qf_ctx* ctx, const int32_t* r, const int32_t* e, int64_t* s_out);
/* ring key: (k+2) polynomials of n coefficients (gpv_ring.rs:70) */
qf_status qf_ring_set_a(qf_ctx* ctx, const int64_t* a);

/* ---- TrapGen (gadget_classical.rs:56-68, gadget_ring.rs:62-81) ------------ */
/* A = [A_bar | tag*G - A_bar*R] mod q from supplied A_bar (n x m_bar), R (m_bar x nk) and
 * tag (n x n, NULL = identity).  Bit-exact against the reference given the same inputs.
 * Writes A (n x m) and installs it as the context key. */
qf_status qf_trap_gen_from(qf_ctx* ctx, const int64_t* a_bar, const int8_t* r, const int64_t* tag, int64_t* a_out);
/* Samples A_bar uniform (gpv.rs:84) and R from PlusMinusOneZero (trapdoor_distribution.rs:82-86)
 * on the device (Philox, `seed`), then as qf_trap_gen_from with tag = I. */
qf_status qf_trap_gen(qf_ctx* ctx, uint64_t seed, int64_t* a_out, int8_t* r_out);
/* Ring: A = [1 | a_bar | g^t - (a_bar*r + e)] mod (X^n+1, q); r, e: k x n small coefficients. */
qf_status qf_ring_trap_gen_from(qf_ctx* ctx, const int64_t* a_bar, const int32_t* r, const int32_t* e,
                                int64_t* a_out);

/* ---- PSF::f_a / check_domain ------------------------------------------------ */
/* u[b] = A * sigma[b] mod q and in_domain[b] = check_domain(sigma[b])
 * (gpv.rs:190-193,219-224; mp_perturbation.rs:366-369,396-402; gpv_ring.rs:243-247,274-283).
 * qf_f_a (host pointers, synchronous) returns QF_ERR_NOT_IN_DOMAIN if any flag is 0 (u rows of such targets are
 * unspecified); the shim turns that into the reference's panic.  Its in_domain may be NULL.
 * qf_f_a_dev is asynchronous and therefore cannot return the verdict: it reports domain failures ONLY through
 * in_domain (device pointer, B bytes), which is mandatory -- NULL is QF_ERR_INVALID, so the assertion of gpv.rs:191
 * can never be dropped silently.  u_out may be NULL (flags only).
 * The squared norm is exact and saturating: entries of any int32 magnitude are handled (no 64-bit wrap-around). */
qf_status qf_f_a(qf_ctx* ctx, const int32_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain);
qf_status qf_f_a_dev(qf_ctx* ctx, const int32_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain);
qf_status qf_check_domain(qf_ctx* ctx, const int32_t* sigma, int64_t batch, uint8_t* in_domain);
/* f_a with a tag per target: u[b] = A_t sigma[b] mod q for t = tag_idx[b], the key of tag t of the table of
 * qf_set_f_a_tags; in_domain[b] = check_domain(sigma[b]), which does not depend on the tag.  u_out is mandatory.
 * qf_f_a_tagged takes host pointers and works as qf_f_a (in_domain may be NULL, QF_ERR_NOT_IN_DOMAIN when a flag is 0);
 * the tag indices are checked on the host before any launch (QF_ERR_INVALID outside [0, ntags)).  qf_f_a_tagged_dev takes
 * device pointers and works as qf_f_a_dev (asynchronous, in_domain mandatory): an index outside the table is never used
 * to address it, its row is unspecified and the next qf_synchronize returns QF_ERR_INVALID.  QF_ERR_NO_KEY without a
 * table, QF_ERR_INVALID on a ring context. */
qf_status qf_f_a_tagged(qf_ctx* ctx, const int32_t* sigma, const int32_t* tag_idx, int64_t batch, int64_t* u_out,
                        uint8_t* in_domain);
qf_status qf_f_a_tagged_dev(qf_ctx* ctx, const int32_t* sigma, const int32_t* tag_idx, int64_t batch, int64_t* u_out,
                            uint8_t* in_domain);

/* ---- ring f_a with a key per target (ring contexts only; QF_ERR_INVALID on a classical context), DESIGN 4.13 ----------
 * A ring public key is (k+2) polynomials of n coefficients, so every signer may hold their own: these calls verify one
 * batch across many keys, as PSF::f_a(&self, a, sigma) takes the key with every call (psf.rs:39-81, gpv_ring.rs:243-247).
 * Install a table of nkeys keys (host, nkeys x (k+2) x n residues in the layout of qf_ring_set_a).  Every coefficient is
 * checked to lie in [0, q) before anything changes: QF_ERR_INVALID names the first bad key and keeps the previous table.
 * QF_ERR_INVALID also for keys == NULL and nkeys outside [1, 2^31 - 1).  Keys need not have a_0 = 1 (f_a reads them only
 * as polynomials); no trapdoor and no installed key are needed, so a verifier-only context works.  The table is
 * independent of qf_ring_set_a (neither call drops the other's state), replaced by the next install and freed with the
 * context.  The keyed calls never use the dense tensor-core path of qf_f_a; the kernel family is chosen at install with
 * the rules of qf_ring_set_a and does not depend on an installed key.  Device memory per key: (k+2) n words of
 *   4 bytes  for primes q < 2^16 with n | q - 1, n a power of two in [64, 2048] (NTT mod q; not with QF_DISABLE_SMALL_NTT=1),
 *   8 bytes  otherwise, for n a power of two in [64, 2048] with (k+2) n (q/2) sqrt(norm bound) < 2^63 (Goldilocks NTT),
 *   8 bytes  for every other n and q (raw residues, schoolbook product);
 * C3 (n = 256, q = 3329, k = 12): 14 336 bytes per key. */
qf_status qf_ring_set_key_table(qf_ctx* ctx, const int64_t* keys, int64_t nkeys);
/* u[b] = sum_j a^(t)_j sigma[b][j] mod (X^n + 1, q) for t = key_idx[b], key t of the table, and in_domain[b] =
 * check_domain(sigma[b]).  For sigma[b] in the domain, row b is bit-identical to qf_f_a on the same context after
 * qf_ring_set_a(key t), for any split into calls and chunks; rows outside the domain have the unspecified u of qf_f_a.
 * u_out is mandatory.  qf_ring_f_a_keyed takes host pointers and works as qf_f_a_tagged: key indices are checked on the
 * host before any launch (QF_ERR_INVALID outside [0, nkeys)), in_domain may be NULL, QF_ERR_NOT_IN_DOMAIN when a flag is
 * 0.  qf_ring_f_a_keyed_dev takes device pointers and is asynchronous (in_domain mandatory): an index outside the table
 * is never used to address it, its row is unspecified and the next qf_synchronize returns QF_ERR_INVALID.  QF_ERR_NO_KEY
 * without a table.  An empty batch is valid.  For int16 or packed sigma, decode first (qf_domain_decode_dev). */
qf_status qf_ring_f_a_keyed(qf_ctx* ctx, const int32_t* sigma, const int32_t* key_idx, int64_t batch, int64_t* u_out,
                            uint8_t* in_domain);
qf_status qf_ring_f_a_keyed_dev(qf_ctx* ctx, const int32_t* sigma, const int32_t* key_idx, int64_t batch, int64_t* u_out,
                                uint8_t* in_domain);
/* count ring TrapGen keys at once (host pointers): a_bar count x n residues in [0, q) (QF_ERR_INVALID otherwise), r and e
 * count x k x n small coefficients; a_out count x (k+2) x n.  Key t is bit-identical to qf_ring_trap_gen_from(a_bar_t,
 * r_t, e_t).  Unlike that call it installs nothing: the context key, its trapdoor and the key table stay as they were.
 * The products a_bar_t r_{t,j} run as one keyed ring product (count k rows, one polynomial per key). */
qf_status qf_ring_trap_gen_batch_from(qf_ctx* ctx, int64_t count, const int64_t* a_bar, const int32_t* r, const int32_t* e,
                                      int64_t* a_out);

/* ---- PSF::samp_d (gpv.rs:113-116, mp_perturbation.rs:264-267, gpv_ring.rs:118-122) --- */
qf_status qf_samp_d(qf_ctx* ctx, int64_t batch, uint64_t seed, uint64_t first_index, int32_t* out);
qf_status qf_samp_d_dev(qf_ctx* ctx, int64_t batch, uint64_t seed, uint64_t first_index, int32_t* out);

/* ---- PSF::samp_p (gpv.rs:152-161, mp_perturbation.rs:304-336, gpv_ring.rs:160-212) --- */
/* e[b] with A e[b] = u[b] mod q, distributed as the reference's sampler. */
qf_status qf_samp_p(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first_index,
                    int32_t* e_out);
qf_status qf_samp_p_dev(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first_index,
                        int32_t* e_out);
/* samp_p with a tag per target: e[b] with A_t e[b] = u[b] mod q for t = tag_idx[b], the key of tag t of the installed tag
 * table (qf_set_tag_table).  For the same seed and first_index, row b is bit-identical to what qf_set_tag(H_t)
 * (PSFGPV: qf_gpv_set_tag(H_t)) followed by qf_samp_p gives for that row.  PSFGPV needs the two-phase recursion
 * (QF_ERR_INVALID otherwise, as for qf_set_tag_table).  qf_samp_p_tagged takes host pointers; targets are range-checked as in qf_samp_p and the
 * tag indices are checked on the host before any launch (QF_ERR_INVALID outside [0, ntags)).  qf_samp_p_tagged_dev takes
 * device pointers and is asynchronous: an index outside the table is not read, its row is unspecified and the next
 * qf_synchronize returns QF_ERR_INVALID.  QF_ERR_NO_KEY without a tag table; QF_ERR_INVALID on a ring context. */
qf_status qf_samp_p_tagged(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed,
                           uint64_t first_index, int32_t* e_out);
qf_status qf_samp_p_tagged_dev(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed,
                               uint64_t first_index, int32_t* e_out);
/* ---- offline / online samp_p (DESIGN 4.12): PSFPerturbation, and PSFGPV on the two-phase recursion -------------------
 * Most of samp_p does not read the target: the perturbation p and A p (PSFPerturbation), phase 1 of the recursion and the
 * products of its z2 (PSFGPV).  qf_samp_p_offline computes that half ahead of time into a device pool of the context; the
 * online calls then do only the target-dependent half.  Row b of an online call that consumed the pool entry of sampler
 * index j is bit-identical to row 0 of qf_samp_p(ctx, u_b, 1, seed, j, ...) (with tag_idx: of qf_samp_p_tagged), for any
 * split into fill calls, online calls and chunks.
 * Caller's responsibility: every entry is served at most once, but refilling an index range already used under the same
 * seed serves the same perturbations / phase-1 draws again -- exactly as calling qf_samp_p twice with one (seed, index).
 * Two preimages that share such a draw leak information about the trapdoor through their difference.
 * Lifetime: one pool per context.  It is dropped by every call that changes A or the trapdoor (qf_set_a, qf_trap_gen,
 * qf_trap_gen_from, qf_set_trapdoor_perturbation, qf_set_trapdoor_gpv, qf_set_tag, qf_gpv_set_tag) and kept by the tag
 * table installs of either form (samp_p and f_a).
 * Device memory per entry: PSFPerturbation 4 m + 8 n bytes (p as int32, A p mod q); PSFGPV 4 m_bar + 8 n + 8 n k bytes
 * (z2 as int32, A_bar z2 mod q, the centre product Mt_1 z2 in fp64). */
/* Fill the pool with the target-independent half of samp_p for the sampler indices first_index .. first_index + count - 1
 * under `seed`; replaces any previous pool (also when the fill fails: there is then no pool).  Synchronous.
 * QF_ERR_UNSUPPORTED on a ring context and on a PSFGPV key that runs the one-pass recursion (its first step, A_P^-1 u,
 * reads the target); QF_ERR_NO_KEY without key or trapdoor; QF_ERR_INVALID for count < 0; QF_ERR_CUDA when the pool does
 * not fit in device memory (nothing is launched). */
qf_status qf_samp_p_offline(qf_ctx* ctx, int64_t count, uint64_t seed, uint64_t first_index);
/* Entries not yet consumed, and the sampler index the next online call starts at (0 and 0 without a pool).  Either
 * pointer may be NULL. */
qf_status qf_samp_p_pool_info(const qf_ctx* ctx, int64_t* remaining, uint64_t* next_index);
/* Consume the next `batch` entries of the pool, in index order, for the targets u (batch x n).  tag_idx == NULL: as
 * qf_samp_p; otherwise as qf_samp_p_tagged (same readiness checks and tag-index checks).  first_index_out (may be NULL)
 * receives the sampler index of row 0.  QF_ERR_NO_KEY without a pool; QF_ERR_INVALID when batch exceeds the remaining
 * entries, before any launch and with nothing consumed.  batch == 0 is valid.  Once the checks pass the entries are
 * consumed, even if the call fails later.  qf_samp_p_online takes host pointers and range-checks the targets as qf_samp_p;
 * qf_samp_p_online_dev takes device pointers and is asynchronous like the other _dev forms (its entries are consumed at
 * enqueue). */
qf_status qf_samp_p_online(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, int32_t* e_out,
                           uint64_t* first_index_out);
qf_status qf_samp_p_online_dev(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, int32_t* e_out,
                               uint64_t* first_index_out);
/* Narrow Domain form: the same preimages as int16 -- |e_i| <= 6 s r is far below 2^15 for the parameter sets of the
 * reference (C2: 6 s = 8568; C3: 3135), so the device->host copy, which bounds the host-buffer path, is halved.  An entry
 * that does not fit is reported as QF_ERR_NUMERIC (then use qf_samp_p).  Targets outside [0,q) are detected on the device
 * (both variants) and reported as QF_ERR_INVALID when the call returns. */
qf_status qf_samp_p_i16(qf_ctx* ctx, const int64_t* u, int64_t batch, uint64_t seed, uint64_t first_index,
                        int16_t* e_out);
/* f_a / check_domain on int16 Domain values (host pointers; otherwise as qf_f_a). */
qf_status qf_f_a_i16(qf_ctx* ctx, const int16_t* sigma, int64_t batch, int64_t* u_out, uint8_t* in_domain);
/* int32 -> int16 on the device (e.g. before the final gather of results over NVLink); *overflow (device int, zeroed by
 * the caller) gets bit 64 set when a value does not fit.  in / out 16-byte aligned. */
qf_status qf_narrow_i32_i16_dev(const int32_t* in, int16_t* out, size_t count, int* overflow, void* cuda_stream);

/* ---- packed Domain values: a lossless Golomb-Rice code of preimages (DESIGN 4.11) ---------------------------------------
 * Entries of a preimage are close to D_{Z,w} (w = s, or s r for PSFPerturbation), about 11 bits of entropy at n = 256,
 * q = 2^24; this code stores them in about 11.3 bits instead of int16's 16, for any int32 value but INT32_MIN.
 * Format.  One row x_0 .. x_{dim-1} (dim = m, or n (k+2) for the ring) is stored in a slot of slot_bytes bytes, a multiple
 * of 16.  Streams are LSB-first: bit j is bit j % 8 of byte j / 8.  Parameter k, 0 <= k <= 30; for each entry a = |x_i|,
 * h_i = floor(a / 2^k), sign = (x_i < 0).
 *  1. Fixed part: entry i is the (k+1)-bit field (a mod 2^k) | sign << k at bit offset i (k+1); it ends at byte
 *     H0 = 16 ceil(dim (k+1) / 128); bits dim (k+1) .. 8 H0 - 1 are zero.
 *  2. High stream from byte H0: for i = 0 .. dim-1 in order, h_i zero bits and then one 1 bit; every bit after the
 *     dim-th 1 bit, to the end of the slot, is zero.
 *  3. Length: nbytes = H0 + ceil(sum_i (h_i + 1) / 8).  A caller may keep the first nbytes bytes and pad with zeros to
 *     read the row back.
 * Canonical form: the decoder rejects a row with an entry of sign 1 and magnitude 0, fewer than dim 1 bits in the high
 * stream, a non-zero padding bit (fixed part or tail), or a magnitude above INT32_MAX.  Every other slot decodes to exactly
 * one row, and encoding that row gives the same bytes back.
 * Overflow: a row whose code does not fit its slot, or that holds INT32_MIN, gets nbytes = -1 and an all-zero slot; the
 * other rows are written and the call returns QF_ERR_NUMERIC.  Samplers are keyed by (seed, index), so qf_samp_p (or
 * qf_samp_p_tagged) with first_index + b and batch 1 returns the int32 preimage of an overflowed row b: nothing is lost.
 * Argument errors are QF_ERR_INVALID before any launch: k outside [0, 30], slot_bytes not a multiple of 16 or below
 * H0 + ceil(dim / 8), NULL pointers. */
/* Recommended parameters for the context's width w and dim: k minimises E[k + 2 + h] for X ~ D_{Z,w} (summed over
 * |x| <= 20 w); slot_bytes = H0 + ceil((dim E[h+1] + 12 sqrt(dim Var[h+1])) / 8), rounded up to 16 (n = 256, q = 2^24
 * PSFGPV: k = 8, 17 696 bytes against 24 704 as int16). */
qf_status qf_domain_code_params(qf_ctx* ctx, int* k, int64_t* slot_bytes);
/* samp_p with packed output (host pointers): out is batch x slot_bytes, nbytes batch lengths.  Row b is byte-identical to
 * the code of row b of qf_samp_p (tag_idx == NULL) or qf_samp_p_tagged (tag_idx: host, as there: same contexts, readiness
 * checks, and indices checked before any launch) for the same seed and first_index.  All three PSF kinds. */
qf_status qf_samp_p_packed(qf_ctx* ctx, const int64_t* u, const int32_t* tag_idx, int64_t batch, uint64_t seed,
                           uint64_t first_index, int k, int64_t slot_bytes, uint8_t* out, int32_t* nbytes);
/* f_a / check_domain on packed Domain values (host pointers): the slots are decoded on the device, then f_a as qf_f_a
 * (tag_idx == NULL) or qf_f_a_tagged (tag_idx: classical contexts, as there).  in_domain[b] = check_domain(sigma[b]) AND
 * slot b is canonical; any 0 gives QF_ERR_NOT_IN_DOMAIN -- a malformed encoding is a rejected signature, not an error of
 * the call.  u_out may be NULL (flags only), in_domain too. */
qf_status qf_f_a_packed(qf_ctx* ctx, const uint8_t* packed, const int32_t* tag_idx, int64_t batch, int k, int64_t slot_bytes,
                        int64_t* u_out, uint8_t* in_domain);
/* Context-free device forms (asynchronous on cuda_stream, NULL = default stream): encode rows x dim int32 into rows slots
 * (nbytes: rows lengths, -1 on overflow -- reported only there), and decode slots into int32 rows with ok[row] = 1 iff the
 * slot is canonical (a rejected row's values are unspecified).  Slots (out / in) 16-byte aligned, int32 rows 4-byte
 * aligned, else QF_ERR_INVALID. */
qf_status qf_domain_encode_dev(const int32_t* in, int64_t rows, int64_t dim, int k, int64_t slot_bytes, uint8_t* out,
                               int32_t* nbytes, void* cuda_stream);
qf_status qf_domain_decode_dev(const uint8_t* in, int64_t rows, int64_t dim, int k, int64_t slot_bytes, int32_t* out,
                               uint8_t* ok, void* cuda_stream);

/* ---- PSFPerturbation::randomized_nearest_plane_gadget (mp_perturbation.rs:173-191), the public helper samp_p calls:
 * z[b] = x0 + SampleD(S, S~, -x0, r sqrt(base^2 + 1)) with x0 = find_solution_gadget_mat(v[b]) -- a preimage of v[b]
 * under the gadget matrix G, Gaussian over the coset Lambda_v^perp(G).  v: B x n residues, z_out: B x (n k).  The gadget
 * short basis (and its GSO) is the one installed with qf_set_trapdoor_perturbation.  Host pointers. */
qf_status qf_randomized_nearest_plane_gadget(qf_ctx* ctx, const int64_t* v, int64_t batch, uint64_t seed,
                                             uint64_t first_index, int32_t* z_out);

/* ---- LossyCompressionFIPS203 (lossy_compression_fips203.rs:89-114, 143-172) ----------- */
/* Flat coefficient streams (a polynomial / matrix of polynomials is just `count` coefficients).
 * u16 variants: q < 2^16, 1 <= d <= 16; device_ptrs != 0 -> in/out are device pointers and the
 * call is asynchronous on `cuda_stream` (may be NULL = default stream). */
qf_status qf_compress_u16(const uint16_t* in, uint16_t* out, size_t count, uint32_t q, uint32_t d,
                          int device_ptrs, void* cuda_stream);
qf_status qf_decompress_u16(const uint16_t* in, uint16_t* out, size_t count, uint32_t q, uint32_t d,
                            int device_ptrs, void* cuda_stream);
/* FLINT-word variants, any q < 2^62, 1 <= d <= 62. */
qf_status qf_compress_i64(const int64_t* in, int64_t* out, size_t count, uint64_t q, uint32_t d,
                          int device_ptrs, void* cuda_stream);
qf_status qf_decompress_i64(const int64_t* in, int64_t* out, size_t count, uint64_t q, uint32_t d,
                            int device_ptrs, void* cuda_stream);

/* ---- FIPS 203 ByteEncode_d / ByteDecode_d fused with Compress_d / Decompress_d (SURVEY 8f rank 4: the step after
 * `lossy_compress` in ML-KEM; the reference stops at the unpacked polynomial, lossy_compression_fips203.rs:62,99-113).
 * Polynomials of degree 256: `in` holds npoly x 256 u16 coefficients, the packed form npoly x 32 d bytes (FIPS 203
 * Algorithm 5: coefficient i supplies stream bits [i d, (i+1) d), bit k of the stream = bit k % 8 of byte k / 8).
 * 1 <= d <= 12, q < 2^16.  compress != 0: ByteEncode_d(Compress_d(x)), else ByteEncode_d(x) (d = 12: x < q).
 * decompress != 0: Decompress_d(ByteDecode_d(b)), else ByteDecode_d(b) (d = 12: reduced mod q, Algorithm 6). */
qf_status qf_compress_encode_u16(const uint16_t* in, uint8_t* out, size_t npoly, uint32_t q, uint32_t d, int compress,
                                 int device_ptrs, void* cuda_stream);
qf_status qf_decode_decompress_u16(const uint8_t* in, uint16_t* out, size_t npoly, uint32_t q, uint32_t d, int decompress,
                                   int device_ptrs, void* cuda_stream);

/* ---- message encodings (src/utils/common_encodings.rs, SURVEY 8f rank 4), batched ------------------------------------
 * encode_value_in_polynomialringzq (:49-92): digit d of the value w.r.t. `base` -> coefficient d * floor(q / base);
 * decode_value_from_polynomialringzq (:125-153): coefficient c (any representative) -> digit
 * floor((c * base + floor(q / (2 base))) / q) mod base.  A batch is a flat stream of `count` digits, one byte each
 * (2 <= base <= 256); coefficients are coeff_bytes wide: 2 (u16, q < 2^16) or 8 (FLINT words, q < 2^62).  The big-integer
 * <-> digit-string conversion of the reference's `value: Z` stays with the caller (one value = up to n digits, padded
 * with zeros).  base < 2 is QF_ERR_INVALID (the reference returns MathError::InvalidIntegerInput).  device_ptrs != 0:
 * device pointers, asynchronous on cuda_stream. */
qf_status qf_encode_digits(const uint8_t* digits, void* coeffs, size_t count, uint64_t q, uint32_t base, int coeff_bytes,
                           int device_ptrs, void* cuda_stream);
qf_status qf_decode_digits(const void* coeffs, uint8_t* digits, size_t count, uint64_t q, uint32_t base, int coeff_bytes,
                           int device_ptrs, void* cuda_stream);
/* base 2 with bit-packed messages (bit j of byte i = coefficient 8 i + j; a 32-byte message <-> 256 u16 coefficients, the
 * mu -> floor(q/2) mu map of the lib.rs example :28-36): nbytes message bytes <-> 8 nbytes coefficients, q < 2^16. */
qf_status qf_encode_bits_u16(const uint8_t* msg, uint16_t* coeffs, size_t nbytes, uint32_t q, int device_ptrs, void* cuda_stream);
qf_status qf_decode_bits_u16(const uint16_t* coeffs, uint8_t* msg, size_t nbytes, uint32_t q, int device_ptrs, void* cuda_stream);

/* ---- Z::sample_discrete_gauss for a batch of (centre) values (qfall-math SampleZ as used at
 * gpv.rs:115 and inside sample_d_precomputed_gso): out[i] <- D_{Z, s, centers[i]}. Host pointers, any count.
 * Value i draws from its own Philox stream (seed, i) under a stream id that no PSF method uses, so equal seeds
 * here and in qf_samp_d give independent outputs.  s < 2e6 (QF_ERR_UNSUPPORTED above); a NaN / infinite centre
 * gives QF_ERR_NUMERIC. */
qf_status qf_sample_z(const double* centers, size_t count, double s, uint64_t seed, int64_t* out);

/* ---- self-test of the tensor-core integer contraction: out = X W^t (mod q if q != 0), exact.
 * x: B x K signed with |x| < 2^(8 LX - 1); w: N x K, residues < 2^(8 LW) (w_signed = 0) or signed
 * |w| < 2^(8 LW - 1) (w_signed = 1).  Host pointers. */
qf_status qf_debug_gemm_i8(const int64_t* x, const int64_t* w, int w_signed, int LX, int LW, int64_t B, int64_t N,
                           int64_t K, uint64_t q, int64_t* out);

/* ---- measured ceiling of the int8 tensor pipe (roofline denominator of the limb contractions; SURVEY 8d: "measure a plain
 * int8 tcgen05 GEMM probe once and use it"): a one-digit-pair B x N x K contraction on random bytes (128 x 256 tiles, K a
 * multiple of 128, <= 65536), `iters` launches timed one by one -> best_tops (burst), then back to back for sustain_ms ->
 * sustained_tops.  TOP/s = 2 B N K / time.  pipe_tops (optional): the tensor pipe on its own -- every SM repeats the MMAs of
 * one shared-memory-resident 128 x 256 x 128 block (no operand traffic), i.e. the rate at 100 % pipe activity; the GEMM probe
 * sits below it because a cta_group::1 tiling is bound by the L2 -> shared-memory operand feed.  Allocates its own buffers. */
qf_status qf_probe_i8_peak(int device, int64_t B, int64_t N, int64_t K, int iters, double sustain_ms, double* best_tops,
                           double* sustained_tops, double* pipe_tops);

/* ---- synthetic inputs for benchmarks (Philox, on device) -------------------------------- */
qf_status qf_fill_uniform_modq_dev(int64_t* out, size_t count, uint64_t q, uint64_t seed, void* cuda_stream);

/* library / build identification */
const char* qf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* QFALL_B200_H */
