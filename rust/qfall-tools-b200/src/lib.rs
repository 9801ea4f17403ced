//! B200 (sm_100a) backend for the batched PSF / FIPS 203 hot path of qfall-tools, behind the reference's own traits.
//!
//! * [`PSFGPVB200`] implements `qfall_tools::primitive::psf::PSF` (src/primitive/psf.rs:39-81) with the associated types
//!   of `PSFGPV` (gpv.rs:59-63), one target per call exactly like the reference, plus [`PSFBatch`] -- the extension the
//!   reference lacks because its methods reject multi-column inputs (gpv.rs:221, pinned by gpv.rs:287-298).
//! * [`PSFPerturbationB200`] (perturbation.rs) and [`PSFGPVRingB200`] (ring.rs) do the same for `PSFPerturbation`
//!   (mp_perturbation.rs:193-197) and `PSFGPVRing` (gpv_ring.rs:69-73).
//! * [`PSFBatch::samp_p_batch_packed`] / [`PSFBatch::f_a_batch_packed`] move preimages in the packed Domain code
//!   ([`PackedDomain`], DESIGN 4.11): about 0.71 of the int16 bytes at n = 256, q = 2^24.
//! * [`PolynomialRingZqB200`] / [`MatPolynomialRingZqB200`] (compression.rs) implement `LossyCompressionFIPS203`
//!   (lossy_compression_fips203.rs:20-59) over [`compress_words`] / [`decompress_words`], which run `Compress_d` /
//!   `Decompress_d` (:101-111, :159-169) for a whole coefficient vector at once.
//!
//! Values cross the boundary as fixed-width words: Range / key entries are residues in [0, q), q < 2^62 (`i64`), Domain
//! entries are `i32`.  Every C entry point returns a status; a non-zero status is turned into the panic (or the
//! `MathError`) the reference raises at the same place.
//!
//! This crate is shipped as SOURCE: the image the backend is built in has no Rust toolchain, so it has not been
//! compiled there.  The `extern "C"` block (ffi.rs) is checked mechanically against include/qfall_b200.h.
pub mod compression;
pub mod ffi;
pub mod perturbation;
pub mod ring;
pub use compression::{MatPolynomialRingZqB200, PolynomialRingZqB200};
pub use perturbation::PSFPerturbationB200;
pub use ring::PSFGPVRingB200;

use ffi::*;
use qfall_math::{
    integer::{MatZ, Z},
    integer_mod_q::MatZq,
    rational::{MatQ, Q},
    traits::{MatrixDimensions, MatrixGetEntry, MatrixSetEntry},
};
use qfall_tools::primitive::psf::{PSF, PSFGPV};
use std::cell::RefCell;
use std::ffi::CStr;

/// Owner of one `qf_ctx` (device memory, stream, installed key).  Neither `Send` nor `Sync`, like the reference's PSF
/// structs (gadget_parameters.rs:51): one caller thread per instance.
pub struct Context {
    pub(crate) raw: *mut qf_ctx,
}

impl Context {
    pub fn new(params: &qf_params, device: i32) -> Result<Self, String> {
        let mut raw: *mut qf_ctx = std::ptr::null_mut();
        let st = unsafe { qf_ctx_create(params, device, &mut raw) };
        if st != QF_OK || raw.is_null() {
            return Err(format!("qf_ctx_create failed with status {st}"));
        }
        Ok(Context { raw })
    }
    fn last_error(&self) -> String {
        unsafe { CStr::from_ptr(qf_last_error(self.raw)) }.to_string_lossy().into_owned()
    }
    /// status -> the reference's failure mode at that call site (`unwrap()` / `assert!`)
    pub(crate) fn check(&self, st: i32, what: &str) {
        assert!(st == QF_OK, "{what}: status {st}: {}", self.last_error());
    }
}

impl Drop for Context {
    fn drop(&mut self) {
        unsafe { qf_ctx_destroy(self.raw) }
    }
}

// ---- value conversion ------------------------------------------------------------------------------------------

/// Residues of a `MatZq` (least non-negative representatives), row-major.
pub fn matzq_to_words(m: &MatZq) -> Vec<i64> {
    let (rows, cols) = (m.get_num_rows(), m.get_num_columns());
    let mut out = Vec::with_capacity((rows * cols) as usize);
    for i in 0..rows {
        for j in 0..cols {
            let z: Z = m.get_entry(i, j).unwrap();
            out.push(i64::try_from(&z).expect("modulus below 2^62"));
        }
    }
    out
}

/// Entries of a `MatZ`, row-major.
pub fn matz_to_words(m: &MatZ) -> Vec<i64> {
    let (rows, cols) = (m.get_num_rows(), m.get_num_columns());
    let mut out = Vec::with_capacity((rows * cols) as usize);
    for i in 0..rows {
        for j in 0..cols {
            let z: Z = m.get_entry(i, j).unwrap();
            out.push(i64::try_from(&z).expect("entry below 2^63"));
        }
    }
    out
}

/// A Domain value (column vector) as `i32`; `None` when an entry does not fit -- such a vector is far outside D_n.
pub fn domain_to_i32(sigma: &MatZ) -> Option<Vec<i32>> {
    matz_to_words(sigma).into_iter().map(|v| i32::try_from(v).ok()).collect()
}

pub fn column_from_i32(e: &[i32]) -> MatZ {
    let mut out = MatZ::new(e.len() as i64, 1);
    for (i, v) in e.iter().enumerate() {
        out.set_entry(i as i64, 0, Z::from(*v as i64)).unwrap();
    }
    out
}

pub fn range_from_words(u: &[i64], q: &Z) -> MatZq {
    let mut out = MatZq::new(u.len() as i64, 1, q);
    for (i, v) in u.iter().enumerate() {
        out.set_entry(i as i64, 0, Z::from(*v)).unwrap();
    }
    out
}

fn matq_to_f64(m: &MatQ) -> Vec<f64> {
    let (rows, cols) = (m.get_num_rows(), m.get_num_columns());
    let mut out = Vec::with_capacity((rows * cols) as usize);
    for i in 0..rows {
        for j in 0..cols {
            let x: Q = m.get_entry(i, j).unwrap();
            out.push(f64::from(&x));
        }
    }
    out
}

// ---- the batch extension -----------------------------------------------------------------------------------------

/// Batched `samp_p` / `f_a` next to the unchanged trait: targets are independent given the key, samplers are keyed by
/// `(seed, first_index + position)`, so a batch split across calls or GPUs gives the same preimages as one call.
pub trait PSFBatch: PSF {
    fn samp_p_batch(&self, a: &Self::A, td: &Self::Trapdoor, us: &[Self::Range], seed: u64, first_index: u64) -> Vec<Self::Domain>;
    fn f_a_batch(&self, a: &Self::A, sigmas: &[Self::Domain]) -> Vec<Self::Range>;
    /// `samp_p_batch` with every preimage in the packed Domain code (qf_samp_p_packed, DESIGN 4.11) at the parameters of
    /// qf_domain_code_params, each row trimmed to its length.  Row b is the code of `samp_p_batch(..)[b]` for the same
    /// seed and first_index.  Panics when a row does not fit its slot (qf_samp_p_packed: QF_ERR_NUMERIC; `samp_p_batch`
    /// at `first_index + b` gives that preimage).
    fn samp_p_batch_packed(&self, a: &Self::A, td: &Self::Trapdoor, us: &[Self::Range], seed: u64, first_index: u64) -> PackedDomain;
    /// `f_a_batch` on packed preimages (qf_f_a_packed): panics like `f_a` when a sigma is outside D_n or its code is not
    /// canonical.
    fn f_a_batch_packed(&self, a: &Self::A, packed: &PackedDomain) -> Vec<Self::Range>;
}

/// Preimages in the packed Domain code (include/qfall_b200.h, DESIGN 4.11): code parameter `k`, slot size, and one code
/// per target trimmed to its length (zero padding up to `slot_bytes` reads it back).
#[derive(Clone, Debug, PartialEq, Eq)]
pub struct PackedDomain {
    pub k: i32,
    pub slot_bytes: i64,
    pub rows: Vec<Vec<u8>>,
}

/// qf_samp_p_packed for the targets `uw` (batch x n words) with the key and trapdoor installed in `ctx`.
/// Online half of samp_p from the context's pool (qf_samp_p_online, DESIGN 4.12): `batch` rows of `m` entries and the
/// sampler index of row 0.  `tag_idx`: one index per target into the installed tag table (qf_samp_p_tagged).
pub(crate) fn samp_p_online_run(ctx: &Context, uw: &[i64], tag_idx: Option<&[i32]>, batch: usize, m: usize) -> (Vec<i32>, u64) {
    let mut e = vec![0i32; batch * m];
    let mut first = 0u64;
    let ti = tag_idx.map(|t| t.as_ptr()).unwrap_or(std::ptr::null());
    let st = unsafe { qf_samp_p_online(ctx.raw, uw.as_ptr(), ti, batch as i64, e.as_mut_ptr(), &mut first) };
    ctx.check(st, "qf_samp_p_online");
    (e, first)
}

/// Remaining entries of the context's pool and the sampler index of the next one (qf_samp_p_pool_info).
pub fn samp_p_pool_info(ctx: &Context) -> (i64, u64) {
    let (mut rem, mut next) = (0i64, 0u64);
    ctx.check(unsafe { qf_samp_p_pool_info(ctx.raw, &mut rem, &mut next) }, "qf_samp_p_pool_info");
    (rem, next)
}

pub(crate) fn samp_p_packed_run(ctx: &Context, uw: &[i64], batch: usize, seed: u64, first_index: u64) -> PackedDomain {
    let (mut k, mut slot) = (0i32, 0i64);
    ctx.check(unsafe { qf_domain_code_params(ctx.raw, &mut k, &mut slot) }, "qf_domain_code_params");
    let mut out = vec![0u8; batch * slot as usize];
    let mut nbytes = vec![0i32; batch];
    let st = unsafe {
        qf_samp_p_packed(ctx.raw, uw.as_ptr(), std::ptr::null(), batch as i64, seed, first_index, k, slot, out.as_mut_ptr(),
                         nbytes.as_mut_ptr())
    };
    ctx.check(st, "qf_samp_p_packed");
    let rows = out.chunks(slot as usize).zip(&nbytes).map(|(row, nb)| row[..*nb as usize].to_vec()).collect();
    PackedDomain { k, slot_bytes: slot, rows }
}

/// qf_f_a_packed against the key installed in `ctx`: u words (batch x n).
pub(crate) fn f_a_packed_run(ctx: &Context, n: usize, packed: &PackedDomain) -> Vec<i64> {
    let slot = packed.slot_bytes as usize;
    let mut buf = vec![0u8; packed.rows.len() * slot];
    for (dst, row) in buf.chunks_mut(slot).zip(&packed.rows) {
        assert!(row.len() <= slot, "a packed row is longer than its slot");
        dst[..row.len()].copy_from_slice(row);
    }
    let b = packed.rows.len();
    let mut u = vec![0i64; b * n];
    let mut ok = vec![0u8; b];
    let st = unsafe {
        qf_f_a_packed(ctx.raw, buf.as_ptr(), std::ptr::null(), b as i64, packed.k, packed.slot_bytes, u.as_mut_ptr(), ok.as_mut_ptr())
    };
    assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n"); // gpv.rs:191
    ctx.check(st, "qf_f_a_packed");
    u
}

// ---- PSFGPV ------------------------------------------------------------------------------------------------------

/// `PSFGPV` (gpv.rs:53-57) evaluated on the GPU.  `inner` keeps the reference struct (parameters, serde), `ctx` the
/// device context; the key and trapdoor most recently used are cached on the device.
pub struct PSFGPVB200 {
    pub inner: PSFGPV,
    ctx: Context,
    installed: RefCell<Option<(Vec<i64>, Vec<i64>)>>, // (A, S) words of the installed key
    /// number of tags in the samp_p tag table on the device (qf_set_tag_table); the device drops it with every key or
    /// trapdoor install and keeps it across set_tag
    installed_tags: RefCell<Option<usize>>,
    fa_tags: FaTags,
    seed: RefCell<u64>,
}

impl PSFGPVB200 {
    pub fn new(inner: PSFGPV, device: i32, seed: u64) -> Result<Self, String> {
        let gp = &inner.gp;
        let params = qf_params {
            kind: QF_PSF_GPV,
            n: i64::try_from(&gp.n).unwrap(),
            k: i64::try_from(&gp.k).unwrap(),
            m_bar: i64::try_from(&gp.m_bar).unwrap(),
            base: i64::try_from(&gp.base).unwrap(),
            q: u64::try_from(&Z::from(&gp.q)).map_err(|_| "modulus must be below 2^62".to_string())?,
            s: f64::from(&inner.s),
            r: 1.0,
            // gpv.rs:223: ||sigma||^2 <= s^2 * m, compared exactly (floor of the exact rational; 0 would make the
            // backend derive it from the f64-rounded s)
            norm_bound: ring::floor_u64(&(&inner.s * &inner.s * Q::from(i64::try_from(&(&gp.m_bar + &gp.n * &gp.k)).unwrap()))),
        };
        Ok(PSFGPVB200 {
            inner,
            ctx: Context::new(&params, device)?,
            installed: RefCell::new(None),
            installed_tags: RefCell::new(None),
            fa_tags: RefCell::new(None),
            seed: RefCell::new(seed),
        })
    }
    fn n(&self) -> usize {
        i64::try_from(&self.inner.gp.n).unwrap() as usize
    }
    fn m(&self) -> usize {
        (i64::try_from(&self.inner.gp.m_bar).unwrap() + i64::try_from(&self.inner.gp.n).unwrap() * i64::try_from(&self.inner.gp.k).unwrap()) as usize
    }
    /// a fresh sampler seed per call (the reference draws from its thread RNG; no seed API, SURVEY finding 1)
    fn next_seed(&self) -> u64 {
        let mut s = self.seed.borrow_mut();
        *s = s.wrapping_mul(6364136223846793005).wrapping_add(1442695040888963407);
        *s
    }
    /// qf_set_a + qf_set_trapdoor_gpv, skipped when the same key is already on the device
    fn install(&self, a: &MatZq, td: &(MatZ, MatQ)) {
        let (aw, sw) = (matzq_to_words(a), matz_to_words(&td.0));
        if let Some((a0, s0)) = self.installed.borrow().as_ref() {
            if *a0 == aw && *s0 == sw {
                return;
            }
        }
        self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
        *self.fa_tags.borrow_mut() = None;
        let gso = matq_to_f64(&td.1);
        self.ctx.check(unsafe { qf_set_trapdoor_gpv(self.ctx.raw, sw.as_ptr(), gso.as_ptr()) }, "qf_set_trapdoor_gpv");
        *self.installed.borrow_mut() = Some((aw, sw));
        *self.installed_tags.borrow_mut() = None;
    }

    /// Tag switch without a new trapdoor install, for a key `a = [A_bar | H G - A_bar R]` (gen_trapdoor with a tag,
    /// gadget_classical.rs:56-68) and its trapdoor `td = (S_H, GSO)` on the two-phase recursion: returns
    /// `(a', (S_H', td.1))` with `a' = [A_bar | H' G - A_bar R]` for `tag` = H' (equal to gen_trapdoor(A_bar, R, H')) and
    /// `S_H'` equal to gen_short_basis_for_trapdoor(H', a', R).  The GSO does not depend on the tag, so it is kept and
    /// nothing is re-installed: the pair is recorded as the installed key (qf_gpv_set_tag).  The samp_p tag table stays;
    /// the f_a tag table is dropped.  Panics off the two-phase recursion and when H' has no unit pivot (the reference
    /// panics in `MatZq::inverse`).
    pub fn set_tag(&self, a: &MatZq, td: &(MatZ, MatQ), tag: &MatZq) -> (MatZq, (MatZ, MatQ)) {
        let (n, m) = (self.n(), self.m());
        assert_eq!((tag.get_num_rows(), tag.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
        self.install(a, td);
        let tw = matzq_to_words(tag);
        let mut aw = vec![0i64; n * m];
        let mut sw = vec![0i64; m * m];
        self.ctx.check(unsafe { qf_gpv_set_tag(self.ctx.raw, tw.as_ptr(), aw.as_mut_ptr(), sw.as_mut_ptr()) }, "qf_gpv_set_tag");
        let q = Z::from(&self.inner.gp.q);
        let mut a_new = MatZq::new(n as i64, m as i64, &q);
        for i in 0..n {
            for j in 0..m {
                a_new.set_entry(i as i64, j as i64, Z::from(aw[i * m + j])).unwrap();
            }
        }
        let mut s_new = MatZ::new(m as i64, m as i64);
        for i in 0..m {
            for j in 0..m {
                s_new.set_entry(i as i64, j as i64, Z::from(sw[i * m + j])).unwrap();
            }
        }
        *self.installed.borrow_mut() = Some((aw, sw));
        *self.fa_tags.borrow_mut() = None; // qf_gpv_set_tag rewrote A
        (a_new, (s_new, td.1.clone()))
    }

    /// Installs the tag table for samp_p with a tag per target: `tags` (T matrices, n x n each, relative to the key `a` =
    /// [A_bar | H_0 G - A_bar R] of any tag H_0 and its trapdoor `td` on the two-phase recursion).  H_t^-1 is computed on
    /// the device (qf_set_tag_table).  The table stays installed until a key or trapdoor is installed; `set_tag` keeps
    /// it.  Panics off the two-phase recursion and when a tag has no unit pivot.
    pub fn set_tag_table(&self, a: &MatZq, td: &(MatZ, MatQ), tags: &[MatZq]) {
        let n = self.n();
        assert!(!tags.is_empty(), "at least one tag");
        self.install(a, td);
        let mut tw = Vec::with_capacity(tags.len() * n * n);
        for tag in tags {
            assert_eq!((tag.get_num_rows(), tag.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
            tw.extend(matzq_to_words(tag));
        }
        self.ctx.check(unsafe { qf_set_tag_table(self.ctx.raw, tw.as_ptr(), tags.len() as i64) }, "qf_set_tag_table");
        *self.installed_tags.borrow_mut() = Some(tags.len());
    }

    /// `set_tag_table` with the tags in polynomial form: tag t is H_t = rot_f(h_t), the matrix of multiplication by
    /// `tags[t]` (an n x 1 vector of coefficients) in Z_q[X]/(f), f = X^n + sum_{i<n} f_i X^i with `f` its n low
    /// coefficients (n x 1).  Rows equal those of `set_tag_table` with the tags rot_f(h_t); the device stores n words per
    /// tag and inverts each in O(n^2) (qf_set_tag_table_poly).  Panics when q is not a prime power and when a tag is not a
    /// unit.
    pub fn set_tag_table_poly(&self, a: &MatZq, td: &(MatZ, MatQ), f: &MatZ, tags: &[MatZq]) {
        assert!(!tags.is_empty(), "at least one tag");
        self.install(a, td);
        let (fw, tw) = poly_tag_words(self.n(), f, tags);
        self.ctx.check(unsafe { qf_set_tag_table_poly(self.ctx.raw, fw.as_ptr(), tw.as_ptr(), tags.len() as i64) },
                       "qf_set_tag_table_poly");
        *self.installed_tags.borrow_mut() = Some(tags.len());
    }

    /// samp_p with a tag per target, against the table of `set_tag_table`: `us[b]` is sampled under
    /// `[A_bar | H_t G - A_bar R]` with `H_t = tags[tag_of[b]]`, in one batch.  Row b equals what `set_tag(H_t)` followed
    /// by `samp_p_batch` gives for it with the same seed (qf_samp_p_tagged).  Panics when no table is installed for this
    /// key and trapdoor or an index is out of range.
    pub fn samp_p_tagged_batch(&self, a: &MatZq, td: &(MatZ, MatQ), us: &[MatZq], tag_of: &[usize], seed: u64) -> Vec<MatZ> {
        let (n, m) = (self.n(), self.m());
        assert_eq!(us.len(), tag_of.len(), "one tag index per target");
        self.install(a, td);
        let ntags = (*self.installed_tags.borrow()).expect("no tag table installed for this key and trapdoor (set_tag_table)");
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        let idx: Vec<i32> = tag_of.iter().map(|t| { assert!(*t < ntags, "tag index out of range"); *t as i32 }).collect();
        let mut e = vec![0i32; us.len() * m];
        let st = unsafe { qf_samp_p_tagged(self.ctx.raw, uw.as_ptr(), idx.as_ptr(), us.len() as i64, seed, 0, e.as_mut_ptr()) };
        self.ctx.check(st, "qf_samp_p_tagged");
        e.chunks(m).map(column_from_i32).collect()
    }

    /// Fills the pool with the target-independent half of samp_p (phase 1 of the two-phase recursion and the products of its
    /// z2) for the sampler indices `first_index .. first_index + count` under `seed` (qf_samp_p_offline).  A new key,
    /// trapdoor or key tag drops the pool; tag tables keep it.  Never refill an index range already served under the same
    /// seed: two preimages sharing a draw leak trapdoor information.  Panics on a one-pass key (QF_ERR_UNSUPPORTED).
    pub fn samp_p_offline(&self, a: &MatZq, td: &(MatZ, MatQ), count: usize, seed: u64, first_index: u64) {
        self.install(a, td);
        self.ctx.check(unsafe { qf_samp_p_offline(self.ctx.raw, count as i64, seed, first_index) }, "qf_samp_p_offline");
    }

    /// Online half for the next `us.len()` pool entries (qf_samp_p_online): row b equals `samp_p_batch` (with `tag_of`:
    /// `samp_p_tagged_batch`) at sampler index `first + b` under the pool's seed; returns the rows and `first`.  Panics
    /// without a pool or when the batch exceeds the remaining entries.
    pub fn samp_p_online_batch(&self, a: &MatZq, td: &(MatZ, MatQ), us: &[MatZq], tag_of: Option<&[usize]>) -> (Vec<MatZ>, u64) {
        let (n, m) = (self.n(), self.m());
        self.install(a, td);
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        let idx: Option<Vec<i32>> = tag_of.map(|t| {
            assert_eq!(us.len(), t.len(), "one tag index per target");
            let ntags = (*self.installed_tags.borrow()).expect("no tag table installed for this key and trapdoor (set_tag_table)");
            t.iter().map(|x| { assert!(*x < ntags, "tag index out of range"); *x as i32 }).collect()
        });
        let (e, first) = samp_p_online_run(&self.ctx, &uw, idx.as_deref(), us.len(), m);
        (e.chunks(m).map(column_from_i32).collect(), first)
    }

    /// `gen_short_basis_for_trapdoor(params, tag, a, r)` (short_basis_classical.rs:54-110) on the device for the key `a`
    /// of this context's parameters: W = digits of -tag^-1 a[:, :m_bar] with tag^-1 and the products computed on the
    /// GPU (qf_gen_short_basis_tagged).  Panics where the reference's `MatZq::inverse(..).unwrap()` does: no unit pivot.
    /// Installs `a` as the context key.
    pub fn gen_short_basis_for_trapdoor(&self, tag: &MatZq, a: &MatZq, r: &MatZ) -> MatZ {
        let (n, m) = (self.n(), self.m());
        let m_bar = i64::try_from(&self.inner.gp.m_bar).unwrap() as usize;
        assert_eq!((tag.get_num_rows(), tag.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
        let (aw, tw) = (matzq_to_words(a), matzq_to_words(tag));
        let r8: Vec<i8> = matz_to_words(r).into_iter().map(|v| i8::try_from(v).expect("R entries must fit i8")).collect();
        assert_eq!(r8.len(), m_bar * (m - m_bar), "R must be m_bar x n k");
        *self.installed_tags.borrow_mut() = None;
        *self.installed.borrow_mut() = None; // qf_set_a drops the installed trapdoor
        *self.fa_tags.borrow_mut() = None;
        self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
        let mut s = vec![0i64; m * m];
        self.ctx.check(unsafe { qf_gen_short_basis_tagged(self.ctx.raw, r8.as_ptr(), tw.as_ptr(), s.as_mut_ptr()) },
                       "qf_gen_short_basis_tagged");
        let mut out = MatZ::new(m as i64, m as i64);
        for i in 0..m {
            for j in 0..m {
                out.set_entry(i as i64, j as i64, Z::from(s[i * m + j])).unwrap();
            }
        }
        out
    }

    /// f_a with a tag per target: `u[b] = A_t sigmas[b]` with `A_t = a + [0 | (H_t - H_0) G]`, `H_t = tags[tag_of[b]]`, for
    /// a key `a = [A_bar | H_0 G - A_bar R]` (`h0` = H_0, None: I) -- the key gen_trapdoor(A_bar, R, H_t) gives, evaluated
    /// from `a` alone (qf_set_f_a_tags, qf_f_a_tagged).  No trapdoor is needed.  The tags cross the boundary once per
    /// table; later batches with the same `a`, `tags` and `h0` pass only sigmas and indices.  Panics like `f_a` when a
    /// sigma is outside D_n, and when an index is out of range.
    pub fn f_a_tagged_batch(&self, a: &MatZq, tags: &[MatZq], h0: Option<&MatZq>, sigmas: &[MatZ], tag_of: &[usize]) -> Vec<MatZq> {
        let aw = matzq_to_words(a);
        // the key of the cached table is on the device too: every key change drops both
        let same = self.installed.borrow().as_ref().map(|(a0, _)| *a0 == aw).unwrap_or(false)
            || self.fa_tags.borrow().as_ref().map(|(a0, _, _, _)| *a0 == aw).unwrap_or(false);
        if !same {
            self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
            *self.installed_tags.borrow_mut() = None;
            *self.installed.borrow_mut() = None;
            *self.fa_tags.borrow_mut() = None;
        }
        let q = Z::from(&self.inner.gp.q);
        f_a_tagged_installed(&self.ctx, &self.fa_tags, aw, self.n(), self.m(), &q, tags, h0, sigmas, tag_of)
    }

    /// `f_a_tagged_batch` with the tags in polynomial form (`f` and `tags` as in `set_tag_table_poly`): A_t = a +
    /// [0 | (rot_f(h_t) - H_0) G] (qf_set_f_a_tags_poly).  Works for every q, singular tags and H_0 = 0.
    pub fn f_a_tagged_batch_poly(&self, a: &MatZq, f: &MatZ, tags: &[MatZq], h0: Option<&MatZq>, sigmas: &[MatZ],
                                 tag_of: &[usize]) -> Vec<MatZq> {
        let aw = matzq_to_words(a);
        let same = self.installed.borrow().as_ref().map(|(a0, _)| *a0 == aw).unwrap_or(false)
            || self.fa_tags.borrow().as_ref().map(|(a0, _, _, _)| *a0 == aw).unwrap_or(false);
        if !same {
            self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
            *self.installed_tags.borrow_mut() = None;
            *self.installed.borrow_mut() = None;
            *self.fa_tags.borrow_mut() = None;
        }
        let q = Z::from(&self.inner.gp.q);
        f_a_tagged_installed_poly(&self.ctx, &self.fa_tags, aw, self.n(), self.m(), &q, f, tags, h0, sigmas, tag_of)
    }
}

/// (f, tags) of tags in polynomial form as words: f is the n x 1 vector of the n low coefficients of the monic modulus,
/// each tag an n x 1 vector of coefficients.
pub(crate) fn poly_tag_words(n: usize, f: &MatZ, tags: &[MatZq]) -> (Vec<i64>, Vec<i64>) {
    assert!(f.is_column_vector() && f.get_num_rows() as usize == n, "f must be the n x 1 vector of its low coefficients");
    let mut tw = Vec::with_capacity(tags.len() * n);
    for tag in tags {
        assert!(tag.is_column_vector() && tag.get_num_rows() as usize == n, "a tag in polynomial form is an n x 1 vector");
        tw.extend(matzq_to_words(tag));
    }
    (matz_to_words(f), tw)
}

/// The f_a tag table on the device (qf_set_f_a_tags[_poly]): (words of the key it belongs to, tag words -- f first in
/// polynomial form, H_0 words; empty for H_0 = I, polynomial form).  The device drops it whenever the key changes, so every
/// key install clears it here too.
pub(crate) type FaTags = RefCell<Option<(Vec<i64>, Vec<i64>, Vec<i64>, bool)>>;

/// f_a with a tag per target against the key installed in `ctx` (qf_f_a_tagged); installs the table when it differs from
/// the cached one.
#[allow(clippy::too_many_arguments)]
pub(crate) fn f_a_tagged_installed(ctx: &Context, fa_tags: &FaTags, aw: Vec<i64>, n: usize, m: usize, q: &Z, tags: &[MatZq],
                                   h0: Option<&MatZq>, sigmas: &[MatZ], tag_of: &[usize]) -> Vec<MatZq> {
    assert!(!tags.is_empty(), "at least one tag");
    assert_eq!(sigmas.len(), tag_of.len(), "one tag index per sigma");
    let square = |t: &MatZq| assert_eq!((t.get_num_rows(), t.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
    let mut tw = Vec::with_capacity(tags.len() * n * n);
    for tag in tags {
        square(tag);
        tw.extend(matzq_to_words(tag));
    }
    let hw = h0.map(|h| { square(h); matzq_to_words(h) }).unwrap_or_default();
    let key = (aw, tw, hw, false);
    if fa_tags.borrow().as_ref() != Some(&key) {
        let hp = if key.2.is_empty() { std::ptr::null() } else { key.2.as_ptr() };
        ctx.check(unsafe { qf_set_f_a_tags(ctx.raw, key.1.as_ptr(), tags.len() as i64, hp) }, "qf_set_f_a_tags");
        *fa_tags.borrow_mut() = Some(key);
    }
    f_a_tagged_run(ctx, n, m, q, tags.len(), sigmas, tag_of)
}

/// `f_a_tagged_installed` with the tags in polynomial form (qf_set_f_a_tags_poly).
#[allow(clippy::too_many_arguments)]
pub(crate) fn f_a_tagged_installed_poly(ctx: &Context, fa_tags: &FaTags, aw: Vec<i64>, n: usize, m: usize, q: &Z, f: &MatZ,
                                        tags: &[MatZq], h0: Option<&MatZq>, sigmas: &[MatZ], tag_of: &[usize]) -> Vec<MatZq> {
    assert!(!tags.is_empty(), "at least one tag");
    assert_eq!(sigmas.len(), tag_of.len(), "one tag index per sigma");
    let (fw, tw) = poly_tag_words(n, f, tags);
    let hw = h0.map(|h| {
        assert_eq!((h.get_num_rows(), h.get_num_columns()), (n as i64, n as i64), "H_0 must be n x n");
        matzq_to_words(h)
    }).unwrap_or_default();
    let key = (aw, [fw, tw].concat(), hw, true);
    if fa_tags.borrow().as_ref() != Some(&key) {
        let hp = if key.2.is_empty() { std::ptr::null() } else { key.2.as_ptr() };
        let st = unsafe { qf_set_f_a_tags_poly(ctx.raw, key.1.as_ptr(), key.1[n..].as_ptr(), tags.len() as i64, hp) };
        ctx.check(st, "qf_set_f_a_tags_poly");
        *fa_tags.borrow_mut() = Some(key);
    }
    f_a_tagged_run(ctx, n, m, q, tags.len(), sigmas, tag_of)
}

/// qf_f_a_tagged against the installed f_a tag table of `ntags` tags.
fn f_a_tagged_run(ctx: &Context, n: usize, m: usize, q: &Z, ntags: usize, sigmas: &[MatZ], tag_of: &[usize]) -> Vec<MatZq> {
    assert_eq!(sigmas.len(), tag_of.len(), "one tag index per sigma");
    let mut sg = Vec::with_capacity(sigmas.len() * m);
    for sigma in sigmas {
        assert!(sigma.is_column_vector() && sigma.get_num_rows() as usize == m, "sigma is not in D_n");
        sg.extend(domain_to_i32(sigma).expect("sigma is not in D_n"));
    }
    let idx: Vec<i32> = tag_of.iter().map(|t| { assert!(*t < ntags, "tag index out of range"); *t as i32 }).collect();
    let mut u = vec![0i64; sigmas.len() * n];
    let mut ok = vec![0u8; sigmas.len()];
    let st = unsafe { qf_f_a_tagged(ctx.raw, sg.as_ptr(), idx.as_ptr(), sigmas.len() as i64, u.as_mut_ptr(), ok.as_mut_ptr()) };
    assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n"); // gpv.rs:191
    ctx.check(st, "qf_f_a_tagged");
    u.chunks(n).map(|row| range_from_words(row, q)).collect()
}

impl PSF for PSFGPVB200 {
    type A = MatZq;
    type Trapdoor = (MatZ, MatQ);
    type Domain = MatZ;
    type Range = MatZq;

    /// gpv.rs:83-94 on the device: uniform A_bar and R, `A = [A_bar | G - A_bar R]` (qf_trap_gen), the short basis
    /// (qf_gen_short_basis, short_basis_classical.rs:54-110) and its GSO (qf_gso; fp64 where the reference is exact).
    fn trap_gen(&self) -> (MatZq, (MatZ, MatQ)) {
        let (n, m) = (self.n(), self.m());
        let m_bar = i64::try_from(&self.inner.gp.m_bar).unwrap() as usize;
        let (mut a, mut r) = (vec![0i64; n * m], vec![0i8; m_bar * (m - m_bar)]);
        self.ctx.check(unsafe { qf_trap_gen(self.ctx.raw, self.next_seed(), a.as_mut_ptr(), r.as_mut_ptr()) }, "qf_trap_gen");
        *self.installed_tags.borrow_mut() = None;
        *self.installed.borrow_mut() = None; // qf_trap_gen installed a new key: whatever trapdoor was cached is gone
        *self.fa_tags.borrow_mut() = None;
        let mut s = vec![0i64; m * m];
        self.ctx.check(unsafe { qf_gen_short_basis(self.ctx.raw, r.as_ptr(), s.as_mut_ptr()) }, "qf_gen_short_basis");
        let mut gso = vec![0f64; m * m];
        self.ctx.check(unsafe { qf_gso(self.ctx.raw, s.as_ptr(), gso.as_mut_ptr()) }, "qf_gso");
        let q = Z::from(&self.inner.gp.q);
        let (mut a_out, mut s_out, mut g_out) = (MatZq::new(n as i64, m as i64, &q), MatZ::new(m as i64, m as i64), MatQ::new(m as i64, m as i64));
        for i in 0..n {
            for j in 0..m {
                a_out.set_entry(i as i64, j as i64, Z::from(a[i * m + j])).unwrap();
            }
        }
        for i in 0..m {
            for j in 0..m {
                s_out.set_entry(i as i64, j as i64, Z::from(s[i * m + j])).unwrap();
                g_out.set_entry(i as i64, j as i64, Q::from(gso[i * m + j])).unwrap();
            }
        }
        (a_out, (s_out, g_out))
    }

    /// gpv.rs:113-116
    fn samp_d(&self) -> MatZ {
        let mut out = vec![0i32; self.m()];
        self.ctx.check(unsafe { qf_samp_d(self.ctx.raw, 1, self.next_seed(), 0, out.as_mut_ptr()) }, "qf_samp_d");
        column_from_i32(&out)
    }

    /// gpv.rs:152-161
    fn samp_p(&self, a: &MatZq, td: &(MatZ, MatQ), u: &MatZq) -> MatZ {
        self.samp_p_batch(a, td, std::slice::from_ref(u), self.next_seed(), 0).pop().unwrap()
    }

    /// gpv.rs:190-193: `assert!(self.check_domain(sigma)); a * sigma`
    fn f_a(&self, a: &MatZq, sigma: &MatZ) -> MatZq {
        self.f_a_batch(a, std::slice::from_ref(sigma)).pop().unwrap()
    }

    /// gpv.rs:219-224: column vector, length m, squared norm at most s^2 m
    fn check_domain(&self, sigma: &MatZ) -> bool {
        if !sigma.is_column_vector() || sigma.get_num_rows() as usize != self.m() {
            return false;
        }
        let Some(sg) = domain_to_i32(sigma) else { return false };
        let mut ok = [0u8; 1];
        self.ctx.check(unsafe { qf_check_domain(self.ctx.raw, sg.as_ptr(), 1, ok.as_mut_ptr()) }, "qf_check_domain");
        ok[0] == 1
    }
}

impl PSFBatch for PSFGPVB200 {
    fn samp_p_batch(&self, a: &MatZq, td: &(MatZ, MatQ), us: &[MatZq], seed: u64, first_index: u64) -> Vec<MatZ> {
        self.install(a, td);
        let (n, m) = (self.n(), self.m());
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        let mut e = vec![0i32; us.len() * m];
        let st = unsafe { qf_samp_p(self.ctx.raw, uw.as_ptr(), us.len() as i64, seed, first_index, e.as_mut_ptr()) };
        self.ctx.check(st, "qf_samp_p"); // the reference unwrap()s here (gpv.rs:155,160)
        e.chunks(m).map(column_from_i32).collect()
    }

    fn f_a_batch(&self, a: &MatZq, sigmas: &[MatZ]) -> Vec<MatZq> {
        let aw = matzq_to_words(a);
        let same = self.installed.borrow().as_ref().map(|(a0, _)| *a0 == aw).unwrap_or(false);
        if !same {
            self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
            *self.installed_tags.borrow_mut() = None;
            *self.installed.borrow_mut() = None;
            *self.fa_tags.borrow_mut() = None;
        }
        let (n, m) = (self.n(), self.m());
        let mut sg = Vec::with_capacity(sigmas.len() * m);
        for sigma in sigmas {
            // the shape half of check_domain (gpv.rs:221-222) stays on the host
            assert!(sigma.is_column_vector() && sigma.get_num_rows() as usize == m, "sigma is not in D_n");
            sg.extend(domain_to_i32(sigma).expect("sigma is not in D_n"));
        }
        let mut u = vec![0i64; sigmas.len() * n];
        let mut ok = vec![0u8; sigmas.len()];
        let st = unsafe { qf_f_a(self.ctx.raw, sg.as_ptr(), sigmas.len() as i64, u.as_mut_ptr(), ok.as_mut_ptr()) };
        assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n"); // gpv.rs:191
        self.ctx.check(st, "qf_f_a");
        let q = Z::from(&self.inner.gp.q);
        u.chunks(n).map(|row| range_from_words(row, &q)).collect()
    }

    fn samp_p_batch_packed(&self, a: &MatZq, td: &(MatZ, MatQ), us: &[MatZq], seed: u64, first_index: u64) -> PackedDomain {
        self.install(a, td);
        let n = self.n();
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        samp_p_packed_run(&self.ctx, &uw, us.len(), seed, first_index)
    }

    fn f_a_batch_packed(&self, a: &MatZq, packed: &PackedDomain) -> Vec<MatZq> {
        let aw = matzq_to_words(a);
        if !self.installed.borrow().as_ref().map(|(a0, _)| *a0 == aw).unwrap_or(false) {
            self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
            *self.installed_tags.borrow_mut() = None;
            *self.installed.borrow_mut() = None;
            *self.fa_tags.borrow_mut() = None;
        }
        let q = Z::from(&self.inner.gp.q);
        f_a_packed_run(&self.ctx, self.n(), packed).chunks(self.n()).map(|row| range_from_words(row, &q)).collect()
    }
}

// ---- LossyCompressionFIPS203 -----------------------------------------------------------------------------------------

/// `Compress_d` of every coefficient word (lossy_compression_fips203.rs:101-111); panics for `d < 1` like `:91-94`.
pub fn compress_words(coeffs: &[i64], d: u32, q: u64) -> Vec<i64> {
    assert!(d >= 1, "Performing this function with d < 1 implies reducing mod 1");
    let mut out = vec![0i64; coeffs.len()];
    let st = unsafe { qf_compress_i64(coeffs.as_ptr(), out.as_mut_ptr(), coeffs.len(), q, d, 0, std::ptr::null_mut()) };
    assert!(st == QF_OK, "qf_compress_i64: status {st}");
    out
}

/// `Decompress_d` (lossy_compression_fips203.rs:159-169), coefficients written unreduced like the reference.
pub fn decompress_words(compressed: &[i64], d: u32, q: u64) -> Vec<i64> {
    assert!(d >= 1, "Performing this function with d < 1 implies reducing mod 1");
    let mut out = vec![0i64; compressed.len()];
    let st = unsafe { qf_decompress_i64(compressed.as_ptr(), out.as_mut_ptr(), compressed.len(), q, d, 0, std::ptr::null_mut()) };
    assert!(st == QF_OK, "qf_decompress_i64: status {st}");
    out
}

/// `ByteEncode_d(Compress_d(f))` for degree-256 polynomials with q < 2^16 (FIPS 203 Algorithm 5): the packed wire form.
pub fn compress_encode(coeffs: &[u16], d: u32, q: u32) -> Vec<u8> {
    assert!(d >= 1 && coeffs.len() % 256 == 0);
    let npoly = coeffs.len() / 256;
    let mut out = vec![0u8; npoly * 32 * d as usize];
    let st = unsafe { qf_compress_encode_u16(coeffs.as_ptr(), out.as_mut_ptr(), npoly, q, d, 1, 0, std::ptr::null_mut()) };
    assert!(st == QF_OK, "qf_compress_encode_u16: status {st}");
    out
}

/// `Decompress_d(ByteDecode_d(b))` (FIPS 203 Algorithm 6).
pub fn decode_decompress(packed: &[u8], d: u32, q: u32) -> Vec<u16> {
    assert!(d >= 1 && packed.len() % (32 * d as usize) == 0);
    let npoly = packed.len() / (32 * d as usize);
    let mut out = vec![0u16; npoly * 256];
    let st = unsafe { qf_decode_decompress_u16(packed.as_ptr(), out.as_mut_ptr(), npoly, q, d, 1, 0, std::ptr::null_mut()) };
    assert!(st == QF_OK, "qf_decode_decompress_u16: status {st}");
    out
}
