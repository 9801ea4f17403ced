//! `PSFPerturbation` (mp_perturbation.rs:57-62, impl :193-403) on the GPU: the MP12 perturbation sampler
//! `p <- D_{sqrt(Sigma_2)}`, `v = u - A p`, `z <- D_{Lambda_v^perp(G)}`, `e = p + [R; I] z` for a batch of targets.
//! Shipped as source (see lib.rs).
use crate::ffi::*;
use crate::{column_from_i32, domain_to_i32, f_a_tagged_installed, f_a_tagged_installed_poly, matz_to_words, matzq_to_words,
            f_a_packed_run, poly_tag_words, range_from_words, samp_p_online_run, samp_p_packed_run, Context, FaTags, PSFBatch, PackedDomain};
use qfall_math::{
    integer::{MatZ, Z},
    integer_mod_q::MatZq,
    rational::{MatQ, Q},
    traits::{MatrixDimensions, MatrixGetEntry, MatrixSetEntry},
};
use qfall_tools::primitive::psf::{PSFPerturbation, PSF};
use std::cell::RefCell;

pub struct PSFPerturbationB200 {
    pub inner: PSFPerturbation,
    ctx: Context,
    installed_a: RefCell<Option<Vec<i64>>>,
    /// the trapdoor on the device: (R words, bit patterns of sqrt(Sigma_2), gadget block S_k, bit patterns of its GSO) --
    /// every component takes part in the comparison: the same R with another covariance (compute_sqrt_sigma_2 with a
    /// custom Sigma, mp_perturbation.rs:94-104) or another gadget basis is a different trapdoor
    installed_r: RefCell<Option<(Vec<i64>, Vec<u64>, Vec<i64>, Vec<u64>)>>,
    /// number of tags in the table on the device (qf_set_tag_table); the device drops it with every key or trapdoor install
    installed_tags: RefCell<Option<usize>>,
    /// the f_a tag table on the device (qf_set_f_a_tags); the device drops it whenever the key changes
    fa_tags: FaTags,
    seed: RefCell<u64>,
}

impl PSFPerturbationB200 {
    pub fn new(inner: PSFPerturbation, device: i32, seed: u64) -> Result<Self, String> {
        let gp = &inner.gp;
        let params = qf_params {
            kind: QF_PSF_PERTURBATION,
            n: i64::try_from(&gp.n).unwrap(),
            k: i64::try_from(&gp.k).unwrap(),
            m_bar: i64::try_from(&gp.m_bar).unwrap(),
            base: i64::try_from(&gp.base).unwrap(),
            q: u64::try_from(&Z::from(&gp.q)).map_err(|_| "modulus must be below 2^62".to_string())?,
            s: f64::from(&inner.s),
            r: f64::from(&inner.r),
            // mp_perturbation.rs:401: ||sigma||^2 <= s^2 r^2 m, compared exactly: floor of the exact rational
            norm_bound: crate::ring::floor_u64(
                &(&inner.s * &inner.s * &inner.r * &inner.r * Q::from(i64::try_from(&(&gp.m_bar + &gp.n * &gp.k)).unwrap())),
            ),
        };
        Ok(PSFPerturbationB200 {
            inner,
            ctx: Context::new(&params, device)?,
            installed_a: RefCell::new(None),
            installed_r: RefCell::new(None),
            installed_tags: RefCell::new(None),
            fa_tags: RefCell::new(None),
            seed: RefCell::new(seed),
        })
    }
    fn n(&self) -> usize {
        i64::try_from(&self.inner.gp.n).unwrap() as usize
    }
    fn k(&self) -> usize {
        i64::try_from(&self.inner.gp.k).unwrap() as usize
    }
    fn m_bar(&self) -> usize {
        i64::try_from(&self.inner.gp.m_bar).unwrap() as usize
    }
    fn m(&self) -> usize {
        self.m_bar() + self.n() * self.k()
    }
    fn next_seed(&self) -> u64 {
        let mut s = self.seed.borrow_mut();
        *s = s.wrapping_mul(6364136223846793005).wrapping_add(1442695040888963407);
        *s
    }
    fn install_a(&self, a: &MatZq) {
        let aw = matzq_to_words(a);
        if self.installed_a.borrow().as_ref() == Some(&aw) {
            return;
        }
        self.ctx.check(unsafe { qf_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_set_a");
        *self.installed_a.borrow_mut() = Some(aw);
        *self.installed_r.borrow_mut() = None;
        *self.installed_tags.borrow_mut() = None;
        *self.fa_tags.borrow_mut() = None;
    }
    /// Trapdoor `(R, sqrt(Sigma_2), (S, S~))` (mp_perturbation.rs:195).  The gadget basis must be `I_n (x) S_k`
    /// (what `short_basis_gadget` returns, gadget_classical.rs:273-286): only its first k x k block crosses the boundary.
    fn install_td(&self, td: &(MatZ, MatQ, (MatZ, MatQ))) {
        let rw = matz_to_words(&td.0);
        let r8: Vec<i8> = rw.iter().map(|v| i8::try_from(*v).expect("R entries are small")).collect();
        let (m, k) = (self.m(), self.k());
        let mut sqrt_sigma_2 = Vec::with_capacity(m * m);
        for i in 0..m {
            for j in 0..m {
                let x: Q = td.1.get_entry(i as i64, j as i64).unwrap();
                sqrt_sigma_2.push(f64::from(&x));
            }
        }
        let (mut s_block, mut s_block_gso) = (Vec::with_capacity(k * k), Vec::with_capacity(k * k));
        for i in 0..k {
            for j in 0..k {
                let z: Z = td.2 .0.get_entry(i as i64, j as i64).unwrap();
                let x: Q = td.2 .1.get_entry(i as i64, j as i64).unwrap();
                s_block.push(i64::try_from(&z).unwrap());
                s_block_gso.push(f64::from(&x));
            }
        }
        let key = (
            rw,
            sqrt_sigma_2.iter().map(|x| x.to_bits()).collect::<Vec<u64>>(),
            s_block.clone(),
            s_block_gso.iter().map(|x| x.to_bits()).collect::<Vec<u64>>(),
        );
        if self.installed_r.borrow().as_ref() == Some(&key) {
            return;
        }
        let st = unsafe {
            qf_set_trapdoor_perturbation(self.ctx.raw, r8.as_ptr(), sqrt_sigma_2.as_ptr(), s_block.as_ptr(), s_block_gso.as_ptr())
        };
        self.ctx.check(st, "qf_set_trapdoor_perturbation");
        *self.installed_r.borrow_mut() = Some(key);
        *self.installed_tags.borrow_mut() = None;
    }

    /// Tag switch for a key `a = [A_bar | H G - A_bar R]` (gen_trapdoor with a tag, gadget_classical.rs:56-68) and its
    /// trapdoor `td`: returns `[A_bar | H' G - A_bar R]` for `tag` = H' (n x n), equal to gen_trapdoor(A_bar, R, H'), and
    /// installs it while R, sqrt(Sigma_2) and the gadget basis stay on the device (qf_set_tag).  Panics when `a` is not such a
    /// key for the R of `td` or when H' has no unit pivot (the reference panics in `MatZq::inverse`).
    pub fn set_tag(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), tag: &MatZq) -> MatZq {
        let (n, m) = (self.n(), self.m());
        assert_eq!((tag.get_num_rows(), tag.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
        self.install_a(a);
        self.install_td(td);
        let tw = matzq_to_words(tag);
        let mut aw = vec![0i64; n * m];
        self.ctx.check(unsafe { qf_set_tag(self.ctx.raw, tw.as_ptr(), aw.as_mut_ptr()) }, "qf_set_tag");
        let q = Z::from(&self.inner.gp.q);
        let mut out = MatZq::new(n as i64, m as i64, &q);
        for i in 0..n {
            for j in 0..m {
                out.set_entry(i as i64, j as i64, Z::from(aw[i * m + j])).unwrap();
            }
        }
        *self.installed_a.borrow_mut() = Some(aw);
        *self.fa_tags.borrow_mut() = None; // qf_set_tag rewrote A
        out
    }

    /// Installs the tag table for samp_p with a tag per target: `tags` (T matrices, n x n each, relative to the key `a` =
    /// [A_bar | H_0 G - A_bar R] of any tag H_0 and its trapdoor `td`).  H_t^-1 is computed on the device
    /// (qf_set_tag_table).  The table stays installed until a key or trapdoor is installed (install_a / install_td of
    /// another `a` or `td`, trap_gen); `set_tag` keeps it.  Panics when a tag has no unit pivot (the reference panics in
    /// `MatZq::inverse`).
    pub fn set_tag_table(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), tags: &[MatZq]) {
        let n = self.n();
        assert!(!tags.is_empty(), "at least one tag");
        self.install_a(a);
        self.install_td(td);
        let mut tw = Vec::with_capacity(tags.len() * n * n);
        for tag in tags {
            assert_eq!((tag.get_num_rows(), tag.get_num_columns()), (n as i64, n as i64), "tag must be n x n");
            tw.extend(matzq_to_words(tag));
        }
        self.ctx.check(unsafe { qf_set_tag_table(self.ctx.raw, tw.as_ptr(), tags.len() as i64) }, "qf_set_tag_table");
        *self.installed_tags.borrow_mut() = Some(tags.len());
    }

    /// `set_tag_table` with the tags in polynomial form: tag t is H_t = rot_f(h_t), the matrix of multiplication by
    /// `tags[t]` (an n x 1 vector of coefficients) in Z_q[X]/(f), `f` the n x 1 vector of the n low coefficients of the
    /// monic modulus (qf_set_tag_table_poly: n words per tag, O(n^2) inverse on the device).  Rows equal those of
    /// `set_tag_table` with the tags rot_f(h_t).  Panics when q is not a prime power and when a tag is not a unit.
    pub fn set_tag_table_poly(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), f: &MatZ, tags: &[MatZq]) {
        assert!(!tags.is_empty(), "at least one tag");
        self.install_a(a);
        self.install_td(td);
        let (fw, tw) = poly_tag_words(self.n(), f, tags);
        self.ctx.check(unsafe { qf_set_tag_table_poly(self.ctx.raw, fw.as_ptr(), tw.as_ptr(), tags.len() as i64) },
                       "qf_set_tag_table_poly");
        *self.installed_tags.borrow_mut() = Some(tags.len());
    }

    /// samp_p with a tag per target, against the table of `set_tag_table`: `us[b]` is sampled under
    /// `[A_bar | H_t G - A_bar R]` with `H_t = tags[tag_of[b]]`, in one batch.  Row b equals what `set_tag(H_t)` followed by
    /// `samp_p_batch` gives for it with the same seed (qf_samp_p_tagged).  The tags do not cross the boundary again, so
    /// repeated batches cost only their targets.  Panics when no table is installed for this key and trapdoor (a key or
    /// trapdoor install drops it: call `set_tag_table` again) or an index is out of range.
    pub fn samp_p_tagged_batch(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), us: &[MatZq], tag_of: &[usize],
                               seed: u64) -> Vec<MatZ> {
        let (n, m) = (self.n(), self.m());
        assert_eq!(us.len(), tag_of.len(), "one tag index per target");
        self.install_a(a);
        self.install_td(td);
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

    /// Fills the pool with the target-independent half of samp_p (the perturbation p and A p) for the sampler indices
    /// `first_index .. first_index + count` under `seed` (qf_samp_p_offline).  A new key, trapdoor or key tag drops the
    /// pool; tag tables keep it.  Never refill an index range already served under the same seed: two preimages sharing a
    /// perturbation leak trapdoor information.
    pub fn samp_p_offline(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), count: usize, seed: u64, first_index: u64) {
        self.install_a(a);
        self.install_td(td);
        self.ctx.check(unsafe { qf_samp_p_offline(self.ctx.raw, count as i64, seed, first_index) }, "qf_samp_p_offline");
    }

    /// Online half for the next `us.len()` pool entries (qf_samp_p_online): row b equals `samp_p_batch` (with `tag_of`:
    /// `samp_p_tagged_batch`) at sampler index `first + b` under the pool's seed; returns the rows and `first`.  Panics
    /// without a pool or when the batch exceeds the remaining entries.
    pub fn samp_p_online_batch(&self, a: &MatZq, td: &(MatZ, MatQ, (MatZ, MatQ)), us: &[MatZq], tag_of: Option<&[usize]>)
                               -> (Vec<MatZ>, u64) {
        let (n, m) = (self.n(), self.m());
        self.install_a(a);
        self.install_td(td);
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

    /// f_a with a tag per target: `u[b] = A_t sigmas[b]` with `A_t = a + [0 | (H_t - H_0) G]`, `H_t = tags[tag_of[b]]`, for
    /// a key `a = [A_bar | H_0 G - A_bar R]` (`h0` = H_0, None: I), evaluated from `a` alone (qf_set_f_a_tags,
    /// qf_f_a_tagged): no trapdoor is needed, singular tags are allowed.  The tags cross the boundary once per table.
    /// Independent of `set_tag_table`.  Panics like `f_a` when a sigma is outside D_n, and when an index is out of range.
    pub fn f_a_tagged_batch(&self, a: &MatZq, tags: &[MatZq], h0: Option<&MatZq>, sigmas: &[MatZ], tag_of: &[usize]) -> Vec<MatZq> {
        self.install_a(a);
        let q = Z::from(&self.inner.gp.q);
        f_a_tagged_installed(&self.ctx, &self.fa_tags, matzq_to_words(a), self.n(), self.m(), &q, tags, h0, sigmas, tag_of)
    }

    /// `f_a_tagged_batch` with the tags in polynomial form (`f` and `tags` as in `set_tag_table_poly`): A_t = a +
    /// [0 | (rot_f(h_t) - H_0) G] (qf_set_f_a_tags_poly).  Works for every q, singular tags and H_0 = 0.
    pub fn f_a_tagged_batch_poly(&self, a: &MatZq, f: &MatZ, tags: &[MatZq], h0: Option<&MatZq>, sigmas: &[MatZ],
                                 tag_of: &[usize]) -> Vec<MatZq> {
        self.install_a(a);
        let q = Z::from(&self.inner.gp.q);
        f_a_tagged_installed_poly(&self.ctx, &self.fa_tags, matzq_to_words(a), self.n(), self.m(), &q, f, tags, h0, sigmas,
                                  tag_of)
    }
}

impl PSF for PSFPerturbationB200 {
    type A = MatZq;
    type Trapdoor = (MatZ, MatQ, (MatZ, MatQ));
    type Domain = MatZ;
    type Range = MatZq;

    /// mp_perturbation.rs:221-244 with the heavy parts on the device: `A = [A_bar | G - A_bar R]` (qf_trap_gen) and the
    /// Cholesky factor of Sigma_2 (qf_compute_sqrt_sigma_2, :111-139); the k x k gadget block and its GSO stay on the host
    /// (`short_basis_gadget`, `MatQ::gso` of a block-diagonal matrix).
    fn trap_gen(&self) -> (MatZq, (MatZ, MatQ, (MatZ, MatQ))) {
        let (n, m, m_bar) = (self.n(), self.m(), self.m_bar());
        let nk = m - m_bar;
        let (mut a, mut r) = (vec![0i64; n * m], vec![0i8; m_bar * nk]);
        self.ctx.check(unsafe { qf_trap_gen(self.ctx.raw, self.next_seed(), a.as_mut_ptr(), r.as_mut_ptr()) }, "qf_trap_gen");
        // qf_trap_gen installed a new key (and thereby dropped the device's trapdoor): forget the cached one
        *self.installed_a.borrow_mut() = None;
        *self.installed_r.borrow_mut() = None;
        *self.installed_tags.borrow_mut() = None;
        *self.fa_tags.borrow_mut() = None;
        let mut l = vec![0f64; m * m];
        let st = unsafe { qf_compute_sqrt_sigma_2(self.ctx.raw, r.as_ptr(), std::ptr::null(), l.as_mut_ptr()) };
        self.ctx.check(st, "qf_compute_sqrt_sigma_2"); // QF_ERR_INVALID = Sigma_2 not positive definite (the reference panics)
        let q = Z::from(&self.inner.gp.q);
        let (mut a_out, mut r_out, mut l_out) = (MatZq::new(n as i64, m as i64, &q), MatZ::new(m_bar as i64, nk as i64), MatQ::new(m as i64, m as i64));
        for i in 0..n {
            for j in 0..m {
                a_out.set_entry(i as i64, j as i64, Z::from(a[i * m + j])).unwrap();
            }
        }
        for i in 0..m_bar {
            for j in 0..nk {
                r_out.set_entry(i as i64, j as i64, Z::from(r[i * nk + j] as i64)).unwrap();
            }
        }
        for i in 0..m {
            for j in 0..=i {
                l_out.set_entry(i as i64, j as i64, Q::from(l[i * m + j])).unwrap();
            }
        }
        let short_basis_gadget = qfall_tools::sample::g_trapdoor::gadget_classical::short_basis_gadget(&self.inner.gp);
        let short_basis_gadget_gso = MatQ::from(&short_basis_gadget).gso();
        (a_out, (r_out, l_out, (short_basis_gadget, short_basis_gadget_gso)))
    }

    /// mp_perturbation.rs:264-267: D_{Z^m, s r}
    fn samp_d(&self) -> MatZ {
        let mut out = vec![0i32; self.m()];
        self.ctx.check(unsafe { qf_samp_d(self.ctx.raw, 1, self.next_seed(), 0, out.as_mut_ptr()) }, "qf_samp_d");
        column_from_i32(&out)
    }

    /// mp_perturbation.rs:304-336
    fn samp_p(&self, a: &MatZq, td: &Self::Trapdoor, u: &MatZq) -> MatZ {
        self.samp_p_batch(a, td, std::slice::from_ref(u), self.next_seed(), 0).pop().unwrap()
    }

    /// mp_perturbation.rs:366-369
    fn f_a(&self, a: &MatZq, sigma: &MatZ) -> MatZq {
        self.f_a_batch(a, std::slice::from_ref(sigma)).pop().unwrap()
    }

    /// mp_perturbation.rs:396-402: column vector, length m, squared norm at most s^2 r^2 m
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

impl PSFBatch for PSFPerturbationB200 {
    fn samp_p_batch(&self, a: &MatZq, td: &Self::Trapdoor, us: &[MatZq], seed: u64, first_index: u64) -> Vec<MatZ> {
        self.install_a(a);
        self.install_td(td);
        let (n, m) = (self.n(), self.m());
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        let mut e = vec![0i32; us.len() * m];
        let st = unsafe { qf_samp_p(self.ctx.raw, uw.as_ptr(), us.len() as i64, seed, first_index, e.as_mut_ptr()) };
        self.ctx.check(st, "qf_samp_p");
        e.chunks(m).map(column_from_i32).collect()
    }

    fn f_a_batch(&self, a: &MatZq, sigmas: &[MatZ]) -> Vec<MatZq> {
        self.install_a(a);
        let (n, m) = (self.n(), self.m());
        let mut sg = Vec::with_capacity(sigmas.len() * m);
        for sigma in sigmas {
            assert!(sigma.is_column_vector() && sigma.get_num_rows() as usize == m, "sigma is not in D_n");
            sg.extend(domain_to_i32(sigma).expect("sigma is not in D_n"));
        }
        let mut u = vec![0i64; sigmas.len() * n];
        let mut ok = vec![0u8; sigmas.len()];
        let st = unsafe { qf_f_a(self.ctx.raw, sg.as_ptr(), sigmas.len() as i64, u.as_mut_ptr(), ok.as_mut_ptr()) };
        assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n"); // mp_perturbation.rs:367
        self.ctx.check(st, "qf_f_a");
        let q = Z::from(&self.inner.gp.q);
        u.chunks(n).map(|row| range_from_words(row, &q)).collect()
    }

    fn samp_p_batch_packed(&self, a: &MatZq, td: &Self::Trapdoor, us: &[MatZq], seed: u64, first_index: u64) -> PackedDomain {
        self.install_a(a);
        self.install_td(td);
        let n = self.n();
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.is_column_vector() && u.get_num_rows() as usize == n, "target must be an n x 1 vector");
            uw.extend(matzq_to_words(u));
        }
        samp_p_packed_run(&self.ctx, &uw, us.len(), seed, first_index)
    }

    fn f_a_batch_packed(&self, a: &MatZq, packed: &PackedDomain) -> Vec<MatZq> {
        self.install_a(a);
        let q = Z::from(&self.inner.gp.q);
        f_a_packed_run(&self.ctx, self.n(), packed).chunks(self.n()).map(|row| range_from_words(row, &q)).collect()
    }
}
