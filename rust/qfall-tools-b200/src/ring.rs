//! `PSFGPVRing` (gpv_ring.rs:62-73, impl :69-284) on the GPU: the ring GPV PSF over `Z_q[X]/(X^n + 1)`.
//!
//! Associated types are the reference's (`A = MatPolynomialRingZq` 1 x (k+2), `Trapdoor = (r, e)` two 1 x k
//! `MatPolyOverZ`, `Domain = MatPolyOverZ` (k+2) x 1, `Range = MatPolynomialRingZq` 1 x 1).  Values cross the boundary in
//! the coefficient embedding (gpv_ring.rs:172-178): a vector of p polynomials is `p * n` words, polynomial-major.
//! The reference rebuilds the short basis and its GSO on every `samp_p` (gpv_ring.rs:169, :205-211); here they are
//! built once per trapdoor (`qf_ring_gen_short_basis` + `qf_set_trapdoor_gpv` with the GSO computed on the device).
//! Shipped as source (see lib.rs).
use crate::ffi::*;
use crate::{f_a_packed_run, samp_p_packed_run, Context, PSFBatch, PackedDomain};
use qfall_math::{
    integer::{MatPolyOverZ, PolyOverZ, Z},
    integer_mod_q::{MatPolynomialRingZq, PolynomialRingZq},
    rational::Q,
    traits::{GetCoefficient, MatrixDimensions, MatrixGetEntry, MatrixSetEntry, SetCoefficient},
};
use qfall_tools::primitive::psf::{PSFGPVRing, PSF};
use std::cell::RefCell;

pub struct PSFGPVRingB200 {
    pub inner: PSFGPVRing,
    ctx: Context,
    installed_a: RefCell<Option<Vec<i64>>>,
    installed_td: RefCell<Option<(Vec<i32>, Vec<i32>)>>,
    // words of the key table on the device (qf_ring_set_key_table); independent of the installed key
    installed_keys: RefCell<Option<Vec<i64>>>,
    seed: RefCell<u64>,
}

/// floor of an exact non-negative rational as u64 (the check_domain bounds are exact rationals in the reference)
pub(crate) fn floor_u64(x: &Q) -> u64 {
    u64::try_from(&x.floor()).expect("norm bound below 2^64")
}

impl PSFGPVRingB200 {
    pub fn new(inner: PSFGPVRing, device: i32, seed: u64) -> Result<Self, String> {
        let gp = &inner.gp;
        let n = gp.modulus.get_degree();
        let k = i64::try_from(&gp.k).unwrap();
        // gpv_ring.rs:281-282: ||sigma||^2 <= s^2 * n * (k + 2), compared exactly
        let bound = &inner.s * &inner.s * Q::from(n * (k + 2));
        let params = qf_params {
            kind: QF_PSF_GPV_RING,
            n,
            k,
            m_bar: k + 2,
            base: i64::try_from(&gp.base).unwrap(),
            q: u64::try_from(&gp.modulus.get_q()).map_err(|_| "modulus must be below 2^62".to_string())?,
            s: f64::from(&inner.s),
            r: 1.0,
            norm_bound: floor_u64(&bound),
        };
        Ok(PSFGPVRingB200 {
            inner,
            ctx: Context::new(&params, device)?,
            installed_a: RefCell::new(None),
            installed_td: RefCell::new(None),
            installed_keys: RefCell::new(None),
            seed: RefCell::new(seed),
        })
    }
    fn n(&self) -> usize {
        self.inner.gp.modulus.get_degree() as usize
    }
    fn k(&self) -> usize {
        i64::try_from(&self.inner.gp.k).unwrap() as usize
    }
    fn next_seed(&self) -> u64 {
        let mut s = self.seed.borrow_mut();
        *s = s.wrapping_mul(6364136223846793005).wrapping_add(1442695040888963407);
        *s
    }
    /// coefficients 0..n of every polynomial of a row or column vector of `PolyOverZ`, polynomial-major
    fn polys_to_words(m: &MatPolyOverZ, n: usize) -> Vec<i64> {
        let (rows, cols) = (m.get_num_rows(), m.get_num_columns());
        let mut out = Vec::with_capacity((rows * cols) as usize * n);
        for i in 0..rows {
            for j in 0..cols {
                let p: PolyOverZ = m.get_entry(i, j).unwrap();
                for t in 0..n {
                    let c: Z = p.get_coeff(t as i64).unwrap();
                    out.push(i64::try_from(&c).expect("coefficient below 2^63"));
                }
            }
        }
        out
    }
    fn key_words(&self, a: &MatPolynomialRingZq) -> Vec<i64> {
        // least non-negative residues of the k + 2 key polynomials
        Self::polys_to_words(&a.get_representative_least_nonnegative_residue(), self.n())
    }
    fn install_a(&self, a: &MatPolynomialRingZq) {
        let aw = self.key_words(a);
        if self.installed_a.borrow().as_ref() == Some(&aw) {
            return;
        }
        self.ctx.check(unsafe { qf_ring_set_a(self.ctx.raw, aw.as_ptr()) }, "qf_ring_set_a");
        *self.installed_a.borrow_mut() = Some(aw);
        *self.installed_td.borrow_mut() = None; // a new key invalidates the trapdoor on the device as well
    }
    fn install_td(&self, td: &(MatPolyOverZ, MatPolyOverZ)) {
        let n = self.n();
        let to32 = |m: &MatPolyOverZ| -> Vec<i32> {
            Self::polys_to_words(m, n).into_iter().map(|v| i32::try_from(v).expect("trapdoor coefficients are small")).collect()
        };
        let (r, e) = (to32(&td.0), to32(&td.1));
        if let Some((r0, e0)) = self.installed_td.borrow().as_ref() {
            if *r0 == r && *e0 == e {
                return;
            }
        }
        let d = n * (self.k() + 2);
        let mut basis = vec![0i64; d * d];
        let st = unsafe { qf_ring_gen_short_basis(self.ctx.raw, r.as_ptr(), e.as_ptr(), basis.as_mut_ptr()) };
        self.ctx.check(st, "qf_ring_gen_short_basis");
        // GSO on the device (s_gso = NULL): the reference computes it inside MatPolyOverZ::sample_d on every call
        self.ctx.check(unsafe { qf_set_trapdoor_gpv(self.ctx.raw, basis.as_ptr(), std::ptr::null()) }, "qf_set_trapdoor_gpv");
        *self.installed_td.borrow_mut() = Some((r, e));
    }
    fn domain_from_words(&self, e: &[i32]) -> MatPolyOverZ {
        let (n, p) = (self.n(), self.k() + 2);
        let mut out = MatPolyOverZ::new(p as i64, 1);
        for i in 0..p {
            let mut poly = PolyOverZ::default();
            for t in 0..n {
                let v = e[i * n + t];
                if v != 0 {
                    poly.set_coeff(t as i64, Z::from(v as i64)).unwrap();
                }
            }
            out.set_entry(i as i64, 0, &poly).unwrap();
        }
        out
    }
    fn range_from_words(&self, u: &[i64]) -> MatPolynomialRingZq {
        let mut poly = PolyOverZ::default();
        for (t, v) in u.iter().enumerate() {
            if *v != 0 {
                poly.set_coeff(t as i64, Z::from(*v)).unwrap();
            }
        }
        let mut m = MatPolyOverZ::new(1, 1);
        m.set_entry(0, 0, &poly).unwrap();
        MatPolynomialRingZq::from((&m, &self.inner.gp.modulus))
    }
    /// Domain value -> i32 words; `None` if the shape is wrong or an entry does not fit (then it is outside D_n)
    fn domain_to_words(&self, sigma: &MatPolyOverZ) -> Option<Vec<i32>> {
        if !sigma.is_column_vector() || sigma.get_num_rows() as usize != self.k() + 2 {
            return None;
        }
        for i in 0..sigma.get_num_rows() {
            let p: PolyOverZ = sigma.get_entry(i, 0).unwrap();
            if p.get_degree() >= self.n() as i64 {
                return None;
            }
        }
        Self::polys_to_words(sigma, self.n()).into_iter().map(|v| i32::try_from(v).ok()).collect()
    }
}

impl PSF for PSFGPVRingB200 {
    type A = MatPolynomialRingZq;
    type Trapdoor = (MatPolyOverZ, MatPolyOverZ);
    type Domain = MatPolyOverZ;
    type Range = MatPolynomialRingZq;

    /// gpv_ring.rs:91-98: uniform `a_bar`, `r`, `e` with coefficients `D_{Z, s_td}` (trapdoor_distribution.rs:112-122) drawn by the
    /// reference's own samplers (k polynomial draws: not the hot path), `A = [1 | a_bar | g^t - (a_bar r + e)]` on the device.
    fn trap_gen(&self) -> (MatPolynomialRingZq, (MatPolyOverZ, MatPolyOverZ)) {
        let (n, k) = (self.n(), self.k());
        let gp = &self.inner.gp;
        let a_bar = PolyOverZ::sample_uniform(gp.modulus.get_degree() - 1, 0, gp.modulus.get_q()).unwrap();
        let r = gp.distribution.sample(&gp.n, &gp.k, &self.inner.s_td);
        let e = gp.distribution.sample(&gp.n, &gp.k, &self.inner.s_td);
        let mut ab = MatPolyOverZ::new(1, 1);
        ab.set_entry(0, 0, &a_bar).unwrap();
        let abw = Self::polys_to_words(&ab, n);
        let to32 = |m: &MatPolyOverZ| -> Vec<i32> { Self::polys_to_words(m, n).into_iter().map(|v| v as i32).collect() };
        let (rw, ew) = (to32(&r), to32(&e));
        let mut a = vec![0i64; (k + 2) * n];
        let st = unsafe { qf_ring_trap_gen_from(self.ctx.raw, abw.as_ptr(), rw.as_ptr(), ew.as_ptr(), a.as_mut_ptr()) };
        self.ctx.check(st, "qf_ring_trap_gen_from"); // the reference unwrap()s gen_trapdoor_ring_lwe (gpv_ring.rs:96)
        let mut am = MatPolyOverZ::new(1, (k + 2) as i64);
        for j in 0..k + 2 {
            let mut poly = PolyOverZ::default();
            for t in 0..n {
                if a[j * n + t] != 0 {
                    poly.set_coeff(t as i64, Z::from(a[j * n + t])).unwrap();
                }
            }
            am.set_entry(0, j as i64, &poly).unwrap();
        }
        let a_out = MatPolynomialRingZq::from((&am, &gp.modulus));
        *self.installed_a.borrow_mut() = Some(a);
        *self.installed_td.borrow_mut() = None;
        (a_out, (r, e))
    }

    /// gpv_ring.rs:118-122: `D_{Z^{n(k+2)}, s}` folded into k + 2 polynomials
    fn samp_d(&self) -> MatPolyOverZ {
        let mut out = vec![0i32; self.n() * (self.k() + 2)];
        self.ctx.check(unsafe { qf_samp_d(self.ctx.raw, 1, self.next_seed(), 0, out.as_mut_ptr()) }, "qf_samp_d");
        self.domain_from_words(&out)
    }

    /// gpv_ring.rs:160-212
    fn samp_p(&self, a: &MatPolynomialRingZq, td: &Self::Trapdoor, u: &MatPolynomialRingZq) -> MatPolyOverZ {
        self.samp_p_batch(a, td, std::slice::from_ref(u), self.next_seed(), 0).pop().unwrap()
    }

    /// gpv_ring.rs:243-247: `assert!(check_domain(sigma))`, lift sigma to R_q, `a * sigma`
    fn f_a(&self, a: &MatPolynomialRingZq, sigma: &MatPolyOverZ) -> MatPolynomialRingZq {
        self.f_a_batch(a, std::slice::from_ref(sigma)).pop().unwrap()
    }

    /// gpv_ring.rs:274-283: column vector of k + 2 polynomials whose coefficient embedding has squared norm <= s^2 n (k+2)
    fn check_domain(&self, sigma: &MatPolyOverZ) -> bool {
        let Some(sg) = self.domain_to_words(sigma) else { return false };
        let mut ok = [0u8; 1];
        self.ctx.check(unsafe { qf_check_domain(self.ctx.raw, sg.as_ptr(), 1, ok.as_mut_ptr()) }, "qf_check_domain");
        ok[0] == 1
    }
}

impl PSFBatch for PSFGPVRingB200 {
    fn samp_p_batch(&self, a: &MatPolynomialRingZq, td: &Self::Trapdoor, us: &[MatPolynomialRingZq], seed: u64, first_index: u64) -> Vec<MatPolyOverZ> {
        self.install_a(a);
        self.install_td(td);
        let (n, d) = (self.n(), self.n() * (self.k() + 2));
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.get_num_rows() == 1 && u.get_num_columns() == 1, "the syndrome is one ring element");
            uw.extend(Self::polys_to_words(&u.get_representative_least_nonnegative_residue(), n));
        }
        let mut e = vec![0i32; us.len() * d];
        let st = unsafe { qf_samp_p(self.ctx.raw, uw.as_ptr(), us.len() as i64, seed, first_index, e.as_mut_ptr()) };
        self.ctx.check(st, "qf_samp_p"); // the reference unwrap()s the solve and the sampler (gpv_ring.rs:185,211)
        e.chunks(d).map(|row| self.domain_from_words(row)).collect()
    }

    fn f_a_batch(&self, a: &MatPolynomialRingZq, sigmas: &[MatPolyOverZ]) -> Vec<MatPolynomialRingZq> {
        self.install_a(a);
        let (n, d) = (self.n(), self.n() * (self.k() + 2));
        let mut sg = Vec::with_capacity(sigmas.len() * d);
        for sigma in sigmas {
            sg.extend(self.domain_to_words(sigma).expect("sigma is not in D_n")); // gpv_ring.rs:244
        }
        let mut u = vec![0i64; sigmas.len() * n];
        let mut ok = vec![0u8; sigmas.len()];
        let st = unsafe { qf_f_a(self.ctx.raw, sg.as_ptr(), sigmas.len() as i64, u.as_mut_ptr(), ok.as_mut_ptr()) };
        assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n");
        self.ctx.check(st, "qf_f_a");
        u.chunks(n).map(|row| self.range_from_words(row)).collect()
    }

    fn samp_p_batch_packed(&self, a: &MatPolynomialRingZq, td: &Self::Trapdoor, us: &[MatPolynomialRingZq], seed: u64,
                           first_index: u64) -> PackedDomain {
        self.install_a(a);
        self.install_td(td);
        let n = self.n();
        let mut uw = Vec::with_capacity(us.len() * n);
        for u in us {
            assert!(u.get_num_rows() == 1 && u.get_num_columns() == 1, "the syndrome is one ring element");
            uw.extend(Self::polys_to_words(&u.get_representative_least_nonnegative_residue(), n));
        }
        samp_p_packed_run(&self.ctx, &uw, us.len(), seed, first_index)
    }

    fn f_a_batch_packed(&self, a: &MatPolynomialRingZq, packed: &PackedDomain) -> Vec<MatPolynomialRingZq> {
        self.install_a(a);
        f_a_packed_run(&self.ctx, self.n(), packed).chunks(self.n()).map(|row| self.range_from_words(row)).collect()
    }
}

impl PSFGPVRingB200 {
    /// f_a with a key per target: `f_a(keys[key_of[b]], sigmas[b])` for every b in one call, e.g. signatures of many
    /// signers (qf_ring_set_key_table + qf_ring_f_a_keyed).  The table is uploaded once and kept while the same keys come
    /// back; the installed key of `f_a` / `samp_p` is not touched.  Panics like `f_a` when a sigma is outside D_n.
    pub fn f_a_keyed_batch(&self, keys: &[MatPolynomialRingZq], sigmas: &[MatPolyOverZ], key_of: &[usize]) -> Vec<MatPolynomialRingZq> {
        assert_eq!(sigmas.len(), key_of.len(), "one key index per sigma");
        self.install_key_table(keys);
        let (n, d) = (self.n(), self.n() * (self.k() + 2));
        let mut sg = Vec::with_capacity(sigmas.len() * d);
        for sigma in sigmas {
            sg.extend(self.domain_to_words(sigma).expect("sigma is not in D_n")); // gpv_ring.rs:244
        }
        let idx: Vec<i32> = key_of.iter().map(|&t| i32::try_from(t).expect("key index below 2^31")).collect();
        let mut u = vec![0i64; sigmas.len() * n];
        let mut ok = vec![0u8; sigmas.len()];
        let st = unsafe {
            qf_ring_f_a_keyed(self.ctx.raw, sg.as_ptr(), idx.as_ptr(), sigmas.len() as i64, u.as_mut_ptr(), ok.as_mut_ptr())
        };
        assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n");
        self.ctx.check(st, "qf_ring_f_a_keyed");
        u.chunks(n).map(|row| self.range_from_words(row)).collect()
    }

    /// `f_a_keyed_batch` on packed signatures (qf_ring_f_a_keyed_packed): row b of `packed` is the code of sigma b, as
    /// `samp_p_batch_packed` returns it, decoded on the device inside the keyed kernels.  Panics like `f_a` when a sigma is
    /// outside D_n or its code is not canonical.
    pub fn f_a_keyed_batch_packed(&self, keys: &[MatPolynomialRingZq], packed: &PackedDomain, key_of: &[usize]) -> Vec<MatPolynomialRingZq> {
        assert_eq!(packed.rows.len(), key_of.len(), "one key index per sigma");
        self.install_key_table(keys);
        let (n, slot) = (self.n(), packed.slot_bytes as usize);
        let mut buf = vec![0u8; packed.rows.len() * slot];
        for (dst, row) in buf.chunks_mut(slot).zip(&packed.rows) {
            assert!(row.len() <= slot, "a packed row is longer than its slot");
            dst[..row.len()].copy_from_slice(row);
        }
        let idx: Vec<i32> = key_of.iter().map(|&t| i32::try_from(t).expect("key index below 2^31")).collect();
        let b = packed.rows.len();
        let mut u = vec![0i64; b * n];
        let mut ok = vec![0u8; b];
        let st = unsafe {
            qf_ring_f_a_keyed_packed(self.ctx.raw, buf.as_ptr(), idx.as_ptr(), b as i64, packed.k, packed.slot_bytes,
                                     u.as_mut_ptr(), ok.as_mut_ptr())
        };
        assert!(st != QF_ERR_NOT_IN_DOMAIN && ok.iter().all(|f| *f == 1), "sigma is not in D_n");
        self.ctx.check(st, "qf_ring_f_a_keyed_packed");
        u.chunks(n).map(|row| self.range_from_words(row)).collect()
    }

    // the key table of the keyed calls: uploaded once and kept while the same keys come back
    fn install_key_table(&self, keys: &[MatPolynomialRingZq]) {
        let mut kw = Vec::with_capacity(keys.len() * self.n() * (self.k() + 2));
        for a in keys {
            kw.extend(self.key_words(a));
        }
        if self.installed_keys.borrow().as_ref() != Some(&kw) {
            let st = unsafe { qf_ring_set_key_table(self.ctx.raw, kw.as_ptr(), keys.len() as i64) };
            self.ctx.check(st, "qf_ring_set_key_table");
            *self.installed_keys.borrow_mut() = Some(kw);
        }
    }

    /// gen_trapdoor_ring_lwe (gadget_ring.rs:62-81) for many (a_bar, r, e) in one call (qf_ring_trap_gen_batch_from): key t
    /// equals the single-key result bit for bit.  Installs nothing.
    pub fn gen_trapdoor_ring_lwe_batch(&self, a_bars: &[PolyOverZ], rs: &[MatPolyOverZ], es: &[MatPolyOverZ]) -> Vec<MatPolynomialRingZq> {
        assert!(a_bars.len() == rs.len() && rs.len() == es.len(), "one (a_bar, r, e) per key");
        let (n, k) = (self.n(), self.k());
        let q = self.inner.gp.modulus.get_q();
        let mut abw = Vec::with_capacity(a_bars.len() * n);
        for a_bar in a_bars {
            let mut ab = MatPolyOverZ::new(1, 1);
            ab.set_entry(0, 0, a_bar).unwrap();
            abw.extend(Self::polys_to_words(&ab, n).into_iter().map(|v| {
                let r = Z::from(v) % &q; // least non-negative residue, as the reference reduces a_bar
                i64::try_from(&r).unwrap()
            }));
        }
        let to32 = |ms: &[MatPolyOverZ]| -> Vec<i32> {
            ms.iter().flat_map(|m| Self::polys_to_words(m, n).into_iter().map(|v| i32::try_from(v).expect("small coefficients"))).collect()
        };
        let (rw, ew) = (to32(rs), to32(es));
        let mut a = vec![0i64; a_bars.len() * (k + 2) * n];
        let st = unsafe {
            qf_ring_trap_gen_batch_from(self.ctx.raw, a_bars.len() as i64, abw.as_ptr(), rw.as_ptr(), ew.as_ptr(), a.as_mut_ptr())
        };
        self.ctx.check(st, "qf_ring_trap_gen_batch_from");
        a.chunks((k + 2) * n)
            .map(|key| {
                let mut am = MatPolyOverZ::new(1, (k + 2) as i64);
                for j in 0..k + 2 {
                    let mut poly = PolyOverZ::default();
                    for t in 0..n {
                        if key[j * n + t] != 0 {
                            poly.set_coeff(t as i64, Z::from(key[j * n + t])).unwrap();
                        }
                    }
                    am.set_entry(0, j as i64, &poly).unwrap();
                }
                MatPolynomialRingZq::from((&am, &self.inner.gp.modulus))
            })
            .collect()
    }
}

#[allow(dead_code)]
fn _ring_element(poly: &PolynomialRingZq) -> PolyOverZ {
    poly.get_representative_least_nonnegative_residue()
}
