"""Host-side mirror of the reference's `PSF` trait (src/primitive/psf.rs:39-81) and its three
implementations, backed by the CUDA library.  Method names, argument meaning and error
behaviour follow the reference; every method has a `_batch` twin (the extension the
reference lacks: its trait methods reject multi-column inputs, gpv.rs:221).

Values cross the boundary as numpy arrays:
  A (classical)   int64  n x m residues            Domain  int32  m      (batch: B x m)
  A (ring)        int64  (k+2) x n residues        Domain  int32  (k+2) x n  (batch: B x (k+2) x n)
  Range           int64  n residues                (batch: B x n)
"""
from __future__ import annotations

import ctypes
import math
import os
from fractions import Fraction

import numpy as np

from . import _ffi, gadget
from ._ffi import NotInDomain, QfError  # noqa: F401


def _seed(seed):
    return int.from_bytes(os.urandom(8), "little") if seed is None else int(seed) & (2**64 - 1)


def _exact_bound(*factors) -> int:
    v = Fraction(1)
    for f in factors:
        v *= Fraction(f)
    return int(v)  # floor for non-negative values


def _domain_i32(values, domain_shape):
    """Domain batch -> (int32 array, per-row "has an entry outside int32" mask).  A plain astype(int32) wraps silently
    (2^32 -> 0), which would report an out-of-domain sigma as in-domain; such rows are zeroed here and reported through
    the mask: their norm exceeds every admissible bound (s r sqrt(m) < 2^31), so they are outside D_n."""
    v = np.asarray(values)
    assert v.shape[1:] == domain_shape, "sigma has the wrong shape"
    if v.dtype == np.int32:
        return np.ascontiguousarray(v), np.zeros(v.shape[0], dtype=bool)
    lim = 2**31 - 1
    if v.dtype == object:
        big = np.array([[abs(int(x)) > lim for x in row.reshape(-1)] for row in v], dtype=bool).reshape(v.shape)
    elif np.issubdtype(v.dtype, np.integer):
        big = (v > lim) | (v < -lim)
    else:
        big = ~(np.abs(v) <= lim) | (v != np.rint(v))  # non-integers (and NaN) are not lattice points
    oob = big.reshape(v.shape[0], -1).any(axis=1) if v.shape[0] else np.zeros(0, dtype=bool)
    if oob.any():
        v = np.where(big, 0, v)
    return np.ascontiguousarray(v, dtype=np.int32), oob


class _PSFBase:
    """Common plumbing: one qf_ctx, cached key/trapdoor uploads."""

    kind = None

    def _make_ctx(self, n, k, m_bar, base, q, s, r, bound, device):
        self.ctx = _ffi.Context(self.kind, n, k, m_bar, base, q, s, r, bound, device)
        self.device = device
        self.ctx_dim = n * (k + 2) if self.kind == _ffi.QF_PSF_GPV_RING else m_bar + n * k
        self._a_id = None
        self._td_id = None
        self._tags_id = None  # samp_p tag table on the device; dropped there with every key / trapdoor install
        self._fa_tags_id = None  # (tags, h0) of the f_a tag table on the device; dropped there whenever A changes
        self._keep = None

    # -- PSF::samp_d ------------------------------------------------------------------------
    def samp_d_batch(self, batch: int, seed=None, first_index: int = 0) -> np.ndarray:
        out = np.empty((batch,) + self._domain_shape, dtype=np.int32)
        self.ctx.call("qf_samp_d", batch, _seed(seed), first_index, _ffi.ptr(out))
        return out

    def samp_d(self, seed=None) -> np.ndarray:
        return self.samp_d_batch(1, seed)[0]

    # -- PSF::check_domain ------------------------------------------------------------------
    def check_domain_batch(self, sigmas: np.ndarray) -> np.ndarray:
        s, oob = _domain_i32(sigmas, self._domain_shape)
        flags = np.empty(s.shape[0], dtype=np.uint8)
        self.ctx.call("qf_check_domain", _ffi.ptr(s), s.shape[0], _ffi.ptr(flags))
        return flags.astype(bool) & ~oob

    def _shape_ok(self, sigma) -> bool:
        raise NotImplementedError

    def check_domain(self, sigma) -> bool:
        sigma = np.asarray(sigma)
        if not self._shape_ok(sigma):
            return False
        return bool(self.check_domain_batch(sigma.reshape((1,) + self._domain_shape))[0])

    # -- PSF::f_a ---------------------------------------------------------------------------
    def f_a_batch(self, a, sigmas: np.ndarray, strict: bool = True):
        """u[b] = A sigma[b]; returns (u, in_domain).  strict=True raises NotInDomain like the
        reference's assert! when some sigma is outside D_n."""
        self._install_a(a)
        if isinstance(sigmas, np.ndarray) and sigmas.dtype == np.int16:  # narrow Domain form: half the host->device bytes
            assert sigmas.shape[1:] == self._domain_shape, "sigma has the wrong shape"
            s, oob, fn = np.ascontiguousarray(sigmas), np.zeros(sigmas.shape[0], dtype=bool), "qf_f_a_i16"
        else:
            (s, oob), fn = _domain_i32(sigmas, self._domain_shape), "qf_f_a"
        b = s.shape[0]
        u = np.empty((b, self.n), dtype=np.int64)
        flags = np.empty(b, dtype=np.uint8)
        st = self.ctx.status(fn, _ffi.ptr(s), b, _ffi.ptr(u), _ffi.ptr(flags))
        if st not in (_ffi.QF_OK, _ffi.QF_ERR_NOT_IN_DOMAIN):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        ok = flags.astype(bool) & ~oob
        if strict and not ok.all():
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not in the domain D_n")
        return u, ok

    def f_a_tagged_batch(self, a, tags, sigmas: np.ndarray, tag_idx, h0=None, strict: bool = True):
        """f_a with a tag per target (classical contexts): u[b] = A_t sigma[b] with A_t = a + [0 | (H_t - H_0) G],
        H_t = tags[tag_idx[b]], for a key a = [A_bar | H_0 G - A_bar R] (h0 = H_0, None: I; H_0 = 0 is allowed).  That is
        the key gen_trapdoor(A_bar, R, H_t) gives, evaluated from a alone: no trapdoor is needed and no tag is inverted.
        tags: T x n x n or PolyTags, h0: n x n (entries taken mod q); the table (qf_set_f_a_tags[_poly]) is cached on the device by the
        identity of tags and h0 until the key on the device changes: the device drops the table there, and every place
        here that installs or rewrites A resets _fa_tags_id.  tag_idx: B indices in [0, T).  Returns (u, in_domain) as
        f_a_batch does."""
        self._install_a(a)
        self._install_fa_tags(tags, h0)
        s, oob = _domain_i32(sigmas, self._domain_shape)
        ti = np.ascontiguousarray(tag_idx, dtype=np.int32)
        b = s.shape[0]
        assert ti.shape == (b,)
        u = np.empty((b, self.n), dtype=np.int64)
        flags = np.empty(b, dtype=np.uint8)
        st = self.ctx.status("qf_f_a_tagged", _ffi.ptr(s), _ffi.ptr(ti), b, _ffi.ptr(u), _ffi.ptr(flags))
        if st not in (_ffi.QF_OK, _ffi.QF_ERR_NOT_IN_DOMAIN):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        ok = flags.astype(bool) & ~oob
        if strict and not ok.all():
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not in the domain D_n")
        return u, ok

    def _install_fa_tags(self, tags, h0):
        """The f_a tag table of f_a_tagged_batch (qf_set_f_a_tags[_poly]), unless it is on the device already."""
        key = self._fa_tags_id
        if key is None or key[0] is not tags or key[1] is not h0:
            hg = None
            if h0 is not None:
                h = np.asarray(h0)
                hg = np.ascontiguousarray(np.array(h % self.gp.q, dtype=np.int64) if h.dtype == object else h, dtype=np.int64)
                assert hg.shape == (self.n, self.n)
            if isinstance(tags, PolyTags):
                fw, tw = tags.words(self.gp.q)
                assert fw.shape == (self.n,)
                self.ctx.call("qf_set_f_a_tags_poly", _ffi.ptr(fw), _ffi.ptr(tw), tw.shape[0], _ffi.ptr(hg))
            else:
                t = np.asarray(tags)
                tg = np.ascontiguousarray(np.array(t % self.gp.q, dtype=np.int64) if t.dtype == object else t, dtype=np.int64)
                assert tg.ndim == 3 and tg.shape[1:] == (self.n, self.n) and tg.shape[0] >= 1
                self.ctx.call("qf_set_f_a_tags", _ffi.ptr(tg), tg.shape[0], _ffi.ptr(hg))
            self._fa_tags_id = (tags, h0)

    def f_a(self, a, sigma) -> np.ndarray:
        sigma = np.asarray(sigma)
        if not self._shape_ok(sigma):
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not a column vector of the right length")
        u, _ = self.f_a_batch(a, sigma.reshape((1,) + self._domain_shape))
        return u[0]

    # -- PSF::samp_p ------------------------------------------------------------------------
    def samp_p_batch(self, a, td, us: np.ndarray, seed=None, first_index: int = 0, dtype=np.int32) -> np.ndarray:
        """dtype=np.int16 returns the same preimages in 16 bits (qf_samp_p_i16: half the device->host bytes; raises
        QfError if an entry does not fit, which needs 6 s r >= 2^15)."""
        self._install_a(a)
        self._install_td(a, td)
        u = np.ascontiguousarray(us, dtype=np.int64)
        assert u.ndim == 2 and u.shape[1] == self.n
        dtype = np.dtype(dtype)
        assert dtype in (np.dtype(np.int32), np.dtype(np.int16))
        e = np.empty((u.shape[0],) + self._domain_shape, dtype=dtype)
        self.ctx.call("qf_samp_p" if dtype == np.int32 else "qf_samp_p_i16", _ffi.ptr(u), u.shape[0], _seed(seed), first_index,
                      _ffi.ptr(e))
        return e

    def samp_p(self, a, td, u, seed=None) -> np.ndarray:
        return self.samp_p_batch(a, td, np.asarray(u, dtype=np.int64).reshape(1, self.n), seed)[0]

    # -- packed Domain values (DESIGN 4.11) -----------------------------------------------------------------------------
    def domain_code_params(self):
        """(k, slot_bytes) recommended for this context's Gaussian width and dim (qf_domain_code_params)."""
        k, sb = ctypes.c_int(), ctypes.c_int64()
        self.ctx.call("qf_domain_code_params", ctypes.byref(k), ctypes.byref(sb))
        return k.value, sb.value

    def _code_params(self, k, slot_bytes):
        if k is None or slot_bytes is None:
            k0, s0 = self.domain_code_params()
            k, slot_bytes = (k0 if k is None else k), (s0 if slot_bytes is None else slot_bytes)
        return int(k), int(slot_bytes)

    def samp_p_packed_batch(self, a, td, us: np.ndarray, seed=None, first_index: int = 0, tags=None, tag_idx=None, k=None,
                            slot_bytes=None):
        """samp_p with packed output (qf_samp_p_packed): returns (packed uint8 B x slot_bytes, nbytes int32 B).  Row b is the
        code of row b of samp_p_batch (tags: samp_p_tagged_batch, same tags and tag_idx) for the same seed and first_index.
        k / slot_bytes default to domain_code_params().  A row whose code does not fit its slot has nbytes -1 and a zero
        slot; samp_p_batch(a, td, us[b:b+1], seed, first_index + b) gives its preimage."""
        self._install_a(a)
        self._install_td(a, td)
        k, slot_bytes = self._code_params(k, slot_bytes)
        u = np.ascontiguousarray(us, dtype=np.int64)
        assert u.ndim == 2 and u.shape[1] == self.n
        b = u.shape[0]
        ti = None
        if tags is not None:
            if not isinstance(self, _TagTable):
                raise QfError(_ffi.QF_ERR_INVALID, "tags need a classical context")
            if self._tags_id is not tags:
                self.set_tag_table(a, td, tags)
            ti = np.ascontiguousarray(tag_idx, dtype=np.int32)
            assert ti.shape == (b,)
        out = np.empty((b, slot_bytes), dtype=np.uint8)
        nbytes = np.empty(b, dtype=np.int32)
        st = self.ctx.status("qf_samp_p_packed", _ffi.ptr(u), _ffi.ptr(ti), b, _seed(seed), first_index, k, slot_bytes,
                             _ffi.ptr(out), _ffi.ptr(nbytes))
        if st != _ffi.QF_OK and not (st == _ffi.QF_ERR_NUMERIC and (nbytes < 0).any()):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        return out, nbytes

    def f_a_packed_batch(self, a, packed: np.ndarray, k=None, tags=None, tag_idx=None, h0=None, strict: bool = True):
        """f_a on packed Domain values (qf_f_a_packed): packed is B x slot_bytes; returns (u, in_domain) as f_a_batch, with
        in_domain[b] False also when slot b is not a canonical code.  tags / tag_idx / h0 as in f_a_tagged_batch
        (classical contexts).  k defaults to domain_code_params()."""
        self._install_a(a)
        p = np.ascontiguousarray(packed, dtype=np.uint8)
        assert p.ndim == 2
        b, slot_bytes = p.shape
        k, _ = self._code_params(k, slot_bytes)
        ti = None
        if tags is not None:
            if not isinstance(self, _TagTable):
                raise QfError(_ffi.QF_ERR_INVALID, "tags need a classical context")
            self._install_fa_tags(tags, h0)
            ti = np.ascontiguousarray(tag_idx, dtype=np.int32)
            assert ti.shape == (b,)
        u = np.empty((b, self.n), dtype=np.int64)
        flags = np.empty(b, dtype=np.uint8)
        st = self.ctx.status("qf_f_a_packed", _ffi.ptr(p), _ffi.ptr(ti), b, k, slot_bytes, _ffi.ptr(u), _ffi.ptr(flags))
        if st not in (_ffi.QF_OK, _ffi.QF_ERR_NOT_IN_DOMAIN):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        ok = flags.astype(bool)
        if strict and not ok.all():
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not canonical or not in the domain D_n")
        return u, ok


class PolyTags:
    """T tags in polynomial form: tag t is H_t = rot_f(tags[t]) (gadget.rot_f), the matrix of multiplication by the ring
    element tags[t] in Z_q[X]/(f), f = X^n + sum_{i<n} f[i] X^i.  f: n low coefficients of the monic modulus; tags: T x n.
    Entries are taken mod q (negatives allowed).  Accepted wherever a T x n x n tag array is (set_tag_table,
    samp_p_tagged_batch, f_a_tagged_batch) and cached on the device by identity as that is; the device stores n words per
    tag instead of n^2 (DESIGN.md 4.10)."""

    def __init__(self, f, tags):
        self.f = np.asarray(f)
        self.tags = np.asarray(tags)
        assert self.f.ndim == 1 and self.tags.ndim == 2 and self.tags.shape[1] == self.f.shape[0] and len(self.tags) >= 1

    def __len__(self):
        return len(self.tags)

    def matrices(self, q: int) -> np.ndarray:
        """The T x n x n tags rot_f(tags[t]) mod q."""
        return np.stack([gadget.rot_f(h, self.f, q) for h in self.tags])

    def words(self, q: int):
        """(f, tags) as contiguous int64 for the C ABI (object entries are reduced mod q first)."""
        def w(x):
            return np.ascontiguousarray(np.array(x % q, dtype=np.int64) if x.dtype == object else x, dtype=np.int64)

        return w(self.f), w(self.tags)


class _TagTable:
    """samp_p with a tag per target for the classical PSFs whose trapdoor serves every tag of (A_bar, R): PSFPerturbation,
    and PSFGPV on the two-phase recursion (DESIGN.md 4.3, 4.4)."""

    def _tag_words(self, tag):
        tg = np.array(np.asarray(tag, dtype=object) % self.gp.q, dtype=np.int64)
        assert tg.shape == (self.n, self.n)
        return tg

    def set_tag_table(self, a, td, tags):
        """Installs the tag table of samp_p_tagged_batch for the key a (any tag H_0) and its trapdoor td: tags is T x n x n,
        entries taken mod q (qf_set_tag_table: H_t^-1 on the device), or PolyTags (qf_set_tag_table_poly: h_t^-1 mod (f, q)
        on the device; QfError QF_ERR_UNSUPPORTED unless q is a prime power).  Raises QfError (QF_ERR_INVALID, naming the index)
        when a tag has no unit pivot; the previous table then stays.  PSFGPV: QF_ERR_INVALID unless a and td run the
        two-phase recursion (a G-trapdoor key with its basis from gen_short_basis_for_trapdoor, m above the tensor-core
        threshold)."""
        self._install_a(a)
        self._install_td(a, td)
        if isinstance(tags, PolyTags):
            fw, tw = tags.words(self.gp.q)
            assert fw.shape == (self.n,)
            self.ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(tw), tw.shape[0])
            self._tags_id = tags
            return
        t = np.asarray(tags)
        if t.dtype == object:
            t = np.array(t % self.gp.q, dtype=np.int64)
        tg = np.ascontiguousarray(t, dtype=np.int64)
        assert tg.ndim == 3 and tg.shape[1:] == (self.n, self.n) and tg.shape[0] >= 1
        self.ctx.call("qf_set_tag_table", _ffi.ptr(tg), tg.shape[0])
        self._tags_id = tags

    def samp_p_tagged_batch(self, a, td, tags, us: np.ndarray, tag_idx, seed=None, first_index: int = 0) -> np.ndarray:
        """samp_p with a tag per target: row b is a preimage of us[b] under [A_bar | H_t G - A_bar R], H_t = tags[tag_idx[b]],
        for the key a = [A_bar | H_0 G - A_bar R] (any tag H_0) and its trapdoor td.  It equals what set_tag(H_t) followed
        by samp_p_batch on the same targets gives for that row with the same seed and first_index (qf_samp_p_tagged).
        tags: T x n x n (entries taken mod q) or PolyTags, cached on the device by identity as keys are; tag_idx: B indices in [0, T).
        Returns B x m int32."""
        self._install_a(a)
        self._install_td(a, td)
        if self._tags_id is not tags:
            self.set_tag_table(a, td, tags)
        u = np.ascontiguousarray(us, dtype=np.int64)
        assert u.ndim == 2 and u.shape[1] == self.n
        ti = np.ascontiguousarray(tag_idx, dtype=np.int32)
        assert ti.shape == (u.shape[0],)
        e = np.empty((u.shape[0], self.m), dtype=np.int32)
        self.ctx.call("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(ti), u.shape[0], _seed(seed), first_index, _ffi.ptr(e))
        return e

    # -- offline / online samp_p (DESIGN.md 4.12) --------------------------------------------------------------------
    def samp_p_offline(self, a, td, count: int, seed=None, first_index: int = 0):
        """Fills the context's pool with the target-independent half of samp_p for the sampler indices first_index ..
        first_index + count - 1 under seed (qf_samp_p_offline), replacing any previous pool.  Installing another key or
        trapdoor, or switching the key's tag, drops the pool; tag tables keep it.  Refilling an index range already used
        under the same seed serves the same perturbations again: the caller must not do that.  PSFGPV needs the two-phase
        recursion (QfError QF_ERR_UNSUPPORTED otherwise)."""
        self._install_a(a)
        self._install_td(a, td)
        self.ctx.call("qf_samp_p_offline", int(count), _seed(seed), int(first_index))

    def pool_info(self):
        """(remaining entries, sampler index of the next one) of the pool; (0, 0) without a pool."""
        rem, nxt = ctypes.c_int64(), ctypes.c_uint64()
        self.ctx.call("qf_samp_p_pool_info", ctypes.byref(rem), ctypes.byref(nxt))
        return rem.value, nxt.value

    def samp_p_online_batch(self, a, td, us: np.ndarray, tags=None, tag_idx=None):
        """Online half of samp_p for the targets us (B x n) from the next B pool entries (qf_samp_p_online).  Returns
        (e, first_index): row b equals row b of samp_p_batch(a, td, us, seed, first_index) for the pool's seed, or of
        samp_p_tagged_batch with tags / tag_idx as there (matrices or PolyTags).  QfError QF_ERR_INVALID when B exceeds the
        remaining entries (nothing is consumed), QF_ERR_NO_KEY without a pool."""
        self._install_a(a)
        self._install_td(a, td)
        u = np.ascontiguousarray(us, dtype=np.int64)
        assert u.ndim == 2 and u.shape[1] == self.n
        ti = None
        if tags is not None:
            if self._tags_id is not tags:
                self.set_tag_table(a, td, tags)
            ti = np.ascontiguousarray(tag_idx, dtype=np.int32)
            assert ti.shape == (u.shape[0],)
        e = np.empty((u.shape[0], self.m), dtype=np.int32)
        first = ctypes.c_uint64()
        self.ctx.call("qf_samp_p_online", _ffi.ptr(u), _ffi.ptr(ti), u.shape[0], _ffi.ptr(e), ctypes.byref(first))
        return e, first.value


class PSFGPV(_TagTable, _PSFBase):
    """src/primitive/psf/gpv.rs:53-225.  Trapdoor = (short basis S_A, its GSO)."""

    kind = _ffi.QF_PSF_GPV

    def __init__(self, gp: gadget.GadgetParameters, s: float, device: int = 0):
        self.gp, self.s = gp, float(s)
        self.n, self.m = gp.n, gp.m
        self._domain_shape = (gp.m,)
        bound = _exact_bound(s, s, gp.m)  # gpv.rs:223
        self._make_ctx(gp.n, gp.k, gp.m_bar, gp.base, gp.q, s, 1.0, bound, device)

    def _shape_ok(self, sigma):
        return (sigma.ndim == 1 or (sigma.ndim == 2 and sigma.shape[1] == 1)) and sigma.shape[0] == self.m

    def _install_a(self, a):
        if self._a_id is not a:
            aa = np.ascontiguousarray(a, dtype=np.int64)  # keep alive across the call
            self.ctx.call("qf_set_a", _ffi.ptr(aa))
            self._a_id, self._td_id, self._tags_id, self._fa_tags_id = a, None, None, None

    def _install_td(self, a, td):
        if self._td_id is not td:
            s, sg = td
            s = np.ascontiguousarray(s, dtype=np.int64)
            # None: the GSO is computed on the device and stays there
            sg = None if sg is None else np.ascontiguousarray(sg, dtype=np.float64)
            assert s.shape == (self.m, self.m) and (sg is None or sg.shape == (self.m, self.m))
            self.ctx.call("qf_set_trapdoor_gpv", _ffi.ptr(s), _ffi.ptr(sg))
            self._td_id, self._tags_id = td, None

    def trap_gen(self, seed=None, dense_gso: bool = None, tag=None):
        """gpv.rs:83-94: uniform A_bar, gen_trapdoor, short basis, GSO -- all on the device.  dense_gso=False
        leaves the second trapdoor component None (the backend computes the GSO when the trapdoor is installed and
        keeps it in HBM instead of moving m x m doubles through the host twice); default: the reference's
        (S, S~) pair up to m = 2048, None above.
        tag: an n x n matrix H invertible mod q (gadget_classical.rs:56-68 with a tag): A = [A_bar | H G - A_bar R] from
        the same device-sampled A_bar and R (qf_trap_gen_from), and the short basis for that tag.  None: H = I."""
        a, r = _trap_gen_classical(self, seed)
        if tag is not None:
            tg = np.array(np.asarray(tag, dtype=object) % self.gp.q, dtype=np.int64)
            assert tg.shape == (self.n, self.n)
            ab = np.ascontiguousarray(a[:, : self.gp.m_bar])
            a = np.empty((self.n, self.m), dtype=np.int64)
            self.ctx.call("qf_trap_gen_from", _ffi.ptr(ab), _ffi.ptr(r), _ffi.ptr(tg), _ffi.ptr(a))
        short_base = self.gen_short_basis_for_trapdoor(r, tag)
        if dense_gso is None:
            dense_gso = self.m <= 2048
        td = (short_base, self.gso(short_base) if dense_gso else None)
        self._a_id = a  # qf_trap_gen installed it
        return a, td

    def gso(self, basis) -> np.ndarray:
        """MatQ::gso (gpv.rs:91): unnormalised Gram-Schmidt of the columns, float64, on the device."""
        return _gso(self, basis)

    def set_tag(self, a, td, tag):
        """Tag switch without a new trapdoor install: for a key a = [A_bar | H G - A_bar R] and its trapdoor td = (S_H, S~)
        on the two-phase recursion, returns (a_new, td_new) with a_new = [A_bar | H' G - A_bar R] for tag = H' (n x n,
        entries taken mod q; None: H' = I), equal to gen_trapdoor(A_bar, R, H'), and td_new = (S_H', td[1]) with S_H' equal
        to gen_short_basis_for_trapdoor(R, H').  The GSO of S_H does not depend on the tag, so td[1] serves S_H' too (None:
        it stays on the device) and nothing is re-installed: both are recorded as installed (qf_gpv_set_tag).  The tag
        table stays; the f_a tag table is dropped.  Raises QfError (QF_ERR_INVALID) off the two-phase recursion or when H'
        has no unit pivot; then the installed key and tag stay as they were."""
        self._install_a(a)
        self._install_td(a, td)
        tg = None if tag is None else self._tag_words(tag)
        a_new = np.empty((self.n, self.m), dtype=np.int64)
        s_new = np.empty((self.m, self.m), dtype=np.int64)
        self.ctx.call("qf_gpv_set_tag", _ffi.ptr(tg), _ffi.ptr(a_new), _ffi.ptr(s_new))
        td_new = (s_new, td[1])
        self._a_id, self._td_id, self._fa_tags_id = a_new, td_new, None
        return a_new, td_new


    def gen_short_basis_for_trapdoor(self, r, tag=None) -> np.ndarray:
        """short_basis_classical.rs:54-110 for the installed A and the tag H (n x n, entries taken mod q; None: H = I):
        H^-1 and every integer product run on the device (qf_gen_short_basis_tagged); exact.  Raises QfError
        (QF_ERR_INVALID) when H is not invertible by unit pivoting, where the reference panics.
        gadget.gen_short_basis_for_trapdoor is the host restatement (tests)."""
        r8 = np.ascontiguousarray(r, dtype=np.int8)
        assert r8.shape == (self.gp.m_bar, self.gp.n * self.gp.k)
        out = np.empty((self.m, self.m), dtype=np.int64)
        if tag is None:
            self.ctx.call("qf_gen_short_basis", _ffi.ptr(r8), _ffi.ptr(out))
            return out
        tg = np.array(np.asarray(tag, dtype=object) % self.gp.q, dtype=np.int64)
        assert tg.shape == (self.n, self.n)
        self.ctx.call("qf_gen_short_basis_tagged", _ffi.ptr(r8), _ffi.ptr(tg), _ffi.ptr(out))
        return out


class PSFPerturbation(_TagTable, _PSFBase):
    """src/primitive/psf/mp_perturbation.rs:57-403.
    Trapdoor = (R, sqrt(Sigma_2), (S, S~)) with S = I_n (x) S_k the gadget short basis."""

    kind = _ffi.QF_PSF_PERTURBATION

    def __init__(self, gp: gadget.GadgetParameters, r: float, s: float, device: int = 0):
        self.gp, self.r, self.s = gp, float(r), float(s)
        self.n, self.m = gp.n, gp.m
        self._domain_shape = (gp.m,)
        bound = _exact_bound(s, s, gp.m, r, r)  # mp_perturbation.rs:401
        self._make_ctx(gp.n, gp.k, gp.m_bar, gp.base, gp.q, s, r, bound, device)

    _shape_ok = PSFGPV._shape_ok
    _install_a = PSFGPV._install_a

    def _install_td(self, a, td):
        if self._td_id is not td:
            r_mat, sqrt_sigma_2, (s_basis, s_gso) = td
            k, n = self.gp.k, self.gp.n
            r8 = np.ascontiguousarray(r_mat, dtype=np.int8)
            assert np.array_equal(r8, np.asarray(r_mat)), "R entries must fit int8"
            # None: the backend derives its own (block-structured) square root of the default Sigma_2
            l = None if sqrt_sigma_2 is None else np.ascontiguousarray(sqrt_sigma_2, dtype=np.float64)
            sb = np.asarray(s_basis)
            sg = np.asarray(s_gso, dtype=np.float64)
            assert r8.shape == (self.gp.m_bar, n * k) and (l is None or l.shape == (self.m, self.m))
            if sb.shape == (n * k, n * k):
                blk = np.ascontiguousarray(sb[:k, :k], dtype=np.int64)
                gblk = np.ascontiguousarray(sg[:k, :k])
                if n * k <= 4096:  # the backend exploits the block-diagonal structure I_n (x) S_k
                    if not (np.array_equal(sb, np.kron(np.eye(n, dtype=np.int64), blk))
                            and np.allclose(sg, np.kron(np.eye(n), gblk))):
                        raise QfError(_ffi.QF_ERR_UNSUPPORTED, "gadget short basis is not I_n (x) S_k")
            else:
                assert sb.shape == (k, k)
                blk, gblk = np.ascontiguousarray(sb, dtype=np.int64), np.ascontiguousarray(sg)
            self.ctx.call("qf_set_trapdoor_perturbation", _ffi.ptr(r8), _ffi.ptr(l), _ffi.ptr(blk), _ffi.ptr(gblk))
            self._td_id, self._tags_id = td, None
            self._keep = (r8, l, blk, gblk)

    def compute_sqrt_sigma_2(self, mat_r, mat_sigma=None) -> np.ndarray:
        """mp_perturbation.rs:111-139: lower Cholesky factor of r^2/(2 pi) (Sigma - (b^2+1) T T^t - I), T = [R; I],
        Sigma = s^2 I by default; blocked Cholesky on the device.  Raises QfError (QF_ERR_INVALID) when Sigma_2 is
        not positive definite, where the reference panics (:109-110)."""
        r8 = np.ascontiguousarray(mat_r, dtype=np.int8)
        assert np.array_equal(r8, np.asarray(mat_r)) and r8.shape == (self.gp.m_bar, self.gp.n * self.gp.k)
        sig = None if mat_sigma is None else np.ascontiguousarray(mat_sigma, dtype=np.float64)
        assert sig is None or sig.shape == (self.m, self.m)
        out = np.empty((self.m, self.m), dtype=np.float64)
        self.ctx.call("qf_compute_sqrt_sigma_2", _ffi.ptr(r8), _ffi.ptr(sig), _ffi.ptr(out))
        return out

    def randomized_nearest_plane_gadget_batch(self, a, td, vs, seed=None, first_index: int = 0) -> np.ndarray:
        """mp_perturbation.rs:173-191 for a batch of syndromes v (B x n): z = x0 + SampleD(S, S~, -x0, r sqrt(b^2+1)),
        x0 the base-b digits of v (find_solution_gadget_mat); G z = v mod q.  Returns B x (n k) int32."""
        self._install_a(a)
        self._install_td(a, td)
        v = np.ascontiguousarray(vs, dtype=np.int64)
        assert v.ndim == 2 and v.shape[1] == self.n
        z = np.empty((v.shape[0], self.gp.n * self.gp.k), dtype=np.int32)
        self.ctx.call("qf_randomized_nearest_plane_gadget", _ffi.ptr(v), v.shape[0], _seed(seed), first_index, _ffi.ptr(z))
        return z

    def randomized_nearest_plane_gadget(self, a, td, v, seed=None) -> np.ndarray:
        return self.randomized_nearest_plane_gadget_batch(a, td, np.asarray(v, dtype=np.int64).reshape(1, self.n), seed)[0]

    def trap_gen(self, seed=None, full_gadget_basis: bool = None, dense_sqrt_sigma_2: bool = None, tag=None):
        """mp_perturbation.rs:221-244.  dense_sqrt_sigma_2=False leaves the second trapdoor component None: the
        backend then uses its block-structured square root of the default Sigma_2 (same law, ~4x less work per
        target); default: dense (the reference's m x m matrix) up to m = 2048, structured above.
        tag: an n x n matrix H invertible mod q (gadget_classical.rs:56-68 with a tag): A = [A_bar | H G - A_bar R] from
        the same device-sampled A_bar and R (qf_trap_gen_from).  The trapdoor does not depend on H; samp_p recognises the
        tag when the trapdoor is installed.  None: H = I."""
        a, r = _trap_gen_classical(self, seed)
        if tag is not None:
            tg = self._tag_words(tag)
            ab = np.ascontiguousarray(a[:, : self.gp.m_bar])
            a = np.empty((self.n, self.m), dtype=np.int64)
            self.ctx.call("qf_trap_gen_from", _ffi.ptr(ab), _ffi.ptr(r), _ffi.ptr(tg), _ffi.ptr(a))
        if dense_sqrt_sigma_2 is None:
            dense_sqrt_sigma_2 = self.m <= 2048
        sqrt_sigma_2 = self.compute_sqrt_sigma_2(r) if dense_sqrt_sigma_2 else None
        k, n = self.gp.k, self.gp.n
        if full_gadget_basis is None:
            full_gadget_basis = n * k <= 1024
        blk = gadget.short_basis_gadget_block(k, self.gp.base, self.gp.q)
        gblk = gadget.gso_small(blk)  # k x k: exact rational Gram-Schmidt on the host, like MatQ::gso
        if full_gadget_basis:
            sb = gadget.short_basis_gadget(self.gp)
            sg = np.kron(np.eye(n), gblk)
        else:  # one diagonal block; the full matrices are I_n (x) these
            sb, sg = blk, gblk
        self._a_id = a
        return a, (r, sqrt_sigma_2, (sb, sg))

    def set_tag(self, a, td, tag) -> np.ndarray:
        """Tag switch without a new trapdoor install: for a key a = [A_bar | H G - A_bar R] and its trapdoor td (R, ...),
        returns a_new = [A_bar | H' G - A_bar R] for tag = H' (n x n, entries taken mod q; None: H' = I), equal to
        gen_trapdoor(A_bar, R, H'), and records it as the installed key; R, sqrt(Sigma_2) and the gadget basis stay on the
        device (qf_set_tag).  Raises QfError (QF_ERR_INVALID) when a is not such a key for td's R or when H' has no unit
        pivot; then the installed key and tag stay as they were."""
        self._install_a(a)
        self._install_td(a, td)
        tg = None if tag is None else self._tag_words(tag)
        a_new = np.empty((self.n, self.m), dtype=np.int64)
        self.ctx.call("qf_set_tag", _ffi.ptr(tg), _ffi.ptr(a_new))
        self._a_id, self._fa_tags_id = a_new, None  # qf_set_tag rewrote A: the f_a table is gone
        return a_new


def _gso(psf, basis) -> np.ndarray:
    b = np.ascontiguousarray(basis, dtype=np.int64)
    d = psf.ctx_dim
    assert b.shape == (d, d)
    out = np.empty((d, d), dtype=np.float64)
    psf.ctx.call("qf_gso", _ffi.ptr(b), _ffi.ptr(out))
    return out


def _trap_gen_classical(psf, seed):
    gp = psf.gp
    a = np.empty((gp.n, gp.m), dtype=np.int64)
    r = np.empty((gp.m_bar, gp.n * gp.k), dtype=np.int8)
    psf.ctx.call("qf_trap_gen", _seed(seed), _ffi.ptr(a), _ffi.ptr(r))
    psf._td_id = psf._tags_id = psf._fa_tags_id = None
    return a, r


def gen_trapdoor(gp: gadget.GadgetParameters, a_bar, r, tag=None, device: int = 0):
    """gadget_classical.rs:56-68 with A_bar, R (and optionally the tag H) supplied:
    A = [A_bar | H G - A_bar R] mod q, computed on the device, bit-exact."""
    ctx = _ffi.Context(_ffi.QF_PSF_GPV, gp.n, gp.k, gp.m_bar, gp.base, gp.q, 1.0, 1.0, 1, device)
    try:
        a = np.empty((gp.n, gp.m), dtype=np.int64)
        ab = np.ascontiguousarray(a_bar, dtype=np.int64)
        r8 = np.ascontiguousarray(r, dtype=np.int8)
        assert ab.shape == (gp.n, gp.m_bar) and r8.shape == (gp.m_bar, gp.n * gp.k)
        tg = None if tag is None else np.ascontiguousarray(tag, dtype=np.int64)
        ctx.call("qf_trap_gen_from", _ffi.ptr(ab), _ffi.ptr(r8), _ffi.ptr(tg), _ffi.ptr(a))
        return a
    finally:
        ctx.close()


class PSFGPVRing(_PSFBase):
    """src/primitive/psf/gpv_ring.rs:62-284.  Trapdoor = (r, e), k polynomials each.
    The reference rebuilds the short basis and its GSO on every samp_p (:169, :205-211);
    here they are built once per trapdoor and cached."""

    kind = _ffi.QF_PSF_GPV_RING

    def __init__(self, gp: gadget.GadgetParametersRing, s: float, s_td: float, device: int = 0):
        self.gp, self.s, self.s_td = gp, float(s), float(s_td)
        self.n = gp.n
        self._domain_shape = (gp.k + 2, gp.n)
        bound = _exact_bound(s, s, gp.n * (gp.k + 2))  # gpv_ring.rs:281-282
        self._make_ctx(gp.n, gp.k, gp.k + 2, gp.base, gp.q, s, 1.0, bound, device)
        self._keys_id = None  # the ring key table on the device (qf_ring_set_key_table); independent of the installed key

    def _shape_ok(self, sigma):
        # a column vector of k+2 polynomials, each given by (at most) n coefficients
        return sigma.ndim == 2 and sigma.shape == (self.gp.k + 2, self.gp.n)

    def _install_a(self, a):
        if self._a_id is not a:
            aa = np.ascontiguousarray(a, dtype=np.int64)
            assert aa.shape == (self.gp.k + 2, self.gp.n)
            self.ctx.call("qf_ring_set_a", _ffi.ptr(aa))
            self._a_id, self._td_id, self._fa_tags_id = a, None, None

    def _install_td(self, a, td):
        if self._td_id is not td:
            r, e = td
            basis = self.gen_short_basis_for_trapdoor_ring(a, r, e)
            self.ctx.call("qf_set_trapdoor_gpv", _ffi.ptr(basis), None)  # GSO computed on the device
            self._td_id = td

    def gen_short_basis_for_trapdoor_ring(self, a, r, e) -> np.ndarray:
        """short_basis_ring.rs:64-166 in the coefficient embedding (D x D, D = n (k + 2), columns = basis vectors), built by
        the library (`qf_ring_gen_short_basis`: polynomial products on the device) for the key `a` and the trapdoor (r, e)."""
        gp = self.gp
        self._install_a(a)
        rr = np.ascontiguousarray(r, dtype=np.int32)
        ee = np.ascontiguousarray(e, dtype=np.int32)
        assert rr.shape == (gp.k, gp.n) and ee.shape == (gp.k, gp.n)
        d = gp.n * (gp.k + 2)
        basis = np.empty((d, d), dtype=np.int64)
        self.ctx.call("qf_ring_gen_short_basis", _ffi.ptr(rr), _ffi.ptr(ee), _ffi.ptr(basis))
        return basis

    def trap_gen(self, seed=None):
        """gpv_ring.rs:91-98 -> gen_trapdoor_ring_lwe (gadget_ring.rs:62-81):
        uniform a_bar, r and e with coefficients D_{Z, s_td} (SampleZ, trapdoor_distribution.rs:112-122)."""
        gp = self.gp
        seed = _seed(seed)
        # r, e: 2k polynomials of n Gaussian coefficients from the device sampler
        tmp = _ffi.Context(_ffi.QF_PSF_GPV, 1, 1, 2 * gp.k * gp.n - 1, 2, 2, self.s_td, 1.0, 1, self.device)
        try:
            re = np.empty((1, 2 * gp.k * gp.n), dtype=np.int32)
            tmp.call("qf_samp_d", 1, seed ^ 0x52494E47, 0, _ffi.ptr(re))
        finally:
            tmp.close()
        r = re[0, : gp.k * gp.n].reshape(gp.k, gp.n).copy()
        e = re[0, gp.k * gp.n:].reshape(gp.k, gp.n).copy()
        rng = np.random.Generator(np.random.Philox(seed))
        a_bar = rng.integers(0, gp.q, gp.n, dtype=np.int64)
        a = self.gen_trapdoor_ring_lwe(a_bar, r, e)
        return a, (r, e)

    def gen_trapdoor_ring_lwe(self, a_bar, r, e) -> np.ndarray:
        """gadget_ring.rs:62-81 with r, e supplied: A = [1 | a_bar | g^t - (a_bar r + e)], bit-exact."""
        gp = self.gp
        a = np.empty((gp.k + 2, gp.n), dtype=np.int64)
        ab = np.ascontiguousarray(a_bar, dtype=np.int64)
        rr = np.ascontiguousarray(r, dtype=np.int32)
        ee = np.ascontiguousarray(e, dtype=np.int32)
        assert ab.shape == (gp.n,) and rr.shape == (gp.k, gp.n) and ee.shape == (gp.k, gp.n)
        self.ctx.call("qf_ring_trap_gen_from", _ffi.ptr(ab), _ffi.ptr(rr), _ffi.ptr(ee), _ffi.ptr(a))
        self._a_id, self._td_id, self._fa_tags_id = a, None, None
        return a

    def f_a_keyed_batch(self, keys, sigmas: np.ndarray, key_idx, strict: bool = True):
        """f_a with a key per target: u[b] = f_a(keys[key_idx[b]], sigmas[b]), for batches that hold signatures of many
        signers.  keys: T x (k+2) x n residues in [0, q) (any a_0); installed as one device table
        (qf_ring_set_key_table) and cached by the identity of `keys`, so pass the same array again to skip the upload.
        key_idx: B indices in [0, T).  Returns (u, in_domain) as f_a_batch does; rows in the domain equal f_a_batch with
        that row's key, bit for bit."""
        if self._keys_id is not keys:
            kk = np.ascontiguousarray(keys, dtype=np.int64)
            assert kk.ndim == 3 and kk.shape[1:] == self._domain_shape and kk.shape[0] >= 1
            self.ctx.call("qf_ring_set_key_table", _ffi.ptr(kk), kk.shape[0])
            self._keys_id = keys
        s, oob = _domain_i32(sigmas, self._domain_shape)
        ki = np.ascontiguousarray(key_idx, dtype=np.int32)
        b = s.shape[0]
        assert ki.shape == (b,)
        u = np.empty((b, self.n), dtype=np.int64)
        flags = np.empty(b, dtype=np.uint8)
        st = self.ctx.status("qf_ring_f_a_keyed", _ffi.ptr(s), _ffi.ptr(ki), b, _ffi.ptr(u), _ffi.ptr(flags))
        if st not in (_ffi.QF_OK, _ffi.QF_ERR_NOT_IN_DOMAIN):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        ok = flags.astype(bool) & ~oob
        if strict and not ok.all():
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not in the domain D_n")
        return u, ok

    def f_a_keyed_packed_batch(self, keys, packed: np.ndarray, key_idx, k=None, strict: bool = True):
        """f_a_keyed_batch on packed Domain values (qf_ring_f_a_keyed_packed): packed is B x slot_bytes, one slot per
        signature in the code of f_a_packed_batch; the table is installed as in f_a_keyed_batch.  k defaults to
        domain_code_params().  Returns (u, in_domain), in_domain[b] False also when slot b is not a canonical code; rows in
        the domain equal f_a_keyed_batch on the decoded sigma, bit for bit.  Pin `packed` (and the outputs) for the copies
        to overlap the computation."""
        if self._keys_id is not keys:
            kk = np.ascontiguousarray(keys, dtype=np.int64)
            assert kk.ndim == 3 and kk.shape[1:] == self._domain_shape and kk.shape[0] >= 1
            self.ctx.call("qf_ring_set_key_table", _ffi.ptr(kk), kk.shape[0])
            self._keys_id = keys
        p = np.ascontiguousarray(packed, dtype=np.uint8)
        assert p.ndim == 2
        b, slot_bytes = p.shape
        k, _ = self._code_params(k, slot_bytes)
        ki = np.ascontiguousarray(key_idx, dtype=np.int32)
        assert ki.shape == (b,)
        u = np.empty((b, self.n), dtype=np.int64)
        flags = np.empty(b, dtype=np.uint8)
        st = self.ctx.status("qf_ring_f_a_keyed_packed", _ffi.ptr(p), _ffi.ptr(ki), b, k, slot_bytes, _ffi.ptr(u),
                             _ffi.ptr(flags))
        if st not in (_ffi.QF_OK, _ffi.QF_ERR_NOT_IN_DOMAIN):
            raise QfError(st, self.ctx._lib.qf_last_error(self.ctx._h).decode())
        ok = flags.astype(bool)
        if strict and not ok.all():
            raise NotInDomain(_ffi.QF_ERR_NOT_IN_DOMAIN, "sigma is not canonical or not in the domain D_n")
        return u, ok

    def gen_trapdoor_ring_lwe_batch(self, a_bars, rs, es) -> np.ndarray:
        """gen_trapdoor_ring_lwe for T keys in one call (qf_ring_trap_gen_batch_from): a_bars T x n residues in [0, q),
        rs and es T x k x n.  Key t equals gen_trapdoor_ring_lwe(a_bars[t], rs[t], es[t]) bit for bit; nothing is
        installed on the context."""
        gp = self.gp
        ab = np.ascontiguousarray(a_bars, dtype=np.int64)
        rr = np.ascontiguousarray(rs, dtype=np.int32)
        ee = np.ascontiguousarray(es, dtype=np.int32)
        t = ab.shape[0]
        assert ab.shape == (t, gp.n) and rr.shape == (t, gp.k, gp.n) and ee.shape == (t, gp.k, gp.n)
        a = np.empty((t, gp.k + 2, gp.n), dtype=np.int64)
        self.ctx.call("qf_ring_trap_gen_batch_from", t, _ffi.ptr(ab), _ffi.ptr(rr), _ffi.ptr(ee), _ffi.ptr(a))
        return a
