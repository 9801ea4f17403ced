"""Keyed ring f_a on packed sigma (qf_ring_f_a_keyed_packed[_dev], DESIGN.md 4.13): slots in the code of DESIGN 4.11,
decoded inside the keyed NTT kernels (ring_small, Goldilocks) or into a staging buffer first (schoolbook, n = 1024).  Every
row is compared bit for bit with qf_ring_f_a_keyed on the int32 rows the slots encode, u and in_domain, for each family."""
import math

import numpy as np
import pytest

from test_domain_code_math import INT32_MAX, h0_bytes, ref_decode, ref_encode_batch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _ring_s(n):
    return ((2 * 2 * 1.005 * math.sqrt(n) + 1) * 2) * 4  # gpv_ring.rs:296-298 (522.6 at n = 256, as in bench.py)


def _psf(T, n, q):
    gp = T.GadgetParametersRing.init_default(n, q)
    return gp, T.PSFGPVRing(gp, float(_ring_s(n)), 1.005)


def _keys(rng, gp, count):
    return rng.integers(0, gp.q, (count, gp.k + 2, gp.n), dtype=np.int64)


def _slot_for(x, k, extra=0):
    """the smallest valid slot that holds every row of x, plus extra bytes"""
    dim = x.shape[1]
    hbits = ((np.abs(x.astype(np.int64)) >> k) + 1).sum(axis=1).max()
    need = h0_bytes(dim, k) + max(-(-int(hbits) // 8), -(-dim // 8))
    return -(-need // 16) * 16 + extra


def _encode(x, k, slot):
    """device encoder (qf_domain_encode_dev); every row must fit"""
    import torch

    from tools_b200 import domain_code

    p, nb = domain_code.encode(torch.from_numpy(np.ascontiguousarray(x.reshape(len(x), -1), dtype=np.int32)).cuda(), k, slot)
    assert bool((nb > 0).all())
    return p.cpu().numpy()


def _int32_rows(psf, keys, sig, idx):
    """u and flags of qf_ring_f_a_keyed on the int32 rows"""
    return psf.f_a_keyed_batch(keys, sig, idx, strict=False)


def _sigmas(psf, gp, count, seed, scaled=(3, 40, 41)):
    """samp_d rows (in the domain) and a few rows out of it: scaled by 3, and one entry of 1.1 s sqrt(dim) (the bound on
    ||x||^2 is dim s^2)"""
    sig = psf.samp_d_batch(count, seed=seed).astype(np.int32)
    big = int(1.1 * psf.s * math.sqrt(sig[0].size)) + 1
    for b in scaled:
        if b < count:
            sig[b] *= 3
            sig[b, 0, 0] = big
    return sig


# (n, q, env): ring_small d = 2 (C3) and complete (257 at n = 64, 7681 at n = 256: the 3-block tile), ring_small at n = 1024
# (decoded first); Goldilocks (C3 with the small NTT disabled, q = 2^16); schoolbook (n < 64, n not a power of two)
FAMILIES = [
    (256, 3329, None),
    (64, 257, None),
    (256, 7681, None),
    (1024, 12289, None),
    (256, 3329, "QF_DISABLE_SMALL_NTT"),
    (128, 2**16, None),
    (32, 257, None),
    (6, 32, None),
]


@pytest.mark.parametrize("n,q,env", FAMILIES)
def test_families_bit_exact(T, monkeypatch, n, q, env):
    if env:
        monkeypatch.setenv(env, "1")
    rng = np.random.default_rng(n * 3 + q % 991)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 37)
    count = 300 if n == 1024 else 700
    sig = _sigmas(psf, gp, count, seed=5)
    idx = rng.integers(0, len(keys), count).astype(np.int32)
    u0, ok0 = _int32_rows(psf, keys, sig, idx)
    assert not ok0[3] and ok0.sum() >= count - 3
    k_rec, slot_rec = psf.domain_code_params()
    flat = sig.reshape(count, -1)
    # the recommended code; k = 0 (a long high stream, about s / 2.5 bits per entry: on fewer rows); a larger k; slots at
    # the size the rows need and larger
    for k, extra in [(k_rec, None), (k_rec, 4096), (0, 0), (0, 48), (min(k_rec + 4, 30), 16)]:
        m = count if k else (24 if n == 1024 else 96)
        slot = max(slot_rec, _slot_for(flat[:m], k)) if extra is None else _slot_for(flat[:m], k, extra)
        p = _encode(flat[:m], k, slot)
        u, ok = psf.f_a_keyed_packed_batch(keys, p, idx[:m], k=k, strict=False)
        assert np.array_equal(ok, ok0[:m]), (k, slot)
        assert np.array_equal(u, u0[:m]), (k, slot)


def _pick_k(dim, k):
    """k or k + 1, whichever leaves padding bits after the fixed fields (none exist when dim (k + 1) is a multiple of 128)"""
    return k if dim * (k + 1) % 128 else k + 1


@pytest.mark.parametrize("n,q,env", [(256, 3329, None), (64, 257, None), (256, 3329, "QF_DISABLE_SMALL_NTT"), (6, 32, None)])
def test_non_canonical_rows(T, monkeypatch, n, q, env):
    """each rejection case of the format on its own row: in_domain 0 there, every other row's u and flag unchanged"""
    if env:
        monkeypatch.setenv(env, "1")
    rng = np.random.default_rng(q + n)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 9)
    count = 64
    sig = psf.samp_d_batch(count, seed=8).astype(np.int32)
    flat = sig.reshape(count, -1)
    dim = flat.shape[1]
    flat[5, 17] = 0  # an entry of magnitude 0 for the sign case
    idx = rng.integers(0, len(keys), count).astype(np.int32)
    u0, ok0 = _int32_rows(psf, keys, sig, idx)
    assert ok0.all()
    k_rec, _ = psf.domain_code_params()
    k = _pick_k(dim, k_rec)
    slot = _slot_for(flat, k, 64)
    p = _encode(flat, k, slot)
    bits = np.unpackbits(p, axis=1, bitorder="little")
    h0b = 8 * h0_bytes(dim, k)
    bad = {}
    if dim * (k + 1) < h0b:  # a padding bit of the fixed part
        bits[2, dim * (k + 1)] = 1
        bad[2] = "fixed padding"
    bits[4, -1] = 1  # a padding bit of the tail
    bad[4] = "tail padding"
    bits[5, 17 * (k + 1) + k] = 1  # sign 1 on magnitude 0
    bad[5] = "negative zero"
    ones = np.flatnonzero(bits[7, h0b:]) + h0b
    bits[7, ones[-1]] = 0  # the last terminator removed: fewer than dim
    bad[7] = "missing terminator"
    ones = np.flatnonzero(bits[9, h0b:]) + h0b
    bits[9, ones[-1] + 1] = 1  # one terminator more than dim
    bad[9] = "extra terminator"
    ones = np.flatnonzero(bits[11, h0b:]) + h0b
    mid = np.flatnonzero(bits[11, h0b:ones[-1]] == 0)
    if len(mid):  # a zero bit of a high part turned into a terminator mid-row
        bits[11, h0b + mid[len(mid) // 2]] = 1
        bad[11] = "split high part"
    pb = np.packbits(bits, axis=1, bitorder="little")
    for b in bad:
        assert not ref_decode(pb[b], dim, k)[1], bad[b]
    u, ok = psf.f_a_keyed_packed_batch(keys, pb, idx, k=k, strict=False)
    want = ok0.copy()
    want[list(bad)] = False
    assert np.array_equal(ok, want), (np.flatnonzero(ok != want), bad)
    keep = np.ones(count, bool)
    keep[list(bad)] = False
    assert np.array_equal(u[keep], u0[keep])
    with pytest.raises(T.NotInDomain):
        psf.f_a_keyed_packed_batch(keys, pb, idx, k=k)


@pytest.mark.parametrize("n,q,env", [(256, 3329, None), (256, 3329, "QF_DISABLE_SMALL_NTT"), (6, 32, None)])
def test_magnitude_above_int32(T, monkeypatch, n, q, env):
    """k = 30: entry 0 of row 1 is INT32_MAX (h = 1); one more zero bit in front of its terminator gives h = 2, a magnitude
    above INT32_MAX"""
    if env:
        monkeypatch.setenv(env, "1")
    rng = np.random.default_rng(31)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 3)
    sig = psf.samp_d_batch(4, seed=2).astype(np.int32)
    flat = sig.reshape(4, -1)
    dim = flat.shape[1]
    flat[1, 0] = INT32_MAX
    idx = np.array([0, 1, 2, 1], np.int32)
    u0, ok0 = _int32_rows(psf, keys, sig, idx)
    k = 30
    slot = _slot_for(flat, k, 16)
    p = _encode(flat, k, slot)
    bits = np.unpackbits(p, axis=1, bitorder="little")
    h0b = 8 * h0_bytes(dim, k)
    assert bits[1, h0b: h0b + 2].tolist() == [0, 1] and bits[1, -1] == 0
    bits[1, h0b + 1:] = bits[1, h0b:-1].copy()
    bits[1, h0b] = 0
    pb = np.packbits(bits, axis=1, bitorder="little")
    assert not ref_decode(pb[1], dim, k)[1]
    u, ok = psf.f_a_keyed_packed_batch(keys, pb, idx, k=k, strict=False)
    assert ok.tolist() == [ok0[0], False, ok0[2], ok0[3]] and ok0[[0, 2, 3]].all()
    assert np.array_equal(u[[0, 2, 3]], u0[[0, 2, 3]])


def test_forms_splits_chunks(T):
    """host and device forms agree; splits over calls and small chunks (the host form's double buffers cross many chunk
    boundaries); an empty batch"""
    import torch

    from tools_b200 import _ffi

    n, q = 256, 3329
    rng = np.random.default_rng(41)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 100)
    count = 3000
    sig = _sigmas(psf, gp, count, seed=6)
    idx = rng.integers(0, len(keys), count).astype(np.int32)
    u0, ok0 = _int32_rows(psf, keys, sig, idx)
    k, slot = psf.domain_code_params()
    slot = max(slot, _slot_for(sig.reshape(count, -1), k))  # (the scaled rows need more than the recommended slot)
    p = _encode(sig.reshape(count, -1), k, slot)
    u, ok = psf.f_a_keyed_packed_batch(keys, p, idx, strict=False)
    assert np.array_equal(u, u0) and np.array_equal(ok, ok0)
    parts = [psf.f_a_keyed_packed_batch(keys, p[i:j], idx[i:j], strict=False) for i, j in ((0, 1), (1, 1333), (1333, count))]
    assert np.array_equal(np.concatenate([a for a, _ in parts]), u)
    assert np.array_equal(np.concatenate([b for _, b in parts]), ok)
    for chunk in (1, 128, 300, 1000):
        _, small = _psf(T, n, q)
        small.ctx.call("qf_set_chunk", chunk)
        m = 260 if chunk == 1 else count
        us, oks = small.f_a_keyed_packed_batch(keys, p[:m], idx[:m], strict=False)
        assert np.array_equal(us, u[:m]) and np.array_equal(oks, ok[:m]), chunk
    # device form, also on a context with small chunks
    dev = torch.device("cuda:0")
    pd, idd = torch.from_numpy(p).to(dev), torch.from_numpy(idx).to(dev)
    for ctx_psf in (psf, small):
        ud = torch.empty((count, n), dtype=torch.int64, device=dev)
        fd = torch.empty(count, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        ctx_psf.ctx.call("qf_ring_f_a_keyed_packed_dev", _ffi.ptr(pd.data_ptr()), _ffi.ptr(idd.data_ptr()), count, k, slot,
                         _ffi.ptr(ud.data_ptr()), _ffi.ptr(fd.data_ptr()))
        ctx_psf.ctx.call("qf_synchronize")
        assert np.array_equal(ud.cpu().numpy(), u) and np.array_equal(fd.cpu().numpy().astype(bool), ok)
    # batch = 0, host and device
    assert psf.ctx.status("qf_ring_f_a_keyed_packed", None, None, 0, k, slot, None, None) == _ffi.QF_OK
    assert psf.ctx.status("qf_ring_f_a_keyed_packed_dev", None, None, 0, k, slot, None, None) == _ffi.QF_OK
    u_e, ok_e = psf.f_a_keyed_packed_batch(keys, p[:0], idx[:0])
    assert u_e.shape == (0, n) and ok_e.shape == (0,)


def test_refusals(T):
    import torch

    from tools_b200 import _ffi

    n, q = 64, 3329
    rng = np.random.default_rng(43)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 4)
    count = 300
    sig = psf.samp_d_batch(count, seed=7)
    idx = rng.integers(0, 4, count).astype(np.int32)
    k, slot = psf.domain_code_params()
    p = _encode(sig.reshape(count, -1), k, slot)
    out, fl = np.full((count, n), -7, np.int64), np.empty(count, np.uint8)
    call = lambda ps, ix=idx, kk=k, ss=slot, pp=p: ps.ctx.status(  # noqa: E731
        "qf_ring_f_a_keyed_packed", _ffi.ptr(pp), _ffi.ptr(ix), count, kk, ss, _ffi.ptr(out), _ffi.ptr(fl))
    # no table
    assert call(psf) == _ffi.QF_ERR_NO_KEY
    u, ok = psf.f_a_keyed_packed_batch(keys, p, idx)
    assert ok.all()
    # a bad index on the host: refused before any launch, u_out untouched
    out[:] = -7
    launches = psf.ctx.launch_count()
    bad = idx.copy()
    bad[17] = 4
    assert call(psf, bad) == _ffi.QF_ERR_INVALID and psf.ctx.launch_count() == launches
    assert "target 17" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert (out == -7).all()
    # bad k or slot_bytes, before any launch
    for kk, ss in [(-1, slot), (31, slot), (k, slot + 8), (k, 16)]:
        assert call(psf, idx, kk, ss) == _ffi.QF_ERR_INVALID, (kk, ss)
    assert psf.ctx.launch_count() == launches
    # NULL pointers: u_out mandatory on the host
    assert psf.ctx.status("qf_ring_f_a_keyed_packed", _ffi.ptr(p), _ffi.ptr(idx), count, k, slot, None,
                          _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_ring_f_a_keyed_packed", _ffi.ptr(p), _ffi.ptr(idx), -1, k, slot, _ffi.ptr(out),
                          _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    # QF_ERR_NOT_IN_DOMAIN with in_domain NULL
    pb = p.copy()
    pb[3, -1] |= 0x80
    assert psf.ctx.status("qf_ring_f_a_keyed_packed", _ffi.ptr(pb), _ffi.ptr(idx), count, k, slot, _ffi.ptr(out),
                          None) == _ffi.QF_ERR_NOT_IN_DOMAIN
    keep = np.arange(count) != 3
    assert np.array_equal(out[keep], u[keep])
    # device: a bad index is never used to address the table, reported at qf_synchronize, other rows exact
    dev = torch.device("cuda:0")
    bad[17], bad[200] = 4, 2**31 - 1
    pd, idd = torch.from_numpy(p).to(dev), torch.from_numpy(bad).to(dev)
    ud = torch.empty((count, n), dtype=torch.int64, device=dev)
    fd = torch.empty(count, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    dcall = lambda pptr, ix=idd, f=fd: psf.ctx.status(  # noqa: E731
        "qf_ring_f_a_keyed_packed_dev", _ffi.ptr(pptr), _ffi.ptr(ix.data_ptr()), count, k, slot, _ffi.ptr(ud.data_ptr()),
        _ffi.ptr(f.data_ptr()) if f is not None else None)
    assert dcall(pd.data_ptr()) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert "key index" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    good = np.ones(count, bool)
    good[[17, 200]] = False
    fh = fd.cpu().numpy()
    assert np.array_equal(ud.cpu().numpy()[good], u[good]) and fh[good].all() and not fh[~good].any()
    # device: NULL in_domain; a slot pointer that is not 16-byte aligned
    assert dcall(pd.data_ptr(), f=None) == _ffi.QF_ERR_INVALID
    big = torch.zeros(count * slot + 16, dtype=torch.uint8, device=dev)
    assert dcall(big.data_ptr() + 8) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    # classical context
    cl = T.PSFGPV(T.GadgetParameters.init_default(8, 127), 30.0)
    assert cl.ctx.status("qf_ring_f_a_keyed_packed", _ffi.ptr(p), _ffi.ptr(idx), 1, k, slot, _ffi.ptr(out),
                         _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    assert cl.ctx.status("qf_ring_f_a_keyed_packed_dev", _ffi.ptr(pd.data_ptr()), _ffi.ptr(idd.data_ptr()), 1, k, slot,
                         _ffi.ptr(ud.data_ptr()), _ffi.ptr(fd.data_ptr())) == _ffi.QF_ERR_INVALID


def test_full_size_c3(T):
    """4096 C3 keys from gen_trapdoor_ring_lwe_batch, 65 536 signatures in random key order, packed on the device and sent
    from pinned host memory; every row against qf_ring_f_a_keyed_dev on the int32 rows"""
    import torch

    from tools_b200 import _ffi

    n, q, B, K = 256, 3329, 1 << 16, 4096
    rng = np.random.default_rng(47)
    gp, psf = _psf(T, n, q)
    a_bars = rng.integers(0, q, (K, n), dtype=np.int64)
    rs = rng.integers(-2, 3, (K, gp.k, n)).astype(np.int32)
    es = rng.integers(-2, 3, (K, gp.k, n)).astype(np.int32)
    keys = psf.gen_trapdoor_ring_lwe_batch(a_bars, rs, es)
    dev = torch.device("cuda:0")
    d = n * (gp.k + 2)
    sig = torch.empty((B, d), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_d_dev", B, 53, 0, _ffi.ptr(sig.data_ptr()))
    psf.ctx.call("qf_synchronize")
    k, slot = psf.domain_code_params()
    from tools_b200 import domain_code

    pd, nb = domain_code.encode(sig, k, slot)
    assert bool((nb > 0).all())
    idx_h = rng.integers(0, K, B).astype(np.int32)
    idd = torch.from_numpy(idx_h).to(dev)
    # reference: the int32 keyed call on the device
    psf.ctx.call("qf_ring_set_key_table", _ffi.ptr(np.ascontiguousarray(keys)), K)
    ur = torch.empty((B, n), dtype=torch.int64, device=dev)
    fr = torch.empty(B, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_ring_f_a_keyed_dev", _ffi.ptr(sig.data_ptr()), _ffi.ptr(idd.data_ptr()), B, _ffi.ptr(ur.data_ptr()),
                 _ffi.ptr(fr.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert bool(fr.all())
    # host form from pinned buffers
    ph = torch.empty((B, slot), dtype=torch.uint8).pin_memory()
    ph.copy_(pd.cpu())
    ih = torch.from_numpy(idx_h).pin_memory()
    uh = torch.empty((B, n), dtype=torch.int64).pin_memory()
    fh = torch.empty(B, dtype=torch.uint8).pin_memory()
    psf.ctx.call("qf_ring_f_a_keyed_packed", _ffi.ptr(ph.data_ptr()), _ffi.ptr(ih.data_ptr()), B, k, slot, _ffi.ptr(uh.data_ptr()),
                 _ffi.ptr(fh.data_ptr()))
    assert bool(fh.all())
    assert bool(torch.equal(uh, ur.cpu()))
    # and the device form
    ud = torch.empty((B, n), dtype=torch.int64, device=dev)
    fd = torch.empty(B, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_ring_f_a_keyed_packed_dev", _ffi.ptr(pd.data_ptr()), _ffi.ptr(idd.data_ptr()), B, k, slot,
                 _ffi.ptr(ud.data_ptr()), _ffi.ptr(fd.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert bool(fd.all()) and bool(torch.equal(ud, ur))


def test_end_to_end_one_signer(T):
    """qf_samp_p_packed output of an installed C3 key, verified through a table that holds that key among others: u equals
    the targets, every row in the domain"""
    n, q = 256, 3329
    rng = np.random.default_rng(59)
    gp, psf = _psf(T, n, q)
    a, td = psf.trap_gen(seed=3)
    us = rng.integers(0, q, (400, n), dtype=np.int64)
    packed, nb = psf.samp_p_packed_batch(a, td, us, seed=11)
    assert (nb > 0).all()
    keys = _keys(rng, gp, 6)
    keys[4] = np.asarray(a).reshape(gp.k + 2, n)
    idx = np.full(len(us), 4, np.int32)
    u, ok = psf.f_a_keyed_packed_batch(keys, packed, idx)
    assert ok.all() and np.array_equal(u, us)
    # rows signed under key 4 checked against another key are in the domain but do not verify
    idx2 = idx.copy()
    idx2[::2] = 1
    u2, ok2 = psf.f_a_keyed_packed_batch(keys, packed, idx2)
    assert ok2.all() and np.array_equal(u2[1::2], us[1::2]) and not (u2[::2] == us[::2]).all(axis=1).any()
    # the numpy reference encoder gives the same slots, hence the same result
    k, slot = psf.domain_code_params()
    e = psf.samp_p_batch(a, td, us[:8], seed=11).reshape(8, -1)
    rp, rnb = ref_encode_batch(e, k, slot)
    assert np.array_equal(rp, packed[:8])
