"""Packed Domain values on the device (domain_code.cu, qf_samp_p_packed, qf_f_a_packed; DESIGN.md 4.11).  The encoder is
compared byte for byte with the numpy reference of test_domain_code_math.py, the decoder with the rows it encoded, and the
packed samp_p / f_a entry points with the int32 ones on the same seeds."""
import math

import numpy as np
import pytest

from test_domain_code_math import INT32_MAX, INT32_MIN, h0_bytes, ref_decode, ref_encode, ref_encode_batch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _slot(dim, k, extra=16):
    return -(-(h0_bytes(dim, k) + -(-dim // 8)) // 16) * 16 + extra


def _dev_encode(x, k, slot):
    import torch

    from tools_b200 import domain_code

    p, nb = domain_code.encode(torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).cuda(), k, slot)
    return p.cpu().numpy(), nb.cpu().numpy()


def _dev_decode(p, dim, k):
    import torch

    from tools_b200 import domain_code

    v, ok = domain_code.decode(torch.from_numpy(np.ascontiguousarray(p, dtype=np.uint8)).cuda(), dim, k)
    return v.cpu().numpy(), ok.cpu().numpy()


def _check_code(x, k, slot):
    """device encode == reference encode; device decode gives x back on every row that fits."""
    p, nb = _dev_encode(x, k, slot)
    rp, rnb = ref_encode_batch(x, k, slot)
    assert np.array_equal(nb, rnb)
    assert np.array_equal(p, rp)
    v, ok = _dev_decode(p, x.shape[1], k)
    fit = nb >= 0
    assert ok[fit].all() and np.array_equal(v[fit], x[fit])
    return p, nb


@pytest.mark.parametrize("dim", [105, 3584, 12352])
@pytest.mark.parametrize("k", [0, 8, 30])
def test_encoder_matches_reference(T, dim, k):
    rng = np.random.default_rng(dim + k)
    w = {0: 3.0, 8: 1428.0, 30: 1428.0}[k]
    x = np.rint(rng.normal(0, w / math.sqrt(2 * math.pi), (24, dim))).astype(np.int64)
    ext = np.array([0, 1, -1, (1 << k) - 1, -((1 << k) - 1), 1 << k, -(1 << k)], dtype=np.int64)
    x[3] = np.resize(ext, dim)
    if k == 30:
        x[4, ::7] = INT32_MAX
        x[5, 1::9] = -INT32_MAX
    x[6, dim // 2] = INT32_MIN  # overflow
    x[7] = 0
    k_slot = _slot(dim, k, 16 * int(dim * (2 + w / (2**k)) / 128) + 64)
    _, nb = _check_code(x, k, k_slot)
    assert nb[6] == -1 and (nb[np.arange(24) != 6] > 0).all()


def test_encoder_on_samp_d_and_global_slot(T):
    """samp_d output of a C2-width PSFGPV context at the recommended parameters, and at k = 2, where the slot (~440 KB) is
    above what shared memory holds and the encoder assembles it in place."""
    gp = T.GadgetParameters.init_default(256, 2**24)
    psf = T.PSFGPV(gp, 1428.0)
    k, slot = psf.domain_code_params()
    assert k == 8 and abs(slot - (h0_bytes(gp.m, 8) + gp.m * 11.31 / 8 - gp.m * 9 / 8)) < 0.03 * slot
    x = psf.samp_d_batch(64, seed=3).astype(np.int64)
    _, nb = _check_code(x, k, slot)
    assert (nb > 0).all() and nb.max() <= slot
    big = _slot(gp.m, 2, 16 * ((gp.m * 300 // 8) // 16))
    assert big > 232448
    _check_code(x[:6], 2, big)


def test_exact_fit_and_one_bit_over(T):
    for dim, k in [(105, 3), (3584, 0), (12352, 8)]:
        slot = _slot(dim, k, 32)
        budget = 8 * (slot - h0_bytes(dim, k))
        x = np.zeros((3, dim), dtype=np.int64)
        x[0, -1] = (budget - dim) << k  # last terminator = last bit of the slot
        x[1, 0] = -(((budget - dim + 1) << k) | ((1 << k) - 1 if k else 0))  # one bit over
        x[2, 5] = 7
        if x[0, -1] > INT32_MAX or -x[1, 0] > INT32_MAX:
            continue
        _, nb = _check_code(x, k, slot)
        assert nb[0] == slot and nb[1] == -1 and nb[2] > 0


def test_decoder_rejects_each_malformed_case(T):
    dim, k = 300, 5
    slot = _slot(dim, k, 512)  # room for the longest row: 13 high-stream bits per entry
    rng = np.random.default_rng(1)
    x = rng.integers(-400, 401, (8, dim))
    x[x == 0] = 3
    p, nb = _check_code(x, k, slot)
    assert (nb > 0).all() and nb.max() < slot
    h0 = h0_bytes(dim, k)
    bits = np.unpackbits(p, axis=1, bitorder="little")
    # row 1: -0 (sign of an entry whose magnitude is 0)
    x0 = x[1].copy()
    x0[10] = 0
    e0, _ = ref_encode(x0, k, slot)
    bits[1] = np.unpackbits(e0, bitorder="little")
    bits[1, 10 * (k + 1) + k] = 1
    # row 2: the last terminator removed (fewer than dim 1 bits)
    bits[2, np.flatnonzero(bits[2])[-1]] = 0
    # row 3: a padding bit of the fixed part
    assert dim * (k + 1) < 8 * h0
    bits[3, dim * (k + 1)] = 1
    # row 4: a bit in the tail after the dim-th terminator
    bits[4, -1] = 1
    bad = np.packbits(bits, axis=1, bitorder="little")
    for b in (1, 2, 3, 4):
        assert not ref_decode(bad[b], dim, k)[1]
    v, ok = _dev_decode(bad, dim, k)
    assert ok.tolist() == [1, 0, 0, 0, 0, 1, 1, 1]
    keep = [0, 5, 6, 7]
    assert np.array_equal(v[keep], x[keep])
    # magnitude above INT32_MAX at k = 30
    d2, k2 = 3, 30
    s2 = _slot(d2, k2)
    y = np.array([[INT32_MAX, -5, 0], [1, 2, 3]], dtype=np.int64)
    p2, _ = _check_code(y, k2, s2)
    b2 = np.unpackbits(p2, axis=1, bitorder="little")
    h0b = 8 * h0_bytes(d2, k2)
    assert b2[0, h0b: h0b + 2].tolist() == [0, 1]
    assert b2[0, h0b: h0b + 5].tolist() == [0, 1, 1, 1, 0]
    b2[0, h0b: h0b + 5] = [0, 0, 1, 1, 1]  # h_0 = 2: magnitude 2^31 + 2^30 - 1
    bad2 = np.packbits(b2, axis=1, bitorder="little")
    assert not ref_decode(bad2[0], d2, k2)[1]
    v2, ok2 = _dev_decode(bad2, d2, k2)
    assert ok2.tolist() == [0, 1] and np.array_equal(v2[1], y[1])


def _gpv_s(gp):
    return float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(gp.n)))


def _unit_poly_tags(n, rng, count):
    """tags h with h(1) odd: units mod (X^n + 1, 2^e)"""
    t = rng.integers(0, 2**16, (count, n), dtype=np.int64)
    t[:, 0] += (t.sum(1) % 2 == 0)
    return t


def _packed_equals_int32(psf, a, td, u, seed, first=0, tags=None, idx=None):
    """qf_samp_p_packed rows == device encode of qf_samp_p[_tagged] rows (and the numpy reference on a sample)"""
    k, slot = psf.domain_code_params()
    p, nb = psf.samp_p_packed_batch(a, td, u, seed=seed, first_index=first, tags=tags, tag_idx=idx)
    e = psf.samp_p_batch(a, td, u, seed=seed, first_index=first) if tags is None else \
        psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=seed, first_index=first)
    flat = e.reshape(len(u), -1).astype(np.int64)
    rp, rnb = _dev_encode(flat, k, slot)
    assert np.array_equal(nb, rnb) and np.array_equal(p, rp)
    sp, snb = ref_encode_batch(flat[:16], k, slot)
    assert np.array_equal(p[:16], sp) and np.array_equal(nb[:16], snb)
    assert (nb > 0).all()
    return p, nb, e


def test_samp_p_packed_every_kind(T):
    rng = np.random.default_rng(7)
    # PSFGPV, small one-pass key and a two-phase key (n = 64, q = 2^16)
    gp8 = T.GadgetParameters.init_default(8, 64)
    g8 = T.PSFGPV(gp8, 90.0)
    a8, td8 = g8.trap_gen(seed=4)
    _packed_equals_int32(g8, a8, td8, rng.integers(0, 64, (300, 8), dtype=np.int64), seed=5, first=11)
    gp64 = T.GadgetParameters.init_default(64, 2**16)
    g64 = T.PSFGPV(gp64, _gpv_s(gp64))
    a64, td64 = g64.trap_gen(seed=8)
    u64 = rng.integers(0, 2**16, (700, 64), dtype=np.int64)
    p64, nb64, e64 = _packed_equals_int32(g64, a64, td64, u64, seed=10)
    # a batch larger than the chunk (overlapped copies) and one smaller, split over calls
    small = T.PSFGPV(gp64, _gpv_s(gp64))
    small.ctx.call("qf_set_chunk", 256)
    ps, nbs = small.samp_p_packed_batch(a64, td64, u64, seed=10)
    assert np.array_equal(ps, p64) and np.array_equal(nbs, nb64)
    pa, _ = small.samp_p_packed_batch(a64, td64, u64[:100], seed=10)
    pb, _ = small.samp_p_packed_batch(a64, td64, u64[100:], seed=10, first_index=100)
    assert np.array_equal(np.concatenate([pa, pb]), p64)
    # tagged PSFGPV: matrix table and polynomial table of the same tags
    f = np.array([1] + [0] * 63, dtype=np.int64)
    ptags = T.PolyTags(f, _unit_poly_tags(64, rng, 3))
    mtags = ptags.matrices(2**16)
    idx = rng.integers(0, 3, len(u64)).astype(np.int32)
    pm, _, _ = _packed_equals_int32(g64, a64, td64, u64, seed=12, tags=mtags, idx=idx)
    pp, _, _ = _packed_equals_int32(g64, a64, td64, u64, seed=12, tags=ptags, idx=idx)
    assert np.array_equal(pm, pp)
    # PSFPerturbation: dense and structured sqrt(Sigma_2), tagged with both table forms
    gp = T.GadgetParameters.init_default(8, 64)
    pd = T.PSFPerturbation(gp, 3.0, 25.0)
    ad, tdd = pd.trap_gen(seed=1)
    assert tdd[1] is not None
    _packed_equals_int32(pd, ad, tdd, rng.integers(0, 64, (500, 8), dtype=np.int64), seed=3)
    gq = T.GadgetParameters.init_default(16, 2**16)
    ps_ = T.PSFPerturbation(gq, 4.0, 80.0)
    aq, tdq = ps_.trap_gen(seed=5, dense_sqrt_sigma_2=False)
    uq = rng.integers(0, 2**16, (600, 16), dtype=np.int64)
    _packed_equals_int32(ps_, aq, tdq, uq, seed=9)
    fq = np.array([1] + [0] * 15, dtype=np.int64)
    pt = T.PolyTags(fq, _unit_poly_tags(16, rng, 4))
    iq = rng.integers(0, 4, len(uq)).astype(np.int32)
    m1, _, _ = _packed_equals_int32(ps_, aq, tdq, uq, seed=9, tags=pt.matrices(2**16), idx=iq)
    m2, _, _ = _packed_equals_int32(ps_, aq, tdq, uq, seed=9, tags=pt, idx=iq)
    assert np.array_equal(m1, m2)
    # PSFGPVRing
    gr = T.GadgetParametersRing.init_default(8, 1024)
    pr = T.PSFGPVRing(gr, 300.0, 1.005)
    ar, tdr = pr.trap_gen(seed=1)
    _packed_equals_int32(pr, ar, tdr, rng.integers(0, 1024, (200, 8), dtype=np.int64), seed=3)


def test_samp_p_packed_overflow_and_recovery(T):
    from tools_b200 import _ffi

    gp = T.GadgetParameters.init_default(64, 2**16)
    g = T.PSFGPV(gp, _gpv_s(gp))
    a, td = g.trap_gen(seed=8)
    u = np.random.default_rng(3).integers(0, 2**16, (300, 64), dtype=np.int64)
    k, slot = g.domain_code_params()
    full, nbf = g.samp_p_packed_batch(a, td, u, seed=4)
    # a slot between the median and the maximum length: some rows overflow
    tight = int(np.sort(nbf)[len(nbf) // 2]) // 16 * 16
    over = nbf > tight
    assert over.any() and (~over).any()
    out = np.empty((len(u), tight), dtype=np.uint8)
    nb = np.empty(len(u), dtype=np.int32)
    st = g.ctx.status("qf_samp_p_packed", _ffi.ptr(u), None, len(u), 4, 0, k, tight, _ffi.ptr(out), _ffi.ptr(nb))
    assert st == _ffi.QF_ERR_NUMERIC
    assert np.array_equal(nb < 0, over) and not out[over].any()
    assert np.array_equal(nb[~over], nbf[~over]) and np.array_equal(out[~over], full[~over][:, :tight])
    b = int(np.flatnonzero(over)[0])
    e = g.samp_p_batch(a, td, u[b:b + 1], seed=4, first_index=b)
    assert ref_encode(e[0], k, tight)[1] == -1 and ref_encode(e[0], k, slot)[1] == nbf[b]


def test_f_a_packed_every_kind(T):
    from tools_b200 import _ffi

    rng = np.random.default_rng(5)
    # two-phase PSFGPV: A e = u end to end from packed preimages, and the f_a tag table
    gp = T.GadgetParameters.init_default(64, 2**16)
    g = T.PSFGPV(gp, _gpv_s(gp))
    a, td = g.trap_gen(seed=8)
    u = rng.integers(0, 2**16, (500, 64), dtype=np.int64)
    p, nb = g.samp_p_packed_batch(a, td, u, seed=2)
    k, slot = g.domain_code_params()
    uu, ok = g.f_a_packed_batch(a, p)
    assert ok.all() and np.array_equal(uu, u)
    e, okd = _dev_decode(p, gp.m, k)
    assert okd.all()
    u2, fl2 = g.f_a_batch(a, e)
    assert np.array_equal(uu, u2) and np.array_equal(ok, fl2)
    # trimmed to nbytes and zero padded reads the same
    pad = p.copy()
    for b in range(len(pad)):
        pad[b, nb[b]:] = 0
    assert np.array_equal(g.f_a_packed_batch(a, pad)[0], u)
    tags = np.stack([np.eye(64, dtype=np.int64), rng.integers(0, 2**16, (64, 64), dtype=np.int64)])
    ti = rng.integers(0, 2, len(u)).astype(np.int32)
    ut, okt = g.f_a_packed_batch(a, p, tags=tags, tag_idx=ti)
    ur, okr = g.f_a_tagged_batch(a, tags, e, ti)
    assert np.array_equal(ut, ur) and np.array_equal(okt, okr)
    # a malformed row: in_domain 0 and QF_ERR_NOT_IN_DOMAIN, other rows unchanged; u_out = NULL gives the flags
    badp = p.copy()
    badp[17, -1] |= 0x80
    flags = np.empty(len(u), dtype=np.uint8)
    uo = np.empty_like(u)
    st = g.ctx.status("qf_f_a_packed", _ffi.ptr(badp), None, len(u), k, slot, _ffi.ptr(uo), _ffi.ptr(flags))
    assert st == _ffi.QF_ERR_NOT_IN_DOMAIN and flags[17] == 0 and flags.sum() == len(u) - 1
    keep = np.arange(len(u)) != 17
    assert np.array_equal(uo[keep], u[keep])
    flags2 = np.empty(len(u), dtype=np.uint8)
    st = g.ctx.status("qf_f_a_packed", _ffi.ptr(badp), None, len(u), k, slot, None, _ffi.ptr(flags2))
    assert st == _ffi.QF_ERR_NOT_IN_DOMAIN and np.array_equal(flags2, flags)
    with pytest.raises(T.NotInDomain):
        g.f_a_packed_batch(a, badp)
    # an out-of-domain but canonical row
    far = e[:3].astype(np.int64).copy()
    far[1, 0] = 10**8
    pf, nbf = _dev_encode(far, 2 * k, _slot(gp.m, 2 * k, 4160))
    assert (nbf > 0).all()
    _, okf = g.f_a_packed_batch(a, pf, k=2 * k, strict=False)
    assert okf.tolist() == [True, False, True]
    # PSFPerturbation with an f_a table, and the ring
    gq = T.GadgetParameters.init_default(16, 2**16)
    pq = T.PSFPerturbation(gq, 4.0, 80.0)
    aq, tdq = pq.trap_gen(seed=5, dense_sqrt_sigma_2=False)
    uq = rng.integers(0, 2**16, (300, 16), dtype=np.int64)
    pp, _ = pq.samp_p_packed_batch(aq, tdq, uq, seed=1)
    kq, _ = pq.domain_code_params()
    eq, _ = _dev_decode(pp, gq.m, kq)
    assert np.array_equal(pq.f_a_packed_batch(aq, pp)[0], uq)
    fq = np.array([1] + [0] * 15, dtype=np.int64)
    pt = T.PolyTags(fq, _unit_poly_tags(16, rng, 3))
    iq = rng.integers(0, 3, len(uq)).astype(np.int32)
    assert np.array_equal(pq.f_a_packed_batch(aq, pp, tags=pt, tag_idx=iq)[0], pq.f_a_tagged_batch(aq, pt, eq, iq)[0])
    gr = T.GadgetParametersRing.init_default(8, 1024)
    pr = T.PSFGPVRing(gr, 300.0, 1.005)
    ar, tdr = pr.trap_gen(seed=1)
    ur = rng.integers(0, 1024, (100, 8), dtype=np.int64)
    prk, _ = pr.samp_p_packed_batch(ar, tdr, ur, seed=3)
    uu, okr = pr.f_a_packed_batch(ar, prk)
    assert okr.all() and np.array_equal(uu, ur)


def test_packed_argument_errors(T):
    import torch

    from tools_b200 import _ffi

    gp = T.GadgetParameters.init_default(16, 2**16)
    pq = T.PSFPerturbation(gp, 4.0, 80.0)
    a, td = pq.trap_gen(seed=5, dense_sqrt_sigma_2=False)
    u = np.random.default_rng(1).integers(0, 2**16, (40, 16), dtype=np.int64)
    pq.samp_p_packed_batch(a, td, u, seed=1)  # installs key and trapdoor
    k, slot = pq.domain_code_params()
    h0 = h0_bytes(gp.m, k)
    out = np.zeros((40, 4 * slot), dtype=np.uint8)
    nb = np.empty(40, dtype=np.int32)
    f = np.array([1] + [0] * 15, dtype=np.int64)
    pt = T.PolyTags(f, _unit_poly_tags(16, np.random.default_rng(2), 2))
    pq.set_tag_table(a, td, pt)
    pq._install_fa_tags(pt, None)
    bad_idx = np.zeros(40, dtype=np.int32)
    bad_idx[9] = 2
    c0 = pq.ctx.launch_count()
    for kk, ss, ti in [(-1, slot, None), (31, slot, None), (k, slot + 8, None), (k, -(-(h0 + 1) // 16) * 16 - 16, None),
                       (k, slot, bad_idx)]:
        st = pq.ctx.status("qf_samp_p_packed", _ffi.ptr(u), _ffi.ptr(ti), 40, 1, 0, kk, ss, _ffi.ptr(out), _ffi.ptr(nb))
        assert st == _ffi.QF_ERR_INVALID, (kk, ss)
        st = pq.ctx.status("qf_f_a_packed", _ffi.ptr(out), _ffi.ptr(ti), 40, kk, ss, None, None)
        assert st == _ffi.QF_ERR_INVALID, (kk, ss)
    assert pq.ctx.status("qf_samp_p_packed", _ffi.ptr(u), None, 40, 1, 0, k, slot, None, _ffi.ptr(nb)) == _ffi.QF_ERR_INVALID
    assert pq.ctx.status("qf_samp_p_packed", _ffi.ptr(u), None, 40, 1, 0, k, slot, _ffi.ptr(out), None) == _ffi.QF_ERR_INVALID
    assert pq.ctx.launch_count() == c0
    lib = _ffi.lib()
    x = torch.zeros((4, 105), dtype=torch.int32, device="cuda")
    pk = torch.zeros((4, 256), dtype=torch.uint8, device="cuda")
    n4 = torch.zeros(4, dtype=torch.int32, device="cuda")
    for kk, ss in [(-1, 256), (31, 256), (8, 200), (8, 128)]:
        assert lib.qf_domain_encode_dev(_ffi.ptr(x.data_ptr()), 4, 105, kk, ss, _ffi.ptr(pk.data_ptr()),
                                        _ffi.ptr(n4.data_ptr()), None) == _ffi.QF_ERR_INVALID
        assert lib.qf_domain_decode_dev(_ffi.ptr(pk.data_ptr()), 4, 105, kk, ss, _ffi.ptr(x.data_ptr()),
                                        _ffi.ptr(n4.data_ptr()), None) == _ffi.QF_ERR_INVALID
    assert lib.qf_domain_encode_dev(None, 4, 105, 8, 256, _ffi.ptr(pk.data_ptr()), _ffi.ptr(n4.data_ptr()), None) == \
        _ffi.QF_ERR_INVALID
    # ring contexts take no tags
    gr = T.GadgetParametersRing.init_default(8, 1024)
    pr = T.PSFGPVRing(gr, 300.0, 1.005)
    ar, tdr = pr.trap_gen(seed=1)
    ur2 = u[:2, :8] % 1024
    pr.samp_p_packed_batch(ar, tdr, ur2, seed=1)
    kr, sr = pr.domain_code_params()
    i0 = np.zeros(2, dtype=np.int32)
    outr = np.zeros((2, sr), dtype=np.uint8)
    assert pr.ctx.status("qf_samp_p_packed", _ffi.ptr(ur2), _ffi.ptr(i0), 2, 1, 0, kr, sr, _ffi.ptr(outr),
                         _ffi.ptr(nb)) == _ffi.QF_ERR_INVALID
    assert pr.ctx.status("qf_f_a_packed", _ffi.ptr(outr), _ffi.ptr(i0), 2, kr, sr, None, None) == _ffi.QF_ERR_INVALID
