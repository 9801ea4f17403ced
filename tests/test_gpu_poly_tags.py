"""Tags in polynomial form on the device (qf_set_tag_table_poly, qf_set_f_a_tags_poly; DESIGN.md 4.10).  The reference of
every test is the matrix table that already exists: in the same context, with the same seed and first_index, a polynomial
table of tags h_t must give bit-identical rows to the matrix table of the tags rot_f(h_t), for samp_p and for f_a.
Preimages are also checked directly: A_t e = u.  The algebra is pinned on the CPU in test_poly_tag_math.py."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


P_OF = {2**16: 2, 4093: 4093, 2**32 - 5: 2**32 - 5, 2**32: 2, 3**10: 3, 2**48: 2, 2**61 - 1: 2**61 - 1, 2**12: 2, 2**24: 2}


def _f(fam, n, rng):
    if fam == "x^n+1":
        return np.array([1] + [0] * (n - 1), dtype=np.int64)
    if fam == "x^n-1":
        return np.array([-1] + [0] * (n - 1), dtype=np.int64)
    return rng.integers(-(2**40), 2**40, n, dtype=np.int64)  # random monic, any sign: taken mod q


def _trim(x, p):
    x = [int(v) % p for v in x]
    while x and x[-1] == 0:
        x.pop()
    return x


def _unit_mod_p(h, f, p):
    """gcd(h, f) = 1 in F_p[X]: for q = p^e, h is a unit mod (f, q) exactly then."""
    a, b = _trim(list(f) + [1], p), _trim(h, p)
    while b:
        inv = pow(b[-1], -1, p)
        while len(a) >= len(b):
            c, sh = a[-1] * inv % p, len(a) - len(b)
            for i, v in enumerate(b):
                a[i + sh] = (a[i + sh] - c * v) % p
            a = _trim(a, p)
        a, b = b, a
    return len(a) == 1


def _unit_tags(n, q, f, rng, count):
    out = []
    while len(out) < count:
        h = rng.integers(0, min(q, 2**62), n, dtype=np.int64)
        if _unit_mod_p(h, f, P_OF[q]):
            out.append(h)
    return np.stack(out)


def _matrices(T, f, tags, q):
    return np.stack([T.rot_f(h, f, q) for h in tags])


def _f_a(a, e, q):
    """A e mod q for a batch of preimages (rows of e), exact."""
    if q >= 2**32:
        return np.array(e.astype(object).dot(a.T.astype(object)) % q, dtype=np.int64)
    ef = e.astype(np.float64)
    lo = np.rint(ef @ (a & 0xFFFF).astype(np.float64).T).astype(np.int64)
    hi = np.rint(ef @ (a >> 16).astype(np.float64).T).astype(np.int64)
    return (lo % q + ((hi % q) << 16) % q) % q


def _assert_preimages(gp, a, h0, mats, idx, e, u):
    """A_t e = u for every row, A_t = A + [0 | (H_t - H_0) G]."""
    q, n, k, mb = gp.q, gp.n, gp.k, gp.m_bar
    ae = _f_a(a, e, q)
    eb = e[:, mb:].astype(object).reshape(len(e), n, k)
    y = (eb * np.array([gp.base**s for s in range(k)], dtype=object)).sum(axis=2) % q
    for t in np.unique(idx):
        rows = idx == t
        d = (np.asarray(mats[t], dtype=object) - np.asarray(h0, dtype=object)) % q
        got = np.array((ae[rows].astype(object) + y[rows].dot(d.T)) % q, dtype=np.int64)
        assert np.array_equal(got, u[rows]), t


def _pert_s(gp):
    return float(math.ceil(1.3 * math.sqrt(5 * ((math.sqrt(gp.m_bar) + math.sqrt(gp.n * gp.k)) ** 2 / 2 + 1) + 1)))


def _dense_unit(n, q, rng):
    while True:
        h = rng.integers(0, min(q, 2**62), (n, n), dtype=np.int64)
        try:
            O.mat_inverse_mod(h.tolist(), q)
            return h
        except ValueError:
            continue


QS = [2**16, 4093, 2**32 - 5, 2**32, 3**10, 2**48, 2**61 - 1]
FAMS = ["x^n+1", "x^n-1", "random"]


@pytest.mark.parametrize("fam", FAMS)
@pytest.mark.parametrize("q", QS)
def test_pert_poly_table_matches_matrix_table(T, q, fam):
    """PSFPerturbation, n = 16: rows of the polynomial table equal the rows of the matrix table of rot_f(h_t), for the
    identity key and for a key with a dense H_0 (set_tag, which keeps the table)."""
    n = 16
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(q % 7919 + FAMS.index(fam))
    f = _f(fam, n, rng)
    tags = _unit_tags(n, q, f, rng, 5)
    poly = T.PolyTags(f, tags)
    mats = _matrices(T, f, tags, q)
    psf = T.PSFPerturbation(gp, 3.0, _pert_s(gp))
    a, td = psf.trap_gen(seed=q % 101 + 1, dense_sqrt_sigma_2=True)
    u = rng.integers(0, min(q, 2**62), (600, n), dtype=np.int64) % q
    idx = rng.integers(0, len(tags), len(u)).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, poly, u, idx, seed=5, first_index=2)
    assert psf.ctx.launch_count() > 0
    ref = psf.samp_p_tagged_batch(a, td, mats, u, idx, seed=5, first_index=2)
    assert np.array_equal(e, ref)
    _assert_preimages(gp, a, np.eye(n, dtype=np.int64), mats, idx, e, u)
    h0 = _dense_unit(n, q, rng)
    a0 = psf.set_tag(a, td, h0)
    e0 = psf.samp_p_tagged_batch(a0, td, mats, u, idx, seed=6)
    psf.set_tag_table(a0, td, poly)
    assert np.array_equal(psf.samp_p_tagged_batch(a0, td, poly, u, idx, seed=6), e0)
    _assert_preimages(gp, a0, h0, mats, idx, e0, u)


def test_pert_poly_entry_points_and_splits(T):
    """Host and device entry points, splits over calls (first_index) and over chunk sizes give the same rows."""
    import torch
    from tools_b200 import _ffi

    n, q = 16, 2**32 - 5
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(3)
    f = _f("random", n, rng)
    poly = T.PolyTags(f, _unit_tags(n, q, f, rng, 7))
    mats = _matrices(T, f, poly.tags, q)
    psf = T.PSFPerturbation(gp, 3.0, _pert_s(gp))
    a, td = psf.trap_gen(seed=7)
    u = rng.integers(0, q, (1500, n), dtype=np.int64)
    idx = rng.integers(0, len(poly), len(u)).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, poly, u, idx, seed=9)
    assert np.array_equal(e, T.PSFPerturbation(gp, 3.0, _pert_s(gp)).samp_p_tagged_batch(a, td, mats, u, idx, seed=9))
    parts = np.concatenate([psf.samp_p_tagged_batch(a, td, poly, u[:700], idx[:700], seed=9, first_index=0),
                            psf.samp_p_tagged_batch(a, td, poly, u[700:], idx[700:], seed=9, first_index=700)])
    assert np.array_equal(parts, e)
    small = T.PSFPerturbation(gp, 3.0, _pert_s(gp))
    small.ctx.call("qf_set_chunk", 256)
    assert np.array_equal(small.samp_p_tagged_batch(a, td, poly, u, idx, seed=9), e)
    dev = torch.device("cuda:0")
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(idx).to(dev)
    ed = torch.empty((len(u), gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(idd.data_ptr()), len(u), 9, 0, _ffi.ptr(ed.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ed.cpu().numpy(), e)


@pytest.mark.parametrize("q", [2**16, 4093, 2**12])
def test_gpv_poly_table_matches_matrix_table(T, monkeypatch, q):
    """PSFGPV on the two-phase recursion (n = 64): polynomial rows equal matrix rows, and A_t e = u."""
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n = 64
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(q % 31)
    psf = T.PSFGPV(gp, float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n))))
    a, td = psf.trap_gen(seed=4)
    for fam in FAMS:
        f = _f(fam, n, rng)
        poly = T.PolyTags(f, _unit_tags(n, q, f, rng, 4))
        mats = _matrices(T, f, poly.tags, q)
        u = rng.integers(0, q, (400, n), dtype=np.int64)
        idx = rng.integers(0, 4, len(u)).astype(np.int32)
        e = psf.samp_p_tagged_batch(a, td, poly, u, idx, seed=3, first_index=1)
        assert np.array_equal(e, psf.samp_p_tagged_batch(a, td, mats, u, idx, seed=3, first_index=1)), fam
        _assert_preimages(gp, a, np.eye(n, dtype=np.int64), mats, idx, e, u)


def test_poly_refusals_and_lifetime(T, monkeypatch):
    import torch
    from tools_b200 import _ffi

    n, q = 16, 4093
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(11)
    f = _f("x^n+1", n, rng)
    poly = T.PolyTags(f, _unit_tags(n, q, f, rng, 5))
    fw, tw = poly.words(q)
    psf = T.PSFPerturbation(gp, 3.0, _pert_s(gp))
    # no key or trapdoor
    assert psf.ctx.status("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(tw), 5) == _ffi.QF_ERR_NO_KEY
    a, td = psf.trap_gen(seed=2)
    u = rng.integers(0, q, (300, n), dtype=np.int64)
    idx = rng.integers(0, 5, len(u)).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, poly, u, idx, seed=4)
    # a tag that is not a unit is refused with its index; the previous table keeps sampling identically
    bad = tw.copy()
    bad[3] = 0  # h = 0
    with pytest.raises(T.QfError) as err:
        psf.set_tag_table(a, td, T.PolyTags(f, bad))
    assert err.value.status == _ffi.QF_ERR_INVALID and "tag 3" in str(err.value)
    out = np.empty((len(u), gp.m), dtype=np.int32)
    psf.ctx.call("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 4, 0, _ffi.ptr(out))
    assert np.array_equal(out, e)
    # bad indices: host before any launch, device at qf_synchronize
    badidx = idx.copy()
    badidx[7] = 5
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(badidx), len(u), 4, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    dev = torch.device("cuda:0")
    ud, bd = torch.from_numpy(u).to(dev), torch.from_numpy(badidx).to(dev)
    ed = torch.empty((len(u), gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    assert psf.ctx.status("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(bd.data_ptr()), len(u), 4, 0,
                          _ffi.ptr(ed.data_ptr())) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    # one form replaces the other: a 3-tag matrix table makes index 4 invalid, the polynomial table makes it valid again
    mats = _matrices(T, f, poly.tags, q)
    psf.set_tag_table(a, td, mats[:3])
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 4, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    psf.set_tag_table(a, td, poly)
    psf.ctx.call("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 4, 0, _ffi.ptr(out))
    assert np.array_equal(out, e)
    # set_tag keeps the table; installing a key drops it
    psf.set_tag(a, td, _dense_unit(n, q, rng))
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 4, 0, _ffi.ptr(out)) == _ffi.QF_OK
    psf.trap_gen(seed=3)
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 4, 0, _ffi.ptr(out)) == _ffi.QF_ERR_NO_KEY
    # q not a prime power: the samp_p table is unsupported, the f_a table works
    for qq in (4095, 2**62 - 1):
        g2 = T.GadgetParameters.init_default(n, qq)
        p2 = T.PSFPerturbation(g2, 3.0, _pert_s(g2))
        a2, td2 = p2.trap_gen(seed=5)
        t2 = T.PolyTags(f, rng.integers(0, 2**40, (3, n), dtype=np.int64))
        with pytest.raises(T.QfError) as err:
            p2.set_tag_table(a2, td2, t2)
        assert err.value.status == _ffi.QF_ERR_UNSUPPORTED
        sig = p2.samp_d_batch(50, seed=1)
        ti = rng.integers(0, 3, 50).astype(np.int32)
        got, ok = p2.f_a_tagged_batch(a2, t2, sig, ti)
        assert np.array_equal(got, p2.f_a_tagged_batch(a2, _matrices(T, f, t2.tags, qq), sig, ti)[0]) and ok.all()
    # PSFGPV without a key, on the one-pass recursion; a ring context
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    g64 = T.GadgetParameters.init_default(64, 2**16)
    s64 = float(math.ceil((math.sqrt(g64.m_bar) + 1.0) * math.sqrt(5.0) * 6.0))
    f64 = _f("x^n+1", 64, rng)
    fw64, tw64 = T.PolyTags(f64, _unit_tags(64, 2**16, f64, rng, 2)).words(2**16)
    bare = T.PSFGPV(g64, s64)
    assert bare.ctx.status("qf_set_tag_table_poly", _ffi.ptr(fw64), _ffi.ptr(tw64), 2) == _ffi.QF_ERR_INVALID
    monkeypatch.setenv("QF_DISABLE_TWO_PHASE", "1")
    one = T.PSFGPV(g64, s64)
    a1, td1 = one.trap_gen(seed=1)
    one._install_a(a1)
    one._install_td(a1, td1)
    assert one.ctx.status("qf_set_tag_table_poly", _ffi.ptr(fw64), _ffi.ptr(tw64), 2) == _ffi.QF_ERR_INVALID
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE")
    ring = T.PSFGPVRing(T.GadgetParametersRing.init_default(8, 257), 20.0, 2.0)
    f8, t8 = np.zeros(8, dtype=np.int64), np.ones((1, 8), dtype=np.int64)
    assert ring.ctx.status("qf_set_tag_table_poly", _ffi.ptr(f8), _ffi.ptr(t8), 1) == _ffi.QF_ERR_INVALID
    assert ring.ctx.status("qf_set_f_a_tags_poly", _ffi.ptr(f8), _ffi.ptr(t8), 1, None) == _ffi.QF_ERR_INVALID


@pytest.mark.parametrize("q", [4093, 2**32, 2**48, 2**62 - 1])
@pytest.mark.parametrize("h0_kind", ["identity", "dense", "zero"])
def test_f_a_poly_matches_matrix(T, q, h0_kind):
    """f_a rows of the polynomial table equal those of the matrix table of rot_f(h_t) (host and device entry points),
    for singular tags too, with out-of-domain sigma; a bad index on the device leaves A sigma and is reported."""
    import torch
    from tools_b200 import _ffi

    n = 16
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(q % 313 + len(h0_kind))
    psf = T.PSFGPV(gp, 40.0)
    a = rng.integers(0, q, (n, gp.m), dtype=np.int64)
    h0 = {"identity": None, "zero": np.zeros((n, n), dtype=np.int64),
          "dense": rng.integers(0, q, (n, n), dtype=np.int64)}[h0_kind]
    for fam in FAMS:
        f = _f(fam, n, rng)
        tags = rng.integers(-(2**40), 2**40, (6, n), dtype=np.int64)
        tags[1] = 0  # singular
        tags[2] = tags[0] * 2
        poly = T.PolyTags(f, tags)
        mats = _matrices(T, f, tags, q)
        sig = rng.integers(-200, 200, (500, gp.m)).astype(np.int32)
        sig[:5] = rng.integers(-(2**31) + 1, 2**31, (5, gp.m))  # outside the domain
        idx = rng.integers(0, 6, len(sig)).astype(np.int32)
        got, ok = psf.f_a_tagged_batch(a, poly, sig, idx, h0=h0, strict=False)
        want, ok2 = psf.f_a_tagged_batch(a, mats, sig, idx, h0=h0, strict=False)
        assert np.array_equal(got, want) and np.array_equal(ok, ok2) and not ok[:5].any(), fam
    psf.f_a_tagged_batch(a, poly, sig[:1], idx[:1], h0=h0, strict=False)
    dev = torch.device("cuda:0")
    bad = idx.copy()
    bad[3] = 6
    sd, bd = torch.from_numpy(sig).to(dev), torch.from_numpy(bad).to(dev)
    ud = torch.empty((len(sig), n), dtype=torch.int64, device=dev)
    fl = torch.empty(len(sig), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    assert psf.ctx.status("qf_f_a_tagged_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(bd.data_ptr()), len(sig),
                          _ffi.ptr(ud.data_ptr()), _ffi.ptr(fl.data_ptr())) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    du = ud.cpu().numpy()
    keep = np.arange(len(sig)) != 3
    assert np.array_equal(du[keep], got[keep])
    assert np.array_equal(du[3], psf.f_a_batch(a, sig[3:4], strict=False)[0][0])
    assert psf.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(bad), len(sig), _ffi.ptr(du), None) == _ffi.QF_ERR_INVALID


def test_2_17_tags_install(T):
    """T = 2^17 distinct tags at n = 64 (a matrix table of that size would take 2 GB): rows of a sample of the tags match
    a small matrix table built from the same tags."""
    n, q = 64, 2**32 - 5
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(17)
    f = _f("x^n+1", n, rng)
    tags = rng.integers(0, q, (2**17, n), dtype=np.int64)  # a non-unit among them has probability about 2^-20
    poly = T.PolyTags(f, tags)
    psf = T.PSFPerturbation(gp, 3.0, _pert_s(gp))
    a, td = psf.trap_gen(seed=6)
    pick = np.unique(np.concatenate([[0, 2**17 - 1], rng.integers(0, 2**17, 30)]))
    u = rng.integers(0, q, (1000, n), dtype=np.int64)
    j = rng.integers(0, len(pick), len(u))
    e = psf.samp_p_tagged_batch(a, td, poly, u, pick[j].astype(np.int32), seed=8)
    mats = _matrices(T, f, tags[pick], q)
    assert np.array_equal(e, psf.samp_p_tagged_batch(a, td, mats, u, j.astype(np.int32), seed=8))


def _full_size(T, psf, gp, a, td, f, B, seed):
    """One fresh tag per target, all on the device: samp_p_tagged_dev, then A_t e = u and check_domain by f_a_tagged_dev."""
    import torch
    from tools_b200 import _ffi

    rng = np.random.default_rng(seed)
    n, q = gp.n, gp.q
    tags = rng.integers(0, q, (B, n), dtype=np.int64)
    if P_OF.get(q) == 2:  # f = X^n + 1 = (X + 1)^n mod 2: h is a unit iff h(1) is odd
        tags[:, 0] += (tags.sum(axis=1) + 1) % 2
    poly = T.PolyTags(f, tags)
    psf.set_tag_table(a, td, poly)
    fw, tw = poly.words(q)
    psf.ctx.call("qf_set_f_a_tags_poly", _ffi.ptr(fw), _ffi.ptr(tw), B, None)
    dev = torch.device("cuda:0")
    u = torch.randint(0, q, (B, n), dtype=torch.int64, device=dev)
    idx = torch.from_numpy(rng.permutation(B).astype(np.int32)).to(dev)
    e = torch.empty((B, gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx.data_ptr()), B, 3, 0, _ffi.ptr(e.data_ptr()))
    got = torch.empty_like(u)
    ok = torch.empty(B, dtype=torch.uint8, device=dev)
    psf.ctx.call("qf_f_a_tagged_dev", _ffi.ptr(e.data_ptr()), _ffi.ptr(idx.data_ptr()), B, _ffi.ptr(got.data_ptr()),
                 _ffi.ptr(ok.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert torch.equal(got, u) and bool(ok.all())
    # rows of two tags against a matrix table of those two tags
    ih = idx[:256].cpu().numpy()
    t0, t1 = int(ih[0]), int(ih[1])
    mats = _matrices(T, f, tags[[t0, t1]], q)
    ref = psf.samp_p_tagged_batch(a, td, mats, u[:256].cpu().numpy(), (ih == t1).astype(np.int32), seed=3)
    rows = (ih == t0) | (ih == t1)
    assert np.array_equal(e[:256].cpu().numpy()[rows], ref[rows])


def test_full_size_c4_shard_fresh_tags(T):
    """C4 shard (n = 512, q = 2^32 - 5, m = 32849): 60 416 targets, each under its own fresh tag."""
    n, q, r = 512, 2**32 - 5, 9.0
    gp = T.GadgetParameters.init_default(n, q)
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
    s = float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=4, dense_sqrt_sigma_2=False)
    _full_size(T, psf, gp, a, td, _f("x^n+1", n, None), 60416, 41)


def test_full_size_c2_gpv_fresh_tags(T, monkeypatch):
    """C2 PSFGPV (n = 256, q = 2^24, m = 12352) on the two-phase recursion: 37 888 targets, each under its own fresh tag."""
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    monkeypatch.delenv("QF_OZAKI_MIN_DIM", raising=False)
    n, q = 256, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFGPV(gp, float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n))))
    a, td = psf.trap_gen(seed=2, dense_gso=False)
    _full_size(T, psf, gp, a, td, _f("x^n+1", n, None), 37888, 42)
