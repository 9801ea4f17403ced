"""f_a with a tag per target (qf_set_f_a_tags, qf_f_a_tagged[_dev], DESIGN.md 4.9).  Every output is compared exactly with
the CPU (A sigma + (H_t - H_0) G sigma_bot mod q, the identity pinned in test_tag_f_a_math.py) and with the per-tag path:
the key of each tag built on its own (gen_trapdoor with H_t, or set_tag(H_t) on PSFPerturbation) and plain f_a_batch."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

G = 8  # QF_F_A_TAG_GROUP


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _mm(x, y, q):
    """x @ y mod q exactly for int64 x (|x| < 2^32) and y in [0, q): 16-bit halves in float64 BLAS for q <= 2^32
    (|partial sums| < 2^32 K < 2^53), object integers above."""
    x, y = np.asarray(x, dtype=np.int64), np.asarray(y, dtype=np.int64)
    if q > 2**32:
        return np.array(x.astype(object).dot(y.astype(object)) % q, dtype=np.int64).reshape(x.shape[0], y.shape[1])
    x0, x1 = (x & 0xFFFF).astype(np.float64), (x >> 16).astype(np.float64)
    y0, y1 = (y & 0xFFFF).astype(np.float64), (y >> 16).astype(np.float64)
    r = lambda a, b: np.rint(a @ b).astype(np.int64) % q  # noqa: E731
    s16 = (1 << 16) % q
    return (r(x0, y0) + (r(x0, y1) + r(x1, y0)) % q * s16 % q + r(x1, y1) * s16 % q * s16 % q) % q


def _ref(gp, a, h0, tags, idx, sig):
    """A_t sigma mod q on the CPU for every row."""
    q, n, k, mb = gp.q, gp.n, gp.k, gp.m_bar
    sig = np.asarray(sig, dtype=np.int64)
    u = _mm(sig, np.asarray(a, dtype=np.int64).T, q)
    gpow = np.array([pow(gp.base, s, q) for s in range(k)], dtype=np.int64).reshape(k, 1)
    y = _mm(sig[:, mb:].reshape(-1, k), gpow, q).reshape(len(sig), n)
    hm = np.eye(n, dtype=np.int64) if h0 is None else np.asarray(h0, dtype=np.int64) % q
    for t in np.unique(idx):
        rows = idx == t
        d = (np.asarray(tags[t], dtype=np.int64) % q - hm) % q
        u[rows] = (u[rows] + _mm(y[rows], d.T, q)) % q
    return u


def _check(psf, gp, a, h0, tags, idx, sig, u, ok):
    """Rows in D_n equal the CPU.  For a sigma outside D_n, f_a leaves A sigma unspecified (qf_f_a), so there the tag
    correction alone is checked: u - f_a(sigma) = (H_t - H_0) G sigma_bot mod q, exact for every int32 sigma."""
    q = gp.q
    ref = _ref(gp, a, h0, tags, idx, sig)
    assert np.array_equal(u[ok], ref[ok])
    h = np.eye(gp.n, dtype=np.int64) if h0 is None else np.asarray(h0, dtype=np.int64)
    base = _ref(gp, a, h0, h[None], np.zeros(len(sig), np.int32), sig)
    u0, ok0 = psf.f_a_batch(a, sig, strict=False)
    assert np.array_equal(ok0, ok) and np.array_equal(u0[ok], base[ok])
    assert np.array_equal((u - u0) % q, (ref - base) % q)


def _tags(n, q, rng, count):
    """dense, unitriangular, singular (two equal rows), zero and identity tags, negative entries included"""
    out = []
    for i in range(count):
        kind = i % 5
        if kind == 0:
            h = rng.integers(0, q, (n, n), dtype=np.int64) - q // 2
        elif kind == 1:
            h = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)
        elif kind == 2:
            h = rng.integers(0, q, (n, n), dtype=np.int64)
            h[-1] = h[0]
        elif kind == 3:
            h = np.zeros((n, n), dtype=np.int64)
        else:
            h = np.eye(n, dtype=np.int64)
        out.append(h)
    return np.stack(out)


def _key(T, gp, rng, h0):
    a_bar = rng.integers(0, gp.q, (gp.n, gp.m_bar), dtype=np.int64)
    r = rng.integers(-1, 2, (gp.m_bar, gp.n * gp.k)).astype(np.int8)
    return a_bar, r, T.psf.gen_trapdoor(gp, a_bar, r, h0)


def _extreme(rng, rows, m):
    lim = 2**31 - 1
    e = rng.integers(-lim, lim + 1, (rows, m), dtype=np.int64)
    e[0], e[1] = lim, -lim
    return e.astype(np.int32)


def _psf(T, gp, kind, s, r=3.0):
    return T.PSFGPV(gp, s) if kind == "gpv" else T.PSFPerturbation(gp, r, s)


SHAPES = [(8, 64, 25.0), (5, 256, 25.0), (6, 128, 25.0), (8, 127, 30.0), (16, 2**20 - 3, 80.0)]


@pytest.mark.parametrize("kind", ["gpv", "pert"])
@pytest.mark.parametrize("h0_kind", ["identity", "tagged", "zero"])
@pytest.mark.parametrize("n,q,s", SHAPES)
def test_f_a_tagged_matches_cpu_and_per_tag_keys(T, n, q, s, h0_kind, kind):
    """A context holding only the key (no trapdoor), H_0 in {I, dense, 0}, mixed tags (singular and zero ones included),
    sigma from samp_d and sigma with extreme int32 entries."""
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 31 + q % 997 + len(h0_kind))
    h0 = {"identity": None, "tagged": rng.integers(0, q, (n, n), dtype=np.int64), "zero": np.zeros((n, n), np.int64)}[h0_kind]
    a_bar, r, a = _key(T, gp, rng, h0)
    psf = _psf(T, gp, kind, s)
    tags = _tags(n, q, rng, 7)
    sig = np.concatenate([psf.samp_d_batch(600, seed=3), _extreme(rng, 40, gp.m)])
    idx = rng.integers(0, len(tags), len(sig)).astype(np.int32)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx, h0=h0, strict=False)
    assert np.array_equal(ok, psf.check_domain_batch(sig))
    assert ok[:600].all() and not ok[600:].any()
    _check(psf, gp, a, h0, tags, idx, sig, u, ok)
    # per-tag keys: gen_trapdoor(A_bar, R, H_t) and plain f_a
    for t in range(len(tags)):
        rows = (idx == t) & ok
        a_t = T.psf.gen_trapdoor(gp, a_bar, r, tags[t] % q)
        ut, _ = psf.f_a_batch(a_t, sig[rows])
        assert np.array_equal(u[rows], ut), t


def test_perturbation_set_tag_path_and_round_trip(T):
    """PSFPerturbation: rows equal set_tag(H_t) + f_a_batch; f_a_tagged(samp_p_tagged(u)) == u with every flag set, with the
    samp_p table and the f_a table built from the same tags, for the identity key and for a tagged installed key."""
    n, q, r, s = 16, 2**20 - 3, 4.0, 80.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(5)
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=4)
    tags = np.stack([np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64) for _ in range(5)])
    u = rng.integers(0, q, (900, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), 900).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=8)
    ua, ok = psf.f_a_tagged_batch(a, tags, e, idx)
    assert np.array_equal(ua, u) and ok.all()
    sig = psf.samp_d_batch(500, seed=1)
    sidx = rng.integers(0, len(tags), 500).astype(np.int32)
    got, _ = psf.f_a_tagged_batch(a, tags, sig, sidx)
    ref = T.PSFPerturbation(gp, r, s)
    for t in range(len(tags)):
        a_t = ref.set_tag(a, td, tags[t])
        ut, _ = ref.f_a_batch(a_t, sig[sidx == t])
        assert np.array_equal(got[sidx == t], ut), t
    h0 = tags[2]
    a0 = psf.set_tag(a, td, h0)
    assert psf._fa_tags_id is None  # qf_set_tag dropped the f_a table
    e0 = psf.samp_p_tagged_batch(a0, td, tags, u, idx, seed=8)
    assert np.array_equal(e0, e)
    ua0, ok0 = psf.f_a_tagged_batch(a0, tags, e0, idx, h0=h0)
    assert np.array_equal(ua0, u) and ok0.all()


@pytest.mark.parametrize("env", [None, "QF_DISABLE_FUSED_FA", "QF_DISABLE_I8"])
def test_entry_points_splits_and_paths(T, monkeypatch, env):
    """host and device entry points, batches split over calls, chunk sizes that cut tag groups, fused and unfused f_a"""
    import torch
    from tools_b200 import _ffi

    if env:
        monkeypatch.setenv(env, "1")
    n, q, s = 16, 2**20 - 3, 80.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(17)
    _, _, a = _key(T, gp, rng, None)
    psf = T.PSFGPV(gp, s)
    tags = _tags(n, q, rng, 6)
    sig = psf.samp_d_batch(3000, seed=6)
    idx = rng.integers(0, len(tags), 3000).astype(np.int32)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx)
    assert np.array_equal(u, _ref(gp, a, None, tags, idx, sig)) and ok.all()
    parts = [psf.f_a_tagged_batch(a, tags, sig[i:j], idx[i:j])[0] for i, j in ((0, 1), (1, 1001), (1001, 3000))]
    assert np.array_equal(np.concatenate(parts), u)
    for chunk in (100, 256):
        small = T.PSFGPV(gp, s)
        small.ctx.call("qf_set_chunk", chunk)
        assert np.array_equal(small.f_a_tagged_batch(a, tags, sig, idx)[0], u)
    dev = torch.device("cuda:0")
    sd, idd = torch.from_numpy(sig).to(dev), torch.from_numpy(idx).to(dev)
    ud = torch.empty((len(sig), n), dtype=torch.int64, device=dev)
    fd = torch.empty(len(sig), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_f_a_tagged_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), len(sig), _ffi.ptr(ud.data_ptr()),
                 _ffi.ptr(fd.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ud.cpu().numpy(), u) and fd.cpu().numpy().all()


@pytest.mark.parametrize("q", [2**32, 2**48, 2**62 - 1])
def test_large_moduli(T, q):
    """q = 2^32 is the last modulus with 4-byte words; 2^48 and 2^62 - 1 take 8-byte words and 192-bit row sums"""
    n = 64
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(q % 1009)
    h0 = rng.integers(0, q, (n, n), dtype=np.int64)
    a_bar, r, a = _key(T, gp, rng, h0)
    s = float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n)))
    psf = T.PSFGPV(gp, s)
    tags = _tags(n, q, rng, 5)
    tags[0] = q - 1  # the largest residue everywhere
    sig = np.concatenate([psf.samp_d_batch(60, seed=2), _extreme(rng, 12, gp.m)])
    idx = (np.arange(len(sig)) % len(tags)).astype(np.int32)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx, h0=h0, strict=False)
    assert ok[:60].all() and not ok[60:].any()
    _check(psf, gp, a, h0, tags, idx, sig, u, ok)
    a_t = T.psf.gen_trapdoor(gp, a_bar, r, tags[1] % q)
    rows = (idx == 1) & ok
    assert np.array_equal(psf.f_a_batch(a_t, sig[rows])[0], u[rows])


@pytest.mark.parametrize("case", ["one_tag", "more_tags_than_targets", "runs_of_g", "runs_of_g_plus_1"])
def test_group_boundaries(T, case):
    n, q, s = 8, 127, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(len(case))
    _, _, a = _key(T, gp, rng, None)
    psf = T.PSFGPV(gp, s)
    if case == "one_tag":
        tags, idx = _tags(n, q, rng, 1), np.zeros(1000, np.int32)
    elif case == "more_tags_than_targets":
        tags, idx = _tags(n, q, rng, 700), rng.integers(0, 700, 300).astype(np.int32)
    else:
        run = G if case == "runs_of_g" else G + 1
        tags = _tags(n, q, rng, 9)
        idx = rng.permutation(np.repeat(np.arange(9), [run, run, 2 * run, 1, run, 3 * run, run, G - 1, run])).astype(np.int32)
    sig = psf.samp_d_batch(len(idx), seed=4)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx)
    assert np.array_equal(u, _ref(gp, a, None, tags, idx, sig)) and ok.all()


def test_table_reinstalled_after_key_switch(T):
    """The device drops the f_a table whenever A changes; the wrapper must install it again when it returns to a key:
    f_a_tagged(a1) -> f_a(a2) -> f_a_tagged(a1), the same across trap_gen, and across set_tag and back (PSFPerturbation)."""
    n, q, s = 8, 127, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(77)
    _, _, a1 = _key(T, gp, rng, None)
    _, _, a2 = _key(T, gp, rng, None)
    tags = _tags(n, q, rng, 4)
    psf = T.PSFGPV(gp, s)
    sig = psf.samp_d_batch(300, seed=2)
    idx = rng.integers(0, 4, 300).astype(np.int32)
    want = _ref(gp, a1, None, tags, idx, sig)
    assert np.array_equal(psf.f_a_tagged_batch(a1, tags, sig, idx)[0], want)
    psf.f_a_batch(a2, sig)
    assert np.array_equal(psf.f_a_tagged_batch(a1, tags, sig, idx)[0], want)
    psf.trap_gen(seed=3)
    assert np.array_equal(psf.f_a_tagged_batch(a1, tags, sig, idx)[0], want)
    pert = T.PSFPerturbation(gp, 3.0, 30.0)
    pa, ptd = pert.trap_gen(seed=5)
    h = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)
    psig = pert.samp_d_batch(300, seed=4)
    pwant = _ref(gp, pa, None, tags, idx, psig)
    assert np.array_equal(pert.f_a_tagged_batch(pa, tags, psig, idx)[0], pwant)
    pert.set_tag(pa, ptd, h)
    assert np.array_equal(pert.f_a_tagged_batch(pa, tags, psig, idx)[0], pwant)


def test_out_of_domain_flags(T):
    from tools_b200 import _ffi

    n, q, s = 8, 127, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(9)
    _, _, a = _key(T, gp, rng, None)
    psf = T.PSFGPV(gp, s)
    tags = _tags(n, q, rng, 3)
    sig = psf.samp_d_batch(200, seed=1)
    sig[[3, 77, 150]] = 10**6
    idx = rng.integers(0, 3, 200).astype(np.int32)
    with pytest.raises(T.NotInDomain):
        psf.f_a_tagged_batch(a, tags, sig, idx)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx, strict=False)
    want = np.ones(200, bool)
    want[[3, 77, 150]] = False
    assert np.array_equal(ok, want)
    _check(psf, gp, a, None, tags, idx, sig, u, ok)
    out, fl = np.empty((200, n), np.int64), np.empty(200, np.uint8)
    assert psf.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(idx), 200, _ffi.ptr(out), None) == _ffi.QF_ERR_NOT_IN_DOMAIN
    assert psf.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(idx), 200, _ffi.ptr(out), _ffi.ptr(fl)) == _ffi.QF_ERR_NOT_IN_DOMAIN
    assert np.array_equal(fl.astype(bool), want)


def test_refusals(T):
    import torch
    from tools_b200 import _ffi

    n, q, s = 8, 127, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(41)
    _, _, a = _key(T, gp, rng, None)
    psf = T.PSFGPV(gp, s)
    tags = _tags(n, q, rng, 3)
    tg = np.ascontiguousarray(tags)
    sig = psf.samp_d_batch(400, seed=3)
    idx = rng.integers(0, 3, 400).astype(np.int32)
    out, fl = np.empty((400, n), np.int64), np.empty(400, np.uint8)
    call = lambda p, ix=idx, o=out: p.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(ix), 400, _ffi.ptr(o), _ffi.ptr(fl))  # noqa: E731
    # no key, no table
    bare = T.PSFGPV(gp, s)
    assert bare.ctx.status("qf_set_f_a_tags", _ffi.ptr(tg), 3, None) == _ffi.QF_ERR_NO_KEY
    assert call(bare) == _ffi.QF_ERR_NO_KEY
    bare._install_a(a)
    assert call(bare) == _ffi.QF_ERR_NO_KEY
    # ntags < 1, NULL tags
    assert bare.ctx.status("qf_set_f_a_tags", _ffi.ptr(tg), 0, None) == _ffi.QF_ERR_INVALID
    assert bare.ctx.status("qf_set_f_a_tags", None, 3, None) == _ffi.QF_ERR_INVALID
    # ring context
    ring = T.PSFGPVRing(T.GadgetParametersRing.init_default(8, 257), 20.0, 2.0)
    assert ring.ctx.status("qf_set_f_a_tags", _ffi.ptr(tg), 3, None) == _ffi.QF_ERR_INVALID
    assert ring.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(idx), 1, _ffi.ptr(out), _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    u, _ = psf.f_a_tagged_batch(a, tags, sig, idx)
    launches = psf.ctx.launch_count()
    # a bad index on the host: refused before any launch; NULL u_out
    bad = idx.copy()
    bad[17] = 3
    assert call(psf, bad) == _ffi.QF_ERR_INVALID and psf.ctx.launch_count() == launches
    bad[17] = -1
    assert call(psf, bad) == _ffi.QF_ERR_INVALID and psf.ctx.launch_count() == launches
    assert psf.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(idx), 400, None, _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    # a bad index on the device: its row is not read from the table, reported at qf_synchronize
    dev = torch.device("cuda:0")
    bad[17], bad[300] = 3, 2**31 - 1
    sd, idd = torch.from_numpy(sig).to(dev), torch.from_numpy(bad).to(dev)
    ud = torch.empty((400, n), dtype=torch.int64, device=dev)
    fd = torch.empty(400, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    args = (_ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), 400, _ffi.ptr(ud.data_ptr()), _ffi.ptr(fd.data_ptr()))
    assert psf.ctx.status("qf_f_a_tagged_dev", *args) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert "tag index outside" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    keep = np.ones(400, bool)
    keep[[17, 300]] = False
    assert np.array_equal(ud.cpu().numpy()[keep], u[keep])
    assert psf.ctx.status("qf_f_a_tagged_dev", args[0], args[1], 400, None, args[4]) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_f_a_tagged_dev", args[0], args[1], 400, args[3], None) == _ffi.QF_ERR_INVALID
    # the table is dropped by qf_set_a and qf_trap_gen
    assert call(psf) == _ffi.QF_OK
    psf.ctx.call("qf_set_a", _ffi.ptr(np.ascontiguousarray(a)))
    assert call(psf) == _ffi.QF_ERR_NO_KEY
    psf.ctx.call("qf_set_f_a_tags", _ffi.ptr(tg), 3, None)
    assert call(psf) == _ffi.QF_OK and np.array_equal(out, u)
    psf.trap_gen(seed=2)
    assert call(psf) == _ffi.QF_ERR_NO_KEY
    # ... and by qf_set_tag (PSFPerturbation), while the samp_p table stays
    pert = T.PSFPerturbation(gp, 3.0, 30.0)
    pa, ptd = pert.trap_gen(seed=5)
    ptags = np.stack([np.eye(n, dtype=np.int64), np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)])
    pidx = (np.arange(400) % 2).astype(np.int32)
    e = pert.samp_p_tagged_batch(pa, ptd, ptags, rng.integers(0, q, (400, n), dtype=np.int64), pidx, seed=1)
    pert.f_a_tagged_batch(pa, ptags, e, pidx)
    assert pert.ctx.status("qf_f_a_tagged", _ffi.ptr(e), _ffi.ptr(pidx), 400, _ffi.ptr(out), _ffi.ptr(fl)) == _ffi.QF_OK
    pa2 = pert.set_tag(pa, ptd, ptags[1])
    assert pert.ctx.status("qf_f_a_tagged", _ffi.ptr(e), _ffi.ptr(pidx), 400, _ffi.ptr(out), _ffi.ptr(fl)) == _ffi.QF_ERR_NO_KEY
    assert pert._tags_id is ptags  # the samp_p table is kept
    uu, ok = pert.f_a_tagged_batch(pa2, ptags, e, pidx, h0=ptags[1])
    assert ok.all()


def _full(T, kind, batch, ntags):
    if kind == "c2":
        n, q = 256, 2**24
        gp = T.GadgetParameters.init_default(n, q)
        psf = T.PSFGPV(gp, float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n))))
    else:
        n, q, r = 512, 2**32 - 5, 9.0
        gp = T.GadgetParameters.init_default(n, q)
        s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
        psf = T.PSFPerturbation(gp, r, float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1))))
    rng = np.random.default_rng(n)
    a_bar, rr, a = _key(T, gp, rng, None)
    tags = np.stack([np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64) for _ in range(ntags)])
    sig = psf.samp_d_batch(batch, seed=7)
    idx = rng.permutation(np.arange(batch) % ntags).astype(np.int32)
    u, ok = psf.f_a_tagged_batch(a, tags, sig, idx)
    assert ok.all()
    assert np.array_equal(u, _ref(gp, a, None, tags, idx, sig))
    for t in (int(idx[0]), int(idx[1])):
        a_t = T.psf.gen_trapdoor(gp, a_bar, rr, tags[t])
        assert np.array_equal(psf.f_a_batch(a_t, sig[idx == t])[0], u[idx == t])


def test_full_size_c2_batch(T):
    """C2 (PSFGPV n = 256, q = 2^24, m = 12352): 8192 targets under 64 tags, every row exact"""
    _full(T, "c2", 8192, 64)


def test_full_size_c4_shard(T):
    """C4 shard (PSFPerturbation n = 512, q = 2^32 - 5, m = 32849): 4096 targets under 64 tags, every row exact"""
    _full(T, "c4", 4096, 64)
