"""PSFPerturbation samp_p with a tag per target (qf_set_tag_table, qf_samp_p_tagged[_dev], DESIGN.md 4.4).  The reference of
every sampling test is the per-tag path: for each tag t, set_tag(H_t) + samp_p_batch on the WHOLE batch with the same
seed and first_index, restricted to the rows with tag_idx == t.  The tag-table output must equal those rows bit for bit,
and A_t e = u must hold exactly on every row.  The identity behind it is pinned on the CPU in test_tag_table_math.py."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _matmul_mod(x, y, q):
    """x y mod q, exact: 16-bit halves in float64 BLAS for q < 2^32, object integers above."""
    x, y = np.asarray(x, dtype=np.int64), np.asarray(y, dtype=np.int64)
    if q >= 2**32:
        return np.array(x.astype(object).dot(y.astype(object)) % q, dtype=np.int64)
    x0, x1 = (x & 0xFFFF).astype(np.float64), (x >> 16).astype(np.float64)
    y0, y1 = (y & 0xFFFF).astype(np.float64), (y >> 16).astype(np.float64)
    p00 = np.rint(x0 @ y0).astype(np.int64) % q
    p01 = (np.rint(x0 @ y1).astype(np.int64) + np.rint(x1 @ y0).astype(np.int64)) % q
    p11 = np.rint(x1 @ y1).astype(np.int64) % q
    return (p00 + (p01 << 16) % q + (((p11 << 16) % q) << 16) % q) % q


def _f_a(a, e, q):
    """A e mod q for a batch of preimages (rows of e), exact."""
    if q >= 2**32:
        return O.f_a_classical_batch(a, e, q)
    ef = e.astype(np.float64)  # |e| < 2^16, 16-bit halves of A: |partial sums| < 2^32 m < 2^53
    lo = np.rint(ef @ (a & 0xFFFF).astype(np.float64).T).astype(np.int64)
    hi = np.rint(ef @ (a >> 16).astype(np.float64).T).astype(np.int64)
    return (lo % q + ((hi % q) << 16) % q) % q


def _assert_preimages(gp, a, h0, tags, idx, e, u):
    """A_t e = u exactly for every row: A_t e = A e + (H_t - H_0) G e_bot with A = [A_bar | H_0 G - A_bar R]."""
    q, n, k, mb = gp.q, gp.n, gp.k, gp.m_bar
    ae = _f_a(a, e, q)
    eb = e[:, mb:].astype(object).reshape(len(e), n, k)
    y = np.array((eb * np.array([gp.base**s for s in range(k)], dtype=object)).sum(axis=2) % q, dtype=np.int64)
    for t in np.unique(idx):
        rows = idx == t
        d = np.array((np.asarray(tags[t], dtype=object) - np.asarray(h0, dtype=object)) % q, dtype=np.int64)
        got = (ae[rows] + _matmul_mod(y[rows], d.T, q)) % q
        assert np.array_equal(got, u[rows]), t


def _per_tag(T, gp, r, s, a, td, tags, u, idx, seed, first_index=0, only=None):
    """The per-tag path: set_tag(H_t) + samp_p_batch on the whole batch, rows of tag t; `done` marks the rows filled."""
    ref = T.PSFPerturbation(gp, r, s)
    out = np.zeros((len(u), gp.m), dtype=np.int32)
    done = np.zeros(len(u), dtype=bool)
    cur = a
    for t in (np.unique(idx) if only is None else only):
        cur = ref.set_tag(cur, td, tags[t])
        e = ref.samp_p_batch(cur, td, u, seed=seed, first_index=first_index)
        out[idx == t] = e[idx == t]
        done |= idx == t
    ref.ctx.close()
    return out, done


def _unitriangular_tag(n, q, rng):
    return np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)


def _dense_tag(n, q, rng):
    while True:
        h = rng.integers(0, q, (n, n), dtype=np.int64)
        try:
            O.mat_inverse_mod(h.tolist(), q)
            return h
        except ValueError:
            continue


def _mixed_tags(n, q, rng, count):
    kinds = [lambda: _dense_tag(n, q, rng), lambda: _unitriangular_tag(n, q, rng), lambda: np.eye(n, dtype=np.int64)]
    return np.stack([kinds[i % 3]() for i in range(count)])


def _midsize():
    n, q = 40, 2**12
    from tools_b200 import gadget

    gp = gadget.GadgetParameters.init_default(n, q)
    s = 1.3 * np.sqrt(5 * ((np.sqrt(gp.m_bar) + np.sqrt(n * gp.k)) ** 2 / 2 + 1) + 1)
    return n, q, float(np.log2(n)), float(s)


PREIMAGE_SHAPES = [(8, 64, 3.0, 25.0), (5, 256, float(np.log2(5)), 25.0), (6, 128, float(np.log2(6)), 25.0),
                   (8, 127, 3.0, 30.0), (16, 2**20 - 3, 4.0, 80.0)]
CASES = [shape + (True,) for shape in PREIMAGE_SHAPES] + [(8, 64, 3.0, 25.0, False), _midsize() + (False,)]


@pytest.mark.parametrize("n,q,r,s,dense", CASES)
def test_tag_table_matches_per_tag_path(T, n, q, r, s, dense):
    """Shapes of test_tagged_matches_reduced_identity_key (dense and structured sqrt(Sigma_2)); dense, unitriangular and
    identity tags in one table, tag indices mixed at random."""
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 17 + q % 991)
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=n + 3, dense_sqrt_sigma_2=dense)
    tags = _mixed_tags(n, q, rng, 5)
    u = rng.integers(0, q, (2000, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), 2000).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=11, first_index=3)
    _assert_preimages(gp, a, np.eye(n, dtype=np.int64), tags, idx, e, u)
    assert psf.check_domain_batch(e).all()
    ref, _ = _per_tag(T, gp, r, s, a, td, tags, u, idx, 11, 3)
    assert np.array_equal(e, ref)


def test_tagged_key_entry_points_and_splits(T):
    """An installed key that is itself tagged (H_0 != I) gives the same preimages as the identity key of the same
    (A_bar, R); the table survives set_tag; host and device entry points, splits over calls (first_index) and over
    chunk sizes give identical preimages."""
    import torch
    from tools_b200 import _ffi

    n, q, r, s = 16, 2**20 - 3, 4.0, 80.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(23)
    psf = T.PSFPerturbation(gp, r, s)
    a_id, td = psf.trap_gen(seed=5)
    tags = _mixed_tags(n, q, rng, 6)
    u = rng.integers(0, q, (1500, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), 1500).astype(np.int32)
    e = psf.samp_p_tagged_batch(a_id, td, tags, u, idx, seed=9)
    ref, _ = _per_tag(T, gp, r, s, a_id, td, tags, u, idx, 9)
    assert np.array_equal(e, ref)
    # tagged installed key: same A_t for every t, so the same preimages; the table is kept across set_tag
    h0 = _dense_tag(n, q, rng)
    a0 = psf.set_tag(a_id, td, h0)
    assert psf._tags_id is tags
    assert np.array_equal(psf.samp_p_tagged_batch(a0, td, tags, u, idx, seed=9), e)
    _assert_preimages(gp, a0, h0, tags, idx, e, u)
    fresh = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(fresh.samp_p_tagged_batch(a0, td, tags, u, idx, seed=9), e)
    # splits over calls and over chunk sizes
    parts = np.concatenate([psf.samp_p_tagged_batch(a0, td, tags, u[:700], idx[:700], seed=9, first_index=0),
                            psf.samp_p_tagged_batch(a0, td, tags, u[700:], idx[700:], seed=9, first_index=700)])
    assert np.array_equal(parts, e)
    small = T.PSFPerturbation(gp, r, s)
    small.ctx.call("qf_set_chunk", 256)
    assert np.array_equal(small.samp_p_tagged_batch(a0, td, tags, u, idx, seed=9), e)
    # device-resident entry point
    dev = torch.device("cuda:0")
    ud = torch.from_numpy(u).to(dev)
    td_idx = torch.from_numpy(idx).to(dev)
    ed = torch.empty((u.shape[0], gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(td_idx.data_ptr()), u.shape[0], 9, 0,
                 _ffi.ptr(ed.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ed.cpu().numpy(), e)
    # the plain samp_p of the tagged key is untouched by the table
    assert np.array_equal(psf.samp_p_batch(a0, td, u, seed=4), T.PSFPerturbation(gp, r, s).samp_p_batch(a0, td, u, seed=4))


def test_tag_table_fp64_branch(T, monkeypatch):
    """QF_DISABLE_I8=1: v = u - A p on the fp64 path, with a tagged installed key."""
    monkeypatch.setenv("QF_DISABLE_I8", "1")
    n, q, r, s = 8, 127, 3.0, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(4)
    psf = T.PSFPerturbation(gp, r, s)
    a_id, td = psf.trap_gen(seed=6)
    h0 = _unitriangular_tag(n, q, rng)
    a0 = psf.set_tag(a_id, td, h0)
    tags = _mixed_tags(n, q, rng, 4)
    u = rng.integers(0, q, (900, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), 900).astype(np.int32)
    e = psf.samp_p_tagged_batch(a0, td, tags, u, idx, seed=2)
    _assert_preimages(gp, a0, h0, tags, idx, e, u)
    ref, _ = _per_tag(T, gp, r, s, a0, td, tags, u, idx, 2)
    assert np.array_equal(e, ref)


@pytest.mark.parametrize("n,q", [(4, 2**48), (64, 2**62 - 1)])
def test_tag_table_large_modulus(T, n, q):
    """64-bit table words.  q = 2^62 - 1 is the largest modulus a context accepts; at n = 64, (q - 1)^2 n >= 2^128, so the
    row sums of the per-target product need their third word."""
    gp = T.GadgetParameters.init_default(n, q)
    r = 3.0
    s = float(math.ceil(1.3 * math.sqrt(5 * ((math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) ** 2 / 2 + 1) + 1)))
    rng = np.random.default_rng(q % 1000 + n)
    psf = T.PSFPerturbation(gp, r, s)
    a_id, td = psf.trap_gen(seed=n + 2, dense_sqrt_sigma_2=n < 16)
    h0 = _dense_tag(n, q, rng)
    a0 = psf.set_tag(a_id, td, h0)
    tags = np.stack([_dense_tag(n, q, rng), _unitriangular_tag(n, q, rng), (q - 1) * np.eye(n, dtype=np.int64)])
    rows = 300 if n < 16 else 96
    u = rng.integers(0, q, (rows, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), rows).astype(np.int32)
    e = psf.samp_p_tagged_batch(a0, td, tags, u, idx, seed=7)
    _assert_preimages(gp, a0, h0, tags, idx, e, u)
    ref, _ = _per_tag(T, gp, r, s, a0, td, tags, u, idx, 7)
    assert np.array_equal(e, ref)


def test_tag_table_larger_than_one_slice(T):
    """T = 300 tags (two inversion slices), negative entries taken mod q: A_t e = u on every row, bit-identical rows for a
    sample of tags on both sides of the slice boundary."""
    n, q, r, s = 4, 127, 3.0, 25.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(300)
    tags = np.stack([_dense_tag(n, q, rng) if i % 2 else _unitriangular_tag(n, q, rng) for i in range(300)])
    tags[::7] -= q  # the same residues
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=12)
    u = rng.integers(0, q, (1200, n), dtype=np.int64)
    idx = rng.integers(0, 300, 1200).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=5)
    _assert_preimages(gp, a, np.eye(n, dtype=np.int64), tags % q, idx, e, u)
    only = [int(t) for t in (idx[0], 0, 255, 256, 299, 7) if (idx == t).any()]
    ref, done = _per_tag(T, gp, r, s, a, td, tags, u, idx, 5, only=only)
    assert done.any() and np.array_equal(e[done], ref[done])


def test_tag_table_refusals(T):
    import torch
    from tools_b200 import _ffi

    n, q, r, s = 8, 127, 3.0, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(41)
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=8)
    tags = _mixed_tags(n, q, rng, 3)
    u = rng.integers(0, q, (400, n), dtype=np.int64)
    idx = rng.integers(0, 3, 400).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=3)
    # a tag without a unit pivot at index 2: refused and named, the old table stays and samples as before
    bad = np.stack([tags[0], tags[1], _unitriangular_tag(n, q, rng)])
    bad[2][:, 1] = 0
    with pytest.raises(T.QfError) as ei:
        psf.set_tag_table(a, td, bad)
    assert ei.value.status == _ffi.QF_ERR_INVALID and "tag 2 " in str(ei.value)
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(np.empty((len(u), gp.m), np.int32))) == _ffi.QF_OK
    assert psf._tags_id is tags  # the wrapper keeps its cache on a refusal
    assert np.array_equal(psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=3), e)
    # an index out of range: host path before any launch, device path through qf_synchronize, no fault
    out = np.empty((len(u), gp.m), dtype=np.int32)
    badidx = idx.copy()
    badidx[17] = 3
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(badidx), len(u), 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    dev = torch.device("cuda:0")
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(badidx).to(dev)
    ed = torch.empty((len(u), gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    assert psf.ctx.status("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(idd.data_ptr()), len(u), 3, 0,
                          _ffi.ptr(ed.data_ptr())) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert "tag index outside the installed tag table" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    assert np.array_equal(psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=3), e)
    # no table, and a table dropped by qf_set_a or by a trapdoor re-install: QF_ERR_NO_KEY
    fresh = T.PSFPerturbation(gp, r, s)
    fresh._install_a(a)
    fresh._install_td(a, td)
    assert fresh.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_NO_KEY
    psf.ctx.call("qf_set_a", _ffi.ptr(np.ascontiguousarray(a)))
    psf._a_id, psf._td_id = a, None
    psf._install_td(a, td)  # key and trapdoor are back, the table is not
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_NO_KEY
    assert psf._tags_id is None
    assert np.array_equal(psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=3), e)
    psf._td_id = None
    psf._install_td(a, td)
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_NO_KEY
    # a key that is not a G-trapdoor for R, a GPV context, no key, bad arguments
    other = T.PSFPerturbation(gp, r, s)
    rand_a = rng.integers(0, q, (n, gp.m), dtype=np.int64)
    other._install_a(rand_a)
    other._install_td(rand_a, td)
    tg = np.ascontiguousarray(tags)
    assert other.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_ERR_INVALID
    g = T.PSFGPV(gp, 90.0)
    assert g.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_ERR_INVALID
    assert g.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    bare = T.PSFPerturbation(gp, r, s)
    assert bare.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_ERR_NO_KEY
    assert psf.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 0) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_set_tag_table", None, 3) == _ffi.QF_ERR_INVALID


def test_full_size_c4_shard_tag_table(T):
    """BASELINE.json configs[3] at full key size (n = 512, q = 2^32 - 5, k = 32, m = 32849, r = 9, structured
    sqrt(Sigma_2)) with T = 64 random unitriangular tags: A_t e = u for 2048 targets (exact, 16-bit splits), check_domain,
    the second moment, and the rows of two tags bit-identical to the per-tag path."""
    n, q, r = 512, 2**32 - 5, 9.0
    gp = T.GadgetParameters.init_default(n, q)
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
    s = float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))
    rng = np.random.default_rng(64)
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=4, dense_sqrt_sigma_2=False)
    tags = np.stack([_unitriangular_tag(n, q, rng) for _ in range(64)])
    u = rng.integers(0, q, (2048, n), dtype=np.int64)
    idx = rng.permutation(np.arange(2048) % 64).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=9)
    _assert_preimages(gp, a, np.eye(n, dtype=np.int64), tags, idx, e, u)
    assert psf.check_domain_batch(e).all()
    ratio = (e.astype(np.float64) ** 2).sum(1).mean() / (gp.m * (s * r) ** 2 / (2 * math.pi))
    assert abs(ratio - 1) < 0.01, ratio
    psf.ctx.close()
    ref, done = _per_tag(T, gp, r, s, a, td, tags, u[:256], idx[:256], 9, only=[int(idx[0]), int(idx[1])])
    assert done.any() and np.array_equal(e[:256][done], ref[done])
