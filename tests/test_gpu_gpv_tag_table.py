"""PSFGPV samp_p with a tag per target and tag switching on one short basis (qf_set_tag_table, qf_samp_p_tagged[_dev],
qf_gpv_set_tag; DESIGN.md 4.3).  The reference of every sampling test is the per-tag path on the same context:
qf_gpv_set_tag(H_t) + samp_p on the WHOLE batch with the same seed and first_index, restricted to the rows with
tag_idx == t.  Both compute the same integer h_t = H_t^-1 (u - A_bar z2) between the phases, so the rows must be
bit-identical; A_t e = u must hold exactly on every row.  The identity behind it is pinned on the CPU in
test_gpv_tag_table_math.py."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _gpv_s(gp):
    return float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(gp.n)))


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


def _f_a(a, e, q):
    """A e mod q for a batch of preimages (rows of e), exact."""
    if q >= 2**32:
        return np.array(e.astype(object).dot(a.T.astype(object)) % q, dtype=np.int64)
    ef = e.astype(np.float64)  # |e| < 2^16, 16-bit halves of A: |partial sums| < 2^32 m < 2^53
    lo = np.rint(ef @ (a & 0xFFFF).astype(np.float64).T).astype(np.int64)
    hi = np.rint(ef @ (a >> 16).astype(np.float64).T).astype(np.int64)
    return (lo % q + ((hi % q) << 16) % q) % q


def _key(T, gp, seed, h0):
    """A context with the key [A_bar | H_0 G - A_bar R] and its basis installed; returns (psf, a, td, A_bar, R)."""
    psf = T.PSFGPV(gp, _gpv_s(gp))
    a0, r = T.psf._trap_gen_classical(psf, seed=seed)
    ab = np.ascontiguousarray(a0[:, : gp.m_bar])
    a = a0 if h0 is None else T.psf.gen_trapdoor(gp, ab, r, h0)
    psf._install_a(a)
    td = (psf.gen_short_basis_for_trapdoor(r, h0), None)
    psf._install_td(a, td)
    return psf, a, td, ab, r


def _mixed_tags(n, q, rng, count):
    kinds = (_dense_tag, _unitriangular_tag, lambda n, q, rng: np.eye(n, dtype=np.int64))
    return np.stack([kinds[i % 3](n, q, rng) for i in range(count)])


def _second_moment(e, gp, s):
    return (e.astype(np.float64) ** 2).sum(1).mean() / (gp.m * s * s / (2 * math.pi))


@pytest.mark.parametrize("installed", ["identity", "tagged"])
@pytest.mark.parametrize("n,q", [(64, 2**16), (128, 2**12), (64, 4093)])
def test_gpv_tag_table_matches_set_tag_and_fresh_keys(T, monkeypatch, n, q, installed):
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(n + q % 1000 + (5 if installed == "tagged" else 0))
    h0 = None if installed == "identity" else _dense_tag(n, q, rng)
    psf, a, td, ab, r = _key(T, gp, n + 1, h0)
    tags = _mixed_tags(n, q, rng, 4)
    B = 1500
    u = rng.integers(0, q, (B, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), B).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=7, first_index=3)
    assert psf.check_domain_batch(e).all()
    assert abs(_second_moment(e, gp, s) - 1) < 0.02
    # round trip: the verifier's tagged f_a gives u back
    got, ok = psf.f_a_tagged_batch(a, tags, e, idx, h0=h0)
    assert np.array_equal(got, u) and ok.all()
    # the per-tag path on the same context: every row bit-identical, A_t e = u with the switched key
    cur, cur_td = a, td
    keys = {}
    for t in range(len(tags)):
        cur, cur_td = psf.set_tag(cur, cur_td, tags[t])
        keys[t] = (cur, cur_td)
        ref = psf.samp_p_batch(cur, cur_td, u, seed=7, first_index=3)
        rows = idx == t
        assert np.array_equal(e[rows], ref[rows]), t
        assert np.array_equal(_f_a(cur, e[rows], q), u[rows]), t
    assert np.array_equal(O.f_a_classical_batch(keys[0][0], e[idx == 0][:3], q), u[idx == 0][:3])
    # the table survived the switches and does not depend on the installed tag
    assert np.array_equal(psf.samp_p_tagged_batch(cur, cur_td, tags, u, idx, seed=7, first_index=3), e)
    # a fresh install per tag (own context, own GSO): exact, and the same preimages up to fp64 rounding of the GSO
    for t in (0, 1):
        fresh = T.PSFGPV(gp, s)
        fresh.ctx.call("qf_set_chunk", 4096)
        a_t = T.psf.gen_trapdoor(gp, ab, r, tags[t])
        fresh._install_a(a_t)
        sb_t = fresh.gen_short_basis_for_trapdoor(r, tags[t])
        assert np.array_equal(a_t, keys[t][0]) and np.array_equal(sb_t, keys[t][1][0])
        ef = fresh.samp_p_batch(a_t, (sb_t, None), u, seed=7, first_index=3)
        rows = idx == t
        assert np.array_equal(_f_a(a_t, ef, q), u)
        same = float((ef[rows] == e[rows]).all(axis=1).mean())
        print(f"n={n} q={q} installed={installed} tag {t}: {same:.4f} of rows bit-identical to a fresh install")
        assert same >= 0.90, same
        fresh.ctx.close()


def test_gpv_set_tag_switch_back_refusals_and_tables(T, monkeypatch):
    from tools_b200 import _ffi, gadget

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(77)
    h0 = _unitriangular_tag(n, q, rng)
    h1 = _dense_tag(n, q, rng)
    psf, a, td, ab, r = _key(T, gp, 11, h0)
    u = rng.integers(0, q, (700, n), dtype=np.int64)
    e0 = psf.samp_p_batch(a, td, u, seed=4)
    tags = _mixed_tags(n, q, rng, 3)
    idx = rng.integers(0, 3, len(u)).astype(np.int32)
    et = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=4)
    psf.f_a_tagged_batch(a, tags, et, idx, h0=h0)  # installs the f_a table
    a1, td1 = psf.set_tag(a, td, h1)
    assert np.array_equal(a1, T.psf.gen_trapdoor(gp, ab, r, h1))
    assert np.array_equal(td1[0], gadget.gen_short_basis_for_trapdoor(gp, a1, r, h1.astype(object)))
    e1 = psf.samp_p_batch(a1, td1, u, seed=4)
    assert np.array_equal(_f_a(a1, e1, q), u)
    # the f_a table went with the old A; the samp_p table stays
    sig = np.ascontiguousarray(et)
    out_u = np.empty((len(u), n), dtype=np.int64)
    flags = np.empty(len(u), dtype=np.uint8)
    assert psf.ctx.status("qf_f_a_tagged", _ffi.ptr(sig), _ffi.ptr(idx), len(u), _ffi.ptr(out_u), _ffi.ptr(flags)) == _ffi.QF_ERR_NO_KEY
    assert psf._tags_id is tags and psf._fa_tags_id is None
    assert np.array_equal(psf.samp_p_tagged_batch(a1, td1, tags, u, idx, seed=4), et)
    # back to H_0: the earlier preimages, bit for bit
    a2, td2 = psf.set_tag(a1, td1, h0)
    assert np.array_equal(a2, a) and np.array_equal(td2[0], td[0])
    assert np.array_equal(psf.samp_p_batch(a2, td2, u, seed=4), e0)
    # a tag without a unit pivot: refused, nothing changes
    bad = _unitriangular_tag(n, q, rng)
    bad[:, 3] = 0
    with pytest.raises(T.QfError) as ei:
        psf.set_tag(a2, td2, bad)
    assert ei.value.status == _ffi.QF_ERR_INVALID
    assert psf._a_id is a2 and psf._td_id is td2
    e_after = np.empty((len(u), gp.m), dtype=np.int32)
    psf.ctx.call("qf_samp_p", _ffi.ptr(u), len(u), 4, 0, _ffi.ptr(e_after))
    assert np.array_equal(e_after, e0)
    # the switched trapdoor installed on a fresh context takes the two-phase path (it accepts a tag table)
    fresh = T.PSFGPV(gp, s)
    ef = fresh.samp_p_batch(a1, td1, u, seed=4)
    assert np.array_equal(_f_a(a1, ef, q), u)
    assert float((ef == e1).all(axis=1).mean()) >= 0.9
    tg = np.ascontiguousarray(tags)
    assert fresh.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_OK
    # the identity tag: back to the untagged key
    a3, td3 = psf.set_tag(a2, td2, None)
    assert np.array_equal(a3, T.psf.gen_trapdoor(gp, ab, r, None))
    plain = T.PSFGPV(gp, s)
    plain._install_a(a3)
    assert np.array_equal(td3[0], plain.gen_short_basis_for_trapdoor(r))
    e3 = psf.samp_p_batch(a3, td3, u, seed=4)
    assert np.array_equal(_f_a(a3, e3, q), u)


def test_gpv_tag_table_entry_points(T, monkeypatch):
    import torch
    from tools_b200 import _ffi

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(91)
    psf, a, td, ab, r = _key(T, gp, 21, None)
    u = rng.integers(0, q, (1300, n), dtype=np.int64)
    # untagged samp_p: same outputs and launches before and after a table is installed
    before = np.empty((len(u), gp.m), dtype=np.int32)
    c0 = psf.ctx.launch_count()
    psf.ctx.call("qf_samp_p", _ffi.ptr(u), len(u), 6, 0, _ffi.ptr(before))
    launches_plain = psf.ctx.launch_count() - c0
    tags = _mixed_tags(n, q, rng, 5)
    idx = rng.integers(0, 5, len(u)).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=6)
    after = np.empty_like(before)
    c0 = psf.ctx.launch_count()
    psf.ctx.call("qf_samp_p", _ffi.ptr(u), len(u), 6, 0, _ffi.ptr(after))
    assert psf.ctx.launch_count() - c0 == launches_plain
    assert np.array_equal(before, after)
    # split over calls and over small chunks
    parts = np.concatenate([psf.samp_p_tagged_batch(a, td, tags, u[:500], idx[:500], seed=6, first_index=0),
                            psf.samp_p_tagged_batch(a, td, tags, u[500:], idx[500:], seed=6, first_index=500)])
    assert np.array_equal(parts, e)
    small = T.PSFGPV(gp, s)
    small.ctx.call("qf_set_chunk", 256)
    assert np.array_equal(small.samp_p_tagged_batch(a, td, tags, u, idx, seed=6), e)
    # device entry point
    dev = torch.device("cuda:0")
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(idx).to(dev)
    ed = torch.empty((len(u), gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(idd.data_ptr()), len(u), 6, 0,
                 _ffi.ptr(ed.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ed.cpu().numpy(), e)
    # bad index: host refuses before any launch, device reports at qf_synchronize
    badidx = idx.copy()
    badidx[33] = 5
    out = np.empty((len(u), gp.m), dtype=np.int32)
    c0 = psf.ctx.launch_count()
    assert psf.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(badidx), len(u), 6, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    assert psf.ctx.launch_count() == c0
    bd = torch.from_numpy(badidx).to(dev)
    torch.cuda.synchronize()
    assert psf.ctx.status("qf_samp_p_tagged_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(bd.data_ptr()), len(u), 6, 0,
                          _ffi.ptr(ed.data_ptr())) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK
    assert np.array_equal(psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=6), e)


def test_gpv_tag_table_refusals(T, monkeypatch):
    from tools_b200 import _ffi

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(5)
    tags = _mixed_tags(n, q, rng, 3)
    tg = np.ascontiguousarray(tags)
    u = rng.integers(0, q, (300, n), dtype=np.int64)
    idx = rng.integers(0, 3, len(u)).astype(np.int32)
    out = np.empty((len(u), gp.m), dtype=np.int32)
    eye = np.eye(n, dtype=np.int64)

    def sample(p):
        return p.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(idx), len(u), 3, 0, _ffi.ptr(out))

    psf, a, td, ab, r = _key(T, gp, 3, None)
    assert sample(psf) == _ffi.QF_ERR_NO_KEY  # two-phase, no table
    psf.set_tag_table(a, td, tags)
    assert sample(psf) == _ffi.QF_OK
    # the table is dropped by qf_set_trapdoor_gpv, qf_set_a and trap_gen
    psf._td_id = None
    psf._install_td(a, td)
    assert psf._tags_id is None and sample(psf) == _ffi.QF_ERR_NO_KEY
    psf.set_tag_table(a, td, tags)
    psf.ctx.call("qf_set_a", _ffi.ptr(np.ascontiguousarray(a)))
    psf._a_id, psf._td_id = a, None
    psf._install_td(a, td)
    assert sample(psf) == _ffi.QF_ERR_NO_KEY
    psf.set_tag_table(a, td, tags)
    a2, td2 = psf.trap_gen(seed=9, dense_gso=False)
    psf._install_td(a2, td2)
    assert psf._tags_id is None and sample(psf) == _ffi.QF_ERR_NO_KEY
    # a key but no trapdoor
    bare = T.PSFGPV(gp, s)
    bare._install_a(a)
    assert bare.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_ERR_INVALID
    assert bare.ctx.status("qf_gpv_set_tag", _ffi.ptr(eye), None, None) == _ffi.QF_ERR_INVALID
    # the one-pass recursion: QF_DISABLE_TWO_PHASE=1, and a dimension below the tensor-core threshold
    monkeypatch.setenv("QF_DISABLE_TWO_PHASE", "1")
    one, a1, td1, _, _ = _key(T, gp, 3, None)
    assert one.ctx.status("qf_set_tag_table", _ffi.ptr(tg), 3) == _ffi.QF_ERR_INVALID
    assert sample(one) == _ffi.QF_ERR_INVALID
    assert one.ctx.status("qf_gpv_set_tag", _ffi.ptr(eye), None, None) == _ffi.QF_ERR_INVALID
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE")
    gs = T.GadgetParameters.init_default(8, 127)
    low, _, _, _, _ = _key(T, gs, 3, None)
    t8 = np.ascontiguousarray(np.eye(8, dtype=np.int64)[None])
    assert low.ctx.status("qf_set_tag_table", _ffi.ptr(t8), 1) == _ffi.QF_ERR_INVALID
    # ring context, PSFPerturbation context
    ring = T.PSFGPVRing(T.GadgetParametersRing.init_default(8, 257), 20.0, 2.0)
    assert ring.ctx.status("qf_set_tag_table", _ffi.ptr(t8), 1) == _ffi.QF_ERR_INVALID
    i8 = np.zeros(1, dtype=np.int32)
    assert ring.ctx.status("qf_samp_p_tagged", _ffi.ptr(u), _ffi.ptr(i8), 1, 3, 0, _ffi.ptr(out)) == _ffi.QF_ERR_INVALID
    assert ring.ctx.status("qf_gpv_set_tag", None, None, None) == _ffi.QF_ERR_INVALID
    pert = T.PSFPerturbation(gp, 3.0, 200.0)
    pa, ptd = pert.trap_gen(seed=2)
    pert._install_a(pa)
    pert._install_td(pa, ptd)
    assert pert.ctx.status("qf_gpv_set_tag", _ffi.ptr(eye), None, None) == _ffi.QF_ERR_INVALID


@pytest.mark.parametrize("n,q,base", [(16, 2**48, 2), (40, 2**61 - 1, 16)])
def test_gpv_tag_table_large_modulus(T, monkeypatch, n, q, base):
    """Residues of 7 and 8 digits (the shapes of test_tagged_key_install_large_modulus).  The tag table gives the set_tag
    path's preimages, or both fail with the same status -- the trapdoor install itself may refuse such a modulus (the
    particular-solution product of qf_set_trapdoor_gpv), and then both paths report that refusal."""
    from tools_b200 import gadget

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    k = gadget._ceil_log(q, base)
    gp = T.GadgetParameters(n=n, k=k, m_bar=n * k + gadget._ceil_log(n, 2) ** 2, base=base, q=q)
    rng = np.random.default_rng(q % 997)
    psf = T.PSFGPV(gp, _gpv_s(gp))
    a, r = T.psf._trap_gen_classical(psf, seed=5)
    ab = np.ascontiguousarray(a[:, : gp.m_bar])
    psf._install_a(a)
    td = (psf.gen_short_basis_for_trapdoor(r), None)  # installed (or refused) by the first call below
    tags = np.stack([_dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)])
    u = rng.integers(0, q, (300, n), dtype=np.int64)
    idx = rng.integers(0, 2, len(u)).astype(np.int32)

    def outcome(f):
        try:
            return f(), None
        except T.QfError as err:
            return None, err.status

    e, st = outcome(lambda: psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=2))
    for t in range(2):
        key, st_t = outcome(lambda: psf.set_tag(a, td, tags[t]))
        if key is not None:
            a, td = key
            assert np.array_equal(a, T.psf.gen_trapdoor(gp, ab, r, tags[t]))
            e_t, st_t = outcome(lambda: psf.samp_p_batch(a, td, u, seed=2))
        assert st == st_t, (st, st_t)
        print(f"n={n} q={q}: tag {t}: status {st}")
        if e is not None:
            rows = idx == t
            assert np.array_equal(e[rows], e_t[rows])
            assert np.array_equal(_f_a(a, e[rows], q), u[rows])


def test_gpv_tag_table_full_size_c2(T, monkeypatch):
    """C2 (n = 256, q = 2^24, m = 12352) with T = 64 random unitriangular tags: A_t e = u for 37 888 targets checked on the
    device (f_a_tagged_batch, with check_domain), the second moment, and the rows of two tags bit-identical to the set_tag
    path."""
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    monkeypatch.delenv("QF_OZAKI_MIN_DIM", raising=False)
    n, q = 256, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(64)
    psf = T.PSFGPV(gp, s)
    a, td = psf.trap_gen(seed=2, dense_gso=False)
    tags = np.stack([_unitriangular_tag(n, q, rng) for _ in range(64)])
    B = 37888
    u = rng.integers(0, q, (B, n), dtype=np.int64)
    idx = rng.permutation(np.arange(B) % 64).astype(np.int32)
    e = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=3)
    got, ok = psf.f_a_tagged_batch(a, tags, e, idx, strict=False)
    assert np.array_equal(got, u) and ok.all()
    assert abs(_second_moment(e, gp, s) - 1) < 0.02
    for t in (int(idx[0]), 63):
        a_t, td_t = psf.set_tag(a, td, tags[t])
        ref = psf.samp_p_batch(a_t, td_t, u, seed=3)
        assert np.array_equal(e[idx == t], ref[idx == t]), t
        a, td = psf.set_tag(a_t, td_t, None)
