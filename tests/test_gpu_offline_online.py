"""Offline / online samp_p (qf_samp_p_offline, qf_samp_p_online[_dev], qf_samp_p_pool_info; DESIGN.md 4.12).  The reference
of every sampling test is qf_samp_p (qf_samp_p_tagged) on the same context with the pool's seed at the same sampler
indices: an online row must be bit-identical to it, whatever the split into fills, online calls and chunks.  A e = u
(A_t e = u) is checked exactly on every row.  Small chunks (qf_set_chunk) make fills and online calls cross chunk
boundaries."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu

SPLITS = (1, 300, 700)  # three online calls over one fill of sum(SPLITS) entries


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _f_a(a, e, q):
    """A e mod q for a batch of preimages (rows of e), exact."""
    if q >= 2**32:
        return O.f_a_classical_batch(a, e, q)
    ef = e.astype(np.float64)  # |e| < 2^16, 16-bit halves of A: |partial sums| < 2^32 m < 2^53
    lo = np.rint(ef @ (a & 0xFFFF).astype(np.float64).T).astype(np.int64)
    hi = np.rint(ef @ (a >> 16).astype(np.float64).T).astype(np.int64)
    return (lo % q + ((hi % q) << 16) % q) % q


def _gpv_s(gp):
    return float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(gp.n)))


def _pert_s(gp):
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(gp.n * gp.k)) / math.sqrt(2)
    return float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))


def _unitriangular_tag(n, q, rng):
    return np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)


def _poly_tags(T, n, q, rng, count):
    """count units of Z_q[X]/(X^n + 1), q a power of two: odd coefficient sum (a unit mod 2 = a unit mod q)."""
    h = rng.integers(0, q, (count, n), dtype=np.int64)
    h[:, 0] += 1 - h.sum(1) % 2
    h %= q
    f = np.zeros(n, dtype=np.int64)
    f[0] = 1
    return T.PolyTags(f, h)


def _online_in_calls(psf, a, td, u, splits, **tags):
    """Online rows for u in len(splits) calls; checks the cursor on the way.  Returns (rows, first index of row 0)."""
    rows, first0 = [], None
    b0 = 0
    for size in splits:
        rem0, nxt0 = psf.pool_info()
        kw = {}
        if tags:
            kw = dict(tags=tags["tags"], tag_idx=tags["tag_idx"][b0:b0 + size])
        e, first = psf.samp_p_online_batch(a, td, u[b0:b0 + size], **kw)
        assert first == nxt0 and psf.pool_info() == (rem0 - size, nxt0 + size)
        first0 = first if first0 is None else first0
        rows.append(e)
        b0 += size
    return np.concatenate(rows), first0


def _check_untagged(T, psf, gp, a, td, rng, seed=7):
    """Two fills (the second at a gap of indices), uneven online calls over each, against qf_samp_p at the same indices."""
    n, q = gp.n, gp.q
    for first, splits in ((5, SPLITS), (5000, (450, 1, 549))):
        B = sum(splits)
        u = rng.integers(0, q, (B, n), dtype=np.int64)
        psf.samp_p_offline(a, td, B, seed=seed, first_index=first)
        assert psf.pool_info() == (B, first)
        e, f0 = _online_in_calls(psf, a, td, u, splits)
        assert f0 == first and psf.pool_info() == (0, first + B)
        ref = psf.samp_p_batch(a, td, u, seed=seed, first_index=first)
        assert np.array_equal(e, ref)
        assert np.array_equal(_f_a(a, e, q), u)


def _check_tagged(T, psf, gp, a, td, rng, tags, seed=9, h0=None):
    """One fill, online calls with a tag per target, against qf_samp_p_tagged; A_t e = u through the f_a tag table."""
    n, q = gp.n, gp.q
    B = sum(SPLITS)
    u = rng.integers(0, q, (B, n), dtype=np.int64)
    idx = rng.integers(0, len(tags), B).astype(np.int32)
    psf.set_tag_table(a, td, tags)
    psf.samp_p_offline(a, td, B, seed=seed, first_index=11)
    psf.set_tag_table(a, td, tags)  # a table install keeps the pool
    assert psf.pool_info() == (B, 11)
    e, _ = _online_in_calls(psf, a, td, u, SPLITS, tags=tags, tag_idx=idx)
    ref = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=seed, first_index=11)
    assert np.array_equal(e, ref)
    got, ok = psf.f_a_tagged_batch(a, tags, e, idx, h0=h0, strict=False)
    assert np.array_equal(got, u) and ok.all()


@pytest.mark.parametrize("installed", ["identity", "tagged"])
@pytest.mark.parametrize("n,q", [(64, 2**16), (64, 2**24)])
def test_gpv_two_phase_online_bit_identical(T, monkeypatch, n, q, installed):
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n + q % 991 + (3 if installed == "tagged" else 0))
    psf = T.PSFGPV(gp, _gpv_s(gp))
    h0 = None if installed == "identity" else _unitriangular_tag(n, q, rng)
    a, td = psf.trap_gen(seed=n + 1, dense_gso=False, tag=h0)
    psf.ctx.call("qf_set_chunk", 384)
    _check_untagged(T, psf, gp, a, td, rng)
    _check_tagged(T, psf, gp, a, td, rng, np.stack([_unitriangular_tag(n, q, rng) for _ in range(3)]), h0=h0)
    _check_tagged(T, psf, gp, a, td, rng, _poly_tags(T, n, q, rng, 5), h0=h0)


# (n, q, r, s, dense sqrt(Sigma_2), tensor-core path); the structured square root needs the tensor-core path
PERT_CASES = [
    (8, 64, 3.0, 25.0, True, True),  # C1 (README example)
    (8, 64, 3.0, 25.0, True, False),
    (16, 2**20, 4.0, 80.0, True, True),
    (16, 2**20, 4.0, 80.0, True, False),
    (16, 2**16, 4.0, None, False, True),
    (64, 2**16, 6.0, None, False, True),
]


@pytest.mark.parametrize("n,q,r,s,dense,i8", PERT_CASES)
def test_perturbation_online_bit_identical(T, monkeypatch, n, q, r, s, dense, i8):
    if not i8:
        monkeypatch.setenv("QF_DISABLE_I8", "1")
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFPerturbation(gp, r, _pert_s(gp) if s is None else s)
    a, td = psf.trap_gen(seed=n + 3, dense_sqrt_sigma_2=dense)
    psf.ctx.call("qf_set_chunk", 256)
    rng = np.random.default_rng(n * 7 + q % 101)
    _check_untagged(T, psf, gp, a, td, rng)
    _check_tagged(T, psf, gp, a, td, rng, np.stack([_unitriangular_tag(n, q, rng) for _ in range(4)]))
    _check_tagged(T, psf, gp, a, td, rng, _poly_tags(T, n, q, rng, 3))


@pytest.mark.parametrize("kind", ["gpv", "pert"])
def test_dev_form_matches_host_form(T, monkeypatch, kind):
    import torch

    from tools_b200 import _ffi

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    if kind == "gpv":
        psf = T.PSFGPV(gp, _gpv_s(gp))
        a, td = psf.trap_gen(seed=5, dense_gso=False)
    else:
        psf = T.PSFPerturbation(gp, 6.0, _pert_s(gp))
        a, td = psf.trap_gen(seed=5, dense_sqrt_sigma_2=False)
    psf.ctx.call("qf_set_chunk", 256)
    rng = np.random.default_rng(17)
    B = 700
    u = rng.integers(0, q, (B, n), dtype=np.int64)
    tags = np.stack([_unitriangular_tag(n, q, rng) for _ in range(3)])
    idx = rng.integers(0, 3, B).astype(np.int32)
    psf.set_tag_table(a, td, tags)
    dev = torch.device("cuda:0")
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(idx).to(dev)
    for tagged in (False, True):
        psf.samp_p_offline(a, td, 2 * B, seed=13, first_index=100)
        host, f_host = psf.samp_p_online_batch(a, td, u, **(dict(tags=tags, tag_idx=idx) if tagged else {}))
        ed = torch.empty((B, gp.m), dtype=torch.int32, device=dev)
        first = _ffi.C.c_uint64()
        torch.cuda.synchronize()
        psf.ctx.call("qf_samp_p_online_dev", _ffi.ptr(ud.data_ptr()), _ffi.ptr(idd.data_ptr()) if tagged else None, B,
                     _ffi.ptr(ed.data_ptr()), _ffi.C.byref(first))
        assert psf.pool_info() == (0, 100 + 2 * B)  # consumed at enqueue
        psf.ctx.call("qf_synchronize")
        assert f_host == 100 and first.value == 100 + B
        got = ed.cpu().numpy()
        if tagged:
            ref = psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=13, first_index=100 + B)
        else:
            ref = psf.samp_p_batch(a, td, u, seed=13, first_index=100 + B)
        assert np.array_equal(got, ref)
        assert np.array_equal(host, psf.samp_p_batch(a, td, u, seed=13, first_index=100) if not tagged
                              else psf.samp_p_tagged_batch(a, td, tags, u, idx, seed=13, first_index=100))


def _online_status(psf, u, tag_idx=None):
    from tools_b200 import _ffi

    uu = np.ascontiguousarray(u, dtype=np.int64)
    e = np.empty((len(uu), psf.m), dtype=np.int32)
    ti = None if tag_idx is None else np.ascontiguousarray(tag_idx, dtype=np.int32)
    return psf.ctx.status("qf_samp_p_online", _ffi.ptr(uu), _ffi.ptr(ti), len(uu), _ffi.ptr(e), None)


def test_cursor_refusals_and_lifetime_perturbation(T):
    from tools_b200 import _ffi

    n, q = 16, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFPerturbation(gp, 4.0, _pert_s(gp))
    a, td = psf.trap_gen(seed=3, dense_sqrt_sigma_2=False)
    rng = np.random.default_rng(1)
    u = rng.integers(0, q, (40, n), dtype=np.int64)
    assert psf.pool_info() == (0, 0)
    assert _online_status(psf, u[:1]) == _ffi.QF_ERR_NO_KEY  # no pool
    psf.samp_p_offline(a, td, 30, seed=2, first_index=7)
    # batch > remaining: refused before any launch, nothing consumed
    assert _online_status(psf, u[:31]) == _ffi.QF_ERR_INVALID and psf.pool_info() == (30, 7)
    # batch 0 is valid and consumes nothing
    e0, f0 = psf.samp_p_online_batch(a, td, u[:0])
    assert e0.shape == (0, gp.m) and f0 == 7 and psf.pool_info() == (30, 7)
    # targets outside [0, q) and bad tag indices are refused as by qf_samp_p / qf_samp_p_tagged
    bad = u[:2].copy()
    bad[1, 3] = q
    assert _online_status(psf, bad) == _ffi.QF_ERR_INVALID
    tags = np.stack([_unitriangular_tag(n, q, rng) for _ in range(2)])
    psf.set_tag_table(a, td, tags)
    assert _online_status(psf, u[:2], [0, 2]) == _ffi.QF_ERR_INVALID
    rem, nxt = psf.pool_info()
    # no entry is served twice: the rest of the pool is the rest of the index range
    e, f = psf.samp_p_online_batch(a, td, u[:rem])
    assert f == nxt and psf.pool_info() == (0, 37)
    assert np.array_equal(e, psf.samp_p_batch(a, td, u[:rem], seed=2, first_index=nxt))
    assert _online_status(psf, u[:1]) == _ffi.QF_ERR_INVALID  # empty pool
    # a refill replaces the pool
    psf.samp_p_offline(a, td, 10, seed=4, first_index=0)
    psf.samp_p_offline(a, td, 5, seed=5, first_index=50)
    assert psf.pool_info() == (5, 50)
    e, f = psf.samp_p_online_batch(a, td, u[:5])
    assert f == 50 and np.array_equal(e, psf.samp_p_batch(a, td, u[:5], seed=5, first_index=50))
    # lifetime: tag tables keep the pool, key / trapdoor / tag changes drop it
    r, l, gb = td
    r8 = np.ascontiguousarray(r, dtype=np.int8)
    tag = _unitriangular_tag(n, q, rng)

    def refill():
        psf.samp_p_offline(a, td, 4, seed=1)
        assert psf.pool_info() == (4, 0)

    refill()
    psf.ctx.call("qf_set_f_a_tags", _ffi.ptr(tags), 2, None)
    f_poly = _poly_tags(T, n, q, rng, 2)
    fw, tw = f_poly.words(q)
    psf.ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(tw), 2)
    psf.ctx.call("qf_set_f_a_tags_poly", _ffi.ptr(fw), _ffi.ptr(tw), 2, None)
    psf.ctx.call("qf_set_tag_table", _ffi.ptr(tags), 2)
    assert psf.pool_info() == (4, 0)
    # every buffer a call reads stays referenced here (a temporary would be freed before the call)
    blk = np.ascontiguousarray(np.asarray(gb[0])[:gp.k, :gp.k], dtype=np.int64)
    gblk = np.ascontiguousarray(np.asarray(gb[1], dtype=np.float64)[:gp.k, :gp.k])
    abar = np.ascontiguousarray(a[:, :gp.m_bar])
    a_out = np.empty((n, gp.m), dtype=np.int64)
    r_out = np.empty((gp.m_bar, n * gp.k), dtype=np.int8)
    drops = [
        lambda: psf.ctx.call("qf_set_tag", _ffi.ptr(tag), None),
        lambda: psf.ctx.call("qf_set_trapdoor_perturbation", _ffi.ptr(r8), None, _ffi.ptr(blk), _ffi.ptr(gblk)),
        lambda: psf.ctx.call("qf_set_a", _ffi.ptr(a)),
        lambda: psf.ctx.call("qf_trap_gen_from", _ffi.ptr(abar), _ffi.ptr(r8), None, _ffi.ptr(a_out)),
        lambda: psf.ctx.call("qf_trap_gen", 9, _ffi.ptr(a_out), _ffi.ptr(r_out)),
    ]
    for i, drop in enumerate(drops):
        psf._a_id = psf._td_id = psf._tags_id = psf._fa_tags_id = None  # re-install the key and trapdoor below
        refill()
        drop()
        assert psf.pool_info() == (0, 0), i
        assert _online_status(psf, u[:1]) == _ffi.QF_ERR_NO_KEY, i


def test_lifetime_gpv_and_refusals(T, monkeypatch):
    from tools_b200 import _ffi

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFGPV(gp, _gpv_s(gp))
    # no key / trapdoor
    assert psf.ctx.status("qf_samp_p_offline", 4, 1, 0) == _ffi.QF_ERR_NO_KEY
    a, td = psf.trap_gen(seed=6, dense_gso=False)
    rng = np.random.default_rng(2)
    u = rng.integers(0, q, (2, n), dtype=np.int64)
    s = np.ascontiguousarray(td[0], dtype=np.int64)
    tag = _unitriangular_tag(n, q, rng)
    for i, drop in enumerate([
        lambda: psf.ctx.call("qf_gpv_set_tag", _ffi.ptr(tag), None, None),
        lambda: psf.ctx.call("qf_set_trapdoor_gpv", _ffi.ptr(s), None),
        lambda: psf.ctx.call("qf_set_a", _ffi.ptr(a)),
    ]):
        psf._a_id = psf._td_id = psf._tags_id = psf._fa_tags_id = None
        psf.samp_p_offline(a, td, 3, seed=1)
        psf.ctx.call("qf_set_tag_table", _ffi.ptr(tag), 1)
        assert psf.pool_info() == (3, 0), i
        drop()
        assert psf.pool_info() == (0, 0), i
        assert _online_status(psf, u[:1]) == _ffi.QF_ERR_NO_KEY, i
    # one-pass recursion (below the tensor-core threshold): the first step reads the target
    gp8 = T.GadgetParameters.init_default(8, 64)
    g8 = T.PSFGPV(gp8, 90.0)
    a8, td8 = g8.trap_gen(seed=4)
    g8._install_a(a8)
    g8._install_td(a8, td8)
    assert g8.ctx.status("qf_samp_p_offline", 4, 1, 0) == _ffi.QF_ERR_UNSUPPORTED
    # ring context
    gpr = T.GadgetParametersRing.init_default(16, 3329)
    ring = T.PSFGPVRing(gpr, 10.0, 1.0)
    assert ring.ctx.status("qf_samp_p_offline", 4, 1, 0) == _ffi.QF_ERR_UNSUPPORTED


def test_full_size_c2_gpv(T, monkeypatch):
    """C2 PSFGPV (n = 256, q = 2^24, m = 12352): 4000 targets from one fill in two online calls."""
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    monkeypatch.delenv("QF_OZAKI_MIN_DIM", raising=False)
    n, q = 256, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFGPV(gp, _gpv_s(gp))
    a, td = psf.trap_gen(seed=2, dense_gso=False)
    rng = np.random.default_rng(3)
    u = rng.integers(0, q, (4000, n), dtype=np.int64)
    psf.samp_p_offline(a, td, 4000, seed=3, first_index=1000)
    e, f = _online_in_calls(psf, a, td, u, (1500, 2500))
    assert f == 1000 and np.array_equal(e, psf.samp_p_batch(a, td, u, seed=3, first_index=1000))
    got, ok = psf.f_a_batch(a, e, strict=False)
    assert np.array_equal(got, u) and ok.all()


def test_full_size_c4_shard_perturbation(T):
    """C4 shard (n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2)): 3000 targets, one fill, two calls."""
    n, q = 512, 2**32 - 5
    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFPerturbation(gp, 9.0, _pert_s(gp))
    a, td = psf.trap_gen(seed=4, dense_sqrt_sigma_2=False)
    rng = np.random.default_rng(5)
    u = rng.integers(0, q, (3000, n), dtype=np.int64)
    psf.samp_p_offline(a, td, 3000, seed=6)
    e, f = _online_in_calls(psf, a, td, u, (1000, 2000))
    assert f == 0 and np.array_equal(e, psf.samp_p_batch(a, td, u, seed=6))
    got, ok = psf.f_a_batch(a, e, strict=False)
    assert np.array_equal(got, u) and ok.all()
