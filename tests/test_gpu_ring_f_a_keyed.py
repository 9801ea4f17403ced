"""Ring f_a with a key per target (qf_ring_set_key_table, qf_ring_f_a_keyed[_dev], DESIGN.md 4.13) and ring TrapGen for many
keys in one call (qf_ring_trap_gen_batch_from).  Every in-domain row is compared bit for bit with qf_f_a after
qf_ring_set_a(key_t) on the same context (f_a_batch with that key) and, on samples, with the oracle's f_a_ring.  The keyed
kernels read key transforms built on the device (ring_small_key_kernel, ring_prepare_kernel) while qf_ring_set_a builds the
ring_small transform on the host (qf_ring_small_key), so equal outputs on many random sigma also pin the device transform to
the host one."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _ring_s(n):
    return ((2 * 2 * 1.005 * math.sqrt(n) + 1) * 2) * 4  # gpv_ring.rs:296-298


def _psf(T, n, q):
    gp = T.GadgetParametersRing.init_default(n, q)
    return gp, T.PSFGPVRing(gp, float(_ring_s(n)), 1.005)


def _per_key(psf, keys, sig, idx):
    """u and flags from plain f_a with each row's own key installed (qf_ring_set_a + qf_f_a)"""
    u = np.empty((len(sig), psf.n), dtype=np.int64)
    ok = np.empty(len(sig), dtype=bool)
    for t in np.unique(idx):
        rows = idx == t
        u[rows], ok[rows] = psf.f_a_batch(keys[t], sig[rows], strict=False)
    return u, ok


def _check(psf, keys, sig, idx, u, ok, oracle_rows=4):
    u0, ok0 = _per_key(psf, keys, sig, idx)
    assert np.array_equal(ok, ok0)
    assert np.array_equal(u[ok], u0[ok])
    n, q = psf.n, psf.gp.q
    for b in np.flatnonzero(ok)[:oracle_rows]:
        assert u[b].tolist() == O.f_a_ring(keys[idx[b]].tolist(), sig[b].tolist(), n, q)


def _keys(rng, gp, count):
    """uniform keys, a_0 != 1 on purpose"""
    return rng.integers(0, gp.q, (count, gp.k + 2, gp.n), dtype=np.int64)


# (n, q, env): ring_small complete (7681, 12289) and incomplete (3329); Goldilocks (small NTT disabled, a q that is not an
# NTT-friendly prime); schoolbook (n not a power of two, n < 64)
FAMILIES = [
    (256, 7681, None),
    (256, 12289, None),
    (256, 3329, None),
    (128, 3329, None),
    (256, 3329, "QF_DISABLE_SMALL_NTT"),
    (128, 2**16, None),
    (64, 2**31 - 1, None),
    (32, 257, None),
    (6, 32, None),
]


@pytest.mark.parametrize("n,q,env", FAMILIES)
def test_families_bit_exact(T, monkeypatch, n, q, env):
    if env:
        monkeypatch.setenv(env, "1")
    rng = np.random.default_rng(n * 7 + q % 1000)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 236)
    sig = psf.samp_d_batch(1500, seed=3)
    idx = rng.integers(0, len(keys), len(sig)).astype(np.int32)
    u, ok = psf.f_a_keyed_batch(keys, sig, idx)
    assert ok.all()
    _check(psf, keys, sig, idx, u, ok)
    # sorted order gives the same rows
    order = np.argsort(idx, kind="stable")
    us, _ = psf.f_a_keyed_batch(keys, sig[order], idx[order])
    assert np.array_equal(us, u[order])
    # T = 1
    u1, ok1 = psf.f_a_keyed_batch(keys[:1], sig[:200], np.zeros(200, np.int32))
    assert ok1.all() and np.array_equal(u1, psf.f_a_batch(keys[0], sig[:200])[0])


def test_domain_flags(T):
    """out-of-domain rows (the edge cases of test_ring_f_a_bit_exact, gpv_ring.rs:355-445): flags as qf_f_a, in-domain rows
    exact; strict raises"""
    n, q = 256, 3329
    rng = np.random.default_rng(5)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 7)
    sig = psf.samp_d_batch(64, seed=9).astype(np.int32)
    big = round(psf.s) * (gp.k + 2) * 8 * (n // 8)
    sig[3, 0, 0] = big
    sig[10, gp.k + 1, n - 1] = -big
    sig[20] = 2**31 - 1
    sig[21] = -(2**31)
    sig[30] = 0
    idx = (np.arange(64) % 7).astype(np.int32)
    u, ok = psf.f_a_keyed_batch(keys, sig, idx, strict=False)
    want = np.ones(64, bool)
    want[[3, 10, 20, 21]] = False
    assert np.array_equal(ok, want)
    _check(psf, keys, sig, idx, u, ok)
    with pytest.raises(AssertionError):
        psf.f_a_keyed_batch(keys, sig, idx)


def test_entry_points_splits_chunks(T):
    """host and device entry points, batches split over calls, several chunk sizes; one table per context"""
    import torch
    from tools_b200 import _ffi

    n, q = 256, 3329
    rng = np.random.default_rng(11)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 236)
    sig = psf.samp_d_batch(3000, seed=4)
    idx = rng.integers(0, len(keys), len(sig)).astype(np.int32)
    u, ok = psf.f_a_keyed_batch(keys, sig, idx)
    assert ok.all()
    parts = [psf.f_a_keyed_batch(keys, sig[i:j], idx[i:j])[0] for i, j in ((0, 1), (1, 1001), (1001, 3000))]
    assert np.array_equal(np.concatenate(parts), u)
    for chunk in (1, 100, 256, 1000):
        _, small = _psf(T, n, q)
        small.ctx.call("qf_set_chunk", chunk)
        m = 300 if chunk == 1 else len(sig)
        assert np.array_equal(small.f_a_keyed_batch(keys, sig[:m], idx[:m])[0], u[:m])
    dev = torch.device("cuda:0")
    sd, idd = torch.from_numpy(sig).to(dev), torch.from_numpy(idx).to(dev)
    ud = torch.empty((len(sig), n), dtype=torch.int64, device=dev)
    fd = torch.empty(len(sig), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_ring_f_a_keyed_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), len(sig), _ffi.ptr(ud.data_ptr()),
                 _ffi.ptr(fd.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ud.cpu().numpy(), u) and fd.cpu().numpy().all()
    _check(psf, keys, sig, idx, u, ok, oracle_rows=2)


def test_table_lifetime_and_independence(T):
    """a table replaced by a second one; qf_ring_set_a and the table leave each other alone, in both directions"""
    n, q = 128, 7681
    rng = np.random.default_rng(13)
    gp, psf = _psf(T, n, q)
    k1, k2 = _keys(rng, gp, 5), _keys(rng, gp, 9)
    a = _keys(rng, gp, 1)[0]
    sig = psf.samp_d_batch(400, seed=5)
    i1 = (np.arange(400) % 5).astype(np.int32)
    i2 = (np.arange(400) % 9).astype(np.int32)
    ua, _ = psf.f_a_batch(a, sig)  # installed key first
    u1, _ = psf.f_a_keyed_batch(k1, sig, i1)
    assert np.array_equal(psf.f_a_batch(a, sig)[0], ua)  # the table install did not drop the key (no reinstall here)
    assert psf._a_id is a
    _check(psf, k1, sig, i1, u1, np.ones(400, bool), oracle_rows=0)
    u2, _ = psf.f_a_keyed_batch(k2, sig, i2)  # replaced
    _check(psf, k2, sig, i2, u2, np.ones(400, bool), oracle_rows=1)
    # qf_ring_set_a of other keys (done inside _check) keeps the table: same table object, no reinstall
    u2b, _ = psf.f_a_keyed_batch(k2, sig, i2)
    assert psf._keys_id is k2 and np.array_equal(u2b, u2)
    # a trapdoor key installed by TrapGen keeps the table as well
    a_bar = rng.integers(0, q, n, dtype=np.int64)
    r = rng.integers(-3, 4, (gp.k, n)).astype(np.int32)
    psf.gen_trapdoor_ring_lwe(a_bar, r, r)
    u2c, _ = psf.f_a_keyed_batch(k2, sig, i2)
    assert np.array_equal(u2c, u2)
    # an index of the first table that is outside the second is refused
    from tools_b200 import _ffi

    with pytest.raises(_ffi.QfError):
        psf.f_a_keyed_batch(k2, sig[:1], np.array([9], np.int32))


def test_refusals(T):
    import torch
    from tools_b200 import _ffi

    n, q = 64, 3329
    rng = np.random.default_rng(17)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 4)
    kk = np.ascontiguousarray(keys)
    sig = psf.samp_d_batch(300, seed=6)
    idx = rng.integers(0, 4, 300).astype(np.int32)
    out, fl = np.empty((300, n), np.int64), np.empty(300, np.uint8)
    call = lambda p, ix=idx, o=out: p.ctx.status("qf_ring_f_a_keyed", _ffi.ptr(sig), _ffi.ptr(ix), 300, _ffi.ptr(o), _ffi.ptr(fl))  # noqa: E731
    # no table
    assert call(psf) == _ffi.QF_ERR_NO_KEY
    # empty batch
    assert psf.ctx.status("qf_ring_f_a_keyed", None, None, 0, None, None) == _ffi.QF_OK
    # nkeys < 1, nkeys >= 2^31 - 1, NULL keys
    assert psf.ctx.status("qf_ring_set_key_table", _ffi.ptr(kk), 0) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_ring_set_key_table", _ffi.ptr(kk), 2**31 - 1) == _ffi.QF_ERR_INVALID
    assert psf.ctx.status("qf_ring_set_key_table", None, 4) == _ffi.QF_ERR_INVALID
    u, _ = psf.f_a_keyed_batch(keys, sig, idx)
    # a bad coefficient names its key and keeps the old table
    bad_keys = _keys(rng, gp, 6)
    bad_keys[4, 2, 7] = q
    msg = None
    try:
        psf.ctx.call("qf_ring_set_key_table", _ffi.ptr(np.ascontiguousarray(bad_keys)), 6)
    except _ffi.QfError as e:
        msg = str(e)
    assert msg is not None and "key 4" in msg and "QF_ERR_INVALID" in msg
    bad_keys[4, 2, 7] = 0
    bad_keys[1, 0, 0] = -1
    assert psf.ctx.status("qf_ring_set_key_table", _ffi.ptr(np.ascontiguousarray(bad_keys)), 6) == _ffi.QF_ERR_INVALID
    assert "key 1" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert call(psf) == _ffi.QF_OK and np.array_equal(out, u)
    # a bad index on the host: refused before any launch; NULL u_out
    launches = psf.ctx.launch_count()
    bad = idx.copy()
    bad[17] = 4
    assert call(psf, bad) == _ffi.QF_ERR_INVALID and psf.ctx.launch_count() == launches
    assert "target 17" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    bad[17] = -1
    assert call(psf, bad) == _ffi.QF_ERR_INVALID and psf.ctx.launch_count() == launches
    assert psf.ctx.status("qf_ring_f_a_keyed", _ffi.ptr(sig), _ffi.ptr(idx), 300, None, _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    # a bad index on the device: never used to address the table, reported at qf_synchronize, other rows exact
    dev = torch.device("cuda:0")
    bad[17], bad[200] = 4, 2**31 - 1
    sd, idd = torch.from_numpy(sig).to(dev), torch.from_numpy(bad).to(dev)
    ud = torch.empty((300, n), dtype=torch.int64, device=dev)
    fd = torch.empty(300, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    assert psf.ctx.status("qf_ring_f_a_keyed_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), 300,
                          _ffi.ptr(ud.data_ptr()), _ffi.ptr(fd.data_ptr())) == _ffi.QF_OK
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_ERR_INVALID
    assert "key index" in psf.ctx._lib.qf_last_error(psf.ctx._h).decode()
    assert psf.ctx.status("qf_synchronize") == _ffi.QF_OK  # reported once
    good = np.ones(300, bool)
    good[[17, 200]] = False
    assert np.array_equal(ud.cpu().numpy()[good], u[good])
    # _dev: NULL in_domain
    assert psf.ctx.status("qf_ring_f_a_keyed_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), 300,
                          _ffi.ptr(ud.data_ptr()), None) == _ffi.QF_ERR_INVALID
    # classical context: every new entry point refuses
    cl = T.PSFGPV(T.GadgetParameters.init_default(8, 127), 30.0)
    assert cl.ctx.status("qf_ring_set_key_table", _ffi.ptr(kk), 4) == _ffi.QF_ERR_INVALID
    assert cl.ctx.status("qf_ring_f_a_keyed", _ffi.ptr(sig), _ffi.ptr(idx), 1, _ffi.ptr(out), _ffi.ptr(fl)) == _ffi.QF_ERR_INVALID
    assert cl.ctx.status("qf_ring_f_a_keyed_dev", _ffi.ptr(sd.data_ptr()), _ffi.ptr(idd.data_ptr()), 1, _ffi.ptr(ud.data_ptr()),
                         _ffi.ptr(fd.data_ptr())) == _ffi.QF_ERR_INVALID
    ab = np.zeros((1, n), np.int64)
    rr = np.zeros((1, gp.k, n), np.int32)
    ao = np.zeros((1, gp.k + 2, n), np.int64)
    assert cl.ctx.status("qf_ring_trap_gen_batch_from", 1, _ffi.ptr(ab), _ffi.ptr(rr), _ffi.ptr(rr), _ffi.ptr(ao)) == _ffi.QF_ERR_INVALID
    # TrapGen batch: count < 1, a_bar outside [0, q)
    assert psf.ctx.status("qf_ring_trap_gen_batch_from", 0, _ffi.ptr(ab), _ffi.ptr(rr), _ffi.ptr(rr), _ffi.ptr(ao)) == _ffi.QF_ERR_INVALID
    ab[0, 3] = q
    assert psf.ctx.status("qf_ring_trap_gen_batch_from", 1, _ffi.ptr(ab), _ffi.ptr(rr), _ffi.ptr(rr), _ffi.ptr(ao)) == _ffi.QF_ERR_INVALID


@pytest.mark.parametrize("n,q,env", [(256, 3329, None), (256, 7681, None), (256, 3329, "QF_DISABLE_SMALL_NTT"), (64, 2**31 - 1, None),
                                     (6, 32, None)])
def test_trap_gen_batch(T, monkeypatch, n, q, env):
    """every key against the oracle and against qf_ring_trap_gen_from one by one; A_t [e_t; r_t; 1] = g for every key;
    the context key and the key table are untouched"""
    if env:
        monkeypatch.setenv(env, "1")
    rng = np.random.default_rng(n + q % 977)
    gp, psf = _psf(T, n, q)
    po = O.GadgetParametersRing.init_default(n, q)
    cnt = 40
    a_bars = rng.integers(0, q, (cnt, n), dtype=np.int64)
    rs = rng.integers(-6, 7, (cnt, gp.k, n)).astype(np.int32)
    es = rng.integers(-6, 7, (cnt, gp.k, n)).astype(np.int32)
    rs[0, 0, 0] = 2**20  # not small: still exact
    keys = _keys(rng, gp, 3)
    a0 = _keys(rng, gp, 1)[0]
    sig = psf.samp_d_batch(30, seed=2)
    idx = (np.arange(30) % 3).astype(np.int32)
    uk, _ = psf.f_a_keyed_batch(keys, sig, idx)
    ua, _ = psf.f_a_batch(a0, sig)
    installed = psf._a_id
    got = psf.gen_trapdoor_ring_lwe_batch(a_bars, rs, es)
    assert psf._a_id is installed
    assert np.array_equal(psf.f_a_keyed_batch(keys, sig, idx)[0], uk)
    assert np.array_equal(psf.f_a_batch(a0, sig)[0], ua)  # context key unchanged (cached: no reinstall)
    _, single = _psf(T, n, q)
    for t in range(cnt):
        if t < 3:
            want = O.gen_trapdoor_ring_lwe(po, a_bars[t].tolist(), rs[t].tolist(), es[t].tolist())
            assert got[t].tolist() == want
        assert np.array_equal(single.gen_trapdoor_ring_lwe(a_bars[t], rs[t], es[t]), got[t])
    # A_t [e_t; r_t; 1] = g: the gadget equation of gadget_ring.rs, sum_j a_{2+j} x + a_1 r_j + e_j = base^j
    for t in range(0, cnt, 7):
        for j in range(gp.k):
            lhs = O.ring_mul_np(got[t, 1].tolist(), [c % q for c in rs[t, j].tolist()], n, q)
            lhs = [(x + y + int(e)) % q for x, y, e in zip(lhs, got[t, 2 + j].tolist(), es[t, j].tolist())]
            assert lhs == [pow(gp.base, j, q)] + [0] * (n - 1)


def test_large_table_c3(T):
    """65 536 keys at C3 (0.9 GB of transforms), random and sorted indices, rows checked against per-key qf_f_a"""
    n, q = 256, 3329
    rng = np.random.default_rng(23)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, 65536)
    sig = psf.samp_d_batch(8192, seed=7)
    idx = rng.integers(0, len(keys), len(sig)).astype(np.int32)
    u, ok = psf.f_a_keyed_batch(keys, sig, idx)
    assert ok.all()
    pick = np.concatenate([np.flatnonzero(idx == idx[0]), np.flatnonzero(idx == 65535), rng.choice(len(sig), 24, replace=False)])
    for b in pick:
        assert np.array_equal(psf.f_a_batch(keys[idx[b]], sig[b:b + 1])[0][0], u[b])
    order = np.argsort(idx, kind="stable")
    us, _ = psf.f_a_keyed_batch(keys, sig[order], idx[order])
    assert np.array_equal(us, u[order])


def test_full_size_c3(T):
    """1 Mi targets over 4096 keys at C3, device-resident sigma; every row checked on the device against qf_f_a after
    qf_ring_set_a(key_t) (the dense tensor-core path of the installed key)"""
    import torch
    from tools_b200 import _ffi

    n, q, B, K = 256, 3329, 1 << 20, 4096
    rng = np.random.default_rng(29)
    gp, psf = _psf(T, n, q)
    keys = _keys(rng, gp, K)
    psf.ctx.call("qf_ring_set_key_table", _ffi.ptr(np.ascontiguousarray(keys)), K)
    dev = torch.device("cuda:0")
    d = gp.n * (gp.k + 2)
    sig = torch.empty((B, d), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_d_dev", B, 31, 0, _ffi.ptr(sig.data_ptr()))
    psf.ctx.call("qf_synchronize")
    idx_h = rng.integers(0, K, B).astype(np.int32)
    idx = torch.from_numpy(idx_h).to(dev)
    u = torch.empty((B, n), dtype=torch.int64, device=dev)
    fl = torch.empty(B, dtype=torch.uint8, device=dev)
    psf.ctx.call("qf_ring_f_a_keyed_dev", _ffi.ptr(sig.data_ptr()), _ffi.ptr(idx.data_ptr()), B, _ffi.ptr(u.data_ptr()),
                 _ffi.ptr(fl.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert bool(fl.all())
    order_h = np.argsort(idx_h, kind="stable")
    starts = np.searchsorted(idx_h[order_h], np.arange(K + 1))
    order = torch.from_numpy(order_h).to(dev)
    sig_s = sig[order].contiguous()
    del sig
    torch.cuda.synchronize()  # the library runs on its own stream
    ref = torch.empty((B, n), dtype=torch.int64, device=dev)
    fr = torch.empty(B, dtype=torch.uint8, device=dev)
    for t in range(K):
        lo, hi = int(starts[t]), int(starts[t + 1])
        if hi == lo:
            continue
        psf._install_a(keys[t])
        psf.ctx.call("qf_f_a_dev", _ffi.ptr(sig_s[lo:hi].data_ptr()), hi - lo, _ffi.ptr(ref[lo:hi].data_ptr()),
                     _ffi.ptr(fr[lo:hi].data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert bool(fr.all())
    assert bool(torch.equal(u[order], ref))
