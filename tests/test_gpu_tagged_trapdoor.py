"""Tagged G-trapdoor keys A = [A_bar | H G - A_bar R] on the device (DESIGN.md 4.3, 4.8): the short basis for a tag
(qf_gen_short_basis_tagged, H^-1 by Gauss-Jordan on the GPU) against the oracle, and samp_p on such keys, which runs
the two-phase recursion on H^-1 A with targets H^-1 u.  The reduction itself is pinned on the CPU in
test_tagged_trapdoor_math.py."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


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


def _inv_unitriangular(h, q):
    """H^-1 mod q of an upper unitriangular H by back substitution (int64: needs n q^2 < 2^63)."""
    n = h.shape[0]
    assert n * q * q < 2**62
    x = np.zeros((n, n), dtype=np.int64)
    for i in range(n - 1, -1, -1):
        row = -(h[i, i + 1:] @ x[i + 1:]) if i + 1 < n else np.zeros(n, dtype=np.int64)
        row[i] += 1
        x[i] = row % q
    return x


def _gpv_s(gp):
    return float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(gp.n)))


def _tagged_key(T, gp, seed, tag):
    """(A_bar, R) from the device sampler and the tagged key A = [A_bar | H G - A_bar R]."""
    psf = T.PSFGPV(gp, 10.0 * gp.n)
    a0, r = T.psf._trap_gen_classical(psf, seed=seed)
    a = T.psf.gen_trapdoor(gp, a0[:, : gp.m_bar], r, tag)
    return psf, a, r


@pytest.mark.parametrize("n,q", [(8, 127), (16, 256), (12, 3329), (24, 2**16), (8, 2**31 - 1), (6, 2**40 + 15)])
def test_tagged_short_basis_matches_oracle(T, n, q):
    gp = T.GadgetParameters.init_default(n, q)
    po = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 7 + q % 1009)
    for tag in (_dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)):
        psf, a, r = _tagged_key(T, gp, n + 3, tag)
        psf._install_a(a)
        got = psf.gen_short_basis_for_trapdoor(r, tag)
        want = O.gen_short_basis_for_trapdoor(po, tag.tolist(), a.tolist(), r.tolist())
        assert got.tolist() == [list(map(int, row)) for row in want]
        assert not (a.astype(object).dot(got.astype(object)) % q).any()  # every column lies in Lambda^perp(A)


def test_tagged_short_basis_matches_host_at_n64(T):
    from tools_b200 import gadget

    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    tag = _dense_tag(n, q, np.random.default_rng(5))
    psf, a, r = _tagged_key(T, gp, 17, tag)
    psf._install_a(a)
    got = psf.gen_short_basis_for_trapdoor(r, tag)
    assert np.array_equal(got, gadget.gen_short_basis_for_trapdoor(gp, a, r, tag.astype(object)))
    assert not (a.astype(object).dot(got.astype(object)) % q).any()


@pytest.mark.parametrize("n,q", [(8, 127), (64, 2**16), (40, 2**20 - 3)])
def test_identity_tag_is_unchanged(T, n, q):
    from tools_b200 import _ffi

    gp = T.GadgetParameters.init_default(n, q)
    psf = T.PSFGPV(gp, 10.0 * n)
    a, r = T.psf._trap_gen_classical(psf, seed=n)
    plain = np.empty((gp.m, gp.m), dtype=np.int64)
    psf.ctx.call("qf_gen_short_basis", _ffi.ptr(r), _ffi.ptr(plain))
    null_tag = np.empty_like(plain)
    psf.ctx.call("qf_gen_short_basis_tagged", _ffi.ptr(r), None, _ffi.ptr(null_tag))
    eye = psf.gen_short_basis_for_trapdoor(r, np.eye(n, dtype=np.int64))
    assert np.array_equal(plain, null_tag) and np.array_equal(plain, eye)
    assert np.array_equal(plain, psf.gen_short_basis_for_trapdoor(r))


def test_non_invertible_tag_is_rejected(T):
    from tools_b200 import _ffi

    n, q = 8, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(3)
    bad = rng.integers(0, q, (n, n), dtype=np.int64)
    bad[:, 0] = 2 * rng.integers(0, q // 2, n)  # no unit in the first column
    psf = T.PSFGPV(gp, 60.0)
    a, r = T.psf._trap_gen_classical(psf, seed=4)
    with pytest.raises(T.QfError) as ei:
        psf.gen_short_basis_for_trapdoor(r, bad)
    assert ei.value.status == _ffi.QF_ERR_INVALID
    # the context stays usable: a valid tag on the same context still matches the oracle
    tag = _unitriangular_tag(n, q, rng)
    a2 = T.psf.gen_trapdoor(gp, a[:, : gp.m_bar], r, tag)
    psf._install_a(a2)
    got = psf.gen_short_basis_for_trapdoor(r, tag)
    want = O.gen_short_basis_for_trapdoor(O.GadgetParameters.init_default(n, q), tag.tolist(), a2.tolist(), r.tolist())
    assert got.tolist() == [list(map(int, row)) for row in want]


@pytest.mark.parametrize("n,q", [(64, 2**16), (128, 2**12), (64, 4093)])
def test_tagged_samp_p_takes_the_two_phase_path(T, monkeypatch, n, q):
    """Shapes of test_gpv_tensor_core_updates_match_fp64_path.  The tagged key's preimages are bit-identical to those of
    the identity key H^-1 A with targets H^-1 u (the already-tested identity two-phase path) and differ from the
    one-pass recursion's, which shows the fast path ran."""
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    gp = T.GadgetParameters.init_default(n, q)
    s = float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n)))
    rng = np.random.default_rng(12)
    tag = _unitriangular_tag(n, q, rng)
    psf = T.PSFGPV(gp, s)
    a, td = psf.trap_gen(seed=31, tag=tag)
    hinv = _inv_unitriangular(tag, q)
    assert np.array_equal((hinv @ tag) % q, np.eye(n, dtype=np.int64))
    u = rng.integers(0, q, (2027, n), dtype=np.int64)
    e = psf.samp_p_batch(a, td, u, seed=77, first_index=5)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    assert psf.check_domain_batch(e).all()
    ratio = (e.astype(np.float64) ** 2).sum(1).mean() / (gp.m * s * s / (2 * math.pi))
    assert abs(ratio - 1) < 0.02, ratio
    # the equivalent identity key on a fresh context
    a_id = (hinv @ a) % q
    u_id = (u @ hinv.T) % q
    ref = T.PSFGPV(gp, s)
    e_id = ref.samp_p_batch(a_id, td, u_id, seed=77, first_index=5)
    assert np.array_equal(e, e_id)
    # the one-pass recursion (what tagged keys took before): exact too, but other draws
    monkeypatch.setenv("QF_DISABLE_TWO_PHASE", "1")
    one = T.PSFGPV(gp, s)
    e1 = one.samp_p_batch(a, td, u, seed=77, first_index=5)
    assert np.array_equal(O.f_a_classical_batch(a, e1, q), u)
    assert not np.array_equal(e, e1)


def test_tagged_samp_p_splits_entry_points_and_key_changes(T, monkeypatch):
    import torch
    from tools_b200 import _ffi

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 2**16
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(21)
    tag = _unitriangular_tag(n, q, rng)
    psf = T.PSFGPV(gp, s)
    a, td = psf.trap_gen(seed=5, tag=tag)
    u = rng.integers(0, q, (1500, n), dtype=np.int64)
    e = psf.samp_p_batch(a, td, u, seed=9)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    # split across calls, and small internal chunks
    parts = np.concatenate([psf.samp_p_batch(a, td, u[:700], seed=9, first_index=0),
                            psf.samp_p_batch(a, td, u[700:], seed=9, first_index=700)])
    assert np.array_equal(parts, e)
    small = T.PSFGPV(gp, s)
    small.ctx.call("qf_set_chunk", 256)
    assert np.array_equal(small.samp_p_batch(a, td, u, seed=9), e)
    # int16 and device-resident entry points
    assert np.array_equal(psf.samp_p_batch(a, td, u, seed=9, dtype=np.int16), e.astype(np.int16))
    dev = torch.device("cuda:0")
    ud = torch.from_numpy(u).to(dev)
    ed = torch.empty((u.shape[0], gp.m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_p_dev", _ffi.ptr(ud.data_ptr()), u.shape[0], 9, 0, _ffi.ptr(ed.data_ptr()))
    psf.ctx.call("qf_synchronize")
    assert np.array_equal(ed.cpu().numpy(), e)
    # an identity key installed after the tagged one gives what a fresh context gives
    a2, td2 = psf.trap_gen(seed=6)
    e2 = psf.samp_p_batch(a2, td2, u, seed=10)
    fresh = T.PSFGPV(gp, s)
    assert np.array_equal(fresh.samp_p_batch(a2, td2, u, seed=10), e2)
    # and the tagged key again
    assert np.array_equal(psf.samp_p_batch(a, td, u, seed=9), e)


def test_tagged_samp_p_full_size_c2(T, monkeypatch):
    """C2 (n = 256, q = 2^24, m = 12352) with a random unitriangular tag: key setup on the device, A e = u and
    check_domain over 37 888 targets, the first 2048 bit-identical to the equivalent identity key and different from the
    one-pass recursion's (so the two-phase path ran)."""
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 256, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(2)
    tag = _unitriangular_tag(n, q, rng)
    psf = T.PSFGPV(gp, s)
    a, td = psf.trap_gen(seed=2, tag=tag, dense_gso=False)
    u = rng.integers(0, q, (37888, n), dtype=np.int64)
    e = psf.samp_p_batch(a, td, u, seed=3)
    got, ok = psf.f_a_batch(a, e, strict=False)
    assert np.array_equal(got, u) and ok.all()
    assert np.array_equal(O.f_a_classical_batch(a, e[:4], q), u[:4])
    hinv = _inv_unitriangular(tag, q)
    ref = T.PSFGPV(gp, s)
    a_id = (hinv @ a) % q
    e_id = ref.samp_p_batch(a_id, td, (u[:2048] @ hinv.T) % q, seed=3)
    assert np.array_equal(e[:2048], e_id)
    ref.ctx.close()
    monkeypatch.setenv("QF_DISABLE_TWO_PHASE", "1")
    one = T.PSFGPV(gp, s)
    e1 = one.samp_p_batch(a, td, u[:2048], seed=3)
    assert np.array_equal(one.f_a_batch(a, e1)[0], u[:2048])
    assert not np.array_equal(e[:2048], e1)


def _outcome(T, gp, s, a, td, u, seed):
    """Preimages of u on a fresh context, or the status the install / sampling failed with."""
    psf = T.PSFGPV(gp, s)
    try:
        return psf.samp_p_batch(a, td, u, seed=seed), None
    except T.QfError as err:
        return None, err.status
    finally:
        psf.ctx.close()


@pytest.mark.parametrize("n,q", [(6, 2**48), (5, 2**61 - 1)])
def test_tagged_short_basis_large_modulus(T, n, q):
    """Residues of 7 and 8 balanced digits: the products with H^-1 run in two digit groups (modq_contract)."""
    gp = T.GadgetParameters.init_default(n, q)
    po = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n)
    for tag in (_dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)):
        psf, a, r = _tagged_key(T, gp, n + 11, tag)
        psf._install_a(a)
        got = psf.gen_short_basis_for_trapdoor(r, tag)
        want = O.gen_short_basis_for_trapdoor(po, tag.tolist(), a.tolist(), r.tolist())
        assert got.tolist() == [list(map(int, row)) for row in want]


@pytest.mark.parametrize("n,q,base", [(16, 2**48, 2), (40, 2**61 - 1, 16)])
def test_tagged_key_install_large_modulus(T, monkeypatch, n, q, base):
    """qf_set_trapdoor_gpv on a tagged key at tensor-core dimensions (tag detection runs) with residues of 7 and 8 digits:
    the tagged key behaves exactly like the identity key H^-1 A with targets H^-1 u -- the same preimages, or the same
    status if that key cannot be sampled at this modulus."""
    from tools_b200 import gadget

    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    k = gadget._ceil_log(q, base)
    gp = T.GadgetParameters(n=n, k=k, m_bar=n * k + gadget._ceil_log(n, 2) ** 2, base=base, q=q)
    assert (n * k) % 128 == 0 and gp.m > 1024
    rng = np.random.default_rng(q % 1000)
    tag = _dense_tag(n, q, rng)
    hinv = np.array(O.mat_inverse_mod(tag.tolist(), q), dtype=object)
    psf, a, r = _tagged_key(T, gp, 5, tag)
    psf._install_a(a)
    sb = psf.gen_short_basis_for_trapdoor(r, tag)
    assert np.array_equal(sb, gadget.gen_short_basis_for_trapdoor(gp, a, r, tag.astype(object)))
    psf.ctx.close()
    s = _gpv_s(gp)
    u = rng.integers(0, q, (300, n), dtype=np.int64)
    a_id = np.array(hinv.dot(a.astype(object)) % q, dtype=np.int64)
    u_id = np.array(u.astype(object).dot(hinv.T) % q, dtype=np.int64)
    e, st = _outcome(T, gp, s, a, (sb, None), u, 7)
    e_id, st_id = _outcome(T, gp, s, a_id, (sb, None), u_id, 7)
    assert st == st_id, (st, st_id)
    if e is not None:
        assert np.array_equal(np.array(e.astype(object).dot(a.T.astype(object)) % q, dtype=np.int64), u)
        assert np.array_equal(e, e_id)


def test_tag_without_unit_pivot_falls_back_to_one_pass(T, monkeypatch):
    """H invertible mod q = 4095 but with no unit in its first column: unit pivoting rejects it, so tag detection leaves
    the key (with its valid basis, built as the identity basis of H^-1 A) on the one-pass recursion -- the preimages are
    exact and equal to those of QF_DISABLE_TWO_PHASE=1."""
    monkeypatch.setenv("QF_OZAKI_MIN_DIM", "1024")
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    n, q = 64, 4095
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(40)
    d = np.eye(n, dtype=np.int64)
    d[:2, :2] = [[3, 5], [5, 3]]                       # det = -16, a unit mod 4095; 3 and 5 are not
    d_inv = np.eye(n, dtype=np.int64)
    di = pow(-16 % q, -1, q)
    d_inv[:2, :2] = np.array([[3, -5], [-5, 3]]) * di % q
    uu = _unitriangular_tag(n, q, rng)
    tag = d @ uu % q
    hinv = _inv_unitriangular(uu, q) @ d_inv % q
    assert np.array_equal(hinv @ tag % q, np.eye(n, dtype=np.int64))
    with pytest.raises(ValueError):
        O.mat_inverse_mod(tag.tolist(), q)
    psf, a, r = _tagged_key(T, gp, 8, tag)
    a_red = hinv @ a % q
    psf._install_a(a_red)
    sb = psf.gen_short_basis_for_trapdoor(r)
    assert not (a.astype(object).dot(sb.astype(object)) % q).any()  # a basis of Lambda^perp(A)
    u = rng.integers(0, q, (700, n), dtype=np.int64)
    e, st = _outcome(T, gp, s, a, (sb, None), u, 3)
    assert st is None
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    monkeypatch.setenv("QF_DISABLE_TWO_PHASE", "1")
    e1, _ = _outcome(T, gp, s, a, (sb, None), u, 3)
    assert np.array_equal(e, e1)
