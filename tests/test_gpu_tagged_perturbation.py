"""PSFPerturbation on tagged G-trapdoor keys A = [A_bar | H G - A_bar R] (DESIGN.md 4.4): qf_set_trapdoor_perturbation
recognises the tag, samp_p samples the gadget preimage of H^-1 (u - A p), and qf_set_tag switches the tag of an installed
key.  The oracle of every sampling test is the reduced identity key A' = [A_bar' | G - A_bar' R] with A_bar = H A_bar':
A = H A', and with targets u = H u' the tagged key must give preimages bit-identical to A' with targets u' (the identity
path is law-tested against the reference loop in test_gpu_stat_parity.py).  The keys are built with forward products
only.  The reduction itself is pinned on the CPU in test_tagged_perturbation_math.py."""
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
    """x y mod q, exact: 16-bit halves in float64 BLAS for q < 2^32 (partial sums < 2^32 K < 2^53), object integers above."""
    x, y = np.asarray(x, dtype=np.int64), np.asarray(y, dtype=np.int64)
    if q >= 2**32:
        return np.array(x.astype(object).dot(y.astype(object)) % q, dtype=np.int64)
    assert x.shape[1] < 2**20
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


def _tag(kind, n, q, rng):
    return _dense_tag(n, q, rng) if kind == "dense" else _unitriangular_tag(n, q, rng)


def _gadget_basis(gp):
    from tools_b200 import gadget

    blk = gadget.short_basis_gadget_block(gp.k, gp.base, gp.q)
    gblk = gadget.gso_small(blk)
    if gp.n * gp.k <= 1024:
        return gadget.short_basis_gadget(gp), np.kron(np.eye(gp.n), gblk)
    return blk, gblk


def _keys(T, gp, r, s, seed, tag, dense=True):
    """The reduced identity key A' = [A_bar' | G - A_bar' R] from the device sampler, the tagged key
    A = qf_trap_gen_from(H A_bar' mod q, R, H) = H A' and the trapdoor (R, sqrt(Sigma_2) or None, gadget basis)."""
    g = T.PSFGPV(gp, 10.0 * gp.n)
    a_red, rm = T.psf._trap_gen_classical(g, seed)
    g.ctx.close()
    a = T.psf.gen_trapdoor(gp, _matmul_mod(tag, a_red[:, : gp.m_bar], gp.q), rm, tag)
    l = None
    if dense:
        p = T.PSFPerturbation(gp, r, s)
        l = p.compute_sqrt_sigma_2(rm)
        p.ctx.close()
    return a, a_red, (rm, l, _gadget_basis(gp))


def _outcome(T, gp, r, s, a, td, u, seed, first_index=0):
    """Preimages of u on a fresh context, or the status the install / sampling failed with."""
    psf = T.PSFPerturbation(gp, r, s)
    try:
        return psf.samp_p_batch(a, td, u, seed=seed, first_index=first_index), None
    except T.QfError as err:
        return None, err.status
    finally:
        psf.ctx.close()


def _midsize():
    n, q = 40, 2**12
    from tools_b200 import gadget

    gp = gadget.GadgetParameters.init_default(n, q)
    s = 1.3 * np.sqrt(5 * ((np.sqrt(gp.m_bar) + np.sqrt(n * gp.k)) ** 2 / 2 + 1) + 1)
    return n, q, float(np.log2(n)), float(s)


PREIMAGE_SHAPES = [(8, 64, 3.0, 25.0), (5, 256, float(np.log2(5)), 25.0), (6, 128, float(np.log2(6)), 25.0),
                   (8, 127, 3.0, 30.0), (16, 2**20 - 3, 4.0, 80.0)]
CASES = ([shape + (kind, True) for shape in PREIMAGE_SHAPES for kind in ("dense", "unitriangular")]
         + [(8, 64, 3.0, 25.0, "dense", False), _midsize() + ("unitriangular", False), _midsize() + ("dense", False)])


@pytest.mark.parametrize("n,q,r,s,kind,dense", CASES)
def test_tagged_matches_reduced_identity_key(T, n, q, r, s, kind, dense):
    """Shapes of test_samp_p_perturbation_preimage_and_domain (dense sqrt(Sigma_2)) and of the structured square root
    (test_samp_p_perturbation_structured_midsize), dense and unitriangular tags."""
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 31 + q % 997)
    tag = _tag(kind, n, q, rng)
    a, a_red, td = _keys(T, gp, r, s, n + 7, tag, dense)
    u_red = rng.integers(0, q, (2000, n), dtype=np.int64)
    u = _matmul_mod(u_red, tag.T, q)
    psf = T.PSFPerturbation(gp, r, s)
    e = psf.samp_p_batch(a, td, u, seed=11, first_index=3)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    assert psf.check_domain_batch(e).all()
    ref = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(ref.samp_p_batch(a_red, td, u_red, seed=11, first_index=3), e)


def test_tagged_entry_points_splits_and_key_changes(T):
    import torch
    from tools_b200 import _ffi

    n, q, r, s = 16, 2**20 - 3, 4.0, 80.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(21)
    tag = _unitriangular_tag(n, q, rng)
    a, a_red, td = _keys(T, gp, r, s, 5, tag)
    u = rng.integers(0, q, (1500, n), dtype=np.int64)
    psf = T.PSFPerturbation(gp, r, s)
    e = psf.samp_p_batch(a, td, u, seed=9)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    ref = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(ref.samp_p_batch(a_red, td, _matmul_mod(u, _inv_unitriangular(tag, q).T, q), seed=9), e)
    # a batch split across calls, and small internal chunks
    parts = np.concatenate([psf.samp_p_batch(a, td, u[:700], seed=9, first_index=0),
                            psf.samp_p_batch(a, td, u[700:], seed=9, first_index=700)])
    assert np.array_equal(parts, e)
    small = T.PSFPerturbation(gp, r, s)
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
    # tagged -> identity -> tagged on one context: what fresh contexts give
    e_id = psf.samp_p_batch(a_red, td, u, seed=10)
    fresh = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(fresh.samp_p_batch(a_red, td, u, seed=10), e_id)
    assert np.array_equal(O.f_a_classical_batch(a_red, e_id, q), u)
    assert np.array_equal(psf.samp_p_batch(a, td, u, seed=9), e)


def test_tagged_fp64_branch(T, monkeypatch):
    """QF_DISABLE_I8=1: u - A p on the fp64 path (and f_a on the fp64 digit matrices of A, which qf_set_tag updates)."""
    monkeypatch.setenv("QF_DISABLE_I8", "1")
    n, q, r, s = 8, 127, 3.0, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(4)
    tag = _dense_tag(n, q, rng)
    a, a_red, td = _keys(T, gp, r, s, 6, tag)
    u_red = rng.integers(0, q, (900, n), dtype=np.int64)
    u = _matmul_mod(u_red, tag.T, q)
    psf = T.PSFPerturbation(gp, r, s)
    e = psf.samp_p_batch(a, td, u, seed=2)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    ref = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(ref.samp_p_batch(a_red, td, u_red, seed=2), e)
    # tag switch on this branch: the fp64 digit matrices of A follow
    tag2 = _unitriangular_tag(n, q, rng)
    a2 = psf.set_tag(a, td, tag2)
    assert np.array_equal(a2, T.psf.gen_trapdoor(gp, a[:, : gp.m_bar], td[0], tag2))
    e2 = psf.samp_p_batch(a2, td, u, seed=3)
    assert np.array_equal(psf.f_a_batch(a2, e2)[0], u)
    assert np.array_equal(T.PSFPerturbation(gp, r, s).samp_p_batch(a2, td, u, seed=3), e2)


def _inv_unitriangular(h, q):
    """H^-1 mod q of an upper unitriangular H by back substitution (object integers)."""
    n = h.shape[0]
    x = np.zeros((n, n), dtype=object)
    ho = h.astype(object)
    for i in range(n - 1, -1, -1):
        row = -(ho[i, i + 1:].dot(x[i + 1:])) if i + 1 < n else np.zeros(n, dtype=object)
        row[i] += 1
        x[i] = row % q
    return np.array(x, dtype=np.int64)


@pytest.mark.parametrize("n,q", [(4, 2**48), (3, 2**61 - 1)])
def test_tagged_large_modulus(T, n, q):
    """Residues of 7 and 8 balanced digits: v' = H^-1 v runs in two digit groups.  Where the context rejects the modulus,
    the tagged key fails with the status the reduced key fails with."""
    gp = T.GadgetParameters.init_default(n, q)
    r = 3.0
    s = float(math.ceil(1.3 * math.sqrt(5 * ((math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) ** 2 / 2 + 1) + 1)))
    rng = np.random.default_rng(q % 1000)
    for tag in (_dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)):
        a, a_red, td = _keys(T, gp, r, s, n + 2, tag)
        u_red = rng.integers(0, q, (300, n), dtype=np.int64)
        u = _matmul_mod(u_red, tag.T, q)
        e, st = _outcome(T, gp, r, s, a, td, u, 7)
        e_red, st_red = _outcome(T, gp, r, s, a_red, td, u_red, 7)
        assert st == st_red, (st, st_red)
        if e is not None:
            assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
            assert np.array_equal(e, e_red)


def test_tag_without_unit_pivot_is_rejected(T):
    """H invertible mod 4095 but without a unit in its first column, and a singular H: both keys have the form
    [A_bar | H G - A_bar R], unit pivoting rejects H, so the trapdoor install fails with QF_ERR_INVALID (as
    qf_gen_short_basis_tagged does).  The context stays usable."""
    from tools_b200 import _ffi

    n, q, r, s = 8, 4095, 3.0, 45.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(40)
    d = np.eye(n, dtype=np.int64)
    d[:2, :2] = [[3, 5], [5, 3]]  # det = -16, a unit mod 4095; 3 and 5 are not
    no_pivot = d @ _unitriangular_tag(n, q, rng) % q
    singular = _unitriangular_tag(n, q, rng)
    singular[:, 0] = 0
    psf = T.PSFPerturbation(gp, r, s)
    u = rng.integers(0, q, (500, n), dtype=np.int64)
    for bad in (no_pivot, singular):
        a, _, td = _keys(T, gp, r, s, 3, bad)
        with pytest.raises(T.QfError) as ei:
            psf.samp_p_batch(a, td, u, seed=1)
        assert ei.value.status == _ffi.QF_ERR_INVALID
    tag = _dense_tag(n, q, rng)
    a, a_red, td = _keys(T, gp, r, s, 4, tag)
    e = psf.samp_p_batch(a, td, u, seed=1)
    assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
    assert np.array_equal(e, T.PSFPerturbation(gp, r, s).samp_p_batch(a, td, u, seed=1))


def test_unrelated_key_installs_as_before(T):
    """A random key, not of the form [A_bar | H G - A_bar R] for the trapdoor's R, installs and samples as before
    (deterministic, in the domain; A e = u does not hold for such a key), and qf_set_tag refuses it."""
    from tools_b200 import _ffi

    n, q, r, s = 8, 127, 3.0, 30.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(8)
    _, _, td = _keys(T, gp, r, s, 9, np.eye(n, dtype=np.int64))
    a = rng.integers(0, q, (n, gp.m), dtype=np.int64)
    u = rng.integers(0, q, (400, n), dtype=np.int64)
    psf = T.PSFPerturbation(gp, r, s)
    e = psf.samp_p_batch(a, td, u, seed=4)
    assert psf.check_domain_batch(e).all()
    assert np.array_equal(T.PSFPerturbation(gp, r, s).samp_p_batch(a, td, u, seed=4), e)
    assert psf.ctx.status("qf_set_tag", None, None) == _ffi.QF_ERR_INVALID
    assert np.array_equal(psf.samp_p_batch(a, td, u, seed=4), e)


def test_set_tag(T):
    from tools_b200 import _ffi

    n, q, r, s = 16, 2**20 - 3, 4.0, 80.0
    gp = T.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(13)
    psf = T.PSFPerturbation(gp, r, s)
    a_id, td = psf.trap_gen(seed=3)
    a_bar, rm = a_id[:, : gp.m_bar], td[0]
    u = rng.integers(0, q, (1200, n), dtype=np.int64)
    sig = psf.samp_d_batch(300, seed=5)

    def same_as_fresh(a, seed):
        e = psf.samp_p_batch(a, td, u, seed=seed)
        assert np.array_equal(O.f_a_classical_batch(a, e, q), u)
        assert np.array_equal(e, T.PSFPerturbation(gp, r, s).samp_p_batch(a, td, u, seed=seed))
        # f_a on the switched key (no re-install: the context's own copies of A)
        got, ok = psf.f_a_batch(a, sig)
        assert ok.all() and np.array_equal(got, O.f_a_classical_batch(a, sig, q))
        return e

    h1, h2 = _dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)
    a1 = psf.set_tag(a_id, td, h1)
    assert np.array_equal(a1, T.psf.gen_trapdoor(gp, a_bar, rm, h1))
    same_as_fresh(a1, 6)
    a2 = psf.set_tag(a1, td, h2 + q)  # entries taken mod q
    assert np.array_equal(a2, T.psf.gen_trapdoor(gp, a_bar, rm, h2))
    e2 = same_as_fresh(a2, 7)
    # a tag without a unit pivot: refused, nothing changes
    bad = _unitriangular_tag(n, q, rng)
    bad[:, 1] = 0
    with pytest.raises(T.QfError) as ei:
        psf.set_tag(a2, td, bad)
    assert ei.value.status == _ffi.QF_ERR_INVALID
    assert psf._a_id is a2
    assert np.array_equal(psf.samp_p_batch(a2, td, u, seed=7), e2)
    assert np.array_equal(psf.f_a_batch(a2, sig)[0], O.f_a_classical_batch(a2, sig, q))
    a3 = psf.set_tag(a2, td, None)
    assert np.array_equal(a3, a_id)
    same_as_fresh(a3, 8)
    # trap_gen with a tag gives the same key as the switch
    tg = T.PSFPerturbation(gp, r, s)
    a4, td4 = tg.trap_gen(seed=3, tag=h1)
    assert np.array_equal(a4, a1)
    e4 = tg.samp_p_batch(a4, td4, u, seed=6)
    assert np.array_equal(O.f_a_classical_batch(a4, e4, q), u)
    # ... and so does qf_trap_gen_from itself for a tag with negative entries (h1 - q), which it takes mod q
    # (the arrays are named: _ffi.ptr does not keep its argument alive through the call)
    ab, r8, neg = np.ascontiguousarray(a_bar), np.ascontiguousarray(rm, dtype=np.int8), np.ascontiguousarray(h1 - q)
    assert neg.min() < 0
    a5 = np.empty_like(a1)
    tg.ctx.call("qf_trap_gen_from", _ffi.ptr(ab), _ffi.ptr(r8), _ffi.ptr(neg), _ffi.ptr(a5))
    assert np.array_equal(a5, a1)
    # refusals: a GPV context, no trapdoor, no key
    g = T.PSFGPV(gp, 90.0)
    assert g.ctx.status("qf_set_tag", None, None) == _ffi.QF_ERR_INVALID
    bare = T.PSFPerturbation(gp, r, s)
    assert bare.ctx.status("qf_set_tag", None, None) == _ffi.QF_ERR_NO_KEY
    bare._install_a(a_id)
    assert bare.ctx.status("qf_set_tag", None, None) == _ffi.QF_ERR_NO_KEY


def test_full_size_c4_shard_tagged(T):
    """BASELINE.json configs[3] at full key size (n = 512, q = 2^32 - 5, k = 32, m = 32849, r = 9, structured
    sqrt(Sigma_2)) with a random unitriangular tag: A e = u for 2048 targets (exact, 16-bit splits), check_domain, the
    second moment, and the first 256 preimages bit-identical to the reduced identity key."""
    n, q, r = 512, 2**32 - 5, 9.0
    gp = T.GadgetParameters.init_default(n, q)
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
    s = float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))
    rng = np.random.default_rng(6)
    tag = _unitriangular_tag(n, q, rng)
    a, a_red, td = _keys(T, gp, r, s, 4, tag, dense=False)
    u_red = rng.integers(0, q, (2048, n), dtype=np.int64)
    u = _matmul_mod(u_red, tag.T, q)
    psf = T.PSFPerturbation(gp, r, s)
    e = psf.samp_p_batch(a, td, u, seed=9)
    assert np.array_equal(_f_a(a, e, q), u)
    assert [int(x) for x in (e[:2].astype(object) @ a.T.astype(object) % q).ravel()] == u[:2].ravel().tolist()
    assert psf.check_domain_batch(e).all()
    ratio = (e.astype(np.float64) ** 2).sum(1).mean() / (gp.m * (s * r) ** 2 / (2 * math.pi))
    assert abs(ratio - 1) < 0.01, ratio
    psf.ctx.close()
    ref = T.PSFPerturbation(gp, r, s)
    assert np.array_equal(ref.samp_p_batch(a_red, td, u_red[:256], seed=9), e[:256])
