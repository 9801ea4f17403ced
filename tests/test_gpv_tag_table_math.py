"""CPU checks (numpy + the oracle) of the identity behind PSFGPV's tag per target (DESIGN.md 4.3, tools_b200/csrc/api.cu
samp_p_np2_chunk with tag indices, qf_gpv_set_tag).  For one (A_bar, R) the basis of tag H is
S_H = [[R S', I + R W_H],[S', W_H]]: its first nk columns [R; I] S' do not depend on H, and Gram-Schmidt removes the
[R; I] W_H part of every later column, so the GSO -- and U_11, U_22, Mt_1, M' -- is the same for every tag; only U_12,
which the two-phase form never reads, changes.  Under common random numbers (test_two_phase_math.py) the two-phase form
with the material of the installed S_H0 and h_t = H_t^-1 (u - A_bar z2) mod q then returns the preimage the reference
loop returns on (A_t, S_t)."""
import numpy as np
import pytest

from oracle import qfall_oracle as O
from test_two_phase_math import _digits, _gso, _sprime


def _dense_tag(n, q, rng):
    while True:
        h = rng.integers(0, q, (n, n))
        try:
            O.mat_inverse_mod(h.tolist(), q)
            return h.astype(np.int64)
        except ValueError:
            continue


def _unitriangular_tag(n, q, rng):
    return np.triu(rng.integers(0, q, (n, n)), 1).astype(np.int64) + np.eye(n, dtype=np.int64)


def _reference(a, s, u_mat, mt, u, alpha, q):
    """gpv.rs:152-161 under common random numbers: centre -sol, all m coordinates."""
    m = len(alpha)
    sol = np.array(O.solve_unit_pivots(a.tolist(), u.tolist(), q), dtype=np.int64)
    c = -(mt @ sol)
    z = np.zeros(m)
    for i in range(m - 1, -1, -1):
        z[i] = np.floor(c[i] + alpha[i])
        c[:i] -= u_mat[:i, i] * z[i]
    return sol + s @ z.astype(np.int64)


def _two_phase(p, a_bar, r, u_mat, mt, hinv, u, alpha):
    """The device's two-phase form with the GSO material (u_mat, mt) of the installed basis and the target's tag H_t."""
    nk, mb, k, q = p.n * p.k, p.m_bar, p.k, p.q
    z2 = np.zeros(mb)
    c2 = np.zeros(mb)
    for i in range(mb - 1, -1, -1):
        z2[i] = np.floor(c2[i] + alpha[nk + i])
        c2[:i] -= u_mat[nk:nk + i, nk + i] * z2[i]
    z2 = z2.astype(np.int64)
    h = (hinv @ ((u - a_bar @ z2) % q)) % q
    g3 = _digits(h, k, p.base)
    mprime = mt[:nk, :mb] @ r + mt[:nk, mb:]
    t1 = -(mprime @ g3) - mt[:nk, :mb] @ z2
    u11 = np.triu(u_mat[:nk, :nk])
    z1 = np.zeros(nk)
    for i in range(nk - 1, -1, -1):
        z1[i] = np.floor(t1[i] + alpha[i])
        t1[:i] -= u11[:i, i] * z1[i]
    e_bot = g3 + _sprime(p) @ z1.astype(np.int64)
    return np.concatenate([z2 + r @ e_bot, e_bot])


@pytest.mark.parametrize("installed", ["identity", "dense"])
@pytest.mark.parametrize("n,q", [(3, 2**6), (4, 2**5), (3, 53), (5, 97)])
def test_gpv_tag_switch_keeps_the_gso_and_the_two_phase_preimage(n, q, installed):
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 1000 + q + (7 if installed == "dense" else 0))
    nk, mb, m = p.n * p.k, p.m_bar, p.m
    a_bar = rng.integers(0, q, (n, mb))
    r_list = O.sample_pm_one_zero(rng, mb, nk)
    r = np.array(r_list, dtype=np.int64)

    def key(tag):
        a = O.gen_trapdoor(p, a_bar.tolist(), tag.tolist(), r_list)
        s = O.gen_short_basis_for_trapdoor(p, tag.tolist(), a, r_list)
        return np.array(a, dtype=np.int64), s

    h0 = np.eye(n, dtype=np.int64) if installed == "identity" else _dense_tag(n, q, rng)
    a0, s0_list = key(h0)
    s0 = np.array(s0_list, dtype=np.int64)
    g0 = O.gso_exact(s0_list)
    u0, mt0 = _gso(s0)
    tags = [np.eye(n, dtype=np.int64), _dense_tag(n, q, rng), _unitriangular_tag(n, q, rng)]
    for tag in tags:
        a_t, s_t_list = key(tag)
        s_t = np.array(s_t_list, dtype=np.int64)
        assert not ((a_t @ s_t) % q).any()
        assert O.gso_exact(s_t_list) == g0
        u_t, mt_t = _gso(s_t)
        assert np.allclose(u_t[:nk, :nk], u0[:nk, :nk], atol=1e-9)     # U_11
        assert np.allclose(u_t[nk:, nk:], u0[nk:, nk:], atol=1e-9)     # U_22
        assert np.allclose(mt_t[:nk, :mb], mt0[:nk, :mb], atol=1e-9)   # Mt_1
        mp_t = mt_t[:nk, :mb] @ r + mt_t[:nk, mb:]
        mp_0 = mt0[:nk, :mb] @ r + mt0[:nk, mb:]
        assert np.allclose(mp_t, mp_0, atol=1e-9)                      # M'
        if not np.array_equal(tag % q, h0 % q):
            assert np.abs(u_t[:nk, nk:] - u0[:nk, nk:]).max() > 1e-3   # U_12 depends on the tag
        hinv = np.array(O.mat_inverse_mod((tag % q).tolist(), q), dtype=np.int64)
        for _ in range(4):
            u = rng.integers(0, q, n)
            alpha = rng.random(m)
            e_ref = _reference(a_t, s_t, u_t, mt_t, u, alpha, q)
            e = _two_phase(p, a_bar, r, u0, mt0, hinv, u, alpha)
            assert np.array_equal((a_t @ e) % q, u)
            assert np.array_equal(e, e_ref)
    # the key of the installed tag is the one the switch starts from
    assert np.array_equal(a0[:, :mb], a_bar)
