"""CPU check (numpy + the oracle) of the offline / online split of two-phase PSFGPV::samp_p (DESIGN.md 4.12,
tools_b200/csrc/api.cu samp_p_offline_chunk / samp_p_online_chunk).  Under the common random numbers of
test_two_phase_math.py (z_i = floor(c'_i + alpha_i)), phase 1 and its products -A_bar z2 mod q and Mt_1 z2 are computed
ONCE, without a target; then several targets u are finished from that state alone.  Each result must equal the two-phase
form computed from scratch for that u, and the reference loop (gpv.rs:152-161)."""
import numpy as np
import pytest

from oracle import qfall_oracle as O

from test_two_phase_math import _digits, _gso, _key, _sprime


@pytest.mark.parametrize("n,q", [(3, 2**6), (4, 2**5), (3, 53), (5, 97)])
def test_offline_state_finishes_every_target(n, q):
    p, a, r, s, rng = _key(n, q, seed=n * 777 + q)
    nk, mb, m, k = p.n * p.k, p.m_bar, p.m, p.k
    sp = _sprime(p)
    u_mat, mt = _gso(s)
    u11 = np.triu(u_mat[:nk, :nk])
    mprime = mt[:nk, :mb] @ r + mt[:nk, mb:]
    alpha = rng.random(m)
    # ---- offline: phase 1 (centres start at 0), -A_bar z2 mod q, Mt_1 z2 -- no target anywhere
    z2 = np.zeros(mb)
    c2 = np.zeros(mb)
    for i in range(mb - 1, -1, -1):
        z2[i] = np.floor(c2[i] + alpha[nk + i])
        c2[:i] -= u_mat[nk:nk + i, nk + i] * z2[i]
    z2 = z2.astype(np.int64)
    neg_abar_z2 = (-(a[:, :mb] @ z2)) % q
    mt1_z2 = mt[:nk, :mb] @ z2
    for trial in range(5):
        u = rng.integers(0, q, n)
        # ---- online: w = u - A_bar z2 from the stored residues, then g3, the centres, phase 2, the tail
        h = (u + neg_abar_z2) % q
        g3 = _digits(h.copy(), k, p.base)
        t1 = -(mprime @ g3)
        t1 = t1 - mt1_z2  # (a) then (b): the order of the composed form
        z1 = np.zeros(nk)
        for i in range(nk - 1, -1, -1):
            z1[i] = np.floor(t1[i] + alpha[i])
            t1[:i] -= u11[:i, i] * z1[i]
        e_bot = g3 + sp @ z1.astype(np.int64)
        e = np.concatenate([z2 + r @ e_bot, e_bot])
        assert np.array_equal((a @ e) % q, u)
        # ---- the two-phase form from scratch for this u (test_two_phase_math.py)
        h2 = (u - a[:, :mb] @ z2) % q
        assert np.array_equal(h, h2)
        t2 = -(mprime @ _digits(h2.copy(), k, p.base)) - mt[:nk, :mb] @ z2
        y1 = np.zeros(nk)
        for i in range(nk - 1, -1, -1):
            y1[i] = np.floor(t2[i] + alpha[i])
            t2[:i] -= u11[:i, i] * y1[i]
        assert np.array_equal(y1, z1)
        # ---- the reference loop: centre -sol over all m coordinates
        sol = np.array(O.solve_unit_pivots(a.tolist(), u.tolist(), q), dtype=np.int64)
        c = -(mt @ sol)
        z = np.zeros(m)
        for i in range(m - 1, -1, -1):
            z[i] = np.floor(c[i] + alpha[i])
            c[:i] -= u_mat[:i, i] * z[i]
        assert np.array_equal(e, sol + s @ z.astype(np.int64)), trial
