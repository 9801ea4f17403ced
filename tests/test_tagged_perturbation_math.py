"""CPU check (the oracle's big-integer restatement) of PSFPerturbation on tagged G-trapdoor keys (DESIGN.md 4.4).
For A = gen_trapdoor(A_bar, H, R) = [A_bar | H G - A_bar R] the trapdoor relation is A [R; I] = H G, so the MP12 sampler
(mp_perturbation.rs:304-336) needs the gadget preimage of v' = H^-1 (u - A p) instead of v = u - A p.  With
A' = H^-1 A = gen_trapdoor(H^-1 A_bar, I, R), H^-1 (u - A p) = H^-1 u - A' p, and p does not depend on A: for the same
random draws the tagged sampler on (A, u) returns exactly what the untagged one returns on (A', H^-1 u)."""
import numpy as np
import pytest

from oracle import qfall_oracle as O


def samp_p_perturbation_tagged(rng, p, a, tag, r_mat, sqrt_sigma_2, s_basis, s_gso, u, r):
    """mp_perturbation.rs:304-336 for a tagged key A = [A_bar | H G - A_bar R]: z solves G z = H^-1 (u - A p) mod q."""
    hinv = np.array(O.mat_inverse_mod(tag, p.q), dtype=object)
    vec_p = O.sample_d_common_non_spherical(rng, sqrt_sigma_2, r)
    ap = O.f_a_classical(a, vec_p, p.q)
    v = np.array([(ui - x) % p.q for ui, x in zip(u, ap)], dtype=object)
    v_tag = [int(x) % p.q for x in hinv.dot(v)]
    z = O.randomized_nearest_plane_gadget(rng, v_tag, p, r, s_basis, s_gso)
    rz = np.array(r_mat, dtype=object).dot(np.array(z, dtype=object))
    top = [int(x) + int(y) for x, y in zip(vec_p[: p.m_bar], rz)]
    bot = [int(x) + int(y) for x, y in zip(vec_p[p.m_bar :], z)]
    return top + bot


def _tag(n, q, rng, kind):
    if kind == "unitriangular":
        h = np.triu(rng.integers(0, q, (n, n)), 1) + np.eye(n, dtype=np.int64)
        return [[int(x) for x in row] for row in h]
    while True:  # a random matrix that MatZq::inverse (unit pivoting) accepts
        h = rng.integers(0, q, (n, n)).tolist()
        try:
            O.mat_inverse_mod(h, q)
            return h
        except ValueError:
            continue


@pytest.mark.parametrize("n,q,kind", [(3, 64, "unitriangular"), (3, 64, "dense"), (4, 127, "dense"), (3, 3329, "unitriangular")])
def test_tagged_perturbation_sampler_is_the_reduced_identity_sampler(n, q, kind):
    r, s = 3.0, 25.0
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 1000 + q)
    a_bar = rng.integers(0, q, (n, p.m_bar)).tolist()
    r_mat = O.sample_pm_one_zero(rng, p.m_bar, p.n * p.k)
    tag = _tag(n, q, rng, kind)
    hinv = np.array(O.mat_inverse_mod(tag, q), dtype=object)
    a = O.gen_trapdoor(p, a_bar, tag, r_mat)
    a_red = O.gen_trapdoor(p, (hinv.dot(np.array(a_bar, dtype=object)) % q).tolist(), O.mat_identity(n), r_mat)
    assert np.array_equal(np.array(a_red, dtype=object), hinv.dot(np.array(a, dtype=object)) % q)
    l = O.compute_sqrt_sigma_2(np.array(r_mat, dtype=np.int64), s, r, p.base)
    sb = np.array(O.short_basis_gadget(p), dtype=np.int64)
    sg = O.gso_f64(sb.astype(np.float64))
    for t in range(4):
        u = rng.integers(0, q, n).tolist()
        e = samp_p_perturbation_tagged(np.random.default_rng(t), p, a, tag, r_mat, l, sb.tolist(), sg, u, r)
        assert O.f_a_classical(a, e, q) == u
        u_red = [int(x) % q for x in hinv.dot(np.array(u, dtype=object))]
        e_red = O.samp_p_perturbation(np.random.default_rng(t), p, a_red, r_mat, l, sb.tolist(), sg, u_red, r)
        assert e == e_red
