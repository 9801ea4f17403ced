"""CPU check (the oracle's big-integer primitives) of the identity behind samp_p with a tag per target (DESIGN.md 4.4).
For the installed key A = [A_bar | H_0 G - A_bar R] and a tag H_t, A_t = [A_bar | H_t G - A_bar R] = A + [0 | (H_t - H_0) G].
With y = G p_bot for a perturbation p (p_bot = p[m_bar:]):
    H_t^-1 (u - A_t p) = H_t^-1 (u - A p + H_0 y) - y   (mod q),
so the per-target kernel turns v = u - A p, which samp_p already computes, into the syndrome of tag t exactly."""
import numpy as np
import pytest

from oracle import qfall_oracle as O


def _tag(n, q, rng, kind):
    if kind == "identity":
        return O.mat_identity(n)
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


def _g_times(p, x):
    """G x for x of length n k: y_i = sum_s base^s x[i k + s] (the layout of gen_gadget_mat)."""
    return [sum(p.base**s * int(x[i * p.k + s]) for s in range(p.k)) for i in range(p.n)]


@pytest.mark.parametrize("n,q,h0_kind", [(3, 64, "identity"), (3, 64, "dense"), (4, 127, "unitriangular"),
                                         (3, 3329, "dense"), (2, 2**61 - 1, "dense"), (3, 2**48, "unitriangular")])
def test_tagged_syndrome_identity(n, q, h0_kind):
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 7919 + q % 10007)
    a_bar = rng.integers(0, q, (n, p.m_bar)).tolist()
    r_mat = O.sample_pm_one_zero(rng, p.m_bar, p.n * p.k)
    h0 = _tag(n, q, rng, h0_kind)
    a = np.array(O.gen_trapdoor(p, a_bar, h0, r_mat), dtype=object)
    g = np.array(O.gen_gadget_mat(p.n, p.k, p.base), dtype=object)
    for kind in ("identity", "dense", "unitriangular", "dense"):
        ht = _tag(n, q, rng, kind)
        a_t = np.array(O.gen_trapdoor(p, a_bar, ht, r_mat), dtype=object)
        ht_inv = np.array(O.mat_inverse_mod(ht, q), dtype=object)
        for _ in range(3):
            u = np.array(rng.integers(0, q, n).tolist(), dtype=object)
            vec_p = np.array(rng.integers(-3000, 3000, p.m).tolist(), dtype=object)
            y = np.array(_g_times(p, vec_p[p.m_bar:]), dtype=object)
            assert np.array_equal(y, g.dot(vec_p[p.m_bar:]))
            lhs = ht_inv.dot((u - a_t.dot(vec_p)) % q) % q
            v = (u - a.dot(vec_p)) % q
            w = (v + np.array(h0, dtype=object).dot(y)) % q
            rhs = (ht_inv.dot(w) - y) % q
            assert np.array_equal(lhs, rhs)
