"""CPU check (the oracle's big-integer primitives) of the identity behind f_a with a tag per target (DESIGN.md 4.9).
For a key A = [A_bar | H_0 G - A_bar R] and any tag H_t, the key of tag t is A_t = [A_bar | H_t G - A_bar R], and
    A_t sigma = A sigma + (H_t - H_0) G sigma_bot   (mod q),   sigma_bot = sigma[m_bar:],
so qf_f_a_tagged needs only A, the differences D_t = H_t - H_0 and y = G sigma_bot: no trapdoor and no inverse.  Singular
tags, H_0 = 0 (the base key [A_bar | -A_bar R]) and int32 sigma of any magnitude are covered."""
import numpy as np
import pytest

from oracle import qfall_oracle as O


def _tag(n, q, rng, kind):
    if kind == "identity":
        return O.mat_identity(n)
    if kind == "zero":
        return [[0] * n for _ in range(n)]
    if kind == "unitriangular":
        h = np.triu(rng.integers(0, q, (n, n)), 1) + np.eye(n, dtype=np.int64)
        return [[int(x) for x in row] for row in h]
    if kind == "singular":  # two equal rows
        h = rng.integers(0, q, (n, n)).tolist()
        h[-1] = list(h[0])
        return h
    return rng.integers(0, q, (n, n)).tolist()  # dense, not necessarily invertible


@pytest.mark.parametrize("n,q,h0_kind", [(3, 64, "identity"), (3, 64, "dense"), (4, 127, "zero"), (3, 3329, "dense"),
                                         (2, 2**32, "identity"), (3, 2**48, "zero"), (2, 2**62 - 1, "dense")])
def test_tagged_f_a_identity(n, q, h0_kind):
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(n * 131 + q % 9973)
    a_bar = rng.integers(0, q, (n, p.m_bar)).tolist()
    r_mat = O.sample_pm_one_zero(rng, p.m_bar, p.n * p.k)
    h0 = _tag(n, q, rng, h0_kind)
    a = np.array(O.gen_trapdoor(p, a_bar, h0, r_mat), dtype=object)
    g = np.array(O.gen_gadget_mat(p.n, p.k, p.base), dtype=object)
    lim = 2**31 - 1
    for kind in ("dense", "unitriangular", "singular", "zero", "identity"):
        ht = _tag(n, q, rng, kind)
        a_t = np.array(O.gen_trapdoor(p, a_bar, ht, r_mat), dtype=object)
        d = (np.array(ht, dtype=object) - np.array(h0, dtype=object)) % q
        for sig in (rng.integers(-3000, 3000, p.m), rng.integers(-lim, lim + 1, p.m), np.full(p.m, -lim), np.full(p.m, lim)):
            sigma = [int(x) for x in sig]
            want = O.f_a_classical(a_t.tolist(), sigma, q)
            y = g.dot(np.array(sigma[p.m_bar:], dtype=object)) % q
            got = (np.array(O.f_a_classical(a.tolist(), sigma, q), dtype=object) + d.dot(y)) % q
            assert [int(x) for x in got] == [int(x) for x in want]
