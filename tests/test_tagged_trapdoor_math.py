"""CPU checks (the oracle's big-integer restatement) of the reduction behind tagged G-trapdoor keys
(DESIGN.md 4.3, tools_b200/csrc/api.cu detect_gpv_structure): for A = gen_trapdoor(A_bar, H, R) = [A_bar | H G - A_bar R]
with H invertible mod q,
  H^-1 A = gen_trapdoor(H^-1 A_bar, I, R)                                                  (same R, identity tag)
  gen_short_basis_for_trapdoor(H, A, R) = gen_short_basis_for_trapdoor(I, H^-1 A mod q, R)  (the same basis)
so samp_p(A, S, u) is samp_p(H^-1 A, S, H^-1 u): the identity-tag two-phase recursion with u' = H^-1 u."""
import numpy as np
import pytest

from oracle import qfall_oracle as O


def _unitriangular_tag(n, q, rng):
    h = np.triu(rng.integers(0, q, (n, n)), 1) + np.eye(n, dtype=np.int64)
    return [[int(x) for x in row] for row in h]


def _dense_tag(n, q, rng):
    while True:  # a random matrix that MatZq::inverse (unit pivoting) accepts
        h = rng.integers(0, q, (n, n)).tolist()
        try:
            O.mat_inverse_mod(h, q)
            return h
        except ValueError:
            continue


def _key(n, q, seed, tag_kind):
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(seed)
    a_bar = rng.integers(0, q, (n, p.m_bar)).tolist()
    r = O.sample_pm_one_zero(rng, p.m_bar, p.n * p.k)
    tag = _unitriangular_tag(n, q, rng) if tag_kind == "unitriangular" else _dense_tag(n, q, rng)
    return p, a_bar, r, tag


CASES = [(3, 2**6, "unitriangular"), (4, 256, "unitriangular"), (5, 3329, "unitriangular"), (3, 2**16, "unitriangular"),
         (4, 127, "dense"), (5, 3329, "dense"), (3, 2**31 - 1, "dense"), (6, 97, "dense")]


@pytest.mark.parametrize("n,q,tag_kind", CASES)
def test_tagged_key_is_identity_key_of_h_inverse_a(n, q, tag_kind):
    p, a_bar, r, tag = _key(n, q, 100 * n + q % 1000, tag_kind)
    h_inv = O.mat_inverse_mod(tag, q)
    assert O.mat_mul(h_inv, tag, q) == O.mat_identity(n)
    a = O.gen_trapdoor(p, a_bar, tag, r)
    a_bar_p = O.mat_mul(h_inv, a_bar, q)
    assert O.mat_mul(h_inv, a, q) == O.gen_trapdoor(p, a_bar_p, O.mat_identity(n), r)


@pytest.mark.parametrize("n,q,tag_kind", CASES)
def test_tagged_short_basis_equals_identity_basis_of_h_inverse_a(n, q, tag_kind):
    p, a_bar, r, tag = _key(n, q, 100 * n + q % 1000 + 1, tag_kind)
    a = O.gen_trapdoor(p, a_bar, tag, r)
    s = O.gen_short_basis_for_trapdoor(p, tag, a, r)
    h_inv_a = O.mat_mul(O.mat_inverse_mod(tag, q), a, q)
    assert s == O.gen_short_basis_for_trapdoor(p, O.mat_identity(n), h_inv_a, r)
    # the basis spans the kernel lattice of both keys, and a preimage for u under A is one for H^-1 u under H^-1 A
    sa = np.array(s, dtype=object)
    assert not (np.array(a, dtype=object).dot(sa) % q).any()
    assert not (np.array(h_inv_a, dtype=object).dot(sa) % q).any()
    rng = np.random.default_rng(n)
    x = rng.integers(-50, 50, p.m).astype(object)
    u = np.array(a, dtype=object).dot(x) % q
    u_p = np.array(O.mat_inverse_mod(tag, q), dtype=object).dot(u) % q
    assert np.array_equal(np.array(h_inv_a, dtype=object).dot(x) % q, u_p)


def test_unit_pivot_rule_rejects_even_first_column():
    """A tag whose first column has no unit mod 2^16 is rejected by unit pivoting (the device inverse follows this rule)."""
    q = 2**16
    tag = [[2, 1, 0], [4, 1, 1], [6, 0, 1]]
    with pytest.raises(ValueError):
        O.mat_inverse_mod(tag, q)
