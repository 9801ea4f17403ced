"""Host-side G-trapdoor machinery (key setup, not per target): the mirror of
src/sample/g_trapdoor/*.rs and src/utils/rotation_matrix.rs in vectorised numpy.
Everything here runs once per key; the per-target work is in the CUDA library."""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np


def _ceil_log(x: int, base: int) -> int:
    e, p = 0, 1
    while p < x:
        p *= base
        e += 1
    return e


@dataclass
class GadgetParameters:
    """gadget_parameters.rs:44-52 (distribution fixed to PlusMinusOneZero, :131)."""

    n: int
    k: int
    m_bar: int
    base: int
    q: int

    @classmethod
    def init_default(cls, n: int, q: int) -> "GadgetParameters":
        """gadget_parameters.rs:113-133."""
        n, q = int(n), int(q)
        if n < 1:
            raise ValueError("n must be positive")
        k = _ceil_log(q, 2)
        return cls(n=n, k=k, m_bar=n * k + _ceil_log(n, 2) ** 2, base=2, q=q)

    @property
    def m(self) -> int:
        return self.m_bar + self.n * self.k


@dataclass
class GadgetParametersRing:
    """gadget_parameters.rs:73-81; modulus X^n + 1 mod q (common_moduli.rs:41-48),
    distribution SampleZ (:183)."""

    n: int
    k: int
    m_bar: int
    base: int
    q: int

    @classmethod
    def init_default(cls, n: int, q: int) -> "GadgetParametersRing":
        """gadget_parameters.rs:165-185."""
        n, q = int(n), int(q)
        if n < 1:
            raise ValueError("n must be positive")
        k = _ceil_log(q, 2)
        return cls(n=n, k=k, m_bar=k + 2, base=2, q=q)


# ---- classical gadget (gadget_classical.rs) -----------------------------------


def gen_gadget_vec(k: int, base: int) -> np.ndarray:
    """gadget_classical.rs:128-136."""
    return np.array([[base**i] for i in range(k)], dtype=object)


def gen_gadget_mat(n: int, k: int, base: int) -> np.ndarray:
    """gadget_classical.rs:91-107: I_n (x) g^t."""
    g = np.array([base**i for i in range(k)], dtype=object)
    out = np.zeros((n, n * k), dtype=object)
    for j in range(n):
        out[j, j * k:(j + 1) * k] = g
    return out


def find_solution_gadget_vec(value: int, q: int, k: int, base: int) -> np.ndarray:
    """gadget_classical.rs:169-182."""
    return find_solution_gadget_mat(np.array([[value]], dtype=object), q, k, base)[:, 0]


def find_solution_gadget_mat(value: np.ndarray, q: int, k: int, base: int) -> np.ndarray:
    """gadget_classical.rs:219-229: digits of row j at rows k*j .. k*j+k-1 (int64 result)."""
    if base**k < q:
        raise ValueError("The modulus is too large, the value is potentially not representable.")
    v = np.asarray(value)
    small = q < 2**62
    v = (v.astype(np.int64) % np.int64(q)) if small and v.dtype != object else np.array(v % q, dtype=object)
    rows, cols = v.shape
    out = np.zeros((rows * k, cols), dtype=np.int64)
    for t in range(k):
        d = v % base
        out[t::k, :] = d.astype(np.int64)
        v = (v - d) // base
    return out


def short_basis_gadget_block(k: int, base: int, q: int) -> np.ndarray:
    """The k x k block S_k of gadget_classical.rs:248-272."""
    sk = np.zeros((k, k), dtype=np.int64)
    for j in range(k):
        sk[j, j] = base
    for i in range(k - 1):
        sk[i + 1, i] = -1
    if base**k != q:
        qq = q
        for i in range(k):
            sk[i, k - 1] = qq % base
            qq //= base
    return sk


def gso_small(basis: np.ndarray) -> np.ndarray:
    """Exact-rational unnormalised Gram-Schmidt of the columns of a SMALL integer matrix (the k x k gadget block;
    MatQ::gso as used at mp_perturbation.rs:234), returned as float64."""
    from fractions import Fraction

    b = [[Fraction(int(x)) for x in row] for row in np.asarray(basis).tolist()]
    rows, cols = len(b), len(b[0])
    out = [[Fraction(0)] * cols for _ in range(rows)]
    for j in range(cols):
        v = [b[t][j] for t in range(rows)]
        for i in range(j):
            gi = [out[t][i] for t in range(rows)]
            den = sum(x * x for x in gi)
            if den:
                mu = sum(x * y for x, y in zip(v, gi)) / den
                v = [x - mu * y for x, y in zip(v, gi)]
        for t in range(rows):
            out[t][j] = v[t]
    return np.array([[float(x) for x in row] for row in out], dtype=np.float64)


def short_basis_gadget(p: GadgetParameters) -> np.ndarray:
    """gadget_classical.rs:248-287: I_n (x) S_k."""
    return np.kron(np.eye(p.n, dtype=np.int64), short_basis_gadget_block(p.k, p.base, p.q))


def _inverse_mod(a: np.ndarray, q: int) -> np.ndarray:
    n = a.shape[0]
    m = [[int(x) % q for x in row] + [int(i == j) for j in range(n)] for i, row in enumerate(a.tolist())]
    for c in range(n):
        piv = next((r for r in range(c, n) if math.gcd(m[r][c], q) == 1), None)
        if piv is None:
            raise ValueError("tag is not invertible by unit pivoting")
        m[c], m[piv] = m[piv], m[c]
        inv = pow(m[c][c], -1, q)
        m[c] = [(x * inv) % q for x in m[c]]
        for r in range(n):
            if r != c and m[r][c]:
                f = m[r][c]
                m[r] = [(x - f * y) % q for x, y in zip(m[r], m[c])]
    return np.array([row[n:] for row in m], dtype=object)


def compute_w(p: GadgetParameters, a: np.ndarray, tag: np.ndarray | None = None) -> np.ndarray:
    """short_basis_classical.rs:105-110: digits of -tag^{-1} A[:, :m_bar]."""
    left = np.asarray(a)[:, : p.m_bar]
    if tag is not None:
        left = np.array(_inverse_mod(np.asarray(tag), p.q).dot(left.astype(object)) % p.q, dtype=object)
        rhs = (-left) % p.q
    else:
        rhs = (-left.astype(np.int64)) % np.int64(p.q)
    return find_solution_gadget_mat(rhs, p.q, p.k, p.base)


def gen_short_basis_for_trapdoor(p: GadgetParameters, a: np.ndarray, r: np.ndarray, tag: np.ndarray | None = None) -> np.ndarray:
    """short_basis_classical.rs:54-110:  [[I,R],[0,I]] * [[0,I],[S',W]] = [[R S', I + R W],[S', W]]
    (S' column-reversed iff base^k = q, :80-82).  Exact: all products are small integers, done
    in float64 BLAS."""
    s = short_basis_gadget(p)
    if p.base**p.k == p.q:
        s = s[:, ::-1]
    w = compute_w(p, a, tag)
    rf = np.asarray(r, dtype=np.float64)
    nk, mb = p.n * p.k, p.m_bar
    out = np.zeros((p.m, p.m), dtype=np.int64)
    out[:mb, :nk] = np.rint(rf @ s.astype(np.float64)).astype(np.int64)
    out[:mb, nk:] = np.rint(rf @ w.astype(np.float64)).astype(np.int64) + np.eye(mb, dtype=np.int64)
    out[mb:, :nk] = s
    out[mb:, nk:] = w
    return out


# ---- rotation matrices (utils/rotation_matrix.rs) ------------------------------


def rot_minus(vec) -> np.ndarray:
    """rotation_matrix.rs:41-63: column j = coefficients of a * X^j mod X^n + 1."""
    v = np.asarray(vec, dtype=object)
    if v.ndim == 2:
        if 1 not in v.shape:
            raise ValueError("The input must be a vector.")
        v = v.reshape(-1)
    n = len(v)
    out = np.zeros((n, n), dtype=object)
    for j in range(n):
        out[j:, j] = v[: n - j]
        out[:j, j] = -v[n - j:]
    return out


def rot_minus_matrix(matrix) -> np.ndarray:
    """rotation_matrix.rs:85-96."""
    m = np.asarray(matrix, dtype=object)
    return np.concatenate([rot_minus(m[:, c]) for c in range(m.shape[1])], axis=1)


def rot_f(h, f, q: int) -> np.ndarray:
    """The tag of h in polynomial form: the n x n matrix of multiplication by h in Z_q[X]/(f), f = X^n + sum_{i<n} f[i] X^i
    monic (f: its n low coefficients).  Column c holds the coefficients of h X^c mod f, reduced mod q (int64).  For
    f = X^n + 1 it is rot_minus(h) mod q."""
    fv = [int(x) for x in np.asarray(f, dtype=object).reshape(-1)]
    col = [int(x) % q for x in np.asarray(h, dtype=object).reshape(-1)]
    n = len(fv)
    assert len(col) == n
    out = np.zeros((n, n), dtype=object)
    for c in range(n):
        out[:, c] = col
        top = col[-1]
        col = [((col[i - 1] if i else 0) - top * fv[i]) % q for i in range(n)]
    return np.array(out, dtype=np.int64)


def _rot_i64(p: np.ndarray) -> np.ndarray:
    n = len(p)
    out = np.zeros((n, n), dtype=np.int64)
    for j in range(n):
        out[j:, j] = p[: n - j]
        out[:j, j] = -p[n - j:]
    return out


# ---- ring gadget / short basis (gadget_ring.rs, short_basis_ring.rs) ------------


def find_solution_gadget_ring(u: np.ndarray, p: GadgetParametersRing) -> np.ndarray:
    """gadget_ring.rs:145-166 -> k x n array: row i, column j = digit i of coefficient j."""
    d = find_solution_gadget_mat(np.asarray(u, dtype=np.int64).reshape(-1, 1) % p.q, p.q, p.k, p.base)
    return d[:, 0].reshape(p.n, p.k).T.copy()


def ring_short_basis_embedded(p: GadgetParametersRing, a: np.ndarray, r: np.ndarray, e: np.ndarray) -> np.ndarray:
    """Coefficient embedding of gen_short_basis_for_trapdoor_ring (short_basis_ring.rs:64-166):
    a (k+2) x n residues, r/e k x n small ints -> D x D int64, D = n (k+2); row = poly_row * n + coeff,
    column = basis vector.  sa_l * sa_r reduced by X^n + 1, built blockwise with rot^- matrices."""
    n, k = p.n, p.k
    D = n * (k + 2)
    s = short_basis_gadget_block(k, p.base, p.q)
    if p.base**k == p.q:
        s = s[:, ::-1]
    w = [find_solution_gadget_ring((-np.asarray(a[c], dtype=np.int64)) % p.q, p) for c in range(2)]  # k x n each
    rot_e = [_rot_i64(np.asarray(e[j], dtype=np.int64)) for j in range(k)]
    rot_r = [_rot_i64(np.asarray(r[j], dtype=np.int64)) for j in range(k)]
    out = np.zeros((D, D), dtype=np.int64)
    eye = np.eye(n, dtype=np.int64)
    # first n*k columns: column i*k + c  = X^i * [sum_j e_j s'_jc ; sum_j r_j s'_jc ; s'_0c ; ... ; s'_{k-1,c}]
    for c in range(k):
        top_e = sum(int(s[j, c]) * rot_e[j] for j in range(k))
        top_r = sum(int(s[j, c]) * rot_r[j] for j in range(k))
        cols = np.arange(n) * k + c
        out[0:n, cols] = top_e
        out[n:2 * n, cols] = top_r
        for j in range(k):
            if s[j, c]:
                out[(2 + j) * n:(3 + j) * n, cols] = int(s[j, c]) * eye
    off = n * k
    for c in range(2):
        cols = off + np.arange(n) * 2 + c
        rot_w = [_rot_i64(w[c][j]) for j in range(k)]
        top_e = sum(rot_e[j] @ rot_w[j] for j in range(k))
        top_r = sum(rot_r[j] @ rot_w[j] for j in range(k))
        if c == 0:
            top_e = top_e + eye
        else:
            top_r = top_r + eye
        out[0:n, cols] = top_e
        out[n:2 * n, cols] = top_r
        for j in range(k):
            out[(2 + j) * n:(3 + j) * n, cols] = rot_w[j]
    return out
