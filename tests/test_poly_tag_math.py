"""CPU check of the algebra behind tags in polynomial form (DESIGN.md 4.10), on big integers.  A tag h in Z_q[X]/(f),
f = X^n + sum_{i<n} f_i X^i monic, stands for the matrix H = rot_f(h) whose column c holds the coefficients of h X^c mod f.
    rot_f(a) rot_f(b) = rot_f(a b),  so  rot_f(h)^-1 = rot_f(h^-1),  and  rot_f(a) v = a * v mod f,
so the tag tables of samp_p and f_a need n words per tag, an O(n^2) inverse and one product mod (f, q) per target.  For
q = p^e, h is a unit iff h mod p is a unit in F_p[X]/(f mod p) (Z_q[X]/(f) is local over p), and Gauss-Jordan with unit
pivots accepts rot_f(h) exactly then.  The reference inverse below (extended Euclid mod p, Newton lifting to q) is the
algorithm the device runs; it is checked here against the oracle's Gauss-Jordan inverse of rot_f(h)."""
import numpy as np
import pytest

from oracle import qfall_oracle as O
from tools_b200 import gadget


# ---- big-integer references --------------------------------------------------------------------------------------------
def rot_f(h, f, q):
    """Column c = coefficients of h X^c mod f, mod q (f: the n low coefficients of the monic modulus)."""
    n = len(f)
    col = [int(x) % q for x in h]
    out = [[0] * n for _ in range(n)]
    for c in range(n):
        for i in range(n):
            out[i][c] = col[i]
        top = col[-1]
        col = [((col[i - 1] if i else 0) - top * int(f[i])) % q for i in range(n)]
    return out


def is_prime_u64(n):
    if n < 2:
        return False
    wit = (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37)
    for w in wit:
        if n % w == 0:
            return n == w
    d, r = n - 1, 0
    while d % 2 == 0:
        d //= 2
        r += 1
    for w in wit:
        x = pow(w, d, n)
        if x in (1, n - 1):
            continue
        for _ in range(r - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


def prime_power(q):
    """(p, e) with q = p^e, p prime, or None: the largest e with an exact e-th root, whose root must be prime."""
    for e in range(q.bit_length(), 0, -1):
        r = max(2, round(q ** (1.0 / e)))
        while r > 2 and r**e > q:
            r -= 1
        while (r + 1) ** e <= q:
            r += 1
        if r**e == q:
            return (r, e) if is_prime_u64(r) else None
    return None


def poly_mulmod(a, b, f, q):
    n = len(f)
    c = [0] * (2 * n - 1)
    for i, x in enumerate(a):
        for j, y in enumerate(b):
            c[i + j] += int(x) * int(y)
    for k in range(2 * n - 2, n - 1, -1):
        t = c[k]
        for i in range(n):
            c[k - n + i] -= t * int(f[i])
    return [x % q for x in c[:n]]


def poly_inverse_mod(h, f, q):
    """h^-1 mod (f, q), q = p^e: extended Euclid in F_p[X], then s <- s (2 - h s) until p^(2^i) >= q.  ValueError when h is
    not a unit or q is not a prime power."""
    pe = prime_power(q)
    if pe is None:
        raise ValueError("q is not a prime power")
    p, e = pe
    n = len(f)

    def trim(x):
        x = [v % p for v in x]
        while x and x[-1] == 0:
            x.pop()
        return x

    def sub_shift(x, y, c, sh):  # x - c X^sh y over F_p
        x = list(x) + [0] * max(0, len(y) + sh - len(x))
        for i, v in enumerate(y):
            x[i + sh] = (x[i + sh] - c * v) % p
        return trim(x)

    r0, r1, t0, t1 = trim(list(f) + [1]), trim(h), [], [1]
    while len(r1) > 1:
        inv = pow(r1[-1], -1, p)
        while len(r0) >= len(r1):
            c, sh = r0[-1] * inv % p, len(r0) - len(r1)
            r0, t0 = sub_shift(r0, r1, c, sh), sub_shift(t0, t1, c, sh)
        r0, r1, t0, t1 = r1, r0, t1, t0
    if not r1:
        raise ValueError("h is not a unit")
    inv = pow(r1[0], -1, p)
    assert len(t1) <= n
    s = [v * inv % p for v in t1] + [0] * (n - len(t1))
    hq, prec = [int(x) % q for x in h], 1
    while prec < e:
        hs = poly_mulmod(hq, s, f, q)
        s = poly_mulmod(s, [((2 if i == 0 else 0) - v) % q for i, v in enumerate(hs)], f, q)
        prec *= 2
    return s


# ---- cases -------------------------------------------------------------------------------------------------------------
QS = [4093, 2**32 - 5, 2**61 - 1, 2**16, 2**32, 3**10]
FAMILIES = ["x^n+1", "x^n-1", "random"]


def _f(kind, n, q, rng):
    if kind == "x^n+1":
        return [1] + [0] * (n - 1)
    if kind == "x^n-1":
        return [-1] + [0] * (n - 1)
    return [int(x) for x in rng.integers(-(2**62), 2**62, n)]  # any sign and size: taken mod q


def _rand(n, q, rng):
    return [int(x) % q for x in rng.integers(0, 2**62, n)]


def _mat_mul(a, b, q):
    return [[int(x) for x in row] for row in (np.array(a, dtype=object).dot(np.array(b, dtype=object)) % q)]


def _eye(n):
    return [[int(i == j) for j in range(n)] for i in range(n)]


@pytest.mark.parametrize("q", QS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_inverse_matches_matrix_inverse(q, fam):
    """s = poly_inverse_mod(h) gives rot_f(h) rot_f(s) = I and rot_f(s) = mat_inverse_mod(rot_f(h)); the tags the
    polynomial inverse refuses are exactly those whose rot_f Gauss-Jordan refuses."""
    n = 4
    rng = np.random.default_rng(q % 10007 + 31 * FAMILIES.index(fam))
    f = _f(fam, n, q, rng)
    p = prime_power(q)[0]
    hs = [_rand(n, q, rng) for _ in range(10)]
    hs += [[p * x % q for x in _rand(n, q, rng)], [0] * n]  # h = 0 mod p: never a unit
    if fam == "x^n-1":
        hs.append([x % q for x in [1, -1, 0, 0]])  # X - 1 divides X^n - 1
    if fam == "random":
        hs.append([x % q for x in [0, 1, 0, 0]])  # X is a unit iff f_0 is a unit mod p
    units = refused = 0
    for h in hs:
        hm = rot_f(h, f, q)
        try:
            ref = O.mat_inverse_mod(hm, q)
        except ValueError:
            ref = None
        try:
            s = poly_inverse_mod(h, f, q)
        except ValueError:
            s = None
        assert (s is None) == (ref is None), h
        if s is None:
            refused += 1
            continue
        units += 1
        sm = rot_f(s, f, q)
        assert _mat_mul(hm, sm, q) == _eye(n)
        assert _mat_mul(sm, hm, q) == _eye(n)
        assert sm == [[x % q for x in row] for row in ref]
        assert poly_mulmod(h, s, f, q) == [1 % q] + [0] * (n - 1)
    assert units >= 3 and refused >= 2


@pytest.mark.parametrize("q", QS)
def test_rot_f_of_x_n_plus_1_is_rot_minus(q):
    rng = np.random.default_rng(q % 997)
    for n in (1, 2, 5, 8):
        h = [int(x) for x in rng.integers(-(2**62), 2**62, n)]
        want = (np.array(gadget.rot_minus(h), dtype=object) % q).tolist()
        assert rot_f(h, [1] + [0] * (n - 1), q) == want
        assert gadget.rot_f(h, [1] + [0] * (n - 1), q).tolist() == want


@pytest.mark.parametrize("q", QS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_product_and_bindings_rot_f(q, fam):
    """rot_f(a) v = a * v mod (f, q), rot_f(a) rot_f(b) = rot_f(a b), and tools_b200.gadget.rot_f is the reference's."""
    n = 5
    rng = np.random.default_rng(q % 4099 + 7 * FAMILIES.index(fam))
    f = _f(fam, n, q, rng)
    a, b = _rand(n, q, rng), _rand(n, q, rng)
    am = rot_f(a, f, q)
    got = (np.array(am, dtype=object).dot(np.array(b, dtype=object)) % q).tolist()
    assert got == poly_mulmod(a, b, f, q)
    assert _mat_mul(am, rot_f(b, f, q), q) == rot_f(poly_mulmod(a, b, f, q), f, q)
    assert gadget.rot_f(a, f, q).tolist() == am


def _h0(kind, n, q, rng):
    if kind == "identity":
        return _eye(n)
    if kind == "zero":
        return [[0] * n for _ in range(n)]
    while True:
        h = rng.integers(0, q, (n, n)).tolist() if q < 2**63 else None
        try:
            O.mat_inverse_mod(h, q)
            return h
        except ValueError:
            continue


@pytest.mark.parametrize("q", QS)
@pytest.mark.parametrize("h0_kind", ["identity", "dense", "zero"])
@pytest.mark.parametrize("fam", FAMILIES)
def test_syndrome_and_f_a_identities(q, h0_kind, fam):
    """samp_p: H_t^-1 (v + H_0 y) - y = s_t * (v + H_0 y) - y mod (f, q) with s_t = h_t^-1 (what the syndrome kernel
    computes in polynomial form).  f_a: A_t sigma = A sigma + h_t * y - H_0 y with y = G sigma_bot, for the keys
    A = [A_bar | H_0 G - A_bar R] and A_t = [A_bar | rot_f(h_t) G - A_bar R] of the oracle's gen_trapdoor.  H_0 = 0 is only
    an f_a key (its trapdoor needs an invertible H_0)."""
    n = 3
    p = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(q % 8191 + 3 * FAMILIES.index(fam) + 11 * len(h0_kind))
    f = _f(fam, n, q, rng)
    h0 = _h0(h0_kind, n, q, rng)
    a_bar = rng.integers(0, min(q, 2**62), (n, p.m_bar)).tolist()
    r_mat = O.sample_pm_one_zero(rng, p.m_bar, p.n * p.k)
    a = O.gen_trapdoor(p, a_bar, h0, r_mat)
    g = np.array(O.gen_gadget_mat(p.n, p.k, p.base), dtype=object)
    h0o = np.array(h0, dtype=object)
    checked = 0
    for _ in range(40):
        if checked == 3:
            break
        h = _rand(n, q, rng)
        hm = rot_f(h, f, q)
        # f_a: every tag, units or not
        a_t = O.gen_trapdoor(p, a_bar, hm, r_mat)
        sigma = [int(x) for x in rng.integers(-(2**31) + 1, 2**31, p.m)]
        y = [int(x) for x in g.dot(np.array(sigma[p.m_bar:], dtype=object)) % q]
        hy = [int(x) for x in h0o.dot(np.array(y, dtype=object)) % q]
        got = [(u + w - z) % q for u, w, z in zip(O.f_a_classical(a, sigma, q), poly_mulmod(h, y, f, q), hy)]
        assert got == O.f_a_classical(a_t, sigma, q)
        # samp_p syndrome
        try:
            s = poly_inverse_mod(h, f, q)
        except ValueError:
            continue
        v = _rand(n, q, rng)
        w = [(x + z) % q for x, z in zip(v, hy)]
        want = [(x - z) % q for x, z in zip(np.array(O.mat_inverse_mod(hm, q), dtype=object).dot(w) % q, y)]
        assert [(x - z) % q for x, z in zip(poly_mulmod(s, w, f, q), y)] == [int(x) for x in want]
        checked += 1
    assert checked == 3


@pytest.mark.parametrize("q,pe", [(4093, (4093, 1)), (2**32 - 5, (2**32 - 5, 1)), (2**61 - 1, (2**61 - 1, 1)),
                                  (2**16, (2, 16)), (2**32, (2, 32)), (3**10, (3, 10)), (2**48, (2, 48)), (4, (2, 2)),
                                  (4095, None), (2**62 - 1, None), (2**24 * 3, None), (6, None)])
def test_prime_power(q, pe):
    """The samp_p table in polynomial form needs q = p^e; these are the moduli the device accepts and refuses."""
    assert prime_power(q) == pe
