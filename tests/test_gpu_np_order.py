"""Order of the tensor-core nearest-plane updates inside a 4096-block (np_block, DESIGN.md 4.3): left-looking (the
default: one launch per 256-block applies everything pending from the finished coordinates of its 4096-block) against
right-looking (QF_NP_ORDER=right: launches after every finished 256- and 1024-block).

The CPU tests run a numpy model of the block schedule: the same partition (ragged tops merged into the block below), every
update inside one scale block and on digitised entries of U, the same entries of U read by both orders, and, in exact
integer arithmetic, both orders equal to the unblocked loop.  The GPU tests compare the two orders on the same key, seed
and targets: both exact (A e = u, check_domain) and nearly all rows bit-identical -- the digit sums of an update are the
same integers, only the fp64 roundings of T -= V * scale are grouped differently."""
import math

import numpy as np
import pytest

from oracle import qfall_oracle as O

# ---------------------------------------------------------------------------------------------------------------------
# numpy model of np_block (tools_b200/csrc/api.cu) at tensor-core dimensions
# ---------------------------------------------------------------------------------------------------------------------
NP_SIZES = (64, 256, 1024, 4096)
NP_TOP = 4
NP_THIN = 512
NP_SCALE_BLOCK = NP_SIZES[3]


def last_block_start(D, S):
    top = (D - 1) // S * S
    if top > 0 and D - top < NP_THIN:
        top -= S
    return top


def block_index(col, D, S):
    return min(col, last_block_start(D, S)) // S


def schedule(D, lo, hi, right):
    """Launch sequence of np_block(lo, hi, NP_TOP): ("diag", lo, hi) samples one 256-block (its own rank-64 updates
    included); ("upd", r0, r1, c0, c1, level) is T[:, r0:r1] -= Z[:, c0:c1] U[r0:r1, c0:c1]^t."""
    ops = []

    def rec(lo, hi, level, q_hi):
        if level == 1:
            ops.append(("diag", lo, hi))
            return
        step = NP_SIZES[level - 1]
        sub_hi = hi
        while sub_hi > lo:
            sub_lo = max(lo, (sub_hi - 1) // step * step)
            if sub_hi == D and sub_lo > lo and sub_hi - sub_lo < NP_THIN:
                sub_lo = max(lo, sub_lo - step)
            if not right and level == 2 and sub_hi < q_hi:
                ops.append(("upd", sub_lo, sub_hi, sub_hi, q_hi, level))
            rec(sub_lo, sub_hi, level - 1, sub_hi if level == NP_TOP else q_hi)
            if sub_lo > lo and (level == NP_TOP or right):
                ops.append(("upd", lo, sub_lo, sub_lo, sub_hi, level))
            sub_hi = sub_lo

    rec(lo, hi, NP_TOP, hi)
    return ops


# (D, phases): C2 two-phase (m = 12352, nk = 6144), the same dimension in one pass, the n = 128 two-phase key of the GPU
# tests (m = 6193, nk = 3072), C3 ring (D = 3584), the shapes of test_gpv_tensor_core_updates_match_fp64_path, and a top
# that is ragged at every level with a 300-wide merged top 256-block
CASES = [
    (12352, [(6144, 12352), (0, 6144)]),
    (12352, [(0, 12352)]),
    (6193, [(3072, 6193), (0, 3072)]),
    (3584, [(0, 3584)]),
    (2084, [(0, 2084)]),
    (3121, [(0, 3121)]),
    (12588, [(0, 12588)]),
]


def _digitised(D, split, i, j):
    """ozaki_digits_kernel (setup.cu): U[i][j] has fixed-point digits."""
    return i < min(j // NP_SIZES[1] * NP_SIZES[1], last_block_start(D, NP_SIZES[1])) and not (i < split <= j)


@pytest.mark.parametrize("D,phases", CASES)
def test_schedule_blocks_and_scales(D, phases):
    split = phases[0][0]
    for right in (False, True):
        for lo, hi in phases:
            ops = schedule(D, lo, hi, right)
            diags = [(a, b) for k, a, b, *_ in ops if k == "diag"]
            # the diagonal blocks tile [lo, hi) in descending order, with the same partition in both orders
            assert diags[0][1] == hi and diags[-1][0] == lo
            assert all(diags[i][0] == diags[i + 1][1] for i in range(len(diags) - 1))
            assert diags == [(a, b) for k, a, b, *_ in schedule(D, lo, hi, not right) if k == "diag"]
            for _, r0, r1, c0, c1, _ in (op for op in ops if op[0] == "upd"):
                assert lo <= r0 < r1 <= c0 < c1 <= hi
                # one scale per row: the K range lies in one column block of the scale partition
                assert block_index(c0, D, NP_SCALE_BLOCK) == block_index(c1 - 1, D, NP_SCALE_BLOCK)
                if c1 - c0 >= NP_SIZES[1]:  # tensor cores: 128-aligned K offset (zero-tile map), entries with digits
                    assert c0 % 128 == 0
                    assert _digitised(D, split, r1 - 1, c0) and _digitised(D, split, r0, c1 - 1)
                    assert c1 - c0 < 2**13  # int32 digit sums (np_update)


def _row_intervals(D, ops):
    rows = [[] for _ in range(D)]
    for _, r0, r1, c0, c1, _ in (op for op in ops if op[0] == "upd"):
        for i in range(r0, r1):
            rows[i].append((c0, c1))
    out = []
    for iv in rows:
        iv.sort()
        assert all(iv[t][1] <= iv[t + 1][0] for t in range(len(iv) - 1)), "an entry of U read twice"
        merged = []
        for a, b in iv:
            if merged and merged[-1][1] == a:
                merged[-1] = (merged[-1][0], b)
            else:
                merged.append((a, b))
        out.append(merged)
    return out


@pytest.mark.parametrize("D,phases", CASES)
def test_schedule_reads_the_same_entries_of_u(D, phases):
    for lo, hi in phases:
        left, right = schedule(D, lo, hi, False), schedule(D, lo, hi, True)
        assert _row_intervals(D, left) == _row_intervals(D, right)
        # left-looking: inside its 4096-block a row is updated by one launch at most (plus the 4096-level launches)
        inner = [op for op in left if op[0] == "upd" and op[5] < NP_TOP]
        per_row = np.zeros(D, dtype=np.int64)
        for _, r0, r1, *_ in inner:
            per_row[r0:r1] += 1
        assert per_row.max() <= 1
        passes = lambda ops: sum(op[2] - op[1] for op in ops if op[0] == "upd" and op[5] < NP_TOP)
        assert passes(left) < passes(right) or passes(right) == 0


def _run_model(D, phases, right, U, c, noise):
    """The schedule in exact integers: z_i = ((T_i mod 7) - 3) + noise_i depends on the whole centre T_i."""
    T = c.copy()
    z = np.zeros(D, dtype=np.int64)
    for lo, hi in phases:
        for op in schedule(D, lo, hi, right):
            if op[0] == "diag":
                _, a, b = op
                for i in range(b - 1, a - 1, -1):
                    z[i] = T[i] % 7 - 3 + noise[i]
                    T[a:i] -= U[a:i, i].astype(np.int64) * z[i]
            else:
                _, r0, r1, c0, c1, _ = op
                T[r0:r1] -= U[r0:r1, c0:c1].astype(np.int64) @ z[c0:c1]
    return T, z


@pytest.mark.parametrize("D,phases", CASES[2:6])
def test_schedule_exact_integers_match_unblocked_loop(D, phases):
    rng = np.random.default_rng(D)
    U = np.triu(rng.integers(-3, 4, (D, D), dtype=np.int8), 1)
    c = rng.integers(-1000, 1000, D, dtype=np.int64)
    noise = rng.integers(-2, 3, D, dtype=np.int64)
    # the reference loop, i = hi - 1 .. lo inside each phase
    T = c.copy()
    z = np.zeros(D, dtype=np.int64)
    for lo, hi in phases:
        for i in range(hi - 1, lo - 1, -1):
            z[i] = T[i] % 7 - 3 + noise[i]
            T[lo:i] -= U[lo:i, i].astype(np.int64) * z[i]
    for right in (False, True):
        Tb, zb = _run_model(D, phases, right, U, c, noise)
        assert np.array_equal(zb, z) and np.array_equal(Tb, T), right


# ---------------------------------------------------------------------------------------------------------------------
# both orders on the GPU
# ---------------------------------------------------------------------------------------------------------------------
MIN_SAME = 0.999


@pytest.fixture(scope="module")
def T():
    import tools_b200

    return tools_b200


def _gpv_s(gp):
    return float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(gp.n)))


def _order(monkeypatch, order):
    """QF_NP_ORDER for the contexts created next (read when a context is created)."""
    if order == "left":
        monkeypatch.delenv("QF_NP_ORDER", raising=False)
    else:
        monkeypatch.setenv("QF_NP_ORDER", order)


def _check_gpv(psf, a, e, u, q):
    got, ok = psf.f_a_batch(a, e, strict=False)
    assert np.array_equal(got, u) and ok.all()
    assert np.array_equal(O.f_a_classical_batch(a, e[:3], q), u[:3])
    assert psf.check_domain_batch(e).all()


def _same(name, e_left, e_right):
    same = (e_left == e_right).reshape(len(e_left), -1).all(axis=1).mean()
    print(f"{name}: {same:.5f} of {len(e_left)} rows bit-identical between the two orders")
    assert same >= MIN_SAME, (name, same)


@pytest.mark.gpu
def test_two_phase_orders_and_offline_online(T, monkeypatch):
    """n = 128, q = 2^24 (m = 6193, nk = 3072): phase 1 covers two 4096-level blocks, the top one ragged at every level
    (305-wide top 256-block, 1073-wide top 1024-block); phase 2 shares the digit-count gate slot of [0, 4096) with phase 1.
    Offline + online stays bit-identical to direct samp_p in the default order."""
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    monkeypatch.delenv("QF_DISABLE_OZAKI", raising=False)
    n, q = 128, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(5)
    u = rng.integers(0, q, (8192, n), dtype=np.int64)
    outs, key = {}, None
    for order in ("left", "right"):
        _order(monkeypatch, order)
        psf = T.PSFGPV(gp, s)
        if key is None:
            key = psf.trap_gen(seed=13, dense_gso=False)
        a, td = key
        e = psf.samp_p_batch(a, td, u, seed=21, first_index=3)
        _check_gpv(psf, a, e, u, q)
        outs[order] = e
        if order == "left":
            psf.samp_p_offline(a, td, 3000, seed=21, first_index=3)
            e_on, first = psf.samp_p_online_batch(a, td, u[:3000])
            assert first == 3 and np.array_equal(e_on, e[:3000])
        psf.ctx.close()
    _same("two-phase n=128", outs["left"], outs["right"])


@pytest.mark.gpu
def test_tagged_two_phase_orders(T, monkeypatch):
    monkeypatch.delenv("QF_DISABLE_TWO_PHASE", raising=False)
    monkeypatch.delenv("QF_DISABLE_OZAKI", raising=False)
    n, q = 128, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(6)
    tag = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)
    u = rng.integers(0, q, (4096, n), dtype=np.int64)
    outs, key = {}, None
    for order in ("left", "right"):
        _order(monkeypatch, order)
        psf = T.PSFGPV(gp, s)
        if key is None:
            key = psf.trap_gen(seed=17, tag=tag, dense_gso=False)
        a, td = key
        e = psf.samp_p_batch(a, td, u, seed=8)
        _check_gpv(psf, a, e, u, q)
        outs[order] = e
        psf.ctx.close()
    _same("tagged two-phase n=128", outs["left"], outs["right"])


@pytest.mark.gpu
def test_one_pass_dense_basis_orders(T, monkeypatch):
    """A short basis that is not of the G-trapdoor form (two columns swapped): the one-pass recursion over the whole
    m = 6193, two 4096-level blocks."""
    monkeypatch.delenv("QF_DISABLE_OZAKI", raising=False)
    n, q = 128, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = _gpv_s(gp)
    rng = np.random.default_rng(7)
    u = rng.integers(0, q, (4096, n), dtype=np.int64)
    outs, key = {}, None
    for order in ("left", "right"):
        _order(monkeypatch, order)
        psf = T.PSFGPV(gp, s)
        if key is None:
            a, (sb, _) = psf.trap_gen(seed=19, dense_gso=False)
            sb = sb.copy()
            sb[:, [0, 1]] = sb[:, [1, 0]]
            key = (a, (sb, None))
        a, td = key
        e = psf.samp_p_batch(a, td, u, seed=9)
        _check_gpv(psf, a, e, u, q)
        outs[order] = e
        psf.ctx.close()
    _same("one-pass dense basis n=128", outs["left"], outs["right"])


@pytest.mark.gpu
def test_ring_orders(T, monkeypatch):
    """C3 shape: PSFGPVRing over X^256 + 1 mod 3329 (D = 3584: one 4096-level block of three 1024-blocks and a 512-wide
    one), the one-pass recursion."""
    monkeypatch.delenv("QF_DISABLE_OZAKI", raising=False)
    n, q = 256, 3329
    gp = T.GadgetParametersRing.init_default(n, q)
    s = ((2 * 2 * 1.005 * np.sqrt(n) + 1) * 2) * 4  # gpv_ring.rs:296-298
    rng = np.random.default_rng(8)
    u = rng.integers(0, q, (4096, n), dtype=np.int64)
    outs, key = {}, None
    for order in ("left", "right"):
        _order(monkeypatch, order)
        psf = T.PSFGPVRing(gp, float(s), 1.005)
        if key is None:
            key = psf.trap_gen(seed=23)
        a, td = key
        e = psf.samp_p_batch(a, td, u, seed=10)
        got, ok = psf.f_a_batch(a, e, strict=False)
        assert np.array_equal(got, u) and ok.all()
        assert O.f_a_ring(a.tolist(), e[0].tolist(), n, q) == u[0].tolist()
        outs[order] = e
        psf.ctx.close()
    _same("ring n=256", outs["left"], outs["right"])
