"""CPU checks of the packed Domain code (DESIGN 4.11): a numpy reference encoder / decoder of the format in
include/qfall_b200.h, its round trips, lengths and canonical rejections, and the rule of qf_domain_code_params.
The GPU tests compare the kernels with this reference (test_gpu_domain_code.py)."""
import math

import numpy as np
import pytest

INT32_MIN, INT32_MAX = -(2**31), 2**31 - 1


def h0_bytes(dim, k):
    return 16 * (-(-dim * (k + 1) // 128))


def ref_encode(x, k, slot_bytes):
    """One row -> (slot bytes, nbytes); (zeros, -1) when the code does not fit or the row holds INT32_MIN."""
    x = [int(v) for v in x]
    dim = len(x)
    h0 = h0_bytes(dim, k)
    bits = np.zeros(8 * slot_bytes, dtype=np.uint8)
    if any(v == INT32_MIN for v in x):
        return np.zeros(slot_bytes, np.uint8), -1
    pos = 8 * h0
    for i, v in enumerate(x):
        a = abs(v)
        f = (a & ((1 << k) - 1)) | (int(v < 0) << k)
        for j in range(k + 1):
            bits[i * (k + 1) + j] = (f >> j) & 1
        pos += a >> k
        if pos >= 8 * slot_bytes:
            return np.zeros(slot_bytes, np.uint8), -1
        bits[pos] = 1
        pos += 1
    return np.packbits(bits, bitorder="little"), h0 + -(-(pos - 8 * h0) // 8)


def ref_decode(slot, dim, k):
    """slot bytes -> (row, ok); ok False for every non-canonical slot."""
    bits = np.unpackbits(np.asarray(slot, np.uint8), bitorder="little")
    h0 = h0_bytes(dim, k)
    if bits[dim * (k + 1): 8 * h0].any():
        return None, False
    ones = np.flatnonzero(bits[8 * h0:])
    if len(ones) < dim or len(ones) > dim:  # fewer terminators, or a 1 bit after the dim-th (tail not zero)
        return None, False
    out, prev = [], -1
    for i in range(dim):
        h = int(ones[i]) - prev - 1
        prev = int(ones[i])
        f = 0
        for j in range(k + 1):
            f |= int(bits[i * (k + 1) + j]) << j
        mag, sign = (h << k) | (f & ((1 << k) - 1)), f >> k
        if mag > INT32_MAX or (sign and mag == 0):
            return None, False
        out.append(-mag if sign else mag)
    return np.array(out, dtype=np.int64), True


def code_params(w, dim):
    """qf_domain_code_params restated: k minimising E[k + 2 + h] over D_{Z,w} (|x| <= 20 w), and the slot of
    H0 + ceil((dim E[h+1] + 12 sqrt(dim Var[h+1])) / 8) rounded up to 16.  Returns (k, slot, bits per entry)."""
    a = np.arange(int(math.floor(20 * w)) + 1, dtype=np.int64)
    p = np.exp(-math.pi * (a / w) ** 2)
    p[1:] *= 2
    p /= p.sum()
    best = None
    for k in range(31):
        h = (a >> k).astype(np.float64)
        eh = float((p * h).sum())
        var = float((p * h * h).sum()) - eh * eh
        if best is None or k + 2 + eh < best[0]:
            best = (k + 2 + eh, k, eh, var)
    bits, k, eh, var = best
    slot = h0_bytes(dim, k) + math.ceil((dim * (eh + 1) + 12 * math.sqrt(dim * var)) / 8)
    return k, -(-slot // 16) * 16, bits


def _min_slot(dim, k):
    return -(-(h0_bytes(dim, k) + -(-dim // 8)) // 16) * 16


@pytest.mark.parametrize("k", [0, 1, 4, 8, 13, 30])
def test_round_trip_random_and_extremes(k):
    rng = np.random.default_rng(k)
    dim = 105
    ext = [0, 1, -1, (1 << k) - 1, -((1 << k) - 1), 1 << k, -(1 << k)]
    if k >= 20:  # at smaller k, h of +-(2^31 - 1) alone takes more than 2^11 bits
        ext += [INT32_MAX, -INT32_MAX]
    rows = [np.array((ext * dim)[:dim]), rng.integers(-3000, 3001, dim), np.zeros(dim, np.int64)]
    for x in rows:
        need = h0_bytes(dim, k) + -(-sum((abs(int(v)) >> k) + 1 for v in x) // 8)
        slot = -(-need // 16) * 16 + 16
        enc, nb = ref_encode(x, k, slot)
        assert nb == need  # nbytes = H0 + ceil(sum (h_i + 1) / 8)
        assert not enc[nb:].any()
        dec, ok = ref_decode(enc, dim, k)
        assert ok and np.array_equal(dec, x)
        # keeping only nbytes bytes and padding with zeros reads the row back
        pad = np.zeros(slot, np.uint8)
        pad[:nb] = enc[:nb]
        assert np.array_equal(pad, enc)


def test_int32_min_overflows():
    x = np.zeros(40, np.int64)
    x[7] = INT32_MIN
    enc, nb = ref_encode(x, 8, 256)
    assert nb == -1 and not enc.any()


def test_exact_fit_and_one_bit_over():
    dim, k = 105, 3
    slot = _min_slot(dim, k) + 16
    budget = 8 * (slot - h0_bytes(dim, k))  # high-stream bits
    x = np.zeros(dim, np.int64)
    x[0] = (budget - dim) << k  # h_0 + 1 + (dim - 1) = budget: the last terminator is the last bit of the slot
    enc, nb = ref_encode(x, k, slot)
    assert nb == slot
    assert ref_decode(enc, dim, k)[1]
    x[0] += 1 << k
    assert ref_encode(x, k, slot)[1] == -1


def _valid(dim=50, k=4, seed=0):
    x = np.random.default_rng(seed).integers(-200, 201, dim)
    x[x == 0] = 1
    slot = _min_slot(dim, k) + 64
    enc, nb = ref_encode(x, k, slot)
    assert nb > 0
    return x, enc, slot


def test_reject_negative_zero():
    dim, k = 50, 4
    x, enc, _ = _valid(dim, k)
    x2 = x.copy()
    x2[3] = 0
    e2, _ = ref_encode(x2, k, len(enc))
    bits = np.unpackbits(e2, bitorder="little")
    bits[3 * (k + 1) + k] = 1  # sign of a zero entry
    assert not ref_decode(np.packbits(bits, bitorder="little"), dim, k)[1]


def test_reject_missing_terminator():
    dim, k = 50, 4
    x, enc, _ = _valid(dim, k)
    bits = np.unpackbits(enc, bitorder="little")
    last = np.flatnonzero(bits)[-1]
    bits[last] = 0
    assert not ref_decode(np.packbits(bits, bitorder="little"), dim, k)[1]


def test_reject_padding_bits():
    dim, k = 50, 4  # dim (k + 1) = 250 bits, H0 = 32 bytes: fixed padding bits 250 .. 255
    x, enc, slot = _valid(dim, k)
    bits = np.unpackbits(enc, bitorder="little")
    b1 = bits.copy()
    b1[dim * (k + 1)] = 1
    assert not ref_decode(np.packbits(b1, bitorder="little"), dim, k)[1]
    b2 = bits.copy()
    b2[-1] = 1  # the tail after the dim-th terminator
    assert not ref_decode(np.packbits(b2, bitorder="little"), dim, k)[1]


def test_reject_magnitude_above_int32():
    dim, k = 1, 30
    slot = _min_slot(dim, k)
    enc, nb = ref_encode([INT32_MAX], k, slot)  # h = 1, low = 2^30 - 1
    assert ref_decode(enc, dim, k)[1]
    bits = np.unpackbits(enc, bitorder="little")
    h0 = h0_bytes(dim, k)
    assert bits[8 * h0: 8 * h0 + 2].tolist() == [0, 1]
    bits[8 * h0 + 1], bits[8 * h0 + 2] = 0, 1  # h = 2: magnitude 2^31 + 2^30 - 1
    assert not ref_decode(np.packbits(bits, bitorder="little"), dim, k)[1]


@pytest.mark.parametrize("name,w,dim,k,bits", [
    ("C2", 1428.0, 12352, 8, 11.31), ("C3", 522.6, 3584, 7, 9.84), ("C4", 450.0 * 9, 32849, 10, 12.80), ("C1", 75.0, 105, 4, 7.05)])
def test_code_params_rule(name, w, dim, k, bits):
    kk, slot, b = code_params(w, dim)
    assert kk == k and abs(b - bits) < 0.01
    mean = h0_bytes(dim, k) + dim * (b - k - 1) / 8
    assert slot % 16 == 0 and mean < slot < 1.1 * mean + 32


def ref_encode_batch(x, k, slot_bytes):
    """ref_encode for a batch of rows (B x dim), vectorised: (B x slot_bytes uint8, nbytes int32 B)."""
    x = np.asarray(x, dtype=np.int64)
    B, dim = x.shape
    h0 = h0_bytes(dim, k)
    a = np.abs(x)
    f = (a & ((1 << k) - 1)) | ((x < 0).astype(np.int64) << k)
    h = a >> k
    ends = 8 * h0 + np.cumsum(h + 1, axis=1) - 1  # terminator bit positions
    fits = (ends[:, -1] < 8 * slot_bytes) & ~(x == INT32_MIN).any(axis=1)
    bits = np.zeros((B, 8 * slot_bytes), dtype=np.uint8)
    cols = np.arange(dim) * (k + 1)
    for j in range(k + 1):
        bits[:, cols + j] = (f >> j) & 1
    rows = np.flatnonzero(fits)
    bits[np.repeat(rows, dim), ends[rows].reshape(-1)] = 1
    bits[~fits] = 0
    out = np.packbits(bits, axis=1, bitorder="little")
    nbytes = np.where(fits, h0 + (ends[:, -1] - 8 * h0 + 8) // 8, -1).astype(np.int32)
    return out, nbytes


@pytest.mark.parametrize("k,slot_extra", [(0, 400), (5, 0), (8, 16), (30, 16)])
def test_batch_reference_matches_scalar(k, slot_extra):
    rng = np.random.default_rng(k)
    dim = 77
    x = np.rint(rng.normal(0, 60, (6, dim))).astype(np.int64)
    x[1, 5] = INT32_MIN
    x[2, :] = 0
    slot = _min_slot(dim, k) + slot_extra
    out, nb = ref_encode_batch(x, k, slot)
    for b in range(len(x)):
        e, n = ref_encode(x[b], k, slot)
        assert n == nb[b] and np.array_equal(e, out[b])
