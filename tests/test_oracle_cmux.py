"""Pins the CMux reference of tests/cmux_ref.py on the CPU, three ways:

(a) meaning: with noise-free GGSW(0) / GGSW(1) (semantics_circuit.noiseless_row) and noise-free t, f the phase of the result is the phase of
    f / t.  Exactly, at res.size * base2k bits, when no limb is truncated (t.size = f.size = res.size = dnum = s.size); within the rounding
    of the truncated limbs otherwise;
(b) t == f gives normalize(f) on f's first res.size limbs, whatever the selector;
(c) the reference equals a restatement of steps 1, 2, 4 and 5 on Python integers (balanced base-2^base2k expansions) around the oracle's
    external product."""
import numpy as np
import pytest

import cmux_ref as CR
import semantics_circuit as SC
from oracle import pyoracle as O
from util import fill_uniform


def prep(o, mat):
    d, ci, sz, co, _ = mat.shape
    pm = o.vmp_pmat_alloc(d, ci, co, sz)
    o.vmp_prepare(pm, mat)
    return pm


def noiseless_ggsw(rng, m, s, k, dnum, size):
    """GGSW(m), m a small integer: row d, column 0 has phase m 2^-(d+1)k, column c >= 1 phase m s_{c-1} 2^-(d+1)k, zero noise."""
    cols, n = len(s) + 1, len(s[0])
    mat = np.zeros((dnum, cols, size, cols, n), dtype=np.int64)
    one = np.zeros(n, dtype=np.int64)
    one[0] = m
    for d in range(dnum):
        for c in range(cols):
            mat[d, c] = SC.noiseless_row(rng, {d: one if c == 0 else s[c - 1] * m}, s, k, size)
    return mat


def centred_diff(a, b, bits):
    mod = 1 << bits
    return max(abs(((x - y + (mod >> 1)) % mod) - (mod >> 1)) for x, y in zip(a, b))


# n, rank, k, res_size, t_size, f_size, dnum, s_size
SHAPES_EXACT = [(64, 1, 12, 2, 2, 2, 2, 2), (64, 2, 13, 3, 3, 3, 3, 3), (128, 1, 18, 1, 1, 1, 1, 1), (128, 2, 10, 4, 4, 4, 4, 4)]
SHAPES_ROUNDED = [(64, 1, 12, 2, 3, 3, 2, 3), (64, 2, 13, 2, 4, 2, 3, 4), (128, 1, 12, 3, 2, 4, 3, 4), (64, 2, 12, 2, 2, 1, 2, 3)]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", SHAPES_EXACT + SHAPES_ROUNDED)
def test_cmux_selects_by_the_ggsw_bit(fl, shape):
    n, rank, k, rs, ts, fs, dnum, ss = shape
    rng = np.random.default_rng(sum(shape) + 100 * fl)
    o = O.OracleModule(n, fl)
    s = [rng.integers(-1, 2, size=n).astype(np.int64) for _ in range(rank)]
    tm, fm = rng.integers(-8, 8, size=n), rng.integers(-8, 8, size=n)
    # messages in the top limb, 4 bits below its top: phase m 2^(size k - 4) units at size * k bits
    t = SC.noiseless_row(rng, {0: tm << (k - 4)}, s, k, ts)
    f = SC.noiseless_row(rng, {0: fm << (k - 4)}, s, k, fs)
    exact = shape in SHAPES_EXACT
    # rounding of the truncated limbs, in units of 2^-(rs k): at most 1/2 (1 + rank n) each for t and f beyond res.size and for the
    # product's limbs beyond res.size (a ternary secret multiplies every coefficient's error)
    tol = 0 if exact else 2 * (1 + rank * n)
    for bit in (0, 1):
        pm = prep(o, noiseless_ggsw(rng, bit, s, k, dnum, ss))
        res = np.zeros((rs, rank + 1, n), dtype=np.int64)
        CR.glwe_cmux(o, res, t, f, k, pm, k)
        sel = t if bit else f
        want = SC.phase_scaled(sel, s, k)
        shift = (sel.shape[0] - rs) * k  # the selected phase at res.size * k bits
        want = [(w >> shift) if shift >= 0 else (w << -shift) for w in want]
        got = SC.phase_scaled(res, s, k)
        err = centred_diff(got, want, rs * k)
        assert err <= tol, (bit, err, tol)
        if not exact:
            assert tol < 1 << (rs * k - 4 - 5)  # 2^5 below the lowest message bit


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", [(64, 1, 12, 2, 3, 2, 2), (64, 2, 13, 3, 3, 2, 4), (128, 1, 18, 1, 2, 3, 1)])
def test_cmux_of_equal_inputs_is_normalised_f(fl, shape):
    n, rank, k, rs, fs, dnum, ss = shape
    rng = np.random.default_rng(sum(shape) + 7 * fl)
    o = O.OracleModule(n, fl)
    f = fill_uniform(rng, (fs, rank + 1, n), 40)
    pm = prep(o, fill_uniform(rng, (dnum, rank + 1, ss, rank + 1, n), k))
    res = np.zeros((rs, rank + 1, n), dtype=np.int64)
    CR.glwe_cmux(o, res, f.copy(), f, k, pm, k)
    want = np.zeros_like(res)
    c = min(rs, fs)
    want[:c] = f[:c]
    for col in range(rank + 1):
        O.vec_znx_normalize_assign(k, want, col)
    assert np.array_equal(res, want)


def balanced(vals, k, size):
    """Python ints -> (size, n) balanced base-2^k digits of each value modulo 2^(size k)."""
    out = np.zeros((size, len(vals)), dtype=np.int64)
    for i, v in enumerate(vals):
        v %= 1 << (size * k)
        for j in range(size - 1, -1, -1):
            dg = v & ((1 << k) - 1)
            if dg >= 1 << (k - 1):
                dg -= 1 << k
            out[j, i] = dg
            v = (v - dg) >> k
    return out


def as_int(limbs, k):
    """(size, n) digits -> the integers sum_j limbs[j] 2^((size-1-j) k)."""
    size, n = limbs.shape
    return [sum(int(limbs[j, i]) << ((size - 1 - j) * k) for j in range(size)) for i in range(n)]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", [(64, 1, 12, 2, 3, 1, 2, 2, 1, 12), (64, 2, 13, 3, 2, 3, 2, 4, 1, 13), (128, 1, 18, 3, 3, 2, 3, 2, 2, 18),
                                   (64, 1, 13, 2, 2, 2, 2, 3, 1, 17)])
def test_cmux_reference_equals_integer_restatement(fl, shape):
    n, rank, k, rs, ts, fs, dnum, ss, dsize, gk = shape
    cols = rank + 1
    rng = np.random.default_rng(sum(shape) + 31 * fl)
    o = O.OracleModule(n, fl)
    t, f = fill_uniform(rng, (ts, cols, n), k + 6), fill_uniform(rng, (fs, cols, n), k + 6)
    pm = prep(o, fill_uniform(rng, (dnum, cols, ss, cols, n), gk))
    res = np.zeros((rs, cols, n), dtype=np.int64)
    CR.glwe_cmux(o, res, t, f, k, pm, gk, dsize)

    def pad(x):
        y = np.zeros((rs, cols, n), dtype=np.int64)
        c = min(rs, x.shape[0])
        y[:c] = x[:c]
        return y

    tp, fp = pad(t), pad(f)
    d = np.zeros((rs, cols, n), dtype=np.int64)
    for c in range(cols):  # steps 1 + 2: the balanced expansion of (t - f) as an integer modulo 2^(rs k)
        d[:, c] = balanced([a - b for a, b in zip(as_int(tp[:, c], k), as_int(fp[:, c], k))], k, rs)
    e = np.zeros((rs, cols, n), dtype=np.int64)
    o.glwe_external_product(e, k, d, k, pm, gk, dsize)
    want = np.zeros_like(e)
    for c in range(cols):  # steps 4 + 5
        want[:, c] = balanced([a + b for a, b in zip(as_int(e[:, c], k), as_int(fp[:, c], k))], k, rs)
    assert np.array_equal(res, want)
