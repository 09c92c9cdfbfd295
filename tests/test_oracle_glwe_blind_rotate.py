"""Pins the blind-rotation reference of tests/glwe_blind_rotate_ref.py on the CPU, three ways:

(a) meaning: with noise-free GGSW(0) / GGSW(1) selectors (test_oracle_cmux.noiseless_ggsw) for the bits of m and a noise-free `a`, the
    phase of the result is the phase of a X^(step m).  Exactly, at res.size * base2k bits, when no limb is truncated (a.size = res.size =
    dnum = s.size); within n_bits times the rounding the CMux test allows per CMux otherwise;
(b) a bit whose rotation p_i = step 2^i is 0 mod 2n leaves a normalised accumulator unchanged, whatever its selector;
(c) one bit is one glwe_cmux with t = X^step a (the rotation restated in numpy)."""
import numpy as np
import pytest

import cmux_ref as CR
import glwe_blind_rotate_ref as BR
import semantics_circuit as SC
from oracle import pyoracle as O
from test_oracle_cmux import centred_diff, noiseless_ggsw, prep
from util import fill_uniform


def rotate_ints(v, p, n):
    """The integers of a polynomial times X^p modulo X^n + 1."""
    out = [0] * n
    for i, x in enumerate(v):
        j = (i + p) % (2 * n)
        if j < n:
            out[j] = x
        else:
            out[j - n] = -x
    return out


def rotate_np(a, p):
    """X^p a on every limb and column of a (size, cols, n) array, negacyclic, in numpy."""
    n = a.shape[-1]
    p %= 2 * n
    r = np.roll(a, p % n, axis=-1)
    sign = np.where(np.arange(n) < p % n, -1, 1) * (-1 if p >= n else 1)
    return (r * sign).astype(np.int64)


# n, rank, k, res_size, a_size, dnum, s_size
SHAPES_EXACT = [(64, 1, 12, 2, 2, 2, 2), (64, 2, 13, 3, 3, 3, 3), (128, 1, 18, 1, 1, 1, 1)]
SHAPES_ROUNDED = [(64, 1, 12, 2, 3, 2, 3), (64, 2, 13, 2, 2, 3, 4), (128, 1, 12, 3, 4, 3, 4)]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", SHAPES_EXACT + SHAPES_ROUNDED)
@pytest.mark.parametrize("step_kind", ["1", "-1", "3", "-n4"])
def test_blind_rotate_rotates_by_the_encrypted_integer(fl, shape, step_kind):
    n, rank, k, rs, as_, dnum, ss = shape
    step = {"1": 1, "-1": -1, "3": 3, "-n4": -(n // 4)}[step_kind]
    rng = np.random.default_rng(sum(shape) + 100 * fl + 7 * (step % 97))
    o = O.OracleModule(n, fl)
    s = [rng.integers(-1, 2, size=n).astype(np.int64) for _ in range(rank)]
    am = rng.integers(-8, 8, size=n)
    a = SC.noiseless_row(rng, {0: am << (k - 4)}, s, k, as_)
    ggsw = [prep(o, noiseless_ggsw(rng, bit, s, k, dnum, ss)) for bit in (0, 1)]
    exact = shape in SHAPES_EXACT
    shift = (as_ - rs) * k  # a's phase at res.size * k bits
    base = [(w >> shift) if shift >= 0 else (w << -shift) for w in SC.phase_scaled(a, s, k)]
    for n_bits, m in [(1, 1), (3, 5), (5, 22), (8, 0), (8, 201), (8, 255)]:
        bits = [(m >> i) & 1 for i in range(n_bits)]
        res = np.zeros((rs, rank + 1, n), dtype=np.int64)
        BR.glwe_blind_rotate_ggsw(o, res, a, k, step, [ggsw[b] for b in bits], k)
        want = rotate_ints(base, step * m, n)
        tol = 0 if exact else n_bits * 2 * (1 + rank * n)
        err = centred_diff(SC.phase_scaled(res, s, k), want, rs * k)
        assert err <= tol, (n_bits, m, err, tol)
        assert tol < 1 << (rs * k - 4 - 5)  # 2^5 below the lowest message bit


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", [(64, 1, 12, 2, 3, 2, 2), (64, 2, 13, 3, 2, 2, 4), (128, 1, 18, 2, 2, 3, 2)])
def test_bits_rotating_by_a_multiple_of_2n_leave_the_accumulator_unchanged(fl, shape):
    n, rank, k, rs, as_, dnum, ss = shape
    cols = rank + 1
    rng = np.random.default_rng(sum(shape) + 11 * fl)
    o = O.OracleModule(n, fl)
    a = fill_uniform(rng, (as_, cols, n), 40)
    sels = [prep(o, fill_uniform(rng, (dnum, cols, ss, cols, n), k)) for _ in range(4)]
    # every p_i = 0: res = normalize(a) on a's first res.size limbs (the CMux of equal inputs), for 2n and for the extreme int64 steps
    want = np.zeros((rs, cols, n), dtype=np.int64)
    c = min(rs, as_)
    want[:c] = a[:c]
    for col in range(cols):
        O.vec_znx_normalize_assign(k, want, col)
    for step in (2 * n, -6 * n, -(1 << 63), 1 << 62):
        res = np.zeros((rs, cols, n), dtype=np.int64)
        BR.glwe_blind_rotate_ggsw(o, res, a, k, step, sels, k)
        assert np.array_equal(res, want), step
    # step = n: only bit 0 rotates; the bits after it see a normalised accumulator and a rotation by 0
    one = np.zeros((rs, cols, n), dtype=np.int64)
    BR.glwe_blind_rotate_ggsw(o, one, a, k, n, sels[:1], k)
    res = np.zeros((rs, cols, n), dtype=np.int64)
    BR.glwe_blind_rotate_ggsw(o, res, a, k, n, sels, k)
    assert np.array_equal(res, one)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", [(64, 1, 12, 2, 3, 2, 2, 1, 12, 5), (64, 2, 13, 3, 2, 2, 4, 2, 13, -7), (128, 1, 13, 2, 2, 3, 3, 1, 17, 131)])
def test_one_bit_is_one_cmux_of_the_rotated_input(fl, shape):
    n, rank, k, rs, as_, dnum, ss, dsize, gk, step = shape
    cols = rank + 1
    rng = np.random.default_rng(sum(map(abs, shape)) + 13 * fl)
    o = O.OracleModule(n, fl)
    a = fill_uniform(rng, (as_, cols, n), k + 6)
    sel = prep(o, fill_uniform(rng, (dnum, cols, ss, cols, n), gk))
    res = np.zeros((rs, cols, n), dtype=np.int64)
    BR.glwe_blind_rotate_ggsw(o, res, a, k, step, [sel], gk, dsize)
    want = np.zeros((rs, cols, n), dtype=np.int64)
    CR.glwe_cmux(o, want, rotate_np(a, step), a, k, sel, gk, dsize)
    assert np.array_equal(res, want)
