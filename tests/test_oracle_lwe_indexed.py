"""The reference of glwe_to_lwe at many coefficients (tests/lwe_indexed_ref.py), CPU only.

The meaning is pinned independently: with a noise-free GLWE -> LWE key, LWE j decrypts to coefficient index[j] of the input's phase
(exactly when no limb is dropped); index {0} is glwe_to_lwe.  Against the per-bit composition (rotate the input, then a whole
glwe_to_lwe), which the entry replaces: both orders agree as integers modulo 2^(size * base2k) within one unit of the last limb, but not
bit for bit.  A rotation negates wrapped digits without renormalising, so a digit -2^(k-1) at a wrapped position comes out as +2^(k-1)
where the composition's final normalisation holds -2^(k-1) and a carry."""
import numpy as np
import pytest

import lwe_indexed_ref as R
import lwe_ref as L
import semantics as S
from oracle import pyoracle as O
from test_oracle_lwe import _binary, _ternary, _tol, embed_secret, lwe_phase, prep
from test_oracle_semantics import noiseless_ksk
from util import fill_uniform

N = 64


def _indices(rng):
    return [0, 1, N - 1] + [int(x) for x in rng.integers(0, N, size=6)]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("rank", [1, 2])
@pytest.mark.parametrize("n_lwe", [3, 41, N])
def test_noiseless_indexed_lwes_carry_the_indexed_coefficients(fl, rank, n_lwe):
    k, a_size = 12, 3
    key_size = a_size + 1
    rng = np.random.default_rng(1100 + 10 * fl + rank + n_lwe)
    o = O.OracleModule(N, fl)
    s = [_ternary(rng, N) for _ in range(rank)]
    s_lwe = _binary(rng, n_lwe)
    key = prep(o, noiseless_ksk(rng, s, [embed_secret(s_lwe, N)], k, a_size, key_size))
    a = fill_uniform(rng, (a_size, rank + 1, N), k)
    want = S.phase(a.tolist(), s, k)
    index = _indices(rng)
    for res_size in (key_size, a_size):
        res = fill_uniform(rng, (len(index), res_size, 1, n_lwe + 1), k)  # garbage pre-fill: every limb is written
        R.glwe_to_lwe_indexed(o, res, k, a, k, index, key, k)
        for j, idx in enumerate(index):
            err = S.centred_mod1(lwe_phase(res[j], s_lwe, k) - want[idx])
            assert abs(err) <= _tol(res_size, k, res_size == key_size), (res_size, j, idx)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("rank", [1, 2])
def test_index_zero_is_glwe_to_lwe(fl, rank):
    a_k, key_k, res_k, a_size, res_size, n_lwe, dsize = 12, 15, 13, 3, 2, 37, 2
    rng = np.random.default_rng(1200 + fl + rank)
    o = O.OracleModule(N, fl)
    in_size = -(-a_size * a_k // key_k)
    key = prep(o, fill_uniform(rng, (-(-in_size // dsize), rank, in_size + 1, 2, N), key_k))
    a = fill_uniform(rng, (a_size, rank + 1, N), a_k)
    got = np.zeros((1, res_size, 1, n_lwe + 1), dtype=np.int64)
    R.glwe_to_lwe_indexed(o, got, res_k, a, a_k, [0], key, key_k, dsize)
    want = np.zeros((res_size, 1, n_lwe + 1), dtype=np.int64)
    L.glwe_to_lwe(o, want, res_k, a, a_k, key, key_k, dsize)
    assert np.array_equal(got[0], want)


def _value(lwe, k):
    """Every coefficient of an LWE (size, 1, n_lwe + 1) as an integer modulo 2^(size k)."""
    size = lwe.shape[0]
    return [sum(int(lwe[l, 0, t]) << ((size - 1 - l) * k) for l in range(size)) % (1 << (size * k)) for t in range(lwe.shape[2])]


def _max_unit_distance(x, y, k):
    mod = 1 << (x.shape[0] * k)
    return max(min((a - b) % mod, (b - a) % mod) for a, b in zip(_value(x, k), _value(y, k)))


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("rank", [1, 2])
@pytest.mark.parametrize("res_k", [12, 13])
def test_per_bit_composition_agrees_within_one_unit(fl, rank, res_k):
    """Key-switching commutes with the rotation up to its final rounding into res.size limbs (input and key in one base2k, so the
    key-switch decomposes the limbs as they are); the rounding need not be odd-symmetric, so a wrapped coefficient may move by one unit."""
    k, a_size, res_size, n_lwe = 12, 3, 2, N
    rng = np.random.default_rng(1300 + fl + rank + res_k)
    o = O.OracleModule(N, fl)
    key = prep(o, fill_uniform(rng, (a_size, rank, a_size + 1, 2, N), k))
    a = fill_uniform(rng, (a_size, rank + 1, N), k)
    index = _indices(rng)
    got = np.zeros((len(index), res_size, 1, n_lwe + 1), dtype=np.int64)
    want = np.zeros_like(got)
    R.glwe_to_lwe_indexed(o, got, res_k, a, k, index, key, k)
    R.glwe_to_lwe_per_bit(o, want, res_k, a, k, index, key, k)
    for j in range(len(index)):
        assert _max_unit_distance(got[j], want[j], res_k) <= 1, (j, index[j])


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
def test_a_wrapped_minus_half_digit_differs_bit_wise(fl):
    """An identity key (row d copies mask limb d to output limb d) leaves a normalised input unchanged.  With -2^(k-1) in the mask's
    coefficient 0, the entry's rotation by X^-idx negates it into +2^(k-1) at t = n - idx; the composition normalises the rotated input
    back to -2^(k-1) and carries one into the limb above.  Same integer, different digits."""
    k, size, idx = 12, 3, 5
    rng = np.random.default_rng(1400 + fl)
    o = O.OracleModule(N, fl)
    mat = np.zeros((size, 1, size, 2, N), dtype=np.int64)
    for d in range(size):
        mat[d, 0, d, 1, 0] = 1
    key = prep(o, mat)
    a = fill_uniform(rng, (size, 2, N), k)
    a[:, 1, 0] = fill_uniform(rng, size, k - 1)  # small digits around the planted one
    a[1, 1, 0] = -(1 << (k - 1))
    g = np.zeros_like(a)
    o.glwe_keyswitch(g, k, a, k, key, k, 1)
    assert np.array_equal(g, a)  # the identity key
    got = np.zeros((1, size, 1, N + 1), dtype=np.int64)
    want = np.zeros_like(got)
    R.glwe_to_lwe_indexed(o, got, k, a, k, [idx], key, k)
    R.glwe_to_lwe_per_bit(o, want, k, a, k, [idx], key, k)
    t = N - idx + 1  # LWE word 1 + (N - idx) reads mask coefficient 0, wrapped
    assert got[0, 1, 0, t] == 1 << (k - 1) and want[0, 1, 0, t] == -(1 << (k - 1))
    assert want[0, 0, 0, t] == got[0, 0, 0, t] + 1
    assert not np.array_equal(got, want)
    assert _max_unit_distance(got[0], want[0], k) == 0
