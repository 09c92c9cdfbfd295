"""Pins the CMux-tree reference of tests/cmux_tree_ref.py on the CPU:

(a) meaning: with noise-free GGSW(0) / GGSW(1) bits of m (test_oracle_cmux.noiseless_ggsw) and noise-free leaves, the phase of the result
    is the phase of leaf m, for every m < 2^n_bits.  Exactly, at res.size * base2k bits, when no limb is truncated (leaf size = res.size =
    dnum = s.size); within n_bits times the rounding the CMux test allows per CMux otherwise;
(b) one bit is one glwe_cmux(t = leaf 1, f = leaf 0);
(c) a table shared by the batch gives what the same table replicated per item gives;
(d) the lookup-table read by vertical packing (circuit.lut_read's composition) of a table with more entries than the ring degree, with
    noise-free bits, is an LWE whose phase is LUT[m]."""
import numpy as np
import pytest

import cmux_ref as CR
import cmux_tree_ref as TR
import semantics_circuit as SC
from oracle import pyoracle as O
from test_oracle_cmux import centred_diff, noiseless_ggsw, prep
from util import fill_uniform

# n, rank, k, res_size, leaf_size, dnum, s_size
SHAPES_EXACT = [(64, 1, 12, 2, 2, 2, 2), (64, 2, 13, 3, 3, 3, 3), (128, 1, 18, 1, 1, 1, 1)]
SHAPES_ROUNDED = [(64, 1, 12, 2, 3, 2, 3), (64, 2, 13, 2, 2, 3, 4), (128, 1, 12, 3, 4, 3, 4)]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", SHAPES_EXACT + SHAPES_ROUNDED)
def test_tree_selects_the_leaf_of_the_encrypted_integer(fl, shape):
    n, rank, k, rs, ls, dnum, ss = shape
    rng = np.random.default_rng(sum(shape) + 100 * fl)
    o = O.OracleModule(n, fl)
    s = [rng.integers(-1, 2, size=n).astype(np.int64) for _ in range(rank)]
    ggsw = [prep(o, noiseless_ggsw(rng, bit, s, k, dnum, ss)) for bit in (0, 1)]
    exact = shape in SHAPES_EXACT
    shift = (ls - rs) * k  # a leaf's phase at res.size * k bits
    for n_bits in (1, 2, 3):
        leaves = [SC.noiseless_row(rng, {0: rng.integers(-8, 8, size=n) << (k - 4)}, s, k, ls) for _ in range(1 << n_bits)]
        tol = 0 if exact else n_bits * 2 * (1 + rank * n)
        assert tol < 1 << (rs * k - 4 - 5)  # 2^5 below the lowest message bit
        for m in range(1 << n_bits):
            res = np.zeros((rs, rank + 1, n), dtype=np.int64)
            TR.glwe_cmux_tree(o, res, leaves, k, [ggsw[(m >> i) & 1] for i in range(n_bits)], k)
            want = [(w >> shift) if shift >= 0 else (w << -shift) for w in SC.phase_scaled(leaves[m], s, k)]
            err = centred_diff(SC.phase_scaled(res, s, k), want, rs * k)
            assert err <= tol, (n_bits, m, err, tol)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("shape", [(64, 1, 12, 2, 3, 2, 2, 1, 12), (64, 2, 13, 3, 2, 2, 4, 2, 13), (128, 1, 13, 2, 2, 3, 3, 1, 17)])
def test_one_bit_is_one_cmux(fl, shape):
    n, rank, k, rs, ls, dnum, ss, dsize, gk = shape
    cols = rank + 1
    rng = np.random.default_rng(sum(shape) + 13 * fl)
    o = O.OracleModule(n, fl)
    leaves = [fill_uniform(rng, (ls, cols, n), k + 6) for _ in range(2)]
    sel = prep(o, fill_uniform(rng, (dnum, cols, ss, cols, n), gk))
    res = np.zeros((rs, cols, n), dtype=np.int64)
    TR.glwe_cmux_tree(o, res, leaves, k, [sel], gk, dsize)
    want = np.zeros((rs, cols, n), dtype=np.int64)
    CR.glwe_cmux(o, want, leaves[1], leaves[0], k, sel, gk, dsize)
    assert np.array_equal(res, want)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
def test_shared_table_equals_the_replicated_table(fl):
    n, cols, k, B, L = 64, 2, 13, 3, 3
    rng = np.random.default_rng(71 + fl)
    o = O.OracleModule(n, fl)
    table = [fill_uniform(rng, (2, cols, n), k + 3) for _ in range(1 << L)]
    sels = [[prep(o, fill_uniform(rng, (2, cols, 2, cols, n), k)) for _ in range(L)] for _ in range(B)]
    shared = np.zeros((B, 2, cols, n), dtype=np.int64)
    TR.glwe_cmux_tree_batch(o, shared, [table], sels, k, k)
    replicated = np.zeros_like(shared)
    TR.glwe_cmux_tree_batch(o, replicated, [table] * B, sels, k, k)
    assert np.array_equal(shared, replicated)
    assert not np.array_equal(shared[0], shared[1])  # the items select differently


def lwe_phase(lwe, s, k):
    """b + <a, s_ext> of an LWE (size, 1, n + 1) as an integer modulo 2^(size k), s_ext(X) = s(X^-1) the key of the extraction."""
    size = lwe.shape[0]
    s_ext = np.concatenate([s[:1], -s[:0:-1]])
    mod = 1 << (size * k)
    return sum(int(lwe[j, 0, 0] + np.dot(lwe[j, 0, 1:], s_ext)) << ((size - 1 - j) * k) for j in range(size)) % mod


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("n,k,size,n_bits,T", [(64, 12, 2, 7, 100), (64, 13, 3, 8, 256), (128, 18, 1, 8, 129), (64, 12, 2, 5, 21)])
def test_lut_read_by_vertical_packing(fl, n, k, size, n_bits, T):
    """T above n (except the last case: n_bits below log2 n, no tree level): noise-free bits of m and exact shapes give the phase LUT[m] exactly."""
    rng = np.random.default_rng(n + k + size + n_bits + T + 7 * fl)
    o = O.OracleModule(n, fl)
    s = rng.integers(-1, 2, size=n).astype(np.int64)
    ggsw = [prep(o, noiseless_ggsw(rng, bit, [s], k, size, size)) for bit in (0, 1)]
    lut = np.zeros((size, T), dtype=np.int64)
    lut[0] = rng.integers(-8, 8, size=T) << (k - 4)
    lut[size - 1] += rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=T)  # low bits in the last limb, kept exactly
    mod = 1 << (size * k)
    want_of = [sum(int(lut[j, t]) << ((size - 1 - j) * k) for j in range(size)) % mod for t in range(T)]
    for m in sorted({0, 1, min(n - 1, T - 1), min(n, T - 1), T - 1, *rng.integers(0, T, size=3).tolist()}):
        lwe = TR.lut_read(o, lut, [ggsw[(m >> i) & 1] for i in range(n_bits)], k)
        assert lwe_phase(lwe, s, k) == want_of[m], m
