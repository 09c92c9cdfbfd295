"""The reference LWE <-> GLWE family of the tests (tests/lwe_ref.py: extraction / embedding copies around the oracle's glwe_keyswitch), CPU
only.

The meaning is pinned independently: sample extraction against its numpy definition, the three key-switching forms with noise-free
keys built from the embedding s_glwe(X) = s_lwe(X^-1) (the phase must survive, exactly when no limb is dropped), and a closed bootstrap
loop LWE(m) -> blind rotation -> glwe_to_lwe -> lwe_keyswitch -> LWE(f(m)) under the original LWE secret, twice in a row.
tests/test_gpu_lwe.py compares the device with these same reference calls."""
from fractions import Fraction

import numpy as np
import pytest

import lwe_ref as L
import semantics as S
import semantics_circuit as SC
from oracle import pyoracle as O
from test_oracle_semantics import noiseless_ksk
from util import fill_uniform

N = 64


def embed_secret(s_lwe, n):
    """s_glwe(X) = s_lwe(X^-1) in Z[X]/(X^n + 1), zero padded: coefficient 0 of c0 + c1 s_glwe is c0[0] + <c1[0..n_lwe), s_lwe>."""
    out = [0] * n
    out[0] = int(s_lwe[0])
    for i in range(1, len(s_lwe)):
        out[n - i] = -int(s_lwe[i])
    return out


def lwe_phase(lwe, s, k):
    """b + <a, s> of an LWE (size, 1, n_lwe + 1) as an unreduced torus Fraction."""
    return sum(Fraction(int(lwe[j, 0, 0]) + int(np.dot(lwe[j, 0, 1:].astype(object), np.asarray(s, dtype=object))), 1 << ((j + 1) * k))
               for j in range(lwe.shape[0]))


def prep(o, mat):
    dnum, cols_in, size, cols_out, _ = mat.shape
    pm = o.vmp_pmat_alloc(dnum, cols_in, cols_out, size)
    o.vmp_prepare(pm, mat)
    return pm


def _binary(rng, n):
    return [int(x) for x in rng.integers(0, 2, size=n)]


def _ternary(rng, n):
    return [int(x) for x in rng.integers(-1, 2, size=n)]


@pytest.mark.parametrize("n_lwe", [1, 37, 64])
@pytest.mark.parametrize("res_size", [1, 3, 5])
def test_sample_extract_equals_numpy_definition(n_lwe, res_size):
    rng = np.random.default_rng(10 * n_lwe + res_size)
    a_size = 3
    a = fill_uniform(rng, (a_size, 2, N), 20)
    res = fill_uniform(rng, (res_size, 1, n_lwe + 1), 20)  # garbage pre-fill: every limb is written
    L.lwe_sample_extract(res, a)
    want = np.zeros_like(res)
    for i in range(min(res_size, a_size)):
        want[i, 0, 0] = a[i, 0, 0]
        want[i, 0, 1:] = a[i, 1, :n_lwe]
    assert np.array_equal(res, want)


def _tol(res_size, k, exact):
    # as test_noiseless_keyswitch_preserves_the_phase: every column rounded at 2^-(res_size k), the masks multiplied by a small secret
    return Fraction(0) if exact else Fraction(1 + N, 1 << (res_size * k))


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("dsize", [1, 2])
def test_noiseless_lwe_keyswitch_preserves_the_phase(fl, dsize):
    k, a_size, n_in, n_out = 12, 4, 50, 37
    key_size = a_size + dsize
    rng = np.random.default_rng(900 + fl + dsize)
    o = O.OracleModule(N, fl)
    s_in, s_out = _binary(rng, n_in), _binary(rng, n_out)
    key = noiseless_ksk(rng, [embed_secret(s_in, N)], [embed_secret(s_out, N)], k, -(-a_size // dsize), key_size, dsize)
    a = fill_uniform(rng, (a_size, 1, n_in + 1), k)
    want = lwe_phase(a, s_in, k)
    for res_size in (key_size, a_size, 2):
        res = fill_uniform(rng, (res_size, 1, n_out + 1), k)
        L.lwe_keyswitch(o, res, k, a, k, prep(o, key), k, dsize)
        assert abs(S.centred_mod1(lwe_phase(res, s_out, k) - want)) <= _tol(res_size, k, res_size == key_size), res_size


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("rank", [1, 2])
def test_noiseless_glwe_to_lwe_extracts_coefficient_zero(fl, rank):
    k, a_size, n_lwe = 12, 3, 41
    key_size = a_size + 1
    rng = np.random.default_rng(950 + fl + rank)
    o = O.OracleModule(N, fl)
    s = [_ternary(rng, N) for _ in range(rank)]
    s_lwe = _binary(rng, n_lwe)
    key = noiseless_ksk(rng, s, [embed_secret(s_lwe, N)], k, a_size, key_size)
    a = fill_uniform(rng, (a_size, rank + 1, N), k)
    want = S.phase(a.tolist(), s, k)[0]
    for res_size in (key_size, a_size):
        res = fill_uniform(rng, (res_size, 1, n_lwe + 1), k)
        L.glwe_to_lwe(o, res, k, a, k, prep(o, key), k)
        assert abs(S.centred_mod1(lwe_phase(res, s_lwe, k) - want)) <= _tol(res_size, k, res_size == key_size), res_size


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("rank", [1, 2])
def test_noiseless_lwe_to_glwe_keeps_the_phase_in_coefficient_zero(fl, rank):
    k, a_size, n_lwe = 12, 3, 64
    key_size = a_size + 1
    rng = np.random.default_rng(970 + fl + rank)
    o = O.OracleModule(N, fl)
    s = [_ternary(rng, N) for _ in range(rank)]
    s_lwe = _binary(rng, n_lwe)
    key = noiseless_ksk(rng, [embed_secret(s_lwe, N)], s, k, a_size, key_size)
    a = fill_uniform(rng, (a_size, 1, n_lwe + 1), k)
    want = lwe_phase(a, s_lwe, k)
    for res_size in (key_size, a_size):
        res = fill_uniform(rng, (res_size, rank + 1, N), k)
        L.lwe_to_glwe(o, res, k, a, k, prep(o, key), k)
        got = S.phase(res.tolist(), s, k)[0]
        assert abs(S.centred_mod1(got - want)) <= _tol(res_size, k, res_size == key_size) * rank, res_size


# ---- closed bootstrap loop ------------------------------------------------------------------------------------------------------------
LOOP = dict(k=12, rank=1, n_lwe=12, block=3, brk_dnum=2, brk_size=3, lwe_size=2, n_mid=40, mid_size=3, log_domain=2)


def f_lut(m, log_domain):
    return (m + 1) % (1 << log_domain)


def loop_material(rng, n, fl):
    """Noise-free keys of the loop: BRK from semantics_circuit.build_keys, the GLWE -> LWE key to a binary s_mid of n_mid coefficients and
    the LWE key-switching key from s_mid back to s_lwe, both built from the embedding; and the LUT of f (one padding bit, drift step / 2
    as circuit_bootstrap_to_constant_ref)."""
    p = LOOP
    k, rank = p["k"], p["rank"]
    s_lwe, s, brk, _, _ = SC.build_keys(rng, n, k, rank, p["n_lwe"], p["block"], p["brk_dnum"], p["brk_size"], 1, 1, 1, 1)
    s_mid = _binary(rng, p["n_mid"])
    ks1 = noiseless_ksk(rng, [list(map(int, x)) for x in s], [embed_secret(s_mid, n)], k, p["brk_size"], p["brk_size"] + 1)
    ks2 = noiseless_ksk(rng, [embed_secret(s_mid, n)], [embed_secret(s_lwe, n)], k, p["mid_size"], p["mid_size"] + 1)
    q = 1 << p["log_domain"]
    step = n // q
    full = np.zeros((1, 1, n), dtype=np.int64)
    for m in range(q):
        full[0, 0, m * step:(m + 1) * step] = f_lut(m, p["log_domain"]) << (k - p["log_domain"] - 1)
    lut = np.zeros_like(full)
    O.vec_znx_rotate((-(step // 2)) % (2 * n), lut, 0, full, 0)
    return dict(s_lwe=s_lwe, s=s, brk=brk, ks1=ks1, ks2=ks2, lut=lut)


def decode(lwe, s_lwe, k, log_domain):
    t = 1 << (log_domain + 1)
    return round(S.centred_mod1(lwe_phase(lwe, s_lwe, k)) * t) % t


def oracle_round(o, lwe, mat, brk_o, xpa, ks1_o, ks2_o):
    """One round on the oracle -> (lwe_2n, acc, lwe_mid, lwe_out)."""
    p, n = LOOP, o.n
    k = p["k"]
    lwe_2n = O.mod_switch_2n(2 * n, lwe, k, True)
    acc = np.zeros((p["brk_size"], p["rank"] + 1, n), dtype=np.int64)
    o.cggi_blind_rotate_block_binary(acc, lwe_2n, mat["lut"], brk_o, xpa, p["block"], k)
    mid = np.zeros((p["mid_size"], 1, p["n_mid"] + 1), dtype=np.int64)
    L.glwe_to_lwe(o, mid, k, acc, k, ks1_o, k)
    out = np.zeros((p["lwe_size"], 1, p["n_lwe"] + 1), dtype=np.int64)
    L.lwe_keyswitch(o, out, k, mid, k, ks2_o, k)
    return lwe_2n, acc, mid, out


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
def test_noiseless_bootstrap_loop_on_the_oracle(fl):
    p = LOOP
    rng = np.random.default_rng(990 + fl)
    o = O.OracleModule(N, fl)
    mat = loop_material(rng, N, fl)
    assert mat["s_lwe"].sum() >= 1
    brk_o = [prep(o, b) for b in mat["brk"]]
    ks1_o, ks2_o, xpa = prep(o, mat["ks1"]), prep(o, mat["ks2"]), o.cggi_x_pow_a()
    for m in range(1 << p["log_domain"]):
        lwe = SC.noiseless_lwe(rng, m, p["log_domain"], mat["s_lwe"], p["k"], p["lwe_size"])
        want = m
        for _ in range(2):
            lwe = oracle_round(o, lwe, mat, brk_o, xpa, ks1_o, ks2_o)[3]
            want = f_lut(want, p["log_domain"])
            assert decode(lwe, mat["s_lwe"], p["k"], p["log_domain"]) == want, (m, want)
