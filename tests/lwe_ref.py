"""Reference LWE <-> GLWE family for the tests, written from the contract of poulpy-core's LWE::sample_extract, LWE::from_glwe
(conversion/glwe_to_lwe.rs), LWE::keyswitch (keyswitching/lwe.rs) and GLWE::from_lwe (conversion/lwe_to_glwe.rs).

An LWE is a one-column VecZnx of n_lwe + 1 coefficients per limb, int64 (size, 1, n_lwe + 1) = (b, a_0, ..), phase b + <a, s_lwe>.  Under the
GLWE embedding s_glwe(X) = s_lwe(X^-1) (zero padded to n) coefficient 0 of c0 + c1 s_glwe is c0[0] + <c1[0..n_lwe), s_lwe>, so extraction and
embedding are copies (numpy here) and all arithmetic is the oracle's glwe_keyswitch (oracle/core.c) on rank-1 GLWEs."""
import numpy as np


def lwe_sample_extract(res, a):
    """res: LWE (size, 1, n_lwe + 1) <- rank-1 GLWE a (size, 2, n): limbs i < min(res.size, a.size) copy (a[i][0][0], a[i][1][0..n_lwe)), the
    other limbs of res are zeroed."""
    assert res.shape[1] == 1 and a.shape[1] == 2 and 2 <= res.shape[2] <= a.shape[2] + 1
    res[:] = 0
    copy = min(res.shape[0], a.shape[0])
    res[:copy, 0, 0] = a[:copy, 0, 0]
    res[:copy, 0, 1:] = a[:copy, 1, : res.shape[2] - 1]


def lwe_embed(a, n):
    """LWE (size, 1, n_lwe + 1) -> zeroed rank-1 GLWE (size, 2, n): column 0 = (b, 0, ..), column 1 = (a_0, .., a_{n_lwe-1}, 0, ..)."""
    assert a.shape[1] == 1 and 2 <= a.shape[2] <= n + 1
    g = np.zeros((a.shape[0], 2, n), dtype=np.int64)
    g[:, 0, 0] = a[:, 0, 0]
    g[:, 1, : a.shape[2] - 1] = a[:, 0, 1:]
    return g


def lwe_keyswitch(o, res, res_base2k, a, a_base2k, key, key_base2k, dsize=1):
    """key = VmpPMat(dnum, 1, 2, key_size) from embed(s_in) to embed(s_out): embed, glwe_keyswitch into res.size limbs, extract."""
    assert key.cols_in == 1 and key.cols_out == 2
    out = np.zeros((res.shape[0], 2, o.n), dtype=np.int64)
    o.glwe_keyswitch(out, res_base2k, lwe_embed(a, o.n), a_base2k, key, key_base2k, dsize)
    lwe_sample_extract(res, out)


def glwe_to_lwe(o, res, res_base2k, a, a_base2k, key, key_base2k, dsize=1):
    """a: GLWE (size, rank + 1, n); key = VmpPMat(dnum, rank, 2, key_size): glwe_keyswitch to rank 1, extract."""
    assert key.cols_in + 1 == a.shape[1] and key.cols_out == 2
    out = np.zeros((res.shape[0], 2, o.n), dtype=np.int64)
    o.glwe_keyswitch(out, res_base2k, a, a_base2k, key, key_base2k, dsize)
    lwe_sample_extract(res, out)


def lwe_to_glwe(o, res, res_base2k, a, a_base2k, key, key_base2k, dsize=1):
    """res: GLWE (size, rank + 1, n); key = VmpPMat(dnum, 1, rank + 1, key_size): embed, glwe_keyswitch into res."""
    assert key.cols_in == 1 and key.cols_out == res.shape[1]
    o.glwe_keyswitch(res, res_base2k, lwe_embed(a, o.n), a_base2k, key, key_base2k, dsize)
