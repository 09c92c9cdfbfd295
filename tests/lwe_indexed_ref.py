"""Reference of glwe_to_lwe at many coefficients (pgb_glwe_to_lwe_indexed_batched, Module.glwe_to_lwe_indexed) for the tests: one
glwe_keyswitch of the GLWE to rank 1 (the oracle's, as lwe_ref.glwe_to_lwe), then per index the rotation X^-index[j] (O.vec_znx_rotate)
and lwe_sample_extract.  Also the per-bit composition it replaces (rotate the input, then a whole glwe_to_lwe per index), which it is
not bit-identical to: see tests/test_oracle_lwe_indexed.py."""
import numpy as np

import lwe_ref as L
from oracle import pyoracle as O


def rotate(a, p):
    """X^p * a for every column of a GLWE (size, cols, n)."""
    n = a.shape[-1]
    out = np.zeros_like(a)
    for c in range(a.shape[1]):
        O.vec_znx_rotate(p % (2 * n), out, c, a, c)
    return out


def glwe_to_lwe_indexed(o, res, res_base2k, a, a_base2k, index, key, key_base2k, dsize=1):
    """res: (n_index, size, 1, n_lwe + 1) <- LWE j = lwe_sample_extract(X^-index[j] * glwe_keyswitch(a)); a: GLWE (size, rank + 1, n),
    key = VmpPMat(dnum, rank, 2, key_size)."""
    assert key.cols_in + 1 == a.shape[1] and key.cols_out == 2 and res.shape[0] == len(index)
    g = np.zeros((res.shape[1], 2, o.n), dtype=np.int64)
    o.glwe_keyswitch(g, res_base2k, a, a_base2k, key, key_base2k, dsize)
    for j, idx in enumerate(index):
        L.lwe_sample_extract(res[j], rotate(g, -int(idx)))


def glwe_to_lwe_per_bit(o, res, res_base2k, a, a_base2k, index, key, key_base2k, dsize=1):
    """The composition with one key-switch per index: LWE j = glwe_to_lwe(X^-index[j] * a)."""
    for j, idx in enumerate(index):
        L.glwe_to_lwe(o, res[j], res_base2k, rotate(a, -int(idx)), a_base2k, key, key_base2k, dsize)
