"""Reference CMux for the tests: the five steps of pgb_glwe_cmux_batched (include/poulpy_b200.h), which restate poulpy-bin-fhe's cmux
(glwe_sub, glwe_normalize_inplace, glwe_external_product_inplace, glwe_add_inplace, glwe_normalize_inplace).  The sub and the add are numpy
(int64 arrays wrap like the reference's i64), the normalisations and the external product are the oracle's (oracle/znx.c, oracle/core.c).

GLWEs are int64 arrays (size, cols, n); s is an oracle VmpPMat(dnum, cols, cols, s_size) -- the selector of this one ciphertext."""
import numpy as np

from oracle import pyoracle as O


def glwe_cmux(o, res, t, f, base2k, s, ggsw_base2k, dsize=1):
    rs, cols, n = res.shape
    assert t.shape[1:] == f.shape[1:] == (cols, n) and s.cols_in == s.cols_out == cols
    # 1. d = t - f into res.size limbs (a limb missing from an operand reads as 0)
    d = np.zeros((rs, cols, n), dtype=np.int64)
    k = min(rs, t.shape[0])
    d[:k] += t[:k]
    k = min(rs, f.shape[0])
    d[:k] -= f[:k]
    # 2. normalise
    for c in range(cols):
        O.vec_znx_normalize_assign(base2k, d, c)
    # 3. external product into res.size limbs of base2k
    e = np.zeros((rs, cols, n), dtype=np.int64)
    o.glwe_external_product(e, base2k, d, base2k, s, ggsw_base2k, dsize)
    # 4. e += f on the common limbs
    k = min(rs, f.shape[0])
    e[:k] += f[:k]
    # 5. normalise
    for c in range(cols):
        O.vec_znx_normalize_assign(base2k, e, c)
    res[:] = e
