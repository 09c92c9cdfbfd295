"""Reference blind rotation by GGSW bits for the tests: the loop of pgb_glwe_blind_rotate_ggsw_batched (include/poulpy_b200.h),

    acc_0 = a;  acc_{i+1} = cmux(t = X^(p_i) acc_i, f = acc_i, s_i) with p_i = (step 2^i) mod 2n;  res = acc_{n_bits},

over cmux_ref.glwe_cmux and the oracle's vec_znx_rotate (oracle/znx.c).  GLWEs are int64 arrays (size, cols, n); sels[i] is the oracle
VmpPMat of bit i of this one ciphertext."""
import numpy as np

import cmux_ref as CR
from oracle import pyoracle as O


def rotation(step, i, n):
    """p_i = (step 2^i) mod 2n, exact for any int64 step and i < 64."""
    return (int(step) << i) % (2 * n)


def glwe_blind_rotate_ggsw(o, res, a, base2k, step, sels, ggsw_base2k, dsize=1):
    rs, cols, n = res.shape
    acc = np.ascontiguousarray(a, dtype=np.int64)
    for i, s in enumerate(sels):
        t = np.zeros_like(acc)
        for c in range(cols):
            O.vec_znx_rotate(rotation(step, i, n), t, c, acc, c)
        nxt = np.zeros((rs, cols, n), dtype=np.int64)
        CR.glwe_cmux(o, nxt, t, acc, base2k, s, ggsw_base2k, dsize)
        acc = nxt
    res[:] = acc
