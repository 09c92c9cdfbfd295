"""Reference CMux tree for the tests: the levels of pgb_glwe_cmux_tree_batched (include/poulpy_b200.h),

    g_0 = leaves;  g_{i+1}[j] = cmux(t = g_i[2j + 1], f = g_i[2j], s_i) for j < 2^(n_bits - 1 - i);  res = g_{n_bits}[0],

over cmux_ref.glwe_cmux, and the lookup-table read by vertical packing of circuit.lut_read over it, glwe_blind_rotate_ref and
lwe_ref.lwe_sample_extract.  GLWEs are int64 arrays (size, cols, n); sels[i] is the oracle VmpPMat of bit i of this one ciphertext."""
import numpy as np

import cmux_ref as CR
import glwe_blind_rotate_ref as BR
import lwe_ref as LR
from poulpy_b200.circuit import lut_split


def glwe_cmux_tree(o, res, leaves, base2k, sels, ggsw_base2k, dsize=1):
    rs, cols, n = res.shape
    assert len(leaves) == 1 << len(sels)
    g = [np.ascontiguousarray(x, dtype=np.int64) for x in leaves]
    for s in sels:
        nxt = []
        for j in range(len(g) // 2):
            out = np.zeros((rs, cols, n), dtype=np.int64)
            CR.glwe_cmux(o, out, g[2 * j + 1], g[2 * j], base2k, s, ggsw_base2k, dsize)
            nxt.append(out)
        g = nxt
    res[:] = g[0]


def lut_leaves(n, lut, n_bits):
    """circuit.lut_read's leaves: the polynomials of lut_split as trivial rank-1 GLWEs (body column 0, mask 0).  -> (nu, leaves)"""
    nu, polys = lut_split(n, lut, n_bits)
    leaves = np.zeros((polys.shape[0], polys.shape[1], 2, n), dtype=np.int64)
    leaves[:, :, 0] = polys
    return nu, leaves


def lut_read(o, lut, sels, base2k, ggsw_base2k=None, dsize=1):
    """The LWE (size, 1, n + 1) of circuit.lut_read for one item whose bit i selects with sels[i]."""
    n = o.n
    gk = base2k if ggsw_base2k is None else ggsw_base2k
    nu, leaves = lut_leaves(n, lut, len(sels))
    size = leaves.shape[1]
    picked = leaves[0]
    if len(sels) > nu:
        picked = np.zeros((size, 2, n), dtype=np.int64)
        glwe_cmux_tree(o, picked, leaves, base2k, sels[nu:], gk, dsize)
    rot = np.zeros((size, 2, n), dtype=np.int64)
    BR.glwe_blind_rotate_ggsw(o, rot, picked, base2k, -1, sels[:nu], gk, dsize)
    out = np.zeros((size, 1, n + 1), dtype=np.int64)
    LR.lwe_sample_extract(out, rot)
    return out


def glwe_cmux_tree_batch(o, res, tables, sels, base2k, ggsw_base2k, dsize=1):
    """res (B, size, cols, n): item b reads table 0 when `tables` holds one table (shared by the batch), table b otherwise; sels[b] are its
    selectors."""
    for b in range(res.shape[0]):
        glwe_cmux_tree(o, res[b], tables[0 if len(tables) == 1 else b], base2k, sels[b], ggsw_base2k, dsize)
