"""CPU pin of what the batched packing entry (pgb_glwe_pack_batched, Module.glwe_pack) must compute, on the maps it is used with:
circuit.glwe_pack over the oracle with zero-mask inputs, so that every key-switch term vanishes and the result is plain integer arithmetic on
the bodies.  Coefficient index[j] of the output carries the constant coefficient of input j, and every other coefficient is cleared: by the
packing rounds (every input is projected onto its constant coefficient, missing partners included) and, for log_gap_out > 0, by the final
partial trace.  The maps are the BDD output maps (a dense prefix of 9, the 8-bit adder's outputs, and of 32, at gap 0), a sparse map at
gap 3, and single inputs (at 0 with the whole trace, and at a non-zero index where every round has one side only)."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import pyoracle as O
from poulpy_b200 import circuit
from util import fill_uniform
from util_circuit import OracleGlweOps, _Ct

N, K, SIZE, LOG_N = 64, 16, 4, 6

MAPS = [
    ("dense9", list(range(9)), 0),
    ("dense32", list(range(32)), 0),
    ("sparse", [0, 8, 24, 40, 56], 3),
    ("one_full_trace", [0], LOG_N),
    ("one_hi_side", [48], 0),
]


def _torus(limbs, K):
    return sum(Fraction(int(v), 1 << ((j + 1) * K)) for j, v in enumerate(limbs))


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("name,index,g", MAPS, ids=[m[0] for m in MAPS])
def test_glwe_pack_maps_place_constant_coefficients(fl, name, index, g):
    rng = np.random.default_rng(3100 + len(index) + g)
    o = O.OracleModule(N, fl)
    atk = []
    for _ in range(LOG_N):
        pm = o.vmp_pmat_alloc(SIZE, 1, 2, SIZE + 1)
        o.vmp_prepare(pm, fill_uniform(rng, (SIZE, 1, SIZE + 1, 2, N), K))
        atk.append(pm)
    ops = OracleGlweOps(o, atk, K, 2, SIZE, 1, N)
    cts, consts = {}, {}
    for i in index:
        a = np.zeros((1, SIZE, 2, N), dtype=np.int64)
        a[0, :, 0] = fill_uniform(rng, (SIZE, N), K)  # body only: zero mask
        cts[i] = _Ct(a)
        consts[i] = _torus(a[0, :, 0, 0], K)
    res = ops.new()
    circuit.glwe_pack(ops, res, cts, g)
    assert not res.arr[0, :, 1].any()
    tol = Fraction(4 * LOG_N, 1 << (SIZE * K))
    for c in range(N):
        err = _torus(res.arr[0, :, 0, c], K) - consts.get(c, 0)
        err -= round(err)
        assert abs(err) <= tol, (name, c, float(err))
