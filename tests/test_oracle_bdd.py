"""Pins the BDD builder (circuit.bdd_from_truth_tables) and the BDD reference of tests/bdd_ref.py on the CPU:

(a) the builder's diagrams reproduce their truth tables in plain integers: the 8-bit adder (9 outputs, 65 nodes with the bits of x and y
    interleaved, most significant first), the 8-bit comparison x < y (23 nodes), the adder in a bad order (2001 nodes), and random tables
    in random orders; every diagram is reduced (no node with equal children, no two equal nodes) and levelled (children in earlier levels);
(b) meaning: with noise-free GGSW bits of x and trivial leaves 0 and scale, every output's phase is f(x) * scale, exactly;
(c) the complete tree written as a circuit equals cmux_tree_ref bit for bit;
(d) a one-node circuit is one glwe_cmux."""
import numpy as np
import pytest

import bdd_ref as BR
import cmux_ref as CR
import cmux_tree_ref as TR
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200.circuit import BddCircuit, bdd_from_truth_tables, bdd_leaves
from test_oracle_cmux import noiseless_ggsw, prep
from util import fill_uniform

X8 = np.arange(1 << 16) & 255
Y8 = np.arange(1 << 16) >> 8
INTERLEAVED = [v for i in range(7, -1, -1) for v in (i, i + 8)]  # x7 y7 x6 y6 ... x0 y0: the root tests x7
ADD8 = [((X8 + Y8) >> i) & 1 for i in range(9)]
LT8 = [(X8 < Y8).astype(np.int64)]


def eval_all(c, n_bits):
    """The circuit in plain integers at every input x < 2^n_bits at once: -> (n_out, 2^n_bits) leaf values."""
    x = np.arange(1 << n_bits)
    state = [np.full(1 << n_bits, v) for v in c.leaves]
    for bit, nodes in c.levels:
        sel = ((x >> bit) & 1).astype(bool)
        state += [np.where(sel, state[t], state[f]) for t, f in nodes]
    return np.stack([state[o] for o in c.outputs])


def check_shape(c, n_bits):
    """Levelled and reduced: children below the level's first state, distinct bits per level, no t == f, no duplicate node."""
    first, seen = len(c.leaves), set()
    bits = [b for b, _ in c.levels]
    assert len(set(bits)) == len(bits) and all(0 <= b < n_bits for b in bits)
    for bit, nodes in c.levels:
        assert nodes
        for t, f in nodes:
            assert t < first and f < first and t != f
            assert (bit, t, f) not in seen
            seen.add((bit, t, f))
        first += len(nodes)
    assert all(0 <= o < first for o in c.outputs)


@pytest.mark.parametrize("name,tables,order,nodes,widest", [
    ("add8", ADD8, INTERLEAVED, 65, 6),
    ("lt8", LT8, INTERLEAVED, 23, 2),
    ("add8-msb-first", ADD8, list(range(7, -1, -1)) + list(range(15, 7, -1)), 2001, None),
])
def test_builder_reproduces_the_truth_tables(name, tables, order, nodes, widest):
    c = bdd_from_truth_tables(tables, 16, order)
    check_shape(c, 16)
    assert c.n_nodes == nodes, (name, c.n_nodes)
    assert len(c.levels) == 16 and [b for b, _ in c.levels] == order[::-1]  # level 0 tests order[-1], the root order[0]
    if widest is not None:
        assert max(len(nodes) for _, nodes in c.levels) == widest
    assert np.array_equal(eval_all(c, 16), np.stack(tables))


@pytest.mark.parametrize("n_bits,n_out", [(1, 1), (3, 2), (5, 4), (9, 3)])
def test_builder_on_random_tables_and_orders(n_bits, n_out):
    rng = np.random.default_rng(31 * n_bits + n_out)
    tables = [rng.integers(0, 2, size=1 << n_bits) for _ in range(n_out)]
    tables.append(np.zeros(1 << n_bits, dtype=np.int64))  # a constant output is a leaf
    tables.append(tables[0].copy())                       # an equal output shares its root
    order = rng.permutation(n_bits).tolist()
    c = bdd_from_truth_tables(tables, n_bits, order)
    check_shape(c, n_bits)
    assert c.outputs[-2] == 0 and c.outputs[-1] == c.outputs[0]
    assert np.array_equal(eval_all(c, n_bits), np.stack(tables))
    for x in (0, (1 << n_bits) - 1, int(rng.integers(0, 1 << n_bits))):
        assert BR.eval_plain(c, [(x >> i) & 1 for i in range(n_bits)]) == [int(t[x]) for t in tables]


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
def test_noise_free_bits_give_the_function_times_scale(fl):
    """A 2-bit adder (3 outputs over 4 bits) and its x < y, in a non-default order: exact shapes (leaf size = res.size = dnum = s.size),
    so the phase of output o at x is tables[o][x] * scale exactly."""
    n, k, size, n_bits = 64, 12, 2, 4
    rng = np.random.default_rng(90 + fl)
    o = O.OracleModule(n, fl)
    s = rng.integers(-1, 2, size=n).astype(np.int64)
    ggsw = [prep(o, noiseless_ggsw(rng, bit, [s], k, size, size)) for bit in (0, 1)]
    x = np.arange(1 << n_bits)
    xs, ys = x & 3, x >> 2
    tables = [((xs + ys) >> i) & 1 for i in range(3)] + [(xs < ys).astype(np.int64)]
    c = bdd_from_truth_tables(tables, n_bits, [1, 3, 0, 2])
    scale = 1 << (k - 2)
    leaves = bdd_leaves(n, c, scale, size)
    for m in range(1 << n_bits):
        got = BR.glwe_bdd_eval(o, size, leaves, c, k, [ggsw[(m >> i) & 1] for i in range(n_bits)], k)
        for j, t in enumerate(tables):
            assert SC.phase_scaled(got[j], [s], k) == SC.phase_scaled(leaves[int(t[m])], [s], k), (m, j)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
@pytest.mark.parametrize("L", [1, 2, 3])
def test_complete_tree_circuit_equals_the_cmux_tree(fl, L):
    n, cols, k, rs, ls = 64, 2, 13, 2, 3
    rng = np.random.default_rng(7 * L + fl)
    o = O.OracleModule(n, fl)
    leaves = fill_uniform(rng, (1 << L, ls, cols, n), k + 4)
    sels = [prep(o, fill_uniform(rng, (2, cols, 2, cols, n), k)) for _ in range(L)]
    want = np.zeros((rs, cols, n), dtype=np.int64)
    TR.glwe_cmux_tree(o, want, leaves, k, sels, k)
    got = BR.glwe_bdd_eval(o, rs, leaves, BR.complete_tree(L), k, sels, k)
    assert got.shape == (1, rs, cols, n) and np.array_equal(got[0], want)


@pytest.mark.parametrize("fl", [O.NTT120, O.FFT64])
def test_one_node_is_one_cmux(fl):
    n, cols, k, rs, ls, gk, dsize = 64, 3, 13, 3, 2, 13, 2
    rng = np.random.default_rng(5 + fl)
    o = O.OracleModule(n, fl)
    leaves = fill_uniform(rng, (3, ls, cols, n), k + 6)
    sel = prep(o, fill_uniform(rng, (2, cols, 4, cols, n), gk))
    c = BddCircuit([0, 1, 2], [(1, [(2, 0)])], [3, 1])  # t = leaf 2, f = leaf 0, bit 1; outputs: the node and leaf 1
    got = BR.glwe_bdd_eval(o, rs, leaves, c, k, [None, sel], gk, dsize)
    want = np.zeros((rs, cols, n), dtype=np.int64)
    CR.glwe_cmux(o, want, leaves[2], leaves[0], k, sel, gk, dsize)
    assert np.array_equal(got[0], want)
    assert np.array_equal(got[1, :ls], leaves[1]) and not got[1, ls:].any()


def test_circuit_struct_matches_the_header():
    """pgb_bdd_circuit: two u64, four pointers, one u64, one pointer (64 bytes); BddCircuit.struct() fills it in level order."""
    import ctypes as C
    from poulpy_b200 import hal
    assert C.sizeof(hal._BDD) == 64
    c = BddCircuit([0, 1], [(3, [(1, 0)]), (0, [(2, 0), (1, 2)])], [3, 4, 1])
    cs, keep = c.struct()
    assert (cs.n_leaves, cs.n_levels, cs.n_out) == (2, 2, 3)
    assert [cs.level_bit[i] for i in range(2)] == [3, 0] and [cs.level_count[i] for i in range(2)] == [1, 2]
    assert [cs.node_t[i] for i in range(3)] == [1, 2, 1] and [cs.node_f[i] for i in range(3)] == [0, 0, 2]
    assert [cs.outputs[i] for i in range(3)] == [3, 4, 1]
