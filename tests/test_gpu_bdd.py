"""GPU parity of the BDD evaluator (pgb_glwe_bdd_eval_batched) with tests/bdd_ref.py, bit for bit, both flavours: n = 256 .. 4096; rank 1
and 2; base2k 13 and 18 and ggsw_base2k != base2k; dsize 1 and 2; leaves at and past the fused routes' bound; random levelled circuits
whose children skip levels, whose levels test the bits in a non-default order and whose outputs include leaves; shared and per-item
leaves with padded strides; shared selectors and per-item selectors in the bit-major and the ciphertext-major layouts; batches 1 .. 512;
default routes against PGB_OPT_NO_FUSION.  Every case also runs today's composition (one glwe_cmux per node, then a glwe_copy per
output) and checks equal outputs, and checks that a chunk launches one CMux's launches per level (on the level's route) plus one; a
forced small scratch runs several chunks with the same result.  Then the complete tree against glwe_cmux_tree, a selector extent above
4 GiB, the rejections, and circuit bootstrapping -> prepare_ggsw -> circuit.bdd_eval of the 8-bit adder, end to end."""
import ctypes as C

import numpy as np
import pytest

import bdd_ref as BR
import lwe_ref as LR
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.circuit import BddCircuit, bdd_from_truth_tables
from poulpy_b200.hal import _BT, lib
from test_gpu_cmux import _glwe, _np, _prep_o, _selectors
from test_gpu_cmux_tree import _tables
from test_gpu_glwe_blind_rotate import _layout, _with_fusion
from test_oracle_bdd import ADD8, INTERLEAVED
from test_oracle_cmux_tree import lwe_phase
from util import fill_uniform

import poulpy_b200 as pb

pytestmark = pytest.mark.gpu


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def _random_circuit(rng, n_leaves, n_bits, widths, n_out):
    """Levels of the given widths testing distinct bits in a random order; every child is a random earlier state (so children skip
    levels and leaves appear on every level); the outputs are the last node, a leaf, and random states."""
    bits = rng.permutation(n_bits)[:len(widths)]
    levels, first = [], n_leaves
    for bit, w in zip(bits, widths):
        levels.append((int(bit), [(int(rng.integers(0, first)), int(rng.integers(0, first))) for _ in range(w)]))
        first += w
    outputs = [first - 1, int(rng.integers(0, n_leaves))] + rng.integers(0, first, size=max(0, n_out - 2)).tolist()
    return BddCircuit(list(range(n_leaves)), levels, outputs[:n_out])


def _level_f_sizes(c, a_size, rs):
    """The f.size of every level: res.size when an f child is a node, min(a.size, res.size) otherwise."""
    nl = len(c.leaves)
    return [rs if any(f >= nl for _, f in nodes) else min(a_size, rs) for _, nodes in c.levels]


def _one_cmux_launches(g, cols, rs, f_size, k, pm, ggsw_stride, sel_offset, gk, dsize, B, cache):
    """Launches of one glwe_cmux of B items on the route a level with this f.size takes: with the level's shared selector, or with B
    per-item (zero) selectors of the same shape."""
    key = (f_size, B, g.get_option(pb.hal.OPT_NO_FUSION), sel_offset if ggsw_stride == 0 else None)
    if key not in cache:
        t, f, out = g.vec_znx_alloc(cols, rs, B), g.vec_znx_alloc(cols, f_size, B), g.vec_znx_alloc(cols, rs, B)
        if ggsw_stride == 0:
            sel = pb.hal.VmpPMat(pm.buf, g.n, pm.rows, cols, cols, pm.size, offset=pm.offset + sel_offset)
        else:
            sel = g.vmp_pmat_alloc(pm.rows, cols, cols, pm.size, batch=max(B, 2))
        before = g.launch_count
        g.glwe_cmux(out, t, f, k, sel, gk, dsize)
        cache[key] = g.launch_count - before
        g.sync()
    return cache[key]


def _expected_launches(g, c, cols, rs, a_size, k, pm, ggsw_stride, bit_stride, gk, dsize, B, chunk, cache):
    widest = max([len(nodes) for _, nodes in c.levels] + [1])
    Bc = min(B, 65535 // widest, chunk or B)
    total = 0
    for b0 in range(0, B, Bc):
        nb = min(Bc, B - b0)
        total += 1 + sum(_one_cmux_launches(g, cols, rs, fs, k, pm, ggsw_stride, bit * bit_stride, gk, dsize, nb * len(nodes), cache)
                         for fs, (bit, nodes) in zip(_level_f_sizes(c, a_size, rs), c.levels))
    return total


def _run(g, c, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, pad, rng, max_chunk=None):
    B, n_out, rs, cols, n = shape
    res = _glwe(fill_uniform(rng, (B * n_out, rs, cols, n), 50), pad)  # garbage pre-fill
    before = g.launch_count
    g.glwe_bdd_eval(res, av, c, k, L, pm, gk, dsize, entry_stride=es, ggsw_stride=ggsw_stride, bit_stride=bit_stride, max_chunk=max_chunk)
    g.sync()
    return _np(res, B * n_out).reshape(shape), g.launch_count - before


def _compose(g, c, shape, av, es, k, pm, ggsw_stride, bit_stride, gk, dsize):
    """Today's composition: one glwe_cmux per node, then one glwe_copy per output."""
    B, n_out, rs, cols, n = shape
    shared = av.batch == 1
    state = [pb.hal.VecZnx(av.buf, n, cols, av.size, offset=av.offset + j * es, batch=1 if shared else B, batch_stride=av.batch_stride)
             for j in range(len(c.leaves))]
    for bit, nodes in c.levels:
        sel = pb.hal.VmpPMat(pm.buf, n, pm.rows, cols, cols, pm.size, offset=pm.offset + bit * bit_stride, batch=B, batch_stride=ggsw_stride)
        for t, f in nodes:
            out = g.vec_znx_alloc(cols, rs, B)
            g.glwe_cmux(out, state[t], state[f], k, sel, gk, dsize)
            state.append(out)
    res = g.vec_znx_alloc(cols, rs, B * n_out)
    for o, s in enumerate(c.outputs):
        src = state[s]
        if src.batch > 1:
            circuit._glwe_copy(g, res.ptr + o * res.batch_stride, n_out * res.batch_stride, rs, src.ptr, src.batch_stride, src.size, cols, B)
        else:  # a shared leaf: one copy per item
            for b in range(B):
                circuit._glwe_copy(g, res.ptr + (b * n_out + o) * res.batch_stride, 0, rs, src.ptr, 0, src.size, cols, 1)
    g.sync()
    return g.vec_znx_to_numpy(res).reshape(shape)


def _check_case(fl, g, o, c, leaves, B, rs, cols, n, k, gk, dsize, mode, pad, L, mats, rng, sample=None, chunk=None):
    shared = leaves.shape[0] == 1
    n_out = len(c.outputs)
    ggsw_items, bit_items, q = _layout(mode, B, L, 1)
    n_sel = L if mode == "shared" else B * L
    idx = rng.integers(0, len(mats), size=n_sel)
    pm = _selectors(g, mats, idx, 8 * (pad // 16), pad)
    ggsw_stride, bit_stride = ggsw_items * pm.batch_stride, bit_items * pm.batch_stride
    pos = [_prep_o(o, m) for m in mats]
    items = range(B) if sample is None else sample
    want = {b: BR.glwe_bdd_eval(o, rs, leaves[0 if shared else b], c, k, [pos[idx[q(b, i)]] for i in range(L)], gk, dsize) for b in items}
    av, es = _tables(leaves, pad)
    shape = (B, n_out, rs, cols, n)
    run = lambda mc=None: _run(g, c, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, pad, rng, mc)  # noqa: E731
    got0, l0 = _with_fusion(g, 0, run)
    got1, l1 = _with_fusion(g, 1, run)
    for b in items:
        assert np.array_equal(got0[b], want[b]), ("default", b)
        assert np.array_equal(got1[b], want[b]), ("no fusion", b)
    comp0 = _with_fusion(g, 0, lambda: _compose(g, c, shape, av, es, k, pm, ggsw_stride, bit_stride, gk, dsize))
    comp1 = _with_fusion(g, 1, lambda: _compose(g, c, shape, av, es, k, pm, ggsw_stride, bit_stride, gk, dsize))
    assert np.array_equal(comp0, got0) and np.array_equal(comp1, got1), "the composition differs"
    cache = {}
    a_size = leaves.shape[2]
    e0 = _with_fusion(g, 0, lambda: _expected_launches(g, c, cols, rs, a_size, k, pm, ggsw_stride, bit_stride, gk, dsize, B, None, cache))
    e1 = _with_fusion(g, 1, lambda: _expected_launches(g, c, cols, rs, a_size, k, pm, ggsw_stride, bit_stride, gk, dsize, B, None, cache))
    assert (l0, l1) == (e0, e1), (l0, l1, e0, e1)
    if chunk is not None:  # a scratch for `chunk` items: several chunks, the same result, the launches of each chunk
        got2, l2 = run(chunk)
        assert np.array_equal(got2, got0)
        assert l2 == _expected_launches(g, c, cols, rs, a_size, k, pm, ggsw_stride, bit_stride, gk, dsize, B, chunk, cache), l2


# n, rank, k, gk, res_size, a_size, dnum, s_size, dsize, batch, selectors, pad, n_bits, level widths, n_leaves, n_out, shared leaves, chunk
CASES = [
    (256, 1, 13, 13, 2, 2, 2, 2, 1, 37, "bit", 16, 4, (3, 1, 5, 2), 3, 4, True, 5),
    (512, 1, 13, 13, 2, 2, 3, 2, 1, 37, "bit", 16, 6, (2, 6, 3, 4, 1), 2, 3, False, 8),  # a.size == res.size == s.size: fused
    (512, 1, 13, 13, 2, 3, 2, 2, 1, 9, "ct", 0, 3, (3, 2, 2), 4, 3, True, None),           # a.size past the bound
    (1024, 2, 13, 13, 3, 3, 2, 2, 1, 5, "bit", 16, 3, (2, 3, 1), 3, 2, False, 2),          # res.size past s.size: limb-wise
    (1024, 2, 13, 13, 2, 1, 2, 2, 1, 9, "ct", 16, 5, (4, 3, 2, 2, 1), 2, 5, True, None),   # a below res
    (1024, 2, 13, 13, 3, 3, 2, 4, 2, 9, "ct", 16, 3, (3, 3, 1), 3, 2, True, 4),            # dsize 2
    (1024, 1, 13, 18, 3, 2, 3, 3, 1, 9, "bit", 0, 2, (1,), 2, 2, False, None),              # ggsw_base2k != base2k, one node
    (1024, 2, 18, 13, 2, 3, 3, 3, 2, 5, "ct", 16, 4, (2, 2, 3), 2, 3, False, None),        # both
    (4096, 1, 18, 18, 2, 2, 2, 3, 1, 3, "bit", 16, 3, (2, 2, 1), 2, 2, True, 1),
    (4096, 2, 13, 13, 1, 1, 1, 1, 1, 2, "ct", 0, 2, (1, 2), 2, 3, False, None),
    (256, 1, 13, 13, 2, 3, 2, 2, 1, 37, "shared", 16, 4, (3, 2, 2), 2, 3, False, 10),
    (1024, 2, 13, 13, 2, 2, 2, 2, 1, 37, "shared", 0, 5, (2, 4, 3, 2, 1), 3, 4, True, None),
    (2048, 1, 18, 13, 3, 2, 3, 3, 2, 5, "shared", 16, 3, (2, 1, 2), 2, 2, False, 2),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-r{c[1]}-k{c[2]}.{c[3]}-s{c[4]}.{c[5]}-d{c[6]}.{c[7]}-ds{c[8]}-b{c[9]}-{c[10]}-p{c[11]}-"
                                             f"L{c[12]}-w{'.'.join(map(str, c[13]))}-l{c[14]}-o{c[15]}{'-lshared' if c[16] else ''}"
                                             f"{'-chunk' + str(c[17]) if c[17] else ''}" for c in CASES])
def test_bdd_matches_reference(fl, case):
    n, rank, k, gk, rs, as_, dnum, ss, dsize, B, mode, pad, L, widths, nl, n_out, shared, chunk = case
    cols = rank + 1
    rng = np.random.default_rng(sum(case[:10]) + 17 * L + 1000 * fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    c = _random_circuit(rng, nl, L, widths, n_out)
    leaves = fill_uniform(rng, (1 if shared else B, nl, as_, cols, n), k + 4)
    mats = [fill_uniform(rng, (dnum, cols, ss, cols, n), gk) for _ in range(3)]
    sample = None if B * c.n_nodes <= 128 else sorted({0, B - 1, *rng.choice(B, 4, replace=False).tolist()})
    _check_case(fl, g, o, c, leaves, B, rs, cols, n, k, gk, dsize, mode, pad, L, mats, rng, sample, chunk)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("B,mode,shared", [(1, "bit", True), (37, "ct", False), (37, "shared", True), (512, "bit", True)])
def test_bdd_bench_shape_adder(fl, B, mode, shared):
    """The 8-bit adder (65 nodes, 16 levels, widest 6) at the circuit-bootstrapping bench shape: n = 1024, rank 2, base2k 13, GGSW dnum 2 x
    2 limbs, GLWEs of 2 limbs.  The reference checks a seeded sample of up to 3 items (the first and the last among them)."""
    n, rank, k, L = 1024, 2, 13, 16
    cols = rank + 1
    rng = np.random.default_rng(B + 3 * fl + len(mode) + 11 * shared)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    c = bdd_from_truth_tables(ADD8, 16, INTERLEAVED)
    leaves = fill_uniform(rng, (1 if shared else B, 2, 2, cols, n), k)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(6)]
    sample = sorted({0, B - 1, int(rng.integers(0, B))})
    _check_case(fl, g, o, c, leaves, B, 2, cols, n, k, k, 1, mode, 0, L, mats, rng, sample, 200 if B == 512 else None)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("nf", [0, 1])
def test_complete_tree_equals_glwe_cmux_tree(fl, nf):
    n, rank, k, L, B = 512, 1, 13, 4, 9
    cols = rank + 1
    rng = np.random.default_rng(44 + fl + 2 * nf)
    g = pb.Module(n, fl)
    tables = fill_uniform(rng, (B, 1 << L, 2, cols, n), k + 3)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(3)]
    pm = _selectors(g, mats, rng.integers(0, 3, size=B * L), 0, 0)
    av, es = _tables(tables, 16)

    def both():
        tree = g.vec_znx_alloc(cols, 2, B)
        g.glwe_cmux_tree(tree, av, k, L, pm, k, entry_stride=es)
        bdd = g.vec_znx_alloc(cols, 2, B)
        g.glwe_bdd_eval(bdd, av, BR.complete_tree(L), k, L, pm, k, entry_stride=es)
        g.sync()
        return g.vec_znx_to_numpy(tree), g.vec_znx_to_numpy(bdd)

    tree, bdd = _with_fusion(g, nf, both)
    assert np.array_equal(tree, bdd)


def test_bdd_selector_extent_above_4_gib():
    """2048 items x 4 bits of per-item NTT120 selectors at the bench shape span 4.8 GB, bit-major: every (b, i) offset must be 64-bit.
    A few distinct GGSWs are replicated with pgb_memcpy_d2d; the first, a middle and the last items are checked."""
    n, rank, k, B, L, G = 1024, 2, 13, 2048, 4, 4
    cols = rank + 1
    rng = np.random.default_rng(4098)
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(G)]
    pm_small = _selectors(g, mats, list(range(G)), 0, 0)
    item = pm_small.batch_stride
    assert item * B * L > 1 << 32
    buf = pb.DevBuf(item * B * L)
    idx = rng.integers(0, G, size=B * L)
    idx[-L:] = np.arange(L) % G
    for q in range(B * L):
        assert lib().pgb_memcpy_d2d(C.c_void_p(buf.ptr + q * item), C.c_void_p(pm_small.buf.ptr + int(idx[q]) * item), item) == 0
    pm = pb.hal.VmpPMat(buf, n, 2, cols, cols, 2, batch=B * L, batch_stride=item)
    c = _random_circuit(rng, 3, L, (2, 3, 2, 1), 3)
    leaves = fill_uniform(rng, (1, 3, 2, cols, n), k)
    av, es = _tables(leaves, 0)
    pos = [_prep_o(o, m) for m in mats]
    for nf in (0, 1):
        got, _ = _with_fusion(g, nf, lambda: _run(g, c, (B, 3, 2, cols, n), av, es, k, L, pm, L * item, item, k, 1, 0, rng))
        for b in (0, B // 2 + 1, B - 1):
            want = BR.glwe_bdd_eval(o, 2, leaves[0], c, k, [pos[idx[b * L + i]] for i in range(L)], k)
            assert np.array_equal(got[b], want), (nf, b)


# ---- rejections: each returns its status and launches nothing ---------------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_bdd_rejections_launch_nothing(fl):
    n, cols, size, B, L, k = 512, 2, 2, 4, 3, 13
    g = pb.Module(n, fl)
    item = n * cols * size * 8
    NL, NO = 2, 3
    good = BddCircuit([0, 1], [(0, [(1, 0)]), (2, [(2, 0), (1, 2)])], [3, 4, 1])  # level 1 skips to a leaf; output 2 is a leaf
    res, a = pb.DevBuf(B * NO * item), pb.DevBuf(B * NL * item)
    pm = g.vmp_pmat_alloc(2, cols, cols, size, batch=B * L + B)  # B spare items after the B * L selectors: room for a misplaced res
    pitem = pm.batch_stride
    S = pm.struct()
    cs, keep = good.struct()

    def tmp(batch, c=cs):
        return lib().pgb_glwe_bdd_eval_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S), C.c_uint64(k),
                                                 C.c_uint64(1), C.byref(c), C.c_uint64(batch))

    def cmux_tmp(batch):
        return lib().pgb_glwe_cmux_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S),
                                             C.c_uint64(k), C.c_uint64(1), C.c_uint64(batch))

    def al(x):
        return -(-x // 256) * 256

    need = tmp(B)
    # the descriptor table (3 nodes x 48 B, 3 outputs x 24 B) | the level blocks | the linear copy of f and one CMux's scratch (widest)
    assert need == al(3 * 48 + 3 * 24) + al(B * item) + al(2 * B * item) + al(2 * B * item) + cmux_tmp(2 * B)
    assert tmp(100000) == tmp(65535 // 2)  # the chunk cap
    scratch = pb.DevBuf(need + 512)
    VZ = pb.hal._VZ

    def vz(ptr, n_=n, cols_=cols, size_=size):
        return VZ(ptr, n_, cols_, size_, size_)

    def circ(**kw):
        d = dict(leaves=good.leaves, levels=good.levels, outputs=good.outputs)
        d.update(kw)
        return BddCircuit(**d).struct()

    def call(r=None, os_=item, aa=None, es=item, nb=L, s=None, gs=L * pitem, bs=pitem, c=None, bt=None, sp=None, sl=None, dsize=1):
        return lib().pgb_glwe_bdd_eval_batched(
            g._h, C.byref(r or vz(res.ptr)), C.c_uint64(os_), C.byref(aa or vz(a.ptr)), C.c_uint64(es), C.c_uint64(k), C.c_uint64(nb),
            C.byref(s or S), C.c_uint64(gs), C.c_uint64(bs), C.c_uint64(k), C.c_uint64(dsize), C.byref(c or cs),
            C.byref(bt or _BT(B, NO * item, NL * item, 0)), C.c_void_p(scratch.ptr if sp is None else sp),
            C.c_size_t(need if sl is None else sl))

    bad_child, kc = circ(levels=[(0, [(1, 0)]), (2, [(2, 0), (1, 4)])])     # a child in its own level
    fwd_child, kf = circ(levels=[(0, [(1, 3)]), (2, [(2, 0), (1, 2)])])     # a child in a later level
    bad_out, ko = circ(outputs=[3, 5])                                       # an output past the last state
    bad_bit, kb = circ(levels=[(0, [(1, 0)]), (3, [(2, 0), (1, 2)])])       # bit 3 with n_bits 3
    no_out, kn = circ(outputs=[])
    null_out, kno = circ()
    null_out.outputs = None
    zero_w, kz = circ(levels=[(0, [(1, 0)]), (2, [])])                     # a level of width 0
    null_t, knt = circ()
    null_t.node_t = None
    last_sel = (B - 1) * L * pitem + 2 * pitem  # the last selector read: (b, i) = (B - 1, 2)
    last_leaf = (B - 1) * NL * item + (NL - 1) * item
    g.sync()
    before = g.launch_count
    bad = [
        (-1, dict(aa=vz(a.ptr, n_=2 * n))),                            # ring degree
        (-1, dict(aa=vz(a.ptr, cols_=3))),                             # columns
        (-1, dict(bt=_BT(0, NO * item, NL * item, 0))),                # count 0
        (-1, dict(bt=_BT(65536, NO * item, NL * item, 0))),            # count > 65535
        (-1, dict(bt=_BT(B, NO * item, NL * item, item))),             # stride_b != 0
        (-1, dict(nb=0)),                                              # n_bits 0
        (-1, dict(nb=65)),                                             # n_bits > 64
        (-1, dict(c=bad_child)),
        (-1, dict(c=fwd_child)),
        (-1, dict(c=bad_out)),
        (-1, dict(c=bad_bit)),
        (-1, dict(c=no_out)),
        (-1, dict(c=null_out)),
        (-1, dict(c=zero_w)),
        (-1, dict(c=null_t)),
        (-1, dict(es=item + 8)),                                       # entry_stride not a multiple of 16
        (-1, dict(es=item - 16)),                                      # entry_stride below one GLWE
        (-1, dict(os_=item + 8)),                                      # out_stride not a multiple of 16
        (-1, dict(os_=item - 16)),                                     # outputs overlapping each other
        (-1, dict(bt=_BT(B, NO * item - 16, NL * item, 0))),           # stride_res below an item's outputs
        (-1, dict(r=vz(res.ptr + 8))),                                 # misaligned res data
        (-1, dict(bt=_BT(B, NO * item, NL * item + 8, 0))),            # misaligned leaf stride
        (-1, dict(gs=L * pitem + 8)),                                  # ggsw_stride not a multiple of 16
        (-1, dict(gs=16)),                                             # ggsw_stride below one GGSW
        (-1, dict(bs=pitem + 8)),                                      # bit_stride not a multiple of 16
        (-1, dict(bs=0)),                                              # bit_stride 0 with n_bits > 1
        (-1, dict(gs=1 << 62, bs=1 << 62)),                            # selectors past the end of the address space
        (-1, dict(es=1 << 63, bt=_BT(B, NO * item, 1 << 62, 0))),      # leaves past the end of the address space
        (-1, dict(os_=1 << 63, bt=_BT(1, 0, 0, 0))),                   # outputs past the end of the address space
        (-4, dict(sl=tmp(1) - 1)),                                     # scratch too small for one item
        (-1, dict(sp=scratch.ptr + 16)),                               # scratch misaligned
        (-3, dict(r=vz(a.ptr))),                                       # res inside the leaves
        (-3, dict(r=vz(a.ptr + last_leaf))),                           # res overlaps only the last leaf
        (-3, dict(r=vz(pm.buf.ptr + last_sel))),                       # res overlaps only the last selector read
        (-3, dict(sp=pm.buf.ptr + last_sel // 256 * 256)),             # scratch overlaps the last selectors
        (-3, dict(sp=res.ptr)),                                        # scratch overlaps res
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert call() == 0  # the same arguments, corrected, run
    assert call(sl=tmp(1)) == 0  # one item per chunk
    g.sync()


# ---- end to end: circuit bootstrapping -> prepare_ggsw -> circuit.bdd_eval ----------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
def test_circuit_bootstrap_then_bdd_eval_on_the_device(fl):
    """The 8-bit adder at n = 256: B * 16 noise-free LWE bits (x in bits 0-7, y in bits 8-15) are circuit-bootstrapped, prepared with
    circuit.prepare_ggsw (bit-major) and evaluated with circuit.bdd_eval.  The 9 LWEs of each item must equal the oracle composition
    (bdd_ref over the oracle's circuit bootstrapping, then sample extraction) bit for bit and decrypt to the bits of x + y."""
    from test_oracle_circuit_semantics import check_ggsw
    n, k, n_lwe, block, log_domain, rank = 256, 12, 12, 3, 2, 1
    brk_size, dnum_res, res_size, lwe_size = 4, 2, 4, 2
    L = 16
    cols = rank + 1
    rng = np.random.default_rng(6400 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    s_lwe, s, brk, atk, tsk = SC.build_keys(rng, n, k, rank, n_lwe, block, brk_size, brk_size, brk_size, brk_size + 1, res_size, res_size + 1)
    per = n * brk_size * cols * cols * brk_size * g.prep_bytes
    brk_buf = pb.DevBuf(per * n_lwe)
    for i, mat in enumerate(brk):
        g.vmp_prepare(pb.hal.VmpPMat(brk_buf, n, brk_size, cols, cols, brk_size, offset=i * per), g.mat_znx_from_numpy(mat))
    brk_g = pb.hal.VmpPMat(brk_buf, n, brk_size, cols, cols, brk_size)

    def prep_g(mat):
        d, ci, sz, co, _ = mat.shape
        pm = g.vmp_pmat_alloc(d, ci, co, sz)
        g.vmp_prepare(pm, g.mat_znx_from_numpy(mat))
        return pm

    brk_o, atk_o, tsk_o = [_prep_o(o, m) for m in brk], [_prep_o(o, m) for m in atk], [_prep_o(o, m) for m in tsk]
    atk_g, tsk_g = [prep_g(m) for m in atk], [prep_g(m) for m in tsk]
    xy = [(255, 1), (173, 94)]
    B = len(xy)
    ms = [x | (y << 8) for x, y in xy]
    bits = [(m >> i) & 1 for m in ms for i in range(L)]
    lwe = np.stack([SC.noiseless_lwe(rng, m, log_domain, s_lwe, k, lwe_size) for m in bits])
    lwe_dev = pb.DevBuf(lwe.nbytes)
    lwe_dev.upload(lwe)
    ggsw = circuit.circuit_bootstrap_to_constant(g, lwe_dev, B * L, n_lwe, lwe_size, k, brk_g, g.cggi_x_pow_a(), block, atk_g, tsk_g, k, rank,
                                                 dnum_res, res_size, log_domain)
    sel = circuit.prepare_ggsw(g, ggsw, B * L, dnum_res, rank, res_size)
    c = bdd_from_truth_tables(ADD8, 16, INTERLEAVED)
    rs = dnum_res
    scale = 1 << (k - 1)  # a bit in the top bit of the phase
    out = circuit.bdd_eval(g, c, sel, B, L, k, scale, size=rs)
    g.sync()
    n_out = len(c.outputs)
    got = out.download(np.int64, (B, n_out, rs, 1, n + 1))
    xpa = o.cggi_x_pow_a()
    leaves = circuit.bdd_leaves(n, c, scale, rs)
    # per CMux as in test_circuit_bootstrap_then_cmux_on_the_device, times the L CMuxes a path passes through at most
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c_ == 0 else n // 8) for c_ in range(cols))
    bound = L * ((dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n))
    assert bound < 1 << (rs * k - 1 - 5)  # 2^5 below the message bit
    mod = 1 << (rs * k)
    for b, (x, y) in enumerate(xy):
        sels = []
        for i in range(L):
            mat = SC.circuit_bootstrap_to_constant_ref(o, lwe[b * L + i], k, brk_o, xpa, block, atk_o, tsk_o, rank, dnum_res, res_size,
                                                       log_domain, brk_size)
            check_ggsw(mat, bits[b * L + i], s, k, res_size)
            sels.append(_prep_o(o, mat))
        glwes = BR.glwe_bdd_eval(o, rs, leaves, c, k, sels, k)
        for j in range(n_out):
            want = np.zeros((rs, 1, n + 1), dtype=np.int64)
            LR.lwe_sample_extract(want, glwes[j])
            assert np.array_equal(got[b, j], want), (b, j)
            bit = ((x + y) >> j) & 1
            e = ((lwe_phase(got[b, j], s[0], k) - (bit << (rs * k - 1)) + (mod >> 1)) % mod) - (mod >> 1)
            assert abs(e) <= bound, (b, j, e, bound)
