"""GPU parity of the CMux tree (pgb_glwe_cmux_tree_batched) with tests/cmux_tree_ref.py, bit for bit, both flavours: n = 256 .. 4096;
rank 1 and 2; base2k 13 and 18 and ggsw_base2k != base2k; dsize 1 and 2; a.size at and past the fused routes' bound (level 0 decides with
a.size, the later levels with res.size); n_bits 1, 2 and 5; shared and per-item tables with padded entry strides; shared selectors and
per-item selectors in the bit-major and the ciphertext-major layouts; batches 1, 37 and 512; default routes against PGB_OPT_NO_FUSION.
Every case also runs today's composition (one glwe_cmux per level and pair j) and checks equal outputs and that the entry launches chunks x
the launches of one CMux per level; a forced small scratch runs several chunks with the same result.  Then n_bits = 16 (one item per
chunk) by the phase of noise-free bits, a table extent above 4 GiB, the rejections, and circuit bootstrapping -> prepare_ggsw ->
circuit.lut_read of a table with more entries than the ring degree, end to end."""
import ctypes as C

import numpy as np
import pytest

import cmux_tree_ref as TR
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.hal import _BT, lib
from test_gpu_cmux import _np, _prep_o, _selectors
from test_gpu_glwe_blind_rotate import _fused_bit, _layout, _with_fusion
from test_oracle_cmux import noiseless_ggsw
from test_oracle_cmux_tree import lwe_phase
from util import fill_uniform

import poulpy_b200 as pb

pytestmark = pytest.mark.gpu


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def _tables(tables, pad):
    """(T, 2^L, size, cols, n) host tables -> (VecZnx of T tables, entry_stride): entries `item + pad` bytes apart, tables 2^L entries
    plus one spare entry apart (so neither stride is the tight one)."""
    T, E, size, cols, n = tables.shape
    item = size * cols * n * 8
    es = item + pad
    ts = (E + 1) * es
    host = np.zeros((T, ts // 8), dtype=np.int64)
    for t in range(T):
        for j in range(E):
            host[t, j * es // 8: j * es // 8 + item // 8] = tables[t, j].reshape(-1)
    buf = pb.DevBuf(host.nbytes)
    buf.upload(host)
    return pb.hal.VecZnx(buf, n, cols, size, batch=T, batch_stride=ts), es


def _run(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, rng, max_chunk=None):
    B, rs, cols, n = shape
    res = g.vec_znx_from_numpy(fill_uniform(rng, shape, 50))  # garbage pre-fill
    before = g.launch_count
    g.glwe_cmux_tree(res, av, k, L, pm, gk, dsize, entry_stride=es, ggsw_stride=ggsw_stride, bit_stride=bit_stride, max_chunk=max_chunk)
    g.sync()
    return g.vec_znx_to_numpy(res).reshape(shape), g.launch_count - before


def _compose(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize):
    """Today's composition: per level i and pair j, glwe_cmux(g_{i+1}[j], t = g_i[2j + 1], f = g_i[2j]).  Returns the result and the
    launches of the first CMux of every level."""
    B, rs, cols, n = shape
    shared = av.batch == 1
    cur = [pb.hal.VecZnx(av.buf, n, cols, av.size, offset=av.offset + j * es, batch=1 if shared else B, batch_stride=av.batch_stride)
           for j in range(1 << L)]
    per_level = []
    for i in range(L):
        sel = pb.hal.VmpPMat(pm.buf, n, pm.rows, cols, cols, pm.size, offset=pm.offset + i * bit_stride, batch=B, batch_stride=ggsw_stride)
        nxt = []
        for j in range(len(cur) // 2):
            out = g.vec_znx_alloc(cols, rs, B)
            before = g.launch_count
            g.glwe_cmux(out, cur[2 * j + 1], cur[2 * j], k, sel, gk, dsize)
            if j == 0:
                per_level.append(g.launch_count - before)
            nxt.append(out)
        cur = nxt
    g.sync()
    return g.vec_znx_to_numpy(cur[0]).reshape(shape), per_level


def _check_case(fl, g, o, tables, B, rs, cols, n, k, gk, dnum, ss, dsize, mode, pad, L, mats, rng, sample=None, chunk=None):
    shared = tables.shape[0] == 1
    ggsw_items, bit_items, q = _layout(mode, B, L, 1)
    n_sel = L if mode == "shared" else B * L
    idx = rng.integers(0, len(mats), size=n_sel)
    pm = _selectors(g, mats, idx, 8 * (pad // 16), pad)
    ggsw_stride, bit_stride = ggsw_items * pm.batch_stride, bit_items * pm.batch_stride
    pos = [_prep_o(o, m) for m in mats]
    items = range(B) if sample is None else sample
    want = {}
    for b in items:
        w = np.zeros((rs, cols, n), dtype=np.int64)
        TR.glwe_cmux_tree(o, w, tables[0 if shared else b], k, [pos[idx[q(b, i)]] for i in range(L)], gk, dsize)
        want[b] = w
    av, es = _tables(tables, pad)
    shape = (B, rs, cols, n)
    got0, l0 = _with_fusion(g, 0, lambda: _run(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, rng))
    got1, l1 = _with_fusion(g, 1, lambda: _run(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, rng))
    for b in items:
        assert np.array_equal(got0[b], want[b]), ("default", b)
        assert np.array_equal(got1[b], want[b]), ("no fusion", b)
    comp0, c0 = _with_fusion(g, 0, lambda: _compose(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize))
    comp1, c1 = _with_fusion(g, 1, lambda: _compose(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize))
    assert np.array_equal(comp0, got0) and np.array_equal(comp1, got1), "the composition differs"
    assert (l0, l1) == (sum(c0), sum(c1)), (l0, l1, c0, c1)  # one chunk: one CMux's launches per level
    fused = [_fused_bit(fl, n, k, gk, tables.shape[2] if i == 0 else rs, rs, ss, dsize, mode) for i in range(L)]
    if all(fused):
        assert l0 < l1 and len(set(c0)) == 1, (l0, l1, c0)
    if chunk is not None:  # a scratch for `chunk` items: several chunks, the same result, chunks x the launches
        got2, l2 = _run(g, shape, av, es, k, L, pm, ggsw_stride, bit_stride, gk, dsize, rng, max_chunk=chunk)
        assert np.array_equal(got2, got0)
        assert l2 == -(-B // chunk) * l0, (l2, B, chunk, l0)


# n, rank, k, gk, res_size, a_size, dnum, s_size, dsize, batch, selectors, pad, n_bits, shared table, chunk
CASES = [
    (256, 1, 13, 13, 2, 2, 2, 2, 1, 37, "bit", 16, 2, True, 5),
    (512, 1, 13, 13, 2, 2, 3, 2, 1, 37, "bit", 16, 5, False, 8),    # a.size == res.size == s.size: fused on every level
    (512, 1, 13, 13, 2, 3, 2, 2, 1, 9, "ct", 0, 2, True, None),     # a.size past the bound: level 0 limb-wise, level 1 fused
    (1024, 2, 13, 13, 3, 3, 2, 2, 1, 5, "bit", 16, 2, False, 2),    # res.size past s.size: limb-wise
    (1024, 2, 13, 13, 2, 1, 2, 2, 1, 9, "ct", 16, 5, True, None),   # a below res
    (1024, 2, 13, 13, 3, 3, 2, 4, 2, 9, "ct", 16, 2, True, 4),      # dsize 2
    (1024, 1, 13, 18, 3, 2, 3, 3, 1, 9, "bit", 0, 1, False, None),  # ggsw_base2k != base2k, one bit
    (1024, 2, 18, 13, 2, 3, 3, 3, 2, 5, "ct", 16, 2, False, None),  # both
    (4096, 1, 18, 18, 2, 2, 2, 3, 1, 3, "bit", 16, 2, True, 1),
    (4096, 2, 13, 13, 1, 1, 1, 1, 1, 2, "ct", 0, 1, False, None),
    (256, 1, 13, 13, 2, 3, 2, 2, 1, 37, "shared", 16, 2, False, 10),
    (1024, 2, 13, 13, 2, 2, 2, 2, 1, 37, "shared", 0, 5, True, None),
    (2048, 1, 18, 13, 3, 2, 3, 3, 2, 5, "shared", 16, 2, False, 2),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-r{c[1]}-k{c[2]}.{c[3]}-s{c[4]}.{c[5]}-d{c[6]}.{c[7]}-ds{c[8]}-b{c[9]}-{c[10]}-p{c[11]}-"
                                             f"L{c[12]}{'-tshared' if c[13] else ''}{'-chunk' + str(c[14]) if c[14] else ''}" for c in CASES])
def test_tree_matches_reference(fl, case):
    n, rank, k, gk, rs, as_, dnum, ss, dsize, B, mode, pad, L, shared, chunk = case
    cols = rank + 1
    rng = np.random.default_rng(sum(case[:10]) + 17 * L + 1000 * fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    tables = fill_uniform(rng, (1 if shared else B, 1 << L, as_, cols, n), k + 4)
    mats = [fill_uniform(rng, (dnum, cols, ss, cols, n), gk) for _ in range(3)]
    sample = None if B * ((1 << L) - 1) <= 128 else sorted({0, B - 1, *rng.choice(B, 4, replace=False).tolist()})
    _check_case(fl, g, o, tables, B, rs, cols, n, k, gk, dnum, ss, dsize, mode, pad, L, mats, rng, sample, chunk)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("B,mode,shared", [(1, "bit", True), (37, "ct", False), (37, "shared", True), (512, "bit", True), (512, "ct", False)])
def test_tree_bench_shape(fl, B, mode, shared):
    """The circuit-bootstrapping bench shape: n = 1024, rank 2, base2k 13, GGSW dnum 2 x 2 limbs, GLWEs of 2 limbs, 5 bits.  The
    reference checks a seeded sample of 6 items (the first and the last among them)."""
    n, rank, k, L = 1024, 2, 13, 5
    cols = rank + 1
    rng = np.random.default_rng(B + 3 * fl + len(mode) + 11 * shared)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    tables = fill_uniform(rng, (1 if shared else B, 1 << L, 2, cols, n), k)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(8)]
    sample = sorted({0, B - 1, *rng.choice(B, min(B, 4), replace=False).tolist()})
    _check_case(fl, g, o, tables, B, 2, cols, n, k, k, 2, 2, 1, mode, 0, L, mats, rng, sample, 100 if B == 512 else None)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_tree_sixteen_bits(fl):
    """n_bits = 16 at a tiny batch: 65536 trivial leaves (mask 0, exact shapes) and noise-free GGSW bits, so the phase of the result is
    leaf m_b's exactly; every level of the 2^16-leaf tree runs (one item per chunk: 2^15 CMuxes at level 0)."""
    n, k, size, L, B = 256, 13, 2, 16, 2
    rng = np.random.default_rng(1600 + fl)
    g = pb.Module(n, fl)
    s = rng.integers(-1, 2, size=n).astype(np.int64)
    mats = [noiseless_ggsw(rng, bit, [s], k, size, size) for bit in (0, 1)]
    ms = [int(rng.integers(0, 1 << L)), (1 << L) - 1]
    idx = [(m >> i) & 1 for m in ms for i in range(L)]  # bit-major
    pm = _selectors(g, mats, idx, 0, 0)
    table = np.zeros((1 << L, size, 2, n), dtype=np.int64)
    table[:, :, 0] = fill_uniform(rng, (1 << L, size, n), k)
    av = g.vec_znx_from_numpy(table)
    av = pb.hal.VecZnx(av.buf, n, 2, size)
    res = g.vec_znx_alloc(2, size, B)
    before = g.launch_count
    g.glwe_cmux_tree(res, av, k, L, pm, k)
    g.sync()
    launches = g.launch_count - before
    got = g.vec_znx_to_numpy(res).reshape(B, size, 2, n)
    for b, m in enumerate(ms):
        assert SC.phase_scaled(got[b], [s], k) == SC.phase_scaled(table[m], [s], k), (b, m)
    assert launches % (B * L) == 0, launches  # two chunks of one item, the same launches on every level


def test_tree_table_extent_above_4_gib():
    """Leaves 1.5 GiB apart (4 leaves: a 4.5 GiB shared table) and per-item tables 2.25 GiB apart: every leaf offset must be 64-bit."""
    n, rank, k, L = 1024, 2, 13, 2
    cols = rank + 1
    rng = np.random.default_rng(4097)
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    item = 2 * cols * n * 8
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(4)]
    pos = [_prep_o(o, m) for m in mats]
    for B, es, ts in [(3, 3 << 29, 0), (3, item, 9 << 28)]:
        T = 1 if ts == 0 else B
        assert (T - 1) * ts + ((1 << L) - 1) * es + item > 1 << 32
        buf = pb.DevBuf((T - 1) * ts + ((1 << L) - 1) * es + item)
        tables = fill_uniform(rng, (T, 1 << L, 2, cols, n), k)
        for t in range(T):
            for j in range(1 << L):
                buf.upload(tables[t, j], offset=t * ts + j * es)
        av = pb.hal.VecZnx(buf, n, cols, 2, batch=T, batch_stride=ts)
        idx = rng.integers(0, len(mats), size=B * L)
        pm = _selectors(g, mats, idx, 0, 0)
        for nf in (0, 1):
            got, _ = _with_fusion(g, nf, lambda: _run(g, (B, 2, cols, n), av, es, k, L, pm, L * pm.batch_stride, pm.batch_stride, k, 1, rng))
            for b in range(B):
                want = np.zeros((2, cols, n), dtype=np.int64)
                TR.glwe_cmux_tree(o, want, tables[0 if T == 1 else b], k, [pos[idx[b * L + i]] for i in range(L)], k)
                assert np.array_equal(got[b], want), (es, ts, nf, b)
        del buf, av


# ---- rejections: each returns its status and launches nothing ---------------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_tree_rejections_launch_nothing(fl):
    n, cols, size, B, L, k = 512, 2, 2, 4, 3, 13
    g = pb.Module(n, fl)
    item = n * cols * size * 8
    E = 1 << L
    res, a = pb.DevBuf(B * item), pb.DevBuf(B * E * item)
    pm = g.vmp_pmat_alloc(2, cols, cols, size, batch=B * L + B)  # B spare items after the B * L selectors: room for a misplaced res
    pitem = pm.batch_stride
    S = pm.struct()

    def tmp(batch, nb=L):
        return lib().pgb_glwe_cmux_tree_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S), C.c_uint64(k),
                                                  C.c_uint64(1), C.c_uint64(nb), C.c_uint64(batch))

    def cmux_tmp(batch):
        return lib().pgb_glwe_cmux_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S),
                                             C.c_uint64(k), C.c_uint64(1), C.c_uint64(batch))

    def al(x):
        return -(-x // 256) * 256

    need = tmp(B)
    P0 = B * E // 2
    # the level-1 and level-2 buffers | level 0's linear copy of f | one CMux's scratch over level 0's CMuxes
    assert need == al(P0 * item) + al(P0 // 2 * item) + al(P0 * item) + cmux_tmp(P0)
    assert tmp(B, 1) == al(B * item) + cmux_tmp(B)
    assert tmp(100000, 16) == tmp(1, 16) and tmp(100000, 8) == tmp(65535 // 128, 8)  # the chunk cap
    scratch = pb.DevBuf(need + 512)
    VZ = pb.hal._VZ

    def vz(ptr, n_=n, cols_=cols, size_=size):
        return VZ(ptr, n_, cols_, size_, size_)

    def call(r=None, aa=None, es=item, nb=L, s=None, gs=L * pitem, bs=pitem, bt=None, sp=None, sl=None, dsize=1):
        return lib().pgb_glwe_cmux_tree_batched(
            g._h, C.byref(r or vz(res.ptr)), C.byref(aa or vz(a.ptr)), C.c_uint64(es), C.c_uint64(k), C.c_uint64(nb), C.byref(s or S),
            C.c_uint64(gs), C.c_uint64(bs), C.c_uint64(k), C.c_uint64(dsize), C.byref(bt or _BT(B, item, E * item, 0)),
            C.c_void_p(scratch.ptr if sp is None else sp), C.c_size_t(need if sl is None else sl))

    last_sel = (B - 1) * L * pitem + (L - 1) * pitem  # the last selector (b, i) = (B - 1, L - 1)
    last_leaf = (B - 1) * E * item + (E - 1) * item    # the last leaf (b, j) = (B - 1, E - 1)
    g.sync()
    before = g.launch_count
    bad = [
        (-1, dict(aa=vz(a.ptr, n_=2 * n))),                            # ring degree
        (-1, dict(aa=vz(a.ptr, cols_=3))),                             # columns
        (-1, dict(bt=_BT(0, item, E * item, 0))),                      # count 0
        (-1, dict(bt=_BT(65536, item, E * item, 0))),                  # count > 65535
        (-1, dict(bt=_BT(B, item, E * item, item))),                   # stride_b != 0
        (-1, dict(nb=0)),                                              # n_bits 0
        (-1, dict(nb=17)),                                             # n_bits > 16
        (-1, dict(es=item + 8)),                                       # entry_stride not a multiple of 16
        (-1, dict(es=item - 16)),                                      # entry_stride below one GLWE
        (-1, dict(r=vz(res.ptr + 8))),                                 # misaligned res data
        (-1, dict(bt=_BT(B, item, E * item + 8, 0))),                  # misaligned table stride
        (-1, dict(gs=L * pitem + 8)),                                  # ggsw_stride not a multiple of 16
        (-1, dict(gs=16)),                                             # ggsw_stride below one GGSW
        (-1, dict(bs=pitem + 8)),                                      # bit_stride not a multiple of 16
        (-1, dict(bs=0)),                                              # bit_stride 0 with n_bits > 1
        (-1, dict(gs=1 << 62, bs=1 << 62)),                            # selectors past the end of the address space
        (-1, dict(es=1 << 62)),                                        # leaves past the end of the address space
        (-4, dict(sl=tmp(1) - 1)),                                     # scratch too small for one item
        (-1, dict(sp=scratch.ptr + 16)),                               # scratch misaligned
        (-3, dict(r=vz(a.ptr))),                                       # res inside the table
        (-3, dict(r=vz(a.ptr + last_leaf))),                           # res overlaps only the last leaf
        (-3, dict(r=vz(pm.buf.ptr + last_sel))),                       # res overlaps only the last selector
        (-3, dict(sp=pm.buf.ptr + last_sel // 256 * 256)),             # scratch overlaps the last selectors
        (-3, dict(sp=res.ptr)),                                        # scratch overlaps res
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert call() == 0  # the same arguments, corrected, run
    assert call(nb=1, bs=0) == 0  # bit_stride is not read for one bit
    assert call(sl=tmp(1)) == 0  # one item per chunk
    g.sync()


# ---- end to end: circuit bootstrapping -> prepare_ggsw -> circuit.lut_read ----------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
def test_circuit_bootstrap_then_lut_read_on_the_device(fl):
    """A lookup table of 300 entries at n = 256 (9 bits: a one-level tree over two polynomials, then a rotation by 8 bits): B * 9
    noise-free LWE bits are circuit-bootstrapped, prepared with circuit.prepare_ggsw (bit-major) and read with circuit.lut_read.  The LWEs
    must equal the oracle composition (tests/cmux_tree_ref.lut_read over the oracle's circuit bootstrapping) bit for bit and decrypt to
    LUT[m_b]."""
    from test_oracle_circuit_semantics import check_ggsw
    n, k, n_lwe, block, log_domain, rank = 256, 12, 12, 3, 2, 1
    brk_size, dnum_res, res_size, lwe_size = 4, 2, 4, 2
    L, T = 9, 300
    cols = rank + 1
    rng = np.random.default_rng(5400 + fl)
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
    ms = [299, 37]
    B = len(ms)
    bits = [(m >> i) & 1 for m in ms for i in range(L)]
    lwe = np.stack([SC.noiseless_lwe(rng, m, log_domain, s_lwe, k, lwe_size) for m in bits])
    lwe_dev = pb.DevBuf(lwe.nbytes)
    lwe_dev.upload(lwe)
    ggsw = circuit.circuit_bootstrap_to_constant(g, lwe_dev, B * L, n_lwe, lwe_size, k, brk_g, g.cggi_x_pow_a(), block, atk_g, tsk_g, k, rank,
                                                 dnum_res, res_size, log_domain)
    sel = circuit.prepare_ggsw(g, ggsw, B * L, dnum_res, rank, res_size)
    rs = dnum_res
    vals = rng.integers(0, 4, size=T)
    lut = np.zeros((rs, T), dtype=np.int64)
    lut[0] = vals << (k - 2)  # 2-bit entries in the top bits
    out = circuit.lut_read(g, lut, sel, B, L, k)
    g.sync()
    got = out.download(np.int64, (B, rs, 1, n + 1))
    xpa = o.cggi_x_pow_a()
    # per CMux as in test_circuit_bootstrap_then_cmux_on_the_device, times the L CMuxes an entry passes through
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c == 0 else n // 8) for c in range(cols))
    bound = L * ((dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n))
    assert bound < 1 << (rs * k - 2 - 5)  # 2^5 below the lowest message bit
    mod = 1 << (rs * k)
    for b, m in enumerate(ms):
        sels = []
        for i in range(L):
            mat = SC.circuit_bootstrap_to_constant_ref(o, lwe[b * L + i], k, brk_o, xpa, block, atk_o, tsk_o, rank, dnum_res, res_size,
                                                       log_domain, brk_size)
            check_ggsw(mat, bits[b * L + i], s, k, res_size)
            sels.append(_prep_o(o, mat))
        want = TR.lut_read(o, lut, sels, k)
        assert np.array_equal(got[b], want), b
        e = ((lwe_phase(got[b], s[0], k) - (int(vals[m]) << (rs * k - 2)) + (mod >> 1)) % mod) - (mod >> 1)
        assert abs(e) <= bound, (b, e, bound)
