"""GPU parity of the CMux (pgb_glwe_cmux_batched) and of the batched GGSW preparation (pgb_vmp_prepare_batched) with tests/cmux_ref.py,
bit for bit, both flavours: n = 256 (NTT120 limb-wise, FFT64 fused), 512, 1024, 4096; rank 1 and 2; sizes 1 .. 4 with t.size, f.size and
res.size apart, f.size at and just past min(res.size, s.size) (where the fused routes hand over to the limb-wise one); dnum 1 .. 4, dsize 1
and 2; base2k 13 and 18 and ggsw_base2k != base2k; shared and per-item selectors with padded strides; batches 1, 37 and 512 at the
circuit-bootstrapping bench shape; default routes against PGB_OPT_NO_FUSION; a per-item selector extent above 4 GiB; the rejections; the
pinned-key invalidation of the batched prepare; and the chain circuit bootstrapping -> prepare_ggsw -> glwe_cmux on the device."""
import ctypes as C

import numpy as np
import pytest

import cmux_ref as CR
import poulpy_b200 as pb
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.hal import _BT, lib
from util import fill_uniform

pytestmark = pytest.mark.gpu


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def _glwe(arr, pad):
    """(B, size, cols, n) -> VecZnx batch, items `item + pad` bytes apart."""
    B, size, cols, n = arr.shape
    item = size * cols * n
    host = np.zeros((B, item + pad // 8), dtype=np.int64)
    host[:, :item] = arr.reshape(B, item)
    buf = pb.DevBuf(host.nbytes)
    buf.upload(host)
    return pb.hal.VecZnx(buf, n, cols, size, batch=B, batch_stride=item * 8 + pad)


def _np(v, B):
    item = v.size * v.cols * v.n
    return v.buf.download(np.int64, (B, v.batch_stride // 8))[:, :item].reshape(B, v.size, v.cols, v.n)


def _selectors(g, mats, idx, mat_pad, pmat_pad, per_item=True):
    """Distinct host MatZnx `mats`, item b = mats[idx[b]]: a device MatZnx batch (stride padded by mat_pad bytes) assembled by device copies,
    prepared with vmp_prepare_batched into a VmpPMat batch (stride padded by pmat_pad bytes)."""
    d, ci, sz, co, n = mats[0].shape
    B = len(idx)
    one = mats[0].nbytes
    mstride = one + mat_pad
    src = pb.DevBuf(one * len(mats))
    src.upload(np.stack(mats))
    mbuf = pb.DevBuf(mstride * B)
    for b, i in enumerate(idx):
        assert lib().pgb_memcpy_d2d(C.c_void_p(mbuf.ptr + b * mstride), C.c_void_p(src.ptr + int(i) * one), one) == 0
    mat = pb.hal.MatZnx(mbuf, n, d, ci, co, sz, batch=B, batch_stride=mstride)
    pitem = n * d * ci * co * sz * g.prep_bytes
    pstride = pitem + pmat_pad
    pm = pb.hal.VmpPMat(pb.DevBuf(pstride * B), n, d, ci, co, sz, batch=B, batch_stride=pstride if per_item else 0)
    g.vmp_prepare_batched(pm, mat)
    return pm


def _prep_o(o, mat):
    d, ci, sz, co, _ = mat.shape
    pm = o.vmp_pmat_alloc(d, ci, co, sz)
    o.vmp_prepare(pm, mat)
    return pm


def _run(g, res_shape, pad, tv, fv, k, pm, gk, dsize, no_fusion, rng):
    g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
    res = _glwe(fill_uniform(rng, res_shape, 50), pad)  # garbage pre-fill
    before = g.launch_count
    g.glwe_cmux(res, tv, fv, k, pm, gk, dsize)
    g.sync()
    return _np(res, res_shape[0]), g.launch_count - before


# n, rank, k, gk, res_size, t_size, f_size, dnum, s_size, dsize, batch, per_item, pad
CASES = [
    (256, 1, 13, 13, 2, 2, 2, 2, 2, 1, 37, True, 16),
    (256, 2, 18, 18, 3, 1, 4, 3, 3, 1, 5, True, 0),
    (512, 1, 13, 13, 3, 4, 2, 3, 2, 1, 37, True, 16),   # f.size == min(res.size, s.size): fused
    (512, 1, 13, 13, 3, 4, 3, 3, 2, 1, 37, True, 16),   # f.size one past it: limb-wise
    (1024, 2, 13, 13, 2, 2, 2, 2, 2, 1, 37, True, 0),
    (1024, 2, 13, 13, 2, 2, 3, 2, 2, 1, 37, True, 16),  # one past
    (1024, 1, 18, 18, 4, 3, 1, 4, 4, 1, 1, True, 0),
    (1024, 2, 13, 13, 3, 3, 3, 2, 4, 2, 9, True, 16),   # dsize 2
    (1024, 1, 13, 18, 3, 2, 2, 3, 3, 1, 9, True, 0),    # ggsw_base2k != base2k
    (1024, 2, 18, 13, 2, 3, 1, 3, 3, 2, 5, True, 16),   # both
    (4096, 1, 18, 18, 2, 2, 2, 2, 3, 1, 3, True, 16),
    (4096, 2, 13, 13, 1, 1, 1, 1, 1, 1, 2, True, 0),
    (256, 1, 13, 13, 2, 3, 2, 2, 2, 1, 37, False, 16),
    (1024, 2, 13, 13, 2, 2, 2, 2, 2, 1, 37, False, 0),
    (1024, 1, 18, 13, 3, 2, 3, 3, 3, 2, 5, False, 16),
    (4096, 2, 18, 18, 2, 2, 1, 2, 2, 1, 3, False, 16),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-r{c[1]}-k{c[2]}.{c[3]}-s{c[4]}{c[5]}{c[6]}-d{c[7]}.{c[8]}-ds{c[9]}-b{c[10]}-"
                                             f"{'item' if c[11] else 'shared'}-p{c[12]}" for c in CASES])
def test_cmux_matches_reference(fl, case):
    n, rank, k, gk, rs, ts, fs, dnum, ss, dsize, B, per_item, pad = case
    cols = rank + 1
    rng = np.random.default_rng(sum(case[:11]) + 1000 * fl + per_item)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    t, f = fill_uniform(rng, (B, ts, cols, n), k + 4), fill_uniform(rng, (B, fs, cols, n), k + 4)
    G = 3 if per_item else 1
    mats = [fill_uniform(rng, (dnum, cols, ss, cols, n), gk) for _ in range(G)]
    idx = rng.integers(0, G, size=B) if per_item else [0]
    pm = _selectors(g, mats, idx, 8 * (pad // 16), pad, per_item)
    pos = [_prep_o(o, m) for m in mats]
    want = np.zeros((B, rs, cols, n), dtype=np.int64)
    for b in range(B):
        CR.glwe_cmux(o, want[b], t[b], f[b], k, pos[idx[b] if per_item else 0], gk, dsize)
    tv, fv = _glwe(t, pad), _glwe(f, pad)
    got0, l0 = _run(g, (B, rs, cols, n), pad, tv, fv, k, pm, gk, dsize, 0, rng)
    got1, l1 = _run(g, (B, rs, cols, n), pad, tv, fv, k, pm, gk, dsize, 1, rng)
    assert np.array_equal(got0, want)
    assert np.array_equal(got1, want)
    assert np.array_equal(_np(tv, B), t) and np.array_equal(_np(fv, B), f), "t / f were written"
    fused = per_item and dsize == 1 and gk == k and fs <= min(rs, ss) and (
        (fl == pb.NTT120 and 512 <= n <= 8192) or (fl == pb.FFT64 and ss * (n // 16) <= 1024))
    if fused:
        assert l0 <= 5 < l1, (l0, l1)  # difference + forward (+ vmp) + fused back end
    elif per_item:
        assert l0 == l1, (l0, l1)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("per_item", [True, False])
def test_cmux_bench_shape_batch_512(fl, per_item):
    """The circuit-bootstrapping bench shape: n = 1024, rank 2, base2k 13, GGSW dnum 2 x 2 limbs, GLWEs of 2 limbs, batch 512."""
    n, rank, k, B = 1024, 2, 13, 512
    cols = rank + 1
    rng = np.random.default_rng(512 + fl + per_item)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    t, f = fill_uniform(rng, (B, 2, cols, n), k), fill_uniform(rng, (B, 2, cols, n), k)
    G = 8 if per_item else 1
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(G)]
    idx = rng.integers(0, G, size=B) if per_item else [0]
    pm = _selectors(g, mats, idx, 0, 0, per_item)
    pos = [_prep_o(o, m) for m in mats]
    want = np.zeros((B, 2, cols, n), dtype=np.int64)
    for b in range(B):
        CR.glwe_cmux(o, want[b], t[b], f[b], k, pos[idx[b] if per_item else 0], k)
    tv, fv = _glwe(t, 0), _glwe(f, 0)
    for nf in (0, 1):
        got, _ = _run(g, (B, 2, cols, n), 0, tv, fv, k, pm, k, 1, nf, rng)
        assert np.array_equal(got, want), nf


def test_cmux_selector_extent_above_4_gib():
    """8192 per-item NTT120 selectors at the bench shape span 4.8 GB: every per-item offset must be 64-bit.  A few distinct GGSWs are
    replicated with pgb_memcpy_d2d; the first and the last items (and one in the middle) are checked."""
    n, rank, k, B, G = 1024, 2, 13, 8192, 4
    cols = rank + 1
    rng = np.random.default_rng(8192)
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(G)]
    pm_small = _selectors(g, mats, list(range(G)), 0, 0)
    item = pm_small.batch_stride
    assert item * B > 1 << 32
    buf = pb.DevBuf(item * B)
    idx = rng.integers(0, G, size=B)
    idx[-1] = G - 1
    for b in range(B):
        assert lib().pgb_memcpy_d2d(C.c_void_p(buf.ptr + b * item), C.c_void_p(pm_small.buf.ptr + int(idx[b]) * item), item) == 0
    pm = pb.hal.VmpPMat(buf, n, 2, cols, cols, 2, batch=B, batch_stride=item)
    t, f = fill_uniform(rng, (B, 2, cols, n), k), fill_uniform(rng, (B, 2, cols, n), k)
    tv, fv = _glwe(t, 0), _glwe(f, 0)
    pos = [_prep_o(o, m) for m in mats]
    for nf in (0, 1):
        got, _ = _run(g, (B, 2, cols, n), 0, tv, fv, k, pm, k, 1, nf, rng)
        for b in (0, B // 2 + 1, B - 1):
            want = np.zeros((2, cols, n), dtype=np.int64)
            CR.glwe_cmux(o, want, t[b], f[b], k, pos[idx[b]], k)
            assert np.array_equal(got[b], want), (nf, b)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("B,mat_pad,pmat_pad", [(1, 0, 0), (37, 8, 16), (5, 24, 48)])
def test_vmp_prepare_batched_equals_single_prepares(fl, B, mat_pad, pmat_pad):
    n, dnum, cols, size = 512, 3, 2, 3
    rng = np.random.default_rng(B + fl)
    g = pb.Module(n, fl)
    mats = [fill_uniform(rng, (dnum, cols, size, cols, n), 18) for _ in range(B)]
    pm = _selectors(g, mats, list(range(B)), mat_pad, pmat_pad)
    g.sync()
    item = n * dnum * cols * cols * size * g.prep_bytes
    got = pm.buf.download(np.uint8, (B * (item + pmat_pad),))
    for b in range(B):
        one = g.vmp_pmat_alloc(dnum, cols, cols, size)
        g.vmp_prepare(one, g.mat_znx_from_numpy(mats[b]))
        ref = one.buf.download(np.uint8, (item,))
        assert np.array_equal(got[b * (item + pmat_pad): b * (item + pmat_pad) + item], ref), b
    # one launch for the whole batch
    mbuf = pb.DevBuf(B * mats[0].nbytes)
    mbuf.upload(np.stack(mats))
    mat = pb.hal.MatZnx(mbuf, n, dnum, cols, cols, size, batch=B, batch_stride=mats[0].nbytes)
    pm2 = g.vmp_pmat_alloc(dnum, cols, cols, size, batch=B)
    before = g.launch_count
    g.vmp_prepare_batched(pm2, mat)
    g.sync()
    assert g.launch_count - before <= (2 if fl == pb.NTT120 else 1)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_vmp_prepare_batched_drops_a_pinned_keys_forms(fl):
    """A pinned key-switching key overwritten by vmp_prepare_batched is re-derived: the key-switch afterwards matches the oracle under the
    new key (the gadget kernel would otherwise keep reading the cached forms of the old one)."""
    n, k, rank, dnum, ksz, B = 1024, 18, 1, 3, 4, 64
    rng = np.random.default_rng(77 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    old, new = (fill_uniform(rng, (dnum, rank, ksz, rank + 1, n), k) for _ in range(2))
    item = n * dnum * rank * (rank + 1) * ksz * g.prep_bytes
    keys = pb.DevBuf(3 * item)
    key = pb.hal.VmpPMat(keys, n, dnum, rank, rank + 1, ksz, offset=item)
    g.vmp_prepare(key, g.mat_znx_from_numpy(old))
    g.gadget_key_pin(key)
    a = fill_uniform(rng, (B, 3, rank + 1, n), k)
    av = g.vec_znx_from_numpy(a)
    for mat in (old, new):
        if mat is new:  # rewrite all three keys in one batched prepare; the pinned one is item 1
            mb = pb.DevBuf(3 * mat.nbytes)
            mb.upload(np.stack([old, new, old]))
            g.vmp_prepare_batched(pb.hal.VmpPMat(keys, n, dnum, rank, rank + 1, ksz, batch=3, batch_stride=item),
                                  pb.hal.MatZnx(mb, n, dnum, rank, rank + 1, ksz, batch=3, batch_stride=mat.nbytes))
        res = g.vec_znx_alloc(rank + 1, 3, B)
        g.glwe_keyswitch(res, k, av, k, key, k)
        g.sync()
        got = g.vec_znx_to_numpy(res)
        want = np.zeros((B, 3, rank + 1, n), dtype=np.int64)
        o.glwe_keyswitch_batch(want, k, a, k, _prep_o(o, mat), k)
        assert np.array_equal(got, want), "new" if mat is new else "old"
    g.gadget_key_unpin(key)


# ---- rejections: each returns its status and launches nothing ---------------------------------------------------------------------------
def _cmux_raw(g, res, t, f, k, s, ggsw_stride, gk, dsize, bt, scratch, length):
    return lib().pgb_glwe_cmux_batched(g._h, C.byref(res), C.byref(t), C.byref(f), C.c_uint64(k), C.byref(s), C.c_uint64(ggsw_stride),
                                       C.c_uint64(gk), C.c_uint64(dsize), C.byref(bt), C.c_void_p(scratch), C.c_size_t(length))


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_cmux_rejections_launch_nothing(fl):
    n, cols, size, B, k = 512, 2, 2, 4, 13
    g = pb.Module(n, fl)
    item = n * cols * size * 8
    res, t, f = (pb.DevBuf(B * item) for _ in range(3))
    pm = g.vmp_pmat_alloc(2, cols, cols, size, batch=B)
    pitem = pm.batch_stride
    S = pm.struct()
    need = lib().pgb_glwe_cmux_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S),
                                         C.c_uint64(k), C.c_uint64(1), C.c_uint64(B))
    scratch = pb.DevBuf(need + 512)
    VZ = pb.hal._VZ

    def vz(buf, off=0, n_=n, cols_=cols, size_=size):
        return VZ(buf.ptr + off, n_, cols_, size_, size_)

    def call(r=None, tt=None, ff=None, s=None, gs=pitem, bt=None, sp=None, sl=None, dsize=1):
        return _cmux_raw(g, r or vz(res), tt or vz(t), ff or vz(f), k, s or S, gs, k, dsize, bt or _BT(B, item, item, item),
                         scratch.ptr if sp is None else sp, need if sl is None else sl)

    g.sync()
    before = g.launch_count
    bad = [
        (-1, dict(tt=vz(t, n_=2 * n))),                                # ring degree
        (-1, dict(ff=vz(f, cols_=3))),                                 # columns
        (-1, dict(bt=_BT(0, item, item, item))),                       # count 0
        (-1, dict(bt=_BT(65536, item, item, item))),                   # count > 65535
        (-1, dict(r=vz(res, 8))),                                      # misaligned res data
        (-1, dict(bt=_BT(B, item + 8, item, item))),                   # misaligned stride
        (-1, dict(bt=_BT(B, item, item - 16, item))),                  # stride below one item
        (-1, dict(gs=pitem + 8)),                                      # ggsw_stride not a multiple of 16
        (-1, dict(gs=16)),                                             # ggsw_stride below one GGSW
        (-4, dict(sl=need - 1)),                                       # scratch too small
        (-1, dict(sp=scratch.ptr + 16)),                               # scratch misaligned
        (-3, dict(r=vz(t))),                                           # res == t
        (-3, dict(r=vz(f, 16 * n))),                                   # res overlaps f
        (-3, dict(r=VZ(pm.buf.ptr, n, cols, size, size))),             # res overlaps a selector
        (-3, dict(sp=res.ptr)),                                        # scratch overlaps res
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert call() == 0  # the same arguments, corrected, run
    g.sync()
    # vmp_prepare_batched
    mb = pb.DevBuf(B * n * 2 * cols * cols * size * 8 + 64)
    M = pb.hal._PM(mb.ptr, n, size, 2, cols, cols)
    before = g.launch_count
    mitem = n * 2 * cols * cols * size * 8
    for status, p_, m_, bt in [(-3, pb.hal._PM(mb.ptr, n, size, 2, cols, cols), M, _BT(B, pitem, mitem, 0)),  # res overlaps a
                               (-1, S, M, _BT(B, pitem + 8, mitem, 0)),                                           # VmpPMat stride % 16
                               (-1, S, M, _BT(B, pitem, mitem + 4, 0)),                                           # MatZnx stride % 8
                               (-1, S, pb.hal._PM(mb.ptr, n, size, 3, cols, cols), _BT(B, pitem, mitem, 0)),      # shape
                               (-1, S, M, _BT(0, pitem, mitem, 0))]:
        assert lib().pgb_vmp_prepare_batched(g._h, C.byref(p_), C.byref(m_), C.byref(bt)) == status
    assert g.launch_count == before


# ---- end to end: circuit bootstrapping -> prepare_ggsw -> glwe_cmux ------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
@pytest.mark.parametrize("rank", [1, 2])
def test_circuit_bootstrap_then_cmux_on_the_device(fl, rank):
    """The noise-free setup of test_noiseless_circuit_bootstrap_on_the_device with bits {0, 1}: the device chain circuit bootstrapping ->
    circuit.prepare_ggsw -> Module.glwe_cmux over noise-free t, f must equal the oracle chain bit for bit and decrypt, exactly, to the
    message the bit selects."""
    from test_oracle_circuit_semantics import check_ggsw
    n, k, n_lwe, block, log_domain = 256, 12, 12, 3, 2
    brk_size, dnum_res, res_size, lwe_size = 4, 2, 4, 2
    cols = rank + 1
    rng = np.random.default_rng(3300 + fl + rank)
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
    bits = [0, 1, 1, 0, 1]
    B = len(bits)
    lwe = np.stack([SC.noiseless_lwe(rng, m, log_domain, s_lwe, k, lwe_size) for m in bits])
    lwe_dev = pb.DevBuf(lwe.nbytes)
    lwe_dev.upload(lwe)
    ggsw = circuit.circuit_bootstrap_to_constant(g, lwe_dev, B, n_lwe, lwe_size, k, brk_g, g.cggi_x_pow_a(), block, atk_g, tsk_g, k, rank,
                                                 dnum_res, res_size, log_domain)
    sel = circuit.prepare_ggsw(g, ggsw, B, dnum_res, rank, res_size)
    # noise-free t, f of dnum_res limbs (no digit of t - f is dropped by the product): 2-bit messages in the top bits
    rs = dnum_res
    tm, fm = rng.integers(0, 4, size=(B, n)), rng.integers(0, 4, size=(B, n))
    t = np.stack([SC.noiseless_row(rng, {0: tm[b] << (k - 2)}, s, k, rs) for b in range(B)])
    f = np.stack([SC.noiseless_row(rng, {0: fm[b] << (k - 2)}, s, k, rs) for b in range(B)])
    res = g.vec_znx_alloc(cols, rs, B)
    g.glwe_cmux(res, g.vec_znx_from_numpy(t), g.vec_znx_from_numpy(f), k, sel, k)
    g.sync()
    got = g.vec_znx_to_numpy(res)
    xpa = o.cggi_x_pow_a()
    # decryption error: the GGSW's (check_ggsw bounds, in units of 2^-(res_size k)) times the product's digits (|digit| <= 2^(k-1), n terms,
    # dnum rows, every column), plus the rounding of the product to rs limbs
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c == 0 else n // 8) for c in range(cols))
    bound = (dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n)
    assert bound < 1 << (rs * k - 2 - 5)  # 2^5 below the lowest message bit
    for b, m in enumerate(bits):
        mat = SC.circuit_bootstrap_to_constant_ref(o, lwe[b], k, brk_o, xpa, block, atk_o, tsk_o, rank, dnum_res, res_size, log_domain, brk_size)
        check_ggsw(mat, m, s, k, res_size)
        want = np.zeros((rs, cols, n), dtype=np.int64)
        CR.glwe_cmux(o, want, t[b], f[b], k, _prep_o(o, mat), k)
        assert np.array_equal(got[b], want), b
        msg = tm[b] if m else fm[b]
        ph = SC.phase_scaled(got[b], s, k)
        mod = 1 << (rs * k)
        err = max(abs(((p - (int(x) << (rs * k - 2)) + (mod >> 1)) % mod) - (mod >> 1)) for p, x in zip(ph, msg))
        assert err <= bound, (b, err, bound)
