"""GPU parity of the blind rotation by GGSW bits (pgb_glwe_blind_rotate_ggsw_batched) with tests/glwe_blind_rotate_ref.py, bit for bit, both
flavours: n = 256 .. 4096; rank 1 and 2; base2k 13 and 18 and ggsw_base2k != base2k; dsize 1 and 2; a.size below, at and above res.size;
res.size at and just past s.size (where the fused routes hand over); n_bits 1, 2, 5, 8 with steps positive, negative, odd and past 2n;
shared selectors, per-item selectors in the bit-major and the ciphertext-major layouts with padded strides, and a shared `a`; batches 1, 37
and 512 at the circuit-bootstrapping bench shape; default routes against PGB_OPT_NO_FUSION.  Every case also runs today's composition on the
device (rotate every column into t, then glwe_cmux) and checks that the entry launches exactly what its CMuxes launch.  Then a selector
extent above 4 GiB, the rejections, and circuit bootstrapping -> prepare_ggsw -> glwe_blind_rotate_ggsw -> sample extraction end to end."""
import ctypes as C

import numpy as np
import pytest

import glwe_blind_rotate_ref as BR
import lwe_ref as LR
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.hal import _BT, lib
from test_gpu_cmux import _glwe, _np, _prep_o, _selectors
from test_oracle_glwe_blind_rotate import rotate_ints
from util import fill_uniform

import poulpy_b200 as pb

pytestmark = pytest.mark.gpu


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def _layout(mode, B, L, item):
    """(ggsw_stride, bit_stride, the selector index of (b, i)) of the three layouts over items `item` bytes apart."""
    if mode == "shared":
        return 0, item, lambda b, i: i
    if mode == "bit":  # bit-major within a ciphertext: circuit.prepare_ggsw over B * L bits
        return L * item, item, lambda b, i: b * L + i
    return item, B * item, lambda b, i: i * B + b  # ciphertext-major


def _with_fusion(g, no_fusion, fn):
    g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
    try:
        return fn()
    finally:
        g.set_option(pb.hal.OPT_NO_FUSION, 0)


def _run(g, res_shape, pad, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize, rng):
    res = _glwe(fill_uniform(rng, res_shape, 50), pad)  # garbage pre-fill
    before = g.launch_count
    g.glwe_blind_rotate_ggsw(res, av, k, step, L, pm, gk, dsize, ggsw_stride=ggsw_stride, bit_stride=bit_stride)
    g.sync()
    return _np(res, res_shape[0]), g.launch_count - before


def _compose(g, res_shape, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize):
    """Today's composition: per bit, rotate every column of acc into t, then glwe_cmux(t, acc).  Returns the result and the launches of the
    CMuxes alone."""
    B, rs, cols, n = res_shape
    cur, cmux_launches = av, 0
    for i in range(L):
        t = g.vec_znx_alloc(cols, cur.size, B)
        bt = _BT(B, t.batch_stride, cur.batch_stride if cur.batch > 1 else 0, 0)
        p = BR.rotation(step, i, n)
        for c in range(cols):
            r, a = t.struct(), cur.struct()
            pb.hal._check(lib().pgb_vec_znx_rotate_batched(g._h, C.c_int64(p), C.byref(r), C.c_uint64(c), C.byref(a), C.c_uint64(c), C.byref(bt)))
        nxt = g.vec_znx_alloc(cols, rs, B)
        sel = pb.hal.VmpPMat(pm.buf, n, pm.rows, cols, cols, pm.size, offset=pm.offset + i * bit_stride, batch=B, batch_stride=ggsw_stride)
        before = g.launch_count
        g.glwe_cmux(nxt, t, cur, k, sel, gk, dsize)
        cmux_launches += g.launch_count - before
        cur = nxt
    g.sync()
    return g.vec_znx_to_numpy(cur).reshape(res_shape), cmux_launches


def _fused_bit(fl, n, k, gk, f_size, rs, ss, dsize, mode):
    """The CMux's condition for its per-item fused routes."""
    return mode != "shared" and dsize == 1 and gk == k and f_size <= min(rs, ss) and (
        (fl == pb.NTT120 and 512 <= n <= 8192) or (fl == pb.FFT64 and ss * (n // 16) <= 1024))


def _check_case(fl, g, o, a, a_shared, B, rs, cols, n, k, gk, dnum, ss, dsize, mode, pad, L, step, mats, rng, sample=None):
    G = len(mats)
    ggsw_stride_items, bit_stride_items, q = _layout(mode, B, L, 1)
    n_sel = L if mode == "shared" else B * L
    idx = rng.integers(0, G, size=n_sel)
    pm = _selectors(g, mats, idx, 8 * (pad // 16), pad)
    item = pm.batch_stride
    ggsw_stride, bit_stride = ggsw_stride_items * item, bit_stride_items * item
    pos = [_prep_o(o, m) for m in mats]
    items = range(B) if sample is None else sample
    want = {}
    for b in items:
        w = np.zeros((rs, cols, n), dtype=np.int64)
        BR.glwe_blind_rotate_ggsw(o, w, a[0 if a_shared else b], k, step, [pos[idx[q(b, i)]] for i in range(L)], gk, dsize)
        want[b] = w
    av = _glwe(a, pad)
    shape = (B, rs, cols, n)
    got0, l0 = _with_fusion(g, 0, lambda: _run(g, shape, pad, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize, rng))
    got1, l1 = _with_fusion(g, 1, lambda: _run(g, shape, pad, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize, rng))
    for b in items:
        assert np.array_equal(got0[b], want[b]), ("default", b)
        assert np.array_equal(got1[b], want[b]), ("no fusion", b)
    assert np.array_equal(_np(av, a.shape[0]), a), "a was written"
    comp0, c0 = _with_fusion(g, 0, lambda: _compose(g, shape, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize))
    comp1, c1 = _with_fusion(g, 1, lambda: _compose(g, shape, av, k, step, L, pm, ggsw_stride, bit_stride, gk, dsize))
    assert np.array_equal(comp0, got0) and np.array_equal(comp1, got1), "the composition differs"
    assert (l0, l1) == (c0, c1), (l0, l1, c0, c1)
    if all(_fused_bit(fl, n, k, gk, a.shape[1] if i == 0 else rs, rs, ss, dsize, mode) for i in range(L)):
        assert l0 < l1, (l0, l1)


# n, rank, k, gk, res_size, a_size, dnum, s_size, dsize, batch, selectors, pad, n_bits, step, a shared
CASES = [
    (256, 1, 13, 13, 2, 2, 2, 2, 1, 37, "bit", 16, 5, 3, False),
    (256, 2, 18, 18, 3, 1, 3, 3, 1, 5, "ct", 0, 2, -1, False),
    (512, 1, 13, 13, 2, 2, 3, 2, 1, 37, "bit", 16, 8, 1, True),      # res.size == s.size: fused on every bit
    (512, 1, 13, 13, 3, 3, 3, 2, 1, 9, "bit", 16, 5, -5, False),     # res.size one past s.size: limb-wise
    (1024, 2, 13, 13, 2, 3, 2, 2, 1, 9, "ct", 16, 8, 37, False),     # a above res: bit 0 limb-wise, the rest fused; step 2^i passes 2n
    (1024, 2, 13, 13, 3, 2, 2, 3, 1, 9, "bit", 0, 5, -300, True),    # a below res
    (1024, 1, 18, 18, 4, 4, 4, 4, 1, 1, "bit", 0, 8, 1023, False),
    (1024, 2, 13, 13, 3, 3, 2, 4, 2, 9, "ct", 16, 2, 7, False),      # dsize 2
    (1024, 1, 13, 18, 3, 2, 3, 3, 1, 9, "bit", 0, 5, -3, False),     # ggsw_base2k != base2k
    (1024, 2, 18, 13, 2, 3, 3, 3, 2, 5, "ct", 16, 2, 5, True),       # both
    (4096, 1, 18, 18, 2, 2, 2, 3, 1, 3, "bit", 16, 5, -1, False),
    (4096, 2, 13, 13, 1, 1, 1, 1, 1, 2, "ct", 0, 2, 4095, False),
    (256, 1, 13, 13, 2, 3, 2, 2, 1, 37, "shared", 16, 5, 3, False),
    (1024, 2, 13, 13, 2, 2, 2, 2, 1, 37, "shared", 0, 8, -1, True),
    (1024, 1, 18, 13, 3, 2, 3, 3, 2, 5, "shared", 16, 2, 5, False),
    (4096, 2, 18, 18, 2, 2, 2, 2, 1, 3, "shared", 16, 1, -7, False),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-r{c[1]}-k{c[2]}.{c[3]}-s{c[4]}.{c[5]}-d{c[6]}.{c[7]}-ds{c[8]}-b{c[9]}-{c[10]}-p{c[11]}-"
                                             f"L{c[12]}-step{c[13]}{'-ashared' if c[14] else ''}" for c in CASES])
def test_blind_rotate_matches_reference(fl, case):
    n, rank, k, gk, rs, as_, dnum, ss, dsize, B, mode, pad, L, step, a_shared = case
    cols = rank + 1
    rng = np.random.default_rng(sum(map(abs, case[:10])) + 17 * L + 1000 * fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    a = fill_uniform(rng, (1 if a_shared else B, as_, cols, n), k + 4)
    mats = [fill_uniform(rng, (dnum, cols, ss, cols, n), gk) for _ in range(3)]
    _check_case(fl, g, o, a, a_shared, B, rs, cols, n, k, gk, dnum, ss, dsize, mode, pad, L, step, mats, rng)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("B,mode", [(1, "bit"), (37, "ct"), (37, "shared"), (512, "bit"), (512, "ct")])
def test_blind_rotate_bench_shape(fl, B, mode):
    """The circuit-bootstrapping bench shape: n = 1024, rank 2, base2k 13, GGSW dnum 2 x 2 limbs, GLWEs of 2 limbs, 8 bits.  At batch 512
    the reference checks a seeded sample of 24 items (the first and the last among them)."""
    n, rank, k, L = 1024, 2, 13, 8
    cols = rank + 1
    rng = np.random.default_rng(B + 3 * fl + len(mode))
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    a = fill_uniform(rng, (B, 2, cols, n), k)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(8)]
    sample = None if B < 512 else sorted({0, B - 1, *rng.choice(B, 22, replace=False).tolist()})
    _check_case(fl, g, o, a, False, B, 2, cols, n, k, k, 2, 2, 1, mode, 0, L, -3, mats, rng, sample)


def test_blind_rotate_selector_extent_above_4_gib():
    """2048 ciphertexts x 4 bits of per-item NTT120 selectors at the bench shape span 4.8 GB, bit-major: every (b, i) offset must be 64-bit.
    A few distinct GGSWs are replicated with pgb_memcpy_d2d; the first, a middle and the last items are checked."""
    n, rank, k, B, L, G = 1024, 2, 13, 2048, 4, 4
    cols = rank + 1
    rng = np.random.default_rng(4096)
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    mats = [fill_uniform(rng, (2, cols, 2, cols, n), k) for _ in range(G)]
    pm_small = _selectors(g, mats, list(range(G)), 0, 0)
    item = pm_small.batch_stride
    assert item * B * L > 1 << 32
    buf = pb.DevBuf(item * B * L)
    idx = rng.integers(0, G, size=B * L)
    idx[-L:] = np.arange(L) % G  # the last item reads every distinct GGSW
    for q in range(B * L):
        assert lib().pgb_memcpy_d2d(C.c_void_p(buf.ptr + q * item), C.c_void_p(pm_small.buf.ptr + int(idx[q]) * item), item) == 0
    pm = pb.hal.VmpPMat(buf, n, 2, cols, cols, 2, batch=B * L, batch_stride=item)
    a = fill_uniform(rng, (B, 2, cols, n), k)
    av = _glwe(a, 0)
    pos = [_prep_o(o, m) for m in mats]
    for nf in (0, 1):
        got, _ = _with_fusion(g, nf, lambda: _run(g, (B, 2, cols, n), 0, av, k, 5, L, pm, L * item, item, k, 1, rng))
        for b in (0, B // 2 + 1, B - 1):
            want = np.zeros((2, cols, n), dtype=np.int64)
            BR.glwe_blind_rotate_ggsw(o, want, a[b], k, 5, [pos[idx[b * L + i]] for i in range(L)], k)
            assert np.array_equal(got[b], want), (nf, b)


# ---- rejections: each returns its status and launches nothing ---------------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_blind_rotate_rejections_launch_nothing(fl):
    n, cols, size, B, L, k = 512, 2, 2, 4, 3, 13
    g = pb.Module(n, fl)
    item = n * cols * size * 8
    res, a = (pb.DevBuf(B * item) for _ in range(2))
    pm = g.vmp_pmat_alloc(2, cols, cols, size, batch=B * L + B)  # B spare items after the B * L selectors: room for a misplaced res
    pitem = pm.batch_stride
    S = pm.struct()
    need = lib().pgb_glwe_blind_rotate_ggsw_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S), C.c_uint64(k),
                                                      C.c_uint64(1), C.c_uint64(L), C.c_uint64(B))
    one = lib().pgb_glwe_cmux_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S), C.c_uint64(k),
                                        C.c_uint64(1), C.c_uint64(B))
    assert need == -(-B * item // 256) * 256 + one  # the ping-pong accumulator + one CMux's scratch
    assert lib().pgb_glwe_blind_rotate_ggsw_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(S), C.c_uint64(k),
                                                      C.c_uint64(1), C.c_uint64(1), C.c_uint64(B)) == one
    scratch = pb.DevBuf(need + 512)
    VZ = pb.hal._VZ

    def vz(buf_ptr, n_=n, cols_=cols, size_=size):
        return VZ(buf_ptr, n_, cols_, size_, size_)

    def call(r=None, aa=None, step=3, nb=L, s=None, gs=L * pitem, bs=pitem, bt=None, sp=None, sl=None, dsize=1):
        return lib().pgb_glwe_blind_rotate_ggsw_batched(
            g._h, C.byref(r or vz(res.ptr)), C.byref(aa or vz(a.ptr)), C.c_uint64(k), C.c_int64(step), C.c_uint64(nb), C.byref(s or S),
            C.c_uint64(gs), C.c_uint64(bs), C.c_uint64(k), C.c_uint64(dsize), C.byref(bt or _BT(B, item, item, 0)),
            C.c_void_p(scratch.ptr if sp is None else sp), C.c_size_t(need if sl is None else sl))

    last = (B - 1) * L * pitem + (L - 1) * pitem  # the last selector (b, i) = (B - 1, L - 1)
    g.sync()
    before = g.launch_count
    bad = [
        (-1, dict(aa=vz(a.ptr, n_=2 * n))),                            # ring degree
        (-1, dict(aa=vz(a.ptr, cols_=3))),                             # columns
        (-1, dict(bt=_BT(0, item, item, 0))),                          # count 0
        (-1, dict(bt=_BT(65536, item, item, 0))),                      # count > 65535
        (-1, dict(bt=_BT(B, item, item, item))),                       # stride_b != 0
        (-1, dict(nb=0)),                                              # n_bits 0
        (-1, dict(nb=65)),                                             # n_bits > 64
        (-1, dict(r=vz(res.ptr + 8))),                                 # misaligned res data
        (-1, dict(bt=_BT(B, item, item + 8, 0))),                      # misaligned a stride
        (-1, dict(gs=L * pitem + 8)),                                  # ggsw_stride not a multiple of 16
        (-1, dict(gs=16)),                                             # ggsw_stride below one GGSW
        (-1, dict(bs=pitem + 8)),                                      # bit_stride not a multiple of 16
        (-1, dict(bs=16)),                                             # bit_stride below one GGSW
        (-1, dict(bs=0)),                                              # bit_stride 0 with n_bits > 1
        (-1, dict(gs=1 << 62, bs=1 << 62)),                            # selectors past the end of the address space
        (-4, dict(sl=need - 1)),                                       # scratch too small
        (-1, dict(sp=scratch.ptr + 16)),                               # scratch misaligned
        (-3, dict(r=vz(a.ptr))),                                       # res == a
        (-3, dict(r=vz(a.ptr + 16 * n))),                              # res overlaps a
        (-3, dict(r=vz(pm.buf.ptr + last))),                           # res overlaps only the last selector
        (-3, dict(sp=pm.buf.ptr + last // 256 * 256)),                 # scratch overlaps the last selectors
        (-3, dict(sp=res.ptr)),                                        # scratch overlaps res
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert call() == 0  # the same arguments, corrected, run
    assert call(nb=1, bs=0) == 0  # bit_stride is not read for one bit
    g.sync()


# ---- end to end: circuit bootstrapping -> prepare_ggsw -> glwe_blind_rotate_ggsw (-> sample extraction) ---------------------------------
@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
@pytest.mark.parametrize("rank", [1, 2])
def test_circuit_bootstrap_then_lut_rotation_on_the_device(fl, rank):
    """Vertical packing of one lookup table on circuit-bootstrapped bits: B * L noise-free LWE bits (bit i of m_b is LWE b * L + i) are
    circuit-bootstrapped, prepared with circuit.prepare_ggsw (bit-major, the default strides) and rotate one shared noise-free LUT GLWE
    sum_j LUT[j] X^(j spacing) by step = -spacing.  The device chain must equal the oracle chain bit for bit and the phase must be the LUT
    rotated by -spacing m_b within L times the CMux test's bound; at rank 1 the extracted LWE must equal the oracle's and decrypt to
    LUT[m_b]."""
    from test_oracle_circuit_semantics import check_ggsw
    n, k, n_lwe, block, log_domain = 256, 12, 12, 3, 2
    brk_size, dnum_res, res_size, lwe_size = 4, 2, 4, 2
    L = 3
    spacing = n >> L
    cols = rank + 1
    rng = np.random.default_rng(5300 + fl + rank)
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
    ms = [5, 0, 7, 2]
    B = len(ms)
    bits = [(m >> i) & 1 for m in ms for i in range(L)]
    lwe = np.stack([SC.noiseless_lwe(rng, m, log_domain, s_lwe, k, lwe_size) for m in bits])
    lwe_dev = pb.DevBuf(lwe.nbytes)
    lwe_dev.upload(lwe)
    ggsw = circuit.circuit_bootstrap_to_constant(g, lwe_dev, B * L, n_lwe, lwe_size, k, brk_g, g.cggi_x_pow_a(), block, atk_g, tsk_g, k, rank,
                                                 dnum_res, res_size, log_domain)
    sel = circuit.prepare_ggsw(g, ggsw, B * L, dnum_res, rank, res_size)
    # one noise-free LUT GLWE of dnum_res limbs: 2-bit entries in the top bits
    rs = dnum_res
    lut = rng.integers(0, 4, size=1 << L)
    poly = np.zeros(n, dtype=np.int64)
    poly[::spacing] = lut
    a = SC.noiseless_row(rng, {0: poly << (k - 2)}, s, k, rs)
    res = g.vec_znx_alloc(cols, rs, B)
    g.glwe_blind_rotate_ggsw(res, g.vec_znx_from_numpy(a), k, -spacing, L, sel, k)
    g.sync()
    got = g.vec_znx_to_numpy(res)
    if rank == 1:
        lwe_out = pb.DevBuf(B * rs * (n + 1) * 8)
        g.lwe_sample_extract(lwe_out, n, rs, res)
        g.sync()
        got_lwe = lwe_out.download(np.int64, (B, rs, 1, n + 1))
        s_ext = np.concatenate([s[0][:1], -s[0][:0:-1]])  # the LWE secret of the extraction: s_glwe(X) = s_lwe(X^-1)
    xpa = o.cggi_x_pow_a()
    # per CMux as in test_circuit_bootstrap_then_cmux_on_the_device, times the L CMuxes
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c == 0 else n // 8) for c in range(cols))
    bound = L * ((dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n))
    assert bound < 1 << (rs * k - 2 - 5)  # 2^5 below the lowest message bit
    mod = 1 << (rs * k)
    base = SC.phase_scaled(a, s, k)
    for b, m in enumerate(ms):
        sels = []
        for i in range(L):
            mat = SC.circuit_bootstrap_to_constant_ref(o, lwe[b * L + i], k, brk_o, xpa, block, atk_o, tsk_o, rank, dnum_res, res_size,
                                                       log_domain, brk_size)
            check_ggsw(mat, bits[b * L + i], s, k, res_size)
            sels.append(_prep_o(o, mat))
        want = np.zeros((rs, cols, n), dtype=np.int64)
        BR.glwe_blind_rotate_ggsw(o, want, a, k, -spacing, sels, k)
        assert np.array_equal(got[b], want), b
        ph = SC.phase_scaled(got[b], s, k)
        err = max(abs(((p - w + (mod >> 1)) % mod) - (mod >> 1)) for p, w in zip(ph, rotate_ints(base, -spacing * m, n)))
        assert err <= bound, (b, err, bound)
        if rank == 1:
            want_lwe = np.zeros((rs, 1, n + 1), dtype=np.int64)
            LR.lwe_sample_extract(want_lwe, want)
            assert np.array_equal(got_lwe[b], want_lwe), b
            dec = sum(int(got_lwe[b, j, 0, 0] + np.dot(got_lwe[b, j, 0, 1:], s_ext)) << ((rs - 1 - j) * k) for j in range(rs))
            e = ((dec - (int(lut[m]) << (rs * k - 2)) + (mod >> 1)) % mod) - (mod >> 1)
            assert abs(e) <= bound, (b, e, bound)
