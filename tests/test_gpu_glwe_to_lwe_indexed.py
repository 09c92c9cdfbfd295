"""GPU parity of glwe_to_lwe at many coefficients (pgb_glwe_to_lwe_indexed_batched, Module.glwe_to_lwe_indexed), both flavours, bit for
bit: against the reference of tests/lwe_indexed_ref.py and against the device twin composition (one glwe_keyswitch, then per index one
batched rotation and one lwe_sample_extract), at n = 256 .. 4096, ranks 1 and 2, mixed base2k, dsize 2, n_index 1, 9, 32 and N, padded
entry and item strides (the padding left untouched), a ragged batch of 37 and a batch of 4096, default routes and PGB_OPT_NO_FUSION.
Then the launch count (that of glwe_to_lwe, whatever n_index), index {0} against Module.glwe_to_lwe, every rejection (each launching
nothing), and two integer additions chained through packed GLWEs on the device: packed -> circuit.ggsw_bits_from_packed -> the 8-bit
adder -> circuit.bdd_eval_packed -> ggsw_bits_from_packed again."""
import ctypes as C
import types
from fractions import Fraction

import numpy as np
import pytest

import lwe_indexed_ref as R
import lwe_ref as LR
import semantics_circuit as SC
import poulpy_b200 as pb
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.circuit import bdd_from_truth_tables
from poulpy_b200.hal import _BT, _VZ, lib
from test_gpu_cmux import _prep_o
from test_gpu_lwe import _glwe, _in_size, _key
from test_oracle_bdd import ADD8, INTERLEAVED
from test_oracle_cmux_tree import lwe_phase as ring_lwe_phase
from test_oracle_lwe import embed_secret
from test_oracle_semantics import noiseless_ksk
from util import fill_uniform

pytestmark = pytest.mark.gpu
SHAPE, ALIAS, SCRATCH = -1, -3, -4


def _index(rng, n, n_index):
    if n_index == n:
        return [int(x) for x in rng.permutation(n)]
    head = [0, 1, n - 1][:n_index]
    return head + [int(x) for x in rng.integers(0, n, size=n_index - len(head))]  # duplicates allowed


def _lwes(raw, n_index, size, n_lwe, entry_stride):
    """-> (B, n_index, size, 1, n_lwe + 1) entries and the bytes between them, from the bytes (B, res_stride) of B items."""
    B, res_stride = raw.shape
    lwe = size * (n_lwe + 1) * 8
    out = np.zeros((B, n_index, size, 1, n_lwe + 1), dtype=np.int64)
    mask = np.ones((B, res_stride), dtype=bool)
    for j in range(n_index):
        out[:, j] = raw[:, j * entry_stride: j * entry_stride + lwe].copy().view(np.int64).reshape(B, size, 1, n_lwe + 1)
        mask[:, j * entry_stride: j * entry_stride + lwe] = False
    return out, raw[mask]


def _twin(g, a, n_lwe, res_size, res_k, a_k, kg, key_k, dsize, index):
    """One glwe_keyswitch of the batch, then per index one batched rotation per column and one lwe_sample_extract (default layout)."""
    B = a.batch
    lwe = res_size * (n_lwe + 1) * 8
    staged, rot = g.vec_znx_alloc(2, res_size, B), g.vec_znx_alloc(2, res_size, B)
    g.glwe_keyswitch(staged, res_k, a, a_k, kg, key_k, dsize)
    out = pb.DevBuf(B * len(index) * lwe)
    r, s = rot.struct(), staged.struct()
    bt = _BT(B, rot.batch_stride, staged.batch_stride, 0)
    for j, idx in enumerate(index):
        for c in range(2):
            pb.hal._check(lib().pgb_vec_znx_rotate_batched(g._h, C.c_int64(-idx), C.byref(r), C.c_uint64(c), C.byref(s), C.c_uint64(c),
                                                         C.byref(bt)))
        g.lwe_sample_extract(types.SimpleNamespace(ptr=out.ptr + j * lwe), n_lwe, res_size, rot, res_stride=len(index) * lwe)
    return out


# n, rank, a_size, res_size, a_k, key_k, res_k, dsize, n_lwe, n_index, batch, pad
CASES = [
    (256, 1, 2, 2, 12, 12, 12, 1, 256, 256, 5, 0),
    (512, 2, 3, 2, 12, 12, 12, 2, 511, 9, 37, 8),
    (1024, 2, 2, 2, 13, 13, 13, 1, 687, 32, 16, 8),
    (1024, 1, 4, 3, 12, 15, 13, 1, 1024, 1, 7, 0),
    (2048, 1, 3, 3, 13, 11, 12, 2, 600, 9, 4, 8),
    (4096, 2, 2, 2, 18, 18, 18, 1, 33, 4096, 2, 0),
    (4096, 1, 1, 2, 18, 18, 18, 2, 1023, 32, 3, 8),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("no_fusion", [0, 1])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-r{c[1]}-s{c[2]}{c[3]}-k{c[4]}.{c[5]}.{c[6]}-d{c[7]}-lwe{c[8]}-idx{c[9]}-b{c[10]}-p{c[11]}"
                                             for c in CASES])
def test_indexed_matches_reference_and_twin(fl, no_fusion, case):
    n, rank, a_size, res_size, a_k, key_k, res_k, dsize, n_lwe, n_index, B, pad = case
    rng = np.random.default_rng(n + 3 * rank + 7 * n_index + dsize + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
    in_size = _in_size(a_size, a_k, key_k)
    kg, ko = _key(rng, g, o, -(-in_size // dsize), rank, 2, in_size + 1, key_k)
    index = _index(rng, n, n_index)
    host = fill_uniform(rng, (B, a_size, rank + 1, n), a_k)
    a = _glwe(g, host, pad)
    lwe = res_size * (n_lwe + 1) * 8
    es, rs = lwe + pad, n_index * (lwe + pad) + 2 * pad
    garbage = fill_uniform(rng, (B * rs // 8,), 64)
    res = pb.DevBuf(B * rs)
    res.upload(garbage)
    g.glwe_to_lwe_indexed(res, n_lwe, res_size, res_k, a, a_k, index, kg, key_k, dsize, entry_stride=es, res_stride=rs)
    twin = _twin(g, a, n_lwe, res_size, res_k, a_k, kg, key_k, dsize, index)
    g.sync()
    got, gaps = _lwes(res.download(np.uint8, (B, rs)), n_index, res_size, n_lwe, es)
    _, want_gaps = _lwes(garbage.view(np.uint8).reshape(B, rs), n_index, res_size, n_lwe, es)
    assert np.array_equal(gaps, want_gaps), "the padding between entries was written"
    assert np.array_equal(got, twin.download(np.int64, got.shape)), "twin"
    want = np.zeros((n_index, res_size, 1, n_lwe + 1), dtype=np.int64)
    for b in range(B):
        R.glwe_to_lwe_indexed(o, want, res_k, host[b], a_k, index, ko, key_k, dsize)
        assert np.array_equal(got[b], want), ("reference", b)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_batch_4096_at_the_bench_shape(fl):
    """n = 1024, rank 2, base2k 13 (the circuit-bootstrapping bench shape), n_index 9, 4096 items: the twin for all, the reference for three."""
    n, rank, k, size, n_lwe, B = 1024, 2, 13, 2, 687, 4096
    rng = np.random.default_rng(5100 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    kg, ko = _key(rng, g, o, size, rank, 2, size + 1, k)
    index = _index(rng, n, 9)
    host = fill_uniform(rng, (B, size, rank + 1, n), k)
    a = g.vec_znx_from_numpy(host)
    res = pb.DevBuf(B * 9 * size * (n_lwe + 1) * 8)
    g.glwe_to_lwe_indexed(res, n_lwe, size, k, a, k, index, kg, k)
    twin = _twin(g, a, n_lwe, size, k, k, kg, k, 1, index)
    g.sync()
    shape = (B, 9, size, 1, n_lwe + 1)
    got = res.download(np.int64, shape)
    assert np.array_equal(got, twin.download(np.int64, shape))
    want = np.zeros(shape[1:], dtype=np.int64)
    for b in (0, 2047, B - 1):
        R.glwe_to_lwe_indexed(o, want, k, host[b], k, index, ko, k)
        assert np.array_equal(got[b], want), b


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("no_fusion", [0, 1])
def test_launch_count_and_index_zero(fl, no_fusion):
    """The entry launches what glwe_to_lwe launches at the same shape, for every n_index; index {0} equals glwe_to_lwe bit for bit."""
    n, rank, k, size, n_lwe, B = 1024, 2, 13, 2, 687, 24
    rng = np.random.default_rng(5200 + fl + no_fusion)
    g = pb.Module(n, fl)
    g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
    kg, _ = _key(rng, g, O.OracleModule(n, fl), size, rank, 2, size + 1, k)
    a = g.vec_znx_from_numpy(fill_uniform(rng, (B, size, rank + 1, n), k))
    lwe = size * (n_lwe + 1) * 8
    plain = pb.DevBuf(B * lwe)
    g.glwe_to_lwe(plain, n_lwe, size, k, a, k, kg, k)  # warm: key forms, scratch
    g.sync()
    before = g.launch_count
    g.glwe_to_lwe(plain, n_lwe, size, k, a, k, kg, k)
    want = g.launch_count - before
    for n_index in (1, 9, 32, n):
        index = [0] if n_index == 1 else _index(rng, n, n_index)
        res = pb.DevBuf(B * n_index * lwe)
        before = g.launch_count
        g.glwe_to_lwe_indexed(res, n_lwe, size, k, a, k, index, kg, k)
        assert g.launch_count - before == want, n_index
        if n_index == 1:
            g.sync()
            assert np.array_equal(res.download(np.int64, (B * lwe // 8,)), plain.download(np.int64, (B * lwe // 8,)))
    g.sync()


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_indexed_rejections_launch_nothing(fl):
    n, k, B, size, rank, n_lwe = 512, 18, 3, 2, 2, 100
    g = pb.Module(n, fl)
    lwe = size * (n_lwe + 1) * 8
    glwe_bs = n * (rank + 1) * size * 8
    n_index = 4
    big = pb.DevBuf(8 * B * n_index * lwe + 2 * B * glwe_bs)
    glwe_off = 4 * B * n_index * lwe
    a = _VZ(big.ptr + glwe_off, n, rank + 1, size, size)
    res = _VZ(big.ptr, n_lwe + 1, 1, size, size)
    key = g.vmp_pmat_alloc(size, rank, 2, size + 1)
    ks = key.struct()
    idx = np.array([0, 1, n - 1, 7], dtype=np.uint32)
    scratch = pb.DevBuf(64 << 20)

    def tmp(ni=n_index, count=B):
        return int(lib().pgb_glwe_to_lwe_indexed_tmp_bytes(g._h, C.c_uint64(size), C.c_uint64(size), C.c_uint64(k), C.byref(ks), C.c_uint64(k),
                                                           C.c_uint64(1), C.c_uint64(ni), C.c_uint64(count)))

    def call(r=res, es=lwe, av=a, ix=idx, ni=n_index, kk=ks, bt=None, sc=scratch.ptr, sl=64 << 20):
        bt = _BT(B, n_index * lwe, glwe_bs, 0) if bt is None else bt
        ip = None if ix is None else ix.ctypes.data_as(C.POINTER(C.c_uint32))
        return lib().pgb_glwe_to_lwe_indexed_batched(g._h, C.byref(r), C.c_uint64(es), C.c_uint64(k), C.byref(av), C.c_uint64(k), ip,
                                                     C.c_uint64(ni), C.byref(kk), C.c_uint64(k), C.c_uint64(1), C.byref(bt),
                                                     C.c_void_p(sc), C.c_size_t(sl))

    before = g.launch_count
    bad = [
        (SHAPE, dict(ix=None)),                                                        # no index table
        (SHAPE, dict(ni=0)),
        (SHAPE, dict(ix=np.arange(n + 1, dtype=np.uint32), ni=n + 1)),                 # more than N entries
        (SHAPE, dict(ix=np.array([0, 1, n, 7], dtype=np.uint32))),                     # an index at N
        (SHAPE, dict(es=lwe - 8)),                                                     # entries overlap
        (SHAPE, dict(es=lwe + 4)),                                                     # entry stride not a multiple of 8
        (SHAPE, dict(bt=_BT(B, n_index * lwe - 8, glwe_bs, 0))),                       # items overlap
        (SHAPE, dict(bt=_BT(B, n_index * lwe + 4, glwe_bs, 0))),
        (SHAPE, dict(es=1 << 61, bt=_BT(B, 1 << 63, glwe_bs, 0))),                     # extents past 2^64 (128-bit arithmetic)
        (SHAPE, dict(bt=_BT(0, n_index * lwe, glwe_bs, 0))),
        (SHAPE, dict(bt=_BT(65536, n_index * lwe, glwe_bs, 0))),
        (SHAPE, dict(r=_VZ(big.ptr + 4, n_lwe + 1, 1, size, size))),                   # misaligned LWE data
        (SHAPE, dict(r=_VZ(big.ptr, n + 2, 1, size, size))),                           # n_lwe > N
        (SHAPE, dict(av=_VZ(a.data, n // 2, rank + 1, size, size))),                   # ring mismatch
        (SHAPE, dict(kk=g.vmp_pmat_alloc(size, rank + 1, 2, size + 1).struct())),      # key rank
        (SHAPE, dict(bt=_BT(B, n_index * lwe, glwe_bs + 8, 0))),                       # GLWE stride not a multiple of 16
        (SHAPE, dict(sc=scratch.ptr + 128)),                                           # misaligned scratch
        (ALIAS, dict(r=_VZ(a.data, n_lwe + 1, 1, size, size))),                        # res on a
        (ALIAS, dict(r=_VZ(a.data - (B - 1) * n_index * lwe - 3 * lwe, n_lwe + 1, 1, size, size))),  # only the last item's last entry on a
        (SCRATCH, dict(sl=tmp() - 1)),
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert tmp(1) < tmp(n) and tmp(n, 2) - tmp(n, 1) == tmp(1, 2) - tmp(1, 1)  # the staged GLWEs are per item, the table per index
    assert call(sl=tmp()) == 0, lib().pgb_last_error()
    assert call(ix=np.array([5, 5, 5, 5], dtype=np.uint32)) == 0  # duplicates
    assert call(es=0, ni=1, bt=_BT(B, lwe, glwe_bs, 0)) == 0       # one entry: any entry stride
    g.sync()


# ---- end to end: two additions chained through packed GLWEs ------------------------------------------------------------------------------
def _lwe_int_phase(lwe, s_lwe, k):
    """b + <a, s_lwe> of an LWE (size, 1, n_lwe + 1) as an integer modulo 2^(size k)."""
    size = lwe.shape[0]
    return sum(int(lwe[j, 0, 0] + np.dot(lwe[j, 0, 1:], s_lwe)) << ((size - 1 - j) * k) for j in range(size)) % (1 << (size * k))


def _centred(x, mod):
    return ((x + (mod >> 1)) % mod) - (mod >> 1)


@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
def test_two_additions_chained_through_packed_glwes_on_the_device(fl):
    """x and y (8 bits, bit i at coefficient i of a noise-free rank-1 GLWE, at the circuit-bootstrapping encoding bit / 2^(log_domain + 1))
    -> ggsw_bits_from_packed -> the 8-bit adder -> bdd_eval_packed (scale 2^(k - log_domain - 1)) gives packed x + y; its low 8 bits and y
    go round again, and the result decrypts to ((x + y) mod 256) + y bit by bit.  The n = 256 noise-free-key setting of
    test_circuit_bootstrap_then_bdd_eval_packed_on_the_device with GGSWs of five limbs: the bound of that test (GGSW error, 16 CMux levels,
    9 outputs summed by the packing, its roundings) must stay under the bootstrapping's margin, half a LUT step less the mod-switch rounding,
    which is itself under half the distance of the encoding.  The first stage's LWEs equal the oracle reference bit for bit."""
    n, k, n_lwe, block, log_domain, rank = 256, 12, 12, 3, 2, 1
    brk_size, dnum_res, res_size, lwe_size = 5, 2, 5, 2
    L, log_n, bits = 16, 8, 8
    cols, rs = rank + 1, dnum_res
    rng = np.random.default_rng(6700 + fl)
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

    atk_g, tsk_g = [prep_g(m) for m in atk], [prep_g(m) for m in tsk]
    ksk = noiseless_ksk(rng, [list(map(int, x)) for x in s], [embed_secret(s_lwe, n)], k, rs, rs + 1)
    ksk_g, ksk_o = prep_g(ksk), _prep_o(o, ksk)
    xpa = g.cggi_x_pow_a()
    c = bdd_from_truth_tables(ADD8, L, INTERLEAVED)
    n_out = len(c.outputs)
    scale = 1 << (k - log_domain - 1)
    gb = n * cols * rs * 8

    # bounds, in units of 2^-(rs k) = 2^-(lwe_size k)
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c_ == 0 else n // 8) for c_ in range(cols))
    bdd_bound = L * ((dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n))
    pack_bound = n_out * bdd_bound + log_n * n_out * 4 * (1 + rank * n)
    ks_round = 1 + n  # the key-switch of the noise-free key into lwe_size < rs + 1 limbs
    unit = 1 << (rs * k)
    alpha = 2  # dnum_res rounded up to a power of two
    half_step = Fraction(n // ((1 << log_domain) * alpha), 4 * n)  # half a LUT step of the blind rotation, as a torus distance
    mod_switch = Fraction(1 + n_lwe, 4 * n)  # rounding of b and n_lwe binary-keyed mask coefficients to 1 / 2n
    assert half_step < Fraction(1, 1 << (log_domain + 2))  # below half the distance of the encoding
    assert pack_bound < 1 << (rs * k - log_domain - 2)

    def packed_int(values):
        """noise-free rank-1 GLWEs (len(values), rs, 2, n): bit i of v at coefficient i, scaled."""
        out = np.zeros((len(values), rs, cols, n), dtype=np.int64)
        for i, v in enumerate(values):
            poly = np.zeros(n, dtype=np.int64)
            poly[:bits] = [((v >> j) & 1) * scale for j in range(bits)]
            out[i] = SC.noiseless_row(rng, {0: poly}, s, k, rs)
        return out

    def check_lwes(packed, values, bound):
        """glwe_to_lwe_indexed of the 2B packed GLWEs -> every LWE decrypts to its bit within `bound` units; returns the LWEs."""
        m = packed.batch
        buf = pb.DevBuf(m * bits * lwe_size * (n_lwe + 1) * 8)
        g.glwe_to_lwe_indexed(buf, n_lwe, lwe_size, k, packed, k, range(bits), ksk_g, k)
        g.sync()
        lwes = buf.download(np.int64, (m, bits, lwe_size, 1, n_lwe + 1))
        for i, v in enumerate(values):
            for j in range(bits):
                e = _centred(_lwe_int_phase(lwes[i, j], s_lwe, k) - (((v >> j) & 1) << (lwe_size * k - log_domain - 1)), unit)
                assert abs(e) <= bound, (i, j, e, bound)
        assert Fraction(bound, unit) + mod_switch < half_step
        return lwes

    def add(packed):
        sel = circuit.ggsw_bits_from_packed(g, packed, range(bits), ksk_g, n_lwe, lwe_size, brk_g, xpa, block, atk_g, tsk_g, k, rank, dnum_res,
                                            res_size, log_domain)
        assert sel.batch == packed.batch * bits
        return circuit.bdd_eval_packed(g, c, sel, packed.batch // 2, L, k, scale, atk_g, size=rs)

    def check_sum(packed_sum, want):
        got = g.vec_znx_to_numpy(packed_sum)
        for b, w in enumerate(want):
            for j in range(n_out):
                rot = R.rotate(got[b], -j)
                ext = np.zeros((rs, 1, n + 1), dtype=np.int64)
                LR.lwe_sample_extract(ext, rot)
                e = _centred(ring_lwe_phase(ext, s[0], k) - (((w >> j) & 1) << (rs * k - log_domain - 1)), unit)
                assert abs(e) <= pack_bound, (b, j, e, pack_bound)

    xy = [(255, 1), (173, 94), (0, 0), (200, 77)]
    B = len(xy)
    # stage 1: item b's selectors are bits 0..7 of x_b, then of y_b: the packed GLWEs interleaved, x_b at 2b and y_b at 2b + 1
    values1 = [v for x, y in xy for v in (x, y)]
    host1 = packed_int(values1)
    packed1 = g.vec_znx_from_numpy(host1)
    lwes = check_lwes(packed1, values1, ks_round)
    want = np.zeros((bits, lwe_size, 1, n_lwe + 1), dtype=np.int64)
    for i in range(2 * B):
        R.glwe_to_lwe_indexed(o, want, k, host1[i], k, range(bits), ksk_o, k)
        assert np.array_equal(lwes[i], want), i
    sum1 = add(packed1)
    g.sync()
    check_sum(sum1, [x + y for x, y in xy])
    # stage 2: the sum's low 8 bits and y, interleaved by device copies
    packed2 = g.vec_znx_alloc(cols, rs, 2 * B)
    circuit._glwe_copy(g, packed2.buf.ptr, 2 * gb, rs, sum1.buf.ptr, sum1.batch_stride, rs, cols, B)
    circuit._glwe_copy(g, packed2.buf.ptr + gb, 2 * gb, rs, packed1.buf.ptr + gb, 2 * gb, rs, cols, B)
    values2 = [v for x, y in xy for v in ((x + y) % 256, y)]
    check_lwes(packed2, values2, pack_bound + ks_round)
    sum2 = add(packed2)
    g.sync()
    check_sum(sum2, [(x + y) % 256 + y for x, y in xy])
