"""GPU parity of the LWE <-> GLWE family (pgb_lwe_sample_extract_batched, pgb_lwe_keyswitch_batched, pgb_glwe_to_lwe_batched,
pgb_lwe_to_glwe_batched) with the reference of tests/lwe_ref.py (copies around the oracle's glwe_keyswitch), bit for bit, both flavours: ring degrees 512 .. 4096 (at 512 the NTT120 key-switch takes the
limb-wise route and FFT64 its single kernel), LWE dimensions 1, even, odd and N, sizes 1 .. 4, mixed base2k, dsize 2, a ragged batch of 37,
LWE batch strides padded by 8 bytes (every LWE limb then only 8-byte aligned) and GLWE batch strides by 16 (the alignment
the key-switch kernels need), default routes and PGB_OPT_NO_FUSION; the rejections; the bench
shapes; and the closed bootstrap loop on the device, whose every intermediate must equal the oracle loop of tests/test_oracle_lwe.py."""
import ctypes as C

import numpy as np
import pytest

import poulpy_b200 as pb
import lwe_ref as L
import semantics_circuit as SC
from oracle import pyoracle as O
from poulpy_b200.hal import _BT, _VZ, lib
from test_oracle_lwe import LOOP, decode, f_lut, loop_material, oracle_round, prep
from util import fill_uniform

pytestmark = pytest.mark.gpu


# ---- helpers -----------------------------------------------------------------------------------------------------------------------------
def _key(rng, g, o, dnum, cols_in, cols_out, size, k):
    mat = fill_uniform(rng, (dnum, cols_in, size, cols_out, g.n), k)
    pm = g.vmp_pmat_alloc(dnum, cols_in, cols_out, size)
    g.vmp_prepare(pm, g.mat_znx_from_numpy(mat))
    return pm, prep(o, mat)


def _dev_items(arr, pad):
    """(B, ...) int64 -> DevBuf with the items `item + pad` bytes apart; returns (buf, stride)."""
    B = arr.shape[0]
    item = arr[0].size
    host = np.zeros((B, item + pad // 8), dtype=np.int64)
    host[:, :item] = arr.reshape(B, item)
    buf = pb.DevBuf(host.nbytes)
    buf.upload(host)
    return buf, (item * 8 + pad)


def _from_dev(buf, shape, pad):
    B = shape[0]
    item = int(np.prod(shape[1:]))
    return buf.download(np.int64, (B, item + pad // 8))[:, :item].reshape(shape)


def _glwe(g, arr, pad):
    """(B, size, cols, n) -> VecZnx batch with a batch stride padded by 2 * `pad` bytes (GLWEs must stay 16-byte aligned)."""
    buf, stride = _dev_items(arr, 2 * pad)
    B, size, cols, n = arr.shape
    return pb.hal.VecZnx(buf, n, cols, size, batch=B, batch_stride=stride)


def _glwe_out(g, shape, pad, rng, k):
    return _glwe(g, fill_uniform(rng, shape, k), pad)  # garbage pre-fill


def _glwe_np(v, shape, pad):
    return _from_dev(v.buf, shape, 2 * pad)


def _in_size(a_size, a_k, key_k):
    return -(-a_size * a_k // key_k)


# N, n_in, n_out, rank, a_size, res_size, a_k, key_k, res_k, dsize, batch, pad
CASES = [
    (512, 512, 511, 3, 1, 1, 18, 18, 18, 1, 37, 0),
    (512, 1, 2, 1, 2, 3, 18, 18, 18, 2, 5, 8),
    (1024, 687, 512, 2, 3, 2, 12, 12, 12, 2, 37, 8),
    (1024, 1024, 1, 1, 4, 4, 12, 15, 13, 1, 7, 0),
    (2048, 1023, 2048, 2, 2, 1, 18, 18, 18, 1, 6, 8),
    (2048, 600, 601, 1, 3, 3, 13, 11, 12, 2, 4, 0),
    (4096, 4096, 1023, 1, 1, 2, 18, 18, 18, 1, 3, 8),
    (4096, 777, 4096, 2, 2, 4, 18, 18, 18, 2, 3, 0),
]


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("no_fusion", [0, 1])
@pytest.mark.parametrize("case", CASES, ids=[f"N{c[0]}-in{c[1]}-out{c[2]}-r{c[3]}-s{c[4]}{c[5]}-k{c[6]}.{c[7]}.{c[8]}-d{c[9]}-b{c[10]}-p{c[11]}"
                                             for c in CASES])
def test_lwe_family_matches_oracle(fl, no_fusion, case):
    n, n_in, n_out, rank, a_size, res_size, a_k, key_k, res_k, dsize, B, pad = case
    rng = np.random.default_rng(n + n_in + 7 * n_out + rank + dsize + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
    in_size = _in_size(a_size, a_k, key_k)
    dnum, key_size = -(-in_size // dsize), in_size + 1

    # sample_extract: rank-1 GLWE (a_size limbs) -> LWE (n_out, res_size)
    a = fill_uniform(rng, (B, a_size, 2, n), a_k)
    res_buf, rs = _dev_items(fill_uniform(rng, (B, res_size, 1, n_out + 1), a_k), pad)
    g.lwe_sample_extract(res_buf, n_out, res_size, _glwe(g, a, pad), res_stride=rs)
    want = np.zeros((B, res_size, 1, n_out + 1), dtype=np.int64)
    for b in range(B):
        L.lwe_sample_extract(want[b], a[b])
    g.sync()
    assert np.array_equal(_from_dev(res_buf, want.shape, pad), want), "sample_extract"

    # lwe_keyswitch n_in -> n_out
    kg, ko = _key(rng, g, o, dnum, 1, 2, key_size, key_k)
    a = fill_uniform(rng, (B, a_size, 1, n_in + 1), a_k)
    a_buf, as_ = _dev_items(a, pad)
    res_buf, rs = _dev_items(fill_uniform(rng, (B, res_size, 1, n_out + 1), res_k), pad)
    g.lwe_keyswitch(res_buf, n_out, res_size, res_k, a_buf, n_in, a_size, a_k, kg, key_k, B, dsize, res_stride=rs, a_stride=as_)
    for b in range(B):
        L.lwe_keyswitch(o, want[b], res_k, a[b], a_k, ko, key_k, dsize)
    g.sync()
    assert np.array_equal(_from_dev(res_buf, want.shape, pad), want), "lwe_keyswitch"
    assert np.array_equal(_from_dev(a_buf, a.shape, pad), a), "lwe_keyswitch wrote its input"

    # glwe_to_lwe: rank `rank` -> LWE n_out
    kg, ko = _key(rng, g, o, dnum, rank, 2, key_size, key_k)
    a = fill_uniform(rng, (B, a_size, rank + 1, n), a_k)
    res_buf, rs = _dev_items(fill_uniform(rng, (B, res_size, 1, n_out + 1), res_k), pad)
    g.glwe_to_lwe(res_buf, n_out, res_size, res_k, _glwe(g, a, pad), a_k, kg, key_k, dsize, res_stride=rs)
    for b in range(B):
        L.glwe_to_lwe(o, want[b], res_k, a[b], a_k, ko, key_k, dsize)
    g.sync()
    assert np.array_equal(_from_dev(res_buf, want.shape, pad), want), "glwe_to_lwe"

    # lwe_to_glwe: LWE n_in -> rank `rank`
    kg, ko = _key(rng, g, o, dnum, 1, rank + 1, key_size, key_k)
    a = fill_uniform(rng, (B, a_size, 1, n_in + 1), a_k)
    a_buf, as_ = _dev_items(a, pad)
    shape = (B, res_size, rank + 1, n)
    res_g = _glwe_out(g, shape, pad, rng, res_k)
    g.lwe_to_glwe(res_g, res_k, a_buf, n_in, a_size, a_k, kg, key_k, dsize, a_stride=as_)
    want_g = np.zeros(shape, dtype=np.int64)
    for b in range(B):
        L.lwe_to_glwe(o, want_g[b], res_k, a[b], a_k, ko, key_k, dsize)
    g.sync()
    assert np.array_equal(_glwe_np(res_g, shape, pad), want_g), "lwe_to_glwe"


# ---- rejections (all of them before any launch) --------------------------------------------------------------------------------------
def _call(name, g, res, rk, a, ak, key, kk, dsize, bt, scratch, length):
    return getattr(lib(), name)(g._h, C.byref(res), C.c_uint64(rk), C.byref(a), C.c_uint64(ak), C.byref(key), C.c_uint64(kk), C.c_uint64(dsize),
                                C.byref(bt), C.c_void_p(scratch), C.c_size_t(length))


def _tmp(name, g, res_size, a_size, ak, key, kk, dsize, B):
    f = getattr(lib(), name)
    return int(f(g._h, C.c_uint64(res_size), C.c_uint64(a_size), C.c_uint64(ak), C.byref(key), C.c_uint64(kk), C.c_uint64(dsize), C.c_uint64(B)))


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_lwe_family_rejections(fl):
    n, k, B, size, rank = 512, 18, 3, 2, 2
    g = pb.Module(n, fl)
    launches = g.launch_count
    lwe_bs = size * (n + 1) * 8  # n_lwe = N: the largest LWE
    big = pb.DevBuf(4 * B * lwe_bs + 4 * B * n * (rank + 1) * size * 8)
    lwe_a = _VZ(big.ptr, n + 1, 1, size, size)
    lwe_r = _VZ(big.ptr + B * lwe_bs, n + 1, 1, size, size)
    glwe_off = 2 * B * lwe_bs
    glwe_bs = n * (rank + 1) * size * 8
    glwe = _VZ(big.ptr + glwe_off, n, rank + 1, size, size)
    glwe1 = _VZ(big.ptr + glwe_off, n, 2, size, size)
    keys = [g.vmp_pmat_alloc(size, 1, 2, size + 1), g.vmp_pmat_alloc(size, rank, 2, size + 1), g.vmp_pmat_alloc(size, 1, rank + 1, size + 1)]
    k_lwe, k_g2l, k_l2g = (x.struct() for x in keys)  # `keys` keeps the buffers alive
    scratch = pb.DevBuf(64 << 20)
    bt_ll = _BT(B, lwe_bs, lwe_bs, 0)
    bt_gl = _BT(B, lwe_bs, glwe_bs, 0)
    bt_lg = _BT(B, glwe_bs, lwe_bs, 0)
    SHAPE, ALIAS, SCRATCH = -1, -3, -4

    def ks(res, a, key, bt, length=64 << 20):
        return _call("pgb_lwe_keyswitch_batched", g, res, k, a, k, key, k, 1, bt, scratch.ptr, length)

    def g2l(res, a, key, bt, length=64 << 20):
        return _call("pgb_glwe_to_lwe_batched", g, res, k, a, k, key, k, 1, bt, scratch.ptr, length)

    def l2g(res, a, key, bt, length=64 << 20):
        return _call("pgb_lwe_to_glwe_batched", g, res, k, a, k, key, k, 1, bt, scratch.ptr, length)

    def extract(res, a, bt):
        return lib().pgb_lwe_sample_extract_batched(g._h, C.byref(res), C.byref(a), C.byref(bt))

    # ring / rank mismatches
    assert extract(lwe_r, _VZ(glwe1.data, n // 2, 2, size, size), bt_gl) == SHAPE
    assert extract(lwe_r, glwe, bt_gl) == SHAPE                                             # rank 2 is not a rank-1 GLWE
    assert g2l(lwe_r, _VZ(glwe.data, n // 2, rank + 1, size, size), k_g2l, bt_gl) == SHAPE
    assert g2l(lwe_r, glwe, g.vmp_pmat_alloc(size, rank + 1, 2, size + 1).struct(), bt_gl) == SHAPE
    assert g2l(lwe_r, glwe, g.vmp_pmat_alloc(size, rank, 3, size + 1).struct(), bt_gl) == SHAPE
    assert l2g(_VZ(glwe.data, n, rank, size, size), lwe_a, k_l2g, bt_lg) == SHAPE            # res rank != key rank_out
    assert ks(lwe_r, lwe_a, k_l2g, bt_ll) == SHAPE                                           # cols_out 3 for an LWE key-switch
    other = pb.Module(2 * n, fl)
    assert ks(lwe_r, lwe_a, other.vmp_pmat_alloc(size, 1, 2, size + 1).struct(), bt_ll) == SHAPE
    # n_lwe > N, n_lwe = 0, more than one column
    assert ks(_VZ(lwe_r.data, n + 2, 1, size, size), lwe_a, k_lwe, _BT(B, size * (n + 2) * 8, lwe_bs, 0)) == SHAPE
    assert ks(lwe_r, _VZ(lwe_a.data, 1, 1, size, size), k_lwe, bt_ll) == SHAPE
    assert l2g(glwe, _VZ(lwe_a.data, n + 1, 2, size, size), k_l2g, bt_lg) == SHAPE
    # layout: stride below one item, not a multiple of 8, misaligned data, batch count out of range, size 0
    assert ks(lwe_r, lwe_a, k_lwe, _BT(B, lwe_bs, lwe_bs - 8, 0)) == SHAPE
    assert ks(lwe_r, lwe_a, k_lwe, _BT(B, lwe_bs + 4, lwe_bs, 0)) == SHAPE
    assert ks(_VZ(lwe_r.data + 4, n + 1, 1, size, size), lwe_a, k_lwe, bt_ll) == SHAPE
    assert ks(lwe_r, lwe_a, k_lwe, _BT(0, lwe_bs, lwe_bs, 0)) == SHAPE
    assert ks(lwe_r, lwe_a, k_lwe, _BT(65536, lwe_bs, lwe_bs, 0)) == SHAPE
    assert ks(lwe_r, _VZ(lwe_a.data, n + 1, 1, 0, 0), k_lwe, bt_ll) == SHAPE
    assert g2l(lwe_r, glwe, k_g2l, _BT(B, lwe_bs, glwe_bs + 8, 0)) == SHAPE                 # GLWEs need 16-byte strides and data
    assert l2g(_VZ(glwe.data + 8, n, rank + 1, size, size), lwe_a, k_l2g, bt_lg) == SHAPE
    assert extract(lwe_r, glwe1, _BT(B, lwe_bs, 2 * n * size * 8 + 8, 0)) == SHAPE
    assert _call("pgb_lwe_keyswitch_batched", g, lwe_r, k, lwe_a, k, k_lwe, k, 1, bt_ll, scratch.ptr + 128, 32 << 20) == SHAPE
    # overlap: in place, shifted by one item, LWE over GLWE
    assert ks(lwe_a, lwe_a, k_lwe, bt_ll) == ALIAS
    assert ks(_VZ(lwe_a.data + lwe_bs, n + 1, 1, size, size), lwe_a, k_lwe, bt_ll) == ALIAS
    assert extract(_VZ(glwe1.data + 8, n + 1, 1, size, size), glwe1, _BT(B, lwe_bs, n * 2 * size * 8, 0)) == ALIAS
    assert g2l(_VZ(glwe.data, n + 1, 1, size, size), glwe, k_g2l, bt_gl) == ALIAS
    assert l2g(glwe, _VZ(glwe.data + glwe_bs, n + 1, 1, size, size), k_l2g, bt_lg) == ALIAS
    assert g.launch_count == launches  # nothing above launched a kernel
    # scratch: exactly _tmp_bytes runs, one byte less is refused
    for name, fn, res, a, key, bt in (("pgb_lwe_keyswitch", ks, lwe_r, lwe_a, k_lwe, bt_ll), ("pgb_glwe_to_lwe", g2l, lwe_r, glwe, k_g2l, bt_gl),
                                      ("pgb_lwe_to_glwe", l2g, glwe, lwe_a, k_l2g, bt_lg)):
        need = _tmp(name + "_tmp_bytes", g, res.size, a.size, k, key, k, 1, B)
        before = g.launch_count
        assert fn(res, a, key, bt, need - 1) == SCRATCH, name
        assert g.launch_count == before
        assert fn(res, a, key, bt, need) == 0, (name, lib().pgb_last_error())
    g.sync()


# ---- bench shapes ----------------------------------------------------------------------------------------------------------------------
BENCH_B = 2368  # bench.py's CGGI batch: 148 SMs x 4 ciphertexts x 4 waves


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_glwe_to_lwe_bench_shape(fl):
    """The blind rotation's output at bench.py's CGGI configuration (N = 512, rank 3, base2k 18, one limb) to an LWE of dimension 512."""
    n, rank, k, B = 512, 3, 18, BENCH_B
    rng = np.random.default_rng(4100 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    kg, ko = _key(rng, g, o, 1, rank, 2, 2, k)
    a = fill_uniform(rng, (B, 1, rank + 1, n), k)
    res = pb.DevBuf(B * (n + 1) * 8)
    g.glwe_to_lwe(res, n, 1, k, g.vec_znx_from_numpy(a), k, kg, k)
    want = np.zeros((B, 1, 1, n + 1), dtype=np.int64)
    for b in range(B):
        L.glwe_to_lwe(o, want[b], k, a[b], k, ko, k)
    g.sync()
    assert np.array_equal(res.download(np.int64, want.shape), want)


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_lwe_keyswitch_bench_shape(fl):
    """LWE key-switch 512 -> 687 (bench.py's n_lwe) on N = 1024, base2k 18, batch 2368."""
    n, n_in, n_out, k, B = 1024, 512, 687, 18, BENCH_B
    rng = np.random.default_rng(4200 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    kg, ko = _key(rng, g, o, 1, 1, 2, 2, k)
    a = fill_uniform(rng, (B, 1, 1, n_in + 1), k)
    a_buf = pb.DevBuf(a.nbytes)
    a_buf.upload(a)
    res = pb.DevBuf(B * (n_out + 1) * 8)
    g.lwe_keyswitch(res, n_out, 1, k, a_buf, n_in, 1, k, kg, k, B)
    want = np.zeros((B, 1, 1, n_out + 1), dtype=np.int64)
    for b in range(B):
        L.lwe_keyswitch(o, want[b], k, a[b], k, ko, k)
    g.sync()
    assert np.array_equal(res.download(np.int64, want.shape), want)


# ---- closed loop ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_noiseless_bootstrap_loop_on_the_device(fl):
    """LWE(m) -> mod_switch_2n -> blind rotation -> glwe_to_lwe -> lwe_keyswitch -> mod_switch_2n -> blind rotation -> .. entirely on the
    device (the LWE key-switch output goes straight into pgb_cggi_mod_switch_2n_batched): every round decrypts to f applied once more, and
    every intermediate equals the oracle loop."""
    p = LOOP
    n, k, rank, cols = 256, p["k"], p["rank"], p["rank"] + 1
    rng = np.random.default_rng(4300 + fl)
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    mat = loop_material(rng, n, fl)
    per = n * p["brk_dnum"] * cols * cols * p["brk_size"] * g.prep_bytes
    brk_buf = pb.DevBuf(per * p["n_lwe"])
    for i, m in enumerate(mat["brk"]):
        g.vmp_prepare(pb.hal.VmpPMat(brk_buf, n, p["brk_dnum"], cols, cols, p["brk_size"], offset=i * per), g.mat_znx_from_numpy(m))
    brk_g = pb.hal.VmpPMat(brk_buf, n, p["brk_dnum"], cols, cols, p["brk_size"])
    brk_o = [prep(o, b) for b in mat["brk"]]

    def prep_g(m):
        d, ci, sz, co, _ = m.shape
        pm = g.vmp_pmat_alloc(d, ci, co, sz)
        g.vmp_prepare(pm, g.mat_znx_from_numpy(m))
        return pm

    ks1_g, ks2_g, ks1_o, ks2_o = prep_g(mat["ks1"]), prep_g(mat["ks2"]), prep(o, mat["ks1"]), prep(o, mat["ks2"])
    xg, xo = g.cggi_x_pow_a(), o.cggi_x_pow_a()
    lut_g = g.vec_znx_from_numpy(mat["lut"])
    msgs = [m % (1 << p["log_domain"]) for m in range(9)]
    B = len(msgs)
    lwe = np.stack([SC.noiseless_lwe(rng, m, p["log_domain"], mat["s_lwe"], k, p["lwe_size"]) for m in msgs])
    lwe_dev = pb.DevBuf(lwe.nbytes)
    lwe_dev.upload(lwe)
    want = list(msgs)
    for rnd in range(2):
        l2n = g.cggi_mod_switch_2n(lwe_dev, B, p["n_lwe"], p["lwe_size"], k, 2 * n, True)
        acc = g.vec_znx_alloc(cols, p["brk_size"], B)
        g.cggi_blind_rotate(acc, l2n, p["n_lwe"], lut_g, brk_g, xg, p["block"], k)
        mid = pb.DevBuf(B * p["mid_size"] * (p["n_mid"] + 1) * 8)
        g.glwe_to_lwe(mid, p["n_mid"], p["mid_size"], k, acc, k, ks1_g, k)
        out = pb.DevBuf(B * p["lwe_size"] * (p["n_lwe"] + 1) * 8)
        g.lwe_keyswitch(out, p["n_lwe"], p["lwe_size"], k, mid, p["n_mid"], p["mid_size"], k, ks2_g, k, B)
        g.sync()
        got = (l2n.download(np.int64, (B, p["n_lwe"] + 1)), g.vec_znx_to_numpy(acc),
               mid.download(np.int64, (B, p["mid_size"], 1, p["n_mid"] + 1)), out.download(np.int64, (B, p["lwe_size"], 1, p["n_lwe"] + 1)))
        want = [f_lut(w, p["log_domain"]) for w in want]
        for b in range(B):
            ref = oracle_round(o, lwe[b], mat, brk_o, xo, ks1_o, ks2_o)
            for name, x, y in zip(("mod_switch_2n", "blind_rotate", "glwe_to_lwe", "lwe_keyswitch"), got, ref):
                assert np.array_equal(x[b], y), (rnd, b, name)
            assert decode(got[3][b], mat["s_lwe"], k, p["log_domain"]) == want[b], (rnd, b)
        lwe, lwe_dev = got[3], out
