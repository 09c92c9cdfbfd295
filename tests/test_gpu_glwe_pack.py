"""GPU parity of the batched packing entry (pgb_glwe_pack_batched, Module.glwe_pack) with the host composition circuit.glwe_pack, both
flavours, bit for bit: over circuit.DeviceGlweOps (the batched ABI calls) and over the oracle (tests/util_circuit.py).  n = 256 (the
limb-wise automorphism route) and n = 1024 (the gadget kernel's automorphism epilogue), dsize 1 and 2, maps with every case of a round
present (pairs, keys with only j, keys with only j + t) and with one case only, the BDD output maps and the gap map of post_process; the
inputs must be unchanged after the call.  Then multi-chunk runs, a shared input batch, the launch count against the documented per-round
formula and against the composition, every rejection (each launching nothing), and circuit bootstrapping -> the 8-bit adder ->
circuit.bdd_eval_packed, end to end."""
import ctypes as C

import numpy as np
import pytest

import bdd_ref as BR
import lwe_ref as LR
import semantics_circuit as SC
import poulpy_b200 as pb
from oracle import pyoracle as O
from poulpy_b200 import circuit
from poulpy_b200.circuit import bdd_from_truth_tables
from poulpy_b200.hal import _BT, _PM, _VZ, lib
from test_gpu_cmux import _np, _prep_o
from test_oracle_bdd import ADD8, INTERLEAVED
from test_oracle_cmux_tree import lwe_phase
from util import fill_uniform
from util_circuit import OracleGlweOps, _Ct

pytestmark = pytest.mark.gpu
RANK, K, SIZE = 1, 13, 2
COLS = RANK + 1


def _maps(n):
    """(name, index, log_gap_out): the adder's 9 outputs and 32 outputs at gap 0, every case in round 0 (pair 0 / n/2, hi only at n/2 + n/4,
    lo only at 40 and 8), one input (lo only in every round; with the whole trace), a hi-only start, and the gap map of post_process."""
    return [("dense9", list(range(9)), 0), ("dense32", list(range(32)), 0), ("all_cases", [0, n // 2, n // 2 + n // 4, 40, 8], 0),
            ("one", [0], 0), ("one_trace", [0], n.bit_length() - 1), ("hi_start", [n // 2 + n // 4], 0),
            ("post_process", [i << 3 for i in range(4)], 3)]


def _keys(g, o, rng, n, dsize):
    log_n = n.bit_length() - 1
    dnum = -(-SIZE // dsize)
    kg, ko = [], []
    for _ in range(log_n):
        mat = fill_uniform(rng, (dnum, RANK, SIZE + 1, COLS, n), K)  # one limb more than the GLWEs
        pg = g.vmp_pmat_alloc(dnum, RANK, COLS, SIZE + 1)
        g.vmp_prepare(pg, g.mat_znx_from_numpy(mat))
        kg.append(pg)
        if o is not None:
            ko.append(_prep_o(o, mat))
    return kg, ko


def _inputs_dev(host, pad=0):
    """(B, n_in, size, cols, n) -> (VecZnx of B items, entry_stride): inputs `item + pad` bytes apart, items one spare input apart."""
    B, n_in, size, cols, n = host.shape
    item = size * cols * n * 8
    es = item + pad
    stride = (n_in + 1) * es
    flat = np.zeros((B, stride // 8), dtype=np.int64)
    for j in range(n_in):
        flat[:, j * es // 8: j * es // 8 + item // 8] = host[:, j].reshape(B, -1)
    buf = pb.DevBuf(flat.nbytes)
    buf.upload(flat)
    return pb.hal.VecZnx(buf, n, cols, size, batch=B, batch_stride=stride), es, flat


def _entry(g, keys, host, index, gap, dsize, pad=0, max_chunk=None, shared=False, B=None):
    B = host.shape[0] if B is None else B
    a, es, flat = _inputs_dev(host, pad)
    if shared:
        a = pb.hal.VecZnx(a.buf, a.n, a.cols, a.size)
    res = g.vec_znx_from_numpy(np.full((B, SIZE, COLS, g.n), 12345, dtype=np.int64))  # garbage: every word must be written
    before = g.launch_count
    g.glwe_pack(res, a, index, gap, keys, K, dsize, entry_stride=es, max_chunk=max_chunk)
    launches = g.launch_count - before
    g.sync()
    assert np.array_equal(a.buf.download(np.int64, flat.shape), flat), "the inputs changed"
    return _np(res, B), launches


def _composition_dev(g, keys, host, index, gap, dsize):
    B = host.shape[0]
    ops = circuit.DeviceGlweOps(g, keys, K, COLS, SIZE, B, dsize)
    cts = {i: g.vec_znx_from_numpy(host[:, j]) for j, i in enumerate(index)}
    res = ops.new()
    before = g.launch_count
    circuit.glwe_pack(ops, res, cts, gap)
    launches = g.launch_count - before
    g.sync()
    return _np(res, B), launches


def _composition_oracle(o, keys_o, host, index, gap, dsize):
    B, n = host.shape[0], host.shape[-1]
    ops = OracleGlweOps(o, keys_o, K, COLS, SIZE, B, n, dsize)
    res = ops.new()
    circuit.glwe_pack(ops, res, {i: _Ct(host[:, j].copy()) for j, i in enumerate(index)}, gap)
    return res.arr


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
@pytest.mark.parametrize("n", [256, 1024])
@pytest.mark.parametrize("dsize", [1, 2])
def test_glwe_pack_matches_the_compositions(fl, n, dsize):
    g = pb.Module(n, fl)
    o = O.OracleModule(n, fl)
    rng = np.random.default_rng(7000 + n + 10 * dsize + fl)
    kg, ko = _keys(g, o, rng, n, dsize)
    B = 3
    for name, index, gap in _maps(n):
        host = fill_uniform(rng, (B, len(index), SIZE, COLS, n), K + 2)  # unnormalised digits
        got, _ = _entry(g, kg, host, index, gap, dsize, pad=16 * (len(index) % 3))
        want, _ = _composition_dev(g, kg, host, index, gap, dsize)
        assert np.array_equal(got, want), (name, "device composition")
        if n == 256 or name in ("dense9", "all_cases"):
            want_o = _composition_oracle(o, ko, host[:1], index, gap, dsize)
            assert np.array_equal(got[:1], want_o), (name, "oracle composition")


# ---- launches ------------------------------------------------------------------------------------------------------------------------------
def _plan(n, index, gap):
    """Per round (pairs, lo only, hi only), as pgb_glwe_pack_batched plans it."""
    cur, rounds = set(index), []
    for i in range(n.bit_length() - 1 - gap):
        t = n >> (i + 1)
        nb = sum(1 for j in range(t) if j in cur and j + t in cur)
        nl = sum(1 for j in range(t) if j in cur and j + t not in cur)
        nh = sum(1 for j in range(t) if j not in cur and j + t in cur)
        rounds.append((nb, nl, nh))
        cur = {k % t for k in cur}
    return rounds


def _measure(g, keys, dsize, cache, kind, count, i=0):
    """Launches of one batched call on zero data: ('plain' | 'op0' | 'op2', count) under keys[i], or ('trace', count) with skip i."""
    key = (kind, count, i)
    if key not in cache:
        x, out = g.vec_znx_alloc(COLS, SIZE, count), g.vec_znx_alloc(COLS, SIZE, count)
        p = g.trace_galois_element(i)
        before = g.launch_count
        if kind == "plain":
            g.glwe_automorphism(out, K, x, K, keys[i], K, p, dsize)
        elif kind == "trace":
            g.glwe_trace_assign(out, K, i, keys, K, dsize)
        else:
            g.glwe_automorphism_op(int(kind[2]), out, K, x, keys[i], K, p, dsize)
        cache[key] = g.launch_count - before
        g.sync()
    return cache[key]


def _expected_launches(g, keys, index, gap, dsize, B, chunk, cache, shared=False):
    """Per chunk: per round one prep launch, one automorphism call per present case, one combine launch when pairs exist; then the trace
    with skip = log_n - gap (none at gap 0); without rounds the state is copied into res first, by a kernel only for a shared input."""
    n, log_n = g.n, g.n.bit_length() - 1
    rounds = _plan(n, index, gap)
    widest = sum(rounds[0]) if rounds else 1
    Bc = min(B, 65535 // widest, chunk or B)
    total = 0
    for b0 in range(0, B, Bc):
        nb = min(Bc, B - b0)
        for i, (p, lo, hi) in enumerate(rounds):
            total += 1 + (p > 0)
            total += (_measure(g, keys, dsize, cache, "plain", nb * p, i) if p else 0)
            total += (_measure(g, keys, dsize, cache, "op0", nb * lo, i) if lo else 0)
            total += (_measure(g, keys, dsize, cache, "op2", nb * hi, i) if hi else 0)
        total += 0 if rounds or not shared else 1  # without rounds: a 2D copy, or a copy kernel for a shared input batch
        total += _measure(g, keys, dsize, cache, "trace", nb, log_n - gap) if gap else 0
    return total


@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_glwe_pack_chunks_shared_inputs_and_launches(fl):
    n, dsize, B = 1024, 1, 5
    g = pb.Module(n, fl)
    rng = np.random.default_rng(7100 + fl)
    kg, _ = _keys(g, None, rng, n, dsize)
    cache = {}
    for name, index, gap in _maps(n):
        host = fill_uniform(rng, (B, len(index), SIZE, COLS, n), K)
        full, _ = _entry(g, kg, host, index, gap, dsize)
        for chunk in (1, 2):  # several chunks: the same result
            got, _ = _entry(g, kg, host, index, gap, dsize, max_chunk=chunk)
            assert np.array_equal(got, full), (name, chunk)
        # a shared input batch equals the replicated one
        rep = np.repeat(host[:1], B, axis=0)
        shared, _ = _entry(g, kg, host[:1], index, gap, dsize, shared=True, B=B)
        want, _ = _entry(g, kg, rep, index, gap, dsize)
        assert np.array_equal(shared, want), name
        # launches on zero data (the NTT120 gadget route is data independent there): the formula, chunked or not, and below the composition
        zero = np.zeros_like(host)
        for chunk in (None, 2):
            _, launches = _entry(g, kg, zero, index, gap, dsize, max_chunk=chunk)
            assert launches == _expected_launches(g, kg, index, gap, dsize, B, chunk, cache), (name, chunk, launches)
        _, launches = _entry(g, kg, zero[:1], index, gap, dsize, shared=True, B=B)
        assert launches == _expected_launches(g, kg, index, gap, dsize, B, None, cache, shared=True), (name, "shared", launches)
        _, comp = _composition_dev(g, kg, zero, index, gap, dsize)
        _, launches = _entry(g, kg, zero, index, gap, dsize)
        # without rounds both are the copy and the trace
        assert launches < comp or (launches == comp and gap == g.n.bit_length() - 1), (name, launches, comp)


def test_glwe_pack_small_scratch_runs_chunks():
    """A scratch that holds two items' worth runs three chunks over five items, with the result of one chunk."""
    n, dsize, B = 256, 2, 5
    g = pb.Module(n, pb.NTT120)
    rng = np.random.default_rng(7200)
    kg, _ = _keys(g, None, rng, n, dsize)
    index, gap = [0, n // 2, n // 2 + n // 4, 40, 8], 0
    host = fill_uniform(rng, (B, len(index), SIZE, COLS, n), K)
    full, _ = _entry(g, kg, host, index, gap, dsize)
    idx = np.asarray(index, dtype=np.uint32)
    arr = (_PM * len(kg))(*[k.struct() for k in kg])
    ip = idx.ctypes.data_as(C.POINTER(C.c_uint32))
    two = lib().pgb_glwe_pack_tmp_bytes(g._h, C.c_uint64(SIZE), C.c_uint64(K), C.byref(arr[0]), C.c_uint64(dsize), ip, C.c_uint64(len(idx)),
                                        C.c_uint64(gap), C.c_uint64(2))
    three = lib().pgb_glwe_pack_tmp_bytes(g._h, C.c_uint64(SIZE), C.c_uint64(K), C.byref(arr[0]), C.c_uint64(dsize), ip, C.c_uint64(len(idx)),
                                          C.c_uint64(gap), C.c_uint64(3))
    assert 0 < two < three
    a, es, _ = _inputs_dev(host)
    res = g.vec_znx_alloc(COLS, SIZE, B)
    scratch = pb.DevBuf(three - 256)
    r, av = res.struct(), a.struct()
    bt = _BT(B, res.batch_stride, a.batch_stride, 0)
    assert lib().pgb_glwe_pack_batched(g._h, C.byref(r), C.byref(av), C.c_uint64(es), ip, C.c_uint64(len(idx)), C.c_uint64(gap), C.c_uint64(K),
                                       arr, C.c_uint64(len(kg)), C.c_uint64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                       C.c_size_t(scratch.nbytes)) == 0
    g.sync()
    assert np.array_equal(_np(res, B), full)


# ---- rejections: each returns its status and launches nothing ---------------------------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.NTT120, pb.FFT64])
def test_glwe_pack_rejections_launch_nothing(fl):
    n, B = 256, 3
    log_n = 8
    g = pb.Module(n, fl)
    rng = np.random.default_rng(7300 + fl)
    kg, _ = _keys(g, None, rng, n, 1)
    item = n * COLS * SIZE * 8
    NI = 5
    index = [0, 128, 192, 40, 8]
    res, a = pb.DevBuf(B * item), pb.DevBuf(B * NI * item)
    keys = (_PM * log_n)(*[k.struct() for k in kg])

    def idx_arr(xs):
        arr = np.asarray(xs, dtype=np.uint32)
        return arr, arr.ctypes.data_as(C.POINTER(C.c_uint32))

    good_idx, good_ip = idx_arr(index)

    def tmp(batch, ip=good_ip, n_in=NI, gap=0):
        return lib().pgb_glwe_pack_tmp_bytes(g._h, C.c_uint64(SIZE), C.c_uint64(K), C.byref(keys[0]), C.c_uint64(1), ip, C.c_uint64(n_in),
                                             C.c_uint64(gap), C.c_uint64(batch))

    need = tmp(B)
    scratch = pb.DevBuf(need + 512)

    def vz(ptr, n_=n, cols_=COLS, size_=SIZE):
        return _VZ(ptr, n_, cols_, size_, size_)

    def call(r=None, aa=None, es=item, ip=good_ip, n_in=NI, gap=0, ks=None, nk=log_n, bt=None, sp=None, sl=None):
        return lib().pgb_glwe_pack_batched(g._h, r if r is not None else C.byref(vz(res.ptr)), aa if aa is not None else C.byref(vz(a.ptr)),
                                           C.c_uint64(es), ip, C.c_uint64(n_in), C.c_uint64(gap), C.c_uint64(K),
                                           keys if ks is None else ks, C.c_uint64(nk), C.c_uint64(1),
                                           bt if bt is not None else C.byref(_BT(B, item, NI * item, 0)),
                                           C.c_void_p(scratch.ptr if sp is None else sp), C.c_size_t(need if sl is None else sl))

    def keys_with(i, **kw):
        ks = (_PM * log_n)(*[k.struct() for k in kg])
        for f, v in kw.items():
            setattr(ks[i], f, v)
        return ks

    dup, dup_ip = idx_arr([0, 128, 128, 40, 8])
    big, big_ip = idx_arr([0, 128, 192, 40, n])
    odd, odd_ip = idx_arr([0, 8, 12])  # 12 is not a multiple of 2^3
    last_input = (B - 1) * NI * item + (NI - 1) * item
    g.sync()
    before = g.launch_count
    null = C.POINTER(C.c_uint32)()
    bad = [
        (-1, dict(r=C.cast(None, C.POINTER(_VZ)))),                     # null res
        (-1, dict(aa=C.cast(None, C.POINTER(_VZ)))),                    # null a
        (-1, dict(ip=null)),                                            # null index
        (-1, dict(ks=C.cast(None, C.POINTER(_PM)))),                    # null keys
        (-1, dict(bt=C.cast(None, C.POINTER(_BT)))),                    # null batch
        (-1, dict(n_in=0)),                                             # n_in 0
        (-1, dict(n_in=n + 1)),                                         # n_in > n
        (-1, dict(ip=dup_ip)),                                          # repeated index
        (-1, dict(ip=big_ip)),                                          # index n
        (-1, dict(ip=odd_ip, n_in=3, gap=3)),                           # index not a multiple of 2^log_gap_out
        (-1, dict(gap=log_n + 1)),                                      # log_gap_out > log_n
        (-1, dict(nk=log_n - 1)),                                       # fewer than log_n keys
        (-1, dict(ks=keys_with(3, cols_in=2))),                         # a key of another rank
        (-1, dict(ks=keys_with(5, size=SIZE + 2))),                     # a key of another shape
        (-1, dict(ks=keys_with(7, n=2 * n))),                           # a key of another ring
        (-1, dict(ks=keys_with(2, data=kg[2].struct().data + 8))),      # a misaligned key
        (-1, dict(bt=C.byref(_BT(0, item, NI * item, 0)))),             # count 0
        (-1, dict(bt=C.byref(_BT(65536, item, NI * item, 0)))),         # count > 65535
        (-1, dict(bt=C.byref(_BT(B, item, NI * item, item)))),          # stride_b != 0
        (-1, dict(aa=C.byref(vz(a.ptr, n_=2 * n)))),                    # ring degree
        (-1, dict(aa=C.byref(vz(a.ptr, cols_=3)))),                     # columns
        (-1, dict(aa=C.byref(vz(a.ptr, size_=SIZE + 1)))),              # a.size != res.size
        (-1, dict(r=C.byref(vz(res.ptr + 8)))),                         # misaligned res data
        (-1, dict(bt=C.byref(_BT(B, item, NI * item + 8, 0)))),         # misaligned input stride
        (-1, dict(bt=C.byref(_BT(B, item - 16, NI * item, 0)))),        # stride_res below one GLWE
        (-1, dict(es=item + 8)),                                        # entry_stride not a multiple of 16
        (-1, dict(es=item - 16)),                                       # entry_stride below one GLWE
        (-1, dict(es=1 << 63, bt=C.byref(_BT(B, item, 1 << 62, 0)))),   # inputs past the end of the address space
        (-1, dict(bt=C.byref(_BT(B, 1 << 63, NI * item, 0)))),          # res past the end of the address space
        (-1, dict(sp=scratch.ptr + 16)),                                # scratch misaligned
        (-4, dict(sl=tmp(1) - 1)),                                      # scratch too small for one item
        (-3, dict(r=C.byref(vz(a.ptr)))),                               # res inside the inputs
        (-3, dict(r=C.byref(vz(a.ptr + last_input)))),                  # res overlaps only the last input
        (-3, dict(r=C.byref(vz(kg[log_n - 1].struct().data)))),         # res overlaps the last key
        (-3, dict(sp=res.ptr)),                                         # scratch overlaps res
        (-3, dict(sp=a.ptr + last_input // 256 * 256)),                 # scratch overlaps the inputs
    ]
    for status, kw in bad:
        assert call(**kw) == status, kw
    assert g.launch_count == before
    assert tmp(B, ip=dup_ip) == 0 and tmp(B, gap=log_n + 1) == 0
    assert call() == 0  # the same arguments, corrected, run
    assert call(sl=tmp(1)) == 0  # one item per chunk
    g.sync()


# ---- end to end: circuit bootstrapping -> prepare_ggsw -> circuit.bdd_eval_packed -------------------------------------------------------
@pytest.mark.parametrize("fl", [pb.FFT64, pb.NTT120])
def test_circuit_bootstrap_then_bdd_eval_packed_on_the_device(fl):
    """The 8-bit adder at n = 256 as in test_circuit_bootstrap_then_bdd_eval_on_the_device, its 9 outputs packed into one GLWE per item
    (output o at coefficient o): equal bit for bit to the oracle composition (bdd_ref, then circuit.glwe_pack over OracleGlweOps), and
    coefficient o decrypts to bit o of x + y."""
    from test_oracle_circuit_semantics import check_ggsw
    n, k, n_lwe, block, log_domain, rank = 256, 12, 12, 3, 2, 1
    brk_size, dnum_res, res_size, lwe_size = 4, 2, 4, 2
    L, log_n = 16, 8
    cols = rank + 1
    rng = np.random.default_rng(6500 + fl)
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
    packed = circuit.bdd_eval_packed(g, c, sel, B, L, k, scale, atk_g, size=rs)
    g.sync()
    got = g.vec_znx_to_numpy(packed)
    n_out = len(c.outputs)
    xpa = o.cggi_x_pow_a()
    leaves = circuit.bdd_leaves(n, c, scale, rs)
    # the bound of test_circuit_bootstrap_then_bdd_eval_on_the_device per output; packing adds the outputs' errors (a round's output error
    # is at most the sum of its two inputs' errors) and, per state and round, at most four roundings of one unit of the last limb on every
    # column (two shifts, the key-switch of the noise-free key into rs limbs, the final normalisation), each (1 + rank n) after decryption
    tol_ggsw = sum(16 * (1 + rank * n) * (1 if c_ == 0 else n // 8) for c_ in range(cols))
    bdd_bound = L * ((dnum_res * (1 << (k - 1)) * n * tol_ggsw >> ((res_size - rs) * k)) + 1 + (1 + rank * n))
    bound = n_out * bdd_bound + log_n * n_out * 4 * (1 + rank * n)
    assert bound < 1 << (rs * k - 2)  # below half the distance to the other bit value
    mod = 1 << (rs * k)
    for b, (x, y) in enumerate(xy):
        sels = []
        for i in range(L):
            mat = SC.circuit_bootstrap_to_constant_ref(o, lwe[b * L + i], k, brk_o, xpa, block, atk_o, tsk_o, rank, dnum_res, res_size,
                                                       log_domain, brk_size)
            check_ggsw(mat, bits[b * L + i], s, k, res_size)
            sels.append(_prep_o(o, mat))
        glwes = BR.glwe_bdd_eval(o, rs, leaves, c, k, sels, k)
        ops = OracleGlweOps(o, atk_o, k, cols, rs, 1, n)
        want = ops.new()
        circuit.glwe_pack(ops, want, {j: _Ct(np.ascontiguousarray(glwes[j])[None].copy()) for j in range(n_out)}, 0)
        assert np.array_equal(got[b], want.arr[0]), b
        for j in range(n_out):
            rot = np.zeros_like(got[b])
            for col in range(cols):
                O.vec_znx_rotate(-j, rot, col, got[b], col)
            ext = np.zeros((rs, 1, n + 1), dtype=np.int64)
            LR.lwe_sample_extract(ext, rot)
            bit = ((x + y) >> j) & 1
            e = ((lwe_phase(ext, s[0], k) - (bit << (rs * k - 1)) + (mod >> 1)) % mod) - (mod >> 1)
            assert abs(e) <= bound, (b, j, e, bound)
