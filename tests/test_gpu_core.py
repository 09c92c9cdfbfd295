"""GPU parity tests of the CoreImpl-tier pipelines (GLWE key-switch C1, GGSW x GLWE external product C2).

The reference's own core tests are statistical (decrypt + noise bound, poulpy-core/src/test_suite/keyswitch/glwe_ct.rs:132-156);
here both sides run the identical call sequence on identical synthetic inputs, so the normalised outputs must be equal bit for
bit -- a strictly stronger check.  Shapes sweep rank_in/out in {1,2}, dsize 1..3 and the mixed-base2k layout of
glwe_ct.rs:34-36 (in = b-1, key = b, out = b-2).
"""
import numpy as np
import pytest

import poulpy_b200 as pb
from oracle import pyoracle as O
from util import fill_uniform

pytestmark = pytest.mark.gpu
FLAVOURS = [pb.NTT120, pb.FFT64]


def _key(g, o, rng, dnum, cols_in, cols_out, size, k):
    mat = fill_uniform(rng, (dnum, cols_in, size, cols_out, g.n), k)
    pg, po = g.vmp_pmat_alloc(dnum, cols_in, cols_out, size), o.vmp_pmat_alloc(dnum, cols_in, cols_out, size)
    g.vmp_prepare(pg, g.mat_znx_from_numpy(mat))
    o.vmp_prepare(po, mat)
    return pg, po


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("dsize", [1, 2, 3])
def test_glwe_keyswitch_shapes(fl, dsize):
    n, batch = 256, 3
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(100 + dsize + fl)
    b = 12 if fl == pb.FFT64 else 40
    for rank_in in (1, 2):
        for rank_out in (1, 2):
            for (a_k, key_k, res_k) in ((b, b, b), (b - 1, b, b - 2)):
                a_size, key_size, res_size = 4, 5, 3
                dnum = -(-a_size // dsize)
                pg, po = _key(g, o, rng, dnum, rank_in, rank_out + 1, key_size, key_k)
                a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), a_k)
                want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), res_k)  # garbage pre-fill on both sides
                res_g = g.vec_znx_from_numpy(want)
                g.glwe_keyswitch(res_g, res_k, g.vec_znx_from_numpy(a), a_k, pg, key_k, dsize)
                g.sync()
                o.glwe_keyswitch_batch(want, res_k, a, a_k, po, key_k, dsize)
                assert np.array_equal(g.vec_znx_to_numpy(res_g), want), (rank_in, rank_out, a_k, key_k, res_k)


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("dsize", [1, 2, 3])
def test_glwe_external_product_shapes(fl, dsize):
    n, batch = 256, 3
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(200 + dsize + fl)
    b = 12 if fl == pb.FFT64 else 40
    for rank in (1, 2):
        for (a_k, g_k, res_k) in ((b, b, b), (b - 1, b, b - 2)):
            a_size, g_size, res_size = 4, 5, 3
            dnum = -(-a_size // dsize)
            pg, po = _key(g, o, rng, dnum, rank + 1, rank + 1, g_size, g_k)
            a = fill_uniform(rng, (batch, a_size, rank + 1, n), a_k)
            want = fill_uniform(rng, (batch, res_size, rank + 1, n), res_k)
            res_g = g.vec_znx_from_numpy(want)
            g.glwe_external_product(res_g, res_k, g.vec_znx_from_numpy(a), a_k, pg, g_k, dsize)
            g.sync()
            o.glwe_external_product_batch(want, res_k, a, a_k, po, g_k, dsize)
            assert np.array_equal(g.vec_znx_to_numpy(res_g), want), (rank, a_k, g_k, res_k)


@pytest.mark.parametrize("fl", FLAVOURS)
def test_keyswitch_bench_shape_c1(fl):
    """BASELINE config 0/M1: n=4096, base2k=18, k=54 (3 limbs), rank=1, dnum=3, key 4 limbs (poulpy-bench/src/params.rs:112-121)."""
    n, k, batch = 4096, 18, 6
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(300 + fl)
    pg, po = _key(g, o, rng, 3, 1, 2, 4, k)
    a = fill_uniform(rng, (batch, 3, 2, n), k)
    want = np.zeros((batch, 3, 2, n), dtype=np.int64)
    res_g = g.vec_znx_alloc(2, 3, batch)
    g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    got = g.vec_znx_to_numpy(res_g)
    assert np.array_equal(got, want)
    # host front end (H2D + compute + D2H inside the call), pageable and pinned callers
    got2 = np.zeros_like(want)
    g.glwe_keyswitch_host(got2, k, a, k, pg, k)
    assert np.array_equal(got2, want)
    ap, rp = pb.pinned_empty(a.shape), pb.pinned_empty(want.shape)
    ap[:] = a
    g.glwe_keyswitch_host(rp, k, ap, k, pg, k)
    assert np.array_equal(rp, want)


@pytest.mark.parametrize("fl", FLAVOURS)
def test_external_product_bench_shape_c3(fl):
    """BASELINE config 2/M3: n=2048, GGSW VmpPMat(3,2,2,3), GLWE VecZnx(2,3) (poulpy-bench/examples/custom_params.json)."""
    n, k, batch = 2048, 18, 8
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(400 + fl)
    pg, po = _key(g, o, rng, 3, 2, 2, 3, k)
    a = fill_uniform(rng, (batch, 3, 2, n), k)
    want = np.zeros((batch, 3, 2, n), dtype=np.int64)
    res_g = g.vec_znx_alloc(2, 3, batch)
    g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_external_product_batch(want, k, a, k, po, k)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)
    got2 = np.zeros_like(want)
    g.glwe_external_product_host(got2, k, a, k, pg, k)
    assert np.array_equal(got2, want)


def test_host_pipeline_many_chunks():
    """More ciphertexts than one staging chunk: exercises the double-buffered H2D/compute/D2H pipeline."""
    n, k, batch = 256, 18, 5000
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(500)
    pg, po = _key(g, o, rng, 2, 1, 2, 3, k)
    a = fill_uniform(rng, (batch, 2, 2, n), k)
    want = np.zeros((batch, 2, 2, n), dtype=np.int64)
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    got = np.full_like(want, -7)
    g.glwe_keyswitch_host(got, k, a, k, pg, k)
    assert np.array_equal(got, want)
    ap, rp = pb.pinned_empty(a.shape), pb.pinned_empty(want.shape)
    ap[:] = a
    rp[:] = -7
    g.glwe_keyswitch_host(rp, k, ap, k, pg, k)
    assert np.array_equal(rp, want)


def test_keyswitch_linearity_full_size():
    """Size-independent property at the bench batch: key-switch is linear over Z, so KS(a1) + KS(a2) and KS(a1 + a2) agree after
    normalisation of both sides to the same digits (checked through their torus value per coefficient on a sample)."""
    n, k, batch = 4096, 18, 256
    g = pb.Module(n, pb.NTT120)
    rng = np.random.default_rng(600)
    mat = fill_uniform(rng, (3, 1, 4, 2, n), k)
    pg = g.vmp_pmat_alloc(3, 1, 2, 4)
    g.vmp_prepare(pg, g.mat_znx_from_numpy(mat))
    a1 = fill_uniform(rng, (batch, 3, 2, n), k - 1)
    a2 = fill_uniform(rng, (batch, 3, 2, n), k - 1)
    outs = []
    for a in (a1, a2, a1 + a2):
        r = g.vec_znx_alloc(2, 3, batch)
        g.glwe_keyswitch(r, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        outs.append(g.vec_znx_to_numpy(r).astype(object))

    def torus(x):  # value * 2^(3k) mod 2^(3k)
        return (x[:, 0] * (1 << (2 * k)) + x[:, 1] * (1 << k) + x[:, 2]) % (1 << (3 * k))

    lhs = (torus(outs[0]) + torus(outs[1])) % (1 << (3 * k))
    rhs = torus(outs[2])
    diff = (lhs - rhs) % (1 << (3 * k))
    diff = np.minimum(diff, (1 << (3 * k)) - diff)
    # each side drops the 4th key limb after rounding: the two sides differ by at most 2 units of the last digit
    assert int(diff.max()) <= 2


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("n", [16384, 65536])
def test_keyswitch_large_n(fl, n):
    """Ring degrees above the single-CTA transforms (global radix-8 top pass + sub-transforms), CKKS-like base2k for NTT120."""
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(900 + n + fl)
    k = 52 if fl == pb.NTT120 else 14
    pg, po = _key(g, o, rng, 2, 1, 2, 3, k)
    a = fill_uniform(rng, (2, 2, 2, n), k)
    want = np.zeros((2, 2, 2, n), dtype=np.int64)
    res_g = g.vec_znx_alloc(2, 2, 2)
    g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)


@pytest.mark.parametrize("n", [512, 2048])
def test_collapsed_key_fast_path_and_guard(n):
    """Batches large enough for the collapsed-key path (one inverse transform per column).  Ciphertexts whose integers could leave
    (-Q/2, Q/2) -- here: a few with 60-bit 'digits' -- must be routed to the per-limb kernel by the on-device bound, and the whole
    batch must still equal the oracle bit for bit."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(1000 + n)
    k, batch = 18, 48
    for rank_in, rank_out, a_size, key_size, res_size in ((1, 1, 3, 4, 3), (2, 1, 3, 4, 4), (1, 2, 2, 3, 2), (1, 1, 3, 5, 6)):
        pg, po = _key(g, o, rng, a_size, rank_in, rank_out + 1, key_size, k)
        a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), k)
        a[5] = fill_uniform(rng, a[5].shape, 61)      # fails the bound: per-limb kernel
        a[17, 0, 0, 3] = -(1 << 62)                   # a single huge body coefficient is enough
        a[30] = 0                                      # all-zero ciphertext
        want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), k)
        res_g = g.vec_znx_from_numpy(want)
        g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_keyswitch_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, (rank_in, rank_out, a_size, key_size, res_size, bad)
    # external product, and a key with huge entries (bound fails for every ciphertext)
    for kbits in (k, 62):
        pg, po = _key(g, o, rng, 3, 2, 2, 3, kbits)
        a = fill_uniform(rng, (batch, 3, 2, n), k)
        want = np.zeros((batch, 3, 2, n), dtype=np.int64)
        res_g = g.vec_znx_alloc(2, 3, batch)
        g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_external_product_batch(want, k, a, k, po, k)
        assert np.array_equal(g.vec_znx_to_numpy(res_g), want), kbits


def test_collapsed_key_wide_base2k():
    """base2k = 52 (CKKS): the collapsed integer would need > 118 bits, every ciphertext takes the per-limb kernel."""
    n, k, batch = 1024, 52, 40
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(1100)
    pg, po = _key(g, o, rng, 2, 1, 2, 3, k)
    a = fill_uniform(rng, (batch, 2, 2, n), k)
    want = np.zeros((batch, 2, 2, n), dtype=np.int64)
    res_g = g.vec_znx_alloc(2, 2, batch)
    g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)


@pytest.mark.parametrize("n", [1024, 2048, 4096])
def test_gadget_single_kernel(n):
    """The cluster kernel of ntt120_gadget.cu (whole key-switch / external product in one launch, n = 2^10..2^12): shape sweep, more
    ciphertexts than resident clusters (persistent loop), ciphertexts that must be flagged for the per-limb route, all bit for bit."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(1200 + n)
    k = 18
    batch = 700 if n == 1024 else 40
    shapes = ((1, 1, 3, 4, 3), (2, 1, 3, 4, 4), (1, 2, 2, 3, 2), (1, 1, 3, 5, 6), (1, 1, 1, 2, 1))
    for rank_in, rank_out, a_size, key_size, res_size in shapes:
        pg, po = _key(g, o, rng, a_size, rank_in, rank_out + 1, key_size, k)
        a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), k)
        a[5] = fill_uniform(rng, a[5].shape, 61)      # fails the bound: per-limb kernels
        a[17, 0, 1, 3] = -(1 << 62)                   # one huge mask coefficient is enough
        a[18, 0, 0, 3] = -(1 << 62)                   # a huge body coefficient is harmless (added after the CRT)
        a[30] = 0
        want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), k)
        res_g = g.vec_znx_from_numpy(want)
        g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_keyswitch_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ks", rank_in, rank_out, a_size, key_size, res_size, bad[:10], len(bad))
    for kbits, rank in ((k, 1), (62, 1), (k, 2)):
        if (rank + 1) * 3 * n * 4 > 96 * 1024:
            continue
        pg, po = _key(g, o, rng, 3, rank + 1, rank + 1, 3, kbits)
        a = fill_uniform(rng, (batch, 3, rank + 1, n), k)
        want = np.zeros((batch, 3, rank + 1, n), dtype=np.int64)
        res_g = g.vec_znx_alloc(rank + 1, 3, batch)
        g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_external_product_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ep", kbits, rank, bad[:10], len(bad))
    # base2k = 25, two digits: S * K = 75 <= 128 and a narrower carry chain
    pg, po = _key(g, o, rng, 2, 1, 2, 3, 25)
    a = fill_uniform(rng, (batch, 2, 2, n), 25)
    want = np.zeros((batch, 3, 2, n), dtype=np.int64)
    res_g = g.vec_znx_alloc(2, 3, batch)
    g.glwe_keyswitch(res_g, 25, g.vec_znx_from_numpy(a), 25, pg, 25)
    g.sync()
    o.glwe_keyswitch_batch(want, 25, a, 25, po, 25)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("n", [256, 2048])
def test_glwe_automorphism(fl, n):
    """glwe_automorphism (poulpy-core/src/automorphism/glwe_ct.rs:51-72) = key-switch + X -> X^p, and the bare vec_znx_automorphism,
    against the oracle for several Galois elements (n = 2048 takes the single-kernel key-switch in the NTT120 flavour)."""
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(1300 + n + fl)
    k, batch = (12 if fl == pb.FFT64 else 18), 5
    pg, po = _key(g, o, rng, 3, 1, 2, 4, k)
    a = fill_uniform(rng, (batch, 3, 2, n), k)
    for p in (3, 5, -1, 2 * n - 1, 2 * 5 ** 3 + 1):
        want = np.zeros((batch, 3, 2, n), dtype=np.int64)
        res_g = g.vec_znx_alloc(2, 3, batch)
        g.glwe_automorphism(res_g, k, g.vec_znx_from_numpy(a), k, pg, k, p)
        g.sync()
        for b in range(batch):
            o.glwe_automorphism(want[b], k, a[b], k, po, k, p)
        assert np.array_equal(g.vec_znx_to_numpy(res_g), want), p
        x = g.vec_znx_from_numpy(a[0])
        y = g.vec_znx_alloc(2, 4)
        g.vec_znx_automorphism(p, y, 1, x, 0)
        wy = np.zeros((4, 2, n), dtype=np.int64)
        O.vec_znx_automorphism(p, wy, 1, a[0], 0)
        assert np.array_equal(g.vec_znx_to_numpy(y)[:, 1], wy[:, 1]), p


def test_gadget_kernel_random_shapes():
    """Randomised shape sweep through the single-kernel gadget product (n = 1024): ranks 1..3, 1..4 input limbs, 1..5 key limbs,
    output sizes below / equal / above the key size, base2k from 4 to 62 (S * K <= 128 selects the kernel, the rest falls back to the
    limb-wise kernels), batch 1..9 -- all bit for bit against the oracle."""
    n = 1024
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(4242)
    for trial in range(28):
        k = int(rng.choice([4, 8, 13, 18, 25, 31, 40, 52, 62]))
        rank_in, rank_out = int(rng.integers(1, 4)), int(rng.integers(1, 4))
        a_size, key_size, res_size = int(rng.integers(1, 5)), int(rng.integers(1, 6)), int(rng.integers(1, 7))
        batch = int(rng.integers(1, 10))
        ext = trial % 3 == 2
        digits = min(k, 50)  # keep |a|, |key| small enough that most ciphertexts stay on the collapsed path
        if ext:
            cols = rank_in + 1
            pg, po = _key(g, o, rng, a_size, cols, cols, key_size, digits)
            a = fill_uniform(rng, (batch, a_size, cols, n), digits)
            want = fill_uniform(rng, (batch, res_size, cols, n), 8)
            res_g = g.vec_znx_from_numpy(want)
            g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
            g.sync()
            o.glwe_external_product_batch(want, k, a, k, po, k)
        else:
            pg, po = _key(g, o, rng, a_size, rank_in, rank_out + 1, key_size, digits)
            a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), digits)
            want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), 8)
            res_g = g.vec_znx_from_numpy(want)
            g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
            g.sync()
            o.glwe_keyswitch_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g).reshape(want.shape)  # batch 1 comes back without the batch axis
        assert np.array_equal(got, want), (trial, ext, k, rank_in, rank_out, a_size, key_size, res_size, batch)


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096])
def test_fft64_gadget_kernel(n):
    """The single-kernel FFT64 gadget product (fft64_gadget.cu: forward FFTs, key products, inverse FFTs, rounding, add_small and the
    carry chain in one launch): key-switch and external product over ranks 1..3, output sizes below / equal / above the key size,
    one / two / four limbs in flight per column (LPR), more ciphertexts than CTAs, one unnormalised body -- bit for bit against the
    oracle's FFT64 restatement."""
    g, o = pb.Module(n, pb.FFT64), O.OracleModule(n, pb.FFT64)
    rng = np.random.default_rng(1300 + n)
    k = 14
    batch = 310 if n == 512 else 37
    #        rank_in rank_out a_size key_size res_size
    shapes = ((1, 1, 3, 4, 3), (2, 1, 3, 4, 5), (1, 2, 2, 3, 2), (1, 1, 2, 5, 6), (1, 1, 1, 2, 1), (1, 0, 2, 3, 3), (2, 3, 2, 2, 2), (1, 1, 4, 1, 2))
    for rank_in, rank_out, a_size, key_size, res_size in shapes:
        pg, po = _key(g, o, rng, a_size, rank_in, rank_out + 1, key_size, k)
        a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), k)
        a[3, :, 0] = fill_uniform(rng, a[3, :, 0].shape, 40)  # an unnormalised body only passes through add_small + normalize
        a[7] = 0
        want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), k)
        res_g = g.vec_znx_from_numpy(want)
        g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_keyswitch_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ks", rank_in, rank_out, a_size, key_size, res_size, bad[:10], len(bad))
    for rank, a_size, g_size, res_size in ((1, 3, 3, 3), (2, 2, 3, 2), (1, 2, 4, 5), (3, 1, 2, 2)):
        pg, po = _key(g, o, rng, a_size, rank + 1, rank + 1, g_size, k)
        a = fill_uniform(rng, (batch, a_size, rank + 1, n), k)
        want = fill_uniform(rng, (batch, res_size, rank + 1, n), k)
        res_g = g.vec_znx_from_numpy(want)
        g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        o.glwe_external_product_batch(want, k, a, k, po, k)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ep", rank, a_size, g_size, res_size, bad[:10], len(bad))


def test_fft64_gadget_more_than_16_input_polys():
    """The FFT64 gadget kernel takes at most 16 input polys (R = min(dnum * rank_in, rank_in * a.size)), though its shared memory would
    hold more at n = 512.  Shapes past that bound run the limb-wise sequence: an external product with R = 18 and a key-switch with R = 20,
    bit for bit against the oracle."""
    n, k, batch = 512, 14, 5
    g, o = pb.Module(n, pb.FFT64), O.OracleModule(n, pb.FFT64)
    rng = np.random.default_rng(1450)
    pg, po = _key(g, o, rng, 9, 2, 2, 3, k)  # rank 1, dnum 9: R = 2 * 9
    a = fill_uniform(rng, (batch, 9, 2, n), k)
    want = fill_uniform(rng, (batch, 3, 2, n), k)
    res_g = g.vec_znx_from_numpy(want)
    g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_external_product_batch(want, k, a, k, po, k)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)
    pg, po = _key(g, o, rng, 5, 4, 4, 3, k)  # rank 4 -> 3, dnum 5: R = 4 * 5
    a = fill_uniform(rng, (batch, 5, 5, n), k)
    want = fill_uniform(rng, (batch, 3, 4, n), k)
    res_g = g.vec_znx_from_numpy(want)
    g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    assert np.array_equal(g.vec_znx_to_numpy(res_g), want)


def test_fft64_gadget_bench_shape():
    """FFT64 key-switch at the bench shape (n = 4096, base2k = 18, three input limbs, key of four): fused kernel == unfused HAL sequence
    == oracle."""
    import os
    n, k, batch = 4096, 18, 24
    g, o = pb.Module(n, pb.FFT64), O.OracleModule(n, pb.FFT64)
    rng = np.random.default_rng(1400)
    pg, po = _key(g, o, rng, 3, 1, 2, 4, k)
    a = fill_uniform(rng, (batch, 3, 2, n), k)
    want = np.zeros((batch, 3, 2, n), dtype=np.int64)
    o.glwe_keyswitch_batch(want, k, a, k, po, k)
    for no_fusion in (0, 1):
        g.set_option(pb.hal.OPT_NO_FUSION, no_fusion)
        try:
            res_g = g.vec_znx_alloc(2, 3, batch)
            g.glwe_keyswitch(res_g, k, g.vec_znx_from_numpy(a), k, pg, k)
            g.sync()
        finally:
            g.set_option(pb.hal.OPT_NO_FUSION, 0)
        assert np.array_equal(g.vec_znx_to_numpy(res_g), want), no_fusion


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("ext", [False, True])
def test_full_bench_batch_4096(fl, ext):
    """BASELINE's full batch (4096 ciphertexts, key-switch at n = 4096 / external product at n = 2048, base2k = 18): 64 distinct
    ciphertexts replicated 64 times in shuffled order, every one of the 4096 outputs compared bit for bit with the oracle's result for
    its source -- the persistent loops of the single-kernel paths run their full length (28-37 ciphertexts per cluster / CTA)."""
    n, k, batch, distinct = (2048 if ext else 4096), 18, 4096, 64
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(1500 + fl + 2 * ext)
    if ext:
        pg, po = _key(g, o, rng, 3, 2, 2, 3, k)
    else:
        pg, po = _key(g, o, rng, 3, 1, 2, 4, k)
    src = fill_uniform(rng, (distinct, 3, 2, n), k)
    want = np.zeros((distinct, 3, 2, n), dtype=np.int64)
    if ext:
        o.glwe_external_product_batch(want, k, src, k, po, k)
    else:
        o.glwe_keyswitch_batch(want, k, src, k, po, k)
    perm = rng.permutation(batch) % distinct
    a = g.vec_znx_from_numpy(src[perm])
    res = g.vec_znx_alloc(2, 3, batch)
    (g.glwe_external_product if ext else g.glwe_keyswitch)(res, k, a, k, pg, k)
    g.sync()
    got = g.vec_znx_to_numpy(res)
    bad = [b for b in range(batch) if not np.array_equal(got[b], want[perm[b]])]
    assert not bad, (bad[:10], len(bad))


@pytest.mark.parametrize("dsize", [2, 3])
@pytest.mark.parametrize("n", [1024, 4096])
def test_gadget_kernel_dsize(dsize, n):
    """dsize > 1 through the single-kernel NTT120 path (the digit groups of keyswitching/glwe.rs:332-379 folded into the collapsed key):
    key-switch and external product, ranks 1..2, input sizes that are / are not multiples of dsize, fewer key rows than digit groups,
    a flagged ciphertext (whole batch redone limb by limb) -- bit for bit against the oracle."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(1600 + dsize + n)
    k, batch = 18, 9
    #        rank_in rank_out a_size dnum key_size res_size
    shapes = ((1, 1, 4, -1, 5, 4), (1, 1, 3, -1, 4, 3), (2, 1, 4, -1, 5, 3), (1, 2, 5, -1, 4, 6), (1, 1, 6, 1, 4, 4), (1, 1, 2, -1, 3, 3))
    for rank_in, rank_out, a_size, dnum, key_size, res_size in shapes:
        dnum = -(-a_size // dsize) if dnum < 0 else dnum
        pg, po = _key(g, o, rng, dnum, rank_in, rank_out + 1, key_size, k)
        for flagged in (False, True):
            a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), k)
            if flagged:
                a[4, 0, 1, 7] = 1 << 61
            want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), k)
            res_g = g.vec_znx_from_numpy(want)
            a_g = g.vec_znx_from_numpy(a)
            l0 = g.launch_count
            g.glwe_keyswitch(res_g, k, a_g, k, pg, k, dsize)
            g.sync()
            launches = g.launch_count - l0
            o.glwe_keyswitch_batch(want, k, a, k, po, k, dsize)
            got = g.vec_znx_to_numpy(res_g)
            bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
            assert not bad, ("ks", rank_in, rank_out, a_size, dnum, key_size, res_size, flagged, bad)
            if key_size <= 4 and not flagged:  # short keys fit the collapsed form: one product kernel + its three key pre-passes
                assert launches <= 5, (launches, rank_in, rank_out, a_size, key_size)
            elif key_size <= 4:
                assert launches > 8, launches  # the flagged batch was redone by the limb-wise sequence
    for rank, a_size, g_size, res_size in ((1, 4, 5, 4), (1, 3, 3, 3), (2, 2, 3, 2), (1, 4, 2, 5)):
        dnum = -(-a_size // dsize)
        pg, po = _key(g, o, rng, dnum, rank + 1, rank + 1, g_size, k)
        a = fill_uniform(rng, (batch, a_size, rank + 1, n), k)
        want = fill_uniform(rng, (batch, res_size, rank + 1, n), k)
        res_g = g.vec_znx_from_numpy(want)
        g.glwe_external_product(res_g, k, g.vec_znx_from_numpy(a), k, pg, k, dsize)
        g.sync()
        o.glwe_external_product_batch(want, k, a, k, po, k, dsize)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ep", rank, a_size, g_size, res_size, bad)


@pytest.mark.parametrize("n", [1024, 4096])
def test_fft64_gadget_kernel_dsize2(n):
    """dsize = 2 through the single-kernel FFT64 path (per-row key limb shift instead of limb_offset vmp + dft_add_assign): key-switch and
    external product against the oracle's FFT64 restatement, with the launch count proving the fused route was taken."""
    g, o = pb.Module(n, pb.FFT64), O.OracleModule(n, pb.FFT64)
    rng = np.random.default_rng(1700 + n)
    k, batch, dsize = 13, 11, 2
    #        rank_in rank_out a_size dnum key_size res_size
    shapes = ((1, 1, 4, -1, 5, 4), (1, 1, 3, -1, 4, 3), (1, 2, 4, -1, 3, 5), (1, 1, 4, 1, 4, 4), (1, 1, 2, -1, 3, 3))
    for rank_in, rank_out, a_size, dnum, key_size, res_size in shapes:
        dnum = -(-a_size // dsize) if dnum < 0 else dnum
        pg, po = _key(g, o, rng, dnum, rank_in, rank_out + 1, key_size, k)
        a = fill_uniform(rng, (batch, a_size, rank_in + 1, n), k)
        want = fill_uniform(rng, (batch, res_size, rank_out + 1, n), k)
        res_g, a_g = g.vec_znx_from_numpy(want), g.vec_znx_from_numpy(a)
        l0 = g.launch_count
        g.glwe_keyswitch(res_g, k, a_g, k, pg, k, dsize)
        g.sync()
        fits = (rank_out + 1) * (n // 16) <= 512 and (rank_in * a_size + rank_out + 1) * (n // 2 + n // 16 + 2) * 16 <= 227 * 1024
        if fits:  # slots and planes fit one CTA: key re-layout + the product kernel, nothing else
            assert g.launch_count - l0 <= 2, (g.launch_count - l0, rank_in, rank_out, a_size, key_size)
        o.glwe_keyswitch_batch(want, k, a, k, po, k, dsize)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ks", rank_in, rank_out, a_size, dnum, key_size, res_size, bad)
    for rank, a_size, g_size, res_size in ((1, 2, 3, 2), (1, 3, 3, 4)):
        if (rank + 1) * a_size > (4 if n == 4096 else 8):
            continue
        dnum = -(-a_size // dsize)
        pg, po = _key(g, o, rng, dnum, rank + 1, rank + 1, g_size, k)
        a = fill_uniform(rng, (batch, a_size, rank + 1, n), k)
        want = fill_uniform(rng, (batch, res_size, rank + 1, n), k)
        res_g, a_g = g.vec_znx_from_numpy(want), g.vec_znx_from_numpy(a)
        l0 = g.launch_count
        g.glwe_external_product(res_g, k, a_g, k, pg, k, dsize)
        g.sync()
        assert g.launch_count - l0 <= 2, (g.launch_count - l0, rank, a_size, g_size)
        o.glwe_external_product_batch(want, k, a, k, po, k, dsize)
        got = g.vec_znx_to_numpy(res_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, ("ep", rank, a_size, g_size, res_size, bad)


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("dsize", [1, 2])
@pytest.mark.parametrize("ext", [False, True])
def test_in_place_with_flagged_ciphertext(fl, dsize, ext):
    """The `_assign` forms (res IS a: keyswitching/glwe.rs:111-165, external_product/glwe.rs:143-195) through every route, with one
    ciphertext outside the collapsed-key bound: with dsize > 1 a flagged ciphertext sends the WHOLE batch to the limb-wise sequence, which
    must still find intact inputs although the single kernel has already produced outputs for the others (ADVICE r1: core.cu:169)."""
    n, k, batch, size = 1024, 18, 7, 4
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(1700 + fl + 2 * dsize + ext)
    cols_in = 2 if ext else 1
    pg, po = _key(g, o, rng, -(-size // dsize), cols_in, 2, size, k)
    for flagged in (False, True):
        a = fill_uniform(rng, (batch, size, 2, n), k)
        if flagged and fl == pb.NTT120:
            a[3, 0, 1, 5] = 1 << 61
        want = np.zeros_like(a)
        (o.glwe_external_product_batch if ext else o.glwe_keyswitch_batch)(want, k, a, k, po, k, dsize)
        a_g = g.vec_znx_from_numpy(a)
        (g.glwe_external_product if ext else g.glwe_keyswitch)(a_g, k, a_g, k, pg, k, dsize)
        g.sync()
        got = g.vec_znx_to_numpy(a_g)
        bad = [b for b in range(batch) if not np.array_equal(got[b], want[b])]
        assert not bad, (flagged, bad)


@pytest.mark.parametrize("fl", FLAVOURS)
def test_partial_overlap_is_rejected(fl):
    """backend_safety_contract.md "Aliasing": overlapping operands that are not the same ciphertexts return PGB_ERR_ALIAS (-3) instead of
    computing garbage: shifted views of one buffer for the compositions, and any overlap for the out-of-place-only helpers."""
    n, k, batch = 1024, 18, 4
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(1750)
    pg, _ = _key(g, o, rng, 3, 1, 2, 3, k)
    big = g.vec_znx_alloc(2, 3, batch + 1)
    item = big.batch_stride
    a = pb.hal.VecZnx(big.buf, n, 2, 3, offset=0, batch=batch, batch_stride=item)
    r = pb.hal.VecZnx(big.buf, n, 2, 3, offset=item // 2, batch=batch, batch_stride=item)
    for fn in (lambda: g.glwe_keyswitch(r, k, a, k, pg, k), lambda: g.vec_znx_automorphism(3, r, 0, a, 0),
               lambda: g.vec_znx_rotate(3, r, 0, a, 0), lambda: g.vec_znx_mul_xp_minus_one(3, a, 0, a, 1)):
        with pytest.raises(pb.PoulpyError, match=r"\[-3\]"):
            fn()


@pytest.mark.parametrize("fl", FLAVOURS)
def test_pinned_key_cache(fl):
    """pgb_gadget_key_pin: the per-key pre-passes of the single-kernel gadget product run once for a pinned key (fewer launches per call,
    identical results), a vmp_prepare into the pinned key drops the cached forms (the next call sees the NEW key), two call shapes on one
    pinned key keep separate forms, and unpin restores the per-call behaviour."""
    n, k, batch = 1024, 18, 5
    g, o = pb.Module(n, fl), O.OracleModule(n, fl)
    rng = np.random.default_rng(1800 + fl)
    mats = [fill_uniform(rng, (3, 1, 4, 2, n), k) for _ in range(2)]
    pg, po = g.vmp_pmat_alloc(3, 1, 2, 4), o.vmp_pmat_alloc(3, 1, 2, 4)

    def run(a_size):
        a = fill_uniform(rng, (batch, a_size, 2, n), k)
        want = np.zeros((batch, a_size, 2, n), dtype=np.int64)
        o.glwe_keyswitch_batch(want, k, a, k, po, k, 1)
        res = g.vec_znx_from_numpy(fill_uniform(rng, want.shape, k))
        a_g = g.vec_znx_from_numpy(a)
        l0 = g.launch_count
        g.glwe_keyswitch(res, k, a_g, k, pg, k, 1)
        g.sync()
        assert np.array_equal(g.vec_znx_to_numpy(res), want)
        return g.launch_count - l0

    g.vmp_prepare(pg, g.mat_znx_from_numpy(mats[0]))
    o.vmp_prepare(po, mats[0])
    unpinned = run(3)
    g.gadget_key_pin(pg)
    first, second = run(3), run(3)
    assert first == unpinned and second < first, (unpinned, first, second)   # pre-passes only on the first pinned call
    other_first, other_second = run(2), run(2)                                # another call shape: its own cached form
    assert other_second < other_first and run(3) == second
    g.vmp_prepare(pg, g.mat_znx_from_numpy(mats[1]))                          # new key bytes in the pinned buffer
    o.vmp_prepare(po, mats[1])
    assert run(3) == first and run(3) == second
    g.gadget_key_unpin(pg)
    assert run(3) == unpinned


def _negacyclic_np(a, b):
    """Exact negacyclic product of two small-integer polynomials with numpy (|result| < 2^62 for the digit sizes used here)."""
    n = len(a)
    full = np.convolve(np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64))
    res = full[:n].copy()
    res[: n - 1] -= full[n:]
    return res


def _phase_int(ct, secrets, k):
    """body + sum mask_c (*) s_c as exact integers scaled by 2^(size k) (Python ints), for ct (size, cols, n)."""
    size, _, n = ct.shape
    out = [0] * n
    for j in range(size):
        v = ct[j, 0].astype(np.int64).copy()
        for c, s in enumerate(secrets):
            v = v + _negacyclic_np(ct[j, 1 + c], s)
        w = 1 << ((size - 1 - j) * k)
        out = [o + int(x) * w for o, x in zip(out, v)]
    return out


@pytest.mark.parametrize("fl", FLAVOURS)
@pytest.mark.parametrize("n", [1024, 4096])
def test_noiseless_keyswitch_preserves_the_phase_on_the_device(fl, n):
    """L4 (SURVEY 8c; reference: poulpy-core/src/test_suite/keyswitch/glwe_ct.rs:132-156): with a NOISE-FREE key-switching key from s to s'
    the single-kernel key-switch maps any ciphertext to one with the same phase under s' -- exactly (no limb is truncated here), checked
    with integer arithmetic that shares nothing with the oracle.  n = 4096 / base2k 18 is the headline shape."""
    k, a_size = 18, 3
    key_size = a_size + 1
    rng = np.random.default_rng(1900 + fl + n)
    g = pb.Module(n, fl)
    s_in = rng.integers(-1, 2, size=n).astype(np.int64)
    s_out = rng.integers(-1, 2, size=n).astype(np.int64)
    key = np.zeros((a_size, 1, key_size, 2, n), dtype=np.int64)
    for d in range(a_size):
        mask = fill_uniform(rng, (key_size, n), k)
        acc = [0] * n  # s_in * 2^-((d+1)k) - mask (*) s_out, scaled by 2^(key_size k)
        for j in range(key_size):
            w = 1 << ((key_size - 1 - j) * k)
            prod = _negacyclic_np(mask[j], s_out)
            for i in range(n):
                acc[i] -= int(prod[i]) * w
        wmsg = 1 << ((key_size - 1 - d) * k)
        for i in range(n):
            acc[i] += int(s_in[i]) * wmsg
        mod = 1 << (key_size * k)
        body = np.zeros((key_size, n), dtype=np.int64)
        for i in range(n):
            v = acc[i] % mod
            for j in range(key_size - 1, -1, -1):
                dgt = v & ((1 << k) - 1)
                if dgt >= 1 << (k - 1):
                    dgt -= 1 << k
                body[j, i] = dgt
                v = (v - dgt) >> k
        key[d, 0, :, 0, :] = body
        key[d, 0, :, 1, :] = mask
    pg = g.vmp_pmat_alloc(a_size, 1, 2, key_size)
    g.vmp_prepare(pg, g.mat_znx_from_numpy(key))
    batch = 3
    a = fill_uniform(rng, (batch, a_size, 2, n), k)
    res = g.vec_znx_alloc(2, key_size, batch)
    g.glwe_keyswitch(res, k, g.vec_znx_from_numpy(a), k, pg, k)
    g.sync()
    got = g.vec_znx_to_numpy(res)
    for b in range(batch):
        want = _phase_int(a[b], [s_in], k)       # scaled by 2^(a_size k)
        have = _phase_int(got[b], [s_out], k)    # scaled by 2^(key_size k)
        mod = 1 << (key_size * k)
        shift = 1 << ((key_size - a_size) * k)
        assert all((h - w * shift) % mod == 0 for h, w in zip(have, want)), b


@pytest.mark.parametrize("two_devices", [False, True])
def test_keyswitch_host_sharded_over_modules(two_devices):
    """pgb_glwe_keyswitch_host_sharded: ONE host call drives several modules from several host threads (Module is Sync + Send in the
    reference, poulpy-hal/src/layouts/module.rs:103-104).  two_devices = False: two modules on device 0 (thread safety of the library on
    one GPU: separate streams, workspaces, thread-local errors); True: one module per GPU, each with its replica of the key (skipped on a
    one-GPU box).  A ragged batch checks the contiguous split; results bit for bit against the oracle."""
    if two_devices and pb.hal.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    n, k, batch = 1024, 18, 37
    devs = (0, 1) if two_devices else (0, 0)
    rng = np.random.default_rng(2000)
    mat = fill_uniform(rng, (3, 1, 4, 2, n), k)
    o = O.OracleModule(n, O.NTT120)
    po = o.vmp_pmat_alloc(3, 1, 2, 4)
    o.vmp_prepare(po, mat)
    mods, keys = [], []
    for d in devs:
        m = pb.Module(n, pb.NTT120, device=d)
        pm = m.vmp_pmat_alloc(3, 1, 2, 4)
        m.vmp_prepare(pm, m.mat_znx_from_numpy(mat))
        m.gadget_key_pin(pm)
        mods.append(m)
        keys.append(pm)
    a = fill_uniform(rng, (batch, 3, 2, n), k)
    want = np.zeros_like(a)
    o.glwe_keyswitch_batch(want, k, a, k, po, k, 1)
    res = np.full_like(a, -3)
    pb.hal.glwe_keyswitch_host_sharded(mods, keys, res, k, a, k, k)
    assert np.array_equal(res, want)
    with pytest.raises(pb.PoulpyError):  # an error inside a shard surfaces in the caller's thread with the shard named
        pb.hal.glwe_keyswitch_host_sharded(mods, keys, res[:, :, :1], k, a, k, k)
