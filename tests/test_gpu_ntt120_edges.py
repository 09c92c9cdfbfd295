"""The NTT120 kernels at the edges of the magnitude arguments that make them bit-exact with the reference.

A. The two-prime blind rotation (cggi_ntt_fused.cu) computes modulo q0 q1 only when the host-side bound
   acc_bits + key_bits + rn_bits + bs_bits <= 58 proves |acc_add| <= 2^58 < q0 q1 / 2; otherwise it falls back to the four-prime
   limb-wise route of cggi.cu.  The cases sit at the bound, one and two bits past it (with an integer that really exceeds q0 q1 / 2),
   and put the one wide key coefficient / LUT word where the device scans end.  The route is witnessed by the launch count: the
   two-prime route costs a handful of launches, the limb-wise route at least one per block.

   The kernel's fail flag (`*handled = false` after the launch, accumulator initialised again) is not reachable from valid inputs: the
   only accumulator values it does not produce itself are the initial X^b * LUT, a negacyclic rotation of the LUT limbs that
   cggi_fused_ntt120 scans (lut_words = n * min(res.size, lut.size), exactly the limbs the rotation copies).  A LUT word of b bits has
   magnitude <= 2^b (-2^b only when negative, and its negation 2^b is still <= acc_limit = 2^acc_bits), so every load passes the
   device check; later loads are balanced base-2^K digits, |d| <= 2^(K-1) <= 2^acc_bits.  No test forces it.

B. Lazily reducing u64 sums (vmp, svp, cnv_apply_dft, cggi_block_ntt120_kernel, the two-prime kernel) fed with operands built from
   -delta_0 (the polynomial -1): every canonical residue is q - 1, the largest term each sum can see.

C. Full-width integers of the big domain: i128 normalisation over the whole centred range, the inverse transform's CRT at
   +-(Q - 1) / 2, and the full-i64 forward transform, for every ring degree.

Every comparison is bit for bit, against the oracle and, where stated, against a Python big-integer model."""
import numpy as np
import pytest

import poulpy_b200 as pb
from poulpy_b200 import hal as H
from oracle import pyoracle as O
from semantics import digits_of_torus_int
from util import fill_uniform, negacyclic_mul

pytestmark = pytest.mark.gpu

Q2 = O.Q[0] * O.Q[1]
QALL = O.Q[0] * O.Q[1] * O.Q[2] * O.Q[3]
HALF_Q = (QALL - 1) // 2


# ---------------------------------------------------------------------------------------------------------------------------------------
# blind-rotation harness
# ---------------------------------------------------------------------------------------------------------------------------------------
class _Rot:
    """n_lwe prepared GGSWs in one device buffer (VmpPMat of GGSW 0 describes the key) + their oracle twins."""

    def __init__(self, n, mats, pin):
        self.n = n
        self.n_lwe, self.dnum, self.cols, self.size = mats.shape[0], mats.shape[1], mats.shape[2], mats.shape[3]
        self.g, self.o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
        self.per = n * self.dnum * self.cols * self.cols * self.size * self.g.prep_bytes
        self.buf = pb.DevBuf(self.per * self.n_lwe)
        self.obrk = [None] * self.n_lwe
        for i in range(self.n_lwe):
            self.prepare(i, mats[i])
        self.brk = H.VmpPMat(self.buf, n, self.dnum, self.cols, self.cols, self.size)
        if pin:
            self.g.gadget_key_pin(self.brk)
        self.xg, self.xo = self.g.cggi_x_pow_a(), self.o.cggi_x_pow_a()
        self.g.sync()

    def prepare(self, i, mat):
        mat = np.ascontiguousarray(mat, dtype=np.int64)
        self.g.vmp_prepare(H.VmpPMat(self.buf, self.n, self.dnum, self.cols, self.cols, self.size, offset=i * self.per),
                           self.g.mat_znx_from_numpy(mat))
        pm = self.o.vmp_pmat_alloc(self.dnum, self.cols, self.cols, self.size)
        self.o.vmp_prepare(pm, mat)
        self.obrk[i] = pm

    def oracle(self, lwe, lut, block, k, out_size, n_lwe=None):
        n_lwe = self.n_lwe if n_lwe is None else n_lwe
        want = np.zeros((lwe.shape[0], out_size, self.cols, self.n), dtype=np.int64)
        for b in range(lwe.shape[0]):
            self.o.cggi_blind_rotate_block_binary(want[b], lwe[b, : n_lwe + 1], lut, self.obrk[:n_lwe], self.xo, block, k)
        return want

    def run(self, lwe, lut, block, k, out_size, primes=0, n_lwe=None):
        """-> (result, kernel launches of the call); primes = 4 forces the limb-wise route"""
        n_lwe = self.n_lwe if n_lwe is None else n_lwe
        g = self.g
        lwe = np.ascontiguousarray(lwe[:, : n_lwe + 1])
        lwe_dev = pb.DevBuf(lwe.nbytes)
        lwe_dev.upload(lwe)
        lut_g = g.vec_znx_from_numpy(lut)
        shape = (lwe.shape[0], out_size, self.cols, self.n)
        res = g.vec_znx_from_numpy(np.full(shape, 12345, dtype=np.int64))  # garbage pre-fill
        g.set_option(H.OPT_CGGI_NTT_PRIMES, primes)
        g.sync()
        l0 = g.launch_count
        g.cggi_blind_rotate(res, lwe_dev, n_lwe, lut_g, self.brk, self.xg, block, k)
        g.sync()
        launches = g.launch_count - l0
        g.set_option(H.OPT_CGGI_NTT_PRIMES, 0)
        return g.vec_znx_to_numpy(res).reshape(shape), launches

    def check(self, lwe, lut, block, k, out_size, two_primes):
        """default route, forced four primes and the oracle all equal; the default route is the one expected"""
        nblk = self.n_lwe // block
        assert nblk >= 12
        want = self.oracle(lwe, lut, block, k, out_size)
        got, launches = self.run(lwe, lut, block, k, out_size)
        got4, launches4 = self.run(lwe, lut, block, k, out_size, primes=4)
        assert np.array_equal(got4, want)
        bad = [b for b in range(lwe.shape[0]) if not np.array_equal(got[b], want[b])]
        assert not bad, bad
        assert launches4 >= nblk, launches4
        if two_primes:
            assert launches < nblk, ("expected the two-prime route", launches, nblk)
        else:
            assert launches >= nblk, ("expected the limb-wise route", launches, nblk)


def _rot_int(p, a):
    """X^a * p in Z[X]/(X^n + 1) on Python ints"""
    n = len(p)
    a %= 2 * n
    res = [0] * n
    for i, v in enumerate(p):
        j = i + a
        s = 1
        while j >= n:
            j -= n
            s = -s
        res[j] += s * v
    return res


def _first_block_acc_add(mats, lut, lwe0, block, dnum, cols):
    """Exact first-block acc_add[c] = sum_t (X^{a_t} - 1) sum_r acc[r] (*) BRK_t[r][c] of one ciphertext, Python ints; acc = X^b LUT in
    column 0 (rows r = limb * cols + col, limbs < dnum)."""
    n = lut.shape[-1]
    size = mats.shape[3]
    acc = [[0] * n for _ in range(cols * dnum)]
    for j in range(min(dnum, lut.shape[0])):
        acc[j * cols] = _rot_int([int(x) for x in lut[j, 0]], int(lwe0[0]))
    memo = {}
    out = [[0] * n for _ in range(size * cols)]
    for t in range(block):
        for c in range(size * cols):
            j, co = divmod(c, cols)
            v = [0] * n
            for r in range(cols * dnum):
                if not any(acc[r]):
                    continue
                d, ci = divmod(r, cols)
                key = mats[t, d, ci, j, co]
                mk = (r, bytes(np.ascontiguousarray(key).data))
                if mk not in memo:
                    memo[mk] = negacyclic_mul(acc[r], key)
                v = [x + y for x, y in zip(v, memo[mk])]
            w = _rot_int(v, int(lwe0[1 + t]))
            out[c] = [o + x - y for o, x, y in zip(out[c], w, v)]
    return out


# ---------------------------------------------------------------------------------------------------------------------------------------
# A. two-prime blind rotation at its bound
# ---------------------------------------------------------------------------------------------------------------------------------------
N, RANK, DNUM, BRK_SIZE, BLOCK = 512, 1, 2, 2, 4   # R = cols * dnum = 4, C = 4, rn_bits = 11, bs_bits = 3
COLS = RANK + 1


def _bound_case(k, lut_bits, key_bits, seed, n_lwe=48, batch=4):
    """LUT digits all -2^lut_bits (lut_bits bits: the LUT scan counts a negative word by its one's complement).  The key scan counts the
    bit length of |key|, so key_bits-bit keys reach 2^key_bits - 1: the first block's keys are -(2^key_bits - 1) in every coefficient,
    the later ones uniform in that range.  Ciphertext 0 has b = 1 and a_t = n in the first block: X^1 LUT is +2^lut_bits at x^0 and
    -2^lut_bits elsewhere, so every term of coefficient 0 of its product with the constant negative key has the same sign, and each
    (X^n - 1) = -2.  -> (mats, lut, lwe, the exact largest |acc_add| of the first block)"""
    rng = np.random.default_rng(seed)
    kmax = (1 << key_bits) - 1
    mats = rng.integers(-kmax, kmax, size=(n_lwe, DNUM, COLS, BRK_SIZE, COLS, N), dtype=np.int64, endpoint=True)
    mats[:BLOCK] = -kmax
    lut = np.full((BRK_SIZE, 1, N), -(1 << lut_bits), dtype=np.int64)
    lwe = rng.integers(-N, N, size=(batch, n_lwe + 1), dtype=np.int64)
    lwe[0, 0] = 1
    lwe[0, 1:BLOCK + 1] = N
    # BLOCK keys x 2 (the (X^n - 1) factors) x DNUM filled rows x N terms of 2^lut_bits kmax
    peak = BLOCK * 2 * DNUM * N * (1 << lut_bits) * kmax
    add = _first_block_acc_add(mats, lut, lwe[0], BLOCK, DNUM, COLS)
    assert max(abs(v) for p in add for v in p) == peak
    return mats, lut, lwe, peak


@pytest.mark.parametrize("k,lut_bits,key_bits", [(18, 17, 27), (30, 29, 15)], ids=["k18_key27", "k30_key15"])
def test_two_primes_at_the_bound(k, lut_bits, key_bits):
    """acc_bits + key_bits + 11 + 3 = 58: the largest sum the host admits.  The first block's integers reach 2^57 (1 - 2^-key_bits): half
    the proven bound 2^58, because only the column-0 rows of X^b LUT are filled; reconstructed exactly from two residues."""
    mats, lut, lwe, peak = _bound_case(k, lut_bits, key_bits, 8000 + k)
    assert peak == (1 << 57) - (1 << (57 - key_bits))
    rot = _Rot(N, mats, pin=True)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=True)


def test_two_primes_one_bit_past_the_bound():
    """28-bit key coefficients: sum = 59.  The integers (< 2^58) would still fit two primes, so only the route tells a bound that is one
    bit too loose."""
    k = 18
    mats, lut, lwe, peak = _bound_case(k, 17, 28, 8101)
    assert (1 << 57) < peak < Q2 // 2
    rot = _Rot(N, mats, pin=True)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)


def test_two_primes_two_bits_past_the_bound():
    """29-bit key coefficients: sum = 60, and the first block's integer 2^59 - 2^30 really exceeds q0 q1 / 2: a two-prime launch would
    return it wrapped, so the values alone catch a bound that is two bits too loose."""
    k = 18
    mats, lut, lwe, peak = _bound_case(k, 17, 29, 8102)
    assert peak > Q2 // 2
    rot = _Rot(N, mats, pin=True)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)


@pytest.mark.parametrize("case", ["lut30", "base2k31"])
def test_two_primes_declines_wide_accumulators(case):
    """A 30-bit LUT word (acc_bits > 29: the kernel's single-word residue conversion needs |acc| < q) and base2k 31 fall back, although
    the keys are small enough for the sum."""
    rng = np.random.default_rng(8200 + len(case))
    mats = fill_uniform(rng, (48, DNUM, COLS, BRK_SIZE, COLS, N), 4)
    if case == "lut30":
        k = 18
        lut = fill_uniform(rng, (BRK_SIZE, 1, N), k)
        lut[0, 0, 7] = -(1 << 30)
        lut[1, 0, N - 1] = (1 << 30) - 1  # 30 bits, above every prime: not a canonical residue
    else:
        k = 31
        lut = fill_uniform(rng, (BRK_SIZE, 1, N), k)
    lwe = rng.integers(-N, N, size=(3, 49), dtype=np.int64)
    rot = _Rot(N, mats, pin=True)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)


def test_two_primes_scan_reaches_the_last_coefficient():
    """brk_max_bits transforms the key in 32 MiB chunks (4096 polys at n = 512): with 260 GGSWs of 16 polys the last GGSW sits in the
    second, partial chunk.  One 2^40 coefficient at the last coefficient of the last poly of the last GGSW, 18-bit digits elsewhere:
    unpinned and pinned, the call must fall back.  Then the same GGSW is prepared again in the pinned key, narrow (the cached bound is
    dropped: two primes) and wide again (dropped again: four primes)."""
    k, n_lwe = 18, 260
    assert n_lwe * COLS * DNUM * COLS * BRK_SIZE > (32 << 20) // (16 * N)
    rng = np.random.default_rng(8300)
    mats = fill_uniform(rng, (n_lwe, DNUM, COLS, BRK_SIZE, COLS, N), 18)
    narrow = mats[-1].copy()
    wide = narrow.copy()
    wide[-1, -1, -1, -1, -1] = 1 << 40
    mats[-1] = wide
    lut = fill_uniform(rng, (BRK_SIZE, 1, N), k)
    lwe = rng.integers(-N, N, size=(2, n_lwe + 1), dtype=np.int64)
    rot = _Rot(N, mats, pin=False)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)
    rot.g.gadget_key_pin(rot.brk)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)
    rot.prepare(n_lwe - 1, narrow)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=True)
    rot.prepare(n_lwe - 1, wide)
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)


def test_two_primes_lut_scan_covers_the_copied_limbs():
    """The LUT scan covers exactly the limbs the rotation copies (min(res.size, lut.size)): one wide word in the last copied limb falls
    back; the same word in a limb beyond res.size is never read and leaves the two-prime route in place."""
    k = 18
    rng = np.random.default_rng(8400)
    mats = fill_uniform(rng, (48, DNUM, COLS, BRK_SIZE, COLS, N), 18)
    rot = _Rot(N, mats, pin=True)
    lwe = rng.integers(-N, N, size=(3, 49), dtype=np.int64)
    lut = fill_uniform(rng, (BRK_SIZE + 1, 1, N), k)
    lut[BRK_SIZE, 0, N - 1] = 1 << 40
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=True)
    lut[BRK_SIZE - 1, 0, N - 1] = 1 << 40
    rot.check(lwe, lut, BLOCK, k, BRK_SIZE, two_primes=False)


def test_gadget_declines_three_primes_for_one_wide_last_coefficient():
    """The gadget kernel's key scan: one 2^40 coefficient at the very end of a pinned 18-bit key sends it to four primes."""
    n, k = 1024, 18
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(8500)
    a = fill_uniform(rng, (5, 3, 2, n), k)
    for wide, primes in ((False, 3), (True, 4)):
        mat = fill_uniform(rng, (3, 1, 3, 2, n), k)
        if wide:
            mat[-1, -1, -1, -1, -1] = 1 << 40
        pg, po = g.vmp_pmat_alloc(3, 1, 2, 3), o.vmp_pmat_alloc(3, 1, 2, 3)
        g.vmp_prepare(pg, g.mat_znx_from_numpy(mat))
        o.vmp_prepare(po, mat)
        g.gadget_key_pin(pg)
        want = np.zeros((5, 3, 2, n), dtype=np.int64)
        o.glwe_keyswitch_batch(want, k, a, k, po, k)
        res = g.vec_znx_alloc(2, 3, 5)
        g.set_option(H.OPT_LAST_GADGET_PRIMES, 0)
        g.glwe_keyswitch(res, k, g.vec_znx_from_numpy(a), k, pg, k)
        g.sync()
        assert g.get_option(H.OPT_LAST_GADGET_PRIMES) == primes, wide
        assert np.array_equal(g.vec_znx_to_numpy(res), want), wide


# ---------------------------------------------------------------------------------------------------------------------------------------
# B. extreme residues (every canonical residue q - 1) through the lazily reducing kernels
# ---------------------------------------------------------------------------------------------------------------------------------------
def _minus_delta(shape):
    x = np.zeros(shape, dtype=np.int64)
    x[..., 0] = -1
    return x


def _all_q_minus_1(planes):
    """planes: uint32 (..., 4, n) canonical residue planes"""
    return all(np.all(planes[..., k, :] == q - 1) for k, q in enumerate(O.Q))


def _vmp_extreme(n, rows, cols_in, cols_out, size, batch, options):
    """-delta_0 inputs and key: every product is (q - 1)^2 and every row sum reaches rows * cols_in (q - 1)^2 before its reduction."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    a = _minus_delta((rows, cols_in, n))
    adg = g.vec_znx_dft_alloc(cols_in, rows, batch)
    ado = o.vec_znx_dft_alloc(cols_in, rows)
    a_g = g.vec_znx_from_numpy(np.broadcast_to(a, (batch,) + a.shape))
    for c in range(cols_in):
        g.vec_znx_dft_apply(1, 0, adg, c, a_g, c)
        o.vec_znx_dft_apply(1, 0, ado, c, a, c)
    assert _all_q_minus_1(adg.buf.download(np.uint32, (batch, rows, cols_in, 4, n)))
    mat = _minus_delta((rows, cols_in, size, cols_out, n))
    pmg, pmo = g.vmp_pmat_alloc(rows, cols_in, cols_out, size), o.vmp_pmat_alloc(rows, cols_in, cols_out, size)
    g.vmp_prepare(pmg, g.mat_znx_from_numpy(mat))
    o.vmp_prepare(pmo, mat)
    assert _all_q_minus_1(pmg.buf.download(np.uint32, (rows * cols_in * size * cols_out, 4, n)))
    ro = o.vec_znx_dft_alloc(cols_out, size)
    o.vmp_apply_dft_to_dft(ro, ado, pmo, 0)
    want = o.vec_znx_idft_apply_consume(ro)
    assert np.array_equal(O.i128_to_int(want[:, :, 0]), np.full((size, cols_out), rows * cols_in, dtype=object))
    for opt, val in options:
        g.set_option(opt, val)
        rg = g.vec_znx_dft_alloc(cols_out, size, batch)
        rg.buf.upload(np.full(rg.buf.nbytes, 0xA5, dtype=np.uint8))
        g.vmp_apply_dft_to_dft(rg, adg, pmg, 0)
        g.vec_znx_idft_apply_consume(rg)  # in place, every batch item
        g.sync()
        g.set_option(opt, 0)
        big = rg.buf.download(np.uint64, (batch, size, cols_out, n, 2))
        for b in range(batch):
            assert np.array_equal(big[b], want), (opt, val, b)


@pytest.mark.parametrize("cols_in", [1, 2])
@pytest.mark.parametrize("rows", [16, 17, 32, 33])
def test_vmp_extreme_residues_per_item(rows, cols_in):
    """The per-item kernel with every output tile width (OPT_VMP_CT 2, 4, 8; C = 8 output polys so CT = 8 is taken)."""
    _vmp_extreme(64, rows, cols_in, 2, 4, 3, [(H.OPT_VMP_CT, 0), (H.OPT_VMP_CT, 2), (H.OPT_VMP_CT, 4), (H.OPT_VMP_CT, 8)])


@pytest.mark.parametrize("cols_in", [1, 2])
@pytest.mark.parametrize("rows", [16, 17, 32, 33])
def test_vmp_extreme_residues_batch_tiled(rows, cols_in):
    """A key of >= 48 MiB with batch >= 4 takes the batch-tiled kernel; OPT_VMP_NO_BT sends the same call to the per-item kernel."""
    cols_out, size = 2, 4
    n = 64
    while rows * cols_in * cols_out * size * 16 * n < (48 << 20):
        n *= 2
    _vmp_extreme(n, rows, cols_in, cols_out, size, 4, [(H.OPT_VMP_NO_BT, 0), (H.OPT_VMP_NO_BT, 1)])


def test_svp_extreme_residues():
    """svp of prepared -delta_0 with the transform of -delta_0: (q - 1)^2 in every frequency, result delta_0."""
    n, size = 256, 3
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    s = _minus_delta((1, n))
    pg, po = g.svp_ppol_alloc(1), o.svp_ppol_alloc(1)
    g.svp_prepare(pg, 0, g.scalar_znx_from_numpy(s), 0)
    o.svp_prepare(po, 0, s, 0)
    assert _all_q_minus_1(pg.buf.download(np.uint32, (1, 4, n)))
    b = _minus_delta((size, 1, n))
    bdg, bdo = g.vec_znx_dft_alloc(1, size), o.vec_znx_dft_alloc(1, size)
    g.vec_znx_dft_apply(1, 0, bdg, 0, g.vec_znx_from_numpy(b), 0)
    o.vec_znx_dft_apply(1, 0, bdo, 0, b, 0)
    rg, ro = g.vec_znx_dft_alloc(1, size), o.vec_znx_dft_alloc(1, size)
    g.svp_apply_dft_to_dft(rg, 0, pg, 0, bdg, 0)
    o.svp_apply_dft_to_dft(ro, 0, po, 0, bdo, 0)
    got, want = g.vec_znx_big_to_numpy(g.vec_znx_idft_apply_consume(rg)), o.vec_znx_idft_apply_consume(ro)
    assert np.array_equal(got, want)
    assert all(O.i128_to_int(want[j, 0, 0]) == 1 for j in range(size))


@pytest.mark.parametrize("limbs", [16, 17, 32])
def test_cnv_apply_dft_extreme_residues(limbs):
    """cnv_apply_dft reduces once per 16 products: with -delta_0 in every limb of both operands the middle output limbs sum `limbs`
    products (q - 1)^2."""
    n = 128
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    a = _minus_delta((limbs, 1, n))
    apg, bpg = g.cnv_pvec_alloc(1, limbs), g.cnv_pvec_alloc(1, limbs)
    g.cnv_prepare_left(apg, g.vec_znx_from_numpy(a), -1)
    g.cnv_prepare_right(bpg, g.vec_znx_from_numpy(a), -1)
    assert _all_q_minus_1(g.vec_znx_dft_to_numpy(apg)) and _all_q_minus_1(g.vec_znx_dft_to_numpy(bpg))
    apo = o.vec_znx_dft_alloc(1, limbs)
    o.cnv_prepare(apo, a, -1)
    res_size = 2 * limbs - 1
    rg, ro = g.vec_znx_dft_alloc(1, res_size), o.vec_znx_dft_alloc(1, res_size)
    g.cnv_apply_dft(0, rg, 0, apg, 0, bpg, 0)
    o.cnv_apply_dft(0, ro, 0, apo, 0, apo, 0)
    got, want = g.vec_znx_big_to_numpy(g.vec_znx_idft_apply_consume(rg)), o.vec_znx_idft_apply_consume(ro)
    assert np.array_equal(got, want)
    assert O.i128_to_int(want[limbs - 1, 0, 0]) == limbs  # the longest sum: `limbs` products of (-1)(-1)


def _adds_for(A, T, k):
    """Even integers x_j such that normalising A + x (base 2^k, limb 0 most significant, carry out of limb 0 dropped) gives the digits
    T; T[-1] is None (free: every acc_add lies in the ideal (X - 1), whose constant terms at X = 1 are even, so the last limb's parity
    cannot be chosen).  Top-down: limb j must receive a carry of the parity that makes x_j even."""
    L = len(A)
    x, cout = [0] * L, 0
    for j in range(L - 1):
        t = T[j] + (cout << k)
        cin = (T[j] - A[j]) & 1
        x[j] = t - A[j] - cin
        cout = cin
    out = A[-1] & 1
    x[-1] = out + (cout << k) - A[-1]
    assert all(v % 2 == 0 for v in x)
    return x


def _normalise_digits(vals, k):
    """balanced base-2^k carry chain of a column of integers (limb 0 most significant), carry out of limb 0 dropped"""
    out, cy = [0] * len(vals), 0
    for j in range(len(vals) - 1, -1, -1):
        t = vals[j] + cy
        d = t & ((1 << k) - 1)
        if d >= 1 << (k - 1):
            d -= 1 << k
        out[j], cy = d, (t - d) >> k
    return out


def _extreme_rotation(n, rank, dnum, brk_size, block, n_lwe, k, seed):
    """Keys whose first block turns the accumulator X^0 LUT (LUT = -delta_0 in limb 0) into -delta_0 in every row (limbs < dnum, every
    column): one key with a_0 = n ((X^n - 1) = -2) carries x_c / 2 delta_0 in the row of LUT limb 0, the other keys of the block have
    a_t = 0.  Every later key is -delta_0 in every poly.  -> (mats, lut, lwe)"""
    cols = rank + 1
    mats = _minus_delta((n_lwe, dnum, cols, brk_size, cols, n))
    T = [-1] * (brk_size - 1) + [None]
    for col in range(cols):
        A = [-1 if (col == 0 and j == 0) else 0 for j in range(brk_size)]
        x = _adds_for(A, T, k)
        assert _normalise_digits([a + v for a, v in zip(A, x)], k)[:brk_size - 1] == T[:-1]
        for j in range(brk_size):
            mats[0, 0, 0, j, col, :] = 0
            mats[0, 0, 0, j, col, 0] = x[j] // 2
    lut = np.zeros((brk_size, 1, n), dtype=np.int64)
    lut[0, 0, 0] = -1
    rng = np.random.default_rng(seed)
    lwe = rng.integers(-n, n, size=(3, n_lwe + 1), dtype=np.int64)
    lwe[:, 0] = 0
    lwe[:, 1] = n
    lwe[:, 2:block + 1] = 0
    return mats, lut, lwe


def _assert_rows_minus_delta(acc, dnum):
    """acc: (batch, size, cols, n) after the first block: limbs < dnum of every column are exactly -delta_0"""
    want = _minus_delta(acc[:, :dnum].shape)
    assert np.array_equal(acc[:, :dnum], want)


def test_cggi_block_kernel_extreme_residues():
    """cggi_block_ntt120_kernel at R = 16 rows (rank 3, dnum 4) and block 8: the second block sums 16 products (q - 1)^2 per frequency,
    0.9995 * 2^64 for Q[0], and 8 lazily reduced (X^a - 1) updates."""
    n, rank, dnum, brk_size, block, k = 512, 3, 4, 5, 8, 18
    mats, lut, lwe = _extreme_rotation(n, rank, dnum, brk_size, block, 2 * block, k, 8600)
    rot = _Rot(n, mats, pin=False)
    first, _ = rot.run(lwe, lut, block, k, brk_size, n_lwe=block)
    assert np.array_equal(first, rot.oracle(lwe, lut, block, k, brk_size, n_lwe=block))
    _assert_rows_minus_delta(first, dnum)
    got, _ = rot.run(lwe, lut, block, k, brk_size)
    assert np.array_equal(got, rot.oracle(lwe, lut, block, k, brk_size))


def test_two_primes_extreme_residues():
    """The two-prime kernel at R = 4 rows, block 4: after the first block every row is -delta_0, then -delta_0 keys: RT = 4 products
    (q - 1)^2 per row sum, every block on the two-prime route."""
    n, rank, dnum, brk_size, block, k = 512, 1, 2, 3, 4, 18
    mats, lut, lwe = _extreme_rotation(n, rank, dnum, brk_size, block, 12 * block, k, 8700)
    rot = _Rot(n, mats, pin=True)
    first, _ = rot.run(lwe, lut, block, k, brk_size, n_lwe=block)
    assert np.array_equal(first, rot.oracle(lwe, lut, block, k, brk_size, n_lwe=block))
    _assert_rows_minus_delta(first, dnum)
    rot.check(lwe, lut, block, k, brk_size, two_primes=True)


# ---------------------------------------------------------------------------------------------------------------------------------------
# C. full-width integers in the NTT120 big domain
# ---------------------------------------------------------------------------------------------------------------------------------------
def _wide_ints(rng, count, k):
    """Python ints over the whole centred range |v| <= (Q - 1) / 2, with the endpoints, +-2^64 +- 1, and low k bits 0 or -2^(k-1)"""
    special = [HALF_Q, -HALF_Q, HALF_Q - 1, -(HALF_Q - 1), (1 << 64) + 1, (1 << 64) - 1, -(1 << 64) + 1, -(1 << 64) - 1, 0, 1, -1,
               (1 << 63), -(1 << 63) - 1]
    vals = list(special)
    while len(vals) < count:
        v = int(rng.integers(0, 1 << 62)) << 58 | int(rng.integers(0, 1 << 58))
        v = v % (2 * HALF_Q + 1) - HALF_Q
        r = len(vals) % 3
        if r == 1:
            v = (v >> k) << k                      # low k bits 0
        elif r == 2:
            v = ((v >> k) << k) - (1 << (k - 1))   # low k bits -2^(k-1)
        vals.append(max(-HALF_Q, min(HALF_Q, v)))
    return vals[:count]


@pytest.mark.parametrize("a_k,res_k", [(12, 17), (17, 12), (18, 19), (19, 18), (52, 50), (50, 52), (7, 51), (18, 18), (50, 50)])
def test_big_normalize_full_width(a_k, res_k):
    """vec_znx_big_normalize (and its +-assign forms) on i128 values over the whole centred range, res_offset grid of
    test_vec_znx_big_normalize_cross_base2k; same-base2k, offset-0 cases also against a Python-int normalisation."""
    n = 64
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(a_k * 100 + res_k + 7)
    for a_size in (1, 2, 4):
        vals = np.array(_wide_ints(rng, a_size * n, a_k), dtype=object).reshape(a_size, 1, n)
        big_o = O.int_to_i128(vals)
        big_g = g.vec_znx_big_alloc(1, a_size)
        big_g.buf.upload(big_o)
        for res_size in (1, 3, 5):
            for res_offset in (-(a_k + 1), -a_k, -3, 0, 2, a_k - 1, a_k, a_k + 1, 2 * a_k + 3):
                init = fill_uniform(rng, (res_size, 1, n), res_k)
                for op in (0, 1, -1):
                    out_g, out_o = g.vec_znx_from_numpy(init), init.copy()
                    g.vec_znx_big_normalize(out_g, res_k, res_offset, 0, big_g, a_k, 0, op=op)
                    o.vec_znx_big_normalize(out_o, res_k, res_offset, 0, big_o, a_k, 0, op=op)
                    got = g.vec_znx_to_numpy(out_g)
                    assert np.array_equal(got, out_o), (a_size, res_size, res_offset, op)
                    if op == 0 and res_offset == 0 and a_k == res_k and res_size >= a_size:
                        w = [sum(int(vals[j, 0, i]) << (a_k * (res_size - 1 - j)) for j in range(a_size)) for i in range(n)]
                        assert np.array_equal(got[:, 0, :], np.array(digits_of_torus_int(w, a_k, res_size), dtype=np.int64))


_N_ALL = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536]


@pytest.mark.parametrize("n", _N_ALL)
def test_idft_crt_at_the_endpoints(n):
    """Integer coefficients up to +-(Q - 1) / 2, reduced mod q_k and transformed by the oracle, uploaded in the [k][n] layout:
    idft_apply, _tmpa and _consume return exactly those integers."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(n + 31)
    vals = _wide_ints(rng, n, 20)
    d = np.array([[v % q for q in O.Q] for v in vals], dtype=np.uint64)
    O.lib().orc_ntt120_ntt(o._h, O._p(d))
    planes = np.stack([(d[:, k] % np.uint64(q)).astype(np.uint32) for k, q in enumerate(O.Q)])
    dg = g.vec_znx_dft_from_bytes(1, 1, planes)
    want = np.array(vals, dtype=object)
    for how in ("apply", "tmpa", "consume"):
        if how == "consume":
            big = g.vec_znx_idft_apply_consume(dg)
        else:
            big = g.vec_znx_big_alloc(1, 1)
            (g.vec_znx_idft_apply if how == "apply" else g.vec_znx_idft_apply_tmpa)(big, 0, dg, 0)
        got = O.i128_to_int(g.vec_znx_big_to_numpy(big)[0, 0])
        assert np.array_equal(got, want), how


@pytest.mark.parametrize("n", _N_ALL)
def test_forward_full_i64_range_all_sizes(n):
    """test_ntt120_full_i64_range's inputs (i64 min / max, -1, 0, uniform 64-bit) at every ring degree."""
    g, o = pb.Module(n, pb.NTT120), O.OracleModule(n, pb.NTT120)
    rng = np.random.default_rng(n + 3)
    a = fill_uniform(rng, (2, 1, n), 64)
    a[0, 0, :4] = [np.iinfo(np.int64).min, np.iinfo(np.int64).max, -1, 0]
    a[1, 0, -4:] = [np.iinfo(np.int64).max, np.iinfo(np.int64).min, 0, -1]
    dg, do = g.vec_znx_dft_alloc(1, 2), o.vec_znx_dft_alloc(1, 2)
    g.vec_znx_dft_apply(1, 0, dg, 0, g.vec_znx_from_numpy(a), 0)
    o.vec_znx_dft_apply(1, 0, do, 0, a, 0)
    got = g.vec_znx_dft_to_numpy(dg)
    for k, q in enumerate(O.Q):
        assert np.array_equal(got[:, :, k, :].astype(np.uint64), do[:, :, :, k] % np.uint64(q)), k
    bg, bo = g.vec_znx_big_alloc(1, 2), o.vec_znx_big_alloc(1, 2)
    g.vec_znx_idft_apply(bg, 0, dg, 0)
    o.vec_znx_idft_apply(bo, 0, do, 0)
    assert np.array_equal(g.vec_znx_big_to_numpy(bg), bo)
    assert np.array_equal(O.i128_to_int(bo[:, 0]), a[:, 0].astype(object))
