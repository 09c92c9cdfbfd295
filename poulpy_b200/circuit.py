"""Circuit bootstrapping, constant mode (SURVEY 8f N4): host orchestration of
`circuit_bootstrap_core(to_exponent = false, ...)` (poulpy-bin-fhe/src/circuit_bootstrapping/circuit.rs:219-380) over the device-resident
entry points of the C ABI:

    LUT f[j * alpha + i] = j * 2^(res_base2k * (dnum - 1 - i))            circuit.rs:278-299, lut.rs:271-338 (lookup_table_set)
    acc  = blind_rotate(lwe, LUT)                                           pgb_cggi_mod_switch_2n_batched + pgb_cggi_blind_rotate_batched
    for i in 0..dnum:  GGSW.at(i, 0) = trace(acc);  acc *= X^{-gap}         pgb_glwe_trace_assign_batched, pgb_vec_znx_rotate_batched
    GGSW columns 1..rank = ggsw_expand_row(GGSW, tsk)                       pgb_ggsw_expand_row_batched

Everything stays on the device; the host only sequences the launches, as `poulpy-bin-fhe` does above `Module<B>`.  All layouts share one
base2k here (the reference converts between the BRK / ATK / result layouts with glwe_normalize when they differ); extension_factor > 1 goes
through the extended blind rotation (`pgb_cggi_blind_rotate_extended_batched`) and the `ext`-component lookup table.

The exponent mode (`to_exponent = true`: circuit.rs:286-290, 352-366 and `post_process` :382-420 with `glwe_pack`,
poulpy-core/src/glwe_packing.rs:15-170) is written once over a small GLWE-operations interface (`DeviceGlweOps` below): the sequencing is
data independent, so the same functions drive a batch of ciphertexts per operand on the device.
"""
import ctypes as C

import numpy as np

from . import hal


def lookup_table_limbs(n, f, k, base2k, ext=1):
    """The un-normalised LookupTable.data of lut.rs:271-327 as a numpy array (ext, limbs, 1, n): the table over the domain n * ext with
    f[i] * scale on blocks of `step` coefficients in its last limb, component j = coefficients j, j + ext, ... (vec_znx_switch_ring after j
    rotations by X^-1).  -> (array, step)"""
    f = [int(x) for x in f]
    domain = n * ext
    assert 0 < len(f) <= domain
    limbs = -(-k // base2k)
    scale = 1 << (base2k - k % base2k) if k % base2k else 1
    step = (domain + len(f) // 2) // len(f)  # usize::div_round (lut.rs:243-247)
    last = np.zeros(domain, dtype=np.int64)
    for i, fi in enumerate(f):
        last[i * step:(i + 1) * step] = fi * scale
    out = np.zeros((ext, limbs, 1, n), dtype=np.int64)
    for j in range(ext):
        out[j, limbs - 1, 0] = last[j::ext]
    return out, step


def lookup_table_rotation_plan(n, ext, k):
    """lookup_table_rotate(k) (lut.rs:340-362): component i is rotated by k_hi (+1 for the last k_lo components) and moves to slot
    (i + k_lo) mod ext.  -> list of (source component, rotation, destination slot)"""
    two_n_ext = 2 * n * ext
    k_pos = (k + two_n_ext) % two_n_ext
    k_hi, k_lo = k_pos // ext, k_pos % ext
    return [(i, k_hi + (1 if i >= ext - k_lo else 0), (i + k_lo) % ext) for i in range(ext)]


def lookup_table_set(module: "hal.Module", f, k, base2k, ext=1):
    """LookupTable::set (lut.rs:271-338) -> (VecZnx(1 col, ceil(k / base2k) limbs) with `ext` batch items on the device, drift)."""
    n = module.n
    raw, step = lookup_table_limbs(n, f, k, base2k, ext)
    lut = module.vec_znx_from_numpy(raw if ext > 1 else raw[0])
    r = lut.struct()
    bt = hal._BT(ext, lut.batch_stride, 0, 0)
    hal._check(hal.lib().pgb_vec_znx_normalize_assign_batched(module._h, C.c_uint64(base2k), C.byref(r), C.c_uint64(0), C.byref(bt)))
    drift = step >> 1
    out = module.vec_znx_alloc(1, raw.shape[1], ext)
    item = n * raw.shape[1] * 8
    for src, rot, dst in lookup_table_rotation_plan(n, ext, -drift):  # res.rotate(-drift) (lut.rs:333)
        o = hal._VZ(out.buf.ptr + dst * item, n, 1, raw.shape[1], raw.shape[1])
        a = hal._VZ(lut.buf.ptr + src * item, n, 1, raw.shape[1], raw.shape[1])
        hal._check(hal.lib().pgb_vec_znx_rotate(module._h, C.c_int64(rot), C.byref(o), C.c_uint64(0), C.byref(a), C.c_uint64(0)))
    return out, drift


def _glwe_copy(module, dst_ptr, dst_stride, dst_size, src_ptr, src_stride, src_size, cols, batch):
    """glwe_copy (vec_znx_copy per column): the first min(size) limbs, the rest of dst zeroed; limb-major containers, so that is one
    contiguous run per ciphertext."""
    n, lib = module.n, hal.lib()
    width = min(dst_size, src_size) * cols * n * 8
    hal._check(lib.pgb_memcpy_d2d_strided(module._h, C.c_void_p(dst_ptr), C.c_uint64(dst_stride), C.c_void_p(src_ptr), C.c_uint64(src_stride),
                                          C.c_uint64(width), C.c_uint64(batch)))
    if dst_size > src_size:
        module.sync()
        for b in range(batch):
            hal._check(lib.pgb_memset(C.c_void_p(dst_ptr + b * dst_stride + width), 0, C.c_size_t((dst_size - src_size) * cols * n * 8)))


def _blind_rotate(module, acc, lwe_dev, batch, n_lwe, lwe_size, lwe_base2k, lut, ext, brk, x_pow_a, block_size, base2k, rot_left):
    """BlindRotationExecute (cggi/algorithm.rs:88-117): mod switch to 2 * n * ext, then the plain or the extended block-binary rotation."""
    lwe_2n = module.cggi_mod_switch_2n(lwe_dev, batch, n_lwe, lwe_size, lwe_base2k, 2 * module.n * ext, rot_left=rot_left)
    if ext == 1:
        module.cggi_blind_rotate(acc, lwe_2n, n_lwe, lut, brk, x_pow_a, block_size, base2k)
    else:
        module.cggi_blind_rotate_extended(acc, lwe_2n, n_lwe, lut, ext, brk, x_pow_a, block_size, base2k)


def circuit_bootstrap_to_constant(module: "hal.Module", lwe_dev: "hal.DevBuf", batch, n_lwe, lwe_size, lwe_base2k, brk: "hal.VmpPMat",
                                  x_pow_a, block_size, atk, tsk, base2k, rank, dnum_res, res_size, log_domain, dsize_atk=1, dsize_tsk=1,
                                  extension_factor=1):
    """-> DevBuf holding `batch` GGSW MatZnx(dnum_res, rank+1, rank+1, res_size) (base2k digits).
    lwe_dev: (batch, lwe_size, 1, n_lwe + 1) int64; brk: the n_lwe prepared GGSWs stored consecutively (VmpPMat of the first);
    atk: log_n prepared automorphism keys, atk[i] for Module.trace_galois_element(i); tsk: rank prepared tensor keys."""
    n, cols = module.n, rank + 1
    assert res_size * 0 == 0 and base2k * (dnum_res - 1) < 64 and log_domain + base2k * max(dnum_res - 1, 0) < 64  # circuit.rs:266-276
    alpha = 1 << (dnum_res - 1).bit_length() if dnum_res > 1 else 1
    f = [0] * ((1 << log_domain) * alpha)
    for j in range(1 << log_domain):
        for i in range(dnum_res):
            f[j * alpha + i] = j * (1 << (base2k * (dnum_res - 1 - i)))
    ext = extension_factor
    lut, drift = lookup_table_set(module, f, base2k * dnum_res, base2k, ext)
    # blind rotation over the BRK layout (k = brk.max_k: brk.size limbs)
    acc_size = brk.size
    acc = module.vec_znx_alloc(cols, acc_size, batch)
    _blind_rotate(module, acc, lwe_dev, batch, n_lwe, lwe_size, lwe_base2k, lut, ext, brk, x_pow_a, block_size, base2k, True)
    gap = 2 * drift // ext  # circuit.rs:336
    assert gap > 0
    ggsw_stride = n * dnum_res * cols * cols * res_size * 8
    ggsw = hal.DevBuf(batch * ggsw_stride, device=module.device)
    tmp_size = max(acc_size, res_size)
    tmp = module.vec_znx_alloc(cols, tmp_size, batch)
    acc2 = module.vec_znx_alloc(cols, acc_size, batch)
    scratch = None
    for i in range(dnum_res):
        # glwe_trace(res.at(i, 0), 0, acc, atk) (glwe_trace.rs:91-127): copy, trace in place, copy out
        _glwe_copy(module, tmp.buf.ptr, tmp.batch_stride, tmp_size, acc.buf.ptr, acc.batch_stride, acc_size, cols, batch)
        scratch = module.glwe_trace_assign(tmp, base2k, 0, atk, base2k, dsize_atk, scratch)
        row_ptr = ggsw.ptr + (i * cols + 0) * (n * cols * res_size * 8)
        _glwe_copy(module, row_ptr, ggsw_stride, res_size, tmp.buf.ptr, tmp.batch_stride, tmp_size, cols, batch)
        if i + 1 < dnum_res:  # glwe_rotate_assign(-gap)
            r, a = acc2.struct(), acc.struct()
            bt = hal._BT(batch, acc2.batch_stride, acc.batch_stride, 0)
            for c in range(cols):
                hal._check(hal.lib().pgb_vec_znx_rotate_batched(module._h, C.c_int64(-gap), C.byref(r), C.c_uint64(c), C.byref(a), C.c_uint64(c),
                                                                C.byref(bt)))
            acc, acc2 = acc2, acc
    module.ggsw_expand_row(ggsw, batch, dnum_res, rank, res_size, base2k, tsk, base2k, dsize_tsk)
    module.sync()
    return ggsw


def prepare_ggsw(module: "hal.Module", ggsw_buf: "hal.DevBuf", batch, dnum, rank, size) -> "hal.VmpPMat":
    """GGSW::prepare of a circuit-bootstrapping output (`batch` consecutive MatZnx(dnum, rank+1, rank+1, size), as returned by
    circuit_bootstrap_to_constant / _to_exponent) -> a batched VmpPMat, one prepared GGSW per item, in one launch; it drives
    Module.glwe_cmux with one selector per ciphertext.  Asynchronous: the module's stream orders it before the next call."""
    cols = rank + 1
    mat = hal.MatZnx(ggsw_buf, module.n, dnum, cols, cols, size, batch=batch, batch_stride=module.n * dnum * cols * cols * size * 8)
    pmat = module.vmp_pmat_alloc(dnum, cols, cols, size, batch=batch)
    module.vmp_prepare_batched(pmat, mat)
    return pmat


# ---- glwe_pack / post_process / exponent mode -----------------------------------------------------------------------------------
class DeviceGlweOps:
    """The GLWE operations `pack_internal` and `post_process` are made of, on batches of device-resident GLWEs (VecZnx with a batch axis)
    of one layout (cols = rank + 1 columns, `size` limbs, one base2k); atk[i] is the prepared automorphism key of
    Module.trace_galois_element(i)."""

    def __init__(self, module, atk, base2k, cols, size, batch, dsize=1):
        self.m, self.atk, self.k, self.cols, self.size, self.batch, self.dsize = module, atk, base2k, cols, size, batch, dsize
        self.log_n = module.n.bit_length() - 1
        self.scratch = None

    def new(self):
        return self.m.vec_znx_alloc(self.cols, self.size, self.batch)

    def _bt(self, res, a=None):
        return hal._BT(self.batch, res.batch_stride, a.batch_stride if a is not None else 0, 0)

    def copy(self, dst, src):
        _glwe_copy(self.m, dst.buf.ptr, dst.batch_stride, dst.size, src.buf.ptr, src.batch_stride, src.size, self.cols, self.batch)

    def rotate(self, k, dst, src):  # glwe_rotate (operations/glwe.rs:982-1003)
        r, a = dst.struct(), src.struct()
        bt = self._bt(dst, src)
        for c in range(self.cols):
            hal._check(hal.lib().pgb_vec_znx_rotate_batched(self.m._h, C.c_int64(k), C.byref(r), C.c_uint64(c), C.byref(a), C.c_uint64(c), C.byref(bt)))

    def rotate_assign(self, k, ct):  # glwe_rotate_assign: through a temporary, then the buffers are swapped
        tmp = self.new()
        self.rotate(k, tmp, ct)
        ct.buf, tmp.buf = tmp.buf, ct.buf

    def _assign(self, fn, res, a):
        r, av = res.struct(), a.struct()
        bt = self._bt(res, a)
        for c in range(self.cols):
            hal._check(fn(self.m._h, C.byref(r), C.c_uint64(c), C.byref(av), C.c_uint64(c), C.byref(bt)))

    def add_assign(self, res, a):
        self._assign(hal.lib().pgb_vec_znx_add_assign_batched, res, a)

    def sub_assign(self, res, a):
        self._assign(hal.lib().pgb_vec_znx_sub_assign_batched, res, a)

    def sub(self, res, a, b):  # glwe_sub: res = a - b
        self.copy(res, a)
        self.sub_assign(res, b)

    def rsh1(self, ct):  # glwe_rsh(1)
        r = ct.struct()
        bt = self._bt(ct)
        for c in range(self.cols):
            hal._check(hal.lib().pgb_vec_znx_rsh_assign_batched(self.m._h, C.c_uint64(self.k), C.c_uint64(1), C.byref(r), C.c_uint64(c), C.byref(bt)))

    def normalize_assign(self, ct):
        r = ct.struct()
        bt = self._bt(ct)
        for c in range(self.cols):
            hal._check(hal.lib().pgb_vec_znx_normalize_assign_batched(self.m._h, C.c_uint64(self.k), C.byref(r), C.c_uint64(c), C.byref(bt)))

    def automorphism_assign(self, ct, i):  # glwe_automorphism_assign: key-switch with atk[i], then X -> X^p
        tmp = self.new()
        self.m.glwe_automorphism(tmp, self.k, ct, self.k, self.atk[i], self.k, self.m.trace_galois_element(i), self.dsize)
        ct.buf, tmp.buf = tmp.buf, ct.buf

    def automorphism_add_assign(self, ct, i):
        self.scratch = self.m.glwe_automorphism_op(0, ct, self.k, ct, self.atk[i], self.k, self.m.trace_galois_element(i), self.dsize, self.scratch)

    def automorphism_sub_negate(self, res, a, i):
        self.scratch = self.m.glwe_automorphism_op(2, res, self.k, a, self.atk[i], self.k, self.m.trace_galois_element(i), self.dsize, self.scratch)

    def trace(self, res, skip, a):  # glwe_trace (glwe_trace.rs:91-127), same layout on both sides
        self.copy(res, a)
        self.scratch = self.m.glwe_trace_assign(res, self.k, skip, self.atk, self.k, self.dsize, self.scratch)


def pack_internal(ops, a, b, i):
    """glwe_packing.rs:15-96: a <- a + b X^t + phi(a - b X^t) with t = 2^(log_n - i - 1) (in place in a, or in b when a is absent)."""
    if a is not None:
        t = 1 << (ops.log_n - i - 1)
        if b is not None:
            tmp_b = ops.new()
            ops.rotate_assign(-t, a)
            ops.sub(tmp_b, a, b)
            ops.rsh1(tmp_b)
            ops.add_assign(a, b)
            ops.rsh1(a)
            ops.normalize_assign(tmp_b)
            ops.automorphism_assign(tmp_b, i)
            ops.sub_assign(a, tmp_b)
            ops.normalize_assign(a)
            ops.rotate_assign(t, a)
        else:
            ops.rsh1(a)
            ops.automorphism_add_assign(a, i)
    elif b is not None:
        t = 1 << (ops.log_n - i - 1)
        tmp_b = ops.new()
        ops.rotate(t, tmp_b, b)
        ops.rsh1(tmp_b)
        ops.automorphism_sub_negate(b, tmp_b, i)


def glwe_pack(ops, res, cts, log_gap_out):
    """glwe_packing.rs:122-170: cts maps a coefficient index to a GLWE (consumed)."""
    cts = dict(cts)
    assert max(cts) < (1 << ops.log_n)
    for i in range(ops.log_n - log_gap_out):
        t = min(1 << ops.log_n, 1 << (ops.log_n - 1 - i))
        for j in range(t):
            lo, hi = cts.pop(j, None), cts.pop(j + t, None)
            pack_internal(ops, lo, hi, i)
            if lo is not None:
                cts[j] = lo
            elif hi is not None:
                cts[j] = hi
    ops.trace(res, ops.log_n - log_gap_out, cts[0])


def post_process(ops, res, a, log_gap_in, log_gap_out, log_domain):
    """circuit.rs:382-420: isolate the coefficients that are multiples of the input gap and repack them at the output gap."""
    if log_gap_in != log_gap_out:
        a_trace = ops.new()
        ops.trace(a_trace, ops.log_n - log_gap_in + 1, a)
        cts = {}
        for i in range(1 << log_domain):
            if i != 0:
                ops.rotate_assign(-(1 << log_gap_in), a_trace)
            ct = ops.new()
            ops.copy(ct, a_trace)
            cts[i * (1 << log_gap_out)] = ct
        glwe_pack(ops, res, cts, log_gap_out)
    else:
        ops.trace(res, ops.log_n - log_gap_in + 1, a)


def exponent_lut(base2k, dnum_res, log_domain):
    """circuit.rs:278-290: f[i] = 2^(base2k * (dnum - 1 - i)) for i < dnum, zero up to 2^log_domain * alpha entries."""
    alpha = 1 << (dnum_res - 1).bit_length() if dnum_res > 1 else 1
    f = [0] * ((1 << log_domain) * alpha)
    for i in range(dnum_res):
        f[i] = 1 << (base2k * (dnum_res - 1 - i))
    return f, alpha


def circuit_bootstrap_to_exponent(module: "hal.Module", log_gap_out, lwe_dev: "hal.DevBuf", batch, n_lwe, lwe_size, lwe_base2k, brk: "hal.VmpPMat",
                                  x_pow_a, block_size, atk, tsk, base2k, rank, dnum_res, size, log_domain, dsize_atk=1, dsize_tsk=1,
                                  extension_factor=1):
    """circuit_bootstrap_core(to_exponent = true) (circuit.rs:219-380): -> DevBuf of `batch` GGSW MatZnx(dnum_res, rank+1, rank+1, size).
    One GLWE layout throughout (`size` limbs = the limbs of the blind-rotation key)."""
    n, cols = module.n, rank + 1
    assert brk.size == size
    f, alpha = exponent_lut(base2k, dnum_res, log_domain)
    ext = extension_factor
    lut, drift = lookup_table_set(module, f, base2k * dnum_res, base2k, ext)
    ops = DeviceGlweOps(module, atk, base2k, cols, size, batch, dsize_atk)
    acc = ops.new()
    _blind_rotate(module, acc, lwe_dev, batch, n_lwe, lwe_size, lwe_base2k, lut, ext, brk, x_pow_a, block_size, base2k, False)  # direction Right (:305-307)
    gap = 2 * drift // ext
    assert gap > 0
    log_gap_in = (gap * alpha - 1).bit_length()
    ggsw_stride = n * dnum_res * cols * cols * size * 8
    ggsw = hal.DevBuf(batch * ggsw_stride, device=module.device)
    row = ops.new()
    for i in range(dnum_res):
        post_process(ops, row, acc, log_gap_in, log_gap_out, log_domain)
        _glwe_copy(module, ggsw.ptr + (i * cols) * (n * cols * size * 8), ggsw_stride, size, row.buf.ptr, row.batch_stride, size, cols, batch)
        if i + 1 < dnum_res:
            ops.rotate_assign(-gap, acc)
    module.sync()
    module.ggsw_expand_row(ggsw, batch, dnum_res, rank, size, base2k, tsk, base2k, dsize_tsk)
    module.sync()
    return ggsw
