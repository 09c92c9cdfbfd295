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


# ---- lookup-table read by vertical packing ----------------------------------------------------------------------------------------
def lut_split(n, lut, n_bits):
    """The vertical-packing leaves of a table of T <= 2^n_bits entries as host polynomials: with nu = min(n_bits, log2 n), polynomial p
    holds entries p 2^nu .. p 2^nu + 2^nu - 1 in its first coefficients (missing entries are 0).  lut is (size, T): limb j of entry t,
    most significant limb first (a 1-d lut is one limb).  -> (nu, array (2^(n_bits - nu), size, n))"""
    lut = np.atleast_2d(np.asarray(lut, dtype=np.int64))
    size, T = lut.shape
    assert n & (n - 1) == 0 and 1 <= n_bits <= 64 and T <= 1 << n_bits, (n, n_bits, T)
    nu = min(n_bits, n.bit_length() - 1)
    full = np.zeros((size, 1 << n_bits), dtype=np.int64)
    full[:, :T] = lut
    polys = np.zeros((1 << (n_bits - nu), size, n), dtype=np.int64)
    polys[:, :, :1 << nu] = full.reshape(size, 1 << (n_bits - nu), 1 << nu).transpose(1, 0, 2)
    return nu, polys


def lut_read(module: "hal.Module", lut, sel: "hal.VmpPMat", batch, n_bits, base2k, ggsw_base2k=None, dsize=1, ggsw_stride=None,
             bit_stride=None, scratch: "hal.DevBuf" = None) -> "hal.DevBuf":
    """LWE encryptions of LUT[m_b] for `batch` encrypted integers m_b = sum_i bit_{b,i} 2^i (n_bits GGSW bits each, rank 1), by vertical
    packing: the table (see lut_split) becomes 2^(n_bits - nu) trivial GLWEs (the polynomial in the body column, the mask zero); a CMux
    tree (Module.glwe_cmux_tree) selects polynomial m_b >> nu with bits [nu, n_bits), a blind rotation (Module.glwe_blind_rotate_ggsw,
    step -1) by bits [0, nu) brings entry m_b to coefficient 0, and lwe_sample_extract extracts it.  Selecting first leaves one polynomial
    per item to rotate.  Selector (b, i) is at sel + b ggsw_stride + i bit_stride, with the defaults of glwe_blind_rotate_ggsw (the
    bit-major output of prepare_ggsw).  -> the LWE batch, int64 (batch, size, 1, n + 1) on the device, size = the table's limbs.
    Asynchronous."""
    n = module.n
    cols = sel.cols_in
    assert cols == 2, "lwe_sample_extract reads rank-1 GLWEs"
    ggsw_base2k = base2k if ggsw_base2k is None else ggsw_base2k
    if bit_stride is None and ggsw_stride is None:
        assert sel.batch >= n_bits * batch, (sel.batch, n_bits, batch)
    bit_stride = sel.batch_stride if bit_stride is None else bit_stride
    ggsw_stride = n_bits * sel.batch_stride if ggsw_stride is None else ggsw_stride
    nu, polys = lut_split(n, lut, n_bits)
    size = polys.shape[1]
    leaves = np.zeros((polys.shape[0], size, cols, n), dtype=np.int64)
    leaves[:, :, 0] = polys
    table = module.vec_znx_from_numpy(leaves)
    table = hal.VecZnx(table.buf, n, cols, size)  # one table of 2^(n_bits - nu) entries, shared by the batch
    if n_bits > nu:
        hi = hal.VmpPMat(sel.buf, n, sel.rows, cols, cols, sel.size, offset=sel.offset + nu * bit_stride, batch=sel.batch,
                         batch_stride=sel.batch_stride)
        picked = module.vec_znx_alloc(cols, size, batch)
        scratch = module.glwe_cmux_tree(picked, table, base2k, n_bits - nu, hi, ggsw_base2k, dsize, ggsw_stride=ggsw_stride,
                                        bit_stride=bit_stride, scratch=scratch)
    else:
        picked = table
    rot = module.vec_znx_alloc(cols, size, batch)
    module.glwe_blind_rotate_ggsw(rot, picked, base2k, -1, nu, sel, ggsw_base2k, dsize, ggsw_stride=ggsw_stride, bit_stride=bit_stride,
                                  scratch=scratch)
    out = hal.DevBuf(batch * size * (n + 1) * 8, device=module.device)
    module.lwe_sample_extract(out, n, size, rot)
    return out


# ---- binary decision diagrams ------------------------------------------------------------------------------------------------------
class BddCircuit:
    """A levelled CMux circuit (the pgb_bdd_circuit of Module.glwe_bdd_eval).  `leaves` are the leaf values (state j < len(leaves) is leaf
    j); `levels` is a list of (bit, [(t, f), ...]): node k, counted in level order, is state len(leaves) + k and selects t when the bit is
    1, f when it is 0; every child must be a leaf or a node of an earlier level.  `outputs` are state indices."""

    def __init__(self, leaves, levels, outputs):
        self.leaves = list(leaves)
        self.levels = [(int(bit), [(int(t), int(f)) for t, f in nodes]) for bit, nodes in levels]
        self.outputs = [int(o) for o in outputs]

    @property
    def n_nodes(self):
        return sum(len(nodes) for _, nodes in self.levels)

    def struct(self):
        """-> (hal._BDD, the arrays it points into: keep them alive while the struct is in use)"""
        u32 = lambda xs: np.ascontiguousarray(np.asarray(xs, dtype=np.uint32).reshape(-1))  # noqa: E731
        bits = u32([b for b, _ in self.levels])
        counts = u32([len(nodes) for _, nodes in self.levels])
        t = u32([t for _, nodes in self.levels for t, _ in nodes])
        f = u32([f for _, nodes in self.levels for _, f in nodes])
        out = u32(self.outputs)
        p = lambda arr: arr.ctypes.data_as(C.POINTER(C.c_uint32))  # noqa: E731
        cs = hal._BDD(len(self.leaves), len(self.levels), p(bits), p(counts), p(t), p(f), len(self.outputs), p(out))
        return cs, (bits, counts, t, f, out)


def bdd_from_truth_tables(tables, n_bits, order):
    """The shared, reduced, ordered BDD of binary functions given by truth tables (tables[o][x] in {0, 1} for x < 2^n_bits, bit i of x
    the input bit i), with the variable order `order` (a permutation of range(n_bits)): the root tests order[0], level 0 tests order[-1],
    and empty levels are left out.  Nodes are merged through a unique table and a node whose two children are equal is dropped, so
    children may skip levels and outputs share nodes.  Leaves are the values 0 and 1.  -> BddCircuit"""
    assert 1 <= n_bits <= 16 and sorted(order) == list(range(n_bits)), (n_bits, order)
    x = np.arange(1 << n_bits)
    pos = np.zeros(1 << n_bits, dtype=np.int64)  # the index of x with order[0] as its most significant bit
    for d, v in enumerate(order):
        pos |= ((x >> v) & 1) << (n_bits - 1 - d)
    unique, nodes = {}, []  # (depth, t, f) -> node id; nodes[id] = (depth, t, f); ids >= 2, leaves are 0 and 1

    def mk(d, t, f):
        if t == f:
            return t
        key = (d, t, f)
        if key not in unique:
            unique[key] = len(nodes) + 2
            nodes.append(key)
        return unique[key]

    roots = []
    for tab in tables:
        tab = np.asarray(tab, dtype=np.int64)
        assert tab.shape == (1 << n_bits,) and np.all((tab == 0) | (tab == 1))
        cur = np.empty(1 << n_bits, dtype=np.int64)
        cur[pos] = tab
        cur = cur.tolist()
        for d in range(n_bits - 1, -1, -1):  # cur[i]: the cofactor of prefix i of order[:d + 1]; its last bit is order[d]
            cur = [mk(d, cur[2 * i + 1], cur[2 * i]) for i in range(len(cur) // 2)]
        roots.append(cur[0])
    state = {0: 0, 1: 1}
    levels = []
    for d in range(n_bits - 1, -1, -1):
        ids = [i + 2 for i, (dd, _, _) in enumerate(nodes) if dd == d]
        if not ids:
            continue
        first = 2 + sum(len(lv) for _, lv in levels)
        for j, i in enumerate(ids):
            state[i] = first + j
        levels.append((order[d], [(state[nodes[i - 2][1]], state[nodes[i - 2][2]]) for i in ids]))
    return BddCircuit([0, 1], levels, [state[r] for r in roots])


def bdd_leaves(n, circuit, scale, size, cols=2):
    """The leaves of bdd_eval as a host array (n_leaves, size, cols, n): trivial GLWEs whose body is the constant leaves[j] * scale in
    the first limb, the rest zero."""
    leaves = np.zeros((len(circuit.leaves), size, cols, n), dtype=np.int64)
    leaves[:, 0, 0, 0] = np.asarray(circuit.leaves, dtype=np.int64) * scale
    return leaves


def bdd_eval(module: "hal.Module", circuit, sel: "hal.VmpPMat", batch, n_bits, base2k, scale, size=1, ggsw_base2k=None, dsize=1,
             ggsw_stride=None, bit_stride=None, scratch: "hal.DevBuf" = None) -> "hal.DevBuf":
    """LWE encryptions of the outputs of a BDD (BddCircuit) for `batch` items of n_bits GGSW bits each (rank 1): the leaves are the
    trivial GLWEs of bdd_leaves (value * scale, `size` limbs), Module.glwe_bdd_eval evaluates the circuit into `size`-limb GLWEs, and
    lwe_sample_extract extracts coefficient 0 of every output.  Selector (b, i) is at sel + b ggsw_stride + i bit_stride, with the
    defaults of glwe_blind_rotate_ggsw (the bit-major output of prepare_ggsw).  -> the LWEs, int64 (batch, n_out, size, 1, n + 1) on the
    device.  Asynchronous."""
    n, cols = module.n, sel.cols_in
    assert cols == 2, "lwe_sample_extract reads rank-1 GLWEs"
    ggsw_base2k = base2k if ggsw_base2k is None else ggsw_base2k
    leaves = module.vec_znx_from_numpy(bdd_leaves(n, circuit, scale, size, cols))
    leaves = hal.VecZnx(leaves.buf, n, cols, size)  # one set of leaves, shared by the batch
    n_out = len(circuit.outputs)
    res = module.vec_znx_alloc(cols, size, batch * n_out)
    module.glwe_bdd_eval(res, leaves, circuit, base2k, n_bits, sel, ggsw_base2k, dsize, ggsw_stride=ggsw_stride, bit_stride=bit_stride,
                         scratch=scratch)
    out = hal.DevBuf(batch * n_out * size * (n + 1) * 8, device=module.device)
    module.lwe_sample_extract(out, n, size, res)
    return out


def bdd_eval_packed(module: "hal.Module", circuit, sel: "hal.VmpPMat", batch, n_bits, base2k, scale, atk, log_gap_out=0, size=1,
                    ggsw_base2k=None, dsize=1, dsize_atk=1, ggsw_stride=None, bit_stride=None, scratch: "hal.DevBuf" = None) -> "hal.VecZnx":
    """The outputs of a BDD packed into one GLWE per item: the leaves and Module.glwe_bdd_eval of bdd_eval, then Module.glwe_pack with
    output o at coefficient o << log_gap_out (n_out << log_gap_out <= n).  atk: log_n prepared automorphism keys, atk[i] for
    Module.trace_galois_element(i), in base2k.  -> VecZnx of `batch` GLWEs (rank 1, `size` limbs) on the device.  Asynchronous."""
    n, cols = module.n, sel.cols_in
    n_out = len(circuit.outputs)
    assert n_out << log_gap_out <= n, (n_out, log_gap_out, n)
    ggsw_base2k = base2k if ggsw_base2k is None else ggsw_base2k
    leaves = module.vec_znx_from_numpy(bdd_leaves(n, circuit, scale, size, cols))
    leaves = hal.VecZnx(leaves.buf, n, cols, size)
    outs = module.vec_znx_alloc(cols, size, batch * n_out)
    scratch = module.glwe_bdd_eval(outs, leaves, circuit, base2k, n_bits, sel, ggsw_base2k, dsize, ggsw_stride=ggsw_stride,
                                   bit_stride=bit_stride, scratch=scratch)
    g = n * cols * size * 8
    a = hal.VecZnx(outs.buf, n, cols, size, batch=batch, batch_stride=n_out * g)  # item b's output o at b n_out + o
    res = module.vec_znx_alloc(cols, size, batch)
    module.glwe_pack(res, a, [o << log_gap_out for o in range(n_out)], log_gap_out, atk, base2k, dsize_atk, entry_stride=g,
                     scratch=scratch)
    return res


def ggsw_bits_from_packed(module: "hal.Module", packed: "hal.VecZnx", index, ksk: "hal.VmpPMat", n_lwe, lwe_size, brk: "hal.VmpPMat",
                          x_pow_a, block_size, atk, tsk, base2k, rank, dnum_res, res_size, log_domain, packed_base2k=None, ksk_base2k=None,
                          dsize_ksk=1, dsize_atk=1, dsize_tsk=1, extension_factor=1) -> "hal.VmpPMat":
    """Packed GLWEs back to prepared GGSW bits, the inverse of bdd_eval_packed: per item b of `packed` (one GLWE per integer, any rank),
    coefficient index[j] is read as an LWE of dimension n_lwe under the blind-rotation key's secret by Module.glwe_to_lwe_indexed (one
    key-switch per item with ksk = VmpPMat(dnum, rank_packed, 2, .) to that secret's embedding, into lwe_size limbs of base2k), then all
    batch * len(index) LWEs are circuit-bootstrapped (circuit_bootstrap_to_constant, same arguments) and prepared (prepare_ggsw).

    Encoding: circuit bootstrapping reads bit m at m / 2^(log_domain + 1) of the LWE's torus (one padding bit), so coefficient index[j]
    must carry its bit at that scale: a GLWE from bdd_eval_packed must have been made with scale = 2^(base2k - log_domain - 1).

    -> a batched VmpPMat of batch * len(index) GGSWs (dnum_res, rank + 1, rank + 1, res_size), GGSW b * len(index) + j holding bit j of
    item b: the bit-major selector default of glwe_blind_rotate_ggsw, glwe_cmux_tree and glwe_bdd_eval with n_bits = len(index)."""
    index = [int(i) for i in index]
    batch, n_bits = packed.batch, len(index)
    packed_base2k = base2k if packed_base2k is None else packed_base2k
    ksk_base2k = base2k if ksk_base2k is None else ksk_base2k
    lwe = hal.DevBuf(batch * n_bits * lwe_size * (n_lwe + 1) * 8, device=module.device)
    module.glwe_to_lwe_indexed(lwe, n_lwe, lwe_size, base2k, packed, packed_base2k, index, ksk, ksk_base2k, dsize_ksk)
    ggsw = circuit_bootstrap_to_constant(module, lwe, batch * n_bits, n_lwe, lwe_size, base2k, brk, x_pow_a, block_size, atk, tsk, base2k,
                                         rank, dnum_res, res_size, log_domain, dsize_atk, dsize_tsk, extension_factor)
    return prepare_ggsw(module, ggsw, batch * n_bits, dnum_res, rank, res_size)


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
