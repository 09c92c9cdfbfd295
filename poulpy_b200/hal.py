"""Host-side mirror of the reference's `Module<B>` HAL API over the C ABI (include/poulpy_b200.h).

The product is `libpoulpy_b200.so`; this module is the thin ctypes binding a Python caller (tests, bench) uses.  Method
names, argument order and error behaviour follow poulpy-hal/src/api/*.rs (`vec_znx_dft_apply`, `vmp_apply_dft_to_dft`,
`vec_znx_big_normalize`, ...): a violated shape contract raises `PoulpyError` where the reference panics.

There is no CPU fallback: importing works anywhere (so the ABI can be checked without a GPU), but creating a `Module`
without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpoulpy_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "poulpy_b200.h")

NTT120, FFT64 = 0, 1
# pgb_option (include/poulpy_b200.h)
(OPT_NO_FUSION, OPT_NO_GADGET, OPT_NO_COLLAPSE, OPT_CGGI_VARIANT, OPT_CGGI_BLOCK_BT1, OPT_VMP_NO_BT, OPT_VMP_CT, OPT_GADGET_MB,
 OPT_HOST_CHUNK_MB, OPT_CGGI_NTT_PRIMES, OPT_GADGET_PRIMES, OPT_LAST_GADGET_PRIMES, OPT_CGGI_CLUSTER) = range(13)
Q = (1073479681, 1071513601, 1070727169, 1068236801)


class PoulpyError(RuntimeError):
    pass


class _VZ(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n", C.c_uint64), ("cols", C.c_uint64), ("size", C.c_uint64), ("max_size", C.c_uint64)]


class _PP(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n", C.c_uint64), ("cols", C.c_uint64)]


class _PM(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n", C.c_uint64), ("size", C.c_uint64), ("rows", C.c_uint64), ("cols_in", C.c_uint64),
                ("cols_out", C.c_uint64)]


class _BT(C.Structure):
    _fields_ = [("count", C.c_uint64), ("stride_res", C.c_uint64), ("stride_a", C.c_uint64), ("stride_b", C.c_uint64)]


class _BDD(C.Structure):
    _fields_ = [("n_leaves", C.c_uint64), ("n_levels", C.c_uint64), ("level_bit", C.POINTER(C.c_uint32)),
                ("level_count", C.POINTER(C.c_uint32)), ("node_t", C.POINTER(C.c_uint32)), ("node_f", C.POINTER(C.c_uint32)),
                ("n_out", C.c_uint64), ("outputs", C.POINTER(C.c_uint32))]


_lib = None


def lib():
    """Load the CUDA library; fails loudly if it has not been built (python __graft_entry__.py / csrc/build.sh)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PoulpyError(f"{LIB_PATH} is missing: build it with poulpy_b200/csrc/build.sh (no CPU fallback exists)")
        _lib = C.CDLL(LIB_PATH)
        _lib.pgb_last_error.restype = C.c_char_p
        for name in ("pgb_alloc_bytes", "pgb_alloc_device_bytes", "pgb_alloc_pinned_bytes"):
            getattr(_lib, name).restype = C.c_void_p
            getattr(_lib, name).argtypes = [C.c_size_t]
        _lib.pgb_free.argtypes = [C.c_void_p]
        _lib.pgb_free_pinned.argtypes = [C.c_void_p]
        for name in ("pgb_memcpy_h2d", "pgb_memcpy_d2h", "pgb_memcpy_d2d"):
            getattr(_lib, name).argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        _lib.pgb_memset.argtypes = [C.c_void_p, C.c_int, C.c_size_t]
        _lib.pgb_recycle_device_bytes.argtypes = [C.c_void_p, C.c_size_t]
        _lib.pgb_module_new.argtypes = [C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        _lib.pgb_module_destroy.argtypes = [C.c_void_p]
        _lib.pgb_module_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int64]
        _lib.pgb_module_get_option.argtypes = [C.c_void_p, C.c_int]
        _lib.pgb_module_get_option.restype = C.c_int64
        _lib.pgb_module_launch_count.restype = C.c_uint64
        _lib.pgb_module_launch_count.argtypes = [C.c_void_p]
        _lib.pgb_module_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        _lib.pgb_module_sync.argtypes = [C.c_void_p]
        _lib.pgb_trace_galois_element.restype = C.c_int64
        _lib.pgb_profile_category_name.restype = C.c_char_p
        _lib.pgb_profile_enable.argtypes = [C.c_void_p, C.c_int]
        _lib.pgb_profile_read.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int]
        for name in ("pgb_glwe_keyswitch_tmp_bytes", "pgb_glwe_external_product_tmp_bytes", "pgb_cggi_blind_rotate_tmp_bytes",
                     "pgb_cggi_blind_rotate_standard_tmp_bytes", "pgb_cggi_blind_rotate_extended_tmp_bytes", "pgb_vmp_apply_dft_tmp_bytes", "pgb_glwe_tensor_apply_tmp_bytes",
                     "pgb_glwe_tensor_relinearize_tmp_bytes", "pgb_glwe_automorphism_tmp_bytes", "pgb_glwe_automorphism_add_assign_tmp_bytes",
                     "pgb_glwe_trace_assign_tmp_bytes", "pgb_glwe_cmux_tmp_bytes", "pgb_glwe_blind_rotate_ggsw_tmp_bytes", "pgb_glwe_cmux_tree_tmp_bytes", "pgb_glwe_bdd_eval_tmp_bytes", "pgb_glwe_pack_tmp_bytes", "pgb_lwe_keyswitch_tmp_bytes", "pgb_glwe_to_lwe_tmp_bytes", "pgb_glwe_to_lwe_indexed_tmp_bytes", "pgb_lwe_to_glwe_tmp_bytes",
                     "pgb_vec_znx_big_automorphism_assign_tmp_bytes", "pgb_ggsw_expand_row_tmp_bytes",
                     "pgb_bytes_of_vmp_pmat", "pgb_size_of_scalar_prep", "pgb_size_of_scalar_big"):
            getattr(_lib, name).restype = C.c_size_t
    return _lib


def _check(status):
    if status != 0:
        raise PoulpyError(f"[{status}] {lib().pgb_last_error().decode()}")


def _u64(x):
    return C.c_uint64(int(x))


_POOL = {}          # (device, nbytes) -> [device pointers] of released DevBufs (cudaMalloc / cudaFree cost milliseconds once GBs are mapped)
_POOL_BYTES = [0]
_POOL_CAP = 8 << 30


class DevBuf:
    """A device (or managed) allocation owned by Python, zero-filled.  Released device blocks go to a size-keyed pool and are handed out
    again after a device-wide synchronisation and a zero fill (pgb_recycle_device_bytes), so loops that allocate their temporaries per
    call do not pay cudaMalloc / cudaFree."""

    def __init__(self, nbytes, managed=False, device=None):
        self.nbytes = int(nbytes)
        self.managed = managed
        self.device = lib().pgb_current_device() if device is None else int(device)
        self._bind()
        self._key = None if managed else (self.device, self.nbytes)
        free = None if managed else _POOL.get(self._key)
        if free:
            self.ptr = free.pop()
            _POOL_BYTES[0] -= self.nbytes
            _check(lib().pgb_recycle_device_bytes(C.c_void_p(self.ptr), C.c_size_t(self.nbytes)))
            return
        f = lib().pgb_alloc_bytes if managed else lib().pgb_alloc_device_bytes
        self.ptr = f(self.nbytes)
        if not self.ptr and _POOL_BYTES[0]:  # out of memory with blocks parked in the pool: release them and retry
            pool_trim()
            self.ptr = f(self.nbytes)
        if not self.ptr:
            raise PoulpyError(f"device allocation of {nbytes} bytes failed")

    def _bind(self):
        """The allocation / copy helpers act on the current device: select this buffer's."""
        if lib().pgb_current_device() != self.device:
            _check(lib().pgb_set_device(C.c_int(self.device)))

    def __del__(self):
        try:
            if getattr(self, "ptr", None):
                if not self.managed and (1 << 12) <= self.nbytes <= _POOL_CAP:
                    if _POOL_BYTES[0] + self.nbytes > _POOL_CAP:
                        pool_trim()  # parked blocks of sizes nobody asks for any more: release them all, then park this one
                    _POOL.setdefault(self._key, []).append(self.ptr)
                    _POOL_BYTES[0] += self.nbytes
                else:
                    lib().pgb_free(self.ptr)
                self.ptr = None
        except Exception:
            pass

    def upload(self, arr: np.ndarray, offset=0):
        arr = np.ascontiguousarray(arr)
        assert offset + arr.nbytes <= self.nbytes
        self._bind()
        _check(lib().pgb_memcpy_h2d(C.c_void_p(self.ptr + offset), C.c_void_p(arr.ctypes.data), arr.nbytes))

    def download(self, dtype, shape, offset=0):
        out = np.empty(shape, dtype=dtype)
        assert offset + out.nbytes <= self.nbytes
        self._bind()
        _check(lib().pgb_memcpy_d2h(C.c_void_p(out.ctypes.data), C.c_void_p(self.ptr + offset), out.nbytes))
        return out

    def host_view(self, dtype, shape):
        """numpy view over managed memory (the reference's `AsRef<[u8]>` contract); only valid for managed buffers."""
        assert self.managed
        n = int(np.prod(shape))
        arr = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))
        return arr.view(dtype)[:n].reshape(shape)


class _Znx:
    """Common base of the limb-major / column-minor containers."""

    scalar_bytes = 8

    def __init__(self, buf, n, cols, size, offset=0, batch=1, batch_stride=0):
        self.buf, self.n, self.cols, self.size, self.max_size = buf, n, cols, size, size
        self.offset = offset
        self.batch, self.batch_stride = batch, batch_stride

    @property
    def ptr(self):
        return self.buf.ptr + self.offset

    def struct(self):
        return _VZ(self.ptr, self.n, self.cols, self.size, self.max_size)

    def set_size(self, size):
        assert size <= self.max_size
        self.size = size


class VecZnx(_Znx):
    pass


class VecZnxDft(_Znx):
    pass


class VecZnxBig(_Znx):
    pass


class SvpPPol:
    def __init__(self, buf, n, cols):
        self.buf, self.n, self.cols = buf, n, cols

    def struct(self):
        return _PP(self.buf.ptr, self.n, self.cols)


class ScalarZnx(SvpPPol):
    pass


class VmpPMat:
    """One matrix, or (batch > 1) `batch` matrices of the same shape laid out batch_stride bytes apart (e.g. one prepared GGSW per
    ciphertext)."""

    def __init__(self, buf, n, rows, cols_in, cols_out, size, offset=0, batch=1, batch_stride=0):
        self.buf, self.n, self.rows, self.cols_in, self.cols_out, self.size = buf, n, rows, cols_in, cols_out, size
        self.offset = offset
        self.batch, self.batch_stride = batch, batch_stride

    def struct(self):
        return _PM(self.buf.ptr + self.offset, self.n, self.size, self.rows, self.cols_in, self.cols_out)


class MatZnx(VmpPMat):
    pass


class Module:
    """`Module<B200Ntt120>` / `Module<B200Fft64>`: poulpy-hal/src/layouts/module.rs:84-104."""

    def __init__(self, n: int, flavour: int = NTT120, device: int = 0, managed: bool = False):
        self.n, self.flavour, self.device, self.managed = n, flavour, device, managed
        h = C.c_void_p()
        _check(lib().pgb_module_new(_u64(n), C.c_int(flavour), C.c_int(device), C.byref(h)))
        self._h = h
        self.prep_bytes = 16 if flavour == NTT120 else 8
        self.big_bytes = 16 if flavour == NTT120 else 8

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().pgb_module_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def sync(self):
        _check(lib().pgb_module_sync(self._h))

    def set_stream(self, cuda_stream_ptr):
        _check(lib().pgb_module_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    @property
    def launch_count(self):
        return int(lib().pgb_module_launch_count(self._h))

    # --- allocation / transfer ---------------------------------------------------------------------------------
    def _buf(self, nbytes):
        return DevBuf(nbytes, managed=self.managed, device=self.device)

    def set_option(self, option, value):
        """pgb_module_set_option (route / tuning knobs; include/poulpy_b200.h pgb_option)."""
        _check(lib().pgb_module_set_option(self._h, C.c_int(option), C.c_int64(int(value))))

    def get_option(self, option):
        """pgb_module_get_option."""
        return int(lib().pgb_module_get_option(self._h, C.c_int(option)))

    def _scratch(self, need):
        """Grow-only scratch owned by the module, handed to every call that was not given one: the calls of one module are ordered on
        its stream, so consecutive operations can share it (a fresh cudaMalloc + clear per call costs more than most operations)."""
        c = getattr(self, "_scratch_cache", None)
        if c is None or c.nbytes < need:
            self._scratch_cache = c = None  # cudaFree of the old block synchronises the device
            self._scratch_cache = c = DevBuf(max(int(need), 1 << 20), device=self.device)
        return c

    def vec_znx_alloc(self, cols, size, batch=1):
        stride = self.n * cols * size * 8
        return VecZnx(self._buf(stride * batch), self.n, cols, size, batch=batch, batch_stride=stride)

    def vec_znx_dft_alloc(self, cols, size, batch=1):
        stride = self.n * cols * size * self.prep_bytes
        return VecZnxDft(self._buf(stride * batch), self.n, cols, size, batch=batch, batch_stride=stride)

    def vec_znx_big_alloc(self, cols, size, batch=1):
        stride = self.n * cols * size * self.big_bytes
        return VecZnxBig(self._buf(stride * batch), self.n, cols, size, batch=batch, batch_stride=stride)

    def svp_ppol_alloc(self, cols):
        return SvpPPol(self._buf(self.n * cols * self.prep_bytes), self.n, cols)

    def vmp_pmat_alloc(self, rows, cols_in, cols_out, size, batch=1):
        stride = self.n * rows * cols_in * cols_out * size * self.prep_bytes
        return VmpPMat(self._buf(stride * batch), self.n, rows, cols_in, cols_out, size, batch=batch, batch_stride=stride if batch > 1 else 0)

    def vec_znx_from_numpy(self, arr):
        """arr: int64 (size, cols, n) or (batch, size, cols, n)."""
        arr = np.ascontiguousarray(arr, dtype=np.int64)
        batch = arr.shape[0] if arr.ndim == 4 else 1
        size, cols, n = arr.shape[-3:]
        assert n == self.n
        v = self.vec_znx_alloc(cols, size, batch)
        v.buf.upload(arr)
        return v

    def vec_znx_to_numpy(self, v: VecZnx):
        shape = (v.max_size, v.cols, v.n) if v.batch == 1 else (v.batch, v.max_size, v.cols, v.n)
        return v.buf.download(np.int64, shape, v.offset)

    def scalar_znx_from_numpy(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.int64)
        b = self._buf(arr.nbytes)
        b.upload(arr)
        return ScalarZnx(b, arr.shape[1], arr.shape[0])

    def mat_znx_from_numpy(self, arr):
        """arr: int64 (rows, cols_in, size, cols_out, n) -- poulpy-hal/src/layouts/mat_znx.rs:161-176."""
        arr = np.ascontiguousarray(arr, dtype=np.int64)
        rows, cols_in, size, cols_out, n = arr.shape
        b = self._buf(arr.nbytes)
        b.upload(arr)
        return MatZnx(b, n, rows, cols_in, cols_out, size)

    def vec_znx_dft_from_bytes(self, cols, size, raw: np.ndarray):
        v = self.vec_znx_dft_alloc(cols, size)
        v.buf.upload(np.ascontiguousarray(raw).view(np.uint8).reshape(-1)[: v.buf.nbytes])
        return v

    def vec_znx_dft_to_numpy(self, v: VecZnxDft):
        """NTT120: uint32 (size, cols, 4, n) canonical residue planes; FFT64: float64 (size, cols, n) = [re | im]."""
        if self.flavour == NTT120:
            return v.buf.download(np.uint32, (v.max_size, v.cols, 4, v.n), v.offset)
        return v.buf.download(np.float64, (v.max_size, v.cols, v.n), v.offset)

    def vec_znx_big_to_numpy(self, v, size=None, cols=None):
        """NTT120: uint64 (size, cols, n, 2) little-endian i128; FFT64: int64 (size, cols, n)."""
        size = v.max_size if size is None else size
        cols = v.cols if cols is None else cols
        if self.flavour == NTT120:
            return v.buf.download(np.uint64, (size, cols, v.n, 2), v.offset)
        return v.buf.download(np.int64, (size, cols, v.n), v.offset)

    # --- batch descriptor ------------------------------------------------------------------------------------------
    @staticmethod
    def _bt(res, a=None, b=None, count=None, stride_b=None):
        cnt = res.batch if count is None else count
        sa = getattr(a, "batch_stride", 0) if a is not None else 0
        sb = getattr(b, "batch_stride", 0) if b is not None else 0
        if stride_b is not None:
            sb = stride_b
        return _BT(cnt, res.batch_stride, sa if (a is not None and getattr(a, "batch", 1) > 1) else 0,
                   sb if (b is not None and getattr(b, "batch", 1) > 1) or stride_b is not None else 0)

    # --- vec_znx_dft (poulpy-hal/src/api/vec_znx_dft.rs) --------------------------------------------------------------
    def vec_znx_dft_apply(self, step, offset, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        if res.batch > 1:
            bt = self._bt(res, a)
            _check(lib().pgb_vec_znx_dft_apply_batched(self._h, _u64(step), _u64(offset), C.byref(r), _u64(res_col), C.byref(av),
                                                       _u64(a_col), C.byref(bt)))
        else:
            _check(lib().pgb_vec_znx_dft_apply(self._h, _u64(step), _u64(offset), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_idft_apply(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        if res.batch > 1:
            bt = self._bt(res, a)
            _check(lib().pgb_vec_znx_idft_apply_batched(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col), C.byref(bt)))
        else:
            _check(lib().pgb_vec_znx_idft_apply(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_idft_apply_tmpa(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_idft_apply_tmpa(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_idft_apply_consume(self, a: VecZnxDft) -> VecZnxBig:
        av = a.struct()
        if a.batch > 1:
            bt = _BT(a.batch, a.batch_stride, 0, 0)
            _check(lib().pgb_vec_znx_idft_apply_consume_batched(self._h, C.byref(av), C.byref(bt)))
        else:
            _check(lib().pgb_vec_znx_idft_apply_consume(self._h, C.byref(av)))
        return VecZnxBig(a.buf, a.n, a.cols, a.size, a.offset, a.batch, a.batch_stride)

    def _dft3(self, fn, res, res_col, a, a_col, b, b_col):
        r, av, bv = res.struct(), a.struct(), b.struct()
        _check(fn(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col), C.byref(bv), _u64(b_col)))

    def _dft2(self, fn, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(fn(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_dft_add_into(self, res, res_col, a, a_col, b, b_col):
        self._dft3(lib().pgb_vec_znx_dft_add_into, res, res_col, a, a_col, b, b_col)

    def vec_znx_dft_sub(self, res, res_col, a, a_col, b, b_col):
        self._dft3(lib().pgb_vec_znx_dft_sub, res, res_col, a, a_col, b, b_col)

    def vec_znx_dft_add_assign(self, res, res_col, a, a_col):
        self._dft2(lib().pgb_vec_znx_dft_add_assign, res, res_col, a, a_col)

    def vec_znx_dft_sub_assign(self, res, res_col, a, a_col):
        self._dft2(lib().pgb_vec_znx_dft_sub_assign, res, res_col, a, a_col)

    def vec_znx_dft_sub_negate_assign(self, res, res_col, a, a_col):
        self._dft2(lib().pgb_vec_znx_dft_sub_negate_assign, res, res_col, a, a_col)

    def vec_znx_dft_add_scaled_assign(self, res, res_col, a, a_col, a_scale):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_dft_add_scaled_assign(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col), C.c_int64(a_scale)))

    def vec_znx_dft_copy(self, step, offset, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_dft_copy(self._h, _u64(step), _u64(offset), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_dft_zero(self, res, res_col):
        r = res.struct()
        _check(lib().pgb_vec_znx_dft_zero(self._h, C.byref(r), _u64(res_col)))

    # --- svp (poulpy-hal/src/api/svp_ppol.rs) -------------------------------------------------------------------------
    def svp_prepare(self, res: SvpPPol, res_col, a: ScalarZnx, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_svp_prepare(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def svp_apply_dft_to_dft(self, res, res_col, a: SvpPPol, a_col, b, b_col):
        r, pv, bv = res.struct(), a.struct(), b.struct()
        if res.batch > 1:
            bt = _BT(res.batch, res.batch_stride, 0, b.batch_stride if b.batch > 1 else 0)
            _check(lib().pgb_svp_apply_dft_to_dft_batched(self._h, C.byref(r), _u64(res_col), C.byref(pv), _u64(a_col), C.byref(bv),
                                                          _u64(b_col), C.byref(bt)))
        else:
            _check(lib().pgb_svp_apply_dft_to_dft(self._h, C.byref(r), _u64(res_col), C.byref(pv), _u64(a_col), C.byref(bv), _u64(b_col)))

    def svp_apply_dft(self, res, res_col, a: SvpPPol, a_col, b, b_col):
        """HalImpl::svp_apply_dft: b is a VecZnx (coefficient domain)."""
        r, pv, bv = res.struct(), a.struct(), b.struct()
        _check(lib().pgb_svp_apply_dft(self._h, C.byref(r), _u64(res_col), C.byref(pv), _u64(a_col), C.byref(bv), _u64(b_col)))

    def svp_apply_dft_to_dft_assign(self, res, res_col, a: SvpPPol, a_col):
        r, pv = res.struct(), a.struct()
        _check(lib().pgb_svp_apply_dft_to_dft_assign(self._h, C.byref(r), _u64(res_col), C.byref(pv), _u64(a_col)))

    # --- vmp (poulpy-hal/src/api/vmp_pmat.rs) ----------------------------------------------------------------------------
    def vmp_prepare(self, pmat: VmpPMat, mat: MatZnx):
        ps, ms = pmat.struct(), mat.struct()
        _check(lib().pgb_vmp_prepare(self._h, C.byref(ps), C.byref(ms)))

    def vmp_prepare_batched(self, pmat: VmpPMat, mat: MatZnx):
        """pgb_vmp_prepare_batched: the pmat.batch matrices of `mat` in one launch (asynchronous: sync() before reading)."""
        assert pmat.batch == mat.batch, (pmat.batch, mat.batch)
        ps, ms = pmat.struct(), mat.struct()
        bt = _BT(pmat.batch, pmat.batch_stride, mat.batch_stride, 0)
        _check(lib().pgb_vmp_prepare_batched(self._h, C.byref(ps), C.byref(ms), C.byref(bt)))

    def vmp_apply_dft_to_dft(self, res, a, pmat: VmpPMat, limb_offset=0):
        r, av, ps = res.struct(), a.struct(), pmat.struct()
        if res.batch > 1:
            bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
            _check(lib().pgb_vmp_apply_dft_to_dft_batched(self._h, C.byref(r), C.byref(av), C.byref(ps), _u64(limb_offset), C.byref(bt)))
        else:
            _check(lib().pgb_vmp_apply_dft_to_dft(self._h, C.byref(r), C.byref(av), C.byref(ps), _u64(limb_offset)))

    def vmp_apply_dft(self, res, a, pmat: VmpPMat):
        """HalImpl::vmp_apply_dft: a is a VecZnx; scratch is taken from a temporary device buffer of vmp_apply_dft_tmp_bytes."""
        r, av, ps = res.struct(), a.struct(), pmat.struct()
        need = lib().pgb_vmp_apply_dft_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(pmat.rows), _u64(pmat.cols_in),
                                                 _u64(pmat.cols_out), _u64(pmat.size))
        scratch = self._scratch(need)
        _check(lib().pgb_vmp_apply_dft(self._h, C.byref(r), C.byref(av), C.byref(ps), C.c_void_p(scratch.ptr), C.c_size_t(need)))

    # --- vec_znx_big (poulpy-hal/src/api/vec_znx_big.rs) ---------------------------------------------------------------------
    def vec_znx_big_add_small_assign(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        if res.batch > 1:
            bt = self._bt(res, a)
            _check(lib().pgb_vec_znx_big_add_small_assign_batched(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col), C.byref(bt)))
        else:
            _check(lib().pgb_vec_znx_big_add_small_assign(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_big_from_small(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_big_from_small(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_big_normalize(self, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, op=0):
        r, av = res.struct(), a.struct()
        args = (self._h, C.byref(r), _u64(res_base2k), C.c_int64(res_offset), _u64(res_col), C.byref(av), _u64(a_base2k), _u64(a_col))
        if op == 0 and res.batch > 1:
            bt = self._bt(res, a)
            _check(lib().pgb_vec_znx_big_normalize_batched(*args, C.byref(bt)))
        elif op == 0:
            _check(lib().pgb_vec_znx_big_normalize(*args))
        elif op > 0:
            _check(lib().pgb_vec_znx_big_normalize_add_assign(*args))
        else:
            _check(lib().pgb_vec_znx_big_normalize_sub_assign(*args))

    def vec_znx_big_normalize_add_assign(self, *a):
        self.vec_znx_big_normalize(*a, op=1)

    def vec_znx_big_normalize_sub_assign(self, *a):
        self.vec_znx_big_normalize(*a, op=-1)

    def vec_znx_normalize(self, res, res_base2k, res_offset, res_col, a, a_base2k, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_normalize(self._h, C.byref(r), _u64(res_base2k), C.c_int64(res_offset), _u64(res_col), C.byref(av),
                                           _u64(a_base2k), _u64(a_col)))

    def vec_znx_rotate(self, p, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_rotate(self._h, C.c_int64(p), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    # --- CoreImpl tier ------------------------------------------------------------------------------------------------------------
    def glwe_keyswitch(self, res: VecZnx, res_base2k, a: VecZnx, a_base2k, key: VmpPMat, key_base2k, dsize=1, scratch: DevBuf = None):
        """Batched over res.batch ciphertexts (device resident, asynchronous: call sync())."""
        ks = key.struct()
        need = lib().pgb_glwe_keyswitch_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(a_base2k), C.byref(ks), _u64(key_base2k),
                                                  _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride, 0)
        _check(lib().pgb_glwe_keyswitch_batched(self._h, C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_base2k), C.byref(ks),
                                                _u64(key_base2k), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_external_product(self, res: VecZnx, res_base2k, a: VecZnx, a_base2k, ggsw: VmpPMat, ggsw_base2k, dsize=1, scratch: DevBuf = None):
        ks = ggsw.struct()
        need = lib().pgb_glwe_external_product_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(a_base2k), C.byref(ks),
                                                         _u64(ggsw_base2k), _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride, 0)
        _check(lib().pgb_glwe_external_product_batched(self._h, C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_base2k), C.byref(ks),
                                                       _u64(ggsw_base2k), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                                       C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_cmux(self, res: VecZnx, t: VecZnx, f: VecZnx, base2k, s: VmpPMat, ggsw_base2k, dsize=1, scratch: DevBuf = None):
        """CMux of res.batch ciphertexts: res = normalize(normalize(t - f) x s + f).  A batched `s` (a VmpPMat with a batch stride, e.g.
        from vmp_pmat_alloc(..., batch=B) or circuit.prepare_ggsw) gives ciphertext b the selector at s + b * s.batch_stride; an `s` without
        one is shared by the batch.  t / f with batch 1 are shared by the batch.  Asynchronous."""
        assert s.batch_stride == 0 or s.batch >= res.batch, (s.batch, res.batch)
        ks = s.struct()
        need = lib().pgb_glwe_cmux_tmp_bytes(self._h, _u64(res.size), _u64(t.size), _u64(f.size), _u64(base2k), C.byref(ks), _u64(ggsw_base2k),
                                             _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, tv, fv = res.struct(), t.struct(), f.struct()
        bt = _BT(res.batch, res.batch_stride, t.batch_stride if t.batch > 1 else 0, f.batch_stride if f.batch > 1 else 0)
        _check(lib().pgb_glwe_cmux_batched(self._h, C.byref(r), C.byref(tv), C.byref(fv), _u64(base2k), C.byref(ks),
                                           _u64(s.batch_stride), _u64(ggsw_base2k), _u64(dsize), C.byref(bt),
                                           C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_blind_rotate_ggsw(self, res: VecZnx, a: VecZnx, base2k, step, n_bits, s: VmpPMat, ggsw_base2k, dsize=1, ggsw_stride=None,
                               bit_stride=None, scratch: DevBuf = None):
        """Rotation of res.batch GLWEs by encrypted integers m_b = sum_i bit_{b,i} 2^i: res_b = a_b X^(step m_b), one CMux per bit
        (acc <- cmux(X^(step 2^i) acc, acc, s_{b,i})).  Selector (b, i) is at s + b * ggsw_stride + i * bit_stride; the defaults are the
        bit-major layout of circuit.prepare_ggsw over res.batch * n_bits bootstrapped bits (bit_stride = s.batch_stride, ggsw_stride =
        n_bits * s.batch_stride); ggsw_stride = 0 shares one integer across the batch.  An `a` with batch 1 is shared by the batch.
        Asynchronous."""
        if bit_stride is None and ggsw_stride is None:
            assert s.batch >= n_bits * res.batch, (s.batch, n_bits, res.batch)
        bit_stride = s.batch_stride if bit_stride is None else bit_stride
        ggsw_stride = n_bits * s.batch_stride if ggsw_stride is None else ggsw_stride
        ks = s.struct()
        need = lib().pgb_glwe_blind_rotate_ggsw_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(base2k), C.byref(ks), _u64(ggsw_base2k),
                                                          _u64(dsize), _u64(n_bits), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_blind_rotate_ggsw_batched(self._h, C.byref(r), C.byref(av), _u64(base2k), C.c_int64(step), _u64(n_bits),
                                                        C.byref(ks), _u64(ggsw_stride), _u64(bit_stride), _u64(ggsw_base2k), _u64(dsize),
                                                        C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_cmux_tree(self, res: VecZnx, a: VecZnx, base2k, n_bits, s: VmpPMat, ggsw_base2k, dsize=1, entry_stride=None, ggsw_stride=None,
                       bit_stride=None, max_chunk=None, scratch: DevBuf = None):
        """Selection of one of 2^n_bits GLWEs per item by encrypted integers m_b = sum_i bit_{b,i} 2^i: res_b = the table's entry m_b,
        normalised, through a tree of CMuxes (level i: g_{i+1,j} = cmux(g_{i,2j+1}, g_{i,2j}, s_{b,i})).  `a` holds the tables: item b's
        table at a + b * a.batch_stride, its entry j at + j * entry_stride (default: one GLWE of a.size limbs, entries consecutive); an `a`
        with batch 1 is one table shared by the batch.  Selector (b, i) is at s + b * ggsw_stride + i * bit_stride, with the defaults and
        rules of glwe_blind_rotate_ggsw.  max_chunk bounds the items per chunk (the scratch grows with it; results do not depend on it).
        Asynchronous."""
        assert a.batch in (1, res.batch), (a.batch, res.batch)
        if bit_stride is None and ggsw_stride is None:
            assert s.batch >= n_bits * res.batch, (s.batch, n_bits, res.batch)
        bit_stride = s.batch_stride if bit_stride is None else bit_stride
        ggsw_stride = n_bits * s.batch_stride if ggsw_stride is None else ggsw_stride
        entry_stride = self.n * a.cols * a.size * 8 if entry_stride is None else entry_stride
        ks = s.struct()
        chunk = res.batch if max_chunk is None else min(res.batch, max_chunk)
        need = lib().pgb_glwe_cmux_tree_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(base2k), C.byref(ks), _u64(ggsw_base2k),
                                                  _u64(dsize), _u64(n_bits), _u64(chunk))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_cmux_tree_batched(self._h, C.byref(r), C.byref(av), _u64(entry_stride), _u64(base2k), _u64(n_bits), C.byref(ks),
                                                _u64(ggsw_stride), _u64(bit_stride), _u64(ggsw_base2k), _u64(dsize), C.byref(bt),
                                                C.c_void_p(scratch.ptr), C.c_size_t(need if max_chunk is not None else scratch.nbytes)))
        return scratch

    def glwe_bdd_eval(self, res: VecZnx, a: VecZnx, circuit, base2k, n_bits, s: VmpPMat, ggsw_base2k, dsize=1, entry_stride=None,
                      out_stride=None, ggsw_stride=None, bit_stride=None, max_chunk=None, scratch: DevBuf = None):
        """Evaluation of a binary decision diagram (circuit.BddCircuit, or anything with a `struct()` giving the pgb_bdd_circuit) over
        GGSW bits: per item b, node k of level i is cmux(state[t_k], state[f_k], s_{b, bit_i}), and output o is the state circuit.outputs[o]
        (a node normalised into res.size limbs, or a leaf copied).  res holds n_out GLWEs per item: res.batch = batch * n_out, item b's
        output o at index b * n_out + o (out_stride: res.batch_stride by default).  `a` holds the leaves: item b's leaf j at
        a + b * a.batch_stride + j * entry_stride (default: one GLWE of a.size limbs, leaves consecutive); an `a` with batch 1 is shared by
        the batch.  Selector (b, i) is at s + b * ggsw_stride + i * bit_stride, with the defaults and rules of glwe_blind_rotate_ggsw.
        max_chunk bounds the items per chunk (the scratch grows with it; results do not depend on it).  Asynchronous."""
        cs, keep = circuit.struct()
        n_out = cs.n_out
        assert n_out >= 1 and res.batch % n_out == 0, (res.batch, n_out)
        B = res.batch // n_out
        assert a.batch in (1, B), (a.batch, B)
        if bit_stride is None and ggsw_stride is None:
            assert s.batch >= n_bits * B, (s.batch, n_bits, B)
        bit_stride = s.batch_stride if bit_stride is None else bit_stride
        ggsw_stride = n_bits * s.batch_stride if ggsw_stride is None else ggsw_stride
        entry_stride = self.n * a.cols * a.size * 8 if entry_stride is None else entry_stride
        out_stride = res.batch_stride if out_stride is None else out_stride
        assert (B - 1) * n_out * out_stride + (n_out - 1) * out_stride + self.n * res.cols * res.size * 8 <= res.buf.nbytes - res.offset
        ks = s.struct()
        chunk = B if max_chunk is None else min(B, max_chunk)
        need = lib().pgb_glwe_bdd_eval_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(base2k), C.byref(ks), _u64(ggsw_base2k),
                                                 _u64(dsize), C.byref(cs), _u64(chunk))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(B, n_out * out_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_bdd_eval_batched(self._h, C.byref(r), _u64(out_stride), C.byref(av), _u64(entry_stride), _u64(base2k),
                                               _u64(n_bits), C.byref(ks), _u64(ggsw_stride), _u64(bit_stride), _u64(ggsw_base2k),
                                               _u64(dsize), C.byref(cs), C.byref(bt), C.c_void_p(scratch.ptr),
                                               C.c_size_t(need if max_chunk is not None else scratch.nbytes)))
        del keep
        return scratch

    def glwe_pack(self, res: VecZnx, a: VecZnx, index, log_gap_out, keys, base2k, dsize=1, entry_stride=None, max_chunk=None,
                  scratch: DevBuf = None):
        """glwe_pack of n_in = len(index) GLWEs per item into one: res_b's coefficient index[j] carries the constant coefficient of item b's
        input j, bit for bit what circuit.glwe_pack computes over circuit.DeviceGlweOps.  `a` holds the inputs: item b's input j at
        a + b * a.batch_stride + j * entry_stride (default: one GLWE of a.size limbs, inputs consecutive); an `a` with batch 1 is shared by
        the batch.  The inputs are read-only.  keys: log_n prepared automorphism keys, keys[i] for trace_galois_element(i).  max_chunk
        bounds the items per chunk (the scratch grows with it; results do not depend on it).  Asynchronous."""
        idx = np.ascontiguousarray(np.asarray(index, dtype=np.uint32).reshape(-1))
        B = res.batch
        assert a.batch in (1, B), (a.batch, B)
        entry_stride = self.n * a.cols * a.size * 8 if entry_stride is None else entry_stride
        arr = (_PM * len(keys))(*[k.struct() for k in keys])
        chunk = B if max_chunk is None else min(B, max_chunk)
        ip = idx.ctypes.data_as(C.POINTER(C.c_uint32))
        need = lib().pgb_glwe_pack_tmp_bytes(self._h, _u64(res.size), _u64(base2k), C.byref(arr[0]), _u64(dsize), ip, _u64(len(idx)),
                                             _u64(log_gap_out), _u64(chunk))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(max(need, 1))
        r, av = res.struct(), a.struct()
        bt = _BT(B, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_pack_batched(self._h, C.byref(r), C.byref(av), _u64(entry_stride), ip, _u64(len(idx)), _u64(log_gap_out),
                                           _u64(base2k), arr, _u64(len(keys)), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                           C.c_size_t(need if max_chunk is not None else scratch.nbytes)))
        return scratch

    def gadget_key_pin(self, key: VmpPMat):
        """pgb_gadget_key_pin: promise that the key's bytes stay unchanged, so its gadget-kernel forms are derived once."""
        ks = key.struct()
        _check(lib().pgb_gadget_key_pin(self._h, C.byref(ks)))

    def gadget_key_unpin(self, key: VmpPMat):
        ks = key.struct()
        _check(lib().pgb_gadget_key_unpin(self._h, C.byref(ks)))

    def glwe_keyswitch_host(self, res: np.ndarray, res_base2k, a: np.ndarray, a_base2k, key: VmpPMat, key_base2k, dsize=1):
        """res/a: host int64 arrays (batch, size, cols, n); synchronous, copies included (the e2e path)."""
        B, a_size, a_cols, n = a.shape
        ks = key.struct()
        _check(lib().pgb_glwe_keyswitch_host(self._h, C.c_void_p(res.ctypes.data), _u64(res.shape[1]), _u64(res_base2k),
                                             C.c_void_p(a.ctypes.data), _u64(a_size), _u64(a_base2k), _u64(a_cols - 1),
                                             _u64(res.shape[2] - 1), C.byref(ks), _u64(key_base2k), _u64(dsize), _u64(B)))

    def glwe_external_product_host(self, res: np.ndarray, res_base2k, a: np.ndarray, a_base2k, ggsw: VmpPMat, ggsw_base2k, dsize=1):
        B, a_size, a_cols, n = a.shape
        ks = ggsw.struct()
        _check(lib().pgb_glwe_external_product_host(self._h, C.c_void_p(res.ctypes.data), _u64(res.shape[1]), _u64(res_base2k),
                                                    C.c_void_p(a.ctypes.data), _u64(a_size), _u64(a_base2k), _u64(a_cols - 1),
                                                    C.byref(ks), _u64(ggsw_base2k), _u64(dsize), _u64(B)))

    def vec_znx_add_assign(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_add_assign(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_sub_assign(self, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_sub_assign(self._h, C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_mul_xp_minus_one(self, p, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_mul_xp_minus_one(self._h, C.c_int64(p), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_normalize_assign(self, base2k, res, res_col):
        r = res.struct()
        _check(lib().pgb_vec_znx_normalize_assign(self._h, _u64(base2k), C.byref(r), _u64(res_col)))

    # --- bivariate convolution (poulpy-hal/src/api/convolution.rs); CnvPVecL/R share the VecZnxDft layout ---------------------
    def cnv_pvec_alloc(self, cols, size, batch=1) -> VecZnxDft:
        return self.vec_znx_dft_alloc(cols, size, batch)

    def cnv_prepare_left(self, res: VecZnxDft, a: VecZnx, mask=-1):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_cnv_prepare_left(self._h, C.byref(r), C.byref(av), C.c_int64(mask)))

    def cnv_prepare_right(self, res: VecZnxDft, a: VecZnx, mask=-1):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_cnv_prepare_right(self._h, C.byref(r), C.byref(av), C.c_int64(mask)))

    def cnv_prepare_self(self, left: VecZnxDft, right: VecZnxDft, a: VecZnx, mask=-1):
        l, r, av = left.struct(), right.struct(), a.struct()
        _check(lib().pgb_cnv_prepare_self(self._h, C.byref(l), C.byref(r), C.byref(av), C.c_int64(mask)))

    def cnv_apply_dft(self, cnv_offset, res, res_col, a, a_col, b, b_col):
        r, av, bv = res.struct(), a.struct(), b.struct()
        _check(lib().pgb_cnv_apply_dft(self._h, _u64(cnv_offset), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col), C.byref(bv), _u64(b_col)))

    def cnv_pairwise_apply_dft(self, cnv_offset, res, res_col, a, b, col_i, col_j):
        r, av, bv = res.struct(), a.struct(), b.struct()
        _check(lib().pgb_cnv_pairwise_apply_dft(self._h, _u64(cnv_offset), C.byref(r), _u64(res_col), C.byref(av), C.byref(bv), _u64(col_i),
                                                _u64(col_j)))

    def cnv_by_const_apply(self, cnv_offset, res: VecZnxBig, res_col, a: VecZnx, a_col, b):
        r, av = res.struct(), a.struct()
        b = np.ascontiguousarray(b, dtype=np.int64)
        _check(lib().pgb_cnv_by_const_apply(self._h, _u64(cnv_offset), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col),
                                            C.c_void_p(b.ctypes.data), _u64(len(b))))

    # --- CKKS multiplication halves (poulpy-core/src/operations/glwe.rs:699-818, :545-610) -------------------------------------
    def glwe_tensor_apply(self, cnv_offset, res: VecZnx, res_base2k, a: VecZnx, a_effective_k, b: VecZnx, b_effective_k, ab_base2k,
                          scratch: DevBuf = None):
        need = lib().pgb_glwe_tensor_apply_tmp_bytes(self._h, _u64(a.cols - 1), _u64(res.size), _u64(res_base2k), _u64(a.size), _u64(b.size),
                                                     _u64(ab_base2k), _u64(cnv_offset), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av, bv = res.struct(), a.struct(), b.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, b.batch_stride if b.batch > 1 else 0)
        _check(lib().pgb_glwe_tensor_apply_batched(self._h, _u64(cnv_offset), C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_effective_k),
                                                   C.byref(bv), _u64(b_effective_k), _u64(ab_base2k), C.byref(bt), C.c_void_p(scratch.ptr),
                                                   C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_tensor_relinearize(self, res: VecZnx, res_base2k, a: VecZnx, a_base2k, tsk: VmpPMat, key_base2k, dsize=1, scratch: DevBuf = None):
        ks = tsk.struct()
        need = lib().pgb_glwe_tensor_relinearize_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(a_base2k), C.byref(ks), _u64(key_base2k),
                                                           _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_tensor_relinearize_batched(self._h, C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_base2k), C.byref(ks),
                                                         _u64(key_base2k), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                                         C.c_size_t(scratch.nbytes)))
        return scratch

    def vec_znx_automorphism(self, p, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_automorphism(self._h, C.c_int64(p), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def glwe_automorphism(self, res: VecZnx, res_base2k, a: VecZnx, a_base2k, key: VmpPMat, key_base2k, p, dsize=1, scratch: DevBuf = None):
        ks = key.struct()
        need = lib().pgb_glwe_automorphism_tmp_bytes(self._h, _u64(res.size), _u64(a.size), _u64(a_base2k), C.byref(ks), _u64(key_base2k),
                                                     _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride if a.batch > 1 else 0, 0)
        _check(lib().pgb_glwe_automorphism_batched(self._h, C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_base2k), C.byref(ks),
                                                   _u64(key_base2k), C.c_int64(p), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                                   C.c_size_t(scratch.nbytes)))
        return scratch

    # --- trace (poulpy-core/src/glwe_trace.rs) and its HAL pieces ---------------------------------------------------------------------
    def vec_znx_rsh_assign(self, base2k, k, res, res_col):
        r = res.struct()
        if res.batch > 1:
            bt = _BT(res.batch, res.batch_stride, 0, 0)
            _check(lib().pgb_vec_znx_rsh_assign_batched(self._h, _u64(base2k), _u64(k), C.byref(r), _u64(res_col), C.byref(bt)))
        else:
            _check(lib().pgb_vec_znx_rsh_assign(self._h, _u64(base2k), _u64(k), C.byref(r), _u64(res_col)))

    def vec_znx_big_automorphism(self, p, res, res_col, a, a_col):
        r, av = res.struct(), a.struct()
        _check(lib().pgb_vec_znx_big_automorphism(self._h, C.c_int64(p), C.byref(r), _u64(res_col), C.byref(av), _u64(a_col)))

    def vec_znx_big_automorphism_assign(self, p, res, res_col):
        r = res.struct()
        _check(lib().pgb_vec_znx_big_automorphism_assign(self._h, C.c_int64(p), C.byref(r), _u64(res_col)))

    def glwe_automorphism_add_assign(self, res: VecZnx, res_base2k, key: VmpPMat, key_base2k, p, dsize=1, scratch: DevBuf = None):
        ks = key.struct()
        need = lib().pgb_glwe_automorphism_add_assign_tmp_bytes(self._h, _u64(res.size), _u64(res_base2k), C.byref(ks), _u64(key_base2k),
                                                                _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r = res.struct()
        bt = _BT(res.batch, res.batch_stride, 0, 0)
        _check(lib().pgb_glwe_automorphism_add_assign_batched(self._h, C.byref(r), _u64(res_base2k), C.byref(ks), _u64(key_base2k), C.c_int64(p),
                                                              _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def glwe_automorphism_op(self, op, res: VecZnx, res_base2k, a: VecZnx, key: VmpPMat, key_base2k, p, dsize=1, scratch: DevBuf = None):
        """op 0: res = aut(ks(a)) + a, 1: aut(ks(a)) - a, 2: a - aut(ks(a)) (automorphism/glwe_ct.rs:95-275); res may be a."""
        ks = key.struct()
        need = lib().pgb_glwe_automorphism_add_assign_tmp_bytes(self._h, _u64(res.size), _u64(res_base2k), C.byref(ks), _u64(key_base2k),
                                                                _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = res.struct(), a.struct()
        bt = _BT(res.batch, res.batch_stride, a.batch_stride, 0)
        _check(lib().pgb_glwe_automorphism_op_batched(self._h, C.c_int(op), C.byref(r), _u64(res_base2k), C.byref(av), C.byref(ks),
                                                      _u64(key_base2k), C.c_int64(p), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr),
                                                      C.c_size_t(scratch.nbytes)))
        return scratch

    def trace_galois_element(self, i):
        return int(lib().pgb_trace_galois_element(self._h, _u64(i)))

    def glwe_trace_assign(self, res: VecZnx, res_base2k, skip, keys, key_base2k, dsize=1, scratch: DevBuf = None):
        """keys: list of log_n prepared automorphism keys, keys[i] for trace_galois_element(i)."""
        arr = (_PM * len(keys))(*[k.struct() for k in keys])
        need = lib().pgb_glwe_trace_assign_tmp_bytes(self._h, _u64(res.size), _u64(res_base2k), C.byref(arr[min(skip, len(keys) - 1)]),
                                                     _u64(key_base2k), _u64(dsize), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r = res.struct()
        bt = _BT(res.batch, res.batch_stride, 0, 0)
        _check(lib().pgb_glwe_trace_assign_batched(self._h, C.byref(r), _u64(res_base2k), _u64(skip), arr, _u64(len(keys)), _u64(key_base2k),
                                                   _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def ggsw_expand_row(self, ggsw_buf: DevBuf, batch, dnum, rank, size, res_base2k, tsk, tsk_base2k, dsize=1, scratch: DevBuf = None):
        """ggsw_buf: `batch` MatZnx(dnum, rank+1, rank+1, size) back to back, column-0 GLWEs filled; tsk: list of rank prepared keys
        (poulpy-core/src/conversion/gglwe_to_ggsw.rs:116-268)."""
        arr = (_PM * len(tsk))(*[k.struct() for k in tsk])
        need = lib().pgb_ggsw_expand_row_tmp_bytes(self._h, _u64(rank), _u64(size), _u64(res_base2k), C.byref(arr[0]), _u64(tsk_base2k),
                                                   _u64(dsize), _u64(batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        g = _PM(ggsw_buf.ptr, self.n, size, dnum, rank + 1, rank + 1)
        stride = self.n * dnum * (rank + 1) * (rank + 1) * size * 8
        bt = _BT(batch, stride, 0, 0)
        _check(lib().pgb_ggsw_expand_row_batched(self._h, C.byref(g), _u64(res_base2k), arr, _u64(len(tsk)), _u64(tsk_base2k), _u64(dsize),
                                                 C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def cggi_x_pow_a(self) -> SvpPPol:
        res = self.svp_ppol_alloc(2 * self.n)
        r = res.struct()
        _check(lib().pgb_cggi_x_pow_a(self._h, C.byref(r)))
        return res

    def cggi_blind_rotate(self, res: VecZnx, lwe_2n: DevBuf, n_lwe, lut: VecZnx, brk: VmpPMat, x_pow_a: SvpPPol, block_size, base2k,
                          scratch: DevBuf = None):
        """brk: the n_lwe prepared GGSWs stored consecutively (VmpPMat describing the first one)."""
        need = lib().pgb_cggi_blind_rotate_tmp_bytes(self._h, _u64(res.cols - 1), _u64(res.size), _u64(brk.rows), _u64(brk.size),
                                                     _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, lv, bs, xp = res.struct(), lut.struct(), brk.struct(), x_pow_a.struct()
        bt = _BT(res.batch, res.batch_stride, 0, 0)
        _check(lib().pgb_cggi_blind_rotate_batched(self._h, C.byref(r), C.c_void_p(lwe_2n.ptr), _u64(n_lwe), C.byref(lv), C.byref(bs),
                                                   C.byref(xp), _u64(block_size), _u64(base2k), C.byref(bt), C.c_void_p(scratch.ptr),
                                                   C.c_size_t(scratch.nbytes)))
        return scratch


    def cggi_blind_rotate_host(self, res: np.ndarray, lwe: np.ndarray, lwe_base2k, lut: VecZnx, brk: VmpPMat, x_pow_a: SvpPPol, block_size,
                               base2k, rot_left=True):
        """res: host int64 (batch, res_size, rank+1, n); lwe: host int64 (batch, lwe_size, 1, n_lwe+1) NOT yet mod-switched; synchronous,
        copies included (the e2e path of the blind rotation)."""
        B, lwe_size, _, len_ = lwe.shape
        assert res.shape[0] == B and res.flags["C_CONTIGUOUS"] and lwe.flags["C_CONTIGUOUS"]
        lv, bs, xp = lut.struct(), brk.struct(), x_pow_a.struct()
        _check(lib().pgb_cggi_blind_rotate_host(self._h, C.c_void_p(res.ctypes.data), _u64(res.shape[2] - 1), _u64(res.shape[1]),
                                                C.c_void_p(lwe.ctypes.data), _u64(len_ - 1), _u64(lwe_size), _u64(lwe_base2k),
                                                C.c_int(1 if rot_left else 0), C.byref(lv), C.byref(bs), C.byref(xp), _u64(block_size),
                                                _u64(base2k), _u64(B)))

    def cggi_blind_rotate_extended(self, res: VecZnx, lwe_2n: DevBuf, n_lwe, luts: VecZnx, ext, brk: VmpPMat, x_pow_a: SvpPPol, block_size,
                                   base2k, scratch: DevBuf = None):
        """execute_block_binary_extended (algorithm.rs:121-273); luts: VecZnx(1 col) with `ext` batch items (LookupTable.data), lwe_2n
        mod-switched to 2 * n * ext."""
        need = lib().pgb_cggi_blind_rotate_extended_tmp_bytes(self._h, _u64(res.cols - 1), _u64(res.size), _u64(brk.rows), _u64(brk.size),
                                                              _u64(ext), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, lv, bs, xp = res.struct(), luts.struct(), brk.struct(), x_pow_a.struct()
        bt = _BT(res.batch, res.batch_stride, 0, 0)
        _check(lib().pgb_cggi_blind_rotate_extended_batched(self._h, C.byref(r), C.c_void_p(lwe_2n.ptr), _u64(n_lwe), C.byref(lv), _u64(ext),
                                                            C.byref(bs), C.byref(xp), _u64(block_size), _u64(base2k), C.byref(bt),
                                                            C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def cggi_mod_switch_2n(self, lwe_dev: DevBuf, batch, n_lwe, size, lwe_base2k, two_n_domain, rot_left=True) -> DevBuf:
        """mod_switch_2n of `batch` LWEs stored as (batch, size, 1, n_lwe + 1) int64 on the device -> DevBuf int64 [batch][n_lwe + 1]."""
        out = DevBuf(batch * (n_lwe + 1) * 8, device=self.device)
        lv = _VZ(lwe_dev.ptr, n_lwe + 1, 1, size, size)
        bt = _BT(batch, 0, size * (n_lwe + 1) * 8, 0)
        _check(lib().pgb_cggi_mod_switch_2n_batched(self._h, C.c_void_p(out.ptr), C.byref(lv), _u64(lwe_base2k), _u64(two_n_domain),
                                                    C.c_int(1 if rot_left else 0), C.byref(bt)))
        return out

    # --- LWE <-> GLWE (poulpy-core/src/conversion/glwe_to_lwe.rs, lwe_to_glwe.rs, keyswitching/lwe.rs) ----------------------------------
    # An LWE batch is a DevBuf of `batch` one-column VecZnx(n_lwe + 1, size) (b, a_0, ..), item b at b * stride bytes (default: back to
    # back, stride = size * (n_lwe + 1) * 8).  Asynchronous like every batched call: sync() before reading the results.
    @staticmethod
    def _lwe(buf: DevBuf, n_lwe, size):
        return _VZ(buf.ptr, n_lwe + 1, 1, size, size)

    @staticmethod
    def _lwe_stride(n_lwe, size, stride):
        return size * (n_lwe + 1) * 8 if stride is None else stride

    def _lwe_call(self, name, r, res_size, res_base2k, av, a_size, a_base2k, key: VmpPMat, key_base2k, dsize, bt, scratch):
        ks = key.struct()
        need = getattr(lib(), name + "_tmp_bytes")(self._h, _u64(res_size), _u64(a_size), _u64(a_base2k), C.byref(ks), _u64(key_base2k),
                                                   _u64(dsize), _u64(bt.count))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        _check(getattr(lib(), name + "_batched")(self._h, C.byref(r), _u64(res_base2k), C.byref(av), _u64(a_base2k), C.byref(ks),
                                                 _u64(key_base2k), _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def lwe_sample_extract(self, res: DevBuf, n_lwe, res_size, a: VecZnx, res_stride=None):
        """LWE::sample_extract of the a.batch rank-1 GLWEs of `a` into the LWE batch `res`."""
        bt = _BT(a.batch, self._lwe_stride(n_lwe, res_size, res_stride), a.batch_stride, 0)
        r, av = self._lwe(res, n_lwe, res_size), a.struct()
        _check(lib().pgb_lwe_sample_extract_batched(self._h, C.byref(r), C.byref(av), C.byref(bt)))

    def lwe_keyswitch(self, res: DevBuf, n_out, res_size, res_base2k, a: DevBuf, n_in, a_size, a_base2k, key: VmpPMat, key_base2k, batch,
                      dsize=1, scratch: DevBuf = None, res_stride=None, a_stride=None):
        """LWE::keyswitch of `batch` LWEs of dimension n_in into dimension n_out; key = VmpPMat(dnum, 1, 2, key_size)."""
        bt = _BT(batch, self._lwe_stride(n_out, res_size, res_stride), self._lwe_stride(n_in, a_size, a_stride), 0)
        return self._lwe_call("pgb_lwe_keyswitch", self._lwe(res, n_out, res_size), res_size, res_base2k, self._lwe(a, n_in, a_size), a_size,
                              a_base2k, key, key_base2k, dsize, bt, scratch)

    def glwe_to_lwe(self, res: DevBuf, n_lwe, res_size, res_base2k, a: VecZnx, a_base2k, key: VmpPMat, key_base2k, dsize=1,
                    scratch: DevBuf = None, res_stride=None):
        """LWE::from_glwe of the a.batch GLWEs of rank k; key = VmpPMat(dnum, k, 2, key_size)."""
        bt = _BT(a.batch, self._lwe_stride(n_lwe, res_size, res_stride), a.batch_stride, 0)
        return self._lwe_call("pgb_glwe_to_lwe", self._lwe(res, n_lwe, res_size), res_size, res_base2k, a.struct(), a.size, a_base2k, key,
                              key_base2k, dsize, bt, scratch)

    def glwe_to_lwe_indexed(self, res: DevBuf, n_lwe, res_size, res_base2k, a: VecZnx, a_base2k, index, key: VmpPMat, key_base2k, dsize=1,
                            entry_stride=None, res_stride=None, scratch: DevBuf = None):
        """glwe_to_lwe at the coefficients `index` (host list, each below n) of the a.batch GLWEs of rank k, with one key-switch per item:
        LWE (b, j) = lwe_sample_extract(X^-index[j] * glwe_keyswitch(a_b)), at res + b * res_stride + j * entry_stride (defaults: one LWE
        apart, res_stride = len(index) * entry_stride, so LWE b * len(index) + j is coefficient index[j] of item b: the item-major order of
        circuit_bootstrap_to_constant).  index = [0] equals glwe_to_lwe.  key = VmpPMat(dnum, k, 2, key_size)."""
        idx = np.ascontiguousarray(np.asarray(index, dtype=np.uint32).reshape(-1))
        entry_stride = self._lwe_stride(n_lwe, res_size, entry_stride)
        res_stride = len(idx) * entry_stride if res_stride is None else res_stride
        ks = key.struct()
        need = lib().pgb_glwe_to_lwe_indexed_tmp_bytes(self._h, _u64(res_size), _u64(a.size), _u64(a_base2k), C.byref(ks), _u64(key_base2k),
                                                       _u64(dsize), _u64(len(idx)), _u64(a.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, av = self._lwe(res, n_lwe, res_size), a.struct()
        bt = _BT(a.batch, res_stride, a.batch_stride, 0)
        _check(lib().pgb_glwe_to_lwe_indexed_batched(self._h, C.byref(r), _u64(entry_stride), _u64(res_base2k), C.byref(av), _u64(a_base2k),
                                                     idx.ctypes.data_as(C.POINTER(C.c_uint32)), _u64(len(idx)), C.byref(ks), _u64(key_base2k),
                                                     _u64(dsize), C.byref(bt), C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch

    def lwe_to_glwe(self, res: VecZnx, res_base2k, a: DevBuf, n_lwe, a_size, a_base2k, key: VmpPMat, key_base2k, dsize=1,
                    scratch: DevBuf = None, a_stride=None):
        """GLWE::from_lwe of res.batch LWEs into GLWEs of rank k; key = VmpPMat(dnum, 1, k + 1, key_size)."""
        bt = _BT(res.batch, res.batch_stride, self._lwe_stride(n_lwe, a_size, a_stride), 0)
        return self._lwe_call("pgb_lwe_to_glwe", res.struct(), res.size, res_base2k, self._lwe(a, n_lwe, a_size), a_size, a_base2k, key,
                              key_base2k, dsize, bt, scratch)

    def cggi_blind_rotate_standard(self, res: VecZnx, res_base2k, lwe_2n: DevBuf, n_lwe, lut: VecZnx, brk: VmpPMat, brk_base2k,
                                   scratch: DevBuf = None):
        """execute_standard (block_size == 1 keys); brk: the n_lwe prepared GGSWs stored consecutively."""
        bs = brk.struct()
        need = lib().pgb_cggi_blind_rotate_standard_tmp_bytes(self._h, _u64(res.cols - 1), _u64(res.size), _u64(res_base2k), C.byref(bs),
                                                              _u64(brk_base2k), _u64(res.batch))
        if scratch is None or scratch.nbytes < need:
            scratch = self._scratch(need)
        r, lv = res.struct(), lut.struct()
        bt = _BT(res.batch, res.batch_stride, 0, 0)
        _check(lib().pgb_cggi_blind_rotate_standard_batched(self._h, C.byref(r), _u64(res_base2k), C.c_void_p(lwe_2n.ptr), _u64(n_lwe),
                                                            C.byref(lv), C.byref(bs), _u64(brk_base2k), C.byref(bt),
                                                            C.c_void_p(scratch.ptr), C.c_size_t(scratch.nbytes)))
        return scratch


def glwe_keyswitch_host_sharded(modules, keys, res: np.ndarray, res_base2k, a: np.ndarray, a_base2k, key_base2k, dsize=1):
    """pgb_glwe_keyswitch_host_sharded: one call, one Module (and one replica of the prepared key) per device; res / a are host int64
    arrays (batch, size, cols, n) split contiguously over the modules."""
    B, a_size, a_cols, n = a.shape
    hs = (C.c_void_p * len(modules))(*[m._h for m in modules])
    ks = (_PM * len(keys))(*[k.struct() for k in keys])
    _check(lib().pgb_glwe_keyswitch_host_sharded(hs, ks, _u64(len(modules)), C.c_void_p(res.ctypes.data), _u64(res.shape[1]), _u64(res_base2k),
                                                 C.c_void_p(a.ctypes.data), _u64(a_size), _u64(a_base2k), _u64(a_cols - 1),
                                                 _u64(res.shape[2] - 1), _u64(key_base2k), _u64(dsize), _u64(B)))


def device_count():
    return int(lib().pgb_device_count())


def pool_trim():
    """cudaFree every block parked in the DevBuf pool."""
    for blocks in _POOL.values():
        while blocks:
            lib().pgb_free(blocks.pop())
    _POOL.clear()
    _POOL_BYTES[0] = 0


def pinned_empty(shape, dtype=np.int64):
    """numpy array over page-locked host memory (for the e2e host front ends)."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = lib().pgb_alloc_pinned_bytes(nbytes)
    if not p:
        raise PoulpyError("pinned allocation failed")
    arr = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p)).view(dtype).reshape(shape)
    return arr
