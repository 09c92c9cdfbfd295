import os, sys, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import poulpy_b200 as pb
lib = pb.lib()
stream = torch.cuda.Stream()
flush = pb.DevBuf(256 << 20)
for fl, nm in ((pb.NTT120, "ntt120"), (pb.FFT64, "fft64")):
    for (log_n, rows, cols_in, cols_out, size) in ((13, 15, 1, 2, 16), (14, 31, 1, 2, 32), (15, 14, 1, 2, 15)):
        n = 1 << log_n
        m = pb.Module(n, fl)
        m.set_stream(stream.cuda_stream)
        pm = m.vmp_pmat_alloc(rows, cols_in, cols_out, size)
        a = m.vec_znx_dft_alloc(cols_in, rows)
        r = m.vec_znx_dft_alloc(cols_out, size)
        rs, as_, ps = r.struct(), a.struct(), pm.struct()
        bt = pb.hal._BT(1, 0, 0, 0)
        R, Cc = rows * cols_in, cols_out * size
        byts = (R + R * Cc + Cc) * n * m.prep_bytes
        times = []
        for it in range(10):
            lib.pgb_memset(C.c_void_p(flush.ptr), it, C.c_size_t(flush.nbytes))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record(stream)
                lib.pgb_vmp_apply_dft_to_dft_batched(m._h, C.byref(rs), C.byref(as_), C.byref(ps), C.c_uint64(0), C.byref(bt))
                e1.record(stream)
            torch.cuda.synchronize()
            if it >= 3:
                times.append(e0.elapsed_time(e1))
        ms = float(np.median(times))
        print(nm, (log_n, rows, cols_in, cols_out, size), "MB", round(byts / 1e6), "ms", round(ms, 4), "GB/s", round(byts / ms / 1e6))
        del m, pm, a, r
