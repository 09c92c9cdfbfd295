import os, sys, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import poulpy_b200 as pb
lib = pb.lib()
log_n, rows, cols_in, cols_out, size = 14, 31, 1, 2, 32
n = 1 << log_n
m = pb.Module(n, pb.NTT120)
pm = m.vmp_pmat_alloc(rows, cols_in, cols_out, size)
a = m.vec_znx_dft_alloc(cols_in, rows)
r = m.vec_znx_dft_alloc(cols_out, size)
for _ in range(3):
    m.vmp_apply_dft_to_dft(r, a, pm, 0)
