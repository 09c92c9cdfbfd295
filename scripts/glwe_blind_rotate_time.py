"""Blind-rotation rates on one GPU at the circuit-bootstrapping bench shape (n = 1024, rank 2, base2k 13, GGSW selectors VmpPMat(2, 3, 3, 2),
GLWEs of 2 limbs), both flavours, 8 bits with per-item selectors in the bit-major layout of circuit.prepare_ggsw, batches 512 and 4096.

    python scripts/glwe_blind_rotate_time.py [--batches 512 4096] [--bits 8] [--reps 10] [--windows 5] [--out FILE.json]

In one process it alternates, window by window, Module.glwe_blind_rotate_ggsw with today's composition (per bit: rotate every column into
a staged t, then glwe_cmux, two host-alternated buffers), asserts that both give equal outputs, and reports both.  Times come from CUDA
events on the module's stream after a warm-up of both; a rate is the median over `windows` windows of `reps` back-to-back calls.  The
selectors are B * bits prepared GGSWs: 4096 * 8 of them are 19 GB (NTT120) / 9.7 GB (FFT64), 512 * 8 are 2.4 GB / 1.2 GB, all above the
126 MB of L2, so every call streams them from HBM.  64 distinct GGSWs are prepared and replicated on the device.  The card's name and power
limit are read in the same run.

Algorithmic bytes of one rotation = bits x those of one per-item CMux (each buffer once; pb = 16 B NTT120 / 8 B FFT64, g = n * cols * 8 B
per i64 limb), as in scripts/cmux_time.py:
  NTT120 fused:  selector dnum*cols*cols*S*n*pb + t, f (2 * size g) + d written and read (2 * size g) + a_dft written and read
                 (2 * size * n * cols * pb) + f again (size g) + res (size g)
  FFT64 fused:   selector + t, f + d written and read + f written into res (size g) + a_dft written and read + res_dft written and read
                 (2 * cols * S * n * pb) + res read and written (2 * size g)
The composition moves, per bit, also the staged t (written and read, 2 * size g); the same formula is used for both, so the two rates are
comparable and the composition's is an upper bound of what it needs."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import poulpy_b200 as pb  # noqa: E402
from poulpy_b200.hal import _BT, _check, lib  # noqa: E402

N, RANK, K, DNUM, S, SIZE = 1024, 2, 13, 2, 2, 2
COLS = RANK + 1
STEP = -3
DISTINCT = 64
HBM_BYTES_PER_S = 7.7e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], text=True)
        power, clock = [x.strip() for x in out.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        power, clock = "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def rand(rng, shape, k=K):
    return rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=shape, dtype=np.int64)


def cmux_bytes(fl):
    pb_ = 16 if fl == pb.NTT120 else 8
    g = N * COLS * 8
    sel = DNUM * COLS * COLS * S * N * pb_
    if fl == pb.NTT120:
        return sel + 2 * SIZE * g + 2 * SIZE * g + 2 * SIZE * N * COLS * pb_ + SIZE * g + SIZE * g
    return sel + 2 * SIZE * g + 2 * SIZE * g + SIZE * g + 2 * SIZE * N * COLS * pb_ + 2 * COLS * S * N * pb_ + 2 * SIZE * g


def selectors(m, rng, count):
    """`count` prepared GGSWs: DISTINCT of them prepared in one batched call, then replicated by doubling device copies."""
    mat_item = DNUM * COLS * COLS * S * N * 8
    mats = pb.DevBuf(DISTINCT * mat_item)
    mats.upload(rand(rng, (DISTINCT, DNUM, COLS, S, COLS, N)))
    sel = m.vmp_pmat_alloc(DNUM, COLS, COLS, S, batch=count)
    item = sel.batch_stride
    m.vmp_prepare_batched(pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S, batch=DISTINCT, batch_stride=item),
                          pb.hal.MatZnx(mats, N, DNUM, COLS, COLS, S, batch=DISTINCT, batch_stride=mat_item))
    m.sync()
    done = DISTINCT
    while done < count:
        cp = min(done, count - done)
        assert lib().pgb_memcpy_d2d(C.c_void_p(sel.buf.ptr + done * item), C.c_void_p(sel.buf.ptr), cp * item) == 0
        done += cp
    return sel


def composition(m, res, bufs, a, sel, B, bits, scratch):
    """Per bit: rotate every column of acc into t, glwe_cmux(t, acc) into the other buffer; the last bit writes res."""
    t, pp = bufs
    cur = a
    item = sel.batch_stride
    for i in range(bits):
        dst = res if (bits - 1 - i) % 2 == 0 else pp
        bt = _BT(B, t.batch_stride, cur.batch_stride, 0)
        p = (STEP << i) % (2 * N)
        for c in range(COLS):
            r, av = t.struct(), cur.struct()
            _check(lib().pgb_vec_znx_rotate_batched(m._h, C.c_int64(p), C.byref(r), C.c_uint64(c), C.byref(av), C.c_uint64(c), C.byref(bt)))
        si = pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S, offset=i * item, batch=B, batch_stride=bits * item)
        m.glwe_cmux(dst, t, cur, K, si, K, scratch=scratch)
        cur = dst


def run(fl, B, bits, reps, windows):
    rng = np.random.default_rng(B + fl)
    m = pb.Module(N, fl)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    sel = selectors(m, rng, B * bits)
    a = m.vec_znx_from_numpy(rand(rng, (B, SIZE, COLS, N)))
    res_new, res_old = m.vec_znx_alloc(COLS, SIZE, B), m.vec_znx_alloc(COLS, SIZE, B)
    bufs = (m.vec_znx_alloc(COLS, SIZE, B), m.vec_znx_alloc(COLS, SIZE, B))

    sc_new = m.glwe_blind_rotate_ggsw(res_new, a, K, STEP, bits, sel, K)
    sc_new = pb.DevBuf(sc_new.nbytes)  # a scratch of its own, apart from the module's (which the composition's CMuxes use)
    sc_old = None

    def new():
        m.glwe_blind_rotate_ggsw(res_new, a, K, STEP, bits, sel, K, scratch=sc_new)

    def old():
        composition(m, res_old, bufs, a, sel, B, bits, sc_old)

    l0 = m.launch_count
    new()
    m.sync()
    l1 = m.launch_count
    old()
    m.sync()
    l2 = m.launch_count
    assert np.array_equal(m.vec_znx_to_numpy(res_new), m.vec_znx_to_numpy(res_old)), "the entry and the composition differ"
    for _ in range(2):
        new()
        old()
    m.sync()
    win = {"entry": [], "composition": []}
    for _ in range(windows):
        for name, fn in (("entry", new), ("composition", old)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            e1.synchronize()
            win[name].append(e0.elapsed_time(e1) / reps)
    assert np.array_equal(m.vec_znx_to_numpy(res_new), m.vec_znx_to_numpy(res_old)), "the entry and the composition differ"
    by = bits * cmux_bytes(fl)
    out = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "batch": B, "bits": bits, "selector_bytes": B * bits * sel.batch_stride}
    for name, launches in (("entry", l1 - l0), ("composition", l2 - l1)):
        ms = float(np.median(win[name]))
        out[name] = {"ms_per_call": ms, "rotations_per_s": B / (ms * 1e-3), "bytes_per_rotation": by, "bytes_per_s": by * B / (ms * 1e-3),
                     "hbm_fraction": by * B / (ms * 1e-3) / HBM_BYTES_PER_S, "launches_per_call": launches, "window_ms": win[name]}
    out["composition_over_entry"] = out["composition"]["ms_per_call"] / out["entry"]["ms_per_call"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--bits", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("glwe_blind_rotate_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "dnum": DNUM, "ggsw_size": S, "glwe_size": SIZE, "step": STEP},
              "runs": []}
    for fl in (pb.NTT120, pb.FFT64):
        for B in args.batches:
            r = run(fl, B, args.bits, args.reps, args.windows)
            result["runs"].append(r)
            print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "window_ms"}) for k, v in r.items()}),
                  flush=True)
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
