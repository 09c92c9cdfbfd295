"""CMux-tree rates on one GPU at the circuit-bootstrapping bench shape (n = 1024, rank 2, base2k 13, GGSW selectors VmpPMat(2, 3, 3, 2),
GLWEs of 2 limbs), both flavours, n_bits 4 and 8, batches 512 and 4096, one table shared by the batch, per-item selectors in the
bit-major layout of circuit.prepare_ggsw.

    python scripts/cmux_tree_time.py [--batches 512 4096] [--bits 4 8] [--reps 3] [--windows 3] [--out FILE.json]

In one process it alternates, window by window, Module.glwe_cmux_tree with today's composition (one glwe_cmux per level and pair j, each
over the whole batch, 2^bits - 1 calls), asserts that both give equal outputs, and reports both.  The composition runs its calls depth
first (a pair as soon as both children exist), so it holds two GLWE batches per level instead of a whole level; the calls and what each
reads are those of level-by-level order.  Times come from CUDA events on the module's stream after a warm-up of both; a rate is the
median over `windows` windows of `reps` back-to-back calls.  The selectors are B * bits prepared GGSWs (at batch 4096 and 8 bits 19 GB
NTT120 / 9.7 GB FFT64, at 512 and 4 bits 1.2 GB / 0.6 GB), all above the 126 MB of L2; 64 distinct GGSWs are prepared and replicated on
the device.  The entry runs with the scratch of one chunk of min(batch, 65535 / 2^(bits-1)) items.  The card's name and power limit are
read in the same run.

Algorithmic bytes of one tree (one item), with sel = one prepared GGSW (dnum*cols*cols*S*n*pb; pb = 16 B NTT120 / 8 B FFT64) and c = the
bytes of one per-item CMux without its selector (the formula of scripts/glwe_blind_rotate_time.py):
  entry:        bits * sel + (2^bits - 1) * c      -- each item's selector once per level
  composition:  (2^bits - 1) * (sel + c)           -- each item's selector once per CMux
bytes/s = batch * that / time."""
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
from poulpy_b200.hal import lib  # noqa: E402

N, RANK, K, DNUM, S, SIZE = 1024, 2, 13, 2, 2, 2
COLS = RANK + 1
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


def sel_bytes(fl):
    return DNUM * COLS * COLS * S * N * (16 if fl == pb.NTT120 else 8)


def cmux_other_bytes(fl):
    """One per-item CMux's bytes without its selector (as in scripts/glwe_blind_rotate_time.py)."""
    pb_ = 16 if fl == pb.NTT120 else 8
    g = N * COLS * 8
    if fl == pb.NTT120:
        return 2 * SIZE * g + 2 * SIZE * g + 2 * SIZE * N * COLS * pb_ + SIZE * g + SIZE * g
    return 2 * SIZE * g + 2 * SIZE * g + SIZE * g + 2 * SIZE * N * COLS * pb_ + 2 * COLS * S * N * pb_ + 2 * SIZE * g


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


def composition(m, res, bufs, table, sel, B, bits, scratch):
    """glwe_cmux(g_{i+1}[j], g_i[2j + 1], g_i[2j]) for every level i and pair j, depth first: bufs[i][0 / 1] hold g_{i+1}[2p] / [2p + 1]
    until their parent runs; the root writes res."""
    item, es = sel.batch_stride, N * COLS * SIZE * 8
    sels = [pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S, offset=i * item, batch=B, batch_stride=bits * item) for i in range(bits)]

    def node(i, j, dst):  # computes g_{i+1}[j] into dst
        if i == 0:
            t = pb.hal.VecZnx(table.buf, N, COLS, SIZE, offset=table.offset + (2 * j + 1) * es)
            f = pb.hal.VecZnx(table.buf, N, COLS, SIZE, offset=table.offset + 2 * j * es)
        else:
            f, t = bufs[i - 1]
            node(i - 1, 2 * j, f)
            node(i - 1, 2 * j + 1, t)
        m.glwe_cmux(dst, t, f, K, sels[i], K, scratch=scratch)

    node(bits - 1, 0, res)


def run(fl, B, bits, reps, windows):
    rng = np.random.default_rng(B + fl + 7 * bits)
    m = pb.Module(N, fl)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    sel = selectors(m, rng, B * bits)
    leaves = m.vec_znx_from_numpy(rand(rng, (1 << bits, SIZE, COLS, N)))
    table = pb.hal.VecZnx(leaves.buf, N, COLS, SIZE)  # one table shared by the batch
    res_new, res_old = m.vec_znx_alloc(COLS, SIZE, B), m.vec_znx_alloc(COLS, SIZE, B)
    bufs = [(m.vec_znx_alloc(COLS, SIZE, B), m.vec_znx_alloc(COLS, SIZE, B)) for _ in range(bits - 1)]

    sc_new = m.glwe_cmux_tree(res_new, table, K, bits, sel, K)
    sc_new = pb.DevBuf(sc_new.nbytes)  # a scratch of its own, apart from the module's (which the composition's CMuxes use)

    def new():
        m.glwe_cmux_tree(res_new, table, K, bits, sel, K, scratch=sc_new)

    def old():
        composition(m, res_old, bufs, table, sel, B, bits, None)

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
    cmuxes = (1 << bits) - 1
    by = {"entry": bits * sel_bytes(fl) + cmuxes * cmux_other_bytes(fl), "composition": cmuxes * (sel_bytes(fl) + cmux_other_bytes(fl))}
    out = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "batch": B, "bits": bits, "selector_bytes": B * bits * sel.batch_stride,
           "entry_scratch_bytes": sc_new.nbytes}
    for name, launches in (("entry", l1 - l0), ("composition", l2 - l1)):
        ms = float(np.median(win[name]))
        out[name] = {"ms_per_call": ms, "trees_per_s": B / (ms * 1e-3), "bytes_per_tree": by[name], "bytes_per_s": by[name] * B / (ms * 1e-3),
                     "hbm_fraction": by[name] * B / (ms * 1e-3) / HBM_BYTES_PER_S, "launches_per_call": launches, "window_ms": win[name]}
    out["composition_over_entry"] = out["composition"]["ms_per_call"] / out["entry"]["ms_per_call"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--bits", type=int, nargs="+", default=[4, 8])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cmux_tree_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "dnum": DNUM, "ggsw_size": S, "glwe_size": SIZE}, "runs": []}
    for fl in (pb.NTT120, pb.FFT64):
        for bits in args.bits:
            for B in args.batches:
                r = run(fl, B, bits, args.reps, args.windows)
                result["runs"].append(r)
                print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "window_ms"})
                                  for k, v in r.items()}), flush=True)
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
