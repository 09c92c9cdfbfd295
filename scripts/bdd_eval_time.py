"""BDD-evaluator rates on one GPU at the circuit-bootstrapping bench shape (n = 1024, rank 2, base2k 13, GGSW selectors VmpPMat(2, 3, 3, 2),
GLWEs of 2 limbs), both flavours, on the 8-bit adder (x + y, 9 outputs: 65 nodes, 16 levels) and the 8-bit comparison x < y (23 nodes,
16 levels), built by circuit.bdd_from_truth_tables with the bits of x and y interleaved, most significant first; batches 512 and 4096,
two leaves shared by the batch, per-item selectors in the bit-major layout of circuit.prepare_ggsw.

    python scripts/bdd_eval_time.py [--batches 512 4096] [--circuits add8 lt8] [--reps 3] [--windows 3] [--out FILE.json]

In one process it alternates, window by window, Module.glwe_bdd_eval with today's composition (one glwe_cmux per node over the whole
batch, level by level, every node's output kept, then one glwe_copy per output), asserts that both give equal outputs, and reports both.
Times come from CUDA events recorded on the module's stream (a torch stream of its own, set with Module.set_stream) after a warm-up of
both; a rate is the median over `windows` windows of `reps` back-to-back calls.  The selectors are B * 16 prepared GGSWs (at batch
4096 38.7 GB NTT120 / 19.3 GB FFT64, at 512 4.8 GB / 2.4 GB), all above the 126 MB of L2; 64 distinct GGSWs are prepared and replicated
on the device.  The card's name and power limit are read in the same run.

Algorithmic bytes of one evaluation (one item), with sel = one prepared GGSW (dnum*cols*cols*S*n*pb; pb = 16 B NTT120 / 8 B FFT64) and
c = the bytes of one per-item CMux without its selector (the formula of scripts/cmux_tree_time.py):
  entry:        levels * sel + nodes * c      -- each item's selector once per level
  composition:  nodes * (sel + c)             -- each item's selector once per node
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
from poulpy_b200 import circuit  # noqa: E402
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


def composition(m, res, states, leaves, c, sel, B, n_out):
    """glwe_cmux(state[n_leaves + k], state[t_k], state[f_k], s_{bit}) for every node in level order, then the outputs copied."""
    item, es, g = sel.batch_stride, N * COLS * SIZE * 8, N * COLS * SIZE * 8
    st = [pb.hal.VecZnx(leaves.buf, N, COLS, SIZE, offset=leaves.offset + j * es) for j in range(len(c.leaves))]
    k = 0
    for bit, nodes in c.levels:
        s = pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S, offset=bit * item, batch=B, batch_stride=16 * item)
        for t, f in nodes:
            m.glwe_cmux(states[k], st[t], st[f], K, s, K)
            st.append(states[k])
            k += 1
    for o, s_ in enumerate(c.outputs):
        src = st[s_]
        if src.batch > 1:
            circuit._glwe_copy(m, res.ptr + o * g, n_out * g, SIZE, src.ptr, g, SIZE, COLS, B)
        else:  # a leaf shared by the batch
            for b in range(B):
                circuit._glwe_copy(m, res.ptr + (b * n_out + o) * g, 0, SIZE, src.ptr, 0, SIZE, COLS, 1)


def circuits():
    x = np.arange(1 << 16)
    xs, ys = x & 255, x >> 8
    order = [v for i in range(7, -1, -1) for v in (i, i + 8)]
    return {"add8": circuit.bdd_from_truth_tables([((xs + ys) >> i) & 1 for i in range(9)], 16, order),
            "lt8": circuit.bdd_from_truth_tables([(xs < ys).astype(np.int64)], 16, order)}


def run(fl, name, c, B, reps, windows):
    rng = np.random.default_rng(B + fl + len(name))
    m = pb.Module(N, fl)
    stream = torch.cuda.Stream()  # not the legacy default stream, which does not order the module's non-blocking stream
    m.set_stream(stream.cuda_stream)
    bits = 16
    sel = selectors(m, rng, B * bits)
    lv = m.vec_znx_from_numpy(rand(rng, (len(c.leaves), SIZE, COLS, N)))
    leaves = pb.hal.VecZnx(lv.buf, N, COLS, SIZE)  # shared by the batch
    n_out = len(c.outputs)
    res_new, res_old = m.vec_znx_alloc(COLS, SIZE, B * n_out), m.vec_znx_alloc(COLS, SIZE, B * n_out)
    states = [m.vec_znx_alloc(COLS, SIZE, B) for _ in range(c.n_nodes)]

    sc_new = m.glwe_bdd_eval(res_new, leaves, c, K, bits, sel, K)
    sc_new = pb.DevBuf(sc_new.nbytes)  # a scratch of its own, apart from the module's (which the composition's CMuxes use)

    def new():
        m.glwe_bdd_eval(res_new, leaves, c, K, bits, sel, K, scratch=sc_new)

    def old():
        composition(m, res_old, states, leaves, c, sel, B, n_out)

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
        for nm, fn in (("entry", new), ("composition", old)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            e1.synchronize()
            win[nm].append(e0.elapsed_time(e1) / reps)
    assert np.array_equal(m.vec_znx_to_numpy(res_new), m.vec_znx_to_numpy(res_old)), "the entry and the composition differ"
    nodes, levels = c.n_nodes, len(c.levels)
    by = {"entry": levels * sel_bytes(fl) + nodes * cmux_other_bytes(fl), "composition": nodes * (sel_bytes(fl) + cmux_other_bytes(fl))}
    out = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "circuit": name, "nodes": nodes, "levels": levels, "batch": B,
           "selector_bytes": B * bits * sel.batch_stride, "entry_scratch_bytes": sc_new.nbytes}
    for nm, launches in (("entry", l1 - l0), ("composition", l2 - l1)):
        ms = float(np.median(win[nm]))
        out[nm] = {"ms_per_call": ms, "evals_per_s": B / (ms * 1e-3), "bytes_per_eval": by[nm], "bytes_per_s": by[nm] * B / (ms * 1e-3),
                   "hbm_fraction": by[nm] * B / (ms * 1e-3) / HBM_BYTES_PER_S, "launches_per_call": launches, "window_ms": win[nm]}
    out["composition_over_entry"] = out["composition"]["ms_per_call"] / out["entry"]["ms_per_call"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--circuits", nargs="+", default=["add8", "lt8"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bdd_eval_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "dnum": DNUM, "ggsw_size": S, "glwe_size": SIZE}, "runs": []}
    cs = circuits()
    for fl in (pb.NTT120, pb.FFT64):
        for name in args.circuits:
            for B in args.batches:
                r = run(fl, name, cs[name], B, args.reps, args.windows)
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
