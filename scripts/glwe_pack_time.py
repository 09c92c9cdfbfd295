"""Packing rates on one GPU: Module.glwe_pack (pgb_glwe_pack_batched) against circuit.glwe_pack over circuit.DeviceGlweOps, at n = 1024,
rank 1, base2k 13, GLWEs of 2 limbs, automorphism keys VmpPMat(2, 1, 2, 3) (one limb more than the GLWEs), dsize 1, both flavours, batches
512 and 4096, on three maps: a dense prefix of 9 (the 8-bit adder's outputs) and of 32 at gap 0, and the map of post_process with
log_domain 4 and log_gap_out 6 (inputs at i << 6, i < 16, then a trace over 6 rounds).

    python scripts/glwe_pack_time.py [--batches 512 4096] [--maps dense9 dense32 post_process] [--reps 3] [--windows 3] [--out FILE.json]

In one process it alternates, window by window, the entry and the composition, asserts that both give equal outputs, and reports both.
The composition consumes its map, so each of its calls starts with one device copy of the inputs (`pgb_memcpy_d2d_strided` on the module's stream, included in its time
and bytes).  Times come from CUDA events recorded on the module's stream (a torch stream of its own, set with Module.set_stream) after a
warm-up of both; a rate is the median over `windows` windows of `reps` back-to-back calls.  Inputs at batch 4096 are 4096 * n_in * 32 KiB
(1.2 GB for dense9, 4.3 GB for dense32), above the 126 MB of L2.  The card's name and power limit are read in the same run.

Algorithmic bytes per item, with g = one GLWE (n * 2 * 2 * 8 B = 32 KiB) and, per round i, nb pairs, nl lo-only and nh hi-only keys:
  entry:        sum_i (9 g nb + 4 g (nl + nh))   -- pair: prep reads lo, hi and writes x, y; automorphism reads x, writes z; combine reads
                                                    y, z and writes out.  lo / hi only: prep reads one and writes x; the op reads x,
                                                    writes out
  composition:  n_in g + sum_i (25 g nb + 5 g nl + 8 g nh)  -- the copy of the inputs, then per pair rotate (2), copy + sub (2 + 3), two
                                                    shifts (2 + 2), add (3), two normalisations (2 + 2), automorphism (2), sub (3),
                                                    rotate (2); lo only: shift (2), op (3); hi only: rotate (2), shift (2), op (3), and
                                                    the buffer swap's temporary (1)
  both:         + 4 g per trace round (shift 2, op 2) and one copy of the state into res (2 g)
Key bytes (one key read per automorphism call) are left out: they are shared by the batch.  bytes/s = batch * that / time."""
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

N, RANK, K, SIZE, KEY_ROWS, KEY_SIZE = 1024, 1, 13, 2, 2, 3
COLS = RANK + 1
LOG_N = 10
HBM_BYTES_PER_S = 7.7e12
MAPS = {"dense9": (list(range(9)), 0), "dense32": (list(range(32)), 0), "post_process": ([i << 6 for i in range(16)], 6)}


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


def plan(index, gap):
    """Per round (pairs, lo only, hi only), as the entry plans it."""
    cur, rounds = set(index), []
    for i in range(LOG_N - gap):
        t = N >> (i + 1)
        rounds.append((sum(1 for j in range(t) if j in cur and j + t in cur), sum(1 for j in range(t) if j in cur and j + t not in cur),
                       sum(1 for j in range(t) if j not in cur and j + t in cur)))
        cur = {k % t for k in cur}
    return rounds


def glwe_bytes(index, gap):
    g = N * COLS * SIZE * 8
    rounds = plan(index, gap)
    tail = 4 * g * gap + 2 * g
    entry = sum(9 * g * p + 4 * g * (lo + hi) for p, lo, hi in rounds) + tail
    comp = len(index) * g + sum(25 * g * p + 5 * g * lo + 8 * g * hi for p, lo, hi in rounds) + tail
    return {"entry": entry, "composition": comp}


def run(fl, name, B, reps, windows):
    index, gap = MAPS[name]
    n_in = len(index)
    rng = np.random.default_rng(B + fl + n_in)
    m = pb.Module(N, fl)
    stream = torch.cuda.Stream()  # not the legacy default stream, which does not order the module's non-blocking stream
    m.set_stream(stream.cuda_stream)
    keys = []
    for _ in range(LOG_N):
        pm = m.vmp_pmat_alloc(KEY_ROWS, RANK, COLS, KEY_SIZE)
        m.vmp_prepare(pm, m.mat_znx_from_numpy(rand(rng, (KEY_ROWS, RANK, KEY_SIZE, COLS, N))))
        keys.append(pm)
    g = N * COLS * SIZE * 8
    # the inputs, input-major (input j of item b at j * B g + b g): the entry reads them with entry_stride = B g and item stride g, and
    # input j is one contiguous batch for the composition
    src = pb.DevBuf(n_in * B * g)
    for j in range(n_in):
        src.upload(rand(rng, (B, SIZE, COLS, N)), offset=j * B * g)
    a = pb.hal.VecZnx(src, N, COLS, SIZE, batch=B, batch_stride=g)
    work = [m.vec_znx_alloc(COLS, SIZE, B) for _ in range(n_in)]
    res_new = m.vec_znx_alloc(COLS, SIZE, B)
    ops = circuit.DeviceGlweOps(m, keys, K, COLS, SIZE, B)
    res_old = ops.new()

    sc_new = m.glwe_pack(res_new, a, index, gap, keys, K, entry_stride=B * g)
    sc_new = pb.DevBuf(sc_new.nbytes)  # a scratch of its own, apart from the module's (which the composition's calls use)

    def new():
        m.glwe_pack(res_new, a, index, gap, keys, K, entry_stride=B * g, scratch=sc_new)

    def old():
        for j in range(n_in):
            assert lib().pgb_memcpy_d2d_strided(m._h, C.c_void_p(work[j].buf.ptr), C.c_uint64(B * g), C.c_void_p(src.ptr + j * B * g),
                                                C.c_uint64(B * g), C.c_uint64(B * g), C.c_uint64(1)) == 0
        circuit.glwe_pack(ops, res_old, {i: work[j] for j, i in enumerate(index)}, gap)

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
    by = glwe_bytes(index, gap)
    out = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "map": name, "n_in": n_in, "log_gap_out": gap, "rounds": plan(index, gap),
           "batch": B, "entry_scratch_bytes": sc_new.nbytes}
    for nm, launches in (("entry", l1 - l0), ("composition", l2 - l1)):
        ms = float(np.median(win[nm]))
        out[nm] = {"ms_per_call": ms, "packs_per_s": B / (ms * 1e-3), "bytes_per_pack": by[nm], "bytes_per_s": by[nm] * B / (ms * 1e-3),
                   "hbm_fraction": by[nm] * B / (ms * 1e-3) / HBM_BYTES_PER_S, "launches_per_call": launches, "window_ms": win[nm]}
    out["composition_over_entry"] = out["composition"]["ms_per_call"] / out["entry"]["ms_per_call"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--maps", nargs="+", default=list(MAPS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    for name in args.maps:
        index, gap = MAPS[name]
        print(json.dumps({"map": name, "rounds": plan(index, gap), "glwe_bytes_per_pack": glwe_bytes(index, gap)}), flush=True)
    if not torch.cuda.is_available():
        sys.exit("glwe_pack_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "glwe_size": SIZE, "key_rows": KEY_ROWS, "key_size": KEY_SIZE},
              "runs": []}
    for fl in (pb.NTT120, pb.FFT64):
        for name in args.maps:
            for B in args.batches:
                r = run(fl, name, B, args.reps, args.windows)
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
