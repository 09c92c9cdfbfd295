"""CMux rates on one GPU at the circuit-bootstrapping bench shape (n = 1024, rank 2, base2k 13, GGSW selectors VmpPMat(2, 3, 3, 2), GLWEs
of 2 limbs), both flavours, batches 512 and 4096: per-item and shared selectors, default routes and PGB_OPT_NO_FUSION; the batched GGSW
preparation against a loop of single prepares (time and launches); algorithmic bytes per CMux and the achieved fraction of the B200's
data-sheet HBM bandwidth (7.7 TB/s).

    python scripts/cmux_time.py [--batches 512 4096] [--reps 20] [--windows 5] [--out FILE.json]

Times come from CUDA events on the module's stream (the module runs on torch's current stream) after a warm-up of every timed call; a rate
is the median over `windows` windows of `reps` back-to-back calls.  Per-item selectors: 512 of them are 302 MB (NTT120) / 151 MB (FFT64),
4096 are 2.4 GB / 1.2 GB, all above the 126 MB of L2, so each call streams them from HBM.  The card's name and power limit are read in the
same run.

Algorithmic bytes of one per-item CMux (what the route has to move, each buffer once; pb = 16 B NTT120 / 8 B FFT64, g = n * cols * 8 B per
i64 limb):
  NTT120 fused:  selector dnum*cols*cols*S*n*pb + t, f (2 * size g) + d written and read (2 * size g) + a_dft written and read
                 (2 * size * n * cols * pb) + f again (size g, added in the back end) + res (size g)
  FFT64 fused:   selector + t, f + d written and read + f written into res (size g) + a_dft written and read + res_dft written and read
                 (2 * cols * S * n * pb) + res read and written (2 * size g)
Shared selectors: the same without the selector (read once per batch)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import poulpy_b200 as pb  # noqa: E402

N, RANK, K, DNUM, S, SIZE = 1024, 2, 13, 2, 2, 2
COLS = RANK + 1
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


def timed(m, fn, reps, windows):
    for _ in range(2):
        fn()
    m.sync()
    out = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / reps)
    return float(np.median(out)), out


def cmux_bytes(fl, per_item):
    pb_ = 16 if fl == pb.NTT120 else 8
    g = N * COLS * 8
    sel = DNUM * COLS * COLS * S * N * pb_ if per_item else 0
    if fl == pb.NTT120:
        return sel + 2 * SIZE * g + 2 * SIZE * g + 2 * SIZE * N * COLS * pb_ + SIZE * g + SIZE * g
    return sel + 2 * SIZE * g + 2 * SIZE * g + SIZE * g + 2 * SIZE * N * COLS * pb_ + 2 * COLS * S * N * pb_ + 2 * SIZE * g


def run(fl, B, reps, windows):
    rng = np.random.default_rng(B + fl)
    m = pb.Module(N, fl)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    out = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "batch": B}
    # selectors: MatZnx batch -> batched prepare, and the same through single prepares
    mat_item = DNUM * COLS * COLS * S * N * 8
    mats = pb.DevBuf(B * mat_item)
    for b0 in range(0, B, 256):
        nb = min(256, B - b0)
        mats.upload(rand(rng, (nb, DNUM, COLS, S, COLS, N)), b0 * mat_item)
    mat = pb.hal.MatZnx(mats, N, DNUM, COLS, COLS, S, batch=B, batch_stride=mat_item)
    sel = m.vmp_pmat_alloc(DNUM, COLS, COLS, S, batch=B)
    singles = [(pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S, offset=b * sel.batch_stride),
                pb.hal.MatZnx(mats, N, DNUM, COLS, COLS, S, offset=b * mat_item)) for b in range(B)]
    l0 = m.launch_count
    m.vmp_prepare_batched(sel, mat)
    m.sync()
    l1 = m.launch_count
    for p, a in singles:
        m.vmp_prepare(p, a)
    l2 = m.launch_count
    ms_b, _ = timed(m, lambda: m.vmp_prepare_batched(sel, mat), max(1, reps // 4), windows)

    def loop():
        for p, a in singles:
            m.vmp_prepare(p, a)

    ms_l, _ = timed(m, loop, 1, max(1, windows // 2))
    out["prepare"] = {"batched_ms": ms_b, "loop_ms": ms_l, "batched_launches": l1 - l0, "loop_launches": l2 - l1,
                      "speedup": ms_l / ms_b}
    t = m.vec_znx_from_numpy(rand(rng, (B, SIZE, COLS, N)))
    f = m.vec_znx_from_numpy(rand(rng, (B, SIZE, COLS, N)))
    res = m.vec_znx_alloc(COLS, SIZE, B)
    shared = pb.hal.VmpPMat(sel.buf, N, DNUM, COLS, COLS, S)
    sc = [None]
    for name, s in (("per_item", sel), ("shared", shared)):
        for nf in (0, 1):
            m.set_option(pb.hal.OPT_NO_FUSION, nf)
            a = m.launch_count
            sc[0] = m.glwe_cmux(res, t, f, K, s, K, scratch=sc[0])
            m.sync()
            launches = m.launch_count - a
            ms, win = timed(m, lambda: m.glwe_cmux(res, t, f, K, s, K, scratch=sc[0]), reps, windows)
            by = cmux_bytes(fl, name == "per_item")
            key = f"{name}_{'no_fusion' if nf else 'default'}"
            out[key] = {"ms_per_call": ms, "cmux_per_s": B / (ms * 1e-3), "launches_per_call": launches, "bytes_per_cmux": by,
                        "hbm_fraction": by * B / (ms * 1e-3) / HBM_BYTES_PER_S, "window_ms": win}
    m.set_option(pb.hal.OPT_NO_FUSION, 0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cmux_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "dnum": DNUM, "ggsw_size": S, "glwe_size": SIZE}, "runs": []}
    for fl in (pb.NTT120, pb.FFT64):
        for B in args.batches:
            r = run(fl, B, args.reps, args.windows)
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
