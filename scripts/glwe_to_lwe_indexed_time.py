"""Rates of glwe_to_lwe at many coefficients on one GPU: Module.glwe_to_lwe_indexed (pgb_glwe_to_lwe_indexed_batched, one key-switch per
item) against the twin composition (one glwe_keyswitch, then per index one batched rotation per column and one lwe_sample_extract) and
the per-bit composition (per index, rotate the input GLWEs and run a whole glwe_to_lwe: n_index key-switches per item), at the
circuit-bootstrapping bench shape (cbt_time.py): n = 1024, rank 2, base2k 13, packed GLWEs of 2 limbs, key VmpPMat(2, 2, 2, 3), LWEs of
dimension 574 and one limb, n_index 9 and 32, batches 512 and 4096, both flavours.

    python scripts/glwe_to_lwe_indexed_time.py [--batches 512 4096] [--n-index 9 32] [--reps 5] [--windows 3] [--share-max 20000] [--out F]

In one process it alternates, window by window, the three, asserts that the entry and the twin give equal outputs (the per-bit
composition is not bit-identical: the key-switch and the rotation do not commute through the final rounding), and reports all three.
Times come from CUDA events on the module's stream (a torch stream of its own) after a warm-up; a rate is the median over `windows`
windows of `reps` back-to-back calls.  The entry's share of one circuit.ggsw_bits_from_packed call (the entry, circuit bootstrapping of
batch * n_index LWEs with random keys of the bench shape, prepare_ggsw) is timed once after a warm-up, where batch * n_index is at most
--share-max (circuit bootstrapping takes at most 65535 LWEs per call).  The card's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import poulpy_b200 as pb  # noqa: E402
from poulpy_b200 import circuit  # noqa: E402
from poulpy_b200.hal import _BT, lib  # noqa: E402

N, LOG_N, RANK, K, SIZE, N_LWE, LWE_SIZE = 1024, 10, 2, 13, 2, 574, 1
COLS = RANK + 1
BLOCK, KEY_ROWS, KEY_SIZE, DNUM_RES, RES_SIZE, LOG_DOMAIN = 7, 3, 4, 2, 2, 1


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


def prep(m, rng, rows, cols_in, cols_out, size):
    pm = m.vmp_pmat_alloc(rows, cols_in, cols_out, size)
    m.vmp_prepare(pm, m.mat_znx_from_numpy(rand(rng, (rows, cols_in, size, cols_out, N))))
    return pm


def events(stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def run(fl, B, n_index, reps, windows, share_max):
    rng = np.random.default_rng(B + n_index + fl)
    m = pb.Module(N, fl)
    stream = torch.cuda.Stream()  # not the legacy default stream, which does not order the module's non-blocking stream
    m.set_stream(stream.cuda_stream)
    key = prep(m, rng, SIZE, RANK, 2, SIZE + 1)
    index = [int(x) for x in rng.choice(N, size=n_index, replace=False)]
    a = m.vec_znx_from_numpy(rand(rng, (B, SIZE, COLS, N)))
    lwe = LWE_SIZE * (N_LWE + 1) * 8
    out = {name: pb.DevBuf(B * n_index * lwe) for name in ("entry", "twin", "per_bit")}
    staged, rot, rot_a = m.vec_znx_alloc(2, LWE_SIZE, B), m.vec_znx_alloc(2, LWE_SIZE, B), m.vec_znx_alloc(COLS, SIZE, B)
    sc = m.glwe_to_lwe_indexed(out["entry"], N_LWE, LWE_SIZE, K, a, K, index, key, K)
    sc = pb.DevBuf(sc.nbytes)  # a scratch of its own, apart from the module's (which the compositions' calls use)

    def rotate(dst, src, p, cols):
        r, s = dst.struct(), src.struct()
        bt = _BT(B, dst.batch_stride, src.batch_stride, 0)
        for c in range(cols):
            pb.hal._check(lib().pgb_vec_znx_rotate_batched(m._h, C.c_int64(p), C.byref(r), C.c_uint64(c), C.byref(s), C.c_uint64(c), C.byref(bt)))

    def at(name, j):
        return types.SimpleNamespace(ptr=out[name].ptr + j * lwe)

    def entry():
        m.glwe_to_lwe_indexed(out["entry"], N_LWE, LWE_SIZE, K, a, K, index, key, K, scratch=sc)

    def twin():
        m.glwe_keyswitch(staged, K, a, K, key, K)
        for j, idx in enumerate(index):
            rotate(rot, staged, -idx, 2)
            m.lwe_sample_extract(at("twin", j), N_LWE, LWE_SIZE, rot, res_stride=n_index * lwe)

    def per_bit():
        for j, idx in enumerate(index):
            rotate(rot_a, a, -idx, COLS)
            m.glwe_to_lwe(at("per_bit", j), N_LWE, LWE_SIZE, K, rot_a, K, key, K, res_stride=n_index * lwe)

    fns = {"entry": entry, "twin": twin, "per_bit": per_bit}
    launches = {}
    for name, fn in fns.items():
        l0 = m.launch_count
        fn()
        m.sync()
        launches[name] = m.launch_count - l0
    words = B * n_index * lwe // 8

    def same():
        return np.array_equal(out["entry"].download(np.int64, (words,)), out["twin"].download(np.int64, (words,)))

    assert same(), "the entry and the twin differ"
    for fn in fns.values():
        fn()
    m.sync()
    win = {name: [] for name in fns}
    for _ in range(windows):
        for name, fn in fns.items():
            win[name].append(events(stream, fn, reps))
    assert same(), "the entry and the twin differ"
    res = {"flavour": "NTT120" if fl == pb.NTT120 else "FFT64", "batch": B, "n_index": n_index}
    for name in fns:
        ms = float(np.median(win[name]))
        res[name] = {"ms_per_call": ms, "lwes_per_s": B * n_index / (ms * 1e-3), "launches_per_call": launches[name], "window_ms": win[name]}
    res["twin_over_entry"] = res["twin"]["ms_per_call"] / res["entry"]["ms_per_call"]
    res["per_bit_over_entry"] = res["per_bit"]["ms_per_call"] / res["entry"]["ms_per_call"]
    if B * n_index <= share_max:
        per = N * COLS * COLS * KEY_ROWS * KEY_SIZE * m.prep_bytes
        brk_buf = pb.DevBuf(per * N_LWE)
        brk = pb.hal.VmpPMat(brk_buf, N, KEY_ROWS, COLS, COLS, KEY_SIZE)
        m.vmp_prepare(brk, m.mat_znx_from_numpy(rand(rng, (KEY_ROWS, COLS, KEY_SIZE, COLS, N))))
        for i in range(1, N_LWE):
            lib().pgb_memcpy_d2d(C.c_void_p(brk_buf.ptr + i * per), C.c_void_p(brk_buf.ptr), C.c_size_t(per))
        atk = [prep(m, rng, KEY_ROWS, RANK, COLS, KEY_SIZE) for _ in range(LOG_N)]
        tsk = [prep(m, rng, KEY_ROWS, RANK, COLS, KEY_SIZE) for _ in range(RANK)]
        lwe_key = prep(m, rng, SIZE, RANK, 2, SIZE + 1)
        xpa = m.cggi_x_pow_a()

        def full():
            return circuit.ggsw_bits_from_packed(m, a, index, lwe_key, N_LWE, LWE_SIZE, brk, xpa, BLOCK, atk, tsk, K, RANK, DNUM_RES, RES_SIZE,
                                                 LOG_DOMAIN)

        full()
        m.sync()
        ms = events(stream, full, 1)
        res["ggsw_bits_from_packed_ms"] = ms
        res["entry_share"] = res["entry"]["ms_per_call"] / ms
    else:
        res["ggsw_bits_from_packed_ms"] = None  # not measured: batch * n_index above --share-max
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--n-index", type=int, nargs="+", default=[9, 32])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--share-max", type=int, default=20000)
    ap.add_argument("--flavours", nargs="+", default=["ntt120", "fft64"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("glwe_to_lwe_indexed_time.py needs a CUDA device")
    result = {"card": card(), "shape": {"n": N, "rank": RANK, "base2k": K, "glwe_size": SIZE, "key": [SIZE, RANK, 2, SIZE + 1],
                                        "n_lwe": N_LWE, "lwe_size": LWE_SIZE}, "runs": []}
    print(json.dumps(result["card"]), flush=True)
    for fl in [pb.NTT120 if f == "ntt120" else pb.FFT64 for f in args.flavours]:
        for n_index in args.n_index:
            for B in args.batches:
                r = run(fl, B, n_index, args.reps, args.windows, args.share_max)
                result["runs"].append(r)
                print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "window_ms"})
                                  for k, v in r.items()}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
