"""Rates of the LWE key-switch and of GLWE -> LWE conversion on one GPU, both flavours, at the shapes of tests/test_gpu_lwe.py's bench-shape
tests, and the share of device time spent in the two layout kernels of lwe.cu (embed / extract).

    python scripts/lwe_time.py [--batch 2368] [--reps 200] [--windows 5] [--out FILE.json]

  lwe_keyswitch : N = 1024, LWE 512 -> 687 (bench.py's n_lwe), base2k 18, one limb in and out, key VmpPMat(1, 1, 2, 2)
  glwe_to_lwe   : N = 512, rank 3, base2k 18 (bench.py's CGGI configuration), one limb, LWE dimension 512, key VmpPMat(1, 3, 2, 2)

The keys are pinned (pgb_gadget_key_pin), as a caller holding a prepared key for its lifetime would.  Times come from CUDA events on the
module's stream (the module runs on torch's current stream), after every shape has been warmed up; a rate is the median over `windows`
windows of `reps` back-to-back calls.  The working set (a few MB) stays in L2 across calls, as it would between the rounds of a
bootstrap loop.  The layout share is measured with pgb_profile_*: the same number of calls of the composite and of its inner
pgb_glwe_keyswitch_batched alone on the staged shapes; the layout kernels are in the profiler's "other" category, so their time is the
difference of that category (the launch difference is printed to show that exactly those kernels are counted)."""
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

NCAT = 7
OTHER = 5


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], text=True)
        power, clock = [x.strip() for x in out.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        power, clock = "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def rand(rng, shape, k=18):
    return rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=shape, dtype=np.int64)


def key(m, rng, dnum, cols_in, cols_out, size):
    pm = m.vmp_pmat_alloc(dnum, cols_in, cols_out, size)
    m.vmp_prepare(pm, m.mat_znx_from_numpy(rand(rng, (dnum, cols_in, size, cols_out, m.n))))
    m.gadget_key_pin(pm)
    return pm


def rate(m, fn, B, reps, windows):
    for _ in range(3):
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
    ms = float(np.median(out))
    return {"ms_per_call": ms, "per_s": B / (ms * 1e-3), "window_ms": out}


def profile(m, fn, reps):
    ms, launches = (C.c_double * NCAT)(), (C.c_uint64 * NCAT)()
    lib().pgb_profile_enable(m._h, 1)
    lib().pgb_profile_read(m._h, ms, launches, 1)
    for _ in range(reps):
        fn()
    lib().pgb_profile_read(m._h, ms, launches, 1)
    lib().pgb_profile_enable(m._h, 0)
    return list(ms), list(launches)


def layout_split(m, composite, inner, reps):
    ms_c, l_c = profile(m, composite, reps)
    ms_i, l_i = profile(m, inner, reps)
    layout_ms = (ms_c[OTHER] - ms_i[OTHER]) / reps
    return {"layout_ms_per_call": layout_ms, "layout_launches_per_call": (l_c[OTHER] - l_i[OTHER]) / reps,
            "profiled_ms_per_call": sum(ms_c) / reps, "layout_share": layout_ms / (sum(ms_c) / reps)}


def run(fl, B, reps, windows):
    rng = np.random.default_rng(7)
    res = {}
    # LWE key-switch 512 -> 687 on N = 1024
    m = pb.Module(1024, fl)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    kk = key(m, rng, 1, 1, 2, 2)
    a = pb.DevBuf(B * 513 * 8)
    a.upload(rand(rng, (B, 1, 1, 513)))
    out = pb.DevBuf(B * 688 * 8)
    sc = [None]

    def ks():
        sc[0] = m.lwe_keyswitch(out, 687, 1, 18, a, 512, 1, 18, kk, 18, B, scratch=sc[0])

    g_in, g_out = m.vec_znx_from_numpy(rand(rng, (B, 1, 2, 1024))), m.vec_znx_alloc(2, 1, B)

    def ks_inner():
        sc[0] = m.glwe_keyswitch(g_out, 18, g_in, 18, kk, 18, scratch=sc[0])

    ks_inner()
    res["lwe_keyswitch"] = rate(m, ks, B, reps, windows)
    res["lwe_keyswitch"].update(layout_split(m, ks, ks_inner, reps))
    del m
    # GLWE (N = 512, rank 3) -> LWE 512
    m = pb.Module(512, fl)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    kg = key(m, rng, 1, 3, 2, 2)
    ga = m.vec_znx_from_numpy(rand(rng, (B, 1, 4, 512)))
    out = pb.DevBuf(B * 513 * 8)
    sc = [None]

    def g2l():
        sc[0] = m.glwe_to_lwe(out, 512, 1, 18, ga, 18, kg, 18, scratch=sc[0])

    g_out = m.vec_znx_alloc(2, 1, B)

    def g2l_inner():
        sc[0] = m.glwe_keyswitch(g_out, 18, ga, 18, kg, 18, scratch=sc[0])

    g2l_inner()
    res["glwe_to_lwe"] = rate(m, g2l, B, reps, windows)
    res["glwe_to_lwe"].update(layout_split(m, g2l, g2l_inner, reps))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=2368)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lwe_time.py measures on a GPU; none is visible")
    report = {"card": card(), "batch": args.batch, "reps": args.reps, "windows": args.windows}
    print(json.dumps(report["card"]), flush=True)
    for fl, name in ((pb.FFT64, "fft64"), (pb.NTT120, "ntt120")):
        r = run(fl, args.batch, args.reps, args.windows)
        report[name] = r
        for op, v in r.items():
            print(f"{name:7s} {op:14s} {v['per_s']:12.0f} /s  {v['ms_per_call'] * 1e3:9.1f} us/call  layout kernels "
                  f"{v['layout_ms_per_call'] * 1e3:7.1f} us/call ({v['layout_launches_per_call']:.0f} launches, "
                  f"{100 * v['layout_share']:.1f} % of profiled device time)", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
