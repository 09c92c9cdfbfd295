#!/usr/bin/env python
"""bench.py -- headline benchmark of the poulpy-hal hot path on B200 (contract: see the task statement).

Workload (config.workload): GLWE key-switch, NTT120 flavour, the reference's own bench defaults
(poulpy-bench/src/params.rs:112-121, poulpy-bench/benches/keyswitch.rs): n=4096, base2k=18, k=54 (3 limbs), rank=1,
dsize=1, dnum=3, key k=72 (4 limbs); a batch of independent ciphertexts against one prepared key.
One "step" = one pass of the hot path over one batch.  Inputs are synthetic uniform digits (the reference's HAL benches
use random bytes, poulpy-bench/src/bench_suite/hal/vmp.rs:154-156).

  value : key-switches/s, inputs resident in HBM, all N ranks (batch sharded, key replicated, no collective)
  e2e   : same metric through pgb_glwe_keyswitch_host with pinned HOST buffers (H2D + compute + D2H in the timed region)
  roofline : dominant kernel, algorithmic bytes / CUDA-event time vs the measured HBM copy bandwidth
  cpu_baseline : the oracle port (C restatement of poulpy-cpu-ref) on the box's host cores, bounded sample

`--impl reference` times that CPU port alone (the Rust reference cannot be built in this image).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NCAT = 7  # PGB_PROFILE_NCAT (include/poulpy_b200.h)
WORK = dict(n=4096, base2k=18, a_size=3, key_size=4, rank=1, dnum=3, dsize=1)


def make_inputs(batch, seed):
    w = WORK
    rng = np.random.default_rng(seed)
    lo, hi = -(1 << (w["base2k"] - 1)), 1 << (w["base2k"] - 1)
    a = rng.integers(lo, hi, size=(batch, w["a_size"], w["rank"] + 1, w["n"]), dtype=np.int64)
    mat = np.random.default_rng(1234).integers(lo, hi, size=(w["dnum"], w["rank"], w["key_size"], w["rank"] + 1, w["n"]), dtype=np.int64)
    return a, mat


DUMP_ROWS = 256  # ciphertexts --dump-outputs writes: 256 x 3 limbs x 2 columns x 4096 coefficients in float64 = 48 MiB


def dump_rows(batch):
    """Indices of the ciphertexts --dump-outputs writes: a fixed, seeded sample of the batch, in ascending order."""
    if batch <= DUMP_ROWS:
        return np.arange(batch)
    return np.sort(np.random.default_rng(2024).choice(batch, DUMP_ROWS, replace=False))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with NVML while the timed region runs."""

    def __init__(self, device):
        self.device, self.samples, self.reasons, self.stop = device, [], set(), False
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80}
        while not self.stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.nv:
            self.t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_port(sample_target_cpu_s=15.0, threads=0, simd=False):
    """Times the oracle port on the host cores on a bounded sample of the same workload.  simd = False: scalar restatement of
    poulpy-cpu-ref; simd = True: the same port with the "cpu-avx-style" data path (four primes per __m256i for the NTT butterflies and
    the bbc products, poulpy-cpu-avx/src/ntt120/ntt.rs:81-110) -- bit-identical values, tests/test_oracle_kat.py."""
    from oracle import pyoracle as O

    w = WORK
    threads = threads or O.num_threads()
    O.ntt120_set_simd(simd)
    try:
        om = O.OracleModule(w["n"], O.NTT120)
        a, mat = make_inputs(4 * threads, 99)
        pm = om.vmp_pmat_alloc(w["dnum"], w["rank"], w["rank"] + 1, w["key_size"])
        om.vmp_prepare(pm, mat)
        res = np.zeros_like(a)
        t0 = time.perf_counter()
        om.glwe_keyswitch_batch(res, w["base2k"], a, w["base2k"], pm, w["base2k"], w["dsize"], threads=threads)
        per_ks_cpu_s = (time.perf_counter() - t0) * threads / a.shape[0]
        count = int(max(4 * threads, min(sample_target_cpu_s / per_ks_cpu_s, 200000)))
        count -= count % threads
        a, _ = make_inputs(count, 98)
        res = np.zeros_like(a)
        t0 = time.perf_counter()
        om.glwe_keyswitch_batch(res, w["base2k"], a, w["base2k"], pm, w["base2k"], w["dsize"], threads=threads)
        dt = time.perf_counter() - t0
    finally:
        O.ntt120_set_simd(False)
    what = ("oracle C port with the cpu-avx-style AVX2 data path (4 primes per __m256i NTT + bbc; restates poulpy-cpu-avx's NTT120 kernels)"
            if simd else "oracle C port (restates poulpy-cpu-ref NTT120, scalar)")
    return {"value": count / dt, "unit": "keyswitch/s", "cores": threads, "kind": "port", "simd": "avx2" if simd else "scalar",
            "sample": f"{count} key-switches of the bench workload, {what}, {threads} threads"}, om, pm


def config_dict(batch, n_gpus):
    w = WORK
    return {"workload": "glwe_keyswitch ntt120 n=4096 base2k=18 k=54 rank=1 dsize=1 dnum=3 key_k=72 (poulpy-bench keyswitch defaults)",
            "batch_per_gpu": batch, "global_batch": batch * n_gpus, "flavour": "ntt120", "parallelism": f"batch-sharded x{n_gpus}, key replicated",
            "l2": "inputs larger than L2 (batch * 196 KB in, 196 KB out per pass)", **w}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path on the host cores.  The Rust reference cannot be built in this
    image (DESIGN.md section 1), so this is the oracle port: scalar (poulpy-cpu-ref) and with the AVX2 data path (poulpy-cpu-avx style);
    `value` is the FASTER of the two, both are reported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as O

    w = WORK
    threads = O.num_threads()
    total = args.steps + args.warmup
    lines = {}
    for simd in (False, True):
        O.ntt120_set_simd(simd)
        try:
            om = O.OracleModule(w["n"], O.NTT120)
            a, mat = make_inputs(8 * threads, 7)
            pm = om.vmp_pmat_alloc(w["dnum"], w["rank"], w["rank"] + 1, w["key_size"])
            om.vmp_prepare(pm, mat)
            res = np.zeros_like(a)
            t0 = time.perf_counter()
            om.glwe_keyswitch_batch(res, w["base2k"], a, w["base2k"], pm, w["base2k"], w["dsize"], threads=threads)
            per = (time.perf_counter() - t0) / a.shape[0]
            per_step = int(max(threads, min(60.0 / total, 2.0) / per))  # each step <= 2 s per variant, whole run within ~2 minutes
            per_step -= per_step % threads
            a, _ = make_inputs(per_step, 8)
            res = np.zeros_like(a)
            for _ in range(args.warmup):
                om.glwe_keyswitch_batch(res, w["base2k"], a, w["base2k"], pm, w["base2k"], w["dsize"], threads=threads)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                om.glwe_keyswitch_batch(res, w["base2k"], a, w["base2k"], pm, w["base2k"], w["dsize"], threads=threads)
            dt = time.perf_counter() - t0
        finally:
            O.ntt120_set_simd(False)
        name = "avx2" if simd else "scalar"
        lines[name] = {"value": per_step * args.steps / dt, "unit": "keyswitch/s", "cores": threads, "kind": "port", "simd": name,
                       "ms_per_step": dt / args.steps * 1e3, "per_step": per_step,
                       "sample": f"{per_step} key-switches per step, oracle C port ({'cpu-avx-style AVX2 data path' if simd else 'scalar, poulpy-cpu-ref'}; "
                                 f"Rust reference not buildable here), {threads} threads"}
    best = max(lines.values(), key=lambda d: d["value"])
    v = best["value"]
    print(json.dumps({
        "impl": "reference", "metric": "glwe_keyswitch_per_s", "value": v, "unit": "keyswitch/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": best["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 (lazy q120b residues)", "data": "synthetic", "config": config_dict(best["per_step"], 1),
        "cpu_baseline": {k: best[k] for k in ("value", "unit", "cores", "kind", "simd", "sample")},
        "cpu_baseline_scalar": lines["scalar"], "cpu_baseline_avx": lines["avx2"],
        "e2e": {"value": v, "unit": "keyswitch/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=4096, help="ciphertexts per GPU per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-aux", action="store_true", help="skip the auxiliary measurements")
    ap.add_argument("--no-cggi", action="store_true", help="skip the CGGI bootstraps/s object")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the key-switch results of the last timed step (rank 0, a fixed seeded sample of the batch) to "
                         "DIR/glwe_keyswitch.npy as float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU implementation only")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    # Libraries write to fd 1 behind Python's back (NCCL prints its version banner there): stdout must carry the ONE JSON line only, so
    # fd 1 is pointed at stderr for the whole run and the line goes to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist

    import poulpy_b200 as pb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w, B = WORK, args.batch
    m = pb.Module(w["n"], pb.NTT120, device=local)
    stream = torch.cuda.Stream(device=local)
    m.set_stream(stream.cuda_stream)

    a_np, mat = make_inputs(B, 1000 + rank)
    pmat = m.vmp_pmat_alloc(w["dnum"], w["rank"], w["rank"] + 1, w["key_size"])
    # setup, not timed: the key is prepared on rank 0 and replicated to the other GPUs over NCCL (SURVEY 8e; the prepared layout is
    # plain bytes); the hot path itself never communicates
    from poulpy_b200.sharding import broadcast_prepared, replicate_prepared

    how = replicate_prepared(lambda: m.vmp_prepare(pmat, m.mat_znx_from_numpy(mat)), lambda: broadcast_prepared(m, pmat.buf))
    if world > 1:  # every rank must hold the same bytes (a CRC per rank, compared everywhere); a mismatch falls back to a local prepare
        import zlib

        probes = [None] * world
        dist.all_gather_object(probes, zlib.crc32(pmat.buf.download(np.uint8, (pmat.buf.nbytes,)).tobytes()))
        if len(set(probes)) != 1:
            print("[bench] replicated key differs across ranks; preparing it on every rank", file=sys.stderr)
            m.vmp_prepare(pmat, m.mat_znx_from_numpy(mat))
            how = "local"
    m.gadget_key_pin(pmat)  # the prepared key is immutable for the whole run (a GGLWEPrepared in the reference): derive its gadget forms once
    a_dev = m.vec_znx_from_numpy(a_np)
    res_dev = m.vec_znx_alloc(w["rank"] + 1, w["a_size"], B)
    scratch = None
    k = w["base2k"]

    def step():
        nonlocal scratch
        scratch = m.glwe_keyswitch(res_dev, k, a_dev, k, pmat, k, w["dsize"], scratch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    import ctypes as C

    lib = pb.lib()
    lib.pgb_profile_enable(m._h, 1)
    launches0 = m.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as cs:
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for _ in range(args.steps):
                step()
            ev1.record(stream)
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    prof_ms = (C.c_double * NCAT)()
    prof_n = (C.c_uint64 * NCAT)()
    lib.pgb_profile_read(m._h, prof_ms, prof_n, 1)
    lib.pgb_profile_enable(m._h, 0)
    launches = m.launch_count - launches0
    barrier()
    t = torch.tensor([ms], device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max * 1e-3)

    # ---- e2e: host buffers, copies inside the timed region --------------------------------------------------------
    a_host = pb.pinned_empty(a_np.shape)
    a_host[:] = a_np
    r_host = pb.pinned_empty(a_np.shape)
    e2e_steps = max(3, min(args.steps, 10))
    m.glwe_keyswitch_host(r_host, k, a_host, k, pmat, k, w["dsize"])  # warm-up (allocates staging)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        m.glwe_keyswitch_host(r_host, k, a_host, k, pmat, k, w["dsize"])  # synchronous: returns when r_host is complete
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / float(t.item())
    check = m.vec_znx_to_numpy(res_dev)
    assert np.array_equal(check, r_host), "device-resident and host-path results differ"
    if args.dump_outputs and rank == 0:
        # res_dev still holds the last timed step (the e2e leg writes r_host only); normalised digits are exact in float64
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "glwe_keyswitch.npy"), check[dump_rows(B)].astype(np.float64))

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------------
    n = w["n"]
    cols_out, R, Cc = w["rank"] + 1, w["dnum"] * w["rank"], (w["rank"] + 1) * w["key_size"]
    key_bytes = R * Cc * 16 * n
    glwe_bytes = (w["rank"] + 1) * w["a_size"] * 8 * n
    bytes_per_launch = {
        # single-kernel gadget product: GLWE in (mask limbs + body limbs) + GLWE out, collapsed key once (fused minimum, SURVEY 8d)
        "gadget_fused": B * 2 * glwe_bytes + R * cols_out * 16 * n,
        "dft_forward": B * w["a_size"] * (8 * n + 16 * n),                # i64 limb in, 16 B/coef DFT limb out (per-limb route only)
        "dft_inverse": B * (R * 16 * n + w["a_size"] * 8 * n + cols_out * w["a_size"] * 8 * n) + key_bytes,
        "vmp_apply": B * (R + Cc) * 16 * n + key_bytes,                   # only on the unfused path
        "normalize": B * (w["key_size"] * 16 * n + w["a_size"] * 8 * n),  # only on the unfused path
        "elementwise": B * (2 * 16 * n + 8 * n),                          # only on the unfused path
    }
    kernel_names = {"gadget_fused": "ntt120_gadget_kernel<12> (dft + vmp + idft + CRT + add_small + normalize, one launch per batch)",
                    "dft_forward": "ntt120_fwd_kernel<12,1>", "dft_inverse": "ntt120_fused_back_kernel<12> (vmp+intt+crt+add_small+normalize)"}
    lib.pgb_profile_category_name.restype = C.c_char_p
    names = [lib.pgb_profile_category_name(i).decode() for i in range(NCAT)]
    peak, peak_src = peaks()
    kernels = {}
    for i, nm in enumerate(names):
        if prof_n[i] == 0:
            continue
        avg_ms = prof_ms[i] / prof_n[i]
        d = {"launches": int(prof_n[i]), "avg_ms": avg_ms, "share_of_step": prof_ms[i] / ms}
        if nm in bytes_per_launch and d["share_of_step"] > 0.05:
            d["algorithmic_bytes_per_launch"] = bytes_per_launch[nm]
            d["achieved_gbs"] = bytes_per_launch[nm] / (avg_ms * 1e-3) / 1e9
            d["frac_of_hbm_peak"] = d["achieved_gbs"] / peak
        kernels[nm] = d
    dom = max((k_ for k_ in kernels if "achieved_gbs" in kernels[k_]), key=lambda k_: kernels[k_]["launches"] * kernels[k_]["avg_ms"])
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (profiles/r2_traffic.json, bytes per key-switch)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(tp):
        tp = os.path.join(ROOT, "profiles", "r1_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if dom in tj:
            traffic = tj[dom]["dram_bytes_per_keyswitch"] * B
    # the kernel is bound by integer issue, not by HBM: butterflies per second against the in-register butterfly rate measured by
    # scripts/pipe_peaks.cu on this GPU model (profiles/r1_pipe_peaks.json), scaled to the SM clock observed during the timed region
    log_n = n.bit_length() - 1
    bf_per_ks = (R + cols_out) * 4 * (n // 2) * log_n
    int_pipe = None
    pp = os.path.join(ROOT, "profiles", "r1_pipe_peaks.json")
    clocks = cs.summary()
    if os.path.exists(pp) and dom == "gadget_fused":
        pk = json.load(open(pp))
        bf_peak = pk["ct_butterfly(harvey,shoup)"]["chip_per_s"]
        bf_ach = bf_per_ks * B / (kernels[dom]["avg_ms"] * 1e-3)
        int_pipe = {"unit": "Shoup/Harvey butterflies/s", "achieved": bf_ach, "peak": bf_peak, "frac": bf_ach / bf_peak,
                    "peak_source": "scripts/pipe_peaks.cu on B200: in-register butterfly loop on all SMs, chip-wide rate from CUDA events "
                                   "(profiles/r1_pipe_peaks.json)",
                    "butterflies_per_keyswitch": bf_per_ks}
    hbm_view = {"achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": kernels[dom]["achieved_gbs"] / peak,
                "peak_source": peak_src, "traffic": traffic,
                "note": "algorithmic bytes per launch (fused minimum: GLWE in + GLWE out + collapsed key once) / CUDA-event duration; "
                        "traffic = ncu dram__bytes of the same kernel"}
    if int_pipe is not None:
        # the binding roof: time at the butterfly peak (0.51 ms per 4096 key-switches) exceeds time at the HBM peak (0.25 ms), so the
        # headline fraction is against integer issue; the HBM view stays as the secondary field
        roofline = {"kernel": kernel_names.get(dom, dom), "category": dom, "bound": "int_issue", "achieved": int_pipe["achieved"],
                    "peak": int_pipe["peak"], "unit": int_pipe["unit"], "frac": int_pipe["frac"], "traffic": traffic,
                    "peak_source": int_pipe["peak_source"], "butterflies_per_keyswitch": bf_per_ks, "hbm": hbm_view,
                    "time_at_peak_ms": {"int_issue": bf_per_ks * B / int_pipe["peak"] * 1e3,
                                        "hbm": bytes_per_launch[dom] / (peak * 1e9) * 1e3},
                    "note": "five NTTs of four primes per key-switch (3 forward + 2 inverse on the collapsed key); achieved = Shoup/Harvey "
                            "butterflies per second of the dominant kernel from CUDA events on the launching stream; the kernel is bound by "
                            "integer issue (IMAD / IMAD.HI on the FMA-heavy pipe), not by bytes: see time_at_peak_ms"}
    else:
        roofline = {"kernel": kernel_names.get(dom, dom), "category": dom, "bound": "hbm", **hbm_view}
    # whole-pipeline view: bytes the fused pipeline must move per key-switch vs what the unfused HAL sequence moves in this backend's
    # 16 B layout (DESIGN.md section 3)
    fused_bytes = bytes_per_launch[dom] / B if dom == "gadget_fused" else (bytes_per_launch["dft_forward"] + bytes_per_launch["dft_inverse"]) / B
    unfused_bytes = 2949504.0
    step_gbs = fused_bytes * B / (ms / args.steps * 1e-3) / 1e9
    out = {
        "metric": "glwe_keyswitch_per_s", "value": value, "unit": "keyswitch/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 (canonical residues mod four 30-bit primes; i128 big)", "data": "synthetic", "config": config_dict(B, world),
        "e2e": {"value": e2e_value, "unit": "keyswitch/s", "h2d_bytes_per_step": int(a_np.nbytes), "d2h_bytes_per_step": int(a_np.nbytes),
                "steps": e2e_steps, "api": "pgb_glwe_keyswitch_host (pinned host buffers)",
                "note": "PCIe bound: 393 KB cross the bus per key-switch; scripts/e2e_probe.py measured 49 GB/s pinned H2D on this box = 250 k key-switches/s ceiling"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels,
        "pipeline": {"fused_bytes_per_keyswitch": fused_bytes, "unfused_bytes_per_keyswitch": unfused_bytes, "achieved_gbs": step_gbs,
                     "frac_of_hbm_peak": step_gbs / peak},
    }

    if not args.no_cggi:
        # CGGI bootstraps/s: measured on every rank under every world size (collectives inside: all ranks must enter)
        try:
            out["cggi"] = cggi_measure(pb, torch, dist, world, rank, local, with_cpu=(world == 1 and not args.no_cpu))
        except Exception as e:
            if world > 1:
                raise  # a one-sided failure would leave the other ranks inside a collective: fail loudly instead
            out["cggi"] = {"error": repr(e)}
    if rank == 0 and world == 1 and not args.no_cpu:
        cb, _, _ = cpu_port(sample_target_cpu_s=8.0)
        cba, _, _ = cpu_port(sample_target_cpu_s=8.0, simd=True)
        out["cpu_baseline"] = cba if cba["value"] > cb["value"] else cb  # the better CPU path is THE baseline; both are reported
        out["cpu_baseline_scalar"] = cb
        out["cpu_baseline_avx"] = cba
    if rank == 0 and world == 1 and not args.no_aux:
        try:
            out["aux"] = aux_measurements(pb, torch, local, peak)
        except Exception as e:  # auxiliary numbers must never break the headline line
            out["aux"] = {"error": repr(e)}
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


CGGI = dict(n=512, n_lwe=687, rank=3, block=3, base2k=18, brk_size=2, dnum=1, acc_size=1, batch=2368)


def cggi_ops_per_bootstrap(fl_name):
    """Algorithmic operation counts of one block-binary blind rotation at the bench shape (DESIGN.md section 7), in the unit of the pipe
    that binds the flavour.
    FFT64: FP64-pipe instructions (FMA / MUL / ADD each count 1): a radix-2 complex butterfly = 2 MUL + 2 FMA + 4 ADD = 8, a complex
    multiply-accumulate of the key products = 4 FMA, the (X^a - 1) update per (frequency, output poly, key) = 2 MUL + 2 FMA + 4 ADD = 8,
    the scaling of the rounded coefficients = 1 MUL.
    NTT120: issue slots of the FMA-heavy integer pipe (the pipe profiles/r1_pipe_peaks.json measures with imad_lo_u32; IMAD.HI is half
    rate = 2 slots): a Shoup / Harvey butterfly = IMAD.HI + 2 IMAD = 4 slots, a modular multiply-accumulate of the key products = 1
    IMAD.WIDE = 1 slot, the (X^a - 1) product per (frequency, output poly, key) = 1 slot; reductions and address arithmetic are not
    counted.  Returned per PRIME: the kernel runs two primes when the device-checked bound allows, the reference always four."""
    c = CGGI
    n, m = c["n"], c["n"] // 2
    cols = c["rank"] + 1
    R, C, bs, blocks = cols * c["dnum"], cols * c["brk_size"], c["block"], c["n_lwe"] // c["block"]
    if fl_name == "fft64":
        log_m = m.bit_length() - 1
        fft = (R + C) * (m // 2) * log_m * 8
        prod = m * C * bs * (R * 4 + 8)
        tail = C * n
        return blocks * (fft + prod + tail), "FP64-pipe instructions (FMA/MUL/ADD)"
    log_n = n.bit_length() - 1
    butterflies = (R + C) * (n // 2) * log_n
    macs = n * C * bs * (R + 1)
    return blocks * (4 * butterflies + macs), "FMA-heavy integer pipe slots (butterfly = 4, modular MAC = 1)"


def cggi_measure(pb, torch, dist, world, rank, local, with_cpu):
    """CGGI gate-bootstrap throughput (the first half of BASELINE.json's metric), measured under EVERY world size: block-binary blind
    rotation at the reference's bench configuration (poulpy-bench/src/bench_suite/schemes/blind_rotation.rs:39-72: n=512, n_lwe=687,
    rank 3, block 3, base2k 18, k_brk=36, k_glwe=18), a batch of 2368 LWEs per GPU (148 SMs x 4 ciphertexts x 4 waves), BRK replicated
    per GPU, no collective.  Per flavour: `value` = bootstraps/s with the LWEs resident in HBM (CUDA events, max over ranks);
    `e2e` = the same through pgb_cggi_blind_rotate_host (pinned HOST LWEs in, mod switch + rotation on the device, HOST GLWEs out; copies
    inside the timed region); `roofline` against the measured FP64 / integer issue rates; `cpu_baseline` = the oracle port on the host
    cores (N = 1 only).  Parity at exactly this configuration: tests/test_gpu_bench_shapes.py."""
    import ctypes as C

    lib = pb.lib()
    c = CGGI
    n, n_lwe, rank_g, block, k, B = c["n"], c["n_lwe"], c["rank"], c["block"], c["base2k"], c["batch"]
    cols = rank_g + 1
    out = {"config": {"workload": "cggi_blind_rotate block-binary n=512 n_lwe=687 rank=3 block=3 base2k=18 k_brk=36 k_glwe=18 "
                                  "(poulpy-bench blind_rotation defaults)", "batch_per_gpu": B, "global_batch": B * world, **c},
           "metric": "cggi_bootstraps_per_s", "unit": "bootstraps/s", "n_gpus": world, "scaling": "weak"}
    stream = torch.cuda.Stream(device=local)
    rng = np.random.default_rng(77 + rank)
    pp = os.path.join(ROOT, "profiles", "r1_pipe_peaks.json")
    pk = json.load(open(pp)) if os.path.exists(pp) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(x):
        t = torch.tensor([x], device=f"cuda:{local}", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for fl, nm in ((pb.FFT64, "fft64"), (pb.NTT120, "ntt120")):
        m = pb.Module(n, fl, device=local)
        m.set_stream(stream.cuda_stream)
        per = n * cols * cols * c["brk_size"] * c["dnum"] * m.prep_bytes
        brk_buf = pb.DevBuf(per * n_lwe, device=local)
        one = pb.hal.VmpPMat(brk_buf, n, c["dnum"], cols, cols, c["brk_size"])
        # synthetic (non-cryptographic) key material as in the reference's HAL benches; 8 distinct random GGSWs cycled over the 687 slots
        mats = np.random.default_rng(4242).integers(-(1 << (k - 1)), 1 << (k - 1), size=(8, c["dnum"], cols, c["brk_size"], cols, n), dtype=np.int64)
        for i in range(8):
            m.vmp_prepare(pb.hal.VmpPMat(brk_buf, n, c["dnum"], cols, cols, c["brk_size"], offset=i * per), m.mat_znx_from_numpy(mats[i]))
        for i in range(8, n_lwe):
            lib.pgb_memcpy_d2d(C.c_void_p(brk_buf.ptr + i * per), C.c_void_p(brk_buf.ptr + (i % 8) * per), C.c_size_t(per))
        m.gadget_key_pin(one)  # the BRK is immutable for the run: its coefficient bound (NTT120 prime count) is derived once
        xpa = m.cggi_x_pow_a()
        lut_np = rng.integers(-(1 << (k - 2)), 1 << (k - 2), size=(1, 1, n), dtype=np.int64)
        lut = m.vec_znx_from_numpy(lut_np)
        lwe_raw = rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=(B, 1, 1, n_lwe + 1), dtype=np.int64)  # base-2^18 LWE digits
        raw_dev = pb.DevBuf(lwe_raw.nbytes, device=local)
        raw_dev.upload(lwe_raw)
        lwe_dev = m.cggi_mod_switch_2n(raw_dev, B, n_lwe, 1, k, 2 * n, True)
        res = m.vec_znx_alloc(cols, c["acc_size"], B)
        sc = [None]

        def br():
            sc[0] = m.cggi_blind_rotate(res, lwe_dev, n_lwe, lut, one, xpa, block, k, sc[0])

        steps = 3
        br()
        barrier()
        l0 = m.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                br()
            e1.record(stream)
        torch.cuda.synchronize()
        launches = (m.launch_count - l0) // steps
        ms = max_ranks(e0.elapsed_time(e1)) / steps
        barrier()
        # e2e: host LWEs -> host GLWEs
        lwe_h = pb.pinned_empty(lwe_raw.shape)
        lwe_h[:] = lwe_raw
        res_h = pb.pinned_empty((B, c["acc_size"], cols, n))
        m.cggi_blind_rotate_host(res_h, lwe_h, k, lut, one, xpa, block, k)  # warm-up: grows the staging workspace
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            m.cggi_blind_rotate_host(res_h, lwe_h, k, lut, one, xpa, block, k)
        barrier()
        e2e_s = max_ranks(time.perf_counter() - t0) / steps
        same = bool(np.array_equal(res_h, m.vec_znx_to_numpy(res)))
        ops, unit = cggi_ops_per_bootstrap(nm)
        d = {"value": world * B / (ms * 1e-3), "ms_per_batch": ms, "launches_per_batch": int(launches),
             "e2e": {"value": world * B / e2e_s, "unit": "bootstraps/s", "h2d_bytes_per_step": int(lwe_raw.nbytes),
                     "d2h_bytes_per_step": int(res_h.nbytes), "api": "pgb_cggi_blind_rotate_host (pinned host LWEs in, host GLWEs out)",
                     "matches_device_resident": same}}
        if pk:
            if nm == "fft64":
                ach, peak_v = ops * B / (ms * 1e-3), pk["dfma"]["chip_per_s"]
                d["roofline"] = {"bound": "fp64_issue", "achieved": ach, "peak": peak_v, "unit": unit + "/s", "frac": ach / peak_v,
                                 "ops_per_bootstrap": ops, "peak_source": "scripts/pipe_peaks.cu on B200 (profiles/r1_pipe_peaks.json: dfma)",
                                 "note": "operation count from cggi_ops_per_bootstrap; ncu: FP64 pipe 40 % busy (profiles/r2_ncu_cggi.md)"}
            else:
                primes = 2 if launches <= 4 else 4  # the whole-rotation kernel (one launch) runs two primes; the limb-wise route four
                ach, peak_v = ops * primes * B / (ms * 1e-3), pk["imad_lo_u32"]["chip_per_s"]
                d["roofline"] = {"bound": "int_issue", "achieved": ach, "peak": peak_v, "unit": unit + "/s", "frac": ach / peak_v,
                                 "ops_per_bootstrap": ops * primes, "primes_computed": primes,
                                 "frac_if_counted_as_four_prime_work": ops * 4 * B / (ms * 1e-3) / peak_v,
                                 "peak_source": "scripts/pipe_peaks.cu on B200 (profiles/r1_pipe_peaks.json: imad_lo_u32)",
                                 "note": "algorithmic slots of the primes actually computed (two when the device-checked bound allows: DESIGN.md "
                                         "3.6); ncu: FMA-heavy pipe 67 % busy including reductions and address arithmetic (profiles/r2_ncu_cggi.md)"}
        out[nm] = d
        if with_cpu and nm == "fft64":  # the reference benches CGGI in FFT64: oracle port on the host cores, bounded sample
            from oracle import pyoracle as O

            om = O.OracleModule(n, O.FFT64)
            opm = []
            for i in range(8):
                pm_ = om.vmp_pmat_alloc(c["dnum"], cols, cols, c["brk_size"])
                om.vmp_prepare(pm_, mats[i])
                opm.append(pm_)
            obrk = [opm[i % 8] for i in range(n_lwe)]
            oxp = om.cggi_x_pow_a()
            threads = O.num_threads()
            cnt = 4 * threads
            l2n = m.cggi_mod_switch_2n(raw_dev, B, n_lwe, 1, k, 2 * n, True).download(np.int64, (B, n_lwe + 1))[:cnt]
            want = np.zeros((cnt, c["acc_size"], cols, n), dtype=np.int64)
            t0 = time.perf_counter()
            om.cggi_blind_rotate_block_binary_batch(want, l2n, lut_np, obrk, oxp, block, k, threads=threads)
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": cnt / dt, "unit": "bootstraps/s", "cores": threads, "kind": "port", "flavour": "fft64",
                                   "sample": f"{cnt} blind rotations of the bench workload, oracle C port of poulpy-cpu-ref (FFT64), {threads} threads",
                                   "matches_gpu": bool(np.array_equal(want, m.vec_znx_to_numpy(res)[:cnt]))}
        del m, brk_buf, xpa, lut, raw_dev, lwe_dev, res, sc
        pb.hal.pool_trim()
    out["value"] = out["fft64"]["value"]  # the reference's CGGI flavour is the headline of this object
    out["e2e"] = out["fft64"]["e2e"]
    return out


def _time_ms(torch, stream, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def aux_measurements(pb, torch, local, peak):
    """Secondary numbers named by BASELINE.json: external products/s (config 2) and vmp_apply HBM GB/s (M5 shapes)."""
    aux = {}
    stream = torch.cuda.Stream(device=local)
    rng = np.random.default_rng(5)
    # GGSW x GLWE external product, n=2048, batch 4096 (BASELINE config "external product batch (4096 ciphertexts) at log_n=11")
    for fl, nm in ((pb.NTT120, "ntt120"), (pb.FFT64, "fft64")):
        n, B, k = 2048, 4096, 18
        m = pb.Module(n, fl, device=local)
        m.set_stream(stream.cuda_stream)
        mat = rng.integers(-(1 << 17), 1 << 17, size=(3, 2, 3, 2, n), dtype=np.int64)
        pm = m.vmp_pmat_alloc(3, 2, 2, 3)
        m.vmp_prepare(pm, m.mat_znx_from_numpy(mat))
        m.gadget_key_pin(pm)
        a = m.vec_znx_from_numpy(rng.integers(-(1 << 17), 1 << 17, size=(B, 3, 2, n), dtype=np.int64))
        r = m.vec_znx_alloc(2, 3, B)
        sc = [None]

        def f():
            sc[0] = m.glwe_external_product(r, k, a, k, pm, k, 1, sc[0])

        ms = _time_ms(torch, stream, f, 10)
        aux[f"glwe_external_product_per_s_{nm}_n2048_b4096"] = B / (ms * 1e-3)
        if fl == pb.NTT120:  # three primes carry the integers of this shape (pinned key, device-checked bound; ntt120_gadget.cu)
            aux["glwe_external_product_ntt120_primes"] = m.get_option(pb.hal.OPT_LAST_GADGET_PRIMES)
        del m, a, r, pm, sc
    # key-switch in the FFT64 flavour (row M1f)
    n, B, k = 4096, 4096, 18
    m = pb.Module(n, pb.FFT64, device=local)
    m.set_stream(stream.cuda_stream)
    mat = rng.integers(-(1 << 17), 1 << 17, size=(3, 1, 4, 2, n), dtype=np.int64)
    pm = m.vmp_pmat_alloc(3, 1, 2, 4)
    m.vmp_prepare(pm, m.mat_znx_from_numpy(mat))
    m.gadget_key_pin(pm)
    a = m.vec_znx_from_numpy(rng.integers(-(1 << 17), 1 << 17, size=(B, 3, 2, n), dtype=np.int64))
    r = m.vec_znx_alloc(2, 3, B)
    sc = [None]

    def f2():
        sc[0] = m.glwe_keyswitch(r, k, a, k, pm, k, 1, sc[0])

    ms = _time_ms(torch, stream, f2, 10)
    aux["glwe_keyswitch_per_s_fft64_n4096_b4096"] = B / (ms * 1e-3)
    del m, a, r, pm, sc
    # vmp_apply_dft_to_dft alone ("vmp_apply HBM GB/s" of BASELINE.json): the reference's whole sweep (poulpy-bench/src/params.rs:75-81)
    # plus the CKKS relinearisation shape, both flavours.  Two regimes per shape:
    #   stream : the batched twin over enough independent products, EACH WITH ITS OWN MATRIX (stride_b = matrix bytes), that the operands
    #            exceed L2 several times -- kernel time from CUDA events, the HBM-streaming number;
    #   single : one product per launch after an L2 flush -- what one HalImpl call costs; for the small shapes this is launch latency
    #            (a few microseconds for < 10 MB), labelled as such.
    import ctypes as C

    lib = pb.lib()
    flush = pb.DevBuf(256 << 20)
    shapes = ((10, 2, 1, 2, 3), (11, 4, 1, 2, 5), (12, 7, 1, 2, 8), (13, 15, 1, 2, 16), (14, 31, 1, 2, 32), (15, 14, 1, 2, 15))
    for fl, nm in ((pb.NTT120, "ntt120"), (pb.FFT64, "fft64")):
        vm = {}
        for (log_n, rows, cols_in, cols_out, size) in shapes:
            n = 1 << log_n
            m = pb.Module(n, fl, device=local)
            m.set_stream(stream.cuda_stream)
            s = m.prep_bytes
            R, Cc = rows * cols_in, cols_out * size
            byts = (R + R * Cc + Cc) * n * s
            count = int(max(1, min(4096, -(-(1 << 30) // byts))))  # >= 1 GB of operands per launch
            pm_one = n * R * Cc * s
            pm = pb.DevBuf(pm_one * count)  # content irrelevant for bandwidth (zeros)
            a = m.vec_znx_dft_alloc(cols_in, rows, count)
            r = m.vec_znx_dft_alloc(cols_out, size, count)
            rs, as_ = r.struct(), a.struct()
            ps = pb.hal._PM(pm.ptr, n, size, rows, cols_in, cols_out)
            bt = pb.hal._BT(count, r.batch_stride, a.batch_stride, pm_one)

            def f3():
                pb.hal._check(lib.pgb_vmp_apply_dft_to_dft_batched(m._h, C.byref(rs), C.byref(as_), C.byref(ps), C.c_uint64(0), C.byref(bt)))

            ms = _time_ms(torch, stream, f3, 5, warm=2)
            e = {"stream": {"products_per_launch": count, "ms": ms, "algorithmic_bytes": byts * count, "achieved_gbs": byts * count / (ms * 1e-3) / 1e9,
                            "frac_of_hbm_peak": byts * count / (ms * 1e-3) / 1e9 / peak}}
            bt1 = pb.hal._BT(1, 0, 0, 0)
            times = []
            for it in range(7):
                lib.pgb_memset(C.c_void_p(flush.ptr), it, C.c_size_t(flush.nbytes))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    e0.record(stream)
                    lib.pgb_vmp_apply_dft_to_dft_batched(m._h, C.byref(rs), C.byref(as_), C.byref(ps), C.c_uint64(0), C.byref(bt1))
                    e1.record(stream)
                torch.cuda.synchronize()
                if it >= 2:
                    times.append(e0.elapsed_time(e1))
            ms1 = float(np.median(times))
            e["single"] = {"ms": ms1, "algorithmic_bytes": byts, "achieved_gbs": byts / (ms1 * 1e-3) / 1e9,
                           "frac_of_hbm_peak": byts / (ms1 * 1e-3) / 1e9 / peak,
                           "regime": "hbm-streaming (operands exceed L2)" if byts > (200 << 20) else
                                     ("launch-latency bound: %.1f MB per launch, time-at-HBM-peak %.1f us" % (byts / 1e6, byts / (peak * 1e3)))}
            vm[f"log_n={log_n},rows={rows},cols_in={cols_in},cols_out={cols_out},size={size}"] = e
            del m, a, r, pm
            pb.hal.pool_trim()
        aux[f"vmp_apply_dft_to_dft_{nm}"] = vm
    del flush

    # CKKS relinearisation core (BASELINE config 4, SURVEY C5): key-switch with VmpPMat(14, 1, 2, 15) at N = 2^15, base2k = 52
    # (poulpy-bench/src/bench_suite/ckks.rs:31-37): R6 + R10 + R7 + R14 + R13 with a 0.22 GB prepared key; tensoring not included
    n, B, k = 1 << 15, 32, 52
    m = pb.Module(n, pb.NTT120, device=local)
    m.set_stream(stream.cuda_stream)
    pm = m.vmp_pmat_alloc(14, 1, 2, 15)
    mat = rng.integers(-(1 << 51), 1 << 51, size=(1, 1, 15, 2, n), dtype=np.int64)
    m.vmp_prepare(pb.hal.VmpPMat(pm.buf, n, 1, 1, 2, 15), m.mat_znx_from_numpy(mat))  # first row random, rest zero (bandwidth only)
    a = m.vec_znx_from_numpy(rng.integers(-(1 << 51), 1 << 51, size=(B, 14, 2, n), dtype=np.int64))
    r = m.vec_znx_alloc(2, 14, B)
    sc = [None]

    def f4():
        sc[0] = m.glwe_keyswitch(r, k, a, k, pm, k, 1, sc[0])

    ms = _time_ms(torch, stream, f4, 5)
    aux["ckks_relinearize_keyswitch_per_s_ntt120_n32768_b32"] = {"value": B / (ms * 1e-3), "ms_per_batch": ms}
    del m, a, r, pm, sc

    # CKKS ciphertext x ciphertext multiplication (BASELINE config 4, SURVEY 8f N2): glwe_tensor_apply + glwe_tensor_relinearize
    # (poulpy-ckks/src/leveled/default/mul.rs:49-86) at the reference's bench parameters (poulpy-bench/src/bench_suite/ckks.rs:31-37:
    # base2k = 52, K = 728 = 14 limbs, rank 1, dsize 1, tensor key 15 limbs); N = 2^15 as in the reference bench and 2^16 as BASELINE asks
    ck = {}
    for log_n, B in ((15, 8), (16, 4)):
        n, k, size = 1 << log_n, 52, 14
        m = pb.Module(n, pb.NTT120, device=local)
        m.set_stream(stream.cuda_stream)
        tsk = m.vmp_pmat_alloc(size, 1, 2, size + 1)
        mat = rng.integers(-(1 << 51), 1 << 51, size=(1, 1, size + 1, 2, n), dtype=np.int64)
        m.vmp_prepare(pb.hal.VmpPMat(tsk.buf, n, 1, 1, 2, size + 1), m.mat_znx_from_numpy(mat))  # first row random, rest zero (timing only)
        a = m.vec_znx_from_numpy(rng.integers(-(1 << 51), 1 << 51, size=(B, size, 2, n), dtype=np.int64))
        b2 = m.vec_znx_from_numpy(rng.integers(-(1 << 51), 1 << 51, size=(B, size, 2, n), dtype=np.int64))
        tensor = m.vec_znx_alloc(3, size, B)
        r = m.vec_znx_alloc(2, size, B)
        sc = [None, None]

        def f5():
            sc[0] = m.glwe_tensor_apply(size * k, tensor, k, a, size * k, b2, size * k, k, sc[0])
            sc[1] = m.glwe_tensor_relinearize(r, k, tensor, k, tsk, k, 1, sc[1])

        ms = _time_ms(torch, stream, f5, 5)
        ck[f"log_n={log_n}"] = {"value": B / (ms * 1e-3), "unit": "ct x ct multiplications/s", "ms_per_batch": ms, "batch": B}
        del m, a, b2, tensor, r, tsk, sc
    aux["ckks_mul_ntt120_base2k52_k728"] = ck

    # prepare paths (SURVEY 8f N3): vmp_prepare (MatZnx i64 -> prepared VmpPMat) and svp_prepare at the key-switch, CGGI and CKKS key shapes;
    # algorithmic bytes per poly = 8n in + prep_bytes * n out
    prep = {}
    for fl, nm, log_n, shape, k in ((pb.NTT120, "ntt120", 12, (3, 1, 2, 4), 18), (pb.FFT64, "fft64", 12, (3, 1, 2, 4), 18),
                                    (pb.FFT64, "fft64", 9, (1, 4, 4, 2), 18), (pb.NTT120, "ntt120", 15, (14, 1, 2, 15), 52)):
        n = 1 << log_n
        m = pb.Module(n, fl, device=local)
        m.set_stream(stream.cuda_stream)
        rows, cols_in, cols_out, size = shape
        polys = rows * cols_in * cols_out * size
        matd = m.mat_znx_from_numpy(np.broadcast_to(rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=(1, 1, 1, 1, n), dtype=np.int64),
                                                    (rows, cols_in, size, cols_out, n)))
        pm = m.vmp_pmat_alloc(rows, cols_in, cols_out, size)
        ms = _time_ms(torch, stream, lambda: m.vmp_prepare(pm, matd), 5)
        byts = polys * n * (8 + m.prep_bytes)
        prep[f"vmp_prepare_{nm}_log_n={log_n}_shape={rows}x{cols_in}x{cols_out}x{size}"] = {
            "ms": ms, "polys_per_s": polys / (ms * 1e-3), "achieved_gbs": byts / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": byts / (ms * 1e-3) / 1e9 / peak,
            "note": "one synchronous call (host launch + stream sync inside the timed region)"}
        sp, sz = m.svp_ppol_alloc(1), m.scalar_znx_from_numpy(rng.integers(-1, 2, size=(1, n), dtype=np.int64))
        ms = _time_ms(torch, stream, lambda: m.svp_prepare(sp, 0, sz, 0), 20)
        prep[f"svp_prepare_{nm}_log_n={log_n}"] = {"ms": ms, "note": "single polynomial, launch-latency bound"}
        del m, matd, pm, sp, sz
    aux["prepare_paths"] = prep

    # batched DFT sweep (BASELINE config 1): forward then inverse over VecZnx(cols=2, size) at log_n 10..16, >= 256 MB of limbs
    sweep = {}
    pp = os.path.join(ROOT, "profiles", "r1_pipe_peaks.json")
    bf_peak = json.load(open(pp))["ct_butterfly(harvey,shoup)"]["chip_per_s"] if os.path.exists(pp) else None
    for fl, nm, k in ((pb.NTT120, "ntt120", 18), (pb.FFT64, "fft64", 18)):
        for log_n, size in ((10, 2), (11, 4), (12, 8), (13, 16), (14, 32), (15, 8), (16, 8)):
            n = 1 << log_n
            m = pb.Module(n, fl, device=local)
            m.set_stream(stream.cuda_stream)
            B = max(1, (256 << 20) // (n * 2 * size * 8))
            a = m.vec_znx_alloc(2, size, B)
            a.buf.upload(rng.integers(-(1 << (k - 1)), 1 << (k - 1), size=(n * 2 * size,), dtype=np.int64))  # first item random, rest zero
            d = m.vec_znx_dft_alloc(2, size, B)
            big = m.vec_znx_big_alloc(2, size, B)

            def fwd():
                for c in range(2):
                    m.vec_znx_dft_apply(1, 0, d, c, a, c)

            def inv():
                for c in range(2):
                    m.vec_znx_idft_apply(big, c, d, c)

            limbs = B * 2 * size
            t_f = _time_ms(torch, stream, fwd, 5)
            t_i = _time_ms(torch, stream, inv, 5)
            pbytes = m.prep_bytes
            e = {"limbs": limbs, "fwd_ms": t_f, "inv_ms": t_i, "fwd_limbs_per_s": limbs / (t_f * 1e-3), "inv_limbs_per_s": limbs / (t_i * 1e-3),
                 "fwd_gbs": limbs * n * (8 + pbytes) / (t_f * 1e-3) / 1e9, "inv_gbs": limbs * n * (pbytes + m.big_bytes) / (t_i * 1e-3) / 1e9}
            if fl == pb.NTT120 and bf_peak:  # the transforms are integer-issue bound: fraction of the measured in-register butterfly rate
                bf = 4 * (n // 2) * log_n
                e["fwd_butterfly_frac"] = limbs * bf / (t_f * 1e-3) / bf_peak
                e["inv_butterfly_frac"] = limbs * bf / (t_i * 1e-3) / bf_peak
            sweep[f"{nm}_log_n={log_n}_size={size}"] = e
            del m, a, d, big
    aux["dft_sweep"] = sweep

    # N4 compositions at the headline key-switch shape (n=4096, base2k=18, rank 1, 3 limbs, key dnum 3 x 4 limbs): automorphism
    # (key-switch + X -> X^p) and trace (log_n key-switch/automorphism/add rounds), batch of ciphertexts per call
    try:
        for fl, nm in ((pb.NTT120, "ntt120"), (pb.FFT64, "fft64")):
            n, B, k = 4096, 1024, 18
            m = pb.Module(n, fl, device=local)
            m.set_stream(stream.cuda_stream)
            keys = []
            for _ in range(12):
                pm = m.vmp_pmat_alloc(3, 1, 2, 4)
                m.vmp_prepare(pm, m.mat_znx_from_numpy(rng.integers(-(1 << 17), 1 << 17, size=(3, 1, 4, 2, n), dtype=np.int64)))
                m.gadget_key_pin(pm)
                keys.append(pm)
            a = m.vec_znx_from_numpy(rng.integers(-(1 << 17), 1 << 17, size=(B, 3, 2, n), dtype=np.int64))
            r = m.vec_znx_alloc(2, 3, B)
            sc = [None, None]

            def f_aut():
                sc[0] = m.glwe_automorphism(r, k, a, k, keys[0], k, 5, 1, sc[0])

            def f_tr():
                sc[1] = m.glwe_trace_assign(r, k, 0, keys, k, 1, sc[1])

            ms = _time_ms(torch, stream, f_aut, 5)
            aux[f"glwe_automorphism_per_s_{nm}_n4096_b{B}"] = B / (ms * 1e-3)
            ms = _time_ms(torch, stream, f_tr, 3, warm=1)
            aux[f"glwe_trace_per_s_{nm}_n4096_b{B}"] = B / (ms * 1e-3)
            del m, keys, a, r, sc
    except Exception as e:
        aux["glwe_trace_per_s"] = {"error": repr(e)}
    pb.hal.pool_trim()  # blocks parked by the sections above are of no use below
    # circuit bootstrapping (poulpy-bench circuit_bootstrapping.rs:47-129 "1-bit"): n=1024, n_lwe=574, block 7, rank 2, base2k 13,
    # BRK/ATK/TSK k=52 dnum=3, result GGSW dnum=2 (constant mode: k=26, 2 limbs; exponent mode keeps the 4-limb layout); synthetic keys;
    # a batch of LWEs per call.  Both flavours for the constant mode (the reference benches FFT64), exponent mode in FFT64.
    from poulpy_b200 import circuit
    for fl, nm, mode in ((pb.FFT64, "fft64", "constant"), (pb.NTT120, "ntt120", "constant"), (pb.FFT64, "fft64", "exponent")):
        key = f"circuit_bootstraps_per_s_{nm}_n1024_nlwe574_rank2" + ("" if mode == "constant" else "_to_exponent")
        try:
            n, log_n, n_lwe, block, rank, K, B = 1024, 10, 574, 7, 2, 13, 512
            cols, ksz, kd, res_size, dnum_res = rank + 1, 4, 3, 2, 2
            m = pb.Module(n, fl, device=local)
            m.set_stream(stream.cuda_stream)
            per = n * cols * cols * kd * ksz * m.prep_bytes
            brk_buf = pb.DevBuf(per * n_lwe)
            one = pb.hal.VmpPMat(brk_buf, n, kd, cols, cols, ksz)
            m.vmp_prepare(one, m.mat_znx_from_numpy(rng.integers(-(1 << 12), 1 << 12, size=(kd, cols, ksz, cols, n), dtype=np.int64)))
            for i in range(1, n_lwe):
                lib.pgb_memcpy_d2d(C.c_void_p(brk_buf.ptr + i * per), C.c_void_p(brk_buf.ptr), C.c_size_t(per))

            def mk(count):
                out = []
                for _ in range(count):
                    pm = m.vmp_pmat_alloc(kd, rank, cols, ksz)
                    m.vmp_prepare(pm, m.mat_znx_from_numpy(rng.integers(-(1 << 12), 1 << 12, size=(kd, rank, ksz, cols, n), dtype=np.int64)))
                    out.append(pm)
                return out

            atk, tsk = mk(log_n), mk(rank)
            lwe = rng.integers(-(1 << 12), 1 << 12, size=(B, 1, 1, n_lwe + 1), dtype=np.int64)
            lwe_dev = pb.DevBuf(lwe.nbytes)
            lwe_dev.upload(lwe)
            xpa = m.cggi_x_pow_a()

            def cbt():
                if mode == "constant":
                    circuit.circuit_bootstrap_to_constant(m, lwe_dev, B, n_lwe, 1, K, one, xpa, block, atk, tsk, K, rank, dnum_res, res_size, 1)
                else:
                    circuit.circuit_bootstrap_to_exponent(m, 2, lwe_dev, B, n_lwe, 1, K, one, xpa, block, atk, tsk, K, rank, dnum_res, ksz, 1)

            l0 = m.launch_count
            ms = _time_ms(torch, stream, cbt, 2, warm=1)
            aux[key + f"_b{B}"] = {"value": B / (ms * 1e-3), "ms_per_batch": ms, "launches_per_batch": (m.launch_count - l0) // 3}
            del m, brk_buf, atk, tsk, lwe_dev, xpa
            pb.hal.pool_trim()
        except Exception as e:
            aux[key] = {"error": repr(e)}
    return aux


if __name__ == "__main__":
    main()
