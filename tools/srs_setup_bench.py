"""Timing of ParamsKZG::setup on the device (h2b_srs_setup) and of its fixed-base kernel; needs a B200.

    python tools/srs_setup_bench.py [--ks 16,20,22,24] [--cpu-ks 16,18] [--window-libs 8=path,12=path] [--out FILE]

One JSON line per measurement (stdout, and appended to --out):
  * device   : card name, power limit and max SM clock, read in this invocation
  * rate     : dependent Fq multiplications per second (h2b_imad_bench kind 2), the roofline's denominator
  * setup    : per k, device time per phase from the profiling tags of a warmed-up call (24 scalars including the derivation
               of w and c, 25 fixed-base, 26 normalisation; both vectors), wall time of h2b_srs_setup without outputs (compute), and separately the extra time of the host download and of
               registering both vectors (window tables on every device)
  * generator_table : the table build of the first call on the device (tag 27)
  * window   : g1_generator_mul on 2^24 uniform scalars with a library built for another window width (--window-libs)
  * cpu      : the CPU restatement of upstream's setup (tests/cpp/srs_setup_oracle.cpp) on all host threads -- a restatement,
               not the reference itself
Work model per point: WINDOWS mixed additions of 10 multiplications (8M + 2S) plus 8 normalisation multiplications
(3 projective products, 3 of Montgomery's trick, 2 for x and y); the scalars are not counted.  Nothing is written to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

TAGS = {24: "scalars", 25: "fixed_base", 26: "normalise", 27: "generator_table"}


def emit(line, out):
    s = json.dumps(line)
    print(s, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(s + "\n")


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(kind="device", name=name, power_limit=power, max_sm_clock=clock)


def windows_of(w):
    return (255 + w - 1) // w


def wall(fn, reps=3):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return sorted(ts)[len(ts) // 2]


def window_only(lib_path, w, out):
    """fixed-base multiplication of 2^24 uniform scalars with the library at lib_path (built for window w)"""
    from halo2_scaffold_b200._lib import Lib
    L = Lib(lib_path)
    L.init_device(0)
    n = 1 << 24
    d_s, d_o = L.dev_alloc(0, n * 32), L.dev_alloc(0, n * 64)
    L.gen_scalars_dev(0, 0x5E7, n, 0, d_s)
    L.dev_sync(0)
    t = time.perf_counter()
    L.g1_generator_mul_dev(0, d_s, 1, d_o)           # builds the table
    L.dev_sync(0)
    table_s = time.perf_counter() - t
    L.g1_generator_mul_dev(0, d_s, n, d_o)
    L.dev_sync(0)

    def run():
        L.g1_generator_mul_dev(0, d_s, n, d_o)
        L.dev_sync(0)
    s = wall(run, 5)
    emit(dict(kind="window", window=w, windows=windows_of(w), table_bytes=windows_of(w) * (1 << (w - 1)) * 64, n=n, ms=s * 1e3,
              table_build_ms=table_s * 1e3, points_per_s=n / s), out)
    L.dev_free(0, d_s)
    L.dev_free(0, d_o)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="16,20,22,24")
    ap.add_argument("--cpu-ks", default="16,18")
    ap.add_argument("--window", type=int, default=16, help="window width the default library was built with")
    ap.add_argument("--window-libs", default="", help="W=path,... libraries built with -DH2B_G1GEN_WINDOW=W")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--window-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.window_only:
        return window_only(args.lib, args.window, args.out)

    import oracle_c as oc
    from halo2_scaffold_b200._lib import Lib, DEFAULT_LIB
    emit(device_line(), args.out)
    L = Lib(args.lib or DEFAULT_LIB)
    L.init_device(0)
    ms, ops = L.imad_bench(2, 4096)
    rate = ops / (ms * 1e-3)
    emit(dict(kind="rate", what="dependent Fq multiplications (imad_bench kind 2)", fq_mul_per_s=rate), args.out)
    s = oc.random_fr(0x5E7, 1)[0]
    W = args.window
    model = windows_of(W) * 10 + 8
    def profiled(k):
        L.profile_enable(True)
        L.srs_setup(k, s, want_host=False, register=False)
        phases = {}
        for tag, t in L.profile_read():
            if tag in TAGS:
                phases[TAGS[tag]] = phases.get(TAGS[tag], 0.0) + t
        L.profile_enable(False)
        return phases
    ks = [int(x) for x in args.ks.split(",") if x]
    first = profiled(ks[0])                           # the first call on the device builds the generator table
    emit(dict(kind="generator_table", window=W, ms=first.get("generator_table")), args.out)
    for k in ks:
        n = 1 << k
        L.srs_setup(k, s, want_host=False, register=False)          # warm-up: module loads, twiddle cache of the power step
        phases = profiled(k)
        compute = wall(lambda: L.srs_setup(k, s, want_host=False, register=False))
        with_host = wall(lambda: L.srs_setup(k, s, want_host=True, register=False))

        def registered():
            r = L.srs_setup(k, s, want_host=False, register=True)
            L.unregister_bases(r["handle_g"])
            L.unregister_bases(r["handle_g_lagrange"])
        with_reg = wall(registered)
        kernel_ms = phases.get("fixed_base", 0.0) + phases.get("normalise", 0.0)
        roofline_ms = 2 * n * model / rate * 1e3
        emit(dict(kind="setup", k=k, window=W, phases_ms=phases, compute_ms=compute * 1e3, host_download_ms=(with_host - compute) * 1e3,
                  register_ms=(with_reg - compute) * 1e3, work_model_fq_mul_per_point=model, roofline_ms=roofline_ms,
                  roofline_share_kernels=roofline_ms / kernel_ms if kernel_ms else None, roofline_share_compute=roofline_ms / (compute * 1e3)), args.out)
    L.shutdown()
    for spec in [x for x in args.window_libs.split(",") if x]:
        w, path = spec.split("=", 1)
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--window-only", "--lib", path, "--window", w] +
                              (["--out", args.out] if args.out else []))
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--window-only", "--lib", args.lib or DEFAULT_LIB, "--window", str(W)] +
                          (["--out", args.out] if args.out else []))
    # the CPU restatement
    import test_srs_setup as t
    threads = os.cpu_count() or 1
    t.setup_oracle()                                  # compiled before the clock starts
    for k in [int(x) for x in args.cpu_ks.split(",") if x]:
        t0 = time.perf_counter()
        t.orc_srs_setup(k, s, threads)
        emit(dict(kind="cpu", what="CPU restatement of upstream ParamsKZG::setup (not the reference)", k=k, threads=threads,
                  s=time.perf_counter() - t0), args.out)


if __name__ == "__main__":
    main()
