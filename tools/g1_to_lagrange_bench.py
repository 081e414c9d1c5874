"""Timing of ParamsKZG::downsize on the device (h2b_srs_downsize) and of the G1 NTT behind it; needs a B200.

    python tools/g1_to_lagrange_bench.py [--K 25] [--ks 16,20,22,24] [--cpu-ks 12,14,16] [--window-libs 2=path,...] [--out FILE]

One JSON line per measurement (stdout, and appended to --out):
  * device   : card name, power limit and max SM clock, read in this invocation
  * rate     : dependent Fq multiplications per second (h2b_imad_bench kind 2), the roofline's denominator
  * downsize : per k, from a registered setup(K) set: device time per phase from the profiling tags of a warmed-up call
               (28 twiddles, 29 butterfly stages, 30 normalisation), and the wall time of the whole h2b_srs_downsize call with the
               host copy of g_lagrange and no registration, and with both new sets registered and no host copy; each result
               is checked against setup(k, s) bit for bit
  * window   : h2b_g1_to_lagrange_dev at 2^20 points with a library built for another window width (--window-libs)
  * cpu      : the CPU restatement of upstream's g_to_lagrange (tests/cpp/g1_to_lagrange_oracle.cpp) on all host threads --
               a restatement, not the reference itself
Work model (Fq multiplications): xyzz_double 9, xyzz_add 14; one scalar multiplication = the table (1 doubling and
2^(W-1) - 2 additions), (windows - 1) W doublings and windows (1 - 2^-W) additions (a Booth digit is 0 with probability
2^-W); per butterfly 2 additions; (n/2) k - (n - 1) butterflies with a non-trivial twiddle plus the n/2 + 1 multiplications by
n^-1 of stage 0; 8 per point for the normalisation.  Nothing is written to the tree.
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

TAGS = {28: "twiddles", 29: "stages", 30: "normalise"}
DBL, ADD = 9, 14


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


def scalar_mul_model(w):
    windows = (255 + w - 1) // w
    table = (DBL if w > 1 else 0) + max((1 << (w - 1)) - 2, 0) * ADD
    return table + (windows - 1) * w * DBL + windows * (1 - 2.0 ** -w) * ADD


def work_model(k, w):
    """Fq multiplications of one g_to_lagrange of 2^k points: (stages, normalisation)"""
    n = 1 << k
    muls = (n // 2) * k - (n - 1) + n // 2 + 1
    return muls * scalar_mul_model(w) + (n // 2) * k * 2 * ADD, 8 * n


def wall(fn, reps):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return sorted(ts)[len(ts) // 2]


def window_only(lib_path, w, out):
    """h2b_g1_to_lagrange_dev of 2^20 points with the library at lib_path (built for window w)"""
    from halo2_scaffold_b200._lib import Lib
    L = Lib(lib_path)
    L.init_device(0)
    k = 20
    n = 1 << k
    d = L.dev_alloc(0, n * 64)
    L.gen_points_dev(0, 0x61, n, d)
    L.g1_to_lagrange_dev(0, d, k, d)              # warm-up: module load, scratch
    L.dev_sync(0)

    def run():
        L.g1_to_lagrange_dev(0, d, k, d)
        L.dev_sync(0)
    s = wall(run, 3)
    stages, norm = work_model(k, w)
    emit(dict(kind="window", window=w, k=k, ms=s * 1e3, work_model_fq_mul=stages + norm), out)
    L.dev_free(0, d)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=25, help="k of the setup the downsizes start from")
    ap.add_argument("--ks", default="16,20,22,24")
    ap.add_argument("--cpu-ks", default="12,14,16")
    ap.add_argument("--window", type=int, default=4, help="window width the default library was built with")
    ap.add_argument("--window-libs", default="", help="W=path,... libraries built with -DH2B_G1_MUL_WINDOW=W")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--window-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.window_only:
        return window_only(args.lib, args.window, args.out)

    import numpy as np
    import oracle_c as oc
    from halo2_scaffold_b200._lib import Lib, DEFAULT_LIB
    emit(device_line(), args.out)
    L = Lib(args.lib or DEFAULT_LIB)
    L.init_device(0)
    ms, ops = L.imad_bench(2, 4096)
    rate = ops / (ms * 1e-3)
    emit(dict(kind="rate", what="dependent Fq multiplications (imad_bench kind 2)", fq_mul_per_s=rate), args.out)
    s = oc.random_fr(0xD0, 1)[0]
    big = L.srs_setup(args.K, s, want_host=False)
    hg = big["handle_g"]
    W = args.window

    def profiled(k):
        L.profile_enable(True)
        r = L.srs_downsize(hg, k, want_host=True, register=False)
        phases = {}
        for tag, t in L.profile_read():
            if tag in TAGS:
                phases[TAGS[tag]] = phases.get(TAGS[tag], 0.0) + t
        L.profile_enable(False)
        return phases, r["g_lagrange"]

    ks = [int(x) for x in args.ks.split(",") if x]
    L.srs_downsize(hg, ks[0], want_host=False, register=False)     # warm-up: module loads
    for k in ks:
        phases, gl = profiled(k)
        want = L.srs_setup(k, s, want_host=True, register=False)["g_lagrange"]
        reps = 3 if k <= 20 else 1
        with_host = wall(lambda: L.srs_downsize(hg, k, want_host=True, register=False), reps)

        def registered():
            r = L.srs_downsize(hg, k, want_host=False, register=True)
            L.unregister_bases(r["handle_g"])
            L.unregister_bases(r["handle_g_lagrange"])
        with_reg = wall(registered, reps)
        stages, norm = work_model(k, W)
        kernel_ms = phases.get("stages", 0.0) + phases.get("normalise", 0.0)
        roofline_ms = (stages + norm) / rate * 1e3
        emit(dict(kind="downsize", K=args.K, k=k, window=W, equals_setup=bool(np.array_equal(gl, want)), phases_ms=phases,
                  call_host_ms=with_host * 1e3, call_registered_ms=with_reg * 1e3,
                  work_model_fq_mul=stages + norm, roofline_ms=roofline_ms,
                  roofline_share_kernels=roofline_ms / kernel_ms if kernel_ms else None), args.out)
    L.unregister_bases(hg)
    L.unregister_bases(big["handle_g_lagrange"])
    L.shutdown()
    for spec in [x for x in args.window_libs.split(",") if x]:
        w, path = spec.split("=", 1)
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--window-only", "--lib", path, "--window", w] +
                              (["--out", args.out] if args.out else []))
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--window-only", "--lib", args.lib or DEFAULT_LIB, "--window", str(W)] +
                          (["--out", args.out] if args.out else []))
    # the CPU restatement
    import test_g1_to_lagrange as t
    threads = os.cpu_count() or 1
    t.oracle()                                        # compiled before the clock starts
    for k in [int(x) for x in args.cpu_ks.split(",") if x]:
        pts = oc.gen_points(0x62, 1 << k)
        t0 = time.perf_counter()
        t.orc_g1_to_lagrange(pts, k, threads)
        emit(dict(kind="cpu", what="CPU restatement of upstream g_to_lagrange (not the reference)", k=k, threads=threads,
                  s=time.perf_counter() - t0), args.out)


if __name__ == "__main__":
    main()
