"""Timing of the permutation keygen on the device (h2b_permutation_sigma_dev, h2b_permutation_build_vk / build_pk) and of
keygen_pk's indicator columns; needs a B200.

    python tools/permutation_keygen_bench.py [--cases 16:4,16:8,16:16,20:4,20:8,20:16,22:4,22:8] [--reps 20] [--baseline] [--out FILE]

One JSON line per measurement (stdout, and appended to --out):
  * device   : card name, power limit and max SM clock, read in this invocation
  * sigma    : the sigma kernel alone on device-resident mapping columns (mean over --reps calls, host clock around calls that end in a
               device synchronise), against the HBM roofline: 16 B read + 32 B written per entry at 7.7 TB/s
  * phases   : device time per phase of one build_vk and one build_pk call from the profiling tags (31 upload, 32 sigma, 33 commitments,
               34 inverse NTTs, 35 coset NTTs, 36 downloads; MSM / NTT tags inside a phase are added to it)
  * calls    : wall time of build_vk and build_pk (all three outputs) with pageable numpy mapping arrays, and of lagrange_indicators
  * baseline : (--baseline) today's path: sigma by the CPU restatement of upstream's construction (tests/cpp/permutation_keygen_oracle.cpp)
               on 16 threads, then the existing host-pointer drop-ins: the batched registered MSM for the commitments and best_fft per
               column for the conversions (the scalings on the host, as upstream does them)
Outputs of the device calls are checked against the oracle's sigma at k <= 16.  Nothing is written to the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

TAGS = {31: "upload", 32: "sigma", 33: "commit", 34: "intt", 35: "coset", 36: "download"}
HBM_BYTES_PER_S = 7.7e12


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


def random_mapping(rng, P, k):
    """valid (column, row) entries; the kernels' cost does not depend on the cycle structure"""
    n = 1 << k
    m = np.empty((P, n, 2), dtype=np.uint64)
    m[:, :, 0] = rng.integers(0, P, size=(P, n), dtype=np.uint64)
    m[:, :, 1] = rng.integers(0, n, size=(P, n), dtype=np.uint64)
    return m


def phases(L):
    out, pending = {v: 0.0 for v in TAGS.values()}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] += pending + v
            pending = 0.0
        else:
            pending += v
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="16:4,16:8,16:16,20:4,20:8,20:16,22:4,22:8")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--baseline", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import halo2_scaffold_b200 as h2
    import oracle_c as oc
    import test_permutation_keygen as t
    L = h2.load()
    L.init(0)
    emit(device_line(), a.out)
    rng = np.random.default_rng(1)
    for case in a.cases.split(","):
        k, P = (int(x) for x in case.split(":"))
        n = 1 << k
        c = t.Consts(L, k)
        mapping = random_mapping(rng, P, k)
        # sigma kernel alone
        dm = [L.dev_alloc(0, n * 16) for _ in range(P)]
        ds = [L.dev_alloc(0, n * 32) for _ in range(P)]
        st = L.dev_alloc(0, 4)
        try:
            for i in range(P):
                L.h2d(0, dm[i], np.ascontiguousarray(mapping[i]))
            for _ in range(3):
                L.permutation_sigma_dev(0, dm, k, c.delta, c.omega, ds, st)
            L.dev_sync(0)
            t0 = time.perf_counter()
            for _ in range(a.reps):
                L.permutation_sigma_dev(0, dm, k, c.delta, c.omega, ds, st)
            L.dev_sync(0)
            ms = (time.perf_counter() - t0) * 1e3 / a.reps
            status = np.zeros(1, dtype=np.uint32)
            L.d2h(0, status, st)
            assert status[0] == 0
            if k <= 16:
                want = np.empty((P, n, 4), dtype=np.uint64)
                t.oracle().orc_permutation_sigma(mapping.ctypes.data, P, k, c.delta.ctypes.data, c.omega.ctypes.data, 16, want.ctypes.data)
                for i in range(P):
                    got = np.empty((n, 4), dtype=np.uint64)
                    L.d2h(0, got, ds[i])
                    assert (got == want[i]).all()
        finally:
            for p in dm + ds + [st]:
                L.dev_free(0, p)
        roof = 48.0 * P * n / HBM_BYTES_PER_S * 1e3
        emit(dict(kind="sigma", k=k, P=P, ms=round(ms, 4), hbm_roofline_ms=round(roof, 4), share_of_hbm_roofline=round(roof / ms, 3),
                  note="includes the twiddle-table build (one per call) and launch overhead"), a.out)
        # end-to-end calls and their phases
        pts = oc.gen_points(7, n)
        h = L.register_bases(pts)
        try:
            cols = [np.ascontiguousarray(mapping[i]) for i in range(P)]
            L.permutation_build_vk(cols, k, c.delta, c.omega, h)           # warm-up (MSM plan, NTT twiddles)
            L.permutation_build_pk(cols, k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            L.profile_enable(True)
            L.permutation_build_vk(cols, k, c.delta, c.omega, h)
            ph_vk = phases(L)
            L.profile_enable(True)
            L.permutation_build_pk(cols, k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            ph_pk = phases(L)
            L.profile_enable(False)
            emit(dict(kind="phases", k=k, P=P, extended_k=c.ek, build_vk_ms=ph_vk, build_pk_ms=ph_pk,
                      note="device 0 only; downloads are synchronous host copies, so 'download' includes their host time"), a.out)
            t0 = time.perf_counter()
            L.permutation_build_vk(cols, k, c.delta, c.omega, h)
            vk_ms = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            L.permutation_build_pk(cols, k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            pk_ms = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            L.keygen_lagrange_indicators(k, c.ek, 5, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            ind_ms = (time.perf_counter() - t0) * 1e3
            emit(dict(kind="calls", k=k, P=P, extended_k=c.ek, devices=L.device_count(), build_vk_ms=round(vk_ms, 2), build_pk_ms=round(pk_ms, 2),
                      lagrange_indicators_ms=round(ind_ms, 2)), a.out)
            if a.baseline:
                t0 = time.perf_counter()
                sig = np.empty((P, n, 4), dtype=np.uint64)
                t.oracle().orc_permutation_sigma(mapping.ctypes.data, P, k, c.delta.ctypes.data, c.omega.ctypes.data, 16, sig.ctypes.data)
                sigma_ms = (time.perf_counter() - t0) * 1e3
                t0 = time.perf_counter()
                L.msm_batch_registered(list(sig), h)
                commit_ms = (time.perf_counter() - t0) * 1e3
                t0 = time.perf_counter()
                en = 1 << c.ek
                zs = [c.zeta[i] for i in range(3)]
                for i in range(P):
                    a_ = np.ascontiguousarray(sig[i])
                    L.ntt(a_, c.omega_inv, k)
                    a_ = oc.fr_scale(a_, c.ifft)
                    ext = np.zeros((en, 4), dtype=np.uint64)
                    for r in range(3):
                        ext[r:n:3] = oc.fr_scale(np.ascontiguousarray(a_[r::3]), zs[r])
                    L.ntt(ext, c.ext_omega, c.ek)
                convert_ms = (time.perf_counter() - t0) * 1e3
                emit(dict(kind="baseline", k=k, P=P, cpu_sigma_16_threads_ms=round(sigma_ms, 2), dropin_commit_ms=round(commit_ms, 2),
                          dropin_convert_ms=round(convert_ms, 2), build_vk_equivalent_ms=round(sigma_ms + commit_ms, 2),
                          build_pk_equivalent_ms=round(sigma_ms + convert_ms, 2),
                          note="conversions: best_fft drop-in per column with the scalings on the host (single thread)"), a.out)
        finally:
            L.unregister_bases(h)


if __name__ == "__main__":
    main()
