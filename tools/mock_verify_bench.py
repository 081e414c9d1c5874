"""Timing of MockProver::verify's row loops on the device (h2b_mock_verify) against the CPU oracle; needs a B200.

    python tools/mock_verify_bench.py [--ks 16,20,22] [--reps 5] [--out FILE]

Shapes (tests/mock_cases.py): halo2_lib -- halo2-lib's q (a + b c - d) gate over rotations 0..3, a standard-plonk gate, a range lookup
(m = 1) and copy constraints over four columns; m3 -- the same plus a lookup of three-element tuples.  Satisfied witnesses, so the call
writes no records.  One JSON line per measurement (stdout, and appended to --out):
  * device : card name, power limit and max SM clock, read in this invocation
  * call   : h2b_mock_verify from pageable host columns, wall time (best / median of --reps), the device phases (profiling tags 49
             uploads, 50 gate check, 51 lookups, 52 copy constraints, 53 scans and records; the median of each over --reps further
             profiled calls, taken apart from the timed ones) and the cost model's inputs
             (bytes uploaded, Fr multiplications of the gate program per row, bitonic passes of the lookups, copy cells)
  * oracle : tests/cpp/mock_verify_oracle.cpp (upstream's three loops over expression trees) on every host core, one run
Neither time includes building the circuit or flattening it for the call; both report the same failures (none).  Nothing is written to
the tree.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from permutation_keygen_bench import device_line, emit  # noqa: E402

TAGS = {49: "upload", 50: "gates", 51: "lookups", 52: "copies", 53: "scans_and_records"}
MUL_OPS = (2, 3)          # h2b_calc_op MUL, SQUARE


def phases(L):
    out, pending = {}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] = out.get(TAGS[t], 0.0) + pending + v
            pending = 0.0
        else:
            pending += v
    return {k: round(v, 3) for k, v in out.items()}


def model(c):
    """the cost model's inputs for circuit c"""
    from halo2_scaffold_b200 import mock
    n, u = c.n, c.usable
    graph, _ = mock.compile_gates(c.gates)
    muls = int(sum(1 for row in graph.calculations if row[0] in MUL_OPS))
    cols = len(c.fixed) + len(c.advice) + len(c.instance)
    upload = 32 * n * cols + ((n + 7) // 8) * (len(c.fixed) + len(c.advice)) + 16 * n * len(c.permutation)
    padded = max(1024, 1 << (u - 1).bit_length())
    lg = padded.bit_length() - 1
    passes = []
    for ins, _ in c.lookups:
        passes.append(("keys_bitonic" if len(ins) == 1 else "index_bitonic", lg * (lg + 1) // 2))
    return dict(upload_bytes=upload, gate_fr_muls_per_row=muls, gate_fr_muls=muls * n, lookup_passes=passes,
                copy_cells=len(c.permutation) * n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="16,20,22")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import oracle_c as oc
    oc.build()
    import mock_cases as mc
    from halo2_scaffold_b200 import load
    L = load()
    L.init(1)
    emit(device_line(), a.out)
    for k in [int(x) for x in a.ks.split(",")]:
        for shape in ("halo2_lib", "m3"):
            c = mc.halo2_lib(k, 1000 + k, m3=shape == "m3")
            args = c.raw_args()
            times = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                count, _ = L.mock_verify(0, *args, capacity=1024)
                times.append((time.perf_counter() - t0) * 1e3)
                assert count == 0
            runs = []
            L.profile_enable(True, 0)
            for _ in range(a.reps):
                L.mock_verify(0, *args, capacity=1024)
                runs.append(phases(L))
            L.profile_enable(False, 0)
            ph = {t: round(float(np.median([r.get(t, 0.0) for r in runs])), 3) for t in TAGS.values()}
            spread = {t: [min(r.get(t, 0.0) for r in runs), max(r.get(t, 0.0) for r in runs)] for t in TAGS.values()}
            times.sort()
            emit(dict(kind="call", shape=shape, k=k, best_ms=round(times[0], 2), median_ms=round(times[len(times) // 2], 2), phases_ms=ph,
                      phases_min_max_ms=spread, profiled_runs=a.reps,
                      **model(c)), a.out)
            t0 = time.perf_counter()
            total, _ = c.oracle(threads=os.cpu_count() or 1)
            emit(dict(kind="oracle", shape=shape, k=k, ms=round((time.perf_counter() - t0) * 1e3, 1), threads=os.cpu_count(), failures=total),
                 a.out)


if __name__ == "__main__":
    main()
