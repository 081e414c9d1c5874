"""Timing of the SHPLONK opening on the device (h2b_shplonk_*, h2b_fr_eval_queries_dev); needs a B200.

    python tools/shplonk_bench.py [--shapes k16,k20,lr22] [--reps 3] [--oracle-k 20] [--out FILE]

Shapes: the three circuits of tools/proof_pipeline_core.py SHAPES (halo2_lib k = 16, linear_regression k = 20, logistic_regression
k = 22), with the query structure of tests/test_shplonk.py's lr_structure (lr22: 36 polynomials, 65 queries, 5 rotation sets).
One JSON line per measurement (stdout, and appended to --out):
  * device   : card name, power limit and max SM clock, read in this invocation
  * resident : begin + finish with device-resident polynomials, wall time (best / median of --reps), and the device phases of one run
               (profiling tags 44 evaluations, 45 scalars, 46 numerators and divisions, 47 MSM, 48 linearisation)
  * host     : begin + finish from pageable host arrays (the upload included), wall time
  * eval     : h2b_fr_eval_queries_dev against one h2b_fr_eval_polynomial_dev per query, wall time after a device synchronise
  * oracle   : tests/cpp/shplonk_oracle.cpp (upstream's algorithm on the CPU) for the same opening at --oracle-k, one run
Every timed h1 / h2 equals the first one, which satisfies the trapdoor identity of tests/test_shplonk.py.  Nothing is written to the tree.
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
from proof_pipeline_core import SHAPES as PIPELINE_SHAPES  # noqa: E402

TAGS = {43: "upload", 44: "evaluations", 45: "scalars", 46: "numerators_and_divisions", 47: "msm", 48: "linearisation"}
SHAPES = {"k16": "halo2_lib_k16", "k20": "linear_regression_k20", "lr22": "logistic_regression_k22"}


def phases(L):
    out, pending = {}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] = out.get(TAGS[t], 0.0) + pending + v
            pending = 0.0
        else:
            pending += v
    return {k: round(v, 3) for k, v in out.items()}


def make_case(oc, shape, seed):
    import bn254 as o
    import test_shplonk as ts
    sh = PIPELINE_SHAPES[shape]
    k = sh["k"]
    c = ts.Case.__new__(ts.Case)
    rng = np.random.default_rng(seed)
    c.k, c.n = k, 1 << k
    c.P, q = ts.lr_structure(sh["A"], sh["LK"], sh["d"])
    c.polys = [oc.random_fr(seed * 100 + i, c.n) for i in range(c.P)]
    R = o.R_MOD
    c.x = int(rng.integers(1, 1 << 62)) * 7919 % R
    w = o.omega_for(k)
    c.queries = [(p, c.x * pow(w, r % c.n, R) % R) for p, r in q]
    c.y, c.v, c.u = (int(rng.integers(1, 1 << 62)) * 104729 % R for _ in range(3))
    c.s = int(rng.integers(2, 1 << 62)) * 65537 % R
    return c


def timed(fn, reps):
    t, outs = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        outs.append(fn())
        t.append((time.perf_counter() - t0) * 1e3)
    return round(min(t), 2), round(float(np.median(t)), 2), outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="k16,k20,lr22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-k", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import oracle_c as oc
    import test_shplonk as ts
    from halo2_scaffold_b200 import load
    oc.build()
    L = load()
    L.init_device(0)
    emit(device_line(), a.out)
    for name in a.shapes.split(","):
        shape = SHAPES[name]
        c = make_case(oc, shape, 22)
        srs = L.srs_setup(c.k, ts._w(c.s))
        g, handle = srs["g"], srs["handle_g"]
        ptrs = ts.device_polys(L, c)
        try:
            ts.device_open(L, c, handle, on_host=False, ptrs=ptrs)          # warm-up: scratch, module load
            best, med, outs = timed(lambda: ts.device_open(L, c, handle, on_host=False, ptrs=ptrs), a.reps)
            h1, h2 = outs[0]
            verified = ts.trapdoor_holds(oc, c, g, h1, h2)
            aff = lambda j: oc.g1_to_affine(j).tobytes()      # Jacobian coordinates depend on the MSM's accumulation order
            same = all(aff(x) == aff(h1) and aff(y) == aff(h2) for x, y in outs)
            L.profile_enable(True)
            ts.device_open(L, c, handle, on_host=False, ptrs=ptrs)
            ph = phases(L)
            L.profile_enable(False)
            emit(dict(kind="resident", shape=name, k=c.k, polys=c.P, queries=len(c.queries), sets=len(ts.sets_of(c)), best_ms=best, median_ms=med,
                      phases_ms=ph, trapdoor=verified, all_equal=same), a.out)
            hb, hm, houts = timed(lambda: ts.device_open(L, c, handle, on_host=True), a.reps)
            emit(dict(kind="host", shape=name, k=c.k, best_ms=hb, median_ms=hm, bytes=c.P * c.n * 32,
                      all_equal=all(aff(x) == aff(h1) and aff(y) == aff(h2) for x, y in houts)), a.out)
            nq = len(c.queries)
            d_out = L.dev_alloc(0, nq * 32)
            try:
                def batched():
                    L.eval_queries_dev(0, ptrs, c.n, c.indexed(), d_out)
                    L.dev_sync(0)

                def single():
                    for i, (p, x) in enumerate(c.indexed()):
                        L.check(L.L.h2b_fr_eval_polynomial_dev(0, ptrs[p], c.n, x.ctypes.data, d_out + 32 * i, None))
                    L.dev_sync(0)
                batched()
                single()
                eb, em, _ = timed(batched, a.reps)
                sb, sm, _ = timed(single, a.reps)
                got = np.empty((nq, 4), dtype=np.uint64)
                batched()
                L.d2h(0, got, d_out)
                ok = all((got[i] == oc.fr_eval_polynomial(c.polys[p], x)).all() for i, (p, x) in enumerate(c.indexed()))
                emit(dict(kind="eval", shape=name, k=c.k, queries=nq, eval_queries_best_ms=eb, eval_queries_median_ms=em,
                          per_query_calls_best_ms=sb, per_query_calls_median_ms=sm, equal_to_oracle=ok), a.out)
            finally:
                L.dev_free(0, d_out)
            if c.k == a.oracle_k:
                t0 = time.perf_counter()
                st, w1, w2 = ts.orc_shplonk(c, g)
                ms = (time.perf_counter() - t0) * 1e3
                emit(dict(kind="oracle", shape=name, k=c.k, threads=ts.threads(), ms=round(ms, 1),
                          equal=bool(st == 0 and (oc.g1_to_affine(w1) == oc.g1_to_affine(h1)).all() and (oc.g1_to_affine(w2) == oc.g1_to_affine(h2)).all())),
                     a.out)
        finally:
            for d in ptrs:
                L.dev_free(0, d)
            L.unregister_bases(handle)
            L.unregister_bases(srs["handle_g_lagrange"])


if __name__ == "__main__":
    main()
