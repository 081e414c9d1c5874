"""Timing of the GWC opening on the device (h2b_gwc_create_proof); needs a B200.

    python tools/gwc_bench.py [--shapes k16,k20,lr22] [--reps 5] [--oracle-k 20] [--out FILE]

Shapes and query structures are those of tools/shplonk_bench.py (tools/proof_pipeline_core.py SHAPES with tests/test_shplonk.py's
lr_structure; lr22: n = 2^22, 36 polynomials, 65 queries, 6 distinct points).  One JSON line per measurement (stdout, and appended to
--out):
  * device   : card name, power limit and max SM clock, read in this invocation
  * resident : h2b_gwc_create_proof on device-resident polynomials, wall time (best / median of --reps), and the median of each device
               phase over --reps profiled calls (tags 55 v powers, 56 numerators, 57 divisions, 58 MSMs)
  * host     : the same from pageable host arrays (tag 54: the upload), wall time and phase medians
  * per_point: the same opening composed of existing entry points, per point one h2b_fr_lincomb_dev, one h2b_fr_kate_division_dev and
               one h2b_msm_bn254_g1_dev_registered, wall time: what the batched divisions and MSMs replace
  * shplonk  : the SHPLONK opening (h2b_shplonk_begin + finish) of the same queries on the same resident polynomials, wall time
  * oracle   : tests/cpp/gwc_oracle.cpp (upstream's algorithm on the CPU) at --oracle-k, one run
Every timed result equals the first one, which satisfies the trapdoor identity of tests/test_gwc.py.  Nothing is written to the tree.
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
from shplonk_bench import SHAPES, make_case, timed  # noqa: E402

TAGS = {54: "upload", 55: "v_powers", 56: "numerators", 57: "divisions", 58: "msm"}


def phases(L):
    """one profiled call -> {phase: ms}; the MSM's own tags count towards the GWC tag that follows them"""
    out, pending = {}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] = out.get(TAGS[t], 0.0) + pending + v
            pending = 0.0
        else:
            pending += v
    return out


def phase_medians(L, fn, reps):
    runs = []
    L.profile_enable(True)
    try:
        for _ in range(reps):
            fn()
            runs.append(phases(L))
    finally:
        L.profile_enable(False)
    return {k: round(float(np.median([r.get(k, 0.0) for r in runs])), 3) for k in runs[0]}


def per_point(L, c, ptrs, handle, d_num, d_q, d_blocks):
    """the opening through one lincomb, one kate_division and one registered MSM per point -> [W]"""
    import bn254
    from halo2_scaffold_b200._lib import _ptr_array
    from test_shplonk import _w
    pts = c.points()
    for i, (z, ps) in enumerate(pts):
        coeffs = np.stack([_w(pow(c.v, j, bn254.R_MOD)) for j in range(len(ps))])
        cols = _ptr_array([ptrs[p] for p in ps])
        L.check(L.L.h2b_fr_lincomb_dev(0, cols, coeffs.ctypes.data, len(ps), c.n, d_num, None))
        zw = _w(z)
        L.check(L.L.h2b_fr_kate_division_dev(0, d_num, c.n, zw.ctypes.data, d_q, None))
        L.check(L.L.h2b_msm_bn254_g1_dev_registered(0, d_q, handle, 0, c.n - 1, d_blocks + 224 * i, None))
    blocks = np.empty((len(pts), 28), dtype=np.uint64)
    L.dev_sync(0)
    L.d2h(0, blocks, d_blocks)
    return blocks[:, :12].copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="k16,k20,lr22")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-k", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import oracle_c as oc
    import test_gwc as tg
    import test_shplonk as ts
    from halo2_scaffold_b200 import load
    oc.build()
    L = load()
    L.init_device(0)
    emit(device_line(), a.out)
    for name in a.shapes.split(","):
        sc = make_case(oc, SHAPES[name], 22)
        c = tg.Case.__new__(tg.Case)
        c.__dict__.update(sc.__dict__)
        srs = L.srs_setup(c.k, ts._w(c.s))
        g, handle = srs["g"], srs["handle_g"]
        ptrs = ts.device_polys(L, c)
        d_num, d_q, d_blocks = L.dev_alloc(0, c.n * 32), L.dev_alloc(0, c.n * 32), L.dev_alloc(0, 224 * len(c.points()))
        aff = lambda ws: b"".join(oc.g1_to_affine(w).tobytes() for w in ws)      # Jacobian coordinates depend on the MSM's order
        try:
            resident = lambda: L.gwc_create_proof(0, ptrs, False, c.n, c.indexed(), handle, ts._w(c.v))
            host = lambda: L.gwc_create_proof(0, c.polys, True, c.n, c.indexed(), handle, ts._w(c.v))
            W = resident()                                                       # warm-up: scratch, module load
            verified = tg.trapdoor_holds(oc, c, g, W)
            best, med, outs = timed(resident, a.reps)
            emit(dict(kind="resident", shape=name, k=c.k, polys=c.P, queries=len(c.queries), points=len(c.points()), best_ms=best, median_ms=med,
                      phases_ms=phase_medians(L, resident, a.reps), trapdoor=verified, all_equal=all(aff(o) == aff(W) for o in outs)), a.out)
            host()
            hb, hm, houts = timed(host, a.reps)
            emit(dict(kind="host", shape=name, k=c.k, best_ms=hb, median_ms=hm, bytes=c.P * c.n * 32, phases_ms=phase_medians(L, host, a.reps),
                      all_equal=all(aff(o) == aff(W) for o in houts)), a.out)
            pp = lambda: per_point(L, c, ptrs, handle, d_num, d_q, d_blocks)
            pp()
            pb, pm, pouts = timed(pp, a.reps)
            emit(dict(kind="per_point", shape=name, k=c.k, best_ms=pb, median_ms=pm, all_equal=all(aff(o) == aff(W) for o in pouts)), a.out)
            sh = lambda: ts.device_open(L, sc, handle, on_host=False, ptrs=ptrs)
            h1, h2 = sh()
            sb, sm, souts = timed(sh, a.reps)
            emit(dict(kind="shplonk", shape=name, k=c.k, best_ms=sb, median_ms=sm, trapdoor=ts.trapdoor_holds(oc, sc, g, h1, h2),
                      all_equal=all(aff(o) == aff((h1, h2)) for o in souts)), a.out)
            if c.k == a.oracle_k:
                t0 = time.perf_counter()
                want = tg.orc_gwc(c, g)
                ms = (time.perf_counter() - t0) * 1e3
                emit(dict(kind="oracle", shape=name, k=c.k, threads=ts.threads(), ms=round(ms, 1), equal=aff(want) == aff(W)), a.out)
        finally:
            for d in ptrs + [d_num, d_q, d_blocks]:
                L.dev_free(0, d)
            L.unregister_bases(handle)
            L.unregister_bases(srs["handle_g_lagrange"])


if __name__ == "__main__":
    main()
