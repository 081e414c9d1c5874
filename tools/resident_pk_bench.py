"""Timing of the proving key resident on the devices (h2b_pk_*); needs a B200.

    python tools/resident_pk_bench.py [--shapes k16,k20,lr22] [--reps 3] [--out FILE]

Shapes, with extended_k = k + 2 and bf = 5:
  * lr22 : the logistic_regression_k22 shape of tools/proof_pipeline_core.py (A = 6, LK = 2): 7 fixed columns (5 of the caller's and 2
           combination columns of 4 disjoint degree-3 selectors), 8 sigma columns, the 3 indicators, k = 22
  * k16 / k20 : the same column counts at k = 16 / 20
One JSON line per measurement (stdout, and appended to --out):
  * device     : card name, power limit and max SM clock, read in this invocation
  * keygen     : (a) keygen_pk's fixed, sigma and indicator columns into host arrays (h2b_keygen_fixed_build_pk, h2b_permutation_build_pk,
                 h2b_keygen_lagrange_indicators_dev + download) against the same into a resident pk (h2b_pk_create and the three resident
                 builds): wall time (best of --reps) and device phases of one call each on device 0 (profiling tags 33 - 42)
  * per_proof  : (b) what a proof no longer pays with the pk resident: uploading the columns create_proof's device steps read (every extended
                 coset, the sigma values of the permutation product and the coefficient forms of the opening) from pageable and from pinned
                 host arrays
  * put        : (c) h2b_pk_put_lagrange of every fixed and sigma column from pageable arrays, plus the indicators
  * memory     : (d) bytes per device in both layouts, at one device and at every visible device
Contents are checked against the host outputs at k <= 16.  Nothing is written to the tree.
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

TAGS = {31: "mapping_upload", 32: "sigma", 34: "intt", 35: "coset", 36: "download", 37: "pack", 39: "fixed_upload", 40: "combination",
        41: "form_copies", 42: "placement"}
SHAPES = {"k16": 16, "k20": 20, "lr22": 22}
N_CALLER_FIXED, N_SELECTORS, N_SIGMA, BF = 5, 4, 8, 5


def phases(L):
    out, pending = {v: 0.0 for v in TAGS.values()}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] += pending + v
            pending = 0.0
        else:
            pending += v
    return {k: round(v, 3) for k, v in out.items() if v}


def inputs(oc, k, seed):
    from halo2_scaffold_b200 import keygen as kg
    n = 1 << k
    rng = np.random.default_rng(seed)
    fixed = [oc.random_fr(seed * 7 + i, n) for i in range(N_CALLER_FIXED)]
    acts = np.zeros((N_SELECTORS, n), dtype=np.uint8)
    for s in range(N_SELECTORS):
        acts[s, s::N_SELECTORS] = 1
    # the identity mapping with random disjoint pairs of cells swapped: a valid permutation of 2-cycles
    mapping = np.zeros((N_SIGMA, n, 2), dtype=np.uint64)
    mapping[:, :, 0] = np.arange(N_SIGMA, dtype=np.uint64)[:, None]
    mapping[:, :, 1] = np.arange(n, dtype=np.uint64)[None, :]
    cells = rng.permutation(N_SIGMA * n)[: 2 * (n // 4)].reshape(-1, 2)
    flat = mapping.reshape(-1, 2)
    flat[cells[:, 0]], flat[cells[:, 1]] = flat[cells[:, 1]].copy(), flat[cells[:, 0]].copy()
    return fixed, list(acts), mapping, kg


def best(fn, reps):
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return round(min(t), 2), round(float(np.median(t)), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="k16,k20,lr22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    import halo2_scaffold_b200 as h2
    import oracle_c as oc
    import test_permutation_keygen as tp
    L = h2.load()
    L.init(0)
    emit(device_line(), a.out)
    for name in a.shapes.split(","):
        k = SHAPES[name]
        c = tp.Consts(L, k)
        n, E = 1 << k, 1 << c.ek
        fixed, acts, mapping, kg = inputs(oc, k, 3)
        asg = kg.compress_selectors(acts, [3] * N_SELECTORS, 4, lib=L)
        F, P = N_CALLER_FIXED + asg["n_combinations"], N_SIGMA
        fx_args = (fixed, acts, asg["combination_of"], asg["root_of"], asg["n_combinations"], k)
        pk_consts = (c.ek, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
        host = {}

        def host_keygen():
            host["fixed"] = L.keygen_fixed_build_pk(*fx_args, *pk_consts)
            host["perm"] = L.permutation_build_pk(mapping, k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            host["ind"] = L.keygen_lagrange_indicators(k, c.ek, BF, c.omega_inv, c.ifft, c.ext_omega, c.zeta)

        def resident_keygen(layout="replicated", keep=False):
            pk = kg.ResidentProvingKey(c.dom, F, P, layout, lib=L)
            pk.build_fixed(fixed, acts, asg)
            pk.build_permutation(mapping)
            pk.build_indicators(BF)
            if keep:
                return pk
            pk.close()

        host_keygen()                   # warm-up: twiddles, staging, kernel loads
        resident_keygen()
        host_ms = best(host_keygen, a.reps)
        res_ms = best(resident_keygen, a.reps)
        L.profile_enable(True)
        host_keygen()
        ph_host = phases(L)
        L.profile_enable(True)
        resident_keygen()
        ph_res = phases(L)
        L.profile_enable(False)
        pk = resident_keygen(keep=True)
        try:
            if k <= 16:
                for i in range(F):
                    vals = fixed[i] if i < N_CALLER_FIXED else host["fixed"]["combination_values"][i - N_CALLER_FIXED]
                    assert (pk.download("fixed", "values", i) == vals).all()
                    assert (pk.download("fixed", "coeff", i) == host["fixed"]["polys"][i]).all()
                    assert (pk.download("fixed", "extended", i) == host["fixed"]["cosets"][i]).all()
                for i in range(P):
                    for form, key in (("values", "permutations"), ("coeff", "polys"), ("extended", "cosets")):
                        assert (pk.download("permutation", form, i) == host["perm"][key][i]).all()
                for i in range(3):
                    assert (pk.download("indicators", "extended", i) == host["ind"][i]).all()
            ext_bytes, n_bytes = (F + P + 3) * E * 32, 2 * (F + P) * n * 32
            emit(dict(kind="keygen", shape=name, k=k, extended_k=c.ek, F=F, P=P, devices=L.device_count(), host_output_ms=host_ms,
                      resident_ms=res_ms, host_output_phases_ms=ph_host, resident_phases_ms=ph_res, pk_bytes=ext_bytes + n_bytes,
                      note="(best, median) of reps; phases of device 0; host outputs land in pageable numpy arrays"), a.out)
            host = {}
            # (b) the uploads a proof pays without the resident pk
            d_buf = L.dev_alloc(0, E * 32)
            try:
                page_ext, page_n = np.ones((E, 4), dtype=np.uint64), np.ones((n, 4), dtype=np.uint64)
                pin_ext = torch.ones((E, 4), dtype=torch.int64).pin_memory().numpy()
                pin_n = torch.ones((n, 4), dtype=torch.int64).pin_memory().numpy()
                up = {}
                for label, ea, na in (("pageable", page_ext, page_n), ("pinned", pin_ext, pin_n)):
                    def upload():
                        for _ in range(F + P + 3):
                            L.h2d(0, d_buf, ea)
                        for _ in range(2 * (F + P)):
                            L.h2d(0, d_buf, na)
                    upload()
                    up[label] = best(upload, a.reps)
                emit(dict(kind="per_proof", shape=name, k=k, bytes=ext_bytes + n_bytes, extended_columns=F + P + 3, n_row_columns=2 * (F + P),
                          upload_pageable_ms=up["pageable"], upload_pinned_ms=up["pinned"],
                          gbps_pageable=round((ext_bytes + n_bytes) / up["pageable"][0] / 1e6, 1),
                          gbps_pinned=round((ext_bytes + n_bytes) / up["pinned"][0] / 1e6, 1),
                          note="one synchronous h2b_memcpy_h2d per column on device 0, (best, median) of reps"), a.out)
            finally:
                L.dev_free(0, d_buf)
            # (c) registering a pk built elsewhere
            values_f = [pk.download("fixed", "values", i) for i in range(F)]
            values_p = [pk.download("permutation", "values", i) for i in range(P)]

            def put():
                with kg.ResidentProvingKey(c.dom, F, P, lib=L) as pk2:
                    pk2.put_lagrange("fixed", values_f)
                    pk2.put_lagrange("permutation", values_p)
                    pk2.build_indicators(BF)
            put()
            put_ms = best(put, a.reps)
            L.profile_enable(True)
            put()
            ph_put = phases(L)
            L.profile_enable(False)
            emit(dict(kind="put", shape=name, k=k, F=F, P=P, put_lagrange_ms=put_ms, phases_ms=ph_put, note="create + put + indicators + release"),
                 a.out)
        finally:
            pk.close()
        # (d) bytes per device
        mem = {}
        for layout, halo in (("replicated", 0), ("row_sharded", 0 if L.device_count() == 1 else 64)):
            with kg.ResidentProvingKey(c.dom, F, P, layout, halo, lib=L) as p:
                mem[layout] = p.info()
        one = 32 * (2 * n * (F + P) + E * (F + P + 3))
        emit(dict(kind="memory", shape=name, k=k, devices=L.device_count(), one_device_bytes=one, replicated_per_device=mem["replicated"],
                  row_sharded_per_device=mem["row_sharded"], halo=0 if L.device_count() == 1 else 64), a.out)


if __name__ == "__main__":
    main()
