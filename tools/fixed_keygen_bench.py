"""Timing of compress_selectors' exclusion matrix and of the fixed columns of keygen_vk / keygen_pk on the device
(h2b_selector_exclusion, h2b_keygen_fixed_build_vk / build_pk); needs a B200.

    python tools/fixed_keygen_bench.py [--ks 16,20,22] [--reps 10] [--baseline] [--out FILE]

Two circuit shapes per k, with extended_k = k + 2:
  * halo2lib     : the halo2-lib shape of tools/proof_pipeline_core.py with A = 8 -- 8 gate selectors of degree 3, each on a random half of
                   the rows (they overlap, so nothing combines), and 2 fixed columns (constants, lookup table); max_degree 4
  * compressible : 32 selectors of degree 2 on disjoint rows (r mod 32), max_degree 5, so process combines them 4 to a column; 2 fixed columns
One JSON line per measurement (stdout, and appended to --out):
  * device    : card name, power limit and max SM clock, read in this invocation
  * exclusion : h2b_selector_exclusion with S = 64 sparse selectors: the call's wall time (pageable uploads and packing included) and the
                exclusion kernel's device time from its profiling tag (38), against the HBM bound of reading the S n / 8 bytes of bitsets
  * phases    : device time per phase of one build_vk and one build_pk call from the profiling tags (37 selector upload + packing,
                39 fixed upload, 40 combination kernel, 33 commitments, 34 inverse NTTs, 35 coset NTTs, 36 downloads; MSM / NTT tags inside
                a phase are added to it)
  * calls     : wall time of compress_selectors (device exclusion + host greedy) and of build_vk / build_pk (all outputs) with pageable arrays
  * baseline  : (--baseline) today's path: the CPU restatement of upstream's process (tests/cpp/fixed_keygen_oracle.cpp, one thread, as
                upstream's is), then the existing drop-ins per column: the batched registered MSM for the commitments and best_fft per column
                for the conversions (the scalings on the host, as upstream does them)
Outputs of the device calls are checked against the oracle at k <= 16.  Nothing is written to the tree.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from permutation_keygen_bench import HBM_BYTES_PER_S, device_line, emit  # noqa: E402

TAGS = {37: "pack", 38: "exclusion", 39: "fixed_upload", 40: "combination", 33: "commit", 34: "intt", 35: "coset", 36: "download"}


def phases(L):
    out, pending = {v: 0.0 for v in TAGS.values()}, 0.0
    for t, v in L.profile_read():
        if t in TAGS:
            out[TAGS[t]] += pending + v
            pending = 0.0
        else:
            pending += v
    return {k: round(v, 3) for k, v in out.items() if v}


def shapes(oc, rng, k):
    n = 1 << k
    fixed = np.stack([oc.random_fr(11 + i, n) for i in range(2)])
    halo2lib = rng.random((8, n)) < 0.5
    comp = np.zeros((32, n), dtype=bool)
    for s in range(32):
        comp[s, s::32] = True
    return [("halo2lib", fixed, halo2lib.astype(np.uint8), [3] * 8, 4), ("compressible", fixed, comp.astype(np.uint8), [2] * 32, 5)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="16,20,22")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--baseline", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import halo2_scaffold_b200 as h2
    import oracle_c as oc
    import test_fixed_keygen as tf
    import test_permutation_keygen as tp
    from halo2_scaffold_b200 import keygen as kg
    L = h2.load()
    L.init(0)
    emit(device_line(), a.out)
    rng = np.random.default_rng(2)
    for k in (int(x) for x in a.ks.split(",")):
        n = 1 << k
        c = tp.Consts(L, k)
        # the exclusion matrix alone, S = 64
        S = 64
        acts = [np.ascontiguousarray(r, dtype=np.uint8) for r in (rng.random((S, n)) < 1.0 / 256)]
        L.selector_exclusion(acts, k)
        t0 = time.perf_counter()
        for _ in range(a.reps):
            got = L.selector_exclusion(acts, k)
        call_ms = (time.perf_counter() - t0) * 1e3 / a.reps
        L.profile_enable(True)
        L.selector_exclusion(acts, k)
        ph = phases(L)
        L.profile_enable(False)
        if k <= 16:
            assert (got == tf.orc_exclusion(np.stack(acts), k)).all()
        bound = S * n / 8 / HBM_BYTES_PER_S * 1e3
        emit(dict(kind="exclusion", k=k, S=S, call_ms=round(call_ms, 3), pack_ms=ph.get("pack"), kernel_ms=ph.get("exclusion"),
                  hbm_bound_ms=round(bound, 4), share_of_hbm_bound=round(bound / ph["exclusion"], 3) if ph.get("exclusion") else None,
                  note="kernel_ms includes the memset of the S x S flags; the bitsets (S n / 8 bytes) fit in L2"), a.out)
        pts = oc.gen_points(7, n)
        h = L.register_bases(pts)
        try:
            for name, fixed, sel, degrees, max_degree in shapes(oc, rng, k):
                cols = list(fixed)
                rows = list(sel)
                t0 = time.perf_counter()
                asg = kg.compress_selectors(rows, degrees, max_degree, lib=L)
                compress_ms = (time.perf_counter() - t0) * 1e3
                C = asg["n_combinations"]
                args = (cols, rows, asg["combination_of"], asg["root_of"], C, k)
                pk_args = args + (c.ek, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
                vk = L.keygen_fixed_build_vk(*args, h)                      # warm-up (MSM plan, NTT twiddles)
                pk = L.keygen_fixed_build_pk(*pk_args)
                if k <= 16:
                    co, ro, lo, comb_cols = tf.orc_compress(sel, degrees, max_degree, k)
                    assert (asg["combination_of"] == co).all() and (asg["root_of"] == ro).all()
                    jac, polys, cosets = tf.orc_fixed_build(np.concatenate([fixed, comb_cols]), c, pts)
                    assert (np.stack(pk["polys"]) == polys).all() and (np.stack(pk["cosets"]) == cosets).all()
                    assert (tp.affine(oc, vk) == tp.affine(oc, jac)).all()
                L.profile_enable(True)
                L.keygen_fixed_build_vk(*args, h)
                ph_vk = phases(L)
                L.profile_enable(True)
                L.keygen_fixed_build_pk(*pk_args)
                ph_pk = phases(L)
                L.profile_enable(False)
                emit(dict(kind="phases", k=k, shape=name, F=len(cols), S=len(rows), C=C, extended_k=c.ek, build_vk_ms=ph_vk, build_pk_ms=ph_pk,
                          note="device 0 only; downloads are synchronous host copies, so 'download' includes their host time"), a.out)
                t0 = time.perf_counter()
                L.keygen_fixed_build_vk(*args, h)
                vk_ms = (time.perf_counter() - t0) * 1e3
                t0 = time.perf_counter()
                L.keygen_fixed_build_pk(*pk_args)
                pk_ms = (time.perf_counter() - t0) * 1e3
                emit(dict(kind="calls", k=k, shape=name, F=len(cols), S=len(rows), C=C, extended_k=c.ek, devices=L.device_count(),
                          compress_selectors_ms=round(compress_ms, 2), build_vk_ms=round(vk_ms, 2), build_pk_ms=round(pk_ms, 2)), a.out)
                if a.baseline:
                    t0 = time.perf_counter()
                    _, _, _, comb_cols = tf.orc_compress(sel, degrees, max_degree, k)
                    process_ms = (time.perf_counter() - t0) * 1e3
                    all_cols = list(fixed) + list(comb_cols)
                    t0 = time.perf_counter()
                    L.msm_batch_registered(all_cols, h)
                    commit_ms = (time.perf_counter() - t0) * 1e3
                    t0 = time.perf_counter()
                    en = 1 << c.ek
                    zs = [c.zeta[i] for i in range(3)]
                    for col in all_cols:
                        a_ = np.ascontiguousarray(col)
                        L.ntt(a_, c.omega_inv, k)
                        a_ = oc.fr_scale(a_, c.ifft)
                        ext = np.zeros((en, 4), dtype=np.uint64)
                        for r in range(3):
                            ext[r:n:3] = oc.fr_scale(np.ascontiguousarray(a_[r::3]), zs[r])
                        L.ntt(ext, c.ext_omega, c.ek)
                    convert_ms = (time.perf_counter() - t0) * 1e3
                    emit(dict(kind="baseline", k=k, shape=name, cpu_process_ms=round(process_ms, 2), dropin_commit_ms=round(commit_ms, 2),
                              dropin_convert_ms=round(convert_ms, 2), keygen_vk_equivalent_ms=round(process_ms + commit_ms, 2),
                              keygen_pk_equivalent_ms=round(process_ms + convert_ms, 2),
                              note="process on one thread; conversions: best_fft drop-in per column with the scalings on the host (single thread)"),
                         a.out)
        finally:
            L.unregister_bases(h)


if __name__ == "__main__":
    main()
