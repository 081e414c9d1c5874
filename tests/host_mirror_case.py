"""Builds tests/cpp/host_mirror_test.cpp against a given libh2b200 build, runs it on seeded inputs and checks every
output file against the oracle (shared by the CPU emulator test and the GPU test)."""
import subprocess

import numpy as np

import bn254 as o
import parity_cases as pc
from harness import build_mirror


def run_host_mirror(oc, lib_path, tmp_path, k=6, j=4):
    n = 1 << k
    exe = build_mirror("host_mirror_test", lib_path, tmp_path)
    s, P, lag = oc.random_fr(0xC0 + k, n), oc.gen_points(0xC1 + k, n), oc.random_fr(0xC2 + k, n)
    s[1] = 0
    P[2] = 0
    rows = 64
    ecols = [oc.random_fr(0xD0 + i, rows) for i in range(6)]
    esc = oc.random_fr(0xDF, 8)
    pool = oc.random_fr(0xE0, 20)
    rng = np.random.default_rng(k)
    ltab = pool[np.concatenate([np.arange(20), rng.integers(0, 20, size=44)])]
    lin = ltab[:58][rng.integers(0, 58, size=64)]
    for name, arr in (("scalars", s), ("bases", P), ("lagrange", lag), ("eval_cols", np.concatenate(ecols)), ("eval_scalars", esc),
                      ("lookup_input", lin), ("lookup_table", ltab)):
        np.ascontiguousarray(arr).tofile(str(tmp_path / (name + ".bin")))
    out = subprocess.run([exe, str(tmp_path), str(j), str(k)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "HOST_MIRROR_OK" in out.stdout, (out.stdout, out.stderr)

    def rd(name, cols):
        return np.fromfile(str(tmp_path / (name + ".bin")), dtype=np.uint64).reshape(-1, cols)

    assert (pc.affine_of(oc, rd("msm", 12)[0]) == pc.affine_of(oc, oc.best_multiexp(s, P))).all()
    dom = o.EvaluationDomain(j, k)
    lag_i = [o.from_mont(v, o.R_MOD) for v in oc.words_to_ints(lag)]
    coeff = dom.lagrange_to_coeff(list(lag_i))
    ext = dom.coeff_to_extended(list(coeff))
    back = dom.extended_to_coeff(list(ext))

    def words(vals):
        return oc.ints_to_words([o.to_mont(v, o.R_MOD) for v in vals])

    assert (rd("coeff", 4) == words(coeff)).all()
    assert (rd("extended", 4) == words(ext)).all()
    assert (rd("back", 4) == words(back)).all()
    assert (rd("fft", 4) == oc.best_fft(lag, pc.omega_words(oc, k), k)).all()
    # the widened rows
    want_div = words(dom.divide_by_vanishing_poly(list(ext)))
    assert (rd("divided", 4) == want_div).all()
    assert (pc.affine_of(oc, rd("commit_after_read", 12)[0]) == pc.affine_of(oc, oc.best_multiexp(s, P))).all()
    # the graph the C++ driver builds through add_calculation, restated in the flat encoding for the oracle
    consts = oc.fr_to_mont(np.array([[0, 0, 0, 0], [1, 0, 0, 0], [2, 0, 0, 0], [0x1234567, 0, 0, 0]], dtype=np.uint64))
    calcs = [[7, 0, 2, 0, 0, 0, 0, 0, 0, 0], [2, 1, 3, 1, 1, 3, 2, 0, 0, 0], [0, 2, 3, 0, 0, 1, 1, 0, 0, 0], [1, 3, 1, 2, 0, 3, 0, 2, 0, 0],
             [2, 4, 1, 0, 0, 1, 3, 0, 0, 0], [3, 5, 1, 4, 0, 0, 0, 0, 0, 0], [2, 6, 4, 0, 0, 0, 3, 0, 0, 0], [6, 7, 10, 0, 0, 9, 0, 0, 0, 4]]
    parts = [[1, 4, 0], [1, 5, 0], [1, 6, 0], [5, 0, 0]]
    graph = (consts, np.array([0, 1, -1], dtype=np.int32), np.array(calcs, dtype=np.uint32), np.array(parts, dtype=np.uint32), 8)
    want = oc.evaluate_graph(graph, ecols[:1], ecols[1:4], ecols[4:5], esc[:1], esc[1], esc[2], esc[3], esc[4], ecols[5], 2)
    assert (rd("eval_out", 4) == want).all()
    w6 = pc.omega_words(oc, 6)
    assert (rd("perm_z", 4) == oc.permutation_product(ecols[1:3], ecols[3:5], esc[1], esc[2], esc[5], esc[6], w6, esc[7])).all()
    assert (rd("lookup_z", 4) == oc.lookup_product(ecols[1], ecols[2], ecols[3], ecols[4], esc[1], esc[2])).all()
    wa, wt = oc.lookup_permute(lin, ltab, 58)
    assert (rd("permuted_input", 4) == wa).all() and (rd("permuted_table", 4) == wt).all()
    c = rd("commit", 12)
    assert (pc.affine_of(oc, c[0]) == pc.affine_of(oc, oc.best_multiexp(s, P))).all()
    h = n // 2
    assert (pc.affine_of(oc, c[1]) == pc.affine_of(oc, oc.best_multiexp(s[:h], P[:h]))).all()
    # batched commitments and the one-upload column pipeline of the C++ mirror
    many = rd("commit_many", 12)
    for got, col in zip(many, (s, s[:h], lag)):
        assert (pc.affine_of(oc, got) == pc.affine_of(oc, oc.best_multiexp(col, P[:col.shape[0]]))).all()
    assert (pc.affine_of(oc, rd("pipeline_commit", 12)[0]) == pc.affine_of(oc, oc.best_multiexp(lag, P))).all()
    assert (rd("pipeline_coeff", 4) == words(coeff)).all()
    assert (rd("pipeline_extended", 4) == words(ext)).all()
