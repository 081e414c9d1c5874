"""
CPU: the shipped kernel sources (csrc/*.cu) compiled for the kernel-logic emulator (tools/emu) and checked
against the oracle and the golden fixtures.  This exercises the real index math, sorting, bucket planning and
reduction code of the CUDA kernels at sizes a CPU finishes in seconds; the GPU tests repeat the same checks through
the C ABI on a B200 at full sizes.
"""
import numpy as np
import pytest

import parity_cases as pc
from harness import run_on_emulated_devices


def test_field_arithmetic(emu, oc):
    pc.check_field(emu, oc, 512)


def test_group_law_edge_cases(emu, oc):
    pc.check_group(emu, oc, 32)


def test_generators_match_oracle_streams(emu, oc):
    assert (emu.gen_points(7, 100) == oc.gen_points(7, 100)).all()
    assert (emu.gen_scalars(11, 300, 0) == oc.random_fr(11, 300)).all()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 7, 10, 11, 12, 13, 15])
def test_ntt_matches_oracle(emu, oc, k):
    pc.check_ntt(emu, oc, k)


def test_ntt_golden(emu, golden):
    pc.check_golden_ntt(emu, golden["ntt"])


def test_ntt_three_and_four_pass_plans(emu, oc, monkeypatch):
    # small B_MAX forces the 3- and 4-pass code paths at CPU-friendly sizes (fresh library instance: the
    # plan is read once per process)
    import os, subprocess, sys
    code = (
        "import sys; sys.path[:0]=[%r,%r,%r]\n"
        "import oracle_c as oc, parity_cases as pc\n"
        "from halo2_scaffold_b200._lib import Lib\n"
        "L=Lib(%r, allow_emulator=True); L.init(1)\n"
        "[pc.check_ntt(L, oc, k) for k in (12, 13, 14, 16)]\n"
        "print('ok')\n") % (pc.__file__.rsplit('/tests/', 1)[0], pc.__file__.rsplit('/tests/', 1)[0] + '/oracle',
                            pc.__file__.rsplit('/', 1)[0], emu.path)
    env = dict(os.environ, H2B_NTT_BMAX="4")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]
    # B_MAX = 5: passes of 3 to 5 stages
    env = dict(os.environ, H2B_NTT_BMAX="5")
    out = subprocess.run([sys.executable, "-c", code.replace("(12, 13, 14, 16)", "(11, 13, 15, 16)")], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]
    # one CTA holding a full 2^11 / 2^12 tile (the tile size of the two-pass plan at 2^22..2^24)
    env = dict(os.environ, H2B_NTT_SINGLE="12")
    out = subprocess.run([sys.executable, "-c", code.replace("(12, 13, 14, 16)", "(11, 12)")], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.parametrize("n", [1, 2, 3, 5, 32, 33, 100, 1000])
def test_msm_matches_oracle(emu, oc, n):
    pc.check_msm(emu, oc, n, kind=0, windows=(0,) if n < 100 else (0, 3, 6))


def test_msm_witness_like_scalars_split_buckets(emu, oc):
    # 50% zero / 20% one / small / small negatives: exercises bucket splitting + warp combine
    pc.check_msm(emu, oc, 3000, kind=1, windows=(0, 5, 10, 12))


def test_msm_golden(emu, oc, golden):
    pc.check_golden_msm(emu, oc, golden["msm"])


def test_msm_registered_prefix_and_offset(emu, oc):
    n = 600
    s, P = oc.random_fr(5, n), oc.gen_points(6, n)
    h = emu.register_bases(P)
    try:
        for off, m in ((0, n), (0, 100), (37, 400)):
            got = pc.affine_of(oc, emu.msm_registered(s[:m], h, off))
            want = pc.affine_of(oc, oc.best_multiexp(s[:m], P[off:off + m]))
            assert (got == want).all()
    finally:
        emu.unregister_bases(h)
    with pytest.raises(Exception):
        emu.msm_registered(s, h, 0)


def test_msm_empty_and_identity(emu, oc):
    out = emu.msm(np.zeros((0, 4), dtype=np.uint64), np.zeros((0, 8), dtype=np.uint64))
    assert (pc.affine_of(oc, out) == 0).all()
    s = oc.random_fr(1, 10)
    out = emu.msm(s, np.zeros((10, 8), dtype=np.uint64))      # all bases are the identity
    assert (pc.affine_of(oc, out) == 0).all()
    out = emu.msm(np.zeros((10, 4), dtype=np.uint64), oc.gen_points(2, 10))   # all scalars zero
    assert (pc.affine_of(oc, out) == 0).all()


def test_length_mismatch_asserts_like_the_reference(emu, oc):
    with pytest.raises(AssertionError):
        emu.msm(oc.random_fr(1, 4), oc.gen_points(1, 5))
    with pytest.raises(AssertionError):
        emu.ntt(np.zeros((3, 4), dtype=np.uint64), np.zeros(4, dtype=np.uint64), 2)


@pytest.mark.parametrize("n,spacing,windows", [(1, 4, (0,)), (3, 6, (0, 3)), (33, 8, (0, 4, 2)), (200, 0, (0,)), (1000, 12, (0, 6, 4, 3)), (700, 10, (0, 5))])
def test_msm_with_window_tables(emu, oc, n, spacing, windows):
    pc.check_msm_tables(emu, oc, n, spacing, windows=windows, ranges=[(0, n), (n // 3, n - n // 3), (n - 1, 1)])


def test_msm_with_window_tables_witness_like(emu, oc):
    # skewed scalars: one bucket holds a large share of the sorted list -> slices cut it into many pieces (heavy combine)
    pc.check_msm_tables(emu, oc, 4000, 8, kind=1, windows=(0, 8))


def test_implicit_base_cache_builds_tables_on_second_use_and_follows_reloaded_srs(emu, oc):
    n = 300
    s, P = pc.edge_msm_inputs(emu, oc, n, 0, 77)
    want = pc.affine_of(oc, oc.best_multiexp(s, P))
    for _ in range(3):      # 1st call: plain upload, 2nd: tables are built, 3rd: tables reused
        assert (pc.affine_of(oc, emu.msm(s, P)) == want).all()
    P2 = P.copy()           # the same SRS vector at a new address (scaffold.rs:174 re-reads the params file per proof)
    assert (pc.affine_of(oc, emu.msm(s, P2)) == want).all()
    P2[0] = P2[11]          # ... and a different vector at that same address (a sampled point differs) must not hit the cache
    want2 = pc.affine_of(oc, oc.best_multiexp(s, P2))
    assert (pc.affine_of(oc, emu.msm(s, P2)) == want2).all()


@pytest.mark.parametrize("tables", [False, True])
def test_msm_one_bucket_holds_everything(emu, oc, tables):
    pc.check_msm_single_bucket(emu, oc, 40000, scalar=1, tables=tables)


def test_cpp_host_mirror_over_the_c_abi(emu, oc, tmp_path):
    # halo2_scaffold_b200/host/h2b200.hpp (best_multiexp / best_fft / EvaluationDomain / ParamsKZG in C++) linked against
    # the emulator build of the same C ABI; the GPU suite repeats this against libh2b200.so
    from host_mirror_case import run_host_mirror
    run_host_mirror(oc, emu.path, tmp_path, k=6, j=4)


def test_msm_chunked_upload_pipeline(emu):
    # host-pointer MSMs cut into upload chunks that are accumulated into the same buckets (fresh process: the chunk
    # size is read once); plain and table mode, uniform and witness-like scalars, ragged last chunk
    import os, subprocess, sys
    root = pc.__file__.rsplit('/tests/', 1)[0]
    code = (
        "import sys; sys.path[:0]=[%r,%r,%r]\n"
        "import oracle_c as oc, parity_cases as pc\n"
        "from halo2_scaffold_b200._lib import Lib\n"
        "L=Lib(%r, allow_emulator=True); L.init(1)\n"
        "pc.check_msm(L, oc, 5000, kind=0, windows=(0, 7))\n"
        "pc.check_msm(L, oc, 4097, kind=1, windows=(0,))\n"
        "pc.check_msm_tables(L, oc, 5000, 8, kind=0, windows=(0, 4), ranges=[(0, 5000), (100, 4500)])\n"
        "pc.check_msm_tables(L, oc, 6000, 10, kind=1)\n"
        "pc.check_msm_single_bucket(L, oc, 9000, scalar=1, tables=True)\n"
        "print('ok')\n") % (root, root + '/oracle', root + '/tests', emu.path)
    env = dict(os.environ, H2B_MSM_UPLOAD_CHUNK_LOG="10")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]
    # the production schedule (1/16 + 3 x 5/16) at a CPU-test size
    env = dict(os.environ, H2B_MSM_UPLOAD_MIN_LOG="10")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]
    # device-resident scalars: 4 (or 3) chunks accumulated into the same buckets
    code2 = (
        "import sys; sys.path[:0]=[%r,%r,%r]\n"
        "import numpy as np, oracle_c as oc, parity_cases as pc\n"
        "from halo2_scaffold_b200._lib import Lib\n"
        "L=Lib(%r, allow_emulator=True); L.init(1)\n"
        "for n, kind, chunks in ((5000, 0, 4), (4099, 1, 3)):\n"
        "    s, P = pc.edge_msm_inputs(L, oc, n, kind, 900 + n)\n"
        "    want = pc.affine_of(oc, oc.best_multiexp(s, P))\n"
        "    h = L.register_bases(P)\n"
        "    d_s, d_p, d_o = L.dev_alloc(0, n * 32), L.dev_alloc(0, n * 64), L.dev_alloc(0, 224)\n"
        "    L.h2d(0, d_s, s); L.h2d(0, d_p, P)\n"
        "    out = np.zeros(28, dtype=np.uint64)\n"
        "    L.msm_dev_registered(0, d_s, h, 0, n, d_o); L.dev_sync(0); L.d2h(0, out, d_o)\n"
        "    assert (pc.affine_of(oc, out[:12]) == want).all()\n"
        "    L.msm_dev_partial(0, d_s, d_p, n, d_o); L.dev_sync(0); L.d2h(0, out, d_o)\n"
        "    assert (pc.affine_of(oc, out[:12]) == want).all()\n"
        "print('ok')\n") % (root, root + '/oracle', root + '/tests', emu.path)
    env = dict(os.environ, H2B_MSM_DEVICE_CHUNK_MIN_LOG="10", H2B_MSM_DEVICE_CHUNKS="4")
    out = subprocess.run([sys.executable, "-c", code2], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_batched_columns_match_single_calls(emu, oc):
    n = 600
    P = oc.gen_points(71, n)
    cols = [oc.random_fr(80 + j, n - 37 * j) for j in range(5)] + [np.zeros((0, 4), dtype=np.uint64)]
    h = emu.register_bases(P)
    try:
        got = emu.msm_batch_registered(cols, h)
        for j, c in enumerate(cols):
            assert (pc.affine_of(oc, got[j]) == pc.affine_of(oc, oc.best_multiexp(c, P[:c.shape[0]]))).all(), j
    finally:
        emu.unregister_bases(h)
    k = 9
    polys = [oc.random_fr(90 + j, 1 << k) for j in range(4)]
    want = [oc.best_fft(a, pc.omega_words(oc, k), k) for a in polys]
    emu.ntt_batch(polys, pc.omega_words(oc, k), k)
    for a, w in zip(polys, want):
        assert (a == w).all()


def test_pageable_host_buffers_go_through_the_pinned_staging_threads(emu):
    # stage.cu: host threads copy pieces of the caller's (pageable) buffers through pinned slots, both directions;
    # tiny pieces force many pieces per worker and the slot recycling at CPU-test sizes
    import os, subprocess, sys
    root = pc.__file__.rsplit('/tests/', 1)[0]
    code = (
        "import sys; sys.path[:0]=[%r,%r,%r]\n"
        "import oracle_c as oc, parity_cases as pc\n"
        "from halo2_scaffold_b200._lib import Lib\n"
        "L=Lib(%r, allow_emulator=True); L.init(1)\n"
        "[pc.check_ntt(L, oc, k) for k in (7, 10, 12)]\n"
        "pc.check_msm(L, oc, 5000, kind=0)\n"
        "pc.check_msm_tables(L, oc, 3000, 8, kind=1, ranges=[(0, 3000), (17, 2500)])\n"
        "print('ok')\n") % (root, root + '/oracle', root + '/tests', emu.path)
    for threads in ("1", "3"):
        env = dict(os.environ, H2B_STAGE_PIECE_LOG="10", H2B_STAGE_THREADS=threads, H2B_MSM_UPLOAD_CHUNK_LOG="11")
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_evaluation_domain_mirror_matches_golden(emu, golden):
    # halo2_scaffold_b200.EvaluationDomain over the h2b_*_dev domain entry points (row a6) against the fixture that
    # tests/golden/make_golden.py produced with the big-int oracle
    import halo2_scaffold_b200 as h2
    g = golden["domain"]
    d = h2.EvaluationDomain(int(g["j"]), int(g["k"]), lib=emu)
    coeff = d.lagrange_to_coeff(g["lagrange"])
    assert (coeff == g["coeff"]).all()
    ext = d.coeff_to_extended(coeff)
    assert (ext == g["extended"]).all()
    assert (d.extended_to_coeff(ext) == g["back"]).all()


def test_msm_randomised_shapes(emu, oc):
    pc.check_msm_random(emu, oc, examples=30, max_n=400, spacings=(-1, 4, 6, 8, 10, 12), windows=(0, 0, 2, 3, 4, 5, 6))


def test_ntt_randomised_inputs(emu, oc):
    """NTT against the oracle for random sizes and structured inputs (zeros, a single spike, all-equal, r-1 everywhere)."""
    rng = np.random.default_rng(5)
    one = oc.fr_to_mont(np.array([[1, 0, 0, 0]], dtype=np.uint64))[0]
    minus_one = oc.field_op("fr", "sub", np.zeros((1, 4), dtype=np.uint64), one.reshape(1, 4))[0]
    for k in (1, 2, 4, 6, 9, 11, 13):
        n = 1 << k
        cases = [np.zeros((n, 4), dtype=np.uint64), np.repeat(minus_one.reshape(1, 4), n, axis=0), oc.random_fr(int(rng.integers(1 << 30)), n)]
        spike = np.zeros((n, 4), dtype=np.uint64)
        spike[int(rng.integers(0, n))] = one
        cases.append(spike)
        for a in cases:
            for inverse in (False, True):
                w = pc.omega_words(oc, k, inverse)
                assert (emu.ntt(a.copy(), w, k) == oc.best_fft(a, w, k)).all(), (k, inverse)


def test_grand_product_building_blocks(emu, oc):
    pc.check_grand_product_blocks(emu, oc, [1, 2, 3, 15, 16, 17, 100, 1023, 1024, 1025, 5000, 20000])


def test_polynomial_evaluation_and_kate_division(emu, oc):
    pc.check_poly_eval_and_division(emu, oc, [1, 2, 3, 15, 16, 17, 255, 256, 257, 4095, 4096, 4097, 70000])


def test_evaluate_graph_random_programs(emu, oc):
    # every Calculation / ValueSource variant, dead code, re-used targets, ragged sizes, negative and large rotations
    cases = [(1, 1, 1, 1), (2, 1, 5, 2), (37, 1, 12, 3), (64, 4, 30, 4), (200, 2, 60, 5), (256, 4, 120, 6), (100, 7, 250, 7), (513, 3, 40, 8),
             (300, 1, 400, 9), (128, 16, 25, 10), (99, 1, 80, 11)]
    pc.check_evaluate_graph(emu, oc, cases)
    slots, ops = emu.evaluate_graph_info()
    assert ops > 0


def test_evaluate_graph_edge_cases(emu, oc):
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200._lib import GraphArrays, H2BError
    size = 40
    adv = [oc.random_fr(5, size)]
    sc = oc.random_fr(6, 4)
    vals = oc.random_fr(7, size)
    none = np.zeros((0, 4), dtype=np.uint64)

    def run(calcs, parts=(), n_inter=4, rotations=(0,)):
        g = (oc.random_fr(8, 3), np.array(rotations, dtype=np.int32), np.array(calcs, dtype=np.uint32).reshape(-1, 10),
             np.array(parts, dtype=np.uint32).reshape(-1, 3), n_inter)
        want = oc.evaluate_graph(g, [], adv, [], none, *sc, vals, 1)
        got = ev.evaluate_graph(emu, GraphArrays(*g), [], adv, [], none, *sc, vals, 1)
        assert (got == want).all()
        return got
    # no calculations: zero, as upstream
    assert not run([], n_inter=0).any()
    # the result is a Store of a column / of the previous value / of an intermediate
    run([[7, 0, 3, 0, 0, 0, 0, 0, 0, 0]])
    assert (run([[7, 0, 10, 0, 0, 0, 0, 0, 0, 0]]) == vals).all()
    run([[2, 0, 3, 0, 0, 10, 0, 0, 0, 0], [7, 1, 1, 0, 0, 0, 0, 0, 0, 0]])
    # Horner without parts is its start value; Horner whose parts repeat one intermediate
    run([[6, 0, 9, 0, 0, 8, 0, 0, 0, 0]])
    run([[3, 0, 3, 0, 0, 0, 0, 0, 0, 0], [6, 1, 10, 0, 0, 9, 0, 0, 0, 3]], parts=[[1, 0, 0], [1, 0, 0], [3, 0, 0]])
    # malformed graphs are refused, not executed
    for bad in ([[0, 0, 1, 2, 0, 0, 0, 0, 0, 0]],          # reads an intermediate that was never written
                [[0, 9, 0, 0, 0, 0, 0, 0, 0, 0]],          # target out of range
                [[0, 0, 3, 5, 0, 0, 0, 0, 0, 0]],          # advice column out of range
                [[0, 0, 3, 0, 4, 0, 0, 0, 0, 0]],          # rotation out of range
                [[6, 0, 0, 0, 0, 0, 0, 0, 0, 2]],          # Horner parts out of range
                [[9, 0, 0, 0, 0, 0, 0, 0, 0, 0]]):         # unknown op
        g = GraphArrays(oc.random_fr(8, 3), np.array([0], dtype=np.int32), np.array(bad, dtype=np.uint32), np.zeros((0, 3), dtype=np.uint32), 4)
        with pytest.raises(H2BError):
            ev.evaluate_graph(emu, g, [], adv, [], none, *sc, vals, 1)


def test_evaluate_graph_many_live_values(emu, oc):
    # 6 / 12 / 24 / 48 values live at once select the 8 / 16 / 32 / 64-slot kernels; more than 64 is refused
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200._lib import H2BError
    size = 33
    adv = [oc.random_fr(5, size)]
    sc = oc.random_fr(6, 4)
    vals = oc.random_fr(7, size)
    none = np.zeros((0, 4), dtype=np.uint64)
    for n_live in (6, 12, 24, 48):
        graph, n_const = pc.wide_graph(n_live)
        g, ga = pc._graph_pair(oc, graph, n_const, n_live)
        want = oc.evaluate_graph(g, [], adv, [], none, *sc, vals, 1)
        got = ev.evaluate_graph(emu, ga, [], adv, [], none, *sc, vals, 1)
        assert (got == want).all(), n_live
        slots, ops = emu.evaluate_graph_info()
        assert n_live <= slots <= n_live + 2, (n_live, slots)
    graph, n_const = pc.wide_graph(70)
    with pytest.raises(H2BError):
        ev.evaluate_graph(emu, pc._graph_pair(oc, graph, n_const, 1)[1], [], adv, [], none, *sc, vals, 1)


def test_evaluate_graph_scheduling_keeps_few_values_live(emu, oc):
    # 40 gate polynomials combined by one Horner in y: upstream keeps one intermediate per gate; the depth-first schedule
    # needs a handful of slots
    from halo2_scaffold_b200 import evaluation as ev
    polys, lookups, nf, na = pc.standard_plonk_like(20)
    E = ev.Evaluator(polys, lookups)
    size = 64
    fixed = [oc.random_fr(100 + j, size) for j in range(nf)]
    advice = [oc.random_fr(300 + j, size) for j in range(na)]
    inst = [oc.random_fr(500, size)]
    sc = oc.random_fr(6, 4)
    none = np.zeros((0, 4), dtype=np.uint64)
    a = E.custom_gates.arrays()
    got = ev.evaluate_graph(emu, a, fixed, advice, inst, none, *sc, np.zeros((size, 4), dtype=np.uint64), 4)
    want = oc.evaluate_graph((a.constants, a.rotations, a.calculations, a.parts, a.n_intermediates), fixed, advice, inst, none, *sc,
                             np.zeros((size, 4), dtype=np.uint64), 4)
    assert (got == want).all()
    slots, ops = emu.evaluate_graph_info()
    assert E.custom_gates.num_intermediates > 300 and slots <= 8, (E.custom_gates.num_intermediates, slots, ops)


def test_evaluate_h_all_three_loops(emu, oc):
    pc.check_evaluate_h(emu, oc, [(5, 3, 1, 1), (7, 5, 2, 2), (6, 6, 1, 3)])


def test_g1_point_codec(emu, oc):
    for n in (1, 2, 33, 300):
        pc.check_g1_codec(emu, oc, n)


def test_srs_file_round_trip(emu, oc, tmp_path):
    pc.check_srs_file_round_trip(emu, oc, tmp_path, 4)
    pc.check_srs_file_round_trip(emu, oc, tmp_path, 7)


def test_srs_reader_rejects_bad_files(emu, oc, tmp_path):
    from halo2_scaffold_b200._lib import H2BError
    p = tmp_path / "short.srs"
    for content in (b"", (3).to_bytes(4, "little") + bytes(100), (40).to_bytes(4, "little"), (2).to_bytes(4, "little") + bytes(2 * 4 * 64 + 10)):
        p.write_bytes(content)
        with pytest.raises(H2BError):
            emu.srs_read(str(p), 1)
    with pytest.raises((H2BError, FileNotFoundError)):
        emu.srs_read(str(tmp_path / "missing.srs"), 1)


def test_srs_reader_keeps_decoded_files_resident(emu, oc, tmp_path):
    # the reference re-reads the params file for every proof (src/scaffold.rs:174): an unchanged file is not decoded twice
    import os
    k, n = 5, 32
    g, gl = oc.gen_points(41, n), oc.gen_points(42, n)
    path = str(tmp_path / "kzg_bn254_5.srs")
    emu.srs_write(path, 0, k, g, gl, bytes(128))
    launches = emu.launch_count()
    a = emu.srs_read(path, 0)
    first = emu.launch_count() - launches
    b = emu.srs_read(path, 0)
    assert emu.launch_count() - launches == first, "the second read decoded again"
    assert (a["handle_g"], a["handle_g_lagrange"]) == (b["handle_g"], b["handle_g_lagrange"])
    assert (b["g"] == g).all() and (b["g_lagrange"] == gl).all() and b["g2_bytes"] == bytes(128)
    s = oc.random_fr(43, n)
    want = pc.affine_of(oc, oc.best_multiexp(s, g))
    # every reader gives its handles back; the sets stay usable until the last one (and the cache) let go
    emu.unregister_bases(a["handle_g"]); emu.unregister_bases(a["handle_g_lagrange"])
    assert (pc.affine_of(oc, emu.msm_registered(s, b["handle_g"], 0)) == want).all()
    emu.unregister_bases(b["handle_g"]); emu.unregister_bases(b["handle_g_lagrange"])
    c = emu.srs_read(path, 0, want_host=False)
    assert c["handle_g"] == a["handle_g"]
    emu.unregister_bases(c["handle_g"]); emu.unregister_bases(c["handle_g_lagrange"])
    # a rewritten file is decoded afresh
    emu.srs_write(path, 0, k, gl, g, bytes(128))
    os.utime(path, ns=(1, 1))
    d = emu.srs_read(path, 0)
    assert d["handle_g"] != a["handle_g"] and (d["g"] == gl).all()
    emu.unregister_bases(d["handle_g"]); emu.unregister_bases(d["handle_g_lagrange"])
    emu.srs_cache_clear()
    from halo2_scaffold_b200._lib import H2BError
    with pytest.raises(H2BError):
        emu.msm_registered(s, d["handle_g"], 0)


def test_divide_by_vanishing_poly(emu, oc):
    pc.check_vanishing_division(emu, oc, [(3, 3), (4, 4), (5, 5), (9, 4), (10, 3), (18, 2)])


def test_permutation_and_lookup_grand_products(emu, oc):
    pc.check_grand_products(emu, oc, [1, 2, 8, 64, 100, 1024, 5000])


def test_linear_combination_of_columns(emu, oc):
    pc.check_lincomb(emu, oc, [(1, 1), (7, 3), (200, 32), (130, 33), (64, 70)])


def test_lookup_permute_async_status(emu, oc):
    pc.check_lookup_permute_async(emu, oc)


def test_lookup_permute_expression_pair(emu, oc):
    pc.check_lookup_permute(emu, oc, [(8, 8, 3, "random", 1), (64, 58, 10, "random", 2), (1024, 1018, 1000, "random", 3), (1024, 1018, 16, "small", 4),
                                      (2048, 2042, 700, "skewed", 5), (3000, 2994, 256, "small", 6), (4096, 4090, 5000, "random", 7), (16, 0, 4, "random", 8),
                                      (1 << 14, (1 << 14) - 6, 3000, "random", 9), (8192 + 77, 8192 + 71, 64, "small", 10)])


def test_prover_rows_golden(emu, golden):
    pc.check_golden_prover(emu, golden["prover"])


def test_evaluate_graph_property(emu, oc):
    pc.check_evaluate_graph_property(emu, oc, examples=80, max_rows=70, max_calcs=160)


def test_msm_duplicate_identity_and_opposite_points(emu, oc, golden):
    # golden vectors (identity bases, duplicate points, P and -P in one bucket), random shapes with forced windows and table
    # spacings, and witness-like columns
    pc.check_golden_msm(emu, oc, golden["msm"])
    pc.check_msm_random(emu, oc, examples=8, max_n=600, spacings=(-1, 4, 6, 8), windows=(0, 2, 3, 4, 6))
    for n, kind in ((3000, 1), (2500, 0)):
        pc.check_msm_opposite_points(emu, oc, n, kind)


def test_quotient_of_a_satisfied_circuit_is_a_polynomial(emu, oc):
    ok, h = pc.check_quotient_is_a_polynomial(emu, oc, k=4, seed=1)
    assert ok and h.any()
    assert pc.check_quotient_is_a_polynomial(emu, oc, k=5, seed=2)[0]
    # and the property is sharp: an unsatisfied gate, a wrong sigma column or a disturbed fill order all break it
    for what in ("witness", "sigma", "fill"):
        assert not pc.check_quotient_is_a_polynomial(emu, oc, k=4, seed=3, break_it=what)[0], what


def test_evaluate_h_row_shards(emu, oc):
    pc.check_evaluate_h_sharded(emu, oc)


def test_argument_prover_mirrors_commit(emu, oc):
    # permutation::Argument::commit / lookup commit_permuted + commit_product through halo2_scaffold_b200.prover with a ParamsKZG:
    # the commitments are commit_lagrange of exactly the columns that are returned
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import prover
    from halo2_scaffold_b200.domain import fr_to_words
    k, n, bf = 5, 32, 5
    params = h2.ParamsKZG(k, oc.gen_points(61, n), oc.gen_points(62, n), lib=emu)
    try:
        cols = [oc.random_fr(70 + j, n) for j in range(3)]
        sig = [oc.random_fr(80 + j, n) for j in range(3)]
        beta, gamma = oc.random_fr(90, 2)
        blind = lambda count: oc.random_fr(91 + count, count)
        zs, coms = prover.permutation_commit(cols, sig, chunk_len=2, blinding_factors=bf, beta=beta, gamma=gamma, omega=pc.omega_words(oc, k), blind=blind,
                                             params=params, lib=emu)
        assert len(zs) == 2 and (zs[1][0] == zs[0][n - bf - 1]).all()
        for z, c in zip(zs, coms):
            assert (z[n - bf:] == blind(bf)).all()
            assert (pc.affine_of(oc, c) == pc.affine_of(oc, oc.best_multiexp(z, params.g_lagrange))).all()
        table = oc.random_fr(95, n)
        inp = table[: n - bf - 1][np.random.default_rng(3).integers(0, n - bf - 1, size=n)]
        pa, pt, (ca, ct) = prover.lookup_commit_permuted(inp, table, blinding_factors=bf, blind=blind, params=params, lib=emu)
        assert pa.shape == (n, 4) and (pa[n - bf - 1:] == blind(bf + 1)).all()
        assert (pc.affine_of(oc, ca) == pc.affine_of(oc, oc.best_multiexp(pa, params.g_lagrange))).all()
        z, cz = prover.lookup_commit_product(inp, table, pa, pt, blinding_factors=bf, beta=beta, gamma=gamma, blind=blind, params=params, lib=emu)
        assert (z[0] == fr_to_words(1)).all() and (z[n - bf - 1] == fr_to_words(1)).all()          # the product closes on the last usable row
        assert (pc.affine_of(oc, cz) == pc.affine_of(oc, oc.best_multiexp(z, params.g_lagrange))).all()
    finally:
        params.close()


def test_lookup_compress_expressions(emu, oc):
    # theta-compression of lookup expressions over the Lagrange rows against field arithmetic of the oracle (rotation wraps inside n)
    from halo2_scaffold_b200 import evaluation as ev, prover
    n = 50
    adv = [oc.random_fr(31 + j, n) for j in range(2)]
    fix = [oc.random_fr(41, n)]
    theta = oc.random_fr(51, 1)[0]
    exprs = [ev.Product(ev.Fixed(0), ev.Advice(0)), ev.Advice(1, 1), ev.Sum(ev.Advice(0, -1), ev.Constant(5))]
    got = prover.lookup_compress_expressions(exprs, fixed=fix, advice=adv, instance=[], challenges=np.zeros((0, 4), dtype=np.uint64), theta=theta, lib=emu)
    mul = lambda a, b: oc.field_op("fr", "mul", a, b)
    add = lambda a, b: oc.field_op("fr", "add", a, b)
    five = np.repeat(oc.fr_to_mont(np.array([[5, 0, 0, 0]], dtype=np.uint64)), n, axis=0)
    th = np.repeat(theta.reshape(1, 4), n, axis=0)
    e0, e1, e2 = mul(fix[0], adv[0]), np.roll(adv[1], -1, axis=0), add(np.roll(adv[0], 1, axis=0), five)
    want = add(mul(add(mul(e0, th), e1), th), e2)
    assert (got == want).all()


def test_implicit_cache_is_content_addressed(emu):
    # digest blocks of 16 points, arrays from 64 points on are cached: the logic of the 1024 / 4096 production values at CPU sizes
    run_on_emulated_devices(None, "pc.check_implicit_cache_is_content_addressed(L, oc, 320, 16)\n"
                                  "pc.check_implicit_cache_under_threads(L, oc, 256, threads=8, rounds=2)", None,
                            dict(H2B_DIGEST_BLOCK_LOG="4", H2B_IMPLICIT_MIN_LOG="6"), timeout=900)


def test_implicit_cache_can_be_disabled(emu):
    run_on_emulated_devices(None, "s, P = oc.random_fr(1, 256), oc.gen_points(2, 256)\n"
                                  "w = pc.affine_of(oc, oc.best_multiexp(s, P))\n"
                                  "assert all((pc.affine_of(oc, L.msm(s, P)) == w).all() for _ in range(2))\n"
                                  "st = L.implicit_cache_stats(); assert st['uploads'] == 0 and st['direct'] == 2, st", None,
                            dict(H2B_DIGEST_BLOCK_LOG="4", H2B_IMPLICIT_MIN_LOG="6", H2B_IMPLICIT_CACHE="0"), timeout=900)


@pytest.mark.parametrize("devices", ["2", "3"])
def test_multi_device_host_logic_on_emulated_devices(emu, devices):
    # the emulator reports several devices, so point-range sharding, sharded base sets (tables per slice),
    # the table all-gather of replicated sets, round-robin + batched columns and the implicit cache's sharded copies all run here
    run_on_emulated_devices(None, "pc.check_sharded_base_set(L, oc, 700, spacing=8)\n"
                                  "pc.check_sharded_base_set(L, oc, 333, spacing=0, kind=1)\n"
                                  "pc.check_msm_tables(L, oc, 600, 8, kind=0, ranges=[(0, 600), (100, 450)])\n"
                                  "pc.check_msm(L, oc, 500, kind=1)\n"
                                  "pc.check_implicit_cache_is_content_addressed(L, oc, 320, 16)\n"
                                  "pc.check_batched_columns(L, oc, 300, 7, spacing=8)", devices,
                            dict(H2B_MULTI_DEVICE_MIN_LOG="7", H2B_DIGEST_BLOCK_LOG="4", H2B_IMPLICIT_MIN_LOG="6"), timeout=900)


def test_fr_transpose(emu, oc):
    pc.check_fr_transpose(emu, oc, shapes=((32, 32), (64, 96), (1, 5), (33, 70), (96, 1)))


@pytest.mark.parametrize("devices", ["2", "4"])
def test_one_ntt_across_emulated_devices(emu, devices):
    # SURVEY.md 8e "one NTT across GPUs": the four-step split of h2b_ntt_bn254_fr (strided uploads of column blocks, transposes,
    # strided-batch transforms, twiddles, 2-D peer copies, strided downloads) against best_fft, both directions, odd and even log_n,
    # pageable host arrays through the staging threads with 1 KiB pieces (several rows per piece, several pieces per thread)
    run_on_emulated_devices(None, "for k in (4, 5, 8, 11, 12, 13):\n"
                                  "    pc.check_ntt(L, oc, k)\n", devices,
                            dict(H2B_NTT_MULTI_MIN_LOG="4", H2B_STAGE_PIECE_LOG="10", H2B_STAGE_THREADS="3"), timeout=900)
    # the strided-batch mode of the multi-pass plans (2, 3 and 4 passes per row / column transform)
    run_on_emulated_devices(None, "for k in (12, 14, 15):\n"
                                  "    pc.check_ntt(L, oc, k)\n", devices,
                            dict(H2B_NTT_MULTI_MIN_LOG="4", H2B_NTT_BMAX="2"), timeout=900)


@pytest.mark.parametrize("n,ncols,spacing,window", [(600, 6, 8, 0), (600, 5, 8, 4), (257, 9, 0, 0), (1200, 4, 12, 6), (40, 33, 6, 0), (300, 4, -1, 0)])
def test_batched_columns_one_kernel_sequence(emu, oc, n, ncols, spacing, window):
    pc.check_batched_columns(emu, oc, n, ncols, spacing=spacing, window=window)


@pytest.mark.parametrize("k,count", [(3, 5), (9, 4), (11, 3), (12, 17), (13, 2)])
def test_batched_ntts_share_pass_launches(emu, oc, k, count):
    pc.check_batched_ntts(emu, oc, k, count)


@pytest.mark.parametrize("shape,batched", [(dict(k=5, A=1, LK=0, d=3), True), (dict(k=6, A=2, LK=1, d=4), True), (dict(k=6, A=3, LK=2, d=4), False)])
def test_device_resident_proof_pipeline_matches_oracle_pipeline(emu, oc, shape, batched):
    # tools/proof_pipeline_core.py (every column resident on the device, batched phase calls) against the same flow recomputed with
    # the CPU oracle: every commitment and every evaluation (VERDICT r1 item 7)
    import pipeline_oracle
    counts = pipeline_oracle.check_pipeline(emu, oc, shape, batched=batched)
    assert counts["msm"] >= 7 and counts["eval"] >= 10


@pytest.mark.parametrize("j,k", [(3, 5), (4, 9), (5, 7)])
def test_column_pipeline_single_upload(emu, oc, j, k):
    pc.check_column_pipeline(emu, oc, j, k)


def test_msm_partitioned_sort(emu):
    # section 2c of msm.cu (two-level sort: partition histogram in shared memory, contiguous runs per partition, chunked placement
    # with shared-memory cursors) forced at CPU sizes -- it needs W <= 16 windows, i.e. 16-bit windows or wider: uniform /
    # witness-like / one-bucket columns (hot partitions), table and plain mode, ragged batches, chunked uploads, tiny chunks
    run_on_emulated_devices(None, "pc.check_msm_tables(L, oc, 3000, 16, kind=0, windows=(16,), ranges=[(0, 3000), (100, 2500)])\n"
                                  "pc.check_msm_tables(L, oc, 2500, 16, kind=1, windows=(16,))\n"
                                  "pc.check_msm_tables(L, oc, 1500, 18, kind=0, windows=(18,))\n"
                                  "pc.check_msm_single_bucket(L, oc, 20000, scalar=1, tables=True)\n"
                                  "pc.check_batched_columns(L, oc, 300, 3, spacing=16, window=16)", None,
                            dict(H2B_MSM_SORT2_MIN_LOG="8", H2B_MSM_SORT2_CHUNK_LOG="7", H2B_MSM_PRECOMP="16"), timeout=2400)
    run_on_emulated_devices(None, "pc.check_msm_tables(L, oc, 4097, 16, kind=1, windows=(16,), ranges=[(0, 4097)])", None,
                            dict(H2B_MSM_SORT2_MIN_LOG="8", H2B_MSM_UPLOAD_CHUNK_LOG="10"), timeout=2400)
    # the bucket scan of a partition in several passes of blockDim buckets (the 4096-bucket partitions of 22-bit tables)
    run_on_emulated_devices(None, "pc.check_msm_tables(L, oc, 3000, 16, kind=0, windows=(16,), ranges=[(0, 3000), (100, 2500)])\n"
                                  "pc.check_msm_tables(L, oc, 2500, 18, kind=1, windows=(18,))", None,
                            dict(H2B_MSM_SORT2_MIN_LOG="8", H2B_MSM_SORT2_CHUNK_LOG="7", H2B_MSM_PLACE_SCAN_THREADS="32"), timeout=2400)
