"""
GPU (B200): the product path through the C ABI (libh2b200.so) against the oracle, the golden fixtures, and -- at the
benchmark's full sizes -- size-independent properties.  Bit-exact everywhere: all arithmetic is integer.
"""
import os

import numpy as np
import pytest

import bn254 as o
import parity_cases as pc

pytestmark = pytest.mark.gpu


def test_library_is_the_cuda_build(gpu):
    assert "sm_100a" in gpu.version() and not gpu.is_emulator
    import torch
    assert gpu.device_count() == torch.cuda.device_count() >= 1      # every visible device is in use


def test_field_arithmetic(gpu, oc):
    pc.check_field(gpu, oc, 1 << 14)


def test_group_law_edge_cases(gpu, oc):
    pc.check_group(gpu, oc, 256)


def test_generators_match_oracle_streams(gpu, oc):
    assert (gpu.gen_points(7, 5000) == oc.gen_points(7, 5000)).all()
    assert (gpu.gen_scalars(11, 5000, 0) == oc.random_fr(11, 5000)).all()


def test_golden_vectors(gpu, oc, golden):
    pc.check_golden_ntt(gpu, golden["ntt"])
    pc.check_golden_msm(gpu, oc, golden["msm"])


@pytest.mark.parametrize("k", list(range(1, 21)) + [22])
def test_ntt_matches_oracle(gpu, oc, k):
    pc.check_ntt(gpu, oc, k)


@pytest.mark.parametrize("n,kind", [(1, 0), (2, 0), (3, 0), (31, 0), (32, 0), (33, 0), (1000, 0), (4096, 1), (1 << 14, 0), (1 << 16, 0),
                                    (1 << 16, 1), ((1 << 17) + 12345, 0), (1 << 18, 0), (1 << 18, 1), (1 << 20, 0)])
def test_msm_matches_oracle(gpu, oc, n, kind):
    windows = (0,) if n < 1000 else ((0, 8, 13) if n <= (1 << 18) else (0,))
    pc.check_msm(gpu, oc, n, kind=kind, windows=windows)


def test_msm_empty_identity_and_cancellation(gpu, oc):
    out = gpu.msm(np.zeros((0, 4), dtype=np.uint64), np.zeros((0, 8), dtype=np.uint64))
    assert (pc.affine_of(oc, out) == 0).all()
    s = oc.random_fr(1, 1000)
    assert (pc.affine_of(oc, gpu.msm(s, np.zeros((1000, 8), dtype=np.uint64))) == 0).all()
    assert (pc.affine_of(oc, gpu.msm(np.zeros((1000, 4), dtype=np.uint64), oc.gen_points(2, 1000))) == 0).all()
    # every scalar equal and every base equal: one bucket holds everything (P + P ... doubling branch, split buckets)
    P = np.repeat(oc.gen_points(3, 1), 5000, axis=0)
    one = oc.fr_to_mont(np.array([[1, 0, 0, 0]], dtype=np.uint64))
    s1 = np.repeat(one, 5000, axis=0)
    want = pc.affine_of(oc, oc.best_multiexp(s1, P))
    assert (pc.affine_of(oc, gpu.msm(s1, P)) == want).all()


def test_msm_implicit_cache_prefix_and_pointer_reuse(gpu, oc):
    n = 1 << 12
    s, P = oc.random_fr(21, n), oc.gen_points(22, n)
    want = pc.affine_of(oc, oc.best_multiexp(s, P))
    assert (pc.affine_of(oc, gpu.msm(s, P)) == want).all()
    assert (pc.affine_of(oc, gpu.msm(s, P)) == want).all()            # second call hits the device-resident copy
    m = 1000                                                              # commit(poly) with len < n: prefix of the same array
    assert (pc.affine_of(oc, gpu.msm(s[:m], P[:m])) == pc.affine_of(oc, oc.best_multiexp(s[:m], P[:m]))).all()
    P[0] = oc.gen_points(99, 1)[0]                                        # same address, new contents (SRS reloaded)
    assert (pc.affine_of(oc, gpu.msm(s, P)) == pc.affine_of(oc, oc.best_multiexp(s, P))).all()


def test_implicit_cache_is_content_addressed(gpu, oc):
    """ADVICE r1 (high): no stale MSM after an in-place edit of any row, at the production thresholds (4096 points, 64 KiB blocks)."""
    pc.check_implicit_cache_is_content_addressed(gpu, oc, 1 << 13, 1024)


def test_implicit_cache_under_concurrent_callers(gpu, oc):
    """8 threads of verifier-sized MSMs over fresh arrays interleaved with 2^18-point commits: one upload of the large vector,
    no eviction, no use-after-free (create_proof followed by verify_proof, /root/reference/src/scaffold.rs:191-230)."""
    pc.check_implicit_cache_under_threads(gpu, oc, 1 << 18, threads=8, rounds=3)


def test_sharded_base_set(gpu, oc):
    pc.check_sharded_base_set(gpu, oc, (1 << 16) + 77, spacing=0)
    pc.check_sharded_base_set(gpu, oc, 1 << 18, spacing=16, kind=1)


@pytest.mark.parametrize("n,ncols,spacing,window", [(1 << 12, 8, 0, 0), (1 << 16, 8, 0, 0), (1 << 16, 5, 16, 8), ((1 << 14) + 5, 33, 8, 0),
                                                     (1 << 14, 4, -1, 0), (1 << 18, 6, 0, 0)])
def test_batched_columns_one_kernel_sequence(gpu, oc, n, ncols, spacing, window):
    pc.check_batched_columns(gpu, oc, n, ncols, spacing=spacing, window=window)


def test_registered_bases_ranges(gpu, oc):
    n = 3000
    s, P = oc.random_fr(5, n), oc.gen_points(6, n)
    h = gpu.register_bases(P)
    try:
        for off, m in ((0, n), (0, 100), (37, 2500)):
            got = pc.affine_of(oc, gpu.msm_registered(s[:m], h, off))
            assert (got == pc.affine_of(oc, oc.best_multiexp(s[:m], P[off:off + m]))).all()
        with pytest.raises(Exception):
            gpu.msm_registered(s, h, 1)
    finally:
        gpu.unregister_bases(h)
    with pytest.raises(Exception):
        gpu.msm_registered(s, h, 0)


@pytest.mark.parametrize("n,spacing,kind,windows", [(1, 4, 0, (0,)), (33, 8, 0, (0, 4)), (1000, 12, 0, (0, 6, 4)), (4096, 0, 1, (0,)),
                                                     (1 << 16, 0, 0, (0,)), (1 << 16, 16, 1, (0, 8)), ((1 << 18) + 777, 18, 0, (0, 9)),
                                                     (1 << 20, 0, 0, (0,)), (1 << 20, 20, 1, (0, 10))])
def test_msm_with_window_tables_matches_oracle(gpu, oc, n, spacing, kind, windows):
    pc.check_msm_tables(gpu, oc, n, spacing, kind=kind, windows=windows, ranges=[(0, n), (n // 3, n - n // 3)])


@pytest.mark.parametrize("n,scalar,tables", [(1 << 20, 1, True), (1 << 20, 3, False), (300000, 0xffff, True)])
def test_msm_one_bucket_holds_everything(gpu, oc, n, scalar, tables):
    pc.check_msm_single_bucket(gpu, oc, n, scalar=scalar, tables=tables)


def test_error_behaviour_matches_reference_asserts(gpu, oc):
    with pytest.raises(AssertionError):
        gpu.msm(oc.random_fr(1, 4), oc.gen_points(1, 5))
    with pytest.raises(AssertionError):
        gpu.ntt(np.zeros((3, 4), dtype=np.uint64), np.zeros(4, dtype=np.uint64), 2)
    with pytest.raises(Exception):
        gpu.ntt(np.zeros((2, 4), dtype=np.uint64), np.zeros(4, dtype=np.uint64), 29)


def test_domain_and_kzg_mirrors(gpu, oc, golden):
    import halo2_scaffold_b200 as h2
    g = golden["domain"]
    d = h2.EvaluationDomain(int(g["j"]), int(g["k"]), lib=gpu)
    coeff = d.lagrange_to_coeff(g["lagrange"])
    assert (coeff == g["coeff"]).all()
    ext = d.coeff_to_extended(coeff)
    assert (ext == g["extended"]).all()
    assert (d.extended_to_coeff(ext) == g["back"]).all()
    # test_commit_lagrange of halo2_proofs: commit_lagrange(evals) == commit(iNTT(evals)) when g_lagrange = iDFT(g)
    k = 8
    n = 1 << k
    dom = h2.EvaluationDomain(3, k, lib=gpu)
    # SRS with known discrete logs: g_i = [s^i] G; g_lagrange_j = [l_j(s)] G -- built from scalars through the oracle generator
    s = 0x1234567
    pows = [pow(s, i, o.R_MOD) for i in range(n)]
    lag = o.best_fft(list(pows), pow(dom.omega, -1, o.R_MOD), k)
    lag = [x * pow(n, -1, o.R_MOD) % o.R_MOD for x in lag]
    G = np.zeros((1, 8), dtype=np.uint64)
    G[0, :4] = oc.ints_to_words([o.to_mont(1, o.P_MOD)])[0]
    G[0, 4:] = oc.ints_to_words([o.to_mont(2, o.P_MOD)])[0]

    def mul_gen(ks):
        out = np.zeros((len(ks), 8), dtype=np.uint64)
        for i, kk in enumerate(ks):
            sc = oc.ints_to_words([o.to_mont(kk, o.R_MOD)])
            out[i] = pc.affine_of(oc, oc.best_multiexp(sc, G, 1))
        return out
    params = h2.ParamsKZG(k, mul_gen(pows), mul_gen(lag), lib=gpu)
    evals = oc.random_fr(77, n)
    c1 = pc.affine_of(oc, params.commit_lagrange(evals))
    c2 = pc.affine_of(oc, params.commit(dom.lagrange_to_coeff(evals)))
    # the same identity through the batched commits and the one-upload column pipeline of the mirror
    many = params.commit_lagrange_many([evals, evals[: n // 2]])
    r = params.commit_lagrange_and_convert(dom, evals)
    c3 = pc.affine_of(oc, params.commit_many([r["coeff"]])[0])
    params.close()
    assert (c1 == c2).all() and (pc.affine_of(oc, many[0]) == c1).all() and (pc.affine_of(oc, r["commitment"]) == c1).all() and (c3 == c1).all()
    assert (r["coeff"] == dom.lagrange_to_coeff(evals)).all() and (r["extended"] == dom.coeff_to_extended(r["coeff"])).all()


def test_cpp_host_mirror_over_the_c_abi(gpu, oc, tmp_path):
    from host_mirror_case import run_host_mirror
    run_host_mirror(oc, gpu.path, tmp_path, k=10, j=4)
    run_host_mirror(oc, gpu.path, tmp_path, k=5, j=3)       # examples/standard_plonk.rs: k = 5, degree 3


def test_grand_product_building_blocks(gpu, oc):
    pc.check_grand_product_blocks(gpu, oc, [1, 17, 1024, 1025, 16385, (1 << 18) + 3, 1 << 22])


def test_polynomial_evaluation_and_kate_division(gpu, oc):
    pc.check_poly_eval_and_division(gpu, oc, [1, 2, 17, 256, 257, 65537, (1 << 20) - 1, 1 << 22])


def test_permutation_and_lookup_grand_products(gpu, oc):
    pc.check_grand_products(gpu, oc, [1, 64, 4096, 1 << 16, (1 << 18) + 5])


def test_quotient_of_a_satisfied_circuit_is_a_polynomial(gpu, oc):
    assert pc.check_quotient_is_a_polynomial(gpu, oc, k=6, seed=4)[0]
    assert not pc.check_quotient_is_a_polynomial(gpu, oc, k=6, seed=5, break_it="sigma")[0]


def test_prover_rows_golden(gpu, golden):
    pc.check_golden_prover(gpu, golden["prover"])


def test_lookup_permute_async_status(gpu, oc):
    pc.check_lookup_permute_async(gpu, oc)


def test_lookup_permute_expression_pair(gpu, oc):
    pc.check_lookup_permute(gpu, oc, [(64, 58, 10, "random", 2), (1 << 12, (1 << 12) - 6, 1000, "random", 3), (1 << 16, (1 << 16) - 6, 1 << 10, "small", 4),
                                      (1 << 17, (1 << 17) - 6, 70000, "skewed", 5), ((1 << 18) + 100, (1 << 18) + 94, 1 << 19, "random", 6)])


def test_linear_combination_of_columns(gpu, oc):
    pc.check_lincomb(gpu, oc, [(1, 1), (5000, 3), (1 << 16, 32), (3001, 45)])


def test_divide_by_vanishing_poly(gpu, oc):
    pc.check_vanishing_division(gpu, oc, [(3, 5), (4, 8), (5, 9), (9, 6), (12, 5)])


def test_g1_point_codec(gpu, oc):
    for n in (1, 33, 5000, 1 << 16):
        pc.check_g1_codec(gpu, oc, n)


def test_srs_file_round_trip(gpu, oc, tmp_path):
    pc.check_srs_file_round_trip(gpu, oc, tmp_path, 5)
    pc.check_srs_file_round_trip(gpu, oc, tmp_path, 14)


def test_evaluate_graph_random_programs(gpu, oc):
    cases = [(1, 1, 3, 21), (1000, 1, 40, 22), (1 << 12, 4, 150, 23), ((1 << 14) + 77, 2, 300, 24), (1 << 16, 4, 80, 25), (1 << 18, 4, 30, 26),
             (1 << 15, 8, 600, 27), (300000, 3, 50, 29)]
    pc.check_evaluate_graph(gpu, oc, cases)


def test_evaluate_graph_many_live_values(gpu, oc):
    from halo2_scaffold_b200 import evaluation as ev
    size = 5000
    adv = [oc.random_fr(5, size)]
    sc = oc.random_fr(6, 4)
    vals = oc.random_fr(7, size)
    none = np.zeros((0, 4), dtype=np.uint64)
    for n_live in (6, 12, 24, 48):
        graph, n_const = pc.wide_graph(n_live)
        g, ga = pc._graph_pair(oc, graph, n_const, n_live)
        assert (ev.evaluate_graph(gpu, ga, [], adv, [], none, *sc, vals, 1) == oc.evaluate_graph(g, [], adv, [], none, *sc, vals, 1)).all(), n_live


def test_evaluate_graph_property(gpu, oc):
    pc.check_evaluate_graph_property(gpu, oc, examples=40, max_rows=20000, max_calcs=400)


def test_evaluate_h_row_shards(gpu, oc):
    pc.check_evaluate_h_sharded(gpu, oc, ek=14, k=12, groups=2, seed=8, shards=((0, 5000, 24), (5000, 6000, 40), (11000, 5384, 24)))


def test_evaluate_h_all_three_loops(gpu, oc):
    pc.check_evaluate_h(gpu, oc, [(5, 3, 1, 1), (12, 10, 2, 2), (16, 14, 3, 3), (18, 16, 1, 4)])


def test_msm_randomised_shapes(gpu, oc):
    pc.check_msm_random(gpu, oc, examples=25, max_n=40000, spacings=(-1, 0, 8, 12, 14, 16), windows=(0, 0, 0, 2, 4, 7, 8))


def test_batched_columns_match_single_calls(gpu, oc):
    n = 1 << 14
    P = oc.gen_points(71, n)
    cols = [gpu.gen_scalars(80 + j, n - 1000 * j, j % 2) for j in range(5)] + [np.zeros((0, 4), dtype=np.uint64)]
    h = gpu.register_bases(P)
    try:
        got = gpu.msm_batch_registered(cols, h)
        for j, c in enumerate(cols):
            assert (pc.affine_of(oc, got[j]) == pc.affine_of(oc, oc.best_multiexp(c, P[:c.shape[0]]))).all(), j
    finally:
        gpu.unregister_bases(h)
    k = 15
    polys = [oc.random_fr(90 + j, 1 << k) for j in range(3)]
    want = [oc.best_fft(a, pc.omega_words(oc, k), k) for a in polys]
    gpu.ntt_batch(polys, pc.omega_words(oc, k), k)
    for a, w in zip(polys, want):
        assert (a == w).all()


@pytest.mark.parametrize("k,count", [(10, 33), (16, 8), (20, 3)])
def test_batched_ntts_share_pass_launches(gpu, oc, k, count):
    pc.check_batched_ntts(gpu, oc, k, count)


@pytest.mark.parametrize("shape,batched", [(dict(k=8, A=1, LK=0, d=3), True), (dict(k=12, A=2, LK=1, d=4), True), (dict(k=11, A=6, LK=2, d=4), True),
                                           (dict(k=10, A=3, LK=1, d=4), False)])
def test_device_resident_proof_pipeline_matches_oracle_pipeline(gpu, oc, shape, batched):
    """tools/proof_pipeline_core.py -- every prover step on device-resident columns, the independent calls of a phase batched --
    against the same flow recomputed with the CPU oracle: every commitment and every evaluation."""
    import pipeline_oracle
    counts = pipeline_oracle.check_pipeline(gpu, oc, shape, batched=batched)
    assert counts["msm"] >= 7 and counts["eval"] >= 10


@pytest.mark.parametrize("j,k", [(3, 10), (4, 16), (4, 20)])
def test_column_pipeline_single_upload(gpu, oc, j, k):
    pc.check_column_pipeline(gpu, oc, j, k)


def test_fr_transpose_tma_and_ragged(gpu, oc):
    # the re-layout step of the split NTT: whole tiles go through cp.async.bulk + mbarrier (UBLKCP), ragged shapes through the LSU kernel
    pc.check_fr_transpose(gpu, oc)
    pc.check_fr_transpose(gpu, oc, shapes=((2048, 4096),))


def test_in_process_multi_device_paths(gpu):
    """Point-range sharding of one MSM across every visible GPU + concurrent callers (fresh process: own library instance)."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "multi_device_check.py")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "MULTI_DEVICE_OK" in out.stdout, (out.stdout[-500:], out.stderr[-2000:])


# ---- full benchmark sizes: size-independent properties -------------------------------------------------------------
def _dot_with_generator_scalars(oc, scalars_mont, seed, n):
    """sum_i s_i * z_i mod r for the synthetic bases P_i = [z_i] G (z_i = SplitMix64 stream `seed`)."""
    st = seed
    zs = np.empty(n, dtype=np.uint64)
    # vectorised SplitMix64 over indices
    idx = np.arange(1, n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    zw = np.zeros((n, 4), dtype=np.uint64)
    zw[:, 0] = z
    prod = oc.field_op("fr", "mul", scalars_mont, oc.fr_to_mont(zw))     # s_i * z_i (Montgomery)
    # tree-sum in Fr with the oracle's vector add
    cur = prod
    while cur.shape[0] > 1:
        if cur.shape[0] & 1:
            cur = np.vstack([cur, np.zeros((1, 4), dtype=np.uint64)])
        half = cur.shape[0] // 2
        cur = oc.field_op("fr", "add", np.ascontiguousarray(cur[:half]), np.ascontiguousarray(cur[half:]))
    return o.from_mont(oc.words_to_ints(cur)[0], o.R_MOD)


@pytest.mark.parametrize("k,kind", [(22, 0), (24, 0), (24, 1)])
def test_msm_full_size_checksum(gpu, oc, k, kind):
    """MSM(s, [z_i]G) must equal [sum s_i z_i]G: an O(n) field-only checksum that is independent of any MSM code."""
    n = 1 << k
    seed_p = 0xB2001000 + k
    s = gpu.gen_scalars(0xB2000000 + k, n, kind)
    d_s, d_p, d_o = gpu.dev_alloc(0, n * 32), gpu.dev_alloc(0, n * 64), gpu.dev_alloc(0, 96)
    try:
        gpu.h2d(0, d_s, s)
        gpu.gen_points_dev(0, seed_p, n, d_p)
        gpu.msm_dev(0, d_s, d_p, n, d_o)
        gpu.dev_sync(0)
        out = np.zeros(12, dtype=np.uint64)
        gpu.d2h(0, out, d_o)
    finally:
        for p in (d_s, d_p, d_o):
            gpu.dev_free(0, p)
    t = _dot_with_generator_scalars(oc, s, seed_p, n)
    want = o.g1_mul(o.G1_GEN, t)
    got_w = oc.words_to_ints(pc.affine_of(oc, out).reshape(2, 4))
    got = (o.from_mont(got_w[0], o.P_MOD), o.from_mont(got_w[1], o.P_MOD))
    assert got == want


@pytest.mark.parametrize("k,kind", [(22, 1), (24, 0), (24, 1)])
def test_msm_window_tables_full_size_checksum(gpu, oc, k, kind):
    """Same O(n) checksum through the registered-SRS path (window tables, one shared bucket set, device-resident scalars)."""
    n = 1 << k
    seed_p = 0xB2001000 + k
    s = gpu.gen_scalars(0xB2000000 + k, n, kind)
    h = gpu.register_bases(gpu.gen_points(seed_p, n))
    d_s, d_o = gpu.dev_alloc(0, n * 32), gpu.dev_alloc(0, 224)
    try:
        assert gpu.base_set_info(h)["n_tables"] > 1
        gpu.h2d(0, d_s, s)
        gpu.msm_dev_registered(0, d_s, h, 0, n, d_o)
        gpu.dev_sync(0)
        out = np.zeros(28, dtype=np.uint64)
        gpu.d2h(0, out, d_o)
        host = gpu.msm_registered(s, h)            # host-pointer entry point over the same tables
    finally:
        gpu.unregister_bases(h)
        for p in (d_s, d_o):
            gpu.dev_free(0, p)
    t = _dot_with_generator_scalars(oc, s, seed_p, n)
    want = o.g1_mul(o.G1_GEN, t)
    for res in (out[:12], host):
        got_w = oc.words_to_ints(pc.affine_of(oc, res).reshape(2, 4))
        assert (o.from_mont(got_w[0], o.P_MOD), o.from_mont(got_w[1], o.P_MOD)) == want


def test_device_checksum_matches_host_dot_product(gpu, oc):
    """h2b_msm_checksum_dev (what bench.py's `verified` flag rests on) against the dot product taken with the oracle's field ops."""
    n, seed_p = (1 << 18) + 77, 0xB2009000
    s = gpu.gen_scalars(0xB2008000, n, 1)
    d_s, d_c = gpu.dev_alloc(0, n * 32), gpu.dev_alloc(0, 32)
    try:
        gpu.h2d(0, d_s, s)
        gpu.msm_checksum_dev(0, d_s, seed_p, n, d_c)
        gpu.dev_sync(0)
        c = np.zeros(4, dtype=np.uint64)
        gpu.d2h(0, c, d_c)
    finally:
        gpu.dev_free(0, d_s)
        gpu.dev_free(0, d_c)
    assert sum(int(c[i]) << (64 * i) for i in range(4)) == _dot_with_generator_scalars(oc, s, seed_p, n)


@pytest.mark.parametrize("k,kind,env", [(25, 0, {}), (22, 0, {"H2B_MSM_SORT2_MIN_LOG": "20"}), (22, 1, {"H2B_MSM_SORT2_MIN_LOG": "20"}),
                                        (20, 0, {"H2B_MSM_SORT2_MIN_LOG": "16", "H2B_MSM_PRECOMP": "22"})])
def test_msm_partitioned_sort_full_size_checksum(gpu, k, kind, env):
    """The two-level partitioned sort (msm.cu section 2c; default from 2^25 points on, forced lower here) at full sizes: uniform and
    witness-like columns, 20- and 22-bit windows, device-resident and host-pointer entry points, against the O(n) checksum.  Fresh
    process per case (the thresholds are read once)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from halo2_scaffold_b200._lib import Lib\n"
        "from halo2_scaffold_b200 import verify as V\n"
        "L = Lib(); L.init_device(0)\n"
        "k, kind = %d, %d; n = 1 << k; seed_p = 0xB2001000 + k\n"
        "h = L.register_bases(L.gen_points(seed_p, n))\n"
        "d_s, d_o, d_c = L.dev_alloc(0, n * 32), L.dev_alloc(0, 224), L.dev_alloc(0, 32)\n"
        "L.gen_scalars_dev(0, 0xB2000000 + k, n, kind, d_s)\n"
        "L.msm_checksum_dev(0, d_s, seed_p, n, d_c)\n"
        "L.msm_dev_registered(0, d_s, h, 0, n, d_o); L.dev_sync(0)\n"
        "out, c = np.zeros(28, dtype=np.uint64), np.zeros(4, dtype=np.uint64)\n"
        "L.d2h(0, out, d_o); L.d2h(0, c, d_c)\n"
        "s = np.empty((n, 4), dtype=np.uint64); L.d2h(0, s, d_s)\n"
        "want = V.scalar_mul_generator(V.words_to_int(c))\n"
        "assert V.jacobian_words_to_affine(out) == want, 'device-resident'\n"
        "assert V.jacobian_words_to_affine(L.msm_registered(s, h)) == want, 'host pointer (chunked upload)'\n"
        "print('SORT2_OK')\n") % (root, k, kind)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "SORT2_OK" in out.stdout, (out.stdout[-500:], out.stderr[-2000:])


def test_ntt_full_size_round_trip_and_spot_values(gpu, oc):
    """k = 24: iNTT(NTT(a)) == n * a, and a handful of output coefficients checked by direct evaluation
    out[i] = sum_j a[j] w^(ij) for a sparse input (so the sum is cheap)."""
    k = 24
    n = 1 << k
    w = pc.omega_words(oc, k)
    wi = pc.omega_words(oc, k, inverse=True)
    a = gpu.gen_scalars(0xA24, n, 0)
    b = gpu.ntt(a.copy(), w, k)
    c = gpu.ntt(b, wi, k)
    ninv = oc.ints_to_words([o.to_mont(pow(n, -1, o.R_MOD), o.R_MOD)])[0]
    step = 4099
    assert (oc.fr_scale(np.ascontiguousarray(c[::step]), ninv) == a[::step]).all()
    assert (oc.fr_scale(np.ascontiguousarray(c[-1000:]), ninv) == a[-1000:]).all()
    # sparse input: 5 non-zero coefficients
    sp = np.zeros((n, 4), dtype=np.uint64)
    pos = [0, 1, 12345, n // 2 + 7, n - 1]
    vals = o.random_fr(5, 5)
    sp[pos] = oc.ints_to_words([o.to_mont(v, o.R_MOD) for v in vals])
    out = gpu.ntt(sp, w, k)
    wint = o.omega_for(k)
    for i in (0, 1, 2, 77777, n // 2, n - 1):
        want = sum(v * pow(wint, (i * j) % n, o.R_MOD) for v, j in zip(vals, pos)) % o.R_MOD
        assert oc.words_to_ints(out[i:i + 1])[0] == o.to_mont(want, o.R_MOD), i


def test_ntt_large_direct_compare(gpu, oc):
    pc.check_ntt(gpu, oc, 23)


def test_msm_window_independence_at_2_22(gpu, oc):
    n = 1 << 22
    s = gpu.gen_scalars(31, n, 1)
    P = gpu.gen_points(32, n)
    res = []
    for cw in (0, 12, 19):
        gpu.set_msm_window(cw)
        res.append(pc.affine_of(oc, gpu.msm(s, P)))
    gpu.set_msm_window(0)
    assert (res[0] == res[1]).all() and (res[0] == res[2]).all()
    # and against the oracle on the witness-like column (mostly 0 / 1 / small: fast on the CPU too)
    assert (res[0] == pc.affine_of(oc, oc.best_multiexp(s, P))).all()


def test_async_upload_overlaps_and_delivers(gpu, oc):
    # a pageable column uploaded with h2b_memcpy_h2d_async while an NTT is in flight on the same stream: later work sees the data
    n = 1 << 18
    a, b = oc.random_fr(0xAB1, n), oc.random_fr(0xAB2, n)
    w = pc.omega_words(oc, 18)
    d_a, d_b = gpu.dev_alloc(0, n * 32), gpu.dev_alloc(0, n * 32)
    try:
        gpu.h2d(0, d_a, a)
        gpu.ntt_dev(0, d_a, w, 18)
        gpu.h2d_async(0, d_b, b)
        gpu.ntt_dev(0, d_b, w, 18)
        gpu.dev_sync(0)
        out_a, out_b = np.empty_like(a), np.empty_like(b)
        gpu.d2h(0, out_a, d_a)
        gpu.d2h(0, out_b, d_b)
        assert (out_a == oc.best_fft(a, w, 18)).all() and (out_b == oc.best_fft(b, w, 18)).all()
    finally:
        gpu.dev_free(0, d_a)
        gpu.dev_free(0, d_b)


def test_msm_duplicate_identity_and_opposite_points(gpu, oc, golden):
    pc.check_golden_msm(gpu, oc, golden["msm"])
    for n, kind in ((1 << 17, 0), (200001, 1)):
        pc.check_msm_opposite_points(gpu, oc, n, kind)


def test_bench_dump_outputs(tmp_path):
    # bench.py --dump-outputs: the outputs of the last timed step of every leg; with one warm-up step both NTT legs have applied
    # the same number of transforms to the same column, and every MSM leg sums the same points
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--k", "12", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                          "--no-widened", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["verified"] and line["steps"] == 2, line["checks"]
    d = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert sorted(d) == ["msm", "msm_e2e", "msm_registered_pinned", "msm_witness", "ntt", "ntt_e2e", "ntt_rows"]
    assert all(a.dtype == np.float64 for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    assert (d["ntt_rows"] == np.arange(1 << 12)).all() and d["ntt"].shape == (1 << 12, 8)
    assert (d["ntt"] == d["ntt_e2e"]).all()
    assert d["msm"].shape == (2, 8) and d["msm"].any()
    assert (d["msm"] == d["msm_e2e"]).all() and (d["msm"] == d["msm_registered_pinned"]).all()
    assert (d["msm_witness"] != d["msm"]).any()
