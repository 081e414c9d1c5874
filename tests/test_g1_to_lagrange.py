"""g_to_lagrange on the device (h2b_g1_to_lagrange_dev), ParamsKZG::downsize built on it (h2b_srs_downsize) and the
variable-base scalar multiplication of its butterflies (h2b_ec_op op 5), against the CPU restatement of upstream's
g_to_lagrange in tests/cpp/g1_to_lagrange_oracle.cpp.

CPU: the kernel sources through the emulator at small k.  GPU: the C ABI on a B200 at k = 10, 16 and 20.  The independent
pin is setup(K, s) then downsize(k) == setup(k, s): setup builds g_lagrange by fixed-base multiplication of L_i(s), so it
shares no code with the G1 NTT."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import bn254 as o
import parity_cases as pc
from harness import affine_ints, build_mirror, build_oracle, mont, orc_srs_setup, run_on_emulated_devices

H2B_ERR_BAD_ARGUMENT = -2


# ---- helpers ---------------------------------------------------------------------------------------------------------
def oracle():
    """tests/cpp/g1_to_lagrange_oracle.cpp"""
    vp = ctypes.c_void_p
    return build_oracle("g1_to_lagrange_oracle", dict(orc_g1_to_lagrange=[vp, ctypes.c_uint32, ctypes.c_int, vp],
                                                      orc_g1_mul_points=[vp, vp, ctypes.c_size_t, ctypes.c_int, vp]))


def orc_g1_to_lagrange(points, k, threads=0):
    p = np.ascontiguousarray(points[:1 << k], dtype=np.uint64)
    out = np.empty((1 << k, 8), dtype=np.uint64)
    oracle().orc_g1_to_lagrange(p.ctypes.data, k, threads or os.cpu_count() or 1, out.ctypes.data)
    return out


def orc_g1_mul_points(points, scalars):
    p = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
    s = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
    out = np.empty_like(p)
    oracle().orc_g1_mul_points(p.ctypes.data, s.ctypes.data, p.shape[0], os.cpu_count() or 1, out.ctypes.data)
    return out


def random_points(oc, seed, n):
    return oc.gen_points(seed, n)


def neg(oc, points):
    """-P for affine Montgomery points (the identity stays (0, 0))"""
    ints = []
    for p in affine_ints(oc, points):
        ints += [0, 0] if p is None else [o.to_mont(p[0], o.P_MOD), o.to_mont(-p[1] % o.P_MOD, o.P_MOD)]
    return oc.ints_to_words(ints).reshape(-1, 8)


def edge_scalars():
    """0, 1, 2, r - 1, (r +- 1) / 2 and 2^(W j) +- 1, 2^(W j) at every window boundary of the windows W = 1 .. 6"""
    r = o.R_MOD
    vals = [0, 1, 2, r - 1, (r - 1) // 2, (r + 1) // 2]
    for W in range(1, 7):
        for j in range(1, 255 // W + 2):
            vals += [(1 << (W * j)) - 1, (1 << (W * j)) + 1, 1 << (W * j)]
    return sorted(set(v % r for v in vals))


def known_answer_cases(oc, k, seed):
    """(input, expected) pairs that need no oracle and drive every exceptional branch of the butterflies"""
    n = 1 << k
    P = random_points(oc, seed, 1)
    minus_P = neg(oc, P)
    Z = np.zeros((1, 8), dtype=np.uint64)
    cases = [(np.repeat(P, n, axis=0), np.concatenate([P, np.repeat(Z, n - 1, axis=0)]))]      # doubling and a - a
    if n >= 2:
        alt = np.concatenate([P, minus_P] * (n // 2))                                           # P, -P, P, -P, ...
        want = np.zeros((n, 8), dtype=np.uint64)
        want[n // 2] = P[0]
        cases.append((alt, want))
    cases.append((np.zeros((n, 8), dtype=np.uint64), np.zeros((n, 8), dtype=np.uint64)))       # all identity
    return cases


def with_scattered_identities(oc, k, seed):
    n = 1 << k
    pts = random_points(oc, seed, n)
    rng = np.random.default_rng(seed)
    pts[rng.choice(n, size=max(1, n // 4), replace=False)] = 0
    pts[0] = 0
    return pts


def check_against_oracle(L, oc, k, seed):
    pts = random_points(oc, seed, 1 << k)
    assert (L.g1_to_lagrange(pts, k) == orc_g1_to_lagrange(pts, k)).all(), k
    pts = with_scattered_identities(oc, k, seed + 1)
    assert (L.g1_to_lagrange(pts, k) == orc_g1_to_lagrange(pts, k)).all(), k


def check_known_answers(L, oc, k):
    for inp, want in known_answer_cases(oc, k, 40 + k):
        assert (L.g1_to_lagrange(inp, k) == want).all(), k


def check_scalar_mul_edges(L, oc, n_random=0):
    e = mont(oc, edge_scalars())
    if n_random:
        e = np.concatenate([e, oc.random_fr(61, n_random)])
    P = random_points(oc, 62, e.shape[0])
    P[1] = 0                                                    # the identity times a scalar
    q = np.zeros((e.shape[0], 8), dtype=np.uint64)
    q[:, :4] = e
    assert (L.ec_op(5, P, q) == orc_g1_mul_points(P, e)).all()


def check_refused(L, oc):
    r = L.srs_setup(4, oc.random_fr(70, 1)[0])
    hs = L.register_bases_sharded(random_points(oc, 71, 16)) if L.device_count() > 1 else None
    try:
        bad = [(r["handle_g"], 29), (r["handle_g"], 5), (0xFFFFFFF0, 2)]
        if hs is not None:
            bad.append((hs, 2))
        for h, k in bad:
            hg, hl = ctypes.c_uint64(0xDEAD), ctypes.c_uint64(0xBEEF)
            rc = L.L.h2b_srs_downsize(h, k, None, ctypes.byref(hg), ctypes.byref(hl))
            assert rc == H2B_ERR_BAD_ARGUMENT, (h, k, rc)
            assert hg.value == 0xDEAD and hl.value == 0xBEEF
        d = L.dev_alloc(0, 64 * 16)
        try:
            assert L.L.h2b_g1_to_lagrange_dev(0, None, 2, d, None) == H2B_ERR_BAD_ARGUMENT
            assert L.L.h2b_g1_to_lagrange_dev(0, d, 2, None, None) == H2B_ERR_BAD_ARGUMENT
            assert L.L.h2b_g1_to_lagrange_dev(0, d, 29, d, None) == H2B_ERR_BAD_ARGUMENT
        finally:
            L.dev_free(0, d)
    finally:
        L.unregister_bases(r["handle_g"])
        L.unregister_bases(r["handle_g_lagrange"])
        if hs is not None:
            L.unregister_bases(hs)


def check_setup_pin(L, oc, K, k, seed):
    """setup(K, s).downsize(k) == setup(k, s), both vectors bit for bit"""
    s = oc.random_fr(seed, 1)[0]
    big = L.srs_setup(K, s)
    try:
        small = L.srs_setup(k, s, register=False)
        r = L.srs_downsize(big["handle_g"], k)
        try:
            assert (r["g_lagrange"] == small["g_lagrange"]).all(), (K, k)
            # the new g set is the prefix: read it back through a second downsize of it at the same k
            r2 = L.srs_downsize(r["handle_g"], k, register=False)
            assert (r2["g_lagrange"] == small["g_lagrange"]).all(), (K, k)
            assert (big["g"][:1 << k] == small["g"]).all()
        finally:
            L.unregister_bases(r["handle_g"])
            L.unregister_bases(r["handle_g_lagrange"])
    finally:
        L.unregister_bases(big["handle_g"])
        L.unregister_bases(big["handle_g_lagrange"])


def check_params_downsize(L, oc, K, k, seed):
    import halo2_scaffold_b200 as h2
    params = h2.ParamsKZG.setup(K, oc.random_fr(seed, 1)[0], lib=L, g2_bytes=bytes(range(256)))
    try:
        old = (params._g, params._g_lagrange)
        g_before = params.g.copy()
        params.downsize(k)
        n = 1 << k
        assert params.k == k and params.n == n
        assert (params.g == g_before[:n]).all() and params.g.shape == (n, 8)
        assert params.g_lagrange.shape == (n, 8)
        assert params.g2_bytes == bytes(range(256))
        for h in old:
            with pytest.raises(RuntimeError):
                L.base_set_info(h)
        e = oc.random_fr(seed + 1, n)
        coeff = oc.fr_scale(oc.best_fft(e, pc.omega_words(oc, k, inverse=True), k), mont(oc, [pow(n, -1, o.R_MOD)])[0])
        assert (pc.affine_of(oc, params.commit_lagrange(e)) == pc.affine_of(oc, params.commit(coeff))).all()
    finally:
        params.close()


def check_handles_on_every_device(L, oc, K, k, seed):
    """both new sets of a downsize commit on every device exactly as the oracle does over the host vectors"""
    n = 1 << k
    s = oc.random_fr(seed, 1)[0]
    big = L.srs_setup(K, s)
    r = L.srs_downsize(big["handle_g"], k)
    L.unregister_bases(big["handle_g"])
    L.unregister_bases(big["handle_g_lagrange"])
    c = oc.random_fr(seed + 1, n)
    want = {r["handle_g"]: pc.affine_of(oc, oc.best_multiexp(c, big["g"][:n])),
            r["handle_g_lagrange"]: pc.affine_of(oc, oc.best_multiexp(c, r["g_lagrange"]))}
    try:
        for h in want:
            for dev in range(L.device_count()):
                d_s, d_b = L.dev_alloc(dev, n * 32), L.dev_alloc(dev, 224)
                try:
                    L.h2d(dev, d_s, c)
                    L.msm_dev_registered(dev, d_s, h, 0, n, d_b)
                    L.dev_sync(dev)
                    blk = np.empty(28, dtype=np.uint64)
                    L.d2h(dev, blk, d_b)
                finally:
                    L.dev_free(dev, d_s)
                    L.dev_free(dev, d_b)
                assert (pc.affine_of(oc, L.msm_fold_partials(blk, dev)) == want[h]).all(), (h, dev)
    finally:
        L.unregister_bases(r["handle_g"])
        L.unregister_bases(r["handle_g_lagrange"])


def check_cpp_mirror(oc, lib_path, tmp_path, K, k):
    """tests/cpp/srs_downsize_mirror.cpp: ParamsKZG::setup(K, s) then downsize(k) of the C++ host mirror"""
    exe = build_mirror("srs_downsize_mirror", lib_path, tmp_path)
    s = oc.random_fr(800 + k, 1)[0]
    s.tofile(str(tmp_path / "s.bin"))
    out = subprocess.run([exe, str(tmp_path), str(K), str(k)], capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and "SRS_DOWNSIZE_MIRROR_OK" in out.stdout, (out.stdout, out.stderr)
    g = np.fromfile(str(tmp_path / "g.bin"), dtype=np.uint64).reshape(-1, 8)
    gl = np.fromfile(str(tmp_path / "g_lagrange.bin"), dtype=np.uint64).reshape(-1, 8)
    wg, wgl = orc_srs_setup(k, s)
    assert (g == wg).all() and (gl == wgl).all()


# ---- the restatement itself, against the big-int definition --------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_restatement_matches_naive_dft(oc, k):
    n = 1 << k
    pts = with_scattered_identities(oc, k, 90 + k) if k >= 2 else random_points(oc, 90 + k, n)
    got = affine_ints(oc, orc_g1_to_lagrange(pts, k, threads=3))
    g = affine_ints(oc, pts)
    w_inv = pow(o.omega_for(k), -1, o.R_MOD)
    n_inv = pow(n, -1, o.R_MOD)
    want = []
    for i in range(n):
        acc = None
        for j in range(n):
            if g[j] is not None:
                acc = o.g1_add(acc, o.g1_mul(g[j], n_inv * pow(w_inv, i * j, o.R_MOD) % o.R_MOD))
        want.append(acc)
    assert got == want
    e = [0, 1, o.R_MOD - 1, 0x1234567890ABCDEF1122334455667788]
    P = random_points(oc, 95, len(e))
    assert affine_ints(oc, orc_g1_mul_points(P, mont(oc, e))) == [o.g1_mul(p, v) for p, v in zip(affine_ints(oc, P), e)]


# ---- CPU: the kernel sources through the emulator ----------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 1, 2, 5, 6])
def test_g1_to_lagrange_matches_restatement_emu(emu, oc, k):
    check_against_oracle(emu, oc, k, 100 + k)


@pytest.mark.parametrize("k", [1, 2, 4])
def test_g1_to_lagrange_known_answers_emu(emu, oc, k):
    check_known_answers(emu, oc, k)


def test_scalar_mul_edge_scalars_emu(emu, oc):
    check_scalar_mul_edges(emu, oc)


def test_downsize_refuses_bad_input_emu(emu, oc):
    check_refused(emu, oc)


@pytest.mark.parametrize("K,k", [(6, 3), (5, 5), (4, 0)])
def test_setup_then_downsize_is_setup_emu(emu, oc, K, k):
    check_setup_pin(emu, oc, K, k, 120 + K + k)


def test_params_downsize_emu(emu, oc):
    check_params_downsize(emu, oc, 6, 4, 130)


def test_cpp_mirror_downsize_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 5, 3)


@pytest.mark.parametrize("devices", ["2", "3"])
def test_downsize_handles_on_emulated_devices(emu, devices):
    run_on_emulated_devices("test_g1_to_lagrange", "t.check_handles_on_every_device(L, oc, 5, 4, 140)\n"
                                                   "t.check_refused(L, oc)", devices)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16])
def test_g1_to_lagrange_matches_restatement(gpu, oc, k):
    check_against_oracle(gpu, oc, k, 200 + k)
    check_known_answers(gpu, oc, k)


@pytest.mark.gpu
def test_scalar_mul_edge_scalars(gpu, oc):
    check_scalar_mul_edges(gpu, oc, 1 << 14)


@pytest.mark.gpu
def test_downsize_refuses_bad_input(gpu, oc):
    check_refused(gpu, oc)


@pytest.mark.gpu
@pytest.mark.parametrize("K,k", [(21, 20), (20, 20)])
def test_setup_then_downsize_is_setup(gpu, oc, K, k):
    check_setup_pin(gpu, oc, K, k, 220 + K + k)


@pytest.mark.gpu
def test_params_downsize_commit_identity(gpu, oc):
    check_params_downsize(gpu, oc, 21, 20, 230)


@pytest.mark.gpu
def test_cpp_mirror_downsize(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 13, 12)


@pytest.mark.gpu
def test_downsize_handles_on_every_device(gpu, oc):
    check_handles_on_every_device(gpu, oc, 15, 14, 240)
