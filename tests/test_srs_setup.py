"""ParamsKZG::setup on the device (h2b_srs_setup) and the fixed-base multiples of the generator it is built on
(h2b_g1_generator_mul_dev), against the CPU restatement of upstream's setup in tests/cpp/srs_setup_oracle.cpp.

CPU: the kernel sources through the emulator at small k.  GPU: the C ABI on a B200 at the sizes the examples use, plus
identities at k = 20 and 24 that share no code with the setup."""
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
def setup_oracle():
    """tests/cpp/srs_setup_oracle.cpp"""
    vp = ctypes.c_void_p
    return build_oracle("srs_setup_oracle", dict(orc_g1_generator_mul=[vp, ctypes.c_size_t, ctypes.c_int, vp]))


def orc_g1_generator_mul(scalars, threads=0):
    s = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
    out = np.empty((s.shape[0], 8), dtype=np.uint64)
    setup_oracle().orc_g1_generator_mul(s.ctypes.data, s.shape[0], threads or os.cpu_count() or 1, out.ctypes.data)
    return out


def edge_scalars():
    """0, 1, 2, r - 1, (r +- 1) / 2, 2^(W j) +- 1 at every window boundary of the candidate windows W = 8 .. 16, and scalars
    whose signed W-bit digits are all -1 (then a top +1) or all 2^(W-1)"""
    r = o.R_MOD
    vals = [0, 1, 2, r - 1, (r - 1) // 2, (r + 1) // 2]
    for W in (8, 12, 16):
        for j in range(1, 255 // W + 2):
            vals += [(1 << (W * j)) - 1, (1 << (W * j)) + 1, 1 << (W * j)]
        for m in range(1, 255 // W + 1):
            vals.append((1 << (W * m)) - sum(1 << (W * i) for i in range(m)))            # digits -1, ..., -1, 1
            vals.append(sum((1 << (W - 1)) << (W * i) for i in range(m)))                  # digits 2^(W-1)
    return [v % r for v in vals]


def omega_int(k):
    return o.omega_for(k)


def check_generator_mul(L, oc, n_random, seed=5):
    edges = mont(oc, edge_scalars())
    s = np.concatenate([edges, oc.random_fr(seed, n_random)]) if n_random else edges
    got = L.g1_generator_mul(s)
    assert (got == orc_g1_generator_mul(s)).all()
    return s.shape[0]


def check_setup_matches_restatement(L, oc, k, s):
    r = L.srs_setup(k, s, want_host=True, register=False)
    wg, wgl = orc_srs_setup(k, s)
    assert (r["g"] == wg).all(), k
    assert (r["g_lagrange"] == wgl).all(), k


def check_refused(L, oc):
    n4 = 1 << 4
    w4 = omega_int(4)
    bad = [(29, mont(oc, [5])[0]),
           (4, np.array([int(x) for x in oc.ints_to_words([o.R_MOD])[0]], dtype=np.uint64)),       # limbs >= r
           (4, mont(oc, [1])[0]), (4, mont(oc, [w4])[0]), (4, mont(oc, [pow(w4, n4 - 1, o.R_MOD)])[0]), (0, mont(oc, [1])[0])]
    for k, s in bad:
        s = np.ascontiguousarray(s, dtype=np.uint64)
        hg, hl = ctypes.c_uint64(0xDEAD), ctypes.c_uint64(0xBEEF)
        rc = L.L.h2b_srs_setup(k, s.ctypes.data, None, None, ctypes.byref(hg), ctypes.byref(hl))
        assert rc == H2B_ERR_BAD_ARGUMENT, (k, rc)
        assert hg.value == 0xDEAD and hl.value == 0xBEEF


def check_s_zero(L, oc, k):
    n = 1 << k
    r = L.srs_setup(k, np.zeros(4, dtype=np.uint64), register=False)
    G = orc_g1_generator_mul(mont(oc, [1]))[0]
    assert (r["g"][0] == G).all() and (r["g"][1:] == 0).all()
    assert (r["g_lagrange"] == orc_g1_generator_mul(mont(oc, [pow(n, -1, o.R_MOD)]))[0]).all()


def check_params_round_trip(L, oc, tmp_path, k, s):
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200.kzg import SerdeFormat
    params = h2.ParamsKZG.setup(k, s, lib=L, g2_bytes=bytes(range(256)))
    try:
        c = oc.random_fr(11, 1 << k)
        assert (pc.affine_of(oc, params.commit(c)) == pc.affine_of(oc, oc.best_multiexp(c, params.g))).all()
        for fmt in (SerdeFormat.Processed, SerdeFormat.RawBytes, SerdeFormat.RawBytesUnchecked):
            params.g2_bytes = bytes(range(128 if fmt == SerdeFormat.Processed else 256))
            path = str(tmp_path / ("setup_%d_%d.srs" % (k, fmt)))
            params.write_custom(path, fmt)
            back = h2.ParamsKZG.read_custom(path, fmt, lib=L)
            try:
                assert (back.g == params.g).all() and (back.g_lagrange == params.g_lagrange).all()
                assert back.g2_bytes == params.g2_bytes
            finally:
                back.close()
    finally:
        params.close()


def check_handles_on_every_device(L, oc, k, s):
    """both resident sets of a setup commit on every device exactly as on device 0 and as the oracle does"""
    n = 1 << k
    r = L.srs_setup(k, s)
    c = oc.random_fr(17, n)
    want = {h: pc.affine_of(oc, oc.best_multiexp(c, pts)) for h, pts in ((r["handle_g"], r["g"]), (r["handle_g_lagrange"], r["g_lagrange"]))}
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


def check_cpp_mirror(oc, lib_path, tmp_path, k):
    """tests/cpp/srs_setup_mirror.cpp against the restatement"""
    exe = build_mirror("srs_setup_mirror", lib_path, tmp_path)
    n = 1 << k
    s, poly = oc.random_fr(500 + k, 1)[0], oc.random_fr(501 + k, n)
    s.tofile(str(tmp_path / "s.bin"))
    poly.tofile(str(tmp_path / "poly.bin"))
    out = subprocess.run([exe, str(tmp_path), str(k)], capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and "SRS_SETUP_MIRROR_OK" in out.stdout, (out.stdout, out.stderr)
    g = np.fromfile(str(tmp_path / "g.bin"), dtype=np.uint64).reshape(-1, 8)
    gl = np.fromfile(str(tmp_path / "g_lagrange.bin"), dtype=np.uint64).reshape(-1, 8)
    wg, wgl = orc_srs_setup(k, s)
    assert (g == wg).all() and (gl == wgl).all()
    c = np.fromfile(str(tmp_path / "commit.bin"), dtype=np.uint64).reshape(2, 12)
    assert (pc.affine_of(oc, c[0]) == pc.affine_of(oc, oc.best_multiexp(poly, wg))).all()
    assert (pc.affine_of(oc, c[1]) == pc.affine_of(oc, oc.best_multiexp(poly, wgl))).all()


# ---- the restatement itself, against the big-int oracle ----------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_setup_restatement_matches_big_int_definition(oc, k):
    n = 1 << k
    s = 0x1234567890ABCDEF1122334455667788 % o.R_MOD
    g, gl = orc_srs_setup(k, mont(oc, [s])[0], threads=3)
    w = omega_int(k)
    c = (pow(s, n, o.R_MOD) - 1) * pow(n, -1, o.R_MOD) % o.R_MOD
    want_g = [o.g1_mul(o.G1_GEN, pow(s, i, o.R_MOD)) for i in range(n)]
    want_gl = [o.g1_mul(o.G1_GEN, c * pow(w, i, o.R_MOD) * pow(s - pow(w, i, o.R_MOD), -1, o.R_MOD)) for i in range(n)]
    assert affine_ints(oc, g) == want_g
    assert affine_ints(oc, gl) == want_gl
    scal = mont(oc, [0, 1, o.R_MOD - 1, s])
    assert affine_ints(oc, orc_g1_generator_mul(scal)) == [o.g1_mul(o.G1_GEN, v) for v in (0, 1, o.R_MOD - 1, s)]


# ---- CPU: the kernel sources through the emulator ----------------------------------------------------------------------
def test_generator_mul_edge_scalars_emu(emu, oc):
    check_generator_mul(emu, oc, 64)


@pytest.mark.parametrize("k", [0, 1, 4, 6])
def test_setup_matches_restatement_emu(emu, oc, k):
    check_setup_matches_restatement(emu, oc, k, oc.random_fr(100 + k, 1)[0])


def test_setup_refuses_bad_input_emu(emu, oc):
    check_refused(emu, oc)


def test_setup_with_s_zero_emu(emu, oc):
    check_s_zero(emu, oc, 3)


def test_setup_params_write_read_round_trip_emu(emu, oc, tmp_path):
    check_params_round_trip(emu, oc, tmp_path, 5, oc.random_fr(7, 1)[0])


def test_cpp_mirror_setup_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 5)


@pytest.mark.parametrize("devices", ["2", "3"])
def test_setup_handles_on_emulated_devices(emu, devices):
    run_on_emulated_devices("test_srs_setup", "t.check_handles_on_every_device(L, oc, 6, oc.random_fr(9, 1)[0])", devices)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_generator_mul_edge_scalars(gpu, oc):
    assert check_generator_mul(gpu, oc, (1 << 16) - len(edge_scalars())) == 1 << 16


@pytest.mark.gpu
def test_setup_refuses_bad_input(gpu, oc):
    check_refused(gpu, oc)
    check_s_zero(gpu, oc, 10)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16])
def test_setup_matches_restatement(gpu, oc, k):
    check_setup_matches_restatement(gpu, oc, k, oc.random_fr(200 + k, 1)[0])


@pytest.mark.gpu
def test_setup_params_write_read_round_trip(gpu, oc, tmp_path):
    check_params_round_trip(gpu, oc, tmp_path, 12, oc.random_fr(8, 1)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 24])
def test_setup_identities_at_scale(gpu, oc, k):
    """at sizes the restatement cannot reach in a test: identities of a genuine [s^i]G / [L_i(s)]G pair"""
    import halo2_scaffold_b200 as h2
    n = 1 << k
    s = oc.random_fr(300 + k, 1)[0]
    params = h2.ParamsKZG.setup(k, s, lib=gpu)
    try:
        # commit(c) = [c(s)] G: Horner evaluation on the CPU, one scalar multiplication of the oracle
        c = oc.random_fr(301 + k, n)
        want = orc_g1_generator_mul(oc.fr_eval_polynomial(c, s).reshape(1, 4))[0]
        assert (pc.affine_of(oc, params.commit(c)) == want).all()
        # commit_lagrange(e) = commit(iNTT(e))
        e = oc.random_fr(302 + k, n)
        coeff = oc.fr_scale(oc.best_fft(e, pc.omega_words(oc, k, inverse=True), k), mont(oc, [pow(n, -1, o.R_MOD)])[0])
        assert (pc.affine_of(oc, params.commit_lagrange(e)) == pc.affine_of(oc, params.commit(coeff))).all()
        # sum_i L_i(s) = 1
        ones = np.repeat(mont(oc, [1]), n, axis=0)
        assert (pc.affine_of(oc, params.commit_lagrange(ones)) == orc_g1_generator_mul(mont(oc, [1]))[0]).all()
        # every point is a valid curve point in range (checked raw decode)
        for v in (params.g, params.g_lagrange):
            gpu.g1_decode(v.view(np.uint8), 1)
    finally:
        params.close()


@pytest.mark.gpu
def test_cpp_mirror_setup(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 12)


@pytest.mark.gpu
def test_setup_handles_on_every_device(gpu, oc):
    check_handles_on_every_device(gpu, oc, 14, oc.random_fr(400, 1)[0])
