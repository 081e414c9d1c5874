"""compress_selectors and the fixed columns of keygen_vk / keygen_pk on the device (h2b_selector_exclusion,
h2b_keygen_fixed_build_vk / build_pk, halo2_scaffold_b200.keygen.compress_selectors), against the CPU restatement of upstream's
process / keygen_vk / keygen_pk in tests/cpp/fixed_keygen_oracle.cpp.

CPU: the kernel sources through the emulator at k = 3 .. 8.  GPU: the C ABI on a B200 at k = 10, 16, 20 and 22.  The pins that need
no recollection of upstream: the exclusion matrix is np.any(a_i & a_j), no two members of a combination share a row, every
combination keeps max(deg - 1) + len <= max_degree, each substitution expression is non-zero exactly on its selector's rows, and
commit_lagrange(column) = commit(poly) with extended_to_coeff(coset) = poly padded with zeros."""
import ctypes
import subprocess

import numpy as np
import pytest

import bn254 as o
from harness import (Consts, W, affine, build_mirror, build_oracle, disjoint, ints, orc_srs_setup, run_on_emulated_devices, sparse,
                     threads)

H2B_ERR_BAD_ARGUMENT = -2
R = o.R_MOD


# ---- helpers ---------------------------------------------------------------------------------------------------------
def oracle():
    """tests/cpp/fixed_keygen_oracle.cpp"""
    vp, u32, i32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int
    return build_oracle("fixed_keygen_oracle", dict(orc_selector_exclusion=[vp, u32, u32, vp], orc_compress_selectors=[vp, vp, u32, u32, u32, vp, vp, vp, vp],
                                                    orc_fixed_build=[vp, u32, u32, u32, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
                        restypes=dict(orc_compress_selectors=u32))


def acts_array(acts, n):
    return np.ascontiguousarray(np.asarray(acts, dtype=np.uint8).reshape(-1, n))


def orc_exclusion(acts, k):
    a = acts_array(acts, 1 << k)
    out = np.empty((a.shape[0], a.shape[0]), dtype=np.uint8)
    oracle().orc_selector_exclusion(a.ctypes.data, a.shape[0], k, out.ctypes.data)
    return out.astype(bool)


def orc_compress(acts, degrees, max_degree, k):
    """process -> (combination_of, root_of, len_of, combination columns (C, n, 4))"""
    n = 1 << k
    a = acts_array(acts, n)
    S = a.shape[0]
    deg = np.ascontiguousarray(degrees, dtype=np.uint32)
    co, ro, lo = (np.zeros(S, dtype=np.uint32) for _ in range(3))
    cols = np.empty((max(S, 1), n, 4), dtype=np.uint64)
    C = oracle().orc_compress_selectors(a.ctypes.data, deg.ctypes.data, S, k, max_degree, co.ctypes.data, ro.ctypes.data, lo.ctypes.data, cols.ctypes.data)
    return co, ro, lo, cols[:C]


def orc_fixed_build(columns, c, g_lagrange=None, want_pk=True):
    cols = np.ascontiguousarray(columns, dtype=np.uint64)
    m = cols.shape[0]
    jac = np.empty((m, 12), dtype=np.uint64) if g_lagrange is not None else None
    polys = np.empty((m, c.n, 4), dtype=np.uint64) if want_pk else None
    cosets = np.empty((m, 1 << c.ek, 4), dtype=np.uint64) if want_pk else None
    gl = np.ascontiguousarray(g_lagrange, dtype=np.uint64) if g_lagrange is not None else None
    p = lambda x: x.ctypes.data if x is not None else None
    oracle().orc_fixed_build(cols.ctypes.data, m, c.k, c.ek, c.omega_inv.ctypes.data, c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data,
                             p(gl), threads(), p(jac), p(polys), p(cosets))
    return jac, polys, cosets


def cases(oc, k, seed):
    """(name, fixed (F, n, 4), activations (S, n) bool, degrees, max_degree)"""
    n = 1 << k
    rng = np.random.default_rng(seed)
    fx = lambda F: np.stack([oc.random_fr(seed * 31 + i, n) for i in range(F)]) if F else np.zeros((0, n, 4), dtype=np.uint64)
    mixed = sparse(rng, 12, n, 1.0 / 16)
    mixed[3] = False                     # never active
    mixed[7] = True                      # active on every row
    overlap = sparse(rng, 4, n, 0.25)
    overlap[:, 0] = True
    lib_acts = sparse(rng, 3, n, 0.5)
    lib_acts[:, 1] = True
    return [
        ("fixed only", fx(3), np.zeros((0, n), dtype=bool), [], 5),
        ("selectors only", fx(0), sparse(rng, 5, n, 1.0 / 8), [1, 2, 3, 4, 2], 5),
        ("all overlapping", fx(1), overlap, [2, 2, 2, 2], 5),
        ("disjoint equal degrees", fx(1), disjoint(10, n), [3] * 10, 5),
        ("random mixed degrees", fx(2), mixed, [int(x) for x in rng.integers(0, 5, size=12)], 5),
        ("more than 16 combinations", fx(2), disjoint(20, n, 24), [0] * 18 + [2, 2], 4),
        ("halo2-lib shape", fx(2), lib_acts, [3, 3, 3], 4),
    ]


def device_assignment(L, acts, degrees, max_degree):
    from halo2_scaffold_b200 import keygen as kg
    return kg.compress_selectors(list(acts), degrees, max_degree, lib=L)


def check_against_oracle(L, oc, k, seed, which=None):
    c = Consts(L, k)
    pts = oc.gen_points(seed, c.n)
    h = L.register_bases(pts)
    try:
        for name, fixed, acts, degrees, max_degree in cases(oc, k, seed):
            if which and name not in which:
                continue
            co, ro, lo, comb_cols = orc_compress(acts, degrees, max_degree, k)
            a = device_assignment(L, acts, degrees, max_degree)
            assert (a["combination_of"] == co).all() and (a["root_of"] == ro).all() and a["n_combinations"] == len(comb_cols), (k, name)
            assert a["expressions"] == [(int(x), int(y), int(z)) for x, y, z in zip(co, ro, lo)], (k, name)
            C = a["n_combinations"]
            r = L.keygen_fixed_build_pk(list(fixed), list(acts), co, ro, C, k, c.ek, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
            all_cols = np.concatenate([fixed, comb_cols]) if C else fixed
            jac, polys, cosets = orc_fixed_build(all_cols, c, pts)
            if C:
                assert (np.stack(r["combination_values"]) == comb_cols).all(), (k, name)
            assert (np.stack(r["polys"]) == polys).all(), (k, name)
            assert (np.stack(r["cosets"]) == cosets).all(), (k, name)
            vk = L.keygen_fixed_build_vk(list(fixed), list(acts), co, ro, C, k, h)
            assert (affine(oc, vk) == affine(oc, jac)).all(), (k, name)
    finally:
        L.unregister_bases(h)


def check_exclusion(L, k, S, seed, density):
    rng = np.random.default_rng(seed)
    acts = sparse(rng, S, 1 << k, density)
    acts[S // 2] = False
    got = L.selector_exclusion(list(acts), k)
    assert (got == orc_exclusion(acts, k)).all()
    want = np.array([[i != j and bool(np.any(acts[i] & acts[j])) for j in range(S)] for i in range(S)])
    assert (got == want).all()
    return got


# ---- pins that need no recollection of upstream ------------------------------------------------------------------------
def check_pins(L, oc, k, fixed, acts, degrees, max_degree, seed):
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import keygen as kg
    c = Consts(L, k)
    n, S = c.n, len(acts)
    a = kg.compress_selectors(list(acts), degrees, max_degree, lib=L)
    simple = [s for s in range(S) if degrees[s] > 0]
    excl = L.selector_exclusion([acts[s] for s in simple], k)
    for i in range(len(simple)):
        for j in range(len(simple)):
            assert excl[i, j] == (i != j and bool(np.any(acts[simple[i]] & acts[simple[j]])))
    params = h2.ParamsKZG.setup(k, oc.random_fr(seed, 1)[0], lib=L)
    try:
        vk = kg.fixed_build_vk(params, c.dom, list(fixed), list(acts), a)
        pk = kg.fixed_build_pk(params, c.dom, list(fixed), list(acts), a)
        cols = list(fixed) + pk["combination_values"]
        assert (affine(oc, vk) == affine(oc, params.commit_lagrange_many(cols))).all()
        assert (affine(oc, vk) == affine(oc, params.commit_many(pk["polys"]))).all()
    finally:
        params.close()
    for poly, coset in zip(pk["polys"], pk["cosets"]):
        coeff = c.dom.extended_to_coeff(coset)
        assert (coeff[:n] == poly).all() and (coeff[n:] == 0).all()
    C = a["n_combinations"]
    for comb in range(C):
        members = [s for s in range(S) if a["combination_of"][s] == comb]
        hits = np.sum([acts[s] for s in members], axis=0)
        assert hits.max() <= 1, comb
        assert max(degrees[s] - 1 for s in members) + len(members) <= max_degree, comb
        # the column as small integers: every row holds F::from(t) for some t in 0 ..= len
        col = pk["combination_values"][comb]
        q = np.full(n, -1, dtype=np.int64)
        for t in range(len(members) + 1):
            q[(col == W(t)).all(axis=1)] = t
        assert (q >= 0).all(), comb
        for s in members:
            comb_s, root, ln = a["expressions"][s]
            assert comb_s == comb and ln == len(members)
            # q * prod_{r = 1..len, r != root} (r - q): a product of integers below len + 1, non-zero mod R exactly when non-zero
            val = q.copy()
            for r in range(1, ln + 1):
                if r != root:
                    val = val * (r - q)
            assert ((val != 0) == acts[s]).all(), (comb, s)


def pins_shapes(oc, k, seed, A=8):
    n = 1 << k
    rng = np.random.default_rng(seed)
    lib_acts = sparse(rng, A, n, 0.5)
    fixed = np.stack([oc.random_fr(seed * 7 + i, n) for i in range(2)])
    return [(fixed, lib_acts, [3] * A, 4),
            (fixed[:1], disjoint(12, n), [1, 2, 3, 3, 2, 1, 0, 3, 3, 2, 1, 3], 5)]


# ---- refused inputs --------------------------------------------------------------------------------------------------------
def check_refused(L, oc, k=4):
    c = Consts(L, k)
    n = c.n
    fixed = [oc.random_fr(3 + i, n) for i in range(2)]
    acts = [np.ascontiguousarray(x, dtype=np.uint8) for x in disjoint(4, n)]
    co, ro = np.array([0, 0, 1, 1], dtype=np.uint32), np.array([1, 2, 1, 2], dtype=np.uint32)
    pts = oc.gen_points(78, n)
    h, h_short = L.register_bases(pts), L.register_bases(pts[:n // 2])
    sentinel = np.uint64(0xA5A5A5A5A5A5A5A5)
    vp = ctypes.c_void_p
    arr = lambda xs: (vp * len(xs))(*[x.ctypes.data if x is not None else None for x in xs]) if xs is not None else None
    overlapping = [a.copy() for a in acts]
    overlapping[1][0] = 1                                          # selectors 0 and 1 of combination 0 both on row 0

    def args(**kw):
        d = dict(fixed=fixed, F=2, acts=acts, S=4, co=co, ro=ro, C=2, k=k)
        d.update(kw)
        return d

    bad = [args(k=29), args(fixed=None), args(fixed=[fixed[0], None]), args(acts=None), args(acts=[acts[0], None, acts[2], acts[3]]),
           args(co=None), args(ro=None), args(co=np.array([0, 0, 2, 1], dtype=np.uint32)), args(ro=np.array([1, 0, 1, 2], dtype=np.uint32)),
           args(C=3), args(acts=overlapping), args(F=0, S=0, C=0), args(S=0)]
    p = lambda x: x.ctypes.data if x is not None else None
    try:
        for a in bad:
            vk = np.full((a["F"] + a["C"], 12), sentinel)
            rc = L.L.h2b_keygen_fixed_build_vk(arr(a["fixed"]), a["F"], arr(a["acts"]), a["S"], p(a["co"]), p(a["ro"]), a["C"], a["k"], h, vk.ctypes.data)
            assert rc == H2B_ERR_BAD_ARGUMENT and (vk == sentinel).all(), {x: y for x, y in a.items() if x in ("F", "S", "C", "k")}
            T = a["F"] + a["C"]
            outs = [[np.full((n, 4), sentinel) for _ in range(a["C"])], [np.full((n, 4), sentinel) for _ in range(T)],
                    [np.full((1 << c.ek, 4), sentinel) for _ in range(T)]]
            rc = L.L.h2b_keygen_fixed_build_pk(arr(a["fixed"]), a["F"], arr(a["acts"]), a["S"], p(a["co"]), p(a["ro"]), a["C"], a["k"], c.ek,
                                               c.omega_inv.ctypes.data, c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data, *[arr(x) for x in outs])
            assert rc == H2B_ERR_BAD_ARGUMENT and all((x == sentinel).all() for xs in outs for x in xs)
        good = args()
        for handle in (0xFFFFFFF0, h_short):
            vk = np.full((4, 12), sentinel)
            rc = L.L.h2b_keygen_fixed_build_vk(arr(fixed), 2, arr(acts), 4, co.ctypes.data, ro.ctypes.data, 2, k, handle, vk.ctypes.data)
            assert rc == H2B_ERR_BAD_ARGUMENT and (vk == sentinel).all()
        assert L.L.h2b_keygen_fixed_build_vk(arr(fixed), 2, arr(acts), 4, co.ctypes.data, ro.ctypes.data, 2, k, h, None) == H2B_ERR_BAD_ARGUMENT
        for ek in (k - 1, 29):
            outs = [None, [np.full((n, 4), sentinel) for _ in range(4)], None]
            rc = L.L.h2b_keygen_fixed_build_pk(arr(fixed), 2, arr(acts), 4, co.ctypes.data, ro.ctypes.data, 2, k, ek, c.omega_inv.ctypes.data,
                                               c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data, *[arr(x) for x in outs])
            assert rc == H2B_ERR_BAD_ARGUMENT and all((x == sentinel).all() for x in outs[1])
        # a null entry in an output array is refused before anything is written
        outs = [None, [np.full((n, 4), sentinel) for _ in range(3)] + [None], None]
        rc = L.L.h2b_keygen_fixed_build_pk(arr(fixed), 2, arr(acts), 4, co.ctypes.data, ro.ctypes.data, 2, k, c.ek, c.omega_inv.ctypes.data,
                                           c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data, *[arr(x) for x in outs])
        assert rc == H2B_ERR_BAD_ARGUMENT and all((x == sentinel).all() for x in outs[1][:3])
        # the exclusion matrix: bad arguments, and S = 0 writes nothing
        out = np.full((4, 4), 7, dtype=np.uint8)
        assert L.L.h2b_selector_exclusion(arr(acts), 4, 29, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT
        assert L.L.h2b_selector_exclusion(None, 4, k, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT
        assert L.L.h2b_selector_exclusion(arr([acts[0], None]), 2, k, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT
        assert L.L.h2b_selector_exclusion(arr(acts), 4, k, None) == H2B_ERR_BAD_ARGUMENT
        assert L.L.h2b_selector_exclusion(None, 0, k, out.ctypes.data) == 0
        assert (out == 7).all()
        assert good["S"] == 4
    finally:
        L.unregister_bases(h)
        L.unregister_bases(h_short)


# ---- the C++ mirror, and every device ----------------------------------------------------------------------------------------
def check_cpp_mirror(oc, lib_path, tmp_path, k):
    exe = build_mirror("fixed_keygen_mirror", lib_path, tmp_path)
    n = 1 << k
    s = oc.random_fr(950 + k, 1)[0]
    s.tofile(str(tmp_path / "s.bin"))
    _, fixed, acts, degrees, max_degree = cases(oc, k, 960 + k)[4]
    fixed.tofile(str(tmp_path / "fixed.bin"))
    acts_array(acts, n).tofile(str(tmp_path / "activations.bin"))
    np.array(degrees, dtype=np.uint32).tofile(str(tmp_path / "degrees.bin"))
    out = subprocess.run([exe, str(tmp_path), str(k), str(len(fixed)), str(len(acts)), str(max_degree)], capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and "FIXED_KEYGEN_MIRROR_OK" in out.stdout, (out.stdout, out.stderr)
    co, ro, lo, comb_cols = orc_compress(acts, degrees, max_degree, k)
    C = len(comb_cols)
    rd = lambda name, shape, dt=np.uint64: np.fromfile(str(tmp_path / name), dtype=dt).reshape(shape)
    assert (rd("assignment.bin", (3, len(acts)), np.uint32) == np.stack([co, ro, lo])).all()
    c = Consts.on_host(k)
    _, gl = orc_srs_setup(k, s)
    jac, polys, cosets = orc_fixed_build(np.concatenate([fixed, comb_cols]), c, gl)
    assert (rd("values.bin", comb_cols.shape) == comb_cols).all()
    assert (rd("polys.bin", polys.shape) == polys).all()
    assert (rd("cosets.bin", cosets.shape) == cosets).all()
    assert (affine(oc, rd("vk.bin", (len(fixed) + C, 12))) == affine(oc, jac)).all()


def check_every_device(L, oc, k, seed):
    """the host entries with columns dealt over every device, with a replicated and a sharded g_lagrange set"""
    c = Consts(L, k)
    _, fixed, acts, degrees, max_degree = cases(oc, k, seed)[5]
    co, ro, lo, comb_cols = orc_compress(acts, degrees, max_degree, k)
    pts = oc.gen_points(seed, c.n)
    jac, polys, cosets = orc_fixed_build(np.concatenate([fixed, comb_cols]), c, pts)
    r = L.keygen_fixed_build_pk(list(fixed), list(acts), co, ro, len(comb_cols), k, c.ek, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
    assert (np.stack(r["polys"]) == polys).all() and (np.stack(r["cosets"]) == cosets).all()
    assert (np.stack(r["combination_values"]) == comb_cols).all()
    for register in (L.register_bases, L.register_bases_sharded):
        h = register(pts)
        try:
            vk = L.keygen_fixed_build_vk(list(fixed), list(acts), co, ro, len(comb_cols), k, h)
            assert (affine(oc, vk) == affine(oc, jac)).all(), register.__name__
        finally:
            L.unregister_bases(h)


# ---- the restatement itself, against big-int arithmetic ------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
def test_oracle_matches_bigint_definition(emu, oc, k):
    c = Consts(emu, k)
    n, ek = c.n, c.ek
    rng = np.random.default_rng(k)
    acts = sparse(rng, 6, n, 0.3)
    degrees = [0, 2, 1, 3, 2, 1]
    co, ro, lo, cols = orc_compress(acts, degrees, 4, k)
    # the columns hold each member's root on its rows, as integers
    for comb in range(len(cols)):
        want = [0] * n
        for s in range(6):
            if co[s] == comb:
                for r in range(n):
                    if acts[s, r]:
                        want[r] = int(ro[s])
        assert ints(cols[comb]) == want
    assert (orc_exclusion(acts, k) == np.array([[i != j and bool(np.any(acts[i] & acts[j])) for j in range(6)] for i in range(6)])).all()
    fixed = np.stack([oc.random_fr(k * 5 + i, n) for i in range(2)])
    all_cols = np.concatenate([fixed, cols])
    _, polys, cosets = orc_fixed_build(all_cols, c)
    w, we, z = c.dom.omega, c.dom.extended_omega, c.dom.g_coset
    for i in range(len(all_cols)):
        v = ints(all_cols[i])
        co_ = [pow(n, -1, R) * sum(v[j] * pow(w, -t * j % n, R) for j in range(n)) % R for t in range(n)]
        assert ints(polys[i]) == co_
        assert ints(cosets[i]) == [sum(co_[t] * pow(z * pow(we, e, R), t, R) for t in range(n)) % R for e in range(1 << ek)]


# ---- CPU: the kernel sources through the emulator ----------------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 5, 8])
def test_build_vk_pk_match_oracle_emu(emu, oc, k):
    check_against_oracle(emu, oc, k, 500 + k)


@pytest.mark.parametrize("k,S", [(3, 5), (6, 64), (8, 64), (7, 130)])
def test_exclusion_matches_bool_zip_emu(emu, k, S):
    check_exclusion(emu, k, S, 510 + k, 2.0 / S)


def test_refuses_bad_input_emu(emu, oc):
    check_refused(emu, oc)


@pytest.mark.parametrize("shape", [0, 1])
def test_pins_emu(emu, oc, shape):
    fixed, acts, degrees, max_degree = pins_shapes(oc, 6, 520, A=4)[shape]
    check_pins(emu, oc, 6, fixed, acts, degrees, max_degree, 521)


def test_cpp_mirror_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 4)


@pytest.mark.parametrize("devices", ["2", "3"])
def test_fixed_keygen_on_emulated_devices(emu, devices):
    run_on_emulated_devices("test_fixed_keygen", "t.check_every_device(L, oc, 4, 530)\n"
                                                 "t.check_against_oracle(L, oc, 3, 531, which=('random mixed degrees', 'fixed only', 'selectors only'))\n"
                                                 "t.check_refused(L, oc)", devices)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16])
def test_build_vk_pk_match_oracle(gpu, oc, k):
    check_against_oracle(gpu, oc, k, 600 + k)


@pytest.mark.gpu
def test_build_vk_pk_match_oracle_k20(gpu, oc):
    check_against_oracle(gpu, oc, 20, 620, which=("random mixed degrees", "halo2-lib shape"))


@pytest.mark.gpu
@pytest.mark.parametrize("k,S", [(10, 64), (16, 64), (20, 64), (12, 200)])
def test_exclusion_matches_bool_zip(gpu, k, S):
    check_exclusion(gpu, k, S, 630 + k, 1.0 / (4 * S))


@pytest.mark.gpu
def test_refuses_bad_input(gpu, oc):
    check_refused(gpu, oc)
    check_refused(gpu, oc, k=12)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1])
def test_pins_k22(gpu, oc, shape):
    fixed, acts, degrees, max_degree = pins_shapes(oc, 22, 640)[shape]
    check_pins(gpu, oc, 22, fixed, acts, degrees, max_degree, 641)


@pytest.mark.gpu
def test_cpp_mirror(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 12)


@pytest.mark.gpu
def test_every_device(gpu, oc):
    check_every_device(gpu, oc, 14, 650)
