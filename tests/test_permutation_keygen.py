"""The permutation argument's keys and keygen_pk's indicator columns on the device (h2b_permutation_sigma_dev,
h2b_permutation_build_vk / build_pk, h2b_keygen_lagrange_indicators_dev), against the CPU restatement of upstream's
Assembly / build_vk / build_pk / keygen_pk in tests/cpp/permutation_keygen_oracle.cpp.

CPU: the kernel sources through the emulator at k = 3 .. 8.  GPU: the C ABI on a B200 at k = 10, 16, 20 and 22.  The pins
that need no recollection of upstream: sigma's cycles are the connected components of the copies, a witness constant on
them closes the permutation product, the toy circuit of parity_cases' quotient check gets its hand-built sigma,
commit_lagrange(sigma) = commit(coefficients), and l_active_row + l_last + l_blind = 1 with l0 = (1/n) sum X^i."""
import ctypes
import subprocess

import numpy as np
import pytest

import bn254 as o
from harness import (Consts, W, affine, build_mirror, build_oracle, ints, orc_mapping, orc_srs_setup, random_copies, run_on_emulated_devices,
                     threads)

H2B_ERR_BAD_ARGUMENT = -2
R = o.R_MOD


# ---- helpers ---------------------------------------------------------------------------------------------------------
def oracle():
    """tests/cpp/permutation_keygen_oracle.cpp"""
    vp, u32, i32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int
    return build_oracle("permutation_keygen_oracle", dict(orc_permutation_sigma=[vp, u32, u32, vp, vp, i32, vp],
                                                          orc_permutation_build_vk=[vp, u32, u32, vp, vp, vp, i32, vp],
                                                          orc_permutation_build_pk=[vp, u32, u32, u32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
                                                          orc_lagrange_indicators=[u32, u32, u32, vp, vp, vp, vp, i32, vp, vp, vp]))


def orc_build_pk(mapping, c):
    P = mapping.shape[0]
    m = np.ascontiguousarray(mapping)
    perm, polys = np.empty((P, c.n, 4), dtype=np.uint64), np.empty((P, c.n, 4), dtype=np.uint64)
    cosets = np.empty((P, 1 << c.ek, 4), dtype=np.uint64)
    oracle().orc_permutation_build_pk(m.ctypes.data, P, c.k, c.ek, c.delta.ctypes.data, c.omega.ctypes.data, c.omega_inv.ctypes.data, c.ifft.ctypes.data,
                                      c.ext_omega.ctypes.data, c.zeta.ctypes.data, threads(), perm.ctypes.data, polys.ctypes.data, cosets.ctypes.data)
    return perm, polys, cosets


def orc_build_vk(mapping, c, g_lagrange):
    P = mapping.shape[0]
    m, gl = np.ascontiguousarray(mapping), np.ascontiguousarray(g_lagrange, dtype=np.uint64)
    out = np.empty((P, 12), dtype=np.uint64)
    oracle().orc_permutation_build_vk(m.ctypes.data, P, c.k, c.delta.ctypes.data, c.omega.ctypes.data, gl.ctypes.data, threads(), out.ctypes.data)
    return out


def orc_indicators(c, bf):
    outs = [np.empty((1 << c.ek, 4), dtype=np.uint64) for _ in range(3)]
    oracle().orc_lagrange_indicators(c.k, c.ek, bf, c.omega_inv.ctypes.data, c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data, threads(),
                                     *[x.ctypes.data for x in outs])
    return outs


def device_pk(L, mapping, c):
    r = L.permutation_build_pk(mapping, c.k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
    return np.stack(r["permutations"]), np.stack(r["polys"]), np.stack(r["cosets"])


def one_cycle(P, n):
    """copies chaining every cell in flat order: one cycle through all P n cells"""
    return [(t // n, t % n, (t + 1) // n, (t + 1) % n) for t in range(P * n - 1)]


def cases(k, seed, big_P=17):
    n = 1 << k
    rng = np.random.default_rng(seed)
    return [("identity", 3, []), ("random", 4, random_copies(rng, 4, n, 2 * n)), ("one cycle", 3, one_cycle(3, n)),
            ("P = 1", 1, random_copies(rng, 1, n, n)), ("P above the launch chunk", big_P, random_copies(rng, big_P, n, 3 * n))]


def check_against_oracle(L, oc, k, seed, which=None, big_P=17):
    c = Consts(L, k)
    pts = oc.gen_points(seed, c.n)
    h = L.register_bases(pts)
    try:
        for name, P, copies in cases(k, seed, big_P):
            if which and name not in which:
                continue
            mapping = orc_mapping(P, k, copies)
            want = orc_build_pk(mapping, c)
            got = device_pk(L, mapping, c)
            for g, w, what in zip(got, want, ("permutations", "polys", "cosets")):
                assert (g == w).all(), (k, name, what)
            vk = L.permutation_build_vk(mapping, k, c.delta, c.omega, h)
            assert (affine(oc, vk) == affine(oc, orc_build_vk(mapping, c, pts))).all(), (k, name)
            # build_vk and build_pk agree on sigma: the commitments are those of build_pk's permutations
            assert (affine(oc, L.msm_batch_registered(list(got[0]), h)) == affine(oc, vk)).all(), (k, name)
    finally:
        L.unregister_bases(h)


def check_indicators(L, k, bfs):
    c = Consts(L, k)
    for bf in bfs:
        got = L.keygen_lagrange_indicators(k, c.ek, bf, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
        for g, w, what in zip(got, orc_indicators(c, bf), ("l0", "l_last", "l_active_row")):
            assert (g == w).all(), (k, bf, what)


def raw_build_pk(L, mapping_cols, P, k, c, outs, ek=None):
    vp = ctypes.c_void_p
    arr = lambda xs: (vp * len(xs))(*[x.ctypes.data if x is not None else None for x in xs]) if xs is not None else None
    return L.L.h2b_permutation_build_pk(arr(mapping_cols) if mapping_cols is not None else None, P, k, c.ek if ek is None else ek, c.delta.ctypes.data,
                                        c.omega.ctypes.data, c.omega_inv.ctypes.data, c.ifft.ctypes.data, c.ext_omega.ctypes.data, c.zeta.ctypes.data,
                                        *[arr(x) for x in outs])


def raw_build_vk(L, mapping_cols, P, k, c, handle, out):
    vp = ctypes.c_void_p
    m = (vp * len(mapping_cols))(*[x.ctypes.data for x in mapping_cols]) if mapping_cols is not None else None
    return L.L.h2b_permutation_build_vk(m, P, k, c.delta.ctypes.data, c.omega.ctypes.data, handle, out.ctypes.data if out is not None else None)


def check_refused(L, oc, k=4):
    c = Consts(L, k)
    n, P = c.n, 3
    good = orc_mapping(P, k, random_copies(np.random.default_rng(5), P, n, n))
    pts = oc.gen_points(77, n)
    h, h_short = L.register_bases(pts), L.register_bases(pts[:n // 2])
    sentinel = np.uint64(0xA5A5A5A5A5A5A5A5)
    try:
        bad_mappings = []
        for (i, j, col, row) in [(1, 3, P, 0), (0, n - 1, 0, n), (2, 0, 1 << 63, 0), (0, 7, 0, 1 << 40)]:
            m = good.copy()
            m[i, j] = (col, row)
            bad_mappings.append(m)
        for m in bad_mappings:
            cols = [np.ascontiguousarray(m[i]) for i in range(P)]
            outs = [[np.full((n, 4), sentinel) for _ in range(P)], [np.full((n, 4), sentinel) for _ in range(P)],
                    [np.full((1 << c.ek, 4), sentinel) for _ in range(P)]]
            assert raw_build_pk(L, cols, P, k, c, outs) == H2B_ERR_BAD_ARGUMENT
            assert all((x == sentinel).all() for xs in outs for x in xs)
            vk = np.full((P, 12), sentinel)
            assert raw_build_vk(L, cols, P, k, c, h, vk) == H2B_ERR_BAD_ARGUMENT
            assert (vk == sentinel).all()
            # the device-pointer entry reports 1 + the flat index of the entry
            flat = [int(i) * n + int(j) for i in range(P) for j in range(n) if m[i, j, 0] >= P or m[i, j, 1] >= n]
            assert flat_status(L, m, c) == flat[-1] + 1
        assert flat_status(L, good, c) == 0
        cols = [np.ascontiguousarray(good[i]) for i in range(P)]
        vk = np.full((P, 12), sentinel)
        for args in [(None, P, k, h), (cols, 0, k, h), (cols, P, 29, h), (cols, P, k, 0xFFFFFFF0), (cols, P, k, h_short)]:
            assert raw_build_vk(L, *args[:3], c, args[3], vk) == H2B_ERR_BAD_ARGUMENT, args[1:]
        assert raw_build_vk(L, cols, P, k, c, h, None) == H2B_ERR_BAD_ARGUMENT
        assert (vk == sentinel).all()
        outs = [[np.full((n, 4), sentinel) for _ in range(P)], None, None]
        for args in [(None, P, k, None), (cols, 0, k, None), (cols, P, 29, None), (cols, P, k, k - 1), (cols, P, k, 29)]:
            assert raw_build_pk(L, args[0], args[1], args[2], c, outs, ek=args[3]) == H2B_ERR_BAD_ARGUMENT, args[1:]
        assert raw_build_pk(L, cols, P, k, c, [[outs[0][0], None, outs[0][2]], None, None]) == H2B_ERR_BAD_ARGUMENT
        assert all((x == sentinel).all() for x in outs[0])
        # indicators and sigma: bad arguments fail before anything is launched
        d = L.dev_alloc(0, 32 << c.ek)
        try:
            ind = lambda kk, ek, bf, p: L.L.h2b_keygen_lagrange_indicators_dev(0, kk, ek, bf, c.omega_inv.ctypes.data, c.ifft.ctypes.data, c.ext_omega.ctypes.data,
                                                                               c.zeta.ctypes.data, p, d, d, None)
            assert ind(k, c.ek, n - 1, d) == H2B_ERR_BAD_ARGUMENT
            assert ind(k, c.ek, 1 << 32 - 1, d) == H2B_ERR_BAD_ARGUMENT
            assert ind(k, k - 1, 1, d) == H2B_ERR_BAD_ARGUMENT
            assert ind(k, 29, 1, d) == H2B_ERR_BAD_ARGUMENT
            assert ind(k, c.ek, 1, None) == H2B_ERR_BAD_ARGUMENT
            vp = ctypes.c_void_p
            one = (vp * 1)(d)
            sig = lambda mp, P_, kk, sg, st: L.L.h2b_permutation_sigma_dev(0, mp, P_, kk, c.delta.ctypes.data, c.omega.ctypes.data, sg, st, None)
            assert sig(one, 1, 29, one, d) == H2B_ERR_BAD_ARGUMENT
            assert sig(one, 0, k, one, d) == H2B_ERR_BAD_ARGUMENT
            assert sig(None, 1, k, one, d) == H2B_ERR_BAD_ARGUMENT
            assert sig(one, 1, k, None, d) == H2B_ERR_BAD_ARGUMENT
            assert sig(one, 1, k, one, None) == H2B_ERR_BAD_ARGUMENT
            assert sig((vp * 1)(None), 1, k, one, d) == H2B_ERR_BAD_ARGUMENT
        finally:
            L.dev_free(0, d)
    finally:
        L.unregister_bases(h)
        L.unregister_bases(h_short)


def flat_status(L, mapping, c, device=0):
    """h2b_permutation_sigma_dev on the device: the status word (and sigma checked against build_pk when it is 0)"""
    P, n = mapping.shape[0], c.n
    dm = [L.dev_alloc(device, n * 16) for _ in range(P)]
    ds = [L.dev_alloc(device, n * 32) for _ in range(P)]
    st = L.dev_alloc(device, 4)
    try:
        for i in range(P):
            L.h2d(device, dm[i], np.ascontiguousarray(mapping[i]))
        L.permutation_sigma_dev(device, dm, c.k, c.delta, c.omega, ds, st)
        L.dev_sync(device)
        status = np.zeros(1, dtype=np.uint32)
        L.d2h(device, status, st)
        if status[0] == 0:
            want = orc_build_pk(mapping, c)[0]
            for i in range(P):
                got = np.empty((n, 4), dtype=np.uint64)
                L.d2h(device, got, ds[i])
                assert (got == want[i]).all(), (device, i)
        return int(status[0])
    finally:
        for p in dm + ds + [st]:
            L.dev_free(device, p)


# ---- pins that need no recollection of upstream ------------------------------------------------------------------------
def components(P, copies):
    """connected components (size > 1) of the copy list, by union-find over the touched cells"""
    parent = {}

    def find(x):
        while parent.setdefault(x, x) != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x
    for (a, b, d, e) in copies:
        ra, rb = find((a, b)), find((d, e))
        if ra != rb:
            parent[ra] = rb
    groups = {}
    for x in list(parent):
        groups.setdefault(find(x), set()).add(x)
    return sorted((frozenset(g) for g in groups.values() if len(g) > 1), key=lambda g: min(g))


def check_cycle_pins(L, oc, k, P, n_copies, seed, bf=5):
    c = Consts(L, k)
    n, u = c.n, c.n - bf - 1
    rng = np.random.default_rng(seed)
    copies = random_copies(rng, P, n, n_copies, rows=u)
    mapping = orc_mapping(P, k, copies)
    ident = np.stack(L.permutation_build_pk(np.stack([np.stack([np.full(n, i, dtype=np.uint64), np.arange(n, dtype=np.uint64)], axis=1) for i in range(P)]),
                                            k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta, want_polys=False, want_cosets=False)["permutations"])
    sig = np.stack(L.permutation_build_pk(mapping, k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta, want_polys=False,
                                          want_cosets=False)["permutations"])
    # the identity sigma against the formula at (up to) 4096 sampled rows of every column
    rows = np.unique(np.concatenate([[0, n - 1], rng.integers(0, n, size=min(n, 4096))]))
    d_int, w_int = o.FR_DELTA, pow(c.dom.omega, 1, R)
    for i in range(P):
        got = ints(ident[i][rows])
        assert got == [pow(d_int, i, R) * pow(w_int, int(r), R) % R for r in rows], i
    # sigma's cycles are the components; cells no copy touches are fixed points
    comps = components(P, copies)
    touched = set().union(*comps) if comps else set()
    value_of = {cell: bytes(ident[cell[0]][cell[1]]) for cell in touched}
    cell_of = {v: cell for cell, v in value_of.items()}
    for comp in comps:
        start = min(comp)
        cyc, cur = {start}, cell_of[bytes(sig[start[0]][start[1]])]
        while cur != start:
            assert cur not in cyc
            cyc.add(cur)
            cur = cell_of[bytes(sig[cur[0]][cur[1]])]
        assert cyc == comp
    fixed = np.ones((P, n), dtype=bool)
    for (i, j) in touched:
        fixed[i, j] = False
    assert (sig[fixed] == ident[fixed]).all()
    # a witness constant on every component closes the permutation product at the last usable row; one changed copied cell breaks it
    vals = [oc.random_fr(seed * 13 + i, n) for i in range(P)]
    for t, comp in enumerate(comps):
        v = oc.random_fr(seed * 17 + t, 1)[0]
        for (i, j) in comp:
            vals[i][j] = v
    beta, gamma = oc.random_fr(seed * 19, 2)
    z = L.permutation_product(vals, list(sig), beta, gamma, c.delta, W(1), c.omega, W(1))
    assert ints(z[u:u + 1]) == [1]
    i, j = min(comps[0])
    vals[i][j] = oc.random_fr(seed * 23, 1)[0]
    z = L.permutation_product(vals, list(sig), beta, gamma, c.delta, W(1), c.omega, W(1))
    assert ints(z[u:u + 1]) != [1]


def check_toy_circuit_sigma(L, k=4, bf=5):
    """the copies of parity_cases.check_quotient_is_a_polynomial's toy circuit, restated from it: (column 0, row i + 1) == (column 2, row i)
    on even usable rows; its hand-built sigma swaps the two cells of every copy in the identity delta^j omega^i"""
    c = Consts(L, k)
    n = c.n
    u = n - (bf + 1)
    copies = [(0, i + 1, 2, i) for i in range(0, u - 1, 2)]
    DELTA = pow(7, 1 << 28, R)
    omega = c.dom.omega
    sigma = [[pow(DELTA, j, R) * pow(omega, i, R) % R for i in range(n)] for j in range(3)]
    for (j0, i0, j1, i1) in copies:
        sigma[j0][i0], sigma[j1][i1] = sigma[j1][i1], sigma[j0][i0]
    got = L.permutation_build_pk(orc_mapping(3, k, copies), k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)["permutations"]
    assert [ints(g) for g in got] == sigma


def check_commitment_and_indicator_pins(L, oc, k, P, seed, bf=5):
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import keygen as kg
    c = Consts(L, k)
    n = c.n
    params = h2.ParamsKZG.setup(k, oc.random_fr(seed, 1)[0], lib=L)
    try:
        mapping = orc_mapping(P, k, random_copies(np.random.default_rng(seed), P, n, min(4 * n, 4096)))
        vk = kg.permutation_build_vk(params, c.dom, mapping)
        pk = kg.permutation_build_pk(params, c.dom, mapping)
        assert (affine(oc, vk) == affine(oc, params.commit_many(pk["polys"]))).all()
        assert (affine(oc, vk) == affine(oc, params.commit_lagrange_many(pk["permutations"]))).all()
    finally:
        params.close()
    l0, l_last, l_active = kg.lagrange_indicators(c.dom, bf)
    blind = np.zeros((n, 4), dtype=np.uint64)
    blind[n - bf:] = W(1)
    l_blind = c.dom.coeff_to_extended(c.dom.lagrange_to_coeff(blind))
    one = oc.field_op("fr", "add", oc.field_op("fr", "add", l_active, l_last), l_blind)
    assert (one == W(1)).all()
    coeff = c.dom.extended_to_coeff(l0)
    assert (coeff[:n] == W(pow(n, -1, R))).all() and (coeff[n:] == 0).all()


def check_cpp_mirror(oc, lib_path, tmp_path, k, P, bf=3):
    exe = build_mirror("permutation_keygen_mirror", lib_path, tmp_path)
    n = 1 << k
    s = oc.random_fr(900 + k, 1)[0]
    s.tofile(str(tmp_path / "s.bin"))
    mapping = orc_mapping(P, k, random_copies(np.random.default_rng(k), P, n, 2 * n))
    mapping.tofile(str(tmp_path / "mapping.bin"))
    out = subprocess.run([exe, str(tmp_path), str(k), str(P), str(bf)], capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and "PERMUTATION_KEYGEN_MIRROR_OK" in out.stdout, (out.stdout, out.stderr)
    c = Consts.on_host(k)
    perm, polys, cosets = orc_build_pk(mapping, c)
    rd = lambda name, shape: np.fromfile(str(tmp_path / name), dtype=np.uint64).reshape(shape)
    assert (rd("permutations.bin", perm.shape) == perm).all()
    assert (rd("polys.bin", polys.shape) == polys).all()
    assert (rd("cosets.bin", cosets.shape) == cosets).all()
    _, gl = orc_srs_setup(k, s)
    assert (affine(oc, rd("vk.bin", (P, 12))) == affine(oc, orc_build_vk(mapping, c, gl))).all()
    for name, want in zip(("l0.bin", "l_last.bin", "l_active.bin"), orc_indicators(c, bf)):
        assert (rd(name, want.shape) == want).all(), name


def check_every_device(L, oc, k, P, seed):
    """the device-pointer sigma entry on every device, and the host entries with a sharded g_lagrange set"""
    c = Consts(L, k)
    mapping = orc_mapping(P, k, random_copies(np.random.default_rng(seed), P, c.n, 2 * c.n))
    for dev in range(L.device_count()):
        assert flat_status(L, mapping, c, dev) == 0, dev
    pts = oc.gen_points(seed, c.n)
    want = affine(oc, orc_build_vk(mapping, c, pts))
    for register in (L.register_bases, L.register_bases_sharded):
        h = register(pts)
        try:
            assert (affine(oc, L.permutation_build_vk(mapping, k, c.delta, c.omega, h)) == want).all(), register.__name__
        finally:
            L.unregister_bases(h)


# ---- the restatement itself, against big-int arithmetic ------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
def test_oracle_matches_bigint_definition(emu, oc, k):
    c = Consts(emu, k)
    n, ek = c.n, c.ek
    P = 3
    copies = random_copies(np.random.default_rng(k), P, n, 2 * n)
    mapping = orc_mapping(P, k, copies)
    perm, polys, cosets = orc_build_pk(mapping, c)
    w, we, z = c.dom.omega, c.dom.extended_omega, c.dom.g_coset
    for i in range(P):
        s = [pow(o.FR_DELTA, int(mapping[i, j, 0]), R) * pow(w, int(mapping[i, j, 1]), R) % R for j in range(n)]
        assert ints(perm[i]) == s
        co = [pow(n, -1, R) * sum(s[j] * pow(w, -t * j % n, R) for j in range(n)) % R for t in range(n)]
        assert ints(polys[i]) == co
        assert ints(cosets[i]) == [sum(co[t] * pow(z * pow(we, e, R), t, R) for t in range(n)) % R for e in range(1 << ek)]
    # Assembly: the mapping is a permutation whose cycles are the components of the copies
    img = {(int(mapping[i, j, 0]), int(mapping[i, j, 1])) for i in range(P) for j in range(n)}
    assert len(img) == P * n
    for bf in (0, 2):
        l0, l_last, l_active = [ints(x) for x in orc_indicators(c, bf)]
        ev = lambda rows: [sum(pow(n, -1, R) * pow(w, -t * r % n, R) * pow(z * pow(we, e, R), t, R) for r in rows for t in range(n)) % R
                           for e in range(1 << ek)]
        assert l0 == ev([0]) and l_last == ev([n - bf - 1]) and l_active == ev(range(n - bf - 1))


# ---- CPU: the kernel sources through the emulator ----------------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 5, 8])
def test_build_vk_pk_match_oracle_emu(emu, oc, k):
    check_against_oracle(emu, oc, k, 300 + k, which=None if k < 8 else ("random", "P above the launch chunk"))


@pytest.mark.parametrize("k", [3, 4, 6, 8])
def test_indicators_match_oracle_emu(emu, k):
    n = 1 << k
    check_indicators(emu, k, sorted({0, 1, 3, n - 2}))


def test_refuses_bad_input_emu(emu, oc):
    check_refused(emu, oc)


def test_cycles_and_product_pins_emu(emu, oc):
    check_cycle_pins(emu, oc, 6, 3, 60, 310)


def test_toy_circuit_sigma_emu(emu):
    check_toy_circuit_sigma(emu)


def test_commitment_and_indicator_pins_emu(emu, oc):
    check_commitment_and_indicator_pins(emu, oc, 5, 3, 320)


def test_cpp_mirror_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 4, 3)


@pytest.mark.parametrize("devices", ["2", "3"])
def test_keygen_on_emulated_devices(emu, devices):
    run_on_emulated_devices("test_permutation_keygen", "t.check_every_device(L, oc, 4, 5, 330)\n"
                                                       "t.check_against_oracle(L, oc, 3, 331, which=('random', 'P = 1'))\n"
                                                       "t.check_refused(L, oc)", devices)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 16])
def test_build_vk_pk_match_oracle(gpu, oc, k):
    check_against_oracle(gpu, oc, k, 400 + k)
    check_indicators(gpu, k, [0, 5, (1 << k) - 2])


@pytest.mark.gpu
def test_build_vk_pk_match_oracle_k20(gpu, oc):
    check_against_oracle(gpu, oc, 20, 420, which=("random",))
    check_indicators(gpu, 20, [5])


@pytest.mark.gpu
def test_refuses_bad_input(gpu, oc):
    check_refused(gpu, oc)
    check_refused(gpu, oc, k=12)


@pytest.mark.gpu
def test_pins_k22(gpu, oc):
    check_cycle_pins(gpu, oc, 22, 8, 4096, 430)
    check_toy_circuit_sigma(gpu)
    check_commitment_and_indicator_pins(gpu, oc, 22, 8, 431)


@pytest.mark.gpu
def test_cpp_mirror(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 12, 4)


@pytest.mark.gpu
def test_every_device(gpu, oc):
    check_every_device(gpu, oc, 14, 6, 440)
