"""The SHPLONK multi-point opening on the device (h2b_shplonk_begin / finish / release, h2b_fr_eval_queries_dev,
halo2_scaffold_b200.multiopen) against tests/cpp/shplonk_oracle.cpp, the CPU restatement of upstream's ProverSHPLONK::create_proof.

The pin that needs no recollection of upstream: with the SRS of ParamsKZG::setup(k, s) for a known s, commit(p) = [p(s)] G, and the
verifier's pairing equation becomes the G1 identity
    (s - u) h2 + Z_{S_0}(u) h1 = [ sum_i v^i (z_i / z_0) sum_j y^j (P_ij(s) - R_ij(u)) ] G,
checked with the oracle's MSM; P_ij(s) and R_ij(u) come from the inputs on the host.  It fails for a verifier handed another
polynomial or an evaluation off by one.

CPU: the kernel sources through the emulator at k = 3 .. 7.  GPU: the product library at k = 10, 14, 16 and the lr22-like structure at
k = 20."""
import ctypes
import os
import sys

import numpy as np
import pytest

import bn254 as o
from harness import ROOT, build_oracle, ints, orc_srs_setup, threads

sys.path.insert(0, os.path.join(ROOT, "tools"))
H2B_ERR_BAD_ARGUMENT = -2
R = o.R_MOD


# ---- query structures --------------------------------------------------------------------------------------------------------
def lr_structure(A=6, LK=2, d=4):
    """(n_polys, [(poly, rotation)]) of a proof_pipeline_core.SHAPES circuit, chained as plonk/prover.rs chains its queries:
    instance {0}; gate advice {0, 1, 2, 3}; lookup advice {0}; permutation z {0, 1, -6} and the last set {0, 1}; lookup z {0, 1},
    permuted input {0, -1}, permuted table {0}; fixed {0}; sigma {0}; h_poly and the random poly {0}"""
    q, nxt = [], [0]

    def new():
        nxt[0] += 1
        return nxt[0] - 1
    q.append((new(), 0))
    for _ in range(A):
        p = new()
        q += [(p, r) for r in (0, 1, 2, 3)]
    q += [(new(), 0) for _ in range(LK)]
    columns = 1 + A + 1
    sets = -(-columns // (d - 2))
    for s in range(sets):
        p = new()
        q += [(p, 0), (p, 1)] + ([(p, -6)] if s < sets - 1 else [])
    for _ in range(LK):
        z, pi, pt = new(), new(), new()
        q += [(z, 0), (z, 1), (pi, 0), (pi, -1), (pt, 0)]
    q += [(new(), 0) for _ in range(A + 1)]
    q += [(new(), 0) for _ in range(columns)]
    q += [(new(), 0), (new(), 0)]
    return nxt[0], q


def structure(name, rng):
    if name == "one_point":
        return 1, [(0, 0)]
    if name == "lr22":
        return lr_structure()
    if name == "shuffled":
        P, q = lr_structure()
        order = rng.permutation(len(q))
        return P, [q[i] for i in order]
    if name == "duplicates":
        return 4, [(0, 0), (1, 1), (0, 0), (2, 0), (1, 1), (1, 0), (3, -1), (2, 0), (3, -1), (3, 0)]
    if name == "equal_contents":
        return 3, [(0, 0), (1, 0), (2, 1), (1, 1), (0, 1)]
    if name == "sixteen_points":
        return 2, [(0, r) for r in range(16)] + [(1, 0)]
    raise KeyError(name)


STRUCTURES = ["one_point", "lr22", "shuffled", "duplicates", "equal_contents", "sixteen_points"]


# ---- inputs, oracle and pin --------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, oc, k, name, seed):
        rng = np.random.default_rng(seed)
        self.k, self.n = k, 1 << k
        self.P, q = structure(name, rng)
        self.polys = [oc.random_fr(seed * 100 + i, self.n) for i in range(self.P)]
        if name == "equal_contents":
            self.polys[1] = self.polys[0].copy()
        self.x = int(rng.integers(1, 1 << 62)) * 7919 % R
        w = o.omega_for(k)
        self.queries = [(p, self.x * pow(w, r % (1 << k), R) % R) for p, r in q]
        self.y, self.v, self.u = (int(rng.integers(1, 1 << 62)) * 104729 % R for _ in range(3))
        self.s = int(rng.integers(2, 1 << 62)) * 65537 % R

    def indexed(self):
        return [(p, _w(x)) for p, x in self.queries]


def _w(x):
    from halo2_scaffold_b200.domain import fr_to_words
    return fr_to_words(int(x) % R)


def srs(case):
    g, _ = orc_srs_setup(case.k, _w(case.s))
    return g


def orc_shplonk(case, g, u=None):
    """tests/cpp/shplonk_oracle.cpp -> (status, h1 Jacobian, h2 Jacobian)"""
    vp, u32, i32, sz = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_size_t
    L = build_oracle("shplonk_oracle", dict(orc_shplonk=[vp, u32, sz, vp, vp, u32, vp, vp, vp, vp, i32, vp, vp]), restypes=dict(orc_shplonk=i32))
    polys = [np.ascontiguousarray(p) for p in case.polys]
    ptrs = (ctypes.c_void_p * len(polys))(*[p.ctypes.data for p in polys])
    qp = np.array([p for p, _ in case.queries], dtype=np.uint32)
    qx = np.stack([_w(x) for _, x in case.queries])
    y, v, uu = _w(case.y), _w(case.v), _w(case.u if u is None else u)
    h1, h2 = np.zeros(12, dtype=np.uint64), np.zeros(12, dtype=np.uint64)
    gg = np.ascontiguousarray(g)
    st = L.orc_shplonk(ptrs, len(polys), case.n, qp.ctypes.data, qx.ctypes.data, len(qp), gg.ctypes.data, y.ctypes.data, v.ctypes.data, uu.ctypes.data,
                       threads(), h1.ctypes.data, h2.ctypes.data)
    return st, h1, h2


def sets_of(case):
    """construct_intermediate_sets restated on integers: [(points, [polys])]"""
    order, pts = [], {}
    for p, x in case.queries:
        if p not in pts:
            order.append(p)
            pts[p] = []
        if x not in pts[p]:
            pts[p].append(x)
    sets = []
    for p in order:
        for s in sets:
            if set(s[0]) == set(pts[p]):
                s[1].append(p)
                break
        else:
            sets.append((pts[p], [p]))
    return sets


def trapdoor_holds(oc, case, g, h1, h2, u=None, poly_override=None, eval_shift=0):
    """(s - u) h2 + Z_{S_0}(u) h1 == [rhs] G, with P_ij(s) and R_ij(u) from the inputs"""
    u = case.u if u is None else u
    polys = list(case.polys)
    if poly_override is not None:
        polys[poly_override[0]] = poly_override[1]

    def ev(p, x):
        return ints(oc.fr_eval_polynomial(polys[p], _w(x)))[0]
    sets = sets_of(case)
    T = []
    for pts, _ in sets:
        T += [x for x in pts if x not in T]

    def vanish(pts):
        r = 1
        for t in pts:
            r = r * (u - t) % R
        return r
    z = [vanish([t for t in T if t not in pts]) for pts, _ in sets]
    z0inv = pow(z[0], -1, R)
    rhs, vi = 0, 1
    for (pts, members), zi in zip(sets, z):
        acc, yj = 0, 1
        for p in members:
            evals = [(ev(p, x) + eval_shift) % R for x in pts]
            r_u = 0
            for k_, xk in enumerate(pts):
                num, den = 1, 1
                for l_, xl in enumerate(pts):
                    if l_ != k_:
                        num, den = num * (u - xl) % R, den * (xk - xl) % R
                r_u = (r_u + evals[k_] * num * pow(den, -1, R)) % R
            acc = (acc + yj * (ev(p, case.s) - r_u)) % R
            yj = yj * case.y % R
        rhs = (rhs + vi * zi % R * z0inv % R * acc) % R
        vi = vi * case.v % R
    zs0 = vanish(sets[0][0])
    lhs = oc.g1_to_affine(oc.best_multiexp(np.stack([_w(case.s - u), _w(zs0)]), np.stack([oc.g1_to_affine(h2), oc.g1_to_affine(h1)])))
    want = oc.g1_to_affine(oc.best_multiexp(np.stack([_w(rhs)]), g[:1]))
    return bool((lhs == want).all())


def device_polys(L, case, device=0):
    ptrs = []
    for p in case.polys:
        d = L.dev_alloc(device, case.n * 32)
        L.h2d(device, d, p)
        ptrs.append(d)
    return ptrs


def device_open(L, case, handle, on_host=True, u=None, device=0, ptrs=None):
    polys = case.polys if on_host else ptrs
    h1, sess = L.shplonk_begin(device, polys, on_host, case.n, case.indexed(), handle, _w(case.y), _w(case.v))
    try:
        h2 = L.shplonk_finish(sess, _w(case.u if u is None else u))
    finally:
        L.shplonk_release(sess)
    return h1, h2


def check_case(L, oc, k, name, seed, device_ptrs=False, device=0):
    import oracle_c
    case = Case(oracle_c, k, name, seed)
    g = srs(case)
    handle = L.register_bases(g)
    ptrs = device_polys(L, case, device) if device_ptrs else None
    try:
        h1, h2 = device_open(L, case, handle, device=device)
        st, w1, w2 = orc_shplonk(case, g)
        assert st == 0
        assert (oc.g1_to_affine(h1) == oc.g1_to_affine(w1)).all(), (name, k, "h1")
        assert (oc.g1_to_affine(h2) == oc.g1_to_affine(w2)).all(), (name, k, "h2")
        assert trapdoor_holds(oc, case, g, h1, h2)
        if device_ptrs:
            d1, d2 = device_open(L, case, handle, on_host=False, ptrs=ptrs, device=device)
            # the MSM's Jacobian coordinates depend on its accumulation order: compare the points
            assert (oc.g1_to_affine(d1) == oc.g1_to_affine(h1)).all() and (oc.g1_to_affine(d2) == oc.g1_to_affine(h2)).all()
    finally:
        for d in ptrs or []:
            L.dev_free(device, d)
        L.unregister_bases(handle)
    return case, g, h1, h2


# ---- CPU: the emulator -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k", list(zip(STRUCTURES, [3, 6, 5, 4, 4, 5])))
def test_matches_oracle_and_trapdoor_emu(emu, oc, name, k):
    check_case(emu, oc, k, name, 900 + k)


def test_host_and_device_sessions_agree_emu(emu, oc):
    check_case(emu, oc, 7, "lr22", 977, device_ptrs=True)


def test_trapdoor_check_has_teeth_emu(emu, oc):
    case, g, h1, h2 = check_case(emu, oc, 4, "duplicates", 41)
    assert not trapdoor_holds(oc, case, g, h1, h2, poly_override=(1, case.polys[2]))
    assert not trapdoor_holds(oc, case, g, h1, h2, eval_shift=1)


def test_u_at_a_point_of_the_first_set_emu(emu, oc):
    import oracle_c
    case = Case(oracle_c, 4, "lr22", 55)
    g = srs(case)
    h = emu.register_bases(g)
    try:
        u = case.x                               # x is a point of every set, S_0 included: valid
        h1, h2 = device_open(emu, case, h, u=u)
        st, w1, w2 = orc_shplonk(case, g, u=u)
        assert st == 0
        assert (oc.g1_to_affine(h2) == oc.g1_to_affine(w2)).all()
        assert trapdoor_holds(oc, case, g, h1, h2, u=u)
        # u in T \ S_0 (x omega: a point of T that S_0 = {x} lacks): refused, output untouched; another u then works
        bad = case.x * o.omega_for(4) % R
        out = np.full(12, 7, dtype=np.uint64)
        h1b, sess = emu.shplonk_begin(0, case.polys, True, case.n, case.indexed(), h, _w(case.y), _w(case.v))
        try:
            assert emu.L.h2b_shplonk_finish(sess, _w(bad).ctypes.data, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT
            assert (out == 7).all()
            assert orc_shplonk(case, g, u=bad)[0] == 1
            assert (oc.g1_to_affine(emu.shplonk_finish(sess, _w(case.u))) == oc.g1_to_affine(device_open(emu, case, h)[1])).all()
            assert emu.L.h2b_shplonk_finish(sess, _w(case.u).ctypes.data, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT     # finished
        finally:
            emu.shplonk_release(sess)
        assert emu.L.h2b_shplonk_finish(sess, _w(case.u).ctypes.data, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT         # released
        assert emu.L.h2b_shplonk_release(sess) == H2B_ERR_BAD_ARGUMENT
    finally:
        emu.unregister_bases(h)


def test_eval_queries_emu(emu, oc):
    import oracle_c
    for k, name in ((3, "duplicates"), (6, "lr22"), (5, "sixteen_points")):
        case = Case(oracle_c, k, name, 300 + k)
        ptrs = device_polys(emu, case)
        nq = len(case.queries)
        d_out = emu.dev_alloc(0, nq * 32)
        try:
            emu.eval_queries_dev(0, ptrs, case.n, case.indexed(), d_out)
            emu.dev_sync(0)
            got = np.empty((nq, 4), dtype=np.uint64)
            emu.d2h(0, got, d_out)
            want = np.stack([oc.fr_eval_polynomial(case.polys[p], _w(x)) for p, x in case.queries])
            assert (got == want).all(), (k, name)
        finally:
            emu.dev_free(0, d_out)
            for d in ptrs:
                emu.dev_free(0, d)


def test_refusals_leave_outputs_untouched_emu(emu, oc):
    import oracle_c
    case = Case(oracle_c, 3, "duplicates", 12)
    g = srs(case)
    h = emu.register_bases(g)
    short = emu.register_bases(g[: case.n - 1])
    Lr = emu.L
    q = case.indexed()
    big = np.array([0xFFFFFFFFFFFFFFFF] * 4, dtype=np.uint64)
    polys = [np.ascontiguousarray(p) for p in case.polys]
    try:
        def begin(queries=q, n_polys=len(polys), n=case.n, handle=h, y=_w(case.y), v=_w(case.v)):
            from halo2_scaffold_b200._lib import _queries
            ptrs = (ctypes.c_void_p * len(polys))(*[p.ctypes.data for p in polys])
            out = np.full(12, 5, dtype=np.uint64)
            sess = ctypes.c_uint64(77)
            rc = Lr.h2b_shplonk_begin(0, ptrs, 1, n_polys, n, _queries(queries), len(queries), handle, y.ctypes.data, v.ctypes.data, out.ctypes.data,
                                      ctypes.byref(sess))
            assert (out == 5).all() and sess.value == 77
            return rc
        assert begin(queries=[(len(polys), q[0][1])] + q[1:]) == H2B_ERR_BAD_ARGUMENT           # poly index out of range
        assert begin(queries=[(p, x) for p, x in q if p != 3]) == H2B_ERR_BAD_ARGUMENT            # a poly no query uses
        assert begin(queries=[(0, big)] + q) == H2B_ERR_BAD_ARGUMENT                                # point >= r
        assert begin(y=big) == H2B_ERR_BAD_ARGUMENT and begin(v=big) == H2B_ERR_BAD_ARGUMENT      # challenge >= r
        assert begin(queries=[]) == H2B_ERR_BAD_ARGUMENT                                            # no queries
        assert begin(n=1) == H2B_ERR_BAD_ARGUMENT and begin(n=(1 << 28) + 1) == H2B_ERR_BAD_ARGUMENT
        seventeen = [(0, _w(case.x * pow(o.omega_for(3), r, R) + r)) for r in range(17)] + [(p, x) for p, x in q if p]
        assert begin(queries=seventeen) == H2B_ERR_BAD_ARGUMENT                                     # more than 16 points
        assert begin(handle=987654) == H2B_ERR_BAD_ARGUMENT and begin(handle=short) == H2B_ERR_BAD_ARGUMENT
        # finish: u >= r refused, output untouched
        h1, sess = emu.shplonk_begin(0, polys, True, case.n, q, h, _w(case.y), _w(case.v))
        out = np.full(12, 9, dtype=np.uint64)
        assert Lr.h2b_shplonk_finish(sess, big.ctypes.data, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT and (out == 9).all()
        emu.shplonk_release(sess)
        # eval_queries: the same refusals on its arguments
        from halo2_scaffold_b200._lib import _queries
        ptrs = (ctypes.c_void_p * len(polys))(*[p.ctypes.data for p in polys])
        assert Lr.h2b_fr_eval_queries_dev(0, ptrs, len(polys), case.n, _queries([(9, q[0][1])]), 1, out.ctypes.data, None) == H2B_ERR_BAD_ARGUMENT
        assert Lr.h2b_fr_eval_queries_dev(0, ptrs, len(polys), case.n, _queries(q), 0, out.ctypes.data, None) == H2B_ERR_BAD_ARGUMENT
        assert (out == 9).all()
    finally:
        emu.unregister_bases(h)
        emu.unregister_bases(short)


def test_python_prover_emu(emu, oc):
    """multiopen.ProverSHPLONK: identity by object, u squeezed after h1"""
    import oracle_c
    from halo2_scaffold_b200 import kzg, multiopen
    case = Case(oracle_c, 4, "equal_contents", 8)
    g = srs(case)
    params = kzg.ParamsKZG(case.k, g, g, lib=emu)
    try:
        seen = []
        queries = [(case.polys[p], _w(x)) for p, x in case.queries]
        h1, h2 = multiopen.ProverSHPLONK(params).create_proof(queries, _w(case.y), _w(case.v), lambda h: seen.append(h) or _w(case.u))
        st, w1, w2 = orc_shplonk(case, g)
        assert len(seen) == 1 and (seen[0] == h1).all()
        assert (oc.g1_to_affine(h2) == oc.g1_to_affine(w2)).all()
    finally:
        params.close()


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 14, 16])
@pytest.mark.parametrize("name", STRUCTURES)
def test_matches_oracle_and_trapdoor(gpu, oc, name, k):
    for device in range(gpu.device_count()):
        check_case(gpu, oc, k, name, 1000 + k + device, device_ptrs=(name == "lr22"), device=device)


@pytest.mark.gpu
def test_lr22_structure_k20(gpu, oc):
    check_case(gpu, oc, 20, "lr22", 2020, device_ptrs=True)


@pytest.mark.gpu
def test_eval_queries_and_memory(gpu, oc):
    import oracle_c
    import torch
    case = Case(oracle_c, 16, "lr22", 16)
    ptrs = device_polys(gpu, case)
    nq = len(case.queries)
    d_out = gpu.dev_alloc(0, nq * 32)
    try:
        gpu.eval_queries_dev(0, ptrs, case.n, case.indexed(), d_out)
        gpu.dev_sync(0)
        got = np.empty((nq, 4), dtype=np.uint64)
        gpu.d2h(0, got, d_out)
        want = np.stack([oc.fr_eval_polynomial(case.polys[p], _w(x)) for p, x in case.queries])
        assert (got == want).all()
        # a session's memory returns after release
        g = srs(case)
        h = gpu.register_bases(g)
        try:
            device_open(gpu, case, h)            # the grow-only scratch of the MSM and the divisions reaches its size first
            gpu.dev_sync(0)
            before = torch.cuda.mem_get_info(0)[0]
            _, sess = gpu.shplonk_begin(0, case.polys, True, case.n, case.indexed(), h, _w(case.y), _w(case.v))
            during = torch.cuda.mem_get_info(0)[0]
            gpu.shplonk_release(sess)
            after = torch.cuda.mem_get_info(0)[0]
            held = (3 + len(case.polys)) * case.n * 32
            assert before - during >= held - (64 << 20), (before, during, held)
            assert after >= before - (64 << 20), (before, after)
        finally:
            gpu.unregister_bases(h)
    finally:
        gpu.dev_free(0, d_out)
        for d in ptrs:
            gpu.dev_free(0, d)


# ---- the C++ mirror ----------------------------------------------------------------------------------------------------------
def check_cpp_mirror(oc, lib_path, tmp_path, k):
    import subprocess
    import oracle_c
    from harness import build_mirror
    exe = build_mirror("shplonk_mirror", lib_path, tmp_path)
    case = Case(oracle_c, k, "lr22", 70 + k)
    _w(case.s).tofile(str(tmp_path / "s.bin"))
    np.stack(case.polys).tofile(str(tmp_path / "polys.bin"))
    np.array([p for p, _ in case.queries], dtype=np.uint32).tofile(str(tmp_path / "qpoly.bin"))
    np.stack([_w(x) for _, x in case.queries]).tofile(str(tmp_path / "qpoint.bin"))
    np.stack([_w(case.y), _w(case.v), _w(case.u)]).tofile(str(tmp_path / "yvu.bin"))
    out = subprocess.run([exe, str(tmp_path), str(k), str(case.P), str(len(case.queries))], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "SHPLONK_MIRROR_OK" in out.stdout, out.stderr
    h = np.fromfile(str(tmp_path / "h.bin"), dtype=np.uint64).reshape(2, 12)
    st, w1, w2 = orc_shplonk(case, srs(case))
    assert st == 0
    assert (oc.g1_to_affine(h[0]) == oc.g1_to_affine(w1)).all() and (oc.g1_to_affine(h[1]) == oc.g1_to_affine(w2)).all()


def test_cpp_mirror_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 5)


@pytest.mark.gpu
def test_cpp_mirror(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 12)
