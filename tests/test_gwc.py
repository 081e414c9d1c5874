"""The GWC multi-point opening on the device (h2b_gwc_create_proof, halo2_scaffold_b200.multiopen.ProverGWC) against
tests/cpp/gwc_oracle.cpp, the CPU restatement of upstream's ProverGWC::create_proof, and the batched kate division it runs on
(h2b_fr_kate_division_batch_dev) against one division at a time.

The pin that needs no recollection of upstream: with the SRS of ParamsKZG::setup(k, s) for a known s, commit(p) = [p(s)] G, and the GWC
verifier's pairing equation for the point z_i becomes the G1 identity
    (s - z_i) W_i = sum_j v^j C_ij - [sum_j v^j p_ij(z_i)] G  =  [ sum_j v^j (p_ij(s) - p_ij(z_i)) ] G,
checked with the oracle's MSM; p_ij(s) and p_ij(z_i) are evaluated on the host.  It fails for another polynomial, an evaluation off by
one, v powers continued across points, and a duplicated query counted once.  The oracle keeps upstream's evaluations and its
subtraction at coefficient 0, which the device drops: their agreement shows that kate_division never reads that coefficient.

CPU: the kernel sources through the emulator at k = 3 .. 7.  GPU: the product library at k = 10, 14, 16 and the lr22-like structure at
k = 20."""
import ctypes

import numpy as np
import pytest

import bn254 as o
import test_shplonk as ts
from harness import build_oracle, ints, orc_srs_setup, threads

H2B_ERR_BAD_ARGUMENT = -2
R = o.R_MOD
MSM_BATCH_MAX = 32                 # msm.cu's MSM_BATCH_MAX: the points of one group


# ---- query structures --------------------------------------------------------------------------------------------------------
def structure(name, rng):
    """(n_polys, [(poly, rotation)], constant polynomials); SHPLONK's structures and three more"""
    if name == "twenty_points":                      # SHPLONK refuses more than 16 points for one polynomial
        return 2, [(0, r) for r in range(20)] + [(1, 0), (1, 3)], False
    if name == "many_points":                        # more points than one MSM batch: the groups run in turn
        return 3, [(r % 3, r) for r in range(MSM_BATCH_MAX + 5)] + [(0, 0), (2, 7)], False
    if name == "constants":                          # every quotient is zero: W is the identity
        return 3, [(0, 0), (1, 0), (2, 1), (0, 1), (1, 2)], True
    P, q = ts.structure(name, rng)
    return P, q, False


STRUCTURES = ts.STRUCTURES + ["twenty_points", "many_points", "constants"]


class Case:
    def __init__(self, oc, k, name, seed):
        rng = np.random.default_rng(seed)
        self.k, self.n = k, 1 << k
        self.P, q, constant = structure(name, rng)
        self.polys = [oc.random_fr(seed * 100 + i, self.n) for i in range(self.P)]
        if constant:
            for p in self.polys:
                p[1:] = 0
        if name == "equal_contents":
            self.polys[1] = self.polys[0].copy()
        self.x = int(rng.integers(1, 1 << 62)) * 7919 % R
        w = o.omega_for(k)
        # rotations beyond n would fold onto others: the structures that need many distinct points take x + r instead
        distinct = name in ("twenty_points", "many_points")
        self.queries = [(p, (self.x + r) % R if distinct else self.x * pow(w, r % (1 << k), R) % R) for p, r in q]
        self.v = int(rng.integers(1, 1 << 62)) * 104729 % R
        self.s = int(rng.integers(2, 1 << 62)) * 65537 % R

    def indexed(self):
        return [(p, _w(x)) for p, x in self.queries]

    def points(self):
        """[(z, [poly of every query at z, in query order])], points in first-appearance order"""
        out = []
        for p, x in self.queries:
            for z, ps in out:
                if z == x:
                    ps.append(p)
                    break
            else:
                out.append((x, [p]))
        return out


_w = ts._w


def srs(case):
    g, _ = orc_srs_setup(case.k, _w(case.s))
    return g


def orc_gwc(case, g):
    """tests/cpp/gwc_oracle.cpp -> (points, 12) Jacobian"""
    vp, u32, i32, sz = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_size_t
    L = build_oracle("gwc_oracle", dict(orc_gwc=[vp, u32, sz, vp, vp, u32, vp, vp, i32, vp]), restypes=dict(orc_gwc=u32))
    polys = [np.ascontiguousarray(p) for p in case.polys]
    ptrs = (ctypes.c_void_p * len(polys))(*[p.ctypes.data for p in polys])
    qp = np.array([p for p, _ in case.queries], dtype=np.uint32)
    qx = np.stack([_w(x) for _, x in case.queries])
    v = _w(case.v)
    out = np.zeros((len(qp), 12), dtype=np.uint64)
    gg = np.ascontiguousarray(g)
    m = L.orc_gwc(ptrs, len(polys), case.n, qp.ctypes.data, qx.ctypes.data, len(qp), gg.ctypes.data, v.ctypes.data, threads(), out.ctypes.data)
    return out[:m]


def trapdoor_holds(oc, case, g, W, poly_override=None, eval_shift=0, continue_v=False, dedup=False):
    """(s - z_i) W_i == [sum_j v^j (p_ij(s) - p_ij(z_i))] G for every point z_i"""
    polys = list(case.polys)
    if poly_override is not None:
        polys[poly_override[0]] = poly_override[1]

    def ev(p, x):
        return ints(oc.fr_eval_polynomial(polys[p], _w(x)))[0]
    pts = case.points()
    if len(W) != len(pts):
        return False
    vj = 1
    for (z, ps), w in zip(pts, W):
        if dedup:
            ps = list(dict.fromkeys(ps))
        if not continue_v:
            vj = 1
        rhs = 0
        for p in ps:
            rhs = (rhs + vj * (ev(p, case.s) - (ev(p, z) + eval_shift))) % R
            vj = vj * case.v % R
        lhs = oc.g1_to_affine(oc.best_multiexp(np.stack([_w(case.s - z)]), np.stack([oc.g1_to_affine(w)])))
        want = oc.g1_to_affine(oc.best_multiexp(np.stack([_w(rhs)]), g[:1]))
        if not (lhs == want).all():
            return False
    return True


def same_points(oc, a, b):
    # the MSM's Jacobian coordinates depend on its accumulation order: compare the points
    return len(a) == len(b) and all((oc.g1_to_affine(x) == oc.g1_to_affine(y)).all() for x, y in zip(a, b))


def check_case(L, oc, k, name, seed, device_ptrs=False, device=0):
    import oracle_c
    case = Case(oracle_c, k, name, seed)
    g = srs(case)
    handle = L.register_bases(g)
    ptrs = ts.device_polys(L, case, device) if device_ptrs else None
    try:
        W = L.gwc_create_proof(device, case.polys, True, case.n, case.indexed(), handle, _w(case.v))
        assert len(W) == len(case.points())
        assert same_points(oc, W, orc_gwc(case, g)), (name, k)
        assert trapdoor_holds(oc, case, g, W), (name, k)
        if name == "constants":
            assert (W[:, 8:] == 0).all()                     # the identity: z = 0
        if device_ptrs:
            Wd = L.gwc_create_proof(device, ptrs, False, case.n, case.indexed(), handle, _w(case.v))
            assert same_points(oc, Wd, W)
    finally:
        for d in ptrs or []:
            L.dev_free(device, d)
        L.unregister_bases(handle)
    return case, g, W


# ---- CPU: the emulator -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k", list(zip(STRUCTURES, [3, 6, 5, 4, 4, 5, 5, 4, 3])))
def test_matches_oracle_and_trapdoor_emu(emu, oc, name, k):
    check_case(emu, oc, k, name, 900 + k)


def test_host_and_device_polynomials_agree_emu(emu, oc):
    check_case(emu, oc, 7, "lr22", 977, device_ptrs=True)


def test_trapdoor_check_has_teeth_emu(emu, oc):
    case, g, W = check_case(emu, oc, 4, "duplicates", 41)
    assert not trapdoor_holds(oc, case, g, W, poly_override=(1, case.polys[2]))
    assert not trapdoor_holds(oc, case, g, W, eval_shift=1)
    assert not trapdoor_holds(oc, case, g, W, continue_v=True)
    assert not trapdoor_holds(oc, case, g, W, dedup=True)


def check_batched_division(L, n, count, seed, device=0):
    """h2b_fr_kate_division_batch_dev equals `count` calls of h2b_fr_kate_division_dev bit for bit, in as many launches as one"""
    import oracle_c
    a = np.stack([oracle_c.random_fr(seed + i, n) for i in range(count)])
    pts = oracle_c.random_fr(seed + 999, count)
    d_a, d_p, d_q = L.dev_alloc(device, a.nbytes), L.dev_alloc(device, pts.nbytes), L.dev_alloc(device, a.nbytes)
    try:
        L.h2d(device, d_a, a)
        L.h2d(device, d_p, pts)
        L.dev_sync(device)
        before = L.launch_count()
        L.fr_kate_division_batch_dev(device, d_a, n, d_p, count, d_q)
        L.dev_sync(device)
        launches = L.launch_count() - before
        got = np.empty((count, n, 4), dtype=np.uint64)
        L.d2h(device, got, d_q)
        got = got[:, : n - 1]
        for i in range(count):
            before = L.launch_count()
            want = L.fr_kate_division(a[i], pts[i], device=device)
            assert L.launch_count() - before == launches, (n, count)
            assert (got[i] == want).all(), (n, count, i)
    finally:
        for d in (d_a, d_p, d_q):
            L.dev_free(device, d)


@pytest.mark.parametrize("n,count", [(2, 1), (2, 3), (17, 5), (100, 1), (256, 7), (4096, 3)])
def test_batched_kate_division_emu(emu, n, count):
    check_batched_division(emu, n, count, 10 * n + count)


def test_refusals_leave_outputs_untouched_emu(emu, oc):
    import oracle_c
    from halo2_scaffold_b200._lib import _queries
    case = Case(oracle_c, 3, "duplicates", 12)
    g = srs(case)
    h = emu.register_bases(g)
    short = emu.register_bases(g[: case.n - 2])
    exact = emu.register_bases(g[: case.n - 1])        # rows [0, n - 1) are all a quotient needs
    Lr = emu.L
    q = case.indexed()
    big = np.array([0xFFFFFFFFFFFFFFFF] * 4, dtype=np.uint64)
    polys = [np.ascontiguousarray(p) for p in case.polys]
    n_pts = len(case.points())
    try:
        def call(queries=q, n_polys=len(polys), n=case.n, handle=h, v=_w(case.v), capacity=n_pts, null=None):
            ptrs = (ctypes.c_void_p * len(polys))(*[p.ctypes.data for p in polys])
            out = np.full((max(capacity, 1), 12), 5, dtype=np.uint64)
            count = ctypes.c_uint32(77)
            args = [0, ptrs, 1, n_polys, n, _queries(queries), len(queries), handle, v.ctypes.data, out.ctypes.data, capacity, ctypes.byref(count)]
            if null is not None:
                args[null] = None
            rc = Lr.h2b_gwc_create_proof(*args)
            if rc != 0:
                assert (out == 5).all() and count.value == 77
            return rc
        assert call() == 0 and call(handle=exact) == 0
        assert call(queries=[(len(polys), q[0][1])] + q[1:]) == H2B_ERR_BAD_ARGUMENT           # poly index out of range
        assert call(queries=[(p, x) for p, x in q if p != 3]) == H2B_ERR_BAD_ARGUMENT            # a poly no query opens
        assert call(queries=[(0, big)] + q) == H2B_ERR_BAD_ARGUMENT                                # point >= r
        assert call(v=big) == H2B_ERR_BAD_ARGUMENT                                                 # v >= r
        assert call(queries=[]) == H2B_ERR_BAD_ARGUMENT                                            # no queries
        assert call(n=1) == H2B_ERR_BAD_ARGUMENT and call(n=(1 << 28) + 1) == H2B_ERR_BAD_ARGUMENT
        for null in (1, 8, 9, 11):                                                                 # polys, v, out, out_points
            assert call(null=null) == H2B_ERR_BAD_ARGUMENT
        assert call(handle=987654) == H2B_ERR_BAD_ARGUMENT and call(handle=short) == H2B_ERR_BAD_ARGUMENT
        assert call(capacity=n_pts - 1) == H2B_ERR_BAD_ARGUMENT
    finally:
        for hh in (h, short, exact):
            emu.unregister_bases(hh)


def test_python_prover_emu(emu, oc):
    """multiopen.ProverGWC: identity by object, one W per point"""
    import oracle_c
    from halo2_scaffold_b200 import kzg, multiopen
    case = Case(oracle_c, 4, "equal_contents", 8)
    g = srs(case)
    params = kzg.ParamsKZG(case.k, g, g, lib=emu)
    try:
        queries = [(case.polys[p], _w(x)) for p, x in case.queries]
        W = multiopen.ProverGWC(params).create_proof(queries, _w(case.v))
        assert same_points(oc, W, orc_gwc(case, g))
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
@pytest.mark.parametrize("n,count", [(2, 3), (17, 5), (1 << 16, 6), ((1 << 20) + 3, 3)])
def test_batched_kate_division(gpu, n, count):
    check_batched_division(gpu, n, count, 10 * n + count)


@pytest.mark.gpu
def test_memory_returns(gpu, oc):
    import oracle_c
    import torch
    case = Case(oracle_c, 16, "lr22", 16)
    g = srs(case)
    h = gpu.register_bases(g)
    try:
        W = gpu.gwc_create_proof(0, case.polys, True, case.n, case.indexed(), h, _w(case.v))   # the grow-only scratch reaches its size
        gpu.dev_sync(0)
        before = torch.cuda.mem_get_info(0)[0]
        W2 = gpu.gwc_create_proof(0, case.polys, True, case.n, case.indexed(), h, _w(case.v))
        gpu.dev_sync(0)
        after = torch.cuda.mem_get_info(0)[0]
        assert after >= before - (64 << 20), (before, after)
        assert same_points(oc, W, W2)
    finally:
        gpu.unregister_bases(h)


# ---- the C++ mirror ----------------------------------------------------------------------------------------------------------
def check_cpp_mirror(oc, lib_path, tmp_path, k):
    import subprocess
    import oracle_c
    from harness import build_mirror
    exe = build_mirror("gwc_mirror", lib_path, tmp_path)
    case = Case(oracle_c, k, "lr22", 70 + k)
    _w(case.s).tofile(str(tmp_path / "s.bin"))
    np.stack(case.polys).tofile(str(tmp_path / "polys.bin"))
    np.array([p for p, _ in case.queries], dtype=np.uint32).tofile(str(tmp_path / "qpoly.bin"))
    np.stack([_w(x) for _, x in case.queries]).tofile(str(tmp_path / "qpoint.bin"))
    _w(case.v).tofile(str(tmp_path / "v.bin"))
    out = subprocess.run([exe, str(tmp_path), str(k), str(case.P), str(len(case.queries))], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "GWC_MIRROR_OK" in out.stdout, out.stderr
    W = np.fromfile(str(tmp_path / "w.bin"), dtype=np.uint64).reshape(-1, 12)
    assert same_points(oc, W, orc_gwc(case, srs(case)))


def test_cpp_mirror_emu(emu, oc, tmp_path):
    check_cpp_mirror(oc, emu.path, tmp_path, 5)


@pytest.mark.gpu
def test_cpp_mirror(gpu, oc, tmp_path):
    check_cpp_mirror(oc, gpu.path, tmp_path, 12)
