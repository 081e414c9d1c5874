"""The proving key resident on the devices (h2b_pk_*, halo2_scaffold_b200.keygen.ResidentProvingKey).

Every form of every column a resident build stores -- read back with h2b_pk_download and as raw device memory through h2b_pk_column --
equals, bit for bit, the host outputs of h2b_keygen_fixed_build_pk, h2b_permutation_build_pk and h2b_keygen_lagrange_indicators_dev,
in the replicated and the row-sharded layout; a row-sharded device holds exactly rows (row0 - halo + t) mod E of each coset.
h2b_pk_put_lagrange of the same Lagrange values gives the same pk.  The toy circuit of the quotient check gets its whole pk from the
resident builders, and evaluate_h reading it through the handle gives the host path's h_ext, unsharded and row-sharded.

CPU: the kernel sources through the emulator on 1, 2 and 3 emulated devices.  GPU: the product library on every visible B200."""
import ctypes

import numpy as np
import pytest

import bn254 as o
from harness import Consts, disjoint, orc_mapping, random_copies, run_on_emulated_devices, sparse

H2B_ERR_BAD_ARGUMENT = -2
R = o.R_MOD
FIXED, PERMUTATION, INDICATORS = 0, 1, 2
VALUES, COEFF, EXTENDED = 0, 1, 2


# ---- inputs and the host reference -----------------------------------------------------------------------------------------
def inputs(L, oc, k, seed, shape):
    """random fixed columns, selectors through compress_selectors (overlapping or disjoint), a random mapping"""
    from halo2_scaffold_b200 import keygen as kg
    n = 1 << k
    rng = np.random.default_rng(seed)
    fixed = np.stack([oc.random_fr(seed * 13 + i, n) for i in range(2)])
    if shape == "overlapping":
        acts = sparse(rng, 4, n, 0.25)
        acts[:, 0] = True
        degrees, max_degree = [2, 2, 2, 2], 5
    else:
        acts = disjoint(6, n)
        degrees, max_degree = [3, 2, 3, 1, 2, 3], 5
    assignment = kg.compress_selectors(list(acts), degrees, max_degree, lib=L)
    P = 3
    mapping = orc_mapping(P, k, random_copies(rng, P, n, max(4, n // 4)))
    return fixed, acts, assignment, mapping


def host_reference(L, c, fixed, acts, assignment, mapping, bf=5):
    """(part, index) -> {form: array} from the existing host-output entry points"""
    C = assignment["n_combinations"]
    fx = L.keygen_fixed_build_pk(list(fixed), list(acts), assignment["combination_of"], assignment["root_of"], C, c.k, c.ek, c.omega_inv, c.ifft,
                                 c.ext_omega, c.zeta)
    pm = L.permutation_build_pk(mapping, c.k, c.ek, c.delta, c.omega, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
    ind = L.keygen_lagrange_indicators(c.k, c.ek, bf, c.omega_inv, c.ifft, c.ext_omega, c.zeta)
    ref = {}
    values = list(fixed) + fx["combination_values"]
    for i in range(len(values)):
        ref[(FIXED, i)] = {VALUES: values[i], COEFF: fx["polys"][i], EXTENDED: fx["cosets"][i]}
    for i in range(len(mapping)):
        ref[(PERMUTATION, i)] = {VALUES: pm["permutations"][i], COEFF: pm["polys"][i], EXTENDED: pm["cosets"][i]}
    for i in range(3):
        ref[(INDICATORS, i)] = {EXTENDED: ind[i]}
    return ref


def resident_build(L, c, fixed, acts, assignment, mapping, layout, halo, bf=5):
    from halo2_scaffold_b200 import keygen as kg
    F = len(fixed) + assignment["n_combinations"]
    pk = kg.ResidentProvingKey(c.dom, F, len(mapping), layout, halo, lib=L)
    pk.build_fixed(list(fixed), list(acts), assignment)
    pk.build_permutation(mapping)
    pk.build_indicators(bf)
    return pk


def raw_column(L, pk, device, part, form, index):
    """the column's device memory on `device`, copied out byte for byte"""
    ptr, (row0, rows, halo) = pk.column(part, form, index, device)
    out = np.empty((rows + 2 * halo, 4), dtype=np.uint64)
    L.d2h(device, out, ptr)
    return out, (row0, rows, halo)


def check_matches(L, c, pk, ref):
    """every form of every column, downloaded and read raw on every device, against the reference"""
    E = 1 << c.ek
    sharded = pk.layout == 1
    for (part, index), forms in ref.items():
        for form, want in forms.items():
            assert (pk.download(part, form, index) == want).all(), (part, index, form)
            for d in range(L.device_count()):
                got, (row0, rows, halo) = raw_column(L, pk, d, part, form, index)
                if form == EXTENDED and sharded:
                    assert rows == E * (d + 1) // L.device_count() - E * d // L.device_count() and row0 == E * d // L.device_count()
                    take = (row0 - halo + np.arange(rows + 2 * halo)) % E
                    assert (got == want[take]).all(), (part, index, form, d)
                else:
                    assert (row0, halo) == (0, 0) and (got == want).all(), (part, index, form, d)


def check_contents(L, oc, k, seed, layout, halo=0, shapes=("overlapping", "disjoint")):
    from halo2_scaffold_b200 import keygen as kg
    c = Consts(L, k)
    for shape in shapes:
        fixed, acts, assignment, mapping = inputs(L, oc, k, seed, shape)
        ref = host_reference(L, c, fixed, acts, assignment, mapping)
        with resident_build(L, c, fixed, acts, assignment, mapping, layout, halo) as pk:
            check_matches(L, c, pk, ref)
            # a ProvingKey built elsewhere: its Lagrange values registered give the same pk
            F = len(fixed) + assignment["n_combinations"]
            with kg.ResidentProvingKey(c.dom, F, len(mapping), layout, halo, lib=L) as pk2:
                pk2.put_lagrange("fixed", [ref[(FIXED, i)][VALUES] for i in range(1)])
                pk2.put_lagrange("fixed", [ref[(FIXED, i)][VALUES] for i in range(1, F)], first=1)
                pk2.put_lagrange("permutation", [ref[(PERMUTATION, i)][VALUES] for i in range(len(mapping))])
                pk2.build_indicators(5)
                check_matches(L, c, pk2, ref)
                assert pk2.info() == pk.info()


# ---- sizes -------------------------------------------------------------------------------------------------------------------
def check_info(L, k, F, P, halo):
    """bytes per device: 2n-row forms of F + P columns everywhere, extended columns whole or as the device's slice"""
    from halo2_scaffold_b200 import keygen as kg
    c = Consts(L, k)
    n, E, D = 1 << k, 1 << c.ek, L.device_count()
    with kg.ResidentProvingKey(c.dom, F, P, "replicated", lib=L) as pk:
        assert pk.info() == [32 * (2 * n * (F + P) + E * (F + P + 3))] * D
    with kg.ResidentProvingKey(c.dom, F, P, "row_sharded", halo, lib=L) as pk:
        rows = [E * (d + 1) // D - E * d // D for d in range(D)]
        assert pk.info() == [32 * (2 * n * (F + P) + (r + 2 * halo) * (F + P + 3)) for r in rows]


# ---- refusals and lifetime ---------------------------------------------------------------------------------------------------------
def check_refused(L, oc, k=4):
    from halo2_scaffold_b200 import keygen as kg
    c = Consts(L, k)
    n, E, D = c.n, 1 << c.ek, L.device_count()
    Lr = L.L
    vp = ctypes.c_void_p
    w = lambda x: x.ctypes.data
    consts = [w(c.omega), w(c.omega_inv), w(c.ifft), w(c.ext_omega), w(c.zeta)]
    h = ctypes.c_uint64(0)
    # create: k, extended_k, layout, null constants, a halo that does not fit
    rows_max = max(E * (d + 1) // D - E * d // D for d in range(D))
    for args in [(29, 29, 0, 0), (k, k - 1, 0, 0), (k, 29, 0, 0), (k, c.ek, 2, 0), (k, c.ek, 1, (E - rows_max) // 2 + 1)]:
        kk, ek, layout, halo = args
        assert Lr.h2b_pk_create(kk, ek, 2, 2, layout, halo, *consts, ctypes.byref(h)) == H2B_ERR_BAD_ARGUMENT, args
    for i in range(5):
        bad = list(consts)
        bad[i] = None
        assert Lr.h2b_pk_create(k, c.ek, 2, 2, 0, 0, *bad, ctypes.byref(h)) == H2B_ERR_BAD_ARGUMENT
    assert Lr.h2b_pk_create(k, c.ek, 2, 2, 1, (E - rows_max) // 2, *consts, ctypes.byref(h)) == 0      # the largest halo that fits
    assert Lr.h2b_pk_release(h.value) == 0

    fixed, acts, assignment, mapping = inputs(L, oc, k, 77, "disjoint")
    F, P = len(fixed) + assignment["n_combinations"], len(mapping)
    pk = resident_build(L, c, fixed, acts, assignment, mapping, "replicated", 0)
    before = {(p, i, f): pk.download(p, f, i) for p, cnt in ((FIXED, F), (PERMUTATION, P)) for i in range(cnt) for f in (VALUES, COEFF, EXTENDED)}
    ptr = vp(0)
    co, ro = assignment["combination_of"], assignment["root_of"]
    arr = lambda xs: (vp * len(xs))(*[x.ctypes.data if x is not None else None for x in xs])
    acts8 = [np.ascontiguousarray(a, dtype=np.uint8) for a in acts]
    try:
        # reading: wrong part / form / index / device, and a column never filled
        for part, form, index, dev in [(3, 0, 0, 0), (-1, 0, 0, 0), (0, 3, 0, 0), (INDICATORS, VALUES, 0, 0), (INDICATORS, COEFF, 0, 0), (FIXED, 0, F, 0),
                                       (PERMUTATION, 0, P, 0), (INDICATORS, EXTENDED, 3, 0), (FIXED, 0, 0, D), (FIXED, 0, 0, -1)]:
            assert Lr.h2b_pk_column(pk.handle, dev, part, form, index, ctypes.byref(ptr), None) == H2B_ERR_BAD_ARGUMENT, (part, form, index, dev)
            out = np.zeros((E, 4), dtype=np.uint64)
            if dev == 0:
                assert Lr.h2b_pk_download(pk.handle, part, form, index, out.ctypes.data) == H2B_ERR_BAD_ARGUMENT and not out.any()
        with kg.ResidentProvingKey(c.dom, 1, 1, lib=L) as empty:
            for part, form in ((FIXED, VALUES), (PERMUTATION, EXTENDED), (INDICATORS, EXTENDED)):
                assert Lr.h2b_pk_column(empty.handle, 0, part, form, 0, ctypes.byref(ptr), None) == H2B_ERR_BAD_ARGUMENT
        # builds that are refused write nothing: a bad mapping entry, two members of one combination on one row, columns past the part
        bad_map = mapping.copy()
        bad_map[1, 3] = (P, 0)
        assert Lr.h2b_permutation_build_pk_resident(arr(list(bad_map)), P, w(c.delta), pk.handle) == H2B_ERR_BAD_ARGUMENT
        bad_map = mapping.copy()
        bad_map[2, n - 1] = (0, n)
        assert Lr.h2b_permutation_build_pk_resident(arr(list(bad_map)), P, w(c.delta), pk.handle) == H2B_ERR_BAD_ARGUMENT
        assert Lr.h2b_permutation_build_pk_resident(arr(list(mapping[:2])), 2, w(c.delta), pk.handle) == H2B_ERR_BAD_ARGUMENT
        overlapping = [a.copy() for a in acts8]
        m0 = [s for s in range(len(acts8)) if co[s] == co[0]]
        assert len(m0) >= 2
        overlapping[m0[1]][np.flatnonzero(acts8[m0[0]])[0]] = 1
        fx = [np.ascontiguousarray(x) for x in fixed]
        C = assignment["n_combinations"]
        assert Lr.h2b_keygen_fixed_build_pk_resident(arr(fx), len(fx), arr(overlapping), len(acts8), w(co), w(ro), C, pk.handle, 0) == H2B_ERR_BAD_ARGUMENT
        assert Lr.h2b_keygen_fixed_build_pk_resident(arr(fx), len(fx), arr(acts8), len(acts8), w(co), w(ro), C, pk.handle, 1) == H2B_ERR_BAD_ARGUMENT
        assert Lr.h2b_keygen_lagrange_indicators_resident(pk.handle, n - 1) == H2B_ERR_BAD_ARGUMENT
        junk = [oc.random_fr(5, n)]
        for part, first in ((INDICATORS, 0), (3, 0), (FIXED, F), (PERMUTATION, P)):
            assert Lr.h2b_pk_put_lagrange(pk.handle, part, first, 1, arr(junk)) == H2B_ERR_BAD_ARGUMENT
        assert Lr.h2b_pk_put_lagrange(pk.handle, FIXED, 0, 1, arr([None])) == H2B_ERR_BAD_ARGUMENT
        for key, want in before.items():
            p, i, f = key
            assert (pk.download(p, f, i) == want).all(), key
        # unknown handles
        for fn in (lambda hh: Lr.h2b_pk_info(hh, None), lambda hh: Lr.h2b_keygen_lagrange_indicators_resident(hh, 5),
                   lambda hh: Lr.h2b_pk_column(hh, 0, 0, 0, 0, ctypes.byref(ptr), None)):
            assert fn(0xFFFFFFF0) == H2B_ERR_BAD_ARGUMENT
    finally:
        handle = pk.handle
        pk.close()
    # after release: every call on the handle fails, and so does a second release
    assert Lr.h2b_pk_info(handle, None) == H2B_ERR_BAD_ARGUMENT
    assert Lr.h2b_pk_column(handle, 0, 0, 0, 0, ctypes.byref(ptr), None) == H2B_ERR_BAD_ARGUMENT
    assert Lr.h2b_pk_release(handle) == H2B_ERR_BAD_ARGUMENT


# ---- the toy circuit of the quotient check, with its pk from the resident builders ------------------------------------------------
def quotient_pin(L, oc, k=5, seed=1, layout="replicated", wrong_mapping=False):
    """-> (top quarter of the quotient is zero, h_ext through the pk, h_ext of the host path).  As
    parity_cases.check_quotient_is_a_polynomial: one multiplication gate q (a b - c), copies a[i+1] = c[i] in two permutation sets and
    one lookup, but q comes from compress_selectors, the table is a fixed column, sigma is built from a mapping of the copies and the
    indicators come from build_indicators; evaluate_h reads all of them through the handle."""
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import evaluation as ev, keygen as kg, prover
    from halo2_scaffold_b200.domain import fr_to_words
    rng = np.random.default_rng(seed)
    n, bf = 1 << k, 5
    u = n - (bf + 1)
    dom = h2.EvaluationDomain(4, k, lib=L)
    en, rot_scale = 1 << dom.extended_k, 1 << (dom.extended_k - k)
    W = lambda vals: np.stack([fr_to_words(int(v)) for v in vals])
    rnd = lambda: int(rng.integers(1, 1 << 62)) * int(rng.integers(1, 1 << 62)) % R
    DELTA = kg.FR_DELTA
    table = [int(v) for v in rng.integers(0, 50, size=n)]
    q = [1 if (i < u and i % 2 == 0) else 0 for i in range(n)]
    a, b, c = ([rnd() for _ in range(n)] for _ in range(3))
    lk = [table[int(rng.integers(0, u))] for _ in range(n)]
    mapping = np.zeros((3, n, 2), dtype=np.uint64)
    mapping[:, :, 0] = np.arange(3)[:, None]
    mapping[:, :, 1] = np.arange(n)[None, :]
    for i in range(0, u - 1, 2):
        c[i] = a[i] * b[i] % R
        a[i + 1] = c[i]
        mapping[0, i + 1], mapping[2, i] = (2, i), (0, i + 1)
    sigma = [[pow(DELTA, int(mapping[j, i, 0]), R) * pow(dom.omega, int(mapping[j, i, 1]), R) % R for i in range(n)] for j in range(3)]
    beta, gamma, theta, y = (rnd() for _ in range(4))
    blind = lambda count: W([rnd() for _ in range(count)])
    ints = lambda wds: [o.from_mont(v, R) for v in oc.words_to_ints(np.ascontiguousarray(wds))]
    zs, _ = prover.permutation_commit([W(cc) for cc in (a, b, c)], [W(sg) for sg in sigma], chunk_len=2, blinding_factors=bf, beta=fr_to_words(beta),
                                      gamma=fr_to_words(gamma), omega=fr_to_words(dom.omega), blind=blind, lib=L)
    z_cols = [ints(z) for z in zs]
    assert z_cols[-1][u] == 1
    pa, pt, _ = prover.lookup_commit_permuted(W(lk), W(table), blinding_factors=bf, blind=blind, lib=L)
    zl, _ = prover.lookup_commit_product(W(lk), W(table), pa, pt, blinding_factors=bf, beta=fr_to_words(beta), gamma=fr_to_words(gamma), blind=blind,
                                         lib=L)
    ext = lambda vals: dom.coeff_to_extended(dom.lagrange_to_coeff(W(vals)))
    ext_w = lambda wds: dom.coeff_to_extended(dom.lagrange_to_coeff(np.ascontiguousarray(wds)))
    E = ev.Evaluator([ev.Product(ev.Fixed(0), ev.Sum(ev.Product(ev.Advice(0), ev.Advice(1)), ev.Negated(ev.Advice(2))))],
                     [([ev.Advice(3)], [ev.Fixed(1)])])
    perm = dict(product_cosets=[ext(z) for z in z_cols], columns=[("advice", 0), ("advice", 1), ("advice", 2)], chunk_len=2, last_rotation=-(bf + 1),
                delta=fr_to_words(DELTA), zeta=fr_to_words(dom.g_coset), extended_omega=fr_to_words(dom.extended_omega))
    common = dict(size=en, rot_scale=rot_scale, advice=[ext(a), ext(b), ext(c), ext(lk)], instance=[], challenges=np.zeros((0, 4), dtype=np.uint64),
                  y=fr_to_words(y), beta=fr_to_words(beta), gamma=fr_to_words(gamma), theta=fr_to_words(theta),
                  lookups=[dict(product_coset=ext_w(zl), permuted_input_coset=ext_w(pa), permuted_table_coset=ext_w(pt))], lib=L)
    l0, l_last, l_active = [1] + [0] * (n - 1), [1 if i == u else 0 for i in range(n)], [1 if i < u else 0 for i in range(n)]
    h_host = E.evaluate_h(fixed=[ext(q), ext(table)], l0=ext(l0), l_last=ext(l_last), l_active_row=ext(l_active),
                          permutation=dict(perm, cosets=[ext(s) for s in sigma]), **common)
    # the pk: q through compress_selectors into fixed column 0, the table as fixed column 1, sigma from the mapping, the indicators
    halo = 6 * rot_scale                               # the largest rotated read: |last_rotation| rows of the permutation argument
    assignment = kg.compress_selectors([np.array(q, dtype=bool)], [3], 4, lib=L)
    with kg.ResidentProvingKey(dom, 2, 3, layout, halo if layout == "row_sharded" else 0, lib=L) as pk:
        pk.build_fixed([], [np.array(q, dtype=bool)], assignment, first_column=0)
        pk.build_fixed([W(table)], [], dict(combination_of=[], root_of=[], n_combinations=0), first_column=1)
        pk.build_permutation(mapping[[1, 0, 2]] if wrong_mapping else mapping)
        pk.build_indicators(bf)
        if layout == "replicated":
            h_pk = E.evaluate_h(permutation=perm, pk=pk, **common)
        else:
            parts = []
            for d in range(L.device_count()):
                parts.append(E.evaluate_h(permutation=perm, pk=pk, device=d, **common))
            h_pk = np.concatenate(parts)
    quotient = dom.divide_by_vanishing_poly(h_pk)
    coeffs = L.ntt(np.ascontiguousarray(quotient), fr_to_words(dom.extended_omega_inv), dom.extended_k)
    return not coeffs[3 * n:].any(), h_pk, h_host


def check_pin(L, oc, k, seed, layouts=("replicated", "row_sharded")):
    for layout in layouts:
        ok, h_pk, h_host = quotient_pin(L, oc, k, seed, layout)
        assert ok and (h_pk == h_host).all(), layout
    ok, h_pk, h_host = quotient_pin(L, oc, k, seed, "replicated", wrong_mapping=True)
    assert not ok, "a pk with sigma from a wrong mapping must break the pin"


# ---- CPU: the kernel sources through the emulator ----------------------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 5, 8])
def test_contents_match_host_keygen_emu(emu, oc, k):
    check_contents(emu, oc, k, 700 + k, "replicated")
    check_contents(emu, oc, k, 710 + k, "row_sharded", 0, shapes=("disjoint",))


def test_info_emu(emu):
    check_info(emu, 5, 3, 2, 0)


def test_refuses_bad_input_emu(emu, oc):
    check_refused(emu, oc)


def test_quotient_pin_emu(emu, oc):
    check_pin(emu, oc, 5, 720, layouts=("replicated",))


@pytest.mark.parametrize("devices", ["2", "3"])
def test_resident_pk_on_emulated_devices(emu, devices):
    # 2 devices: the slices wrap at the start (device 0) and at the end (device 1); 3 devices: D does not divide E
    run_on_emulated_devices("test_resident_pk", "oc.build()\n"
                                                "t.check_contents(L, oc, 4, 730, 'row_sharded', 5)\n"
                                                "t.check_contents(L, oc, 3, 731, 'row_sharded', 3, shapes=('overlapping',))\n"
                                                "t.check_contents(L, oc, 4, 732, 'replicated', shapes=('disjoint',))\n"
                                                "t.check_info(L, 4, 3, 2, 7)\n"
                                                "t.check_refused(L, oc)\n"
                                                "t.check_pin(L, oc, 5, 733)", devices)


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _layouts(L):
    return ("replicated", "row_sharded") if L.device_count() > 1 else ("replicated",)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 12, 16])
def test_contents_match_host_keygen(gpu, oc, k):
    check_contents(gpu, oc, k, 800 + k, "replicated")
    # one device: the sharded layout holds the whole coset (a halo cannot fit), still through the slice path
    check_contents(gpu, oc, k, 810 + k, "row_sharded", 0 if gpu.device_count() == 1 else 1 << 4, shapes=("disjoint",))


@pytest.mark.gpu
def test_contents_match_host_keygen_k20(gpu, oc):
    check_contents(gpu, oc, 20, 820, "replicated", shapes=("disjoint",))


@pytest.mark.gpu
def test_info_and_refusals(gpu, oc):
    check_info(gpu, 10, 3, 2, 0 if gpu.device_count() == 1 else 64)
    check_refused(gpu, oc)
    check_refused(gpu, oc, k=12)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 12])
def test_quotient_pin(gpu, oc, k):
    check_pin(gpu, oc, k, 830 + k, layouts=_layouts(gpu))


@pytest.mark.gpu
def test_device_memory_returns_after_release(gpu):
    """cudaMemGetInfo on every device: back to its value before create after release (the pk reserves its storage at create)"""
    from halo2_scaffold_b200 import keygen as kg
    import torch

    def free_bytes():
        return [torch.cuda.mem_get_info(d)[0] for d in range(gpu.device_count())]
    c = Consts(gpu, 20)
    slack = 64 << 20
    before = free_bytes()
    pk = kg.ResidentProvingKey(c.dom, 6, 6, lib=gpu)
    held = pk.info()
    during = free_bytes()
    assert all(b - d >= h - slack for b, d, h in zip(before, during, held)), (before, during, held)
    pk.close()
    after = free_bytes()
    assert all(a >= b - slack for a, b in zip(after, before)), (before, after)

