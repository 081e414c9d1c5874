"""MockProver::verify's gate, lookup and permutation loops on the device (h2b_mock_verify, halo2_scaffold_b200.mock) against
tests/cpp/mock_verify_oracle.cpp, which restates upstream's three loops over the expression trees with the Value enum and
evaluate_lazy -- not through a GraphEvaluator.

Every case compares the failures of mock.verify (upstream's order, lookups re-sorted by tuple) with the oracle's, and the raw
records of the C ABI (lookups by row) with the oracle's in that order.  CPU: the kernel sources through the emulator at k = 3 .. 8.
GPU: the product library at k = 10, 14, 16 and a halo2-lib-like circuit at k = 20."""
import numpy as np
import pytest

import mock_cases as mc
from halo2_scaffold_b200 import _lib
from halo2_scaffold_b200.evaluation import ADVICE, Advice, Evaluator, Fixed, Product, Sum

H2B_ERR_BAD_ARGUMENT = -2


def check(L, c, capacity=1024):
    """mock.verify and the raw records against the oracle -> the number of failures"""
    total, recs = c.oracle()
    assert c.device(L, capacity=capacity) == mc.as_failures(recs)
    count, raw = c.device_raw(L, capacity=max(total, 1))
    assert count == total
    assert [tuple(r) for r in raw.tolist()] == mc.device_order(recs)
    return total


# ---- faults injected into a satisfied circuit --------------------------------------------------------------------------------
def fault(c, name, rng):
    n, u, ix = c.n, c.usable, c.ix
    if name == "corrupt_advice":                 # one cell read by the gate at rotations 0..3 of four rows
        r = 4 * int(rng.integers(max(u // 4 - 1, 1))) + 2
        c.advice[ix["a"]][r] = mc.random_words(rng, 1)[0]
    elif name == "poisoned_read":                # an enabled selector whose rotations reach the blinding rows, and a zero one
        c.fixed[ix["q"]][u - 2] = mc.words([1])[0]
        c.fixed[ix["q"]][u - 1] = mc.words([0])[0]
    elif name == "lookup_missing":               # inputs outside the table, one of them twice, and one row at a zero selector
        rows = [r for r in range(u) if c.fixed[ix["ql"]][r].any()][:3]
        vals = [ix["T"] + 9, ix["T"] + 3, ix["T"] + 9]
        for r, v in zip(rows, vals):
            c.advice[ix["x"]][r] = mc.words([v])[0]
        c.advice[ix["x"]][next(r for r in range(u) if not c.fixed[ix["ql"]][r].any())] = mc.words([ix["T"] + 1])[0]
    elif name == "lookup_m3_missing":
        for j, r in enumerate((1, 3, 3)):
            c.advice[ix["m3_inputs"][j]][r] = mc.random_words(rng, 1)[0]
    elif name == "lookup_blinding":              # an input reaching a blinding row through a rotation: Poison, absent from the table
        c.lookups.append(([Advice(ix["x"], 1)], [Fixed(ix["t"])]))
    elif name == "lookup_fill_poison":           # fill_row is Poison here, so the Poison input at the last usable row is skipped
        c.lookups.append(([Advice(ix["x"], 1)], [Advice(ix["x"], 1)]))
    elif name == "unassigned_copy":              # Unassigned copied to Assigned(0)
        e, f = ix["e"], ix["f"]
        r1 = next(r for r in range(u) if int(c.mapping[1][r][0]) == 1 and int(c.mapping[1][r][1]) == r)
        r2 = next(r for r in range(u) if int(c.mapping[2][r][0]) == 2 and int(c.mapping[2][r][1]) == r)
        c.advice_assigned[e][r1] = False
        c.fixed[f][r2] = 0
        c.mapping[1][r1] = (2, r2)
        c.mapping[2][r2] = (1, r1)
    elif name == "copy_mismatch":                # one cell of a copy cycle changed
        x, y = next((cc, r) for cc in (1, 2, 3) for r in range(u) if (int(c.mapping[cc][r][0]), int(c.mapping[cc][r][1])) != (cc, r))
        kind, idx = c.permutation[x]
        c.cols(kind)[idx][y] = mc.random_words(rng, 1)[0]
    elif name == "copy_blinding":                # Poison(i) == Poison(j) only for i = j
        c.mapping[0][u], c.mapping[0][u + 1] = (0, u + 1), (0, u)
    else:
        raise KeyError(name)
    return c


FAULTS = ["corrupt_advice", "poisoned_read", "lookup_missing", "lookup_m3_missing", "lookup_blinding", "lookup_fill_poison", "unassigned_copy",
          "copy_mismatch", "copy_blinding"]


def faulted(k, name, seed):
    rng = np.random.default_rng(seed)
    return fault(mc.halo2_lib(k, seed, m3=name == "lookup_m3_missing"), name, rng)


def many_failures(k, seed):
    """a circuit that fails everywhere: every gate, lookup and copy kind"""
    c = mc.halo2_lib(k, seed, m3=True)
    rng = np.random.default_rng(seed + 1)
    for name in ("lookup_missing", "lookup_blinding", "unassigned_copy", "copy_blinding"):
        fault(c, name, rng)
    c.advice[c.ix["a"]][:] = mc.random_words(rng, c.n)
    return c


# ---- CPU: the kernel sources through the emulator ------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 4, 5, 6, 7, 8])
def test_satisfied_circuits_emu(emu, k):
    c = mc.halo2_lib(k, 10 + k, bf=2 if k == 3 else 5, m3=k >= 6)
    assert check(emu, c) == 0


@pytest.mark.parametrize("name", FAULTS)
def test_faults_emu(emu, name):
    assert (check(emu, faulted(6, name, 31)) > 0) == (name != "lookup_fill_poison")


def test_poison_algebra_emu(emu):
    """Scaled, Product with a zero side on either side, x + 0, x * 1, x * 2, x * x, -x, x - x, x * 0, Poison * Poison, each read one or
    two rows ahead so that the last usable rows read Poison"""
    c = mc.poison_algebra(6, 5)
    failures = c.device(emu)
    assert check(emu, c) > 0
    poisoned = {f[1] for f in failures if f[0] == "ConstraintPoisoned"}
    assert {0, 2, 3, 4, 5, 6, 7, 8, 9, 11}.issubset(poisoned)
    assert not {1, 10} & poisoned                  # Scaled(x, 0) and x * 0 are Real(0)


def test_poisoned_rows_merge_into_one_failure_emu(emu):
    """a polynomial poisoned on several blinding rows is one ConstraintPoisoned (upstream's dedup), while the C ABI reports every row"""
    c = mc.poison_algebra(6, 5)
    c.gates = [c.gates[0]]                         # Scaled(advice[r + 1], 5): Poison from row usable - 1 to row n - 2
    count, raw = c.device_raw(emu, capacity=64)
    assert count == c.n - c.usable and {tuple(r[:3]) for r in raw.tolist()} == {(1, 0, 0)}
    assert c.device(emu) == [("ConstraintPoisoned", 0, 0)]


@pytest.mark.parametrize("parts", ["no_gates", "no_lookups", "no_permutation", "nothing"])
def test_missing_parts_emu(emu, parts):
    c = many_failures(5, 3)
    if parts in ("no_gates", "nothing"):
        c.gates = []
    if parts in ("no_lookups", "nothing"):
        c.lookups = []
    if parts in ("no_permutation", "nothing"):
        c.permutation, c.mapping = [], []
    total = check(emu, c)
    assert (total == 0) == (parts == "nothing")


def test_capacity_emu(emu):
    c = many_failures(6, 8)
    total, recs = c.oracle()
    order = mc.device_order(recs)
    assert total > 20
    for cap in (0, 1, 7, total - 1, total, total + 5):
        count, raw = c.device_raw(emu, capacity=cap)
        assert count == total
        assert [tuple(r) for r in raw.tolist()] == order[:min(cap, total)]
    assert c.device(emu, capacity=3) == mc.as_failures(recs)      # mock.verify asks again with room for all


def test_refusals_emu(emu):
    c = mc.halo2_lib(5, 4, m3=True)

    def refused(hook=None, capacity=16, **edit):
        args = list(c.raw_args())
        names = ["k", "bf", "fixed", "fa", "advice", "aa", "instance", "ch", "graph", "roots", "lookups", "perm", "mapping"]
        for key, v in edit.items():
            args[names.index(key)] = v
        with pytest.raises(_lib.H2BError) as e:
            emu.mock_verify(0, *args, capacity=capacity, circuit_hook=hook)
        assert e.value.code == H2B_ERR_BAD_ARGUMENT, e.value

    def set_field(name, value):
        return lambda s: setattr(s, name, value)

    refused(set_field("k", 0))
    refused(set_field("k", 29))
    refused(set_field("blinding_factors", 31))
    refused(set_field("fixed", None))
    refused(set_field("advice_assigned", None))
    refused(set_field("roots", None))
    refused(set_field("mapping", None))
    refused(set_field("n_fixed", 0))                                     # the gates read fixed columns that are not there
    refused(set_field("n_advice", 1))
    refused(perm=[(ADVICE, 99)] + c.raw_args()[11][1:])
    refused(perm=[(0, 0)] + c.raw_args()[11][1:])                          # a constant is no column
    graph, roots = c.raw_args()[8], c.raw_args()[9]
    refused(roots=list(reversed(roots)) + [(0, 0, roots[0][2])])         # out of gate order
    refused(roots=roots + [(9, 0, (1, 10_000, 0))])                      # an intermediate no calculation wrote
    refused(roots=roots + [(9, 0, (0, 10_000, 0))])                      # a constant out of range
    refused(roots=roots + [(9, 0, (5, 0, 0))])                           # no challenges
    lk = c.raw_args()[10]
    g0, ins, tbs = lk[0]
    refused(lookups=[(g0, [], [])])
    refused(lookups=[(g0, ins * 17, tbs * 17)])
    bad_map = [m.copy() for m in c.mapping]
    bad_map[2][3] = (len(c.permutation), 0)
    refused(mapping=bad_map)
    bad_map[2][3] = (0, c.n)
    refused(mapping=bad_map)
    # a graph that keeps more than 64 values live, and one with more rotations than the interpreter indexes
    deep = Product(Fixed(0), Advice(0))
    for i in range(1, 70):
        deep = Sum(Product(Fixed(0, i), Advice(0, i)), deep)
    from halo2_scaffold_b200 import mock
    g, r = mock.compile_gates([[deep]])
    refused(graph=g, roots=r)
    g, r = mock.compile_gates([[Advice(0, i)] for i in range(1100)])
    refused(graph=g, roots=r)
    # null records with a non-zero capacity and a null count
    with pytest.raises(_lib.H2BError):
        import ctypes
        emu.check(emu.L.h2b_mock_verify(0, None, None, 0, ctypes.byref(ctypes.c_uint64())))
    c.device_raw(emu, capacity=4)                                        # the circuit itself is fine


# evaluate_h's graphs compile as they did before the compiler took roots: (slots, micro-operations) of the custom-gate graph and
# of each lookup graph, as the compiler without roots gave them; the evaluate_h parity tests pin their values
def _evaluators():
    a, b, c_, q = Advice(0), Advice(0, 1), Advice(0, 2), Fixed(0)
    gate = Product(q, Sum(Sum(a, Product(b, c_)), Product(Fixed(1), Advice(0, 3))))
    plonk = Sum(Sum(Product(Fixed(2), a), Product(Fixed(3), Advice(1))), Product(Fixed(4), Product(a, Advice(1))))
    return [Evaluator([gate]), Evaluator([gate, plonk], [([Product(q, a)], [Fixed(5)]), ([a, b, Advice(1)], [Fixed(5), Fixed(6), Fixed(7)])])]


EXISTING_STREAMS = [(2, 6), (3, 13), (2, 6), (2, 9)]


def test_existing_graphs_compile_unchanged_emu(emu):
    import halo2_scaffold_b200.evaluation as ev
    got = []
    n = 16
    zero = np.zeros((n, 4), dtype=np.uint64)
    w = np.zeros(4, dtype=np.uint64)
    for e in _evaluators():
        for graph in [e.custom_gates] + e.lookups:
            ev.evaluate_graph(emu, graph.arrays(), [zero] * 8, [zero] * 2, [], [], w, w, w, w, zero, 1)
            got.append(emu.evaluate_graph_info())
    assert got == EXISTING_STREAMS


# ---- GPU: the product library ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 14, 16])
def test_matches_oracle(gpu, k):
    assert check(gpu, mc.halo2_lib(k, 100 + k, m3=True)) == 0
    for name in FAULTS:
        assert (check(gpu, faulted(k, name, 200 + k)) > 0) == (name != "lookup_fill_poison"), name
    assert check(gpu, mc.poison_algebra(k, 7)) > 0
    c = many_failures(k, 300 + k)
    total, recs = c.oracle()
    order = mc.device_order(recs)
    for cap in (0, 5, total - 1, total):
        count, raw = c.device_raw(gpu, capacity=cap)
        assert count == total and [tuple(r) for r in raw.tolist()] == order[:cap]


@pytest.mark.gpu
def test_halo2_lib_k20(gpu):
    assert check(gpu, mc.halo2_lib(20, 20)) == 0
    assert check(gpu, faulted(20, "corrupt_advice", 21)) > 0
