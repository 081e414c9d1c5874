"""Circuits for the MockProver::verify tests (tests/test_mock_verify.py, tools/mock_verify_bench.py): seeded random witnesses that
satisfy a standard-plonk gate, halo2-lib's q * (a + b c - d) gate over rotations 0..3, a range lookup, an m = 3 lookup and copy
constraints across fixed, advice and instance columns, plus the faults the tests inject into them.  The reference is
tests/cpp/mock_verify_oracle.cpp, which evaluates the same expression trees with upstream's Value arithmetic."""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bn254 as o  # noqa: E402
from halo2_scaffold_b200 import _lib  # noqa: E402
from halo2_scaffold_b200 import mock  # noqa: E402
from halo2_scaffold_b200.evaluation import (ADVICE, FIXED, INSTANCE, Advice, Challenge, Constant, Fixed, Instance, Negated,  # noqa: E402
                                            Product, Scaled, Sum)

R = o.R_MOD
KIND = {"fixed": FIXED, "advice": ADVICE, "instance": INSTANCE}


def words(vals):
    """canonical integers -> Montgomery words"""
    import oracle_c as oc
    v = np.asarray(vals)
    if v.dtype.kind in "iu" and (v.size == 0 or (v.min() >= 0 and v.max() < 1 << 62)):
        w = np.zeros((v.size, 4), dtype=np.uint64)
        w[:, 0] = v.reshape(-1)
        return oc.fr_to_mont(w)
    return oc.fr_to_mont(oc.ints_to_words([int(x) % R for x in vals]))


def random_words(rng, n):
    """n uniformly random field elements (Montgomery words), any 256-bit pattern below 2^253 < r"""
    w = rng.integers(0, 1 << 63, size=(n, 4), dtype=np.uint64, endpoint=False)
    w[:, 3] &= np.uint64((1 << 61) - 1)
    return w


def fmul(a, b):
    import oracle_c as oc
    return oc.field_op("fr", "mul", a, b)


def fadd(a, b):
    import oracle_c as oc
    return oc.field_op("fr", "add", a, b)


class Circuit:
    """What MockProver holds after `run`, as host arrays: columns (Montgomery words), assigned flags, gates, lookups, permutation"""

    def __init__(self, k, bf=5):
        self.k, self.bf, self.n = k, bf, 1 << k
        self.usable = self.n - (bf + 1)
        self.fixed, self.fixed_assigned, self.advice, self.advice_assigned, self.instance = [], [], [], [], []
        self.challenges = np.zeros((0, 4), dtype=np.uint64)
        self.gates, self.lookups, self.permutation, self.copies = [], [], [], []
        self.mapping = None
        self.ix = {}            # column names of the builders -> index

    def column(self, kind, vals=None, assigned=None):
        vals = np.zeros((self.n, 4), dtype=np.uint64) if vals is None else np.ascontiguousarray(vals, dtype=np.uint64).reshape(self.n, 4)
        if kind == "instance":
            self.instance.append(vals)
            return len(self.instance) - 1
        assigned = np.ones(self.n, dtype=bool) if assigned is None else np.asarray(assigned, dtype=bool)
        if kind == "advice":
            assigned = assigned.copy()
            assigned[self.usable:] = False
            self.advice.append(vals)
            self.advice_assigned.append(assigned)
            return len(self.advice) - 1
        self.fixed.append(vals)
        self.fixed_assigned.append(assigned)
        return len(self.fixed) - 1

    def cols(self, kind):
        return {"fixed": self.fixed, "advice": self.advice, "instance": self.instance}[kind]

    def finish_permutation(self):
        """the mapping of upstream's Assembly after self.copies, and every cycle's cells made equal to its first cell"""
        from harness import orc_mapping
        P = len(self.permutation)
        if P == 0:
            self.mapping = []
            return
        self.mapping = orc_mapping(P, self.k, self.copies) if self.copies else np.stack(
            [np.stack([np.full(self.n, c, dtype=np.uint64), np.arange(self.n, dtype=np.uint64)], axis=1) for c in range(P)])
        seen = np.zeros((P, self.n), dtype=bool)
        for c in range(P):
            for r in range(self.n):
                if seen[c, r]:
                    continue
                cyc, (x, y) = [], (c, r)
                while not seen[x, y]:
                    seen[x, y] = True
                    cyc.append((x, y))
                    x, y = (int(v) for v in self.mapping[x][y])
                if len(cyc) < 2:
                    continue
                # an instance cell fixes the value; every other cell takes it and is assigned
                src = next((q for q in cyc if self.permutation[q[0]][0] == "instance"), cyc[0])
                kind, idx = self.permutation[src[0]]
                v = self.cols(kind)[idx][src[1]].copy()
                for x, y in cyc:
                    kd, ix = self.permutation[x]
                    self.cols(kd)[ix][y] = v
                    if kd == "fixed":
                        self.fixed_assigned[ix][y] = True
                    elif kd == "advice":
                        self.advice_assigned[ix][y] = True

    # ---- the two entry points and the oracle ------------------------------------------------------------------------------
    def raw_args(self):
        graph, roots = mock.compile_gates(self.gates)
        lks = [mock.compile_lookup(i, t) for i, t in self.lookups]
        return (self.k, self.bf, self.fixed, [mock.bitmap(a) for a in self.fixed_assigned], self.advice, [mock.bitmap(a) for a in self.advice_assigned],
                self.instance, self.challenges, graph, roots, lks, [(KIND[kd], ix) for kd, ix in self.permutation], list(self.mapping))

    def device_raw(self, L, capacity, device=0, hook=None):
        return L.mock_verify(device, *self.raw_args(), capacity=capacity, circuit_hook=hook)

    def device(self, L, device=0, capacity=1024):
        return mock.verify(self.k, self.bf, fixed=self.fixed, fixed_assigned=self.fixed_assigned, advice=self.advice,
                           advice_assigned=self.advice_assigned, instance=self.instance, challenges=self.challenges, gates=self.gates,
                           lookups=self.lookups, permutation=self.permutation, mapping=self.mapping, lib=L, device=device, capacity=capacity)

    def oracle(self, threads=0, cap=None):
        """-> (count, records (kind, index, poly, row) in upstream's order)"""
        from harness import build_oracle
        vp, u32 = ctypes.c_void_p, ctypes.c_uint32
        L = build_oracle("mock_verify_oracle", dict(orc_mock_verify=[u32, u32, vp, vp, u32, vp, vp, u32, vp, u32, vp, vp, vp, u32, vp, u32, vp, vp, u32,
                                                                      ctypes.c_int, vp, ctypes.c_uint64]),
                         dict(orc_mock_verify=ctypes.c_uint64))
        tokens, roots, lks = [], [], []
        for g, polys in enumerate(self.gates):
            for p, e in enumerate(polys):
                roots += [g, p, len(tokens)]
                serialize(e, tokens)
        for ins, tbs in self.lookups:
            lks.append(len(ins))
            offs = []
            for e in list(ins) + list(tbs):
                offs.append(len(tokens))
                serialize(e, tokens)
            lks += offs
        nb = (self.n + 7) // 8

        def cat(arrs, shape, dtype):
            return np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=dtype).reshape(shape) for a in arrs]) if arrs else np.zeros(8, dtype=dtype))

        fx, ad, ins = cat(self.fixed, (-1, 4), np.uint64), cat(self.advice, (-1, 4), np.uint64), cat(self.instance, (-1, 4), np.uint64)
        fb = cat([mock.bitmap(a) for a in self.fixed_assigned], (nb,), np.uint8)
        ab = cat([mock.bitmap(a) for a in self.advice_assigned], (nb,), np.uint8)
        ch = np.ascontiguousarray(self.challenges if len(self.challenges) else np.zeros((1, 4), dtype=np.uint64), dtype=np.uint64)
        tk = np.array(tokens + [0], dtype=np.uint64)
        rt, lk = np.array(roots + [0], dtype=np.uint32), np.array(lks + [0], dtype=np.uint32)
        pm = np.array([[{"fixed": 1, "advice": 2, "instance": 3}[kd], ix] for kd, ix in self.permutation] + [[0, 0]], dtype=np.uint32)
        mp = cat(list(self.mapping), (-1, 2), np.uint64)
        total = L.orc_mock_verify(self.k, self.bf, fx.ctypes.data, fb.ctypes.data, len(self.fixed), ad.ctypes.data, ab.ctypes.data, len(self.advice),
                                  ins.ctypes.data, len(self.instance), ch.ctypes.data, tk.ctypes.data, rt.ctypes.data, len(roots) // 3, lk.ctypes.data,
                                  len(self.lookups), pm.ctypes.data, mp.ctypes.data, len(self.permutation), threads or os.cpu_count() or 1, None, 0)
        cap = total if cap is None else min(cap, total)
        out = np.zeros((max(cap, 1), 4), dtype=np.uint32)
        L.orc_mock_verify(self.k, self.bf, fx.ctypes.data, fb.ctypes.data, len(self.fixed), ad.ctypes.data, ab.ctypes.data, len(self.advice), ins.ctypes.data,
                          len(self.instance), ch.ctypes.data, tk.ctypes.data, rt.ctypes.data, len(roots) // 3, lk.ctypes.data, len(self.lookups),
                          pm.ctypes.data, mp.ctypes.data, len(self.permutation), threads or os.cpu_count() or 1, out.ctypes.data, cap)
        return total, out[:cap]


def serialize(e, out):
    """an Expression in the oracle's prefix form"""
    def w4(v):
        out.extend(int(x) for x in words([v])[0])
    if isinstance(e, Constant):
        out.append(0); w4(e.value)
    elif isinstance(e, (Fixed, Advice, Instance)):
        out += [1 if isinstance(e, Fixed) else 2 if isinstance(e, Advice) else 3, e.column_index, e.rotation & 0xFFFFFFFFFFFFFFFF]
    elif isinstance(e, Challenge):
        out += [4, e.index]
    elif isinstance(e, Negated):
        out.append(5); serialize(e.a, out)
    elif isinstance(e, Sum):
        out.append(6); serialize(e.a, out); serialize(e.b, out)
    elif isinstance(e, Product):
        out.append(7); serialize(e.a, out); serialize(e.b, out)
    elif isinstance(e, Scaled):
        out.append(8); serialize(e.a, out); w4(e.f)
    else:
        raise TypeError(e)


NAMES = {0: "ConstraintNotSatisfied", 1: "ConstraintPoisoned", 2: "Lookup", 3: "Permutation"}


def as_failures(records):
    """oracle records -> MockProver::verify's failures: ConstraintPoisoned has no location, and verify_at_rows_par ends with
    `errors.dedup_by(|a, b| both ConstraintPoisoned && a == b)`"""
    out = []
    for k, i, p, r in np.asarray(records).tolist():
        f = (NAMES[k], i, p, r) if k == 0 else (NAMES[k], i, p) if k == 1 else (NAMES[k], i, r)
        if k == 1 and out and out[-1] == f:
            continue
        out.append(f)
    return out


def device_order(records):
    """upstream's order -> the device's: lookup records by (lookup, row) instead of (tuple, row)"""
    recs = [tuple(r) for r in np.asarray(records).tolist()]
    lk = sorted((r for r in recs if r[0] == 2), key=lambda r: (r[1], r[3]))
    first = next((i for i, r in enumerate(recs) if r[0] == 2), None)
    if first is None:
        return recs
    rest = [r for r in recs if r[0] != 2]
    return rest[:first] + lk + rest[first:]


# ---- circuits ------------------------------------------------------------------------------------------------------------
def halo2_lib(k, seed, bf=5, lookup=True, permutation=True, m3=False, plonk=True, assign_frac=1.0, pairs=None):
    """halo2-lib's shape: one advice column with q (a + b c - d) over rotations 0..3 every 4 rows, a standard-plonk gate over three
    more advice columns, a range lookup of an advice column against a fixed table, optionally an m = 3 lookup, and copy
    constraints across advice, fixed and instance columns.  pairs (default from k = 18 on): the copies are disjoint pairs of cells,
    built without upstream's Assembly, which the host walks cell by cell."""
    rng = np.random.default_rng(seed)
    c = Circuit(k, bf)
    n, u = c.n, c.usable
    # halo2-lib's gate
    q = np.zeros(n, dtype=np.int64)
    q[0:max(u - 3, 0):4] = 1
    a = random_words(rng, n)
    r0 = np.arange(0, max(u - 3, 0), 4)
    a[r0 + 3] = fadd(a[r0], fmul(a[r0 + 1], a[r0 + 2]))
    qcol = c.column("fixed", words(q))
    acol = c.column("advice", a, rng.random(n) < assign_frac if assign_frac < 1 else None)
    if assign_frac < 1:      # the cells the gate reads stay assigned
        for d in range(4):
            c.advice_assigned[acol][r0 + d] = True
    c.ix.update(q=qcol, a=acol)
    c.gates.append([Product(Fixed(qcol), Sum(Sum(Advice(acol, 0), Product(Advice(acol, 1), Advice(acol, 2))), Negated(Advice(acol, 3))))])
    if plonk:
        # q_a a + q_b b + q_m a b + q_c c + q_const = 0 with q_c = -1
        qa, qb, qm, qk = (random_words(rng, n) for _ in range(4))
        x, y = random_words(rng, n), random_words(rng, n)
        z = fadd(fadd(fadd(fmul(qa, x), fmul(qb, y)), fmul(qm, fmul(x, y))), qk)
        on = rng.random(n) < 0.7
        on[u:] = False
        qs = [c.column("fixed", np.where(on[:, None], v, 0).astype(np.uint64)) for v in (qa, qb, qm, qk)]
        qc = c.column("fixed", np.where(on[:, None], words([R - 1]), 0).astype(np.uint64))
        xs = [c.column("advice", v) for v in (x, y, z)]
        A, B, C = (Advice(i) for i in xs)
        c.gates.append([Sum(Sum(Sum(Product(Fixed(qs[0]), A), Product(Fixed(qs[1]), B)), Sum(Product(Fixed(qs[2]), Product(A, B)), Product(Fixed(qc), C))),
                            Fixed(qs[3]))])
    if lookup:
        T = min(256, u)
        t = np.arange(n) % T
        t[u:] = T - 1
        tcol = c.column("fixed", words(t))
        ql = (rng.random(n) < 0.5).astype(np.int64)
        ql[u:] = 0
        xcol = c.column("advice", words(rng.integers(0, T, size=n)))
        qlc = c.column("fixed", words(ql))
        c.ix.update(t=tcol, x=xcol, ql=qlc, T=T)
        c.lookups.append(([Product(Fixed(qlc), Advice(xcol))], [Fixed(tcol)]))
    if m3:
        T = min(64, u)
        tab = [random_words(rng, n) for _ in range(3)]
        for tb in tab:
            tb[T:] = tb[T - 1]
        tcols = [c.column("fixed", tb) for tb in tab]
        pick = rng.integers(0, T, size=n)
        ins = [c.column("advice", tb[pick]) for tb in tab]
        c.ix.update(m3_inputs=ins, m3_lookup=len(c.lookups))
        c.lookups.append(([Advice(i) for i in ins], [Fixed(t) for t in tcols]))
    if permutation:
        e = c.column("advice", random_words(rng, n))
        f = c.column("fixed", random_words(rng, n))
        i = c.column("instance", random_words(rng, n))
        c.ix.update(e=e, f=f, i=i)
        c.permutation = [("advice", acol), ("advice", e), ("fixed", f), ("instance", i)]
        P = len(c.permutation)
        if pairs or (pairs is None and k >= 18):
            # disjoint pairs of cells of the copy-only columns (1..3) at usable rows, the second taking the first one's value
            cells = rng.choice((P - 1) * u, size=2 * max(4, n // 8), replace=False)
            col, row = 1 + cells // u, cells % u
            c.mapping = np.stack([np.stack([np.full(n, q, dtype=np.uint64), np.arange(n, dtype=np.uint64)], axis=1) for q in range(P)])
            a_, b_ = slice(0, None, 2), slice(1, None, 2)
            c.mapping[col[a_], row[a_]] = np.stack([col[b_], row[b_]], axis=1)
            c.mapping[col[b_], row[b_]] = np.stack([col[a_], row[a_]], axis=1)
            vals = {q: c.cols(c.permutation[q][0])[c.permutation[q][1]] for q in range(1, P)}
            for q in range(1, P):
                for q2 in range(1, P):
                    sel = (col[a_] == q) & (col[b_] == q2)
                    vals[q2][row[b_][sel]] = vals[q][row[a_][sel]]
            return c
        # copies between the copy-only columns (1..3) at usable rows; column 0 (the gate's) only as its own identity
        c.copies = [(int(rng.integers(1, P)), int(rng.integers(u)), int(rng.integers(1, P)), int(rng.integers(u))) for _ in range(max(4, n // 4))]
    c.finish_permutation()
    return c


def poison_algebra(k, seed, bf=5):
    """gates that read an all-zero advice column one and two rows ahead, so that the last usable rows read Poison: a Scaled term, a
    Product with a zero side on either side, x + 0, x * 1, x * 2, x * x, -x, x - x, x * 0 and Poison * Poison"""
    rng = np.random.default_rng(seed)
    c = Circuit(k, bf)
    n, u = c.n, c.usable
    pcol = c.column("advice", np.zeros((n, 4), dtype=np.uint64))
    qv = (rng.random(n) < 0.3).astype(np.int64)
    qv[u - 2:u + 1] = [1, 0, 1]          # an enabled and a zero selector on rows that read Poison
    qcol = c.column("fixed", words(qv))
    x, x2 = Advice(pcol, 1), Advice(pcol, 2)
    c.gates = [[Scaled(x, 5)], [Scaled(x, 0)], [Product(x, Fixed(qcol))], [Product(Fixed(qcol), x)], [Sum(x, Constant(0))], [Product(x, Constant(1))],
               [Product(x, Constant(2))], [Product(x, x)], [Negated(x)], [Sum(x, Negated(x))], [Product(x, Constant(0))], [Product(x2, x)],
               [Product(Fixed(qcol), Sum(x2, Scaled(x, 3))), Scaled(Product(Fixed(qcol), x2), 7)]]
    c.finish_permutation()
    return c
