"""
MockProver::verify's row loops on the device ([UP] halo2_proofs/src/dev.rs, `verify_par`): every gate polynomial on every row, every
lookup input row against its table and every copy constraint, through h2b_mock_verify.

The circuit comes as MockProver holds it after `run`: host columns (2^k x 4 uint64, Montgomery) with a per-cell `assigned` flag for
the fixed and advice columns, the instance columns, the challenges, the gates as lists of `evaluation` Expressions (selectors already
compressed into fixed columns), the lookups as (input expressions, table expressions) and the permutation's columns with their
mapping.  Advice rows from usable_rows = 2^k - (blinding_factors + 1) on are Poison, as upstream poisons them.  The expressions are
compiled with `evaluation.GraphEvaluator`, one root per polynomial.

Failures come back in upstream's order and shape:
    ("ConstraintNotSatisfied", gate, poly, row) / ("ConstraintPoisoned", gate, poly)          gates, rows, polynomials
    ("Lookup", lookup, row)                                                                  per lookup in (input tuple, row) order
    ("Permutation", column, row)                                                             columns, rows
The device reports lookup failures by row; they are put back in upstream's (tuple, row) order here, evaluating the few failing
input tuples on the host.  As upstream's ConstraintPoisoned carries no location, consecutive equal ones are merged into one, as
upstream's closing `errors.dedup_by(..)` merges them (one poisoned polynomial fails on every blinding row its rotations reach).  Region checks (CellNotAssigned) and failure locations stay with the caller, as in upstream's own code.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np

from . import _lib
from .domain import FR_MODULUS
from .evaluation import (ADVICE, FIXED, INSTANCE, Advice, Challenge, Constant, Fixed, GraphEvaluator, Instance, Negated, Product, Scaled,
                         Sum)

_KINDS = {"fixed": FIXED, "advice": ADVICE, "instance": INSTANCE}
_NAMES = {_lib.MOCK_CONSTRAINT_NOT_SATISFIED: "ConstraintNotSatisfied", _lib.MOCK_CONSTRAINT_POISONED: "ConstraintPoisoned",
          _lib.MOCK_LOOKUP: "Lookup", _lib.MOCK_PERMUTATION: "Permutation"}
_R_INV = pow(1 << 256, -1, FR_MODULUS)


def bitmap(assigned) -> np.ndarray:
    """per-row assigned flags (2^k bools) -> the (2^k + 7) // 8 bitmap bytes of h2b_mock_verify (bit r % 8 of byte r / 8)"""
    return np.packbits(np.asarray(assigned, dtype=bool).reshape(-1), bitorder="little")


def _canonical(words) -> int:
    w = [int(x) for x in np.asarray(words, dtype=np.uint64).reshape(4)]
    return (w[0] | w[1] << 64 | w[2] << 128 | w[3] << 192) * _R_INV % FR_MODULUS


class _HostCells:
    """Value of an expression at one row on the host ([UP] Expression::evaluate_lazy over MockProver's cells): None is Poison"""

    def __init__(self, n, usable, fixed, fixed_assigned, advice, advice_assigned, instance, challenges):
        self.n, self.usable = n, usable
        self.fixed, self.fixed_assigned, self.advice, self.advice_assigned = fixed, fixed_assigned, advice, advice_assigned
        self.instance, self.challenges = instance, challenges

    def value(self, e, row):
        if isinstance(e, Constant):
            return e.value % FR_MODULUS
        if isinstance(e, (Fixed, Advice, Instance)):
            r = (row + e.rotation) % self.n
            if isinstance(e, Instance):
                return _canonical(self.instance[e.column_index][r])
            if isinstance(e, Advice) and r >= self.usable:
                return None
            cols, flags = (self.fixed, self.fixed_assigned) if isinstance(e, Fixed) else (self.advice, self.advice_assigned)
            return _canonical(cols[e.column_index][r]) if flags[e.column_index][r] else 0
        if isinstance(e, Challenge):
            return _canonical(self.challenges[e.index])
        if isinstance(e, Negated):
            a = self.value(e.a, row)
            return None if a is None else -a % FR_MODULUS
        if isinstance(e, Sum):
            a, b = self.value(e.a, row), self.value(e.b, row)
            return None if a is None or b is None else (a + b) % FR_MODULUS
        if isinstance(e, Product):
            a = self.value(e.a, row)
            if a == 0:
                return 0
            b = self.value(e.b, row)
            if a is not None and b is not None:
                return a * b % FR_MODULUS
            return 0 if b == 0 else None
        if isinstance(e, Scaled):
            a, f = self.value(e.a, row), e.f % FR_MODULUS
            if a is None:
                return 0 if f == 0 else None
            return a * f % FR_MODULUS
        raise TypeError("unsupported expression %r" % (e,))


def _order_key(v):
    """Value's derived Ord: Real < Poison, Reals by their canonical integer"""
    return (1, 0) if v is None else (0, v)


def compile_gates(gates: Sequence[Sequence]):
    """-> (GraphArrays, roots [(gate, poly, value source)]) of every gate polynomial"""
    graph, roots = GraphEvaluator(), []
    for g, polys in enumerate(gates):
        for p, poly in enumerate(polys):
            roots.append((g, p, graph.add_expression(poly)))
    return graph.arrays(), roots


def compile_lookup(input_expressions, table_expressions):
    """-> (GraphArrays, input roots, table roots) of one lookup argument"""
    graph = GraphEvaluator()
    ins = [graph.add_expression(e) for e in input_expressions]
    tbs = [graph.add_expression(e) for e in table_expressions]
    return graph.arrays(), ins, tbs


def verify(k: int, blinding_factors: int, *, fixed=(), fixed_assigned=(), advice=(), advice_assigned=(), instance=(), challenges=(),
           gates: Sequence[Sequence] = (), lookups: Sequence[tuple] = (), permutation: Sequence[tuple] = (), mapping=(), lib=None, device: int = 0,
           capacity: int = 1024) -> list:
    """The failures of MockProver::verify's gate, lookup and permutation loops, in upstream's order (module docstring).
    fixed_assigned / advice_assigned: per column, 2^k bools; permutation: [("fixed" | "advice" | "instance", index)] with its mapping,
    per column 2^k (column, row) pairs.  `capacity` is the first record buffer; a circuit with more failures is asked again with room
    for all of them."""
    L = lib or _lib.load()
    n = 1 << k
    graph, roots = compile_gates(gates)
    lks = [compile_lookup(i, t) for i, t in lookups]
    perm = [(_KINDS[kind], index) for kind, index in permutation]
    ch = np.ascontiguousarray(challenges, dtype=np.uint64).reshape(-1, 4) if len(challenges) else np.zeros((0, 4), dtype=np.uint64)
    args = (device, k, blinding_factors, fixed, [bitmap(a) for a in fixed_assigned], advice, [bitmap(a) for a in advice_assigned], instance, ch,
            graph, roots, lks, perm, list(mapping))
    count, records = L.mock_verify(*args, capacity=capacity)
    if count > capacity:
        count, records = L.mock_verify(*args, capacity=count)
    cells = _HostCells(n, n - (blinding_factors + 1), [np.asarray(c, dtype=np.uint64).reshape(-1, 4) for c in fixed],
                       [np.asarray(a, dtype=bool).reshape(-1) for a in fixed_assigned], [np.asarray(c, dtype=np.uint64).reshape(-1, 4) for c in advice],
                       [np.asarray(a, dtype=bool).reshape(-1) for a in advice_assigned], [np.asarray(c, dtype=np.uint64).reshape(-1, 4) for c in instance],
                       ch)
    out, lookup_rows = [], {}
    for kind, index, poly, row in records.tolist():
        if kind == _lib.MOCK_LOOKUP:
            lookup_rows.setdefault(index, []).append(row)
            continue
        if kind == _lib.MOCK_PERMUTATION and lookup_rows:
            out += _lookup_failures(lookups, lookup_rows, cells)
            lookup_rows = {}
        if kind == _lib.MOCK_CONSTRAINT_POISONED:
            out.append((_NAMES[kind], index, poly))
        elif kind == _lib.MOCK_CONSTRAINT_NOT_SATISFIED:
            out.append((_NAMES[kind], index, poly, row))
        else:
            out.append((_NAMES[kind], index, row))
    return dedup_poisoned(out + _lookup_failures(lookups, lookup_rows, cells))


def dedup_poisoned(failures: list) -> list:
    """upstream's `errors.dedup_by`: a ConstraintPoisoned equal to the one before it is dropped; nothing else is merged"""
    out = []
    for f in failures:
        if not (out and f[0] == "ConstraintPoisoned" and out[-1] == f):
            out.append(f)
    return out


def _lookup_failures(lookups, lookup_rows, cells) -> list:
    """upstream sorts a lookup's (input tuple, row) pairs before it searches: its failures come out in that order"""
    out = []
    for index in sorted(lookup_rows):
        inputs = lookups[index][0]
        keyed = sorted((tuple(_order_key(cells.value(e, row)) for e in inputs), row) for row in lookup_rows[index])
        out += [("Lookup", index, row) for _, row in keyed]
    return out
