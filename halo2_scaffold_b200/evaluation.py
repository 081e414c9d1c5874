"""
Host-side mirror of halo2_proofs::plonk::evaluation ([UP] halo2_proofs/src/plonk/evaluation.rs, SURVEY.md
section 8f rank 2): `GraphEvaluator` (how the prover flattens the gate / lookup expressions once per proving
key) and `Evaluator::evaluate_h` (the per-proof quotient evaluation over the extended coset).

The graph construction is scalar host work, exactly as in the Rust code; every per-row loop of evaluate_h
runs on the GPU on device-resident columns:
    custom gates  -> h2b_evaluate_graph_dev
    permutations  -> h2b_evaluate_h_permutation_dev
    lookups       -> h2b_evaluate_h_lookup_dev   (one call per lookup argument)
Names and argument meaning follow upstream (ValueSource, Calculation, add_expression, add_calculation, ...).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np

from . import _lib
from .domain import FR_MODULUS, fr_to_words

# enum ValueSource, in declaration order (the derived PartialOrd upstream sorts by variant, then fields)
CONSTANT, INTERMEDIATE, FIXED, ADVICE, INSTANCE, CHALLENGE, BETA, GAMMA, THETA, Y, PREVIOUS_VALUE = range(11)
# enum Calculation
ADD, SUB, MUL, SQUARE, DOUBLE, NEGATE, HORNER, STORE = range(8)


def ValueSource(kind: int, index: int = 0, rotation: int = 0):
    return (kind, index, rotation)


# ---- plonk::Expression ----------------------------------------------------------------------------------
@dataclass(frozen=True)
class Constant:
    value: int


@dataclass(frozen=True)
class Fixed:
    column_index: int
    rotation: int = 0


@dataclass(frozen=True)
class Advice:
    column_index: int
    rotation: int = 0


@dataclass(frozen=True)
class Instance:
    column_index: int
    rotation: int = 0


@dataclass(frozen=True)
class Challenge:
    index: int


@dataclass(frozen=True)
class Negated:
    a: object


@dataclass(frozen=True)
class Sum:
    a: object
    b: object


@dataclass(frozen=True)
class Product:
    a: object
    b: object


@dataclass(frozen=True)
class Scaled:
    a: object
    f: int


class GraphEvaluator:
    """[UP] evaluation.rs `struct GraphEvaluator` (Default: constants 0, 1, 2)."""

    def __init__(self):
        self.constants = [0, 1, 2]
        self.rotations: list[int] = []
        self.calculations: list[tuple] = []      # CalculationInfo: ((op, a, b, parts), target)
        self.num_intermediates = 0

    def add_rotation(self, rotation: int) -> int:
        if rotation in self.rotations:
            return self.rotations.index(rotation)
        self.rotations.append(rotation)
        return len(self.rotations) - 1

    def add_constant(self, constant: int):
        constant %= FR_MODULUS
        if constant in self.constants:
            return ValueSource(CONSTANT, self.constants.index(constant))
        self.constants.append(constant)
        return ValueSource(CONSTANT, len(self.constants) - 1)

    def add_calculation(self, op: int, a, b=(0, 0, 0), parts: Sequence = ()):
        calc = (op, tuple(a), tuple(b), tuple(tuple(p) for p in parts))
        for existing, target in self.calculations:
            if existing == calc:
                return ValueSource(INTERMEDIATE, target)
        target = self.num_intermediates
        self.calculations.append((calc, target))
        self.num_intermediates += 1
        return ValueSource(INTERMEDIATE, target)

    def add_expression(self, expr):
        zero, one, two = ValueSource(CONSTANT, 0), ValueSource(CONSTANT, 1), ValueSource(CONSTANT, 2)
        if isinstance(expr, Constant):
            return self.add_constant(expr.value)
        if isinstance(expr, (Fixed, Advice, Instance)):
            rot_idx = self.add_rotation(expr.rotation)
            kind = FIXED if isinstance(expr, Fixed) else ADVICE if isinstance(expr, Advice) else INSTANCE
            return self.add_calculation(STORE, ValueSource(kind, expr.column_index, rot_idx))
        if isinstance(expr, Challenge):
            return self.add_calculation(STORE, ValueSource(CHALLENGE, expr.index))
        if isinstance(expr, Negated):
            if isinstance(expr.a, Constant):
                return self.add_constant(-expr.a.value)
            result_a = self.add_expression(expr.a)
            return result_a if result_a == zero else self.add_calculation(NEGATE, result_a)
        if isinstance(expr, Sum):
            if isinstance(expr.b, Negated):          # a + (-b) is stored back as a subtraction
                result_a, result_b = self.add_expression(expr.a), self.add_expression(expr.b.a)
                if result_a == zero:
                    return self.add_calculation(NEGATE, result_b)
                if result_b == zero:
                    return result_a
                return self.add_calculation(SUB, result_a, result_b)
            result_a, result_b = self.add_expression(expr.a), self.add_expression(expr.b)
            if result_a == zero:
                return result_b
            if result_b == zero:
                return result_a
            return self.add_calculation(ADD, result_a, result_b) if result_a <= result_b else self.add_calculation(ADD, result_b, result_a)
        if isinstance(expr, Product):
            result_a, result_b = self.add_expression(expr.a), self.add_expression(expr.b)
            if result_a == zero or result_b == zero:
                return zero
            if result_a == one:
                return result_b
            if result_b == one:
                return result_a
            if result_a == two:
                return self.add_calculation(DOUBLE, result_b)
            if result_b == two:
                return self.add_calculation(DOUBLE, result_a)
            if result_a == result_b:
                return self.add_calculation(SQUARE, result_a)
            return self.add_calculation(MUL, result_a, result_b) if result_a <= result_b else self.add_calculation(MUL, result_b, result_a)
        if isinstance(expr, Scaled):
            f = expr.f % FR_MODULUS
            if f == 0:
                return zero
            if f == 1:
                return self.add_expression(expr.a)
            cst = self.add_constant(f)
            result_a = self.add_expression(expr.a)
            return self.add_calculation(MUL, result_a, cst)
        raise TypeError("unsupported expression %r (selectors are replaced before the evaluator is built)" % (expr,))

    def arrays(self) -> _lib.GraphArrays:
        """flatten into the arrays of `h2b_graph` (include/h2b200.h)"""
        calcs = np.zeros((len(self.calculations), 10), dtype=np.uint32)
        parts: list[tuple] = []
        for i, ((op, a, b, ps), target) in enumerate(self.calculations):
            calcs[i] = [op, target, *a, *b, len(parts) if ps else 0, len(ps)]
            parts.extend(ps)
        constants = np.stack([fr_to_words(c) for c in self.constants]) if self.constants else np.zeros((0, 4), dtype=np.uint64)
        return _lib.GraphArrays(constants, np.array(self.rotations, dtype=np.int32), calcs,
                                np.array(parts, dtype=np.uint32).reshape(-1, 3), self.num_intermediates)


class _Device:
    """uploads host columns for the duration of one call"""

    def __init__(self, lib, device: int, size: int):
        self.L, self.device, self.size, self.held = lib, device, size, []

    def up(self, a) -> int:
        a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
        assert a.shape[0] == self.size, (a.shape, self.size)
        d = self.L.dev_alloc(self.device, max(self.size, 1) * 32)
        self.held.append(d)
        self.L.h2d(self.device, d, a)
        return d

    def down(self, d: int) -> np.ndarray:
        self.L.dev_sync(self.device)
        out = np.empty((self.size, 4), dtype=np.uint64)
        self.L.d2h(self.device, out, d)
        return out

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for d in self.held:
            self.L.dev_free(self.device, d)


def evaluate_graph(lib, graph: _lib.GraphArrays, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale: int,
                   device: int = 0) -> np.ndarray:
    """values[idx] = graph.evaluate(.., previous_value = values[idx], idx, rot_scale, isize) on host arrays, through the device"""
    values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
    with _Device(lib, device, values.shape[0]) as dev:
        cols = _lib.EvalColumns([dev.up(c) for c in fixed], [dev.up(c) for c in advice], [dev.up(c) for c in instance], challenges, beta, gamma,
                                theta, y)
        d_values = dev.up(values)
        lib.evaluate_graph_dev(device, graph, cols, d_values, values.shape[0], rot_scale)
        return dev.down(d_values)


def evaluate_h_lookup(lib, graph: _lib.GraphArrays, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale: int, product_coset,
                      permuted_input_coset, permuted_table_coset, l0, l_last, l_active_row, device: int = 0) -> np.ndarray:
    values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
    with _Device(lib, device, values.shape[0]) as dev:
        cols = _lib.EvalColumns([dev.up(c) for c in fixed], [dev.up(c) for c in advice], [dev.up(c) for c in instance], challenges, beta, gamma,
                                theta, y)
        d_values = dev.up(values)
        lib.evaluate_h_lookup_dev(device, graph, cols, d_values, values.shape[0], rot_scale, dev.up(product_coset), dev.up(permuted_input_coset),
                                  dev.up(permuted_table_coset), dev.up(l0), dev.up(l_last), dev.up(l_active_row))
        return dev.down(d_values)


def evaluate_h_permutation(lib, values, rot_scale: int, product_cosets, columns, perm_cosets, chunk_len: int, last_rotation: int, l0, l_last,
                           l_active_row, beta, gamma, y, delta, zeta, extended_omega, device: int = 0) -> np.ndarray:
    values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
    with _Device(lib, device, values.shape[0]) as dev:
        d_values = dev.up(values)
        lib.evaluate_h_permutation_dev(device, d_values, values.shape[0], rot_scale, [dev.up(c) for c in product_cosets],
                                       [dev.up(c) for c in columns], [dev.up(c) for c in perm_cosets], chunk_len, last_rotation, dev.up(l0),
                                       dev.up(l_last), dev.up(l_active_row), beta, gamma, y, delta, zeta, extended_omega)
        return dev.down(d_values)


class Evaluator:
    """[UP] evaluation.rs `struct Evaluator { custom_gates, lookups }` and `Evaluator::new(cs)`."""

    def __init__(self, gate_polynomials: Sequence, lookups: Sequence[tuple] = ()):
        """gate_polynomials: the polynomials of every gate in cs.gates order;
        lookups: (input_expressions, table_expressions) per lookup argument"""
        self.custom_gates = GraphEvaluator()
        parts = [self.custom_gates.add_expression(poly) for poly in gate_polynomials]
        self.custom_gates.add_calculation(HORNER, ValueSource(PREVIOUS_VALUE), ValueSource(Y), parts)
        self.lookups: list[GraphEvaluator] = []
        for input_expressions, table_expressions in lookups:
            graph = GraphEvaluator()

            def evaluate_lc(expressions):
                ps = [graph.add_expression(e) for e in expressions]
                return graph.add_calculation(HORNER, ValueSource(CONSTANT, 0), ValueSource(THETA), ps)

            compressed_input_coset = evaluate_lc(input_expressions)
            compressed_table_coset = evaluate_lc(table_expressions)
            right_gamma = graph.add_calculation(ADD, compressed_table_coset, ValueSource(GAMMA))
            lc = graph.add_calculation(ADD, compressed_input_coset, ValueSource(BETA))
            graph.add_calculation(MUL, lc, right_gamma)
            self.lookups.append(graph)

    def evaluate_h(self, *, size: int, rot_scale: int, fixed=None, advice, instance, challenges, y, beta, gamma, theta, l0=None, l_last=None,
                   l_active_row=None, permutation: dict | None = None, lookups: Sequence[dict] = (), values: np.ndarray | None = None, lib=None,
                   device: int = 0, shard: tuple | None = None, pk=None) -> np.ndarray:
        """One proof's pass of evaluate_h.  Columns are host arrays (size x 4 u64, Montgomery) of extended-coset
        evaluations; they are uploaded once and all three loops run on the device.
        permutation = dict(product_cosets=[..], columns=[("advice"|"fixed"|"instance", index), ..], cosets=[..], chunk_len=,
                           last_rotation=, delta=, zeta=, extended_omega=)       (words: 4 x u64 Montgomery)
        lookups[n]  = dict(product_coset=, permuted_input_coset=, permuted_table_coset=)
        pk = a keygen.ResidentProvingKey: the fixed cosets, the permutation's sigma cosets and l0 / l_last / l_active_row are then read
        from it on `device` and not uploaded (fixed, permutation["cosets"] and the indicators are not needed); a row-sharded pk gives the
        shard of `device`.
        shard = (row0, rows, halo): rows [row0, row0 + rows) only; every column is cut to its slice with `halo` rows on both sides
        (wrap-around included) before it is uploaded -- what each device of a row-sharded evaluate_h holds (a row-sharded pk holds its
        columns that way already).  -> the `rows` values of the shard"""
        L = lib or _lib.load()
        pk_cols = pk.eval_columns(device) if pk is not None else None
        if pk_cols is not None:
            assert shard is None or pk_cols["shard"] is not None, "a replicated pk feeds the unsharded evaluate_h"
            assert shard is None or tuple(shard) == tuple(pk_cols["shard"]), "this device's shard of the pk is %r" % (pk_cols["shard"],)
            shard = pk_cols["shard"]
        assert len(lookups) == len(self.lookups)
        row0, rows, halo = shard if shard is not None else (0, size, 0)
        if values is None:
            values = np.zeros((rows, 4), dtype=np.uint64)
        elif shard is not None:
            values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)[row0:row0 + rows]
        with _Device(L, device, rows + 2 * halo) as dev, _Device(L, device, rows) as vdev:
            if shard is None:
                up = dev.up
            else:
                take = np.arange(row0 - halo, row0 + rows + halo) % size
                up = lambda a: dev.up(np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)[take])
            d_advice, d_instance = [up(c) for c in advice], [up(c) for c in instance]
            if pk_cols is None:
                d_fixed, d_l0, d_l_last, d_l_active = [up(c) for c in fixed], up(l0), up(l_last), up(l_active_row)
            else:
                d_fixed, d_l0, d_l_last, d_l_active = pk_cols["fixed"], pk_cols["l0"], pk_cols["l_last"], pk_cols["l_active_row"]
            d_values = vdev.up(values)
            cols = _lib.EvalColumns(d_fixed, d_advice, d_instance, challenges, beta, gamma, theta, y)
            # Custom gates
            L.evaluate_graph_dev(device, self.custom_gates.arrays(), cols, d_values, size, rot_scale, shard=shard)
            # Permutations
            if permutation is not None and permutation["product_cosets"]:
                by_type = {"advice": d_advice, "fixed": d_fixed, "instance": d_instance}
                d_sigma = [up(c) for c in permutation["cosets"]] if pk_cols is None else pk_cols["permutation"]
                L.evaluate_h_permutation_dev(device, d_values, size, rot_scale, [up(c) for c in permutation["product_cosets"]],
                                             [by_type[t][i] for t, i in permutation["columns"]], d_sigma,
                                             permutation["chunk_len"], permutation["last_rotation"], d_l0, d_l_last, d_l_active, beta, gamma, y,
                                             permutation["delta"], permutation["zeta"], permutation["extended_omega"], shard=shard)
            # Lookups
            for graph, lk in zip(self.lookups, lookups):
                L.evaluate_h_lookup_dev(device, graph.arrays(), cols, d_values, size, rot_scale, up(lk["product_coset"]),
                                        up(lk["permuted_input_coset"]), up(lk["permuted_table_coset"]), d_l0, d_l_last, d_l_active, shard=shard)
            return vdev.down(d_values)
