"""
Lazily reduced field arithmetic (values in [0, 2p), no final subtraction after a Montgomery product) that the MSM
bucket accumulation and the NTT butterflies run on: the primitives at the edge values of their range, and the lazy
mixed addition on an accumulator that is not canonical, including the doubling and opposite-point cases.  The same
checks run on the kernel-logic emulator (CPU) and, marked gpu, on the device.
"""
import random

import numpy as np
import pytest

import bn254 as o

R = 1 << 256
MODS = {"fr": o.R_MOD, "fq": o.P_MOD}


def words(vals):
    return np.array([[(v >> (64 * i)) & ((1 << 64) - 1) for i in range(4)] for v in vals], dtype=np.uint64)


def ints(w):
    return [sum(int(x) << (64 * i) for i, x in enumerate(row)) for row in w]


def lazy_operands(mod, n_random=256, seed=0):
    """pairs (a, b) in [0, 2p): edge values 0, 1, p - 1, p, p + 1, 2p - 1, long runs of one-bits, then random ones."""
    rng = random.Random(seed)
    edge = [0, 1, 2, mod - 1, mod, mod + 1, 2 * mod - 1, 2 * mod - 2, R % mod, mod + R % mod, 0xFFFFFFFF,
            (1 << 64) - 1, (1 << 224) - 1, mod - 0xFFFFFFFF, mod + 0xFFFFFFFF]
    for sh in range(0, 256, 32):
        edge += [((1 << 256) - (1 << sh)) % (2 * mod), ((1 << sh) - 1) % (2 * mod)]
    pairs = [(x, y) for x in edge for y in edge]
    pairs += [(rng.randrange(2 * mod), rng.randrange(2 * mod)) for _ in range(n_random)]
    return [x for x, _ in pairs], [y for _, y in pairs]


def check_lazy_field(L, oc):
    for f, mod in MODS.items():
        A, B = lazy_operands(mod, seed=len(f) + mod % 97)
        a, b = words(A), words(B)
        a_c, b_c = words([x % mod for x in A]), words([y % mod for y in B])
        pinv = pow(mod, -1, R)
        for op, want_canon in (("mul_lazy", oc.field_op(f, "mul", a_c, b_c)), ("add_lazy", oc.field_op(f, "add", a_c, b_c)),
                               ("sub_lazy", oc.field_op(f, "sub", a_c, b_c)), ("sqr_lazy", oc.field_op(f, "mul", a_c, a_c))):
            got = ints(L.field_op(f, op, a, b) if op != "sqr_lazy" else L.field_op(f, op, a))
            assert all(g < 2 * mod for g in got), (f, op)
            assert (words([g % mod for g in got]) == want_canon).all(), (f, op)
            if op in ("mul_lazy", "sqr_lazy"):
                # the Montgomery value before the final subtraction is unique: (xy + Mp) / 2^256, M = -xy/p mod 2^256
                for x, y, g in zip(A, A if op == "sqr_lazy" else B, got):
                    assert g == (x * y + (-x * y * pinv % R) * mod) // R, (f, op, hex(x), hex(y))
        assert ints(L.field_op(f, "canon", a)) == [x % mod for x in A], f
        assert ints(L.field_op(f, "is_zero_lazy", a)) == [int(x % mod == 0) for x in A], f


def check_lazy_mixed_addition(L, oc, n=32):
    """ec op 4: the accumulator holds P with x, y, ZZ and ZZZ all offset by p; the incoming point is P (doubling),
    -P (opposite point), the identity, or a random point."""
    def aff(w):
        v = oc.words_to_ints(np.ascontiguousarray(w).reshape(-1, 4))
        return [None if (v[2 * i] == 0 and v[2 * i + 1] == 0) else (o.from_mont(v[2 * i], o.P_MOD), o.from_mont(v[2 * i + 1], o.P_MOD))
                for i in range(len(v) // 2)]
    P, Q = oc.gen_points(21, n), oc.gen_points(23, n)
    for i in range(0, n, 4):
        Q[i] = P[i]                                                          # doubling
        Q[i + 1, :4] = P[i + 1, :4]                                          # opposite point
        Q[i + 1, 4:] = oc.field_op("fq", "sub", np.zeros((1, 4), dtype=np.uint64), P[i + 1:i + 2, 4:])[0]
    Q[2] = 0                                                                 # identity operand
    P[6] = 0                                                                 # identity accumulator
    pa, qa = aff(P), aff(Q)
    got = aff(L.ec_op(4, P, Q))
    for i in range(n):
        assert got[i] == o.g1_add(pa[i], qa[i]), i
    assert got[1] is None and got[0] == o.g1_mul(pa[0], 2)


def test_lazy_field_primitives(emu, oc):
    check_lazy_field(emu, oc)


def test_lazy_mixed_addition_on_offset_accumulator(emu, oc):
    check_lazy_mixed_addition(emu, oc)


@pytest.mark.gpu
def test_gpu_lazy_field_primitives(gpu, oc):
    check_lazy_field(gpu, oc)


@pytest.mark.gpu
def test_gpu_lazy_mixed_addition_on_offset_accumulator(gpu, oc):
    check_lazy_mixed_addition(gpu, oc, 256)
