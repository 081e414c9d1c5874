"""
The lazily reduced a*b + c*d with one Montgomery reduction that gives the MSM's mixed addition its Y3
(Y3 = R (Q - X3) + Y1 (p - PPP)): the exact bits (a*b + c*d + M p) / 2^256 and the [0, 2p) bound at the edge values of
the lazy range, with b and d canonical as the bound needs.  The same checks run on the kernel-logic emulator (CPU) and,
marked gpu, on the device; the generator's interpreter proves the PTX itself on the same kind of operands.
"""
import os
import sys

import pytest

from test_lazy_field import MODS, R, ints, lazy_operands, words

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check_mul2_lazy(L):
    for f, mod in MODS.items():
        A, B = lazy_operands(mod, seed=3 + mod % 89)
        got = ints(L.field_op(f, "mul2_lazy", words(A), words(B)))
        pinv = pow(mod, -1, R)
        for x, y, g in zip(A, B, got):
            t = x * (y % mod) + y * (mod - x % mod)          # a (b mod p) + b (p - (a mod p))
            assert g == (t + (-t * pinv % R) * mod) // R, (f, hex(x), hex(y))
            assert g < 2 * mod, (f, hex(x), hex(y))


def test_generator_proves_mul2_lazy_and_neg_lazy():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_field_ptx as g
    for mod in (g.FR, g.FQ):
        assert g.check_lazy(g.gen_mont_mul("mul2_lazy", mod, lazy=True, pair=True), mod, "mul2", trials=300) > 0
        assert g.check_lazy(g.gen_neg("neg_lazy", mod), mod, "neg", trials=300) > 0
        assert g.check(g.gen_mont_mul("mul2", mod, pair=True), mod, "mul2", trials=300) > 0


def test_mul2_lazy(emu):
    check_mul2_lazy(emu)


@pytest.mark.gpu
def test_gpu_mul2_lazy(gpu):
    check_mul2_lazy(gpu)
