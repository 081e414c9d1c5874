#!/usr/bin/env python3
"""
Generator + simulator for the 254-bit Montgomery field arithmetic (8 x 32-bit limbs) used by
every kernel in halo2_scaffold_b200/csrc.  It emits `field_asm.inc`: one inline-PTX block per
operation and modulus (BN254 Fr and Fq), built from `mad.lo.cc/madc.hi.cc` carry chains that
ptxas fuses into IMAD.WIDE.U32(.X) pairs (the "even/odd accumulator" scheme, so that no 64-bit
partial product ever overlaps a pending carry).

Because there is no GPU in the build container, the exact instruction stream that is emitted is
first *executed here* by a tiny PTX-subset interpreter (32-bit registers + the CC.CF carry flag)
and checked against Python big-int arithmetic on random and edge-case inputs; generation aborts
if any check fails.

  python tools/gen_field_ptx.py            # verify + write csrc/field_asm.inc
"""
from __future__ import annotations

import os
import random
import sys

M32 = 0xFFFFFFFF
NL = 8  # limbs

FR = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
FQ = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47


def limbs(x, n=NL):
    return [(x >> (32 * i)) & M32 for i in range(n)]


class Prog:
    """A straight-line PTX program over named 32-bit registers."""

    def __init__(self, name, inputs, outputs):
        self.name = name
        self.inputs = inputs      # list of register names (operands, read-only)
        self.outputs = outputs    # list of register names (written)
        self.ins = []             # (op, dst, [srcs])  srcs: reg name or int immediate
        self.temps = []

    def tmp(self, name):
        if name not in self.temps:
            self.temps.append(name)
        return name

    def emit(self, op, dst, *srcs):
        self.ins.append((op, dst, list(srcs)))

    # ---------------- interpreter ----------------
    def run(self, env):
        reg = dict(env)
        cf = 0

        def val(s):
            return s if isinstance(s, int) else reg[s]

        for op, dst, srcs in self.ins:
            v = [val(s) for s in srcs]
            if op == "mov":
                reg[dst] = v[0]
            elif op == "mul.lo":
                reg[dst] = (v[0] * v[1]) & M32
            elif op == "mul.hi":
                reg[dst] = (v[0] * v[1]) >> 32
            elif op in ("mad.lo", "mad.lo.cc", "madc.lo", "madc.lo.cc", "mad.hi", "mad.hi.cc", "madc.hi", "madc.hi.cc"):
                prod = v[0] * v[1]
                part = (prod & M32) if ".lo" in op else (prod >> 32)
                s = part + v[2] + (cf if op.startswith("madc") else 0)
                reg[dst] = s & M32
                if op.endswith(".cc"):
                    cf = s >> 32
            elif op in ("add", "add.cc", "addc", "addc.cc"):
                s = v[0] + v[1] + (cf if op.startswith("addc") else 0)
                reg[dst] = s & M32
                if op.endswith(".cc"):
                    cf = s >> 32
            elif op in ("sub", "sub.cc", "subc", "subc.cc"):
                s = v[0] - v[1] - (cf if op.startswith("subc") else 0)
                reg[dst] = s & M32
                if op.endswith(".cc"):
                    cf = 1 if s < 0 else 0
            elif op == "and":
                reg[dst] = v[0] & v[1]
            elif op == "shl1":        # dst = low 32 bits of ((v1:v0) << 1) >> 32 = (v1 << 1) | (v0 >> 31)   (shf.l.wrap)
                reg[dst] = ((v[1] << 1) | (v[0] >> 31)) & M32
            elif op == "chk0":        # generator-side assertion: the carry flag must be clear here (emits nothing)
                if cf:
                    raise OverflowError("lost carry in %s" % self.name)
            elif op == "selnz":       # dst = (v0 != 0) ? v1 : v2   (emitted as setp + selp)
                reg[dst] = v[1] if v[0] != 0 else v[2]
            else:
                raise ValueError(op)
        return [reg[o] for o in self.outputs]

    # ---------------- emitter ----------------
    def to_cuda(self, signature):
        opnum = {}
        for i, o in enumerate(self.outputs):
            opnum[o] = i
        for i, a in enumerate(self.inputs):
            opnum[a] = len(self.outputs) + i

        def r(s):
            if isinstance(s, int):
                return "0x%08x" % s
            if s in opnum:
                return "%%%d" % opnum[s]
            return s

        lines = []
        if self.temps:
            lines.append(".reg .u32 " + ", ".join(self.temps) + ";")
        lines.append(".reg .pred pz;")
        for op, dst, srcs in self.ins:
            if op == "selnz":
                lines.append("setp.ne.u32 pz, %s, 0;" % r(srcs[0]))
                lines.append("selp.u32 %s, %s, %s, pz;" % (r(dst), r(srcs[1]), r(srcs[2])))
            elif op == "mov":
                lines.append("mov.u32 %s, %s;" % (r(dst), r(srcs[0])))
            elif op == "shl1":
                lines.append("shf.l.wrap.b32 %s, %s, %s, 1;" % (r(dst), r(srcs[0]), r(srcs[1])))
            elif op == "chk0":
                pass
            elif op == "and":
                lines.append("and.b32 %s, %s, %s;" % (r(dst), r(srcs[0]), r(srcs[1])))
            else:
                base, *suffix = op.split(".")
                # mad.lo.cc -> mad.lo.cc.u32 ; add.cc -> add.cc.u32
                lines.append("%s.u32 %s, %s;" % (op, r(dst), ", ".join(r(s) for s in srcs)))
        body = "\n".join('        "%s\\n\\t"' % l for l in ["{"] + lines + ["}"])
        outs = ", ".join('"=r"(%s)' % self._cname(o) for o in self.outputs)
        ins = ", ".join('"r"(%s)' % self._cname(a) for a in self.inputs)
        return "%s {\n    asm(\n%s\n        : %s\n        : %s);\n}\n" % (signature, body, outs, ins)

    @staticmethod
    def _cname(reg):
        # register names like r3 / a5 / b0 map to C array elements r[3] / a[5] / b[0]; z0 is the opaque zero
        if reg == "z0":
            return "z"
        return "%s[%s]" % (reg[0], reg[1:])


# =====================================================================================
# Montgomery multiplication, even/odd accumulators
#   T = E + O*2^32 ; E gets the products a_j*b_i with j even, O those with j odd.
#   After each row the low limb of E is zero, T is divided by 2^32 by *renaming*:
#   new E = old O (+ old e1 at limb 0), new O = old E >> 64.
# =====================================================================================
def gen_mont_mul(name, mod, square=False, lazy=False):
    p = limbs(mod)
    inv = (-pow(mod, -1, 1 << 32)) & M32
    A = ["a%d" % i for i in range(NL)]
    B = A if square else ["b%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A + ([] if square else B), R)
    ev = [P.tmp("e%d" % i) for i in range(NL)]
    od = [P.tmp("o%d" % i) for i in range(NL)]
    m = P.tmp("m")

    def chain_mad(acc, mul_src, scalar, first_has_carry_in=False):
        """acc[0..7] += sum_j mul_src[j]*scalar << 64*j (4 wide products), one carry chain."""
        for j in range(NL // 2):
            lo_op = "madc.lo.cc" if (j > 0 or first_has_carry_in) else "mad.lo.cc"
            P.emit(lo_op, acc[2 * j], mul_src[j], scalar, acc[2 * j])
            P.emit("madc.hi.cc", acc[2 * j + 1], mul_src[j], scalar, acc[2 * j + 1])

    a_even = [A[0], A[2], A[4], A[6]]
    a_odd = [A[1], A[3], A[5], A[7]]
    p_even = [p[0], p[2], p[4], p[6]]
    p_odd = [p[1], p[3], p[5], p[7]]

    E, O = ev, od
    for i in range(NL):
        bi = B[i]
        if i == 0:
            for j in range(NL // 2):
                P.emit("mul.lo", O[2 * j], a_odd[j], bi)
                P.emit("mul.hi", O[2 * j + 1], a_odd[j], bi)
            for j in range(NL // 2):
                P.emit("mul.lo", E[2 * j], a_even[j], bi)
                P.emit("mul.hi", E[2 * j + 1], a_even[j], bi)
        else:
            # divide by 2^32 by renaming: E' = O (limb0 += e1), O' = E >> 64, then add row i
            P.emit("add.cc", O[0], O[0], E[1])
            # new odd accumulator lives in E's registers, shifted down by two limbs
            for j in range(NL // 2):
                src_lo = E[2 * j + 2] if 2 * j + 2 < NL else 0
                src_hi = E[2 * j + 3] if 2 * j + 3 < NL else 0
                P.emit("madc.lo.cc", E[2 * j], a_odd[j], bi, src_lo)
                P.emit("madc.hi.cc", E[2 * j + 1], a_odd[j], bi, src_hi)
            E, O = O, E
            chain_mad(E, a_even, bi)
            P.emit("addc", O[NL - 1], O[NL - 1], 0)
        P.emit("mul.lo", m, E[0], inv)
        chain_mad(O, p_odd, m)
        chain_mad(E, p_even, m)
        P.emit("addc", O[NL - 1], O[NL - 1], 0)
    # T = (E >> 32) + O   (E[0] == 0);  T < 2p whenever a*b < p * 2^256
    t = R if lazy else [P.tmp("t%d" % i) for i in range(NL)]
    for i in range(NL):
        op = "add.cc" if i == 0 else ("addc.cc" if i < NL - 1 else "addc")
        P.emit(op, t[i], O[i], E[i + 1] if i + 1 < NL else 0)
    if lazy:
        return P
    # canonical: r = T - p if T >= p
    s = [P.tmp("s%d" % i) for i in range(NL)]
    bw = P.tmp("bw")
    for i in range(NL):
        P.emit("sub.cc" if i == 0 else "subc.cc", s[i], t[i], p[i])
    P.emit("subc", bw, 0, 0)            # bw = 0xffffffff iff T < p
    for i in range(NL):
        P.emit("selnz", R[i], bw, t[i], s[i])
    return P



# =====================================================================================
# Separated product / reduction ("full-width even/odd accumulators")
#   AE holds the 64-bit product slots that start at even limbs, AO those that start at odd limbs
#   (AO[k] is limb k+1 of the total); every row of partial products is one mad.lo.cc/madc.hi.cc
#   chain inside ONE accumulator, so ptxas keeps it as IMAD.WIDE.U32(.X).  The Montgomery
#   reduction adds its m_i * p rows into the same accumulators; a carry that leaves a chain goes
#   into a small per-limb counter C[pos] (or initialises a still untouched limb), never ripples.
#   Used for the operations whose product phase differs from a plain a*b:
#     * squaring (28 doubled cross products + 8 squares instead of 64 products),
#     * a*b + c*d with ONE reduction (the Y3 of the XYZZ mixed addition).
# =====================================================================================
class WideAcc:
    def __init__(self, P, nlimbs=16):
        self.P = P
        self.n = nlimbs
        self.ae = [P.tmp("x%d" % k) for k in range(nlimbs)]          # limb k
        self.ao = [P.tmp("y%d" % k) for k in range(nlimbs)]          # limb k + 1
        self.te = [False] * nlimbs
        self.to = [False] * nlimbs
        self.c = {}                                                  # total limb position -> counter register

    def _counter(self, pos):
        if pos not in self.c:
            self.c[pos] = self.P.tmp("k%d" % pos)
            return self.c[pos], 0
        return self.c[pos], self.c[pos]

    def chain(self, limb, products):
        """add sum_j products[j] << 64*j at total limb position `limb` (one carry chain)."""
        P = self.P
        even = (limb % 2 == 0)
        regs, touched, start = (self.ae, self.te, limb) if even else (self.ao, self.to, limb - 1)
        for j, (x, y) in enumerate(products):
            k = start + 2 * j
            lo_src = regs[k] if touched[k] else 0
            hi_src = regs[k + 1] if touched[k + 1] else 0
            P.emit("mad.lo.cc" if j == 0 else "madc.lo.cc", regs[k], x, y, lo_src)
            P.emit("madc.hi.cc", regs[k + 1], x, y, hi_src)
            touched[k] = touched[k + 1] = True
        top = start + 2 * len(products)
        if top >= self.n:
            P.emit("chk0", None)
            return
        if not touched[top]:
            P.emit("addc", regs[top], 0, 0)
            touched[top] = True
        else:
            pos = top if even else top + 1
            if pos >= self.n:
                P.emit("chk0", None)
            else:
                creg, csrc = self._counter(pos)
                P.emit("addc", creg, csrc, 0)

    def limb_e(self, k):
        return self.ae[k] if (0 <= k < self.n and self.te[k]) else 0

    def limb_o(self, k):          # AO register that holds total limb k
        return self.ao[k - 1] if (1 <= k <= self.n and self.to[k - 1]) else 0

    def double(self):
        """AE <- 2*AE, AO <- 2*AO with funnel shifts (no carry chain); the small carry counters are doubled too."""
        P = self.P
        for creg in self.c.values():
            P.emit("add", creg, creg, creg)
        for regs, touched in ((self.ae, self.te), (self.ao, self.to)):
            for k in range(self.n - 1, -1, -1):
                if not touched[k]:
                    if k > 0 and touched[k - 1]:
                        P.emit("shl1", regs[k], regs[k - 1], 0)       # only the bit shifted out of the limb below
                        touched[k] = True
                    continue
                P.emit("shl1", regs[k], regs[k - 1] if (k > 0 and touched[k - 1]) else 0, regs[k])


def redc_tail(P, acc, p, inv, R, lazy=False):
    """Montgomery reduction of the value held in acc (< p * 2^256) into R (canonical; lazy: < 2p, no final subtraction)."""
    NLp = NL
    p_even = [p[0], p[2], p[4], p[6]]
    p_odd = [p[1], p[3], p[5], p[7]]
    m = P.tmp("m")
    v = P.tmp("v")
    cw = None                      # carry word into limb i (0..2)
    s1, s2, c1 = P.tmp("s1"), P.tmp("s2"), P.tmp("c1")
    for i in range(NLp):
        if i > 0:
            # limb i-1 of the running total is 0 mod 2^32; its carry goes into limb i
            P.emit("add.cc", s1, acc.limb_e(i - 1), acc.limb_o(i - 1))
            P.emit("addc", c1, 0, 0)
            ncw = P.tmp("w%d" % i)
            if cw is None:
                P.emit("mov", ncw, c1)
            else:
                P.emit("add.cc", s2, s1, cw)
                P.emit("addc", ncw, c1, 0)
            cw = ncw
        P.emit("add", v, acc.limb_e(i), acc.limb_o(i))
        if cw is not None:
            P.emit("add", v, v, cw)
        P.emit("mul.lo", m, v, inv)
        acc.chain(i, [(m, pj) for pj in p_even])
        acc.chain(i + 1, [(m, pj) for pj in p_odd])
    # carry out of limb 7 into limb 8
    P.emit("add.cc", s1, acc.limb_e(NLp - 1), acc.limb_o(NLp - 1))
    P.emit("addc", c1, 0, 0)
    P.emit("add.cc", s2, s1, cw)
    cw8 = P.tmp("w8")
    P.emit("addc", cw8, c1, 0)
    creg, csrc = acc._counter(NLp)
    P.emit("add", creg, csrc, cw8)
    # t = limbs 8..15 of AE + (AO << 32) + counters
    x = [P.tmp("q%d" % k) for k in range(NLp)]
    t = R if lazy else [P.tmp("t%d" % k) for k in range(NLp)]
    for k in range(NLp):
        op = "add.cc" if k == 0 else ("addc.cc" if k < NLp - 1 else "addc")
        P.emit(op, x[k], acc.limb_e(NLp + k), acc.limb_o(NLp + k))
    for k in range(NLp):
        op = "add.cc" if k == 0 else ("addc.cc" if k < NLp - 1 else "addc")
        P.emit(op, t[k], x[k], acc.c.get(NLp + k, 0))
    if lazy:
        return
    s = [P.tmp("s%d" % i) for i in range(NLp)]
    bw = P.tmp("bw")
    for i in range(NLp):
        P.emit("sub.cc" if i == 0 else "subc.cc", s[i], t[i], p[i])
    P.emit("subc", bw, 0, 0)
    for i in range(NLp):
        P.emit("selnz", R[i], bw, t[i], s[i])


def product_rows(acc, X, Y):
    """acc += X * Y (8 x 8 limbs), operand scanning, two chains per row."""
    for i in range(NL):
        acc.chain(i, [(X[j], Y[i]) for j in (0, 2, 4, 6)])
        acc.chain(i + 1, [(X[j], Y[i]) for j in (1, 3, 5, 7)])


def gen_mont_sqr_sep(name, mod, lazy=False):
    p = limbs(mod)
    inv = (-pow(mod, -1, 1 << 32)) & M32
    A = ["a%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A, R)
    acc = WideAcc(P)
    # cross products a_i * a_j, i < j: row i has one chain per parity class of j
    for i in range(NL):
        for par in (1, 0):
            js = [j for j in range(i + 1, NL) if (j - i) % 2 == par]
            if js:
                acc.chain(i + js[0], [(A[i], A[j]) for j in js])
    acc.double()
    # squares a_i^2 at limb 2i: one chain over the whole even accumulator
    acc.chain(0, [(A[i], A[i]) for i in range(NL)])
    redc_tail(P, acc, p, inv, R, lazy)
    return P


def gen_mont_mul2_sep(name, mod):
    """r = (a*b + c*d) / R mod p with a single reduction (a*b + c*d < 2 p^2 < p * 2^256)."""
    p = limbs(mod)
    inv = (-pow(mod, -1, 1 << 32)) & M32
    A = ["a%d" % i for i in range(NL)]
    B = ["b%d" % i for i in range(NL)]
    C = ["c%d" % i for i in range(NL)]
    D = ["d%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A + B + C + D, R)
    acc = WideAcc(P)
    product_rows(acc, A, B)
    product_rows(acc, C, D)
    redc_tail(P, acc, p, inv, R)
    return P




def gen_add(name, mod, lazy=False):
    p = limbs(2 * mod if lazy else mod)      # lazy: inputs and output in [0, 2p), correction by 2p
    A = ["a%d" % i for i in range(NL)]
    B = ["b%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A + B, R)
    t = [P.tmp("t%d" % i) for i in range(NL)]
    s = [P.tmp("s%d" % i) for i in range(NL)]
    bw = P.tmp("bw")
    for i in range(NL):
        P.emit("add.cc" if i == 0 else ("addc.cc" if i < NL - 1 else "addc"), t[i], A[i], B[i])
    for i in range(NL):
        P.emit("sub.cc" if i == 0 else "subc.cc", s[i], t[i], p[i])
    P.emit("subc", bw, 0, 0)
    for i in range(NL):
        P.emit("selnz", R[i], bw, t[i], s[i])
    return P


def gen_sub(name, mod, lazy=False):
    p = limbs(2 * mod if lazy else mod)
    A = ["a%d" % i for i in range(NL)]
    B = ["b%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A + B, R)
    t = [P.tmp("t%d" % i) for i in range(NL)]
    q = [P.tmp("q%d" % i) for i in range(NL)]
    bw = P.tmp("bw")
    for i in range(NL):
        P.emit("sub.cc" if i == 0 else "subc.cc", t[i], A[i], B[i])
    P.emit("subc", bw, 0, 0)            # all-ones iff a < b
    for i in range(NL):
        P.emit("and", q[i], bw, p[i])
    for i in range(NL):
        P.emit("add.cc" if i == 0 else ("addc.cc" if i < NL - 1 else "addc"), R[i], t[i], q[i])
    return P


def gen_canon(name, mod):
    """[0, 2p) -> [0, p): r = a - p if a >= p."""
    p = limbs(mod)
    A = ["a%d" % i for i in range(NL)]
    R = ["r%d" % i for i in range(NL)]
    P = Prog(name, A, R)
    s = [P.tmp("s%d" % i) for i in range(NL)]
    bw = P.tmp("bw")
    for i in range(NL):
        P.emit("sub.cc" if i == 0 else "subc.cc", s[i], A[i], p[i])
    P.emit("subc", bw, 0, 0)
    for i in range(NL):
        P.emit("selnz", R[i], bw, A[i], s[i])
    return P


# =====================================================================================
# verification
# =====================================================================================
def check(prog, mod, kind, trials=3000):
    rng = random.Random(0xB200 + mod % 9973 + len(prog.ins))
    Rinv = pow(1 << 256, -1, mod)
    edge = [0, 1, 2, mod - 1, mod - 2, (1 << 256) % mod, (1 << 255) % mod, (mod - 1) // 2, (mod + 1) // 2,
            0xFFFFFFFF, 0xFFFFFFFF00000000, (1 << 224) - 1, mod - 0xFFFFFFFF]
    cases = [(x, y) for x in edge for y in edge]
    cases += [(rng.randrange(mod), rng.randrange(mod)) for _ in range(trials)]
    # values with long runs of one-bits in every limb position (carry propagation across accumulator tops)
    for sh in range(0, 256, 16):
        v1 = ((1 << 256) - 1 - ((1 << sh) - 1)) % mod
        v2 = ((1 << sh) - 1) % mod
        cases += [(v1, v1), (v1, v2), (v2, v2), (mod - 1 - v2 if v2 < mod else 0, v1)]
    for idx, (x, y) in enumerate(cases):
        env = {}
        for i, l in enumerate(limbs(x)):
            env["a%d" % i] = l
        for i, l in enumerate(limbs(y)):
            env["b%d" % i] = l
        z, w = 0, 0
        if kind == "mul2":
            z, w = cases[(idx * 7 + 3) % len(cases)]
            if idx % 5 == 0:
                z, w = mod - 1, mod - 1
            for i, l in enumerate(limbs(z)):
                env["c%d" % i] = l
            for i, l in enumerate(limbs(w)):
                env["d%d" % i] = l
        env["z0"] = 0
        out = prog.run(env)
        got = sum(v << (32 * i) for i, v in enumerate(out))
        if kind == "mul":
            want = x * y * Rinv % mod
        elif kind == "mul2":
            want = (x * y + z * w) * Rinv % mod
        elif kind == "sqr":
            want = x * x * Rinv % mod
        elif kind == "add":
            want = (x + y) % mod
        elif kind == "sub":
            want = (x - y) % mod
        if got != want:
            raise SystemExit("FAIL %s: x=%x y=%x got=%x want=%x" % (prog.name, x, y, got, want))
    return len(cases)


def check_lazy(prog, mod, kind, trials=3000):
    """Lazily reduced operations: operands in [0, 2p).  Checks the
    congruence, the output bound and, for products, the exact value: (a*b + M*p) / 2^256 with M = -a*b/p mod 2^256
    is the unique Montgomery value before a final subtraction, so every other implementation must give these bits."""
    rng = random.Random(0x1A2B + mod % 9973 + len(prog.ins))
    R = 1 << 256
    Rinv = pow(R, -1, mod)
    pinv = pow(mod, -1, R)
    two_p = 2 * mod
    edge = [0, 1, 2, mod - 1, mod, mod + 1, two_p - 1, two_p - 2, R % mod, mod + R % mod, (mod - 1) // 2, (mod + 1) // 2,
            0xFFFFFFFF, 0xFFFFFFFF00000000, (1 << 224) - 1, mod - 0xFFFFFFFF, mod + 0xFFFFFFFF, two_p - 0xFFFFFFFF]
    for sh in range(0, 256, 16):                     # long runs of one-bits at every limb position
        edge += [((1 << 256) - 1 - ((1 << sh) - 1)) % two_p, ((1 << sh) - 1) % two_p]
    cases = [(x, y) for x in edge for y in edge]
    cases += [(rng.randrange(two_p), rng.randrange(two_p)) for _ in range(trials)]
    for x, y in cases:
        if kind == "sqr":
            y = x
        env = {"z0": 0}
        for i, l in enumerate(limbs(x)):
            env["a%d" % i] = l
        for i, l in enumerate(limbs(y)):
            env["b%d" % i] = l
        got = sum(v << (32 * i) for i, v in enumerate(prog.run(env)))
        if kind in ("mul", "sqr"):
            ok = got == (x * y + (-x * y * pinv % R) * mod) // R and got < two_p and got % mod == x * y * Rinv % mod
        elif kind == "add":
            ok = got < two_p and got % mod == (x + y) % mod
        elif kind == "sub":
            ok = got < two_p and got % mod == (x - y) % mod
        elif kind == "canon":
            ok = got == x % mod
        if not ok:
            raise SystemExit("FAIL %s: x=%x y=%x got=%x" % (prog.name, x, y, got))
    return len(cases)


def main():
    out_path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "halo2_scaffold_b200", "csrc", "field_asm.inc")
    chunks = [
        "// GENERATED by tools/gen_field_ptx.py -- do not edit. Every instruction stream below was\n"
        "// executed by the generator's PTX interpreter and checked against big-int arithmetic.\n"
        "// 8 x 32-bit little-endian limbs, Montgomery R = 2^256, canonical (fully reduced) in/out.\n\n"
    ]
    total = 0
    for tag, mod in (("fr", FR), ("fq", FQ)):
        for kind, gen in (("mul", gen_mont_mul), ("sqr", gen_mont_sqr_sep), ("mul2", gen_mont_mul2_sep),
                          ("add", gen_add), ("sub", gen_sub)):
            prog = gen("%s_%s" % (tag, kind), mod)
            total += check(prog, mod, kind)
            if kind == "mul2":
                sig = ("__device__ __forceinline__ void %s_%s_asm(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8], "
                       "const uint32_t (&c)[8], const uint32_t (&d)[8])" % (tag, kind))
            elif kind == "sqr":
                sig = "__device__ __forceinline__ void %s_%s_asm(uint32_t (&r)[8], const uint32_t (&a)[8])" % (tag, kind)
            else:
                sig = "__device__ __forceinline__ void %s_%s_asm(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8])" % (tag, kind)
            chunks.append("// %s: %d PTX instructions\n" % (prog.name, len(prog.ins)))
            chunks.append(prog.to_cuda(sig))
            chunks.append("\n")
    chunks.append("// Lazily reduced operations: operands and results in [0, 2p) (canon: result in [0, p)).\n"
                  "// BN254's p and r are below 2^256 / 5.29, so a Montgomery product of two values < 2p is already < 2p\n"
                  "// without the final conditional subtraction.\n\n")
    for tag, mod in (("fr", FR), ("fq", FQ)):
        for kind, gen in (("mul", lambda n, m: gen_mont_mul(n, m, lazy=True)), ("sqr", lambda n, m: gen_mont_sqr_sep(n, m, lazy=True)),
                          ("add", lambda n, m: gen_add(n, m, lazy=True)), ("sub", lambda n, m: gen_sub(n, m, lazy=True)),
                          ("canon", gen_canon)):
            name = "%s_%s" % (tag, kind) if kind == "canon" else "%s_%s_lazy" % (tag, kind)
            prog = gen(name, mod)
            total += check_lazy(prog, mod, kind)
            if kind in ("sqr", "canon"):
                sig = "__device__ __forceinline__ void %s_asm(uint32_t (&r)[8], const uint32_t (&a)[8])" % name
            else:
                sig = "__device__ __forceinline__ void %s_asm(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8])" % name
            chunks.append("// %s: %d PTX instructions\n" % (prog.name, len(prog.ins)))
            chunks.append(prog.to_cuda(sig))
            chunks.append("\n")
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        f.write("".join(chunks))
    print("verified %d cases; wrote %s" % (total, os.path.normpath(out_path)))


if __name__ == "__main__":
    main()
