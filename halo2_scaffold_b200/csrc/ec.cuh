// BN254 G1 (y^2 = x^3 + 3 over Fq) group law for the MSM kernels.
//
// Bucket sums are kept in extended-Jacobian "XYZZ" coordinates (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2):
// the mixed addition of an affine SRS point costs 8M + 2S with no inversion. The identity is
// ZZ = 0.  Affine inputs follow halo2curves' G1Affine layout (x|y Montgomery, (0,0) = identity,
// [UP] halo2curves 0.3.x src/derive/curve.rs; SURVEY.md section 8 "Sizes").  Every routine is
// complete: P + P, P + (-P) and identity operands are handled, because real witness columns make
// equal points meet in a bucket (duplicate bases, repeated small scalars).
#pragma once
#include "field.cuh"

namespace h2b {

struct Affine {
    Fq x, y;
};
struct XYZZ {
    Fq x, y, zz, zzz;
};

__device__ __forceinline__ bool affine_is_identity(const Affine& p) { return fp_is_zero(p.x) && fp_is_zero(p.y); }
__device__ __forceinline__ bool xyzz_is_identity(const XYZZ& p) { return fp_is_zero(p.zz); }
__device__ __forceinline__ XYZZ xyzz_identity() {
    XYZZ r;
    r.x = fp_zero<FQ>(); r.y = fp_zero<FQ>(); r.zz = fp_zero<FQ>(); r.zzz = fp_zero<FQ>();
    return r;
}
__device__ __forceinline__ Affine affine_load(const void* p) {
    Affine a;
    a.x = fp_load<FQ>(p);
    a.y = fp_load<FQ>(reinterpret_cast<const uint4*>(p) + 2);
    return a;
}
__device__ __forceinline__ void affine_store(void* p, const Affine& a) {
    fp_store<FQ>(p, a.x);
    fp_store<FQ>(reinterpret_cast<uint4*>(p) + 2, a.y);
}
__device__ __forceinline__ XYZZ xyzz_load(const void* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    XYZZ r;
    r.x = fp_load<FQ>(q); r.y = fp_load<FQ>(q + 2); r.zz = fp_load<FQ>(q + 4); r.zzz = fp_load<FQ>(q + 6);
    return r;
}
__device__ __forceinline__ void xyzz_store(void* p, const XYZZ& v) {
    uint4* q = reinterpret_cast<uint4*>(p);
    fp_store<FQ>(q, v.x); fp_store<FQ>(q + 2, v.y); fp_store<FQ>(q + 4, v.zz); fp_store<FQ>(q + 6, v.zzz);
}
__device__ __forceinline__ XYZZ xyzz_from_affine(const Affine& p) {
    XYZZ r;
    if (affine_is_identity(p)) return xyzz_identity();
    r.x = p.x; r.y = p.y; r.zz = fp_one<FQ>(); r.zzz = fp_one<FQ>();
    return r;
}

// 2 * (affine point), result in XYZZ  (EFD mdbl-2008-s-1, a = 0)
__device__ __forceinline__ XYZZ xyzz_double_affine(const Affine& p) {
    XYZZ r;
    Fq u = fp_dbl(p.y);
    Fq v = fp_sqr(u);
    Fq w = fp_mul(u, v);
    Fq s = fp_mul(p.x, v);
    Fq xx = fp_sqr(p.x);
    Fq m = fp_add(fp_dbl(xx), xx);
    r.x = fp_sub(fp_sqr(m), fp_dbl(s));
    r.y = fp_sub(fp_mul(m, fp_sub(s, r.x)), fp_mul(w, p.y));
    r.zz = v;
    r.zzz = w;
    return r;
}

// One shared, NON-inlined copy of the Fq multiplier for the kernels that run a few warps through long chains of dependent group
// additions (bucket reduction, combine of cut buckets, final Horner).  With every multiplication expanded in line an addition is
// ~4000 straight-line instructions and those warps stall on instruction fetch as often as on the arithmetic itself (ncu of
// msm_reduce_level_kernel: "no instruction" 3.1 and fixed-latency wait 3.2 cycles per issue, 0.19 IPC at 1.7 warps per scheduler).
// (A product-scanning C version with 64 independent addend-free products -- 560 instructions instead of 216, no carry chain through
// the products -- was tried here for its instruction-level parallelism: a lone warp issued it at 5.5 instead of 9 clocks per
// instruction, but 2.6x as many: reduction 0.91 -> 1.41 ms.  profiles/r02_shared_multiplier_latency_kernels.jsonl.)
static __device__ __noinline__ Fq fq_mul_shared(Fq a, Fq b) { return fp_mul(a, b); }
template <bool SHARED> __device__ __forceinline__ Fq fq_m(const Fq& a, const Fq& b) {
    if (SHARED) return fq_mul_shared(a, b);
    return fp_mul(a, b);
}
template <bool SHARED> __device__ __forceinline__ Fq fq_s(const Fq& a) {
    if (SHARED) return fq_mul_shared(a, a);
    return fp_sqr(a);
}

// 2 * P in XYZZ  (EFD dbl-2008-s-1, a = 0).  y = 0 never happens on this curve (odd order).
template <bool SHARED = false>
__device__ __forceinline__ XYZZ xyzz_double(const XYZZ& p) {
    if (xyzz_is_identity(p)) return p;
    XYZZ r;
    Fq u = fp_dbl(p.y);
    Fq v = fq_s<SHARED>(u);
    Fq w = fq_m<SHARED>(u, v);
    Fq s = fq_m<SHARED>(p.x, v);
    Fq xx = fq_s<SHARED>(p.x);
    Fq m = fp_add(fp_dbl(xx), xx);
    r.x = fp_sub(fq_s<SHARED>(m), fp_dbl(s));
    r.y = fp_sub(fq_m<SHARED>(m, fp_sub(s, r.x)), fq_m<SHARED>(w, p.y));
    r.zz = fq_m<SHARED>(v, p.zz);
    r.zzz = fq_m<SHARED>(w, p.zzz);
    return r;
}

// acc += (neg ? -q : q), q affine  (EFD madd-2008-s: 8M + 2S)
__device__ __forceinline__ void xyzz_add_affine(XYZZ& acc, const Affine& q_in, bool neg) {
    if (affine_is_identity(q_in)) return;
    Affine q = q_in;
    if (neg) q.y = fp_neg(q.y);
    if (xyzz_is_identity(acc)) {
        acc.x = q.x; acc.y = q.y; acc.zz = fp_one<FQ>(); acc.zzz = fp_one<FQ>();
        return;
    }
    Fq u2 = fp_mul(q.x, acc.zz);
    Fq s2 = fp_mul(q.y, acc.zzz);
    Fq p = fp_sub(u2, acc.x);
    Fq r = fp_sub(s2, acc.y);
    if (fp_is_zero(p)) {
        if (fp_is_zero(r)) acc = xyzz_double_affine(q);
        else acc = xyzz_identity();
        return;
    }
    Fq pp = fp_sqr(p);
    Fq ppp = fp_mul(p, pp);
    Fq qq = fp_mul(acc.x, pp);
    Fq x3 = fp_sub(fp_sub(fp_sqr(r), ppp), fp_dbl(qq));
    // Y3 = R*(Q - X3) - Y1*PPP.  fp_mul2 (two products, one Montgomery reduction) saves 72 of this addition's 1260
    // FMA-pipe instructions, but measured 2 % SLOWER here (profiles/r01_field_primitives.jsonl): at the 16 warps per
    // SM this kernel's 126 registers allow, the longer dependency chains of the separated product/reduction form
    // cost more than the saved dispatch cycles.  Kept behind a switch for kernels with more resident warps.
#ifdef H2B_MADD_MUL2
    Fq y3 = fp_mul2(r, fp_sub(qq, x3), fp_neg(acc.y), ppp);
#else
    Fq y3 = fp_sub(fp_mul(r, fp_sub(qq, x3)), fp_mul(acc.y, ppp));
#endif
    acc.x = x3;
    acc.y = y3;
    acc.zz = fp_mul(acc.zz, pp);
    acc.zzz = fp_mul(acc.zzz, ppp);
}

// The same mixed addition on a lazily reduced accumulator (every coordinate in [0, 2p), see field.cuh); q is canonical.
// It drops the final conditional subtraction of all ten products (17 ALU instructions each).  The
// exceptional cases are tested modulo p: P == 0 or P == p.  ZZ of a non-identity accumulator is never 0 mod p, so the
// identity test on ZZ == 0 stays exact.  Pass the result through xyzz_canon before it is stored.
__device__ __forceinline__ void xyzz_add_affine_lazy(XYZZ& acc, const Affine& q_in, bool neg) {
    if (affine_is_identity(q_in)) return;
    Affine q = q_in;
    if (neg) q.y = fp_neg(q.y);
    if (xyzz_is_identity(acc)) {
        acc.x = q.x; acc.y = q.y; acc.zz = fp_one<FQ>(); acc.zzz = fp_one<FQ>();
        return;
    }
    Fq u2 = fp_mul_lazy(q.x, acc.zz);
    Fq s2 = fp_mul_lazy(q.y, acc.zzz);
    Fq p = fp_sub_lazy(u2, acc.x);
    Fq r = fp_sub_lazy(s2, acc.y);
    if (fp_is_zero_lazy(p)) {
        if (fp_is_zero_lazy(r)) acc = xyzz_double_affine(q);
        else acc = xyzz_identity();
        return;
    }
    Fq pp = fp_sqr_lazy(p);
    Fq ppp = fp_mul_lazy(p, pp);
    Fq qq = fp_mul_lazy(acc.x, pp);
    Fq yppp = fp_mul_lazy(acc.y, ppp);      // before X3: in the order of xyzz_add_affine this kernel spills at 128 registers
    Fq x3 = fp_sub_lazy(fp_sub_lazy(fp_sqr_lazy(r), ppp), fp_add_lazy(qq, qq));
    Fq y3 = fp_sub_lazy(fp_mul_lazy(r, fp_sub_lazy(qq, x3)), yppp);
    acc.x = x3;
    acc.y = y3;
    acc.zz = fp_mul_lazy(acc.zz, pp);
    acc.zzz = fp_mul_lazy(acc.zzz, ppp);
}
__device__ __forceinline__ XYZZ xyzz_canon(const XYZZ& a) {
    XYZZ r;
    r.x = fp_canon(a.x); r.y = fp_canon(a.y); r.zz = fp_canon(a.zz); r.zzz = fp_canon(a.zzz);
    return r;
}

// acc += b, both XYZZ  (EFD add-2008-s: 12M + 2S)
template <bool SHARED> __device__ __forceinline__ void xyzz_add_body(XYZZ& acc, const XYZZ& b);
// ONE copy of the general addition for the latency-bound kernels: with the addition inlined at every call site the loop of
// msm_reduce_level_kernel (three additions + a doubling) is 34 KB of straight-line code, more than the 32 KB L1.5 instruction
// cache, and a lone warp waits for instruction fetch on everything but the shared multiplier
static __device__ __noinline__ XYZZ xyzz_add_shared(XYZZ acc, XYZZ b) {
    xyzz_add_body<true>(acc, b);
    return acc;
}
template <bool SHARED = false>
__device__ __forceinline__ void xyzz_add(XYZZ& acc, const XYZZ& b) {
    if (SHARED) acc = xyzz_add_shared(acc, b);
    else xyzz_add_body<false>(acc, b);
}
template <bool SHARED>
__device__ __forceinline__ void xyzz_add_body(XYZZ& acc, const XYZZ& b) {
    if (xyzz_is_identity(b)) return;
    if (xyzz_is_identity(acc)) { acc = b; return; }
    Fq u1 = fq_m<SHARED>(acc.x, b.zz);
    Fq u2 = fq_m<SHARED>(b.x, acc.zz);
    Fq s1 = fq_m<SHARED>(acc.y, b.zzz);
    Fq s2 = fq_m<SHARED>(b.y, acc.zzz);
    Fq p = fp_sub(u2, u1);
    Fq r = fp_sub(s2, s1);
    if (fp_is_zero(p)) {
        if (fp_is_zero(r)) acc = xyzz_double<SHARED>(acc);
        else acc = xyzz_identity();
        return;
    }
    Fq pp = fq_s<SHARED>(p);
    Fq ppp = fq_m<SHARED>(p, pp);
    Fq qq = fq_m<SHARED>(u1, pp);
    Fq x3 = fp_sub(fp_sub(fq_s<SHARED>(r), ppp), fp_dbl(qq));
    Fq y3 = fp_sub(fq_m<SHARED>(r, fp_sub(qq, x3)), fq_m<SHARED>(s1, ppp));
    acc.x = x3;
    acc.y = y3;
    acc.zz = fq_m<SHARED>(fq_m<SHARED>(acc.zz, b.zz), pp);
    acc.zzz = fq_m<SHARED>(fq_m<SHARED>(acc.zzz, b.zzz), ppp);
}

// [e] P for a canonical (non-Montgomery) e < 2^254 and any P, the variable-base multiplication of the G1 NTT (g1gen.cu).
// Left to right over Booth (signed radix-2^W) digits d_j = ((x + 1) >> 1) - 2^W (x >> W) in [-2^(W-1), 2^(W-1)], x the W + 1
// bits [jW - 1, jW + W - 1] of e (bit -1 = 0): each digit is read straight off the scalar, with no carry from the digits
// below, so the loop consumes them top down.  A per-thread table T[m - 1] = m P, m = 1 .. 2^(W-1); per window W doublings
// and one complete general addition of +-T[|d| - 1].  W = H2B_G1_MUL_WINDOW is chosen by measurement (DESIGN.md 5.8).
#ifndef H2B_G1_MUL_WINDOW
#define H2B_G1_MUL_WINDOW 4
#endif
static const int G1_MUL_W = H2B_G1_MUL_WINDOW;
static const int G1_MUL_WINDOWS = (255 + G1_MUL_W - 1) / G1_MUL_W;     // W * windows >= 255: the top digit is never negative
static_assert(G1_MUL_W >= 1 && G1_MUL_W <= 6, "variable-base window out of range");

__device__ __forceinline__ XYZZ xyzz_mul_scalar(const XYZZ& p, const Fp<FR>& e) {
    const int TAB = 1 << (G1_MUL_W - 1);
    XYZZ tab[TAB];
    tab[0] = p;
    if (TAB > 1) tab[1] = xyzz_double(p);
#pragma unroll 1
    for (int m = 2; m < TAB; ++m) { tab[m] = tab[m - 1]; xyzz_add(tab[m], p); }
    // z = 2 e in 9 words; after t windows it is shifted left by t W, so the field of the current window is always at bit TOP
    uint32_t z[9];
    z[0] = e.l[0] << 1;
#pragma unroll
    for (int i = 1; i < 8; ++i) z[i] = __funnelshift_l(e.l[i - 1], e.l[i], 1);
    z[8] = e.l[7] >> 31;
    const int TOP = G1_MUL_W * (G1_MUL_WINDOWS - 1), TW = TOP / 32, TS = TOP % 32;
    XYZZ acc = xyzz_identity();
#pragma unroll 1
    for (int t = 0; t < G1_MUL_WINDOWS; ++t) {
        if (t) {
#pragma unroll
            for (int b = 0; b < G1_MUL_W; ++b) acc = xyzz_double(acc);
        }
        const uint32_t x = __funnelshift_r(z[TW], z[TW + 1], TS) & ((2u << G1_MUL_W) - 1);
#pragma unroll
        for (int i = 8; i > 0; --i) z[i] = __funnelshift_l(z[i - 1], z[i], G1_MUL_W);
        z[0] <<= G1_MUL_W;
        const int d = (int)((x + 1) >> 1) - (int)((x >> G1_MUL_W) << G1_MUL_W);
        if (d != 0) {
            XYZZ q = tab[(d < 0 ? -d : d) - 1];
            if (d < 0) q.y = fp_neg(q.y);
            xyzz_add(acc, q);
        }
    }
    return acc;
}

// XYZZ -> a Jacobian representative (X', Y', Z') of the same point without an inversion:
// Z' = ZZ*ZZZ, X' = X*ZZ*ZZZ^2, Y' = Y*ZZ^3*ZZZ^2  (then X'/Z'^2 = X/ZZ and Y'/Z'^3 = Y/ZZZ).
// Identity -> (0, 1, 0), matching halo2curves' G1::identity().
__device__ __forceinline__ void xyzz_to_jacobian(const XYZZ& p, Fq& X, Fq& Y, Fq& Z) {
    if (xyzz_is_identity(p)) { X = fp_zero<FQ>(); Y = fp_one<FQ>(); Z = fp_zero<FQ>(); return; }
    Fq zzz2 = fp_sqr(p.zzz);
    Fq t = fp_mul(p.zz, zzz2);          // ZZ * ZZZ^2
    X = fp_mul(p.x, t);
    Y = fp_mul(fp_mul(p.y, fp_sqr(p.zz)), t);
    Z = fp_mul(p.zz, p.zzz);
}

// XYZZ -> affine (one field inversion; used for a handful of points only)
__device__ __forceinline__ Affine xyzz_to_affine(const XYZZ& p) {
    Affine a;
    if (xyzz_is_identity(p)) { a.x = fp_zero<FQ>(); a.y = fp_zero<FQ>(); return a; }
    Fq zi = fp_inv(fp_mul(p.zz, p.zzz));     // 1/(ZZ*ZZZ)
    a.x = fp_mul(p.x, fp_mul(p.zzz, zi));    // X/ZZ
    a.y = fp_mul(p.y, fp_mul(p.zz, zi));     // Y/ZZZ
    return a;
}

}  // namespace h2b
