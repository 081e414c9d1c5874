// BN254 Fr / Fq arithmetic for sm_100a: 8 x 32-bit limbs, Montgomery form with R = 2^256, values
// always fully reduced -- the same representation halo2curves keeps in its 4 x u64 limbs
// ([UP] halo2curves 0.3.x src/bn256/{fr,fq}.rs; SURVEY.md section 8 "Sizes"), so arrays of Rust
// `Fr`/`Fq` can be copied to the device byte-for-byte.
//
// The multiply/add/sub bodies are the generated IMAD.WIDE carry chains in field_asm.inc
// (tools/gen_field_ptx.py, which also proves them against big-int arithmetic).
//
// The *_lazy operations keep values in [0, 2p) instead: BN254's p and r are below 2^256 / 5.29, so a Montgomery
// product of two values < 2p is (ab + Mp) / 2^256 < 1.76p and needs no final conditional subtraction, and sums and
// differences are corrected by 2p.  Loops that chain many products (the MSM bucket accumulation, the NTT butterflies)
// run on them and call fp_canon before a value leaves the loop; everything stored in memory stays canonical.
#pragma once
#include <cstdint>

#ifdef H2B_EMU
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#define H2B_LAUNCH(kern, grid, block, smem, stream, ...) \
    (h2b::count_launch(), kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__))
#define H2B_DYN_SMEM(T, name)                                   \
    extern __shared__ __align__(16) unsigned char _h2b_dsm[];   \
    T* name = reinterpret_cast<T*>(_h2b_dsm)
#include "field_asm.inc"
#endif

namespace h2b {

// number of kernels this library has launched (reported by bench.py as `gpu_launches`)
extern unsigned long long g_launch_count;
inline void count_launch() { __atomic_fetch_add(&g_launch_count, 1ull, __ATOMIC_RELAXED); }

enum FieldId { FR = 0, FQ = 1 };

template <int F> struct FpParams;
template <> struct FpParams<FR> {
    __host__ __device__ static constexpr uint32_t P(int i) {
        constexpr uint32_t t[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return t[i];
    }
    __host__ __device__ static constexpr uint32_t ONE(int i) {
        constexpr uint32_t t[8] = {0x4ffffffbu, 0xac96341cu, 0x9f60cd29u, 0x36fc7695u, 0x7879462eu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return t[i];
    }
    __host__ __device__ static constexpr uint32_t R2(int i) {
        constexpr uint32_t t[8] = {0xae216da7u, 0x1bb8e645u, 0xe35c59e3u, 0x53fe3ab1u, 0x53bb8085u, 0x8c49833du, 0x7f4e44a5u, 0x0216d0b1u};
        return t[i];
    }
    static constexpr uint32_t INV = 0xefffffffu;
};
template <> struct FpParams<FQ> {
    __host__ __device__ static constexpr uint32_t P(int i) {
        constexpr uint32_t t[8] = {0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return t[i];
    }
    __host__ __device__ static constexpr uint32_t ONE(int i) {
        constexpr uint32_t t[8] = {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return t[i];
    }
    __host__ __device__ static constexpr uint32_t R2(int i) {
        constexpr uint32_t t[8] = {0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u};
        return t[i];
    }
    static constexpr uint32_t INV = 0xe4866389u;
};

template <int F>
struct Fp {
    uint32_t l[8];
};
typedef Fp<FR> Fr;
typedef Fp<FQ> Fq;

template <int F> __device__ __forceinline__ Fp<F> fp_zero() {
    Fp<F> r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.l[i] = 0;
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_one() {
    Fp<F> r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.l[i] = FpParams<F>::ONE(i);
    return r;
}
template <int F> __device__ __forceinline__ bool fp_is_zero(const Fp<F>& a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a.l[i];
    return o == 0;
}
template <int F> __device__ __forceinline__ bool fp_eq(const Fp<F>& a, const Fp<F>& b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a.l[i] ^ b.l[i];
    return o == 0;
}

// 32-byte element <-> two 128-bit accesses
template <int F> __device__ __forceinline__ Fp<F> fp_load(const void* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    Fp<F> r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
    r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
template <int F> __device__ __forceinline__ void fp_store(void* p, const Fp<F>& v) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    q[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

#ifndef H2B_EMU
template <int F> __device__ __forceinline__ Fp<F> fp_mul(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_mul_asm(r.l, a.l, b.l); else fq_mul_asm(r.l, a.l, b.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_sqr(const Fp<F>& a) {
#ifdef H2B_SQR_AS_MUL
    return fp_mul(a, a);
#else
    Fp<F> r;
    if (F == FR) fr_sqr_asm(r.l, a.l); else fq_sqr_asm(r.l, a.l);
    return r;
#endif
}
// a*b + c*d with a single Montgomery reduction (a*b + c*d < 2 p^2 < p * 2^256)
template <int F> __device__ __forceinline__ Fp<F> fp_mul2(const Fp<F>& a, const Fp<F>& b, const Fp<F>& c, const Fp<F>& d) {
    Fp<F> r;
    if (F == FR) fr_mul2_asm(r.l, a.l, b.l, c.l, d.l); else fq_mul2_asm(r.l, a.l, b.l, c.l, d.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_add(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_add_asm(r.l, a.l, b.l); else fq_add_asm(r.l, a.l, b.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_sub(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_sub_asm(r.l, a.l, b.l); else fq_sub_asm(r.l, a.l, b.l);
    return r;
}
// lazily reduced: a, b < 2p -> result < 2p; products are the Montgomery value before the final subtraction
template <int F> __device__ __forceinline__ Fp<F> fp_mul_lazy(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_mul_lazy_asm(r.l, a.l, b.l); else fq_mul_lazy_asm(r.l, a.l, b.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_sqr_lazy(const Fp<F>& a) {
#ifdef H2B_SQR_AS_MUL
    return fp_mul_lazy(a, a);
#else
    Fp<F> r;
    if (F == FR) fr_sqr_lazy_asm(r.l, a.l); else fq_sqr_lazy_asm(r.l, a.l);
    return r;
#endif
}
// a*b + c*d with one Montgomery reduction: a, c < 2p, b, d CANONICAL (< p) -> result < 2p.  With b or d lazy the sum of
// the products can exceed p * 2^256 and the result 2p.
template <int F> __device__ __forceinline__ Fp<F> fp_mul2_lazy(const Fp<F>& a, const Fp<F>& b, const Fp<F>& c, const Fp<F>& d) {
    Fp<F> r;
    if (F == FR) fr_mul2_lazy_asm(r.l, a.l, b.l, c.l, d.l); else fq_mul2_lazy_asm(r.l, a.l, b.l, c.l, d.l);
    return r;
}
// p - a for a in [0, p]: a canonical negation whose result is p, not 0, for a == 0
template <int F> __device__ __forceinline__ Fp<F> fp_neg_lazy(const Fp<F>& a) {
    Fp<F> r;
    if (F == FR) fr_neg_lazy_asm(r.l, a.l); else fq_neg_lazy_asm(r.l, a.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_add_lazy(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_add_lazy_asm(r.l, a.l, b.l); else fq_add_lazy_asm(r.l, a.l, b.l);
    return r;
}
template <int F> __device__ __forceinline__ Fp<F> fp_sub_lazy(const Fp<F>& a, const Fp<F>& b) {
    Fp<F> r;
    if (F == FR) fr_sub_lazy_asm(r.l, a.l, b.l); else fq_sub_lazy_asm(r.l, a.l, b.l);
    return r;
}
// [0, 2p) -> [0, p)
template <int F> __device__ __forceinline__ Fp<F> fp_canon(const Fp<F>& a) {
    Fp<F> r;
    if (F == FR) fr_canon_asm(r.l, a.l); else fq_canon_asm(r.l, a.l);
    return r;
}
#else
// portable bodies for the kernel-logic emulator (tools/emu); same contract, canonical in/out
template <int F> inline bool fp_geq_p(const uint32_t* t) {
    for (int i = 7; i >= 0; --i) {
        if (t[i] > FpParams<F>::P(i)) return true;
        if (t[i] < FpParams<F>::P(i)) return false;
    }
    return true;
}
template <int F> inline void fp_sub_p(uint32_t* t) {
    int64_t bw = 0;
    for (int i = 0; i < 8; ++i) {
        int64_t d = (int64_t)t[i] - FpParams<F>::P(i) + bw;
        t[i] = (uint32_t)d;
        bw = d >> 32;
    }
}
// Montgomery product without the final subtraction: t[0..8] = (ab + Mp) / 2^256 (with c, d: (ab + cd + Mp) / 2^256)
template <int F> inline void fp_mont_emu(const Fp<F>& a, const Fp<F>& b, uint32_t (&t)[10], const Fp<F>* c2 = nullptr, const Fp<F>* d2 = nullptr) {
    for (int i = 0; i < 8; ++i) {
        for (int k = 0; k < (c2 ? 2 : 1); ++k) {
            const Fp<F>& x = k ? *c2 : a;
            const uint32_t y = k ? d2->l[i] : b.l[i];
            uint64_t c = 0;
            for (int j = 0; j < 8; ++j) { c += (uint64_t)x.l[j] * y + t[j]; t[j] = (uint32_t)c; c >>= 32; }
            c += t[8]; t[8] = (uint32_t)c; t[9] += (uint32_t)(c >> 32);
        }
        uint32_t m = t[0] * FpParams<F>::INV;
        uint64_t c = (uint64_t)m * FpParams<F>::P(0) + t[0]; c >>= 32;
        for (int j = 1; j < 8; ++j) { c += (uint64_t)m * FpParams<F>::P(j) + t[j]; t[j - 1] = (uint32_t)c; c >>= 32; }
        c += t[8]; t[7] = (uint32_t)c; t[8] = t[9] + (uint32_t)(c >> 32); t[9] = 0;
    }
}
template <int F> inline Fp<F> fp_mul(const Fp<F>& a, const Fp<F>& b) {
    uint32_t t[10] = {0};
    fp_mont_emu(a, b, t);
    Fp<F> r;
    if (t[8] || fp_geq_p<F>(t)) fp_sub_p<F>(t);
    for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
template <int F> inline Fp<F> fp_sqr(const Fp<F>& a) { return fp_mul(a, a); }
template <int F> inline Fp<F> fp_add(const Fp<F>& a, const Fp<F>& b);
template <int F> inline Fp<F> fp_mul2(const Fp<F>& a, const Fp<F>& b, const Fp<F>& c, const Fp<F>& d) { return fp_add(fp_mul(a, b), fp_mul(c, d)); }
template <int F> inline Fp<F> fp_add(const Fp<F>& a, const Fp<F>& b) {
    uint32_t t[8]; uint64_t c = 0;
    for (int i = 0; i < 8; ++i) { c += (uint64_t)a.l[i] + b.l[i]; t[i] = (uint32_t)c; c >>= 32; }
    if (fp_geq_p<F>(t)) fp_sub_p<F>(t);
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
template <int F> inline Fp<F> fp_sub(const Fp<F>& a, const Fp<F>& b) {
    uint32_t t[8]; int64_t bw = 0;
    for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)a.l[i] - b.l[i] + bw; t[i] = (uint32_t)d; bw = d >> 32; }
    if (bw) { uint64_t c = 0; for (int i = 0; i < 8; ++i) { c += (uint64_t)t[i] + FpParams<F>::P(i); t[i] = (uint32_t)c; c >>= 32; } }
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
// lazily reduced bodies: the same bits as the generated chains ((ab + Mp) / 2^256 is unique; sums and differences
// are corrected by 2p exactly when the chains correct them)
template <int F> inline void fp_2p(uint32_t (&q)[8]) {
    uint64_t c = 0;
    for (int i = 0; i < 8; ++i) { c += 2 * (uint64_t)FpParams<F>::P(i); q[i] = (uint32_t)c; c >>= 32; }
}
template <int F> inline Fp<F> fp_mul_lazy(const Fp<F>& a, const Fp<F>& b) {
    uint32_t t[10] = {0};
    fp_mont_emu(a, b, t);
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
template <int F> inline Fp<F> fp_sqr_lazy(const Fp<F>& a) { return fp_mul_lazy(a, a); }
template <int F> inline Fp<F> fp_mul2_lazy(const Fp<F>& a, const Fp<F>& b, const Fp<F>& c, const Fp<F>& d) {
    uint32_t t[10] = {0};
    fp_mont_emu(a, b, t, &c, &d);
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
template <int F> inline Fp<F> fp_neg_lazy(const Fp<F>& a) {
    Fp<F> r; int64_t bw = 0;
    for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)FpParams<F>::P(i) - a.l[i] + bw; r.l[i] = (uint32_t)d; bw = d >> 32; }
    return r;
}
template <int F> inline Fp<F> fp_add_lazy(const Fp<F>& a, const Fp<F>& b) {
    uint32_t q[8], t[8], s[8]; fp_2p<F>(q);
    uint64_t c = 0; int64_t bw = 0;
    for (int i = 0; i < 8; ++i) { c += (uint64_t)a.l[i] + b.l[i]; t[i] = (uint32_t)c; c >>= 32; }
    for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)t[i] - q[i] + bw; s[i] = (uint32_t)d; bw = d >> 32; }
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = bw ? t[i] : s[i];
    return r;
}
template <int F> inline Fp<F> fp_sub_lazy(const Fp<F>& a, const Fp<F>& b) {
    uint32_t q[8], t[8]; fp_2p<F>(q);
    int64_t bw = 0;
    for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)a.l[i] - b.l[i] + bw; t[i] = (uint32_t)d; bw = d >> 32; }
    if (bw) { uint64_t c = 0; for (int i = 0; i < 8; ++i) { c += (uint64_t)t[i] + q[i]; t[i] = (uint32_t)c; c >>= 32; } }
    Fp<F> r; for (int i = 0; i < 8; ++i) r.l[i] = t[i];
    return r;
}
template <int F> inline Fp<F> fp_canon(const Fp<F>& a) {
    Fp<F> r = a;
    if (fp_geq_p<F>(r.l)) fp_sub_p<F>(r.l);
    return r;
}
#endif

// x == 0 (mod p) for x in [0, 2p): x == 0 or x == p
template <int F> __device__ __forceinline__ bool fp_is_zero_lazy(const Fp<F>& a) {
    uint32_t o = 0, d = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o |= a.l[i]; d |= a.l[i] ^ FpParams<F>::P(i); }
    return o == 0 || d == 0;
}

template <int F> __device__ __forceinline__ Fp<F> fp_neg(const Fp<F>& a) { return fp_sub(fp_zero<F>(), a); }
template <int F> __device__ __forceinline__ Fp<F> fp_dbl(const Fp<F>& a) { return fp_add(a, a); }
// leave / enter Montgomery form
template <int F> __device__ __forceinline__ Fp<F> fp_from_mont(const Fp<F>& a) {
    Fp<F> o = fp_zero<F>();
    o.l[0] = 1;
    return fp_mul(a, o);
}
template <int F> __device__ __forceinline__ Fp<F> fp_to_mont(const Fp<F>& a) {
    Fp<F> r2;
#pragma unroll
    for (int i = 0; i < 8; ++i) r2.l[i] = FpParams<F>::R2(i);
    return fp_mul(a, r2);
}
// a^(p-2) (Fermat); 0 -> 0.  Only used off the hot path (normalising a handful of points).
template <int F> __device__ __noinline__ Fp<F> fp_inv(const Fp<F>& a) {
    Fp<F> r = fp_one<F>();
#pragma unroll
    for (int w = 7; w >= 0; --w) {
        uint32_t word = FpParams<F>::P(w);
        if (w == 0) word -= 2;       // exponent p - 2 (low limb of p is > 2, no borrow)
#pragma unroll 1
        for (int i = 31; i >= 0; --i) {
            r = fp_sqr(r);
            if ((word >> i) & 1) r = fp_mul(r, a);
        }
    }
    return r;
}

// base^e for a small exponent (row indices: omega^i), square-and-multiply from the low bit
template <int F> __device__ __noinline__ Fp<F> fp_pow_u32(Fp<F> base, uint32_t e) {
    Fp<F> r = fp_one<F>();
    while (e) {
        if (e & 1) r = fp_mul(r, base);
        base = fp_sqr(base);
        e >>= 1;
    }
    return r;
}

}  // namespace h2b
