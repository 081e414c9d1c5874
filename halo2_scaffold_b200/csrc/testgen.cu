// Synthetic inputs, device self-tests and integer-pipe micro-benchmarks.
//
// * gen_scalars (and gen_points, g1gen.cu) build the benchmark workload of SURVEY.md section 8(d) on the device
//   (valid distinct G1 points, uniform or witness-like Fr scalars) so that bench.py never needs the
//   CPU oracle to produce inputs.  The definitions match oracle/h2_oracle.cpp (orc_gen_points,
//   orc_random_fr) bit for bit, which the parity tests exploit.
// * field/ec self-tests expose single field / group operations through the C ABI for the parity
//   tests of the arithmetic layer.
// * imad_bench measures the achievable 32-bit multiply-add rate of the SMs: the denominator of the
//   MSM roofline (SURVEY.md section 8(d): "IMAD peak: to be measured on the box").
#include "common.h"
#include "ec.cuh"

namespace h2b {

// kind 0: uniform in [0, r): 512-bit SplitMix64 draw (big-endian word order) reduced mod r.
// kind 1: witness-like skew (SURVEY.md 8d): 50 % zero, 20 % one, 20 % uniform < 2^19, 10 % r - small.
__global__ void __launch_bounds__(256) gen_scalars_kernel(uint64_t seed, uint64_t first, uint32_t n, int kind, uint4* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t idx = first + i;
    Fr r = fp_zero<FR>();
    if (kind == 0) {
        Fr two64 = fp_zero<FR>();
        two64.l[2] = 1;
        two64 = fp_to_mont(two64);
        for (int w = 0; w < 8; ++w) {
            uint64_t v = splitmix64_at(seed, 8 * idx + w);
            Fr x = fp_zero<FR>();
            x.l[0] = (uint32_t)v;
            x.l[1] = (uint32_t)(v >> 32);
            r = fp_add(fp_mul(r, two64), fp_to_mont(x));
        }
    } else {
        uint64_t v = splitmix64_at(seed, 2 * idx), u = splitmix64_at(seed, 2 * idx + 1);
        uint32_t sel = (uint32_t)(v % 10);
        Fr x = fp_zero<FR>();
        if (sel < 5) { /* zero */ }
        else if (sel < 7) x.l[0] = 1;
        else if (sel < 9) x.l[0] = (uint32_t)(u & 0x7ffff);
        else x.l[0] = (uint32_t)(u & 0xffff) + 1;
        r = fp_to_mont(x);
        if (sel == 9) r = fp_neg(r);
    }
    fp_store<FR>(out + 2 * (size_t)i, r);
}

int gen_scalars_run(DeviceCtx& ctx, uint64_t seed, size_t n, int kind, void* d_out, cudaStream_t stream) {
    (void)ctx;
    if (kind != 0 && kind != 1) { set_error("gen_scalars: kind must be 0 (uniform) or 1 (witness-like)"); return H2B_ERR_BAD_ARGUMENT; }
    for (size_t done = 0; done < n; done += (size_t)1 << 24) {
        uint32_t m = (uint32_t)((n - done < ((size_t)1 << 24)) ? n - done : (size_t)1 << 24);
        H2B_LAUNCH(gen_scalars_kernel, (m + 255) / 256, 256, 0, stream, seed, (uint64_t)done, m, kind, (uint4*)d_out + 2 * done);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- O(n) checksum of an MSM over the synthetic points ----------------------------------------------------------------
// For P_i = [z_i] G (gen_points, stream `seed`):  sum_i s_i P_i = [ sum_i s_i z_i mod r ] G.  The dot product is field
// arithmetic only -- no group law, no buckets, no sorting -- so it checks a timed 2^24 .. 2^27-point MSM result against
// something that shares no code with the MSM (bench.py `verified`, tests at the full benchmark sizes).
__global__ void __launch_bounds__(256) checksum_partial_kernel(const uint4* __restrict__ scalars, uint64_t seed, uint64_t first, uint64_t n,
                                                             uint4* __restrict__ partial) {
    __shared__ uint4 sh[256 * 2];
    Fr acc = fp_zero<FR>();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t z = splitmix64_at(seed, first + i);
        Fr zf = fp_zero<FR>();
        zf.l[0] = (uint32_t)z;
        zf.l[1] = (uint32_t)(z >> 32);
        // s is held in Montgomery form (s R) and z is canonical: their Montgomery product (s R) z / R = s z is canonical
        acc = fp_add(acc, fp_mul(fp_load<FR>(scalars + 2 * i), zf));
    }
    fp_store<FR>(sh + 2 * threadIdx.x, acc);
    __syncthreads();
    for (uint32_t d = blockDim.x >> 1; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            acc = fp_add(acc, fp_load<FR>(sh + 2 * (threadIdx.x + d)));
            fp_store<FR>(sh + 2 * threadIdx.x, acc);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) fp_store<FR>(partial + 2 * (size_t)blockIdx.x, acc);
}
__global__ void __launch_bounds__(256) checksum_final_kernel(const uint4* __restrict__ partial, uint32_t count, uint4* __restrict__ out) {
    __shared__ uint4 sh[256 * 2];
    Fr acc = fp_zero<FR>();
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) acc = fp_add(acc, fp_load<FR>(partial + 2 * (size_t)i));
    fp_store<FR>(sh + 2 * threadIdx.x, acc);
    __syncthreads();
    for (uint32_t d = blockDim.x >> 1; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            acc = fp_add(acc, fp_load<FR>(sh + 2 * (threadIdx.x + d)));
            fp_store<FR>(sh + 2 * threadIdx.x, acc);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) fp_store<FR>(out, acc);
}
// d_out: one Fr (32 B), CANONICAL (not Montgomery) value of sum_i s_i z_i mod r, i over [0, n), z from stream `seed` at first + i
int msm_checksum_run(DeviceCtx& ctx, const void* d_scalars, uint64_t seed, uint64_t first, size_t n, void* d_out, cudaStream_t stream) {
    const uint32_t blocks = (uint32_t)ctx.sm_count * 8;
    H2B_TRY(ctx.scan_scratch.reserve((size_t)blocks * 32));
    H2B_LAUNCH(checksum_partial_kernel, blocks, 256, 0, stream, (const uint4*)d_scalars, seed, first, (uint64_t)n, (uint4*)ctx.scan_scratch.p);
    H2B_LAUNCH(checksum_final_kernel, 1, 256, 0, stream, (const uint4*)ctx.scan_scratch.p, blocks, (uint4*)d_out);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- arithmetic self-tests -------------------------------------------------------------------------------
// op: 0 add, 1 sub, 2 mul, 3 sqr(a), 4 inv(a), 5 from_mont(a), 6 to_mont(a); lazily reduced (operands < 2p):
// 7 mul_lazy, 8 sqr_lazy(a), 9 add_lazy, 10 sub_lazy, 11 canon(a), 12 is_zero_lazy(a) (1 or 0 in the low limb),
// 13 mul2_lazy(a, canon(b), b, neg_lazy(canon(a))) = a (b mod p) + b (p - (a mod p)), the form of the mixed addition's Y3
template <int F>
__global__ void __launch_bounds__(128) field_selftest_kernel(int op, const uint4* __restrict__ a, const uint4* __restrict__ b, uint32_t n, uint4* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fp<F> x = fp_load<F>(a + 2 * (size_t)i), y = fp_load<F>(b + 2 * (size_t)i), r;
    switch (op) {
        case 0: r = fp_add(x, y); break;
        case 1: r = fp_sub(x, y); break;
        case 2: r = fp_mul(x, y); break;
        case 3: r = fp_sqr(x); break;
        case 4: r = fp_inv(x); break;
        case 5: r = fp_from_mont(x); break;
        case 6: r = fp_to_mont(x); break;
        case 7: r = fp_mul_lazy(x, y); break;
        case 8: r = fp_sqr_lazy(x); break;
        case 9: r = fp_add_lazy(x, y); break;
        case 10: r = fp_sub_lazy(x, y); break;
        case 11: r = fp_canon(x); break;
        case 13: r = fp_mul2_lazy(x, fp_canon(y), y, fp_neg_lazy(fp_canon(x))); break;
        default: r = fp_zero<F>(); r.l[0] = fp_is_zero_lazy(x) ? 1u : 0u; break;
    }
    fp_store<F>(out + 2 * (size_t)i, r);
}

int field_selftest_run(DeviceCtx& ctx, int field, int op, const void* d_a, const void* d_b, size_t n, void* d_out, cudaStream_t stream) {
    (void)ctx;
    if (n == 0) return H2B_OK;
    if (field == 0) { H2B_LAUNCH(field_selftest_kernel<FR>, (unsigned)((n + 127) / 128), 128, 0, stream, op, (const uint4*)d_a, (const uint4*)d_b, (uint32_t)n, (uint4*)d_out); }
    else { H2B_LAUNCH(field_selftest_kernel<FQ>, (unsigned)((n + 127) / 128), 128, 0, stream, op, (const uint4*)d_a, (const uint4*)d_b, (uint32_t)n, (uint4*)d_out); }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// op 0: affine p + affine q (mixed-add path, through XYZZ);  op 1: p - q;  op 2: general XYZZ add of 2p+q and q
// (exercises xyzz_add / xyzz_double);  op 3: Jacobian conversion round trip of p+q;  op 4: p + q by the lazily reduced
// mixed addition of the MSM accumulation, on an accumulator that holds p with every coordinate offset by the modulus
// (non-canonical, as a lazily reduced accumulator may be);  op 5: [e] p by the variable-base multiplication of the G1 NTT,
// e = the first 4 words of q (Fr, Montgomery).  Output affine (64 B).
__device__ __forceinline__ Fq fq_plus_modulus(const Fq& a) {
    Fq r;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { c += (uint64_t)a.l[i] + FpParams<FQ>::P(i); r.l[i] = (uint32_t)c; c >>= 32; }
    return r;
}

__global__ void __launch_bounds__(128) ec_selftest_kernel(int op, const uint4* __restrict__ P, const uint4* __restrict__ Q, uint32_t n, uint4* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine p = affine_load(P + 4 * (size_t)i), q = affine_load(Q + 4 * (size_t)i);
    XYZZ acc = xyzz_identity();
    Affine res;
    if (op == 0 || op == 1) {
        xyzz_add_affine(acc, p, false);
        xyzz_add_affine(acc, q, op == 1);
        res = xyzz_to_affine(acc);
    } else if (op == 2) {
        xyzz_add_affine(acc, p, false);
        acc = xyzz_double(acc);
        xyzz_add_affine(acc, q, false);       // 2p + q
        XYZZ o = xyzz_from_affine(q);
        xyzz_add(acc, o);                      // 2p + 2q
        xyzz_add(acc, acc);                    // 4p + 4q (doubling branch of the general add)
        res = xyzz_to_affine(acc);
    } else if (op == 5) {
        Fr e;
#pragma unroll
        for (int l = 0; l < 8; ++l) e.l[l] = q.x.l[l];
        res = xyzz_to_affine(xyzz_mul_scalar(xyzz_from_affine(p), fp_from_mont(e)));
    } else if (op == 4) {
        if (!affine_is_identity(p)) {
            acc.x = fq_plus_modulus(p.x); acc.y = fq_plus_modulus(p.y);
            acc.zz = fq_plus_modulus(fp_one<FQ>()); acc.zzz = fq_plus_modulus(fp_one<FQ>());
        }
        xyzz_add_affine_lazy(acc, q, false);
        res = xyzz_to_affine(xyzz_canon(acc));
    } else {
        xyzz_add_affine(acc, p, false);
        xyzz_add_affine(acc, q, false);
        Fq X, Y, Z;
        xyzz_to_jacobian(acc, X, Y, Z);
        if (fp_is_zero(Z)) { res.x = fp_zero<FQ>(); res.y = fp_zero<FQ>(); }
        else {
            Fq zi = fp_inv(Z), zi2 = fp_sqr(zi);
            res.x = fp_mul(X, zi2);
            res.y = fp_mul(Y, fp_mul(zi2, zi));
        }
    }
    affine_store(out + 4 * (size_t)i, res);
}

int ec_selftest_run(DeviceCtx& ctx, int op, const void* d_p, const void* d_q, size_t n, void* d_out, cudaStream_t stream) {
    (void)ctx;
    if (n == 0) return H2B_OK;
    H2B_LAUNCH(ec_selftest_kernel, (unsigned)((n + 127) / 128), 128, 0, stream, op, (const uint4*)d_p, (const uint4*)d_q, (uint32_t)n, (uint4*)d_out);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- integer-pipe micro-benchmarks ------------------------------------------------------------------------
// kind 0: independent 32-bit mad.lo chains (IMAD);  kind 1: independent mad.wide.u32 chains (IMAD.WIDE, 64-bit
// accumulate);  kind 2: dependent Fq Montgomery multiplications (the real inner loop: 128 IMAD.WIDE + 8 IMAD each);
// kind 3: dependent XYZZ mixed additions.   ops_out = multiply-adds (kind 0/1), field muls (2), point adds (3).
#ifndef H2B_EMU
template <int kind>
__global__ void __launch_bounds__(256) imad_bench_kernel(int iters, uint32_t* sink) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (kind == 0) {
        uint32_t a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7, m = t | 1, k = t * 3 + 1;
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                asm volatile("mad.lo.u32 %0, %0, %8, %9;\n\tmad.lo.u32 %1, %1, %8, %9;\n\tmad.lo.u32 %2, %2, %8, %9;\n\tmad.lo.u32 %3, %3, %8, %9;\n\t"
                             "mad.lo.u32 %4, %4, %8, %9;\n\tmad.lo.u32 %5, %5, %8, %9;\n\tmad.lo.u32 %6, %6, %8, %9;\n\tmad.lo.u32 %7, %7, %8, %9;"
                             : "+r"(a0), "+r"(a1), "+r"(a2), "+r"(a3), "+r"(a4), "+r"(a5), "+r"(a6), "+r"(a7) : "r"(m), "r"(k));
            }
        }
        sink[t] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
    } else if (kind == 1) {
        unsigned long long a0 = t, a1 = t + 1, a2 = t + 2, a3 = t + 3, a4 = t + 4, a5 = t + 5, a6 = t + 6, a7 = t + 7;
        uint32_t m = t | 1, k = t * 3 + 1;
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                asm volatile("mad.wide.u32 %0, %8, %9, %0;\n\tmad.wide.u32 %1, %8, %9, %1;\n\tmad.wide.u32 %2, %8, %9, %2;\n\tmad.wide.u32 %3, %8, %9, %3;\n\t"
                             "mad.wide.u32 %4, %8, %9, %4;\n\tmad.wide.u32 %5, %8, %9, %5;\n\tmad.wide.u32 %6, %8, %9, %6;\n\tmad.wide.u32 %7, %8, %9, %7;"
                             : "+l"(a0), "+l"(a1), "+l"(a2), "+l"(a3), "+l"(a4), "+l"(a5), "+l"(a6), "+l"(a7) : "r"(m), "r"(k));
                m += (uint32_t)a0;
            }
        }
        unsigned long long x = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
        sink[t] = (uint32_t)x ^ (uint32_t)(x >> 32);
    } else if (kind == 2) {
        Fq a = fp_one<FQ>(), b = fp_one<FQ>();
        a.l[0] ^= t; b.l[1] ^= t;
        for (int i = 0; i < iters; ++i) {
            Fq c = fp_mul(a, b);
            a = b; b = c;
        }
        sink[t] = b.l[0] ^ b.l[7];
    } else if (kind == 4) {
        Fq a = fp_one<FQ>();
        a.l[0] ^= t; a.l[3] ^= t * 7;
        for (int i = 0; i < iters; ++i) a = fp_sqr(a);
        sink[t] = a.l[0] ^ a.l[7];
    } else if (kind == 5) {
        Fq a = fp_one<FQ>(), b = fp_one<FQ>();
        a.l[0] ^= t; b.l[1] ^= t;
        for (int i = 0; i < iters; ++i) {
            Fq c = fp_mul2(a, b, b, a);
            a = b; b = c;
        }
        sink[t] = b.l[0] ^ b.l[7];
    } else {
        Affine g;
        g.x = fp_one<FQ>();
        g.y = fp_dbl(fp_one<FQ>());
        XYZZ acc = xyzz_double_affine(g);
        acc.x.l[0] ^= 0;   // keep the point valid: 2G, then repeatedly add G
        for (int i = 0; i < iters; ++i) xyzz_add_affine_lazy(acc, g, (i & 7) == 7 && t == 0xffffffffu);     // the MSM accumulation's addition
        sink[t] = acc.x.l[0] ^ acc.zzz.l[3];
    }
}
#endif

int imad_bench_run(DeviceCtx& ctx, int kind, int iters, int blocks, int threads, float* ms_out, double* ops_out, cudaStream_t stream) {
#ifdef H2B_EMU
    (void)ctx; (void)kind; (void)iters; (void)blocks; (void)threads; (void)ms_out; (void)ops_out; (void)stream;
    set_error("imad_bench: not available in the kernel-logic emulator");
    return H2B_ERR_BAD_ARGUMENT;
#else
    if (kind < 0 || kind > 5 || iters < 1 || blocks < 1 || threads < 32 || threads > 256) { set_error("imad_bench: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
    (void)ctx;
    DevBuf sink;
    H2B_TRY(sink.reserve((size_t)blocks * threads * 4));
    cudaEvent_t e0, e1;
    H2B_CUDA(cudaEventCreate(&e0));
    H2B_CUDA(cudaEventCreate(&e1));
    void (*kfn)(int, uint32_t*) = kind == 0 ? imad_bench_kernel<0> : kind == 1 ? imad_bench_kernel<1> : kind == 2 ? imad_bench_kernel<2> : kind == 3 ? imad_bench_kernel<3> :
                                   kind == 4 ? imad_bench_kernel<4> : imad_bench_kernel<5>;
    H2B_LAUNCH(kfn, blocks, threads, 0, stream, iters / 8 + 1, (uint32_t*)sink.p);   // warm-up
    H2B_CUDA(cudaEventRecord(e0, stream));
    H2B_LAUNCH(kfn, blocks, threads, 0, stream, iters, (uint32_t*)sink.p);
    H2B_CUDA(cudaEventRecord(e1, stream));
    H2B_CUDA(cudaEventSynchronize(e1));
    H2B_CUDA(cudaGetLastError());
    H2B_CUDA(cudaEventElapsedTime(ms_out, e0, e1));
    double per_thread = (kind <= 1) ? 64.0 * iters : (double)iters;
    *ops_out = per_thread * blocks * threads;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    sink.release();
    return H2B_OK;
#endif
}

}  // namespace h2b
