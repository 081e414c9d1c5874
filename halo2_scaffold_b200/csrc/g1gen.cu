// Fixed-base multiples of the G1 generator and the KZG setup built on them.
//
// * g1_generator_mul: out[i] = [z_i] G for 254-bit scalars.  Each scalar is recoded into signed W-bit digits d_j in
//   (-2^(W-1), 2^(W-1)], and the point is  sum_j d_j 2^(W j) G: one complete mixed addition per non-zero digit of a table
//   entry T[j][|d_j|] = |d_j| 2^(W j) G, no doublings.  The table is built on the device once per device (DeviceCtx) and
//   stays resident.  W is chosen by measurement (DESIGN.md section 5.7).
// * Normalisation: the kernel leaves (X ZZZ, Y ZZ) in the output and ZZ ZZZ in a scratch column; one batch inversion of
//   that column (scan.cu, Montgomery's trick) and one more pass give x = X/ZZ, y = Y/ZZZ.  The identity has ZZ = ZZZ = 0:
//   its inverse stays 0 and the point comes out as (0, 0).  Large inputs run in chunks of 2^24 points.
// * gen_points (synthetic benchmark bases, [z]G for 64-bit SplitMix64 z) and the SRS setup both use it; only the scalar
//   source differs (a template parameter, so the synthetic scalars need no column of their own).
// * srs_setup: [UP] halo2_proofs/src/poly/kzg/commitment.rs ParamsKZG::setup computes g[i] = [s^i] G and
//   g_lagrange[i] = [L_i(s)] G, L_i(s) = w^i (s^n - 1) / (n (s - w^i)), by one scalar multiplication per point on the CPU.
//   Here L_i(s) = c / (s w^-i - 1) with c = (s^n - 1) / n: the denominators are one power table, one batch inversion and
//   one scaling, and both vectors go through the fixed-base kernel.
// * g1_to_lagrange (ParamsKZG::downsize): a radix-2 NTT over G1 points, see the section at the end; it shares the
//   normalisation with the two above.
#include "common.h"
#include "ec.cuh"

namespace h2b {

#ifndef H2B_G1GEN_WINDOW
#define H2B_G1GEN_WINDOW 16
#endif
static const int GEN_W = H2B_G1GEN_WINDOW;
static const int GEN_WINDOWS = (255 + GEN_W - 1) / GEN_W;     // W * windows >= 255: the top digit never carries out (r < 2^254)
static const uint32_t GEN_ROWS = 1u << (GEN_W - 1);          // T[j][m - 1] = m 2^(W j) G, m = 1 .. 2^(W-1)
static const size_t GEN_CHUNK = (size_t)1 << 24;
static_assert(GEN_W >= 2 && GEN_W <= 20, "fixed-base window out of range");

// scalar sources: the canonical (non-Montgomery) value of scalar i
struct ScalarSplitMix {       // z = SplitMix64 value #(first + i) of stream `seed`
    uint64_t seed, first;
    __device__ __forceinline__ Fr at(size_t i) const {
        const uint64_t z = splitmix64_at(seed, first + i);
        Fr r = fp_zero<FR>();
        r.l[0] = (uint32_t)z;
        r.l[1] = (uint32_t)(z >> 32);
        return r;
    }
};
struct ScalarArray {          // Fr array in Montgomery form
    const uint4* a;
    __device__ __forceinline__ Fr at(size_t i) const { return fp_from_mont(fp_load<FR>(a + 2 * i)); }
};

// (X ZZZ, Y ZZ) -> out, ZZ ZZZ -> den: the half of the normalisation that needs no inverse
__device__ __forceinline__ void gen_store_projective(const XYZZ& p, uint4* out, uint4* den) {
    Affine a;
    a.x = fp_mul(p.x, p.zzz);
    a.y = fp_mul(p.y, p.zz);
    affine_store(out, a);
    fp_store<FQ>(den, fp_mul(p.zz, p.zzz));
}

// B_j = 2^(W j) G, affine (one thread; W * GEN_WINDOWS doublings and GEN_WINDOWS inversions, once per device)
__global__ void g1gen_bases_kernel(uint4* bases) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    Affine g;
    g.x = fp_one<FQ>();
    g.y = fp_dbl(fp_one<FQ>());
    XYZZ t = xyzz_from_affine(g);
    for (int j = 0; j < GEN_WINDOWS; ++j) {
        affine_store(bases + 4 * j, xyzz_to_affine(t));
        for (int b = 0; b < GEN_W; ++b) t = xyzz_double(t);
    }
}

// T[j][m - 1] = m B_j by double-and-add over the bits of m, left projective for the batch normalisation
__global__ void __launch_bounds__(128) g1gen_table_kernel(const uint4* __restrict__ bases, uint4* __restrict__ table, uint4* __restrict__ den) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint32_t)GEN_WINDOWS * GEN_ROWS) return;
    const uint32_t j = idx / GEN_ROWS, m = idx % GEN_ROWS + 1;
    const Affine b = affine_load(bases + 4 * j);
    XYZZ acc = xyzz_identity();
    for (int bit = GEN_W - 1; bit >= 0; --bit) {
        acc = xyzz_double(acc);
        if ((m >> bit) & 1) xyzz_add_affine(acc, b, false);
    }
    gen_store_projective(acc, table + 4 * (size_t)idx, den + 2 * (size_t)idx);
}

// out[i] = [scalar i] G, projective half of the normalisation (see gen_store_projective)
template <class Src>
__global__ void __launch_bounds__(128) g1gen_mul_kernel(const uint4* __restrict__ table, Src src, uint32_t n, uint4* __restrict__ out, uint4* __restrict__ den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr z = src.at(i);
    XYZZ acc = xyzz_identity();
    uint32_t carry = 0;
#pragma unroll 1
    for (int j = 0; j < GEN_WINDOWS; ++j) {
        const uint32_t v = (z.l[0] & ((1u << GEN_W) - 1)) + carry;
#pragma unroll
        for (int l = 0; l < 7; ++l) z.l[l] = __funnelshift_r(z.l[l], z.l[l + 1], GEN_W);
        z.l[7] >>= GEN_W;
        carry = v > GEN_ROWS ? 1u : 0u;
        const uint32_t mag = carry ? (1u << GEN_W) - v : v;        // digit v - 2^W < 0 when carrying
        if (mag != 0) xyzz_add_affine_lazy(acc, affine_load(table + 4 * ((size_t)j * GEN_ROWS + mag - 1)), carry != 0);
    }
    gen_store_projective(xyzz_canon(acc), out + 4 * (size_t)i, den + 2 * (size_t)i);
}

// out[i] = (x' inv[i], y' inv[i]) with inv = 1 / (ZZ ZZZ) (0 for the identity)
__global__ void __launch_bounds__(128) g1gen_finish_kernel(uint4* __restrict__ pts, const uint4* __restrict__ inv, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Fq d = fp_load<FQ>(inv + 2 * i);
    Affine a = affine_load(pts + 4 * i);
    a.x = fp_mul(a.x, d);
    a.y = fp_mul(a.y, d);
    affine_store(pts + 4 * i, a);
}

static int g1gen_normalise(DeviceCtx& ctx, uint4* pts, uint4* den, size_t n, cudaStream_t stream) {
    H2B_TRY(fq_batch_invert_run(ctx, den, n, stream));
    H2B_LAUNCH(g1gen_finish_kernel, (unsigned)((n + 127) / 128), 128, 0, stream, pts, (const uint4*)den, n);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// the resident table of this device, built on first use; `built` tells the caller whether this call built it
static int g1gen_table(DeviceCtx& ctx, cudaStream_t stream, bool* built) {
    *built = false;
    if (ctx.gen_table.p) return H2B_OK;
    const size_t entries = (size_t)GEN_WINDOWS * GEN_ROWS;
    DevBuf bases, den;
    int rc = ctx.gen_table.reserve(entries * 64);
    if (!rc) rc = bases.reserve((size_t)GEN_WINDOWS * 64);
    if (!rc) rc = den.reserve(entries * 32);
    if (!rc) {
        H2B_LAUNCH(g1gen_bases_kernel, 1, 32, 0, stream, (uint4*)bases.p);
        H2B_LAUNCH(g1gen_table_kernel, (unsigned)((entries + 127) / 128), 128, 0, stream, (const uint4*)bases.p, (uint4*)ctx.gen_table.p, (uint4*)den.p);
        rc = g1gen_normalise(ctx, (uint4*)ctx.gen_table.p, (uint4*)den.p, entries, stream);
    }
    cudaError_t e = cudaStreamSynchronize(stream);      // the temporaries go now
    bases.release();
    den.release();
    if (!rc && e != cudaSuccess) { set_error("g1 generator table: %s", cudaGetErrorString(e)); rc = H2B_ERR_CUDA; }
    if (rc) { ctx.gen_table.release(); return rc; }
    *built = true;
    return H2B_OK;
}

// n points [scalar i] G into d_out, chunk by chunk; `before_chunk(done, m)` may fill the scalar source of the chunk
template <class SrcOf, class Before>
static int g1gen_run(DeviceCtx& ctx, size_t n, uint4* d_out, cudaStream_t stream, SrcOf src_of, Before before_chunk, bool mark) {
    const size_t chunk = n < GEN_CHUNK ? n : GEN_CHUNK;
    H2B_TRY(ctx.gen_scratch.reserve(chunk * 64 + 128));         // den | chunk scalars | setup constants
    H2B_TRY(ctx.scan_scratch.reserve(chunk * 32));               // the batch inversions: allocated before any phase is timed
    uint4* den = (uint4*)ctx.gen_scratch.p;
    for (size_t done = 0; done < n; done += GEN_CHUNK) {
        const uint32_t m = (uint32_t)(n - done < GEN_CHUNK ? n - done : GEN_CHUNK);
        if (mark) ctx.prof.mark(PROF_BEGIN, stream);
        H2B_TRY(before_chunk(done, m));
        if (mark) ctx.prof.mark(PROF_SRS_SCALARS, stream);
        H2B_LAUNCH(g1gen_mul_kernel<decltype(src_of(done))>, (m + 127) / 128, 128, 0, stream, (const uint4*)ctx.gen_table.p, src_of(done), m, d_out + 4 * done, den);
        if (mark) ctx.prof.mark(PROF_SRS_FIXED_BASE, stream);
        H2B_TRY(g1gen_normalise(ctx, d_out + 4 * done, den, m, stream));
        if (mark) ctx.prof.mark(PROF_SRS_NORMALISE, stream);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

void g1gen_release_scratch(DeviceCtx& ctx, size_t scan_cap_before) {
    ctx.gen_scratch.release();
    if (ctx.scan_scratch.cap != scan_cap_before) ctx.scan_scratch.release();
}

// synchronous; keeps only the generator table (32 MiB at W = 16) resident, not the chunk scratch
int gen_points_run(DeviceCtx& ctx, uint64_t seed, size_t n, void* d_out, cudaStream_t stream) {
    if (n == 0) return H2B_OK;
    const size_t scan_cap = ctx.scan_scratch.cap;
    bool built;
    H2B_TRY(g1gen_table(ctx, stream, &built));
    int rc = g1gen_run(ctx, n, (uint4*)d_out, stream, [&](size_t done) { return ScalarSplitMix{seed, (uint64_t)done}; },
                       [](size_t, uint32_t) { return (int)H2B_OK; }, false);
    cudaError_t e = cudaStreamSynchronize(stream);
    g1gen_release_scratch(ctx, scan_cap);
    if (rc) return rc;
    H2B_CUDA(e);
    return H2B_OK;
}

int g1_generator_mul_run(DeviceCtx& ctx, const void* d_scalars, size_t n, void* d_out, cudaStream_t stream) {
    if (n == 0) return H2B_OK;
    if (!d_scalars || !d_out) { set_error("g1_generator_mul: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    bool built;
    H2B_TRY(g1gen_table(ctx, stream, &built));
    return g1gen_run(ctx, n, (uint4*)d_out, stream, [&](size_t done) { return ScalarArray{(const uint4*)d_scalars + 2 * done}; },
                     [](size_t, uint32_t) { return (int)H2B_OK; }, false);
}

// ---- ParamsKZG::setup ---------------------------------------------------------------------------------------------------
// Fr Montgomery product on the host: only for checking the caller's s before anything runs
static void fr_mul_host(const uint64_t* a, const uint64_t* b, uint64_t* r) {
    uint32_t x[8], y[8], t[10] = {0};
    memcpy(x, a, 32);
    memcpy(y, b, 32);
    for (int i = 0; i < 8; ++i) {
        uint64_t c = 0;
        for (int j = 0; j < 8; ++j) { c += (uint64_t)x[j] * y[i] + t[j]; t[j] = (uint32_t)c; c >>= 32; }
        c += t[8]; t[8] = (uint32_t)c; t[9] = (uint32_t)(c >> 32);
        const uint32_t m = t[0] * FpParams<FR>::INV;
        c = (uint64_t)m * FpParams<FR>::P(0) + t[0]; c >>= 32;
        for (int j = 1; j < 8; ++j) { c += (uint64_t)m * FpParams<FR>::P(j) + t[j]; t[j - 1] = (uint32_t)c; c >>= 32; }
        c += t[8]; t[7] = (uint32_t)c; t[8] = t[9] + (uint32_t)(c >> 32);
    }
    bool geq = t[8] != 0;
    if (!geq) {
        geq = true;
        for (int i = 7; i >= 0; --i) { if (t[i] != FpParams<FR>::P(i)) { geq = t[i] > FpParams<FR>::P(i); break; } }
    }
    if (geq) { int64_t bw = 0; for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)t[i] - FpParams<FR>::P(i) + bw; t[i] = (uint32_t)d; bw = d >> 32; } }
    memcpy(r, t, 32);
}

int srs_setup_check(uint32_t k, const uint64_t s[4]) {
    if (k > 28) { set_error("h2b_srs_setup: k = %u (at most 28)", k); return H2B_ERR_BAD_ARGUMENT; }
    if (!fr_canonical(s)) { set_error("h2b_srs_setup: s is not below the scalar field modulus"); return H2B_ERR_BAD_ARGUMENT; }
    // s^n == 1 means s = w^j for some j: a denominator s - w^j vanishes (upstream panics in invert().unwrap())
    uint64_t p[4];
    memcpy(p, s, 32);
    for (uint32_t i = 0; i < k; ++i) fr_mul_host(p, p, p);
    uint32_t one[8];
    for (int i = 0; i < 8; ++i) one[i] = FpParams<FR>::ONE(i);
    if (memcmp(p, one, 32) == 0) { set_error("h2b_srs_setup: s^(2^%u) = 1 (s is a power of the root of unity)", k); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

// halo2curves' Fr::ROOT_OF_UNITY (order 2^28), Montgomery form
static const uint64_t FR_ROOT_OF_UNITY_MONT[4] = {0x9632c7c5b639feb8ull, 0x985ce3400d0ff299ull, 0xb2dd880001b0ecd8ull, 0x1d69070d6d98ce29ull};

// consts[0] = w (from ntt_root_powers_run) -> consts[0] = w^-1, consts[1] = (s^n - 1) / n
__global__ void srs_constants_kernel(Fr s, uint32_t k, uint4* consts) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const Fr w = fp_load<FR>(consts);
    Fr sn = s;
    for (uint32_t i = 0; i < k; ++i) sn = fp_sqr(sn);
    Fr n = fp_zero<FR>();
    n.l[0] = 1u << k;
    fp_store<FR>(consts, fp_inv(w));
    fp_store<FR>(consts + 2, fp_mul(fp_sub(sn, fp_one<FR>()), fp_inv(fp_to_mont(n))));
}

// out[i] = mul base^(first + i) - sub; RUN consecutive powers per thread, the first by square-and-multiply
static const uint32_t SRS_RUN = 32;
struct SrsPowers { Fr base, mul, sub; };
__global__ void __launch_bounds__(128) srs_powers_kernel(SrsPowers p, uint32_t first, uint32_t m, uint4* __restrict__ out) {
    const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * SRS_RUN;
    if (i0 >= m) return;
    Fr cur = fp_mul(p.mul, fp_pow_u32(p.base, first + i0));
    for (uint32_t i = i0; i < i0 + SRS_RUN && i < m; ++i) {
        fp_store<FR>(out + 2 * (size_t)i, fp_sub(cur, p.sub));
        cur = fp_mul(cur, p.base);
    }
}

// which = 0: g[i] = [s^i] G;  which = 1: g_lagrange[i] = [L_i(s)] G.  srs_setup_check has passed.
int srs_setup_run(DeviceCtx& ctx, uint32_t k, const uint64_t s_words[4], int which, void* d_out, cudaStream_t stream) {
    const size_t n = (size_t)1 << k, chunk = n < GEN_CHUNK ? n : GEN_CHUNK;
    bool built;
    H2B_TRY(ctx.gen_scratch.reserve(chunk * 64 + 128));
    H2B_TRY(ctx.scan_scratch.reserve(chunk * 32));
    ctx.prof.mark(PROF_BEGIN, stream);
    H2B_TRY(g1gen_table(ctx, stream, &built));
    if (built) ctx.prof.mark(PROF_SRS_TABLE, stream);
    uint4* scal = (uint4*)ctx.gen_scratch.p + 2 * chunk;
    uint4* consts = scal + 2 * chunk;
    SrsPowers p;
    memcpy(p.base.l, s_words, 32);
    for (int i = 0; i < 8; ++i) { p.mul.l[i] = FpParams<FR>::ONE(i); p.sub.l[i] = 0; }
    Fr c;
    if (which == 1) {
        // w = ROOT_OF_UNITY^(2^(28 - k)) as EvaluationDomain derives it, w^-1 and c = (s^n - 1) / n, all on the device
        H2B_TRY(ntt_root_powers_run(ctx, FR_ROOT_OF_UNITY_MONT, 28 - k, 28 - k, consts, stream));
        Fr s = p.base;
        H2B_LAUNCH(srs_constants_kernel, 1, 32, 0, stream, s, k, consts);
        uint32_t host[16];
        H2B_CUDA(cudaMemcpyAsync(host, consts, 64, cudaMemcpyDeviceToHost, stream));
        H2B_CUDA(cudaStreamSynchronize(stream));
        memcpy(p.base.l, host, 32);                 // w^-1
        memcpy(c.l, host + 8, 32);
        p.mul = s;
        for (int i = 0; i < 8; ++i) p.sub.l[i] = FpParams<FR>::ONE(i);   // s w^-i - 1
        ctx.prof.mark(PROF_SRS_SCALARS, stream);
    }
    auto fill = [&](size_t done, uint32_t m) -> int {
        H2B_LAUNCH(srs_powers_kernel, (m + 128 * SRS_RUN - 1) / (128 * SRS_RUN), 128, 0, stream, p, (uint32_t)done, m, scal);
        if (which == 1) {
            H2B_TRY(fr_batch_invert_run(ctx, scal, m, stream));
            uint64_t f[4];
            memcpy(f, c.l, 32);
            H2B_TRY(ntt_scale_run(ctx, scal, m, f, 1, stream));
        }
        H2B_CUDA(cudaGetLastError());
        return H2B_OK;
    };
    return g1gen_run(ctx, n, (uint4*)d_out, stream, [&](size_t) { return ScalarArray{scal}; }, fill, true);
}

// ---- g_to_lagrange: a radix-2 NTT over G1 points -----------------------------------------------------------------------
// [UP] halo2_proofs/src/arithmetic.rs g_to_lagrange: g_lagrange[i] = n^-1 sum_j w^(-ij) g[j] (best_fft over C::Curve with
// omega_inv, *= n_inv, batch_normalize).  One butterfly is two general additions and one variable-base scalar multiplication
// (xyzz_mul_scalar, ~3300 Fq multiplications) on 256 bytes of points, so the transform is arithmetic-bound by three orders of
// magnitude: one launch per radix-2 stage, one thread per butterfly, in place on an n x 128 B XYZZ work buffer.
// Decimation in frequency on the natural-order input: stage s pairs i and i + n / 2^(s+1) and gives (a + b, w^(-j 2^s) (a - b)).
// Stage 0 reads the affine input and folds n^-1 in (n^-1 (a + b), (n^-1 w^-j) (a - b): n / 2 extra multiplications instead of
// n); the last stage has only trivial twiddles and stores the projective half of the normalisation at the bit-reversed index.

// consts[0] = w (from ntt_root_powers_run) -> consts[0] = w^-1, consts[1] = 1 / 2^k
__global__ void g1ntt_constants_kernel(uint32_t k, uint4* consts) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    Fr n = fp_zero<FR>();
    n.l[0] = 1u << k;
    fp_store<FR>(consts, fp_inv(fp_load<FR>(consts)));
    fp_store<FR>(consts + 2, fp_inv(fp_to_mont(n)));
}

// tw[i] = w^-i for i < m (Montgomery), SRS_RUN consecutive powers per thread as srs_powers_kernel does; the base is read
// from the device, so the call stays asynchronous
__global__ void __launch_bounds__(128) g1ntt_twiddle_kernel(const uint4* __restrict__ consts, uint32_t m, uint4* __restrict__ tw) {
    const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * SRS_RUN;
    if (i0 >= m) return;
    const Fr base = fp_load<FR>(consts);
    Fr cur = fp_pow_u32(base, i0);
    for (uint32_t i = i0; i < i0 + SRS_RUN && i < m; ++i) {
        fp_store<FR>(tw + 2 * (size_t)i, cur);
        cur = fp_mul(cur, base);
    }
}

// one DIF stage; MODE bit 0: the first stage (affine input, n^-1 folded in), bit 1: the last (projective normalisation half
// stored at the bit-reversed index into out / den)
template <int MODE>
__global__ void __launch_bounds__(128) g1ntt_stage_kernel(const uint4* __restrict__ in, uint4* __restrict__ work, const uint4* __restrict__ tw,
                                                           const uint4* __restrict__ consts, uint32_t log_n, uint32_t s, uint4* __restrict__ out,
                                                           uint4* __restrict__ den) {
    const bool FIRST = MODE & 1, LAST = MODE & 2;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (1u << (log_n - 1))) return;
    const uint32_t lh = log_n - 1 - s, j = t & ((1u << lh) - 1);
    const uint32_t i0 = ((t >> lh) << (lh + 1)) | j, i1 = i0 + (1u << lh);
    XYZZ a, b;
    if (FIRST) {
        a = xyzz_from_affine(affine_load(in + 4 * (size_t)i0));
        b = xyzz_from_affine(affine_load(in + 4 * (size_t)i1));
    } else {
        a = xyzz_load(work + 8 * (size_t)i0);
        b = xyzz_load(work + 8 * (size_t)i1);
    }
    XYZZ sum = a;
    xyzz_add(sum, b);
    b.y = fp_neg(b.y);
    xyzz_add(a, b);                                 // a - b
    if (FIRST) {
        const Fr ninv = fp_load<FR>(consts + 2);
        sum = xyzz_mul_scalar(sum, fp_from_mont(ninv));
        a = xyzz_mul_scalar(a, fp_from_mont(fp_mul(ninv, fp_load<FR>(tw + 2 * (size_t)j))));
    } else if (j != 0) {
        a = xyzz_mul_scalar(a, fp_from_mont(fp_load<FR>(tw + 2 * ((size_t)j << s))));
    }
    if (LAST) {
        const uint32_t r0 = __brev(i0) >> (32 - log_n), r1 = __brev(i1) >> (32 - log_n);
        gen_store_projective(sum, out + 4 * (size_t)r0, den + 2 * (size_t)r0);
        gen_store_projective(a, out + 4 * (size_t)r1, den + 2 * (size_t)r1);
    } else {
        xyzz_store(work + 8 * (size_t)i0, sum);
        xyzz_store(work + 8 * (size_t)i1, a);
    }
}

// d_out[i] = g_to_lagrange(d_g)[i] for i < 2^k (d_out may be d_g); asynchronous, the scratch stays reserved in gen_scratch
int g1_to_lagrange_run(DeviceCtx& ctx, const void* d_g, uint32_t k, void* d_out, cudaStream_t stream) {
    if (k > 28) { set_error("g1_to_lagrange: k = %u (at most 28)", k); return H2B_ERR_BAD_ARGUMENT; }
    if (!d_g || !d_out) { set_error("g1_to_lagrange: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (k == 0) {                                   // n^-1 = 1, a transform of length one
        if (d_out != d_g) H2B_CUDA(cudaMemcpyAsync(d_out, d_g, 64, cudaMemcpyDeviceToDevice, stream));
        return H2B_OK;
    }
    const size_t n = (size_t)1 << k;
    H2B_TRY(ctx.gen_scratch.reserve(n * 128 + n * 32 + (n / 2) * 32 + 64));      // work | den | twiddles | constants
    H2B_TRY(ctx.scan_scratch.reserve(n * 32));
    uint4* work = (uint4*)ctx.gen_scratch.p;
    uint4* den = work + 8 * n;
    uint4* tw = den + 2 * n;
    uint4* consts = tw + n;
    ctx.prof.mark(PROF_BEGIN, stream);
    H2B_TRY(ntt_root_powers_run(ctx, FR_ROOT_OF_UNITY_MONT, 28 - k, 28 - k, consts, stream));
    H2B_LAUNCH(g1ntt_constants_kernel, 1, 32, 0, stream, k, consts);
    const uint32_t half = (uint32_t)(n / 2);
    H2B_LAUNCH(g1ntt_twiddle_kernel, (half + 128 * SRS_RUN - 1) / (128 * SRS_RUN), 128, 0, stream, (const uint4*)consts, half, tw);
    ctx.prof.mark(PROF_G1NTT_TWIDDLE, stream);
    const unsigned grid = (half + 127) / 128;
    const uint4* g = (const uint4*)d_g;
    uint4* out = (uint4*)d_out;
    if (k == 1) {
        H2B_LAUNCH(g1ntt_stage_kernel<3>, grid, 128, 0, stream, g, work, (const uint4*)tw, (const uint4*)consts, k, 0u, out, den);
    } else {
        H2B_LAUNCH(g1ntt_stage_kernel<1>, grid, 128, 0, stream, g, work, (const uint4*)tw, (const uint4*)consts, k, 0u, out, den);
        for (uint32_t s = 1; s + 1 < k; ++s)
            H2B_LAUNCH(g1ntt_stage_kernel<0>, grid, 128, 0, stream, g, work, (const uint4*)tw, (const uint4*)consts, k, s, out, den);
        H2B_LAUNCH(g1ntt_stage_kernel<2>, grid, 128, 0, stream, g, work, (const uint4*)tw, (const uint4*)consts, k, k - 1, out, den);
    }
    ctx.prof.mark(PROF_G1NTT_STAGES, stream);
    H2B_TRY(g1gen_normalise(ctx, out, den, n, stream));
    ctx.prof.mark(PROF_G1NTT_NORMALISE, stream);
    return H2B_OK;
}

}  // namespace h2b
