// Grand-product building blocks on device-resident Fr columns (SURVEY.md section 8f, rank 3): the permutation and lookup
// arguments of the prover ([UP] halo2_proofs/src/plonk/permutation/prover.rs, plonk/lookup/prover.rs) build z(X) as the
// running product of numerator[i] / denominator[i]; the denominators are inverted with ff::BatchInvert (zeros stay
// zero) and z(omega^i) is the exclusive prefix product.  Both are one pass over the column on the CPU; here:
//   * batch inversion: Montgomery's trick per thread over K strided elements (3 multiplications per element + one Fermat
//     inversion per thread), prefix products parked in a scratch column;
//   * exclusive prefix product: chunk products of 16 consecutive elements, recursive scan of the chunk products (one CTA
//     Hillis-Steele at the bottom), then every chunk replays its elements from its scanned offset.
#include "common.h"

namespace h2b {

// ---- batch inversion (Fr; Fq for the point normalisation of g1gen.cu) ---------------------------------------------
template <int F>
__global__ void __launch_bounds__(128) fp_batch_invert_kernel(uint4* __restrict__ a, uint4* __restrict__ pre, size_t n, uint32_t K, uint32_t G) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= G) return;
    Fp<F> run = fp_one<F>();
    for (uint32_t j = 0; j < K; ++j) {
        const size_t idx = (size_t)j * G + t;
        if (idx >= n) break;
        Fp<F> x = fp_load<F>(a + 2 * idx);
        fp_store<F>(pre + 2 * idx, run);
        if (!fp_is_zero(x)) run = fp_mul(run, x);
    }
    Fp<F> inv = fp_inv(run);
    for (uint32_t j = K; j-- > 0;) {
        const size_t idx = (size_t)j * G + t;
        if (idx >= n) continue;
        Fp<F> x = fp_load<F>(a + 2 * idx);
        if (fp_is_zero(x)) continue;
        Fp<F> p = fp_load<F>(pre + 2 * idx);
        fp_store<F>(a + 2 * idx, fp_mul(inv, p));
        inv = fp_mul(inv, x);
    }
}

template <int F>
static int batch_invert_run(DeviceCtx& ctx, void* d_a, size_t n, cudaStream_t stream) {
    if (n == 0) return H2B_OK;
    if (!d_a) { set_error("batch_invert: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(ctx.scan_scratch.reserve(n * 32));
    // K elements per thread: enough threads to fill the GPU, at most 128 so that the Fermat inversion (about 380
    // multiplications) costs 3 more multiplications per element
    const size_t resident = (size_t)ctx.sm_count * 1024;
    size_t K = n / resident;
    if (K < 8) K = 8;
    if (K > 128) K = 128;
    const uint32_t G = (uint32_t)((n + K - 1) / K);
    H2B_LAUNCH(fp_batch_invert_kernel<F>, (G + 127) / 128, 128, 0, stream, (uint4*)d_a, (uint4*)ctx.scan_scratch.p, n, (uint32_t)K, G);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}
int fr_batch_invert_run(DeviceCtx& ctx, void* d_a, size_t n, cudaStream_t stream) { return batch_invert_run<FR>(ctx, d_a, n, stream); }
int fq_batch_invert_run(DeviceCtx& ctx, void* d_a, size_t n, cudaStream_t stream) { return batch_invert_run<FQ>(ctx, d_a, n, stream); }

// ---- exclusive prefix product ----------------------------------------------------------------------------------------
static const uint32_t SCAN_K = 16;          // consecutive elements per thread
static const uint32_t SCAN_BASE = 1024;     // the bottom of the recursion: one CTA

__global__ void __launch_bounds__(128) fr_chunk_product_kernel(const uint4* __restrict__ in, size_t n, uint4* __restrict__ prod, uint32_t chunks) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const size_t lo = (size_t)t * SCAN_K;
    Fr run = fp_load<FR>(in + 2 * lo);
    for (uint32_t i = 1; i < SCAN_K && lo + i < n; ++i) run = fp_mul(run, fp_load<FR>(in + 2 * (lo + i)));
    fp_store<FR>(prod + 2 * (size_t)t, run);
}

// out[i] = offset[t] * in[lo] * ... * in[i-1] for the chunk t that holds i; in-place safe (each element is read before it is written)
__global__ void __launch_bounds__(128) fr_chunk_replay_kernel(const uint4* __restrict__ in, size_t n, const uint4* __restrict__ offset, uint4* __restrict__ out,
                                                            uint32_t chunks) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const size_t lo = (size_t)t * SCAN_K;
    Fr run = fp_load<FR>(offset + 2 * (size_t)t);
    for (uint32_t i = 0; i < SCAN_K && lo + i < n; ++i) {
        Fr x = fp_load<FR>(in + 2 * (lo + i));
        fp_store<FR>(out + 2 * (lo + i), run);
        run = fp_mul(run, x);
    }
}

// one CTA: exclusive prefix product of count <= SCAN_BASE elements (Hillis-Steele in shared memory), in place
__global__ void __launch_bounds__(1024) fr_scan_base_kernel(uint4* __restrict__ a, uint32_t count) {
    H2B_DYN_SMEM(uint4, sh);
    const uint32_t tid = threadIdx.x;
    Fr x = tid < count ? fp_load<FR>(a + 2 * (size_t)tid) : fp_one<FR>();
    for (uint32_t d = 1; d < count; d <<= 1) {
        fp_store<FR>(sh + 2 * tid, x);
        __syncthreads();
        if (tid >= d) x = fp_mul(x, fp_load<FR>(sh + 2 * (tid - d)));
        __syncthreads();
    }
    // inclusive -> exclusive
    fp_store<FR>(sh + 2 * tid, x);
    __syncthreads();
    if (tid < count) fp_store<FR>(a + 2 * (size_t)tid, tid ? fp_load<FR>(sh + 2 * (tid - 1)) : fp_one<FR>());
}

static int prefix_product_rec(DeviceCtx& ctx, const uint4* in, uint4* out, size_t n, uint4* scratch, cudaStream_t stream) {
    if (n <= SCAN_BASE) {
        if (in != out) H2B_CUDA(cudaMemcpyAsync(out, in, n * 32, cudaMemcpyDeviceToDevice, stream));
        uint32_t threads = 32;
        while (threads < n) threads <<= 1;
        H2B_LAUNCH(fr_scan_base_kernel, 1, threads, (size_t)threads * 32, stream, out, (uint32_t)n);
        H2B_CUDA(cudaGetLastError());
        return H2B_OK;
    }
    const uint32_t chunks = (uint32_t)((n + SCAN_K - 1) / SCAN_K);
    H2B_LAUNCH(fr_chunk_product_kernel, (chunks + 127) / 128, 128, 0, stream, in, n, scratch, chunks);
    H2B_TRY(prefix_product_rec(ctx, scratch, scratch, chunks, scratch + 2 * (size_t)chunks, stream));
    H2B_LAUNCH(fr_chunk_replay_kernel, (chunks + 127) / 128, 128, 0, stream, in, n, (const uint4*)scratch, out, chunks);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

int fr_prefix_product_run(DeviceCtx& ctx, const void* d_in, void* d_out, size_t n, cudaStream_t stream) {
    if (n == 0) return H2B_OK;
    if (!d_in || !d_out) { set_error("prefix_product: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n > ((size_t)1 << 31)) { set_error("prefix_product: at most 2^31 elements"); return H2B_ERR_BAD_ARGUMENT; }
    // chunk products of all levels: n/16 + n/256 + ... < n/15 elements (+ slack)
    H2B_TRY(ctx.scan_scratch.reserve((n / 15 + 4 * SCAN_BASE) * 32));
    return prefix_product_rec(ctx, (const uint4*)d_in, (uint4*)d_out, n, (uint4*)ctx.scan_scratch.p, stream);
}

// ---- polynomial evaluation and division by (X - b) ---------------------------------------------------------------------
// [UP] halo2_proofs::arithmetic::{eval_polynomial, kate_division} (SURVEY.md section 1, layer L0): the prover evaluates
// every committed polynomial at the challenge points and divides by (X - x) for the multi-open argument.
// Both are first-order linear recurrences with a constant multiplier, so they telescope through levels of 16:
//   eval:  P(x) = sum_t p_t * (x^16)^t with p_t the Horner value of 16 consecutive coefficients -> evaluate {p_t} at x^16;
//   kate:  q[i-1] = a[i] + b * q[i]  (q = all suffix Horner values): chunk sums with zero carry-in, the same recurrence
//          on the chunk sums with multiplier b^16 gives every chunk's carry-in, then the chunks replay.
static const uint32_t POLY_K = 16;
static const uint32_t POLY_LEVELS_MAX = 9;          // 16^8 > 2^31

// pts[l] = x^(16^l), l < levels (one thread; a handful of squarings)
__global__ void fr_point_powers_kernel(const uint4* __restrict__ x, uint32_t levels, uint4* __restrict__ pts) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    Fr p = fp_load<FR>(x);
    for (uint32_t l = 0; l < levels; ++l) {
        fp_store<FR>(pts + 2 * l, p);
        for (int k = 0; k < 4; ++k) p = fp_sqr(p);
    }
}

// out[t] = sum_{i < 16} in[16 t + i] * x^i
__global__ void __launch_bounds__(128) fr_horner_chunk_kernel(const uint4* __restrict__ in, size_t n, const uint4* __restrict__ x, uint4* __restrict__ out, uint32_t chunks) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const size_t lo = (size_t)t * POLY_K;
    const size_t hi = lo + POLY_K < n ? lo + POLY_K : n;
    const Fr xx = fp_load<FR>(x);
    Fr r = fp_load<FR>(in + 2 * (hi - 1));
    for (size_t i = hi - 1; i-- > lo;) r = fp_add(fp_mul(r, xx), fp_load<FR>(in + 2 * i));
    fp_store<FR>(out + 2 * (size_t)t, r);
}

int fr_eval_polynomial_run(DeviceCtx& ctx, const void* d_coeffs, size_t n, const uint64_t x[4], void* d_out, cudaStream_t stream) {
    if (!d_out || !x || (n && !d_coeffs)) { set_error("eval_polynomial: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) { H2B_CUDA(cudaMemsetAsync(d_out, 0, 32, stream)); return H2B_OK; }
    if (n > ((size_t)1 << 31)) { set_error("eval_polynomial: at most 2^31 coefficients"); return H2B_ERR_BAD_ARGUMENT; }
    // scratch: point powers (POLY_LEVELS_MAX + 1 elements) | the partial values of all levels (< n/15 + slack)
    H2B_TRY(ctx.scan_scratch.reserve((n / 15 + 64) * 32));
    uint4* pts = (uint4*)ctx.scan_scratch.p;
    uint4* buf = pts + 2 * (POLY_LEVELS_MAX + 1);
    H2B_CUDA(cudaMemcpyAsync(pts + 2 * POLY_LEVELS_MAX, x, 32, cudaMemcpyHostToDevice, stream));
    H2B_LAUNCH(fr_point_powers_kernel, 1, 32, 0, stream, (const uint4*)(pts + 2 * POLY_LEVELS_MAX), POLY_LEVELS_MAX, pts);
    const uint4* in = (const uint4*)d_coeffs;
    size_t m = n;
    for (uint32_t l = 0;; ++l) {
        const uint32_t chunks = (uint32_t)((m + POLY_K - 1) / POLY_K);
        uint4* out = chunks == 1 ? (uint4*)d_out : buf;
        H2B_LAUNCH(fr_horner_chunk_kernel, (chunks + 127) / 128, 128, 0, stream, in, m, (const uint4*)(pts + 2 * l), out, chunks);
        if (chunks == 1) break;
        in = buf;
        buf += 2 * (size_t)chunks;
        m = chunks;
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// chunk sums with zero carry-in: s[t] = sum_{i < 16} a[16 t + i] * b^i   (the same kernel as the Horner chunks), then
// carry[t] = s[t+1] + b^16 * carry[t+1] solved recursively, then the replay:
//   q[i-1] = a[i] + b * q[i] inside chunk t, starting from q[hi-1] = carry[t]
// `q` has n - 1 coefficients (q[i-1] for i = 1 .. n-1); a[0] only enters the remainder, which the caller does not need.
__global__ void __launch_bounds__(128) fr_kate_replay_kernel(const uint4* __restrict__ a, size_t n, const uint4* __restrict__ b, const uint4* __restrict__ carry,
                                                           uint4* __restrict__ q, uint32_t chunks) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const size_t lo = (size_t)t * POLY_K;
    const size_t hi = lo + POLY_K < n ? lo + POLY_K : n;
    const Fr bb = fp_load<FR>(b);
    Fr run = carry ? fp_load<FR>(carry + 2 * (size_t)t) : fp_zero<FR>();       // value of q at index hi - 1
    for (size_t i = hi; i-- > lo;) {
        // run = q[i];  q[i-1] = a[i] + b * q[i]
        if (i == 0) break;
        run = fp_add(fp_load<FR>(a + 2 * i), fp_mul(bb, run));
        fp_store<FR>(q + 2 * (i - 1), run);
    }
}

// carry-in of every chunk at one level: c[t] = value the recurrence has reached when it enters chunk t from above,
// i.e. c[chunks-1] = 0 and c[t] = s[t+1] + m * c[t+1] with m = b^(16^(level+1)).  Solved by recursion on {s[t+1]}.
static int kate_carries(DeviceCtx& ctx, const uint4* s, uint32_t chunks, const uint4* pts, uint32_t level, uint4* carry, uint4* scratch, cudaStream_t stream);

// q_out[i-1] = a[i] + m * q[i] for a vector a of length n with multiplier pts[level]; writes n - 1 values ... as a reusable
// step: solve the recurrence for `a` (length n) at `level`, producing q (length n - 1, q[n-1] taken as 0)
static int kate_level(DeviceCtx& ctx, const uint4* a, size_t n, const uint4* pts, uint32_t level, uint4* q, uint4* scratch, cudaStream_t stream) {
    const uint32_t chunks = (uint32_t)((n + POLY_K - 1) / POLY_K);
    if (chunks == 1) {
        H2B_LAUNCH(fr_kate_replay_kernel, 1, 128, 0, stream, a, n, pts + 2 * level, (const uint4*)nullptr, q, 1u);
        return H2B_OK;
    }
    uint4* s = scratch;                     // chunk sums
    uint4* carry = s + 2 * (size_t)chunks;  // carry-ins
    uint4* rest = carry + 2 * (size_t)chunks;
    H2B_LAUNCH(fr_horner_chunk_kernel, (chunks + 127) / 128, 128, 0, stream, a, n, pts + 2 * level, s, chunks);
    H2B_TRY(kate_carries(ctx, s, chunks, pts, level, carry, rest, stream));
    H2B_LAUNCH(fr_kate_replay_kernel, (chunks + 127) / 128, 128, 0, stream, a, n, pts + 2 * level, (const uint4*)carry, q, chunks);
    return H2B_OK;
}

static int kate_carries(DeviceCtx& ctx, const uint4* s, uint32_t chunks, const uint4* pts, uint32_t level, uint4* carry, uint4* scratch, cudaStream_t stream) {
    // c[t-1] = s[t] + m * c[t] for t = chunks-1 .. 1, c[chunks-1] = 0: exactly the kate recurrence on the vector s with
    // multiplier m = pts[level + 1]; its solution q has q[t-1] = c[t-1], and c[chunks-1] = 0 completes it
    H2B_CUDA(cudaMemsetAsync(carry + 2 * (size_t)(chunks - 1), 0, 32, stream));
    return kate_level(ctx, s, chunks, pts, level + 1, carry, scratch, stream);
}

// b on the host (kind = cudaMemcpyHostToDevice) or on the device (cudaMemcpyDeviceToDevice)
static int kate_division(DeviceCtx& ctx, const void* d_a, size_t n, const void* b, cudaMemcpyKind kind, void* d_q, cudaStream_t stream) {
    if (!b || (n && (!d_a || !d_q))) { set_error("kate_division: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n <= 1) return H2B_OK;                 // the quotient of a constant is empty
    if (n > ((size_t)1 << 31)) { set_error("kate_division: at most 2^31 coefficients"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(ctx.scan_scratch.reserve((n / 7 + 256) * 32));
    uint4* pts = (uint4*)ctx.scan_scratch.p;
    uint4* buf = pts + 2 * (POLY_LEVELS_MAX + 1);
    H2B_CUDA(cudaMemcpyAsync(pts + 2 * POLY_LEVELS_MAX, b, 32, kind, stream));
    H2B_LAUNCH(fr_point_powers_kernel, 1, 32, 0, stream, (const uint4*)(pts + 2 * POLY_LEVELS_MAX), POLY_LEVELS_MAX, pts);
    H2B_TRY(kate_level(ctx, (const uint4*)d_a, n, pts, 0, (uint4*)d_q, buf, stream));
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}
int fr_kate_division_run(DeviceCtx& ctx, const void* d_a, size_t n, const uint64_t b[4], void* d_q, cudaStream_t stream) {
    return kate_division(ctx, d_a, n, b, cudaMemcpyHostToDevice, d_q, stream);
}
int fr_kate_division_at_run(DeviceCtx& ctx, const void* d_a, size_t n, const void* d_b, void* d_q, cudaStream_t stream) {
    return kate_division(ctx, d_a, n, d_b, cudaMemcpyDeviceToDevice, d_q, stream);
}

// ---- the grand products themselves --------------------------------------------------------------------------------------
// [UP] halo2_proofs/src/plonk/permutation/prover.rs `Argument::commit` (one call per chunk of columns = one set) and
// [UP] halo2_proofs/src/plonk/lookup/prover.rs `Permuted::commit_product`: both build
//     z[0] = start,  z[i + 1] = z[i] * numerator[i] / denominator[i]
// with the denominators inverted in one batch.  On the device: one elementwise kernel for the denominators, the batch
// inversion, one elementwise kernel for the numerators, the exclusive prefix product, and the scaling by `start`
// (last_z of the previous set).  The blinding rows at the end of z are the caller's (they are random).
static const uint32_t PERM_MAX_COLUMNS = 16;        // columns per launch; a set holds cs.degree() - 2 columns and longer sets run in pieces

struct PermProductParams {
    const uint4* values[PERM_MAX_COLUMNS];
    const uint4* sigma[PERM_MAX_COLUMNS];
    uint32_t m;
    uint32_t j0;            // index of values[0] inside the set (pieces after the first multiply into `out`)
    Fr beta, gamma, delta, deltaomega, omega;
};

// out[i] = prod_j (beta * sigma_j[i] + gamma + v_j[i])
__global__ void __launch_bounds__(128) perm_denominator_kernel(PermProductParams p, size_t n, uint4* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = fp_one<FR>();
    for (uint32_t j = 0; j < p.m; ++j) {
        const Fr t = fp_add(fp_add(fp_mul(p.beta, fp_load<FR>(p.sigma[j] + 2 * i)), p.gamma), fp_load<FR>(p.values[j] + 2 * i));
        acc = j ? fp_mul(acc, t) : t;
    }
    if (p.j0) acc = fp_mul(acc, fp_load<FR>(out + 2 * i));
    fp_store<FR>(out + 2 * i, acc);
}

// out[i] *= prod_j (deltaomega * delta^j * omega^i * beta + gamma + v_j[i])
__global__ void __launch_bounds__(128) perm_numerator_kernel(PermProductParams p, size_t n, uint4* __restrict__ out) {
    const uint32_t stride = gridDim.x * blockDim.x, t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    Fr w = fp_mul(fp_mul(p.deltaomega, p.beta), fp_pow_u32<FR>(p.omega, t));      // deltaomega * beta * omega^i
    if (p.j0) w = fp_mul(w, fp_pow_u32<FR>(p.delta, p.j0));                        // ... * delta^j0 for a later piece of the set
    const Fr step = fp_pow_u32<FR>(p.omega, stride);
    for (size_t i = t; i < n; i += stride) {
        Fr acc = fp_load<FR>(out + 2 * i);
        Fr d = w;
        for (uint32_t j = 0; j < p.m; ++j) {
            acc = fp_mul(acc, fp_add(fp_add(d, p.gamma), fp_load<FR>(p.values[j] + 2 * i)));
            d = fp_mul(d, p.delta);
        }
        fp_store<FR>(out + 2 * i, acc);
        w = fp_mul(w, step);
    }
}

static bool is_montgomery_one(const uint64_t* w) {
    Fr one;
    for (int i = 0; i < 8; ++i) one.l[i] = FpParams<FR>::ONE(i);
    return memcmp(w, one.l, 32) == 0;
}

int permutation_product_run(DeviceCtx& ctx, const void* const* d_values, const void* const* d_sigma, uint32_t m, size_t n, const uint64_t* beta,
                            const uint64_t* gamma, const uint64_t* delta, const uint64_t* deltaomega, const uint64_t* omega, const uint64_t* last_z,
                            void* d_z, cudaStream_t stream) {
    if (!d_z || !beta || !gamma || !delta || !deltaomega || !omega || !last_z || (m && (!d_values || !d_sigma))) {
        set_error("permutation_product: null pointer");
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (m == 0) { set_error("permutation_product: a set has at least one column"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) return H2B_OK;
    if (n > ((size_t)1 << 31)) { set_error("permutation_product: at most 2^31 rows"); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t j = 0; j < m; ++j) if (!d_values[j] || !d_sigma[j]) { set_error("permutation_product: null column"); return H2B_ERR_BAD_ARGUMENT; }
    // sets of more than PERM_MAX_COLUMNS columns (cs.degree() > 18) run in pieces: denominators multiplied up piece by piece,
    // one batch inversion, numerators piece by piece with delta^j carried on
    auto piece = [&](uint32_t j0) {
        PermProductParams p;
        memset(&p, 0, sizeof(p));
        p.m = m - j0 < PERM_MAX_COLUMNS ? m - j0 : PERM_MAX_COLUMNS;
        p.j0 = j0;
        for (uint32_t j = 0; j < p.m; ++j) {
            p.values[j] = (const uint4*)d_values[j0 + j];
            p.sigma[j] = (const uint4*)d_sigma[j0 + j];
        }
        memcpy(p.beta.l, beta, 32); memcpy(p.gamma.l, gamma, 32); memcpy(p.delta.l, delta, 32);
        memcpy(p.deltaomega.l, deltaomega, 32); memcpy(p.omega.l, omega, 32);
        return p;
    };
    for (uint32_t j0 = 0; j0 < m; j0 += PERM_MAX_COLUMNS)
        H2B_LAUNCH(perm_denominator_kernel, (unsigned)((n + 127) / 128), 128, 0, stream, piece(j0), n, (uint4*)d_z);
    H2B_TRY(fr_batch_invert_run(ctx, d_z, n, stream));
    const size_t want = (n + 127) / 128, cap = (size_t)ctx.sm_count * 8;
    for (uint32_t j0 = 0; j0 < m; j0 += PERM_MAX_COLUMNS)
        H2B_LAUNCH(perm_numerator_kernel, (unsigned)(want < cap ? want : cap), 128, 0, stream, piece(j0), n, (uint4*)d_z);
    H2B_TRY(fr_prefix_product_run(ctx, d_z, d_z, n, stream));
    if (!is_montgomery_one(last_z)) H2B_TRY(ntt_scale_run(ctx, d_z, n, last_z, 1, stream));
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// out[i] = (a'[i] + beta) * (s'[i] + gamma)        (denominators)
// out[i] *= (a[i] + beta) * (s[i] + gamma)         (numerators; a, s = the theta-compressed input / table expressions)
struct LookupProductParams { Fr beta, gamma; };
__global__ void __launch_bounds__(128) lookup_product_terms_kernel(const uint4* __restrict__ x, const uint4* __restrict__ y, LookupProductParams p, size_t n,
                                                                 uint4* __restrict__ out, int multiply) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr t = fp_mul(fp_add(fp_load<FR>(x + 2 * i), p.beta), fp_add(fp_load<FR>(y + 2 * i), p.gamma));
    if (multiply) t = fp_mul(t, fp_load<FR>(out + 2 * i));
    fp_store<FR>(out + 2 * i, t);
}

int lookup_product_run(DeviceCtx& ctx, const void* d_compressed_input, const void* d_compressed_table, const void* d_permuted_input,
                       const void* d_permuted_table, size_t n, const uint64_t* beta, const uint64_t* gamma, void* d_z, cudaStream_t stream) {
    if (!beta || !gamma || (n && (!d_compressed_input || !d_compressed_table || !d_permuted_input || !d_permuted_table || !d_z))) {
        set_error("lookup_product: null pointer");
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (n == 0) return H2B_OK;
    if (n > ((size_t)1 << 31)) { set_error("lookup_product: at most 2^31 rows"); return H2B_ERR_BAD_ARGUMENT; }
    LookupProductParams p;
    memcpy(p.beta.l, beta, 32); memcpy(p.gamma.l, gamma, 32);
    const unsigned grid = (unsigned)((n + 127) / 128);
    H2B_LAUNCH(lookup_product_terms_kernel, grid, 128, 0, stream, (const uint4*)d_permuted_input, (const uint4*)d_permuted_table, p, n, (uint4*)d_z, 0);
    H2B_TRY(fr_batch_invert_run(ctx, d_z, n, stream));
    H2B_LAUNCH(lookup_product_terms_kernel, grid, 128, 0, stream, (const uint4*)d_compressed_input, (const uint4*)d_compressed_table, p, n, (uint4*)d_z, 1);
    H2B_TRY(fr_prefix_product_run(ctx, d_z, d_z, n, stream));
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- linear combination of columns -------------------------------------------------------------------------------------
// out[i] (+)= sum_j coeffs[j] * cols[j][i]: the y- and v-weighted sums of committed polynomials in the multi-open argument
// ([UP] halo2_proofs/src/poly/kzg/multiopen/shplonk/prover.rs) and the theta-compression of lookup expressions
// ([UP] plonk/lookup/prover.rs `compress_expressions`).  One pass: every column is read once, out is written once.
static const uint32_t LINCOMB_MAX = 32;
struct LincombParams {
    const uint4* cols[LINCOMB_MAX];
    Fr coeffs[LINCOMB_MAX];
    uint32_t m;
    uint32_t accumulate;
};
__global__ void __launch_bounds__(128) fr_lincomb_kernel(LincombParams p, size_t n, uint4* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = p.accumulate ? fp_load<FR>(out + 2 * i) : fp_zero<FR>();
    for (uint32_t j = 0; j < p.m; ++j) acc = fp_add(acc, fp_mul(p.coeffs[j], fp_load<FR>(p.cols[j] + 2 * i)));
    fp_store<FR>(out + 2 * i, acc);
}

int fr_lincomb_run(DeviceCtx& ctx, const void* const* d_cols, const uint64_t* coeffs, uint32_t m, size_t n, void* d_out, cudaStream_t stream) {
    (void)ctx;
    if (!d_out || (m && (!d_cols || !coeffs))) { set_error("lincomb: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) return H2B_OK;
    if (m == 0) { H2B_CUDA(cudaMemsetAsync(d_out, 0, n * 32, stream)); return H2B_OK; }
    for (uint32_t lo = 0; lo < m; lo += LINCOMB_MAX) {
        LincombParams p;
        memset(&p, 0, sizeof(p));
        p.m = m - lo < LINCOMB_MAX ? m - lo : LINCOMB_MAX;
        p.accumulate = lo ? 1u : 0u;
        for (uint32_t j = 0; j < p.m; ++j) {
            if (!d_cols[lo + j]) { set_error("lincomb: null column"); return H2B_ERR_BAD_ARGUMENT; }
            p.cols[j] = (const uint4*)d_cols[lo + j];
            memcpy(p.coeffs[j].l, coeffs + 4 * (size_t)(lo + j), 32);
        }
        H2B_LAUNCH(fr_lincomb_kernel, (unsigned)((n + 127) / 128), 128, 0, stream, p, n, (uint4*)d_out);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

}  // namespace h2b
