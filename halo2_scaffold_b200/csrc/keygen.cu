// Key generation on the device: the σ columns of the permutation argument ([UP] halo2_proofs/src/plonk/permutation/keygen.rs
// Assembly::build_vk / build_pk @ v2023_02_02), the l_0 / l_last / l_active_row columns of keygen_pk ([UP] plonk/keygen.rs), and
// the exclusion matrix and combination columns of compress_selectors ([UP] plonk/circuit/compress_selectors.rs).
//
// σ_i[j] = δ^c · ω^r for (c, r) = mapping[i][j].  Upstream tabulates deltaomega[c][r] for every (c, r), P x n values; here the
// exponent is split at h = ⌈k/2⌉: ω^r = ω^(r mod 2^h) · ω^(2^h ⌊r / 2^h⌋), and δ^c is folded into the high factor, so that
// σ = lo[r mod 2^h] · hi[c][⌊r / 2^h⌋] with lo 2^h and hi P · 2^(k-h) entries (64 KiB + P · 64 KiB at k = 22): one Fr
// multiplication per entry out of L2-resident tables.  Every output is a unique field value, so this is bit-identical to
// upstream's table lookup.
#include "common.h"

namespace h2b {

static const uint32_t SIGMA_BATCH_MAX = 16;      // columns per launch (blockIdx.y)

struct SigmaTableParams {
    uint32_t delta[8], omega[8];
    uint32_t h, hi_len, lo_len, n_columns;
    uint4* lo;
    uint4* hi;
};

// entry t < lo_len: lo[t] = ω^t;  entry lo_len + c · hi_len + j: hi[c][j] = δ^c · ω^(j · 2^h)
__global__ void __launch_bounds__(128) keygen_sigma_table_kernel(SigmaTableParams p) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = p.lo_len + (size_t)p.n_columns * p.hi_len;
    if (t >= total) return;
    Fr w, d;
#pragma unroll
    for (int i = 0; i < 8; ++i) { w.l[i] = p.omega[i]; d.l[i] = p.delta[i]; }
    if (t < p.lo_len) {
        fp_store<FR>(p.lo + 2 * t, fp_pow_u32(w, (uint32_t)t));
        return;
    }
    const size_t u = t - p.lo_len;
    const uint32_t c = (uint32_t)(u / p.hi_len), j = (uint32_t)(u % p.hi_len);
    fp_store<FR>(p.hi + 2 * u, fp_mul(fp_pow_u32(d, c), fp_pow_u32(w, j << p.h)));
}

struct SigmaCols {
    const uint4* map[SIGMA_BATCH_MAX];   // n pairs of u64 (column, row) = 16 bytes per entry
    uint4* out[SIGMA_BATCH_MAX];
};

// out_y[j] = lo[row mod 2^h] · hi[column][row >> h]; an entry outside [0, n_columns) x [0, n) raises the status word to
// 1 + its flat index (col0 + y) · n + j (saturated at 2^32 - 1) and writes nothing
__global__ void __launch_bounds__(256) keygen_sigma_kernel(SigmaCols cols, uint32_t col0, uint32_t k, uint32_t h, uint32_t n_columns,
                                                           const uint4* __restrict__ lo, const uint4* __restrict__ hi, unsigned* status) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >> k) return;
    const uint4 e = cols.map[blockIdx.y][j];
    const uint64_t column = (uint64_t)e.x | ((uint64_t)e.y << 32), row = (uint64_t)e.z | ((uint64_t)e.w << 32);
    if (column >= n_columns || (row >> k) != 0) {
        const uint64_t flat = ((uint64_t)(col0 + blockIdx.y) << k) + j + 1;
        atomicMax(status, flat > 0xFFFFFFFFull ? 0xFFFFFFFFu : (unsigned)flat);
        return;
    }
    const uint32_t r = (uint32_t)row;
    const Fr a = fp_load<FR>(lo + 2 * (size_t)(r & ((1u << h) - 1)));
    const Fr b = fp_load<FR>(hi + 2 * (((size_t)column << (k - h)) + (r >> h)));
    fp_store<FR>(cols.out[blockIdx.y] + 2 * j, fp_mul(a, b));
}

int permutation_sigma_tables_run(DeviceCtx& ctx, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4], cudaStream_t stream) {
    SigmaTableParams p;
    memcpy(p.delta, delta, 32);
    memcpy(p.omega, omega, 32);
    p.h = (k + 1) / 2;
    p.lo_len = 1u << p.h;
    p.hi_len = 1u << (k - p.h);
    p.n_columns = n_columns;
    const size_t total = p.lo_len + (size_t)n_columns * p.hi_len;
    H2B_TRY(ctx.keygen_tables.reserve(total * 32));
    p.lo = (uint4*)ctx.keygen_tables.p;
    p.hi = p.lo + 2 * (size_t)p.lo_len;
    H2B_LAUNCH(keygen_sigma_table_kernel, (unsigned)((total + 127) / 128), 128, 0, stream, p);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

int permutation_sigma_run(DeviceCtx& ctx, const void* const* d_mapping, uint32_t count, uint32_t col0, uint32_t n_columns, uint32_t k,
                          void* const* d_sigma, void* d_status, cudaStream_t stream) {
    const uint32_t h = (k + 1) / 2;
    const uint4* lo = (const uint4*)ctx.keygen_tables.p;
    const uint4* hi = lo + 2 * ((size_t)1 << h);
    const size_t n = (size_t)1 << k;
    for (uint32_t j0 = 0; j0 < count; j0 += SIGMA_BATCH_MAX) {
        const uint32_t m = count - j0 < SIGMA_BATCH_MAX ? count - j0 : SIGMA_BATCH_MAX;
        SigmaCols c;
        memset(&c, 0, sizeof(c));
        for (uint32_t y = 0; y < m; ++y) {
            c.map[y] = (const uint4*)d_mapping[j0 + y];
            c.out[y] = (uint4*)d_sigma[j0 + y];
        }
        H2B_LAUNCH(keygen_sigma_kernel, dim3((unsigned)((n + 255) / 256), m), 256, 0, stream, c, col0 + j0, k, h, n_columns, lo, hi, (unsigned*)d_status);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// rows [0, n): l0 = e_0, l_last = e_(n-bf-1), l_active_row = 1 on rows 0 .. n-bf-2
__global__ void __launch_bounds__(256) keygen_indicator_kernel(uint4* l0, uint4* l_last, uint4* l_active, uint32_t k, uint32_t last) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >> k) return;
    const Fr one = fp_one<FR>(), zero = fp_zero<FR>();
    fp_store<FR>(l0 + 2 * i, i == 0 ? one : zero);
    fp_store<FR>(l_last + 2 * i, i == last ? one : zero);
    fp_store<FR>(l_active + 2 * i, i < last ? one : zero);
}

// keygen_pk's three indicator columns: filled in Lagrange form, then lagrange_to_coeff and coeff_to_extended as one batch.
// By linearity l_active_row = 1 - (l_last + l_blind) = ext(coeff(1 on rows 0 .. n-bf-2)), so l_blind is never formed.
int keygen_indicators_run(DeviceCtx& ctx, uint32_t k, uint32_t extended_k, uint32_t blinding_factors, const uint64_t omega_inv[4],
                          const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], void* const* d_cols /*3*/,
                          cudaStream_t stream) {
    const size_t n = (size_t)1 << k;
    H2B_LAUNCH(keygen_indicator_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (uint4*)d_cols[0], (uint4*)d_cols[1], (uint4*)d_cols[2], k,
               (uint32_t)(n - blinding_factors - 1));
    H2B_CUDA(cudaGetLastError());
    H2B_TRY(lagrange_to_coeff_batch_run(ctx, d_cols, 3, k, omega_inv, ifft_divisor, stream));
    return coeff_to_extended_batch_run(ctx, d_cols, 3, k, extended_k, extended_omega, zeta_powers, stream);
}

// ---- selectors: compress_selectors' exclusion matrix and combination columns ([UP] plonk/circuit/compress_selectors.rs) --------
// A selector's activations (Rust Vec<bool>: n bytes of 0 / 1) are packed into n / 32 words, bit j of word w = row 32 w + j.

__device__ __forceinline__ uint32_t nonzero_bytes(uint32_t y) {
    return ((y & 0xFFu) ? 1u : 0u) | ((y & 0xFF00u) ? 2u : 0u) | ((y & 0xFF0000u) ? 4u : 0u) | ((y & 0xFF000000u) ? 8u : 0u);
}

__global__ void __launch_bounds__(256) keygen_selector_pack_kernel(const uint8_t* __restrict__ act, size_t n, uint32_t* __restrict__ bits) {
    const size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= selector_words(n)) return;
    uint32_t x = 0;
    if (32 * (w + 1) <= n) {
        const uint4* p = (const uint4*)(act + 32 * w);
        const uint4 a = p[0], b = p[1];
        const uint32_t y[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) x |= nonzero_bytes(y[i]) << (4 * i);
    } else {
        for (size_t r = 32 * w; r < n; ++r) x |= (act[r] ? 1u : 0u) << (r - 32 * w);
    }
    bits[w] = x;
}

int selector_pack_run(DeviceCtx&, const void* d_activations, size_t n, void* d_bits, cudaStream_t stream) {
    const size_t W = selector_words(n);
    H2B_LAUNCH(keygen_selector_pack_kernel, (unsigned)((W + 255) / 256), 256, 0, stream, (const uint8_t*)d_activations, n, (uint32_t*)d_bits);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

static const uint32_t EXCL_TILE = 64;     // selectors per side of a tile pair
static const uint32_t EXCL_WORDS = 32;    // bitset words (1024 rows) per block

// One block: a chunk of EXCL_WORDS words of the selectors of tile pair (ti, tj), ti >= tj (blockIdx.y = ti (ti + 1) / 2 + tj).  Each
// word of every bitset is read from memory once per tile pair -- once in all when S <= 64 -- and thread (i, q) ORs a_i & a_j over the
// chunk for the 16 selectors j = q, q + 4, ..; a pair that meets sets flags[i S + j] (i > j).
__global__ void __launch_bounds__(256) keygen_selector_exclusion_kernel(const uint32_t* __restrict__ bits, uint32_t S, size_t W, uint32_t* flags) {
    __shared__ uint32_t a[EXCL_TILE][EXCL_WORDS + 1], b[EXCL_TILE][EXCL_WORDS + 1];
    const uint32_t p = blockIdx.y;
    uint32_t ti = 0;
    while ((ti + 1) * (ti + 2) / 2 <= p) ++ti;
    const uint32_t tj = p - ti * (ti + 1) / 2;
    const size_t w0 = (size_t)blockIdx.x * EXCL_WORDS;
    for (uint32_t t = threadIdx.x; t < EXCL_TILE * EXCL_WORDS; t += blockDim.x) {
        const uint32_t s = t / EXCL_WORDS, w = t % EXCL_WORDS;
        const uint32_t si = ti * EXCL_TILE + s, sj = tj * EXCL_TILE + s;
        const size_t ww = w0 + w;
        a[s][w] = (si < S && ww < W) ? bits[(size_t)si * W + ww] : 0u;
        b[s][w] = (sj < S && ww < W) ? bits[(size_t)sj * W + ww] : 0u;
    }
    __syncthreads();
    const uint32_t i = threadIdx.x >> 2, q = threadIdx.x & 3;
    uint32_t acc[EXCL_TILE / 4];
#pragma unroll
    for (uint32_t u = 0; u < EXCL_TILE / 4; ++u) acc[u] = 0;
    for (uint32_t w = 0; w < EXCL_WORDS; ++w) {
        const uint32_t x = a[i][w];
#pragma unroll
        for (uint32_t u = 0; u < EXCL_TILE / 4; ++u) acc[u] |= x & b[q + 4 * u][w];
    }
    const uint32_t gi = ti * EXCL_TILE + i;
    if (gi >= S) return;
#pragma unroll
    for (uint32_t u = 0; u < EXCL_TILE / 4; ++u) {
        const uint32_t gj = tj * EXCL_TILE + q + 4 * u;
        uint32_t* f = flags + (size_t)gi * S + gj;
        if (gj < gi && acc[u] && !*f) *f = 1;
    }
}

int selector_exclusion_run(DeviceCtx&, const void* d_bits, uint32_t n_selectors, size_t n, void* d_flags, cudaStream_t stream) {
    const size_t W = selector_words(n);
    const uint32_t tiles = (n_selectors + EXCL_TILE - 1) / EXCL_TILE;
    H2B_CUDA(cudaMemsetAsync(d_flags, 0, (size_t)n_selectors * n_selectors * 4, stream));
    const dim3 grid((unsigned)((W + EXCL_WORDS - 1) / EXCL_WORDS), tiles * (tiles + 1) / 2);
    H2B_LAUNCH(keygen_selector_exclusion_kernel, grid, 256, 0, stream, (const uint32_t*)d_bits, n_selectors, W, (uint32_t*)d_flags);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// out[j] = F::from(root_m) (Montgomery) for the member m active on row j, 0 on rows where none is.  Members are (bitset slot, root)
// pairs.  A row where two members are active raises the status word to 1 + (combination << k) + j (saturated) and writes nothing.
__global__ void __launch_bounds__(256) keygen_combination_kernel(const uint32_t* __restrict__ bits, size_t W, const uint2* __restrict__ members,
                                                                 uint32_t n_members, uint32_t combination, uint32_t k, uint4* out, unsigned* status) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >> k) return;
    uint32_t root = 0, hits = 0;
    for (uint32_t m = 0; m < n_members; ++m) {
        const uint2 e = members[m];
        if ((bits[(size_t)e.x * W + (j >> 5)] >> (j & 31)) & 1u) { root = e.y; ++hits; }
    }
    if (hits > 1) {
        const uint64_t flat = ((uint64_t)combination << k) + j + 1;
        atomicMax(status, flat > 0xFFFFFFFFull ? 0xFFFFFFFFu : (unsigned)flat);
        return;
    }
    Fr v = fp_zero<FR>();
    if (root) {
        v.l[0] = root;
        v = fp_to_mont(v);
    }
    fp_store<FR>(out + 2 * j, v);
}

int combination_column_run(DeviceCtx&, const void* d_bits, const void* d_members, uint32_t n_members, uint32_t combination, uint32_t k, void* d_out,
                           void* d_status, cudaStream_t stream) {
    const size_t n = (size_t)1 << k;
    H2B_LAUNCH(keygen_combination_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (const uint32_t*)d_bits, selector_words(n), (const uint2*)d_members,
               n_members, combination, k, (uint4*)d_out, (unsigned*)d_status);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

}  // namespace h2b
