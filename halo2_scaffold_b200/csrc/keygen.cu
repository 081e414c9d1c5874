// Key generation on the device: the σ columns of the permutation argument ([UP] halo2_proofs/src/plonk/permutation/keygen.rs
// Assembly::build_vk / build_pk @ v2023_02_02) and the l_0 / l_last / l_active_row columns of keygen_pk ([UP] plonk/keygen.rs).
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

}  // namespace h2b
