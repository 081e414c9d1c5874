// The lookup argument's permutation of its input / table columns on the device:
// [UP] halo2_proofs/src/plonk/lookup/prover.rs `permute_expression_pair`.  Upstream, per lookup and on one core:
//     A' = sort(A[..usable_rows])                                   (Fr's Ord = order of the canonical integers)
//     leftover = multiset(S[..usable_rows]) as a BTreeMap value -> count
//     row by row: a first occurrence of a value in A' puts that value into S' at the same row and takes one instance out of
//     leftover (an input value that is not in the table is an error); repeated rows are collected;
//     then the leftover table values, ascending, fill the repeated rows taken from the END of that list.
// Here:
//   * both columns leave Montgomery form and are sorted by a bitonic network on the 8-limb canonical keys.  Equal keys are
//     indistinguishable, so no stability is needed; compare-exchange distances below the tile run in shared memory
//     (limb-major layout), larger ones as streaming passes, two distances per pass.  Padding up to a power of two is the all-ones key;
//   * first occurrences, the match of every distinct input value to the first equal table entry (binary search in the
//     sorted table) and the fill are elementwise kernels; the ranks of the repeated rows and of the unmatched table entries are two
//     exclusive scans (scan.cu's u32_exclusive_scan).  The order of the fill is exactly upstream's: the i-th smallest leftover value goes to the
//     i-th repeated row counted from the end.
// Rows at and beyond usable_rows (the blinding rows) are the caller's.
#include "keys.cuh"

namespace h2b {

// canonical keys of the first `usable` rows, all-ones padding up to `padded`
__global__ void __launch_bounds__(256) lookup_keys_kernel(const uint4* __restrict__ in, uint32_t usable, uint32_t padded, uint4* __restrict__ keys) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= padded) return;
    if (i < usable) {
        fp_store<FR>(keys + 2 * (size_t)i, fp_from_mont(fp_load<FR>(in + 2 * (size_t)i)));
    } else {
        keys[2 * (size_t)i] = make_uint4(~0u, ~0u, ~0u, ~0u);
        keys[2 * (size_t)i + 1] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
}

// one compare-exchange pass of the bitonic network at distance j inside sorted runs of length k (global memory)
__global__ void __launch_bounds__(256) bitonic_global_kernel(uint4* __restrict__ keys, uint32_t half, uint32_t j, uint32_t k) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= half) return;
    const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), p = i | j;
    const bool up = (i & k) == 0;
    Key a = key_load(keys, i), b = key_load(keys, p);
    if (key_less(b, a) == up) {
        key_store(keys, i, b);
        key_store(keys, p, a);
    }
}

// two consecutive passes (distances j and j / 2, both >= SORT_TILE) in one sweep over memory: a thread owns the four keys of one
// two-level butterfly, so every key is read and written once for two levels of the network
__device__ __forceinline__ void key_cmpx(Key& a, Key& b, bool up) {
    if (key_less(b, a) == up) { const Key t = a; a = b; b = t; }
}
__global__ void __launch_bounds__(256) bitonic_global2_kernel(uint4* __restrict__ keys, uint32_t quarter, uint32_t j, uint32_t k) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= quarter) return;
    const uint32_t h = j >> 1;
    const uint32_t i00 = ((t & ~(h - 1)) << 2) | (t & (h - 1)), i01 = i00 | h, i10 = i00 | j, i11 = i10 | h;
    const bool up = (i00 & k) == 0;                    // j < k: the four keys lie in the same run of length k
    Key a = key_load(keys, i00), b = key_load(keys, i01), c = key_load(keys, i10), d = key_load(keys, i11);
    key_cmpx(a, c, up); key_cmpx(b, d, up);            // distance j
    key_cmpx(a, b, up); key_cmpx(c, d, up);            // distance j / 2
    key_store(keys, i00, a); key_store(keys, i01, b); key_store(keys, i10, c); key_store(keys, i11, d);
}

// three consecutive passes (distances j, j / 2, j / 4, all >= SORT_TILE) in one sweep: a thread owns the eight keys of a three-level
// butterfly (64 registers of keys).  The sort is bound by its sweeps over HBM: 2^22 rows need 30 + 13 of them instead of 42 + 13
__global__ void __launch_bounds__(256) bitonic_global3_kernel(uint4* __restrict__ keys, uint32_t eighth, uint32_t j, uint32_t k) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= eighth) return;
    const uint32_t h = j >> 1, q = j >> 2;
    const uint32_t i0 = ((t & ~(q - 1)) << 3) | (t & (q - 1));
    const bool up = (i0 & k) == 0;
    Key v[8];
#pragma unroll
    for (int x = 0; x < 8; ++x) v[x] = key_load(keys, i0 | ((x & 4) ? j : 0u) | ((x & 2) ? h : 0u) | ((x & 1) ? q : 0u));
#pragma unroll
    for (int x = 0; x < 4; ++x) key_cmpx(v[x], v[x + 4], up);                          // distance j
#pragma unroll
    for (int x = 0; x < 8; ++x) if (!(x & 2)) key_cmpx(v[x], v[x + 2], up);            // distance j / 2
#pragma unroll
    for (int x = 0; x < 8; x += 2) key_cmpx(v[x], v[x + 1], up);                       // distance j / 4
#pragma unroll
    for (int x = 0; x < 8; ++x) key_store(keys, i0 | ((x & 4) ? j : 0u) | ((x & 2) ? h : 0u) | ((x & 1) ? q : 0u), v[x]);
}

// all passes with distance < SORT_TILE of one tile in shared memory.  k_lo == 0: the whole network up to runs of SORT_TILE
// (the first phase); otherwise the tail j = min(k_lo, SORT_TILE) / 2 ... 1 of the stage with run length k_lo.
__global__ void __launch_bounds__(512) bitonic_shared_kernel(uint4* __restrict__ keys, uint32_t count, uint32_t k_lo) {
    __shared__ uint32_t sh[8][SORT_TILE];
    const uint32_t base = blockIdx.x * SORT_TILE;
    for (uint32_t e = threadIdx.x; e < SORT_TILE; e += blockDim.x) {
        Key v;
        if (base + e < count) v = key_load(keys, base + e);
        else {
#pragma unroll
            for (int l = 0; l < 8; ++l) v.l[l] = ~0u;
        }
#pragma unroll
        for (int l = 0; l < 8; ++l) sh[l][e] = v.l[l];
    }
    __syncthreads();
    const uint32_t k_first = k_lo ? k_lo : 2, k_last = k_lo ? k_lo : SORT_TILE;
    for (uint32_t k = k_first; k <= k_last; k <<= 1) {
        uint32_t j = k >> 1;
        if (j >= SORT_TILE) j = SORT_TILE >> 1;
        for (; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < SORT_TILE / 2; t += blockDim.x) {
                const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), p = i | j;
                const bool up = ((base + i) & k) == 0;
                Key a, b;
#pragma unroll
                for (int l = 0; l < 8; ++l) { a.l[l] = sh[l][i]; b.l[l] = sh[l][p]; }
                if (key_less(b, a) == up) {
#pragma unroll
                    for (int l = 0; l < 8; ++l) { sh[l][i] = b.l[l]; sh[l][p] = a.l[l]; }
                }
            }
            __syncthreads();
        }
        if (k == 0x80000000u) break;
    }
    for (uint32_t e = threadIdx.x; e < SORT_TILE; e += blockDim.x) {
        if (base + e >= count) continue;
        Key v;
#pragma unroll
        for (int l = 0; l < 8; ++l) v.l[l] = sh[l][e];
        key_store(keys, base + e, v);
    }
}

int bitonic_sort(uint4* keys, uint32_t padded, cudaStream_t stream) {      // padded: a power of two
    const uint32_t tiles = (padded + SORT_TILE - 1) / SORT_TILE;
    H2B_LAUNCH(bitonic_shared_kernel, tiles, 512, 0, stream, keys, padded, 0u);
    for (uint32_t k = SORT_TILE << 1; k != 0 && k <= padded; k <<= 1) {
        uint32_t j = k >> 1;
        static int three = -1;
        if (three < 0) { const char* e = getenv("H2B_SORT_THREE"); three = e ? atoi(e) : 1; }
        for (; three && j >= 4 * SORT_TILE; j >>= 3)    // three distances per sweep while all are >= SORT_TILE
            H2B_LAUNCH(bitonic_global3_kernel, (padded / 8 + 255) / 256, 256, 0, stream, keys, padded / 8, j, k);
        for (; j >= 2 * SORT_TILE; j >>= 2)             // two distances per sweep while both are >= SORT_TILE
            H2B_LAUNCH(bitonic_global2_kernel, (padded / 4 + 255) / 256, 256, 0, stream, keys, padded / 4, j, k);
        if (j >= SORT_TILE) H2B_LAUNCH(bitonic_global_kernel, (padded / 2 + 255) / 256, 256, 0, stream, keys, padded / 2, j, k);
        H2B_LAUNCH(bitonic_shared_kernel, tiles, 512, 0, stream, keys, padded, k);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- matching the sorted input against the sorted table --------------------------------------------------------------------
// repeated[r] = 1 when A'[r] == A'[r-1]; a first occurrence claims the first table entry equal to it (used[p] = 1)
__global__ void __launch_bounds__(256) lookup_match_kernel(const uint4* __restrict__ a, const uint4* __restrict__ t, uint32_t usable,
                                                         uint32_t* __restrict__ repeated, uint32_t* __restrict__ used, uint32_t* __restrict__ missing) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= usable) return;
    const Key v = key_load(a, r);
    const bool rep = r > 0 && key_eq(v, key_load(a, r - 1));
    repeated[r] = rep ? 1u : 0u;
    if (rep) return;
    uint32_t lo = 0, hi = usable;                    // lower bound of v in t[0, usable)
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (key_less(key_load(t, mid), v)) lo = mid + 1; else hi = mid;
    }
    if (lo < usable && key_eq(key_load(t, lo), v)) used[lo] = 1u;
    else atomicMax(missing, r + 1);                  // an input value that the table does not hold
}
__global__ void __launch_bounds__(256) lookup_invert_flags_kernel(const uint32_t* __restrict__ used, uint32_t usable, uint32_t* __restrict__ unused) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < usable) unused[p] = used[p] ? 0u : 1u;
}
// rows_of_rank[rank of repeated row r] = r
__global__ void __launch_bounds__(256) lookup_repeated_rows_kernel(const uint32_t* __restrict__ repeated, const uint32_t* __restrict__ rank_r, uint32_t usable,
                                                                 uint32_t* __restrict__ rows_of_rank) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < usable && repeated[r]) rows_of_rank[rank_r[r]] = r;
}
// S'[r] = A'[r] on first occurrences; the i-th unmatched table entry (ascending) goes to the i-th repeated row from the end.
// Outputs return to Montgomery form.
__global__ void __launch_bounds__(256) lookup_fill_kernel(const uint4* __restrict__ a, const uint4* __restrict__ t, uint32_t usable,
                                                        const uint32_t* __restrict__ repeated, const uint32_t* __restrict__ rank_r,
                                                        const uint32_t* __restrict__ unused, const uint32_t* __restrict__ rank_l,
                                                        const uint32_t* __restrict__ rows_of_rank, uint4* __restrict__ out_input, uint4* __restrict__ out_table) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= usable) return;
    const Fr av = fp_to_mont(fp_load<FR>(a + 2 * (size_t)i));
    fp_store<FR>(out_input + 2 * (size_t)i, av);
    if (!repeated[i]) fp_store<FR>(out_table + 2 * (size_t)i, av);
    if (unused[i]) {
        const uint32_t n_repeated = rank_r[usable], n_left = rank_l[usable];
        const uint32_t q = rank_l[i];
        if (n_left == n_repeated && q < n_repeated) {
            const uint32_t row = rows_of_rank[n_repeated - 1 - q];
            fp_store<FR>(out_table + 2 * (size_t)row, fp_to_mont(fp_load<FR>(t + 2 * (size_t)i)));
        }
    }
}

int lookup_permute_run(DeviceCtx& ctx, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                       void* d_status, cudaStream_t stream) {
    if (usable_rows == 0) {
        if (d_status) H2B_CUDA(cudaMemsetAsync(d_status, 0, 4, stream));
        return H2B_OK;
    }
    if (!d_input || !d_table || !d_permuted_input || !d_permuted_table) { set_error("lookup_permute: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (usable_rows > (1u << 28)) { set_error("lookup_permute: at most 2^28 rows"); return H2B_ERR_BAD_ARGUMENT; }
    uint32_t padded = SORT_TILE;
    while (padded < usable_rows) padded <<= 1;
    const size_t key_bytes = (size_t)padded * 32, flag_bytes = ((size_t)usable_rows + 1 + 3) / 4 * 16;
    const uint32_t nblocks = (usable_rows + SCAN_BLOCK - 1) / SCAN_BLOCK;
    H2B_TRY(ctx.lookup_scratch.reserve(2 * key_bytes + 7 * flag_bytes + ((size_t)nblocks + 2) * 4 + 64));
    char* base = (char*)ctx.lookup_scratch.p;
    uint4* ka = (uint4*)base;
    uint4* kt = (uint4*)(base + key_bytes);
    uint32_t* repeated = (uint32_t*)(base + 2 * key_bytes);
    uint32_t* used = (uint32_t*)((char*)repeated + flag_bytes);
    uint32_t* unused = (uint32_t*)((char*)used + flag_bytes);
    uint32_t* rank_r = (uint32_t*)((char*)unused + flag_bytes);
    uint32_t* rank_l = (uint32_t*)((char*)rank_r + flag_bytes);
    uint32_t* rows_of_rank = (uint32_t*)((char*)rank_l + flag_bytes);
    uint32_t* missing = (uint32_t*)((char*)rows_of_rank + flag_bytes);
    uint32_t* sums = missing + 16;
    const unsigned gp = (padded + 255) / 256, gu = (usable_rows + 255) / 256;
    H2B_LAUNCH(lookup_keys_kernel, gp, 256, 0, stream, (const uint4*)d_input, usable_rows, padded, ka);
    H2B_LAUNCH(lookup_keys_kernel, gp, 256, 0, stream, (const uint4*)d_table, usable_rows, padded, kt);
    H2B_TRY(bitonic_sort(ka, padded, stream));
    H2B_TRY(bitonic_sort(kt, padded, stream));
    H2B_CUDA(cudaMemsetAsync(used, 0, flag_bytes, stream));
    H2B_CUDA(cudaMemsetAsync(missing, 0, 4, stream));
    H2B_LAUNCH(lookup_match_kernel, gu, 256, 0, stream, (const uint4*)ka, (const uint4*)kt, usable_rows, repeated, used, missing);
    H2B_LAUNCH(lookup_invert_flags_kernel, gu, 256, 0, stream, (const uint32_t*)used, usable_rows, unused);
    H2B_TRY(u32_exclusive_scan(repeated, usable_rows, rank_r, nullptr, sums, stream));
    H2B_TRY(u32_exclusive_scan(unused, usable_rows, rank_l, nullptr, sums, stream));
    H2B_LAUNCH(lookup_repeated_rows_kernel, gu, 256, 0, stream, (const uint32_t*)repeated, (const uint32_t*)rank_r, usable_rows, rows_of_rank);
    H2B_LAUNCH(lookup_fill_kernel, gu, 256, 0, stream, (const uint4*)ka, (const uint4*)kt, usable_rows, (const uint32_t*)repeated, (const uint32_t*)rank_r,
               (const uint32_t*)unused, (const uint32_t*)rank_l, (const uint32_t*)rows_of_rank, (uint4*)d_permuted_input, (uint4*)d_permuted_table);
    H2B_CUDA(cudaGetLastError());
    // upstream returns Err(ConstraintSystemFailure) for an input value the table does not hold.  With a status word the verdict is left
    // on the device (0 = satisfied, otherwise 1 + the sorted row of a missing value) and the call stays asynchronous; without one
    // the call synchronises and fails
    if (d_status) {
        H2B_CUDA(cudaMemcpyAsync(d_status, missing, 4, cudaMemcpyDeviceToDevice, stream));
        return H2B_OK;
    }
    uint32_t miss = 0;
    H2B_CUDA(cudaMemcpyAsync(&miss, missing, 4, cudaMemcpyDeviceToHost, stream));
    H2B_CUDA(cudaStreamSynchronize(stream));
    if (miss) { set_error("lookup_permute: the input value at sorted row %u is not in the table (ConstraintSystemFailure)", miss - 1); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

}  // namespace h2b
