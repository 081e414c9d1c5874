// BN254 G1 multi-scalar multiplication for sm_100a -- the device side of `best_multiexp`
// ([UP] halo2_proofs/src/arithmetic.rs::best_multiexp / multiexp_serial @ v2023_02_02; SURVEY.md
// section 8 rows a1/a2; reached through ParamsKZG::commit{,_lagrange} from src/scaffold.rs:132,135,
// 191-199,207-214,223,284,287,322-346,354 and examples/standard_plonk.rs:33,34,41-49,57).
//
// Contract (identical to the reference): scalars n x 32 B (Fr, Montgomery), bases n x 64 B
// (G1Affine x|y Montgomery, (0,0) = identity) -> sum_i s_i * P_i as a Jacobian triple whose
// affine value is the unique group element the reference computes.
//
// Algorithm (all on the device, no host arithmetic):
//   0. (registered SRS vectors only, once) precompute T_j[i] = 2^(c0*j) * P_i, j < W0, in affine form.  With the
//      tables resident every window of a scalar lands in ONE shared bucket set, so the MSM needs no doublings at
//      all and its bucket reduction shrinks from W sets to c0/c sets (SURVEY.md 8d: "precomputed multiples");
//   1. decompose: leave Montgomery form, map s > (r-1)/2 to (r - s, -P) so that "small negative" witness values
//      stay small, recode into W signed c-bit digits |d| <= 2^(c-1); window w uses table w / m and bucket set
//      w % m (plain, table-less mode: m = W, i.e. one bucket set per window); histogram with global reductions;
//   2. exclusive scan of the histogram; counting-sort scatter of (table row | sign) by bucket;
//   3. accumulate: the sorted list is cut into G equal slices, one per thread, regardless of bucket boundaries
//      (perfect balance for any scalar distribution: 50 % zeros, a bucket holding 20 % of the column ...).  A
//      thread adds the gathered affine points of its slice into an XYZZ accumulator (8M + 2S per point, next
//      point prefetched) and flushes it whenever the bucket changes; the piece of a bucket that started in an
//      earlier slice goes to a per-thread "head partial" instead;
//   4. combine: buckets cut by a slice boundary get their head partials added (one thread per bucket; one CTA
//      per bucket for buckets cut into many pieces);
//   5. bucket reduction sum_b b * B_b per set as a hierarchy of chunked running sums, Horner over the (few)
//      sets, conversion to Jacobian.
#include "common.h"
#include "ec.cuh"

namespace h2b {

static const uint32_t SIGN_BIT = 0x80000000u;

// scattered 4-byte stores of the counting sort: evict-first, so that they do not push the bucket cursors out of L2
#if defined(H2B_EMU) || defined(H2B_NO_STREAMING_STORES)
#define H2B_STORE_STREAMING(ptr, val) (*(ptr) = (val))
#else
#define H2B_STORE_STREAMING(ptr, val) __stcs((ptr), (val))
#endif

struct MsmPlan {
    uint32_t n;          // scalars in this (sub-)MSM
    uint32_t c;          // window bits
    uint32_t W;          // windows over the scalar
    uint32_t m;          // bucket sets: window w -> set w % m, table w / m
    uint32_t Nb;         // buckets per set = 2^(c-1), ids 1..Nb
    uint32_t B;          // m * Nb
    uint32_t stride;     // rows between consecutive tables
    uint32_t row0;       // first row of this call inside each table
    uint32_t G;          // slices (accumulate threads)
    uint32_t add_into;   // 1: chunked MSM -- each chunk's bucket sums are merged into running accumulators
    uint32_t top_bins;   // > 0: the top window only has this many digit values (few scalar bits left): its histogram and
                         //      cursor atomics are aggregated per CTA in shared memory instead of hammering 2-4 counters
    uint32_t ncols;      // batched MSM: independent scalar columns over the same points (blockIdx.y of the sort kernels); column j owns
                         //      bucket sets [j * m, (j + 1) * m), so B = ncols * m * Nb and everything after the sort is unchanged
    uint32_t pb;         // > 0: partitioned sort (section 2c): buckets are grouped into partitions of 2^pb, P = ceil(B / 2^pb) of them
};

// scalar columns of a batched MSM (one sort / accumulate / reduce sequence for all of them): the columns a proof phase commits
// are independent MSMs over the same SRS vector ([UP] plonk/prover.rs commits advice / lookup / permutation columns one by one);
// at k <= 20 a single column is latency bound (bucket reduction depth), a batch shares every dependent step
static const uint32_t MSM_BATCH_MAX = 32;
struct MsmCols {
    const uint4* scalars[MSM_BATCH_MAX];
    uint32_t len[MSM_BATCH_MAX];
};

static const uint32_t TOP_BINS_MAX = 1026;      // top windows of up to 10 bits (+ carry) are aggregated

// (r - 1) / 2 as canonical 32-bit limbs
__device__ __forceinline__ bool fr_gt_half(const Fr& s) {
    const uint32_t H[8] = {0xf8000000u, 0xa1f0fac9u, 0x3cdcb848u, 0x9419f424u, 0x40c0ac2eu, 0xdc2822dbu, 0x7098d014u, 0x18322739u};
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        if (s.l[i] > H[i]) return true;
        if (s.l[i] < H[i]) return false;
    }
    return false;
}

// s >>= c (0 < c < 32): the window loop takes the low c bits and shifts, instead of selecting two limbs by a run-time index per window
// (8 funnel shifts against ~35 compare / select instructions: the recoding is what bounds the decompose kernels on sparse columns)
__device__ __forceinline__ void fr_shift_right(Fr& s, uint32_t c) {
#pragma unroll
    for (int i = 0; i < 7; ++i) s.l[i] = (s.l[i] >> c) | (s.l[i + 1] << (32 - c));
    s.l[7] >>= c;
}

// scalar -> signed window digits.  Calls emit(w, set, d, sign) for every window (d == 0: no entry)
template <class F>
__device__ __forceinline__ void msm_recode(const uint4* __restrict__ scalars, uint32_t i, bool live, const MsmPlan& pl, F emit) {
    const uint32_t c = pl.c, half = 1u << (c - 1);
    Fr s = fp_zero<FR>();
    uint32_t neg = 0;
    if (live) {
        s = fp_from_mont(fp_load<FR>(scalars + 2 * (size_t)i));
        if (fr_gt_half(s)) {
            Fr r;
#pragma unroll
            for (int k = 0; k < 8; ++k) r.l[k] = FpParams<FR>::P(k);
            uint32_t borrow = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                uint64_t d = (uint64_t)r.l[k] - s.l[k] - borrow;
                s.l[k] = (uint32_t)d;
                borrow = (uint32_t)(d >> 63);
            }
            neg = SIGN_BIT;
        }
    }
    uint32_t carry = 0, set = 0;
    const uint32_t mask = (1u << c) - 1;
    for (uint32_t w = 0; w < pl.W; ++w) {
        uint32_t d = (s.l[0] & mask) + carry;
        fr_shift_right(s, c);
        uint32_t sign = neg;
        if (d > half) { d = (1u << c) - d; carry = 1; sign ^= SIGN_BIT; }
        else carry = 0;
        emit(w, set, d, sign);
        if (++set == pl.m) set = 0;
    }
}

// ---- 2c. partitioned sort ------------------------------------------------------------------------------------------------
// The one-pass counting sort (sections 1-2) issues one returning L2 atomic and one scattered 4-byte store per entry.  At 2^24
// points that is 218 M of each: ncu shows the kernel waiting on them (long-scoreboard 226 cycles per issue, L2 45 %, DRAM write
// amplification 2.7x because 2^19 half-written 128-byte lines do not stay in the L2), 4.1 ms + 1.2 ms for the histogram's
// reductions.  Here the sort is done in two levels that keep every random access on chip:
//   digits    (msm_decompose_kernel, pb > 0): digits as before, but only a histogram over P ~ 512 PARTITIONS of 2^pb buckets,
//             taken in shared memory and flushed with P global reductions per CTA;
//   partition (msm_partition_kernel): a CTA takes a tile of scalars, groups its entries by partition in shared memory and
//             appends each group to the partition's region of an intermediate list as one contiguous run (8-byte entries
//             bucket | row+sign): coalesced writes, P global atomics per tile instead of one per entry;
//   place     (msm_place_kernel): one CTA per partition counts its buckets in shared memory, scans them -- this yields
//             offsets[] -- and places every entry at its final position with shared-memory cursors; the partition's slice of
//             the sorted list (a few MB) is written while it is L2-resident.
static const uint32_t PART_MAX = 2048;            // partitions (shared-memory histogram of the first two kernels)
static const uint32_t PART_TILE_ENTRIES = 12288;  // entries staged per tile: 96 KiB of shared memory
static const uint32_t PART_W_MAX = 16;            // windows per scalar kept in registers by msm_partition_kernel
static const uint32_t PLACE_MAX_LOG = 13;         // buckets per partition in the place kernels: 32 KiB of cursors

__device__ __forceinline__ void msm_decompose_partitions(const MsmCols& cols, const MsmPlan& pl, uint32_t* __restrict__ digits, uint32_t* __restrict__ part_counts) {
    __shared__ uint32_t part_hist[PART_MAX];
    const uint32_t col = blockIdx.y;
    digits += (size_t)col * pl.W * pl.n;
    const uint4* __restrict__ scalars = cols.scalars[col];
    const uint32_t col_len = cols.len[col];
    const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
    const uint32_t gbase = col * pl.m * pl.Nb;
    for (uint32_t b = threadIdx.x; b < P; b += blockDim.x) part_hist[b] = 0;
    __syncthreads();
    const uint32_t rounds = (pl.n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (uint32_t round = 0; round < rounds; ++round) {
        const uint32_t i = (round * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        if (i >= col_len) continue;
        // the digits are kept (window-major, like the one-pass sort's): msm_partition_kernel reads them back instead of recoding the
        // scalar -- the recoding (one Montgomery multiplication + 13 extractions) made both kernels instruction bound
        msm_recode(scalars, i, true, pl, [&](uint32_t w, uint32_t set, uint32_t d, uint32_t sign) {
            if (d) atomicAdd(&part_hist[(gbase + set * pl.Nb + d - 1) >> pl.pb], 1u);
            digits[(size_t)w * pl.n + i] = d ? (d | sign) : 0u;
        });
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < P; b += blockDim.x)
        if (part_hist[b]) atomicAdd(&part_counts[b], part_hist[b]);
}

// exclusive scans over the P partition totals: entries -> part_off[0..P] (+ a copy: the append cursors), and chunks of
// 2^chunk_log entries -> chunk0[0..P] (the place kernels work on chunks, so that a partition holding far more than its share --
// the narrow top window of uniform scalars, the ones and zeros of a witness column -- is spread over many CTAs)
__global__ void __launch_bounds__(1024) msm_partition_scan_kernel(const uint32_t* __restrict__ part_counts, uint32_t P, uint32_t chunk_log,
                                                                uint32_t* __restrict__ part_off, uint32_t* __restrict__ part_cursor, uint32_t* __restrict__ chunk0) {
    __shared__ uint32_t sh[1024], sh2[1024];
    __shared__ uint32_t carry_sh, carry2_sh;
    if (threadIdx.x == 0) { carry_sh = 0; carry2_sh = 0; }
    __syncthreads();
    for (uint32_t start = 0; start < P; start += 1024) {
        const uint32_t idx = start + threadIdx.x;
        const uint32_t v = idx < P ? part_counts[idx] : 0;
        const uint32_t v2 = (v + (1u << chunk_log) - 1) >> chunk_log;
        sh[threadIdx.x] = v;
        sh2[threadIdx.x] = v2;
        __syncthreads();
        for (uint32_t o = 1; o < 1024; o <<= 1) {
            const uint32_t add = threadIdx.x >= o ? sh[threadIdx.x - o] : 0, add2 = threadIdx.x >= o ? sh2[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += add;
            sh2[threadIdx.x] += add2;
            __syncthreads();
        }
        const uint32_t incl = sh[threadIdx.x], carry = carry_sh, incl2 = sh2[threadIdx.x], carry2 = carry2_sh;
        if (idx < P) { part_off[idx] = carry + incl - v; part_cursor[idx] = carry + incl - v; chunk0[idx] = carry2 + incl2 - v2; }
        __syncthreads();
        if (threadIdx.x == 1023) { carry_sh = carry + incl; carry2_sh = carry2 + incl2; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { part_off[P] = carry_sh; chunk0[P] = carry2_sh; }
}

// one thread per scalar of the tile (blockDim.x == tile): the W <= 16 digits are recoded once and stay in registers
__global__ void __launch_bounds__(1024) msm_partition_kernel(MsmCols cols, MsmPlan pl, const uint32_t* __restrict__ digits, uint32_t* __restrict__ part_cursor,
                                                           uint2* __restrict__ inter) {
    H2B_DYN_SMEM(uint32_t, smem);
    const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
    uint32_t* cnt = smem;                    // entries of this tile per partition, then the fill cursor
    uint32_t* start = smem + P;              // first staging slot of the partition
    uint32_t* base = smem + 2 * P;           // first slot of this tile's run in the partition's region
    uint2* staging = (uint2*)(smem + 3 * P + (P & 1));
    __shared__ uint32_t warp_tot[32];
    const uint32_t col = blockIdx.y;
    const uint32_t col_len = cols.len[col];
    const uint32_t gbase = col * pl.m * pl.Nb;
    const uint32_t tile = blockDim.x;
    const uint32_t ntiles = (pl.n + tile - 1) / tile;
    digits += (size_t)col * pl.W * pl.n;
    for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint32_t i = t * tile + threadIdx.x;
        const bool live = i < col_len;
        for (uint32_t b = threadIdx.x; b < P; b += blockDim.x) cnt[b] = 0;
        uint32_t dig[PART_W_MAX];            // bucket (global index + 1, 0 = no entry) with the sign in bit 31
#pragma unroll
        for (uint32_t w = 0; w < PART_W_MAX; ++w) dig[w] = 0;
        if (live) {
            uint32_t set = 0;
#pragma unroll
            for (uint32_t w = 0; w < PART_W_MAX; ++w) {
                if (w < pl.W) {
                    const uint32_t e = digits[(size_t)w * pl.n + i];
                    if (e) dig[w] = (gbase + set * pl.Nb + (e & ~SIGN_BIT)) | (e & SIGN_BIT);
                    if (++set == pl.m) set = 0;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (uint32_t w = 0; w < PART_W_MAX; ++w)
            if (dig[w]) atomicAdd(&cnt[((dig[w] & ~SIGN_BIT) - 1) >> pl.pb], 1u);
        __syncthreads();
        // exclusive scan of cnt over the P partitions, reserve the runs, reset cnt as fill cursor
        {
            const uint32_t per = (P + blockDim.x - 1) / blockDim.x;
            const uint32_t lo = threadIdx.x * per < P ? threadIdx.x * per : P, hi = lo + per < P ? lo + per : P;
            uint32_t sum = 0;
            for (uint32_t b = lo; b < hi; ++b) sum += cnt[b];
            uint32_t incl = sum;
            const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += v;
            }
            if (lane == 31) warp_tot[wid] = incl;
            __syncthreads();
            uint32_t run = incl - sum;
            for (uint32_t k = 0; k < wid; ++k) run += warp_tot[k];
            for (uint32_t b = lo; b < hi; ++b) {
                const uint32_t c = cnt[b];
                start[b] = run;
                base[b] = c ? atomicAdd(&part_cursor[b], c) : 0u;
                cnt[b] = 0;
                run += c;
            }
        }
        __syncthreads();
        // stage the entries grouped by partition: (global bucket, table row | sign)
        {
            uint32_t set = 0, row = pl.row0 + i;
#pragma unroll
            for (uint32_t w = 0; w < PART_W_MAX; ++w) {
                if (w < pl.W) {
                    if (dig[w]) {
                        const uint32_t g = (dig[w] & ~SIGN_BIT) - 1;
                        const uint32_t p = g >> pl.pb;
                        staging[start[p] + atomicAdd(&cnt[p], 1u)] = make_uint2(g, row | (dig[w] & SIGN_BIT));
                    }
                    if (++set == pl.m) { set = 0; row += pl.stride; }
                }
            }
        }
        __syncthreads();
        // write-out: every partition's group goes to its region of the intermediate list as one contiguous run
        const uint32_t total = start[P - 1] + cnt[P - 1];
        for (uint32_t j = threadIdx.x; j < total; j += blockDim.x) {
            const uint2 ent = staging[j];
            const uint32_t p = ent.x >> pl.pb;
            inter[base[p] + (j - start[p])] = ent;
        }
        __syncthreads();
    }
}

// chunk c -> (partition, entry range).  chunk0 is ascending; the partition is the last one whose first chunk is <= c.
__device__ __forceinline__ bool msm_chunk_range(const uint32_t* __restrict__ chunk0, const uint32_t* __restrict__ part_off, uint32_t P, uint32_t chunk_log,
                                                uint32_t c, uint32_t& p, uint32_t& e0, uint32_t& e1) {
    if (c >= chunk0[P]) return false;
    uint32_t lo = 0, hi = P;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (chunk0[mid] <= c) lo = mid; else hi = mid;
    }
    p = lo;           // chunk0[p] <= c < chunk0[p + 1]: partitions without entries (chunk0[p] == chunk0[p + 1]) are never selected
    e0 = part_off[p] + ((c - chunk0[p]) << chunk_log);
    e1 = e0 + (1u << chunk_log) < part_off[p + 1] ? e0 + (1u << chunk_log) : part_off[p + 1];
    return true;
}

// per-chunk bucket histogram (shared memory) -> chunk_hist[c][0 .. 2^pb)
__global__ void __launch_bounds__(1024) msm_place_count_kernel(MsmPlan pl, uint32_t chunk_log, const uint32_t* __restrict__ chunk0, const uint32_t* __restrict__ part_off,
                                                             const uint2* __restrict__ inter, uint32_t* __restrict__ chunk_hist) {
    H2B_DYN_SMEM(uint32_t, cur);
    const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
    const uint32_t NB = 1u << pl.pb;
    for (uint32_t c = blockIdx.x;; c += gridDim.x) {
        uint32_t p, e0, e1;
        if (!msm_chunk_range(chunk0, part_off, P, chunk_log, c, p, e0, e1)) return;
        const uint32_t g0 = p << pl.pb;
        const bool hot = (uint64_t)(part_off[p + 1] - part_off[p]) * P > 8ull * part_off[P];
        for (uint32_t b = threadIdx.x; b < NB; b += blockDim.x) cur[b] = 0;
        __syncthreads();
        for (uint32_t base = e0; base < e1; base += 4 * blockDim.x) {
            uint32_t bk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t j = base + u * blockDim.x + threadIdx.x;
                bk[u] = j < e1 ? inter[j].x - g0 : 0xffffffffu;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (hot) {
                    const unsigned peers = __match_any_sync(0xffffffffu, bk[u]);
                    if (bk[u] != 0xffffffffu && (threadIdx.x & 31) == (uint32_t)(__ffs((int)peers) - 1)) atomicAdd(&cur[bk[u]], (uint32_t)__popc(peers));
                } else if (bk[u] != 0xffffffffu) atomicAdd(&cur[bk[u]], 1u);
            }
        }
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < NB; b += blockDim.x) chunk_hist[(size_t)c * NB + b] = cur[b];
        __syncthreads();
    }
}

// one CTA per partition: bucket totals over the partition's chunks, exclusive scan -> offsets[], and every chunk's histogram
// row is replaced by the positions at which that chunk starts writing each bucket
__global__ void __launch_bounds__(1024) msm_place_scan_kernel(MsmPlan pl, const uint32_t* __restrict__ chunk0, const uint32_t* __restrict__ part_off,
                                                            uint32_t* __restrict__ chunk_hist, uint32_t* __restrict__ offsets) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t base_sh;
    const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
    const uint32_t NB = 1u << pl.pb;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    for (uint32_t p = blockIdx.x; p < P; p += gridDim.x) {
        const uint32_t c0 = chunk0[p], c1 = chunk0[p + 1];
        const uint32_t g0 = p << pl.pb;
        const uint32_t nb = (pl.B - g0 < NB) ? pl.B - g0 : NB;
        if (threadIdx.x == 0) base_sh = part_off[p];
        __syncthreads();
        // blockDim.x buckets at a time, bucket = q + threadIdx.x: every walk over the chunk rows is coalesced (with a thread owning
        // `per` CONSECUTIVE buckets a 4096-bucket partition took 0.93 ms here at 2^24 points, 30x the 1024-bucket case)
        for (uint32_t q = 0; q < NB; q += blockDim.x) {
            const uint32_t bkt = q + threadIdx.x;
            uint32_t tot = 0;
            if (bkt < NB) {
#pragma unroll 4
                for (uint32_t c = c0; c < c1; ++c) tot += chunk_hist[(size_t)c * NB + bkt];
            }
            uint32_t incl = tot;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += v;
            }
            if (lane == 31) warp_tot[wid] = incl;
            __syncthreads();
            const uint32_t base = base_sh;
            uint32_t run = base + incl - tot;
            for (uint32_t k = 0; k < wid; ++k) run += warp_tot[k];
            if (bkt < NB) {
                if (bkt < nb) offsets[g0 + bkt] = run;
                uint32_t r = run;
                for (uint32_t c = c0; c < c1; ++c) {
                    const uint32_t v = chunk_hist[(size_t)c * NB + bkt];
                    chunk_hist[(size_t)c * NB + bkt] = r;
                    r += v;
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t t = base;
                for (uint32_t k = 0; k < nwarps; ++k) t += warp_tot[k];
                base_sh = t;
            }
            __syncthreads();
        }
        if (p == P - 1 && threadIdx.x == 0) offsets[pl.B] = part_off[P];
        __syncthreads();
    }
}

// per chunk: cursors from the scanned histogram row, every entry to its final position
__global__ void __launch_bounds__(1024) msm_place_kernel(MsmPlan pl, uint32_t chunk_log, const uint32_t* __restrict__ chunk0, const uint32_t* __restrict__ part_off,
                                                       const uint2* __restrict__ inter, const uint32_t* __restrict__ chunk_hist, uint32_t* __restrict__ sorted) {
    H2B_DYN_SMEM(uint32_t, cur);
    const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
    const uint32_t NB = 1u << pl.pb;
    for (uint32_t c = blockIdx.x;; c += gridDim.x) {
        uint32_t p, e0, e1;
        if (!msm_chunk_range(chunk0, part_off, P, chunk_log, c, p, e0, e1)) return;
        const uint32_t g0 = p << pl.pb;
        const bool hot = (uint64_t)(part_off[p + 1] - part_off[p]) * P > 8ull * part_off[P];
        for (uint32_t b = threadIdx.x; b < NB; b += blockDim.x) cur[b] = chunk_hist[(size_t)c * NB + b];
        __syncthreads();
        for (uint32_t base = e0; base < e1; base += 4 * blockDim.x) {
            uint2 ent[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t j = base + u * blockDim.x + threadIdx.x;
                ent[u] = j < e1 ? inter[j] : make_uint2(0xffffffffu, 0u);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool live = ent[u].x != 0xffffffffu;
                const uint32_t b = ent[u].x - g0;
                if (hot) {
                    const unsigned peers = __match_any_sync(0xffffffffu, live ? b : 0xffffffffu);
                    const uint32_t lane = threadIdx.x & 31, leader = (uint32_t)(__ffs((int)peers) - 1);
                    uint32_t first = 0;
                    if (live && lane == leader) first = atomicAdd(&cur[b], (uint32_t)__popc(peers));
                    first = __shfl_sync(0xffffffffu, first, (int)leader);
                    if (live) sorted[first + (uint32_t)__popc(peers & ((1u << lane) - 1))] = ent[u].y;
                } else if (live) {
                    sorted[atomicAdd(&cur[b], 1u)] = ent[u].y;
                }
            }
        }
        __syncthreads();
    }
}

// ---- 1. decompose + histogram ------------------------------------------------------------------
// (grid-stride over blocks of 256 scalars so that the per-CTA aggregation of a narrow top window is flushed rarely)
__global__ void __launch_bounds__(256) msm_decompose_kernel(MsmCols cols, MsmPlan pl,
                                                          uint32_t* __restrict__ digits, uint32_t* __restrict__ counts) {
    __shared__ uint32_t top_hist[TOP_BINS_MAX];
    const uint32_t col = blockIdx.y;
    const uint4* __restrict__ scalars = cols.scalars[col];
    const uint32_t col_len = cols.len[col];
    if (pl.pb) {
        // partitioned sort: only the P partition totals are needed here (the per-bucket counts are taken per partition, in shared
        // memory, by msm_place_kernel): a per-CTA histogram, flushed with one global reduction per partition
        msm_decompose_partitions(cols, pl, digits, counts);
        return;
    }
    counts += (size_t)col * pl.m * pl.Nb;
    digits += (size_t)col * pl.W * pl.n;
    const uint32_t top_set = (pl.W - 1) % pl.m;
    if (pl.top_bins) {
        for (uint32_t b = threadIdx.x; b < pl.top_bins; b += blockDim.x) top_hist[b] = 0;
        __syncthreads();
    }
    const uint32_t c = pl.c, half = 1u << (c - 1);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t rounds = (pl.n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (uint32_t round = 0; round < rounds; ++round) {
        const uint32_t i = (round * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        const bool live = i < col_len;
        Fr s = fp_zero<FR>();
        uint32_t neg = 0;
        if (live) {
            s = fp_from_mont(fp_load<FR>(scalars + 2 * (size_t)i));
            if (fr_gt_half(s)) {
                // s <- r - s  (canonical, non-zero)
                Fr r;
#pragma unroll
                for (int k = 0; k < 8; ++k) r.l[k] = FpParams<FR>::P(k);
                uint32_t borrow = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    uint64_t d = (uint64_t)r.l[k] - s.l[k] - borrow;
                    s.l[k] = (uint32_t)d;
                    borrow = (uint32_t)(d >> 63);
                }
                neg = SIGN_BIT;
            }
        }
        uint32_t carry = 0, set = 0;
        const uint32_t mask = (1u << c) - 1;
        for (uint32_t w = 0; w < pl.W; ++w) {
            uint32_t d = (s.l[0] & mask) + carry;
            fr_shift_right(s, c);
            uint32_t sign = neg;
            if (d > half) { d = (1u << c) - d; carry = 1; sign ^= SIGN_BIT; }
            else carry = 0;
            if (w == 0) {
                // Window 0 is where witness columns pile up (a fifth of the rows equal to 1, small lookup limbs ...):
                // lanes of a warp that hit the same bucket send ONE reduction.  (Every lane takes part; d == 0 = no entry.)
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                if (d != 0 && lane == (uint32_t)(__ffs((int)peers) - 1)) atomicAdd(&counts[d - 1], (uint32_t)__popc(peers));
            } else if (d != 0) {
                if (pl.top_bins && w + 1 == pl.W) atomicAdd(&top_hist[d], 1u);
                else atomicAdd(&counts[set * pl.Nb + d - 1], 1u);
            }
            if (live) digits[(size_t)w * pl.n + i] = d ? (d | sign) : 0u;
            if (++set == pl.m) set = 0;
        }
    }
    if (pl.top_bins) {
        __syncthreads();
        for (uint32_t b = 1 + threadIdx.x; b < pl.top_bins; b += blockDim.x)
            if (top_hist[b]) atomicAdd(&counts[top_set * pl.Nb + b - 1], top_hist[b]);
    }
}

// ---- 2. exclusive scan of the counts (scan.cu's u32_exclusive_scan) + scatter -------------------------

__global__ void __launch_bounds__(256) msm_scatter_kernel(MsmCols cols, MsmPlan pl, const uint32_t* __restrict__ digits, uint32_t* __restrict__ cursor,
                                                        uint32_t* __restrict__ sorted) {
    __shared__ uint32_t top_cnt[TOP_BINS_MAX];      // per-round count, then the round's base position, of each top-window digit
    const uint32_t col = blockIdx.y;
    const uint32_t col_len = cols.len[col];
    cursor += (size_t)col * pl.m * pl.Nb;
    digits += (size_t)col * pl.W * pl.n;
    const uint32_t top_set = (pl.W - 1) % pl.m;
    const uint32_t rounds = (pl.n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (uint32_t round = 0; round < rounds; ++round) {
        const uint32_t i = (round * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        const bool live = i < col_len;
        uint32_t set = 0, row = pl.row0 + i;
        const uint32_t lower = pl.top_bins ? pl.W - 1 : pl.W;
        {   // window 0: one cursor update per warp and bucket (see msm_decompose_kernel)
            const uint32_t e = live ? digits[i] : 0u;
            const uint32_t d = e & ~SIGN_BIT;
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            const uint32_t lane = threadIdx.x & 31, leader = (uint32_t)(__ffs((int)peers) - 1);
            uint32_t base = 0;
            if (d != 0 && lane == leader) base = atomicAdd(&cursor[d - 1], (uint32_t)__popc(peers));
            base = __shfl_sync(0xffffffffu, base, (int)leader);
            if (d != 0) sorted[base + (uint32_t)__popc(peers & ((1u << lane) - 1))] = row | (e & SIGN_BIT);
            if (++set == pl.m) { set = 0; row += pl.stride; }
        }
        if (live) {
            for (uint32_t w = 1; w < lower; ++w) {
                uint32_t e = digits[(size_t)w * pl.n + i];
                if (e != 0) {
                    uint32_t d = e & ~SIGN_BIT;
                    uint32_t pos = atomicAdd(&cursor[set * pl.Nb + d - 1], 1u);
                    H2B_STORE_STREAMING(&sorted[pos], row | (e & SIGN_BIT));
                }
                if (++set == pl.m) { set = 0; row += pl.stride; }
            }
        }
        if (pl.top_bins) {
            // narrow top window: rank inside the CTA in shared memory, one global cursor update per digit value and round
            for (uint32_t b = threadIdx.x; b < pl.top_bins; b += blockDim.x) top_cnt[b] = 0;
            __syncthreads();
            uint32_t e = live ? digits[(size_t)(pl.W - 1) * pl.n + i] : 0u;
            uint32_t d = e & ~SIGN_BIT, rank = 0;
            if (d) rank = atomicAdd(&top_cnt[d], 1u);
            __syncthreads();
            for (uint32_t b = 1 + threadIdx.x; b < pl.top_bins; b += blockDim.x)
                if (top_cnt[b]) top_cnt[b] = atomicAdd(&cursor[top_set * pl.Nb + b - 1], top_cnt[b]);
            __syncthreads();
            if (d) sorted[top_cnt[d] + rank] = (pl.row0 + i + ((pl.W - 1) / pl.m) * pl.stride) | (e & SIGN_BIT);
            __syncthreads();
        }
    }
}

// ---- 3. accumulate: equal slices of the sorted list ----------------------------------------------------
// slice length for `total` sorted entries cut into at most G slices.  The host sizes G for the worst case (every
// digit non-zero); skewed columns sort far fewer entries, so slices never get shorter than SLICE_MIN and the
// surplus threads simply exit.
static const uint32_t SLICE_MIN = 16;
__device__ __forceinline__ uint32_t slice_len(uint32_t total, uint32_t G) {
    uint32_t S = (total + G - 1) / G;
    return S < SLICE_MIN ? SLICE_MIN : S;
}

// ctrl[0] = buckets cut by a slice boundary (split_list), ctrl[1] = those cut into many pieces (heavy_list)
__global__ void __launch_bounds__(256, 2) msm_accumulate_kernel(MsmPlan pl, const uint4* __restrict__ tables, const uint32_t* __restrict__ offsets,
                                                           const uint32_t* __restrict__ sorted, uint32_t* __restrict__ ctrl,
                                                           uint32_t* __restrict__ split_list, uint4* __restrict__ bucket_acc,
                                                           uint4* __restrict__ head_partial) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= pl.G) return;
    const uint32_t total = offsets[pl.B];
    const uint32_t S = slice_len(total, pl.G);
    if ((uint64_t)t * S >= total) return;
    const uint32_t start = t * S;
    const uint32_t end = (total - start > S) ? start + S : total;
    // b = the bucket that holds entry `start`: offsets[b] <= start < offsets[b + 1]
    uint32_t lo = 0, hi = pl.B;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= start) lo = mid; else hi = mid;
    }
    uint32_t b = lo;
    uint32_t next = offsets[b + 1];
    bool head = offsets[b] < start;      // the bucket began in an earlier slice

    // The next point is gathered into shared memory while this one is added, not into 16 registers held across the
    // whole addition: with those registers free the addition fits 128 (16 warps per SM) without spilling.  Two slots
    // per thread, so the copy never overwrites the point being read.
    __shared__ uint4 pt[2][4][256];
    const uint32_t tid = threadIdx.x;
    XYZZ acc = xyzz_identity();
    uint32_t e = sorted[start];
#pragma unroll
    for (int k = 0; k < 4; ++k) copy16_async(&pt[0][k][tid], tables + 4 * (size_t)(e & ~SIGN_BIT) + k);
    uint32_t e_next = start + 1 < end ? sorted[start + 1] : 0;
    for (uint32_t j = start; j < end; ++j) {
        const uint32_t s = (j - start) & 1;
        copy_async_wait_all();
        if (j + 1 < end) {
#pragma unroll
            for (int k = 0; k < 4; ++k) copy16_async(&pt[s ^ 1][k][tid], tables + 4 * (size_t)(e_next & ~SIGN_BIT) + k);
        }
        Affine p;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint4 v = pt[s][k][tid];
            uint32_t* l = (k < 2 ? p.x.l : p.y.l) + 4 * (k & 1);
            l[0] = v.x; l[1] = v.y; l[2] = v.z; l[3] = v.w;
        }
        const uint32_t e_cur = e;
        e = e_next;
        e_next = j + 2 < end ? sorted[j + 2] : 0;
        if (j == next) {        // bucket b is complete: flush, move to the next non-empty bucket
            if (head) xyzz_store(head_partial + 8 * (size_t)t, xyzz_canon(acc));
            else xyzz_store(bucket_acc + 8 * (size_t)b, xyzz_canon(acc));
            head = false;
            acc = xyzz_identity();
            do { ++b; next = offsets[b + 1]; } while (next <= j);
        }
        xyzz_add_affine_lazy(acc, p, (e_cur & SIGN_BIT) != 0);      // acc lazily reduced, canonical when stored
    }
    if (head) {
        xyzz_store(head_partial + 8 * (size_t)t, xyzz_canon(acc));
    } else {
        xyzz_store(bucket_acc + 8 * (size_t)b, xyzz_canon(acc));
        if (next > end) split_list[atomicAdd(&ctrl[0], 1u)] = b;      // continues in later slices
    }
}

// ---- 4. combine the pieces of buckets cut by slice boundaries --------------------------------------------
// Light buckets (a few pieces: the common case, one thread each) are finished by msm_combine_light_kernel.  A bucket
// cut into many pieces (a witness column whose value 1 fills 20 % of the rows ...) is reduced by a two-level tree:
// chunks of COMBINE_CHUNK pieces by one CTA each, then one CTA per bucket over the chunk sums.
static const uint32_t COMBINE_HEAVY = 24;      // more pieces than this: tree
static const uint32_t COMBINE_CHUNK = 1024;    // pieces per CTA in the first tree level
static const uint32_t COMBINE_THREADS = 256;   // CTAs of the two tree levels; two per SM (capped at 128 registers).  64-thread CTAs over 256-piece chunks were tried for the
                                               // ~1500 moderately heavy buckets of a narrow top window (22-bit tables: combine 0.63 -> 0.41 ms) but cost a witness-like column, whose
                                               // one bucket is cut into 13 000 pieces, 0.11 ms

struct HeavyDesc { uint32_t bucket, chunk0, nchunks, pad; };

// ctrl[0] = split buckets, ctrl[1] = heavy buckets, ctrl[2] = chunks
__global__ void __launch_bounds__(128) msm_combine_light_kernel(MsmPlan pl, const uint32_t* __restrict__ offsets, uint32_t* __restrict__ ctrl,
                                                              const uint32_t* __restrict__ split_list, HeavyDesc* __restrict__ heavy,
                                                              uint2* __restrict__ chunk_desc, const uint4* __restrict__ head_partial,
                                                              uint4* __restrict__ bucket_acc) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ctrl[0]) return;
    const uint32_t S = slice_len(offsets[pl.B], pl.G);
    const uint32_t b = split_list[idx];
    const uint32_t first = offsets[b] / S, last = (offsets[b + 1] - 1) / S;
    const uint32_t pieces = last - first;
    if (pieces > COMBINE_HEAVY) {
        HeavyDesc d;
        d.bucket = b;
        d.nchunks = (pieces + COMBINE_CHUNK - 1) / COMBINE_CHUNK;
        d.chunk0 = atomicAdd(&ctrl[2], d.nchunks);
        d.pad = 0;
        const uint32_t h = atomicAdd(&ctrl[1], 1u);
        heavy[h] = d;
        for (uint32_t i = 0; i < d.nchunks; ++i) chunk_desc[d.chunk0 + i] = make_uint2(h, i);
        return;
    }
    XYZZ acc = xyzz_load(bucket_acc + 8 * (size_t)b);
    for (uint32_t t = first + 1; t <= last; ++t) {
        XYZZ q = xyzz_load(head_partial + 8 * (size_t)t);
        xyzz_add(acc, q);
    }
    xyzz_store(bucket_acc + 8 * (size_t)b, acc);
}

// sum of `acc` over the threads of the CTA, valid in thread 0
__device__ __forceinline__ void block_sum_xyzz(XYZZ& acc, uint4* sh) {
    xyzz_store(sh + 8 * threadIdx.x, acc);
    __syncthreads();
    for (uint32_t d = blockDim.x >> 1; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            XYZZ o = xyzz_load(sh + 8 * (threadIdx.x + d));
            xyzz_add<true>(acc, o);
            xyzz_store(sh + 8 * threadIdx.x, acc);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(COMBINE_THREADS, 2) msm_combine_chunk_kernel(MsmPlan pl, const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ ctrl,
                                                              const HeavyDesc* __restrict__ heavy, const uint2* __restrict__ chunk_desc,
                                                              const uint4* __restrict__ head_partial, uint4* __restrict__ chunk_out) {
    __shared__ uint4 sh[COMBINE_THREADS * 8];
    const uint32_t S = slice_len(offsets[pl.B], pl.G);
    const uint32_t nchunks = ctrl[2];
    for (uint32_t item = blockIdx.x; item < nchunks; item += gridDim.x) {
        const uint2 cd = chunk_desc[item];
        const uint32_t b = heavy[cd.x].bucket;
        const uint32_t first = offsets[b] / S, last = (offsets[b + 1] - 1) / S;
        const uint32_t lo = first + 1 + cd.y * COMBINE_CHUNK;
        uint32_t hi = lo + COMBINE_CHUNK;
        if (hi > last + 1) hi = last + 1;
        XYZZ acc = xyzz_identity();
        for (uint32_t t = lo + threadIdx.x; t < hi; t += blockDim.x) {
            XYZZ q = xyzz_load(head_partial + 8 * (size_t)t);
            xyzz_add<true>(acc, q);
        }
        block_sum_xyzz(acc, sh);
        if (threadIdx.x == 0) xyzz_store(chunk_out + 8 * (size_t)item, acc);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(COMBINE_THREADS, 2) msm_combine_heavy_kernel(const uint32_t* __restrict__ ctrl, const HeavyDesc* __restrict__ heavy,
                                                              const uint4* __restrict__ chunk_out, uint4* __restrict__ bucket_acc) {
    __shared__ uint4 sh[COMBINE_THREADS * 8];
    const uint32_t nheavy = ctrl[1];
    for (uint32_t h = blockIdx.x; h < nheavy; h += gridDim.x) {
        const HeavyDesc d = heavy[h];
        XYZZ acc = xyzz_identity();
        for (uint32_t i = threadIdx.x; i < d.nchunks; i += blockDim.x) {
            XYZZ q = xyzz_load(chunk_out + 8 * (size_t)(d.chunk0 + i));
            xyzz_add<true>(acc, q);
        }
        block_sum_xyzz(acc, sh);
        if (threadIdx.x == 0) {
            XYZZ cur = xyzz_load(bucket_acc + 8 * (size_t)d.bucket);
            xyzz_add<true>(cur, acc);
            xyzz_store(bucket_acc + 8 * (size_t)d.bucket, cur);
        }
        __syncthreads();
    }
}

// ---- 4b. chunked MSMs: add the bucket sums of one chunk into the running bucket accumulators -------------------
// (a separate, uniform kernel: doing this addition inside the accumulate kernel's flush would make every lane's
// flush a divergent 14-multiplication detour for the whole warp)
__global__ void __launch_bounds__(128) msm_merge_kernel(uint32_t B, const uint32_t* __restrict__ offsets, const uint4* __restrict__ chunk_acc,
                                                      uint4* __restrict__ bucket_acc) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || offsets[b + 1] == offsets[b]) return;
    XYZZ cur = xyzz_load(bucket_acc + 8 * (size_t)b);
    XYZZ add = xyzz_load(chunk_acc + 8 * (size_t)b);
    xyzz_add(cur, add);
    xyzz_store(bucket_acc + 8 * (size_t)b, cur);
}

// ---- 5. bucket reduction ------------------------------------------------------------------------------
// One level of  S_w = sum_u (u+1) * Bw[u] + sum_u Dw[u]  over N items per set, m items per thread:
//   A_j = sum_i B[jm+i],  C_j = sum_i (i+1) B[jm+i] + sum_i D[jm+i]
//   S_w = sum_j C_j + m * sum_{j>=1} j * A_j  ->  next level: B'[j-1] = m*A_j, B'[J-1] = 0, D'[j] = C_j.
// Level 0 reads the bucket accumulators; `offsets` (level 0 only) tells which buckets are empty and were
// therefore never written.
__global__ void __launch_bounds__(128) msm_reduce_level_kernel(const uint4* __restrict__ Bin, const uint4* __restrict__ Din, const uint32_t* __restrict__ offsets,
                                                             uint32_t N, uint32_t logm, uint32_t W, uint4* __restrict__ Bout, uint4* __restrict__ Dout) {
    uint32_t m = 1u << logm;
    uint32_t J = (N + m - 1) >> logm;
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= W * J) return;
    uint32_t w = t / J, j = t - w * J;
    const uint4* Bw = Bin + 8 * (size_t)w * N;
    const uint4* Dw = Din ? Din + 8 * (size_t)w * N : nullptr;
    const uint32_t* Ow = offsets ? offsets + (size_t)w * N : nullptr;
    uint32_t lo = j << logm, hi = lo + m;
    if (hi > N) hi = N;
    XYZZ running = xyzz_identity(), acc = xyzz_identity();
    for (uint32_t u = hi; u-- > lo;) {
        if (!Ow || Ow[u + 1] != Ow[u]) {
            XYZZ bu = xyzz_load(Bw + 8 * (size_t)u);
            xyzz_add<true>(running, bu);
        }
        xyzz_add<true>(acc, running);
        if (Dw) {
            XYZZ du = xyzz_load(Dw + 8 * (size_t)u);
            xyzz_add<true>(acc, du);
        }
    }
    xyzz_store(Dout + 8 * ((size_t)w * J + j), acc);
    if (j >= 1) {
        for (uint32_t k = 0; k < logm; ++k) running = xyzz_double<true>(running);
        xyzz_store(Bout + 8 * ((size_t)w * J + j - 1), running);
    } else {
        xyzz_store(Bout + 8 * ((size_t)w * J + J - 1), xyzz_identity());
    }
}

// Block level of the reduction: a CTA of M = blockDim.x threads (a power of two, 32..512) owns M consecutive items of one set and
// computes, 2 log2(M) + 1 additions deep,
//     A_j = sum_i B[jM + i]   and   C_j = sum_i (i + 1) B[jM + i] + sum_i D[jM + i]
// as a suffix scan (sum_i (i + 1) B_i = sum_i suffix_i; A_j = suffix_0) followed by a tree sum, both in shared memory.  With more
// than one block per set the outputs feed the next level like those of msm_reduce_level_kernel (B'[j-1] = M * A_j, B'[J-1] = 0,
// D'[j] = C_j): 2.1 additions per bit of the item index, where the chunked running sums of one thread need 5.6 (2m additions + log2 m
// doublings per log2 m bits) -- and a lone warp takes ~10 us per addition whatever the GPU has idle.  The tree sum runs MIRRORED
// (the result lands in the last thread) so that thread 0, in another warp, does the log2(M) doublings of A_j in its shadow, one per
// tree step.  Work is M log M additions per block: only for levels that no longer fill the GPU (the host picks: section
// "bucket reduction hierarchy").  One block per set (gridDim.x == 1) is the tail: out[w] = S_w.
static const uint32_t REDUCE_TAIL_MAX = 512;
static const uint32_t REDUCE_BLOCK = 128;
__global__ void __launch_bounds__(512) msm_reduce_block_kernel(const uint4* __restrict__ Bin, const uint4* __restrict__ Din, const uint32_t* __restrict__ offsets,
                                                             uint32_t N, uint4* __restrict__ Bout, uint4* __restrict__ Dout) {
    H2B_DYN_SMEM(uint4, sh);
    const uint32_t w = blockIdx.y, j = blockIdx.x, J = gridDim.x, tid = threadIdx.x, M = blockDim.x;
    const uint32_t u = j * M + tid;
    const bool live = u < N;
    XYZZ x = xyzz_identity();
    if (live && (!offsets || offsets[(size_t)w * N + u + 1] != offsets[(size_t)w * N + u])) x = xyzz_load(Bin + 8 * ((size_t)w * N + u));
    for (uint32_t d = 1; d < M; d <<= 1) {
        xyzz_store(sh + 8 * tid, x);
        __syncthreads();
        if (tid + d < M) {
            XYZZ o = xyzz_load(sh + 8 * (tid + d));
            xyzz_add<true>(x, o);
        }
        __syncthreads();
    }
    XYZZ a = x;                                 // thread 0: A_j
    if (Din && live) {
        XYZZ dd = xyzz_load(Din + 8 * ((size_t)w * N + u));
        xyzz_add<true>(x, dd);
    }
    xyzz_store(sh + 8 * tid, x);
    __syncthreads();
    for (uint32_t d = M >> 1; d > 0; d >>= 1) {
        if (tid >= M - d) {
            XYZZ o = xyzz_load(sh + 8 * (tid - d));
            xyzz_add<true>(x, o);
            xyzz_store(sh + 8 * tid, x);
        } else if (tid == 0 && J > 1 && M >= 64) {
            a = xyzz_double<true>(a);           // log2(M) tree steps = log2(M) doublings
        }
        __syncthreads();
    }
    if (tid == M - 1) xyzz_store(Dout + 8 * ((size_t)w * J + j), x);
    if (tid == 0 && J > 1) {
        if (M < 64) for (uint32_t d = M >> 1; d > 0; d >>= 1) a = xyzz_double<true>(a);
        if (j >= 1) xyzz_store(Bout + 8 * ((size_t)w * J + j - 1), a);
        else xyzz_store(Bout + 8 * ((size_t)w * J + J - 1), xyzz_identity());
    }
}

// Horner over the set sums (S[w] = Dfinal[w], weight 2^(c*w)) and conversion to a Jacobian triple; one block per column of a
// batched MSM (sets [col * W, (col + 1) * W), result block col)
__global__ void msm_final_kernel(const uint4* __restrict__ S, uint32_t W, uint32_t c, uint4* __restrict__ out_jac, uint32_t accumulate) {
    if (threadIdx.x != 0) return;
    S += 8 * (size_t)blockIdx.x * W;
    out_jac += 14 * (size_t)blockIdx.x;
    XYZZ acc = xyzz_load(S + 8 * (size_t)(W - 1));
    for (uint32_t w = W - 1; w-- > 0;) {
        for (uint32_t k = 0; k < c; ++k) acc = xyzz_double<true>(acc);
        XYZZ sw = xyzz_load(S + 8 * (size_t)w);
        xyzz_add<true>(acc, sw);
    }
    if (accumulate) {       // running total across sub-MSMs is kept in XYZZ right behind the Jacobian slot
        XYZZ prev = xyzz_load(out_jac + 6);
        xyzz_add<true>(acc, prev);
    }
    xyzz_store(out_jac + 6, acc);
    Fq X, Y, Z;
    xyzz_to_jacobian(acc, X, Y, Z);
    fp_store<FQ>(out_jac, X);
    fp_store<FQ>(out_jac + 2, Y);
    fp_store<FQ>(out_jac + 4, Z);
}

// ---- 0. table precomputation: dst[i] = 2^c0 * src[i], affine in, affine out --------------------------------
// Each thread owns PRE_G points so that one field inversion (Fermat) serves PRE_G conversions to affine.
static const int PRE_G = 8;
__global__ void __launch_bounds__(128) msm_precompute_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, uint32_t n, uint32_t c0) {
    const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * PRE_G;
    if (i0 >= n) return;
    XYZZ q[PRE_G];
    Fq pre[PRE_G];
    Fq run = fp_one<FQ>();
#pragma unroll 1
    for (int g = 0; g < PRE_G; ++g) {
        XYZZ v = xyzz_identity();
        if (i0 + g < n) {
            v = xyzz_from_affine(affine_load(src + 4 * (size_t)(i0 + g)));
#pragma unroll 1
            for (uint32_t k = 0; k < c0; ++k) v = xyzz_double(v);
        }
        q[g] = v;
        pre[g] = run;
        if (!xyzz_is_identity(v)) run = fp_mul(run, fp_mul(v.zz, v.zzz));
    }
    Fq inv = fp_inv(run);
#pragma unroll 1
    for (int g = PRE_G - 1; g >= 0; --g) {
        if (i0 + g >= n) continue;
        XYZZ v = q[g];
        Affine a;
        if (xyzz_is_identity(v)) {
            a.x = fp_zero<FQ>();
            a.y = fp_zero<FQ>();
        } else {
            Fq zi = fp_mul(inv, pre[g]);                 // 1 / (ZZ * ZZZ)
            inv = fp_mul(inv, fp_mul(v.zz, v.zzz));
            a.x = fp_mul(v.x, fp_mul(v.zzz, zi));        // X / ZZ
            a.y = fp_mul(v.y, fp_mul(v.zz, zi));         // Y / ZZZ
        }
        affine_store(dst + 4 * (size_t)(i0 + g), a);
    }
}

int msm_precompute_run(DeviceCtx& ctx, const void* d_src, void* d_dst, size_t n, uint32_t c0, cudaStream_t stream) {
    (void)ctx;
    if (n == 0) return H2B_OK;
    if (n > ((size_t)1 << 26)) { set_error("msm precompute: at most 2^26 points per table"); return H2B_ERR_BAD_ARGUMENT; }
    const uint32_t threads = (uint32_t)((n + PRE_G - 1) / PRE_G);
    H2B_LAUNCH(msm_precompute_kernel, (threads + 127) / 128, 128, 0, stream, (const uint4*)d_src, (uint4*)d_dst, (uint32_t)n, c0);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- host orchestration ----------------------------------------------------------------------------------
struct MsmScratch {
    DevBuf digits, counts, offsets, cursor, block_sums, sorted, ctrl, split_list, heavy, chunk_desc, chunk_out, bucket_acc, bucket_tmp, head_partial, redA, redB, redC, redD, result;
    DevBuf batch_out;                                                   // result blocks of a batched host-pointer call
    DevBuf part_counts, part_off, part_cursor, chunk0, chunk_hist, inter; // partitioned sort (section 2c)
    bool part_attr_set = false;
};

static int g_forced_c = 0;
int msm_set_window(int c) {
    if (c != 0 && (c < 2 || c > 24)) { set_error("msm window must be 0 (auto) or in [2, 24]"); return H2B_ERR_BAD_ARGUMENT; }
    g_forced_c = c;
    return H2B_OK;
}

static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

static uint32_t windows_for(uint32_t c) { return 253 / c + 1; }

// Cost model in units of one sorted entry (sort + one mixed addition, 0.18 ns on a B200), fitted to measurements at
// 2^16..2^26 (profiles/r01_msm_spacing.jsonl): the counting sort slows down by about 3.5 % per bit once the bucket set
// outgrows the L2-friendly 2^19 counters, and a bucket costs about 8 entries (the reduction is latency bound).
static double msm_cost(double n, uint32_t c, uint32_t sets) {
    double per_entry = 1.0 + (c > 20 ? 0.035 * (c - 20) : 0.0);
    double cost = n * windows_for(c) * per_entry + 8.0 * sets * (double)(1u << (c - 1));
    // a top window with only a few scalar bits left puts n / 2^bits entries into each of its 2^bits buckets; cutting those
    // into slices and folding the pieces back is a latency-bound tree (0.2 - 0.9 ms at 2^16): worth about 1.5 windows
    const uint32_t top_bits = 253 - c * (windows_for(c) - 1);
    if (top_bits <= 4) cost += 1.5 * n;
    return cost;
}

// plain mode (no tables): one bucket set per window
static uint32_t msm_pick_window_plain(size_t n) {
    if (g_forced_c) return (uint32_t)g_forced_c;
    static int env_c = -1;
    if (env_c < 0) env_c = env_int("H2B_MSM_C", 0);
    if (env_c >= 2 && env_c <= 24) return (uint32_t)env_c;
    uint32_t best = 2;
    double best_cost = 1e300;
    for (uint32_t c = 2; c <= 20; ++c) {
        double cost = msm_cost((double)n, c, windows_for(c));
        if (cost < best_cost) { best_cost = cost; best = c; }
    }
    return best;
}

// table spacing for a base set of n points: even c0 minimising the cost of a full-length MSM, within `max_tables`
uint32_t msm_pick_table_spacing(size_t n, uint32_t max_tables) {
    // measured on B200 (profiles/r01_msm_spacing.jsonl, r01_sweep.jsonl): small sets are latency bound and want few
    // buckets (8-bit windows, whose 5-bit top window is harmless), the mid range 16 bits, large sets 20 bits; 10/12/14/18
    // bits leave a 1-3 bit top window whose hot buckets cost more than they save
    // from 2^25 points on 22 bits (12 tables): the accumulation saves 1/13 of its additions, and the costs that come with 2^21 buckets
    // -- the partitioned sort, a throughput-bound first reduction level -- no longer grow with n (2^26: 163.5 -> 157.1 ms uniform,
    // 15.7 -> 15.4 ms witness-like; 2^24: 41.1 against 41.3 ms uniform but +1 ms on every witness-like column, so 20 bits there)
    const uint32_t preferred = n < ((size_t)1 << 15) ? 8u : (n < ((size_t)1 << 20) ? 16u : (n < ((size_t)1 << 25) ? 20u : 22u));
    if (windows_for(preferred) <= max_tables) return preferred;
    uint32_t best = 0;
    double best_cost = 1e300;
    for (uint32_t c0 = 4; c0 <= 24; c0 += 2) {
        if (windows_for(c0) > max_tables) continue;
        double cost = msm_cost((double)n, c0, 1);
        if (cost < best_cost) { best_cost = cost; best = c0; }
    }
    return best;
}
uint32_t msm_tables_for(uint32_t c0) { return windows_for(c0); }

// precomputed mode: window bits must divide the table spacing c0
static uint32_t msm_pick_window_tables(size_t n, uint32_t c0) {
    if (g_forced_c && c0 % (uint32_t)g_forced_c == 0) return (uint32_t)g_forced_c;
    uint32_t best = c0;
    double best_cost = 1e300;
    for (uint32_t sets = 1; sets <= c0 / 2; ++sets) {
        if (c0 % sets) continue;
        uint32_t c = c0 / sets;
        double cost = msm_cost((double)n, c, sets);
        if (cost < best_cost) { best_cost = cost; best = c; }
    }
    return best;
}

// ---- an MSM = plan + one or more chunks of scalars accumulated into the same buckets + one bucket reduction ----
static int msm_plan(DeviceCtx& ctx, MsmScratch& s, const MsmBases& bases, size_t n_total, bool chunked, cudaStream_t stream, MsmPlan& pl, uint32_t ncols = 1) {
    (void)ctx;
    const bool tables = bases.n_tables > 1;
    memset(&pl, 0, sizeof(pl));
    pl.c = tables ? msm_pick_window_tables(n_total, bases.c0) : msm_pick_window_plain(n_total);
    pl.W = windows_for(pl.c);
    pl.m = tables ? bases.c0 / pl.c : pl.W;
    pl.Nb = 1u << (pl.c - 1);
    pl.ncols = ncols;
    if ((uint64_t)ncols * pl.m * pl.Nb >= 0x40000000ull) { set_error("msm: %u columns x %u sets x 2^%u buckets exceed the bucket index", ncols, pl.m, pl.c - 1); return H2B_ERR_BAD_ARGUMENT; }
    pl.B = ncols * pl.m * pl.Nb;
    pl.stride = tables ? (uint32_t)bases.stride : 0u;
    pl.add_into = chunked ? 1u : 0u;
    {   // scalar bits left for the top window (the recoded scalar is < 2^253) -> number of digit values it can take
        const uint32_t top_bits = 253 - pl.c * (pl.W - 1);
        const uint64_t bins = ((uint64_t)1 << top_bits) + 2;      // digits 0 .. 2^top_bits (carry) inclusive
        pl.top_bins = (bins <= TOP_BINS_MAX && bins <= (uint64_t)pl.Nb + 1) ? (uint32_t)bins : 0u;
    }
    if (tables && (pl.W + pl.m - 1) / pl.m > bases.n_tables) { set_error("msm: %u tables cannot serve %u windows in %u sets", bases.n_tables, pl.W, pl.m); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(s.counts.reserve((size_t)pl.B * 4));
    H2B_TRY(s.offsets.reserve(((size_t)pl.B + 1) * 4));
    H2B_TRY(s.cursor.reserve((size_t)pl.B * 4));
    H2B_TRY(s.ctrl.reserve(16));
    H2B_TRY(s.bucket_acc.reserve((size_t)pl.B * 128));
    if (chunked) {
        H2B_TRY(s.bucket_tmp.reserve((size_t)pl.B * 128));
        H2B_CUDA(cudaMemsetAsync(s.bucket_acc.p, 0, (size_t)pl.B * 128, stream));     // XYZZ identity = all zero
    }
    return H2B_OK;
}

static uint32_t msm_sort2_chunk_log() {
    static int v = -1;
    if (v < 0) { v = env_int("H2B_MSM_SORT2_CHUNK_LOG", 15); if (v < 5 || v > 20) v = 15; }
    return (uint32_t)v;
}

// where chunk [done, done + m) of the call finds its points
static void chunk_points(const MsmBases& bases, size_t done, const void** tables, size_t* row0) {
    *row0 = bases.row0 + done;
    *tables = bases.tables;
    if (bases.n_tables <= 1) {       // plain mode: rows are relative to the first point of the chunk
        *tables = (const char*)bases.tables + *row0 * 64;
        *row0 = 0;
    }
}

// slices and scratch of one chunk
static int msm_size_chunk(DeviceCtx& ctx, MsmScratch& s, MsmPlan& pl, size_t row0, uint32_t n) {
    pl.n = n;
    pl.row0 = (uint32_t)row0;
    const uint64_t upper = (uint64_t)n * pl.W * pl.ncols;          // sorted entries, at most
    if (upper >= 0xffffffffull) { set_error("msm: %u columns x %u points x %u windows exceed the 32-bit sort index", pl.ncols, n, pl.W); return H2B_ERR_BAD_ARGUMENT; }
    // slices: about 256 entries each once the GPU is full; below one full wave they shrink down to SLICE_MIN entries
    // (a small MSM is latency bound, and a slice is a serial chain of mixed additions)
    const uint64_t resident = (uint64_t)ctx.sm_count * 512;
    static int env_slice = -1;
    if (env_slice < 0) env_slice = env_int("H2B_MSM_SLICE", 256);
    if (upper >= resident * 64) pl.G = (uint32_t)(resident * ((upper + resident * env_slice - 1) / (resident * env_slice)));
    else if (upper >= resident * SLICE_MIN) pl.G = (uint32_t)resident;
    else pl.G = (uint32_t)((upper + SLICE_MIN - 1) / SLICE_MIN);
    if (pl.G == 0) pl.G = 1;
    // partitioned sort for large lists (H2B_MSM_SORT2=0 keeps the one-pass counting sort; H2B_MSM_SORT2_MIN_LOG lowers the threshold: tests)
    {
        static int env_on = -1, env_min = -1;
        if (env_on < 0) env_on = env_int("H2B_MSM_SORT2", 1);
        if (env_min < 0) env_min = env_int("H2B_MSM_SORT2_MIN_LOG", 28);      // sorted entries, log2: 2^25 points x 12 windows and up (profiles/r02_partitioned_sort.jsonl: equal at 2^24 points on uniform scalars, behind on witness-like ones; ahead from 2^25 on)
        pl.pb = 0;
        // with 2^21 buckets and more (22-bit tables) the one-pass scatter loses its L2 residency: the partitioned sort also takes the shorter lists of
        // the upload chunks of a host-pointer call (2^25 points end to end: 87.5 ms with one-pass sorted chunks)
        const uint64_t min_entries = (pl.B >= (1u << 21) && env_min > 24) ? ((uint64_t)1 << 24) : ((uint64_t)1 << env_min);
        if (env_on && upper >= min_entries && pl.W <= PART_W_MAX && pl.B <= (1u << 24) && pl.B >= 64) {
            uint32_t lb = 0;
            while ((1u << lb) < pl.B) ++lb;
            uint32_t pb = lb > 9 ? lb - 9 : 1;            // about 512 partitions
            if (pb > PLACE_MAX_LOG) pb = PLACE_MAX_LOG;
            if (((pl.B + (1u << pb) - 1) >> pb) <= PART_MAX) pl.pb = pb;
        }
        if (pl.pb) {
            const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
            H2B_TRY(s.part_counts.reserve((size_t)P * 4));
            H2B_TRY(s.part_off.reserve(((size_t)P + 1) * 4));
            H2B_TRY(s.part_cursor.reserve((size_t)P * 4));
            H2B_TRY(s.chunk0.reserve(((size_t)P + 1) * 4));
            H2B_TRY(s.chunk_hist.reserve((((size_t)upper >> msm_sort2_chunk_log()) + P + 1) * ((size_t)4 << pl.pb)));
            H2B_TRY(s.inter.reserve((size_t)upper * 8 + 8));
        }
    }
    H2B_TRY(s.digits.reserve((size_t)upper * 4));
    H2B_TRY(s.sorted.reserve((size_t)upper * 4 + 4));
    H2B_TRY(s.offsets.reserve(((size_t)pl.B + 1) * 4));
    H2B_TRY(s.split_list.reserve((size_t)pl.G * 4));
    const size_t max_heavy = pl.G / COMBINE_HEAVY + 1, max_chunks = pl.G / COMBINE_CHUNK + max_heavy + 1;
    H2B_TRY(s.heavy.reserve(max_heavy * sizeof(HeavyDesc)));
    H2B_TRY(s.chunk_desc.reserve(max_chunks * 8));
    H2B_TRY(s.chunk_out.reserve(max_chunks * 128));
    H2B_TRY(s.head_partial.reserve((size_t)pl.G * 128));
    return H2B_OK;
}

// stage 1 of a chunk: digits, histogram, scan, counting-sort scatter -> offsets, sorted
static int msm_sort_chunk(DeviceCtx& ctx, MsmScratch& s, const MsmPlan& pl, const MsmCols& cols, cudaStream_t stream) {
    uint32_t* counts = (uint32_t*)s.counts.p;
    uint32_t* offsets = (uint32_t*)s.offsets.p;
    uint32_t* cursor = (uint32_t*)s.cursor.p;
    uint32_t* sorted = (uint32_t*)s.sorted.p;
    const uint32_t nblk = (pl.n + 255) / 256;
    if (pl.pb) {
        // partitioned sort (section 2c)
        const uint32_t P = (pl.B + (1u << pl.pb) - 1) >> pl.pb;
        uint32_t* part_counts = (uint32_t*)s.part_counts.p;
        H2B_CUDA(cudaMemsetAsync(part_counts, 0, (size_t)P * 4, stream));
        ctx.prof.mark(PROF_BEGIN, stream);
        const uint32_t dgrid = nblk > (uint32_t)ctx.sm_count * 16 ? (uint32_t)ctx.sm_count * 16 : nblk;
        const uint32_t chunk_log = msm_sort2_chunk_log();
        H2B_LAUNCH(msm_decompose_kernel, dim3(dgrid, pl.ncols), 256, 0, stream, cols, pl, (uint32_t*)s.digits.p, part_counts);
        ctx.prof.mark(PROF_MSM_DECOMPOSE, stream);
        H2B_LAUNCH(msm_partition_scan_kernel, 1, 1024, 0, stream, (const uint32_t*)part_counts, P, chunk_log, (uint32_t*)s.part_off.p, (uint32_t*)s.part_cursor.p,
                   (uint32_t*)s.chunk0.p);
        ctx.prof.mark(PROF_MSM_SCAN, stream);
        uint32_t tile = (PART_TILE_ENTRIES / pl.W) & ~31u;
        if (tile > 1024) tile = 1024;
        const size_t smem1 = ((size_t)3 * P + 1) * 4 + (size_t)tile * pl.W * 8;
        const size_t smem2 = (size_t)4 << pl.pb;
        if (!s.part_attr_set) {
            H2B_CUDA(cudaFuncSetAttribute(msm_partition_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(((size_t)3 * PART_MAX + 1) * 4 + (size_t)PART_TILE_ENTRIES * 8)));
            H2B_CUDA(cudaFuncSetAttribute(msm_place_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)4 << PLACE_MAX_LOG)));
            H2B_CUDA(cudaFuncSetAttribute(msm_place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)4 << PLACE_MAX_LOG)));
            s.part_attr_set = true;
        }
        const uint32_t ntiles = (pl.n + tile - 1) / tile;
        const uint32_t pgrid = ntiles > (uint32_t)ctx.sm_count * 8 ? (uint32_t)ctx.sm_count * 8 : ntiles;
        H2B_LAUNCH(msm_partition_kernel, dim3(pgrid, pl.ncols), tile, smem1, stream, cols, pl, (const uint32_t*)s.digits.p, (uint32_t*)s.part_cursor.p, (uint2*)s.inter.p);
        ctx.prof.mark(PROF_MSM_PLAN, stream);
        const uint64_t upper = (uint64_t)pl.n * pl.W * pl.ncols;
        const uint32_t max_chunks = (uint32_t)(upper >> chunk_log) + P + 1;
        const uint32_t cgrid = max_chunks > (uint32_t)ctx.sm_count * 16 ? (uint32_t)ctx.sm_count * 16 : max_chunks;
        H2B_LAUNCH(msm_place_count_kernel, cgrid, 1024, smem2, stream, pl, chunk_log, (const uint32_t*)s.chunk0.p, (const uint32_t*)s.part_off.p, (const uint2*)s.inter.p,
                   (uint32_t*)s.chunk_hist.p);
        static int scan_threads = -1;      // tests: fewer threads than buckets per partition (several passes per partition)
        if (scan_threads < 0) { scan_threads = env_int("H2B_MSM_PLACE_SCAN_THREADS", 1024); if (scan_threads < 32 || scan_threads > 1024 || (scan_threads & 31)) scan_threads = 1024; }
        H2B_LAUNCH(msm_place_scan_kernel, P, (unsigned)scan_threads, 0, stream, pl, (const uint32_t*)s.chunk0.p, (const uint32_t*)s.part_off.p, (uint32_t*)s.chunk_hist.p, offsets);
        H2B_LAUNCH(msm_place_kernel, cgrid, 1024, smem2, stream, pl, chunk_log, (const uint32_t*)s.chunk0.p, (const uint32_t*)s.part_off.p, (const uint2*)s.inter.p,
                   (const uint32_t*)s.chunk_hist.p, sorted);
        H2B_CUDA(cudaGetLastError());
        ctx.prof.mark(PROF_MSM_SCATTER, stream);
        return H2B_OK;
    }
    H2B_CUDA(cudaMemsetAsync(counts, 0, (size_t)pl.B * 4, stream));
    // grid-stride only when a narrow top window is aggregated per CTA (fewer, longer-lived CTAs flush less often)
    const uint32_t sort_grid = (pl.top_bins && nblk > (uint32_t)ctx.sm_count * 32) ? (uint32_t)ctx.sm_count * 32 : nblk;
    ctx.prof.mark(PROF_BEGIN, stream);
    H2B_LAUNCH(msm_decompose_kernel, dim3(sort_grid, pl.ncols), 256, 0, stream, cols, pl, (uint32_t*)s.digits.p, counts);
    ctx.prof.mark(PROF_MSM_DECOMPOSE, stream);
    H2B_TRY(s.block_sums.reserve((((size_t)pl.B + SCAN_BLOCK - 1) / SCAN_BLOCK + 1) * 4));
    H2B_TRY(u32_exclusive_scan(counts, pl.B, offsets, cursor, (uint32_t*)s.block_sums.p, stream));
    ctx.prof.mark(PROF_MSM_SCAN, stream);
    H2B_LAUNCH(msm_scatter_kernel, dim3(sort_grid, pl.ncols), 256, 0, stream, cols, pl, (const uint32_t*)s.digits.p, cursor, sorted);
    H2B_CUDA(cudaGetLastError());
    ctx.prof.mark(PROF_MSM_SCATTER, stream);
    return H2B_OK;
}

// stage 2 of a chunk: accumulate the sorted list into the buckets, combine cut buckets, merge (chunked MSMs)
static int msm_accumulate_chunk(DeviceCtx& ctx, MsmScratch& s, const MsmPlan& pl, const void* tables, cudaStream_t stream) {
    const uint32_t* offsets = (const uint32_t*)s.offsets.p;
    const uint32_t* sorted = (const uint32_t*)s.sorted.p;
    uint32_t* ctrl = (uint32_t*)s.ctrl.p;
    uint4* target = (uint4*)(pl.add_into ? s.bucket_tmp.p : s.bucket_acc.p);
    H2B_CUDA(cudaMemsetAsync(ctrl, 0, 16, stream));
    ctx.prof.mark(PROF_BEGIN, stream);
    H2B_LAUNCH(msm_accumulate_kernel, (pl.G + 255) / 256, 256, 0, stream, pl, (const uint4*)tables, offsets, sorted, ctrl, (uint32_t*)s.split_list.p, target,
               (uint4*)s.head_partial.p);
    ctx.prof.mark(PROF_MSM_ACCUMULATE, stream);
    H2B_LAUNCH(msm_combine_light_kernel, (pl.G + 127) / 128, 128, 0, stream, pl, offsets, ctrl, (const uint32_t*)s.split_list.p,
               (HeavyDesc*)s.heavy.p, (uint2*)s.chunk_desc.p, (const uint4*)s.head_partial.p, target);
    H2B_LAUNCH(msm_combine_chunk_kernel, ctx.sm_count * 2, COMBINE_THREADS, 0, stream, pl, offsets, (const uint32_t*)ctrl, (const HeavyDesc*)s.heavy.p,
               (const uint2*)s.chunk_desc.p, (const uint4*)s.head_partial.p, (uint4*)s.chunk_out.p);
    H2B_LAUNCH(msm_combine_heavy_kernel, ctx.sm_count * 2, COMBINE_THREADS, 0, stream, (const uint32_t*)ctrl, (const HeavyDesc*)s.heavy.p, (const uint4*)s.chunk_out.p,
               target);
    if (pl.add_into)
        H2B_LAUNCH(msm_merge_kernel, (pl.B + 127) / 128, 128, 0, stream, pl.B, offsets, (const uint4*)target, (uint4*)s.bucket_acc.p);
    H2B_CUDA(cudaGetLastError());
    ctx.prof.mark(PROF_MSM_COMBINE, stream);
    return H2B_OK;
}

// All chunks of one MSM, each sorted and then accumulated on `stream`.  uploaded[j], when given, is the event after which
// chunk j's scalars are in device memory.
// bounds: nchunks + 1 ascending scalar indices, bounds[0] = 0, bounds[nchunks] = n
static int msm_run_chunks(DeviceCtx& ctx, MsmScratch& s, MsmPlan pl, const void* d_scalars, const MsmBases& bases, const std::vector<size_t>& bounds,
                          const cudaEvent_t* uploaded, cudaStream_t stream, const std::function<int(size_t)>* before_chunk = nullptr) {
    const size_t nchunks = bounds.size() - 1;
    for (size_t j = 0; j < nchunks; ++j) {
        const size_t done = bounds[j], m = bounds[j + 1] - bounds[j];
        const void* tables;
        size_t row0;
        chunk_points(bases, done, &tables, &row0);
        H2B_TRY(msm_size_chunk(ctx, s, pl, row0, (uint32_t)m));
        if (before_chunk) H2B_TRY((*before_chunk)(j));          // e.g. the staged upload of this chunk's scalars onto `stream`
        if (uploaded) H2B_CUDA(cudaStreamWaitEvent(stream, uploaded[j], 0));
        MsmCols cols;
        memset(&cols, 0, sizeof(cols));
        cols.scalars[0] = (const uint4*)((const char*)d_scalars + done * 32);
        cols.len[0] = (uint32_t)m;
        H2B_TRY(msm_sort_chunk(ctx, s, pl, cols, stream));
        H2B_TRY(msm_accumulate_chunk(ctx, s, pl, tables, stream));
    }
    return H2B_OK;
}

// bucket reduction hierarchy + Horner over the sets -> 224-byte result block (Jacobian | XYZZ)
static int msm_finish(DeviceCtx& ctx, MsmScratch& s, const MsmPlan& pl, void* d_result, bool accumulate, cudaStream_t stream) {
    // running sums over m = 2^logm buckets per thread and level: 16 while a level still fills the GPU (throughput),
    // 4 below that (each level is then a serial chain of 2m additions, and latency is all that matters)
    static int env_logm = -1;
    if (env_logm < 0) env_logm = env_int("H2B_MSM_REDUCE_LOGM", 0);
    const uint32_t sets = pl.ncols * pl.m;      // bucket sets in flight (batched MSM: m per column)
    uint32_t logm = (uint64_t)sets * pl.Nb >= (1u << 21) ? 4u : 2u;
    if (env_logm >= 1 && env_logm <= 6) logm = (uint32_t)env_logm;
    uint32_t N = pl.Nb;
    uint32_t J0 = (N + (1u << logm) - 1) >> logm;
    if (J0 < 1) J0 = 1;
    H2B_TRY(s.redA.reserve((size_t)sets * J0 * 128));
    H2B_TRY(s.redB.reserve((size_t)sets * J0 * 128));
    H2B_TRY(s.redC.reserve((size_t)sets * J0 * 128));
    H2B_TRY(s.redD.reserve((size_t)sets * J0 * 128));
    ctx.prof.mark(PROF_BEGIN, stream);
    const uint4* Bin = (const uint4*)s.bucket_acc.p;
    const uint4* Din = nullptr;
    // single-chunk MSMs never wrote their empty buckets: level 0 skips them by their sorted count
    const uint32_t* offs = pl.add_into ? nullptr : (const uint32_t*)s.offsets.p;
    uint4* Bping[2] = {(uint4*)s.redA.p, (uint4*)s.redB.p};
    uint4* Dping[2] = {(uint4*)s.redC.p, (uint4*)s.redD.p};
    int pp = 0;
    if (!ctx.msm_attr_set) {      // a per-device function attribute
        H2B_CUDA(cudaFuncSetAttribute(msm_reduce_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(REDUCE_TAIL_MAX * 128)));
        ctx.msm_attr_set = true;
    }
    // Levels that fill the GPU: chunked running sums, one thread per 2^logm items (work-efficient: 2 additions per item).  From
    // 2^14 items in flight down a level is pure latency: block levels (msm_reduce_block_kernel, 2.1 instead of 5.6 additions deep
    // per bit).  Measured (profiles/r02_block_reduce.jsonl): reduction 0.52 -> 0.31 ms at 2^15 buckets (a 2^16-point MSM: 0.87 ->
    // 0.66 ms), 0.96 -> 0.75 ms at 2^19; switching at 2^16 items is 0.05 ms slower, 128- and 64-item blocks are equal, 256 slower.
    // H2B_MSM_REDUCE_BLOCK_MAX_LOG moves the switch (0 = chunked levels all the way down to the tail, as in round 1).
    static int env_block_log = -1;
    if (env_block_log < 0) { env_block_log = env_int("H2B_MSM_REDUCE_BLOCK_MAX_LOG", 14); if (env_block_log > 24) env_block_log = 24; }
    static int env_block = -1, env_tail = -1;
    if (env_block < 0) { env_block = env_int("H2B_MSM_REDUCE_BLOCK", (int)REDUCE_BLOCK); if (env_block != 64 && env_block != 128 && env_block != 256 && env_block != 512) env_block = (int)REDUCE_BLOCK; }
    if (env_tail < 0) { env_tail = env_int("H2B_MSM_REDUCE_TAIL", (int)REDUCE_TAIL_MAX); if (env_tail != 64 && env_tail != 128 && env_tail != 256 && env_tail != 512) env_tail = (int)REDUCE_TAIL_MAX; }
    const uint32_t block_m = (uint32_t)env_block, tail_max = (uint32_t)env_tail;
    while (N > tail_max) {
        if (env_block_log > 0 && (uint64_t)sets * N <= ((uint64_t)1 << env_block_log)) {
            const uint32_t J = (N + block_m - 1) / block_m;
            H2B_LAUNCH(msm_reduce_block_kernel, dim3(J, sets), block_m, (size_t)block_m * 128, stream, Bin, Din, offs, N, Bping[pp], Dping[pp]);
            Bin = Bping[pp];
            Din = Dping[pp];
            offs = nullptr;
            pp ^= 1;
            N = J;
            continue;
        }
        uint32_t J = (N + (1u << logm) - 1) >> logm;
        uint32_t threads = sets * J;
        H2B_LAUNCH(msm_reduce_level_kernel, (threads + 127) / 128, 128, 0, stream, Bin, Din, offs, N, logm, sets, Bping[pp], Dping[pp]);
        Bin = Bping[pp];
        Din = Dping[pp];
        offs = nullptr;
        pp ^= 1;
        N = J;
        if (env_logm < 1 && (uint64_t)sets * N < (1u << 21)) logm = 2;
    }
    {
        uint32_t tthreads = 32;
        while (tthreads < N) tthreads <<= 1;
        H2B_LAUNCH(msm_reduce_block_kernel, dim3(1, sets), tthreads, (size_t)tthreads * 128, stream, Bin, Din, offs, N, (uint4*)nullptr, Dping[pp]);
        Din = Dping[pp];
    }
    ctx.prof.mark(PROF_MSM_REDUCE, stream);
    H2B_LAUNCH(msm_final_kernel, pl.ncols, 32, 0, stream, Din, pl.m, pl.c, (uint4*)d_result, accumulate ? 1u : 0u);
    H2B_CUDA(cudaGetLastError());
    ctx.prof.mark(PROF_MSM_FINAL, stream);
    return H2B_OK;
}

static int msm_check_args(const void* scalars, const MsmBases& bases, size_t n, const void* out) {
    if (!scalars || !bases.tables || !out) { set_error("msm: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (bases.n_tables > 1 && (bases.row0 + n > bases.stride || (uint64_t)bases.stride * bases.n_tables >= 0x80000000ull)) {
        set_error("msm: range [%zu, %zu) does not fit the %u x %zu table set", bases.row0, bases.row0 + n, bases.n_tables, bases.stride);
        return H2B_ERR_BAD_ARGUMENT;
    }
    return H2B_OK;
}

static int msm_identity(void* d_out, size_t out_bytes, cudaStream_t stream) {
    // identity: Jacobian (0, 1, 0), XYZZ all-zero
    uint32_t host[56];
    memset(host, 0, sizeof(host));
    for (int i = 0; i < 8; ++i) host[8 + i] = FpParams<FQ>::ONE(i);
    H2B_CUDA(cudaMemcpyAsync(d_out, host, out_bytes, cudaMemcpyHostToDevice, stream));
    H2B_CUDA(cudaStreamSynchronize(stream));
    return H2B_OK;
}

// Scalars already on the device.  d_out_jac: 96 bytes (x|y|z Montgomery), or the 224-byte block (Jacobian | XYZZ).
int msm_run(DeviceCtx& ctx, const void* d_scalars, const MsmBases& bases, size_t n, void* d_out_jac, bool with_xyzz, cudaStream_t stream) {
    if (!ctx.msm) ctx.msm = new MsmScratch();
    MsmScratch& s = *ctx.msm;
    H2B_TRY(s.result.reserve(256));
    const size_t out_bytes = with_xyzz ? 224 : 96;
    if (n == 0) return msm_identity(d_out_jac, out_bytes, stream);
    H2B_TRY(msm_check_args(d_scalars, bases, n, d_out_jac));
    // device-resident scalars need no chunks below 2^26 points (H2B_MSM_DEVICE_CHUNKS > 1 splits anyway: tests, tuning)
    const size_t MAX_CHUNK = (size_t)1 << 26;
    static int env_dev_chunks = -1;
    if (env_dev_chunks < 0) env_dev_chunks = env_int("H2B_MSM_DEVICE_CHUNKS", 1);
    size_t chunk = n;
    static int env_dev_min = -1;
    if (env_dev_min < 0) env_dev_min = env_int("H2B_MSM_DEVICE_CHUNK_MIN_LOG", 22);      // tests lower it
    if (env_dev_chunks > 1 && n >= ((size_t)1 << env_dev_min)) chunk = (n + env_dev_chunks - 1) / env_dev_chunks;
    if (chunk > MAX_CHUNK) chunk = MAX_CHUNK;
    MsmPlan pl;
    H2B_TRY(msm_plan(ctx, s, bases, n, chunk < n, stream, pl));
    std::vector<size_t> bounds;
    for (size_t done = 0; done < n; done += chunk) bounds.push_back(done);
    bounds.push_back(n);
    H2B_TRY(msm_run_chunks(ctx, s, pl, d_scalars, bases, bounds, nullptr, stream));
    H2B_TRY(msm_finish(ctx, s, pl, s.result.p, false, stream));
    H2B_CUDA(cudaMemcpyAsync(d_out_jac, s.result.p, out_bytes, cudaMemcpyDeviceToDevice, stream));
    return H2B_OK;
}

// Scalars in host memory (the drop-in entry points): the upload is cut into chunks on a second stream, and chunk
// j + 1 crosses PCIe while chunk j is sorted and accumulated, so only the first chunk's transfer is exposed.
// d_staging: device buffer of at least n * 32 bytes.  Synchronous: returns with the result block in `h_out_block`.
int msm_run_host(DeviceCtx& ctx, const void* h_scalars, void* d_staging, const MsmBases& bases, size_t n, void* h_out_block /* 224 B */) {
    if (!ctx.msm) ctx.msm = new MsmScratch();
    MsmScratch& s = *ctx.msm;
    cudaStream_t stream = ctx.stream;
    H2B_TRY(s.result.reserve(256));
    if (n == 0) {
        H2B_TRY(msm_identity(s.result.p, 224, stream));
        H2B_CUDA(cudaMemcpyAsync(h_out_block, s.result.p, 224, cudaMemcpyDeviceToHost, stream));
        H2B_CUDA(cudaStreamSynchronize(stream));
        return H2B_OK;
    }
    H2B_TRY(msm_check_args(h_scalars, bases, n, h_out_block));
    // From 2^22 points up the upload is cut into a short first chunk (1/16: the only transfer nothing can hide) and three
    // chunks of 5/16 whose transfers hide behind the previous chunk's kernels (profiles/r01_msm_e2e_chunks.txt).
    // H2B_MSM_UPLOAD_CHUNK_LOG forces a uniform chunk size (tests).
    static int env_chunk = -1;
    if (env_chunk < 0) env_chunk = env_int("H2B_MSM_UPLOAD_CHUNK_LOG", 0);
    std::vector<size_t> bounds;
    if (env_chunk >= 10 && env_chunk <= 26 && n >= ((size_t)2 << env_chunk)) {
        for (size_t done = 0; done < n; done += (size_t)1 << env_chunk) bounds.push_back(done);
    } else if (env_chunk == 0 && n >= ((size_t)1 << env_int("H2B_MSM_UPLOAD_MIN_LOG", host_is_pageable(h_scalars) ? 20 : 21))) {
        // (measured, profiles/r02_e2e_matrix.jsonl: chunking pays from 2^21 points with pinned scalars -- 7.20 -> 6.96 ms; 2^20: 4.10 -> 4.29 ms --
        // and from 2^20 with pageable ones -- 5.81 -> 5.10 ms, 2^21: 8.48 -> 8.23 ms: the per-device share of a point-range split is that small)
        const size_t u = n / 16;
        // Pinned scalars: every DMA is queued up front and PCIe is 4x faster than the kernels consume scalars: a short first chunk
        // (1/32: the only transfer nothing can hide), then 4 : 11 : 16.  Pageable scalars are copied by host threads (stage.cu) right
        // before a chunk's kernels are queued, at only ~3x the rate the GPU consumes them: chunk j + 1 has to be copied within the
        // GPU time of chunk j, so the chunks grow 1 : 3 : 7 : 5 sixteenths (with 1 : 5 : 5 : 5 the GPU idled ~2 ms waiting for chunk 1).
        // Measured at 2^24 (profiles/r02_e2e_matrix.jsonl): pageable 46.1 -> 44.2 ms, pinned 42.9 -> 42.3 ms (41.4 device-resident).
        if (host_is_pageable(h_scalars)) bounds = {0, u, 4 * u, 11 * u};
        else bounds = {0, u / 2, 5 * (u / 2), 8 * u};
        if (const char* sched = getenv("H2B_MSM_UPLOAD_SCHED")) {      // tuning: chunk weights, e.g. "1,3,12,16" (any sum)
            std::vector<size_t> wts;
            size_t total = 0;
            for (const char* q = sched; *q;) { char* end; const unsigned long v = strtoul(q, &end, 10); if (end == q) break; wts.push_back(v); total += v; q = *end ? end + 1 : end; }
            if (wts.size() >= 1 && wts.size() <= 16 && total > 0) {
                bounds.clear();
                size_t acc = 0;
                for (size_t v : wts) { bounds.push_back((size_t)((unsigned __int128)n * acc / total)); acc += v; }
                for (size_t j = 1; j < bounds.size(); ++j) if (bounds[j] <= bounds[j - 1]) { bounds = {0}; break; }
            }
        }
    } else {
        bounds.push_back(0);
    }
    bounds.push_back(n);
    const size_t nchunks = bounds.size() - 1;
    if (!ctx.copy_stream) H2B_CUDA(cudaStreamCreateWithFlags(&ctx.copy_stream, cudaStreamNonBlocking));
    while (ctx.copy_events.size() < nchunks) {
        cudaEvent_t e;
        H2B_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx.copy_events.push_back(e);
    }
    MsmPlan pl;
    H2B_TRY(msm_plan(ctx, s, bases, n, nchunks > 1, stream, pl));
    if (host_is_pageable(h_scalars)) {
        // pageable caller memory (a Rust Vec): chunk j is copied through pinned slots by a few host threads right before
        // its kernels are queued, so the CPU copy of chunk j + 1 overlaps the GPU work of chunk j (stage.cu)
        std::function<int(size_t)> upload = [&](size_t j) -> int {
            const size_t done = bounds[j], m = bounds[j + 1] - bounds[j];
            // only chunk 0 has to wait for the previous call's kernels (they may still read the staging buffer); the
            // other chunks land in regions nothing in flight touches, so their DMA overlaps the GPU work of chunk j - 1
            return host_upload(ctx, (char*)d_staging + done * 32, (const char*)h_scalars + done * 32, m * 32, stream, j == 0);
        };
        H2B_TRY(msm_run_chunks(ctx, s, pl, d_staging, bases, bounds, nullptr, stream, &upload));
    } else {
        // pinned caller memory: every chunk's DMA is queued up front on the copy stream
        // (the staging buffer may still be read by the previous call's kernels on `stream`: order the copies after them)
        if (nchunks > 1) {
            H2B_CUDA(cudaEventRecord(ctx.copy_events[0], stream));
            H2B_CUDA(cudaStreamWaitEvent(ctx.copy_stream, ctx.copy_events[0], 0));
        }
        for (size_t j = 0; j < nchunks; ++j) {
            const size_t done = bounds[j], m = bounds[j + 1] - bounds[j];
            cudaStream_t cs = nchunks > 1 ? ctx.copy_stream : stream;
            H2B_CUDA(cudaMemcpyAsync((char*)d_staging + done * 32, (const char*)h_scalars + done * 32, m * 32, cudaMemcpyHostToDevice, cs));
            if (nchunks > 1) H2B_CUDA(cudaEventRecord(ctx.copy_events[j], cs));
        }
        H2B_TRY(msm_run_chunks(ctx, s, pl, d_staging, bases, bounds, nchunks > 1 ? ctx.copy_events.data() : nullptr, stream));
    }
    H2B_TRY(msm_finish(ctx, s, pl, s.result.p, false, stream));
    H2B_CUDA(cudaMemcpyAsync(h_out_block, s.result.p, 224, cudaMemcpyDeviceToHost, stream));
    H2B_CUDA(cudaStreamSynchronize(stream));
    return H2B_OK;
}

// ---- batched MSM: `count` independent scalar columns over the same points, one kernel sequence ----------------------------
// d_cols[j]: lens[j] scalars on the device; every column uses rows [row0, row0 + lens[j]) of the point set.  d_out_blocks:
// count x 224 bytes (Jacobian | XYZZ per column).  The window is chosen for the longest column.
int msm_run_batch(DeviceCtx& ctx, const void* const* d_cols, const size_t* lens, uint32_t count, const MsmBases& bases, void* d_out_blocks, cudaStream_t stream) {
    if (count == 0) return H2B_OK;
    if (count > MSM_BATCH_MAX) { set_error("msm batch: at most %u columns per call", MSM_BATCH_MAX); return H2B_ERR_BAD_ARGUMENT; }
    if (!ctx.msm) ctx.msm = new MsmScratch();
    MsmScratch& s = *ctx.msm;
    size_t n_max = 0;
    for (uint32_t j = 0; j < count; ++j) n_max = lens[j] > n_max ? lens[j] : n_max;
    H2B_TRY(s.result.reserve((size_t)MSM_BATCH_MAX * 224));
    if (n_max == 0) {
        uint32_t host[56];
        memset(host, 0, sizeof(host));
        for (int i = 0; i < 8; ++i) host[8 + i] = FpParams<FQ>::ONE(i);
        for (uint32_t j = 0; j < count; ++j) H2B_CUDA(cudaMemcpyAsync((char*)d_out_blocks + 224 * (size_t)j, host, 224, cudaMemcpyHostToDevice, stream));
        H2B_CUDA(cudaStreamSynchronize(stream));
        return H2B_OK;
    }
    MsmCols cols;
    memset(&cols, 0, sizeof(cols));
    for (uint32_t j = 0; j < count; ++j) {
        if (lens[j] && !d_cols[j]) { set_error("msm batch: column %u is null", j); return H2B_ERR_BAD_ARGUMENT; }
        cols.scalars[j] = (const uint4*)d_cols[j];
        cols.len[j] = (uint32_t)lens[j];
    }
    H2B_TRY(msm_check_args(d_cols, bases, n_max, d_out_blocks));
    if (n_max > ((size_t)1 << 26)) { set_error("msm batch: columns of at most 2^26 scalars"); return H2B_ERR_BAD_ARGUMENT; }
    MsmPlan pl;
    H2B_TRY(msm_plan(ctx, s, bases, n_max, false, stream, pl, count));
    const void* tables;
    size_t row0;
    chunk_points(bases, 0, &tables, &row0);
    H2B_TRY(msm_size_chunk(ctx, s, pl, row0, (uint32_t)n_max));
    H2B_TRY(msm_sort_chunk(ctx, s, pl, cols, stream));
    H2B_TRY(msm_accumulate_chunk(ctx, s, pl, tables, stream));
    H2B_TRY(msm_finish(ctx, s, pl, s.result.p, false, stream));
    H2B_CUDA(cudaMemcpyAsync(d_out_blocks, s.result.p, 224 * (size_t)count, cudaMemcpyDeviceToDevice, stream));
    return H2B_OK;
}

// the same with the columns in host memory: uploads into d_staging (count x n_max x 32 bytes at least), synchronous,
// h_out_blocks: count x 224 bytes
int msm_run_host_batch(DeviceCtx& ctx, const void* const* h_cols, const size_t* lens, uint32_t count, void* d_staging, const MsmBases& bases, void* h_out_blocks) {
    if (count == 0) return H2B_OK;
    if (count > MSM_BATCH_MAX) { set_error("msm batch: at most %u columns per call", MSM_BATCH_MAX); return H2B_ERR_BAD_ARGUMENT; }
    cudaStream_t stream = ctx.stream;
    const void* d_cols[MSM_BATCH_MAX];
    size_t off = 0;
    for (uint32_t j = 0; j < count; ++j) {
        d_cols[j] = (char*)d_staging + off;
        if (lens[j]) {
            if (!h_cols[j]) { set_error("msm batch: column %u is null", j); return H2B_ERR_BAD_ARGUMENT; }
            H2B_TRY(host_upload(ctx, (char*)d_staging + off, h_cols[j], lens[j] * 32, stream, j == 0));
        }
        off += lens[j] * 32;
    }
    if (!ctx.msm) ctx.msm = new MsmScratch();
    H2B_TRY(ctx.msm->batch_out.reserve((size_t)MSM_BATCH_MAX * 224));
    H2B_TRY(msm_run_batch(ctx, d_cols, lens, count, bases, ctx.msm->batch_out.p, stream));
    H2B_CUDA(cudaMemcpyAsync(h_out_blocks, ctx.msm->batch_out.p, 224 * (size_t)count, cudaMemcpyDeviceToHost, stream));
    H2B_CUDA(cudaStreamSynchronize(stream));
    return H2B_OK;
}
uint32_t msm_batch_max() { return MSM_BATCH_MAX; }

// sum of `count` partial results (224-byte blocks: Jacobian | XYZZ) -> Jacobian.  Used to fold the per-device
// partial sums of a point-range-sharded MSM (SURVEY.md section 8e).
__global__ void msm_sum_partials_kernel(const uint4* __restrict__ blocks, uint32_t count, uint4* __restrict__ out_jac) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    XYZZ acc = xyzz_identity();
    for (uint32_t i = 0; i < count; ++i) {
        XYZZ p = xyzz_load(blocks + 14 * (size_t)i + 6);
        xyzz_add<true>(acc, p);
    }
    Fq X, Y, Z;
    xyzz_to_jacobian(acc, X, Y, Z);
    fp_store<FQ>(out_jac, X);
    fp_store<FQ>(out_jac + 2, Y);
    fp_store<FQ>(out_jac + 4, Z);
}
int msm_sum_partials_run(DeviceCtx& ctx, const void* d_blocks, uint32_t count, void* d_out_jac, cudaStream_t stream) {
    (void)ctx;
    H2B_LAUNCH(msm_sum_partials_kernel, 1, 32, 0, stream, (const uint4*)d_blocks, count, (uint4*)d_out_jac);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

void msm_release(DeviceCtx& ctx) {
    if (!ctx.msm) return;
    MsmScratch& s = *ctx.msm;
    DevBuf* all[] = {&s.digits, &s.counts, &s.offsets, &s.cursor, &s.block_sums, &s.sorted, &s.ctrl, &s.split_list, &s.heavy, &s.chunk_desc, &s.chunk_out,
                     &s.bucket_acc, &s.bucket_tmp, &s.head_partial, &s.redA, &s.redB, &s.redC, &s.redD, &s.result, &s.batch_out,
                     &s.part_counts, &s.part_off, &s.part_cursor, &s.chunk0, &s.chunk_hist, &s.inter};
    for (DevBuf* b : all) b->release();
    delete ctx.msm;
    ctx.msm = nullptr;
}

}  // namespace h2b
