// Shared host-side plumbing of libh2b200: per-device context, error reporting, scratch buffers.
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/h2b200.h"   // H2B_OK / H2B_ERR_* codes
#include "field.cuh"

namespace h2b {

void set_error(const char* fmt, ...);
const char* get_error();

#define H2B_CUDA(expr)                                                                           \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            h2b::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return (_e == cudaErrorMemoryAllocation) ? H2B_ERR_OOM : H2B_ERR_CUDA;     \
        }                                                                                        \
    } while (0)

#define H2B_TRY(expr)             \
    do {                          \
        int _r = (expr);          \
        if (_r != 0) return _r;   \
    } while (0)

// 16-byte global -> shared copy that does not pass through registers (LDGSTS): a thread issues its copies back to
// back and waits once, so a tile load costs one memory latency instead of one per element (NTT), and a gathered point
// waits in shared memory instead of registers (MSM accumulation).
__device__ __forceinline__ void copy16_async(uint4* smem_dst, const uint4* gmem_src) {
#ifdef H2B_EMU
    *smem_dst = *gmem_src;
#else
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem_src) : "memory");
#endif
}
__device__ __forceinline__ void copy_async_wait_all() {
#ifndef H2B_EMU
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
#endif
}

// A grow-only device buffer (scratch space reused across calls on one device).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return H2B_OK;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&p, want);
        // a failed allocation stays the thread's last error, which the next launch check would report: clear it
        if (e != cudaSuccess) {
            cudaGetLastError();
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
            return H2B_ERR_OOM;
        }
        cap = want;
        return H2B_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// value #index (0-based) of the SplitMix64 stream `seed`: the synthetic points and scalars (g1gen.cu, testgen.cu)
__host__ __device__ __forceinline__ uint64_t splitmix64_at(uint64_t seed, uint64_t index) {
    uint64_t z = seed + (index + 1) * 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

// w (4 little-endian words) is below the scalar field modulus r
inline bool fr_canonical(const uint64_t w[4]) {
    uint32_t l[8];
    memcpy(l, w, 32);
    for (int i = 7; i >= 0; --i) {
        if (l[i] < FpParams<FR>::P(i)) return true;
        if (l[i] > FpParams<FR>::P(i)) return false;
    }
    return false;
}

// Optional per-kernel timing with CUDA events on the launching stream (bench.py's roofline numbers).
enum ProfTag { PROF_BEGIN = 0, PROF_MSM_DECOMPOSE = 1, PROF_MSM_SCAN = 2, PROF_MSM_SCATTER = 3, PROF_MSM_PLAN = 4, PROF_MSM_ACCUMULATE = 5,
               PROF_MSM_COMBINE = 6, PROF_MSM_REDUCE = 7, PROF_MSM_FINAL = 8, PROF_MSM_PRECOMPUTE = 9, PROF_NTT_TWIDDLE = 15, PROF_NTT_PASS0 = 16,
               PROF_SRS_SCALARS = 24, PROF_SRS_FIXED_BASE = 25, PROF_SRS_NORMALISE = 26, PROF_SRS_TABLE = 27,
               PROF_G1NTT_TWIDDLE = 28, PROF_G1NTT_STAGES = 29, PROF_G1NTT_NORMALISE = 30,
               PROF_KEYGEN_UPLOAD = 31, PROF_KEYGEN_SIGMA = 32, PROF_KEYGEN_COMMIT = 33, PROF_KEYGEN_INTT = 34, PROF_KEYGEN_COSET = 35,
               PROF_KEYGEN_DOWNLOAD = 36, PROF_KEYGEN_PACK = 37, PROF_KEYGEN_EXCLUSION = 38, PROF_KEYGEN_FIXED_UPLOAD = 39,
               PROF_KEYGEN_COMBINATION = 40, PROF_PK_FORM_COPY = 41, PROF_PK_PLACE = 42,
               PROF_OPEN_UPLOAD = 43, PROF_OPEN_EVAL = 44, PROF_OPEN_SCALARS = 45, PROF_OPEN_NUMERATORS = 46, PROF_OPEN_MSM = 47,
               PROF_OPEN_LINEARISE = 48, PROF_MOCK_UPLOAD = 49, PROF_MOCK_GATES = 50, PROF_MOCK_LOOKUPS = 51, PROF_MOCK_PERMUTATION = 52,
               PROF_MOCK_RECORDS = 53, PROF_GWC_UPLOAD = 54, PROF_GWC_SCALARS = 55, PROF_GWC_NUMERATORS = 56, PROF_GWC_DIVISIONS = 57,
               PROF_GWC_MSM = 58 };
struct Profiler {
    bool enabled = false;
    std::vector<cudaEvent_t> ev;
    std::vector<int> tag;
    size_t used = 0;
    void mark(int t, cudaStream_t stream) {
        if (!enabled || used >= ev.size()) return;
        cudaEventRecord(ev[used], stream);
        tag[used++] = t;
    }
};

struct Stager;        // stage.cu
struct NttTwiddles;   // ntt.cu
struct MsmScratch;    // msm.cu
struct EvalScratch;   // evaluate.cu

struct DeviceCtx {
    int device = -1;
    int sm_count = 148;
    cudaStream_t stream = nullptr;     // stream used by the host-pointer entry points
    cudaStream_t copy_stream = nullptr;   // chunked scalar uploads of the host-pointer MSM (overlap with compute)
    std::vector<cudaEvent_t> copy_events;
    std::mutex mu;                     // serialises calls that share this context's scratch
    DevBuf ntt_work;                   // ping-pong buffer of the multi-pass NTT
    bool ntt_attr_set = false;
    bool msm_attr_set = false;
    DevBuf ntt_io;                     // staging for the host-pointer NTT entry point
    DevBuf ntt_fs[2];                  // the two other matrices of the multi-device four-step NTT (api_sets.cu: ntt_multi_device)
    DevBuf col_ext;                    // extended form of h2b_column_pipeline when the caller only wants it on the host
    DevBuf scale_table;                // factor table of h2b_fr_scale_dev with more than 8 factors
    DevBuf msm_scalars;                // staging for host-pointer MSM scalars
    DevBuf msm_out;                    // 96-byte result
    DevBuf msm_bases;                  // points of an uncached host-pointer MSM (small / odd-length calls: uploaded per call)
    DevBuf scan_scratch;               // batch inversion / prefix product scratch (scan.cu)
    DevBuf srs_status, srs_io;         // first-invalid-point flag and encoded-bytes staging of the SRS reader (srs.cu)
    DevBuf lookup_scratch;             // sorted keys, flags and ranks of permute_expression_pair (lookup.cu)
    DevBuf gen_table;                  // fixed-base table of the G1 generator, built on first use (g1gen.cu)
    DevBuf gen_scratch;                // normalisation denominators and SRS scalars of one chunk; the G1 NTT work buffer (g1gen.cu)
    DevBuf keygen_tables;              // the two-level delta^c omega^r tables of the sigma kernel (keygen.cu)
    DevBuf open_scratch;               // point powers and level values of the query evaluation (multiopen.cu)
    DevBuf open_tables;                // plan tables and pair values of h2b_fr_eval_queries_dev (api_open.cu)
    EvalScratch* eval = nullptr;       // compiled-program ring of the quotient evaluation (evaluate.cu)
    std::vector<NttTwiddles*> twiddles;  // small LRU cache keyed by (omega, log_n)
    MsmScratch* msm = nullptr;
    Profiler prof;
    Stager* stager = nullptr;          // pinned slots + worker streams for pageable host buffers
    void* pinned = nullptr;            // small pinned bounce buffer
    size_t pinned_cap = 0;
};

// ---- stage.cu ----
int host_upload(DeviceCtx& ctx, void* d_dst, const void* h_src, size_t bytes, cudaStream_t consumer, bool order_after_consumer = true);
int host_download(DeviceCtx& ctx, void* h_dst, const void* d_src, size_t bytes, cudaStream_t producer);
// `height` rows of `width` bytes: host rows are `h_pitch` bytes apart, the device side is packed
int host_upload_2d(DeviceCtx& ctx, void* d_dst, const void* h_src, size_t h_pitch, size_t width, size_t height, cudaStream_t consumer);
int host_download_2d(DeviceCtx& ctx, void* h_dst, size_t h_pitch, const void* d_src, size_t width, size_t height, cudaStream_t producer);
void stager_release(DeviceCtx& ctx);
bool host_is_pageable(const void* p);
// ---- scan.cu ----
// polynomial evaluation and division by (X - b) run in levels of POLY_K coefficients; the powers x^(16^l), l < POLY_LEVELS_MAX, of one
// point take POLY_PTS elements, the last of them the point itself
static const uint32_t POLY_K = 16;
static const uint32_t POLY_LEVELS_MAX = 9;                 // 16^8 > 2^31
static const uint32_t POLY_PTS = POLY_LEVELS_MAX + 1;
static const uint32_t SCAN_BLOCK = 1024;                   // elements per CTA of u32_exclusive_scan (256 threads x 4)
int fr_batch_invert_run(DeviceCtx& ctx, void* d_a, size_t n, cudaStream_t stream);
int fq_batch_invert_run(DeviceCtx& ctx, void* d_a, size_t n, cudaStream_t stream);
int fr_prefix_product_run(DeviceCtx& ctx, const void* d_in, void* d_out, size_t n, cudaStream_t stream);
int fr_eval_polynomial_run(DeviceCtx& ctx, const void* d_coeffs, size_t n, const uint64_t x[4], void* d_out, cudaStream_t stream);
int fr_kate_division_run(DeviceCtx& ctx, const void* d_a, size_t n, const uint64_t b[4], void* d_q, cudaStream_t stream);
// the same with the point b already on the device (d_b: one Fr, outside ctx.scan_scratch)
int fr_kate_division_at_run(DeviceCtx& ctx, const void* d_a, size_t n, const void* d_b, void* d_q, cudaStream_t stream);
// `count` divisions of length n in one launch sequence: division d divides the n Fr at d_a + d n by (X - d_b[d]) into d_q + d n (n - 1
// coefficients; d_b: count consecutive Fr on the device, outside ctx.scan_scratch).  count = 1 is fr_kate_division_at_run.
int fr_kate_division_batch_run(DeviceCtx& ctx, const void* d_a, size_t n, const void* d_b, uint32_t count, void* d_q, cudaStream_t stream);
// the powers of `count` points (back to back at d_x) into d_pts, point y's at d_pts + y POLY_PTS
int fr_point_powers_run(const void* d_x, uint32_t count, void* d_pts, cudaStream_t stream);
// `count` vectors of m values back to back at d_in, vector y at the point whose powers are at d_pts + y POLY_PTS, from `level` on:
// one launch per level, the partial values of every level in d_buf (count (m / 15 + 1) elements), the count values to d_out
int fr_horner_levels_run(const void* d_in, size_t m, const void* d_pts, uint32_t level, uint32_t count, void* d_buf, void* d_out, cudaStream_t stream);
// exclusive scan of `count` 32-bit values: out[i] = in[0] + .. + in[i-1], out[count] = total, out2 (optional) = out[0, count) again;
// `sums` holds ceil(count / SCAN_BLOCK) + 1 words
int u32_exclusive_scan(const uint32_t* in, uint32_t count, uint32_t* out, uint32_t* out2, uint32_t* sums, cudaStream_t stream);
int fr_lincomb_run(DeviceCtx& ctx, const void* const* d_cols, const uint64_t* coeffs, uint32_t m, size_t n, void* d_out, cudaStream_t stream);
int permutation_product_run(DeviceCtx& ctx, const void* const* d_values, const void* const* d_sigma, uint32_t m, size_t n, const uint64_t* beta,
                            const uint64_t* gamma, const uint64_t* delta, const uint64_t* deltaomega, const uint64_t* omega, const uint64_t* last_z,
                            void* d_z, cudaStream_t stream);
int lookup_product_run(DeviceCtx& ctx, const void* d_compressed_input, const void* d_compressed_table, const void* d_permuted_input,
                       const void* d_permuted_table, size_t n, const uint64_t* beta, const uint64_t* gamma, void* d_z, cudaStream_t stream);
// ---- lookup.cu ----
int lookup_permute_run(DeviceCtx& ctx, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                       void* d_status, cudaStream_t stream);
// ---- srs.cu ----
int g1_decode_run(DeviceCtx& ctx, const void* d_bytes, size_t n, int format, void* d_out, uint64_t* first_invalid, cudaStream_t stream);
int g1_encode_run(DeviceCtx& ctx, const void* d_affine, size_t n, void* d_out_bytes, cudaStream_t stream);
// ---- evaluate.cu ----
int evaluate_graph_run(DeviceCtx& ctx, const h2b_graph* g, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                       const h2b_eval_shard* shard, cudaStream_t stream);
int evaluate_h_lookup_run(DeviceCtx& ctx, const h2b_graph* g, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                          const void* d_product, const void* d_permuted_input, const void* d_permuted_table, const void* d_l0, const void* d_l_last,
                          const void* d_l_active_row, const h2b_eval_shard* shard, cudaStream_t stream);
int evaluate_h_permutation_run(DeviceCtx& ctx, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                               const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len, int32_t last_rotation,
                               const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t* beta, const uint64_t* gamma,
                               const uint64_t* y, const uint64_t* delta, const uint64_t* zeta, const uint64_t* extended_omega, const h2b_eval_shard* shard,
                               cudaStream_t stream);
void evaluate_graph_last_info(uint32_t* slots, uint32_t* micro_ops);
void evaluate_release(DeviceCtx& ctx);
// ---- ntt.cu ----
int ntt_run(DeviceCtx& ctx, void* d_a, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream);
int ntt_run_batch(DeviceCtx& ctx, void* const* d_polys, size_t count, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream);
uint32_t ntt_batch_max();
int ntt_run_strided(DeviceCtx& ctx, void* d_base, size_t count, size_t stride_elems, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream);
int fr_transpose_run(DeviceCtx& ctx, const void* d_in, void* d_out, uint32_t rows, uint32_t cols, cudaStream_t stream);
int ntt_fourstep_twiddle_run(DeviceCtx& ctx, void* d_y, uint32_t rows, uint32_t log_len, uint32_t row0, const uint64_t omega[4], cudaStream_t stream);
int ntt_root_powers_run(DeviceCtx& ctx, const uint64_t omega[4], uint32_t e0, uint32_t e1, void* d_out, cudaStream_t stream);
int ntt_scale_run(DeviceCtx& ctx, void* d_a, size_t n, const uint64_t* factors /*host, count x 4*/, int count, cudaStream_t stream);
int ntt_scale_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t ncols, size_t n, const uint64_t* factors, int count, cudaStream_t stream);
int lagrange_to_coeff_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t count, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4],
                                cudaStream_t stream);
int coeff_to_extended_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t count, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4],
                                const uint64_t zeta_powers[12], cudaStream_t stream);
void ntt_release(DeviceCtx& ctx);
// ---- msm.cu ----
// The points of an MSM: table j (j < n_tables) holds 2^(c0*j) * P_i at rows [0, stride); the call uses rows
// [row0, row0 + n) of every table.  n_tables == 1 is the plain, table-less mode (c0 ignored).
struct MsmBases {
    const void* tables = nullptr;
    uint32_t n_tables = 1;
    uint32_t c0 = 0;
    size_t stride = 0;
    size_t row0 = 0;
};
int msm_run(DeviceCtx& ctx, const void* d_scalars, const MsmBases& bases, size_t n, void* d_out, bool with_xyzz, cudaStream_t stream);
int msm_run_host(DeviceCtx& ctx, const void* h_scalars, void* d_staging, const MsmBases& bases, size_t n, void* h_out_block);
int msm_run_batch(DeviceCtx& ctx, const void* const* d_cols, const size_t* lens, uint32_t count, const MsmBases& bases, void* d_out_blocks, cudaStream_t stream);
int msm_run_host_batch(DeviceCtx& ctx, const void* const* h_cols, const size_t* lens, uint32_t count, void* d_staging, const MsmBases& bases, void* h_out_blocks);
uint32_t msm_batch_max();
int msm_precompute_run(DeviceCtx& ctx, const void* d_src, void* d_dst, size_t n, uint32_t c0, cudaStream_t stream);
uint32_t msm_pick_table_spacing(size_t n, uint32_t max_tables);
uint32_t msm_tables_for(uint32_t c0);
int msm_sum_partials_run(DeviceCtx& ctx, const void* d_blocks, uint32_t count, void* d_out_jac, cudaStream_t stream);
void msm_release(DeviceCtx& ctx);
int msm_set_window(int c);   // 0 = automatic
// ---- g1gen.cu ----
int gen_points_run(DeviceCtx& ctx, uint64_t seed, size_t n, void* d_out_affine, cudaStream_t stream);
int g1_generator_mul_run(DeviceCtx& ctx, const void* d_scalars, size_t n, void* d_out_affine, cudaStream_t stream);
int srs_setup_check(uint32_t k, const uint64_t s[4]);
int srs_setup_run(DeviceCtx& ctx, uint32_t k, const uint64_t s[4], int which, void* d_out_affine, cudaStream_t stream);
// g_to_lagrange of the first 2^k affine points of d_g into d_out (may equal d_g); asynchronous, scratch in gen_scratch
int g1_to_lagrange_run(DeviceCtx& ctx, const void* d_g, uint32_t k, void* d_out_affine, cudaStream_t stream);
// after a synchronous call: drop the chunk scratch, and scan_scratch if the call grew it (the generator table stays)
void g1gen_release_scratch(DeviceCtx& ctx, size_t scan_cap_before);
// ---- keygen.cu ----
// the lo / hi tables of sigma for n_columns columns at k into ctx.keygen_tables (stream-ordered; must precede permutation_sigma_run)
int permutation_sigma_tables_run(DeviceCtx& ctx, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4], cudaStream_t stream);
// sigma of `count` mapping columns (flat column index col0 + y for the status word), with the tables of the last permutation_sigma_tables_run
int permutation_sigma_run(DeviceCtx& ctx, const void* const* d_mapping, uint32_t count, uint32_t col0, uint32_t n_columns, uint32_t k,
                          void* const* d_sigma, void* d_status, cudaStream_t stream);
// selector activations: n bytes (0 / 1) -> selector_words(n) words, bit j of word w = row 32 w + j
__host__ __device__ __forceinline__ size_t selector_words(size_t n) { return (n + 31) / 32; }
int selector_pack_run(DeviceCtx& ctx, const void* d_activations, size_t n, void* d_bits, cudaStream_t stream);
// d_flags (S x S u32, zeroed here): flags[i S + j] = 1 for j < i when bitsets i and j (S consecutive ones in d_bits) share a row
int selector_exclusion_run(DeviceCtx& ctx, const void* d_bits, uint32_t n_selectors, size_t n, void* d_flags, cudaStream_t stream);
// one combination column: d_members holds n_members (bitset slot in d_bits, root) u32 pairs; two members on one row raise d_status
int combination_column_run(DeviceCtx& ctx, const void* d_bits, const void* d_members, uint32_t n_members, uint32_t combination, uint32_t k, void* d_out,
                           void* d_status, cudaStream_t stream);
// l0, l_last, l_active_row (d_cols[0..3), 2^extended_k elements each) of keygen_pk
int keygen_indicators_run(DeviceCtx& ctx, uint32_t k, uint32_t extended_k, uint32_t blinding_factors, const uint64_t omega_inv[4],
                          const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], void* const* d_cols,
                          cudaStream_t stream);
// ---- multiopen.cu ----
// construct_intermediate_sets of a list of queries over n_polys polynomials: slots are the polynomials in first-appearance order,
// pairs the distinct (slot, point) queries grouped by slot, T the distinct points in first-appearance order; a set holds the slots
// of one point set (points in its first slot's order).  Only index and byte comparisons: no field arithmetic on the host.
static const uint32_t SHPLONK_MAX_POINTS = 16;
struct ShplonkPlan {
    std::vector<uint32_t> used;                   // caller's polynomial index of each slot
    std::vector<const void*> d_polys;             // device coefficients of each slot (filled by the caller of the plan)
    std::vector<uint64_t> points;                 // T, 4 Montgomery words per point
    std::vector<uint32_t> pair_point;             // T index of each pair
    std::vector<uint32_t> slot_first, slot_count; // the pairs of each slot
    std::vector<uint32_t> query_pair;             // pair of each query
    std::vector<uint32_t> slot_set, slot_member;  // set of each slot and its place j in the set
    std::vector<std::vector<uint32_t>> set_slots, set_points;
    uint32_t n_points() const { return (uint32_t)(points.size() / 4); }
};
// need_every_poly: a polynomial that no query names is refused
int shplonk_plan_build(const char* who, const h2b_opening_query* queries, uint32_t n_queries, uint32_t n_polys, bool need_every_poly, ShplonkPlan* out);
size_t shplonk_tables_bytes(const ShplonkPlan& p);
size_t shplonk_scalars_count(const ShplonkPlan& p);
int shplonk_tables_upload(const ShplonkPlan& p, const void* const* d_polys_by_slot, void* d_tables, cudaStream_t stream);
const void* shplonk_tables_status(const ShplonkPlan& p, const void* d_tables);      // u32, 1 when z_0 = 0
const void* shplonk_tables_jac(const ShplonkPlan& p, const void* d_tables);         // 96 B for an MSM result
int shplonk_eval_pairs_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, void* d_evals, cudaStream_t stream);
int shplonk_eval_queries_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, void* d_pair_evals, void* d_out, cudaStream_t stream);
int shplonk_begin_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, const uint64_t y[4], const uint64_t v[4], void* d_evals,
                      void* d_scal, void* d_hx, void* d_a, void* d_b, cudaStream_t stream);
int shplonk_finish_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, const uint64_t u[4], const void* d_evals, void* d_scal,
                       const void* d_hx, void* d_a, void* d_b, cudaStream_t stream);
// GWC's construct_intermediate_sets: the distinct points in first-appearance order, each with the polynomial of every query there in
// query order (the j-th is weighted by v^j; a query listed twice is there twice).  The refusals of shplonk_plan_build, no point cap.
struct GwcPlan {
    std::vector<uint64_t> points;                    // 4 Montgomery words per point
    std::vector<std::vector<uint32_t>> polys_at;
    uint32_t max_queries = 0;                        // the longest list of polys_at
    uint32_t n_points() const { return (uint32_t)(points.size() / 4); }
};
int gwc_plan_build(const char* who, const h2b_opening_query* queries, uint32_t n_queries, uint32_t n_polys, GwcPlan* out);
// device bytes of one call's work block
size_t gwc_work_bytes(const GwcPlan& p, size_t n);
// every W_i (Jacobian, 12 words each) into the host array out_jac, over rows [0, n - 1) of g; d_polys by the caller's index.  Synchronous.
int gwc_run(DeviceCtx& ctx, const GwcPlan& p, const void* const* d_polys, size_t n, const uint64_t v[4], const MsmBases& g, void* d_work,
            uint64_t* out_jac, cudaStream_t stream);
// ---- mock.cu ----
// the refusals that need the compiler (graph and root contents); the caller has checked pointers, sizes and indices
int mock_verify_check(const h2b_mock_circuit* c);
// h2b_mock_verify on one device after every check: synchronous, the call's device memory given back before it returns
int mock_verify_run(DeviceCtx& ctx, const h2b_mock_circuit* c, h2b_mock_record* records, uint64_t capacity, uint64_t* count);
// ---- testgen.cu ----
int msm_checksum_run(DeviceCtx& ctx, const void* d_scalars, uint64_t seed, uint64_t first, size_t n, void* d_out, cudaStream_t stream);
int gen_scalars_run(DeviceCtx& ctx, uint64_t seed, size_t n, int kind, void* d_out, cudaStream_t stream);
int field_selftest_run(DeviceCtx& ctx, int field, int op, const void* d_a, const void* d_b, size_t n, void* d_out, cudaStream_t stream);
int ec_selftest_run(DeviceCtx& ctx, int op, const void* d_p, const void* d_q, size_t n, void* d_out, cudaStream_t stream);
int imad_bench_run(DeviceCtx& ctx, int kind, int iters, int blocks, int threads, float* ms_out, double* ops_out, cudaStream_t stream);

}  // namespace h2b
