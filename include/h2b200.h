/*
 * h2b200 -- B200-native (sm_100a) replacement for the data-parallel hot path of the Halo2 KZG
 * prover as DCMMC/halo2-scaffold exercises it: BN254 G1 multi-scalar multiplication and the
 * radix-2 NTT over BN254 Fr.  Plain C ABI: pointers and sizes only, no C++ types, no exceptions.
 *
 * What each entry point replaces (the arithmetic lives in un-vendored git dependencies of the
 * reference, marked [UP]; the reference's own call sites are given as file:line under
 * /root/reference):
 *
 *   h2b_msm_bn254_g1   <- [UP] halo2_proofs::arithmetic::best_multiexp::<G1Affine>
 *                         (halo2_proofs/src/arithmetic.rs, PSE tag v2023_02_02 -- Cargo.toml:13 --
 *                          and the Axiom fork `axiom/dev` -- Cargo.toml:16), reached through
 *                         ParamsKZG::commit / commit_lagrange from keygen_vk / keygen_pk
 *                         (src/scaffold.rs:132,135,146,149,284,287,298,301), create_proof
 *                         (src/scaffold.rs:191-199,207-214,322-330,338-346;
 *                          examples/standard_plonk.rs:41-49) and verify_proof
 *                         (src/scaffold.rs:223-230,354-361; examples/standard_plonk.rs:57-64).
 *   h2b_ntt_bn254_fr   <- [UP] halo2_proofs::arithmetic::best_fft::<Fr>, reached through
 *                         EvaluationDomain::{lagrange_to_coeff, coeff_to_extended,
 *                         extended_to_coeff} from keygen_pk (src/scaffold.rs:135,149,287,301) and
 *                         create_proof (same lines as above).
 *
 * Data layouts are exactly halo2curves 0.3.x's in-memory layouts, so Rust slices can be passed
 * by pointer cast (SURVEY.md section 8):
 *   Fr / Fq   : 4 x u64 little-endian limbs, Montgomery form (R = 2^256), fully reduced.
 *   G1Affine  : x | y (8 x u64); the identity is (0, 0).
 *   G1        : x | y | z Jacobian (12 x u64); z == 0 is the identity.
 *
 * Errors: every function returns 0 on success and a negative H2B_ERR_* code otherwise;
 * h2b_last_error() returns a thread-local description.  The upstream Rust functions are
 * infallible (they assert/panic), so the Rust shim turns a non-zero return into a panic.
 * Threading: all entry points may be called concurrently from several host threads; host-pointer
 * calls are synchronous (they return after the result is in caller memory).
 * There is no CPU fallback: without a usable CUDA device h2b_init fails.
 */
#ifndef H2B200_H
#define H2B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define H2B_OK 0
#define H2B_ERR_NOT_INITIALIZED (-1)
#define H2B_ERR_BAD_ARGUMENT (-2)
#define H2B_ERR_CUDA (-3)
#define H2B_ERR_OOM (-4)
#define H2B_ERR_NO_DEVICE (-5)
#define H2B_ERR_BAD_HANDLE (-6)

/* ---- lifecycle ------------------------------------------------------------------------------- */
/* Use CUDA devices 0..n_devices-1 (0 = every visible device).  Idempotent. */
int h2b_init(int n_devices);
/* Use exactly one device, by CUDA ordinal (one-process-per-GPU launches: pass LOCAL_RANK). */
int h2b_init_device(int device);
void h2b_shutdown(void);
int h2b_device_count(void);
const char* h2b_last_error(void);
const char* h2b_version(void);
/* 1 if this binary is the CPU kernel-logic emulator build used by unit tests, 0 for the CUDA build. */
int h2b_is_emulator(void);

/* ---- drop-in entry points (host pointers, synchronous) ------------------------------------------- */
/* best_multiexp(coeffs, bases): out_jac = sum_i scalars[i] * bases[i].  n may be any value >= 0
 * (n == 0 gives the identity).  A pure function of its arguments, like upstream's:
 *  - arrays of fewer than 4096 points, or whose length is not a multiple of 1024 points (verifier MSMs,
 *    odd prefixes), are uploaded for the call and never cached;
 *  - longer arrays -- in a prover only the SRS vectors `g` and `g_lagrange` (SURVEY.md row a7) -- are kept
 *    resident (window tables from the second use on) and found again by CONTENT: a 128-bit digest of
 *    every 64 KiB block is taken at upload time, and a resident copy is used for a call only if every block
 *    of the caller's array still matches (host threads verify while the GPU runs the MSM; a mismatch discards
 *    the result, re-uploads and recomputes).  In-place edits and address reuse can therefore not return stale
 *    results, and the same vector re-loaded at another address (src/scaffold.rs:174) is recognised.
 * With more than one device the resident copy is sharded by point range (device d holds rows
 * [d n/D, (d+1) n/D)), every device runs a complete Pippenger on its slice and the partial sums are
 * added on device 0.  H2B_IMPLICIT_CACHE=0 disables the cache. */
int h2b_msm_bn254_g1(const uint64_t* scalars, const uint64_t* bases, size_t n, uint64_t out_jac[12]);

/* best_fft(a, omega, log_n) for G = Fr: in place, natural order in and out, no scaling;
 * a has 2^log_n elements, log_n <= 28.
 * With D = 2^j > 1 devices and log_n >= 22 (H2B_NTT_MULTI_MIN_LOG; H2B_NTT_MULTI=0 turns it off) the ONE transform is split over
 * the devices as a four-step NTT (SURVEY.md 8e "one NTT across GPUs"): device d uploads the column block [d C/D, (d+1) C/D) of the
 * R x C matrix straight from `a` (D PCIe links in parallel), runs its column transforms and the twiddle step, the devices exchange
 * n/D^2-element blocks by 2-D peer copies over NVLink (the only exchange; no collective), and every device runs its row transforms
 * and writes its part of the result into `a`. */
int h2b_ntt_bn254_fr(uint64_t* a, const uint64_t omega[4], uint32_t log_n);

/* Explicit device residency for an SRS vector (copied; the host array may be freed afterwards).  Registration
 * also precomputes the window tables T_j[i] = 2^(spacing*j) * bases[i] on the device (one-off cost of a few MSMs;
 * memory n_tables x n x 64 B, see h2b_base_set_info) so that later MSMs over the set need no doublings and a
 * single shared bucket set.  ParamsKZG's `g` and `g_lagrange` ([UP] halo2_proofs/src/poly/kzg/commitment.rs) are
 * the two vectors a prover registers.  Implicitly cached arrays (h2b_msm_bn254_g1) get their tables on second use. */
int h2b_register_bases(const uint64_t* bases, size_t n, uint64_t* handle);
/* The same with the rows split over the devices of h2b_init: device d keeps rows [d n/D, (d+1) n/D) and their tables
 * (1/D of the memory and of the registration time; table spacing chosen for n/D points).  MSMs over such a set are split
 * by point range over the devices that hold the rows (SURVEY.md section 8e row 1); with one device it equals
 * h2b_register_bases. */
int h2b_register_bases_sharded(const uint64_t* bases, size_t n, uint64_t* handle);
/* Drops one reference; calls still running on the set finish on it (device memory is released afterwards). */
int h2b_unregister_bases(uint64_t handle);
/* MSM over bases[offset .. offset+n) of a registered set. */
int h2b_msm_bn254_g1_registered(const uint64_t* scalars, uint64_t handle, size_t offset, size_t n, uint64_t out_jac[12]);

/* ---- batched drop-ins: independent columns / polynomials, distributed round-robin over the devices ------------------
 * The advice, lookup and permutation columns a proof phase commits are independent MSMs over the same SRS vector, and
 * its per-polynomial (i)NTTs are independent too (SURVEY.md section 8e): with D devices, D columns are in flight at
 * once, each on a device that holds its own copy of the SRS tables.  Results are identical to `count` single calls. */
int h2b_msm_bn254_g1_batch_registered(const uint64_t* const* scalars, const size_t* lens, size_t count, uint64_t handle,
                                      uint64_t* out_jac /* count x 12 */);
/* Columns that land on the same device and are short enough to be latency bound (<= 2^21 scalars) share ONE
 * decompose / sort / accumulate / reduce sequence (column id in the bucket index; up to 32 columns and 2^23 scalars per
 * group): the examples the reference ships run k = 16..20, where a single MSM is dominated by dependent steps. */
int h2b_ntt_bn254_fr_batch(uint64_t* const* a, size_t count, const uint64_t omega[4], uint32_t log_n);

/* ---- device-resident entry points (device pointers on `device`, caller's CUDA stream) ------------- */
/* Asynchronous with respect to the host: work is enqueued on `stream` (a cudaStream_t; NULL = the
 * legacy default stream).  `device` is an index into the devices given to h2b_init.
 * Stream contract: the *_dev entry points of one device share that device's grow-only scratch buffers (sort lists, NTT work
 * buffer, scan / lookup scratch), so calls on the SAME device must be ordered with respect to each other -- issue them on one
 * stream (what a prover thread does), or order the streams with events.  Different devices are independent.  (The compiled
 * programs of evaluate_h are the exception: they rotate through a small ring guarded by events.) */
int h2b_ntt_bn254_fr_dev(int device, void* d_a, const uint64_t omega[4], uint32_t log_n, void* stream);
/* `count` device-resident polynomials of 2^log_n elements each (d_polys: host array of device pointers), same omega: groups of up
 * to 16 polynomials share every pass launch (polynomial index in blockIdx.y) -- the per-column (i)NTTs of a proof phase. */
int h2b_ntt_bn254_fr_dev_batch(int device, void* const* d_polys, size_t count, const uint64_t omega[4], uint32_t log_n, void* stream);
int h2b_msm_bn254_g1_dev(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_jac /* 96 B */, void* stream);
/* Point-range sharding across processes (one process per GPU, SURVEY.md section 8e): each rank computes a partial
 * result block (224 B: Jacobian x|y|z followed by the XYZZ form) for its slice, the blocks are gathered by the
 * caller (e.g. torch.distributed.all_gather) and folded on one device. */
int h2b_msm_bn254_g1_dev_partial(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_block /* 224 B */, void* stream);
/* same over rows [offset, offset + n) of a registered base set (uses its window tables); d_scalars on `device` */
int h2b_msm_bn254_g1_dev_registered(int device, const void* d_scalars, uint64_t handle, size_t offset, size_t n, void* d_out_block /* 224 B */, void* stream);
/* `count` device-resident columns (d_scalars: host array of device pointers, lens[j] scalars each) over rows [0, lens[j]) of a
 * registered set in one batched kernel sequence; d_out_blocks: count x 224 B.  Asynchronous on `stream`. */
int h2b_msm_bn254_g1_dev_batch_registered(int device, const void* const* d_scalars, const size_t* lens, size_t count, uint64_t handle,
                                          void* d_out_blocks, void* stream);
int h2b_msm_fold_partials(int device, const uint64_t* host_blocks /* count x 28 u64 */, size_t count, uint64_t out_jac[12]);
/* same, blocks and result in device memory, asynchronous on `stream` */
int h2b_msm_fold_partials_dev(int device, const void* d_blocks, size_t count, void* d_out_jac /* 96 B */, void* stream);
/* a[i] *= factors[i % count], 1 <= count <= 4096 (more than 8 factors go through a device table and synchronise the stream once): the 1/n scaling of lagrange_to_coeff / extended_to_coeff (count 1), the
 * (1, zeta, zeta^2) coset pattern of coeff_to_extended (count 3) and EvaluationDomain::divide_by_vanishing_poly, whose
 * t_evaluations repeat with period 2^(extended_k - k) ([UP] halo2_proofs/src/poly/domain.rs). */
int h2b_fr_scale_dev(int device, void* d_a, size_t n, const uint64_t* factors, int count, void* stream);

/* EvaluationDomain's three conversions on a device-resident column ([UP] halo2_proofs/src/poly/domain.rs, SURVEY.md row
 * a6); the domain constants are the caller's (computed once per domain on the host, as EvaluationDomain::new does):
 *   lagrange_to_coeff : best_fft(a, omega_inv, k); a[i] *= ifft_divisor                         (2^k elements, in place)
 *   coeff_to_extended : a[i] *= zeta_powers[i mod 3] for i < 2^k; zero-pad to 2^extended_k; best_fft(a, extended_omega, extended_k)
 *                       (d_a must hold 2^extended_k elements; zeta_powers = 1, zeta, zeta^2)
 *   extended_to_coeff : best_fft(a, extended_omega_inv, extended_k); a[i] *= factors[i mod 3]
 *                       (factors = extended_ifft_divisor * (1, zeta^2, zeta); the caller truncates to n * (j - 1)) */
int h2b_lagrange_to_coeff_dev(int device, void* d_a, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], void* stream);
int h2b_coeff_to_extended_dev(int device, void* d_a, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                              void* stream);
int h2b_extended_to_coeff_dev(int device, void* d_a, uint32_t extended_k, const uint64_t extended_omega_inv[4], const uint64_t factors[12], void* stream);
/* lagrange_to_coeff / coeff_to_extended for `count` columns at once (d_cols: host array of device pointers; every column as in the
 * single-column call): the transform passes and the scalings are launched once per batch of up to 16 columns */
int h2b_lagrange_to_coeff_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4],
                                    void* stream);
int h2b_coeff_to_extended_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4],
                                    const uint64_t zeta_powers[12], void* stream);

/* ONE column through commit_lagrange -> lagrange_to_coeff -> coeff_to_extended with a single upload (SURVEY.md 8f rank 1; [UP]
 * plonk/prover.rs commits every advice / permuted / product column in Lagrange form and then converts it twice): `lagrange` is the
 * host column (2^k x 4 words), handle_g_lagrange a registered copy of ParamsKZG::g_lagrange resident on `device`.  Writes the
 * commitment (Jacobian), and -- each optional, NULL to skip -- the coefficient form (host, 2^k x 4), the extended-coset form to the
 * host (2^extended_k x 4) and/or leaves it on the device (*d_extended, to be released with h2b_dev_free) for h2b_evaluate_*_dev.
 * Synchronous.  Against three host-pointer drop-in calls it saves two uploads and one download of the column. */
int h2b_column_pipeline(int device, const uint64_t* lagrange, uint64_t handle_g_lagrange, uint32_t k, uint32_t extended_k, const uint64_t omega_inv[4],
                        const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], uint64_t out_commitment_jac[12],
                        uint64_t* out_coeff, uint64_t* out_extended, void** d_extended);

/* Grand-product building blocks on a device-resident Fr column (SURVEY.md section 8f rank 3; [UP] halo2_proofs
 * plonk/permutation/prover.rs, plonk/lookup/prover.rs): z(omega^i) is the exclusive running product of
 * numerator[i] / denominator[i], the denominators inverted with ff::BatchInvert.
 *   batch_invert   : a[i] <- 1 / a[i] in place; zeros stay zero
 *   prefix_product : out[0] = 1, out[i] = in[0] * ... * in[i-1]   (n outputs; out may alias in) */
int h2b_fr_batch_invert_dev(int device, void* d_a, size_t n, void* stream);
int h2b_fr_prefix_product_dev(int device, const void* d_in, void* d_out, size_t n, void* stream);
/* [UP] halo2_proofs::arithmetic::eval_polynomial(poly, point) = sum_i poly[i] * point^i  -> one Fr (32 B) at d_out;
 * [UP] halo2_proofs::arithmetic::kate_division(a, b): the n - 1 coefficients of a(X) / (X - b) -> d_q (must not alias d_a) */
int h2b_fr_eval_polynomial_dev(int device, const void* d_coeffs, size_t n, const uint64_t x[4], void* d_out, void* stream);
int h2b_fr_kate_division_dev(int device, const void* d_a, size_t n, const uint64_t b[4], void* d_q, void* stream);

/* out[i] = sum_j coeffs[j] * cols[j][i] (m columns of n elements; out may alias none of them): the y- / v-weighted sums of
 * the multi-open argument ([UP] poly/kzg/multiopen/shplonk/prover.rs) and the theta-compression of lookup expressions
 * ([UP] plonk/lookup/prover.rs compress_expressions) */
int h2b_fr_lincomb_dev(int device, const void* const* d_cols, const uint64_t* coeffs /* m x 4 */, uint32_t m, size_t n, void* d_out, void* stream);
/* out[c * rows + r] = in[r * cols + c] for a rows x cols matrix of Fr elements (out must not alias in): the re-layout step of the
 * four-step NTT that splits one transform over several devices (h2b_ntt_bn254_fr), usable on its own for row / column blocks of
 * device-resident columns.  Whole 32 x 32 tiles are moved by the TMA unit (cp.async.bulk + mbarrier). */
int h2b_fr_transpose_dev(int device, const void* d_in, void* d_out, uint32_t rows, uint32_t cols, void* stream);
/* The grand products themselves, on device-resident Lagrange-basis columns of n = 2^k rows:
 *   [UP] plonk/permutation/prover.rs Argument::commit, one call per set (chunk of cs.degree() - 2 columns; any number, 16 per launch):
 *        z[0] = last_z,  z[i+1] = z[i] * prod_j (v_j[i] + deltaomega * delta^j * omega^i * beta + gamma)
 *                                      / prod_j (v_j[i] + beta * s_j[i] + gamma)
 *        d_values[j] / d_permutations[j]: the j-th column of the set and its permutation column s_j; deltaomega = delta^(index of
 *        the set's first column in the whole argument); last_z = one for the first set, z[n - (blinding_factors + 1)] of the
 *        previous set afterwards.  All n entries of d_z are written; the caller overwrites the blinding rows.
 *   [UP] plonk/lookup/prover.rs Permuted::commit_product:
 *        z[0] = 1,  z[i+1] = z[i] * (a[i] + beta) (s[i] + gamma) / ((a'[i] + beta) (s'[i] + gamma))
 *        a, s: theta-compressed input / table expressions; a', s': their permuted versions. */
int h2b_permutation_product_dev(int device, const void* const* d_values, const void* const* d_permutations, uint32_t n_columns, size_t n,
                                const uint64_t beta[4], const uint64_t gamma[4], const uint64_t delta[4], const uint64_t deltaomega[4], const uint64_t omega[4],
                                const uint64_t last_z[4], void* d_z, void* stream);
int h2b_lookup_product_dev(int device, const void* d_compressed_input, const void* d_compressed_table, const void* d_permuted_input,
                           const void* d_permuted_table, size_t n, const uint64_t beta[4], const uint64_t gamma[4], void* d_z, void* stream);

/* [UP] plonk/lookup/prover.rs permute_expression_pair on the first usable_rows = n - (blinding_factors + 1) rows of the
 * theta-compressed input and table columns (device, Montgomery): permuted_input = the input sorted by canonical value;
 * permuted_table: every first occurrence of a value in permuted_input has that value at the same row, the remaining rows
 * receive the leftover table values exactly as upstream assigns them (ascending leftovers onto the repeated rows taken from
 * the end).  The outputs may alias the inputs; rows from usable_rows on (the blinding rows) are not touched.  The call
 * synchronises the stream: an input value that the table does not hold fails with H2B_ERR_BAD_ARGUMENT, as upstream returns
 * Error::ConstraintSystemFailure. */
int h2b_lookup_permute_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                           void* stream);
/* The same without the synchronisation: the verdict is written to the 32-bit device word d_status on `stream` (0 = every input value
 * is in the table, otherwise 1 + the sorted row of one that is not -- the outputs are then meaningless); the caller reads it when it
 * next synchronises.  Lets several devices permute their lookups concurrently. */
int h2b_lookup_permute_async_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input,
                                 void* d_permuted_table, void* d_status, void* stream);

/* ---- quotient evaluation: evaluate_h on device-resident extended-coset columns (SURVEY.md section 8f rank 2) ----------
 * [UP] halo2_proofs/src/plonk/evaluation.rs.  A GraphEvaluator is passed in the vocabulary upstream builds it in
 * (ValueSource / Calculation / CalculationInfo), flattened into plain arrays; the Rust shim fills these structs from
 * `Evaluator { custom_gates, lookups }` once per proving key.  Every column is a device pointer to `size` Fr elements
 * (the 2^extended_k evaluations over the zeta coset that coeff_to_extended produced). */
enum h2b_value_kind {          /* [UP] evaluation.rs `enum ValueSource`; index / rotation as upstream's tuple fields */
    H2B_VS_CONSTANT = 0,       /* constants[index] */
    H2B_VS_INTERMEDIATE = 1,   /* intermediates[index] */
    H2B_VS_FIXED = 2,          /* fixed[index][rotations[rotation]] */
    H2B_VS_ADVICE = 3,         /* advice[index][rotations[rotation]] */
    H2B_VS_INSTANCE = 4,       /* instance[index][rotations[rotation]] */
    H2B_VS_CHALLENGE = 5,      /* challenges[index] */
    H2B_VS_BETA = 6, H2B_VS_GAMMA = 7, H2B_VS_THETA = 8, H2B_VS_Y = 9,
    H2B_VS_PREVIOUS_VALUE = 10
};
enum h2b_calc_op {             /* [UP] evaluation.rs `enum Calculation` */
    H2B_CALC_ADD = 0, H2B_CALC_SUB = 1, H2B_CALC_MUL = 2, H2B_CALC_SQUARE = 3, H2B_CALC_DOUBLE = 4, H2B_CALC_NEGATE = 5,
    H2B_CALC_HORNER = 6,       /* value = a; for part in parts: value = value * b + part */
    H2B_CALC_STORE = 7
};
typedef struct h2b_value_source { uint32_t kind, index, rotation; } h2b_value_source;
typedef struct h2b_calculation {
    uint32_t op, target;                 /* intermediates[target] = op(...) */
    h2b_value_source a, b;               /* Horner: a = start value, b = factor */
    uint32_t parts_offset, parts_len;    /* Horner only: parts[parts_offset .. parts_offset + parts_len) */
} h2b_calculation;
typedef struct h2b_graph {               /* [UP] evaluation.rs `struct GraphEvaluator` */
    const uint64_t* constants; uint32_t n_constants;     /* n x 4, Montgomery */
    const int32_t* rotations; uint32_t n_rotations;
    const h2b_calculation* calculations; uint32_t n_calculations;
    const h2b_value_source* parts; uint32_t n_parts;
    uint32_t n_intermediates;
} h2b_graph;
typedef struct h2b_eval_columns {        /* host arrays of device pointers + the per-proof scalars of evaluate_h */
    const void* const* fixed; uint32_t n_fixed;
    const void* const* advice; uint32_t n_advice;
    const void* const* instance; uint32_t n_instance;
    const uint64_t* challenges; uint32_t n_challenges;    /* n x 4 */
    const uint64_t* beta; const uint64_t* gamma; const uint64_t* theta; const uint64_t* y;   /* 4 words each */
} h2b_eval_columns;
/* values[idx] = graph.evaluate(.., previous_value = values[idx], idx, rot_scale, isize = size) for every idx < size: the
 * "Custom gates" loop of evaluate_h.  The same call on Lagrange-basis columns (size = 2^k, rot_scale = 1) is the lookup argument's
 * compress_expressions ([UP] plonk/lookup/prover.rs).  A graph without calculations writes zero, as upstream does.  The rotated row is
 * get_rotation_idx(idx, rot, rot_scale, isize) = (idx + rot * rot_scale).rem_euclid(isize). */
int h2b_evaluate_graph_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                           void* stream);
/* The "Permutations" loop of evaluate_h: values[idx] is advanced by the l_0 / l_last / set-chaining / product terms.
 *   d_product_cosets[n_sets]   : permutation_product_coset of every set (z_i)
 *   d_columns[n_columns]       : the value coset of every column of the argument, in p.columns order (the caller resolves
 *                                Any::{Advice, Fixed, Instance} to a pointer); d_perm_cosets[n_columns] = pk.permutation.cosets
 *   chunk_len = cs.degree() - 2; last_rotation = -(blinding_factors + 1); delta = Fr::DELTA; zeta = Fr::ZETA */
int h2b_evaluate_h_permutation_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                   const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                   int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                   const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                   const uint64_t extended_omega[4], void* stream);
/* One iteration of the "Lookups" loop of evaluate_h: table_value = graph.evaluate(.., previous_value = 0, ..) and the five
 * lookup terms on product_coset (z), permuted_input_coset (a') and permuted_table_coset (s'). */
int h2b_evaluate_h_lookup_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                              const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                              const void* d_l_last, const void* d_l_active_row, void* stream);
/* Row-sharded variants (evaluate_h across devices): this call produces rows [row0, row0 + rows) of the domain.  Every column pointer
 * (fixed / advice / instance, product / permuted / sigma cosets, l_0, l_last, l_active) is then a SLICE of rows + 2 * halo rows that
 * starts at global row (row0 - halo) mod size -- wrap-around included -- and d_values is the halo-free slice of `rows` rows.  halo must
 * cover the largest rotated read: max |rotation| * rot_scale of the graph, rot_scale for lookups, max(1, |last_rotation|) * rot_scale
 * for the permutation argument; otherwise the call is refused.  Row values do not depend on the sharding. */
typedef struct h2b_eval_shard { uint32_t row0, rows, halo; } h2b_eval_shard;
int h2b_evaluate_graph_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                 const h2b_eval_shard* shard, void* stream);
int h2b_evaluate_h_permutation_shard_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                         const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                         int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                         const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                         const uint64_t extended_omega[4], const h2b_eval_shard* shard, void* stream);
int h2b_evaluate_h_lookup_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                    const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                                    const void* d_l_last, const void* d_l_active_row, const h2b_eval_shard* shard, void* stream);
/* slots (live values per row) and micro-operations the last compiled graph of this thread needed -- diagnostics / tests */
int h2b_evaluate_graph_info(uint32_t* slots, uint32_t* micro_ops);

/* ---- SRS on-disk format (SURVEY.md section 8f rank 4) ------------------------------------------------------------------
 * [UP] halo2_proofs/src/poly/kzg/commitment.rs ParamsKZG::{read_custom, write_custom} / halo2_proofs::SerdeFormat and
 * [UP] halo2curves 0.3.x GroupEncoding / SerdeObject for G1Affine; the reference loads params/kzg_bn254_{k}.srs at
 * src/scaffold.rs:119,174,271.  File: k (u32 LE) | g[2^k] | g_lagrange[2^k] | g2 | s_g2. */
enum h2b_serde_format {
    H2B_SERDE_PROCESSED = 0,            /* compressed: 32 B = canonical LE x, (y & 1) << 7 in byte 31, all-zero = identity */
    H2B_SERDE_RAW_BYTES = 1,            /* x | y Montgomery limbs (64 B), range- and curve-checked */
    H2B_SERDE_RAW_BYTES_UNCHECKED = 2   /* the same bytes, unchecked */
};
/* n encoded points (device) -> n affine points x | y Montgomery (device; may alias the input for the raw formats).
 * With first_invalid != NULL the call synchronises the stream, stores the index of the first invalid encoding (or
 * UINT64_MAX) and fails with H2B_ERR_BAD_ARGUMENT if there is one (upstream unwraps / returns io::Error); with NULL it
 * stays asynchronous and invalid points decode to the identity. */
int h2b_g1_decode_dev(int device, const void* d_bytes, size_t n, int format, void* d_out_affine, uint64_t* first_invalid, void* stream);
/* n affine points (device) -> n x 32 compressed bytes (device): G1Affine::to_bytes */
int h2b_g1_encode_dev(int device, const void* d_affine, size_t n, void* d_out_bytes, void* stream);
/* ParamsKZG::read_custom: reads the file, decodes g and g_lagrange on the device and leaves both resident as registered
 * base sets (window tables built, every device of h2b_init) -> *handle_g, *handle_g_lagrange for
 * h2b_msm_bn254_g1_registered (commit / commit_lagrange).  out_g / out_g_lagrange (2^k x 8 words each, may be NULL) receive
 * the decoded points for the host-side ParamsKZG; the G2 section (g2 | s_g2, 2 x 64 B compressed or 2 x 128 B raw) is
 * returned as bytes for the host to parse.  Either handle pointer may be NULL (that vector is then only decoded). */
int h2b_srs_read(const char* path, int format, uint32_t* k, uint64_t* out_g, uint64_t* out_g_lagrange, uint8_t* g2_bytes, size_t g2_cap,
                 size_t* g2_len, uint64_t* handle_g, uint64_t* handle_g_lagrange);
/* A file that was read before and has not changed since (same path, format, size and mtime) is NOT decoded again: the call
 * hands out the resident base sets (reference counted -- every handle still has to be given back with
 * h2b_unregister_bases) and, if asked, downloads the points.  The reference re-reads the SRS file for every proof
 * (src/scaffold.rs:174).  H2B_SRS_CACHE=0 in the environment disables this; h2b_srs_cache_clear drops the cache's references. */
int h2b_srs_cache_clear(void);
/* ParamsKZG::write_custom for host arrays (Processed: compressed on the device) */
int h2b_srs_write(const char* path, int format, uint32_t k, const uint64_t* g, const uint64_t* g_lagrange, const uint8_t* g2_bytes, size_t g2_len);

/* ParamsKZG::setup ([UP] halo2_proofs/src/poly/kzg/commitment.rs) with the caller's toxic waste s (Montgomery, < r):
 * g[i] = [s^i] G, g_lagrange[i] = [L_i(s)] G for i < 2^k, k <= 28, G = (1, 2), computed on device 0 by fixed-base
 * multiplication (w = ROOT_OF_UNITY^(2^(28 - k)) is derived on the device).  Output convention of h2b_srs_read:
 * out_g / out_g_lagrange (2^k x 8 words, may be NULL) receive the points; handle_g / handle_g_lagrange (may be NULL)
 * receive registered, replicated base sets with window tables.  Synchronous.  k > 28, s >= r and s^(2^k) = 1 (s a power
 * of w, s = 1 included: a denominator s - w^i vanishes) fail with H2B_ERR_BAD_ARGUMENT before anything is allocated;
 * s = 0 is legal (g = [G, O, O, ...], g_lagrange[i] = [1/n] G). */
int h2b_srs_setup(uint32_t k, const uint64_t s[4], uint64_t* out_g, uint64_t* out_g_lagrange, uint64_t* handle_g, uint64_t* handle_g_lagrange);
/* out[i] = [scalars[i]] G (G = (1, 2)); scalars n x 4 words Montgomery (< r), out n x 8 words affine, identity (0, 0);
 * asynchronous on `stream`.  The first call on a device builds its fixed-base table (32 MiB, kept until h2b_shutdown, as are
 * h2b_srs_setup's and h2b_gen_points_dev's); being asynchronous, this call also keeps its scratch (64 B per point up to 2^24
 * points, plus the batch-inversion scratch) reserved until h2b_shutdown, as the other device-pointer entry points do. */
int h2b_g1_generator_mul_dev(int device, const void* d_scalars, size_t n, void* d_out_affine, void* stream);
/* g_to_lagrange ([UP] halo2_proofs/src/arithmetic.rs) of the first 2^k affine points at d_g_affine (n x 8 words, identity
 * (0, 0) allowed anywhere): d_out[i] = n^-1 sum_j w^(-ij) g[j], w = ROOT_OF_UNITY^(2^(28 - k)) the root of the Fr NTT of the
 * same k, batch-normalised affine, bit-identical to upstream's.  d_out may equal d_g.  Asynchronous on `stream`; its
 * scratch (about 200 B per point) stays reserved until h2b_shutdown, as h2b_g1_generator_mul_dev's does.  k > 28 and null
 * pointers fail with H2B_ERR_BAD_ARGUMENT. */
int h2b_g1_to_lagrange_dev(int device, const void* d_g_affine, uint32_t k, void* d_out_affine, void* stream);
/* ParamsKZG::downsize(k) ([UP] halo2_proofs/src/poly/kzg/commitment.rs) of the resident g of a REPLICATED registered set
 * (h2b_srs_read, h2b_srs_setup, h2b_register_bases): handle_g_out (may be NULL) receives a new registered set holding the
 * 2^k-point prefix of g (a device-to-device copy, window tables sized for 2^k), handle_g_lagrange_out (may be NULL) a new
 * registered set of g_to_lagrange of that prefix, and out_g_lagrange (2^k x 8 words, may be NULL) its host copy.  The caller
 * truncates its own host g and drops the old handles when it wants to.  Synchronous; gives its scratch back before it returns.
 * k > 28, 2^k above the set's n, an unknown handle and a sharded set fail with H2B_ERR_BAD_ARGUMENT before anything is
 * allocated, and leave the output handles untouched. */
int h2b_srs_downsize(uint64_t handle_g, uint32_t k, uint64_t* out_g_lagrange, uint64_t* handle_g_out, uint64_t* handle_g_lagrange_out);

/* ---- key generation: the permutation argument's sigma columns and keygen_pk's indicator columns -------------------------
 * [UP] halo2_proofs/src/plonk/permutation/keygen.rs (Assembly::build_vk / build_pk) and plonk/keygen.rs (keygen_pk).  A mapping
 * column is upstream's Vec<(usize, usize)> as it sits in memory: n = 2^k pairs of u64 (column, row).  sigma_i[j] = delta^c * omega^r
 * for (c, r) = mapping[i][j], Montgomery form, canonical; delta is Fr::DELTA and omega the domain's root, both from the caller. */
/* sigma of n_columns mapping columns (d_mapping[i]: n x 16 B on `device`) into d_sigma[i] (n x 32 B), for every column in one launch
 * sequence.  An entry with c >= n_columns or r >= n is refused as upstream's out-of-range index panics: the 32-bit word at d_status
 * receives 1 + the flat index i * n + j of the last such entry (saturated at 2^32 - 1), 0 when every entry is valid; sigma is
 * unspecified when it is non-zero (the convention of h2b_lookup_permute_async_dev).  Asynchronous on `stream`; the twiddle tables
 * (2^ceil(k/2) + n_columns * 2^floor(k/2) entries of 32 B) stay reserved until h2b_shutdown.  k > 28, n_columns = 0 and null pointers
 * fail with H2B_ERR_BAD_ARGUMENT before anything is launched. */
int h2b_permutation_sigma_dev(int device, const void* const* d_mapping, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4],
                              void* const* d_sigma, void* d_status, void* stream);
/* keygen_pk's l0 = ext(coeff(e_0)), l_last = ext(coeff(e_(n-bf-1))) and l_active_row = 1 - (l_last + l_blind) = ext(coeff(1 on rows
 * 0 .. n-bf-2)), each 2^extended_k x 32 B on `device`, with ext / coeff the EvaluationDomain conversions of
 * h2b_lagrange_to_coeff_dev_batch / h2b_coeff_to_extended_dev_batch (same constants).  Nothing is uploaded.  Asynchronous on `stream`.
 * bf + 1 >= n, extended_k < k, extended_k > 28 and null pointers fail with H2B_ERR_BAD_ARGUMENT. */
int h2b_keygen_lagrange_indicators_dev(int device, uint32_t k, uint32_t extended_k, uint32_t blinding_factors, const uint64_t omega_inv[4],
                                       const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], void* d_l0,
                                       void* d_l_last, void* d_l_active_row, void* stream);
/* Assembly::build_vk: out_commitments[12 i ..] = commit_lagrange(sigma_i) (Jacobian) over the registered set handle_g_lagrange (the
 * handles h2b_msm_bn254_g1_batch_registered accepts: replicated or sharded, at least n points).  mapping[i]: the caller's n x 2 u64
 * column (pageable is fine); columns go round-robin over the devices, and each is staged through pinned buffers while the previous
 * one's sigma kernel runs.  Synchronous; gives its scratch back before it returns.  k > 28, n_columns = 0, null pointers, an unknown
 * handle, a set shorter than n and an invalid mapping entry fail with H2B_ERR_BAD_ARGUMENT and leave out_commitments untouched. */
int h2b_permutation_build_vk(const uint64_t* const* mapping, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4],
                             uint64_t handle_g_lagrange, uint64_t* out_commitments);
/* Assembly::build_pk: per column i, out_permutations[i] = sigma_i (n x 32 B), out_polys[i] = lagrange_to_coeff(sigma_i) (n x 32 B) and
 * out_cosets[i] = coeff_to_extended(out_polys[i]) (2^extended_k x 32 B); any of the three arrays may be NULL.  The domain constants
 * are those of h2b_lagrange_to_coeff_dev_batch / h2b_coeff_to_extended_dev_batch.  Columns are dealt as in h2b_permutation_build_vk
 * and processed a bounded number (at most 2 GiB of device memory per device) at a time.  Every entry is checked before any caller
 * memory is written: bad arguments and invalid entries fail with H2B_ERR_BAD_ARGUMENT and leave every output untouched.  Synchronous;
 * gives its scratch back before it returns. */
int h2b_permutation_build_pk(const uint64_t* const* mapping, uint32_t n_columns, uint32_t k, uint32_t extended_k, const uint64_t delta[4],
                             const uint64_t omega[4], const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4],
                             const uint64_t zeta_powers[12], uint64_t* const* out_permutations, uint64_t* const* out_polys, uint64_t* const* out_cosets);

/* ---- key generation: compress_selectors and the fixed columns of keygen_vk / keygen_pk -------------------------------------------
 * [UP] halo2_proofs/src/plonk/circuit/compress_selectors.rs (process) and plonk/keygen.rs.  A selector's activations are upstream's
 * Vec<bool> as it sits in memory: n = 2^k bytes, a non-zero byte is an active row.  An assignment gives each selector s a combination
 * combination_of[s] < n_combinations and a root root_of[s] > 0; combination column c holds F::from(root_of[s]) (Montgomery form) on
 * the rows where its member s is active and zero on every other row -- what process fills -- so no two members of a combination may
 * be active on one row.  n_selectors is at most 2^14. */
/* out (n_selectors x n_selectors bytes, row-major): out[i][j] = 1 when selectors i and j are both active on some row, else 0; symmetric,
 * zero diagonal -- process's exclusion matrix.  activations[s] may be pageable.  Synchronous.  k > 28, more than 2^14 selectors and
 * null pointers fail with H2B_ERR_BAD_ARGUMENT before anything is written; n_selectors = 0 writes nothing. */
int h2b_selector_exclusion(const uint8_t* const* activations, uint32_t n_selectors, uint32_t k, uint8_t* out);
/* keygen_vk's fixed commitments: out_commitments[12 i ..] = commit_lagrange(column i) (Jacobian) over the registered set
 * handle_g_lagrange (replicated or sharded, at least n points), for the n_fixed caller columns fixed[i] (n x 32 B Montgomery, pageable
 * is fine) and then the n_combinations combination columns -- upstream's order, fixed.extend(selector_polys).  n_fixed = 0 or
 * n_selectors = 0 are fine, both n_fixed = n_combinations = 0 is not.  Columns go round-robin over the devices as in
 * h2b_permutation_build_vk; each device uploads and packs the selectors of its combinations once.  Synchronous.  k > 28, null
 * pointers, a combination index >= n_combinations, a root of 0, a combination no selector uses, an unknown handle, a set shorter than n
 * and two members of one combination active on one row fail with H2B_ERR_BAD_ARGUMENT and leave out_commitments untouched. */
int h2b_keygen_fixed_build_vk(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                              const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint32_t k, uint64_t handle_g_lagrange,
                              uint64_t* out_commitments);
/* keygen_pk's fixed columns: out_combination_values[c] = combination column c (n x 32 B; the caller holds its fixed columns), and for
 * all n_fixed + n_combinations columns i in the order of h2b_keygen_fixed_build_vk out_polys[i] = lagrange_to_coeff(column i) (n x 32 B)
 * and out_cosets[i] = coeff_to_extended(out_polys[i]) (2^extended_k x 32 B), with the constants of h2b_lagrange_to_coeff_dev_batch /
 * h2b_coeff_to_extended_dev_batch.  Any of the three arrays may be NULL.  Refuses what h2b_keygen_fixed_build_vk refuses, and
 * extended_k < k or > 28; every combination column is built and checked before any caller memory is written, so a refused call leaves
 * every output untouched.  Synchronous. */
int h2b_keygen_fixed_build_pk(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                              const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint32_t k, uint32_t extended_k,
                              const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                              uint64_t* const* out_combination_values, uint64_t* const* out_polys, uint64_t* const* out_cosets);

/* ---- the proving key resident on the devices ----------------------------------------------------------------------------------------
 * [UP] halo2_proofs/src/plonk.rs ProvingKey: fixed_values / fixed_polys / fixed_cosets, permutation.{permutations, polys, cosets} and
 * l0 / l_last / l_active_row, held on the devices of h2b_init from keygen to the last proof, so that create_proof's device steps read
 * them instead of uploading them again for every proof.  A pk is a reference-counted object behind a handle, like a registered base set:
 * a call holds it while it runs, h2b_pk_release drops the handle's reference, and device memory goes when the last holder lets go.
 *   parts : FIXED       n_fixed columns -- the caller's fixed columns, then the combination columns (upstream's fixed.extend(selector_polys))
 *           PERMUTATION n_permutation sigma columns
 *           INDICATORS  l0, l_last, l_active_row (in that order)
 *   forms : VALUES (Lagrange, 2^k rows), COEFF (2^k), EXTENDED (2^extended_k); FIXED and PERMUTATION hold all three, INDICATORS EXTENDED only
 *   layout: REPLICATED  every device holds every form of every column
 *           ROW_SHARDED every device holds the 2^k-row forms; of every EXTENDED column, device d of D holds its rows
 *                       [floor(d E / D), floor((d + 1) E / D)) plus `halo` rows on each side, wrap-around included, starting at global row
 *                       (row0 - halo) mod E (E = 2^extended_k): the slice h2b_evaluate_*_shard_dev takes, halo its largest rotated read. */
enum h2b_pk_part { H2B_PK_FIXED = 0, H2B_PK_PERMUTATION = 1, H2B_PK_INDICATORS = 2 };
enum h2b_pk_form { H2B_PK_VALUES = 0, H2B_PK_COEFF = 1, H2B_PK_EXTENDED = 2 };
enum h2b_pk_layout { H2B_PK_REPLICATED = 0, H2B_PK_ROW_SHARDED = 1 };
/* An empty pk with every byte of its storage reserved on every device now (H2B_ERR_OOM if it does not fit, before any key generation).
 * The domain constants (those of h2b_lagrange_to_coeff_dev_batch / h2b_coeff_to_extended_dev_batch, plus omega) are stored with it and
 * used by every later build.  k > 28, extended_k < k or > 28, an unknown layout, a null pointer and, in the sharded layout,
 * rows + 2 halo > 2^extended_k for some device fail with H2B_ERR_BAD_ARGUMENT.  halo is ignored in the replicated layout. */
int h2b_pk_create(uint32_t k, uint32_t extended_k, uint32_t n_fixed, uint32_t n_permutation, int layout, uint32_t halo, const uint64_t omega[4],
                  const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                  uint64_t* handle);
/* h2b_keygen_fixed_build_pk with the pk as its destination: the n_fixed + n_combinations columns go to FIXED columns first_column ..,
 * all three forms.  Refuses what h2b_keygen_fixed_build_pk refuses (k and the constants are the pk's), an unknown handle and columns past
 * the pk's n_fixed; every combination column is checked before anything is stored, so a refused call leaves the pk as it was.  Nothing
 * passes through the host: forms are copied off the group buffers on the device and placed on the other devices by peer copies.
 * Synchronous. */
int h2b_keygen_fixed_build_pk_resident(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                                       const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint64_t pk, uint32_t first_column);
/* h2b_permutation_build_pk into the pk's PERMUTATION part (n_columns must equal its n_permutation); every mapping entry is checked first. */
int h2b_permutation_build_pk_resident(const uint64_t* const* mapping, uint32_t n_columns, const uint64_t delta[4], uint64_t pk);
/* h2b_keygen_lagrange_indicators_dev into the pk's INDICATORS (computed on device 0, placed on the others).  bf + 1 >= 2^k fails. */
int h2b_keygen_lagrange_indicators_resident(uint64_t pk, uint32_t blinding_factors);
/* Registers a proving key built elsewhere (the CPU keygen, ProvingKey::read): values[j] (2^k x 32 B Lagrange form, pageable is fine)
 * becomes column first + j of `part` (FIXED or PERMUTATION), and COEFF / EXTENDED are derived on the device by the conversions keygen
 * uses -- the pk then equals what the device keygen stores.  INDICATORS are built with h2b_keygen_lagrange_indicators_resident. */
int h2b_pk_put_lagrange(uint64_t pk, int part, uint32_t first, uint32_t count, const uint64_t* const* values);
/* *d_ptr = the column on `device` (an index into the devices of h2b_init), valid while the handle is held.  shard (may be NULL) receives
 * {row0, rows, halo} of the slice: of a sharded EXTENDED column, this device's; of any other column {0, its length, 0}.  A column never
 * filled, a form the part does not hold, an index out of range, a device outside h2b_init and an unknown handle fail with
 * H2B_ERR_BAD_ARGUMENT. */
int h2b_pk_column(uint64_t pk, int device, int part, int form, uint32_t index, void** d_ptr, h2b_eval_shard* shard);
/* a host copy of one column (2^k or 2^extended_k x 32 B) -- a sharded EXTENDED column is assembled from the devices' slices */
int h2b_pk_download(uint64_t pk, int part, int form, uint32_t index, uint64_t* host_out);
/* per_device_bytes[d] (h2b_device_count() entries, may be NULL): the storage the pk holds on device d */
int h2b_pk_info(uint64_t pk, uint64_t* per_device_bytes);
/* drops the handle; freeing waits for the work queued on the pk's devices.  An unknown or already released handle fails. */
int h2b_pk_release(uint64_t pk);

/* ---- the multi-point opening: [UP] halo2_proofs/src/poly/kzg/multiopen/shplonk/prover.rs ProverSHPLONK::create_proof ----------
 * A query opens polynomial `poly` (an index into the caller's list; polynomials are identified by index, as upstream identifies them
 * by pointer) at `point` (Montgomery form).  Every polynomial has n coefficients.  Refused with H2B_ERR_BAD_ARGUMENT, every output
 * untouched: no queries, a poly index >= n_polys, a polynomial that no query opens, a point >= r, more than 16 distinct points for one
 * polynomial, n < 2 or n > 2^28. */
typedef struct h2b_opening_query { uint32_t poly; uint32_t reserved; uint64_t point[4]; } h2b_opening_query;
/* eval_polynomial(poly, point) of every query -> d_out (one Fr per query, in query order).  d_polys: n_polys device pointers.
 * Each coefficient is read from device memory once per polynomial however many points open it.  Asynchronous on `stream`; its
 * tables and scratch stay reserved on the device until h2b_shutdown. */
int h2b_fr_eval_queries_dev(int device, const void* const* d_polys, uint32_t n_polys, size_t n, const h2b_opening_query* queries, uint32_t n_queries,
                            void* d_out, void* stream);
/* Steps 1-6 of create_proof: construct_intermediate_sets, the evaluations, interpolants, numerators, quotients and h_x, and
 * h1 = commit(h_x) over the registered set handle_g (Jacobian, out_h1_jac) -- for the y and v the caller squeezed.  With
 * polys_on_host, polys[i] are host arrays (pageable is fine), uploaded once into the session; otherwise they are device pointers on
 * `device`, borrowed: they must stay unchanged until h2b_shplonk_finish returns.  Synchronous.  Besides the refusals above, a
 * challenge >= r, an unknown handle_g and one that does not hold rows [0, n) on `device` are refused.  The session is a
 * reference-counted handle like a proving key.  The scratch of the evaluations (about n / 15 Fr per (polynomial, point) pair) is
 * shared with h2b_fr_eval_queries_dev and stays reserved on the device until h2b_shutdown, so that later openings allocate nothing
 * but their session. */
int h2b_shplonk_begin(int device, const void* const* polys, int polys_on_host, uint32_t n_polys, size_t n, const h2b_opening_query* queries,
                      uint32_t n_queries, uint64_t handle_g, const uint64_t y[4], const uint64_t v[4], uint64_t out_h1_jac[12], uint64_t* session);
/* Step 7 for the u the caller squeezed after writing h1: h2 = commit(kate_division(L, u) / z_0) (Jacobian, out_h2_jac).  Synchronous.
 * u >= r and u in T \ S_0 (z_0 = 0, where upstream panics in invert().unwrap()) are refused, output untouched, and the session can
 * be finished with another u; after a successful finish every further call on the session is refused. */
int h2b_shplonk_finish(uint64_t session, const uint64_t u[4], uint64_t out_h2_jac[12]);
/* drops the handle; device memory goes when the last call holding the session returns.  An unknown or released handle fails. */
int h2b_shplonk_release(uint64_t session);

/* ---- raw device memory helpers (so that non-CUDA hosts -- ctypes, Rust -- can hold device buffers) --- */
int h2b_dev_alloc(int device, size_t bytes, void** out);
int h2b_dev_free(int device, void* p);
int h2b_memcpy_h2d(int device, void* d_dst, const void* h_src, size_t bytes);
int h2b_memcpy_d2h(int device, void* h_dst, const void* d_src, size_t bytes);
/* Upload a fresh column while the device keeps working: nothing in flight may touch d_dst; work queued on `stream` after the
 * call sees the data.  Pageable sources are consumed before the call returns (pinned staging threads), pinned sources must
 * stay valid until the stream reaches the copy. */
int h2b_memcpy_h2d_async(int device, void* d_dst, const void* h_src, size_t bytes, void* stream);
/* column copies / zero padding on the caller's stream (the padding of coeff_to_extended, copies that keep the Lagrange form) */
int h2b_memcpy_d2d_async(int device, void* d_dst, const void* d_src, size_t bytes, void* stream);
int h2b_memset_zero_async(int device, void* d_dst, size_t bytes, void* stream);
int h2b_dev_sync(int device);

/* ---- synthetic workload + diagnostics ---------------------------------------------------------------- */
/* P_i = [z_i] G with z_i the i-th SplitMix64 value of stream `seed` (valid, distinct G1 points). */
int h2b_gen_points_dev(int device, uint64_t seed, size_t n, void* d_out_affine, void* stream);
/* kind 0: uniform in [0, r);  kind 1: witness-like (50% 0, 20% 1, 20% < 2^19, 10% r - small). */
int h2b_gen_scalars_dev(int device, uint64_t seed, size_t n, int kind, void* d_out, void* stream);
/* O(n) checksum of an MSM over the synthetic points: for P_i = [z_i] G (h2b_gen_points_dev, stream `seed`, indices first + i),
 * sum_i s_i P_i = [sum_i s_i z_i mod r] G.  Writes the CANONICAL (non-Montgomery) value of sum_i s_i z_i mod r as 32 bytes at d_out;
 * field arithmetic only, so it shares no code with the MSM it checks (bench.py `verified`). */
int h2b_msm_checksum_dev(int device, const void* d_scalars /* n x 32 B Montgomery */, uint64_t seed, uint64_t first, size_t n, void* d_out, void* stream);
/* element-wise field op on host arrays.  field: 0 Fr, 1 Fq.  op: 0 add, 1 sub, 2 mul, 3 sqr(a), 4 inv(a),
 * 5 from_mont(a), 6 to_mont(a); the lazily reduced operations of the MSM and NTT loops (operands in [0, 2p)):
 * 7 mul, 8 sqr(a), 9 add, 10 sub (results in [0, 2p)), 11 canonical form of a, 12 a == 0 mod p (1 or 0 in limb 0) */
int h2b_field_op(int field, int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out);
/* element-wise group op on host arrays of affine points; op: 0 p+q, 1 p-q, 2 4(p+q) via the general
 * XYZZ adder and doubling, 3 p+q through the Jacobian conversion, 4 p+q by the lazily reduced mixed addition
 * on a non-canonical accumulator, 5 [e] p by the variable-base multiplication of h2b_g1_to_lagrange_dev with e the
 * first 4 words of q (Fr, Montgomery).  out: affine. */
int h2b_ec_op(int op, const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out);
/* integer-pipe micro-benchmark; kind 0 IMAD, 1 IMAD.WIDE, 2 dependent Fq multiplications, 3 dependent
 * XYZZ mixed additions (the lazily reduced one of the MSM accumulation), 4 dependent Fq squarings, 5 dependent a*b + c*d with one reduction.  Returns elapsed milliseconds and the number of operations executed. */
int h2b_imad_bench(int device, int kind, int iters, float* ms_out, double* ops_out);
/* number of CUDA kernels this library has launched since it was loaded */
unsigned long long h2b_launch_count(void);
/* per-kernel timing with CUDA events recorded on the launching stream. After h2b_profile_enable(device, 1) every
 * MSM / NTT call records one event per phase; h2b_profile_read synchronises the device and returns (tag, ms) pairs
 * in launch order.  MSM tags: 1 decompose, 2 scan, 3 scatter, 4 plan, 5 accumulate, 6 combine, 7 bucket reduction,
 * 8 final;  NTT tags: 15 twiddle tables, 16 + p = pass p;  h2b_srs_setup tags (per vector and chunk of 2^24 points):
 * 24 scalars (powers, inversion, scaling), 25 fixed-base multiplication, 26 normalisation, 27 generator table (first use
 * on the device only); registering the results records 9 (window tables) as every registered base set does;
 * h2b_g1_to_lagrange_dev / h2b_srs_downsize tags: 28 twiddles (w^-1, n^-1 and the power table), 29 butterfly stages (all
 * k of them), 30 normalisation (batch inversion and the affine finish);  h2b_permutation_build_vk / h2b_permutation_build_pk tags
 * (per column or group of columns): 31 mapping upload, 32 sigma kernel (the first also builds the twiddle tables), 33 commitments,
 * 34 inverse NTTs (lagrange_to_coeff), 35 coset NTTs (coeff_to_extended), 36 downloads; the MSM / NTT tags recorded inside a phase
 * belong to the keygen tag that follows them;  h2b_selector_exclusion and h2b_keygen_fixed_build_vk / _pk add 37 selector uploads
 * and packing (all selectors of the call or device at once), 38 exclusion kernel, 39 fixed column upload, 40 combination column
 * kernel, with 33 - 36 as above;  the resident pk builds (h2b_*_resident, h2b_pk_put_lagrange) add 41 form copies into the pk's storage on
 * the computing device and 42 placement on the other devices (peer copies, sharded slices), in place of 36. */
int h2b_profile_enable(int device, int on);
int h2b_profile_read(int device, int* tags, float* ms, int cap, int* count);
/* force the MSM window size (0 = automatic) -- tuning / tests only */
int h2b_set_msm_window(int c);
/* window-table policy for base sets registered from now on: -1 no tables, 0 automatic spacing, 2..24 forced
 * spacing (tuning / tests; the environment variable H2B_MSM_PRECOMP sets the initial value) */
int h2b_set_msm_precomp(int spacing);
/* tables, spacing (bits) and device bytes per device (the largest share) of a registered base set */
int h2b_base_set_info(uint64_t handle, uint32_t* n_tables, uint32_t* spacing, uint64_t* device_bytes);
/* implicit cache of h2b_msm_bn254_g1: out = {uploads, verified hits, stale copies discarded, uncached (direct) calls,
 * resident implicit sets, of which with tables} -- diagnostics / tests */
int h2b_implicit_cache_stats(uint64_t out[6]);

#ifdef __cplusplus
}
#endif
#endif /* H2B200_H */
