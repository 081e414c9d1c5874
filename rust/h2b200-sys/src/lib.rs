//! `extern "C"` declarations of include/h2b200.h plus the two safe wrappers the `halo2_proofs` patches call.
//!
//! Layout contract (halo2curves 0.3.x): `Fr`/`Fq` are `#[repr(transparent)]`-compatible `[u64; 4]` in Montgomery form,
//! `G1Affine` is `x | y` (64 bytes, (0,0) = identity), `G1` is `x | y | z` Jacobian (96 bytes).  Slices of those types are
//! therefore passed by pointer cast, no conversion and no copy on the host.
#![allow(non_camel_case_types)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

/// Row range of a sharded `evaluate_h` call (include/h2b200.h `h2b_eval_shard`).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct h2b_eval_shard { pub row0: u32, pub rows: u32, pub halo: u32 }
/// `enum ValueSource` of halo2_proofs/src/plonk/evaluation.rs, flattened: kind = variant index in declaration order
/// (Constant, Intermediate, Fixed, Advice, Instance, Challenge, Beta, Gamma, Theta, Y, PreviousValue).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct h2b_value_source { pub kind: u32, pub index: u32, pub rotation: u32 }
/// `enum Calculation` + `CalculationInfo::target`: op = variant index (Add, Sub, Mul, Square, Double, Negate, Horner, Store).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct h2b_calculation { pub op: u32, pub target: u32, pub a: h2b_value_source, pub b: h2b_value_source, pub parts_offset: u32, pub parts_len: u32 }
#[repr(C)]
pub struct h2b_graph {
    pub constants: *const u64, pub n_constants: u32,
    pub rotations: *const i32, pub n_rotations: u32,
    pub calculations: *const h2b_calculation, pub n_calculations: u32,
    pub parts: *const h2b_value_source, pub n_parts: u32,
    pub n_intermediates: u32,
}
#[repr(C)]
pub struct h2b_eval_columns {
    pub fixed: *const *const c_void, pub n_fixed: u32,
    pub advice: *const *const c_void, pub n_advice: u32,
    pub instance: *const *const c_void, pub n_instance: u32,
    pub challenges: *const u64, pub n_challenges: u32,
    pub beta: *const u64, pub gamma: *const u64, pub theta: *const u64, pub y: *const u64,
}

extern "C" {
    pub fn h2b_init(n_devices: c_int) -> c_int;
    pub fn h2b_init_device(device: c_int) -> c_int;
    pub fn h2b_shutdown();
    pub fn h2b_device_count() -> c_int;
    pub fn h2b_last_error() -> *const c_char;
    pub fn h2b_msm_bn254_g1(scalars: *const u64, bases: *const u64, n: usize, out_jac: *mut u64) -> c_int;
    pub fn h2b_ntt_bn254_fr(a: *mut u64, omega: *const u64, log_n: u32) -> c_int;
    pub fn h2b_register_bases(bases: *const u64, n: usize, handle: *mut u64) -> c_int;
    pub fn h2b_unregister_bases(handle: u64) -> c_int;
    pub fn h2b_msm_bn254_g1_registered(scalars: *const u64, handle: u64, offset: usize, n: usize, out_jac: *mut u64) -> c_int;
    pub fn h2b_ntt_bn254_fr_dev(device: c_int, d_a: *mut c_void, omega: *const u64, log_n: u32, stream: *mut c_void) -> c_int;
    pub fn h2b_msm_bn254_g1_dev(device: c_int, d_scalars: *const c_void, d_bases: *const c_void, n: usize, d_out_jac: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_msm_bn254_g1_dev_registered(device: c_int, d_scalars: *const c_void, handle: u64, offset: usize, n: usize, d_out_block: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_scale_dev(device: c_int, d_a: *mut c_void, n: usize, factors: *const u64, count: c_int, stream: *mut c_void) -> c_int;
    // EvaluationDomain conversions and the prover's column primitives on device-resident columns
    pub fn h2b_lagrange_to_coeff_dev(device: c_int, d_a: *mut c_void, k: u32, omega_inv: *const u64, ifft_divisor: *const u64, stream: *mut c_void) -> c_int;
    pub fn h2b_coeff_to_extended_dev(device: c_int, d_a: *mut c_void, k: u32, extended_k: u32, extended_omega: *const u64, zeta_powers: *const u64, stream: *mut c_void) -> c_int;
    pub fn h2b_extended_to_coeff_dev(device: c_int, d_a: *mut c_void, extended_k: u32, extended_omega_inv: *const u64, factors: *const u64, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_batch_invert_dev(device: c_int, d_a: *mut c_void, n: usize, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_prefix_product_dev(device: c_int, d_in: *const c_void, d_out: *mut c_void, n: usize, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_eval_polynomial_dev(device: c_int, d_coeffs: *const c_void, n: usize, x: *const u64, d_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_kate_division_dev(device: c_int, d_a: *const c_void, n: usize, b: *const u64, d_q: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_transpose_dev(device: c_int, d_in: *const c_void, d_out: *mut c_void, rows: u32, cols: u32, stream: *mut c_void) -> c_int;
    pub fn h2b_fr_lincomb_dev(device: c_int, d_cols: *const *const c_void, coeffs: *const u64, m: u32, n: usize, d_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_permutation_product_dev(device: c_int, d_values: *const *const c_void, d_permutations: *const *const c_void, n_columns: u32, n: usize,
                                       beta: *const u64, gamma: *const u64, delta: *const u64, deltaomega: *const u64, omega: *const u64,
                                       last_z: *const u64, d_z: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_lookup_permute_dev(device: c_int, d_input: *const c_void, d_table: *const c_void, usable_rows: u32, d_permuted_input: *mut c_void,
                                  d_permuted_table: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_lookup_permute_async_dev(device: c_int, d_input: *const c_void, d_table: *const c_void, usable_rows: u32, d_permuted_input: *mut c_void,
                                        d_permuted_table: *mut c_void, d_status: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_lookup_product_dev(device: c_int, d_compressed_input: *const c_void, d_compressed_table: *const c_void, d_permuted_input: *const c_void,
                                  d_permuted_table: *const c_void, n: usize, beta: *const u64, gamma: *const u64, d_z: *mut c_void, stream: *mut c_void) -> c_int;
    // plonk::evaluation (evaluate_h)
    pub fn h2b_evaluate_graph_dev(device: c_int, graph: *const h2b_graph, cols: *const h2b_eval_columns, d_values: *mut c_void, size: u32, rot_scale: i32,
                                  stream: *mut c_void) -> c_int;
    pub fn h2b_evaluate_h_permutation_dev(device: c_int, d_values: *mut c_void, size: u32, rot_scale: i32, d_product_cosets: *const *const c_void, n_sets: u32,
                                          d_columns: *const *const c_void, d_perm_cosets: *const *const c_void, n_columns: u32, chunk_len: u32,
                                          last_rotation: i32, d_l0: *const c_void, d_l_last: *const c_void, d_l_active_row: *const c_void, beta: *const u64,
                                          gamma: *const u64, y: *const u64, delta: *const u64, zeta: *const u64, extended_omega: *const u64,
                                          stream: *mut c_void) -> c_int;
    pub fn h2b_evaluate_h_lookup_dev(device: c_int, graph: *const h2b_graph, cols: *const h2b_eval_columns, d_values: *mut c_void, size: u32, rot_scale: i32,
                                     d_product_coset: *const c_void, d_permuted_input_coset: *const c_void, d_permuted_table_coset: *const c_void,
                                     d_l0: *const c_void, d_l_last: *const c_void, d_l_active_row: *const c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_evaluate_graph_shard_dev(device: c_int, graph: *const h2b_graph, cols: *const h2b_eval_columns, d_values: *mut c_void, size: u32, rot_scale: i32,
                                        shard: *const h2b_eval_shard, stream: *mut c_void) -> c_int;
    pub fn h2b_evaluate_h_permutation_shard_dev(device: c_int, d_values: *mut c_void, size: u32, rot_scale: i32, d_product_cosets: *const *const c_void,
                                                n_sets: u32, d_columns: *const *const c_void, d_perm_cosets: *const *const c_void, n_columns: u32, chunk_len: u32,
                                                last_rotation: i32, d_l0: *const c_void, d_l_last: *const c_void, d_l_active_row: *const c_void,
                                                beta: *const u64, gamma: *const u64, y: *const u64, delta: *const u64, zeta: *const u64,
                                                extended_omega: *const u64, shard: *const h2b_eval_shard, stream: *mut c_void) -> c_int;
    pub fn h2b_evaluate_h_lookup_shard_dev(device: c_int, graph: *const h2b_graph, cols: *const h2b_eval_columns, d_values: *mut c_void, size: u32,
                                           rot_scale: i32, d_product_coset: *const c_void, d_permuted_input_coset: *const c_void,
                                           d_permuted_table_coset: *const c_void, d_l0: *const c_void, d_l_last: *const c_void,
                                           d_l_active_row: *const c_void, shard: *const h2b_eval_shard, stream: *mut c_void) -> c_int;
    // SRS file -> resident base sets (ParamsKZG::read_custom / write_custom)
    pub fn h2b_g1_decode_dev(device: c_int, d_bytes: *const c_void, n: usize, format: c_int, d_out_affine: *mut c_void, first_invalid: *mut u64, stream: *mut c_void) -> c_int;
    pub fn h2b_g1_encode_dev(device: c_int, d_affine: *const c_void, n: usize, d_out_bytes: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_srs_read(path: *const c_char, format: c_int, k: *mut u32, out_g: *mut u64, out_g_lagrange: *mut u64, g2_bytes: *mut u8, g2_cap: usize,
                        g2_len: *mut usize, handle_g: *mut u64, handle_g_lagrange: *mut u64) -> c_int;
    pub fn h2b_srs_write(path: *const c_char, format: c_int, k: u32, g: *const u64, g_lagrange: *const u64, g2_bytes: *const u8, g2_len: usize) -> c_int;
    pub fn h2b_srs_cache_clear() -> c_int;
    // ParamsKZG::setup on the device and the fixed-base multiples of the generator it is built on
    pub fn h2b_srs_setup(k: u32, s: *const u64, out_g: *mut u64, out_g_lagrange: *mut u64, handle_g: *mut u64, handle_g_lagrange: *mut u64) -> c_int;
    pub fn h2b_g1_generator_mul_dev(device: c_int, d_scalars: *const c_void, n: usize, d_out_affine: *mut c_void, stream: *mut c_void) -> c_int;
    // ParamsKZG::downsize on the device and the G1 NTT (g_to_lagrange) it is built on
    pub fn h2b_g1_to_lagrange_dev(device: c_int, d_g_affine: *const c_void, k: u32, d_out_affine: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_srs_downsize(handle_g: u64, k: u32, out_g_lagrange: *mut u64, handle_g_out: *mut u64, handle_g_lagrange_out: *mut u64) -> c_int;
    // the permutation argument's sigma columns (Assembly::build_vk / build_pk) and keygen_pk's l0 / l_last / l_active_row
    pub fn h2b_permutation_sigma_dev(device: c_int, d_mapping: *const *const c_void, n_columns: u32, k: u32, delta: *const u64, omega: *const u64,
                                     d_sigma: *const *mut c_void, d_status: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_keygen_lagrange_indicators_dev(device: c_int, k: u32, extended_k: u32, blinding_factors: u32, omega_inv: *const u64, ifft_divisor: *const u64,
                                              extended_omega: *const u64, zeta_powers: *const u64, d_l0: *mut c_void, d_l_last: *mut c_void,
                                              d_l_active_row: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_permutation_build_vk(mapping: *const *const u64, n_columns: u32, k: u32, delta: *const u64, omega: *const u64, handle_g_lagrange: u64,
                                    out_commitments: *mut u64) -> c_int;
    pub fn h2b_permutation_build_pk(mapping: *const *const u64, n_columns: u32, k: u32, extended_k: u32, delta: *const u64, omega: *const u64,
                                    omega_inv: *const u64, ifft_divisor: *const u64, extended_omega: *const u64, zeta_powers: *const u64,
                                    out_permutations: *const *mut u64, out_polys: *const *mut u64, out_cosets: *const *mut u64) -> c_int;
    // compress_selectors' exclusion matrix and the fixed columns of keygen_vk / keygen_pk
    pub fn h2b_selector_exclusion(activations: *const *const u8, n_selectors: u32, k: u32, out: *mut u8) -> c_int;
    pub fn h2b_keygen_fixed_build_vk(fixed: *const *const u64, n_fixed: u32, activations: *const *const u8, n_selectors: u32, combination_of: *const u32,
                                     root_of: *const u32, n_combinations: u32, k: u32, handle_g_lagrange: u64, out_commitments: *mut u64) -> c_int;
    pub fn h2b_keygen_fixed_build_pk(fixed: *const *const u64, n_fixed: u32, activations: *const *const u8, n_selectors: u32, combination_of: *const u32,
                                     root_of: *const u32, n_combinations: u32, k: u32, extended_k: u32, omega_inv: *const u64, ifft_divisor: *const u64,
                                     extended_omega: *const u64, zeta_powers: *const u64, out_combination_values: *const *mut u64,
                                     out_polys: *const *mut u64, out_cosets: *const *mut u64) -> c_int;
    // the proving key resident on the devices (h2b_pk_*)
    pub fn h2b_pk_create(k: u32, extended_k: u32, n_fixed: u32, n_permutation: u32, layout: c_int, halo: u32, omega: *const u64, omega_inv: *const u64,
                         ifft_divisor: *const u64, extended_omega: *const u64, zeta_powers: *const u64, handle: *mut u64) -> c_int;
    pub fn h2b_keygen_fixed_build_pk_resident(fixed: *const *const u64, n_fixed: u32, activations: *const *const u8, n_selectors: u32,
                                              combination_of: *const u32, root_of: *const u32, n_combinations: u32, pk: u64, first_column: u32) -> c_int;
    pub fn h2b_permutation_build_pk_resident(mapping: *const *const u64, n_columns: u32, delta: *const u64, pk: u64) -> c_int;
    pub fn h2b_keygen_lagrange_indicators_resident(pk: u64, blinding_factors: u32) -> c_int;
    pub fn h2b_pk_put_lagrange(pk: u64, part: c_int, first: u32, count: u32, values: *const *const u64) -> c_int;
    pub fn h2b_pk_column(pk: u64, device: c_int, part: c_int, form: c_int, index: u32, d_ptr: *mut *mut c_void, shard: *mut h2b_eval_shard) -> c_int;
    pub fn h2b_pk_download(pk: u64, part: c_int, form: c_int, index: u32, host_out: *mut u64) -> c_int;
    pub fn h2b_pk_info(pk: u64, per_device_bytes: *mut u64) -> c_int;
    pub fn h2b_pk_release(pk: u64) -> c_int;
    pub fn h2b_fr_eval_queries_dev(device: c_int, d_polys: *const *const c_void, n_polys: u32, n: usize, queries: *const h2b_opening_query, n_queries: u32,
                                   d_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_shplonk_begin(device: c_int, polys: *const *const c_void, polys_on_host: c_int, n_polys: u32, n: usize, queries: *const h2b_opening_query,
                             n_queries: u32, handle_g: u64, y: *const u64, v: *const u64, out_h1_jac: *mut u64, session: *mut u64) -> c_int;
    pub fn h2b_shplonk_finish(session: u64, u: *const u64, out_h2_jac: *mut u64) -> c_int;
    pub fn h2b_shplonk_release(session: u64) -> c_int;
    pub fn h2b_dev_alloc(device: c_int, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn h2b_dev_free(device: c_int, p: *mut c_void) -> c_int;
    pub fn h2b_memcpy_h2d(device: c_int, d_dst: *mut c_void, h_src: *const c_void, bytes: usize) -> c_int;
    pub fn h2b_memcpy_h2d_async(device: c_int, d_dst: *mut c_void, h_src: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn h2b_memcpy_d2h(device: c_int, h_dst: *mut c_void, d_src: *const c_void, bytes: usize) -> c_int;
    pub fn h2b_dev_sync(device: c_int) -> c_int;
    // round 2: sharded residency, batched columns / polynomials, one-upload column pipeline, column copies
    pub fn h2b_register_bases_sharded(bases: *const u64, n: usize, handle: *mut u64) -> c_int;
    pub fn h2b_msm_bn254_g1_batch_registered(scalars: *const *const u64, lens: *const usize, count: usize, handle: u64, out_jac: *mut u64) -> c_int;
    pub fn h2b_ntt_bn254_fr_batch(a: *const *mut u64, count: usize, omega: *const u64, log_n: u32) -> c_int;
    pub fn h2b_msm_bn254_g1_dev_batch_registered(device: c_int, d_scalars: *const *const c_void, lens: *const usize, count: usize, handle: u64,
                                                 d_out_blocks: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn h2b_ntt_bn254_fr_dev_batch(device: c_int, d_polys: *const *mut c_void, count: usize, omega: *const u64, log_n: u32, stream: *mut c_void) -> c_int;
    pub fn h2b_lagrange_to_coeff_dev_batch(device: c_int, d_cols: *const *mut c_void, count: usize, k: u32, omega_inv: *const u64, ifft_divisor: *const u64,
                                           stream: *mut c_void) -> c_int;
    pub fn h2b_coeff_to_extended_dev_batch(device: c_int, d_cols: *const *mut c_void, count: usize, k: u32, extended_k: u32, extended_omega: *const u64,
                                           zeta_powers: *const u64, stream: *mut c_void) -> c_int;
    pub fn h2b_column_pipeline(device: c_int, lagrange: *const u64, handle_g_lagrange: u64, k: u32, extended_k: u32, omega_inv: *const u64,
                               ifft_divisor: *const u64, extended_omega: *const u64, zeta_powers: *const u64, out_commitment_jac: *mut u64,
                               out_coeff: *mut u64, out_extended: *mut u64, d_extended: *mut *mut c_void) -> c_int;
    pub fn h2b_memcpy_d2d_async(device: c_int, d_dst: *mut c_void, d_src: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn h2b_memset_zero_async(device: c_int, d_dst: *mut c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn h2b_implicit_cache_stats(out: *mut u64) -> c_int;
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(h2b_last_error()).to_string_lossy().into_owned() }
}

/// Initialise every visible B200 once; panics (like the upstream functions' asserts) when no device is usable --
/// there is no CPU fallback.
pub fn ensure_init() {
    use std::sync::Once;
    static INIT: Once = Once::new();
    INIT.call_once(|| {
        let rc = unsafe { h2b_init(0) };
        if rc != 0 {
            panic!("h2b200: initialisation failed ({rc}): {}", last_error());
        }
    });
}

/// `best_multiexp::<G1Affine>`: `scalars` = `&[Fr]` as `n x 4` u64, `bases` = `&[G1Affine]` as `n x 8` u64;
/// returns the Jacobian triple `x | y | z`.
pub fn msm_bn254_g1(scalars: &[[u64; 4]], bases: &[[u64; 8]]) -> [u64; 12] {
    assert_eq!(scalars.len(), bases.len());
    ensure_init();
    let mut out = [0u64; 12];
    let rc = unsafe { h2b_msm_bn254_g1(scalars.as_ptr() as *const u64, bases.as_ptr() as *const u64, scalars.len(), out.as_mut_ptr()) };
    if rc != 0 {
        panic!("h2b_msm_bn254_g1 failed ({rc}): {}", last_error());
    }
    out
}

/// `best_fft::<Fr>`: in place, natural order, no scaling.
pub fn ntt_bn254_fr(a: &mut [[u64; 4]], omega: &[u64; 4], log_n: u32) {
    assert_eq!(a.len(), 1usize << log_n);
    ensure_init();
    let rc = unsafe { h2b_ntt_bn254_fr(a.as_mut_ptr() as *mut u64, omega.as_ptr(), log_n) };
    if rc != 0 {
        panic!("h2b_ntt_bn254_fr failed ({rc}): {}", last_error());
    }
}

/// The G1 half of `ParamsKZG::<Bn256>::setup(k, rng)` for the toxic waste `s` (Montgomery limbs, `Fr::random(rng)` drawn by
/// the caller): `g[i] = [s^i] G`, `g_lagrange[i] = [L_i(s)] G` as `2^k x 8` u64 each, plus the handles of both vectors as
/// registered base sets (window tables built on every device).  Panics like upstream's `invert().unwrap()` when `s` is a
/// `2^k`-th root of unity, and on `k > 28`.
pub fn srs_setup(k: u32, s: &[u64; 4]) -> (Vec<[u64; 8]>, Vec<[u64; 8]>, u64, u64) {
    assert!(k <= 28);
    ensure_init();
    let n = 1usize << k;
    let (mut g, mut g_lagrange) = (vec![[0u64; 8]; n], vec![[0u64; 8]; n]);
    let (mut hg, mut hl) = (0u64, 0u64);
    let rc = unsafe { h2b_srs_setup(k, s.as_ptr(), g.as_mut_ptr() as *mut u64, g_lagrange.as_mut_ptr() as *mut u64, &mut hg, &mut hl) };
    if rc != 0 {
        panic!("h2b_srs_setup failed ({rc}): {}", last_error());
    }
    (g, g_lagrange, hg, hl)
}

/// The G1 half of `ParamsKZG::<Bn256>::downsize(k)` on the resident g of the registered, replicated set `handle_g`:
/// `g_lagrange` of the `2^k`-point prefix of g (`g_to_lagrange`, computed on the device) as `2^k x 8` u64, plus the handles of
/// two new registered sets, the prefix of g and that g_lagrange.  The old handles stay valid; the caller gives them back.
/// Panics like upstream's `assert!(k <= self.k)` when `2^k` exceeds the set.
pub fn srs_downsize(handle_g: u64, k: u32) -> (Vec<[u64; 8]>, u64, u64) {
    assert!(k <= 28);
    ensure_init();
    let mut g_lagrange = vec![[0u64; 8]; 1usize << k];
    let (mut hg, mut hl) = (0u64, 0u64);
    let rc = unsafe { h2b_srs_downsize(handle_g, k, g_lagrange.as_mut_ptr() as *mut u64, &mut hg, &mut hl) };
    if rc != 0 {
        panic!("h2b_srs_downsize failed ({rc}): {}", last_error());
    }
    (g_lagrange, hg, hl)
}

/// The domain constants the keygen calls take, as Montgomery limbs (`EvaluationDomain`'s fields; `zeta_powers` = 1, g_coset,
/// g_coset_inv).
pub struct KeygenDomain {
    pub k: u32,
    pub extended_k: u32,
    pub omega: [u64; 4],
    pub omega_inv: [u64; 4],
    pub ifft_divisor: [u64; 4],
    pub extended_omega: [u64; 4],
    pub zeta_powers: [[u64; 4]; 3],
}

/// A mapping column as the C ABI reads it: `2^k` pairs of u64 (column, row).  Upstream's `Vec<(usize, usize)>` is passed as is
/// when `(usize, usize)` is laid out that way on this target (64-bit usize, field 0 first); otherwise it is converted once.
fn mapping_columns(mapping: &[Vec<(usize, usize)>], n: usize) -> (Vec<Vec<[u64; 2]>>, Vec<*const u64>) {
    let same_layout = std::mem::size_of::<(usize, usize)>() == 16
        && std::mem::size_of::<usize>() == 8
        && std::mem::offset_of!((usize, usize), 0) == 0
        && std::mem::offset_of!((usize, usize), 1) == 8;
    let mut owned = Vec::new();
    let mut ptrs = Vec::with_capacity(mapping.len());
    for col in mapping {
        assert_eq!(col.len(), n, "mapping column length != 2^k");
        if same_layout {
            ptrs.push(col.as_ptr() as *const u64);
        } else {
            owned.push(col.iter().map(|&(c, r)| [c as u64, r as u64]).collect::<Vec<_>>());
            ptrs.push(owned.last().unwrap().as_ptr() as *const u64);
        }
    }
    (owned, ptrs)
}

/// `Assembly::build_vk`: `commit_lagrange(sigma_i)` (Jacobian, 12 u64) for every column of `mapping`, over the registered set
/// `handle_g_lagrange`.  Panics like upstream's out-of-range index on an invalid mapping entry.
pub fn permutation_build_vk(mapping: &[Vec<(usize, usize)>], delta: &[u64; 4], dom: &KeygenDomain, handle_g_lagrange: u64) -> Vec<[u64; 12]> {
    ensure_init();
    let (_owned, ptrs) = mapping_columns(mapping, 1usize << dom.k);
    let mut out = vec![[0u64; 12]; mapping.len()];
    let rc = unsafe {
        h2b_permutation_build_vk(ptrs.as_ptr(), ptrs.len() as u32, dom.k, delta.as_ptr(), dom.omega.as_ptr(), handle_g_lagrange, out.as_mut_ptr() as *mut u64)
    };
    if rc != 0 {
        panic!("h2b_permutation_build_vk failed ({rc}): {}", last_error());
    }
    out
}

/// `Assembly::build_pk`: per column sigma (Lagrange), its coefficients and its extended coset, as `2^k`, `2^k` and `2^extended_k`
/// Montgomery scalars.  Panics like upstream's out-of-range index on an invalid mapping entry.
#[allow(clippy::type_complexity)]
pub fn permutation_build_pk(mapping: &[Vec<(usize, usize)>], delta: &[u64; 4], dom: &KeygenDomain) -> (Vec<Vec<[u64; 4]>>, Vec<Vec<[u64; 4]>>, Vec<Vec<[u64; 4]>>) {
    ensure_init();
    let n = 1usize << dom.k;
    let (_owned, ptrs) = mapping_columns(mapping, n);
    let mut perms = vec![vec![[0u64; 4]; n]; mapping.len()];
    let mut polys = vec![vec![[0u64; 4]; n]; mapping.len()];
    let mut cosets = vec![vec![[0u64; 4]; 1usize << dom.extended_k]; mapping.len()];
    let outs = |v: &mut Vec<Vec<[u64; 4]>>| v.iter_mut().map(|c| c.as_mut_ptr() as *mut u64).collect::<Vec<_>>();
    let (p, c, e) = (outs(&mut perms), outs(&mut polys), outs(&mut cosets));
    let rc = unsafe {
        h2b_permutation_build_pk(ptrs.as_ptr(), ptrs.len() as u32, dom.k, dom.extended_k, delta.as_ptr(), dom.omega.as_ptr(), dom.omega_inv.as_ptr(),
                                 dom.ifft_divisor.as_ptr(), dom.extended_omega.as_ptr(), dom.zeta_powers.as_ptr() as *const u64, p.as_ptr(), c.as_ptr(),
                                 e.as_ptr())
    };
    if rc != 0 {
        panic!("h2b_permutation_build_pk failed ({rc}): {}", last_error());
    }
    (perms, polys, cosets)
}

/// keygen_pk's `(l0, l_last, l_active_row)` on the extended coset, each `2^extended_k` Montgomery scalars, computed on device 0.
pub fn keygen_lagrange_indicators(dom: &KeygenDomain, blinding_factors: u32) -> [Vec<[u64; 4]>; 3] {
    ensure_init();
    let en = 1usize << dom.extended_k;
    let mut d = [std::ptr::null_mut::<c_void>(); 3];
    for p in d.iter_mut() {
        assert_eq!(unsafe { h2b_dev_alloc(0, en * 32, p) }, 0, "h2b_dev_alloc: {}", last_error());
    }
    let mut out = [vec![[0u64; 4]; en], vec![[0u64; 4]; en], vec![[0u64; 4]; en]];
    let rc = unsafe {
        h2b_keygen_lagrange_indicators_dev(0, dom.k, dom.extended_k, blinding_factors, dom.omega_inv.as_ptr(), dom.ifft_divisor.as_ptr(),
                                           dom.extended_omega.as_ptr(), dom.zeta_powers.as_ptr() as *const u64, d[0], d[1], d[2], std::ptr::null_mut())
    };
    let mut ok = rc == 0 && unsafe { h2b_dev_sync(0) } == 0;
    for (o, p) in out.iter_mut().zip(d.iter()) {
        ok = ok && unsafe { h2b_memcpy_d2h(0, o.as_mut_ptr() as *mut c_void, *p, en * 32) } == 0;
    }
    for p in d {
        unsafe { h2b_dev_free(0, p) };
    }
    if !ok {
        panic!("keygen_pk indicators failed: {}", last_error());
    }
    out
}

/// compress_selectors' assignment: per selector its combination (the index of the fixed column `process` allocates for it, counted
/// from the first one) and its root; `n_combinations` columns in all.
pub struct SelectorAssignment {
    pub combination_of: Vec<u32>,
    pub root_of: Vec<u32>,
    pub n_combinations: u32,
}

/// Rust's `bool` is one byte, 0 or 1: a `Vec<bool>` goes to the C ABI as it sits in memory.
fn activation_rows(activations: &[Vec<bool>], n: usize) -> Vec<*const u8> {
    activations.iter().map(|a| {
        assert_eq!(a.len(), n, "selector activations length != 2^k");
        a.as_ptr() as *const u8
    }).collect()
}

fn fixed_rows(fixed: &[&[[u64; 4]]], n: usize) -> Vec<*const u64> {
    fixed.iter().map(|c| {
        assert_eq!(c.len(), n, "fixed column length != 2^k");
        c.as_ptr() as *const u64
    }).collect()
}

/// `process`'s exclusion matrix: `out[i][j]` is true when selectors i and j are both active on some row (symmetric, false on the
/// diagonal).
pub fn selector_exclusion(activations: &[Vec<bool>], k: u32) -> Vec<Vec<bool>> {
    ensure_init();
    let s = activations.len();
    let rows = activation_rows(activations, 1usize << k);
    let mut out = vec![0u8; s * s];
    let rc = unsafe { h2b_selector_exclusion(rows.as_ptr(), s as u32, k, out.as_mut_ptr()) };
    if rc != 0 {
        panic!("h2b_selector_exclusion failed ({rc}): {}", last_error());
    }
    out.chunks(s.max(1)).take(s).map(|r| r.iter().map(|&b| b != 0).collect()).collect()
}

/// keygen_vk's `fixed_commitments`: `commit_lagrange` (Jacobian, 12 u64) of each fixed column, then of each combination column.
pub fn keygen_fixed_build_vk(fixed: &[&[[u64; 4]]], activations: &[Vec<bool>], a: &SelectorAssignment, k: u32, handle_g_lagrange: u64) -> Vec<[u64; 12]> {
    ensure_init();
    let n = 1usize << k;
    let (f, rows) = (fixed_rows(fixed, n), activation_rows(activations, n));
    let mut out = vec![[0u64; 12]; fixed.len() + a.n_combinations as usize];
    let rc = unsafe {
        h2b_keygen_fixed_build_vk(f.as_ptr(), f.len() as u32, rows.as_ptr(), rows.len() as u32, a.combination_of.as_ptr(), a.root_of.as_ptr(),
                                  a.n_combinations, k, handle_g_lagrange, out.as_mut_ptr() as *mut u64)
    };
    if rc != 0 {
        panic!("h2b_keygen_fixed_build_vk failed ({rc}): {}", last_error());
    }
    out
}

/// keygen_pk's fixed columns: the combination columns (Lagrange), and the coefficients and extended cosets of every fixed and
/// combination column, as Montgomery scalars.
#[allow(clippy::type_complexity)]
pub fn keygen_fixed_build_pk(fixed: &[&[[u64; 4]]], activations: &[Vec<bool>], a: &SelectorAssignment, dom: &KeygenDomain)
    -> (Vec<Vec<[u64; 4]>>, Vec<Vec<[u64; 4]>>, Vec<Vec<[u64; 4]>>) {
    ensure_init();
    let n = 1usize << dom.k;
    let (f, rows) = (fixed_rows(fixed, n), activation_rows(activations, n));
    let total = fixed.len() + a.n_combinations as usize;
    let mut values = vec![vec![[0u64; 4]; n]; a.n_combinations as usize];
    let mut polys = vec![vec![[0u64; 4]; n]; total];
    let mut cosets = vec![vec![[0u64; 4]; 1usize << dom.extended_k]; total];
    let outs = |v: &mut Vec<Vec<[u64; 4]>>| v.iter_mut().map(|c| c.as_mut_ptr() as *mut u64).collect::<Vec<_>>();
    let (v, p, e) = (outs(&mut values), outs(&mut polys), outs(&mut cosets));
    let rc = unsafe {
        h2b_keygen_fixed_build_pk(f.as_ptr(), f.len() as u32, rows.as_ptr(), rows.len() as u32, a.combination_of.as_ptr(), a.root_of.as_ptr(),
                                  a.n_combinations, dom.k, dom.extended_k, dom.omega_inv.as_ptr(), dom.ifft_divisor.as_ptr(), dom.extended_omega.as_ptr(),
                                  dom.zeta_powers.as_ptr() as *const u64, v.as_ptr(), p.as_ptr(), e.as_ptr())
    };
    if rc != 0 {
        panic!("h2b_keygen_fixed_build_pk failed ({rc}): {}", last_error());
    }
    (values, polys, cosets)
}

// ---- the proving key resident on the devices ------------------------------------------------------------------------------------
pub const PK_FIXED: c_int = 0;
pub const PK_PERMUTATION: c_int = 1;
pub const PK_INDICATORS: c_int = 2;
pub const PK_VALUES: c_int = 0;
pub const PK_COEFF: c_int = 1;
pub const PK_EXTENDED: c_int = 2;
pub const PK_REPLICATED: c_int = 0;
pub const PK_ROW_SHARDED: c_int = 1;

/// A `ProvingKey`'s fixed, permutation and indicator columns held on the devices (`h2b_pk_*`).  Every call panics on a non-zero
/// return code, as the upstream functions' asserts do; `Drop` releases the handle.
pub struct ResidentProvingKey {
    pub handle: u64,
    pub k: u32,
    pub extended_k: u32,
}

impl ResidentProvingKey {
    pub fn new(dom: &KeygenDomain, n_fixed: u32, n_permutation: u32, layout: c_int, halo: u32) -> Self {
        ensure_init();
        let mut handle = 0u64;
        let rc = unsafe {
            h2b_pk_create(dom.k, dom.extended_k, n_fixed, n_permutation, layout, halo, dom.omega.as_ptr(), dom.omega_inv.as_ptr(), dom.ifft_divisor.as_ptr(),
                          dom.extended_omega.as_ptr(), dom.zeta_powers.as_ptr() as *const u64, &mut handle)
        };
        if rc != 0 {
            panic!("h2b_pk_create failed ({rc}): {}", last_error());
        }
        ResidentProvingKey { handle, k: dom.k, extended_k: dom.extended_k }
    }

    fn check(rc: c_int, what: &str) {
        if rc != 0 {
            panic!("{what} failed ({rc}): {}", last_error());
        }
    }

    /// keygen_pk's fixed columns (the caller's, then the combination columns) into FIXED columns `first_column ..`
    pub fn build_fixed(&self, fixed: &[&[[u64; 4]]], activations: &[Vec<bool>], a: &SelectorAssignment, first_column: u32) {
        let n = 1usize << self.k;
        let (f, rows) = (fixed_rows(fixed, n), activation_rows(activations, n));
        Self::check(unsafe {
            h2b_keygen_fixed_build_pk_resident(f.as_ptr(), f.len() as u32, rows.as_ptr(), rows.len() as u32, a.combination_of.as_ptr(), a.root_of.as_ptr(),
                                               a.n_combinations, self.handle, first_column)
        }, "h2b_keygen_fixed_build_pk_resident");
    }

    /// `Assembly::build_pk` into the PERMUTATION part; panics like upstream's out-of-range index on an invalid mapping entry
    pub fn build_permutation(&self, mapping: &[Vec<(usize, usize)>], delta: &[u64; 4]) {
        let (_owned, ptrs) = mapping_columns(mapping, 1usize << self.k);
        Self::check(unsafe { h2b_permutation_build_pk_resident(ptrs.as_ptr(), ptrs.len() as u32, delta.as_ptr(), self.handle) },
                    "h2b_permutation_build_pk_resident");
    }

    pub fn build_indicators(&self, blinding_factors: u32) {
        Self::check(unsafe { h2b_keygen_lagrange_indicators_resident(self.handle, blinding_factors) }, "h2b_keygen_lagrange_indicators_resident");
    }

    /// columns of a `ProvingKey` built elsewhere, in Lagrange form
    pub fn put_lagrange(&self, part: c_int, first: u32, values: &[&[[u64; 4]]]) {
        let v = fixed_rows(values, 1usize << self.k);
        Self::check(unsafe { h2b_pk_put_lagrange(self.handle, part, first, v.len() as u32, v.as_ptr()) }, "h2b_pk_put_lagrange");
    }

    /// the column on `device` and its slice (row0, rows, halo); the pointer is valid while `self` lives
    pub fn column(&self, device: c_int, part: c_int, form: c_int, index: u32) -> (*mut c_void, h2b_eval_shard) {
        let mut p = std::ptr::null_mut();
        let mut shard = h2b_eval_shard { row0: 0, rows: 0, halo: 0 };
        Self::check(unsafe { h2b_pk_column(self.handle, device, part, form, index, &mut p, &mut shard) }, "h2b_pk_column");
        (p, shard)
    }

    /// a host copy of one column, for `ProvingKey`'s host fields and `pk.write`
    pub fn download(&self, part: c_int, form: c_int, index: u32) -> Vec<[u64; 4]> {
        let rows = 1usize << if form == PK_EXTENDED { self.extended_k } else { self.k };
        let mut out = vec![[0u64; 4]; rows];
        Self::check(unsafe { h2b_pk_download(self.handle, part, form, index, out.as_mut_ptr() as *mut u64) }, "h2b_pk_download");
        out
    }
}

impl Drop for ResidentProvingKey {
    fn drop(&mut self) {
        unsafe { h2b_pk_release(self.handle) };
    }
}

/// `h2b_opening_query`: polynomial index and point (Montgomery limbs)
#[repr(C)]
#[derive(Clone, Copy)]
pub struct h2b_opening_query {
    pub poly: u32,
    pub reserved: u32,
    pub point: [u64; 4],
}

/// One SHPLONK opening between its two commitments (`h2b_shplonk_*`): `begin` returns h1, `finish` h2; `Drop` releases the session on
/// every path, a panic included.  Polynomials are host slices of n Fr limbs, uploaded once by `begin`.
pub struct ShplonkSession {
    handle: u64,
}

impl ShplonkSession {
    pub fn begin(polys: &[&[[u64; 4]]], queries: &[h2b_opening_query], handle_g: u64, y: &[u64; 4], v: &[u64; 4]) -> (Self, [u64; 12]) {
        ensure_init();
        let n = polys.first().map(|p| p.len()).unwrap_or(0);
        assert!(polys.iter().all(|p| p.len() == n), "ProverSHPLONK: polynomials of different lengths");
        let ptrs: Vec<*const c_void> = polys.iter().map(|p| p.as_ptr() as *const c_void).collect();
        let mut h1 = [0u64; 12];
        let mut handle = 0u64;
        let rc = unsafe {
            h2b_shplonk_begin(0, ptrs.as_ptr(), 1, ptrs.len() as u32, n, queries.as_ptr(), queries.len() as u32, handle_g, y.as_ptr(), v.as_ptr(),
                              h1.as_mut_ptr(), &mut handle)
        };
        if rc != 0 {
            panic!("h2b_shplonk_begin failed ({rc}): {}", last_error());
        }
        (ShplonkSession { handle }, h1)
    }

    pub fn finish(&self, u: &[u64; 4]) -> [u64; 12] {
        let mut h2 = [0u64; 12];
        let rc = unsafe { h2b_shplonk_finish(self.handle, u.as_ptr(), h2.as_mut_ptr()) };
        if rc != 0 {
            // upstream: z_0.invert().unwrap() panics when u is a point of T outside S_0
            panic!("h2b_shplonk_finish failed ({rc}): {}", last_error());
        }
        h2
    }
}

impl Drop for ShplonkSession {
    fn drop(&mut self) {
        unsafe { h2b_shplonk_release(self.handle) };
    }
}
