// Written to spec, NOT compiled here (no cargo / rustc in the build image).  What a maintainer adds to the patched
// halo2_proofs (both forks: PSE v2023_02_02 and axiom/dev keep these names) to run the quotient evaluation and the SRS
// load through libh2b200.  Everything else in plonk/evaluation.rs, plonk/prover.rs and poly/kzg/commitment.rs stays.
//
// ---- halo2_proofs/src/plonk/evaluation.rs ---------------------------------------------------------------------------------
// `GraphEvaluator` already is a flat program; the shim only re-encodes its enums as the repr(C) structs of h2b200-sys.
use h2b200_sys::{h2b_calculation, h2b_eval_columns, h2b_graph, h2b_value_source};

pub(crate) fn encode_source(s: &ValueSource) -> h2b_value_source {
    let (kind, index, rotation) = match *s {
        ValueSource::Constant(i) => (0, i, 0),
        ValueSource::Intermediate(i) => (1, i, 0),
        ValueSource::Fixed(c, r) => (2, c, r),
        ValueSource::Advice(c, r) => (3, c, r),
        ValueSource::Instance(c, r) => (4, c, r),
        ValueSource::Challenge(i) => (5, i, 0),
        ValueSource::Beta() => (6, 0, 0),
        ValueSource::Gamma() => (7, 0, 0),
        ValueSource::Theta() => (8, 0, 0),
        ValueSource::Y() => (9, 0, 0),
        ValueSource::PreviousValue() => (10, 0, 0),
    };
    h2b_value_source { kind, index: index as u32, rotation: rotation as u32 }
}

/// Owns the flattened arrays; built once per `Evaluator` (i.e. once per proving key).
pub struct FlatGraph { constants: Vec<[u64; 4]>, rotations: Vec<i32>, calcs: Vec<h2b_calculation>, parts: Vec<h2b_value_source>, n_intermediates: u32 }

impl FlatGraph {
    pub fn new<C: CurveAffine>(g: &GraphEvaluator<C>) -> Self {
        let mut parts = Vec::new();
        let calcs = g.calculations.iter().map(|info| {
            let z = h2b_value_source::default();
            let (op, a, b, po, pl) = match &info.calculation {
                Calculation::Add(a, b) => (0, encode_source(a), encode_source(b), 0, 0),
                Calculation::Sub(a, b) => (1, encode_source(a), encode_source(b), 0, 0),
                Calculation::Mul(a, b) => (2, encode_source(a), encode_source(b), 0, 0),
                Calculation::Square(a) => (3, encode_source(a), z, 0, 0),
                Calculation::Double(a) => (4, encode_source(a), z, 0, 0),
                Calculation::Negate(a) => (5, encode_source(a), z, 0, 0),
                Calculation::Horner(start, ps, factor) => {
                    let po = parts.len();
                    parts.extend(ps.iter().map(encode_source));
                    (6, encode_source(start), encode_source(factor), po, ps.len())
                }
                Calculation::Store(a) => (7, encode_source(a), z, 0, 0),
            };
            h2b_calculation { op, target: info.target as u32, a, b, parts_offset: po as u32, parts_len: pl as u32 }
        }).collect();
        FlatGraph {
            constants: g.constants.iter().map(|c| unsafe { std::mem::transmute_copy::<C::ScalarExt, [u64; 4]>(c) }).collect(),   // Fr = [u64; 4] Montgomery
            rotations: g.rotations.clone(), calcs, parts, n_intermediates: g.num_intermediates as u32,
        }
    }
    pub fn as_ffi(&self) -> h2b_graph {
        h2b_graph { constants: self.constants.as_ptr() as *const u64, n_constants: self.constants.len() as u32,
                    rotations: self.rotations.as_ptr(), n_rotations: self.rotations.len() as u32,
                    calculations: self.calcs.as_ptr(), n_calculations: self.calcs.len() as u32,
                    parts: self.parts.as_ptr(), n_parts: self.parts.len() as u32, n_intermediates: self.n_intermediates }
    }
}

// In `Evaluator::evaluate_h`, with the fixed / advice / instance cosets kept in device buffers (DeviceColumn = a pointer from
// h2b_dev_alloc filled by h2b_coeff_to_extended_dev) instead of `Polynomial<_, ExtendedLagrangeCoeff>`:
//
//   // Custom gates                       (was: multicore::scope over chunks calling custom_gates.evaluate per row)
//   check(h2b_evaluate_graph_dev(dev, &self.flat_custom_gates.as_ffi(), &cols, d_values, size as u32, rot_scale, stream));
//   // Permutations                       (was: parallelize(&mut values, ...) with the l_0 / l_last / product terms)
//   check(h2b_evaluate_h_permutation_dev(dev, d_values, size as u32, rot_scale, z_cosets.as_ptr(), sets.len() as u32,
//         perm_columns.as_ptr(), sigma_cosets.as_ptr(), p.columns.len() as u32, chunk_len as u32, last_rotation.0,
//         d_l0, d_l_last, d_l_active_row, &beta, &gamma, &y, &C::Scalar::DELTA, &C::Scalar::ZETA, &extended_omega, stream));
//   // Lookups                            (was: one parallelize per lookup)
//   for (n, lookup) in lookups.iter().enumerate() {
//       check(h2b_evaluate_h_lookup_dev(dev, &self.flat_lookups[n].as_ffi(), &cols, d_values, size as u32, rot_scale,
//             lookup.d_product_coset, lookup.d_permuted_input_coset, lookup.d_permuted_table_coset, d_l0, d_l_last, d_l_active_row, stream));
//   }
//   // then, still on the device: h2b_fr_scale_dev(t_evaluations, 2^(extended_k - k))   = divide_by_vanishing_poly
//   //                            h2b_extended_to_coeff_dev                              = extended_to_coeff
//   //                            h2b_msm_bn254_g1_dev_registered per n-sized piece      = commit of the h pieces
//
// ---- halo2_proofs/src/poly/kzg/commitment.rs ------------------------------------------------------------------------------
// ParamsKZG gains two handles; read_custom fills them from the file, commit / commit_lagrange use them.
//
//   pub fn read_custom<R: io::Read>(..)  ->  for a file path:
//       let mut k = 0u32; let (mut hg, mut hl) = (0u64, 0u64); let mut g2 = [0u8; 256]; let mut g2_len = 0usize;
//       let mut g = vec![G1Affine::default(); n]; let mut g_lagrange = vec![G1Affine::default(); n];
//       check(h2b_srs_read(path, format as c_int, &mut k, g.as_mut_ptr() as *mut u64, g_lagrange.as_mut_ptr() as *mut u64,
//                          g2.as_mut_ptr(), 256, &mut g2_len, &mut hg, &mut hl));
//       let g2 = G2Affine::read(&mut &g2[..g2_len / 2], format)?; let s_g2 = G2Affine::read(&mut &g2[g2_len / 2..g2_len], format)?;
//   fn commit(&self, poly, _: Blind)           -> h2b_msm_bn254_g1_registered(poly.as_ptr(), self.handle_g, 0, poly.len(), &mut out)
//   fn commit_lagrange(&self, poly, _: Blind)  -> h2b_msm_bn254_g1_registered(poly.as_ptr(), self.handle_g_lagrange, 0, poly.len(), &mut out)
//   impl Drop: h2b_unregister_bases(handle_g); h2b_unregister_bases(handle_g_lagrange)   (reference counted: an unchanged file read
//       again by the next prove_private call -- src/scaffold.rs:174 -- gets the same resident sets without decoding)
