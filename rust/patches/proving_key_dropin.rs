// Written to spec, NOT compiled here (no cargo / rustc in the build image).  What a maintainer adds to the patched halo2_proofs so that
// keygen_pk leaves its proving key on the devices and create_proof's device steps read it from there instead of uploading it for every
// proof.  The ProvingKey struct, its host fields and pk.write / ProvingKey::read behave as upstream's.
//
// ---- halo2_proofs/src/plonk.rs --------------------------------------------------------------------------------------------------
// `ProvingKey<C>` gains one field (not serialized, default empty):
//
//     #[doc(hidden)]
//     pub h2b_resident: std::cell::OnceCell<h2b200_sys::ResidentProvingKey>,
//
// `ResidentProvingKey`'s Drop releases the handle, so dropping the ProvingKey frees its device copy (after the work queued on the
// devices).  `ProvingKey::read` leaves the cell empty; the first `create_proof` fills it through `h2b_resident_of` below, from the host
// fields, with h2b_pk_put_lagrange (the device derives the coefficient and extended forms bit for bit as keygen does).

use h2b200_sys::{KeygenDomain, ResidentProvingKey, SelectorAssignment, PK_COEFF, PK_EXTENDED, PK_FIXED, PK_INDICATORS, PK_PERMUTATION,
                 PK_REPLICATED, PK_VALUES};

/// The layout a prover process wants: every column on every device (each device proves whole columns), or, with a row-sharded
/// evaluate_h, the extended cosets split by row with `halo` = the largest rotated read (DESIGN section 7).
pub fn h2b_layout() -> (std::os::raw::c_int, u32) {
    (PK_REPLICATED, 0)
}

// ---- halo2_proofs/src/plonk/keygen.rs, keygen_pk (G1Affine dispatch as in fixed_keygen_dropin.rs) ---------------------------------
// After upstream has built `fixed` (the caller's fixed columns, extended by the selector columns), `assembly.mapping` and the vk, the
// patched body replaces the fixed_polys / fixed_cosets, permutation::Assembly::build_pk and l0 / l_last / l_active_row blocks with:
pub fn keygen_pk_h2b<C: CurveAffine>(
    dom: &KeygenDomain,
    fixed: &[&[[u64; 4]]],                  // the caller's fixed columns after batch_invert_assigned (Lagrange, Montgomery)
    selectors: &[Vec<bool>],
    assignment: &SelectorAssignment,        // from compress_selectors_h2b
    mapping: &[Vec<(usize, usize)>],
    delta: &[u64; 4],
    blinding_factors: u32,
) -> (ResidentProvingKey, HostPkColumns) {
    let n_fixed = (fixed.len() as u32) + assignment.n_combinations;
    let (layout, halo) = h2b_layout();
    let pk = ResidentProvingKey::new(dom, n_fixed, mapping.len() as u32, layout, halo);
    pk.build_fixed(fixed, selectors, assignment, 0);
    pk.build_permutation(mapping, delta);
    pk.build_indicators(blinding_factors);
    // upstream's host fields, so that the struct and pk.write stay as they are
    let host = HostPkColumns {
        fixed_values: (0..n_fixed).map(|i| pk.download(PK_FIXED, PK_VALUES, i)).collect(),
        fixed_polys: (0..n_fixed).map(|i| pk.download(PK_FIXED, PK_COEFF, i)).collect(),
        fixed_cosets: (0..n_fixed).map(|i| pk.download(PK_FIXED, PK_EXTENDED, i)).collect(),
        permutations: (0..mapping.len() as u32).map(|i| pk.download(PK_PERMUTATION, PK_VALUES, i)).collect(),
        permutation_polys: (0..mapping.len() as u32).map(|i| pk.download(PK_PERMUTATION, PK_COEFF, i)).collect(),
        permutation_cosets: (0..mapping.len() as u32).map(|i| pk.download(PK_PERMUTATION, PK_EXTENDED, i)).collect(),
        l0: pk.download(PK_INDICATORS, PK_EXTENDED, 0),
        l_last: pk.download(PK_INDICATORS, PK_EXTENDED, 1),
        l_active_row: pk.download(PK_INDICATORS, PK_EXTENDED, 2),
    };
    (pk, host)
}

/// The host copies keygen_pk stores in `ProvingKey { fixed_values, fixed_polys, fixed_cosets, permutation: permutation::ProvingKey
/// { permutations, polys, cosets }, l0, l_last, l_active_row }`; the caller wraps each in `Polynomial` (domain.lagrange_from_vec /
/// coeff_from_vec / the extended equivalent; `[u64; 4]` is Fr's memory layout) and sets `pk.h2b_resident` to the handle.
pub struct HostPkColumns {
    pub fixed_values: Vec<Vec<[u64; 4]>>,
    pub fixed_polys: Vec<Vec<[u64; 4]>>,
    pub fixed_cosets: Vec<Vec<[u64; 4]>>,
    pub permutations: Vec<Vec<[u64; 4]>>,
    pub permutation_polys: Vec<Vec<[u64; 4]>>,
    pub permutation_cosets: Vec<Vec<[u64; 4]>>,
    pub l0: Vec<[u64; 4]>,
    pub l_last: Vec<[u64; 4]>,
    pub l_active_row: Vec<[u64; 4]>,
}

/// A ProvingKey from ProvingKey::read or from the CPU keygen: its Lagrange values registered once, on first use.
pub fn h2b_resident_of<'a>(cell: &'a std::cell::OnceCell<ResidentProvingKey>, dom: &KeygenDomain, fixed_values: &[&[[u64; 4]]],
                           permutations: &[&[[u64; 4]]], blinding_factors: u32) -> &'a ResidentProvingKey {
    cell.get_or_init(|| {
        let (layout, halo) = h2b_layout();
        let pk = ResidentProvingKey::new(dom, fixed_values.len() as u32, permutations.len() as u32, layout, halo);
        pk.put_lagrange(PK_FIXED, 0, fixed_values);
        pk.put_lagrange(PK_PERMUTATION, 0, permutations);
        pk.build_indicators(blinding_factors);
        pk
    })
}

// ---- halo2_proofs/src/plonk/evaluation.rs, Evaluator::evaluate_h (continuing evaluation_dropin.rs) --------------------------------
// The pointers evaluation_dropin.rs passed without saying where they come from now come from the handle (device `dev`):
//
//   let rpk = h2b_resident_of(&pk.h2b_resident, &dom, &fixed_values, &permutations, cs.blinding_factors() as u32);
//   let fixed: Vec<*const c_void> = (0..n_fixed).map(|i| rpk.column(dev, PK_FIXED, PK_EXTENDED, i).0 as *const c_void).collect();
//   let sigma_cosets: Vec<*const c_void> = (0..n_perm).map(|i| rpk.column(dev, PK_PERMUTATION, PK_EXTENDED, i).0 as *const c_void).collect();
//   let (d_l0, shard) = rpk.column(dev, PK_INDICATORS, PK_EXTENDED, 0);
//   let d_l_last = rpk.column(dev, PK_INDICATORS, PK_EXTENDED, 1).0;
//   let d_l_active_row = rpk.column(dev, PK_INDICATORS, PK_EXTENDED, 2).0;
//
// and the calls of evaluation_dropin.rs take them unchanged (with a row-sharded pk: the *_shard_dev entry points with `shard`).  The
// permutation product of create_proof reads sigma in Lagrange form (PK_PERMUTATION, PK_VALUES) and the opening the coefficient forms
// (PK_COEFF) the same way.  Nothing of the pk is uploaded per proof.
