// Written to spec, NOT compiled here (no cargo / rustc in the build image).  Appended by rust/patches/apply_dropin.py to
// halo2_proofs/src/plonk/circuit/compress_selectors.rs (`process_h2b`) and to src/plonk/keygen.rs (`fixed_keygen_h2b`).
//
// compress_selectors: apply_dropin.py copies upstream's `ConstraintSystem::compress_selectors` (plonk/circuit.rs) to
// `compress_selectors_h2b`, with only the call `compress_selectors::process(` renamed to `compress_selectors::process_h2b(` and the
// return type `(Self, Vec<Vec<F>>)` changed to `(Self, h2b200_sys::SelectorAssignment)`.  process_h2b allocates the fixed columns
// through the caller's closure in process's order and builds the same substitution expressions, so the new fixed columns, the
// substituted gates and therefore the VK's pinned representation come from upstream's own code; it returns the assignment
// (combination and root per selector) in place of the filled columns.  The exclusion matrix comes from the device.
//
// keygen_vk / keygen_pk: apply_dropin.py wraps upstream's
//     let (cs, selector_polys) = cs.compress_selectors(<selectors>);
//     fixed.extend(selector_polys.into_iter().map(|poly| <domain>.lagrange_from_vec(poly)));
// and the fixed commitment / fixed_polys / fixed_cosets statements in
//     if TypeId::of::<C>() == TypeId::of::<G1Affine>() { if let Some(h) = params.h2b_g_lagrange_handle() { ... fixed_keygen_h2b ... } }
// as permutation_keygen_dropin.rs does; assembly.selectors (Vec<Vec<bool>>) is passed as it sits in memory.

// ---- compress_selectors.rs -----------------------------------------------------------------------------------------------------
pub fn process_h2b<F: FieldExt, E>(
    mut selectors: Vec<SelectorDescription>,
    max_degree: usize,
    mut allocate_fixed_column: E,
) -> (h2b200_sys::SelectorAssignment, Vec<SelectorAssignment<F>>)
where
    E: FnMut() -> Expression<F>,
{
    let total = selectors.len();
    let mut assignment = h2b200_sys::SelectorAssignment { combination_of: vec![0; total], root_of: vec![0; total], n_combinations: 0 };
    let mut selector_assignments = vec![];
    if selectors.is_empty() {
        return (assignment, selector_assignments);
    }
    let k = selectors[0].activations.len().trailing_zeros();
    // degree-0 selectors first, each in a column of its own (root 1), in selector order
    selectors.retain(|selector| {
        if selector.max_degree != 0 {
            return true;
        }
        let expression = allocate_fixed_column();
        assignment.combination_of[selector.selector] = assignment.n_combinations;
        assignment.root_of[selector.selector] = 1;
        selector_assignments.push(SelectorAssignment { selector: selector.selector, combination_index: assignment.n_combinations as usize, expression });
        assignment.n_combinations += 1;
        false
    });
    let activations: Vec<Vec<bool>> = selectors.iter().map(|s| s.activations.clone()).collect();
    let exclusion = if activations.is_empty() { vec![] } else { h2b200_sys::selector_exclusion(&activations, k) };
    let mut added = vec![false; selectors.len()];
    for (i, selector) in selectors.iter().enumerate() {
        if added[i] {
            continue;
        }
        added[i] = true;
        assert!(selector.max_degree <= max_degree);
        let mut d = selector.max_degree - 1;
        let mut combination = vec![selector];
        let mut combination_added = vec![i];
        'try_selectors: for (j, selector) in selectors.iter().enumerate().skip(i + 1) {
            if d + combination.len() == max_degree {
                break 'try_selectors;
            }
            if added[j] {
                continue 'try_selectors;
            }
            for &i in combination_added.iter() {
                if exclusion[j][i] {
                    continue 'try_selectors;
                }
            }
            let new_d = std::cmp::max(d, selector.max_degree - 1);
            if new_d + combination.len() + 1 > max_degree {
                continue 'try_selectors;
            }
            d = new_d;
            combination.push(selector);
            combination_added.push(j);
            added[j] = true;
        }
        let combination_len = combination.len();
        let combination_index = assignment.n_combinations as usize;
        let query = allocate_fixed_column();
        let mut assigned_root = F::one();
        for (t, selector) in combination.iter().enumerate() {
            let mut expression = query.clone();
            let mut root = F::one();
            for _ in 0..combination_len {
                if root != assigned_root {
                    expression = expression * (Expression::Constant(root) - query.clone());
                }
                root += F::one();
            }
            assigned_root += F::one();
            assignment.combination_of[selector.selector] = combination_index as u32;
            assignment.root_of[selector.selector] = t as u32 + 1;
            selector_assignments.push(SelectorAssignment { selector: selector.selector, combination_index, expression });
        }
        assignment.n_combinations += 1;
    }
    (assignment, selector_assignments)
}

// ---- keygen.rs ----------------------------------------------------------------------------------------------------------------------
// F == Fr (checked through TypeId by every caller): Montgomery limbs, plain old data
fn h2b_fixed_rows<F>(fixed: &[Polynomial<F, LagrangeCoeff>]) -> Vec<&[[u64; 4]]> {
    fixed.iter().map(|p| unsafe { std::slice::from_raw_parts(p.values.as_ptr() as *const [u64; 4], p.values.len()) }).collect()
}

/// keygen_vk's fixed_commitments: the fixed columns (after batch_invert_assigned), then the combination columns
pub(crate) fn fixed_commitments_h2b<C: CurveAffine>(
    fixed: &[Polynomial<C::Scalar, LagrangeCoeff>],
    selectors: &[Vec<bool>],
    assignment: &h2b200_sys::SelectorAssignment,
    k: u32,
    handle_g_lagrange: u64,
) -> Vec<C> {
    let jac = h2b200_sys::keygen_fixed_build_vk(&h2b_fixed_rows(fixed), selectors, assignment, k, handle_g_lagrange);
    jac.iter().map(|p| unsafe { std::mem::transmute_copy::<[u64; 12], C::Curve>(p) }.to_affine()).collect()
}

/// keygen_pk's fixed_values (the caller's fixed columns followed by the combination columns), fixed_polys and fixed_cosets
#[allow(clippy::type_complexity)]
pub(crate) fn fixed_keygen_h2b<F: ff::PrimeField>(
    mut fixed: Vec<Polynomial<F, LagrangeCoeff>>,
    selectors: &[Vec<bool>],
    assignment: &h2b200_sys::SelectorAssignment,
    domain: &EvaluationDomain<F>,
) -> (Vec<Polynomial<F, LagrangeCoeff>>, Vec<Polynomial<F, Coeff>>, Vec<Polynomial<F, ExtendedLagrangeCoeff>>) {
    let (values, polys, cosets) =
        h2b200_sys::keygen_fixed_build_pk(&h2b_fixed_rows(&fixed), selectors, assignment, &crate::plonk::permutation::keygen::h2b_domain(domain));
    fixed.extend(values.into_iter().map(|v| domain.lagrange_from_vec(crate::plonk::permutation::keygen::h2b_columns(v))));
    let polys = polys.into_iter().map(|v| domain.coeff_from_vec(crate::plonk::permutation::keygen::h2b_columns(v))).collect();
    let cosets = cosets
        .into_iter()
        .map(|v| {
            let mut e = domain.empty_extended();
            e.values = crate::plonk::permutation::keygen::h2b_columns(v);
            e
        })
        .collect();
    (fixed, polys, cosets)
}
