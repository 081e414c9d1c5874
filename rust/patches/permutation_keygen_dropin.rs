// Written to spec, NOT compiled here (no cargo / rustc in the build image).  Appended by rust/patches/apply_dropin.py to
// halo2_proofs/src/plonk/permutation/keygen.rs, which also inserts the dispatch lines at the top of the two methods:
//
//     pub(crate) fn build_vk<'params, C: CurveAffine, P: Params<'params, C>>(self, params: &P, domain: &EvaluationDomain<C::Scalar>, p: &Argument)
//         -> VerifyingKey<C> {
//         if TypeId::of::<C>() == TypeId::of::<G1Affine>() { if let Some(h) = params.h2b_g_lagrange_handle() { return self.build_vk_h2b(h, domain); } }
//         ... upstream's body, unchanged: every other curve, and params without a resident g_lagrange, run it ...
//     pub(crate) fn build_pk<'params, C: CurveAffine, P: Params<'params, C>>(self, params: &P, domain: &EvaluationDomain<C::Scalar>, p: &Argument)
//         -> ProvingKey<C> {
//         if TypeId::of::<C>() == TypeId::of::<G1Affine>() { return self.build_pk_h2b(domain); }
//         ...
//
// Where the g_lagrange handle comes from: build_vk only sees `P: Params`, so apply_dropin.py adds a defaulted method to the
// `Params` trait (halo2_proofs/src/poly/commitment.rs)
//
//     fn h2b_g_lagrange_handle(&self) -> Option<u64> { None }
//
// and overrides it in `impl Params for ParamsKZG<E>` (poly/kzg/commitment.rs) with `Some(self.handle_g_lagrange)` when
// TypeId::of::<E>() == TypeId::of::<Bn256>() -- the registered set the kzg drop-ins (evaluation_dropin.rs, kzg_setup_dropin.rs,
// kzg_downsize_dropin.rs) keep.  Every other Params keeps None and upstream's host path.
//
// The mapping: upstream's `mapping: Vec<Vec<(usize, usize)>>` goes to the C ABI as it sits in memory when `(usize, usize)` is
// two u64 with field 0 first, and is converted once otherwise (h2b200_sys::permutation_build_vk / build_pk); apply_dropin.py
// refuses a halo2_proofs whose Assembly holds another mapping type.  The l0 / l_blind / l_last block of keygen_pk is replaced by
// `keygen_indicators_h2b` below (plonk/keygen.rs), by the same TypeId dispatch.

pub(crate) fn h2b_domain<F: ff::PrimeField>(domain: &EvaluationDomain<F>) -> h2b200_sys::KeygenDomain {
    // F == halo2curves::bn256::Fr here (checked through TypeId by every caller): Montgomery limbs, plain old data
    let w = |x: &F| unsafe { std::mem::transmute_copy::<F, [u64; 4]>(x) };
    let n = F::from(1u64 << domain.k());
    let zeta = F::ZETA;
    h2b200_sys::KeygenDomain {
        k: domain.k(),
        extended_k: domain.extended_k(),
        omega: w(&domain.get_omega()),
        omega_inv: w(&domain.get_omega_inv()),
        ifft_divisor: w(&n.invert().unwrap()),
        extended_omega: w(&domain.get_extended_omega()),
        zeta_powers: [w(&F::ONE), w(&zeta), w(&zeta.square())],
    }
}

fn h2b_delta<F: ff::PrimeField>() -> [u64; 4] {
    unsafe { std::mem::transmute_copy::<F, [u64; 4]>(&F::DELTA) }
}

pub(crate) fn h2b_columns<F: Copy>(v: Vec<[u64; 4]>) -> Vec<F> {
    // F == Fr: 32 bytes of Montgomery limbs per element
    v.iter().map(|x| unsafe { std::mem::transmute_copy::<[u64; 4], F>(x) }).collect()
}

impl Assembly {
    fn build_vk_h2b<C: CurveAffine>(self, handle_g_lagrange: u64, domain: &EvaluationDomain<C::Scalar>) -> VerifyingKey<C> {
        let jac = h2b200_sys::permutation_build_vk(&self.mapping, &h2b_delta::<C::Scalar>(), &h2b_domain(domain), handle_g_lagrange);
        // C::Curve == G1: x | y | z Montgomery limbs (Jacobian), then to_affine as upstream does
        let commitments = jac.iter().map(|p| unsafe { std::mem::transmute_copy::<[u64; 12], C::Curve>(p) }.to_affine()).collect();
        VerifyingKey { commitments }
    }

    fn build_pk_h2b<C: CurveAffine>(self, domain: &EvaluationDomain<C::Scalar>) -> ProvingKey<C> {
        let (perms, polys, cosets) = h2b200_sys::permutation_build_pk(&self.mapping, &h2b_delta::<C::Scalar>(), &h2b_domain(domain));
        ProvingKey {
            permutations: perms.into_iter().map(|v| domain.lagrange_from_vec(h2b_columns(v))).collect(),
            polys: polys.into_iter().map(|v| domain.coeff_from_vec(h2b_columns(v))).collect(),
            cosets: cosets
                .into_iter()
                .map(|v| {
                    let mut e = domain.empty_extended();
                    e.values = h2b_columns(v);
                    e
                })
                .collect(),
        }
    }
}

// keygen_pk (plonk/keygen.rs): apply_dropin.py replaces upstream's block from `let mut l0 = vk.domain.empty_lagrange();` to the end
// of the `l_active_row` computation by
//     let (l0, l_last, l_active_row) = if TypeId::of::<C>() == TypeId::of::<G1Affine>() {
//         crate::plonk::permutation::keygen::keygen_indicators_h2b(&vk.domain, cs.blinding_factors())
//     } else { <upstream's block, unchanged, ending in (l0, l_last, l_active_row)> };
#[allow(clippy::type_complexity)]
pub(crate) fn keygen_indicators_h2b<F: ff::PrimeField>(
    domain: &EvaluationDomain<F>,
    blinding_factors: usize,
) -> (Polynomial<F, ExtendedLagrangeCoeff>, Polynomial<F, ExtendedLagrangeCoeff>, Polynomial<F, ExtendedLagrangeCoeff>) {
    let [l0, l_last, l_active] = h2b200_sys::keygen_lagrange_indicators(&h2b_domain(domain), blinding_factors as u32);
    let ext = |v: Vec<[u64; 4]>| {
        let mut e = domain.empty_extended();
        e.values = h2b_columns(v);
        e
    };
    (ext(l0), ext(l_last), ext(l_active))
}
