// Written to spec, NOT compiled here (no cargo / rustc in the build image).  REPLACES the body of upstream's generic
// `impl<E: Engine + Debug> ParamsKZG<E> { pub fn setup<R: RngCore>(k: u32, rng: R) -> Self }` in the patched
// halo2_proofs/src/poly/kzg/commitment.rs (there is no second, Bn256-only `setup`: it would clash with the generic one).
// For E = Bn256 both G1 vectors are computed on the device by h2b_srs_setup and stay resident as the two registered base
// sets that commit / commit_lagrange use (the handle fields of evaluation_dropin.rs); G2 stays on the host with halo2curves.
// Any other engine runs upstream's body unchanged (`setup_generic`, the upstream code renamed).
//
// The RNG is consumed exactly as upstream consumes it -- one `E::Scalar::random(rng)` and nothing else -- so a seeded
// caller (the proof-parity harness, rust/harness) gets the same toxic waste, hence the same SRS and the same proofs, as
// with the upstream body.  To check against the fork when a machine has it: upstream v2023_02_02 draws
// `let s = <E::Scalar>::random(rng);` once, after `assert!(k <= E::Scalar::S)` and before any other use of `rng`.

impl<E: Engine + Debug> ParamsKZG<E> {
    pub fn setup<R: RngCore>(k: u32, rng: R) -> Self {
        if TypeId::of::<E>() != TypeId::of::<Bn256>() {
            return Self::setup_generic(k, rng);
        }
        // Largest root of unity exponent of the Engine is `2^E::Scalar::S`, so we can
        // only support FFTs of polynomials below degree `2^E::Scalar::S`.
        assert!(k <= E::Scalar::S);
        let n: u64 = 1 << k;
        let s = <E::Scalar>::random(rng);

        // E::Scalar == Fr: its Montgomery limbs are what h2b_srs_setup takes (the field is pub(crate) in halo2curves)
        let s_limbs: [u64; 4] = unsafe { std::mem::transmute_copy::<E::Scalar, [u64; 4]>(&s) };
        let (g, g_lagrange, handle_g, handle_g_lagrange) = h2b200_sys::srs_setup(k, &s_limbs);
        // E::G1Affine == G1Affine = x | y Montgomery limbs: element-wise, as arithmetic_dropin.rs converts results
        let to_affine = |v: Vec<[u64; 8]>| -> Vec<E::G1Affine> {
            v.iter().map(|p| unsafe { std::mem::transmute_copy::<[u64; 8], E::G1Affine>(p) }).collect()
        };
        let (g, g_lagrange) = (to_affine(g), to_affine(g_lagrange));

        let g2 = <E::G2Affine as PrimeCurveAffine>::generator();
        let s_g2 = (g2 * s).into();

        Self { k, n, g, g_lagrange, g2, s_g2, handle_g, handle_g_lagrange }
    }
}
