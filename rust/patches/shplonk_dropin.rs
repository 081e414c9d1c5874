// Written to spec, NOT compiled here (no cargo / rustc in the build image).  REPLACES the body of upstream's
// `impl<'params, E: Engine + Debug> Prover<'params, KZGCommitmentScheme<E>> for ProverSHPLONK<'params, E> { fn create_proof }` in the
// patched halo2_proofs/src/poly/kzg/multiopen/shplonk/prover.rs: apply_dropin.py puts
// `if TypeId::of::<E>() == TypeId::of::<Bn256>() { return self.create_proof_h2b(transcript, queries); }` at the top of upstream's
// `create_proof` and appends this inherent method.  Any other engine runs upstream's body unchanged.
//
// The transcript sees what upstream writes, in upstream's order: squeeze y, squeeze v, write h1, squeeze u, write h2.  The RNG is not
// touched (upstream's KZG ignores it and every blind).  Polynomials are identified by `ptr::eq`, as upstream's PolynomialPointer
// equality does, and passed to h2b_shplonk_begin as indices in first-appearance order; the session is released on every path by
// ShplonkSession's Drop.

impl<'params, E: Engine + Debug> ProverSHPLONK<'params, E> {
    fn create_proof_h2b<'com, Ch: EncodedChallenge<E::G1Affine>, T: TranscriptWrite<E::G1Affine, Ch>, I>(
        &self,
        transcript: &mut T,
        queries: I,
    ) -> io::Result<()>
    where
        I: IntoIterator<Item = ProverQuery<'com, E::G1Affine>> + Clone,
    {
        // E::Scalar == Fr and E::G1 == G1 (TypeId dispatch above): their Montgomery limbs are the C ABI's layout
        let limbs = |x: &E::Scalar| -> [u64; 4] { unsafe { std::mem::transmute_copy::<E::Scalar, [u64; 4]>(x) } };
        let mut polys: Vec<&'com Polynomial<E::Scalar, Coeff>> = Vec::new();
        let mut abi_queries = Vec::new();
        for q in queries.into_iter() {
            let index = match polys.iter().position(|p| std::ptr::eq(*p, q.poly)) {
                Some(i) => i,
                None => {
                    polys.push(q.poly);
                    polys.len() - 1
                }
            };
            abi_queries.push(h2b200_sys::h2b_opening_query { poly: index as u32, reserved: 0, point: limbs(&q.point) });
        }
        let slices: Vec<&[[u64; 4]]> = polys
            .iter()
            .map(|p| unsafe { std::slice::from_raw_parts(p.values.as_ptr() as *const [u64; 4], p.values.len()) })
            .collect();

        let y: ChallengeY<_> = transcript.squeeze_challenge_scalar();
        let v: ChallengeV<_> = transcript.squeeze_challenge_scalar();
        let (session, h1) = h2b200_sys::ShplonkSession::begin(&slices, &abi_queries, self.params.handle_g, &limbs(&*y), &limbs(&*v));
        let h1: E::G1 = unsafe { std::mem::transmute_copy::<[u64; 12], E::G1>(&h1) };
        transcript.write_point(h1.to_affine())?;
        let u: ChallengeU<_> = transcript.squeeze_challenge_scalar();
        let h2 = session.finish(&limbs(&*u));
        let h2: E::G1 = unsafe { std::mem::transmute_copy::<[u64; 12], E::G1>(&h2) };
        transcript.write_point(h2.to_affine())?;
        Ok(())
    }
}
