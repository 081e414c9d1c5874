// Written to spec, NOT compiled here (no cargo / rustc in the build image).  `downsize` is a method of upstream's
// `impl<'params, E: Engine + Debug> Params<'params, E::G1Affine> for ParamsKZG<E>` in halo2_proofs/src/poly/kzg/commitment.rs
// and cannot be renamed, so rust/patches/apply_dropin.py inserts one dispatch line at the top of its body:
//
//     fn downsize(&mut self, k: u32) {
//         if TypeId::of::<E>() == TypeId::of::<Bn256>() { return self.downsize_h2b(k); }
//         ... upstream's body, unchanged: every other engine runs it ...
//
// and appends this inherent method.  For E = Bn256 the g_lagrange of the 2^k-point prefix of g is computed on the device by
// h2b_srs_downsize (g_to_lagrange as a G1 NTT) from the resident g of this params' registered set; both vectors become new
// registered sets (the handle fields of evaluation_dropin.rs), the old ones are given back.  g2 and s_g2 are unchanged, as
// upstream leaves them.

impl<E: Engine + Debug> ParamsKZG<E> {
    fn downsize_h2b(&mut self, k: u32) {
        assert!(k <= self.k);
        let (g_lagrange, handle_g, handle_g_lagrange) = h2b200_sys::srs_downsize(self.handle_g, k);
        unsafe {
            h2b200_sys::h2b_unregister_bases(self.handle_g);
            h2b200_sys::h2b_unregister_bases(self.handle_g_lagrange);
        }
        self.k = k;
        self.n = 1 << k;
        self.g.truncate(self.n as usize);
        // E::G1Affine == G1Affine = x | y Montgomery limbs: element-wise, as arithmetic_dropin.rs converts results
        self.g_lagrange = g_lagrange.iter().map(|p| unsafe { std::mem::transmute_copy::<[u64; 8], E::G1Affine>(p) }).collect();
        self.handle_g = handle_g;
        self.handle_g_lagrange = handle_g_lagrange;
    }
}
