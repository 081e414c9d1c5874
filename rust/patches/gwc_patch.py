"""The text transform that apply_dropin.py uses to wire rust/patches/gwc_dropin.rs into a halo2_proofs checkout.  A pure function on
source text, so that it can be checked without a checkout; it asserts what it relies on and stops instead of guessing.

  * patch_gwc_prover(src, dropin)  src/poly/kzg/multiopen/gwc/prover.rs: the Bn256 dispatch at the top of `ProverGWC::create_proof`,
                                   the `use`s it needs, and the drop-in's `create_proof_h2b` appended.  Idempotent.
"""
import re

DISPATCH = "if TypeId::of::<E>() == TypeId::of::<Bn256>() { return self.create_proof_h2b(transcript, queries); }"
USES = ["use std::any::TypeId;", "use halo2curves::bn256::Bn256;", "use crate::poly::Coeff;"]
# upstream's signature, rustfmt's layout or one line: generics, parameters, return type, where clause, opening brace
SIGNATURE = (r"\n    fn create_proof<\s*'com,\s*Ch: EncodedChallenge<E::G1Affine>,\s*T: TranscriptWrite<E::G1Affine, Ch>,\s*R,\s*I,?\s*>"
             r"\(.*?\)\s*->\s*io::Result<\(\)>(?:\s*where[^{]*)?\{")


def patch_gwc_prover(src: str, dropin: str) -> str:
    if "create_proof_h2b" in src:
        return src
    heads = list(re.finditer(SIGNATURE, src, re.S))
    assert len(heads) == 1, "ProverGWC::create_proof: %d matches of its signature" % len(heads)
    assert "for ProverGWC<'params, E>" in src[:heads[0].start()], "create_proof is not in the Prover impl of ProverGWC"
    assert re.search(r"^use crate::poly::\{[^}]*\bPolynomial\b", src, re.M), "gwc/prover.rs does not import Polynomial from crate::poly"
    end = heads[0].end()
    src = src[:end] + "\n        " + DISPATCH + src[end:]
    for use in USES:
        if use not in src:
            src = use + "\n" + src
    return src + "\n// ---- libh2b200 drop-in (rust/patches/gwc_dropin.rs) ----\n" + dropin + "\n"
