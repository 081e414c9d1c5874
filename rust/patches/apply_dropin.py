#!/usr/bin/env python3
"""apply_dropin.py <path to a halo2_proofs crate> <path to this repository's rust/ directory>

Turns a checkout of halo2_proofs (PSE tag v2023_02_02 or axiom-crypto branch axiom/dev) into the GPU arm:
  * src/arithmetic.rs: the bodies of `best_multiexp` and `best_fft` are renamed to `*_generic` and the dispatching versions of
    rust/patches/arithmetic_dropin.rs are appended (public signatures unchanged);
  * src/poly/kzg/commitment.rs: a dispatch to `downsize_h2b` for Bn256 is inserted at the top of `fn downsize` and
    rust/patches/kzg_downsize_dropin.rs is appended (the method of the `Params` trait keeps its name and signature);
  * src/plonk/permutation/keygen.rs, src/plonk/keygen.rs, src/poly/commitment.rs, src/poly/kzg/commitment.rs: the permutation keygen
    drop-in (rust/patches/permutation_keygen_dropin.rs, whose header states the mechanism): G1Affine dispatches at the top of
    `Assembly::build_vk` / `build_pk` and around keygen_pk's l0 / l_blind / l_last block, and the defaulted
    `Params::h2b_g_lagrange_handle` that `ParamsKZG<Bn256>` overrides.  Each substitution is asserted, and so is upstream's
    `mapping: Vec<Vec<(usize, usize)>>` layout of `Assembly`;
  * src/plonk/circuit/compress_selectors.rs, src/plonk/circuit.rs, src/plonk/keygen.rs: the fixed-column keygen drop-in
    (rust/patches/fixed_keygen_dropin.rs): `process_h2b`, a copy of `ConstraintSystem::compress_selectors` that calls it, and G1Affine
    dispatches around keygen_vk's fixed commitments and keygen_pk's fixed values / polys / cosets.  Each substitution is asserted;
  * Cargo.toml: `h2b200-sys = { path = ".../rust/h2b200-sys" }` is added to [dependencies].
Idempotent.  Not run in the build container (no Rust sources of halo2_proofs are available there)."""
import pathlib
import re
import sys

crate, rust = pathlib.Path(sys.argv[1]), pathlib.Path(sys.argv[2]).resolve()
arith = crate / "src" / "arithmetic.rs"
src = arith.read_text()
if "h2b200_sys" not in src:
    src, n1 = re.subn(r"\bpub fn best_multiexp<", "pub fn best_multiexp_generic<", src, count=1)
    src, n2 = re.subn(r"\bpub fn best_fft<", "pub fn best_fft_generic<", src, count=1)
    assert n1 == 1 and n2 == 1, "best_multiexp / best_fft not found in %s" % arith
    dropin = (rust / "patches" / "arithmetic_dropin.rs").read_text()
    dropin = "\n".join(l for l in dropin.splitlines() if not l.startswith("use halo2curves::CurveAffine") and not l.startswith("use group::Group"))
    arith.write_text(src + "\n// ---- libh2b200 drop-in (rust/patches/arithmetic_dropin.rs) ----\n" + dropin + "\n")
kzg = crate / "src" / "poly" / "kzg" / "commitment.rs"
src = kzg.read_text()
if "downsize_h2b" not in src:
    src, n = re.subn(r"(\bfn downsize\(&mut self, k: u32\)\s*\{)",
                     r"\1\n        if TypeId::of::<E>() == TypeId::of::<Bn256>() { return self.downsize_h2b(k); }", src, count=1)
    assert n == 1, "fn downsize not found in %s" % kzg
    for use in ("use std::any::TypeId;", "use halo2curves::bn256::Bn256;"):
        if use not in src:
            src = use + "\n" + src
    kzg.write_text(src + "\n// ---- libh2b200 drop-in (rust/patches/kzg_downsize_dropin.rs) ----\n" + (rust / "patches" / "kzg_downsize_dropin.rs").read_text() + "\n")

def substitute(path, pattern, repl, what, flags=0):
    text = path.read_text()
    text, n = re.subn(pattern, repl, text, count=1, flags=flags)
    assert n == 1, "%s not found in %s" % (what, path)
    path.write_text(text)


def add_uses(path, uses):
    text = path.read_text()
    for use in uses:
        if use not in text:
            text = use + "\n" + text
    path.write_text(text)


perm_keygen = crate / "src" / "plonk" / "permutation" / "keygen.rs"
if "build_vk_h2b" not in perm_keygen.read_text():
    src = perm_keygen.read_text()
    assert re.search(r"\bmapping:\s*Vec<Vec<\(usize,\s*usize\)>>", src), \
        "%s: Assembly's mapping is not Vec<Vec<(usize, usize)>>; the shim must convert it (see permutation_keygen_dropin.rs)" % perm_keygen
    dispatch_vk = ("\\1\n        if TypeId::of::<C>() == TypeId::of::<G1Affine>() {\n"
                   "            if let Some(h) = params.h2b_g_lagrange_handle() { return self.build_vk_h2b(h, domain); }\n        }")
    substitute(perm_keygen, r"(\bpub\(crate\) fn build_vk<[^{]*?\)\s*->\s*VerifyingKey<C>\s*\{)", dispatch_vk, "Assembly::build_vk", re.S)
    substitute(perm_keygen, r"(\bpub\(crate\) fn build_pk<[^{]*?\)\s*->\s*ProvingKey<C>\s*\{)",
               "\\1\n        if TypeId::of::<C>() == TypeId::of::<G1Affine>() { return self.build_pk_h2b(domain); }", "Assembly::build_pk", re.S)
    add_uses(perm_keygen, ["use std::any::TypeId;", "use halo2curves::bn256::G1Affine;",
                           "use crate::poly::{Coeff, ExtendedLagrangeCoeff, LagrangeCoeff, Polynomial};"])
    perm_keygen.write_text(perm_keygen.read_text() + "\n// ---- libh2b200 drop-in (rust/patches/permutation_keygen_dropin.rs) ----\n"
                           + (rust / "patches" / "permutation_keygen_dropin.rs").read_text() + "\n")
keygen = crate / "src" / "plonk" / "keygen.rs"
if "keygen_indicators_h2b" not in keygen.read_text():
    substitute(keygen, r"(let mut l0 = vk\.domain\.empty_lagrange\(\);.*?\*value = one - \(l_last\[idx\] \+ l_blind\[idx\]\);\s*\}\s*\}\);)",
               "let (l0, l_last, l_active_row) = if TypeId::of::<C>() == TypeId::of::<G1Affine>() {\n"
               "        crate::plonk::permutation::keygen::keygen_indicators_h2b(&vk.domain, cs.blinding_factors())\n"
               "    } else {\n    \\1\n    (l0, l_last, l_active_row)\n    };", "keygen_pk's l0 / l_blind / l_last block", re.S)
    add_uses(keygen, ["use std::any::TypeId;", "use halo2curves::bn256::G1Affine;"])
params_trait = crate / "src" / "poly" / "commitment.rs"
if "h2b_g_lagrange_handle" not in params_trait.read_text():
    substitute(params_trait, r"(\bpub trait Params<'params, C: CurveAffine>[^{]*\{)",
               "\\1\n    /// the registered g_lagrange set of libh2b200 (Bn256 KZG params only)\n    fn h2b_g_lagrange_handle(&self) -> Option<u64> { None }",
               "trait Params", re.S)
if "fn h2b_g_lagrange_handle" not in kzg.read_text():
    substitute(kzg, r"(\bimpl<'params, E: Engine \+ Debug> Params<'params, E::G1Affine> for ParamsKZG<E>[^{]*\{)",
               "\\1\n    fn h2b_g_lagrange_handle(&self) -> Option<u64> {\n"
               "        if TypeId::of::<E>() == TypeId::of::<Bn256>() { Some(self.handle_g_lagrange) } else { None }\n    }",
               "impl Params for ParamsKZG", re.S)
# compress_selectors and the fixed columns of keygen_vk / keygen_pk (rust/patches/fixed_keygen_dropin.rs, whose header states the mechanism)
fixed_dropin = (rust / "patches" / "fixed_keygen_dropin.rs").read_text()
process_part, keygen_part = fixed_dropin.split("// ---- keygen.rs ----", 1)
compress = crate / "src" / "plonk" / "circuit" / "compress_selectors.rs"
if "process_h2b" not in compress.read_text():
    assert re.search(r"\bpub fn process<F: FieldExt, E>\(", compress.read_text()), "compress_selectors::process not found in %s" % compress
    compress.write_text(compress.read_text() + "\n// ---- libh2b200 drop-in (rust/patches/fixed_keygen_dropin.rs) ----\n" + process_part + "\n")
circuit = crate / "src" / "plonk" / "circuit.rs"
if "compress_selectors_h2b" not in circuit.read_text():
    text = circuit.read_text()
    m = re.search(r"\n(    pub\(crate\) fn compress_selectors\(mut self, selectors: Vec<Vec<bool>>\) -> \(Self, Vec<Vec<F>>\) \{.*?\n    \})\n", text, re.S)
    assert m, "ConstraintSystem::compress_selectors not found in %s" % circuit
    body = m.group(1)
    assert body.count("compress_selectors::process(") == 1, "compress_selectors does not call process exactly once"
    copy = body.replace("fn compress_selectors(", "fn compress_selectors_h2b(", 1).replace("-> (Self, Vec<Vec<F>>)", "-> (Self, h2b200_sys::SelectorAssignment)", 1)
    copy = copy.replace("compress_selectors::process(", "compress_selectors::process_h2b(", 1)
    circuit.write_text(text[:m.end(1)] + "\n\n    // libh2b200: upstream's body above with process -> process_h2b (rust/patches/fixed_keygen_dropin.rs)\n" + copy + text[m.end(1):])
if "fixed_keygen_h2b" not in keygen.read_text():
    # keygen_vk: the assignment instead of the filled columns, and the fixed commitments from the device
    substitute(keygen, r"(let \(cs, selector_polys\) = cs\.compress_selectors\(assembly\.selectors\);\s*fixed\.extend\(\s*selector_polys\s*\.into_iter\(\)\s*"
               r"\.map\(\|poly\| domain\.lagrange_from_vec\(poly\)\),?\s*\);)",
               "let h2b_handle = if TypeId::of::<C>() == TypeId::of::<G1Affine>() { params.h2b_g_lagrange_handle() } else { None };\n"
               "    let (cs, h2b_fixed_commitments) = if let Some(h) = h2b_handle {\n"
               "        let (cs, assignment) = cs.compress_selectors_h2b(assembly.selectors.clone());\n"
               "        let com = fixed_commitments_h2b::<C>(&fixed, &assembly.selectors, &assignment, params.k(), h);\n"
               "        (cs, Some(com))\n"
               "    } else {\n    \\1\n    (cs, None)\n    };", "keygen_vk's compress_selectors", re.S)
    substitute(keygen, r"(let fixed_commitments = )(fixed\s*\.iter\(\)\s*\.map\(\|poly\| params\.commit_lagrange\(poly, Blind::default\(\)\)\.to_affine\(\)\)\s*\.collect\(\));",
               "\\1h2b_fixed_commitments.unwrap_or_else(|| \\2);", "keygen_vk's fixed_commitments", re.S)
    # keygen_pk: fixed_values, fixed_polys and fixed_cosets from the device
    substitute(keygen, r"(let \(cs, selector_polys\) = cs\.compress_selectors\(assembly\.selectors\.clone\(\)\);\s*fixed\.extend\(\s*selector_polys\s*\.into_iter\(\)\s*"
               r"\.map\(\|poly\| vk\.domain\.lagrange_from_vec\(poly\)\),?\s*\);\s*"
               r"let fixed_polys: Vec<_> = fixed\s*\.iter\(\)\s*\.map\(\|poly\| vk\.domain\.lagrange_to_coeff\(poly\.clone\(\)\)\)\s*\.collect\(\);\s*"
               r"let fixed_cosets = fixed_polys\s*\.iter\(\)\s*\.map\(\|poly\| vk\.domain\.coeff_to_extended\(poly\.clone\(\)\)\)\s*\.collect\(\);)",
               "let (cs, fixed, fixed_polys, fixed_cosets) = if TypeId::of::<C>() == TypeId::of::<G1Affine>() {\n"
               "        let (cs, assignment) = cs.compress_selectors_h2b(assembly.selectors.clone());\n"
               "        let (fixed, fixed_polys, fixed_cosets) = fixed_keygen_h2b(fixed, &assembly.selectors, &assignment, &vk.domain);\n"
               "        (cs, fixed, fixed_polys, fixed_cosets)\n"
               "    } else {\n    \\1\n    (cs, fixed, fixed_polys, fixed_cosets)\n    };", "keygen_pk's fixed columns", re.S)
    keygen.write_text(keygen.read_text() + "\n// ---- libh2b200 drop-in (rust/patches/fixed_keygen_dropin.rs) ----\n" + keygen_part + "\n")
# ProverSHPLONK::create_proof (rust/patches/shplonk_dropin.rs, whose header states the mechanism)
shplonk = crate / "src" / "poly" / "kzg" / "multiopen" / "shplonk" / "prover.rs"
if "create_proof_h2b" not in shplonk.read_text():
    m = re.search(r"(\n    fn create_proof<'com, Ch: EncodedChallenge<E::G1Affine>, T: TranscriptWrite<E::G1Affine, Ch>, R, I>\((.*?)\)\s*->\s*io::Result<\(\)>(.*?)\{)",
                  shplonk.read_text(), re.S)
    assert m, "ProverSHPLONK::create_proof not found in %s" % shplonk
    substitute(shplonk, re.escape(m.group(1)), lambda _: m.group(1) + "\n        if TypeId::of::<E>() == TypeId::of::<Bn256>() { return self.create_proof_h2b(transcript, queries); }",
               "ProverSHPLONK::create_proof", re.S)
    add_uses(shplonk, ["use std::any::TypeId;", "use halo2curves::bn256::Bn256;", "use crate::poly::{Coeff, Polynomial};"])
    shplonk.write_text(shplonk.read_text() + "\n// ---- libh2b200 drop-in (rust/patches/shplonk_dropin.rs) ----\n" + (rust / "patches" / "shplonk_dropin.rs").read_text() + "\n")
toml = crate / "Cargo.toml"
t = toml.read_text()
if "h2b200-sys" not in t:
    t = t.replace("[dependencies]", '[dependencies]\nh2b200-sys = { path = "%s" }' % (rust / "h2b200-sys"), 1)
    toml.write_text(t)
print("patched", crate)
