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
toml = crate / "Cargo.toml"
t = toml.read_text()
if "h2b200-sys" not in t:
    t = t.replace("[dependencies]", '[dependencies]\nh2b200-sys = { path = "%s" }' % (rust / "h2b200-sys"), 1)
    toml.write_text(t)
print("patched", crate)
