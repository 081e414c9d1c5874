#!/usr/bin/env python3
"""apply_dropin.py <path to a halo2_proofs crate> <path to this repository's rust/ directory>

Turns a checkout of halo2_proofs (PSE tag v2023_02_02 or axiom-crypto branch axiom/dev) into the GPU arm:
  * src/arithmetic.rs: the bodies of `best_multiexp` and `best_fft` are renamed to `*_generic` and the dispatching versions of
    rust/patches/arithmetic_dropin.rs are appended (public signatures unchanged);
  * src/poly/kzg/commitment.rs: a dispatch to `downsize_h2b` for Bn256 is inserted at the top of `fn downsize` and
    rust/patches/kzg_downsize_dropin.rs is appended (the method of the `Params` trait keeps its name and signature);
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
toml = crate / "Cargo.toml"
t = toml.read_text()
if "h2b200-sys" not in t:
    t = t.replace("[dependencies]", '[dependencies]\nh2b200-sys = { path = "%s" }' % (rust / "h2b200-sys"), 1)
    toml.write_text(t)
print("patched", crate)
