"""Text transforms that apply_dropin.py uses to wire rust/patches/mock_prover_dropin.rs into a halo2_proofs checkout.  Pure functions
on source text, so that they can be checked without a checkout; each one asserts what it relies on and stops instead of guessing.

  * patch_plonk(src)       src/plonk.rs: the `evaluation` module visible in the crate (dev.rs uses its GraphEvaluator and FlatGraph)
  * patch_evaluation(src)  src/plonk/evaluation.rs: appends `encode_source` and `FlatGraph` from evaluation_dropin.rs (the part
                           between its `use h2b200_sys` line and its commentary on evaluate_h), both visible in the crate
  * patch_dev(src)         src/dev.rs: the Fr dispatch at the top of `MockProver::verify_par`, `selector_errors_h2b` (upstream's own
                           region-check statement of `verify_at_rows_par`, cut out by bracket balance) and the drop-in itself
"""
import re

EVALUATION_MARKER = "// In `Evaluator::evaluate_h`"
DISPATCH = "if TypeId::of::<F>() == TypeId::of::<halo2curves::bn256::Fr>() { return self.verify_par_h2b(); }"


def statement_after(src: str, head: str) -> str:
    """the expression of the statement that starts with `head` (e.g. "let x =") up to its closing `;` at bracket depth 0.  String and
    char literals and comments are skipped, so a `;` or a bracket inside them does not end or unbalance the statement."""
    start = src.index(head) + len(head)
    depth, i = 0, start
    while i < len(src):
        c = src[i]
        if src.startswith("//", i):
            i = src.index("\n", i)
            continue
        if src.startswith("/*", i):
            i = src.index("*/", i) + 2
            continue
        if c == '"':
            i += 1
            while src[i] != '"':
                i += 2 if src[i] == "\\" else 1
        elif c == "'" and re.match(r"'(\\.|[^\\'])'", src[i:i + 4]):
            i = src.index("'", i + 1 + (src[i + 1] == "\\"))
        elif c in "([{":
            depth += 1
        elif c in ")]}":
            depth -= 1
            assert depth >= 0, "unbalanced brackets after %r" % head
        elif c == ";" and depth == 0:
            return src[start:i].strip()
        i += 1
    raise AssertionError("no end of the statement after %r" % head)


def patch_plonk(src: str) -> str:
    if re.search(r"\bpub(\([a-z]+\))? mod evaluation;", src):
        return src
    assert re.search(r"^mod evaluation;", src, re.M), "`mod evaluation;` not found in plonk.rs"
    return re.sub(r"^mod evaluation;", "pub(crate) mod evaluation;", src, count=1, flags=re.M)


def patch_evaluation(src: str, evaluation_dropin: str) -> str:
    if "struct FlatGraph" in src:
        return src
    head, sep, _ = evaluation_dropin.partition(EVALUATION_MARKER)
    assert sep, "evaluation_dropin.rs lost its %r marker" % EVALUATION_MARKER
    defs = head[head.index("use h2b200_sys"):]
    assert "pub(crate) fn encode_source" in defs and "pub struct FlatGraph" in defs and "impl FlatGraph" in defs
    return src + "\n// ---- libh2b200: the flat form of a GraphEvaluator (rust/patches/evaluation_dropin.rs) ----\n" + defs.rstrip() + "\n"


def patch_dev(src: str, mock_dropin: str) -> str:
    if "verify_par_h2b" in src:
        return src
    fn = re.search(r"\n    pub fn verify_par\(&self\) -> Result<\(\), Vec<VerifyFailure>> \{", src)
    assert fn, "MockProver::verify_par not found in dev.rs"
    at = src.index("fn verify_at_rows_par")
    region_check = statement_after(src[at:], "let selector_errors =")
    assert "self.regions" in region_check and "CellNotAssigned" in region_check, "verify_at_rows_par's region check not recognised"
    src = src[:fn.end()] + "\n        " + DISPATCH + src[fn.end():]
    uses = ["use std::any::TypeId;", "use crate::plonk::evaluation::{encode_source, FlatGraph, GraphEvaluator};"]
    first_use = re.search(r"^use ", src, re.M)
    assert first_use, "no `use` line in dev.rs"
    src = src[:first_use.start()] + "\n".join(u for u in uses if u not in src) + "\n" + src[first_use.start():]
    # the region check reads verify_at_rows_par's `n` and, where it filters by them, its gate rows: verify_par passes the usable rows
    helper = ("\nimpl<F: FieldExt> MockProver<F> {\n"
              "    /// verify_at_rows_par's region check (CellNotAssigned), as verify_par runs it\n"
              "    fn selector_errors_h2b(&self) -> Vec<VerifyFailure> {\n"
              "        let n = self.n as i32;\n"
              "        let gate_row_ids: Vec<usize> = self.usable_rows.clone().collect();\n"
              "        let _ = (&n, &gate_row_ids);\n"
              "        let selector_errors = " + region_check + ";\n"
              "        selector_errors.collect()\n"
              "    }\n}\n")
    return src + "\n// ---- libh2b200 drop-in (rust/patches/mock_prover_dropin.rs) ----" + helper + "\n" + mock_dropin + "\n"
