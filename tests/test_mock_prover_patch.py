"""CPU: the text transforms that wire rust/patches/mock_prover_dropin.rs into halo2_proofs (rust/patches/mock_prover_patch.py), run on
excerpts laid out as PSE v2023_02_02's src/dev.rs, src/plonk.rs and src/plonk/evaluation.rs (restated from recollection, not copied:
the checkout is not vendored).  What they pin is what the transforms rely on: the whole region-check statement is carried over even
though its closures hold inner `;`-terminated statements and its comment comes before it, the helper defines the `n` it reads,
`FlatGraph` and `encode_source` reach evaluation.rs and are visible from dev.rs, and every transform is idempotent."""
import os
import re
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust", "patches"))

import mock_prover_patch as mpp  # noqa: E402

DEV_RS = '''use std::collections::HashMap;
use std::iter;

use crate::plonk::Expression;

impl<F: FieldExt> MockProver<F> {
    pub fn verify_at_rows_par<I: Clone + Iterator<Item = usize>>(
        &self,
        gate_row_ids: I,
        lookup_input_row_ids: I,
    ) -> Result<(), Vec<VerifyFailure>> {
        let n = self.n as i32;

        let gate_row_ids = gate_row_ids.collect::<Vec<_>>();
        let lookup_input_row_ids = lookup_input_row_ids.collect::<Vec<_>>();

        // Check that within each region, all cells used in instantiated gates have been
        // assigned to.
        let selector_errors = self.regions.iter().enumerate().flat_map(|(r_i, r)| {
            r.enabled_selectors.iter().flat_map(move |(selector, at)| {
                // Find the gates enabled by this selector
                self.cs
                    .gates
                    .iter()
                    // Assume that if a queried selector is enabled, the user wants to use the
                    // corresponding gate in some way.
                    .filter(move |g| g.queried_selectors().contains(selector))
                    .enumerate()
                    .flat_map(move |(gate_index, gate)| {
                        at.iter().flat_map(move |selector_row| {
                            // Selectors are queried with no rotation.
                            let gate_row = *selector_row as i32;

                            gate.queried_cells().iter().filter_map(move |cell| {
                                // Determine where this cell should have been assigned.
                                let cell_row = ((gate_row + n + cell.rotation.0) % n) as usize;

                                // Check that it was assigned!
                                if r.cells.get(&(cell.column, cell_row)).is_some() {
                                    None
                                } else {
                                    Some(VerifyFailure::CellNotAssigned {
                                        gate: (gate_index, gate.name()).into(),
                                        region: (r_i, r.name.clone()).into(),
                                        gate_offset: *selector_row,
                                        column: cell.column,
                                        offset: cell_row as isize - r.rows.unwrap().0 as isize,
                                    })
                                }
                            })
                        })
                    })
            })
        });

        let gate_errors = self.cs.gates.iter().enumerate().flat_map(|(gate_index, gate)| { iter::empty() });
        let mut errors: Vec<_> = iter::empty().chain(selector_errors).chain(gate_errors).collect();
        if errors.is_empty() { Ok(()) } else { Err(errors) }
    }

    pub fn verify_par(&self) -> Result<(), Vec<VerifyFailure>> {
        self.verify_at_rows_par(self.usable_rows.clone(), self.usable_rows.clone())
    }
}
'''

PLONK_RS = "mod circuit;\nmod error;\nmod evaluation;\nmod keygen;\n\npub use circuit::*;\n"
EVALUATION_RS = "use crate::plonk::Expression;\n\npub struct GraphEvaluator<C: CurveAffine> { pub constants: Vec<C::ScalarExt> }\n"


def read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def balanced(text):
    stack, pairs = [], {")": "(", "]": "[", "}": "{"}
    for c in re.sub(r'//[^\n]*|"(\\.|[^"\\])*"', "", text):
        if c in "([{":
            stack.append(c)
        elif c in pairs:
            if not stack or stack.pop() != pairs[c]:
                return False
    return not stack


def test_dev_rs_gets_the_dispatch_and_the_whole_region_check():
    out = mpp.patch_dev(DEV_RS, read("rust", "patches", "mock_prover_dropin.rs"))
    verify_par = out[out.index("pub fn verify_par(&self)"):]
    assert verify_par.splitlines()[1].strip() == mpp.DISPATCH
    start = out.index("impl<F: FieldExt> MockProver<F> {\n    /// verify_at_rows_par's region check")
    helper = out[start:out.index("\n}\n", start) + 2]
    assert mpp.statement_after(DEV_RS, "let selector_errors =") in helper
    assert "let cell_row = ((gate_row + n + cell.rotation.0) % n) as usize;" in helper
    assert "let n = self.n as i32;" in helper and balanced(helper)
    assert "use crate::plonk::evaluation::{encode_source, FlatGraph, GraphEvaluator};" in out and "use std::any::TypeId;" in out
    assert balanced(out)
    assert mpp.patch_dev(out, "") == out


def test_region_check_statement_is_cut_by_bracket_balance():
    region = mpp.statement_after(DEV_RS, "let selector_errors =")
    assert region.startswith("self.regions.iter()") and region.endswith("})") and balanced(region)
    assert "offset: cell_row as isize - r.rows.unwrap().0 as isize," in region
    with pytest.raises(AssertionError):
        mpp.patch_dev(DEV_RS.replace("CellNotAssigned", "Other"), "")


def test_statement_after_skips_literals_and_comments():
    src = 'let x = f(";", \'}\', /* ) */ g(a; b)) // ;\n + 1;\nlet y = 2;'
    assert mpp.statement_after(src, "let x =") == 'f(";", \'}\', /* ) */ g(a; b)) // ;\n + 1'


def test_evaluation_and_module_visibility():
    ev = mpp.patch_evaluation(EVALUATION_RS, read("rust", "patches", "evaluation_dropin.rs"))
    assert "pub(crate) fn encode_source(" in ev and "pub struct FlatGraph" in ev and "impl FlatGraph" in ev
    assert "Evaluator::evaluate_h" not in ev and balanced(ev)
    assert mpp.patch_evaluation(ev, "") == ev
    plonk = mpp.patch_plonk(PLONK_RS)
    assert "pub(crate) mod evaluation;" in plonk and mpp.patch_plonk(plonk) == plonk
    with pytest.raises(AssertionError):
        mpp.patch_plonk("mod circuit;\n")


def test_apply_dropin_calls_the_transforms():
    src = read("rust", "patches", "apply_dropin.py")
    for name in ("patch_plonk", "patch_evaluation", "patch_dev"):
        assert "mpp.%s" % name in src
    assert "dedup_by" in read("rust", "patches", "mock_prover_dropin.rs")
