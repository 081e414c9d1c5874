// Written to spec, NOT compiled here (no cargo / rustc in the build image).  REPLACES the gate, lookup and permutation loops of
// `MockProver::verify_par` in the patched halo2_proofs/src/dev.rs for F == Fr:
//   * PSE v2023_02_02: `verify_par` calls `verify_at_rows_par(self.usable_rows.clone(), self.usable_rows.clone())`, whose
//     `gate_errors`, `lookup_errors` and `perm_errors` are the three loops replaced here; `selector_errors` (the region checks)
//     stays.  apply_dropin.py (through mock_prover_patch.py) copies upstream's whole `let selector_errors = ...;` statement of
//     `verify_at_rows_par`, cut out by bracket balance, into `fn selector_errors_h2b(&self)`, which defines the `n` and the gate rows
//     (the usable rows, as verify_par passes them) it reads; puts
//     `if TypeId::of::<F>() == TypeId::of::<Fr>() { return self.verify_par_h2b(); }` at the top of `verify_par`, so `verify` /
//     `assert_satisfied` (which call it) take the same path; appends `encode_source` and `FlatGraph` (evaluation_dropin.rs) to
//     plonk/evaluation.rs and makes that module visible in the crate.
//   * axiom/dev: believed to share these loops under the same names; apply_dropin.py asserts each pattern it patches and stops on a
//     fork where one is missing instead of guessing.
// `verify_at_rows` / `verify_at_rows_par` with caller-chosen rows keep upstream's code.
//
// The shim flattens `CellValue<Fr>` into Montgomery words plus one assigned bit per cell (Poison rows are implied by usable_rows),
// compiles the gates and lookups with upstream's own `GraphEvaluator` (one root per polynomial; FlatGraph from
// evaluation_dropin.rs), and maps each record back to `VerifyFailure` with upstream's `FailureLocation::find_expressions` /
// `FailureLocation::find` and the same constructors `verify_at_rows_par` uses.  Lookup failures arrive by (lookup, row); they are
// re-sorted here by (input tuple, row) with upstream's own `load` / `Value` ordering, which touches only the failing rows.

impl<F: FieldExt> MockProver<F> {
    /// `load` of verify_at_rows_par's lookup loop: an expression's Value at one row
    fn load_value_h2b(&self, e: &Expression<F>, row: usize) -> Value<F> {
        let n = self.n as i32;
        let at = |rot: Rotation| ((row as i32 + n + rot.0) % n) as usize;
        e.evaluate_lazy(
            &|scalar| Value::Real(scalar),
            &|_| panic!("virtual selectors are removed during optimization"),
            &|query| self.fixed[query.column_index][at(query.rotation)].into(),
            &|query| self.advice[query.column_index][at(query.rotation)].into(),
            &|query| Value::Real(self.instance[query.column_index][at(query.rotation)].value()),
            &|challenge| Value::Real(self.challenges[challenge.index()]),
            &|a| -a,
            &|a, b| a + b,
            &|a, b| a * b,
            &|a, scalar| a * scalar,
            &Value::Real(F::zero()),
        )
    }

    fn verify_par_h2b(&self) -> Result<(), Vec<VerifyFailure>> {
        use h2b200_sys::*;
        // F == Fr (TypeId dispatch above): every F below is an Fr and its limbs are the C ABI's Montgomery words
        let limbs = |x: &F| -> [u64; 4] { unsafe { std::mem::transmute_copy::<F, [u64; 4]>(x) } };
        let n = self.n as usize;
        let cell_words = |col: &[CellValue<F>]| -> (Vec<[u64; 4]>, Vec<u8>) {
            let mut words = vec![[0u64; 4]; n];
            let mut bits = vec![0u8; (n + 7) / 8];
            for (r, c) in col.iter().enumerate() {
                if let CellValue::Assigned(v) = c {
                    words[r] = limbs(v);
                    bits[r / 8] |= 1 << (r % 8);
                }
            }
            (words, bits)
        };
        let fixed: Vec<_> = self.fixed.iter().map(|c| cell_words(c)).collect();
        let advice: Vec<_> = self.advice.iter().map(|c| cell_words(c)).collect();
        let instance: Vec<Vec<[u64; 4]>> = self.instance.iter().map(|c| c.iter().map(|v| limbs(&v.value())).collect()).collect();
        let challenges: Vec<[u64; 4]> = self.challenges.iter().map(limbs).collect();

        // gates: one GraphEvaluator, a root per polynomial in (gate, poly) order
        let mut gates = GraphEvaluator::<halo2curves::bn256::G1Affine>::default();
        let as_fr = |e: &Expression<F>| -> &Expression<halo2curves::bn256::Fr> { unsafe { &*(e as *const Expression<F> as *const _) } };
        let mut roots = Vec::new();
        for (g, gate) in self.cs.gates.iter().enumerate() {
            for (p, poly) in gate.polynomials().iter().enumerate() {
                let v = gates.add_expression(as_fr(poly));
                roots.push(h2b_mock_root { gate: g as u32, poly: p as u32, value: encode_source(&v) });
            }
        }
        let flat_gates = FlatGraph::new(&gates);
        let ffi_gates = flat_gates.as_ffi();
        // lookups: a graph per lookup with its m input and m table roots
        let lookups: Vec<(FlatGraph, Vec<h2b_value_source>, Vec<h2b_value_source>)> = self.cs.lookups.iter().map(|lookup| {
            let mut g = GraphEvaluator::<halo2curves::bn256::G1Affine>::default();
            let ins = lookup.input_expressions.iter().map(|e| encode_source(&g.add_expression(as_fr(e)))).collect();
            let tbs = lookup.table_expressions.iter().map(|e| encode_source(&g.add_expression(as_fr(e)))).collect();
            (FlatGraph::new(&g), ins, tbs)
        }).collect();
        let ffi_lookups: Vec<h2b_mock_lookup> = lookups.iter().map(|(g, ins, tbs)| {
            h2b_mock_lookup { graph: g.as_ffi(), inputs: ins.as_ptr(), tables: tbs.as_ptr(), m: ins.len() as u32 }
        }).collect();
        // the permutation's columns and Assembly's mapping, as (u64 column, u64 row) pairs
        let perm_cols: Vec<h2b_mock_column> = self.cs.permutation.get_columns().iter().map(|c| match c.column_type() {
            Any::Fixed => h2b_mock_column { kind: 2, index: c.index() as u32 },
            Any::Advice(_) => h2b_mock_column { kind: 3, index: c.index() as u32 },
            Any::Instance => h2b_mock_column { kind: 4, index: c.index() as u32 },
        }).collect();
        let mapping: Vec<Vec<[u64; 2]>> = self.permutation.mapping.iter().map(|col| col.iter().map(|&(c, r)| [c as u64, r as u64]).collect()).collect();

        let ptrs = |v: &[(Vec<[u64; 4]>, Vec<u8>)]| -> (Vec<*const u64>, Vec<*const u8>) {
            (v.iter().map(|(w, _)| w.as_ptr() as *const u64).collect(), v.iter().map(|(_, b)| b.as_ptr()).collect())
        };
        let (fx, fb) = ptrs(&fixed);
        let (ad, ab) = ptrs(&advice);
        let ins: Vec<*const u64> = instance.iter().map(|c| c.as_ptr() as *const u64).collect();
        let mp: Vec<*const u64> = mapping.iter().map(|c| c.as_ptr() as *const u64).collect();
        let circuit = h2b_mock_circuit {
            k: self.k, blinding_factors: self.cs.blinding_factors() as u32,
            fixed: fx.as_ptr(), fixed_assigned: fb.as_ptr(), n_fixed: fx.len() as u32,
            advice: ad.as_ptr(), advice_assigned: ab.as_ptr(), n_advice: ad.len() as u32,
            instance: ins.as_ptr(), n_instance: ins.len() as u32,
            challenges: challenges.as_ptr() as *const u64, n_challenges: challenges.len() as u32,
            gates: &ffi_gates, roots: roots.as_ptr(), n_roots: roots.len() as u32,
            lookups: ffi_lookups.as_ptr(), n_lookups: ffi_lookups.len() as u32,
            permutation: perm_cols.as_ptr(), mapping: mp.as_ptr(), n_permutation: perm_cols.len() as u32,
        };
        let records = h2b200_sys::mock_verify(&circuit, 1024);

        // records -> VerifyFailure, with upstream's constructors and location finders (the bodies of verify_at_rows_par)
        let mut errors: Vec<VerifyFailure> = self.selector_errors_h2b();        // the region checks, unchanged
        let mut lookup_failures: Vec<(usize, Vec<Value<F>>, usize)> = Vec::new();
        for rec in &records {
            let (index, row) = (rec.index as usize, rec.row as usize);
            match rec.kind {
                H2B_MOCK_CONSTRAINT_NOT_SATISFIED | H2B_MOCK_CONSTRAINT_POISONED => {
                    let gate = &self.cs.gates[index];
                    let poly = &gate.polynomials()[rec.poly as usize];
                    let constraint = ((index, gate.name()).into(), rec.poly as usize, gate.constraint_name(rec.poly as usize)).into();
                    errors.push(if rec.kind == H2B_MOCK_CONSTRAINT_NOT_SATISFIED {
                        VerifyFailure::ConstraintNotSatisfied {
                            constraint,
                            location: FailureLocation::find_expressions(&self.cs, &self.regions, row, Some(poly).into_iter()),
                            cell_values: util::cell_values(gate, poly, &util::load(n as i32, row as i32, &self.cs.fixed_queries, &self.fixed),
                                                           &util::load(n as i32, row as i32, &self.cs.advice_queries, &self.advice),
                                                           &util::load_instance(n as i32, row as i32, &self.cs.instance_queries, &self.instance)),
                        }
                    } else {
                        VerifyFailure::ConstraintPoisoned { constraint }
                    });
                }
                H2B_MOCK_LOOKUP => {
                    let input = self.cs.lookups[index].input_expressions.iter().map(|e| self.load_value_h2b(e, row)).collect();
                    lookup_failures.push((index, input, row));
                }
                _ => {
                    let column = self.cs.permutation.get_columns()[index];
                    errors.push(VerifyFailure::Permutation { column: (*column.column_type(), column.index()).into(),
                                                             location: FailureLocation::find(&self.regions, row, Some(column).into_iter().collect()) });
                }
            }
        }
        // upstream sorts (input tuple, row) before it searches, per lookup
        lookup_failures.sort_by(|a, b| (a.0, &a.1, a.2).cmp(&(b.0, &b.1, b.2)));
        let at = errors.iter().position(|e| matches!(e, VerifyFailure::Permutation { .. })).unwrap_or(errors.len());
        let lookup_errors: Vec<VerifyFailure> = lookup_failures.into_iter().map(|(index, _, row)| {
            let lookup = &self.cs.lookups[index];
            VerifyFailure::Lookup { name: lookup.name, lookup_index: index,
                                    location: FailureLocation::find_expressions(&self.cs, &self.regions, row, lookup.input_expressions.iter()) }
        }).collect();
        errors.splice(at..at, lookup_errors);
        if errors.is_empty() {
            Ok(())
        } else {
            // as verify_at_rows_par ends: ConstraintPoisoned carries no location, and every unusable row a poisoned polynomial
            // reaches gives one, so consecutive equal ones are merged
            errors.dedup_by(|a, b| match (a, b) {
                (a @ VerifyFailure::ConstraintPoisoned { .. }, b @ VerifyFailure::ConstraintPoisoned { .. }) => a == b,
                _ => false,
            });
            Err(errors)
        }
    }
}
