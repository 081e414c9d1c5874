"""CPU: the text transform that wires rust/patches/gwc_dropin.rs into halo2_proofs (rust/patches/gwc_patch.py), run on an excerpt laid
out as PSE v2023_02_02's src/poly/kzg/multiopen/gwc/prover.rs (restated from recollection, not copied: the checkout is not vendored).
What it pins: the Bn256 dispatch is the first statement of `create_proof`, before upstream squeezes v, in rustfmt's multi-line
signature as well as on one line; the imports the drop-in needs are added without repeating one upstream has; the drop-in is appended
once; and a file without that signature stops the transform instead of being patched somewhere else."""
import os
import re
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "rust", "patches"))

import gwc_patch  # noqa: E402

PROVER_RS = '''use super::{construct_intermediate_sets, ChallengeV, Query};
use crate::arithmetic::{eval_polynomial, kate_division, powers, CurveAffine};
use crate::helpers::SerdeCurveAffine;
use crate::poly::commitment::ParamsProver;
use crate::poly::commitment::Prover;
use crate::poly::kzg::commitment::{KZGCommitmentScheme, ParamsKZG};
use crate::poly::query::ProverQuery;
use crate::poly::{commitment::Blind, Polynomial};
use crate::transcript::{EncodedChallenge, TranscriptWrite};

use group::Curve;
use halo2curves::pairing::Engine;
use rand_core::RngCore;
use std::fmt::Debug;
use std::io;
use std::marker::PhantomData;

/// Concrete KZG prover with GWC variant
#[derive(Debug)]
pub struct ProverGWC<'params, E: Engine> {
    params: &'params ParamsKZG<E>,
}

/// Create a multi-opening proof
impl<'params, E: Engine + Debug> Prover<'params, KZGCommitmentScheme<E>> for ProverGWC<'params, E>
where
    E::G1Affine: SerdeCurveAffine,
    E::G2Affine: SerdeCurveAffine,
{
    const QUERY_INSTANCE: bool = false;

    fn new(params: &'params ParamsKZG<E>) -> Self {
        Self { params }
    }

    /// Create a multi-opening proof
    fn create_proof<
        'com,
        Ch: EncodedChallenge<E::G1Affine>,
        T: TranscriptWrite<E::G1Affine, Ch>,
        R,
        I,
    >(
        &self,
        _: R,
        transcript: &mut T,
        queries: I,
    ) -> io::Result<()>
    where
        I: IntoIterator<Item = ProverQuery<'com, E::G1Affine>> + Clone,
        R: RngCore,
    {
        let v: ChallengeV<_> = transcript.squeeze_challenge_scalar();
        let commitment_data = construct_intermediate_sets(queries);

        for commitment_at_a_point in commitment_data.iter() {
            let z = commitment_at_a_point.point;
            let (poly_batch, eval_batch) = commitment_at_a_point
                .queries
                .iter()
                .zip(powers(*v))
                .map(|(query, power_of_v)| {
                    assert_eq!(query.get_point(), z);

                    let poly = query.get_commitment().poly;
                    let eval = query.get_eval();

                    (poly.clone() * power_of_v, eval * power_of_v)
                })
                .reduce(|(poly_acc, eval_acc), (poly, eval)| (poly_acc + &poly, eval_acc + eval))
                .unwrap();

            let poly_batch = &poly_batch - eval_batch;
            let witness_poly = Polynomial {
                values: kate_division(&poly_batch.values, z),
                _marker: PhantomData,
            };
            let w = self
                .params
                .commit(&witness_poly, Blind::default())
                .to_affine();

            transcript.write_point(w)?;
        }
        Ok(())
    }
}
'''

ONE_LINE = PROVER_RS.replace('''    fn create_proof<
        'com,
        Ch: EncodedChallenge<E::G1Affine>,
        T: TranscriptWrite<E::G1Affine, Ch>,
        R,
        I,
    >(
        &self,
        _: R,
        transcript: &mut T,
        queries: I,
    ) -> io::Result<()>''', "    fn create_proof<'com, Ch: EncodedChallenge<E::G1Affine>, T: TranscriptWrite<E::G1Affine, Ch>, R, I>(&self, _: R, transcript: &mut T, queries: I) -> io::Result<()>")


def dropin():
    with open(os.path.join(ROOT, "rust", "patches", "gwc_dropin.rs")) as f:
        return f.read()


@pytest.mark.parametrize("src", [PROVER_RS, ONE_LINE], ids=["rustfmt", "one_line"])
def test_dispatch_comes_first_and_dropin_is_appended(src):
    out = gwc_patch.patch_gwc_prover(src, dropin())
    patched, appended = out.split("// ---- libh2b200 drop-in (rust/patches/gwc_dropin.rs) ----\n")
    assert appended == dropin() + "\n" and out.count("fn create_proof_h2b<") == 1
    # the first statement of create_proof's body, before upstream squeezes v
    open_brace = "        R: RngCore,\n    {\n"
    body = patched[patched.index(open_brace) + len(open_brace):]
    assert body.lstrip().startswith(gwc_patch.DISPATCH + "\n        let v: ChallengeV<_> = transcript.squeeze_challenge_scalar();")
    assert patched.count(gwc_patch.DISPATCH) == 1
    uses = [l for l in patched.splitlines() if l.startswith("use ")]
    for use in gwc_patch.USES:
        assert uses.count(use) == 1
    assert sum(bool(re.search(r"\bPolynomial\b", l)) for l in uses) == 1            # upstream's import is not repeated
    assert gwc_patch.patch_gwc_prover(out, dropin()) == out                          # idempotent


def test_refuses_a_file_it_does_not_recognise():
    with pytest.raises(AssertionError):
        gwc_patch.patch_gwc_prover(PROVER_RS.replace("fn create_proof<", "fn create_proof_renamed<"), dropin())
    with pytest.raises(AssertionError):
        gwc_patch.patch_gwc_prover(PROVER_RS.replace("for ProverGWC<'params, E>", "for ProverOther<'params, E>"), dropin())
    with pytest.raises(AssertionError):
        gwc_patch.patch_gwc_prover(PROVER_RS.replace("use crate::poly::{commitment::Blind, Polynomial};", "use crate::poly::commitment::Blind;"), dropin())
