//! proof_bytes <case> <seed> <out-file>
//!
//! Proves one of the reference's circuits under a ChaCha20 rng seeded with <seed> (SRS, witness and prover randomness all come from
//! it), checks the proof with the reference's verifier call, writes the proof bytes to <out-file> and prints their Blake2b digest.
//! Run once per arm (stock halo2_proofs / forks patched with libh2b200) and compare the files: scripts/proof_parity.sh.
//!
//! Cases (BASELINE.json configs):  standard_plonk  -- /root/reference/examples/standard_plonk.rs:25-64 (PSE prover, k = 5)
//!                                 standard_plonk_gwc -- the same circuit opened with ProverGWC / VerifierGWC instead of SHPLONK
//!                                 halo2_lib       -- /root/reference/examples/halo2_lib.rs through the scaffold::prove flow
//!                                                    (/root/reference/src/scaffold.rs:246-365; Axiom prover; DEGREE / LOOKUP_BITS env)
//! The circuits themselves are the reference's own types (halo2_scaffold::circuits / ::scaffold); only the rng differs: every call
//! site of the reference passes OsRng (src/scaffold.rs:198,214,329,345), which cannot be replayed.
use std::{env, fs};

use rand::SeedableRng;
use rand_chacha::ChaCha20Rng;

fn digest(bytes: &[u8]) -> String {
    blake2b_simd::Params::new().hash_length(32).hash(bytes).to_hex().to_string()
}

/// keygen + create_proof + verify_proof for any circuit of the PSE crate; `mk(None)` is the keygen circuit, `mk(Some(rng))` the proving one
mod pse {
    use super::*;
    use halo2_proofs::{
        halo2curves::bn256::{Bn256, Fr, G1Affine},
        plonk::{create_proof, keygen_pk, keygen_vk, verify_proof, Circuit},
        poly::commitment::ParamsProver,
        poly::kzg::{
            commitment::{KZGCommitmentScheme, ParamsKZG},
            multiopen::{ProverGWC, ProverSHPLONK, VerifierGWC, VerifierSHPLONK},
            strategy::SingleStrategy,
        },
        transcript::{Blake2bRead, Blake2bWrite, Challenge255, TranscriptReadBuffer, TranscriptWriterBuffer},
    };

    /// gwc: open with ProverGWC / VerifierGWC instead of ProverSHPLONK / VerifierSHPLONK
    pub fn prove<C: Circuit<Fr>>(k: u32, seed: u64, keygen: C, proving: impl FnOnce(&mut ChaCha20Rng) -> C, instances: &[&[Fr]], gwc: bool) -> Vec<u8> {
        let mut rng = ChaCha20Rng::seed_from_u64(seed);
        let params = ParamsKZG::<Bn256>::setup(k, &mut rng);
        let pk = keygen_pk(&params, keygen_vk(&params, &keygen).expect("vk"), &keygen).expect("pk");
        let circuit = proving(&mut rng);
        let mut w = Blake2bWrite::<_, G1Affine, Challenge255<_>>::init(vec![]);
        if gwc {
            create_proof::<KZGCommitmentScheme<Bn256>, ProverGWC<'_, Bn256>, _, _, _, _>(&params, &pk, &[circuit], &[instances], &mut rng, &mut w)
        } else {
            create_proof::<KZGCommitmentScheme<Bn256>, ProverSHPLONK<'_, Bn256>, _, _, _, _>(&params, &pk, &[circuit], &[instances], &mut rng, &mut w)
        }
        .expect("create_proof");
        let proof = w.finalize();
        let mut r = Blake2bRead::<_, G1Affine, Challenge255<_>>::init(&proof[..]);
        if gwc {
            verify_proof::<KZGCommitmentScheme<Bn256>, VerifierGWC<'_, Bn256>, _, _, SingleStrategy<'_, Bn256>>(
                params.verifier_params(), pk.get_vk(), SingleStrategy::new(&params), &[instances], &mut r)
        } else {
            verify_proof::<KZGCommitmentScheme<Bn256>, VerifierSHPLONK<'_, Bn256>, _, _, SingleStrategy<'_, Bn256>>(
                params.verifier_params(), pk.get_vk(), SingleStrategy::new(&params), &[instances], &mut r)
        }
        .expect("the reference verifier rejected the proof");
        proof
    }
}

/// the scaffold flow (GateThreadBuilder keygen -> break points -> prover builder) on the Axiom fork, with a seeded rng
mod axiom {
    use super::*;
    use halo2_base::{
        gates::builder::{GateCircuitBuilder, GateThreadBuilder, RangeCircuitBuilder},
        gates::{GateChip, GateInstructions},
        halo2_proofs::{
            halo2curves::bn256::{Bn256, Fr, G1Affine},
            plonk::{create_proof, keygen_pk, keygen_vk, verify_proof},
            poly::kzg::{
                commitment::{KZGCommitmentScheme, ParamsKZG},
                multiopen::{ProverSHPLONK, VerifierSHPLONK},
                strategy::SingleStrategy,
            },
            transcript::{Blake2bRead, Blake2bWrite, Challenge255, TranscriptReadBuffer, TranscriptWriterBuffer},
        },
        AssignedValue, Context,
    };
    use halo2_scaffold::scaffold::{GateWithInstanceCircuitBuilder, RangeWithInstanceCircuitBuilder};

    /// x -> x^2 + 27, the computation of the reference's halo2_lib example, written against the halo2-base gate API
    fn square_plus_27(ctx: &mut Context<Fr>, x: Fr, public: &mut Vec<AssignedValue<Fr>>) {
        let gate = GateChip::<Fr>::default();
        let x = ctx.load_witness(x);
        public.push(x);
        let sq = gate.mul(ctx, x, x);
        let out = gate.add(ctx, sq, halo2_base::QuantumCell::Constant(Fr::from(27)));
        public.push(out);
    }

    pub fn prove(seed: u64) -> Vec<u8> {
        let k: u32 = env::var("DEGREE").unwrap_or_else(|_| "16".into()).parse().unwrap();
        let lookup_bits: Option<usize> = env::var("LOOKUP_BITS").ok().map(|s| s.parse().unwrap());
        let mut rng = ChaCha20Rng::seed_from_u64(seed);
        let params = ParamsKZG::<Bn256>::setup(k, &mut rng);
        let x = Fr::from(rand::Rng::gen::<u64>(&mut rng));

        let mut kb = GateThreadBuilder::keygen();
        let mut kpub = vec![];
        square_plus_27(kb.main(0), Fr::zero(), &mut kpub);
        kb.config(k as usize, Some(9));
        let mut pb = GateThreadBuilder::prover();
        let mut ppub = vec![];
        square_plus_27(pb.main(0), x, &mut ppub);
        let io: Vec<Fr> = ppub.iter().map(|v| *v.value()).collect();

        macro_rules! run {
            ($wrapper:ident, $inner:ident, $bp:expr) => {{
                let kc = $wrapper { circuit: $inner::keygen(kb), assigned_instances: kpub };
                let pk = keygen_pk(&params, keygen_vk(&params, &kc).expect("vk"), &kc).expect("pk");
                let bp = $bp(&kc);
                let pc = $wrapper { circuit: $inner::prover(pb, bp), assigned_instances: ppub };
                let mut w = Blake2bWrite::<_, G1Affine, Challenge255<_>>::init(vec![]);
                create_proof::<KZGCommitmentScheme<Bn256>, ProverSHPLONK<'_, Bn256>, _, _, _, _>(&params, &pk, &[pc], &[&[&io]], &mut rng, &mut w)
                    .expect("create_proof");
                let proof = w.finalize();
                let mut r = Blake2bRead::<_, G1Affine, Challenge255<_>>::init(&proof[..]);
                verify_proof::<KZGCommitmentScheme<Bn256>, VerifierSHPLONK<'_, Bn256>, _, _, SingleStrategy<'_, Bn256>>(
                    &params, pk.get_vk(), SingleStrategy::new(&params), &[&[&io]], &mut r)
                    .expect("the reference verifier rejected the proof");
                proof
            }};
        }
        if lookup_bits.is_some() {
            run!(RangeWithInstanceCircuitBuilder, RangeCircuitBuilder, |c: &RangeWithInstanceCircuitBuilder<Fr>| c.circuit.0.break_points.take())
        } else {
            run!(GateWithInstanceCircuitBuilder, GateCircuitBuilder, |c: &GateWithInstanceCircuitBuilder<Fr>| c.circuit.break_points.take())
        }
    }
}

fn main() {
    let args: Vec<String> = env::args().collect();
    if args.len() != 4 {
        eprintln!("usage: proof_bytes <standard_plonk|standard_plonk_gwc|halo2_lib> <seed> <out-file>");
        std::process::exit(2);
    }
    let seed: u64 = args[2].parse().expect("seed");
    let proof = match args[1].as_str() {
        case @ ("standard_plonk" | "standard_plonk_gwc") => {
            use halo2_proofs::{circuit::Value, halo2curves::bn256::Fr};
            use halo2_scaffold::circuits::standard_plonk::StandardPlonk;
            pse::prove(5, seed, StandardPlonk { x: Value::unknown() }, |rng| StandardPlonk { x: Value::known(<Fr as ff::Field>::random(rng)) }, &[],
                       case == "standard_plonk_gwc")
        }
        "halo2_lib" => axiom::prove(seed),
        other => panic!("unknown case {other}"),
    };
    fs::write(&args[3], &proof).expect("write proof");
    println!("{} seed {} bytes {} blake2b {}", args[1], seed, proof.len(), digest(&proof));
}
