#!/usr/bin/env bash
# One command on a machine with cargo + a B200:   rust/harness/scripts/proof_parity.sh [seed]
# Builds the harness twice -- arm "cpu": stock halo2_proofs; arm "gpu": both halo2 forks patched to call libh2b200 -- proves every case
# with the same seed in both arms and compares the proof bytes.  Exit status 0 = byte-identical proofs, each accepted by the
# reference verifier (the binary panics otherwise).
set -euo pipefail
SEED="${1:-20240406}"
HERE="$(cd "$(dirname "$0")/.." && pwd)"          # rust/harness
REPO="$(cd "$HERE/../.." && pwd)"                 # this repository
WORK="$(cd "$REPO/.." && pwd)"                    # holds halo2-scaffold/ next to this repository
FORKS="$REPO/rust/forks"

[ -d "$WORK/halo2-scaffold" ] || git clone https://github.com/DCMMC/halo2-scaffold "$WORK/halo2-scaffold"
mkdir -p "$FORKS"
[ -d "$FORKS/halo2-pse-v2023_02_02" ] || git clone --depth 1 --branch v2023_02_02 https://github.com/privacy-scaling-explorations/halo2 "$FORKS/halo2-pse-v2023_02_02"
[ -d "$FORKS/halo2-axiom-dev" ] || git clone --depth 1 --branch axiom/dev https://github.com/axiom-crypto/halo2 "$FORKS/halo2-axiom-dev"
# the drop-in: best_multiexp / best_fft bodies + the h2b200-sys dependency (INTEGRATION.md section 3)
for f in "$FORKS/halo2-pse-v2023_02_02" "$FORKS/halo2-axiom-dev"; do
    python3 "$REPO/rust/patches/apply_dropin.py" "$f/halo2_proofs" "$REPO/rust"
done

python3 -c "import __graft_entry__ as g; g.build()" 2>/dev/null || make -C "$REPO/halo2_scaffold_b200/csrc"
export H2B200_LIB_DIR="$REPO/halo2_scaffold_b200/lib" LD_LIBRARY_PATH="$REPO/halo2_scaffold_b200/lib:${LD_LIBRARY_PATH:-}"

build_arm() {   # $1 = cpu | gpu
    cp "$HERE/Cargo.toml" "$HERE/Cargo.toml.orig"
    if [ "$1" = gpu ]; then
        cat >> "$HERE/Cargo.toml" <<PATCH
[patch."https://github.com/privacy-scaling-explorations/halo2.git"]
halo2_proofs = { path = "$FORKS/halo2-pse-v2023_02_02/halo2_proofs" }
[patch."https://github.com/axiom-crypto/halo2.git"]
halo2_proofs = { path = "$FORKS/halo2-axiom-dev/halo2_proofs" }
PATCH
    fi
    (cd "$HERE" && cargo build --release --target-dir "target-$1")
    mv "$HERE/Cargo.toml.orig" "$HERE/Cargo.toml"
}
build_arm cpu
build_arm gpu

OUT="$HERE/proofs"; mkdir -p "$OUT"; status=0
for case in standard_plonk standard_plonk_gwc halo2_lib; do
    for arm in cpu gpu; do
        DEGREE=16 "$HERE/target-$arm/release/proof_bytes" "$case" "$SEED" "$OUT/$case.$arm.proof"
    done
    if cmp -s "$OUT/$case.cpu.proof" "$OUT/$case.gpu.proof"; then echo "PARITY OK   $case (seed $SEED)"; else echo "PARITY FAIL $case"; status=1; fi
done
DEGREE=20 LOOKUP_BITS=19 "$HERE/target-cpu/release/proof_bytes" halo2_lib "$SEED" "$OUT/halo2_lib_k20.cpu.proof"
DEGREE=20 LOOKUP_BITS=19 "$HERE/target-gpu/release/proof_bytes" halo2_lib "$SEED" "$OUT/halo2_lib_k20.gpu.proof"
cmp -s "$OUT/halo2_lib_k20.cpu.proof" "$OUT/halo2_lib_k20.gpu.proof" && echo "PARITY OK   halo2_lib k=20 lookup" || { echo "PARITY FAIL halo2_lib k=20"; status=1; }
exit $status
