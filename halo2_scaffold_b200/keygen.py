"""
Host-side mirror of the key-generation steps of halo2_proofs that build the permutation argument's keys
([UP] halo2_proofs/src/plonk/permutation/keygen.rs Assembly::{build_vk, build_pk}) and keygen_pk's indicator columns
([UP] halo2_proofs/src/plonk/keygen.rs).  The mapping -- upstream's Vec<Vec<(usize, usize)>>, here a (P, n, 2) uint64 array
of (column, row) pairs -- comes from the circuit's synthesis (Assembly::copy), which stays on the host; everything per row
runs on the device: sigma, its commitments, its coefficient and extended-coset forms, and l0 / l_last / l_active_row.

The fixed half of keygen_vk / keygen_pk ([UP] plonk/circuit/compress_selectors.rs, plonk/keygen.rs) runs here too: compress_selectors
takes process's exclusion matrix from the device and keeps upstream's greedy step on the host, and the fixed and combination columns
get their commitments, coefficients and extended cosets on the device.  batch_invert_assigned stays with the caller.
"""
from __future__ import annotations

import numpy as np

from .domain import FR_MODULUS, FR_S, fr_to_words

FR_GENERATOR = 7
FR_DELTA = pow(FR_GENERATOR, 1 << FR_S, FR_MODULUS)     # Fr::DELTA = GENERATOR^(2^S)


def _zeta_powers(domain) -> np.ndarray:
    return np.stack([fr_to_words(1), fr_to_words(domain.g_coset), fr_to_words(domain.g_coset_inv)])


def permutation_build_vk(params, domain, mapping) -> np.ndarray:
    """Assembly::build_vk: commitments[i] = params.commit_lagrange(sigma_i) -> (P, 12) Jacobian"""
    return params.lib.permutation_build_vk(mapping, domain.k, fr_to_words(FR_DELTA), fr_to_words(domain.omega), params._g_lagrange)


def permutation_build_pk(params, domain, mapping) -> dict:
    """Assembly::build_pk -> dict(permutations, polys, cosets): sigma_i in Lagrange form, lagrange_to_coeff(sigma_i) and
    coeff_to_extended of that, one list entry per column.  `params` only supplies the library (upstream's is unused too)."""
    return params.lib.permutation_build_pk(mapping, domain.k, domain.extended_k, fr_to_words(FR_DELTA), fr_to_words(domain.omega),
                                           fr_to_words(domain.omega_inv), fr_to_words(domain.ifft_divisor), fr_to_words(domain.extended_omega),
                                           _zeta_powers(domain))


def lagrange_indicators(domain, blinding_factors: int):
    """keygen_pk's (l0, l_last, l_active_row) on the extended coset, each (2^extended_k, 4)"""
    return domain.lib.keygen_lagrange_indicators(domain.k, domain.extended_k, blinding_factors, fr_to_words(domain.omega_inv),
                                                 fr_to_words(domain.ifft_divisor), fr_to_words(domain.extended_omega), _zeta_powers(domain),
                                                 device=domain.device)


# ---- compress_selectors and the fixed columns of keygen_vk / keygen_pk ([UP] plonk/circuit/compress_selectors.rs, plonk/keygen.rs) ----
def compress_selectors(activations, degrees, max_degree: int, lib=None) -> dict:
    """compress_selectors::process over selectors with these activations ((S, 2^k) bool) and gate degrees (upstream's
    SelectorDescription::max_degree; 0 for a selector in no gate polynomial), against max_degree = cs.degree().  The exclusion matrix
    comes from the device; the greedy step is upstream's, on the host.  Returns dict(combination_of, root_of: (S,) uint32,
    n_combinations, expressions: per selector (combination, root, len), standing for the substitution q * prod_{r = 1..len, r != root} (r - q)
    with q the combination's fixed column)."""
    if lib is None:
        from . import load
        lib = load()
    S = len(activations)
    degrees = [int(d) for d in degrees]
    assert len(degrees) == S, "one degree per selector"
    combination_of = np.zeros(S, dtype=np.uint32)
    root_of = np.zeros(S, dtype=np.uint32)
    expressions = [None] * S
    n_comb = 0
    # degree-0 selectors first, each in a column of its own with root 1
    for s in range(S):
        if degrees[s] == 0:
            combination_of[s], root_of[s], expressions[s] = n_comb, 1, (n_comb, 1, 1)
            n_comb += 1
    simple = [s for s in range(S) if degrees[s] > 0]
    if simple:
        k = int(np.asarray(activations[simple[0]]).reshape(-1).shape[0]).bit_length() - 1
        excl = lib.selector_exclusion([activations[s] for s in simple], k)
    added = [False] * len(simple)
    for i in range(len(simple)):
        if added[i]:
            continue
        added[i] = True
        assert degrees[simple[i]] <= max_degree
        d = degrees[simple[i]] - 1
        combination = [i]
        for j in range(i + 1, len(simple)):
            if d + len(combination) == max_degree:
                break
            if added[j] or any(excl[j][m] for m in combination):
                continue
            new_d = max(d, degrees[simple[j]] - 1)
            if new_d + len(combination) + 1 > max_degree:
                continue
            d = new_d
            combination.append(j)
            added[j] = True
        for t, m in enumerate(combination, start=1):
            s = simple[m]
            combination_of[s], root_of[s], expressions[s] = n_comb, t, (n_comb, t, len(combination))
        n_comb += 1
    return dict(combination_of=combination_of, root_of=root_of, n_combinations=n_comb, expressions=expressions)


def fixed_build_vk(params, domain, fixed, activations, assignment) -> np.ndarray:
    """keygen_vk's fixed_commitments: commit_lagrange of each fixed column, then of each combination column of `assignment`
    (compress_selectors' result) -> (F + C, 12) Jacobian"""
    return params.lib.keygen_fixed_build_vk(fixed, activations, assignment["combination_of"], assignment["root_of"], assignment["n_combinations"],
                                            domain.k, params._g_lagrange)


def fixed_build_pk(params, domain, fixed, activations, assignment) -> dict:
    """keygen_pk's fixed columns -> dict(combination_values, polys, cosets): the combination columns in Lagrange form (fixed_values
    is the caller's fixed columns followed by these), and lagrange_to_coeff / coeff_to_extended of every fixed and combination column"""
    return params.lib.keygen_fixed_build_pk(fixed, activations, assignment["combination_of"], assignment["root_of"], assignment["n_combinations"],
                                            domain.k, domain.extended_k, fr_to_words(domain.omega_inv), fr_to_words(domain.ifft_divisor),
                                            fr_to_words(domain.extended_omega), _zeta_powers(domain))
