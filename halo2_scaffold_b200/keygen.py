"""
Host-side mirror of the key-generation steps of halo2_proofs that build the permutation argument's keys
([UP] halo2_proofs/src/plonk/permutation/keygen.rs Assembly::{build_vk, build_pk}) and keygen_pk's indicator columns
([UP] halo2_proofs/src/plonk/keygen.rs).  The mapping -- upstream's Vec<Vec<(usize, usize)>>, here a (P, n, 2) uint64 array
of (column, row) pairs -- comes from the circuit's synthesis (Assembly::copy), which stays on the host; everything per row
runs on the device: sigma, its commitments, its coefficient and extended-coset forms, and l0 / l_last / l_active_row.
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
