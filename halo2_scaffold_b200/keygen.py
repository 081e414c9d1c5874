"""
Host-side mirror of the key-generation steps of halo2_proofs that build the permutation argument's keys
([UP] halo2_proofs/src/plonk/permutation/keygen.rs Assembly::{build_vk, build_pk}) and keygen_pk's indicator columns
([UP] halo2_proofs/src/plonk/keygen.rs).  The mapping -- upstream's Vec<Vec<(usize, usize)>>, here a (P, n, 2) uint64 array
of (column, row) pairs -- comes from the circuit's synthesis (Assembly::copy), which stays on the host; everything per row
runs on the device: sigma, its commitments, its coefficient and extended-coset forms, and l0 / l_last / l_active_row.

The fixed half of keygen_vk / keygen_pk ([UP] plonk/circuit/compress_selectors.rs, plonk/keygen.rs) runs here too: compress_selectors
takes process's exclusion matrix from the device and keeps upstream's greedy step on the host, and the fixed and combination columns
get their commitments, coefficients and extended cosets on the device.  batch_invert_assigned stays with the caller.

ResidentProvingKey keeps those columns on the devices as one handle (h2b_pk_*), built there by the same kernels, so that the prover's
device steps read them instead of uploading them for every proof.
"""
from __future__ import annotations

import numpy as np

from . import _lib
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


# ---- the proving key resident on the devices (include/h2b200.h h2b_pk_*) ------------------------------------------------------------
_PARTS = {"fixed": _lib.PK_FIXED, "permutation": _lib.PK_PERMUTATION, "indicators": _lib.PK_INDICATORS}
_FORMS = {"values": _lib.PK_VALUES, "coeff": _lib.PK_COEFF, "extended": _lib.PK_EXTENDED}
_LAYOUTS = {"replicated": _lib.PK_REPLICATED, "row_sharded": _lib.PK_ROW_SHARDED}


def _code(table, x):
    return table[x] if isinstance(x, str) else int(x)


class ResidentProvingKey:
    """A ProvingKey's fixed, permutation and indicator columns held on the devices of the library from keygen to the last proof.

    Fixed and permutation columns keep three forms each (values: Lagrange, coeff: lagrange_to_coeff, extended: coeff_to_extended), the
    indicators l0 / l_last / l_active_row their extended form.  layout "replicated" puts every column on every device; "row_sharded"
    keeps the n-row forms on every device and gives device d of D only its rows of each extended column plus `halo` rows on each side
    -- the slice the row-sharded evaluate_h reads.  A context manager: the handle is released on exit."""

    def __init__(self, domain, n_fixed: int, n_permutation: int, layout="replicated", halo: int = 0, lib=None):
        self.lib = lib or domain.lib
        self.domain = domain
        self.n_fixed, self.n_permutation = int(n_fixed), int(n_permutation)
        self.layout = _code(_LAYOUTS, layout)
        d = domain
        self.handle = self.lib.pk_create(d.k, d.extended_k, self.n_fixed, self.n_permutation, self.layout, halo, fr_to_words(d.omega),
                                         fr_to_words(d.omega_inv), fr_to_words(d.ifft_divisor), fr_to_words(d.extended_omega), _zeta_powers(d))

    def close(self):
        if self.handle:
            h, self.handle = self.handle, 0
            self.lib.pk_release(h)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- building ----
    def build_fixed(self, fixed, activations, assignment, first_column: int = 0):
        """keygen_pk's fixed columns (the caller's, then compress_selectors' combination columns) into FIXED columns first_column .."""
        self.lib.keygen_fixed_build_pk_resident(fixed, activations, assignment["combination_of"], assignment["root_of"], assignment["n_combinations"],
                                                self.domain.k, self.handle, first_column)

    def build_permutation(self, mapping):
        """Assembly::build_pk's sigma columns from the mapping ((P, 2^k, 2) (column, row) pairs)"""
        self.lib.permutation_build_pk_resident(mapping, self.domain.k, fr_to_words(FR_DELTA), self.handle)

    def build_indicators(self, blinding_factors: int):
        """keygen_pk's l0, l_last, l_active_row"""
        self.lib.keygen_lagrange_indicators_resident(self.handle, blinding_factors)

    def put_lagrange(self, part, values, first: int = 0):
        """columns of a ProvingKey built elsewhere, in Lagrange form; the other forms are derived on the device"""
        self.lib.pk_put_lagrange(self.handle, _code(_PARTS, part), first, list(values), self.domain.k)

    # ---- reading ----
    def column(self, part, form, index: int, device: int = 0):
        """-> (device pointer, (row0, rows, halo)) of one column on `device`"""
        return self.lib.pk_column(self.handle, device, _code(_PARTS, part), _code(_FORMS, form), index)

    def download(self, part, form, index: int) -> np.ndarray:
        rows = 1 << (self.domain.extended_k if _code(_FORMS, form) == _lib.PK_EXTENDED else self.domain.k)
        return self.lib.pk_download(self.handle, _code(_PARTS, part), _code(_FORMS, form), index, rows)

    def info(self) -> list:
        """bytes held on each device"""
        return self.lib.pk_info(self.handle)

    def eval_columns(self, device: int = 0) -> dict:
        """what the h2b_evaluate_* entry points take from the pk on `device`: dict(fixed, permutation: lists of extended-coset pointers,
        l0, l_last, l_active_row, shard: (row0, rows, halo) for the row-sharded entry points, None in the replicated layout)"""
        ext = lambda part, i: self.column(part, "extended", i, device)
        fixed = [ext("fixed", i) for i in range(self.n_fixed)]
        perm = [ext("permutation", i) for i in range(self.n_permutation)]
        ind = [ext("indicators", i) for i in range(3)]
        return dict(fixed=[p for p, _ in fixed], permutation=[p for p, _ in perm], l0=ind[0][0], l_last=ind[1][0], l_active_row=ind[2][0],
                    shard=ind[0][1] if self.layout == _lib.PK_ROW_SHARDED else None)
