// ORACLE (test infrastructure only): CPU restatement of halo2_proofs' compress_selectors and of the fixed half of keygen_vk /
// keygen_pk ([UP] halo2_proofs/src/plonk/circuit/compress_selectors.rs and plonk/keygen.rs @ v2023_02_02, as recalled), on the field,
// NTT and MSM code of oracle/h2_oracle.cpp.  It follows upstream's algorithm, deliberately not the device's:
//
//   process(selectors, max_degree): every degree-0 selector, in order, gets a column of its own (its activations as 0 / 1); the rest
//       get the lower-triangular exclusion matrix excl[i][j] = activations_i.iter().zip(activations_j).any(|(l, r)| l & r), then the
//       greedy combination (d = deg_i - 1; stop at d + len == max_degree; skip added or excluded j and any j with
//       max(d, deg_j - 1) + len + 1 > max_degree), and each combination is filled row by row into vec![F::zero(); n] with
//       assigned_root = 1, 2, .. counted by repeated F::one() additions
//   keygen_vk: fixed_commitments = commit_lagrange(each of fixed ++ selector columns) = best_multiexp(column, g_lagrange)
//   keygen_pk: fixed_polys = lagrange_to_coeff(each), fixed_cosets = coeff_to_extended(each poly)
//
// EvaluationDomain::lagrange_to_coeff: best_fft(a, omega_inv, k), a[i] *= ifft_divisor;  coeff_to_extended: a[i] *= zeta_powers[i mod 3],
// zero-pad to 2^extended_k, best_fft(a, extended_omega, extended_k).  Also the timed CPU path of tools/fixed_keygen_bench.py.
#include "../../oracle/h2_oracle.cpp"

namespace {

Fr fr_of(const u64* w) { Fr r; memcpy(r.l, w, 32); return r; }

bool any_both(const uint8_t* a, const uint8_t* b, size_t n) {
    for (size_t r = 0; r < n; ++r)
        if ((a[r] != 0) & (b[r] != 0)) return true;
    return false;
}

}  // namespace

extern "C" {

// the full symmetric exclusion matrix (S x S bytes) of S selectors (S x 2^k bytes), by the bool zip of every pair
void orc_selector_exclusion(const uint8_t* acts, uint32_t S, uint32_t k, uint8_t* out) {
    const size_t n = (size_t)1 << k;
    for (size_t i = 0; i < S; ++i) {
        out[i * S + i] = 0;
        for (size_t j = 0; j < i; ++j) out[i * S + j] = out[j * S + i] = any_both(acts + i * n, acts + j * n, n) ? 1 : 0;
    }
}

// process: per selector its combination, root and combination length; returns the number of combinations.  out_columns (C x n x 4,
// may be null) receives the combination columns as process fills them.
uint32_t orc_compress_selectors(const uint8_t* acts, const uint32_t* degrees, uint32_t S, uint32_t k, uint32_t max_degree, uint32_t* combination_of,
                                uint32_t* root_of, uint32_t* len_of, u64* out_columns) {
    const size_t n = (size_t)1 << k;
    std::vector<std::vector<Fr>> columns;
    std::vector<uint32_t> simple;
    for (uint32_t s = 0; s < S; ++s) {
        if (degrees[s] != 0) { simple.push_back(s); continue; }
        std::vector<Fr> col(n);
        for (size_t r = 0; r < n; ++r) col[r] = acts[s * n + r] ? Fr::one() : Fr::zero();
        combination_of[s] = (uint32_t)columns.size(); root_of[s] = 1; len_of[s] = 1;
        columns.push_back(std::move(col));
    }
    const size_t m = simple.size();
    std::vector<std::vector<bool>> excl(m);
    for (size_t i = 0; i < m; ++i) {
        excl[i].assign(i, false);
        for (size_t j = 0; j < i; ++j) excl[i][j] = any_both(acts + simple[i] * n, acts + simple[j] * n, n);
    }
    std::vector<bool> added(m, false);
    for (size_t i = 0; i < m; ++i) {
        if (added[i]) continue;
        added[i] = true;
        size_t d = degrees[simple[i]] - 1;
        std::vector<size_t> comb{i};
        for (size_t j = i + 1; j < m; ++j) {
            if (d + comb.size() == max_degree) break;
            if (added[j]) continue;
            bool excluded = false;
            for (size_t a : comb) excluded = excluded || excl[j][a];
            if (excluded) continue;
            const size_t new_d = std::max(d, (size_t)degrees[simple[j]] - 1);
            if (new_d + comb.size() + 1 > max_degree) continue;
            d = new_d;
            comb.push_back(j);
            added[j] = true;
        }
        std::vector<Fr> col(n, Fr::zero());
        Fr assigned_root = Fr::one();
        for (size_t t = 0; t < comb.size(); ++t) {
            const uint32_t s = simple[comb[t]];
            for (size_t r = 0; r < n; ++r)
                if (acts[s * n + r]) col[r] = assigned_root;
            assigned_root = assigned_root + Fr::one();
            combination_of[s] = (uint32_t)columns.size(); root_of[s] = (uint32_t)(t + 1); len_of[s] = (uint32_t)comb.size();
        }
        columns.push_back(std::move(col));
    }
    if (out_columns)
        for (size_t c = 0; c < columns.size(); ++c) memcpy(out_columns + 4 * n * c, columns[c].data(), n * 32);
    return (uint32_t)columns.size();
}

// keygen_vk / keygen_pk over m columns (m x n x 4, fixed ++ selector columns): commitments (m x 12 Jacobian, over g_lagrange) when
// out_jac is non-null, polys (m x n x 4) and cosets (m x 2^ek x 4) when non-null
void orc_fixed_build(const u64* columns, uint32_t m, uint32_t k, uint32_t ek, const u64* omega_inv, const u64* ifft_divisor, const u64* ext_omega,
                     const u64* zeta_powers, const u64* g_lagrange, int threads, u64* out_jac, u64* out_polys, u64* out_cosets) {
    const size_t n = (size_t)1 << k, en = (size_t)1 << ek;
    const Fr zeta[3] = {fr_of(zeta_powers), fr_of(zeta_powers + 4), fr_of(zeta_powers + 8)};
    std::vector<Fr> poly(n), ext(en);
    for (size_t i = 0; i < m; ++i) {
        const Fr* col = (const Fr*)columns + i * n;
        if (out_jac) {
            G1 r = best_multiexp(col, (const G1Affine*)g_lagrange, n, threads);
            memcpy(out_jac + 12 * i, &r, 96);
        }
        if (!out_polys && !out_cosets) continue;
        memcpy(poly.data(), col, n * 32);
        best_fft(poly.data(), fr_of(omega_inv), k, threads);
        for (size_t t = 0; t < n; ++t) poly[t] = poly[t] * fr_of(ifft_divisor);
        if (out_polys) memcpy(out_polys + 4 * n * i, poly.data(), n * 32);
        if (!out_cosets) continue;
        for (size_t t = 0; t < en; ++t) ext[t] = t < n ? poly[t] * zeta[t % 3] : Fr::zero();
        best_fft(ext.data(), fr_of(ext_omega), ek, threads);
        memcpy(out_cosets + 4 * en * i, ext.data(), en * 32);
    }
}

}  // extern "C"
