// ORACLE (test infrastructure only): CPU restatement of halo2_proofs' permutation keygen and of keygen_pk's indicator block
// ([UP] halo2_proofs/src/plonk/permutation/keygen.rs and plonk/keygen.rs @ v2023_02_02, as recalled), on the field, NTT and MSM
// code of oracle/h2_oracle.cpp.  It follows upstream's algorithm, deliberately not the device's:
//
//   Assembly::new(n, p): mapping[i][j] = aux[i][j] = (i, j), sizes[i][j] = 1
//   Assembly::copy(l, r): if aux[l] == aux[r] return; the larger cycle by `sizes` becomes the left one (ties keep the order),
//       sizes[left] += sizes[right], walk the right cycle through `mapping` setting aux to the left cycle, swap(mapping[l], mapping[r])
//   build_vk: omega_powers[j] = omega^j, deltaomega[i][j] = delta^i omega_powers[j] (the P x n table), sigma_i[j] =
//       deltaomega[mapping[i][j]], commitments[i] = commit_lagrange(sigma_i) = best_multiexp(sigma_i, g_lagrange)
//   build_pk: the same sigma_i, polys[i] = lagrange_to_coeff(sigma_i), cosets[i] = coeff_to_extended(polys[i])
//   keygen_pk: l0 = ext(coeff(e_0)), l_blind = ext(coeff(1 on the last bf rows)), l_last = ext(coeff(e_(n-bf-1))),
//       l_active_row[t] = 1 - (l_last[t] + l_blind[t])
//
// EvaluationDomain::lagrange_to_coeff: best_fft(a, omega_inv, k), a[i] *= ifft_divisor;  coeff_to_extended: a[i] *= zeta_powers[i mod 3],
// zero-pad to 2^extended_k, best_fft(a, extended_omega, extended_k).  std::thread in place of rayon.  Also the timed CPU sigma baseline of
// tools/permutation_keygen_bench.py.
#include "../../oracle/h2_oracle.cpp"

namespace {

typedef std::pair<u64, u64> Cell;

struct Assembly {
    std::vector<std::vector<Cell>> mapping, aux;
    std::vector<std::vector<u64>> sizes;
    Assembly(size_t n, size_t p) : mapping(p), aux(p), sizes(p, std::vector<u64>(n, 1)) {
        for (size_t i = 0; i < p; ++i) {
            mapping[i].resize(n);
            for (size_t j = 0; j < n; ++j) mapping[i][j] = Cell(i, j);
            aux[i] = mapping[i];
        }
    }
    void copy(size_t lc, size_t lr, size_t rc, size_t rr) {
        Cell left = aux[lc][lr], right = aux[rc][rr];
        if (left == right) return;
        if (sizes[left.first][left.second] < sizes[right.first][right.second]) std::swap(left, right);
        sizes[left.first][left.second] += sizes[right.first][right.second];
        Cell i = right;
        for (;;) {
            aux[i.first][i.second] = left;
            i = mapping[i.first][i.second];
            if (i == right) break;
        }
        std::swap(mapping[lc][lr], mapping[rc][rr]);
    }
};

template <class F>
void parallel_for(size_t n, int threads, F f) {
    if (threads < 1) threads = 1;
    const size_t per = (n + threads - 1) / threads;
    std::vector<std::thread> th;
    for (int t = 0; t < threads; ++t) {
        const size_t lo = t * per, hi = std::min(n, lo + per);
        if (lo >= hi) break;
        th.emplace_back(f, lo, hi);
    }
    for (auto& x : th) x.join();
}

Fr fr_pow(const Fr& b, u64 e) { const u64 w[4] = {e, 0, 0, 0}; return b.pow(w); }
Fr fr_of(const u64* w) { Fr r; memcpy(r.l, w, 32); return r; }

// build_vk / build_pk's sigma through upstream's P x n deltaomega table
void sigma_columns(const u64* mapping, uint32_t P, uint32_t k, const Fr& delta, const Fr& omega, int threads, Fr* out) {
    const size_t n = (size_t)1 << k;
    std::vector<Fr> omega_powers(n), deltaomega((size_t)P * n);
    parallel_for(n, threads, [&](size_t lo, size_t hi) {
        Fr cur = fr_pow(omega, lo);
        for (size_t j = lo; j < hi; ++j) { omega_powers[j] = cur; cur = cur * omega; }
    });
    parallel_for(P, threads, [&](size_t lo, size_t hi) {
        Fr cur = fr_pow(delta, lo);
        for (size_t i = lo; i < hi; ++i) {
            for (size_t j = 0; j < n; ++j) deltaomega[i * n + j] = omega_powers[j] * cur;
            cur = cur * delta;
        }
    });
    parallel_for((size_t)P * n, threads, [&](size_t lo, size_t hi) {
        for (size_t t = lo; t < hi; ++t) {
            const u64 c = mapping[2 * t], r = mapping[2 * t + 1];
            out[t] = deltaomega[c * n + r];
        }
    });
}

void lagrange_to_coeff(Fr* a, uint32_t k, const Fr& omega_inv, const Fr& ifft_divisor, int threads) {
    best_fft(a, omega_inv, k, threads);
    for (size_t i = 0; i < ((size_t)1 << k); ++i) a[i] = a[i] * ifft_divisor;
}

void coeff_to_extended(const Fr* coeff, uint32_t k, uint32_t ek, const Fr& ext_omega, const Fr zeta[3], int threads, Fr* out) {
    const size_t n = (size_t)1 << k, en = (size_t)1 << ek;
    for (size_t i = 0; i < en; ++i) out[i] = i < n ? coeff[i] * zeta[i % 3] : Fr::zero();
    best_fft(out, ext_omega, ek, threads);
}

}  // namespace

extern "C" {

// Assembly::new(2^k, P) then copy(l_col, l_row, r_col, r_row) for each of the `count` copies (4 u64 each), in order -> mapping (P x n x 2)
void orc_assembly_mapping(uint32_t P, uint32_t k, const u64* copies, size_t count, u64* out_mapping) {
    const size_t n = (size_t)1 << k;
    Assembly a(n, P);
    for (size_t c = 0; c < count; ++c) a.copy(copies[4 * c], copies[4 * c + 1], copies[4 * c + 2], copies[4 * c + 3]);
    for (size_t i = 0; i < P; ++i)
        for (size_t j = 0; j < n; ++j) { out_mapping[2 * (i * n + j)] = a.mapping[i][j].first; out_mapping[2 * (i * n + j) + 1] = a.mapping[i][j].second; }
}

// sigma of every column (P x n x 4 words)
void orc_permutation_sigma(const u64* mapping, uint32_t P, uint32_t k, const u64* delta, const u64* omega, int threads, u64* out) {
    sigma_columns(mapping, P, k, fr_of(delta), fr_of(omega), threads, (Fr*)out);
}

// build_vk: commitments (P x 12, Jacobian) over the first n points of g_lagrange
void orc_permutation_build_vk(const u64* mapping, uint32_t P, uint32_t k, const u64* delta, const u64* omega, const u64* g_lagrange, int threads,
                              u64* out_jac) {
    const size_t n = (size_t)1 << k;
    std::vector<Fr> sigma((size_t)P * n);
    sigma_columns(mapping, P, k, fr_of(delta), fr_of(omega), threads, sigma.data());
    for (size_t i = 0; i < P; ++i) {
        G1 r = best_multiexp(sigma.data() + i * n, (const G1Affine*)g_lagrange, n, threads);
        memcpy(out_jac + 12 * i, &r, 96);
    }
}

// build_pk: permutations (P x n x 4), polys (P x n x 4), cosets (P x 2^ek x 4)
void orc_permutation_build_pk(const u64* mapping, uint32_t P, uint32_t k, uint32_t ek, const u64* delta, const u64* omega, const u64* omega_inv,
                              const u64* ifft_divisor, const u64* ext_omega, const u64* zeta_powers, int threads, u64* out_perm, u64* out_polys,
                              u64* out_cosets) {
    const size_t n = (size_t)1 << k, en = (size_t)1 << ek;
    sigma_columns(mapping, P, k, fr_of(delta), fr_of(omega), threads, (Fr*)out_perm);
    const Fr zeta[3] = {fr_of(zeta_powers), fr_of(zeta_powers + 4), fr_of(zeta_powers + 8)};
    for (size_t i = 0; i < P; ++i) {
        Fr* poly = (Fr*)out_polys + i * n;
        memcpy(poly, (Fr*)out_perm + i * n, n * 32);
        lagrange_to_coeff(poly, k, fr_of(omega_inv), fr_of(ifft_divisor), threads);
        coeff_to_extended(poly, k, ek, fr_of(ext_omega), zeta, threads, (Fr*)out_cosets + i * en);
    }
}

// keygen_pk's indicator block -> l0, l_last, l_active_row (2^ek x 4 each)
void orc_lagrange_indicators(uint32_t k, uint32_t ek, uint32_t bf, const u64* omega_inv, const u64* ifft_divisor, const u64* ext_omega,
                             const u64* zeta_powers, int threads, u64* out_l0, u64* out_l_last, u64* out_l_active) {
    const size_t n = (size_t)1 << k, en = (size_t)1 << ek;
    const Fr zeta[3] = {fr_of(zeta_powers), fr_of(zeta_powers + 4), fr_of(zeta_powers + 8)};
    auto ext = [&](std::vector<Fr> lagrange, Fr* out) {
        lagrange_to_coeff(lagrange.data(), k, fr_of(omega_inv), fr_of(ifft_divisor), threads);
        coeff_to_extended(lagrange.data(), k, ek, fr_of(ext_omega), zeta, threads, out);
    };
    std::vector<Fr> l0(n, Fr::zero()), l_blind(n, Fr::zero()), l_last(n, Fr::zero());
    l0[0] = Fr::one();
    for (size_t t = 0; t < bf; ++t) l_blind[n - 1 - t] = Fr::one();
    l_last[n - bf - 1] = Fr::one();
    std::vector<Fr> blind_ext(en);
    ext(l0, (Fr*)out_l0);
    ext(l_blind, blind_ext.data());
    ext(l_last, (Fr*)out_l_last);
    Fr* active = (Fr*)out_l_active;
    const Fr* last = (const Fr*)out_l_last;
    for (size_t t = 0; t < en; ++t) active[t] = Fr::one() - (last[t] + blind_ext[t]);
}

}  // extern "C"
