// ORACLE (test infrastructure only): CPU restatement of ProverSHPLONK::create_proof ([UP] halo2_proofs/src/poly/kzg/multiopen/shplonk/
// prover.rs and shplonk.rs's construct_intermediate_sets @ v2023_02_02, as recalled), step by step in upstream's order, on the field and
// MSM code of oracle/h2_oracle.cpp.  It follows upstream's algorithm, deliberately not the device's:
//
//   construct_intermediate_sets: every distinct polynomial (identity = index here, pointer upstream) collects its points; polynomials
//       with equal point sets form a rotation set, sets ordered by their first polynomial's first appearance, members likewise;
//   per set: every member evaluated at every point with eval_polynomial, r_ij = lagrange_interpolate(points, evals) (upstream's
//       algorithm: pairwise denominators batch-inverted, the basis products built one factor at a time), the numerator
//       sum_j y^j (p_ij - r_ij), div_by_vanishing = one kate_division per point, resized to n;
//   h_x = sum_i v^i q_i, h1 = commit(h_x);
//   per set: z_i = prod over T \ S_i of (u - t), l_i = z_i sum_j y^j (p_ij - r_ij(u)); l = sum_i v^i l_i - Z_T(u) h_x, l(u) == 0 asserted;
//   h' = kate_division(l, u) * z_0^-1 (n - 1 coefficients), h2 = commit(h').
// Also the timed CPU reference of tools/shplonk_bench.py.
#include "../../oracle/h2_oracle.cpp"

namespace {

Fr fr_of(const u64* w) { Fr r; memcpy(r.l, w, 32); return r; }

// [UP] arithmetic.rs eval_polynomial
Fr eval_poly(const std::vector<Fr>& a, const Fr& x) {
    Fr r = Fr::zero();
    for (size_t i = a.size(); i-- > 0;) r = r * x + a[i];
    return r;
}

// [UP] arithmetic.rs kate_division: a(X) / (X - b), a.len() - 1 coefficients
std::vector<Fr> kate_division(const std::vector<Fr>& a, const Fr& b) {
    if (a.size() <= 1) return {};
    std::vector<Fr> q(a.size() - 1, Fr::zero());
    Fr tmp = Fr::zero();
    for (size_t i = a.size() - 1; i >= 1; --i) {
        Fr lead = a[i] + tmp;
        q[i - 1] = lead;
        tmp = lead * b;
    }
    return q;
}

// [UP] arithmetic.rs lagrange_interpolate
std::vector<Fr> lagrange_interpolate(const std::vector<Fr>& points, const std::vector<Fr>& evals) {
    const size_t m = points.size();
    if (m == 1) return {evals[0]};
    std::vector<std::vector<Fr>> denoms(m);
    for (size_t j = 0; j < m; ++j)
        for (size_t k = 0; k < m; ++k) if (k != j) denoms[j].push_back(points[j] - points[k]);
    for (auto& d : denoms) for (auto& x : d) x = x.inv();      // batch_invert: the same values
    std::vector<Fr> final_poly(m, Fr::zero());
    for (size_t j = 0; j < m; ++j) {
        std::vector<Fr> tmp{Fr::one()};
        size_t di = 0;
        for (size_t k = 0; k < m; ++k) {
            if (k == j) continue;
            const Fr denom = denoms[j][di++], x_k = points[k];
            std::vector<Fr> product(tmp.size() + 1, Fr::zero());
            // product[c] = a[c] * (-denom * x_k) + b[c] * denom with a = tmp ++ [0], b = [0] ++ tmp
            for (size_t c = 0; c < product.size(); ++c) {
                const Fr a = c < tmp.size() ? tmp[c] : Fr::zero();
                const Fr b = c > 0 ? tmp[c - 1] : Fr::zero();
                product[c] = a * (denom * x_k).neg() + b * denom;
            }
            tmp.swap(product);
        }
        for (size_t c = 0; c < m; ++c) final_poly[c] = final_poly[c] + tmp[c] * evals[j];
    }
    return final_poly;
}

Fr vanishing_at(const std::vector<Fr>& pts, const Fr& u) {
    Fr r = Fr::one();
    for (auto& t : pts) r = r * (u - t);
    return r;
}

G1 commit(const std::vector<Fr>& poly, const u64* g_affine, int threads) {
    return best_multiexp(poly.data(), (const G1Affine*)g_affine, poly.size(), threads);
}

void put_jac(const G1& p, u64* out) { memcpy(out, &p, 96); }

}  // namespace

extern "C" {

// polys: n_polys host arrays of n coefficients; queries (q_poly[i], q_points[4 i]); g_affine: at least n points.
// Returns 0, or 1 where upstream panics (z_0 = 0, u in T \ S_0).  h1_jac / h2_jac: 12 words each.
int orc_shplonk(const u64* const* polys, uint32_t n_polys, size_t n, const uint32_t* q_poly, const u64* q_points, uint32_t nq, const u64* g_affine,
                const u64* y_w, const u64* v_w, const u64* u_w, int threads, u64* h1_jac, u64* h2_jac) {
    (void)n_polys;
    const Fr y = fr_of(y_w), v = fr_of(v_w), u = fr_of(u_w);
    // construct_intermediate_sets
    std::vector<uint32_t> order;                       // distinct polynomials, first appearance
    std::map<uint32_t, std::vector<Fr>> points_of;     // their distinct points, first appearance
    std::vector<Fr> super_set;
    auto contains = [](const std::vector<Fr>& s, const Fr& x) { for (auto& e : s) if (e == x) return true; return false; };
    for (uint32_t i = 0; i < nq; ++i) {
        const Fr x = fr_of(q_points + 4 * (size_t)i);
        if (!points_of.count(q_poly[i])) order.push_back(q_poly[i]);
        std::vector<Fr>& ps = points_of[q_poly[i]];
        if (!contains(ps, x)) ps.push_back(x);
        if (!contains(super_set, x)) super_set.push_back(x);
    }
    auto same_set = [&](const std::vector<Fr>& a, const std::vector<Fr>& b) {
        if (a.size() != b.size()) return false;
        for (auto& x : a) if (!contains(b, x)) return false;
        return true;
    };
    std::vector<std::vector<uint32_t>> set_polys;
    std::vector<std::vector<Fr>> set_points;
    for (uint32_t p : order) {
        size_t i = 0;
        while (i < set_points.size() && !same_set(set_points[i], points_of[p])) ++i;
        if (i == set_points.size()) { set_points.push_back(points_of[p]); set_polys.emplace_back(); }
        set_polys[i].push_back(p);
    }
    auto poly_of = [&](uint32_t p) { return std::vector<Fr>((const Fr*)polys[p], (const Fr*)polys[p] + n); };
    // quotient_contribution of every set
    std::vector<Fr> h_x(n, Fr::zero());
    std::vector<std::vector<std::vector<Fr>>> r_of(set_polys.size());
    Fr vi = Fr::one();
    for (size_t i = 0; i < set_polys.size(); ++i) {
        std::vector<Fr> numerator(n, Fr::zero());
        Fr yj = Fr::one();
        for (uint32_t p : set_polys[i]) {
            const std::vector<Fr> poly = poly_of(p);
            std::vector<Fr> evals;
            for (auto& x : set_points[i]) evals.push_back(eval_poly(poly, x));
            std::vector<Fr> r = lagrange_interpolate(set_points[i], evals);
            std::vector<Fr> diff = poly;
            for (size_t c = 0; c < r.size(); ++c) diff[c] = diff[c] - r[c];
            for (size_t c = 0; c < n; ++c) numerator[c] = numerator[c] + diff[c] * yj;
            r_of[i].push_back(r);
            yj = yj * y;
        }
        std::vector<Fr> q = numerator;
        for (auto& x : set_points[i]) q = kate_division(q, x);
        q.resize(n, Fr::zero());
        for (size_t c = 0; c < n; ++c) h_x[c] = h_x[c] + q[c] * vi;
        vi = vi * v;
    }
    const G1 h1 = commit(h_x, g_affine, threads);
    // linearisation_contribution of every set
    std::vector<Fr> l_x(n, Fr::zero());
    Fr z0 = Fr::zero();
    vi = Fr::one();
    for (size_t i = 0; i < set_polys.size(); ++i) {
        std::vector<Fr> diffs;
        for (auto& t : super_set) if (!contains(set_points[i], t)) diffs.push_back(t);
        const Fr z_i = vanishing_at(diffs, u);
        if (i == 0) z0 = z_i;
        std::vector<Fr> acc(n, Fr::zero());
        Fr yj = Fr::one();
        for (size_t j = 0; j < set_polys[i].size(); ++j) {
            std::vector<Fr> poly = poly_of(set_polys[i][j]);
            poly[0] = poly[0] - eval_poly(r_of[i][j], u);
            for (size_t c = 0; c < n; ++c) acc[c] = acc[c] + poly[c] * yj;
            yj = yj * y;
        }
        for (size_t c = 0; c < n; ++c) l_x[c] = l_x[c] + acc[c] * z_i * vi;
        vi = vi * v;
    }
    const Fr zt = vanishing_at(super_set, u);
    for (size_t c = 0; c < n; ++c) l_x[c] = l_x[c] - h_x[c] * zt;
    if (!eval_poly(l_x, u).is_zero()) return 2;         // upstream's sanity assertion
    if (z0.is_zero()) return 1;                          // invert().unwrap()
    std::vector<Fr> h = kate_division(l_x, u);
    const Fr z0_inv = z0.inv();
    for (auto& c : h) c = c * z0_inv;
    const G1 h2 = commit(h, g_affine, threads);
    put_jac(h1, h1_jac);
    put_jac(h2, h2_jac);
    return 0;
}

}  // extern "C"
