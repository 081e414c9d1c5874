// ORACLE (test infrastructure only): CPU restatement of ProverGWC::create_proof ([UP] halo2_proofs/src/poly/kzg/multiopen/gwc/prover.rs
// and gwc.rs's construct_intermediate_sets @ v2023_02_02, as recalled), step by step in upstream's order, on the field and MSM code of
// oracle/h2_oracle.cpp.  It follows upstream literally, deliberately not the device:
//
//   construct_intermediate_sets: the distinct points in first-appearance order, each with every query at it in query order (a query
//       listed twice stays twice);
//   per point z: poly_batch = sum_j v^j p_j, eval_batch = sum_j v^j eval_polynomial(p_j, z) (j restarts at 0 for every point),
//       poly_batch[0] -= eval_batch (Sub<F> for Polynomial<Coeff>), W = commit(kate_division(poly_batch, z)) over g[0 .. n-1).
// The device drops the evaluations and the subtraction (kate_division never reads coefficient 0); agreement with this file is the
// test of that.  Also the timed CPU reference of tools/gwc_bench.py.
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

}  // namespace

extern "C" {

// polys: n_polys host arrays of n coefficients; queries (q_poly[i], q_points[4 i]); g_affine: at least n - 1 points.
// Writes one Jacobian W (12 words) per distinct point to w_jac and returns the number of points.
uint32_t orc_gwc(const u64* const* polys, uint32_t n_polys, size_t n, const uint32_t* q_poly, const u64* q_points, uint32_t nq, const u64* g_affine,
                 const u64* v_w, int threads, u64* w_jac) {
    (void)n_polys;
    const Fr v = fr_of(v_w);
    std::vector<Fr> points;
    std::vector<std::vector<uint32_t>> at;
    for (uint32_t i = 0; i < nq; ++i) {
        const Fr x = fr_of(q_points + 4 * (size_t)i);
        size_t t = 0;
        while (t < points.size() && !(points[t] == x)) ++t;
        if (t == points.size()) { points.push_back(x); at.emplace_back(); }
        at[t].push_back(q_poly[i]);
    }
    for (size_t t = 0; t < points.size(); ++t) {
        std::vector<Fr> poly_batch(n, Fr::zero());
        Fr eval_batch = Fr::zero(), vj = Fr::one();
        for (uint32_t p : at[t]) {
            const std::vector<Fr> poly((const Fr*)polys[p], (const Fr*)polys[p] + n);
            for (size_t c = 0; c < n; ++c) poly_batch[c] = poly_batch[c] + poly[c] * vj;
            eval_batch = eval_batch + eval_poly(poly, points[t]) * vj;
            vj = vj * v;
        }
        poly_batch[0] = poly_batch[0] - eval_batch;
        const std::vector<Fr> q = kate_division(poly_batch, points[t]);
        const G1 w = best_multiexp(q.data(), (const G1Affine*)g_affine, q.size(), threads);
        memcpy(w_jac + 12 * t, &w, 96);
    }
    return (uint32_t)points.size();
}

}  // extern "C"
