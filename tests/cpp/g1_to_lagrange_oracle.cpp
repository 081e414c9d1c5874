// ORACLE (test infrastructure only): CPU restatement of halo2_proofs' g_to_lagrange ([UP] halo2_proofs/src/arithmetic.rs
// @ v2023_02_02, as recalled; SURVEY.md Appendix B restates best_fft the same way), on the field and group code of
// oracle/h2_oracle.cpp and the scalar multiplication of srs_setup_oracle.cpp:
//
//     pub fn g_to_lagrange<C: CurveAffine>(g_projective: Vec<C::Curve>, k: u32) -> Vec<C> {
//         let n_inv = C::Scalar::TWO_INV.pow_vartime(&[k as u64, 0, 0, 0]);
//         let mut omega_inv = C::Scalar::ROOT_OF_UNITY_INV;
//         for _ in k..C::Scalar::S { omega_inv = omega_inv.square(); }
//         let mut g_lagrange_projective = g_projective;
//         best_fft(&mut g_lagrange_projective, omega_inv, k);
//         parallelize(&mut g_lagrange_projective, |g, _| for g in g.iter_mut() { *g *= n_inv; });
//         // then C::Curve::batch_normalize per parallelize chunk
//     }
//
// best_fft over C::Curve: bit-reversal permutation, then recursive_butterfly_arithmetic with `t = b; t *= twiddle;
// b = a - t; a += t` (the twiddle-one case without the multiplication), each `*=` a full double-and-add.  It follows
// upstream's algorithm, deliberately not the device's (DIT here, DIF there).  std::thread in place of rayon.  Also the timed
// CPU baseline of tools/g1_to_lagrange_bench.py ("CPU restatement", not the reference itself).
#include "srs_setup_oracle.cpp"

namespace {

G1 g1_neg(const G1& p) {
    G1 r = p;
    r.y = p.y.neg();
    return r;
}

void recursive_butterfly_g1(G1* a, size_t n, size_t twiddle_chunk, const Fr* tw, int par_depth) {
    if (n == 2) { G1 t = a[1]; a[1] = g1_add(a[0], g1_neg(t)); a[0] = g1_add(a[0], t); return; }
    const size_t half = n / 2;
    if (par_depth > 0) {       // rayon::join
        std::thread other([=] { recursive_butterfly_g1(a + half, half, twiddle_chunk * 2, tw, par_depth - 1); });
        recursive_butterfly_g1(a, half, twiddle_chunk * 2, tw, par_depth - 1);
        other.join();
    } else {
        recursive_butterfly_g1(a, half, twiddle_chunk * 2, tw, 0);
        recursive_butterfly_g1(a + half, half, twiddle_chunk * 2, tw, 0);
    }
    G1* l = a;
    G1* r = a + half;
    { G1 t = r[0]; r[0] = g1_add(l[0], g1_neg(t)); l[0] = g1_add(l[0], t); }      // twiddle one
    auto body = [=](size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; ++i) { G1 t = g1_mul(r[i], tw[i * twiddle_chunk]); r[i] = g1_add(l[i], g1_neg(t)); l[i] = g1_add(l[i], t); }
    };
    if (par_depth > 0 && half >= 64) {
        const int T = 1 << par_depth;
        std::vector<std::thread> th;
        const size_t per = (half + T - 1) / T;
        for (int t = 0; t < T; ++t) {
            const size_t lo = std::max<size_t>(1, t * per), hi = std::min(half, (t + 1) * per);
            if (lo < hi) th.emplace_back(body, lo, hi);
        }
        for (auto& x : th) x.join();
    } else body(1, half);
}

}  // namespace

extern "C" {

// g_to_lagrange of n = 2^k affine points (identity (0, 0)) -> n affine points
void orc_g1_to_lagrange(const u64* g_aff, uint32_t k, int threads, u64* out_aff) {
    const size_t n = (size_t)1 << k;
    if (threads < 1) threads = 1;
    std::vector<G1> a(n);
    for (size_t i = 0; i < n; ++i) {
        G1Affine p; memcpy(&p, g_aff + 8 * i, 64);
        a[i].x = p.x; a[i].y = p.is_identity() ? Fq::one() : p.y; a[i].z = p.is_identity() ? Fq::zero() : Fq::one();
    }
    // omega_inv = ROOT_OF_UNITY_INV squared S - k times; n_inv = TWO_INV^k
    Fr root; const u64 rou[4] = {0x9632c7c5b639feb8ULL, 0x985ce3400d0ff299ULL, 0xb2dd880001b0ecd8ULL, 0x1d69070d6d98ce29ULL};
    memcpy(root.l, rou, 32);
    Fr omega_inv = root.inv();
    for (uint32_t i = k; i < 28; ++i) omega_inv = omega_inv.sqr();
    Fr two = Fr::one().dbl();
    const Fr n_inv = pow_u64(two.inv(), k);
    // best_fft
    for (size_t i = 0; i < n; ++i) { const size_t ri = bitreverse(i, k); if (i < ri) std::swap(a[i], a[ri]); }
    if (n >= 2) {
        std::vector<Fr> tw(n / 2);
        tw[0] = Fr::one();
        for (size_t i = 1; i < n / 2; ++i) tw[i] = tw[i - 1] * omega_inv;
        int depth = 0;
        while ((1 << (depth + 1)) <= threads) ++depth;
        if ((unsigned)depth >= k) depth = k > 1 ? (int)k - 1 : 0;
        recursive_butterfly_g1(a.data(), n, 1, tw.data(), depth);
    }
    parallelize(n, threads, [&](size_t lo, size_t hi) {
        std::vector<G1> chunk(a.begin() + lo, a.begin() + hi);
        for (G1& p : chunk) p = g1_mul(p, n_inv);
        batch_normalize(chunk, out_aff + 8 * lo);
    });
}

// out[i] = [scalars[i]] points[i], affine
void orc_g1_mul_points(const u64* points_aff, const u64* scalars, size_t n, int threads, u64* out_aff) {
    parallelize(n, threads, [=](size_t lo, size_t hi) {
        std::vector<G1> jac(hi - lo);
        for (size_t i = lo; i < hi; ++i) {
            G1Affine p; memcpy(&p, points_aff + 8 * i, 64);
            G1 q; q.x = p.x; q.y = p.is_identity() ? Fq::one() : p.y; q.z = p.is_identity() ? Fq::zero() : Fq::one();
            Fr e; memcpy(e.l, scalars + 4 * i, 32);
            jac[i - lo] = g1_mul(q, e);
        }
        batch_normalize(jac, out_aff + 8 * lo);
    });
}

}  // extern "C"
