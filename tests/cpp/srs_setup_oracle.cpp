// ORACLE (test infrastructure only): CPU restatement of halo2_proofs ParamsKZG::setup
// ([UP] halo2_proofs/src/poly/kzg/commitment.rs @ v2023_02_02) and of a plain [k]G, on the field and group code of
// oracle/h2_oracle.cpp.  It follows upstream's algorithm, deliberately not the device's: per chunk of `parallelize` a
// `current_g *= s` chain of full variable-base scalar multiplications for g, and per point one pow_vartime, one inversion
// and one scalar multiplication of the generator for g_lagrange, then batch normalisation.  std::thread in place of rayon.
// Also the timed CPU baseline of tools/srs_setup_bench.py ("CPU restatement", not the reference itself).
#include "../../oracle/h2_oracle.cpp"

namespace {

// [e]P by double-and-add over the canonical bits of e (halo2curves' `impl Mul<Fr> for G1`)
G1 g1_mul(const G1& p, const Fr& e_mont) {
    const Fr e = e_mont.from_mont();
    G1 acc = G1::identity();
    for (int i = 255; i >= 0; --i) {
        acc = g1_double(acc);
        if ((e.l[i / 64] >> (i % 64)) & 1) acc = g1_add(acc, p);
    }
    return acc;
}

G1 generator() {
    G1 g;
    g.x = Fq::one();
    g.y = Fq::one().dbl();
    g.z = Fq::one();
    return g;
}

// C::Curve::batch_normalize of one chunk (Montgomery's trick, identity -> (0, 0))
void batch_normalize(const std::vector<G1>& jac, u64* out_aff) {
    const size_t m = jac.size();
    std::vector<Fq> pre(m);
    Fq run = Fq::one();
    for (size_t i = 0; i < m; ++i) { pre[i] = run; if (!jac[i].z.is_zero()) run = run * jac[i].z; }
    Fq inv = run.inv();
    for (size_t i = m; i-- > 0;) {
        G1Affine a;
        if (jac[i].z.is_zero()) { a.x = Fq::zero(); a.y = Fq::zero(); }
        else {
            Fq zi = inv * pre[i];
            inv = inv * jac[i].z;
            Fq zi2 = zi.sqr();
            a.x = jac[i].x * zi2;
            a.y = jac[i].y * zi2 * zi;
        }
        memcpy(out_aff + 8 * i, &a, 64);
    }
}

// rayon-style `parallelize`: f(lo, hi) on `threads` contiguous chunks
template <class F>
void parallelize(size_t n, int threads, F f) {
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

Fr pow_u64(const Fr& b, u64 e) {
    const u64 w[4] = {e, 0, 0, 0};
    return b.pow(w);
}

}  // namespace

extern "C" {

// out[i] = [scalars[i]] G, affine (identity (0, 0))
void orc_g1_generator_mul(const u64* scalars, size_t n, int threads, u64* out_aff) {
    parallelize(n, threads, [=](size_t lo, size_t hi) {
        std::vector<G1> jac(hi - lo);
        for (size_t i = lo; i < hi; ++i) { Fr e; memcpy(e.l, scalars + 4 * i, 32); jac[i - lo] = g1_mul(generator(), e); }
        batch_normalize(jac, out_aff + 8 * lo);
    });
}

// ParamsKZG::<Bn256>::setup(k, rng) with s = the rng's Fr::random; out_g, out_gl: 2^k affine points each
void orc_srs_setup(uint32_t k, const u64* s_words, int threads, u64* out_g, u64* out_gl) {
    const size_t n = (size_t)1 << k;
    Fr s; memcpy(s.l, s_words, 32);
    const G1 g1 = generator();
    parallelize(n, threads, [&](size_t lo, size_t hi) {
        std::vector<G1> g(hi - lo);
        G1 current_g = g1_mul(g1, pow_u64(s, lo));
        for (size_t i = lo; i < hi; ++i) { g[i - lo] = current_g; current_g = g1_mul(current_g, s); }
        batch_normalize(g, out_g + 8 * lo);
    });
    // root = Fr::ROOT_OF_UNITY squared S - k times; n_inv = Fr::from(n).invert(); multiplier = (s^n - 1) n_inv
    Fr root; const u64 rou[4] = {0x9632c7c5b639feb8ULL, 0x985ce3400d0ff299ULL, 0xb2dd880001b0ecd8ULL, 0x1d69070d6d98ce29ULL};
    memcpy(root.l, rou, 32);
    for (uint32_t i = k; i < 28; ++i) root = root.sqr();
    Fr nf = Fr::zero(); nf.l[0] = n; nf = nf.to_mont();
    const Fr multiplier = (pow_u64(s, n) - Fr::one()) * nf.inv();
    parallelize(n, threads, [&](size_t lo, size_t hi) {
        std::vector<G1> g(hi - lo);
        for (size_t i = lo; i < hi; ++i) {
            const Fr root_pow = pow_u64(root, i);
            const Fr scalar = multiplier * root_pow * (s - root_pow).inv();
            g[i - lo] = g1_mul(g1, scalar);
        }
        batch_normalize(g, out_gl + 8 * lo);
    });
}

}  // extern "C"
