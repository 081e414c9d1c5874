// h2b200.hpp -- C++ host-side mirror of the reference's operator interface for the hot path, over the C ABI of
// include/h2b200.h.  The reference is Rust (halo2_proofs / halo2curves, un-vendored git dependencies of
// DCMMC/halo2-scaffold: Cargo.toml:13,16); this image has no Rust toolchain, so the host side above the C ABI is
// written in C++ with the SAME names, argument meaning and error behaviour as the Rust items it mirrors:
//
//   h2b200::arithmetic::best_multiexp   <- [UP] halo2_proofs::arithmetic::best_multiexp   (SURVEY.md row a1)
//   h2b200::arithmetic::best_fft        <- [UP] halo2_proofs::arithmetic::best_fft        (row a3)
//   h2b200::poly::EvaluationDomain      <- [UP] halo2_proofs::poly::EvaluationDomain      (row a6, Appendix B)
//   h2b200::poly::kzg::ParamsKZG        <- [UP] halo2_proofs::poly::kzg::commitment::ParamsKZG::{commit, commit_lagrange,
//                                          read_custom, write_custom} (rows a7, f4)
//   h2b200::plonk::evaluation::GraphEvaluator, h2b200::plonk::{permutation, lookup}::*
//                                       <- [UP] halo2_proofs::plonk::evaluation / permutation::prover / lookup::prover (rows f2, f3)
//
// Rust `assert!`/`panic!` become h2b200::Panic (a std::logic_error); a non-zero return of the C ABI becomes
// h2b200::Panic carrying h2b_last_error(), exactly what the Rust shim of INTEGRATION.md does.
// Vector work runs on the GPU; only the per-domain scalar constants (omega, divisors, zeta powers) are computed on
// the host, as EvaluationDomain::new does in the reference.  Header-only; link with -lh2b200.
#pragma once
#include <cstdint>
#include <cstring>
#include <cstdio>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/h2b200.h"

namespace h2b200 {

struct Panic : std::logic_error {
    using std::logic_error::logic_error;
};

inline void check(int rc, const char* what) {
    if (rc != H2B_OK) throw Panic(std::string(what) + ": " + h2b_last_error());
}

// halo2curves 0.3.x memory layouts (SURVEY.md section 8 "Sizes")
struct Fr { uint64_t l[4]; };                 // Montgomery, R = 2^256, fully reduced
struct Fq { uint64_t l[4]; };
struct G1Affine { Fq x, y; };                 // (0, 0) = identity
struct G1 { Fq x, y, z; };                    // Jacobian, z == 0 = identity
static_assert(sizeof(Fr) == 32 && sizeof(G1Affine) == 64 && sizeof(G1) == 96, "layouts must match halo2curves");

inline bool operator==(const Fr& a, const Fr& b) { return std::memcmp(&a, &b, sizeof(Fr)) == 0; }

// ---- scalar Fr arithmetic on the host (domain constants only) ----------------------------------------------------
namespace fr {
typedef unsigned __int128 u128;
static const uint64_t MODULUS[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
static const uint64_t INV = 0xc2e1f593efffffffull;                 // -r^-1 mod 2^64
static const uint64_t R2[4] = {0x1bb8e645ae216da7ull, 0x53fe3ab1e35c59e3ull, 0x8c49833d53bb8085ull, 0x0216d0b17f4e44a5ull};
static const uint32_t S = 28;                                      // two-adicity
// canonical (non-Montgomery) integers
static const uint64_t ROOT_OF_UNITY_CANON[4] = {0xd34f1ed960c37c9cull, 0x3215cf6dd39329c8ull, 0x98865ea93dd31f74ull, 0x03ddb9f5166d18b7ull};
static const uint64_t ZETA_CANON[4] = {0xb8ca0b2d36636f23ull, 0xcc37a73fec2bc5e9ull, 0x048b6e193fd84104ull, 0x30644e72e131a029ull};

inline bool geq_modulus(const uint64_t t[4]) {
    for (int i = 3; i >= 0; --i) {
        if (t[i] > MODULUS[i]) return true;
        if (t[i] < MODULUS[i]) return false;
    }
    return true;
}
// Montgomery product a * b / R mod r (coarsely integrated operand scanning)
inline Fr mul(const Fr& a, const Fr& b) {
    uint64_t t[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 4; ++i) {
        u128 carry = 0;
        for (int j = 0; j < 4; ++j) {
            u128 cur = (u128)a.l[j] * b.l[i] + t[j] + carry;
            t[j] = (uint64_t)cur;
            carry = cur >> 64;
        }
        u128 top = (u128)t[4] + carry;
        t[4] = (uint64_t)top;
        t[5] = (uint64_t)(top >> 64);
        uint64_t m = t[0] * INV;
        carry = ((u128)m * MODULUS[0] + t[0]) >> 64;
        for (int j = 1; j < 4; ++j) {
            u128 cur = (u128)m * MODULUS[j] + t[j] + carry;
            t[j - 1] = (uint64_t)cur;
            carry = cur >> 64;
        }
        top = (u128)t[4] + carry;
        t[3] = (uint64_t)top;
        t[4] = t[5] + (uint64_t)(top >> 64);
    }
    if (t[4] || geq_modulus(t)) {
        u128 borrow = 0;
        for (int i = 0; i < 4; ++i) {
            u128 d = (u128)t[i] - MODULUS[i] - borrow;
            t[i] = (uint64_t)d;
            borrow = (d >> 64) & 1;
        }
    }
    Fr r;
    std::memcpy(r.l, t, 32);
    return r;
}
inline Fr from_canonical(const uint64_t c[4]) {
    Fr a, r2;
    std::memcpy(a.l, c, 32);
    std::memcpy(r2.l, R2, 32);
    return mul(a, r2);
}
inline Fr from_u64(uint64_t v) {
    uint64_t c[4] = {v, 0, 0, 0};
    return from_canonical(c);
}
inline Fr one() { return from_u64(1); }
inline Fr sub(const Fr& a, const Fr& b) {
    Fr r; u128 bw = 0;
    for (int i = 0; i < 4; ++i) { u128 d = (u128)a.l[i] - b.l[i] - (uint64_t)bw; r.l[i] = (uint64_t)d; bw = (d >> 64) & 1; }
    if (bw) { u128 c = 0; for (int i = 0; i < 4; ++i) { c += (u128)r.l[i] + MODULUS[i]; r.l[i] = (uint64_t)c; c >>= 64; } }
    return r;
}
inline Fr square(const Fr& a) { return mul(a, a); }
inline Fr pow(const Fr& a, const uint64_t e[4]) {
    Fr r = one();
    for (int w = 3; w >= 0; --w)
        for (int i = 63; i >= 0; --i) {
            r = square(r);
            if ((e[w] >> i) & 1) r = mul(r, a);
        }
    return r;
}
inline Fr invert(const Fr& a) {                       // a^(r-2)
    uint64_t e[4] = {MODULUS[0] - 2, MODULUS[1], MODULUS[2], MODULUS[3]};
    return pow(a, e);
}
inline Fr root_of_unity() { return from_canonical(ROOT_OF_UNITY_CANON); }
inline Fr zeta() { return from_canonical(ZETA_CANON); }
}  // namespace fr

// ---- process-wide initialisation ---------------------------------------------------------------------------------
inline void ensure_init() {
    if (h2b_device_count() == 0) check(h2b_init(0), "h2b_init");
}

// ---- halo2_proofs::arithmetic -----------------------------------------------------------------------------------
namespace arithmetic {

// pub fn best_multiexp<C: CurveAffine>(coeffs: &[C::Scalar], bases: &[C]) -> C::Curve
inline G1 best_multiexp(const Fr* coeffs, size_t coeffs_len, const G1Affine* bases, size_t bases_len) {
    if (coeffs_len != bases_len) throw Panic("assertion failed: `(left == right)` coeffs.len() == bases.len()");
    ensure_init();
    G1 out;
    check(h2b_msm_bn254_g1(reinterpret_cast<const uint64_t*>(coeffs), reinterpret_cast<const uint64_t*>(bases), coeffs_len,
                           reinterpret_cast<uint64_t*>(&out)), "best_multiexp");
    return out;
}
inline G1 best_multiexp(const std::vector<Fr>& coeffs, const std::vector<G1Affine>& bases) {
    return best_multiexp(coeffs.data(), coeffs.size(), bases.data(), bases.size());
}

// pub fn best_fft<G: Group>(a: &mut [G], omega: G::Scalar, log_n: u32)      (G = Fr)
inline void best_fft(Fr* a, size_t len, const Fr& omega, uint32_t log_n) {
    if (log_n > 63 || len != ((size_t)1 << log_n)) throw Panic("assertion failed: a.len() == 1 << log_n");
    ensure_init();
    check(h2b_ntt_bn254_fr(reinterpret_cast<uint64_t*>(a), omega.l, log_n), "best_fft");
}
inline void best_fft(std::vector<Fr>& a, const Fr& omega, uint32_t log_n) { best_fft(a.data(), a.size(), omega, log_n); }

}  // namespace arithmetic

// ---- a device buffer (RAII) for the device-resident callers --------------------------------------------------------
class DeviceBuffer {
  public:
    DeviceBuffer(int device, size_t bytes) : device_(device) { check(h2b_dev_alloc(device, bytes, &p_), "h2b_dev_alloc"); }
    ~DeviceBuffer() { if (p_) h2b_dev_free(device_, p_); }
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    void* get() const { return p_; }
  private:
    int device_;
    void* p_ = nullptr;
};

namespace poly {

// pub struct EvaluationDomain<G: Group>; EvaluationDomain::new(j, k)
class EvaluationDomain {
  public:
    EvaluationDomain(uint32_t j, uint32_t k, int device = 0) : device_(device), k_(k) {
        ensure_init();
        if (j < 2) throw Panic("EvaluationDomain::new: j must be at least 2");
        quotient_poly_degree_ = j - 1;
        n_ = (uint64_t)1 << k;
        extended_k_ = k;
        while (((uint64_t)1 << extended_k_) < n_ * quotient_poly_degree_) ++extended_k_;
        if (extended_k_ > fr::S) throw Panic("EvaluationDomain::new: extended domain exceeds the two-adicity of the field");
        extended_omega_ = fr::root_of_unity();
        for (uint32_t i = extended_k_; i < fr::S; ++i) extended_omega_ = fr::square(extended_omega_);
        omega_ = extended_omega_;
        for (uint32_t i = k; i < extended_k_; ++i) omega_ = fr::square(omega_);
        omega_inv_ = fr::invert(omega_);
        extended_omega_inv_ = fr::invert(extended_omega_);
        ifft_divisor_ = fr::invert(fr::from_u64(n_));
        extended_ifft_divisor_ = fr::invert(fr::from_u64((uint64_t)1 << extended_k_));
        g_coset_ = fr::zeta();
        g_coset_inv_ = fr::square(g_coset_);
        // t_evaluations: 1 / (X^n - 1) on the zeta coset repeats with period 2^(extended_k - k)
        const uint64_t e[4] = {n_, 0, 0, 0};
        const Fr orig = fr::pow(g_coset_, e), step = fr::pow(extended_omega_, e);
        Fr cur = orig;
        do {
            t_evaluations_.push_back(fr::invert(fr::sub(cur, fr::one())));
            cur = fr::mul(cur, step);
        } while (!(cur == orig));
        if (t_evaluations_.size() != ((size_t)1 << (extended_k_ - k_))) throw Panic("EvaluationDomain::new: unexpected t_evaluations period");
    }
    uint32_t k() const { return k_; }
    uint32_t extended_k() const { return extended_k_; }
    size_t extended_len() const { return (size_t)1 << extended_k_; }
    uint64_t get_quotient_poly_degree() const { return quotient_poly_degree_; }
    const Fr& get_omega() const { return omega_; }
    const Fr& get_omega_inv() const { return omega_inv_; }
    const Fr& get_extended_omega() const { return extended_omega_; }
    const Fr& get_ifft_divisor() const { return ifft_divisor_; }
    const Fr& get_g_coset() const { return g_coset_; }
    const Fr& get_g_coset_inv() const { return g_coset_inv_; }
    int device() const { return device_; }

    // pub fn lagrange_to_coeff(&self, a: Polynomial<_, LagrangeCoeff>) -> Polynomial<_, Coeff>
    std::vector<Fr> lagrange_to_coeff(const std::vector<Fr>& a) const {
        if (a.size() != n_) throw Panic("assertion failed: a.len() == 1 << self.k");
        return run(a, n_, n_, n_, [&](void* d) {
            check(h2b_lagrange_to_coeff_dev(device_, d, k_, omega_inv_.l, ifft_divisor_.l, nullptr), "lagrange_to_coeff");
        });
    }
    // pub fn coeff_to_extended(&self, a: Polynomial<_, Coeff>) -> Polynomial<_, ExtendedLagrangeCoeff>
    std::vector<Fr> coeff_to_extended(const std::vector<Fr>& a) const {
        if (a.size() != n_) throw Panic("assertion failed: a.len() == 1 << self.k");
        const Fr z[3] = {fr::one(), g_coset_, g_coset_inv_};
        // only the 2^k coefficients cross PCIe; scaling by zeta powers, zero-padding and the extended FFT run on the device
        return run(a, extended_len(), n_, extended_len(), [&](void* d) {
            check(h2b_coeff_to_extended_dev(device_, d, k_, extended_k_, extended_omega_.l, z[0].l, nullptr), "coeff_to_extended");
        });
    }
    // pub fn extended_to_coeff(&self, a: Polynomial<_, ExtendedLagrangeCoeff>) -> Vec<G>
    std::vector<Fr> extended_to_coeff(const std::vector<Fr>& a) const {
        if (a.size() != extended_len()) throw Panic("assertion failed: a.len() == self.extended_len()");
        const Fr z[3] = {extended_ifft_divisor_, fr::mul(extended_ifft_divisor_, g_coset_inv_), fr::mul(extended_ifft_divisor_, g_coset_)};
        return run(a, n_ * quotient_poly_degree_, extended_len(), extended_len(), [&](void* d) {
            check(h2b_extended_to_coeff_dev(device_, d, extended_k_, extended_omega_inv_.l, z[0].l, nullptr), "extended_to_coeff");
        });
    }

    // pub fn divide_by_vanishing_poly(&self, a: Polynomial<_, ExtendedLagrangeCoeff>) -> Polynomial<_, ExtendedLagrangeCoeff>
    std::vector<Fr> divide_by_vanishing_poly(const std::vector<Fr>& a) const {
        if (a.size() != extended_len()) throw Panic("assertion failed: a.len() == self.extended_len()");
        return run(a, extended_len(), extended_len(), extended_len(), [&](void* d) {
            check(h2b_fr_scale_dev(device_, d, extended_len(), t_evaluations_[0].l, (int)t_evaluations_.size(), nullptr), "divide_by_vanishing_poly");
        });
    }

  private:
    // upload `upload_len` elements of `a` into a device buffer of `alloc_len`, run `steps`, download `out_len`
    template <class F>
    std::vector<Fr> run(const std::vector<Fr>& a, size_t out_len, size_t upload_len, size_t alloc_len, F steps) const {
        DeviceBuffer d(device_, alloc_len * sizeof(Fr));
        check(h2b_memcpy_h2d(device_, d.get(), a.data(), upload_len * sizeof(Fr)), "h2d");
        steps(d.get());
        check(h2b_dev_sync(device_), "sync");
        std::vector<Fr> out(out_len);
        check(h2b_memcpy_d2h(device_, out.data(), d.get(), out_len * sizeof(Fr)), "d2h");
        return out;
    }
    int device_;
    uint32_t k_, extended_k_;
    uint64_t n_, quotient_poly_degree_;
    Fr omega_, omega_inv_, extended_omega_, extended_omega_inv_, ifft_divisor_, extended_ifft_divisor_, g_coset_, g_coset_inv_;
    std::vector<Fr> t_evaluations_;
};

namespace kzg {

// pub struct ParamsKZG<E: Engine> { k, n, g: Vec<G1Affine>, g_lagrange: Vec<G1Affine>, ... }
// Both SRS vectors are registered once (device resident, window tables precomputed).
// pub enum SerdeFormat { Processed, RawBytes, RawBytesUnchecked }
enum class SerdeFormat : int { Processed = H2B_SERDE_PROCESSED, RawBytes = H2B_SERDE_RAW_BYTES, RawBytesUnchecked = H2B_SERDE_RAW_BYTES_UNCHECKED };

class ParamsKZG {
    friend class ProverSHPLONK;

  public:
    ParamsKZG(uint32_t k, const std::vector<G1Affine>& g, const std::vector<G1Affine>& g_lagrange, std::vector<uint8_t> g2_bytes = {})
        : k_(k), n_((uint64_t)1 << k), host_g_(g), host_g_lagrange_(g_lagrange), g2_bytes_(std::move(g2_bytes)) {
        ensure_init();
        if (g.size() != n_ || g_lagrange.size() != n_) throw Panic("ParamsKZG: g and g_lagrange must hold 2^k points");
        check(h2b_register_bases(reinterpret_cast<const uint64_t*>(g.data()), g.size(), &g_), "register g");
        check(h2b_register_bases(reinterpret_cast<const uint64_t*>(g_lagrange.data()), g_lagrange.size(), &g_lagrange_), "register g_lagrange");
    }
    // pub fn read_custom<R: io::Read>(reader, format) -> io::Result<Self>: decoded on the device, both vectors stay resident there
    ParamsKZG(const std::string& path, SerdeFormat format) {
        ensure_init();
        FILE* f = fopen(path.c_str(), "rb");
        unsigned char kb[4];
        if (!f || fread(kb, 1, 4, f) != 4) { if (f) fclose(f); throw Panic("ParamsKZG::read_custom: cannot read " + path); }
        fclose(f);
        k_ = (uint32_t)kb[0] | ((uint32_t)kb[1] << 8) | ((uint32_t)kb[2] << 16) | ((uint32_t)kb[3] << 24);
        if (k_ > 28) throw Panic("ParamsKZG::read_custom: k out of range");
        n_ = (uint64_t)1 << k_;
        host_g_.resize(n_); host_g_lagrange_.resize(n_);
        g2_bytes_.resize(256);
        size_t g2_len = 0;
        uint32_t k = 0;
        check(h2b_srs_read(path.c_str(), (int)format, &k, reinterpret_cast<uint64_t*>(host_g_.data()), reinterpret_cast<uint64_t*>(host_g_lagrange_.data()),
                           g2_bytes_.data(), g2_bytes_.size(), &g2_len, &g_, &g_lagrange_), "ParamsKZG::read_custom");
        g2_bytes_.resize(g2_len);
    }
    // pub fn setup<R: RngCore>(k: u32, rng: R) -> Self with the toxic waste s = Fr::random(rng) drawn by the caller: both vectors are
    // computed on the device and stay resident there.  g2_bytes (g2 | s_g2 as write_custom stores them) are the caller's (G2 is host work).
    static std::unique_ptr<ParamsKZG> setup(uint32_t k, const Fr& s, std::vector<uint8_t> g2_bytes = {}) {
        return std::unique_ptr<ParamsKZG>(new ParamsKZG(k, s, std::move(g2_bytes)));
    }
    // pub fn write_custom<W: io::Write>(&self, writer, format)
    void write_custom(const std::string& path, SerdeFormat format) const {
        check(h2b_srs_write(path.c_str(), (int)format, k_, reinterpret_cast<const uint64_t*>(host_g_.data()), reinterpret_cast<const uint64_t*>(host_g_lagrange_.data()),
                            g2_bytes_.data(), g2_bytes_.size()), "ParamsKZG::write_custom");
    }
    // fn downsize(&mut self, k: u32): g keeps its first 2^k points, g_lagrange is recomputed from them on the device
    // (g_to_lagrange); both become new resident sets and the old ones are given back.  g2_bytes are kept.
    void downsize(uint32_t k) {
        if (k > k_) throw Panic("ParamsKZG::downsize: k above the params' k");
        uint64_t hg = 0, hl = 0;
        std::vector<G1Affine> gl((size_t)1 << k);
        check(h2b_srs_downsize(g_, k, reinterpret_cast<uint64_t*>(gl.data()), &hg, &hl), "ParamsKZG::downsize");
        h2b_unregister_bases(g_);
        h2b_unregister_bases(g_lagrange_);
        g_ = hg; g_lagrange_ = hl;
        k_ = k; n_ = (uint64_t)1 << k;
        host_g_.resize(n_);
        host_g_lagrange_ = std::move(gl);
    }
    const std::vector<G1Affine>& get_g() const { return host_g_; }
    const std::vector<G1Affine>& get_g_lagrange() const { return host_g_lagrange_; }
    const std::vector<uint8_t>& g2_bytes() const { return g2_bytes_; }
    // the registered g_lagrange set (what Assembly::build_vk commits sigma over)
    uint64_t g_lagrange_handle() const { return g_lagrange_; }
    ~ParamsKZG() {
        if (g_) h2b_unregister_bases(g_);
        if (g_lagrange_) h2b_unregister_bases(g_lagrange_);
    }
    ParamsKZG(const ParamsKZG&) = delete;
    ParamsKZG& operator=(const ParamsKZG&) = delete;
    uint32_t k() const { return k_; }
    uint64_t n() const { return n_; }
    // fn commit(&self, poly: &Polynomial<_, Coeff>, _: Blind<_>) -> G1     (best_multiexp(&scalars, &self.g[..len]))
    G1 commit(const std::vector<Fr>& poly) const { return msm(poly, g_); }
    // fn commit_lagrange(&self, poly: &Polynomial<_, LagrangeCoeff>, _: Blind<_>) -> G1
    G1 commit_lagrange(const std::vector<Fr>& poly) const { return msm(poly, g_lagrange_); }
    // The independent commitments of one prover phase ([UP] plonk/prover.rs commits the advice / permuted / product columns of a phase
    // one after the other): ONE batched kernel sequence per device, columns dealt round-robin over the devices.  Same results as
    // commit_lagrange / commit called column by column.
    std::vector<G1> commit_lagrange_many(const std::vector<std::vector<Fr>>& polys) const { return msm_many(polys, g_lagrange_); }
    std::vector<G1> commit_many(const std::vector<std::vector<Fr>>& polys) const { return msm_many(polys, g_); }

    // One witness / product column through commit_lagrange -> lagrange_to_coeff -> coeff_to_extended with a single upload
    // (h2b_column_pipeline; SURVEY.md 8f rank 1).  `extended` receives the 2^extended_k coset evaluations when non-null.
    struct CommittedColumn { G1 commitment; std::vector<Fr> coeff; std::vector<Fr> extended; };
    CommittedColumn commit_lagrange_and_convert(const EvaluationDomain& dom, const std::vector<Fr>& lagrange, bool want_extended = true) const {
        if (lagrange.size() != n_ || dom.k() != k_) throw Panic("assertion failed: a.len() == 1 << self.k");
        CommittedColumn out;
        out.coeff.resize(n_);
        if (want_extended) out.extended.resize(dom.extended_len());
        const Fr z[3] = {fr::one(), dom.get_g_coset(), dom.get_g_coset_inv()};
        check(h2b_column_pipeline(dom.device(), reinterpret_cast<const uint64_t*>(lagrange.data()), g_lagrange_, k_, dom.extended_k(), dom.get_omega_inv().l,
                                  dom.get_ifft_divisor().l, dom.get_extended_omega().l, z[0].l, reinterpret_cast<uint64_t*>(&out.commitment),
                                  reinterpret_cast<uint64_t*>(out.coeff.data()), want_extended ? reinterpret_cast<uint64_t*>(out.extended.data()) : nullptr,
                                  nullptr), "commit_lagrange_and_convert");
        return out;
    }

  private:
    ParamsKZG(uint32_t k, const Fr& s, std::vector<uint8_t> g2_bytes) : k_(k), g2_bytes_(std::move(g2_bytes)) {
        ensure_init();
        if (k > 28) throw Panic("ParamsKZG::setup: k out of range");
        n_ = (uint64_t)1 << k;
        host_g_.resize(n_); host_g_lagrange_.resize(n_);
        check(h2b_srs_setup(k, s.l, reinterpret_cast<uint64_t*>(host_g_.data()), reinterpret_cast<uint64_t*>(host_g_lagrange_.data()), &g_, &g_lagrange_),
              "ParamsKZG::setup");
    }
    std::vector<G1> msm_many(const std::vector<std::vector<Fr>>& polys, uint64_t handle) const {
        std::vector<const uint64_t*> ptrs;
        std::vector<size_t> lens;
        for (const auto& p : polys) {
            if (p.size() > n_) throw Panic("assertion failed: bases.len() >= size");
            ptrs.push_back(reinterpret_cast<const uint64_t*>(p.data()));
            lens.push_back(p.size());
        }
        std::vector<G1> out(polys.size());
        check(h2b_msm_bn254_g1_batch_registered(ptrs.data(), lens.data(), polys.size(), handle, reinterpret_cast<uint64_t*>(out.data())), "commit (batched)");
        return out;
    }
    G1 msm(const std::vector<Fr>& poly, uint64_t handle) const {
        if (poly.size() > n_) throw Panic("assertion failed: bases.len() >= size");
        G1 out;
        check(h2b_msm_bn254_g1_registered(reinterpret_cast<const uint64_t*>(poly.data()), handle, 0, poly.size(), reinterpret_cast<uint64_t*>(&out)), "commit");
        return out;
    }
    uint32_t k_ = 0;
    uint64_t n_ = 0;
    std::vector<G1Affine> host_g_, host_g_lagrange_;
    std::vector<uint8_t> g2_bytes_;           // g2 | s_g2 as stored: G2 arithmetic is the verifier's (host) business
    uint64_t g_ = 0, g_lagrange_ = 0;
};

// ProverSHPLONK::create_proof ([UP] poly/kzg/multiopen/shplonk/prover.rs): queries are (polynomial, point) with the polynomial an
// index into `polys` (upstream compares PolynomialPointers by address; a caller maps them to indices the same way).  y and v are the
// challenges the caller squeezed; squeeze_u(h1) writes h1 to the transcript and returns u.  The session is released on every path.
struct Query { uint32_t poly; Fr point; };
class ProverSHPLONK {
  public:
    explicit ProverSHPLONK(const ParamsKZG& params, int device = 0) : params_(params), device_(device) {}
    template <class SqueezeU>
    std::pair<G1, G1> create_proof(const std::vector<std::vector<Fr>>& polys, const std::vector<Query>& queries, const Fr& y, const Fr& v,
                                   SqueezeU squeeze_u) const {
        std::vector<const void*> ptrs;
        for (const auto& p : polys) ptrs.push_back(p.data());
        std::vector<h2b_opening_query> q(queries.size());
        for (size_t i = 0; i < queries.size(); ++i) { q[i].poly = queries[i].poly; q[i].reserved = 0; memcpy(q[i].point, queries[i].point.l, 32); }
        const size_t n = polys.empty() ? 0 : polys[0].size();
        for (const auto& p : polys) if (p.size() != n) throw Panic("ProverSHPLONK::create_proof: polynomials of different lengths");
        G1 h1, h2;
        uint64_t session = 0;
        check(h2b_shplonk_begin(device_, ptrs.data(), 1, (uint32_t)polys.size(), n, q.data(), (uint32_t)q.size(), params_.g_, y.l, v.l,
                                reinterpret_cast<uint64_t*>(&h1), &session), "ProverSHPLONK::create_proof (h1)");
        struct Release { uint64_t s; ~Release() { h2b_shplonk_release(s); } } release{session};
        const Fr u = squeeze_u(h1);
        check(h2b_shplonk_finish(session, u.l, reinterpret_cast<uint64_t*>(&h2)), "ProverSHPLONK::create_proof (h2)");
        return {h1, h2};
    }

  private:
    const ParamsKZG& params_;
    int device_;
};

}  // namespace kzg
}  // namespace poly

// ---- plonk: quotient evaluation, grand products, lookup permutation (SURVEY.md section 8f ranks 2 and 3) -----------------------
namespace plonk {

// host columns of equal length, uploaded for the duration of one call
class DeviceColumns {
  public:
    DeviceColumns(int device, size_t rows) : device_(device), rows_(rows) {}
    const void* upload(const std::vector<Fr>& col) {
        if (col.size() != rows_) throw Panic("column length mismatch");
        bufs_.emplace_back(new DeviceBuffer(device_, (rows_ ? rows_ : 1) * sizeof(Fr)));
        if (rows_) check(h2b_memcpy_h2d(device_, bufs_.back()->get(), col.data(), rows_ * sizeof(Fr)), "h2d");
        return bufs_.back()->get();
    }
    void* scratch() {
        bufs_.emplace_back(new DeviceBuffer(device_, (rows_ ? rows_ : 1) * sizeof(Fr)));
        return bufs_.back()->get();
    }
    std::vector<Fr> download(const void* d, size_t rows) const {
        std::vector<Fr> out(rows);
        check(h2b_dev_sync(device_), "sync");
        if (rows) check(h2b_memcpy_d2h(device_, out.data(), d, rows * sizeof(Fr)), "d2h");
        return out;
    }
  private:
    int device_;
    size_t rows_;
    std::vector<std::unique_ptr<DeviceBuffer>> bufs_;
};

namespace evaluation {

// pub enum ValueSource / pub enum Calculation, as include/h2b200.h flattens them
struct ValueSource : h2b_value_source {
    static ValueSource make(uint32_t kind, uint32_t index = 0, uint32_t rotation = 0) { ValueSource v; v.kind = kind; v.index = index; v.rotation = rotation; return v; }
    static ValueSource Constant(uint32_t i) { return make(H2B_VS_CONSTANT, i); }
    static ValueSource Intermediate(uint32_t i) { return make(H2B_VS_INTERMEDIATE, i); }
    static ValueSource Fixed(uint32_t c, uint32_t r) { return make(H2B_VS_FIXED, c, r); }
    static ValueSource Advice(uint32_t c, uint32_t r) { return make(H2B_VS_ADVICE, c, r); }
    static ValueSource Instance(uint32_t c, uint32_t r) { return make(H2B_VS_INSTANCE, c, r); }
    static ValueSource Challenge(uint32_t i) { return make(H2B_VS_CHALLENGE, i); }
    static ValueSource Beta() { return make(H2B_VS_BETA); }
    static ValueSource Gamma() { return make(H2B_VS_GAMMA); }
    static ValueSource Theta() { return make(H2B_VS_THETA); }
    static ValueSource Y() { return make(H2B_VS_Y); }
    static ValueSource PreviousValue() { return make(H2B_VS_PREVIOUS_VALUE); }
    bool operator==(const ValueSource& o) const { return kind == o.kind && index == o.index && rotation == o.rotation; }
};

// pub enum Expression<F> (plonk/circuit.rs) -- the variants the evaluator sees (selectors are replaced before it is built)
struct Expression {
    enum Kind { Constant, Fixed, Advice, Instance, Challenge, Negated, Sum, Product, Scaled } kind;
    Fr scalar{};                              // Constant / Scaled
    uint32_t index = 0;                       // column or challenge index
    int32_t rotation = 0;
    std::shared_ptr<Expression> a, b;
    static std::shared_ptr<Expression> make(Kind k) { auto e = std::make_shared<Expression>(); e->kind = k; return e; }
};
typedef std::shared_ptr<Expression> Expr;
inline Expr constant(const Fr& c) { Expr e = Expression::make(Expression::Constant); e->scalar = c; return e; }
inline Expr column(Expression::Kind k, uint32_t index, int32_t rotation = 0) { Expr e = Expression::make(k); e->index = index; e->rotation = rotation; return e; }
inline Expr fixed(uint32_t i, int32_t r = 0) { return column(Expression::Fixed, i, r); }
inline Expr advice(uint32_t i, int32_t r = 0) { return column(Expression::Advice, i, r); }
inline Expr instance(uint32_t i, int32_t r = 0) { return column(Expression::Instance, i, r); }
inline Expr challenge(uint32_t i) { return column(Expression::Challenge, i); }
inline Expr negated(Expr a) { Expr e = Expression::make(Expression::Negated); e->a = std::move(a); return e; }
inline Expr sum(Expr a, Expr b) { Expr e = Expression::make(Expression::Sum); e->a = std::move(a); e->b = std::move(b); return e; }
inline Expr product(Expr a, Expr b) { Expr e = Expression::make(Expression::Product); e->a = std::move(a); e->b = std::move(b); return e; }
inline Expr scaled(Expr a, const Fr& f) { Expr e = Expression::make(Expression::Scaled); e->a = std::move(a); e->scalar = f; return e; }

// pub struct GraphEvaluator<C> { constants, rotations, calculations, num_intermediates }  (Default: constants 0, 1, 2)
class GraphEvaluator {
  public:
    GraphEvaluator() : constants_{fr::from_u64(0), fr::one(), fr::from_u64(2)} {}
    // fn add_rotation(&mut self, rotation: &Rotation) -> usize
    uint32_t add_rotation(int32_t rotation) {
        for (size_t i = 0; i < rotations_.size(); ++i) if (rotations_[i] == rotation) return (uint32_t)i;
        rotations_.push_back(rotation);
        return (uint32_t)rotations_.size() - 1;
    }
    // fn add_constant(&mut self, constant: &C::ScalarExt) -> ValueSource
    ValueSource add_constant(const Fr& c) {
        for (size_t i = 0; i < constants_.size(); ++i) if (constants_[i] == c) return ValueSource::Constant((uint32_t)i);
        constants_.push_back(c);
        return ValueSource::Constant((uint32_t)constants_.size() - 1);
    }
    // fn add_calculation(&mut self, calculation: Calculation) -> ValueSource   (an existing identical calculation is reused)
    ValueSource add_calculation(uint32_t op, const ValueSource& a, const ValueSource& b = ValueSource::Constant(0), const std::vector<ValueSource>& parts = {}) {
        for (size_t i = 0; i < calcs_.size(); ++i) {
            const h2b_calculation& c = calcs_[i];
            if (c.op != op || !(ValueSource::make(c.a.kind, c.a.index, c.a.rotation) == a) || !(ValueSource::make(c.b.kind, c.b.index, c.b.rotation) == b) ||
                c.parts_len != parts.size()) continue;
            bool same = true;
            for (size_t j = 0; j < parts.size() && same; ++j) same = static_cast<const ValueSource&>(parts_[c.parts_offset + j]) == parts[j];
            if (same) return ValueSource::Intermediate(c.target);
        }
        h2b_calculation c;
        c.op = op; c.target = num_intermediates_++; c.a = a; c.b = b;
        c.parts_offset = (uint32_t)parts_.size(); c.parts_len = (uint32_t)parts.size();
        for (const ValueSource& p : parts) parts_.push_back(p);
        calcs_.push_back(c);
        return ValueSource::Intermediate(c.target);
    }
    // fn add_expression(&mut self, expr: &Expression<C::ScalarExt>) -> ValueSource
    ValueSource add_expression(const Expr& expr) {
        const ValueSource zero = ValueSource::Constant(0), one = ValueSource::Constant(1), two = ValueSource::Constant(2);
        auto ordered = [&](uint32_t op, const ValueSource& x, const ValueSource& y) {     // derived PartialOrd: variant, then fields
            const bool le = x.kind != y.kind ? x.kind < y.kind : (x.index != y.index ? x.index < y.index : x.rotation <= y.rotation);
            return le ? add_calculation(op, x, y) : add_calculation(op, y, x);
        };
        switch (expr->kind) {
            case Expression::Constant: return add_constant(expr->scalar);
            case Expression::Fixed: return add_calculation(H2B_CALC_STORE, ValueSource::Fixed(expr->index, add_rotation(expr->rotation)));
            case Expression::Advice: return add_calculation(H2B_CALC_STORE, ValueSource::Advice(expr->index, add_rotation(expr->rotation)));
            case Expression::Instance: return add_calculation(H2B_CALC_STORE, ValueSource::Instance(expr->index, add_rotation(expr->rotation)));
            case Expression::Challenge: return add_calculation(H2B_CALC_STORE, ValueSource::Challenge(expr->index));
            case Expression::Negated: {
                if (expr->a->kind == Expression::Constant) return add_constant(fr::sub(fr::from_u64(0), expr->a->scalar));
                const ValueSource ra = add_expression(expr->a);
                return ra == zero ? ra : add_calculation(H2B_CALC_NEGATE, ra);
            }
            case Expression::Sum: {
                if (expr->b->kind == Expression::Negated) {                 // a + (-b) is stored back as a subtraction
                    const ValueSource ra = add_expression(expr->a), rb = add_expression(expr->b->a);
                    if (ra == zero) return add_calculation(H2B_CALC_NEGATE, rb);
                    if (rb == zero) return ra;
                    return add_calculation(H2B_CALC_SUB, ra, rb);
                }
                const ValueSource ra = add_expression(expr->a), rb = add_expression(expr->b);
                if (ra == zero) return rb;
                if (rb == zero) return ra;
                return ordered(H2B_CALC_ADD, ra, rb);
            }
            case Expression::Product: {
                const ValueSource ra = add_expression(expr->a), rb = add_expression(expr->b);
                if (ra == zero || rb == zero) return zero;
                if (ra == one) return rb;
                if (rb == one) return ra;
                if (ra == two) return add_calculation(H2B_CALC_DOUBLE, rb);
                if (rb == two) return add_calculation(H2B_CALC_DOUBLE, ra);
                if (ra == rb) return add_calculation(H2B_CALC_SQUARE, ra);
                return ordered(H2B_CALC_MUL, ra, rb);
            }
            case Expression::Scaled: {
                if (expr->scalar == fr::from_u64(0)) return zero;
                if (expr->scalar == fr::one()) return add_expression(expr->a);
                const ValueSource cst = add_constant(expr->scalar);
                const ValueSource ra = add_expression(expr->a);
                return add_calculation(H2B_CALC_MUL, ra, cst);
            }
        }
        throw Panic("unreachable: Expression::Selector");
    }
    // pub fn evaluate(..) for every row idx < isize: values[idx] = evaluate(.., previous_value = values[idx], idx, rot_scale, isize)
    std::vector<Fr> evaluate(const std::vector<std::vector<Fr>>& fixed, const std::vector<std::vector<Fr>>& advice, const std::vector<std::vector<Fr>>& instance,
                             const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma, const Fr& theta, const Fr& y, const std::vector<Fr>& values,
                             int32_t rot_scale, int device = 0) const {
        ensure_init();
        const size_t size = values.size();
        DeviceColumns dev(device, size);
        std::vector<const void*> f, a, i;
        for (auto& c : fixed) f.push_back(dev.upload(c));
        for (auto& c : advice) a.push_back(dev.upload(c));
        for (auto& c : instance) i.push_back(dev.upload(c));
        void* d_values = const_cast<void*>(dev.upload(values));
        h2b_graph g;
        g.constants = reinterpret_cast<const uint64_t*>(constants_.data()); g.n_constants = (uint32_t)constants_.size();
        g.rotations = rotations_.data(); g.n_rotations = (uint32_t)rotations_.size();
        g.calculations = calcs_.data(); g.n_calculations = (uint32_t)calcs_.size();
        g.parts = parts_.data(); g.n_parts = (uint32_t)parts_.size();
        g.n_intermediates = num_intermediates_;
        h2b_eval_columns c;
        c.fixed = f.data(); c.n_fixed = (uint32_t)f.size();
        c.advice = a.data(); c.n_advice = (uint32_t)a.size();
        c.instance = i.data(); c.n_instance = (uint32_t)i.size();
        c.challenges = reinterpret_cast<const uint64_t*>(challenges.data()); c.n_challenges = (uint32_t)challenges.size();
        c.beta = beta.l; c.gamma = gamma.l; c.theta = theta.l; c.y = y.l;
        check(h2b_evaluate_graph_dev(device, &g, &c, d_values, (uint32_t)size, rot_scale, nullptr), "GraphEvaluator::evaluate");
        return dev.download(d_values, size);
    }
    uint32_t num_intermediates() const { return num_intermediates_; }

  private:
    std::vector<Fr> constants_;
    std::vector<int32_t> rotations_;
    std::vector<h2b_calculation> calcs_;
    std::vector<h2b_value_source> parts_;
    uint32_t num_intermediates_ = 0;
};

// Evaluator::new(cs), custom gates: every gate polynomial through add_expression, combined by one Horner in y over the previous value
inline GraphEvaluator custom_gates_evaluator(const std::vector<Expr>& gate_polynomials) {
    GraphEvaluator g;
    std::vector<ValueSource> parts;
    for (const Expr& poly : gate_polynomials) parts.push_back(g.add_expression(poly));
    g.add_calculation(H2B_CALC_HORNER, ValueSource::PreviousValue(), ValueSource::Y(), parts);
    return g;
}

}  // namespace evaluation

namespace permutation {
// permutation::Argument::commit for one set of columns: z[0] = last_z, z[i+1] = z[i] * numerator_i / denominator_i
inline std::vector<Fr> commit_product(const std::vector<std::vector<Fr>>& values, const std::vector<std::vector<Fr>>& permutations, const Fr& beta, const Fr& gamma,
                                      const Fr& delta, const Fr& deltaomega, const Fr& omega, const Fr& last_z, int device = 0) {
    ensure_init();
    if (values.empty() || values.size() != permutations.size()) throw Panic("permutation::commit: column / permutation count mismatch");
    const size_t n = values[0].size();
    DeviceColumns dev(device, n);
    std::vector<const void*> v, p;
    for (auto& c : values) v.push_back(dev.upload(c));
    for (auto& c : permutations) p.push_back(dev.upload(c));
    void* z = dev.scratch();
    check(h2b_permutation_product_dev(device, v.data(), p.data(), (uint32_t)v.size(), n, beta.l, gamma.l, delta.l, deltaomega.l, omega.l, last_z.l, z, nullptr),
          "permutation::commit");
    return dev.download(z, n);
}

// Assembly::build_vk / build_pk (plonk/permutation/keygen.rs) from the mapping that Assembly::copy built on the host:
// mapping[i][j] = (column, row), sigma_i[j] = DELTA^column omega^row, all per-row work on the device.
namespace keygen {
typedef std::vector<std::vector<std::pair<uint64_t, uint64_t>>> Mapping;      // upstream's Vec<Vec<(usize, usize)>>
static_assert(sizeof(std::pair<uint64_t, uint64_t>) == 16, "a mapping entry is two u64");

inline Fr delta() {                      // Fr::DELTA = GENERATOR^(2^S)
    const uint64_t e[4] = {(uint64_t)1 << fr::S, 0, 0, 0};
    return fr::pow(fr::from_u64(7), e);
}
inline std::vector<const uint64_t*> columns_of(const Mapping& mapping, size_t n) {
    std::vector<const uint64_t*> cols;
    for (const auto& c : mapping) {
        if (c.size() != n) throw Panic("permutation keygen: mapping column length != 2^k");
        cols.push_back(reinterpret_cast<const uint64_t*>(c.data()));
    }
    return cols;
}
// VerifyingKey { commitments }: commit_lagrange(sigma_i) for every column
inline std::vector<G1> build_vk(const poly::kzg::ParamsKZG& params, const poly::EvaluationDomain& domain, const Mapping& mapping) {
    ensure_init();
    const auto cols = columns_of(mapping, (size_t)1 << domain.k());
    std::vector<G1> out(cols.size());
    check(h2b_permutation_build_vk(cols.data(), (uint32_t)cols.size(), domain.k(), delta().l, domain.get_omega().l, params.g_lagrange_handle(),
                                   reinterpret_cast<uint64_t*>(out.data())), "permutation::keygen::build_vk");
    return out;
}
// ProvingKey { permutations, polys, cosets }
struct ProvingKey { std::vector<std::vector<Fr>> permutations, polys, cosets; };
inline ProvingKey build_pk(const poly::kzg::ParamsKZG&, const poly::EvaluationDomain& domain, const Mapping& mapping) {
    ensure_init();
    const size_t n = (size_t)1 << domain.k();
    const auto cols = columns_of(mapping, n);
    ProvingKey pk;
    std::vector<uint64_t*> p, c, e;
    for (size_t i = 0; i < cols.size(); ++i) {
        pk.permutations.emplace_back(n); pk.polys.emplace_back(n); pk.cosets.emplace_back(domain.extended_len());
        p.push_back(reinterpret_cast<uint64_t*>(pk.permutations.back().data()));
        c.push_back(reinterpret_cast<uint64_t*>(pk.polys.back().data()));
        e.push_back(reinterpret_cast<uint64_t*>(pk.cosets.back().data()));
    }
    const Fr z[3] = {fr::one(), domain.get_g_coset(), domain.get_g_coset_inv()};
    check(h2b_permutation_build_pk(cols.data(), (uint32_t)cols.size(), domain.k(), domain.extended_k(), delta().l, domain.get_omega().l,
                                   domain.get_omega_inv().l, domain.get_ifft_divisor().l, domain.get_extended_omega().l, z[0].l, p.data(), c.data(), e.data()),
          "permutation::keygen::build_pk");
    return pk;
}
}  // namespace keygen
}  // namespace permutation

// keygen_pk's l0, l_last and l_active_row on the extended coset (plonk/keygen.rs), computed on the device
namespace keygen {
struct LagrangeIndicators { std::vector<Fr> l0, l_last, l_active_row; };
inline LagrangeIndicators lagrange_indicators(const poly::EvaluationDomain& domain, uint32_t blinding_factors) {
    ensure_init();
    const size_t en = domain.extended_len();
    DeviceBuffer d0(domain.device(), en * sizeof(Fr)), d1(domain.device(), en * sizeof(Fr)), d2(domain.device(), en * sizeof(Fr));
    const Fr z[3] = {fr::one(), domain.get_g_coset(), domain.get_g_coset_inv()};
    check(h2b_keygen_lagrange_indicators_dev(domain.device(), domain.k(), domain.extended_k(), blinding_factors, domain.get_omega_inv().l,
                                             domain.get_ifft_divisor().l, domain.get_extended_omega().l, z[0].l, d0.get(), d1.get(), d2.get(), nullptr),
          "keygen_pk: lagrange indicators");
    check(h2b_dev_sync(domain.device()), "sync");
    LagrangeIndicators out{std::vector<Fr>(en), std::vector<Fr>(en), std::vector<Fr>(en)};
    check(h2b_memcpy_d2h(domain.device(), out.l0.data(), d0.get(), en * sizeof(Fr)), "d2h");
    check(h2b_memcpy_d2h(domain.device(), out.l_last.data(), d1.get(), en * sizeof(Fr)), "d2h");
    check(h2b_memcpy_d2h(domain.device(), out.l_active_row.data(), d2.get(), en * sizeof(Fr)), "d2h");
    return out;
}

// compress_selectors (plonk/circuit/compress_selectors.rs process) and the fixed half of keygen_vk / keygen_pk.  A selector's
// activations are one byte per row (Rust's Vec<bool> layout; std::vector<bool> is bit-packed, so it is not used).
typedef std::vector<std::vector<uint8_t>> Activations;
// per selector: its combination, its root and the combination's length -- the substitution is q * prod_{r = 1..len, r != root} (r - q)
struct SelectorAssignment { std::vector<uint32_t> combination_of, root_of, len_of; uint32_t n_combinations = 0; };

inline std::vector<const uint8_t*> activation_rows(const Activations& acts, size_t n) {
    std::vector<const uint8_t*> rows;
    for (const auto& a : acts) {
        if (a.size() != n) throw Panic("compress_selectors: activations length != 2^k");
        rows.push_back(a.data());
    }
    return rows;
}
// process over selectors of these gate degrees (0: in no gate polynomial) against max_degree = cs.degree(); the exclusion matrix comes
// from the device, the greedy step is upstream's
inline SelectorAssignment compress_selectors(const Activations& acts, const std::vector<uint32_t>& degrees, uint32_t max_degree, uint32_t k) {
    ensure_init();
    const size_t S = acts.size();
    if (degrees.size() != S) throw Panic("compress_selectors: one degree per selector");
    SelectorAssignment a;
    a.combination_of.assign(S, 0); a.root_of.assign(S, 0); a.len_of.assign(S, 0);
    std::vector<uint32_t> simple;
    for (uint32_t s = 0; s < S; ++s) {
        if (degrees[s] != 0) { simple.push_back(s); continue; }
        a.combination_of[s] = a.n_combinations++; a.root_of[s] = 1; a.len_of[s] = 1;
    }
    const auto all_rows = activation_rows(acts, (size_t)1 << k);
    const size_t m = simple.size();
    std::vector<uint8_t> excl(m * m);
    std::vector<const uint8_t*> rows;
    for (uint32_t s : simple) rows.push_back(all_rows[s]);
    if (m) check(h2b_selector_exclusion(rows.data(), (uint32_t)m, k, excl.data()), "compress_selectors: exclusion matrix");
    std::vector<bool> added(m, false);
    for (size_t i = 0; i < m; ++i) {
        if (added[i]) continue;
        added[i] = true;
        if (degrees[simple[i]] > max_degree) throw Panic("compress_selectors: selector degree above max_degree");
        size_t d = degrees[simple[i]] - 1;
        std::vector<size_t> comb{i};
        for (size_t j = i + 1; j < m; ++j) {
            if (d + comb.size() == max_degree) break;
            if (added[j]) continue;
            bool excluded = false;
            for (size_t x : comb) excluded = excluded || excl[j * m + x];
            if (excluded) continue;
            const size_t new_d = std::max(d, (size_t)degrees[simple[j]] - 1);
            if (new_d + comb.size() + 1 > max_degree) continue;
            d = new_d;
            comb.push_back(j);
            added[j] = true;
        }
        for (size_t t = 0; t < comb.size(); ++t) {
            const uint32_t s = simple[comb[t]];
            a.combination_of[s] = a.n_combinations; a.root_of[s] = (uint32_t)(t + 1); a.len_of[s] = (uint32_t)comb.size();
        }
        ++a.n_combinations;
    }
    return a;
}

inline std::vector<const uint64_t*> fixed_columns_of(const std::vector<std::vector<Fr>>& fixed, size_t n) {
    std::vector<const uint64_t*> cols;
    for (const auto& c : fixed) {
        if (c.size() != n) throw Panic("keygen: fixed column length != 2^k");
        cols.push_back(reinterpret_cast<const uint64_t*>(c.data()));
    }
    return cols;
}
// keygen_vk's fixed_commitments: commit_lagrange of each fixed column, then of each combination column
inline std::vector<G1> fixed_build_vk(const poly::kzg::ParamsKZG& params, const poly::EvaluationDomain& domain, const std::vector<std::vector<Fr>>& fixed,
                                      const Activations& acts, const SelectorAssignment& a) {
    ensure_init();
    const size_t n = (size_t)1 << domain.k();
    const auto cols = fixed_columns_of(fixed, n);
    const auto rows = activation_rows(acts, n);
    std::vector<G1> out(cols.size() + a.n_combinations);
    check(h2b_keygen_fixed_build_vk(cols.data(), (uint32_t)cols.size(), rows.data(), (uint32_t)rows.size(), a.combination_of.data(), a.root_of.data(),
                                    a.n_combinations, domain.k(), params.g_lagrange_handle(), reinterpret_cast<uint64_t*>(out.data())),
          "keygen::fixed_build_vk");
    return out;
}
// keygen_pk's fixed columns: the combination columns in Lagrange form (fixed_values = fixed ++ these), and fixed_polys / fixed_cosets
// of every column
struct FixedProvingKey { std::vector<std::vector<Fr>> combination_values, polys, cosets; };
inline FixedProvingKey fixed_build_pk(const poly::kzg::ParamsKZG&, const poly::EvaluationDomain& domain, const std::vector<std::vector<Fr>>& fixed,
                                      const Activations& acts, const SelectorAssignment& a) {
    ensure_init();
    const size_t n = (size_t)1 << domain.k();
    const auto cols = fixed_columns_of(fixed, n);
    const auto rows = activation_rows(acts, n);
    FixedProvingKey pk;
    std::vector<uint64_t*> v, p, e;
    for (uint32_t c = 0; c < a.n_combinations; ++c) {
        pk.combination_values.emplace_back(n);
        v.push_back(reinterpret_cast<uint64_t*>(pk.combination_values.back().data()));
    }
    for (size_t i = 0; i < cols.size() + a.n_combinations; ++i) {
        pk.polys.emplace_back(n); pk.cosets.emplace_back(domain.extended_len());
        p.push_back(reinterpret_cast<uint64_t*>(pk.polys.back().data()));
        e.push_back(reinterpret_cast<uint64_t*>(pk.cosets.back().data()));
    }
    const Fr z[3] = {fr::one(), domain.get_g_coset(), domain.get_g_coset_inv()};
    check(h2b_keygen_fixed_build_pk(cols.data(), (uint32_t)cols.size(), rows.data(), (uint32_t)rows.size(), a.combination_of.data(), a.root_of.data(),
                                    a.n_combinations, domain.k(), domain.extended_k(), domain.get_omega_inv().l, domain.get_ifft_divisor().l,
                                    domain.get_extended_omega().l, z[0].l, v.data(), p.data(), e.data()),
          "keygen::fixed_build_pk");
    return pk;
}
}  // namespace keygen

// ProvingKey's fixed, permutation and indicator columns held on the devices from keygen to the last proof (h2b_pk_*): built there by
// the keygen kernels, or registered from a key built elsewhere, and read by the device steps of create_proof through column().  RAII:
// the destructor releases the handle (freeing waits for the work queued on the devices).
class ProvingKeyOnDevice {
  public:
    ProvingKeyOnDevice(const poly::EvaluationDomain& domain, uint32_t n_fixed, uint32_t n_permutation, int layout = H2B_PK_REPLICATED,
                       uint32_t halo = 0)
        : k_(domain.k()), extended_k_(domain.extended_k()) {
        ensure_init();
        const Fr z[3] = {fr::one(), domain.get_g_coset(), domain.get_g_coset_inv()};
        check(h2b_pk_create(k_, extended_k_, n_fixed, n_permutation, layout, halo, domain.get_omega().l, domain.get_omega_inv().l,
                            domain.get_ifft_divisor().l, domain.get_extended_omega().l, z[0].l, &handle_),
              "ProvingKeyOnDevice: create");
    }
    ~ProvingKeyOnDevice() { if (handle_) h2b_pk_release(handle_); }
    ProvingKeyOnDevice(const ProvingKeyOnDevice&) = delete;
    ProvingKeyOnDevice& operator=(const ProvingKeyOnDevice&) = delete;

    void build_fixed(const std::vector<std::vector<Fr>>& fixed, const keygen::Activations& acts, const keygen::SelectorAssignment& a,
                     uint32_t first_column = 0) {
        const size_t n = (size_t)1 << k_;
        const auto cols = keygen::fixed_columns_of(fixed, n);
        const auto rows = keygen::activation_rows(acts, n);
        check(h2b_keygen_fixed_build_pk_resident(cols.data(), (uint32_t)cols.size(), rows.data(), (uint32_t)rows.size(), a.combination_of.data(),
                                                 a.root_of.data(), a.n_combinations, handle_, first_column),
              "ProvingKeyOnDevice::build_fixed");
    }
    void build_permutation(const permutation::keygen::Mapping& mapping) {
        const auto cols = permutation::keygen::columns_of(mapping, (size_t)1 << k_);
        check(h2b_permutation_build_pk_resident(cols.data(), (uint32_t)cols.size(), permutation::keygen::delta().l, handle_),
              "ProvingKeyOnDevice::build_permutation");
    }
    void build_indicators(uint32_t blinding_factors) {
        check(h2b_keygen_lagrange_indicators_resident(handle_, blinding_factors), "ProvingKeyOnDevice::build_indicators");
    }
    // columns of a ProvingKey built elsewhere (the CPU keygen, ProvingKey::read), in Lagrange form
    void put_lagrange(int part, uint32_t first, const std::vector<std::vector<Fr>>& values) {
        const auto cols = keygen::fixed_columns_of(values, (size_t)1 << k_);
        check(h2b_pk_put_lagrange(handle_, part, first, (uint32_t)cols.size(), cols.data()), "ProvingKeyOnDevice::put_lagrange");
    }
    // the column on `device`, valid while this object lives; *shard (optional) receives its slice
    const void* column(int device, int part, int form, uint32_t index, h2b_eval_shard* shard = nullptr) const {
        void* p = nullptr;
        check(h2b_pk_column(handle_, device, part, form, index, &p, shard), "ProvingKeyOnDevice::column");
        return p;
    }
    std::vector<Fr> download(int part, int form, uint32_t index) const {
        std::vector<Fr> out((size_t)1 << (form == H2B_PK_EXTENDED ? extended_k_ : k_));
        check(h2b_pk_download(handle_, part, form, index, reinterpret_cast<uint64_t*>(out.data())), "ProvingKeyOnDevice::download");
        return out;
    }
    std::vector<uint64_t> info() const {
        std::vector<uint64_t> bytes((size_t)h2b_device_count());
        check(h2b_pk_info(handle_, bytes.data()), "ProvingKeyOnDevice::info");
        return bytes;
    }
    uint64_t handle() const { return handle_; }

  private:
    uint32_t k_, extended_k_;
    uint64_t handle_ = 0;
};

namespace lookup {
// fn permute_expression_pair(..) -> Result<(Vec<F>, Vec<F>), Error>: the first usable_rows rows of (A', S')
inline std::pair<std::vector<Fr>, std::vector<Fr>> permute_expression_pair(const std::vector<Fr>& input_expression, const std::vector<Fr>& table_expression,
                                                                            size_t usable_rows, int device = 0) {
    ensure_init();
    if (input_expression.size() != table_expression.size() || usable_rows > input_expression.size()) throw Panic("permute_expression_pair: bad lengths");
    DeviceColumns dev(device, input_expression.size());
    const void* a = dev.upload(input_expression);
    const void* t = dev.upload(table_expression);
    void* pa = dev.scratch();
    void* pt = dev.scratch();
    check(h2b_lookup_permute_dev(device, a, t, (uint32_t)usable_rows, pa, pt, nullptr), "Error::ConstraintSystemFailure");
    return {dev.download(pa, usable_rows), dev.download(pt, usable_rows)};
}
// Permuted::commit_product: z[0] = 1, z[i+1] = z[i] (a + beta)(s + gamma) / ((a' + beta)(s' + gamma))
inline std::vector<Fr> commit_product(const std::vector<Fr>& compressed_input, const std::vector<Fr>& compressed_table, const std::vector<Fr>& permuted_input,
                                      const std::vector<Fr>& permuted_table, const Fr& beta, const Fr& gamma, int device = 0) {
    ensure_init();
    const size_t n = compressed_input.size();
    DeviceColumns dev(device, n);
    const void* c[4] = {dev.upload(compressed_input), dev.upload(compressed_table), dev.upload(permuted_input), dev.upload(permuted_table)};
    void* z = dev.scratch();
    check(h2b_lookup_product_dev(device, c[0], c[1], c[2], c[3], n, beta.l, gamma.l, z, nullptr), "lookup::commit_product");
    return dev.download(z, n);
}
}  // namespace lookup
}  // namespace plonk
}  // namespace h2b200
