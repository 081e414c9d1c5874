// ORACLE (test infrastructure only): CPU restatement of the three row loops of MockProver::verify_par ([UP] halo2_proofs/src/dev.rs
// @ v2023_02_02, as recalled) on the field code of oracle/h2_oracle.cpp.  It evaluates the circuit's EXPRESSION TREES with
// `evaluate_lazy` and the `Value` enum, deliberately not a compiled GraphEvaluator, so that the device's compiled route is checked
// against an independent evaluation:
//
//   cells    : CellValue::{Unassigned, Assigned(F), Poison(row)}; advice rows >= usable_rows are Poison(row); instance cells are
//              Assigned(value).  Loading: Unassigned -> Real(0), Assigned(v) -> Real(v), Poison -> Poison
//   Value    : +, -, negation: Poison if an operand is; a * b: Real(0) when either side is Real(0), else Poison if either is;
//              Poison * f (Scaled): Real(0) for f = 0, Poison otherwise.  Product short-circuits a left side equal to Real(0)
//   gates    : for gate, for row in 0..n, for poly: Real(0) passes, Real(!= 0) ConstraintNotSatisfied, Poison ConstraintPoisoned
//   lookups  : fill_row = table expressions at row usable_rows - 1; table = sorted tuples of the usable rows except fill_row;
//              inputs = (tuple, row) of the usable rows except fill_row, sorted; an input not found by binary search fails.
//              Order: Real < Poison, Reals by canonical integer; failures come out in (tuple, row) order
//   copies   : for column, for row: cell(c, r) != cell(mapping[c][r]) under CellValue equality fails
//
// Expressions arrive in prefix form, one u64 per token: 0 Constant (+4 Montgomery words), 1 Fixed, 2 Advice, 3 Instance (each + column,
// rotation as i64), 4 Challenge (+ index), 5 Negated (+ a), 6 Sum (+ a, b), 7 Product (+ a, b), 8 Scaled (+ a, 4 words).
// The gate and copy loops run on `threads` threads, each over a block of rows, as verify_par spreads rows over rayon's pool.
#include "../../oracle/h2_oracle.cpp"

#include <algorithm>
#include <cstdio>
#include <thread>

namespace {

struct Val {
    bool poison;
    Fr v;
    bool operator==(const Val& o) const { return poison == o.poison && (poison || v == o.v); }
};
struct Canon { u64 l[4]; };
static Canon canon(const Fr& x) { Fr c = x.from_mont(); Canon o; memcpy(o.l, c.l, 32); return o; }
static int canon_cmp(const Fr& a, const Fr& b) {
    const Canon x = canon(a), y = canon(b);
    for (int i = 3; i >= 0; --i) if (x.l[i] != y.l[i]) return x.l[i] < y.l[i] ? -1 : 1;
    return 0;
}
static int val_cmp(const Val& a, const Val& b) {      // derived Ord of enum Value { Real(F), Poison }
    if (a.poison != b.poison) return a.poison ? 1 : -1;
    return a.poison ? 0 : canon_cmp(a.v, b.v);
}
static int tuple_cmp(const std::vector<Val>& a, const std::vector<Val>& b) {
    for (size_t i = 0; i < a.size(); ++i) { const int c = val_cmp(a[i], b[i]); if (c) return c; }
    return 0;
}

struct Circuit {
    uint32_t k, n, usable;
    std::vector<const u64*> fixed, advice, instance;
    std::vector<const uint8_t*> fixed_bits, advice_bits;
    const u64* challenges;
    const u64* tokens;
    bool assigned(const uint8_t* bits, uint32_t r) const { return (bits[r >> 3] >> (r & 7)) & 1; }
    Val load(uint32_t kind, uint64_t col, int64_t rot, uint32_t row) const {
        const uint32_t r = (uint32_t)((((int64_t)row + rot) % (int64_t)n + n) % n);
        if (kind == 3) return Val{false, fr_at(instance[col], r)};
        if (kind == 2 && r >= usable) return Val{true, Fr::zero()};
        const u64* c = kind == 1 ? fixed[col] : advice[col];
        const uint8_t* b = kind == 1 ? fixed_bits[col] : advice_bits[col];
        return Val{false, assigned(b, r) ? fr_at(c, r) : Fr::zero()};
    }
    // evaluate_lazy of the expression at tokens[pos]; pos moves past it
    Val eval(size_t& pos, uint32_t row) const {
        const u64 t = tokens[pos++];
        auto word4 = [&]() { Fr x; memcpy(x.l, tokens + pos, 32); pos += 4; return x; };
        auto skip = [&]() { Val dummy = eval(pos, row); (void)dummy; };
        switch (t) {
            case 0: return Val{false, word4()};
            case 1: case 2: case 3: { const u64 col = tokens[pos], rot = tokens[pos + 1]; pos += 2; return load((uint32_t)t, col, (int64_t)rot, row); }
            case 4: { const u64 i = tokens[pos++]; return Val{false, fr_at(challenges, i)}; }
            case 5: { Val a = eval(pos, row); return a.poison ? a : Val{false, a.v.neg()}; }
            case 6: { Val a = eval(pos, row), b = eval(pos, row); return (a.poison || b.poison) ? Val{true, Fr::zero()} : Val{false, a.v + b.v}; }
            case 7: {
                Val a = eval(pos, row);
                if (!a.poison && a.v.is_zero()) { skip(); return a; }       // evaluate_lazy: a zero left side skips the right one
                Val b = eval(pos, row);
                if (!a.poison && !b.poison) return Val{false, a.v * b.v};
                if ((!a.poison && a.v.is_zero()) || (!b.poison && b.v.is_zero())) return Val{false, Fr::zero()};
                return Val{true, Fr::zero()};
            }
            case 8: {
                Val a = eval(pos, row);
                const Fr f = word4();
                if (!a.poison) return Val{false, a.v * f};
                return f.is_zero() ? Val{false, Fr::zero()} : Val{true, Fr::zero()};
            }
        }
        fprintf(stderr, "mock oracle: bad token %llu\n", (unsigned long long)t);
        abort();
    }
    Val eval_at(size_t offset, uint32_t row) const { size_t p = offset; return eval(p, row); }
};

struct Rec { uint32_t kind, index, poly, row; };

template <class F> static void rows_in_blocks(uint32_t n, int threads, std::vector<std::vector<Rec>>& parts, F&& body) {
    threads = std::max(1, std::min<int>(threads, (int)n));
    parts.assign(threads, {});
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t)
        pool.emplace_back([&, t] {
            const uint32_t lo = (uint32_t)((uint64_t)n * t / threads), hi = (uint32_t)((uint64_t)n * (t + 1) / threads);
            for (uint32_t r = lo; r < hi; ++r) body(r, parts[t]);
        });
    for (auto& th : pool) th.join();
}

}  // namespace

extern "C" {

// roots: n_roots x (gate, poly, token offset), gates ascending.  lookups: per lookup m, then m input and m table token offsets.
// perm: n_perm x (kind 1 fixed / 2 advice / 3 instance, index); mapping: n_perm x n x (column, row).  Writes the first `cap` records
// (kind, index, poly, row) in upstream's order and returns the total.
uint64_t orc_mock_verify(uint32_t k, uint32_t bf, const u64* fixed, const uint8_t* fixed_bits, uint32_t nf, const u64* advice, const uint8_t* advice_bits,
                         uint32_t na, const u64* instance, uint32_t ni, const u64* challenges, const u64* tokens, const uint32_t* roots, uint32_t n_roots,
                         const uint32_t* lookups, uint32_t n_lookups, const uint32_t* perm, const u64* mapping, uint32_t n_perm, int threads,
                         uint32_t* out, uint64_t cap) {
    Circuit c;
    c.k = k; c.n = 1u << k; c.usable = c.n - (bf + 1);
    const size_t nb = (c.n + 7) / 8;
    for (uint32_t i = 0; i < nf; ++i) { c.fixed.push_back(fixed + (size_t)4 * c.n * i); c.fixed_bits.push_back(fixed_bits + nb * i); }
    for (uint32_t i = 0; i < na; ++i) { c.advice.push_back(advice + (size_t)4 * c.n * i); c.advice_bits.push_back(advice_bits + nb * i); }
    for (uint32_t i = 0; i < ni; ++i) c.instance.push_back(instance + (size_t)4 * c.n * i);
    c.challenges = challenges; c.tokens = tokens;
    std::vector<Rec> all;
    std::vector<std::vector<Rec>> parts;
    // gates
    for (uint32_t z0 = 0; z0 < n_roots;) {
        uint32_t z1 = z0;
        while (z1 < n_roots && roots[3 * z1] == roots[3 * z0]) ++z1;
        rows_in_blocks(c.n, threads, parts, [&](uint32_t row, std::vector<Rec>& out_) {
            for (uint32_t z = z0; z < z1; ++z) {
                const Val v = c.eval_at(roots[3 * z + 2], row);
                if (v.poison) out_.push_back(Rec{1, roots[3 * z], roots[3 * z + 1], row});
                else if (!v.v.is_zero()) out_.push_back(Rec{0, roots[3 * z], roots[3 * z + 1], row});
            }
        });
        for (auto& p : parts) all.insert(all.end(), p.begin(), p.end());
        z0 = z1;
    }
    // lookups
    const uint32_t* d = lookups;
    for (uint32_t l = 0; l < n_lookups; ++l) {
        const uint32_t m = *d++;
        const uint32_t* in_off = d;
        const uint32_t* tb_off = d + m;
        d += 2 * m;
        auto tuple = [&](const uint32_t* offs, uint32_t row) { std::vector<Val> t; for (uint32_t j = 0; j < m; ++j) t.push_back(c.eval_at(offs[j], row)); return t; };
        const std::vector<Val> fill = tuple(tb_off, c.usable - 1);
        std::vector<std::vector<Val>> table;
        for (uint32_t r = 0; r < c.usable; ++r) { auto t = tuple(tb_off, r); if (tuple_cmp(t, fill) != 0) table.push_back(std::move(t)); }
        std::sort(table.begin(), table.end(), [](const std::vector<Val>& a, const std::vector<Val>& b) { return tuple_cmp(a, b) < 0; });
        std::vector<std::pair<std::vector<Val>, uint32_t>> inputs;
        for (uint32_t r = 0; r < c.usable; ++r) { auto t = tuple(in_off, r); if (tuple_cmp(t, fill) != 0) inputs.emplace_back(std::move(t), r); }
        std::sort(inputs.begin(), inputs.end(), [](const auto& a, const auto& b) { const int x = tuple_cmp(a.first, b.first); return x ? x < 0 : a.second < b.second; });
        for (const auto& in : inputs) {
            const bool found = std::binary_search(table.begin(), table.end(), in.first, [](const std::vector<Val>& a, const std::vector<Val>& b) { return tuple_cmp(a, b) < 0; });
            if (!found) all.push_back(Rec{2, l, 0, in.second});
        }
    }
    // copy constraints: CellValue of (column, row) as (state, value): 0 Unassigned, 1 Assigned, 2 Poison(row)
    auto cell = [&](uint64_t col, uint64_t row, Fr& v) -> uint32_t {
        const uint32_t kind = perm[2 * col], idx = perm[2 * col + 1];
        if (kind == 3) { v = fr_at(c.instance[idx], row); return 1; }
        if (kind == 2 && row >= c.usable) return 2;
        const uint8_t* b = kind == 1 ? c.fixed_bits[idx] : c.advice_bits[idx];
        if (!c.assigned(b, (uint32_t)row)) return 0;
        v = fr_at(kind == 1 ? c.fixed[idx] : c.advice[idx], row);
        return 1;
    };
    for (uint32_t col = 0; col < n_perm; ++col) {
        rows_in_blocks(c.n, threads, parts, [&](uint32_t row, std::vector<Rec>& out_) {
            const u64* m = mapping + 2 * ((size_t)col * c.n + row);
            Fr a = Fr::zero(), b = Fr::zero();
            const uint32_t sa = cell(col, row, a), sb = cell(m[0], m[1], b);
            const bool equal = sa == sb && (sa == 0 || (sa == 1 && a == b) || (sa == 2 && row == m[1]));
            if (!equal) out_.push_back(Rec{3, col, 0, row});
        });
        for (auto& p : parts) all.insert(all.end(), p.begin(), p.end());
    }
    for (size_t i = 0; i < all.size() && i < cap; ++i) memcpy(out + 4 * i, &all[i], 16);
    return all.size();
}

}  // extern "C"
