// Drives compress_selectors and the fixed-column keygen of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp):
// ParamsKZG::setup(k, s) with s from <dir>/s.bin, EvaluationDomain(5, k), F fixed columns (F x 2^k x 4 u64) from <dir>/fixed.bin,
// S selectors (S x 2^k bytes) from <dir>/activations.bin and their degrees (S u32) from <dir>/degrees.bin, then
// keygen::compress_selectors(max_degree), fixed_build_vk and fixed_build_pk; writes assignment.bin (combination_of, root_of, len_of),
// vk.bin, values.bin, polys.bin and cosets.bin.
//   usage: fixed_keygen_mirror <dir> <k> <F> <S> <max_degree>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../halo2_scaffold_b200/host/h2b200.hpp"

using namespace h2b200;

static bool write_all(const std::string& path, const void* p, size_t bytes) {
    FILE* w = fopen(path.c_str(), "wb");
    if (!w) return false;
    const bool ok = fwrite(p, 1, bytes, w) == bytes;
    fclose(w);
    return ok;
}

template <class T>
static bool write_columns(const std::string& path, const std::vector<std::vector<T>>& cols) {
    std::vector<T> flat;
    for (const auto& c : cols) flat.insert(flat.end(), c.begin(), c.end());
    return write_all(path, flat.data(), flat.size() * sizeof(T));
}

template <class T>
static bool read_columns(const std::string& path, std::vector<std::vector<T>>& cols) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    bool ok = true;
    for (auto& c : cols) ok = ok && fread(c.data(), sizeof(T), c.size(), f) == c.size();
    fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc < 6) return 2;
    const std::string dir = argv[1];
    const uint32_t k = (uint32_t)atoi(argv[2]), F = (uint32_t)atoi(argv[3]), S = (uint32_t)atoi(argv[4]), max_degree = (uint32_t)atoi(argv[5]);
    const size_t n = (size_t)1 << k;
    std::vector<std::vector<Fr>> s(1, std::vector<Fr>(1)), fixed(F, std::vector<Fr>(n));
    plonk::keygen::Activations acts(S, std::vector<uint8_t>(n));
    std::vector<std::vector<uint32_t>> degrees(1, std::vector<uint32_t>(S));
    if (!read_columns(dir + "/s.bin", s) || !read_columns(dir + "/fixed.bin", fixed) || !read_columns(dir + "/activations.bin", acts) ||
        !read_columns(dir + "/degrees.bin", degrees))
        return 2;
    try {
        auto params = poly::kzg::ParamsKZG::setup(k, s[0][0]);
        poly::EvaluationDomain domain(5, k);
        const plonk::keygen::SelectorAssignment a = plonk::keygen::compress_selectors(acts, degrees[0], max_degree, k);
        const std::vector<G1> vk = plonk::keygen::fixed_build_vk(*params, domain, fixed, acts, a);
        const plonk::keygen::FixedProvingKey pk = plonk::keygen::fixed_build_pk(*params, domain, fixed, acts, a);
        if (!write_columns(dir + "/assignment.bin", std::vector<std::vector<uint32_t>>{a.combination_of, a.root_of, a.len_of}) ||
            !write_all(dir + "/vk.bin", vk.data(), vk.size() * sizeof(G1)) || !write_columns(dir + "/values.bin", pk.combination_values) ||
            !write_columns(dir + "/polys.bin", pk.polys) || !write_columns(dir + "/cosets.bin", pk.cosets))
            return 2;
        // two members of one combination on the same row are refused
        plonk::keygen::SelectorAssignment bad = a;
        for (uint32_t t = 0; t < S; ++t) { bad.combination_of[t] = 0; bad.root_of[t] = t + 1; }
        for (auto& row : acts) row[0] = 1;
        bad.n_combinations = 1;
        bool refused = false;
        try { plonk::keygen::fixed_build_pk(*params, domain, fixed, acts, bad); }
        catch (const Panic&) { refused = true; }
        if (S > 1 && !refused) { fprintf(stderr, "overlapping members of a combination were not refused\n"); return 1; }
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("FIXED_KEYGEN_MIRROR_OK\n");
    return 0;
}
