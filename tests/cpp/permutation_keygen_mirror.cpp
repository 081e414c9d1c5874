// Drives the permutation keygen of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp): ParamsKZG::setup(k, s) with s from
// <dir>/s.bin, EvaluationDomain(5, k), the mapping (P x 2^k x 2 u64) from <dir>/mapping.bin, then permutation::keygen::build_vk /
// build_pk and keygen::lagrange_indicators(bf); writes vk.bin, permutations.bin, polys.bin, cosets.bin, l0.bin, l_last.bin, l_active.bin.
//   usage: permutation_keygen_mirror <dir> <k> <P> <bf>
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

int main(int argc, char** argv) {
    if (argc < 5) return 2;
    const std::string dir = argv[1];
    const uint32_t k = (uint32_t)atoi(argv[2]), P = (uint32_t)atoi(argv[3]), bf = (uint32_t)atoi(argv[4]);
    const size_t n = (size_t)1 << k;
    Fr s;
    FILE* f = fopen((dir + "/s.bin").c_str(), "rb");
    if (!f || fread(s.l, 8, 4, f) != 4) return 2;
    fclose(f);
    plonk::permutation::keygen::Mapping mapping(P, std::vector<std::pair<uint64_t, uint64_t>>(n));
    f = fopen((dir + "/mapping.bin").c_str(), "rb");
    if (!f) return 2;
    for (auto& c : mapping)
        if (fread(c.data(), 16, n, f) != n) return 2;
    fclose(f);
    try {
        auto params = poly::kzg::ParamsKZG::setup(k, s);
        poly::EvaluationDomain domain(5, k);
        const std::vector<G1> vk = plonk::permutation::keygen::build_vk(*params, domain, mapping);
        const plonk::permutation::keygen::ProvingKey pk = plonk::permutation::keygen::build_pk(*params, domain, mapping);
        const plonk::keygen::LagrangeIndicators ind = plonk::keygen::lagrange_indicators(domain, bf);
        if (!write_all(dir + "/vk.bin", vk.data(), vk.size() * sizeof(G1)) || !write_columns(dir + "/permutations.bin", pk.permutations) ||
            !write_columns(dir + "/polys.bin", pk.polys) || !write_columns(dir + "/cosets.bin", pk.cosets) ||
            !write_all(dir + "/l0.bin", ind.l0.data(), ind.l0.size() * sizeof(Fr)) ||
            !write_all(dir + "/l_last.bin", ind.l_last.data(), ind.l_last.size() * sizeof(Fr)) ||
            !write_all(dir + "/l_active.bin", ind.l_active_row.data(), ind.l_active_row.size() * sizeof(Fr)))
            return 2;
        // an out-of-range entry is refused as upstream's index panics
        mapping[0][1] = {P, 0};
        bool refused = false;
        try { plonk::permutation::keygen::build_pk(*params, domain, mapping); }
        catch (const Panic&) { refused = true; }
        if (!refused) { fprintf(stderr, "an out-of-range mapping entry was not refused\n"); return 1; }
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("PERMUTATION_KEYGEN_MIRROR_OK\n");
    return 0;
}
