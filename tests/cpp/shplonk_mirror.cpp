// Drives ProverSHPLONK::create_proof of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp): ParamsKZG::setup(k, s) with s from
// <dir>/s.bin, P polynomials (P x 2^k x 4 u64) from <dir>/polys.bin, Q queries (poly u32 per query in <dir>/qpoly.bin, points Q x 4 u64 in
// <dir>/qpoint.bin) and y | v | u from <dir>/yvu.bin; writes h1 | h2 (2 x 12 u64, Jacobian) to <dir>/h.bin.
//   usage: shplonk_mirror <dir> <k> <P> <Q>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../halo2_scaffold_b200/host/h2b200.hpp"

using namespace h2b200;

template <class T>
static bool read_all(const std::string& path, T* p, size_t count) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    const bool ok = fread(p, sizeof(T), count, f) == count;
    fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc < 5) return 2;
    const std::string dir = argv[1];
    const uint32_t k = (uint32_t)atoi(argv[2]), P = (uint32_t)atoi(argv[3]), Q = (uint32_t)atoi(argv[4]);
    const size_t n = (size_t)1 << k;
    Fr s, yvu[3];
    std::vector<std::vector<Fr>> polys(P, std::vector<Fr>(n));
    std::vector<uint32_t> qpoly(Q);
    std::vector<Fr> qpoint(Q);
    bool ok = read_all(dir + "/s.bin", &s, 1) && read_all(dir + "/yvu.bin", yvu, 3) && read_all(dir + "/qpoly.bin", qpoly.data(), Q) &&
              read_all(dir + "/qpoint.bin", qpoint.data(), Q);
    FILE* f = fopen((dir + "/polys.bin").c_str(), "rb");
    for (auto& p : polys) ok = ok && f && fread(p.data(), sizeof(Fr), n, f) == n;
    if (f) fclose(f);
    if (!ok) return 2;
    try {
        auto params = poly::kzg::ParamsKZG::setup(k, s);
        std::vector<poly::kzg::Query> queries;
        for (uint32_t i = 0; i < Q; ++i) queries.push_back(poly::kzg::Query{qpoly[i], qpoint[i]});
        int squeezed = 0;
        const auto h = poly::kzg::ProverSHPLONK(*params).create_proof(polys, queries, yvu[0], yvu[1], [&](const G1&) { ++squeezed; return yvu[2]; });
        if (squeezed != 1) return 1;
        FILE* w = fopen((dir + "/h.bin").c_str(), "wb");
        if (!w || fwrite(&h.first, sizeof(G1), 1, w) != 1 || fwrite(&h.second, sizeof(G1), 1, w) != 1) return 2;
        fclose(w);
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("SHPLONK_MIRROR_OK\n");
    return 0;
}
