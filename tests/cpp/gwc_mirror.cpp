// Drives ProverGWC::create_proof of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp): ParamsKZG::setup(k, s) with s from
// <dir>/s.bin, P polynomials (P x 2^k x 4 u64) from <dir>/polys.bin, Q queries (poly u32 per query in <dir>/qpoly.bin, points Q x 4 u64 in
// <dir>/qpoint.bin) and v from <dir>/v.bin; writes W of every distinct point (points x 12 u64, Jacobian) to <dir>/w.bin.
//   usage: gwc_mirror <dir> <k> <P> <Q>
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
    Fr s, v;
    std::vector<std::vector<Fr>> polys(P, std::vector<Fr>(n));
    std::vector<uint32_t> qpoly(Q);
    std::vector<Fr> qpoint(Q);
    bool ok = read_all(dir + "/s.bin", &s, 1) && read_all(dir + "/v.bin", &v, 1) && read_all(dir + "/qpoly.bin", qpoly.data(), Q) &&
              read_all(dir + "/qpoint.bin", qpoint.data(), Q);
    FILE* f = fopen((dir + "/polys.bin").c_str(), "rb");
    for (auto& p : polys) ok = ok && f && fread(p.data(), sizeof(Fr), n, f) == n;
    if (f) fclose(f);
    if (!ok) return 2;
    try {
        auto params = poly::kzg::ParamsKZG::setup(k, s);
        std::vector<poly::kzg::Query> queries;
        for (uint32_t i = 0; i < Q; ++i) queries.push_back(poly::kzg::Query{qpoly[i], qpoint[i]});
        const std::vector<G1> w = poly::kzg::ProverGWC(*params).create_proof(polys, queries, v);
        if (w.empty()) return 1;
        FILE* out = fopen((dir + "/w.bin").c_str(), "wb");
        if (!out || fwrite(w.data(), sizeof(G1), w.size(), out) != w.size()) return 2;
        fclose(out);
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("GWC_MIRROR_OK\n");
    return 0;
}
