// Drives ParamsKZG::setup of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp): reads s (4 words, Montgomery) from
// <dir>/s.bin, writes g.bin / g_lagrange.bin and a commitment of <dir>/poly.bin over each resident vector for the test to
// compare with the oracle.
//   usage: srs_setup_mirror <dir> <k>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../halo2_scaffold_b200/host/h2b200.hpp"

using namespace h2b200;

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    const std::string dir = argv[1];
    const uint32_t k = (uint32_t)atoi(argv[2]);
    const size_t n = (size_t)1 << k;
    Fr s;
    std::vector<Fr> poly(n);
    FILE* f = fopen((dir + "/s.bin").c_str(), "rb");
    if (!f || fread(s.l, 8, 4, f) != 4) return 2;
    fclose(f);
    f = fopen((dir + "/poly.bin").c_str(), "rb");
    if (!f || fread(poly.data(), sizeof(Fr), n, f) != n) return 2;
    fclose(f);
    try {
        auto params = poly::kzg::ParamsKZG::setup(k, s);
        G1 c[2] = {params->commit(poly), params->commit_lagrange(poly)};
        const struct { const char* name; const void* p; size_t bytes; } outs[] = {
            {"/g.bin", params->get_g().data(), n * sizeof(G1Affine)}, {"/g_lagrange.bin", params->get_g_lagrange().data(), n * sizeof(G1Affine)},
            {"/commit.bin", c, sizeof(c)}};
        for (const auto& o : outs) {
            FILE* w = fopen((dir + o.name).c_str(), "wb");
            if (!w || fwrite(o.p, 1, o.bytes, w) != o.bytes) return 2;
            fclose(w);
        }
        // the caller's s is checked: s = 1 is refused as upstream's setup panics on it
        bool refused = false;
        try { poly::kzg::ParamsKZG::setup(k, Fr{{0xac96341c4ffffffbULL, 0x36fc76959f60cd29ULL, 0x666ea36f7879462eULL, 0x0e0a77c19a07df2fULL}}); }
        catch (const Panic&) { refused = true; }
        if (!refused) { fprintf(stderr, "setup(k, 1) was not refused\n"); return 1; }
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("SRS_SETUP_MIRROR_OK\n");
    return 0;
}
