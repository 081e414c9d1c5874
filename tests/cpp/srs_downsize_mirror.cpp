// Drives ParamsKZG::downsize of the C++ host mirror (halo2_scaffold_b200/host/h2b200.hpp): setup(K, s) with s (4 words,
// Montgomery) from <dir>/s.bin, then downsize(k); writes g.bin / g_lagrange.bin for the test to compare with setup(k, s).
//   usage: srs_downsize_mirror <dir> <K> <k>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../halo2_scaffold_b200/host/h2b200.hpp"

using namespace h2b200;

int main(int argc, char** argv) {
    if (argc < 4) return 2;
    const std::string dir = argv[1];
    const uint32_t K = (uint32_t)atoi(argv[2]), k = (uint32_t)atoi(argv[3]);
    const size_t n = (size_t)1 << k;
    Fr s;
    FILE* f = fopen((dir + "/s.bin").c_str(), "rb");
    if (!f || fread(s.l, 8, 4, f) != 4) return 2;
    fclose(f);
    try {
        auto params = poly::kzg::ParamsKZG::setup(K, s);
        params->downsize(k);
        if (params->k() != k || params->n() != n || params->get_g().size() != n || params->get_g_lagrange().size() != n) {
            fprintf(stderr, "downsize left k / n / the vectors inconsistent\n");
            return 1;
        }
        const struct { const char* name; const void* p; size_t bytes; } outs[] = {
            {"/g.bin", params->get_g().data(), n * sizeof(G1Affine)}, {"/g_lagrange.bin", params->get_g_lagrange().data(), n * sizeof(G1Affine)}};
        for (const auto& o : outs) {
            FILE* w = fopen((dir + o.name).c_str(), "wb");
            if (!w || fwrite(o.p, 1, o.bytes, w) != o.bytes) return 2;
            fclose(w);
        }
        // upstream asserts k <= self.k
        bool refused = false;
        try { params->downsize(k + 1); }
        catch (const Panic&) { refused = true; }
        if (!refused) { fprintf(stderr, "downsize(k + 1) was not refused\n"); return 1; }
    } catch (const std::exception& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    printf("SRS_DOWNSIZE_MIRROR_OK\n");
    return 0;
}
