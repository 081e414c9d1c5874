// C ABI of libh2b200, MockProver::verify's row loops: h2b_mock_verify.
#include "host.h"

namespace h2b {

// everything about a circuit that can be refused on the host, before the device is touched
static int mock_args_check(const h2b_mock_circuit* c, const h2b_mock_record* records, uint64_t capacity, const uint64_t* count) {
    static const char* who = "h2b_mock_verify";
    if (!c || !count || (capacity && !records)) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    if (c->k == 0 || c->k > 28) { set_error("%s: k = %u (1 <= k <= 28)", who, c->k); return H2B_ERR_BAD_ARGUMENT; }
    const uint64_t n = 1ull << c->k;
    if ((uint64_t)c->blinding_factors + 1 >= n) { set_error("%s: blinding_factors + 1 = %llu leaves no usable row of %llu", who, (unsigned long long)c->blinding_factors + 1, (unsigned long long)n); return H2B_ERR_BAD_ARGUMENT; }
    if ((c->n_fixed && (!c->fixed || !c->fixed_assigned)) || (c->n_advice && (!c->advice || !c->advice_assigned)) || (c->n_instance && !c->instance) ||
        (c->n_challenges && !c->challenges) || (c->n_roots && (!c->gates || !c->roots)) || (c->n_lookups && !c->lookups) ||
        (c->n_permutation && (!c->permutation || !c->mapping))) {
        set_error("%s: null array with a non-zero count", who);
        return H2B_ERR_BAD_ARGUMENT;
    }
    for (uint32_t i = 0; i < c->n_fixed; ++i) if (!c->fixed[i] || !c->fixed_assigned[i]) { set_error("%s: fixed column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < c->n_advice; ++i) if (!c->advice[i] || !c->advice_assigned[i]) { set_error("%s: advice column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < c->n_instance; ++i) if (!c->instance[i]) { set_error("%s: instance column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    const uint64_t usable = n - (c->blinding_factors + 1), limit = 1ull << 31;
    for (uint32_t z = 1; z < c->n_roots; ++z)
        if (c->roots[z].gate < c->roots[z - 1].gate) { set_error("%s: root %u of gate %u follows a root of gate %u (roots go in gate order)", who, z, c->roots[z].gate, c->roots[z - 1].gate); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t l = 0; l < c->n_lookups; ++l) {
        const h2b_mock_lookup& lk = c->lookups[l];
        if (lk.m == 0 || lk.m > H2B_MOCK_MAX_LOOKUP_WIDTH) { set_error("%s: lookup %u has %u expressions per side (1 .. %u)", who, l, lk.m, H2B_MOCK_MAX_LOOKUP_WIDTH); return H2B_ERR_BAD_ARGUMENT; }
        if (!lk.inputs || !lk.tables) { set_error("%s: lookup %u: null root list", who, l); return H2B_ERR_BAD_ARGUMENT; }
    }
    for (uint32_t i = 0; i < c->n_permutation; ++i) {
        const h2b_mock_column& col = c->permutation[i];
        const uint32_t count_of = col.kind == H2B_VS_FIXED ? c->n_fixed : col.kind == H2B_VS_ADVICE ? c->n_advice : col.kind == H2B_VS_INSTANCE ? c->n_instance : 0;
        if (col.index >= count_of) { set_error("%s: permutation column %u: (kind %u, index %u) is not a column of the circuit", who, i, col.kind, col.index); return H2B_ERR_BAD_ARGUMENT; }
        if (!c->mapping[i]) { set_error("%s: mapping column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    }
    if ((uint64_t)c->n_roots * n >= limit || (uint64_t)c->n_lookups * usable >= limit || (uint64_t)c->n_permutation * n >= limit) {
        set_error("%s: more than 2^31 (root, row), (lookup, row) or (column, row) pairs", who);
        return H2B_ERR_BAD_ARGUMENT;
    }
    return mock_verify_check(c);
}

}  // namespace h2b

using namespace h2b;

extern "C" {

int h2b_mock_verify(int device, const h2b_mock_circuit* circuit, h2b_mock_record* records, uint64_t capacity, uint64_t* count) {
    return on_device(device, [&]() -> int { return mock_args_check(circuit, records, capacity, count); },
                     [&](DeviceCtx& c) -> int { return mock_verify_run(c, circuit, records, capacity, count); });
}

}  // extern "C"
