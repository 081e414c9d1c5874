// 256-bit sort keys (canonical Fr values, limb 7 most significant) and their sort: shared by the lookup argument's permutation
// (lookup.cu, which implements the sort) and the MockProver checker (mock.cu).
#pragma once
#include "common.h"

namespace h2b {

static const uint32_t SORT_TILE_LOG = 10, SORT_TILE = 1u << SORT_TILE_LOG;       // elements per CTA in the shared-memory phases

struct Key { uint32_t l[8]; };
__device__ __forceinline__ bool key_less(const Key& a, const Key& b) {
#pragma unroll
    for (int i = 7; i >= 0; --i) {
        if (a.l[i] != b.l[i]) return a.l[i] < b.l[i];
    }
    return false;
}
__device__ __forceinline__ bool key_eq(const Key& a, const Key& b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a.l[i] ^ b.l[i];
    return o == 0;
}
__device__ __forceinline__ Key key_load(const uint4* p, size_t i) {
    const uint4 a = p[2 * i], b = p[2 * i + 1];
    Key k;
    k.l[0] = a.x; k.l[1] = a.y; k.l[2] = a.z; k.l[3] = a.w; k.l[4] = b.x; k.l[5] = b.y; k.l[6] = b.z; k.l[7] = b.w;
    return k;
}
__device__ __forceinline__ void key_store(uint4* p, size_t i, const Key& k) {
    p[2 * i] = make_uint4(k.l[0], k.l[1], k.l[2], k.l[3]);
    p[2 * i + 1] = make_uint4(k.l[4], k.l[5], k.l[6], k.l[7]);
}

// ---- lookup.cu ----
// ascending bitonic sort of `padded` keys (a power of two, at least SORT_TILE)
int bitonic_sort(uint4* keys, uint32_t padded, cudaStream_t stream);

}  // namespace h2b
