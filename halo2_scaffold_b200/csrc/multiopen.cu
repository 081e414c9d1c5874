// The SHPLONK multi-point opening on device-resident polynomials ([UP] halo2_proofs/src/poly/kzg/multiopen/shplonk/prover.rs,
// ProverSHPLONK::create_proof) and the query evaluation it starts from (every committed polynomial at every point it is opened at,
// plonk/prover.rs's "evaluations at x" and ProverQuery::get_eval).
//
//   * plan (host, no field arithmetic): construct_intermediate_sets -- polynomials in first-appearance order with their distinct
//     points, grouped into rotation sets by equal point sets, the super point set T -- packed into one table block on the device;
//   * query evaluation: one kernel reads a polynomial's 16-coefficient chunk once and runs the chunk Horner of scan.cu for every
//     point of that polynomial (up to 16, in groups of 4 accumulators); the chunk values of every (polynomial, point) pair then go
//     down the levels of 16 together, one launch per level for all pairs;
//   * scalars (one CTA): y^j, v^i and the combined interpolant of every set, R_i = sum_j y^j R_ij = interpolate(S_i, sum_j y^j P_ij(S_i))
//     (the interpolation is linear, so one interpolation per set replaces one per polynomial); after u: z_i = Z_{T \ S_i}(u), z_0^-1,
//     every linearisation coefficient v^i z_i y^j / z_0, -Z_T(u) / z_0 and the constant -sum_i v^i z_i R_i(u) / z_0, and a status
//     word when z_0 = 0.  Nothing goes back to the host between the steps;
//   * numerators and divisions, per set: N_i = sum_j y^j P_ij - R_i in one pass, then one kate_division (scan.cu's levels) per point
//     of S_i, ping-ponging between two buffers, then h_x += v^i Q_i;
//   * linearisation: one combination of every polynomial and h_x with the constant at coefficient 0, already scaled by z_0^-1, and
//     one division by (X - u): h' = kate_division(L, u) / z_0.
#include <algorithm>

#include "common.h"

namespace h2b {

static const uint32_t MO_K = 16;                 // coefficients per chunk at every level (scan.cu's POLY_K)
static const uint32_t MO_LEVELS = 9;             // 16^8 > 2^31
static const uint32_t MO_GROUP = 4;              // points evaluated together per pass over a chunk
static const uint32_t MO_SCALAR_THREADS = 128;

// ---- plan -------------------------------------------------------------------------------------------------------------------
static bool fr_words_canonical(const uint64_t* w) {
    uint32_t l[8];
    memcpy(l, w, 32);
    for (int i = 7; i >= 0; --i) {
        if (l[i] < FpParams<FR>::P(i)) return true;
        if (l[i] > FpParams<FR>::P(i)) return false;
    }
    return false;
}
bool fr_canonical(const uint64_t w[4]) { return fr_words_canonical(w); }

int shplonk_plan_build(const char* who, const h2b_opening_query* queries, uint32_t n_queries, uint32_t n_polys, bool need_every_poly, ShplonkPlan* out) {
    if (!queries || n_queries == 0) { set_error("%s: no queries", who); return H2B_ERR_BAD_ARGUMENT; }
    ShplonkPlan p;
    std::vector<uint32_t> slot_of(n_polys, UINT32_MAX);
    std::vector<std::vector<uint32_t>> slot_points;          // T indices, first-appearance order, no repeats
    p.query_pair.resize(n_queries);
    std::vector<uint32_t> query_slot(n_queries), query_point(n_queries);
    for (uint32_t q = 0; q < n_queries; ++q) {
        const uint32_t poly = queries[q].poly;
        if (poly >= n_polys) { set_error("%s: query %u names polynomial %u of %u", who, q, poly, n_polys); return H2B_ERR_BAD_ARGUMENT; }
        if (!fr_words_canonical(queries[q].point)) { set_error("%s: the point of query %u is not below the scalar field modulus", who, q); return H2B_ERR_BAD_ARGUMENT; }
        uint32_t t = 0;
        while (t < p.n_points() && memcmp(&p.points[4 * (size_t)t], queries[q].point, 32) != 0) ++t;
        if (t == p.n_points()) p.points.insert(p.points.end(), queries[q].point, queries[q].point + 4);
        if (slot_of[poly] == UINT32_MAX) { slot_of[poly] = (uint32_t)p.used.size(); p.used.push_back(poly); slot_points.emplace_back(); }
        std::vector<uint32_t>& sp = slot_points[slot_of[poly]];
        if (std::find(sp.begin(), sp.end(), t) == sp.end()) {
            if (sp.size() == SHPLONK_MAX_POINTS) { set_error("%s: polynomial %u is opened at more than %u points", who, poly, SHPLONK_MAX_POINTS); return H2B_ERR_BAD_ARGUMENT; }
            sp.push_back(t);
        }
        query_slot[q] = slot_of[poly];
        query_point[q] = t;
    }
    if (need_every_poly && p.used.size() != n_polys) {
        for (uint32_t i = 0; i < n_polys; ++i)
            if (slot_of[i] == UINT32_MAX) { set_error("%s: no query opens polynomial %u", who, i); return H2B_ERR_BAD_ARGUMENT; }
    }
    const uint32_t P = (uint32_t)p.used.size();
    // pairs grouped by slot, in the slot's point order
    for (uint32_t s = 0; s < P; ++s) {
        p.slot_first.push_back((uint32_t)p.pair_point.size());
        p.slot_count.push_back((uint32_t)slot_points[s].size());
        for (uint32_t t : slot_points[s]) p.pair_point.push_back(t);
    }
    if (p.pair_point.size() > 65535 || P > 65535) { set_error("%s: more than 65535 distinct (polynomial, point) pairs", who); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t q = 0; q < n_queries; ++q) {
        const std::vector<uint32_t>& sp = slot_points[query_slot[q]];
        p.query_pair[q] = p.slot_first[query_slot[q]] + (uint32_t)(std::find(sp.begin(), sp.end(), query_point[q]) - sp.begin());
    }
    // rotation sets: slots with equal point sets (compared as sets), in the order their first slot appeared
    std::vector<std::vector<uint32_t>> keys;
    p.slot_set.resize(P);
    p.slot_member.resize(P);
    for (uint32_t s = 0; s < P; ++s) {
        std::vector<uint32_t> key = slot_points[s];
        std::sort(key.begin(), key.end());
        uint32_t i = 0;
        while (i < keys.size() && keys[i] != key) ++i;
        if (i == keys.size()) { keys.push_back(key); p.set_slots.emplace_back(); p.set_points.push_back(slot_points[s]); }
        p.slot_set[s] = i;
        p.slot_member[s] = (uint32_t)p.set_slots[i].size();
        p.set_slots[i].push_back(s);
    }
    *out = std::move(p);
    return H2B_OK;
}

// ---- the plan's tables on the device -----------------------------------------------------------------------------------------
struct MoSet { uint32_t member0, members, point0, points, pair0, comp0, comps, r0; };

struct MoLayout { size_t ptrs, slot_pairs, pair_pt, query_pair, sets, members, set_pts, pairidx, comp, status, jac, T, end; };
static size_t up32(size_t b) { return (b + 31) & ~(size_t)31; }
static MoLayout mo_layout(const ShplonkPlan& p) {
    size_t sum_points = 0, sum_pairs = 0, sum_comp = 0;
    for (size_t i = 0; i < p.set_slots.size(); ++i) {
        sum_points += p.set_points[i].size();
        sum_pairs += p.set_points[i].size() * p.set_slots[i].size();
        sum_comp += p.n_points() - p.set_points[i].size();
    }
    MoLayout L;
    size_t o = 0;
    L.ptrs = o;       o = up32(o + 8 * p.used.size());
    L.slot_pairs = o; o = up32(o + 8 * p.used.size());
    L.pair_pt = o;    o = up32(o + 4 * p.pair_point.size());
    L.query_pair = o; o = up32(o + 4 * p.query_pair.size());
    L.sets = o;       o = up32(o + sizeof(MoSet) * p.set_slots.size());
    L.members = o;    o = up32(o + 4 * p.used.size());
    L.set_pts = o;    o = up32(o + 4 * sum_points);
    L.pairidx = o;    o = up32(o + 4 * sum_pairs);
    L.comp = o;       o = up32(o + 4 * sum_comp + 4);
    L.status = o;     o = up32(o + 4);
    L.jac = o;        o = up32(o + 96);
    L.T = o;          o = up32(o + 32 * p.n_points());
    L.end = o;
    return L;
}
size_t shplonk_tables_bytes(const ShplonkPlan& p) { return mo_layout(p).end; }

size_t shplonk_scalars_count(const ShplonkPlan& p) {
    size_t r = 0;
    for (auto& s : p.set_points) r += s.size();
    return 2 * p.used.size() + p.set_slots.size() + r + 3;
}

int shplonk_tables_upload(const ShplonkPlan& p, const void* const* d_polys_by_slot, void* d_tables, cudaStream_t stream) {
    const MoLayout L = mo_layout(p);
    std::vector<uint8_t> h(L.end, 0);
    auto u32s = [&](size_t off) { return (uint32_t*)(h.data() + off); };
    for (size_t s = 0; s < p.used.size(); ++s) {
        const uint64_t ptr = (uint64_t)(uintptr_t)d_polys_by_slot[s];
        memcpy(h.data() + L.ptrs + 8 * s, &ptr, 8);
        u32s(L.slot_pairs)[2 * s] = p.slot_first[s];
        u32s(L.slot_pairs)[2 * s + 1] = p.slot_count[s];
    }
    if (!p.pair_point.empty()) memcpy(h.data() + L.pair_pt, p.pair_point.data(), 4 * p.pair_point.size());
    memcpy(h.data() + L.query_pair, p.query_pair.data(), 4 * p.query_pair.size());
    uint32_t member0 = 0, point0 = 0, pair0 = 0, comp0 = 0;
    for (size_t i = 0; i < p.set_slots.size(); ++i) {
        const std::vector<uint32_t>& sl = p.set_slots[i];
        const std::vector<uint32_t>& pt = p.set_points[i];
        MoSet s;
        s.member0 = member0; s.members = (uint32_t)sl.size(); s.point0 = point0; s.points = (uint32_t)pt.size();
        s.pair0 = pair0; s.comp0 = comp0; s.comps = (uint32_t)(p.n_points() - pt.size()); s.r0 = point0;
        memcpy(h.data() + L.sets + sizeof(MoSet) * i, &s, sizeof(MoSet));
        for (uint32_t j = 0; j < sl.size(); ++j) {
            u32s(L.members)[member0 + j] = sl[j];
            // pair of (member j, point k): the member's pairs hold the same points, possibly in another order
            const uint32_t f = p.slot_first[sl[j]], c = p.slot_count[sl[j]];
            for (uint32_t k = 0; k < pt.size(); ++k) {
                uint32_t e = 0;
                while (e < c && p.pair_point[f + e] != pt[k]) ++e;
                u32s(L.pairidx)[pair0 + j * pt.size() + k] = f + e;
            }
        }
        for (uint32_t k = 0; k < pt.size(); ++k) u32s(L.set_pts)[point0 + k] = pt[k];
        for (uint32_t t = 0; t < p.n_points(); ++t)
            if (std::find(pt.begin(), pt.end(), t) == pt.end()) u32s(L.comp)[comp0++] = t;
        member0 += s.members; point0 += s.points; pair0 += s.members * s.points;
    }
    memcpy(h.data() + L.T, p.points.data(), 32 * p.n_points());
    H2B_CUDA(cudaMemcpyAsync(d_tables, h.data(), L.end, cudaMemcpyHostToDevice, stream));
    // a pageable source: the copy has consumed `h` when cudaMemcpyAsync returns, but the order of the later kernels needs no wait
    return H2B_OK;
}

const void* shplonk_tables_status(const ShplonkPlan& p, const void* d_tables) { return (const char*)d_tables + mo_layout(p).status; }
const void* shplonk_tables_jac(const ShplonkPlan& p, const void* d_tables) { return (const char*)d_tables + mo_layout(p).jac; }

// ---- query evaluation ---------------------------------------------------------------------------------------------------------
// pow[t * MO_LEVELS + l] = T[t]^(16^l)
__global__ void __launch_bounds__(128) mo_point_powers_kernel(const uint4* __restrict__ T, uint32_t t_count, uint4* __restrict__ pow) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= t_count) return;
    Fr p = fp_load<FR>(T + 2 * (size_t)t);
    for (uint32_t l = 0; l < MO_LEVELS; ++l) {
        fp_store<FR>(pow + 2 * ((size_t)t * MO_LEVELS + l), p);
        for (int k = 0; k < 4; ++k) p = fp_sqr(p);
    }
}

// level 0: polynomial blockIdx.y, chunk t: out[pair * chunks + t] = sum_{i < 16} a[16 t + i] * x_pair^i for every pair (point) of the
// polynomial; the chunk is read from HBM once, the groups of MO_GROUP points after the first re-read it from L1
__global__ void __launch_bounds__(128) mo_eval_chunk_kernel(const uint64_t* __restrict__ ptrs, const uint32_t* __restrict__ slot_pairs,
                                                          const uint32_t* __restrict__ pair_pt, const uint4* __restrict__ pow, size_t n, uint32_t chunks,
                                                          uint4* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const uint32_t slot = blockIdx.y, first = slot_pairs[2 * slot], count = slot_pairs[2 * slot + 1];
    const uint4* in = (const uint4*)(uintptr_t)ptrs[slot];
    const size_t lo = (size_t)t * MO_K, hi = lo + MO_K < n ? lo + MO_K : n;
    for (uint32_t g0 = 0; g0 < count; g0 += MO_GROUP) {
        const uint32_t gm = count - g0 < MO_GROUP ? count - g0 : MO_GROUP;      // uniform over the block
        Fr x[MO_GROUP], r[MO_GROUP];
        const Fr top = fp_load<FR>(in + 2 * (hi - 1));
#pragma unroll
        for (uint32_t g = 0; g < MO_GROUP; ++g) {
            if (g < gm) { x[g] = fp_load<FR>(pow + 2 * (size_t)pair_pt[first + g0 + g] * MO_LEVELS); r[g] = top; }
        }
        for (size_t i = hi - 1; i-- > lo;) {
            const Fr a = fp_load<FR>(in + 2 * i);
#pragma unroll
            for (uint32_t g = 0; g < MO_GROUP; ++g)
                if (g < gm) r[g] = fp_add(fp_mul(r[g], x[g]), a);
        }
#pragma unroll
        for (uint32_t g = 0; g < MO_GROUP; ++g)
            if (g < gm) fp_store<FR>(out + 2 * ((size_t)(first + g0 + g) * chunks + t), r[g]);
    }
}

// level l >= 1, pair blockIdx.y: out[pair * out_stride + t] = sum_{i < 16} in[pair * m + 16 t + i] * (x_pair^(16^l))^i
__global__ void __launch_bounds__(128) mo_eval_level_kernel(const uint4* __restrict__ in, size_t m, const uint32_t* __restrict__ pair_pt,
                                                          const uint4* __restrict__ pow, uint32_t level, uint32_t chunks, uint4* __restrict__ out,
                                                          uint32_t out_stride) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= chunks) return;
    const uint32_t pair = blockIdx.y;
    const uint4* a = in + 2 * (size_t)pair * m;
    const size_t lo = (size_t)t * MO_K, hi = lo + MO_K < m ? lo + MO_K : m;
    const Fr x = fp_load<FR>(pow + 2 * ((size_t)pair_pt[pair] * MO_LEVELS + level));
    Fr r = fp_load<FR>(a + 2 * (hi - 1));
    for (size_t i = hi - 1; i-- > lo;) r = fp_add(fp_mul(r, x), fp_load<FR>(a + 2 * i));
    fp_store<FR>(out + 2 * ((size_t)pair * out_stride + t), r);
}

__global__ void __launch_bounds__(128) mo_gather_kernel(const uint4* __restrict__ evals, const uint32_t* __restrict__ query_pair, uint32_t n_queries,
                                                      uint4* __restrict__ out) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_queries) return;
    fp_store<FR>(out + 2 * (size_t)q, fp_load<FR>(evals + 2 * (size_t)query_pair[q]));
}

// every (polynomial, point) pair of the plan -> d_evals (one Fr per pair); scratch in ctx.open_scratch
int shplonk_eval_pairs_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, void* d_evals, cudaStream_t stream) {
    const MoLayout L = mo_layout(p);
    const char* tb = (const char*)d_tables;
    const uint32_t pairs = (uint32_t)p.pair_point.size(), slots = (uint32_t)p.used.size(), tc = p.n_points();
    const uint32_t chunks0 = (uint32_t)((n + MO_K - 1) / MO_K);
    size_t level_elems = 0;
    for (size_t m = chunks0; m > 1; m = (m + MO_K - 1) / MO_K) level_elems += m;
    H2B_TRY(ctx.open_scratch.reserve(((size_t)tc * MO_LEVELS + (size_t)pairs * level_elems + 2) * 32));
    uint4* pow = (uint4*)ctx.open_scratch.p;
    uint4* buf = pow + 2 * (size_t)tc * MO_LEVELS;
    const uint32_t* pair_pt = (const uint32_t*)(tb + L.pair_pt);
    H2B_LAUNCH(mo_point_powers_kernel, (tc + 127) / 128, 128, 0, stream, (const uint4*)(tb + L.T), tc, pow);
    uint4* out0 = chunks0 == 1 ? (uint4*)d_evals : buf;
    H2B_LAUNCH(mo_eval_chunk_kernel, dim3((chunks0 + 127) / 128, slots), 128, 0, stream, (const uint64_t*)(tb + L.ptrs), (const uint32_t*)(tb + L.slot_pairs),
               pair_pt, (const uint4*)pow, n, chunks0, out0);
    const uint4* in = buf;
    size_t m = chunks0;
    for (uint32_t l = 1; m > 1; ++l) {
        const uint32_t chunks = (uint32_t)((m + MO_K - 1) / MO_K);
        uint4* out = chunks == 1 ? (uint4*)d_evals : (uint4*)in + 2 * (size_t)pairs * m;
        H2B_LAUNCH(mo_eval_level_kernel, dim3((chunks + 127) / 128, pairs), 128, 0, stream, in, m, pair_pt, (const uint4*)pow, l, chunks, out,
                   chunks == 1 ? 1u : chunks);
        in = out;
        m = chunks;
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

int shplonk_eval_queries_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, void* d_pair_evals, void* d_out, cudaStream_t stream) {
    H2B_TRY(shplonk_eval_pairs_run(ctx, p, d_tables, n, d_pair_evals, stream));
    const uint32_t nq = (uint32_t)p.query_pair.size();
    H2B_LAUNCH(mo_gather_kernel, (nq + 127) / 128, 128, 0, stream, (const uint4*)d_pair_evals, (const uint32_t*)((const char*)d_tables + mo_layout(p).query_pair),
               nq, (uint4*)d_out);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// ---- scalars ------------------------------------------------------------------------------------------------------------------
// The scalar block of a session (Fr entries), P polynomials, S sets, sum_i |S_i| = Rn:
//   [0, P) y^j of each polynomial (j = its place in its set) | [P, P + S) v^i | [P + S, P + S + Rn) -R_i, |S_i| coefficients per set |
//   F0 = P + S + Rn: [F0, F0 + P) linearisation coefficient v^i z_i y^j / z_0 of each polynomial | F0 + P: -Z_T(u) / z_0 |
//   F0 + P + 1: -sum_i v^i z_i R_i(u) / z_0 | F0 + P + 2: u
struct MoScalarArgs {
    const MoSet* sets;
    const uint32_t* members;
    const uint32_t* set_pts;
    const uint32_t* pairidx;
    const uint32_t* comp;
    const uint4* T;
    const uint4* evals;
    uint4* scal;
    uint32_t* status;
    uint32_t n_sets, n_points, P, F0;
    Fr y, v;
};

// one CTA, a thread per set: y^j, v^i and R_i = interpolate(S_i, E_i) with E_i(x_k) = sum_j y^j P_ij(x_k), negated:
//   w_k = E_i(x_k) / prod_{l != k} (x_k - x_l)  (the denominators inverted in one batch),  R_i = sum_k w_k Z_{S_i}(X) / (X - x_k)
__global__ void __launch_bounds__(MO_SCALAR_THREADS) shplonk_begin_scalars_kernel(MoScalarArgs a) {
    for (uint32_t i = threadIdx.x; i < a.n_sets; i += blockDim.x) {
        const MoSet s = a.sets[i];
        const uint32_t np = s.points;
        fp_store<FR>(a.scal + 2 * (size_t)(a.P + i), fp_pow_u32<FR>(a.v, i));
        Fr e[SHPLONK_MAX_POINTS], x[SHPLONK_MAX_POINTS], pre[SHPLONK_MAX_POINTS], z[SHPLONK_MAX_POINTS + 1];
        for (uint32_t k = 0; k < np; ++k) { e[k] = fp_zero<FR>(); x[k] = fp_load<FR>(a.T + 2 * (size_t)a.set_pts[s.point0 + k]); }
        Fr yj = fp_one<FR>();
        for (uint32_t j = 0; j < s.members; ++j) {
            fp_store<FR>(a.scal + 2 * (size_t)a.members[s.member0 + j], yj);
            for (uint32_t k = 0; k < np; ++k)
                e[k] = fp_add(e[k], fp_mul(yj, fp_load<FR>(a.evals + 2 * (size_t)a.pairidx[s.pair0 + j * np + k])));
            yj = fp_mul(yj, a.y);
        }
        // denominators d_k = prod_{l != k} (x_k - x_l), inverted with Montgomery's trick
        Fr run = fp_one<FR>();
        for (uint32_t k = 0; k < np; ++k) {
            pre[k] = run;
            for (uint32_t l = 0; l < np; ++l) if (l != k) run = fp_mul(run, fp_sub(x[k], x[l]));
        }
        Fr inv = fp_inv(run);
        for (uint32_t k = np; k-- > 0;) {
            Fr d = fp_one<FR>();
            for (uint32_t l = 0; l < np; ++l) if (l != k) d = fp_mul(d, fp_sub(x[k], x[l]));
            e[k] = fp_mul(e[k], fp_mul(inv, pre[k]));
            inv = fp_mul(inv, d);
        }
        // Z(X) = prod_k (X - x_k): np + 1 coefficients
        z[0] = fp_one<FR>();
        for (uint32_t k = 0; k < np; ++k) {
            z[k + 1] = z[k];
            for (uint32_t c = k; c > 0; --c) z[c] = fp_sub(z[c - 1], fp_mul(x[k], z[c]));
            z[0] = fp_neg(fp_mul(x[k], z[0]));
        }
        // R = sum_k w_k Z / (X - x_k); the quotient by synthetic division q[np-1] = z[np] = 1, q[c-1] = z[c] + x_k q[c]
        Fr r[SHPLONK_MAX_POINTS];
        for (uint32_t c = 0; c < np; ++c) r[c] = fp_zero<FR>();
        for (uint32_t k = 0; k < np; ++k) {
            Fr q = fp_one<FR>();
            for (uint32_t c = np; c-- > 0;) {
                r[c] = fp_add(r[c], fp_mul(e[k], q));
                if (c) q = fp_add(z[c], fp_mul(x[k], q));
            }
        }
        for (uint32_t c = 0; c < np; ++c) fp_store<FR>(a.scal + 2 * (size_t)(a.P + a.n_sets + s.r0 + c), fp_neg(r[c]));
    }
}

// one CTA after u: thread 0 takes Z_T(u), z_0 and its inverse (status 1 when z_0 = 0), then a thread per set
__global__ void __launch_bounds__(MO_SCALAR_THREADS) shplonk_finish_scalars_kernel(MoScalarArgs a) {
    __shared__ Fr sh[MO_SCALAR_THREADS + 2];
    const uint32_t tid = threadIdx.x;
    const uint32_t iu = a.F0 + a.P + 2;
    const Fr u = fp_load<FR>(a.scal + 2 * (size_t)iu);
    if (tid == 0) {
        Fr zt = fp_one<FR>(), z0 = fp_one<FR>();
        for (uint32_t t = 0; t < a.n_points; ++t) zt = fp_mul(zt, fp_sub(u, fp_load<FR>(a.T + 2 * (size_t)t)));
        const MoSet s0 = a.sets[0];
        for (uint32_t c = 0; c < s0.comps; ++c) z0 = fp_mul(z0, fp_sub(u, fp_load<FR>(a.T + 2 * (size_t)a.comp[s0.comp0 + c])));
        *a.status = fp_is_zero(z0) ? 1u : 0u;
        sh[MO_SCALAR_THREADS] = fp_inv(z0);
        sh[MO_SCALAR_THREADS + 1] = zt;
    }
    __syncthreads();
    const Fr z0inv = sh[MO_SCALAR_THREADS];
    Fr acc = fp_zero<FR>();
    for (uint32_t i = tid; i < a.n_sets; i += blockDim.x) {
        const MoSet s = a.sets[i];
        Fr zi = fp_one<FR>();
        for (uint32_t c = 0; c < s.comps; ++c) zi = fp_mul(zi, fp_sub(u, fp_load<FR>(a.T + 2 * (size_t)a.comp[s.comp0 + c])));
        const Fr w = fp_mul(fp_mul(fp_load<FR>(a.scal + 2 * (size_t)(a.P + i)), zi), z0inv);
        const uint4* nr = a.scal + 2 * (size_t)(a.P + a.n_sets + s.r0);
        Fr h = fp_load<FR>(nr + 2 * (size_t)(s.points - 1));
        for (uint32_t c = s.points - 1; c-- > 0;) h = fp_add(fp_mul(h, u), fp_load<FR>(nr + 2 * (size_t)c));
        acc = fp_add(acc, fp_mul(w, h));
        for (uint32_t j = 0; j < s.members; ++j) {
            const uint32_t slot = a.members[s.member0 + j];
            fp_store<FR>(a.scal + 2 * (size_t)(a.F0 + slot), fp_mul(w, fp_load<FR>(a.scal + 2 * (size_t)slot)));
        }
    }
    __syncthreads();
    sh[tid] = acc;
    __syncthreads();
    if (tid == 0) {
        Fr c = sh[0];
        for (uint32_t t = 1; t < blockDim.x; ++t) c = fp_add(c, sh[t]);
        fp_store<FR>(a.scal + 2 * (size_t)(a.F0 + a.P + 1), c);
        fp_store<FR>(a.scal + 2 * (size_t)(a.F0 + a.P), fp_neg(fp_mul(sh[MO_SCALAR_THREADS + 1], z0inv)));
    }
}

// ---- combinations with coefficients on the device -------------------------------------------------------------------------------
// out[i] (+)= sum_j scal[coef[j]] * cols[j][i]  (+ scal[low0 + i] for i < lows), i < len
static const uint32_t MO_COMBINE_MAX = 32;
struct MoCombine {
    const uint4* cols[MO_COMBINE_MAX];
    uint32_t coef[MO_COMBINE_MAX];
    uint32_t m, accumulate, low0, lows;
};
__global__ void __launch_bounds__(128) mo_combine_kernel(MoCombine p, const uint4* __restrict__ scal, size_t len, uint4* __restrict__ out) {
    __shared__ Fr c[MO_COMBINE_MAX];
    if (threadIdx.x < p.m) c[threadIdx.x] = fp_load<FR>(scal + 2 * (size_t)p.coef[threadIdx.x]);
    __syncthreads();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len) return;
    Fr acc = p.accumulate ? fp_load<FR>(out + 2 * i) : fp_zero<FR>();
    for (uint32_t j = 0; j < p.m; ++j) acc = fp_add(acc, fp_mul(c[j], fp_load<FR>(p.cols[j] + 2 * i)));
    if (i < p.lows) acc = fp_add(acc, fp_load<FR>(scal + 2 * ((size_t)p.low0 + i)));
    fp_store<FR>(out + 2 * i, acc);
}

// cols[j] with scalar indices coef[j], in launches of MO_COMBINE_MAX columns; the low constants go with the first launch
static int mo_combine(const std::vector<const void*>& cols, const std::vector<uint32_t>& coef, bool accumulate, uint32_t low0, uint32_t lows,
                      const uint4* scal, size_t len, void* d_out, cudaStream_t stream) {
    if (len == 0) return H2B_OK;
    for (size_t lo = 0; lo < cols.size() || lo == 0; lo += MO_COMBINE_MAX) {
        MoCombine p;
        memset(&p, 0, sizeof(p));
        p.m = (uint32_t)(cols.size() - lo < MO_COMBINE_MAX ? cols.size() - lo : MO_COMBINE_MAX);
        for (uint32_t j = 0; j < p.m; ++j) { p.cols[j] = (const uint4*)cols[lo + j]; p.coef[j] = coef[lo + j]; }
        p.accumulate = (accumulate || lo) ? 1u : 0u;
        if (lo == 0) { p.low0 = low0; p.lows = lows; }
        H2B_LAUNCH(mo_combine_kernel, (unsigned)((len + 127) / 128), 128, 0, stream, p, scal, len, (uint4*)d_out);
        if (cols.empty()) break;
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

static MoScalarArgs mo_scalar_args(const ShplonkPlan& p, const void* d_tables, const void* d_evals, void* d_scal) {
    const MoLayout L = mo_layout(p);
    const char* tb = (const char*)d_tables;
    MoScalarArgs a;
    memset(&a, 0, sizeof(a));
    a.sets = (const MoSet*)(tb + L.sets); a.members = (const uint32_t*)(tb + L.members); a.set_pts = (const uint32_t*)(tb + L.set_pts);
    a.pairidx = (const uint32_t*)(tb + L.pairidx); a.comp = (const uint32_t*)(tb + L.comp); a.T = (const uint4*)(tb + L.T);
    a.status = (uint32_t*)(tb + L.status); a.evals = (const uint4*)d_evals; a.scal = (uint4*)d_scal;
    a.n_sets = (uint32_t)p.set_slots.size(); a.n_points = p.n_points(); a.P = (uint32_t)p.used.size();
    a.F0 = (uint32_t)(shplonk_scalars_count(p) - a.P - 3);
    return a;
}

// steps 2-5 up to h_x: evaluations, interpolants, numerators, divisions, the v-sum.  d_a, d_b, d_hx: n Fr each.
int shplonk_begin_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, const uint64_t y[4], const uint64_t v[4], void* d_evals,
                      void* d_scal, void* d_hx, void* d_a, void* d_b, cudaStream_t stream) {
    H2B_TRY(shplonk_eval_pairs_run(ctx, p, d_tables, n, d_evals, stream));
    ctx.prof.mark(PROF_OPEN_EVAL, stream);
    MoScalarArgs a = mo_scalar_args(p, d_tables, d_evals, d_scal);
    memcpy(a.y.l, y, 32);
    memcpy(a.v.l, v, 32);
    H2B_LAUNCH(shplonk_begin_scalars_kernel, 1, MO_SCALAR_THREADS, 0, stream, a);
    ctx.prof.mark(PROF_OPEN_SCALARS, stream);
    H2B_CUDA(cudaMemsetAsync(d_hx, 0, n * 32, stream));
    const MoLayout L = mo_layout(p);
    const uint4* T = (const uint4*)((const char*)d_tables + L.T);
    const uint4* scal = (const uint4*)d_scal;
    uint32_t r0 = 0;
    for (uint32_t i = 0; i < a.n_sets; ++i) {
        const std::vector<uint32_t>& sl = p.set_slots[i];
        const std::vector<uint32_t>& pt = p.set_points[i];
        std::vector<const void*> cols;
        std::vector<uint32_t> coef;
        for (uint32_t s : sl) { cols.push_back(p.d_polys[s]); coef.push_back(s); }
        H2B_TRY(mo_combine(cols, coef, false, a.P + a.n_sets + r0, (uint32_t)pt.size(), scal, n, d_a, stream));
        void* cur = d_a;
        void* nxt = d_b;
        size_t len = n;
        for (uint32_t t : pt) {
            if (len <= 1) { len = 0; break; }
            H2B_TRY(fr_kate_division_at_run(ctx, cur, len, T + 2 * (size_t)t, nxt, stream));
            --len;
            std::swap(cur, nxt);
        }
        H2B_TRY(mo_combine(std::vector<const void*>{cur}, std::vector<uint32_t>{a.P + i}, true, 0, 0, scal, len, d_hx, stream));
        r0 += (uint32_t)pt.size();
    }
    ctx.prof.mark(PROF_OPEN_NUMERATORS, stream);
    return H2B_OK;
}

// step 7 up to h' = kate_division(L, u) / z_0 in d_b (n - 1 coefficients); the status word of the tables is 1 when z_0 = 0
int shplonk_finish_run(DeviceCtx& ctx, const ShplonkPlan& p, const void* d_tables, size_t n, const uint64_t u[4], const void* d_evals, void* d_scal,
                       const void* d_hx, void* d_a, void* d_b, cudaStream_t stream) {
    MoScalarArgs a = mo_scalar_args(p, d_tables, d_evals, d_scal);
    uint4* uslot = (uint4*)d_scal + 2 * (size_t)(a.F0 + a.P + 2);
    H2B_CUDA(cudaMemcpyAsync(uslot, u, 32, cudaMemcpyHostToDevice, stream));
    H2B_LAUNCH(shplonk_finish_scalars_kernel, 1, MO_SCALAR_THREADS, 0, stream, a);
    ctx.prof.mark(PROF_OPEN_SCALARS, stream);
    std::vector<const void*> cols;
    std::vector<uint32_t> coef;
    for (uint32_t s = 0; s < a.P; ++s) { cols.push_back(p.d_polys[s]); coef.push_back(a.F0 + s); }
    cols.push_back(d_hx);
    coef.push_back(a.F0 + a.P);
    H2B_TRY(mo_combine(cols, coef, false, a.F0 + a.P + 1, 1, (const uint4*)d_scal, n, d_a, stream));
    H2B_TRY(fr_kate_division_at_run(ctx, d_a, n, uslot, d_b, stream));
    ctx.prof.mark(PROF_OPEN_LINEARISE, stream);
    return H2B_OK;
}

}  // namespace h2b
