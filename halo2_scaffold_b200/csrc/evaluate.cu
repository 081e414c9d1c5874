// Quotient evaluation on device-resident extended-coset columns (SURVEY.md section 8f, rank 2):
// [UP] halo2_proofs/src/plonk/evaluation.rs -- `GraphEvaluator::evaluate` for the custom gates and the lookup
// compressions, and the fixed-function permutation / lookup terms of `Evaluator::evaluate_h`.  On the CPU every row walks
// the calculation list and keeps one `intermediates` vector per thread; here
//   * the host COMPILES the calculation list once per call into micro-operations: dead calculations are dropped, `Store`s
//     of columns / constants are forwarded to their consumers, `Horner` is unrolled into multiply-add steps, and the
//     calculations are re-scheduled depth-first so that a value is produced right before its consumer.  A Horner over all
//     gate polynomials (how upstream combines them with y) then needs a handful of live values instead of one per gate.
//     Field arithmetic is exact, so any schedule gives the bits upstream's sequential walk gives;
//   * live values get physical slots by reference counting; a result consumed by the very next micro-operation is
//     forwarded in registers and never stored;
//   * one thread evaluates one row (grid-stride, consecutive threads on consecutive rows, so every column read is a
//     coalesced 32-byte-per-lane access); the slots live in per-thread local memory (hardware-interleaved, L1-resident).
// The kernels are bound by the Fr multiplication rate (IMAD), like everything else on this path.
#include <algorithm>
#include <cstdlib>

#include "evaluate.cuh"

namespace h2b {

struct LookupTerms {            // the lookup argument's extra columns
    const uint4 *product, *permuted_input, *permuted_table, *l0, *l_last, *l_active_row;
    uint32_t off_next, off_prev;    // rot_scale and -rot_scale, reduced mod size
    uint32_t beta, gamma, y;        // indices into the constants table
};

template <int S>
__device__ __forceinline__ Fr eval_row(const EvalProgram& p, uint32_t idx, Fr* slots) {
    Fr r = fp_zero<FR>();
#pragma unroll 1
    for (uint32_t i = 0; i < p.n_ops; ++i) {
        const uint4 op = __ldg(p.ops + i);
        const uint32_t code = op.x & 0x7f;
        Fr a = eval_fetch(p, op.y, idx, slots, r);
        Fr out;
        if (code == MOP_MUL || code == MOP_FMA) {
            Fr b = eval_fetch(p, op.z, idx, slots, r);
            out = fp_mul(a, b);
            if (code == MOP_FMA) out = fp_add(out, eval_fetch(p, op.w, idx, slots, r));
        } else if (code == MOP_ADD) {
            out = fp_add(a, eval_fetch(p, op.z, idx, slots, r));
        } else if (code == MOP_SUB) {
            out = fp_sub(a, eval_fetch(p, op.z, idx, slots, r));
        } else if (code == MOP_SQR) {
            out = fp_sqr(a);
        } else if (code == MOP_DBL) {
            out = fp_dbl(a);
        } else if (code == MOP_NEG) {
            out = fp_neg(a);
        } else {
            out = a;
        }
        r = out;
        if (!(op.x & MOP_NOSTORE)) slots[(op.x >> 8) & (S - 1)] = out;
    }
    return r;
}

// MODE 0: values[idx] = graph(idx) (custom gates).  MODE 1: lookup terms with table_value = graph(idx).
template <int S, int MODE>
__global__ void __launch_bounds__(128) evaluate_graph_kernel(EvalProgram p, uint4* __restrict__ values, LookupTerms lk) {
    Fr slots[S];
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.rows; i += stride) {
        const uint32_t idx = p.row0 + i;                           // global row; `i` indexes the (halo-free) values slice
        const uint32_t li = shard_local(idx, p.base, p.size);        // the same row inside the column slices
        Fr g = eval_row<S>(p, idx, slots);
        if (MODE == 0) {
            fp_store<FR>(values + 2 * (size_t)i, g);
        } else {
            const Fr beta = fp_load<FR>(p.consts + 2 * (size_t)lk.beta), gamma = fp_load<FR>(p.consts + 2 * (size_t)lk.gamma);
            const Fr y = fp_load<FR>(p.consts + 2 * (size_t)lk.y);
            uint32_t r_next = idx + lk.off_next, r_prev = idx + lk.off_prev;
            if (r_next >= p.size) r_next -= p.size;
            if (r_prev >= p.size) r_prev -= p.size;
            r_next = shard_local(r_next, p.base, p.size);
            r_prev = shard_local(r_prev, p.base, p.size);
            const Fr z = fp_load<FR>(lk.product + 2 * (size_t)li), z_next = fp_load<FR>(lk.product + 2 * (size_t)r_next);
            const Fr a = fp_load<FR>(lk.permuted_input + 2 * (size_t)li), a_prev = fp_load<FR>(lk.permuted_input + 2 * (size_t)r_prev);
            const Fr s = fp_load<FR>(lk.permuted_table + 2 * (size_t)li);
            const Fr l0 = fp_load<FR>(lk.l0 + 2 * (size_t)li), l_last = fp_load<FR>(lk.l_last + 2 * (size_t)li);
            const Fr l_active = fp_load<FR>(lk.l_active_row + 2 * (size_t)li);
            const Fr a_minus_s = fp_sub(a, s);
            Fr v = fp_load<FR>(values + 2 * (size_t)i);
            // l_0(X) * (1 - z(X)) = 0
            v = fp_add(fp_mul(v, y), fp_mul(fp_sub(fp_one<FR>(), z), l0));
            // l_last(X) * (z(X)^2 - z(X)) = 0
            v = fp_add(fp_mul(v, y), fp_mul(fp_sub(fp_sqr(z), z), l_last));
            // (1 - (l_last + l_blind)) * (z(wX) (a' + beta) (s' + gamma) - z(X) * table_value) = 0
            Fr t = fp_mul(fp_mul(z_next, fp_add(a, beta)), fp_add(s, gamma));
            v = fp_add(fp_mul(v, y), fp_mul(fp_sub(t, fp_mul(z, g)), l_active));
            // l_0(X) * (a'(X) - s'(X)) = 0
            v = fp_add(fp_mul(v, y), fp_mul(a_minus_s, l0));
            // (1 - (l_last + l_blind)) * (a' - s') * (a' - a'(w^-1 X)) = 0
            v = fp_add(fp_mul(v, y), fp_mul(fp_mul(a_minus_s, fp_sub(a, a_prev)), l_active));
            fp_store<FR>(values + 2 * (size_t)i, v);
        }
    }
}

// ---- host: compile a GraphEvaluator --------------------------------------------------------------------------------
namespace {

struct Ref {            // a resolved operand: either an external source (already encoded) or the value of calculation `def`
    int32_t def = -1;
    uint32_t enc = 0;
};

thread_local uint32_t t_last_slots = 0, t_last_ops = 0;

// whole domain when `sh` is null; otherwise rows [row0, row0 + rows) with `halo` rows of every column on both sides
static int make_shard(const h2b_eval_shard* sh, uint32_t size, Shard& out) {
    if (!sh) { out = Shard{0, size, 0, 0}; return H2B_OK; }
    if (sh->rows == 0 || sh->row0 >= size || sh->rows > size - sh->row0 || (uint64_t)sh->rows + 2ull * sh->halo > size) {
        set_error("evaluate: shard [%u, %u) + halo %u does not fit a domain of %u rows", sh->row0, sh->row0 + sh->rows, sh->halo, size);
        return H2B_ERR_BAD_ARGUMENT;
    }
    out.row0 = sh->row0; out.rows = sh->rows; out.halo = sh->halo;
    out.base = sh->row0 >= sh->halo ? sh->row0 - sh->halo : size - (sh->halo - sh->row0);
    return H2B_OK;
}
// a rotated read at offset `off` (already reduced mod size) must stay inside the halo
static bool offset_within_halo(uint32_t off, uint32_t size, const Shard& sh) {
    if (sh.rows == size && sh.halo == 0) return true;
    return off <= sh.halo || size - off <= sh.halo;
}

static uint32_t rem_euclid_u32(int64_t v, uint32_t size) {
    int64_t m = v % (int64_t)size;
    if (m < 0) m += size;
    return (uint32_t)m;
}

}  // namespace

int compile_graph(const h2b_graph* g, const h2b_eval_columns* cols, const void* d_values, uint32_t size, int32_t rot_scale, bool previous_is_zero,
                  const Shard& shard, const h2b_value_source* roots, uint32_t n_roots, Compiled& out) {
    if (n_roots && !roots) { set_error("evaluate: null root list"); return H2B_ERR_BAD_ARGUMENT; }
    if (!g || !cols) { set_error("evaluate: null graph / columns"); return H2B_ERR_BAD_ARGUMENT; }
    if (size == 0 || size > (1u << 30)) { set_error("evaluate: size must be in [1, 2^30]"); return H2B_ERR_BAD_ARGUMENT; }
    if ((g->n_constants && !g->constants) || (g->n_rotations && !g->rotations) || (g->n_calculations && !g->calculations) || (g->n_parts && !g->parts) ||
        (cols->n_fixed && !cols->fixed) || (cols->n_advice && !cols->advice) || (cols->n_instance && !cols->instance) ||
        (cols->n_challenges && !cols->challenges) || !cols->beta || !cols->gamma || !cols->theta || !cols->y) {
        set_error("evaluate: null array with a non-zero count");
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (g->n_rotations + 1 > MAX_ROT) { set_error("evaluate: at most %u rotations", MAX_ROT - 1); return H2B_ERR_BAD_ARGUMENT; }
    const uint64_t total_cols = (uint64_t)cols->n_fixed + cols->n_advice + cols->n_instance + 1;
    if (total_cols > MAX_COLS) { set_error("evaluate: too many columns"); return H2B_ERR_BAD_ARGUMENT; }

    // constants table: graph constants | challenges | beta gamma theta y | zero
    const uint32_t nc = g->n_constants, nch = cols->n_challenges;
    out.consts.assign((size_t)(nc + nch + 5) * 4, 0);
    if (nc) memcpy(out.consts.data(), g->constants, (size_t)nc * 32);
    if (nch) memcpy(out.consts.data() + (size_t)nc * 4, cols->challenges, (size_t)nch * 32);
    out.c_beta = nc + nch; out.c_gamma = nc + nch + 1; out.c_theta = nc + nch + 2; out.c_y = nc + nch + 3; out.c_zero = nc + nch + 4;
    memcpy(out.consts.data() + (size_t)out.c_beta * 4, cols->beta, 32);
    memcpy(out.consts.data() + (size_t)out.c_gamma * 4, cols->gamma, 32);
    memcpy(out.consts.data() + (size_t)out.c_theta * 4, cols->theta, 32);
    memcpy(out.consts.data() + (size_t)out.c_y * 4, cols->y, 32);
    // rotations (get_rotation_idx with the row added on the device) and the unified column table
    out.rot_off.resize(g->n_rotations + 1);
    for (uint32_t i = 0; i < g->n_rotations; ++i) out.rot_off[i] = rem_euclid_u32((int64_t)g->rotations[i] * rot_scale, size);
    out.rot_off[g->n_rotations] = 0;
    out.cols.clear();
    for (uint32_t i = 0; i < cols->n_fixed; ++i) out.cols.push_back(cols->fixed[i]);
    for (uint32_t i = 0; i < cols->n_advice; ++i) out.cols.push_back(cols->advice[i]);
    for (uint32_t i = 0; i < cols->n_instance; ++i) out.cols.push_back(cols->instance[i]);
    for (uint32_t i = 0; i < g->n_rotations; ++i)
        if (!offset_within_halo(out.rot_off[i], size, shard)) { set_error("evaluate: rotation %d x %d exceeds the shard's halo of %u rows", g->rotations[i], rot_scale, shard.halo); return H2B_ERR_BAD_ARGUMENT; }
    // the values slice carries no halo: shifting its pointer back by `halo` rows makes the column indexing (row - base) land on it
    out.cols.push_back((const char*)d_values - (size_t)shard.halo * 32);
    for (const void* p : out.cols) if (!p) { set_error("evaluate: null column pointer"); return H2B_ERR_BAD_ARGUMENT; }
    const uint32_t values_col = (uint32_t)out.cols.size() - 1;

    const uint32_t n = g->n_calculations;
    out.ops.clear();
    out.n_slots = 0;
    if (n == 0 && n_roots == 0) return H2B_OK;

    // 1. resolve operands: intermediates become references to the calculation that defined them, Stores are forwarded
    std::vector<int32_t> cur_def(g->n_intermediates, -1);
    std::vector<Ref> alias(n);                       // for a Store: what it stands for
    std::vector<uint32_t> first(n + 1, 0);           // operand list of calculation c: refs[first[c] .. first[c+1])
    std::vector<Ref> refs;
    bool bad = false;
    auto resolve = [&](const h2b_value_source& s, uint32_t c) -> Ref {
        Ref r;
        auto column = [&](uint32_t base, uint32_t count) {
            if (s.index >= count || s.rotation >= g->n_rotations) { set_error("evaluate: calculation %u: column %u / rotation %u out of range", c, s.index, s.rotation); bad = true; return; }
            r.enc = OPK_COL | ((base + s.index) << 10) | s.rotation;
        };
        switch (s.kind) {
            case H2B_VS_CONSTANT:
                if (s.index >= nc) { set_error("evaluate: calculation %u: constant %u out of range", c, s.index); bad = true; }
                r.enc = OPK_CONST | s.index;
                break;
            case H2B_VS_INTERMEDIATE:
                if (s.index >= g->n_intermediates || cur_def[s.index] < 0) {
                    set_error("evaluate: calculation %u reads intermediate %u before it is written", c, s.index);
                    bad = true;
                } else {
                    const int32_t d = cur_def[s.index];
                    r = g->calculations[d].op == H2B_CALC_STORE ? alias[d] : Ref{d, 0};
                }
                break;
            case H2B_VS_FIXED: column(0, cols->n_fixed); break;
            case H2B_VS_ADVICE: column(cols->n_fixed, cols->n_advice); break;
            case H2B_VS_INSTANCE: column(cols->n_fixed + cols->n_advice, cols->n_instance); break;
            case H2B_VS_CHALLENGE:
                if (s.index >= nch) { set_error("evaluate: calculation %u: challenge %u out of range", c, s.index); bad = true; }
                r.enc = OPK_CONST | (nc + s.index);
                break;
            case H2B_VS_BETA: r.enc = OPK_CONST | out.c_beta; break;
            case H2B_VS_GAMMA: r.enc = OPK_CONST | out.c_gamma; break;
            case H2B_VS_THETA: r.enc = OPK_CONST | out.c_theta; break;
            case H2B_VS_Y: r.enc = OPK_CONST | out.c_y; break;
            case H2B_VS_PREVIOUS_VALUE:
                r.enc = previous_is_zero ? (OPK_CONST | out.c_zero) : (OPK_COL | (values_col << 10) | g->n_rotations);
                break;
            default: set_error("evaluate: calculation %u: unknown value source kind %u", c, s.kind); bad = true;
        }
        return r;
    };
    for (uint32_t c = 0; c < n; ++c) {
        const h2b_calculation& k = g->calculations[c];
        first[c] = (uint32_t)refs.size();
        if (k.op > H2B_CALC_STORE) { set_error("evaluate: calculation %u: unknown op %u", c, k.op); return H2B_ERR_BAD_ARGUMENT; }
        if (k.target >= g->n_intermediates) { set_error("evaluate: calculation %u: target %u out of range", c, k.target); return H2B_ERR_BAD_ARGUMENT; }
        refs.push_back(resolve(k.a, c));
        if (k.op == H2B_CALC_ADD || k.op == H2B_CALC_SUB || k.op == H2B_CALC_MUL || k.op == H2B_CALC_HORNER) refs.push_back(resolve(k.b, c));
        if (k.op == H2B_CALC_HORNER) {
            if ((uint64_t)k.parts_offset + k.parts_len > g->n_parts) { set_error("evaluate: calculation %u: Horner parts out of range", c); return H2B_ERR_BAD_ARGUMENT; }
            for (uint32_t j = 0; j < k.parts_len; ++j) refs.push_back(resolve(g->parts[k.parts_offset + j], c));
        }
        if (bad) return H2B_ERR_BAD_ARGUMENT;
        if (k.op == H2B_CALC_STORE) alias[c] = refs[first[c]];
        cur_def[k.target] = (int32_t)c;
    }
    first[n] = (uint32_t)refs.size();
    std::vector<Ref> root_refs(n_roots);
    for (uint32_t i = 0; i < n_roots; ++i) {
        root_refs[i] = resolve(roots[i], n);
        if (bad) { set_error("evaluate: root %u: out-of-range or unwritten value source", i); return H2B_ERR_BAD_ARGUMENT; }
    }

    // 2. the result is the last calculation's value, or every root; count the uses of every reachable calculation
    const uint32_t root = n ? n - 1 : 0;
    const bool root_is_store = n_roots == 0 && g->calculations[root].op == H2B_CALC_STORE;
    std::vector<uint32_t> uses(n, 0);
    std::vector<uint8_t> reach(n, 0);
    std::vector<uint32_t> stack;
    auto visit = [&](const Ref& r) {
        if (r.def < 0) return;
        ++uses[r.def];
        if (!reach[r.def]) { reach[r.def] = 1; stack.push_back((uint32_t)r.def); }
    };
    if (n_roots) for (const Ref& r : root_refs) visit(r);
    else if (root_is_store) visit(alias[root]);
    else { reach[root] = 1; stack.push_back(root); }
    while (!stack.empty()) {
        const uint32_t c = stack.back();
        stack.pop_back();
        for (uint32_t i = first[c]; i < first[c + 1]; ++i) visit(refs[i]);
    }

    // 3. depth-first emission with reference-counted slots
    std::vector<int32_t> slot_of(n, -1);
    std::vector<uint32_t> free_slots;
    uint32_t n_slots = 0;
    auto alloc_slot = [&]() -> uint32_t {
        if (!free_slots.empty()) { uint32_t s = free_slots.back(); free_slots.pop_back(); return s; }
        return n_slots++;
    };
    auto enc_of = [&](const Ref& r) -> uint32_t { return r.def < 0 ? r.enc : (OPK_SLOT | (uint32_t)slot_of[r.def]); };
    auto release = [&](const Ref& r) {
        if (r.def >= 0 && --uses[r.def] == 0) free_slots.push_back((uint32_t)slot_of[r.def]);
    };
    auto emit = [&](uint32_t code, uint32_t dst, uint32_t a, uint32_t b, uint32_t c) { out.ops.push_back(make_uint4(code | (dst << 8), a, b, c)); };
    struct Frame { uint32_t c, stage; int32_t acc; };       // stage = number of operands already ensured / consumed
    std::vector<Frame> frames;
    std::vector<uint8_t> done(n, 0);
    auto push = [&](uint32_t c) { frames.push_back(Frame{c, 0, -1}); };
    auto drain = [&]() {
        while (!frames.empty()) {
            Frame& f = frames.back();
            const uint32_t c = f.c;
            if (done[c]) { frames.pop_back(); continue; }
            const h2b_calculation& k = g->calculations[c];
            const uint32_t lo = first[c], cnt = first[c + 1] - lo;
            if (k.op != H2B_CALC_HORNER) {
                // make sure every operand exists, then emit
                bool pushed = false;
                for (uint32_t i = f.stage; i < cnt; ++i) {
                    const Ref& r = refs[lo + i];
                    if (r.def >= 0 && !done[r.def]) { f.stage = i; push((uint32_t)r.def); pushed = true; break; }
                }
                if (pushed) continue;
                const uint32_t a = enc_of(refs[lo]), b = cnt > 1 ? enc_of(refs[lo + 1]) : 0;
                for (uint32_t i = 0; i < cnt; ++i) release(refs[lo + i]);
                const uint32_t dst = alloc_slot();
                static const uint32_t code_of[8] = {MOP_ADD, MOP_SUB, MOP_MUL, MOP_SQR, MOP_DBL, MOP_NEG, MOP_FMA, MOP_MOV};
                emit(code_of[k.op], dst, a, b, 0);
                slot_of[c] = (int32_t)dst;
                done[c] = 1;
                frames.pop_back();
                continue;
            }
            // Horner(start = refs[lo], factor = refs[lo+1], parts = refs[lo+2 ..]): value = start; value = value * factor + part
            // stage 0/1: ensure start and factor; stage 2 + j: part j
            if (f.stage < 2) {
                const Ref& r = refs[lo + f.stage];
                ++f.stage;
                if (r.def >= 0 && !done[r.def]) { push((uint32_t)r.def); continue; }
                continue;
            }
            const uint32_t parts = cnt - 2;
            const uint32_t j = f.stage - 2;
            if (parts == 0) {
                const uint32_t a = enc_of(refs[lo]);
                release(refs[lo]); release(refs[lo + 1]);
                const uint32_t dst = alloc_slot();
                emit(MOP_MOV, dst, a, 0, 0);
                slot_of[c] = (int32_t)dst; done[c] = 1; frames.pop_back();
                continue;
            }
            const Ref& part = refs[lo + 2 + j];
            if (part.def >= 0 && !done[part.def]) { push((uint32_t)part.def); continue; }      // same stage again afterwards
            {
                const uint32_t acc = f.acc < 0 ? enc_of(refs[lo]) : (OPK_SLOT | (uint32_t)f.acc);
                const uint32_t fac = enc_of(refs[lo + 1]), pe = enc_of(part);
                if (f.acc < 0) release(refs[lo]); else free_slots.push_back((uint32_t)f.acc);
                release(part);
                if (j + 1 == parts) release(refs[lo + 1]);
                const uint32_t dst = alloc_slot();
                emit(MOP_FMA, dst, acc, fac, pe);
                f.acc = (int32_t)dst;
                ++f.stage;
                if (j + 1 == parts) { slot_of[c] = (int32_t)dst; done[c] = 1; frames.pop_back(); }
            }
        }
    };
    if (n_roots) {
        // each root right after what it needs, then its check; a root shared with a later one keeps its slot until then
        for (uint32_t i = 0; i < n_roots; ++i) {
            const Ref& r = root_refs[i];
            if (r.def >= 0 && !done[r.def]) { push((uint32_t)r.def); drain(); }
            emit(MOP_CHECK | MOP_NOSTORE, 0, enc_of(r), i, 0);
            release(r);
        }
    } else {
        if (root_is_store) { if (alias[root].def >= 0) push((uint32_t)alias[root].def); } else push(root);
        drain();
        if (root_is_store || out.ops.empty()) {
            const Ref& r = alias[root];
            emit(MOP_MOV, alloc_slot(), enc_of(r), 0, 0);
        }
    }
    if (n_slots > MAX_SLOTS) { set_error("evaluate: graph needs %u live values per row (limit %u)", n_slots, MAX_SLOTS); return H2B_ERR_BAD_ARGUMENT; }

    // 4. register forwarding: a slot operand produced by the previous micro-operation is read from registers; a result
    //    with no other reader is not stored (backward liveness over the slots)
    std::vector<uint4>& ops = out.ops;
    auto n_operands = [](uint32_t code) { return code == MOP_FMA ? 3u : (code == MOP_ADD || code == MOP_SUB || code == MOP_MUL) ? 2u : 1u; };
    for (size_t i = 1; i < ops.size(); ++i) {
        if ((ops[i - 1].x & 0x7f) == MOP_CHECK) continue;          // a check writes no slot
        const uint32_t prev_dst = OPK_SLOT | (ops[i - 1].x >> 8);
        uint32_t* e[3] = {&ops[i].y, &ops[i].z, &ops[i].w};
        for (uint32_t q = 0; q < n_operands(ops[i].x & 0x7f); ++q) if (*e[q] == prev_dst) *e[q] = OPK_PREV;
    }
    std::vector<uint8_t> live(n_slots ? n_slots : 1, 0);
    for (size_t i = ops.size(); i-- > 0;) {
        const uint32_t dst = ops[i].x >> 8;
        if ((ops[i].x & 0x7f) != MOP_CHECK) {
            if (!live[dst]) ops[i].x |= MOP_NOSTORE;
            live[dst] = 0;
        }
        const uint32_t e[3] = {ops[i].y, ops[i].z, ops[i].w};
        for (uint32_t q = 0; q < n_operands(ops[i].x & 0x7f); ++q) if ((e[q] & OPK_MASK) == OPK_SLOT) live[e[q] & ~OPK_MASK] = 1;
    }
    out.n_slots = n_slots;
    return H2B_OK;
}


struct EvalScratch {
    ProgramBuf ring[4];
    unsigned next = 0;
};

static size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

// resident CTAs (of 128 threads) per SM for the grid-stride row kernels; H2B_EVAL_CTAS_PER_SM overrides (tuning)
// (measured at 2^22 rows, profiles/r01_evaluate_h.jsonl: the 48-register interpreter gains 8 % from 16 over 8, the 128-register
// permutation kernel is best at 8)
static uint32_t eval_ctas_per_sm(uint32_t dflt) {
    static const int forced = [] {
        const char* e = getenv("H2B_EVAL_CTAS_PER_SM");
        const int x = e ? atoi(e) : 0;
        return x >= 1 && x <= 32 ? x : 0;
    }();
    return forced ? (uint32_t)forced : dflt;
}

int upload_program(DeviceCtx& ctx, const Compiled& c, uint32_t size, const Shard& shard, cudaStream_t stream, EvalProgram& dev, ProgramBuf** used) {
    if (!ctx.eval) ctx.eval = new EvalScratch();
    ProgramBuf& pb = ctx.eval->ring[ctx.eval->next++ & 3];
    const size_t o_ops = 0, o_consts = align16(o_ops + c.ops.size() * 16), o_rot = align16(o_consts + c.consts.size() * 8),
                 o_cols = align16(o_rot + c.rot_off.size() * 4), total = align16(o_cols + c.cols.size() * sizeof(void*));
    std::vector<unsigned char> host(total, 0);
    if (!c.ops.empty()) memcpy(host.data() + o_ops, c.ops.data(), c.ops.size() * 16);
    memcpy(host.data() + o_consts, c.consts.data(), c.consts.size() * 8);
    memcpy(host.data() + o_rot, c.rot_off.data(), c.rot_off.size() * 4);
    memcpy(host.data() + o_cols, c.cols.data(), c.cols.size() * sizeof(void*));
    if (pb.done) H2B_CUDA(cudaStreamWaitEvent(stream, pb.done, 0));     // the previous user of this ring slot
    else H2B_CUDA(cudaEventCreateWithFlags(&pb.done, cudaEventDisableTiming));
    H2B_TRY(pb.buf.reserve(total));
    // pageable source: the runtime stages it before returning, so `host` may die at the end of this function
    H2B_CUDA(cudaMemcpyAsync(pb.buf.p, host.data(), total, cudaMemcpyHostToDevice, stream));
    unsigned char* d = (unsigned char*)pb.buf.p;
    dev.ops = (const uint4*)(d + o_ops);
    dev.consts = (const uint4*)(d + o_consts);
    dev.rot_off = (const uint32_t*)(d + o_rot);
    dev.cols = (const void* const*)(d + o_cols);
    dev.n_ops = (uint32_t)c.ops.size();
    dev.size = size;
    dev.row0 = shard.row0; dev.rows = shard.rows; dev.base = shard.base;
    *used = &pb;
    return H2B_OK;
}

template <int MODE>
static int launch_graph(DeviceCtx& ctx, const EvalProgram& p, uint32_t n_slots, void* d_values, const LookupTerms& lk, cudaStream_t stream) {
    const uint32_t want = (p.rows + 127) / 128, cap = (uint32_t)ctx.sm_count * eval_ctas_per_sm(16);
    const uint32_t grid = want < cap ? want : cap;
    if (n_slots <= 8) H2B_LAUNCH((evaluate_graph_kernel<8, MODE>), grid, 128, 0, stream, p, (uint4*)d_values, lk);
    else if (n_slots <= 16) H2B_LAUNCH((evaluate_graph_kernel<16, MODE>), grid, 128, 0, stream, p, (uint4*)d_values, lk);
    else if (n_slots <= 32) H2B_LAUNCH((evaluate_graph_kernel<32, MODE>), grid, 128, 0, stream, p, (uint4*)d_values, lk);
    else H2B_LAUNCH((evaluate_graph_kernel<64, MODE>), grid, 128, 0, stream, p, (uint4*)d_values, lk);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

int evaluate_graph_run(DeviceCtx& ctx, const h2b_graph* g, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                       const h2b_eval_shard* sh, cudaStream_t stream) {
    if (!d_values) { set_error("evaluate_graph: null values"); return H2B_ERR_BAD_ARGUMENT; }
    if (size == 0 || size > (1u << 30)) { set_error("evaluate: size must be in [1, 2^30]"); return H2B_ERR_BAD_ARGUMENT; }
    Shard shard;
    H2B_TRY(make_shard(sh, size, shard));
    Compiled c;
    H2B_TRY(compile_graph(g, cols, d_values, size, rot_scale, false, shard, nullptr, 0, c));
    t_last_slots = c.n_slots;
    t_last_ops = (uint32_t)c.ops.size();
    if (c.ops.empty()) {        // no calculations: upstream returns zero for every row
        H2B_CUDA(cudaMemsetAsync(d_values, 0, (size_t)shard.rows * 32, stream));
        return H2B_OK;
    }
    EvalProgram p;
    ProgramBuf* pb = nullptr;
    H2B_TRY(upload_program(ctx, c, size, shard, stream, p, &pb));
    LookupTerms lk;
    memset(&lk, 0, sizeof(lk));
    H2B_TRY(launch_graph<0>(ctx, p, c.n_slots, d_values, lk, stream));
    H2B_CUDA(cudaEventRecord(pb->done, stream));
    return H2B_OK;
}

int evaluate_h_lookup_run(DeviceCtx& ctx, const h2b_graph* g, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                          const void* d_product, const void* d_permuted_input, const void* d_permuted_table, const void* d_l0, const void* d_l_last,
                          const void* d_l_active_row, const h2b_eval_shard* sh, cudaStream_t stream) {
    if (!d_values || !d_product || !d_permuted_input || !d_permuted_table || !d_l0 || !d_l_last || !d_l_active_row) {
        set_error("evaluate_h_lookup: null pointer");
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (size == 0 || size > (1u << 30)) { set_error("evaluate: size must be in [1, 2^30]"); return H2B_ERR_BAD_ARGUMENT; }
    Shard shard;
    H2B_TRY(make_shard(sh, size, shard));
    if (!offset_within_halo(rem_euclid_u32((int64_t)rot_scale, size), size, shard)) { set_error("evaluate_h_lookup: rot_scale exceeds the shard's halo"); return H2B_ERR_BAD_ARGUMENT; }
    Compiled c;
    H2B_TRY(compile_graph(g, cols, d_values, size, rot_scale, true, shard, nullptr, 0, c));
    if (c.ops.empty()) c.ops.push_back(make_uint4(MOP_MOV | MOP_NOSTORE, OPK_CONST | c.c_zero, 0, 0));      // table_value = 0
    t_last_slots = c.n_slots;
    t_last_ops = (uint32_t)c.ops.size();
    EvalProgram p;
    ProgramBuf* pb = nullptr;
    H2B_TRY(upload_program(ctx, c, size, shard, stream, p, &pb));
    LookupTerms lk;
    lk.product = (const uint4*)d_product; lk.permuted_input = (const uint4*)d_permuted_input; lk.permuted_table = (const uint4*)d_permuted_table;
    lk.l0 = (const uint4*)d_l0; lk.l_last = (const uint4*)d_l_last; lk.l_active_row = (const uint4*)d_l_active_row;
    lk.off_next = rem_euclid_u32((int64_t)rot_scale, size);
    lk.off_prev = rem_euclid_u32(-(int64_t)rot_scale, size);
    lk.beta = c.c_beta; lk.gamma = c.c_gamma; lk.y = c.c_y;
    H2B_TRY(launch_graph<1>(ctx, p, c.n_slots, d_values, lk, stream));
    H2B_CUDA(cudaEventRecord(pb->done, stream));
    return H2B_OK;
}

void evaluate_graph_last_info(uint32_t* slots, uint32_t* micro_ops) {
    if (slots) *slots = t_last_slots;
    if (micro_ops) *micro_ops = t_last_ops;
}

// ---- permutation argument terms --------------------------------------------------------------------------------------
struct PermParams {
    const void* const* product;     // n_sets
    const void* const* columns;     // n_columns
    const void* const* cosets;      // n_columns
    const uint4 *l0, *l_last, *l_active_row;
    uint32_t n_sets, n_columns, chunk_len, size, off_next, off_last, row0, rows, base;
    Fr beta, gamma, y, delta, zeta, omega;
};

__global__ void __launch_bounds__(128) evaluate_h_permutation_kernel(PermParams p, uint4* __restrict__ values) {
    const uint32_t stride = gridDim.x * blockDim.x, t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.rows) return;
    Fr beta_term = fp_pow_u32<FR>(p.omega, p.row0 + t);         // extended_omega^idx
    const Fr omega_step = fp_pow_u32<FR>(p.omega, stride);
    const Fr delta_start = fp_mul(p.beta, p.zeta);
    const uint4* z_first = (const uint4*)p.product[0];
    const uint4* z_last = (const uint4*)p.product[p.n_sets - 1];
    for (uint32_t i = t; i < p.rows; i += stride) {
        const uint32_t idx = p.row0 + i, li = shard_local(idx, p.base, p.size);
        uint32_t r_next = idx + p.off_next, r_last = idx + p.off_last;
        if (r_next >= p.size) r_next -= p.size;
        if (r_last >= p.size) r_last -= p.size;
        r_next = shard_local(r_next, p.base, p.size);
        r_last = shard_local(r_last, p.base, p.size);
        const Fr l0 = fp_load<FR>(p.l0 + 2 * (size_t)li), l_last = fp_load<FR>(p.l_last + 2 * (size_t)li);
        const Fr l_active = fp_load<FR>(p.l_active_row + 2 * (size_t)li);
        Fr v = fp_load<FR>(values + 2 * (size_t)i);
        // l_0(X) * (1 - z_0(X)) = 0
        v = fp_add(fp_mul(v, p.y), fp_mul(fp_sub(fp_one<FR>(), fp_load<FR>(z_first + 2 * (size_t)li)), l0));
        // l_last(X) * (z_l(X)^2 - z_l(X)) = 0
        {
            const Fr z = fp_load<FR>(z_last + 2 * (size_t)li);
            v = fp_add(fp_mul(v, p.y), fp_mul(fp_sub(fp_sqr(z), z), l_last));
        }
        // l_0(X) * (z_i(X) - z_{i-1}(w^(last) X)) = 0
        for (uint32_t s = 1; s < p.n_sets; ++s) {
            const Fr zi = fp_load<FR>((const uint4*)p.product[s] + 2 * (size_t)li);
            const Fr zp = fp_load<FR>((const uint4*)p.product[s - 1] + 2 * (size_t)r_last);
            v = fp_add(fp_mul(v, p.y), fp_mul(fp_sub(zi, zp), l0));
        }
        // (1 - (l_last + l_blind)) * (z_i(wX) prod (p + beta s_j + gamma) - z_i(X) prod (p + delta^j beta X + gamma)) = 0
        Fr current_delta = fp_mul(delta_start, beta_term);
        for (uint32_t s = 0, c0 = 0; s < p.n_sets && c0 < p.n_columns; ++s, c0 += p.chunk_len) {
            const uint32_t c1 = c0 + p.chunk_len < p.n_columns ? c0 + p.chunk_len : p.n_columns;
            const uint4* z = (const uint4*)p.product[s];
            Fr left = fp_load<FR>(z + 2 * (size_t)r_next), right = fp_load<FR>(z + 2 * (size_t)li);
            for (uint32_t c = c0; c < c1; ++c) {
                const Fr val = fp_load<FR>((const uint4*)p.columns[c] + 2 * (size_t)li);
                const Fr perm = fp_load<FR>((const uint4*)p.cosets[c] + 2 * (size_t)li);
                left = fp_mul(left, fp_add(fp_add(val, fp_mul(p.beta, perm)), p.gamma));
                right = fp_mul(right, fp_add(fp_add(val, current_delta), p.gamma));
                current_delta = fp_mul(current_delta, p.delta);
            }
            v = fp_add(fp_mul(v, p.y), fp_mul(fp_sub(left, right), l_active));
        }
        fp_store<FR>(values + 2 * (size_t)i, v);
        beta_term = fp_mul(beta_term, omega_step);
    }
}

static void load_fr(Fr& dst, const uint64_t* w) { memcpy(dst.l, w, 32); }

int evaluate_h_permutation_run(DeviceCtx& ctx, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                               const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len, int32_t last_rotation,
                               const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t* beta, const uint64_t* gamma,
                               const uint64_t* y, const uint64_t* delta, const uint64_t* zeta, const uint64_t* extended_omega, const h2b_eval_shard* sh,
                               cudaStream_t stream) {
    if (n_sets == 0) return H2B_OK;                         // upstream: `if !sets.is_empty()`
    if (!d_values || !d_product_cosets || (n_columns && (!d_columns || !d_perm_cosets)) || !d_l0 || !d_l_last || !d_l_active_row || !beta || !gamma || !y ||
        !delta || !zeta || !extended_omega) {
        set_error("evaluate_h_permutation: null pointer");
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (size == 0 || size > (1u << 30)) { set_error("evaluate_h_permutation: size must be in [1, 2^30]"); return H2B_ERR_BAD_ARGUMENT; }
    if (chunk_len == 0) { set_error("evaluate_h_permutation: chunk_len must be positive"); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < n_sets; ++i) if (!d_product_cosets[i]) { set_error("evaluate_h_permutation: null product coset"); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < n_columns; ++i) if (!d_columns[i] || !d_perm_cosets[i]) { set_error("evaluate_h_permutation: null column"); return H2B_ERR_BAD_ARGUMENT; }
    if (!ctx.eval) ctx.eval = new EvalScratch();
    ProgramBuf& pb = ctx.eval->ring[ctx.eval->next++ & 3];
    const size_t n_ptrs = (size_t)n_sets + 2 * (size_t)n_columns;
    const size_t total = align16(n_ptrs * sizeof(void*));
    std::vector<unsigned char> host(total, 0);
    const void** hp = (const void**)host.data();
    for (uint32_t i = 0; i < n_sets; ++i) hp[i] = d_product_cosets[i];
    for (uint32_t i = 0; i < n_columns; ++i) { hp[n_sets + i] = d_columns[i]; hp[n_sets + n_columns + i] = d_perm_cosets[i]; }
    if (pb.done) H2B_CUDA(cudaStreamWaitEvent(stream, pb.done, 0));
    else H2B_CUDA(cudaEventCreateWithFlags(&pb.done, cudaEventDisableTiming));
    H2B_TRY(pb.buf.reserve(total));
    H2B_CUDA(cudaMemcpyAsync(pb.buf.p, host.data(), total, cudaMemcpyHostToDevice, stream));
    unsigned char* d = (unsigned char*)pb.buf.p;
    PermParams p;
    p.product = (const void* const*)d;
    p.columns = (const void* const*)d + n_sets;
    p.cosets = (const void* const*)d + n_sets + n_columns;
    p.l0 = (const uint4*)d_l0; p.l_last = (const uint4*)d_l_last; p.l_active_row = (const uint4*)d_l_active_row;
    p.n_sets = n_sets; p.n_columns = n_columns; p.chunk_len = chunk_len; p.size = size;
    p.off_next = rem_euclid_u32((int64_t)rot_scale, size);
    p.off_last = rem_euclid_u32((int64_t)last_rotation * rot_scale, size);
    Shard shard;
    H2B_TRY(make_shard(sh, size, shard));
    if (!offset_within_halo(p.off_next, size, shard) || !offset_within_halo(p.off_last, size, shard)) {
        set_error("evaluate_h_permutation: rot_scale / last_rotation exceed the shard's halo of %u rows", shard.halo);
        return H2B_ERR_BAD_ARGUMENT;
    }
    p.row0 = shard.row0; p.rows = shard.rows; p.base = shard.base;
    load_fr(p.beta, beta); load_fr(p.gamma, gamma); load_fr(p.y, y); load_fr(p.delta, delta); load_fr(p.zeta, zeta); load_fr(p.omega, extended_omega);
    const uint32_t want = (shard.rows + 127) / 128, cap = (uint32_t)ctx.sm_count * eval_ctas_per_sm(8);
    H2B_LAUNCH(evaluate_h_permutation_kernel, want < cap ? want : cap, 128, 0, stream, p, (uint4*)d_values);
    H2B_CUDA(cudaGetLastError());
    H2B_CUDA(cudaEventRecord(pb.done, stream));
    return H2B_OK;
}

void evaluate_release(DeviceCtx& ctx) {
    if (!ctx.eval) return;
    for (ProgramBuf& pb : ctx.eval->ring) {
        pb.buf.release();
        if (pb.done) cudaEventDestroy(pb.done);
    }
    delete ctx.eval;
    ctx.eval = nullptr;
}

}  // namespace h2b
