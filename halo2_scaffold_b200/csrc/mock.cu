// MockProver::verify on the device: [UP] halo2_proofs/src/dev.rs, the gate, lookup and permutation loops of verify_par.
// Upstream walks every row on the CPU with an enum per cell (CellValue::{Unassigned, Assigned, Poison}) and per value
// (Value::{Real, Poison}).  Here
//   * the gates are one GraphEvaluator compiled with a root per polynomial (evaluate.cuh): the row interpreter of the quotient
//     evaluation carries one poison bit per live value (a 64-bit mask for the 64 slots) and a MOP_CHECK classifies each root.
//     Only a product with a poisoned operand tests the other operand for zero (Poison * Real(0) = Real(0)); every other micro-op
//     ORs the bits, so the unpoisoned path does the arithmetic of evaluate.cu.  A thread counts the failures of each gate on its
//     row; an exclusive scan of the (gate, row) counts places every record, so they come out in upstream's (gate, row, poly) order
//     without atomics;
//   * a lookup evaluates its m input and m table roots over the usable rows into canonical 256-bit keys (Poison = 2^255, above
//     every canonical value, so tuples order as Value's derived Ord does).  The table is sorted -- the keys themselves through
//     lookup.cu's bitonic sort when m = 1, row indices compared as whole tuples when m > 1 -- and every input tuple is
//     binary-searched: exact membership, no compression;
//   * a copy constraint is one thread per (column, row) that gathers the mapped cell and compares CellValues.
// Unassigned fixed / advice cells are zeroed on the device before the gates run (they read Real(0)); the bitmaps stay for the
// copy constraints, where Unassigned != Assigned(0).
#include <memory>

#include "evaluate.cuh"
#include "keys.cuh"

namespace h2b {

static const uint32_t MOCK_BLOCK = 128;

// what a program's column operands mean for poison: columns [adv_lo, adv_hi) of its table are advice, Poison from row `usable`
struct MockRows { uint32_t usable, adv_lo, adv_hi; };

__device__ __forceinline__ Fr mock_fetch(const EvalProgram& p, const MockRows& mr, uint32_t enc, uint32_t idx, const Fr* slots, uint64_t slot_poison,
                                         const Fr& prev, bool prev_poison, bool& poison) {
    const uint32_t kind = enc & OPK_MASK, v = enc & ~OPK_MASK;
    if (kind == OPK_PREV) { poison = prev_poison; return prev; }
    if (kind == OPK_SLOT) { poison = (slot_poison >> v) & 1; return slots[v]; }
    poison = false;
    if (kind == OPK_CONST) return fp_load<FR>(p.consts + 2 * (size_t)v);
    const uint32_t row = eval_operand_row(p, v, idx), c = v >> 10;
    poison = c >= mr.adv_lo && c < mr.adv_hi && row >= mr.usable;
    const uint4* col = reinterpret_cast<const uint4*>(__ldg(reinterpret_cast<const unsigned long long*>(p.cols) + c));
    return fp_load<FR>(col + 2 * (size_t)row);
}

__device__ __forceinline__ void mock_key_store(uint4* keys, size_t i, const Fr& v, bool poison) {
    if (poison) {
        keys[2 * i] = make_uint4(0, 0, 0, 0);
        keys[2 * i + 1] = make_uint4(0, 0, 0, 0x80000000u);
    } else {
        fp_store<FR>(keys + 2 * i, fp_from_mont(v));
    }
}

// MODE 0 (gates): status[root * n + row] = 0 Real(0), 1 Real(!= 0), 2 Poison; counts[group * n + row] = the failures of the root group
// (CHECK's w) on the row.  MODE 1 (lookups): root z's canonical key at keys[z * key_stride + row].
struct MockOut {
    uint8_t* status;
    uint32_t* counts;
    uint4* keys;
    size_t key_stride;
};

template <int S, int MODE>
__global__ void __launch_bounds__(MOCK_BLOCK, 1) mock_graph_kernel(EvalProgram p, MockRows mr, MockOut o) {
    Fr slots[S];
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < p.rows; idx += stride) {
        Fr r = fp_zero<FR>();
        bool rp = false;
        uint64_t sp = 0;
        uint32_t group = ~0u, fails = 0;
#pragma unroll 1
        for (uint32_t i = 0; i < p.n_ops; ++i) {
            const uint4 op = __ldg(p.ops + i);
            const uint32_t code = op.x & 0x7f;
            bool pa, pb;
            const Fr a = mock_fetch(p, mr, op.y, idx, slots, sp, r, rp, pa);
            if (code == MOP_CHECK) {
                if (MODE == 0) {
                    const uint8_t st = pa ? 2 : fp_is_zero(a) ? 0 : 1;
                    o.status[(size_t)op.z * p.size + idx] = st;
                    if (op.w != group) {
                        if (group != ~0u) o.counts[(size_t)group * p.size + idx] = fails;
                        group = op.w;
                        fails = 0;
                    }
                    fails += st != 0;
                } else {
                    mock_key_store(o.keys + 2 * o.key_stride * op.z, idx, a, pa);
                }
                continue;
            }
            Fr out;
            bool po = pa;
            if (code == MOP_MUL || code == MOP_FMA) {
                const Fr b = mock_fetch(p, mr, op.z, idx, slots, sp, r, rp, pb);
                out = fp_mul(a, b);
                po = pa || pb;
                // Value's Mul: Poison times Real(0) is Real(0)
                if (po && ((!pa && fp_is_zero(a)) || (!pb && fp_is_zero(b)))) { out = fp_zero<FR>(); po = false; }
                if (code == MOP_FMA) {
                    bool pc;
                    out = fp_add(out, mock_fetch(p, mr, op.w, idx, slots, sp, r, rp, pc));
                    po = po || pc;
                }
            } else if (code == MOP_ADD || code == MOP_SUB) {
                const Fr b = mock_fetch(p, mr, op.z, idx, slots, sp, r, rp, pb);
                out = code == MOP_ADD ? fp_add(a, b) : fp_sub(a, b);
                po = pa || pb;
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
            rp = po;
            if (!(op.x & MOP_NOSTORE)) {
                const uint32_t d = (op.x >> 8) & (S - 1);
                slots[d] = out;
                sp = po ? sp | (1ull << d) : sp & ~(1ull << d);
            }
        }
        if (MODE == 0 && group != ~0u) o.counts[(size_t)group * p.size + idx] = fails;
    }
}

// Unassigned cells read Real(0): zero the value words whose bitmap bit is clear
__global__ void __launch_bounds__(256) mock_mask_kernel(uint4* __restrict__ col, const uint8_t* __restrict__ bits, uint32_t n) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n || ((bits[r >> 3] >> (r & 7)) & 1)) return;
    col[2 * (size_t)r] = make_uint4(0, 0, 0, 0);
    col[2 * (size_t)r + 1] = make_uint4(0, 0, 0, 0);
}

// ---- lookups ----------------------------------------------------------------------------------------------------------
static const uint32_t NO_ROW = ~0u;      // padding of the index sort: above every tuple

// tuple of table row a vs tuple of row b (m keys, `stride` keys apart): < 0, 0, > 0
__device__ __forceinline__ int tuple_cmp(const uint4* ka, size_t a, const uint4* kb, size_t b, uint32_t m, size_t stride) {
    for (uint32_t j = 0; j < m; ++j) {
        const Key x = key_load(ka + 2 * stride * j, a), y = key_load(kb + 2 * stride * j, b);
        if (!key_eq(x, y)) return key_less(x, y) ? -1 : 1;
    }
    return 0;
}
__device__ __forceinline__ bool row_less(const uint4* t, uint32_t a, uint32_t b, uint32_t m, size_t stride) {
    if (a == NO_ROW) return false;
    if (b == NO_ROW) return true;
    return tuple_cmp(t, a, t, b, m, stride) < 0;
}

__global__ void __launch_bounds__(256) mock_index_init_kernel(uint32_t* idx, uint32_t usable, uint32_t padded) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < padded) idx[i] = i < usable ? i : NO_ROW;
}
// one compare-exchange pass of a bitonic network over row indices, ordered by their table tuples
__global__ void __launch_bounds__(256) mock_index_bitonic_kernel(uint32_t* idx, uint32_t half, uint32_t j, uint32_t k, const uint4* __restrict__ table,
                                                               uint32_t m, size_t stride) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= half) return;
    const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), q = i | j;
    const bool up = (i & k) == 0;
    const uint32_t a = idx[i], b = idx[q];
    if (row_less(table, b, a, m, stride) == up) { idx[i] = b; idx[q] = a; }
}

// flags[r] = 1 when the input tuple of row r is neither fill_row nor in the table.  m = 1: `table` is sorted; otherwise `order`
// lists the table rows by tuple
__global__ void __launch_bounds__(256) mock_lookup_check_kernel(const uint4* __restrict__ input, const uint4* __restrict__ table, const uint32_t* __restrict__ order,
                                                              const uint4* __restrict__ fill, uint32_t usable, uint32_t m, size_t stride,
                                                              uint32_t* __restrict__ flags) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= usable) return;
    bool is_fill = true;
    for (uint32_t j = 0; j < m && is_fill; ++j) is_fill = key_eq(key_load(input + 2 * stride * j, r), key_load(fill, j));
    if (is_fill) { flags[r] = 0; return; }
    uint32_t lo = 0, hi = usable;                    // lower bound of the input tuple among the sorted table tuples
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        const int c = m == 1 ? (key_less(key_load(table, mid), key_load(input, r)) ? -1 : 0) : tuple_cmp(table, order[mid], input, r, m, stride);
        if (c < 0) lo = mid + 1; else hi = mid;
    }
    bool found = false;
    if (lo < usable) found = m == 1 ? key_eq(key_load(table, lo), key_load(input, r)) : tuple_cmp(table, order[lo], input, r, m, stride) == 0;
    flags[r] = found ? 0u : 1u;
}

// ---- copy constraints -------------------------------------------------------------------------------------------------
struct MockPermCols {
    const uint4* const* values;      // per permutation column
    const uint8_t* const* bits;      // assigned bitmaps (null for instance columns)
    const uint64_t* const* mapping;  // n x (column, row)
    const uint32_t* is_advice;
    uint32_t n_columns, n, usable;
};

// CellValue of (c, r): state 0 Unassigned, 1 Assigned(value), 2 Poison(r)
__device__ __forceinline__ uint32_t mock_cell(const MockPermCols& pc, uint32_t c, uint32_t r, Fr& v) {
    if (pc.is_advice[c] && r >= pc.usable) return 2;
    const uint8_t* b = pc.bits[c];
    if (b && !((b[r >> 3] >> (r & 7)) & 1)) return 0;
    v = fp_load<FR>(pc.values[c] + 2 * (size_t)r);
    return 1;
}
__global__ void __launch_bounds__(256) mock_permutation_kernel(MockPermCols pc, uint32_t* __restrict__ flags, uint32_t* __restrict__ bad_entry) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)pc.n_columns * pc.n) return;
    const uint32_t c = (uint32_t)(t / pc.n), r = (uint32_t)(t % pc.n);
    const uint64_t mc = pc.mapping[c][2 * (size_t)r], mr = pc.mapping[c][2 * (size_t)r + 1];
    if (mc >= pc.n_columns || mr >= pc.n) { atomicMax(bad_entry, (uint32_t)t + 1); flags[t] = 0; return; }
    Fr a = fp_zero<FR>(), b = fp_zero<FR>();
    const uint32_t sa = mock_cell(pc, c, r, a), sb = mock_cell(pc, (uint32_t)mc, (uint32_t)mr, b);
    const bool equal = sa == sb && (sa == 0 || (sa == 1 && fp_eq(a, b)) || (sa == 2 && r == (uint32_t)mr));
    flags[t] = equal ? 0u : 1u;
}

// ---- records ----------------------------------------------------------------------------------------------------------
// one thread per (root group, row): the group's failing roots in root order at offsets[g n + row] + base
__global__ void __launch_bounds__(256) mock_gate_records_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets, const uint8_t* __restrict__ status,
                                                              const uint32_t* __restrict__ group_first, const uint32_t* __restrict__ group_gate,
                                                              const uint32_t* __restrict__ root_poly, uint32_t n_groups, uint32_t n, uint32_t cap,
                                                              h2b_mock_record* __restrict__ out) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)n_groups * n || counts[t] == 0) return;
    const uint32_t g = (uint32_t)(t / n), row = (uint32_t)(t % n);
    uint32_t at = offsets[t];
    for (uint32_t z = group_first[g]; z < group_first[g + 1] && at < cap; ++z) {
        const uint8_t st = status[(size_t)z * n + row];
        if (!st) continue;
        h2b_mock_record rec;
        rec.kind = st == 1 ? H2B_MOCK_CONSTRAINT_NOT_SATISFIED : H2B_MOCK_CONSTRAINT_POISONED;
        rec.index = group_gate[g]; rec.poly = root_poly[z]; rec.row = row;
        out[at++] = rec;
    }
}
// one thread per (index, row) of a flag array with `rows` rows per index: a record at base + offsets[t] when flagged
__global__ void __launch_bounds__(256) mock_flag_records_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ offsets, uint32_t count, uint32_t rows,
                                                              uint32_t kind, uint32_t base, uint32_t cap, h2b_mock_record* __restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count || !flags[t]) return;
    const uint32_t at = base + offsets[t];
    if (at >= cap) return;
    h2b_mock_record rec;
    rec.kind = kind; rec.index = t / rows; rec.poly = 0; rec.row = t % rows;
    out[at] = rec;
}

// ---- host ---------------------------------------------------------------------------------------------------------------
namespace {

// device allocations of one call, given back when it returns
struct CallMemory {
    std::vector<void*> held;
    ~CallMemory() {
        for (void* p : held) cudaFree(p);
        cudaGetLastError();
    }
    int get(void** out, size_t bytes, const char* what) {
        *out = nullptr;
        cudaError_t e = cudaMalloc(out, bytes ? bytes : 16);
        if (e != cudaSuccess) {
            cudaGetLastError();
            *out = nullptr;
            set_error("h2b_mock_verify: cudaMalloc(%zu) for %s failed: %s", bytes, what, cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? H2B_ERR_OOM : H2B_ERR_CUDA;
        }
        held.push_back(*out);
        return H2B_OK;
    }
    template <class T> int get(T** out, size_t count, const char* what) { return get((void**)out, count * sizeof(T), what); }
};

template <int MODE>
int mock_launch_graph(DeviceCtx& ctx, const EvalProgram& p, uint32_t n_slots, const MockRows& mr, const MockOut& o, cudaStream_t stream) {
    const uint32_t want = (p.rows + MOCK_BLOCK - 1) / MOCK_BLOCK, cap = (uint32_t)ctx.sm_count * 16;
    const uint32_t grid = want < cap ? want : cap;
    if (n_slots <= 8) H2B_LAUNCH((mock_graph_kernel<8, MODE>), grid, MOCK_BLOCK, 0, stream, p, mr, o);
    else if (n_slots <= 16) H2B_LAUNCH((mock_graph_kernel<16, MODE>), grid, MOCK_BLOCK, 0, stream, p, mr, o);
    else if (n_slots <= 32) H2B_LAUNCH((mock_graph_kernel<32, MODE>), grid, MOCK_BLOCK, 0, stream, p, mr, o);
    else H2B_LAUNCH((mock_graph_kernel<64, MODE>), grid, MOCK_BLOCK, 0, stream, p, mr, o);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

uint32_t blocks_of(size_t count, uint32_t block) { return (uint32_t)((count + block - 1) / block); }

}  // namespace

// compiles a graph of the circuit with its roots.  With d_cols null it only validates: a placeholder stands in for every column.
// The values column of the quotient evaluation is never read (no PREVIOUS_VALUE: it reads zero), so it is a placeholder too.
static int mock_compile(const h2b_mock_circuit* c, const h2b_graph* g, const h2b_value_source* roots, uint32_t n_roots, const void* const* d_cols,
                        Compiled& out) {
    static const uint64_t placeholder[4] = {0, 0, 0, 0};
    const uint32_t n = 1u << c->k, n_cols = c->n_fixed + c->n_advice + c->n_instance;
    std::vector<const void*> cols(n_cols + 1, (const void*)placeholder);
    for (uint32_t i = 0; i < n_cols && d_cols; ++i) cols[i] = d_cols[i];
    h2b_eval_columns ec;
    ec.fixed = cols.data(); ec.n_fixed = c->n_fixed;
    ec.advice = cols.data() + c->n_fixed; ec.n_advice = c->n_advice;
    ec.instance = cols.data() + c->n_fixed + c->n_advice; ec.n_instance = c->n_instance;
    ec.challenges = c->challenges; ec.n_challenges = c->n_challenges;
    ec.beta = ec.gamma = ec.theta = ec.y = placeholder;
    const Shard whole{0, n, 0, 0};
    return compile_graph(g, &ec, cols[n_cols], n, 1, true, whole, roots, n_roots, out);
}

int mock_verify_check(const h2b_mock_circuit* c) {
    Compiled tmp;
    std::vector<h2b_value_source> rs;
    for (uint32_t i = 0; i < c->n_roots; ++i) rs.push_back(c->roots[i].value);
    if (c->n_roots) H2B_TRY(mock_compile(c, c->gates, rs.data(), c->n_roots, nullptr, tmp));
    for (uint32_t l = 0; l < c->n_lookups; ++l) {
        const h2b_mock_lookup& lk = c->lookups[l];
        rs.assign(lk.inputs, lk.inputs + lk.m);
        rs.insert(rs.end(), lk.tables, lk.tables + lk.m);
        H2B_TRY(mock_compile(c, &lk.graph, rs.data(), 2 * lk.m, nullptr, tmp));
    }
    return H2B_OK;
}

int mock_verify_run(DeviceCtx& ctx, const h2b_mock_circuit* c, h2b_mock_record* records, uint64_t capacity, uint64_t* count) {
    const cudaStream_t st = ctx.stream;
    const uint32_t n = 1u << c->k, usable = n - (c->blinding_factors + 1);
    const uint32_t NF = c->n_fixed, NA = c->n_advice, NI = c->n_instance, NC = NF + NA + NI, P = c->n_permutation;
    const size_t bitmap_bytes = (n + 7) / 8;
    CallMemory mem;
    ctx.prof.mark(PROF_BEGIN, st);

    // columns: fixed | advice | instance, and the fixed / advice bitmaps
    std::vector<void*> d_cols(NC);
    std::vector<uint8_t*> d_bits(NF + NA);
    for (uint32_t i = 0; i < NC; ++i) {
        H2B_TRY(mem.get(&d_cols[i], (size_t)n * 32, "a column"));
        const uint64_t* src = i < NF ? c->fixed[i] : i < NF + NA ? c->advice[i - NF] : c->instance[i - NF - NA];
        H2B_TRY(host_upload(ctx, d_cols[i], src, (size_t)n * 32, st));
    }
    for (uint32_t i = 0; i < NF + NA; ++i) {
        H2B_TRY(mem.get(&d_bits[i], bitmap_bytes, "a bitmap"));
        H2B_TRY(host_upload(ctx, d_bits[i], i < NF ? c->fixed_assigned[i] : c->advice_assigned[i - NF], bitmap_bytes, st));
        H2B_LAUNCH(mock_mask_kernel, blocks_of(n, 256), 256, 0, st, (uint4*)d_cols[i], (const uint8_t*)d_bits[i], n);
    }
    std::vector<uint64_t*> d_map(P);
    for (uint32_t i = 0; i < P; ++i) {
        H2B_TRY(mem.get(&d_map[i], (size_t)n * 2, "a mapping column"));
        H2B_TRY(host_upload(ctx, d_map[i], c->mapping[i], (size_t)n * 16, st));
    }
    H2B_CUDA(cudaGetLastError());
    ctx.prof.mark(PROF_MOCK_UPLOAD, st);
    const MockRows mr{usable, NF, NF + NA};
    uint32_t* sums = nullptr;
    size_t max_scan = std::max<size_t>({(size_t)P * n, (size_t)c->n_lookups * usable, 1});

    // gates: root groups are the runs of roots of one gate
    uint32_t n_groups = 0;
    std::vector<uint32_t> group_first, group_gate, root_poly;
    for (uint32_t z = 0; z < c->n_roots; ++z) {
        if (z == 0 || c->roots[z].gate != c->roots[z - 1].gate) { group_first.push_back(z); group_gate.push_back(c->roots[z].gate); ++n_groups; }
        root_poly.push_back(c->roots[z].poly);
    }
    group_first.push_back(c->n_roots);
    max_scan = std::max(max_scan, (size_t)n_groups * n);
    H2B_TRY(mem.get(&sums, max_scan / SCAN_BLOCK + 2, "scan sums"));
    uint8_t* status = nullptr;
    uint32_t *counts = nullptr, *gate_off = nullptr;
    uint32_t totals[3] = {0, 0, 0};
    uint32_t* d_totals = nullptr;
    H2B_TRY(mem.get(&d_totals, 4, "totals"));
    H2B_CUDA(cudaMemsetAsync(d_totals, 0, 16, st));
    if (n_groups) {
        H2B_TRY(mem.get(&status, (size_t)c->n_roots * n, "gate status"));
        H2B_TRY(mem.get(&counts, (size_t)n_groups * n, "gate counts"));
        H2B_TRY(mem.get(&gate_off, (size_t)n_groups * n + 1, "gate offsets"));
        std::vector<h2b_value_source> rs;
        for (uint32_t z = 0; z < c->n_roots; ++z) rs.push_back(c->roots[z].value);
        Compiled cg;
        H2B_TRY(mock_compile(c, c->gates, rs.data(), c->n_roots, (const void* const*)d_cols.data(), cg));
        for (uint4& op : cg.ops) if ((op.x & 0x7f) == MOP_CHECK) op.w = (uint32_t)(std::upper_bound(group_first.begin(), group_first.end() - 1, op.z) - group_first.begin()) - 1;
        EvalProgram p;
        ProgramBuf* pb = nullptr;
        H2B_TRY(upload_program(ctx, cg, n, Shard{0, n, 0, 0}, st, p, &pb));
        H2B_TRY(mock_launch_graph<0>(ctx, p, cg.n_slots, mr, MockOut{status, counts, nullptr, 0}, st));
        H2B_CUDA(cudaEventRecord(pb->done, st));
        ctx.prof.mark(PROF_MOCK_GATES, st);
        H2B_TRY(u32_exclusive_scan(counts, n_groups * n, gate_off, nullptr, sums, st));
        H2B_CUDA(cudaMemcpyAsync(d_totals, gate_off + (size_t)n_groups * n, 4, cudaMemcpyDeviceToDevice, st));
    }

    // lookups, one after another through one key buffer
    uint32_t *lk_flags = nullptr, *lk_off = nullptr;
    if (c->n_lookups) {
        uint32_t m_max = 0;
        for (uint32_t l = 0; l < c->n_lookups; ++l) m_max = std::max(m_max, c->lookups[l].m);
        uint32_t padded = SORT_TILE;
        while (padded < usable) padded <<= 1;
        uint4 *keys = nullptr, *fill = nullptr;
        uint32_t* order = nullptr;
        H2B_TRY(mem.get(&keys, (size_t)2 * m_max * padded * 2, "lookup keys"));
        H2B_TRY(mem.get(&fill, (size_t)m_max * 2, "fill row"));
        H2B_TRY(mem.get(&order, padded, "table order"));
        H2B_TRY(mem.get(&lk_flags, (size_t)c->n_lookups * usable, "lookup flags"));
        H2B_TRY(mem.get(&lk_off, (size_t)c->n_lookups * usable + 1, "lookup offsets"));
        for (uint32_t l = 0; l < c->n_lookups; ++l) {
            const h2b_mock_lookup& lk = c->lookups[l];
            const uint32_t m = lk.m;
            std::vector<h2b_value_source> rs(lk.inputs, lk.inputs + m);
            rs.insert(rs.end(), lk.tables, lk.tables + m);
            Compiled cg;
            H2B_TRY(mock_compile(c, &lk.graph, rs.data(), 2 * m, (const void* const*)d_cols.data(), cg));
            EvalProgram p;
            ProgramBuf* pb = nullptr;
            H2B_TRY(upload_program(ctx, cg, n, Shard{0, n, 0, 0}, st, p, &pb));
            p.rows = usable;                        // input and table rows are the usable ones
            H2B_TRY(mock_launch_graph<1>(ctx, p, cg.n_slots, mr, MockOut{nullptr, nullptr, keys, padded}, st));
            H2B_CUDA(cudaEventRecord(pb->done, st));
            uint4* input = keys;
            uint4* table = keys + 2 * (size_t)padded * m;
            for (uint32_t j = 0; j < m; ++j)        // fill_row: the table tuple of the last usable row
                H2B_CUDA(cudaMemcpyAsync(fill + 2 * (size_t)j, table + 2 * ((size_t)padded * j + usable - 1), 32, cudaMemcpyDeviceToDevice, st));
            if (m == 1) {
                H2B_CUDA(cudaMemsetAsync(table + 2 * (size_t)usable, 0xff, (size_t)(padded - usable) * 32, st));
                H2B_TRY(bitonic_sort(table, padded, st));
            } else {
                H2B_LAUNCH(mock_index_init_kernel, blocks_of(padded, 256), 256, 0, st, order, usable, padded);
                for (uint32_t k = 2; k <= padded; k <<= 1)
                    for (uint32_t j = k >> 1; j > 0; j >>= 1)
                        H2B_LAUNCH(mock_index_bitonic_kernel, blocks_of(padded / 2, 256), 256, 0, st, order, padded / 2, j, k, (const uint4*)table, m,
                                   (size_t)padded);
            }
            H2B_LAUNCH(mock_lookup_check_kernel, blocks_of(usable, 256), 256, 0, st, (const uint4*)input, (const uint4*)table, (const uint32_t*)order,
                       (const uint4*)fill, usable, m, (size_t)padded, lk_flags + (size_t)l * usable);
            H2B_CUDA(cudaGetLastError());
        }
        ctx.prof.mark(PROF_MOCK_LOOKUPS, st);
        H2B_TRY(u32_exclusive_scan(lk_flags, c->n_lookups * usable, lk_off, nullptr, sums, st));
        H2B_CUDA(cudaMemcpyAsync(d_totals + 1, lk_off + (size_t)c->n_lookups * usable, 4, cudaMemcpyDeviceToDevice, st));
    }

    // copy constraints
    uint32_t *pm_flags = nullptr, *pm_off = nullptr;
    if (P) {
        std::vector<const void*> tab(3 * (size_t)P);
        std::vector<uint32_t> is_advice(P);
        for (uint32_t i = 0; i < P; ++i) {
            const h2b_mock_column& col = c->permutation[i];
            const uint32_t flat = col.kind == H2B_VS_FIXED ? col.index : col.kind == H2B_VS_ADVICE ? NF + col.index : NF + NA + col.index;
            tab[i] = d_cols[flat];
            tab[P + i] = col.kind == H2B_VS_INSTANCE ? nullptr : d_bits[flat];
            tab[2 * (size_t)P + i] = d_map[i];
            is_advice[i] = col.kind == H2B_VS_ADVICE;
        }
        void* d_tab = nullptr;
        uint32_t* d_adv = nullptr;
        H2B_TRY(mem.get(&d_tab, tab.size() * sizeof(void*), "permutation tables"));
        H2B_TRY(mem.get(&d_adv, P, "permutation kinds"));
        H2B_CUDA(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(void*), cudaMemcpyHostToDevice, st));
        H2B_CUDA(cudaMemcpyAsync(d_adv, is_advice.data(), (size_t)P * 4, cudaMemcpyHostToDevice, st));
        H2B_TRY(mem.get(&pm_flags, (size_t)P * n, "permutation flags"));
        H2B_TRY(mem.get(&pm_off, (size_t)P * n + 1, "permutation offsets"));
        MockPermCols pc;
        pc.values = (const uint4* const*)d_tab;
        pc.bits = (const uint8_t* const*)d_tab + P;
        pc.mapping = (const uint64_t* const*)d_tab + 2 * (size_t)P;
        pc.is_advice = d_adv;
        pc.n_columns = P; pc.n = n; pc.usable = usable;
        H2B_LAUNCH(mock_permutation_kernel, blocks_of((size_t)P * n, 256), 256, 0, st, pc, pm_flags, d_totals + 3);
        ctx.prof.mark(PROF_MOCK_PERMUTATION, st);
        H2B_TRY(u32_exclusive_scan(pm_flags, P * n, pm_off, nullptr, sums, st));
        H2B_CUDA(cudaMemcpyAsync(d_totals + 2, pm_off + (size_t)P * n, 4, cudaMemcpyDeviceToDevice, st));
    }
    uint32_t got[4];
    H2B_CUDA(cudaMemcpyAsync(got, d_totals, 16, cudaMemcpyDeviceToHost, st));
    H2B_CUDA(cudaStreamSynchronize(st));
    if (got[3]) {
        const uint32_t t = got[3] - 1;
        set_error("h2b_mock_verify: mapping entry (column %u, row %u) points outside the permutation's %u columns and %u rows", t / n, t % n, P, n);
        return H2B_ERR_BAD_ARGUMENT;
    }
    memcpy(totals, got, 12);
    const uint64_t total = (uint64_t)totals[0] + totals[1] + totals[2];
    const uint32_t cap = (uint32_t)std::min<uint64_t>(capacity, total);
    if (cap) {
        h2b_mock_record* d_rec = nullptr;
        H2B_TRY(mem.get(&d_rec, cap, "records"));
        if (n_groups && totals[0]) {
            uint32_t* d_meta = nullptr;
            std::vector<uint32_t> meta(group_first);
            meta.insert(meta.end(), group_gate.begin(), group_gate.end());
            meta.insert(meta.end(), root_poly.begin(), root_poly.end());
            H2B_TRY(mem.get(&d_meta, meta.size(), "gate tables"));
            H2B_CUDA(cudaMemcpyAsync(d_meta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, st));
            H2B_LAUNCH(mock_gate_records_kernel, blocks_of((size_t)n_groups * n, 256), 256, 0, st, (const uint32_t*)counts, (const uint32_t*)gate_off,
                       (const uint8_t*)status, (const uint32_t*)d_meta, (const uint32_t*)d_meta + n_groups + 1, (const uint32_t*)d_meta + 2 * n_groups + 1,
                       n_groups, n, cap, d_rec);
        }
        if (totals[1] && totals[0] < cap)
            H2B_LAUNCH(mock_flag_records_kernel, blocks_of((size_t)c->n_lookups * usable, 256), 256, 0, st, (const uint32_t*)lk_flags, (const uint32_t*)lk_off,
                       c->n_lookups * usable, usable, (uint32_t)H2B_MOCK_LOOKUP, totals[0], cap, d_rec);
        if (totals[2] && totals[0] + totals[1] < cap)
            H2B_LAUNCH(mock_flag_records_kernel, blocks_of((size_t)P * n, 256), 256, 0, st, (const uint32_t*)pm_flags, (const uint32_t*)pm_off, P * n, n,
                       (uint32_t)H2B_MOCK_PERMUTATION, totals[0] + totals[1], cap, d_rec);
        H2B_CUDA(cudaGetLastError());
        std::vector<h2b_mock_record> host(cap);
        H2B_CUDA(cudaMemcpyAsync(host.data(), d_rec, (size_t)cap * sizeof(h2b_mock_record), cudaMemcpyDeviceToHost, st));
        H2B_CUDA(cudaStreamSynchronize(st));
        memcpy(records, host.data(), (size_t)cap * sizeof(h2b_mock_record));
    }
    ctx.prof.mark(PROF_MOCK_RECORDS, st);
    *count = total;
    return H2B_OK;
}

}  // namespace h2b
