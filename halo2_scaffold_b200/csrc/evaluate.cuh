// The row interpreter of a compiled GraphEvaluator, shared by the quotient evaluation (evaluate.cu) and the MockProver checker
// (mock.cu): the micro-operation encoding, the device view of a program and its operand fetch, and the host compiler's interface.
#pragma once
#include "common.h"

namespace h2b {

enum MicroOp : uint32_t { MOP_ADD = 0, MOP_SUB = 1, MOP_MUL = 2, MOP_SQR = 3, MOP_DBL = 4, MOP_NEG = 5, MOP_FMA = 6, MOP_MOV = 7,
                          MOP_CHECK = 8 };      // CHECK: operand a is the value of root #z (only in programs compiled with roots)
// operand encoding: kind in the top two bits
static const uint32_t OPK_SLOT = 0u << 30, OPK_CONST = 1u << 30, OPK_COL = 2u << 30, OPK_PREV = 3u << 30, OPK_MASK = 3u << 30;
static const uint32_t MOP_NOSTORE = 0x80;       // flag in the op word: the result is only consumed through OPK_PREV
static const uint32_t MAX_ROT = 1024, MAX_COLS = 1u << 20, MAX_SLOTS = 64;

struct EvalProgram {            // device view of a compiled graph
    const uint4* ops;
    const uint4* consts;        // Fr table: graph constants, challenges, beta, gamma, theta, y, zero
    const uint32_t* rot_off;    // (rot * rot_scale).rem_euclid(size) per rotation index; last entry 0
    const void* const* cols;    // fixed..., advice..., instance..., values
    uint32_t n_ops;
    uint32_t size;
    // row shard: this launch evaluates rows [row0, row0 + rows) of the domain; every column pointer is a slice that starts at global row
    // `base` = row0 - halo (mod size) and holds rows + 2 * halo rows.  The whole domain is row0 = base = 0, rows = size.
    uint32_t row0, rows, base;
};

__device__ __forceinline__ uint32_t shard_local(uint32_t row, uint32_t base, uint32_t size) { return row >= base ? row - base : row + (size - base); }

// the global row a column operand reads at row idx
__device__ __forceinline__ uint32_t eval_operand_row(const EvalProgram& p, uint32_t v, uint32_t idx) {
    uint32_t row = idx + __ldg(p.rot_off + (v & (MAX_ROT - 1)));
    if (row >= p.size) row -= p.size;
    return row;
}

__device__ __forceinline__ Fr eval_fetch(const EvalProgram& p, uint32_t enc, uint32_t idx, const Fr* slots, const Fr& prev) {
    const uint32_t kind = enc & OPK_MASK, v = enc & ~OPK_MASK;
    if (kind == OPK_PREV) return prev;
    if (kind == OPK_SLOT) return slots[v];
    if (kind == OPK_CONST) return fp_load<FR>(p.consts + 2 * (size_t)v);
    const uint32_t row = shard_local(eval_operand_row(p, v, idx), p.base, p.size);
    const uint4* col = reinterpret_cast<const uint4*>(__ldg(reinterpret_cast<const unsigned long long*>(p.cols) + (v >> 10)));
    return fp_load<FR>(col + 2 * (size_t)row);
}

// ---- host: the compiler ------------------------------------------------------------------------------------------------
struct Shard { uint32_t row0, rows, halo, base; };

struct Compiled {
    std::vector<uint4> ops;
    std::vector<uint64_t> consts;       // 4 words per entry
    std::vector<uint32_t> rot_off;
    std::vector<const void*> cols;
    uint32_t n_slots = 0;
    uint32_t c_beta = 0, c_gamma = 0, c_theta = 0, c_y = 0, c_zero = 0;
};

// Compiles graph `g` over the columns `cols` (device pointers) into micro-operations.  Without roots (n_roots = 0) the program's
// result is the last calculation's value, as evaluate_h reads it.  With roots, the program computes every root in order and
// follows each with a MOP_CHECK of its value (z = the root's position); a root stays live until its check.
int compile_graph(const h2b_graph* g, const h2b_eval_columns* cols, const void* d_values, uint32_t size, int32_t rot_scale, bool previous_is_zero,
                  const Shard& shard, const h2b_value_source* roots, uint32_t n_roots, Compiled& out);

// device copy of a compiled program: a small ring of buffers per device so that calls on different streams do not
// overwrite a program a running kernel still reads.  Record `(*used)->done` on `stream` after the last launch that reads it.
struct ProgramBuf { DevBuf buf; cudaEvent_t done = nullptr; };
int upload_program(DeviceCtx& ctx, const Compiled& c, uint32_t size, const Shard& shard, cudaStream_t stream, EvalProgram& dev, ProgramBuf** used);

}  // namespace h2b
