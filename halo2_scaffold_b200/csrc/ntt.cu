// Radix-2 NTT over BN254 Fr for sm_100a -- the device side of `best_fft`
// ([UP] halo2_proofs/src/arithmetic.rs::best_fft @ v2023_02_02; SURVEY.md section 8 rows a3/a4;
// reached from src/scaffold.rs:135,149,287,301 (keygen_pk) and :191-214,322-346 (create_proof)).
//
// Contract (identical to the reference): a[0..2^log_n) in Montgomery form, natural order in,
// natural order out, out[i] = sum_j a[j] * omega^(i*j), no scaling.
//
// Design (tools/ntt_model.py proves the index math against the O(n^2) DFT):
//   n = N_1 * ... * N_P, N_p = 2^(b_p) <= 2^9.  Pass p works on segments of length
//   L_p = n / (N_1..N_{p-1}); one CTA stages a tile of N_p x T elements in shared memory (T
//   consecutive elements per stride so that global accesses are T*32-byte runs), runs the b_p DIF
//   butterfly stages out of shared memory with an N_p/2-entry twiddle table that also lives in
//   shared memory, leaves the digit bit-reversed in place and applies the inter-pass twiddle
//   w^(S_p * jr * bitrev(q)) from a two-level table (w^e = hi[e >> h] * lo[e & mask], both tables
//   L2-resident).  The bit-reversal permutation of the reference is never materialised: the last
//   pass scatters straight to out[bitrev(pos)], tiling over the top index bits so that those
//   writes are T*32-byte runs as well.  HBM traffic: P reads + P writes of the vector.
#include "common.h"

namespace h2b {

static const int NTT_MAX_TILE_LOG = 12;      // 4096 elements: 146 KiB of (skewed) shared memory + 73 KiB of stage twiddles
static const int NTT_DEFAULT_TILE_LOG = 11;  // measured best on B200 (profiles/r01_ntt_tiles.jsonl): 2048-element tiles, two CTAs per SM
static const int NTT_MAX_PASSES = 4;
static const int NTT_SINGLE_CTA_LOG = 10;    // up to 2^10 elements one CTA does the whole transform (latency)

static const uint32_t NTT_BATCH_MAX = 16;    // polynomials per launch (blockIdx.y): independent (i)NTTs of one proof phase share the passes
struct NttPassParams {
    const uint4* ins[NTT_BATCH_MAX];
    uint4* outs[NTT_BATCH_MAX];
    size_t in_stride, out_stride;   // != 0: polynomial y is ins[0] + y * in_stride / outs[0] + y * out_stride (uint4 units): any number of equally
                                    // spaced transforms in one launch (the row / column transforms of the multi-device four-step NTT)
    const uint4* tw_small;   // Omega^t, t < N/2, Omega = w^(n/N)
    const uint4* tw_lo;      // w^j,          j < 2^h
    const uint4* tw_hi;      // w^(j * 2^h),  j < 2^(log_n - h)
    const uint4* tw_direct;  // optional: w^(S * jr * bitrev(q)) at [q * M + jr] -- the inter-pass twiddle in ONE load, no multiplication
    uint32_t log_n;
    uint32_t b;              // digit bits of this pass
    uint32_t logT;           // tile width
    uint32_t logL;           // segment length
    uint32_t h;              // split of the two-level table
    uint32_t last;
};

// Shared-memory slot of element e.  Elements live in two 16-byte planes; the skew keeps every access pattern of the
// radix-8 rounds (strides 1, 8, 64, 512 elements) spread over all 32 banks.
__host__ __device__ __forceinline__ uint32_t sm_slot(uint32_t e) { return e + (e >> 3) + (e >> 6) + (e >> 9); }

__device__ __forceinline__ Fr sm_get(const uint4* lo, const uint4* hi, uint32_t e) {
    const uint32_t k = sm_slot(e);
    uint4 a = lo[k], b = hi[k];
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
    r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
__device__ __forceinline__ void sm_put(uint4* lo, uint4* hi, uint32_t e, const Fr& v) {
    const uint32_t k = sm_slot(e);
    lo[k] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    hi[k] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

// 16-byte global -> shared copy that does not pass through registers (LDGSTS): a thread issues all its copies of a
// tile back to back and waits once, so the tile load costs one memory latency instead of one per element.
__device__ __forceinline__ void copy16_async(uint4* smem_dst, const uint4* gmem_src) {
#ifdef H2B_EMU
    *smem_dst = *gmem_src;
#else
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem_src) : "memory");
#endif
}
__device__ __forceinline__ void copy_async_wait_all() {
#ifndef H2B_EMU
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
#endif
}

// R consecutive DIF stages (first stage index s) on 2^R elements held in registers: the elements of one work item
// differ in bits [b-s-R, b-s) of the digit q.  Stage s' multiplies the lower output of each butterfly by
// Omega^(r * 2^s'), r = position inside the half block (the table index never exceeds N/2).
template <int R>
__device__ __forceinline__ void ntt_round(uint4* lo, uint4* hi, const uint4* tlo, const uint4* thi, uint32_t item, uint32_t b, uint32_t s,
                                          uint32_t logT, bool last) {
    constexpr int K = 1 << R;
    const uint32_t loghmin = b - s - R;
    uint32_t t, g;
    if (!last) { t = item & ((1u << logT) - 1); g = item >> logT; }
    else { g = item & ((1u << (b - R)) - 1); t = item >> (b - R); }
    const uint32_t lo_part = g & ((1u << loghmin) - 1);
    const uint32_t q0 = ((g >> loghmin) << (loghmin + R)) + lo_part;
    Fr x[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const uint32_t q = q0 + ((uint32_t)j << loghmin);
        x[j] = sm_get(lo, hi, last ? ((t << b) + q) : ((q << logT) + t));
    }
#pragma unroll
    for (int st = 0; st < R; ++st) {
        const int dj = K >> (st + 1);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (j & dj) continue;
            const uint32_t r = ((uint32_t)(j & (dj - 1)) << loghmin) + lo_part;
            const uint32_t twi = r << (s + st);
            // lazily reduced (field.cuh): x stays in [0, 2p) through all rounds, in shared memory too.  (Leaving the
            // twiddled difference uncorrected, a - b + 2p < 4p, also keeps the product < 2p but spills at 128 registers.)
            Fr sum = fp_add_lazy(x[j], x[j + dj]), dif = fp_sub_lazy(x[j], x[j + dj]);
            if (twi != 0) dif = fp_mul_lazy(dif, sm_get(tlo, thi, twi));
            x[j] = sum;
            x[j + dj] = dif;
        }
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const uint32_t q = q0 + ((uint32_t)j << loghmin);
        sm_put(lo, hi, last ? ((t << b) + q) : ((q << logT) + t), x[j]);
    }
}

__global__ void __launch_bounds__(512, 1) ntt_pass_kernel(NttPassParams p) {
    H2B_DYN_SMEM(uint4, sm);
    const uint4* __restrict__ p_in = p.out_stride ? p.ins[0] + p.in_stride * blockIdx.y : p.ins[blockIdx.y];
    uint4* __restrict__ p_out = p.out_stride ? p.outs[0] + p.out_stride * blockIdx.y : p.outs[blockIdx.y];
    const uint32_t b = p.b, logT = p.logT;
    const uint32_t N = 1u << b, T = 1u << logT, E = N << logT;
    const uint32_t data_slots = sm_slot(E - 1) + 1, tw_slots = sm_slot((N >> 1) ? (N >> 1) - 1 : 0) + 1;
    uint4* lo = sm;
    uint4* hi = sm + data_slots;
    uint4* tlo = sm + 2 * data_slots;       // stage twiddles, same two planes
    uint4* thi = tlo + tw_slots;
    const uint32_t tid = threadIdx.x, nthr = blockDim.x;
    const bool last = p.last != 0;
    // non-last pass: tile (q, t), q < N, t < T  <->  global base + q*M + t ; shared e = q*T + t
    // last pass: T segments that differ in the TOP logT bits of the position;
    //            element (q, t) <-> global ((t*nseg + tile) << b) + q ; shared e = t*N + q
    const uint32_t logM = last ? 0u : p.logL - b;
    const uint32_t M = 1u << logM;
    const uint32_t log_tiles_per_seg = logM - (last ? 0u : logT);
    const uint32_t nseg = (1u << (p.log_n - b)) >> logT;

    // stage twiddles: once per CTA
    for (uint32_t idx = tid; idx < N; idx += nthr) {
        uint32_t half = idx & 1, j = idx >> 1;
        copy16_async((half ? thi : tlo) + sm_slot(j), p.tw_small + 2 * j + half);
    }
    // this CTA's tile
    const uint32_t tile = blockIdx.x;
    if (!last) {
        const uint32_t seg = tile >> log_tiles_per_seg, tau = tile & ((1u << log_tiles_per_seg) - 1);
        const uint32_t base = (seg << p.logL) + (tau << logT);
        for (uint32_t idx = tid; idx < 2 * E; idx += nthr) {
            uint32_t half = idx & 1, t = (idx >> 1) & (T - 1), q = idx >> (1 + logT);
            copy16_async((half ? hi : lo) + sm_slot((q << logT) + t), p_in + 2 * (size_t)(base + q * M + t) + half);
        }
    } else {
        for (uint32_t idx = tid; idx < 2 * E; idx += nthr) {
            uint32_t half = idx & 1, q = (idx >> 1) & (N - 1), t = idx >> (1 + b);
            copy16_async((half ? hi : lo) + sm_slot((t << b) + q), p_in + 2 * (size_t)(((t * nseg + tile) << b) + q) + half);
        }
    }
    copy_async_wait_all();
    __syncthreads();

    // b DIF stages: one partial round (b mod 3 stages) followed by radix-8 rounds, all out of registers
    uint32_t s = 0;
    if (b % 3 == 1) {
        for (uint32_t item = tid; item < (E >> 1); item += nthr) ntt_round<1>(lo, hi, tlo, thi, item, b, 0, logT, last);
        s = 1;
        __syncthreads();
    } else if (b % 3 == 2) {
        for (uint32_t item = tid; item < (E >> 2); item += nthr) ntt_round<2>(lo, hi, tlo, thi, item, b, 0, logT, last);
        s = 2;
        __syncthreads();
    }
    for (; s < b; s += 3) {
        for (uint32_t item = tid; item < (E >> 3); item += nthr) ntt_round<3>(lo, hi, tlo, thi, item, b, s, logT, last);
        __syncthreads();
    }

    // Write-out: non-last passes multiply by the inter-pass twiddles, the last pass scatters to bit-reversed positions.
    // The tile geometry is recomputed here: kept live across the radix-8 rounds, it spills at the 128-register cap.
    {
        const uint32_t logM = last ? 0u : p.logL - b;
        const uint32_t M = 1u << logM;
        const uint32_t log_tiles_per_seg = logM - (last ? 0u : logT);
        const uint32_t nseg = (1u << (p.log_n - b)) >> logT;
        if (!last) {
            const uint32_t seg = tile >> log_tiles_per_seg, tau = tile & ((1u << log_tiles_per_seg) - 1);
            const uint32_t base = (seg << p.logL) + (tau << logT);
            const uint32_t logS = p.log_n - p.logL;          // S_p = n / L_p
            const uint32_t hmask = (1u << p.h) - 1;
#pragma unroll 2
            for (uint32_t i = tid; i < E; i += nthr) {
                uint32_t t = i & (T - 1), q = i >> logT;
                Fr v = sm_get(lo, hi, i);      // in [0, 2p): the canonical inter-pass product, or fp_canon, reduces it
                uint32_t ip = __brev(q) >> (32 - b);
                uint32_t jr = (tau << logT) + t;
                uint32_t ex = (jr * ip) << logS;
                if (ex != 0) {
                    Fr w;
                    if (p.tw_direct) {
                        w = fp_load<FR>(p.tw_direct + 2 * (((size_t)q << logM) + jr));
                    } else {
                        w = fp_load<FR>(p.tw_lo + 2 * (size_t)(ex & hmask));
                        uint32_t eh = ex >> p.h;
                        if (eh != 0) w = fp_mul(w, fp_load<FR>(p.tw_hi + 2 * (size_t)eh));
                    }
                    v = fp_mul(v, w);
                } else {
                    v = fp_canon(v);
                }
                fp_store<FR>(p_out + 2 * (size_t)(base + q * M + t), v);
            }
        } else {
            for (uint32_t i = tid; i < E; i += nthr) {
                uint32_t tr = i & (T - 1), q = i >> logT;
                uint32_t t = logT ? (__brev(tr) >> (32 - logT)) : 0u;
                const uint32_t e = (t << b) + q;
                Fr v = fp_canon(sm_get(lo, hi, e));
                uint32_t pos = ((t * nseg + tile) << b) + q;
                uint32_t oidx = __brev(pos) >> (32 - p.log_n);
                fp_store<FR>(p_out + 2 * (size_t)oidx, v);
            }
        }
    }
}

// ---- twiddle tables ---------------------------------------------------------------------------
struct TwTableDesc {
    uint32_t start;    // first flat thread index of this table
    uint32_t count;    // entries
    uint32_t shift;    // table base = w^(2^shift)
    uint32_t offset;   // element offset of the table in the output buffer
};
struct TwGenParams {
    uint32_t l[8];     // omega, Montgomery limbs
    TwTableDesc tab[NTT_MAX_PASSES + 2];
    uint32_t ntab;
    uint32_t total;
    uint4* out;
};

__global__ void __launch_bounds__(128) ntt_twiddle_kernel(TwGenParams g) {
    uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= g.total) return;
    uint32_t k = 0;
    for (uint32_t i = 1; i < g.ntab; ++i) if (idx >= g.tab[i].start) k = i;
    uint32_t j = idx - g.tab[k].start;
    Fr base;
#pragma unroll
    for (int i = 0; i < 8; ++i) base.l[i] = g.l[i];
    for (uint32_t s = 0; s < g.tab[k].shift; ++s) base = fp_sqr(base);
    Fr r = fp_one<FR>();
    for (uint32_t e = j; e != 0; e >>= 1) {
        if (e & 1) r = fp_mul(r, base);
        base = fp_sqr(base);
    }
    fp_store<FR>(g.out + 2 * (size_t)(g.tab[k].offset + j), r);
}

// direct inter-pass twiddle table of one pass: entry [q * M + jr] = w^(S * jr * bitrev_b(q)), built from the two-level tables
struct TwDirectParams {
    const uint4* tw_lo;
    const uint4* tw_hi;
    uint4* out;
    uint32_t log_n, b, logL, h;
};
__global__ void __launch_bounds__(256) ntt_direct_twiddle_kernel(TwDirectParams g) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >> g.logL) return;
    const uint32_t logM = g.logL - g.b;
    const uint32_t q = (uint32_t)(idx >> logM), jr = (uint32_t)idx & ((1u << logM) - 1);
    const uint32_t ip = g.b ? (__brev(q) >> (32 - g.b)) : 0u;
    const uint32_t ex = (jr * ip) << (g.log_n - g.logL);
    Fr w = fp_load<FR>(g.tw_lo + 2 * (size_t)(ex & ((1u << g.h) - 1)));
    const uint32_t eh = ex >> g.h;
    if (eh != 0) w = fp_mul(w, fp_load<FR>(g.tw_hi + 2 * (size_t)eh));
    fp_store<FR>(g.out + 2 * idx, w);
}

struct NttPass { uint32_t b, logT, logL; };
struct NttTwiddles {
    uint64_t omega[4];
    uint32_t log_n;
    uint64_t last_use;
    DevBuf buf;
    uint32_t npass;
    NttPass pass[NTT_MAX_PASSES];
    uint32_t small_off[NTT_MAX_PASSES];
    uint32_t lo_off, hi_off, h;
    DevBuf direct;                              // direct inter-pass tables of the non-last passes (optional)
    size_t direct_off[NTT_MAX_PASSES];          // element offsets into `direct`
    bool has_direct = false;
};

static uint64_t g_use_counter = 0;

static int ntt_tile_log() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("H2B_NTT_TILE");
        v = e ? atoi(e) : NTT_DEFAULT_TILE_LOG;
        if (v < 3 || v > NTT_MAX_TILE_LOG) v = NTT_DEFAULT_TILE_LOG;
    }
    return v;
}

static int ntt_bmax() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("H2B_NTT_BMAX");
        v = e ? atoi(e) : ntt_tile_log();
        if (v < 1 || v > ntt_tile_log()) v = ntt_tile_log();
    }
    return v;
}

static void ntt_plan(uint32_t log_n, NttTwiddles& tw) {
    uint32_t P;
    static int single_env = -1;
    if (single_env < 0) {
        const char* e = getenv("H2B_NTT_SINGLE");
        single_env = e ? atoi(e) : NTT_SINGLE_CTA_LOG;
        if (single_env < 1 || single_env > ntt_tile_log()) single_env = NTT_SINGLE_CTA_LOG;
    }
    const uint32_t single = (uint32_t)(ntt_bmax() < single_env ? ntt_bmax() : single_env);
    if (log_n <= single) P = 1;
    else P = (log_n + ntt_bmax() - 1) / ntt_bmax();
    if (P < 2 && log_n > single) P = 2;
    if (P > (uint32_t)NTT_MAX_PASSES) P = NTT_MAX_PASSES;   // log_n <= 28 < 4 * 7 needs H2B_NTT_BMAX >= 7
    tw.npass = P;
    uint32_t logL = log_n;
    for (uint32_t p = 0; p < P; ++p) {
        uint32_t b = log_n / P + (p < log_n % P ? 1 : 0);
        uint32_t logT = (uint32_t)ntt_tile_log() - b;
        uint32_t room = (p + 1 < P) ? (logL - b) : (log_n - b);   // tile cannot exceed the stride / segment count
        if (logT > room) logT = room;
        tw.pass[p].b = b;
        tw.pass[p].logT = logT;
        tw.pass[p].logL = logL;
        logL -= b;
    }
}

static int ntt_get_twiddles(DeviceCtx& ctx, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream, NttTwiddles** out) {
    for (NttTwiddles* t : ctx.twiddles) {
        if (t->log_n == log_n && memcmp(t->omega, omega, 32) == 0) {
            t->last_use = ++g_use_counter;
            *out = t;
            return H2B_OK;
        }
    }
    // the direct tables are big (32 * n bytes): keep the cache under a byte budget as well as under 16 entries
    for (;;) {
        size_t bytes = 0, victim = 0;
        for (size_t i = 0; i < ctx.twiddles.size(); ++i) {
            bytes += ctx.twiddles[i]->direct.cap;
            if (ctx.twiddles[i]->last_use < ctx.twiddles[victim]->last_use) victim = i;
        }
        if (bytes <= ((size_t)12 << 30) || ctx.twiddles.size() <= 1) break;
        H2B_CUDA(cudaStreamSynchronize(stream));
        NttTwiddles* v = ctx.twiddles[victim];
        ctx.twiddles.erase(ctx.twiddles.begin() + victim);
        v->buf.release();
        v->direct.release();
        delete v;
    }
    NttTwiddles* t;
    if (ctx.twiddles.size() >= 16) {   // evict the least recently used entry
        size_t victim = 0;
        for (size_t i = 1; i < ctx.twiddles.size(); ++i)
            if (ctx.twiddles[i]->last_use < ctx.twiddles[victim]->last_use) victim = i;
        t = ctx.twiddles[victim];
        ctx.twiddles.erase(ctx.twiddles.begin() + victim);
        H2B_CUDA(cudaStreamSynchronize(stream));
    } else {
        t = new NttTwiddles();
    }
    memcpy(t->omega, omega, 32);
    t->log_n = log_n;
    t->last_use = ++g_use_counter;
    ntt_plan(log_n, *t);

    TwGenParams g;
    memset(&g, 0, sizeof(g));
    memcpy(g.l, omega, 32);
    uint32_t off = 0, start = 0, nt = 0;
    for (uint32_t p = 0; p < t->npass; ++p) {
        uint32_t b = t->pass[p].b, cnt = b ? (1u << (b - 1)) : 1u;
        t->small_off[p] = off;
        g.tab[nt++] = TwTableDesc{start, cnt, log_n - b, off};
        off += cnt; start += cnt;
    }
    t->h = (log_n + 1) / 2;
    t->lo_off = off;
    g.tab[nt++] = TwTableDesc{start, 1u << t->h, 0, off};
    off += 1u << t->h; start += 1u << t->h;
    t->hi_off = off;
    g.tab[nt++] = TwTableDesc{start, 1u << (log_n - t->h), t->h, off};
    off += 1u << (log_n - t->h); start += 1u << (log_n - t->h);
    g.ntab = nt;
    g.total = start;
    int rc = t->buf.reserve((size_t)off * 32);
    if (rc != H2B_OK) { delete t; return rc; }
    g.out = (uint4*)t->buf.p;
    H2B_LAUNCH(ntt_twiddle_kernel, (g.total + 127) / 128, 128, 0, stream, g);
    H2B_CUDA(cudaGetLastError());
    // Direct inter-pass tables (one 32-byte load replaces two loads and a multiplication per element and pass
    // boundary; about n entries in total).  Only while they stay affordable: H2B_NTT_DIRECT_MB per (omega, log n),
    // default 2304 MiB = up to 2^26.
    static long direct_mb = -1;
    if (direct_mb < 0) { const char* e = getenv("H2B_NTT_DIRECT_MB"); direct_mb = e ? atol(e) : 2304; }
    t->has_direct = false;
    if (t->npass > 1) {
        size_t entries = 0;
        for (uint32_t p = 0; p + 1 < t->npass; ++p) { t->direct_off[p] = entries; entries += (size_t)1 << t->pass[p].logL; }
        if (entries * 32 <= (size_t)direct_mb << 20 && t->direct.reserve(entries * 32) == H2B_OK) {
            for (uint32_t p = 0; p + 1 < t->npass; ++p) {
                TwDirectParams d;
                d.tw_lo = (const uint4*)t->buf.p + 2 * (size_t)t->lo_off;
                d.tw_hi = (const uint4*)t->buf.p + 2 * (size_t)t->hi_off;
                d.out = (uint4*)t->direct.p + 2 * t->direct_off[p];
                d.log_n = log_n; d.b = t->pass[p].b; d.logL = t->pass[p].logL; d.h = t->h;
                const size_t cnt = (size_t)1 << d.logL;
                H2B_LAUNCH(ntt_direct_twiddle_kernel, (unsigned)((cnt + 255) / 256), 256, 0, stream, d);
            }
            H2B_CUDA(cudaGetLastError());
            t->has_direct = true;
        } else {
            t->direct.release();
            cudaGetLastError();
        }
    } else {
        t->direct.release();
    }
    ctx.twiddles.push_back(t);
    *out = t;
    return H2B_OK;
}

// `count` <= NTT_BATCH_MAX transforms of the same (omega, log_n) in one launch per pass (polynomial = blockIdx.y)
static int ntt_run_group(DeviceCtx& ctx, void* const* d_polys, uint32_t count, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream, size_t stride_elems = 0) {
    NttTwiddles* tw = nullptr;
    ctx.prof.mark(PROF_BEGIN, stream);
    H2B_TRY(ntt_get_twiddles(ctx, omega, log_n, stream, &tw));
    ctx.prof.mark(PROF_NTT_TWIDDLE, stream);
    const size_t n = (size_t)1 << log_n;
    if (tw->npass > 1) H2B_TRY(ctx.ntt_work.reserve(n * 32 * count));
    auto kfn = ntt_pass_kernel;
    if (!ctx.ntt_attr_set) {
        H2B_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      32 * (int)(sm_slot((1u << NTT_MAX_TILE_LOG) - 1) + 1 + sm_slot((1u << (NTT_MAX_TILE_LOG - 1)) - 1) + 1)));
        ctx.ntt_attr_set = true;
    }
    const uint4* tbl = (const uint4*)tw->buf.p;
    for (uint32_t p = 0; p < tw->npass; ++p) {
        NttPassParams a;
        memset(&a, 0, sizeof(a));
        const bool first = (p == 0), last = (p + 1 == tw->npass);
        // pass 1: a -> work, middle passes in place in work, last pass: work -> a (scatter)
        if (stride_elems) {      // `count` transforms spaced stride_elems apart, starting at d_polys[0]
            uint4* work = (uint4*)ctx.ntt_work.p;
            a.ins[0] = first ? (const uint4*)d_polys[0] : work;
            a.outs[0] = last ? (uint4*)d_polys[0] : work;
            a.in_stride = first ? 2 * stride_elems : 2 * n;
            a.out_stride = last ? 2 * stride_elems : 2 * n;
        } else {
            for (uint32_t j = 0; j < count; ++j) {
                uint4* work = (uint4*)ctx.ntt_work.p + 2 * n * j;
                a.ins[j] = first ? (const uint4*)d_polys[j] : work;
                a.outs[j] = last ? (uint4*)d_polys[j] : work;
            }
        }
        a.tw_small = tbl + 2 * (size_t)tw->small_off[p];
        a.tw_lo = tbl + 2 * (size_t)tw->lo_off;
        a.tw_hi = tbl + 2 * (size_t)tw->hi_off;
        a.tw_direct = (tw->has_direct && !last) ? (const uint4*)tw->direct.p + 2 * tw->direct_off[p] : nullptr;
        a.log_n = log_n;
        a.b = tw->pass[p].b;
        a.logT = tw->pass[p].logT;
        a.logL = tw->pass[p].logL;
        a.h = tw->h;
        a.last = last ? 1u : 0u;
        const uint32_t logE = a.b + a.logT;
        const uint32_t ntiles = 1u << (log_n - logE);
        uint32_t threads = (1u << logE) / 8;
        if (threads > 512) threads = 512;
        if (threads < 32) threads = 32;
        const size_t smem = 32 * ((size_t)sm_slot((1u << logE) - 1) + 1 + sm_slot(a.b > 1 ? (1u << (a.b - 1)) - 1 : 0) + 1);
        // one CTA per tile: CTAs of different ages overlap their load, butterfly and store phases on an SM
        H2B_LAUNCH(kfn, dim3(ntiles, count), threads, smem, stream, a);
        H2B_CUDA(cudaGetLastError());
        ctx.prof.mark(PROF_NTT_PASS0 + (int)p, stream);
    }
    return H2B_OK;
}

int ntt_run(DeviceCtx& ctx, void* d_a, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream) {
    if (log_n > 28) { set_error("ntt: log_n = %u exceeds the two-adicity of Fr (28)", log_n); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n == 0) return H2B_OK;
    if (!d_a) { set_error("ntt: null data pointer"); return H2B_ERR_BAD_ARGUMENT; }
    void* one[1] = {d_a};
    return ntt_run_group(ctx, one, 1, omega, log_n, stream);
}

// Independent transforms of equal size (the per-polynomial (i)NTTs of a proof phase): groups of up to NTT_BATCH_MAX polynomials
// and 2^26 elements share every pass launch, so that 2^16-element transforms (32 tiles each) fill the 148 SMs together.
int ntt_run_batch(DeviceCtx& ctx, void* const* d_polys, size_t count, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream) {
    if (log_n > 28) { set_error("ntt: log_n = %u exceeds the two-adicity of Fr (28)", log_n); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n == 0 || count == 0) return H2B_OK;
    for (size_t j = 0; j < count; ++j) if (!d_polys[j]) { set_error("ntt batch: polynomial %zu is null", j); return H2B_ERR_BAD_ARGUMENT; }
    size_t group = NTT_BATCH_MAX;
    while (group > 1 && (group << log_n) > ((size_t)1 << 26)) group >>= 1;
    for (size_t j0 = 0; j0 < count; j0 += group) {
        const size_t m = count - j0 < group ? count - j0 : group;
        H2B_TRY(ntt_run_group(ctx, d_polys + j0, (uint32_t)m, omega, log_n, stream));
    }
    return H2B_OK;
}
uint32_t ntt_batch_max() { return NTT_BATCH_MAX; }

// `count` in-place transforms of 2^log_n elements each, spaced stride_elems >= 2^log_n elements apart from d_base on: the rows of a matrix
int ntt_run_strided(DeviceCtx& ctx, void* d_base, size_t count, size_t stride_elems, const uint64_t omega[4], uint32_t log_n, cudaStream_t stream) {
    if (log_n > 28 || log_n == 0) { set_error("strided ntt: log_n = %u out of range", log_n); return H2B_ERR_BAD_ARGUMENT; }
    if (count == 0) return H2B_OK;
    if (!d_base || stride_elems < ((size_t)1 << log_n)) { set_error("strided ntt: bad base or stride"); return H2B_ERR_BAD_ARGUMENT; }
    size_t group = 32768;                                        // gridDim.y
    while (group > 1 && (group << log_n) > ((size_t)1 << 27)) group >>= 1;      // work buffer: at most 4 GiB
    for (size_t j0 = 0; j0 < count; j0 += group) {
        const size_t m = count - j0 < group ? count - j0 : group;
        void* one[1] = {(char*)d_base + j0 * stride_elems * 32};
        H2B_TRY(ntt_run_group(ctx, one, (uint32_t)m, omega, log_n, stream, stride_elems));
    }
    return H2B_OK;
}

// ---- pieces of the four-step NTT across the devices of one process (api_sets.cu: ntt_multi_device) ------------------------------------
// out[c * rows + r] = in[r * cols + c] for a rows x cols matrix of Fr elements (32-byte tiles through shared memory: both sides coalesced)
__global__ void __launch_bounds__(256) fr_transpose_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, uint32_t rows, uint32_t cols) {
    __shared__ uint4 tile[2][32][33];
    const uint32_t c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (uint32_t dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const uint32_t r = r0 + dy, c = c0 + threadIdx.x;
        if (r < rows && c < cols) {
            tile[0][dy][threadIdx.x] = in[2 * ((size_t)r * cols + c)];
            tile[1][dy][threadIdx.x] = in[2 * ((size_t)r * cols + c) + 1];
        }
    }
    __syncthreads();
    for (uint32_t dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const uint32_t c = c0 + dy, r = r0 + threadIdx.x;
        if (r < rows && c < cols) {
            out[2 * ((size_t)c * rows + r)] = tile[0][threadIdx.x][dy];
            out[2 * ((size_t)c * rows + r) + 1] = tile[1][threadIdx.x][dy];
        }
    }
}
#ifndef H2B_EMU
// The same transpose with the tile brought in by the TMA unit: one thread arms an mbarrier with the tile's byte count and issues 32
// bulk copies (cp.async.bulk.shared::cluster.global, 1 KiB = one tile row each; UBLKCP in SASS) into rows padded by 16 bytes, every
// thread waits on the barrier's phase and the transposed reads are conflict-free (row stride 260 words: lanes 4 banks apart).  No
// thread touches the incoming data before it sits in shared memory and no register or LSU slot is spent on it.  Whole tiles only
// (rows and cols multiples of 32); other shapes take fr_transpose_kernel.
static const uint32_t TR_ROW_BYTES = 32 * 32 + 16;
__global__ void __launch_bounds__(256) fr_transpose_bulk_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, uint32_t rows, uint32_t cols) {
    __shared__ __align__(128) unsigned char tile[32 * TR_ROW_BYTES];
    __shared__ __align__(8) unsigned long long mbar;
    const uint32_t c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const uint32_t tid = threadIdx.y * 32 + threadIdx.x;
    const unsigned mbar_s = (unsigned)__cvta_generic_to_shared(&mbar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_s) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar_s), "r"(32u * 1024u) : "memory");
        for (uint32_t r = 0; r < 32; ++r) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(tile + r * TR_ROW_BYTES);
            const uint4* src = in + 2 * ((size_t)(r0 + r) * cols + c0);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(1024u), "r"(mbar_s)
                         : "memory");
        }
    }
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra TR_DONE;\n"
        "bra TR_WAIT;\n"
        "TR_DONE:\n"
        "}" ::"r"(mbar_s), "r"(0u)
        : "memory");
    for (uint32_t dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const uint4* e = reinterpret_cast<const uint4*>(tile + threadIdx.x * TR_ROW_BYTES + dy * 32);
        const size_t o = 2 * ((size_t)(c0 + dy) * rows + r0 + threadIdx.x);
        out[o] = e[0];
        out[o + 1] = e[1];
    }
}
#endif

int fr_transpose_run(DeviceCtx& ctx, const void* d_in, void* d_out, uint32_t rows, uint32_t cols, cudaStream_t stream) {
    (void)ctx;
    if (rows == 0 || cols == 0) return H2B_OK;
    const uint32_t gy = (rows + 31) / 32;
    if (gy > 65535) { set_error("transpose: too many rows"); return H2B_ERR_BAD_ARGUMENT; }
#ifndef H2B_EMU
    static int bulk = -1;
    if (bulk < 0) { const char* e = getenv("H2B_TRANSPOSE_BULK"); bulk = e ? atoi(e) : 1; }
    if (bulk && rows % 32 == 0 && cols % 32 == 0 && ((uintptr_t)d_in & 15) == 0) {
        H2B_LAUNCH(fr_transpose_bulk_kernel, dim3(cols / 32, gy), dim3(32, 8), 0, stream, (const uint4*)d_in, (uint4*)d_out, rows, cols);
        H2B_CUDA(cudaGetLastError());
        return H2B_OK;
    }
#endif
    H2B_LAUNCH(fr_transpose_kernel, dim3((cols + 31) / 32, gy), dim3(32, 8), 0, stream, (const uint4*)d_in, (uint4*)d_out, rows, cols);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// y[row][k] *= w^((row0 + row) * k) for a rows x 2^log_len matrix (row-major): the twiddle step between the column and the row transforms.
// A thread owns FS_RUN consecutive k of one row: g = w^(row0 + row), start g^(k0) by square-and-multiply, then one multiplication per step.
static const uint32_t FS_RUN = 64;
struct FsOmega { uint32_t w[8]; };
__global__ void __launch_bounds__(128) ntt_fourstep_twiddle_kernel(uint4* __restrict__ y, uint32_t rows, uint32_t log_len, uint32_t row0, FsOmega om) {
    const uint32_t len = 1u << log_len;
    const uint32_t run = len < FS_RUN ? len : FS_RUN;
    const uint32_t runs_per_row = len / run;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)rows * runs_per_row) return;
    const uint32_t row = (uint32_t)(t / runs_per_row), k0 = (uint32_t)(t % runs_per_row) * run;
    Fr w;
#pragma unroll
    for (int i = 0; i < 8; ++i) w.l[i] = om.w[i];
    const Fr g = fp_pow_u32(w, row0 + row);
    Fr cur = fp_pow_u32(g, k0);
    uint4* p = y + 2 * ((size_t)row * len + k0);
    for (uint32_t k = 0; k < run; ++k) {
        fp_store<FR>(p + 2 * k, fp_mul(fp_load<FR>(p + 2 * k), cur));
        cur = fp_mul(cur, g);
    }
}
int ntt_fourstep_twiddle_run(DeviceCtx& ctx, void* d_y, uint32_t rows, uint32_t log_len, uint32_t row0, const uint64_t omega[4], cudaStream_t stream) {
    (void)ctx;
    if (rows == 0) return H2B_OK;
    FsOmega om;
    memcpy(om.w, omega, 32);
    const uint32_t len = 1u << log_len, run = len < FS_RUN ? len : FS_RUN;
    const size_t threads = (size_t)rows * (len / run);
    H2B_LAUNCH(ntt_fourstep_twiddle_kernel, (unsigned)((threads + 127) / 128), 128, 0, stream, (uint4*)d_y, rows, log_len, row0, om);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// out[0] = w^(2^e0), out[1] = w^(2^e1): the roots of the column and row transforms (no field arithmetic on the host)
__global__ void ntt_root_powers_kernel(FsOmega om, uint32_t e0, uint32_t e1, uint4* out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    Fr w;
#pragma unroll
    for (int i = 0; i < 8; ++i) w.l[i] = om.w[i];
    Fr a = w, b = w;
    for (uint32_t i = 0; i < e0; ++i) a = fp_sqr(a);
    for (uint32_t i = 0; i < e1; ++i) b = fp_sqr(b);
    fp_store<FR>(out, a);
    fp_store<FR>(out + 2, b);
}
int ntt_root_powers_run(DeviceCtx& ctx, const uint64_t omega[4], uint32_t e0, uint32_t e1, void* d_out /*64 B*/, cudaStream_t stream) {
    (void)ctx;
    FsOmega om;
    memcpy(om.w, omega, 32);
    H2B_LAUNCH(ntt_root_powers_kernel, 1, 32, 0, stream, om, e0, e1, (uint4*)d_out);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// a[i] *= factors[i % count]   (count 1 / 3: the 1/n of lagrange_to_coeff / extended_to_coeff and the zeta-coset pattern
// of coeff_to_extended; count 2^(extended_k - k) <= 8: the t_evaluations of divide_by_vanishing_poly --
// [UP] halo2_proofs/src/poly/domain.rs; SURVEY.md row a6)
struct ScaleParams { uint32_t f[8][8]; uint32_t count; };
__global__ void __launch_bounds__(256) ntt_scale_kernel(uint4* a, size_t n, ScaleParams s) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr f;
    if (s.count <= 3) {
        uint32_t k = s.count == 1 ? 0u : (uint32_t)(i % s.count);
#pragma unroll
        for (int j = 0; j < 8; ++j) f.l[j] = k == 0 ? s.f[0][j] : (k == 1 ? s.f[1][j] : s.f[2][j]);
    } else {
        const uint32_t k = (uint32_t)(i % s.count);
#pragma unroll
        for (int j = 0; j < 8; ++j) f.l[j] = s.f[k][j];
    }
    Fr v = fp_load<FR>(a + 2 * i);
    fp_store<FR>(a + 2 * i, fp_mul(v, f));
}

// count > 8 (divide_by_vanishing_poly of a circuit with cs.degree() > 9: 2^(extended_k - k) t_evaluations): factors from a device table
__global__ void __launch_bounds__(256) ntt_scale_table_kernel(uint4* a, size_t n, const uint4* __restrict__ factors, uint32_t count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Fr f = fp_load<FR>(factors + 2 * (size_t)(i % count));
    fp_store<FR>(a + 2 * i, fp_mul(fp_load<FR>(a + 2 * i), f));
}

// the same factor pattern on up to NTT_BATCH_MAX columns in one launch (column = blockIdx.y)
struct ScaleBatch { uint4* a[NTT_BATCH_MAX]; };
__global__ void __launch_bounds__(256) ntt_scale_batch_kernel(ScaleBatch cols, size_t n, ScaleParams s) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4* a = cols.a[blockIdx.y];
    const uint32_t k = s.count == 1 ? 0u : (uint32_t)(i % s.count);
    Fr f;
#pragma unroll
    for (int j = 0; j < 8; ++j) f.l[j] = s.f[k][j];
    Fr v = fp_load<FR>(a + 2 * i);
    fp_store<FR>(a + 2 * i, fp_mul(v, f));
}
int ntt_scale_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t ncols, size_t n, const uint64_t* factors, int count, cudaStream_t stream) {
    (void)ctx;
    if (count < 1 || count > 8) { set_error("batched scale: count must be in [1, 8]"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) return H2B_OK;
    ScaleParams s;
    memset(&s, 0, sizeof(s));
    s.count = (uint32_t)count;
    memcpy(s.f, factors, (size_t)count * 32);
    for (size_t j0 = 0; j0 < ncols; j0 += NTT_BATCH_MAX) {
        const size_t m = ncols - j0 < NTT_BATCH_MAX ? ncols - j0 : NTT_BATCH_MAX;
        ScaleBatch b;
        memset(&b, 0, sizeof(b));
        for (size_t j = 0; j < m; ++j) b.a[j] = (uint4*)d_cols[j0 + j];
        H2B_LAUNCH(ntt_scale_batch_kernel, dim3((unsigned)((n + 255) / 256), (unsigned)m), 256, 0, stream, b, n, s);
    }
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

int ntt_scale_run(DeviceCtx& ctx, void* d_a, size_t n, const uint64_t* factors, int count, cudaStream_t stream) {
    if (count < 1 || count > 4096) { set_error("scale: count must be in [1, 4096]"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) return H2B_OK;
    if (count > 8) {
        // the table is staged through a small device buffer of its own (grow-only; the copy is ordered on `stream`)
        H2B_TRY(ctx.scale_table.reserve((size_t)count * 32));
        H2B_CUDA(cudaMemcpyAsync(ctx.scale_table.p, factors, (size_t)count * 32, cudaMemcpyHostToDevice, stream));
        H2B_CUDA(cudaStreamSynchronize(stream));      // `factors` is the caller's (pageable) memory: do not outlive the call
        H2B_LAUNCH(ntt_scale_table_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (uint4*)d_a, n, (const uint4*)ctx.scale_table.p, (uint32_t)count);
        H2B_CUDA(cudaGetLastError());
        return H2B_OK;
    }
    ScaleParams s;
    memset(&s, 0, sizeof(s));
    s.count = (uint32_t)count;
    memcpy(s.f, factors, (size_t)count * 32);
    H2B_LAUNCH(ntt_scale_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (uint4*)d_a, n, s);
    H2B_CUDA(cudaGetLastError());
    return H2B_OK;
}

// EvaluationDomain::lagrange_to_coeff / coeff_to_extended ([UP] halo2_proofs/src/poly/domain.rs) of `count` columns in place: the (i)NTT
// passes and the scaling are launched once for the whole batch.  coeff_to_extended needs 2^extended_k elements per column.
int lagrange_to_coeff_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t count, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4],
                                cudaStream_t stream) {
    H2B_TRY(ntt_run_batch(ctx, d_cols, count, omega_inv, k, stream));
    return ntt_scale_batch_run(ctx, d_cols, count, (size_t)1 << k, ifft_divisor, 1, stream);
}

int coeff_to_extended_batch_run(DeviceCtx& ctx, void* const* d_cols, size_t count, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4],
                                const uint64_t zeta_powers[12], cudaStream_t stream) {
    const size_t n = (size_t)1 << k, en = (size_t)1 << extended_k;
    H2B_TRY(ntt_scale_batch_run(ctx, d_cols, count, n, zeta_powers, 3, stream));                     // a[i] *= zeta^(i mod 3)
    if (en > n)
        for (size_t j = 0; j < count; ++j) H2B_CUDA(cudaMemsetAsync((char*)d_cols[j] + n * 32, 0, (en - n) * 32, stream));   // zero-pad
    return ntt_run_batch(ctx, d_cols, count, extended_omega, extended_k, stream);
}

void ntt_release(DeviceCtx& ctx) {
    for (NttTwiddles* t : ctx.twiddles) { t->buf.release(); t->direct.release(); delete t; }
    ctx.twiddles.clear();
    ctx.ntt_work.release();
    ctx.ntt_io.release();
    ctx.ntt_fs[0].release();
    ctx.ntt_fs[1].release();
    ctx.scale_table.release();
}

}  // namespace h2b
