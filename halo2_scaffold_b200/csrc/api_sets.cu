// C ABI of libh2b200, resident base sets: registration, the implicit SRS cache of h2b_msm_bn254_g1 and the host-pointer drop-ins for
// best_multiexp / best_fft (single, batched, point-range sharded across the GPUs of one box, one NTT across them), and
// h2b_column_pipeline.
#include <thread>

#include "host.h"

namespace h2b {

static const size_t IMPLICIT_CACHE_MAX_SETS = 8;
// MSMs below this many points stay on one device (H2B_MULTI_DEVICE_MIN_LOG lowers it: tests)
static size_t multi_device_min_points() {
    static size_t v = 0;
    if (!v) { const char* e = getenv("H2B_MULTI_DEVICE_MIN_LOG"); int lg = e ? atoi(e) : 18; v = (size_t)1 << (lg < 1 || lg > 28 ? 18 : lg); }
    return v;
}
#define MULTI_DEVICE_MIN_POINTS (multi_device_min_points())
static const uint64_t IMPLICIT_TABLES_AFTER_USES = 2;   // an implicitly cached SRS vector gets its tables on the 2nd MSM

static int env_int_or(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}
// the implicit cache works on blocks of 2^H2B_DIGEST_BLOCK_LOG points (default 1024 = 64 KiB) and only takes arrays of at
// least 2^H2B_IMPLICIT_MIN_LOG points (default 4096) whose length is a whole number of blocks; tests lower both
static size_t digest_block() {
    static size_t v = 0;
    if (!v) { int lg = env_int_or("H2B_DIGEST_BLOCK_LOG", 10); v = (size_t)1 << (lg < 2 || lg > 16 ? 10 : lg); }
    return v;
}
static size_t implicit_min_points() {
    static size_t v = 0;
    if (!v) { int lg = env_int_or("H2B_IMPLICIT_MIN_LOG", 12); v = (size_t)1 << (lg < 2 || lg > 28 ? 12 : lg); if (v < digest_block()) v = digest_block(); }
    return v;
}
static bool implicit_cache_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("H2B_IMPLICIT_CACHE"); v = (e && e[0] == '0') ? 0 : 1; }
    return v == 1;
}

// table policy: -1 never build tables, 0 automatic spacing, > 0 forced spacing (tests / tuning)
static int g_table_policy = -2;
static int table_policy() {
    if (g_table_policy == -2) {
        const char* e = getenv("H2B_MSM_PRECOMP");
        g_table_policy = e ? atoi(e) : 0;
        if (e && g_table_policy == 0 && e[0] == '0') g_table_policy = -1;      // H2B_MSM_PRECOMP=0 disables
    }
    return g_table_policy;
}

// ---- content digests of host arrays (implicit cache) --------------------------------------------------------------------
// best_multiexp is a pure function of its arguments: a device copy may only be reused if the caller's array still holds exactly
// what was uploaded.  Every block of digest_block() points gets a 128-bit digest (multiply-fold over 64-bit words, four
// independent lanes: memory-bound on one core); a cached set is reused only after ALL blocks of the call's range matched.
static inline uint64_t mum64(uint64_t a, uint64_t b) {
    unsigned __int128 r = (unsigned __int128)a * b;
    return (uint64_t)r ^ (uint64_t)(r >> 64);
}
static void digest_words(const uint64_t* p, size_t words, uint64_t out[2]) {
    uint64_t a0 = 0xa0761d6478bd642full, a1 = 0xe7037ed1a0b428dbull, a2 = 0x8ebc6af09c88c6e3ull, a3 = 0x589965cc75374cc3ull;
    size_t i = 0;
    for (; i + 8 <= words; i += 8) {
        a0 = mum64(p[i] ^ 0x2d358dccaa6c78a5ull, p[i + 1] ^ a0);
        a1 = mum64(p[i + 2] ^ 0x8bb84b93962eacc9ull, p[i + 3] ^ a1);
        a2 = mum64(p[i + 4] ^ 0x4b33a62ed433d4a3ull, p[i + 5] ^ a2);
        a3 = mum64(p[i + 6] ^ 0x4d5a2da51de1aa47ull, p[i + 7] ^ a3);
    }
    for (; i < words; ++i) a0 = mum64(p[i] ^ 0x2d358dccaa6c78a5ull, a0 ^ (0x9e3779b97f4a7c15ull + i));
    out[0] = mum64(a0 ^ a2 ^ (uint64_t)words, a1 ^ 0xa0761d6478bd642full) ^ a3;
    out[1] = mum64(a1 + a3, a2 ^ 0xe7037ed1a0b428dbull) ^ mum64(a0, a3 ^ 0x589965cc75374cc3ull);
}
static unsigned digest_threads() {
    static unsigned v = 0;
    if (!v) {
        unsigned hw = std::thread::hardware_concurrency();
        v = hw >= 16 ? 8 : (hw >= 8 ? 4 : 2);
        int e = env_int_or("H2B_DIGEST_THREADS", 0);
        if (e >= 1 && e <= 64) v = (unsigned)e;
    }
    return v;
}
// blocks [b0, b1) of `bases`: mode 0 writes the digests to out, mode 1 compares them with `want` (early exit) -> all equal?
static bool digest_blocks(const uint64_t* bases, size_t b0, size_t b1, uint64_t* out, const uint64_t* want) {
    const size_t blk = digest_block();
    std::atomic<bool> ok{true};
    std::atomic<size_t> next{b0};
    auto work = [&] {
        for (;;) {
            const size_t b = next.fetch_add(16);
            if (b >= b1 || !ok.load(std::memory_order_relaxed)) return;
            for (size_t x = b; x < b + 16 && x < b1; ++x) {
                uint64_t d[2];
                digest_words(bases + x * blk * 8, blk * 8, d);
                if (want) { if (d[0] != want[2 * x] || d[1] != want[2 * x + 1]) { ok = false; return; } }
                else { out[2 * x] = d[0]; out[2 * x + 1] = d[1]; }
            }
        }
    };
    const size_t count = b1 - b0;
    unsigned T = digest_threads();
    if (count < 256) T = 1;                     // below 16 MiB a thread launch costs more than it saves
    if (T <= 1) { work(); return ok; }
    std::vector<std::thread> th;
    for (unsigned t = 1; t < T; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    return ok;
}

// ---- building resident sets ------------------------------------------------------------------------------------------------
// a set of n points laid out over every device, nothing allocated yet
static SetRef new_set(size_t n, bool sharded) {
    const size_t nd = G.devs.size();
    SetRef bs(new BaseSet());
    bs->n = n;
    bs->sharded = sharded;
    bs->lo.assign(nd, 0);
    bs->rows.assign(nd, n);
    if (sharded)
        for (size_t d = 0; d < nd; ++d) { bs->lo[d] = n * d / nd; bs->rows[d] = n * (d + 1) / nd - bs->lo[d]; }
    for (size_t d = 0; d < nd; ++d) bs->ordinal.push_back(G.devs[d]->device);
    bs->dev.assign(nd, nullptr);
    return bs;
}

static SetRef new_set_like(const BaseSet& src) {
    SetRef bs = new_set(src.n, src.sharded);
    bs->handle = src.handle; bs->implicit = src.implicit; bs->host_ptr = src.host_ptr; bs->digest = src.digest;
    bs->last_use = src.last_use; bs->uses = src.uses; bs->refs = src.refs;
    return bs;
}

// device 0's rows of a replicated set -> every other device, one peer copy each
static int replicate_device0(BaseSet& bs) {
    for (size_t d = 1; d < G.devs.size(); ++d) {
        DeviceCtx& c = *G.devs[d];
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        H2B_TRY(dev_malloc(&bs.dev[d], bs.n * 64 + 64, "SRS bases"));
        const cudaError_t e = cudaMemcpyPeer(bs.dev[d], c.device, bs.dev[0], G.devs[0]->device, bs.n * 64);
        if (e != cudaSuccess) { set_error("device %zu: peer copy of SRS bases: %s", d, cudaGetErrorString(e)); return H2B_ERR_CUDA; }
    }
    return H2B_OK;
}

// The table set of msm.cu step 0 for a resident point set (table 0 = the points themselves) as a NEW set; the source stays
// untouched (calls in flight keep using it).  Best effort: returns the source itself when tables are off or do not fit.
// Work split: a sharded set's device builds the tables of its own rows; the devices of a replicated set each build 1/D of
// the rows and all-gather the rest over NVLink (peer copies run at hundreds of GB/s, recomputation at 18 G points/s), so
// registration time falls with the device count instead of growing with it.
static SetRef build_tables(const SetRef& src) {
    const int policy = table_policy();
    const size_t nd = G.devs.size();
    if (policy < 0 || src->n_tables > 1 || src->n == 0) return src;
    size_t max_rows = 0;
    for (size_t d = 0; d < nd; ++d) max_rows = src->rows[d] > max_rows ? src->rows[d] : max_rows;
    if (max_rows > ((size_t)1 << 26)) return src;
    // spacing for the MSMs this layout runs: whole-set MSMs on one device (replicated) or 1/D of the set (sharded)
    uint32_t c0 = 0;
    if (policy > 0) c0 = (uint32_t)policy;
    else {
        size_t free_b = 0, total_b = 0;
        cudaSetDevice(G.devs[0]->device);
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return src;
        size_t max_tables = (free_b / 3) / (max_rows * 64);
        if ((uint64_t)max_rows * max_tables >= 0x7fffffffull) max_tables = (size_t)(0x7fffffffull / max_rows);
        c0 = msm_pick_table_spacing(max_rows, (uint32_t)(max_tables > 128 ? 128 : max_tables));
    }
    if (c0 < 2 || c0 > 24) return src;
    const uint32_t nt = msm_tables_for(c0);
    if ((uint64_t)max_rows * nt >= 0x7fffffffull) return src;
    SetRef out = new_set_like(*src);
    out->n_tables = nt;
    out->c0 = c0;
    bool ok = true;
    std::vector<std::unique_lock<std::mutex>> locks;
    for (size_t d = 0; d < nd; ++d) locks.emplace_back(G.devs[d]->mu);
    const bool gather = !src->sharded && nd > 1;
    // phase 1: every device computes its share (kernels of all devices queued first, awaited afterwards)
    for (size_t d = 0; d < nd && ok; ++d) {
        DeviceCtx& c = *G.devs[d];
        const size_t R = src->rows[d];
        if (R == 0) continue;
        cudaSetDevice(c.device);
        if (dev_malloc(&out->dev[d], (size_t)nt * R * 64 + 64, "window tables") != H2B_OK) { ok = false; break; }
        const size_t r0 = gather ? R * d / nd : 0, r1 = gather ? R * (d + 1) / nd : R;
        c.prof.mark(PROF_BEGIN, c.stream);
        if (cudaMemcpyAsync(out->dev[d], src->dev[d], R * 64, cudaMemcpyDeviceToDevice, c.stream) != cudaSuccess) ok = false;
        for (uint32_t j = 1; j < nt && ok && r1 > r0; ++j)
            ok = msm_precompute_run(c, (const char*)out->dev[d] + ((size_t)(j - 1) * R + r0) * 64, (char*)out->dev[d] + ((size_t)j * R + r0) * 64, r1 - r0, c0, c.stream) == H2B_OK;
        c.prof.mark(PROF_MSM_PRECOMPUTE, c.stream);
    }
    for (size_t d = 0; d < nd; ++d) {
        if (!out->dev[d]) continue;
        cudaSetDevice(G.devs[d]->device);
        if (cudaStreamSynchronize(G.devs[d]->stream) != cudaSuccess) ok = false;
    }
    // phase 2 (replicated sets on several devices): every device pulls the other devices' shares
    if (ok && gather) {
        const size_t R = src->n;
        for (size_t d = 0; d < nd && ok; ++d) {
            cudaSetDevice(G.devs[d]->device);
            for (size_t e = 0; e < nd && ok; ++e) {
                if (e == d) continue;
                const size_t r0 = R * e / nd, r1 = R * (e + 1) / nd;
                for (uint32_t j = 1; j < nt && ok && r1 > r0; ++j)
                    ok = cudaMemcpyPeerAsync((char*)out->dev[d] + ((size_t)j * R + r0) * 64, G.devs[d]->device, (const char*)out->dev[e] + ((size_t)j * R + r0) * 64,
                                             G.devs[e]->device, (r1 - r0) * 64, G.devs[d]->stream) == cudaSuccess;
            }
        }
        for (size_t d = 0; d < nd; ++d) {
            cudaSetDevice(G.devs[d]->device);
            if (cudaStreamSynchronize(G.devs[d]->stream) != cudaSuccess) ok = false;
        }
    }
    locks.clear();
    if (!ok) { cudaGetLastError(); return src; }      // `out` frees whatever it allocated
    return out;
}

// upload `bases` (host) as a new resident set
static int create_set(const uint64_t* bases, size_t n, bool sharded, bool with_tables, SetRef* out) {
    SetRef bs = new_set(n, sharded && G.devs.size() > 1);
    // sharded: disjoint slices, one upload per device, concurrently (each over its own PCIe link).  Replicated: one trip over PCIe
    // to device 0, then peer copies: D concurrent uploads of the same host array only fight for the host's memory
    std::vector<size_t> devs;
    for (size_t d = 0; d < (bs->sharded ? G.devs.size() : 1); ++d) if (bs->rows[d]) devs.push_back(d);
    H2B_TRY(on_devices(devs, [&](size_t d) -> int {
        DeviceCtx& c = *G.devs[d];
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        H2B_TRY(dev_malloc(&bs->dev[d], bs->rows[d] * 64 + 64, "SRS bases"));
        H2B_TRY(host_upload(c, bs->dev[d], bases + 8 * bs->lo[d], bs->rows[d] * 64, c.stream));
        if (cudaStreamSynchronize(c.stream) != cudaSuccess) { set_error("SRS upload: %s", cudaGetErrorString(cudaGetLastError())); return H2B_ERR_CUDA; }
        return H2B_OK;
    }));
    if (!bs->sharded) H2B_TRY(replicate_device0(*bs));
    *out = with_tables ? build_tables(bs) : bs;
    return H2B_OK;
}

// hands a new set out under a fresh handle.  Caller holds G.mu.
static uint64_t publish_new_locked(const SetRef& bs) {
    bs->last_use = ++G.use_counter;
    return G.sets.publish_locked(bs);
}

int device0_points_locked(size_t n, const char* caller, const char* what, bool release_g1gen,
                          const std::function<int(DeviceCtx&, void*)>& produce, uint64_t* host_out, uint64_t* handle) {
    DeviceCtx& c = *G.devs[0];
    SetRef bs = new_set(n, false);      // owns the points from here on: every failure path frees them
    int rc;
    {
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        const size_t scan_cap = c.scan_scratch.cap;
        rc = dev_malloc(&bs->dev[0], n * 64 + 64, "SRS bases");
        if (!rc) rc = produce(c, bs->dev[0]);
        if (!rc && host_out) rc = host_download(c, host_out, bs->dev[0], n * 64, c.stream);
        if (!rc && cudaStreamSynchronize(c.stream) != cudaSuccess) { set_error("%s", cudaGetErrorString(cudaGetLastError())); rc = H2B_ERR_CUDA; }
        if (release_g1gen) g1gen_release_scratch(c, scan_cap);
    }
    if (!rc && handle) rc = replicate_device0(*bs);
    if (rc) { set_error("%s: %s: %s", caller, what, std::string(get_error()).c_str()); return rc; }
    if (handle) *handle = publish_new_locked(build_tables(bs));
    return H2B_OK;
}

// ---- the implicit cache of h2b_msm_bn254_g1 ---------------------------------------------------------------------------------
// quick filter before the (concurrent) full verification: up to 16 evenly spaced blocks of the call's range. Caller holds G.mu.
static bool spot_check(const BaseSet& bs, const uint64_t* bases, size_t nblocks) {
    const size_t blk = digest_block();
    for (int k = 0; k < 16; ++k) {
        const size_t b = nblocks <= 1 ? 0 : (size_t)(((unsigned __int128)k * (nblocks - 1)) / 15);
        uint64_t d[2];
        digest_words(bases + b * blk * 8, blk * 8, d);
        if (d[0] != bs.digest[2 * b] || d[1] != bs.digest[2 * b + 1]) return false;
    }
    return true;
}

// a resident copy that may hold bases[0, n): same address first, then any cached array (the same SRS vector re-loaded at
// another address: src/scaffold.rs:174 re-reads the params file for every proof).  Tables are built on the 2nd use.
static SetRef implicit_candidate_locked(const uint64_t* bases, size_t n) {
    const size_t nblocks = n / digest_block();
    for (int pass = 0; pass < 2; ++pass) {
        for (auto& sp : G.sets.all) {
            if (!sp->implicit || sp->n < n || (pass == 0) != (sp->host_ptr == (const void*)bases)) continue;
            if (!spot_check(*sp, bases, nblocks)) continue;
            SetRef hit = sp;
            hit->last_use = ++G.use_counter;
            if (++hit->uses == IMPLICIT_TABLES_AFTER_USES && hit->n_tables == 1) {
                SetRef with = build_tables(hit);
                if (with != hit) { sp = with; hit = with; }
            }
            return hit;
        }
    }
    return SetRef();
}

static int implicit_insert_locked(const uint64_t* bases, size_t n, SetRef* out) {
    // stale entries for this address (their contents no longer match, or they are shorter), then LRU beyond the budget
    std::vector<SetRef>& sets = G.sets.all;
    for (size_t i = 0; i < sets.size();) {
        if (sets[i]->implicit && sets[i]->host_ptr == (const void*)bases) sets.erase(sets.begin() + i);
        else ++i;
    }
    size_t total_b = 0, free_b = 0;
    cudaSetDevice(G.devs[0]->device);
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); total_b = (size_t)64 << 30; }
    const size_t budget = total_b / 2;
    for (;;) {
        size_t implicit = 0, bytes = 0, victim = (size_t)-1;
        for (size_t i = 0; i < sets.size(); ++i) {
            if (!sets[i]->implicit) continue;
            ++implicit;
            bytes += sets[i]->bytes_on(0);
            if (victim == (size_t)-1 || sets[i]->last_use < sets[victim]->last_use) victim = i;
        }
        if (victim == (size_t)-1 || (implicit < IMPLICIT_CACHE_MAX_SETS && bytes + n * 64 * 14 <= budget)) break;
        sets.erase(sets.begin() + victim);
    }
    SetRef bs;
    H2B_TRY(create_set(bases, n, n >= MULTI_DEVICE_MIN_POINTS, false, &bs));
    bs->implicit = true;
    bs->host_ptr = bases;
    bs->uses = 1;
    bs->refs = 0;
    const size_t nblocks = n / digest_block();
    bs->digest.resize(2 * nblocks);
    digest_blocks(bases, 0, nblocks, bs->digest.data(), nullptr);
    publish_new_locked(bs);
    G.implicit_uploads++;
    *out = bs;
    return H2B_OK;
}

// ---- running an MSM over a resident set --------------------------------------------------------------------------------------
static int msm_on_device(DeviceCtx& c, const uint64_t* scalars, const MsmBases& d_bases, size_t n, uint64_t* out_block /*28 x u64*/) {
    H2B_CUDA(cudaSetDevice(c.device));
    H2B_TRY(c.msm_scalars.reserve(n * 32 + 32));
    return msm_run_host(c, scalars, c.msm_scalars.p, d_bases, n, out_block);
}

// the devices an MSM over rows [offset, offset + n) runs on: {device, first scalar, scalars}; device == SIZE_MAX: any idle one
struct Piece { size_t d, lo, n; };
static std::vector<Piece> split_call(const BaseSet& bs, size_t offset, size_t n) {
    const size_t nd = G.devs.size();
    std::vector<Piece> pieces;
    if (bs.sharded) {
        for (size_t d = 0; d < nd; ++d) {
            const size_t a = offset > bs.lo[d] ? offset : bs.lo[d];
            const size_t b = offset + n < bs.lo[d] + bs.rows[d] ? offset + n : bs.lo[d] + bs.rows[d];
            if (a < b) pieces.push_back(Piece{d, a - offset, b - a});
        }
    } else if (nd == 1 || n < MULTI_DEVICE_MIN_POINTS) {
        pieces.push_back(Piece{(size_t)-1, 0, n});
    } else {
        for (size_t d = 0; d < nd; ++d) pieces.push_back(Piece{d, n * d / nd, n * (d + 1) / nd - n * d / nd});
    }
    return pieces;
}

int msm_host(const uint64_t* scalars, const BaseSet& bs, size_t offset, size_t n, uint64_t out_jac[12]) {
    const std::vector<Piece> pieces = split_call(bs, offset, n);
    if (pieces.size() == 1) {
        const Piece& p = pieces[0];
        std::unique_lock<std::mutex> lk;
        size_t d = p.d;
        DeviceCtx* c;
        if (d == (size_t)-1) c = pick_device(lk, &d);
        else { c = G.devs[d].get(); lk = std::unique_lock<std::mutex>(c->mu); }
        uint64_t block[28];
        H2B_TRY(msm_on_device(*c, scalars + 4 * p.lo, bases_of(bs, d, offset + p.lo), p.n, block));
        memcpy(out_jac, block, 96);
        return H2B_OK;
    }
    // point-range sharding: every piece is a complete Pippenger on its device; the partial sums are folded on device 0
    const size_t np = pieces.size();
    std::vector<uint64_t> blocks(28 * np);
    std::vector<size_t> devs, piece_on(G.devs.size());
    for (size_t i = 0; i < np; ++i) { devs.push_back(pieces[i].d); piece_on[pieces[i].d] = i; }
    H2B_TRY(on_devices(devs, [&](size_t d) -> int {
        const size_t i = piece_on[d];
        DeviceCtx& c = *G.devs[d];
        std::lock_guard<std::mutex> lk(c.mu);
        return msm_on_device(c, scalars + 4 * pieces[i].lo, bases_of(bs, d, offset + pieces[i].lo), pieces[i].n, &blocks[28 * i]);
    }));
    DeviceCtx& c0 = *G.devs[0];
    std::lock_guard<std::mutex> lk(c0.mu);
    H2B_CUDA(cudaSetDevice(c0.device));
    H2B_TRY(c0.msm_scalars.reserve(224 * np));
    H2B_TRY(c0.msm_out.reserve(256));
    H2B_CUDA(cudaMemcpyAsync(c0.msm_scalars.p, blocks.data(), 224 * np, cudaMemcpyHostToDevice, c0.stream));
    H2B_TRY(msm_sum_partials_run(c0, c0.msm_scalars.p, (uint32_t)np, c0.msm_out.p, c0.stream));
    H2B_CUDA(cudaMemcpyAsync(out_jac, c0.msm_out.p, 96, cudaMemcpyDeviceToHost, c0.stream));
    H2B_CUDA(cudaStreamSynchronize(c0.stream));
    return H2B_OK;
}

// best_multiexp over an array that is NOT resident: points and scalars are uploaded for this call only (verifier MSMs of a few
// dozen fresh points, odd-length prefixes).  No device allocation in steady state, nothing cached, nothing to go stale.
static int msm_direct(const uint64_t* scalars, const uint64_t* bases, size_t n, uint64_t out_jac[12]) {
    std::unique_lock<std::mutex> lk;
    DeviceCtx* c = pick_device(lk);
    H2B_CUDA(cudaSetDevice(c->device));
    H2B_TRY(c->msm_bases.reserve(n * 64 + 64));
    H2B_TRY(host_upload(*c, c->msm_bases.p, bases, n * 64, c->stream));
    MsmBases b;
    b.tables = c->msm_bases.p;
    b.stride = n;
    uint64_t block[28];
    H2B_TRY(msm_on_device(*c, scalars, b, n, block));
    memcpy(out_jac, block, 96);
    G.direct_calls++;
    return H2B_OK;
}

static void jac_identity(uint64_t out_jac[12]) {
    memset(out_jac, 0, 96);
    for (int i = 0; i < 4; ++i) out_jac[4 + i] = (uint64_t)FpParams<FQ>::ONE(2 * i) | ((uint64_t)FpParams<FQ>::ONE(2 * i + 1) << 32);
}

static int register_bases(const char* who, const uint64_t* bases, size_t n, bool sharded, uint64_t* handle) {
    H2B_TRY(require_init());
    if (!bases || !handle || n == 0) { set_error("%s: bad argument", who); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(G.mu);
    SetRef bs;
    H2B_TRY(create_set(bases, n, sharded, true, &bs));
    *handle = publish_new_locked(bs);
    return H2B_OK;
}

int registered_set(const char* who, uint64_t handle, size_t offset, size_t n, SetRef* out) {
    SetRef bs = G.sets.find(handle);
    if (!bs) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
    if (offset > bs->n || n > bs->n - offset) { set_error("%s: range [%zu, %zu) exceeds the registered set of %zu points", who, offset, offset + n, bs->n); return H2B_ERR_BAD_ARGUMENT; }
    *out = bs;
    return H2B_OK;
}

// ---- ONE NTT across the devices of the process (SURVEY.md section 8e, "one NTT across GPUs") ---------------------------------------
// Four-step transform of the n = R x C matrix a[i1 * C + i2] (R = 2^(log_n / 2) rows):
//   A. device d takes the columns i2 in [d C/D, (d+1) C/D) straight from the caller's array (one strided upload per device: D PCIe links
//      in parallel), transposes them, runs the C/D column transforms of length R (root w^C) and multiplies by w^(i2 k1);
//   B. the one exchange step: device e pulls, from every device, the k1 in [e R/D, (e+1) R/D) part of its rows (2-D peer copies over
//      NVLink: n/D^2 elements per pair);
//   C. device e transposes, runs its R/D row transforms of length C (root w^R), transposes back and writes a_hat[k1 + R k2] into the
//      caller's array (one strided download per device).
// Transposes are HBM-bound passes over n/D elements (tens of microseconds); the transforms are the single-device kernels in their
// strided-batch mode.  No collective: the exchange is D (D - 1) independent copies.
static bool ntt_multi_applicable(uint32_t log_n, uint32_t* log_d) {
    const size_t nd = G.devs.size();
    if (nd < 2 || (nd & (nd - 1))) return false;
    static int on = -1, min_log = -1;
    if (on < 0) on = env_int_or("H2B_NTT_MULTI", 1);
    if (min_log < 0) min_log = env_int_or("H2B_NTT_MULTI_MIN_LOG", 22);
    uint32_t ld = 0;
    while (((size_t)1 << ld) < nd) ++ld;
    if (!on || log_n < (uint32_t)min_log || log_n / 2 < ld || log_n < 2) return false;
    *log_d = ld;
    return true;
}

static int ntt_multi_device(uint64_t* a, const uint64_t omega[4], uint32_t log_n, uint32_t log_d) {
    const size_t D = (size_t)1 << log_d;
    const uint32_t r1 = log_n / 2, r2 = log_n - r1;
    const size_t R = (size_t)1 << r1, C = (size_t)1 << r2, Rd = R >> log_d, Cd = C >> log_d;
    const size_t slice = (size_t)32 << (log_n - log_d);
    std::vector<std::unique_lock<std::mutex>> locks;      // every device, in index order
    for (size_t d = 0; d < D; ++d) locks.emplace_back(G.devs[d]->mu);
    uint64_t roots[8];                                    // w^C (order R) | w^R (order C)
    {
        DeviceCtx& c0 = *G.devs[0];
        H2B_CUDA(cudaSetDevice(c0.device));
        H2B_TRY(c0.msm_out.reserve(256));
        H2B_TRY(ntt_root_powers_run(c0, omega, r2, r1, c0.msm_out.p, c0.stream));
        H2B_CUDA(cudaMemcpyAsync(roots, c0.msm_out.p, 64, cudaMemcpyDeviceToHost, c0.stream));
        H2B_CUDA(cudaStreamSynchronize(c0.stream));
    }
    const std::vector<size_t> devs = first_devices(D);
    H2B_TRY(on_devices(devs, [&](size_t d) -> int {
        DeviceCtx& c = *G.devs[d];
        H2B_CUDA(cudaSetDevice(c.device));
        H2B_TRY(c.ntt_io.reserve(slice));
        H2B_TRY(c.ntt_fs[0].reserve(slice));
        H2B_TRY(c.ntt_fs[1].reserve(slice));
        H2B_TRY(host_upload_2d(c, c.ntt_io.p, (const char*)a + d * Cd * 32, C * 32, Cd * 32, R, c.stream));          // R x Cd
        H2B_TRY(fr_transpose_run(c, c.ntt_io.p, c.ntt_fs[0].p, (uint32_t)R, (uint32_t)Cd, c.stream));                 // Cd x R
        H2B_TRY(ntt_run_strided(c, c.ntt_fs[0].p, Cd, R, roots, r1, c.stream));
        H2B_TRY(ntt_fourstep_twiddle_run(c, c.ntt_fs[0].p, (uint32_t)Cd, r1, (uint32_t)(d * Cd), omega, c.stream));
        H2B_CUDA(cudaStreamSynchronize(c.stream));
        return H2B_OK;
    }));
    return on_devices(devs, [&](size_t e) -> int {
        DeviceCtx& c = *G.devs[e];
        H2B_CUDA(cudaSetDevice(c.device));
        for (size_t k = 0; k < D; ++k) {                  // C x Rd, rows [d Cd, (d+1) Cd) from device d; every device starts with its own block
            const size_t d = (e + k) & (D - 1);
            H2B_CUDA(cudaMemcpy2DAsync((char*)c.ntt_io.p + d * Cd * Rd * 32, Rd * 32, (const char*)G.devs[d]->ntt_fs[0].p + e * Rd * 32, R * 32, Rd * 32, Cd,
                                       cudaMemcpyDefault, c.stream));
        }
        H2B_TRY(fr_transpose_run(c, c.ntt_io.p, c.ntt_fs[1].p, (uint32_t)C, (uint32_t)Rd, c.stream));                 // Rd x C
        H2B_TRY(ntt_run_strided(c, c.ntt_fs[1].p, Rd, C, roots + 4, r2, c.stream));
        H2B_TRY(fr_transpose_run(c, c.ntt_fs[1].p, c.ntt_io.p, (uint32_t)Rd, (uint32_t)C, c.stream));                 // C x Rd: [k2][k1]
        return host_download_2d(c, (char*)a + e * Rd * 32, R * 32, c.ntt_io.p, Rd * 32, C, c.stream);
    });
}

// columns of up to BATCH_COLUMN_MAX scalars are latency bound and share one kernel sequence per device (msm_run_batch): up to
// MSM_BATCH_MAX columns and 2^23 scalars per group; longer columns run one by one (they fill the GPU on their own)
static const size_t BATCH_GROUP_POINTS = (size_t)1 << 23;

}  // namespace h2b

using namespace h2b;

extern "C" {

int h2b_msm_bn254_g1(const uint64_t* scalars, const uint64_t* bases, size_t n, uint64_t out_jac[12]) {
    H2B_TRY(require_init());
    if (!out_jac || (n && (!scalars || !bases))) { set_error("h2b_msm_bn254_g1: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) { jac_identity(out_jac); return H2B_OK; }
    // Short arrays (verifier MSMs, openings of a few dozen points) and lengths that are not a whole number of digest blocks
    // are never cached: both arrays are uploaded for this call.
    if (!implicit_cache_enabled() || n < implicit_min_points() || n % digest_block() != 0) return msm_direct(scalars, bases, n, out_jac);
    const size_t nblocks = n / digest_block();
    for (int attempt = 0; attempt < 2; ++attempt) {
        SetRef set;
        bool fresh = false;
        {
            std::lock_guard<std::mutex> lk(G.mu);
            set = implicit_candidate_locked(bases, n);
            if (!set) { H2B_TRY(implicit_insert_locked(bases, n, &set)); fresh = true; }
        }
        if (fresh) return msm_host(scalars, *set, 0, n, out_jac);      // digests were taken from the very bytes that were uploaded
        // A resident copy passed the spot check.  The MSM runs on it while host threads verify EVERY block of the caller's
        // array against the digests taken at upload time; the result is only returned if all of them match (best_multiexp is a
        // pure function: an array mutated in place, or a freed Vec whose address was reused, must not see the old points).
        std::atomic<int> verdict{-1};
        std::thread verifier([&] { verdict = digest_blocks(bases, 0, nblocks, nullptr, set->digest.data()) ? 1 : 0; });
        const int rc = msm_host(scalars, *set, 0, n, out_jac);
        verifier.join();
        if (verdict == 1) { if (rc == H2B_OK) G.implicit_hits++; return rc; }
        G.implicit_stale++;
        std::lock_guard<std::mutex> lk(G.mu);
        if (set->host_ptr == (const void*)bases) G.sets.take_locked(set->handle);      // that address holds something else now
        // (a copy uploaded from another address stays: its own array may well be intact); second attempt: the spot check of the
        // remaining candidates runs again, and a miss uploads the array
    }
    return msm_direct(scalars, bases, n, out_jac);      // unreachable in practice: the array changed twice while we looked at it
}

int h2b_register_bases(const uint64_t* bases, size_t n, uint64_t* handle) {
    return register_bases("h2b_register_bases", bases, n, false, handle);
}

int h2b_register_bases_sharded(const uint64_t* bases, size_t n, uint64_t* handle) {
    return register_bases("h2b_register_bases_sharded", bases, n, true, handle);
}

int h2b_unregister_bases(uint64_t handle) {
    H2B_TRY(require_init());
    std::lock_guard<std::mutex> lk(G.mu);
    SetRef bs = G.sets.find_locked(handle);
    if (!bs || bs->implicit) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
    if (--bs->refs > 0) return H2B_OK;
    G.sets.take_locked(handle);      // calls still running on the set keep it alive until they return
    return H2B_OK;
}

int h2b_msm_bn254_g1_registered(const uint64_t* scalars, uint64_t handle, size_t offset, size_t n, uint64_t out_jac[12]) {
    H2B_TRY(require_init());
    if (!out_jac || (n && !scalars)) { set_error("h2b_msm_bn254_g1_registered: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs;
    H2B_TRY(registered_set("h2b_msm_bn254_g1_registered", handle, offset, n, &bs));
    if (n == 0) { jac_identity(out_jac); return H2B_OK; }
    return msm_host(scalars, *bs, offset, n, out_jac);
}

int h2b_ntt_bn254_fr(uint64_t* a, const uint64_t omega[4], uint32_t log_n) {
    H2B_TRY(require_init());
    if (!a || !omega) { set_error("h2b_ntt_bn254_fr: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n > 28) { set_error("h2b_ntt_bn254_fr: log_n = %u exceeds the two-adicity of Fr (28)", log_n); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n == 0) return H2B_OK;
    uint32_t log_d = 0;
    if (ntt_multi_applicable(log_n, &log_d)) return ntt_multi_device(a, omega, log_n, log_d);
    std::unique_lock<std::mutex> lk;
    DeviceCtx* c = pick_device(lk);
    H2B_CUDA(cudaSetDevice(c->device));
    const size_t bytes = (size_t)32 << log_n;
    H2B_TRY(c->ntt_io.reserve(bytes));
    H2B_TRY(host_upload(*c, c->ntt_io.p, a, bytes, c->stream));
    H2B_TRY(ntt_run(*c, c->ntt_io.p, omega, log_n, c->stream));
    return host_download(*c, a, c->ntt_io.p, bytes, c->stream);
}

int h2b_msm_bn254_g1_batch_registered(const uint64_t* const* scalars, const size_t* lens, size_t count, uint64_t handle, uint64_t* out_jac) {
    H2B_TRY(require_init());
    if (count == 0) return H2B_OK;
    if (!scalars || !lens || !out_jac) { set_error("h2b_msm_bn254_g1_batch_registered: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs;
    H2B_TRY(registered_set("h2b_msm_bn254_g1_batch_registered", handle, 0, 0, &bs));
    for (size_t j = 0; j < count; ++j) {
        if (lens[j] > bs->n) { set_error("column %zu: %zu scalars exceed the registered set of %zu points", j, lens[j], bs->n); return H2B_ERR_BAD_ARGUMENT; }
        if (lens[j] && !scalars[j]) { set_error("column %zu: null scalars", j); return H2B_ERR_BAD_ARGUMENT; }
    }
    if (bs->sharded) {
        // every column is split by point range over the devices that hold its rows
        for (size_t j = 0; j < count; ++j) {
            if (lens[j] == 0) jac_identity(out_jac + 12 * j);
            else H2B_TRY(msm_host(scalars[j], *bs, 0, lens[j], out_jac + 12 * j));
        }
        return H2B_OK;
    }
    // groups of columns; group g runs on device g mod D
    struct Group { std::vector<size_t> cols; };
    std::vector<Group> groups;
    static int env_batch = -1;
    if (env_batch < 0) env_batch = env_int_or("H2B_MSM_BATCH", 1);
    const size_t nd = G.devs.size();
    {
        const size_t group_cols = env_batch ? msm_batch_max() : 1;
        // spread the columns over the devices first, then batch what lands on one device
        std::vector<std::vector<size_t>> per_dev(nd);
        for (size_t j = 0; j < count; ++j) per_dev[j % nd].push_back(j);
        for (size_t d = 0; d < nd; ++d) {
            Group cur;
            size_t pts = 0;
            for (size_t j : per_dev[d]) {
                const bool solo = lens[j] > BATCH_COLUMN_MAX;
                if (!cur.cols.empty() && (solo || cur.cols.size() >= group_cols || pts + lens[j] > BATCH_GROUP_POINTS)) { groups.push_back(cur); cur = Group(); pts = 0; }
                cur.cols.push_back(j);
                pts += lens[j];
                if (solo) { groups.push_back(cur); cur = Group(); pts = 0; }
            }
            if (!cur.cols.empty()) groups.push_back(cur);
        }
    }
    // group -> device: the device its columns were dealt to
    std::vector<std::vector<size_t>> dev_groups(nd);
    for (size_t g = 0; g < groups.size(); ++g) dev_groups[groups[g].cols[0] % nd].push_back(g);
    auto run_device = [&](size_t d) -> int {
        DeviceCtx& c = *G.devs[d];
        for (size_t g : dev_groups[d]) {
            const std::vector<size_t>& cols = groups[g].cols;
            std::lock_guard<std::mutex> lk(c.mu);
            if (cols.size() == 1) {
                uint64_t block[28];
                H2B_TRY(msm_on_device(c, scalars[cols[0]], bases_of(*bs, d, 0), lens[cols[0]], block));
                memcpy(out_jac + 12 * cols[0], block, 96);
                continue;
            }
            H2B_CUDA(cudaSetDevice(c.device));
            std::vector<const void*> hp;
            std::vector<size_t> ln;
            size_t total = 0;
            for (size_t j : cols) { hp.push_back(scalars[j]); ln.push_back(lens[j]); total += lens[j]; }
            H2B_TRY(c.msm_scalars.reserve(total * 32 + 32));
            std::vector<uint64_t> blocks(28 * cols.size());
            H2B_TRY(msm_run_host_batch(c, hp.data(), ln.data(), (uint32_t)cols.size(), c.msm_scalars.p, bases_of(*bs, d, 0), blocks.data()));
            for (size_t i = 0; i < cols.size(); ++i) memcpy(out_jac + 12 * cols[i], &blocks[28 * i], 96);
        }
        return H2B_OK;
    };
    std::vector<size_t> busy;
    for (size_t d = 0; d < nd; ++d) if (!dev_groups[d].empty()) busy.push_back(d);
    return on_devices(busy, run_device);
}

int h2b_ntt_bn254_fr_batch(uint64_t* const* a, size_t count, const uint64_t omega[4], uint32_t log_n) {
    H2B_TRY(require_init());
    if (count == 0) return H2B_OK;
    if (!a || !omega) { set_error("h2b_ntt_bn254_fr_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n > 28) { set_error("h2b_ntt_bn254_fr_batch: log_n = %u exceeds the two-adicity of Fr (28)", log_n); return H2B_ERR_BAD_ARGUMENT; }
    for (size_t j = 0; j < count; ++j) if (!a[j]) { set_error("polynomial %zu: null pointer", j); return H2B_ERR_BAD_ARGUMENT; }
    if (log_n == 0) return H2B_OK;
    const size_t bytes = (size_t)32 << log_n;
    // polynomial j goes to device j mod D; what lands on one device is transformed in groups that share every pass launch
    const size_t nd = G.devs.size();
    size_t group = ntt_batch_max();
    while (group > 1 && group * bytes > ((size_t)1 << 31)) group >>= 1;
    auto run_device = [&](size_t d) -> int {
        DeviceCtx& c = *G.devs[d];
        std::vector<size_t> mine;
        for (size_t j = d; j < count; j += nd) mine.push_back(j);
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        for (size_t g0 = 0; g0 < mine.size(); g0 += group) {
            const size_t m = mine.size() - g0 < group ? mine.size() - g0 : group;
            H2B_TRY(c.ntt_io.reserve(bytes * m));
            std::vector<void*> ptrs(m);
            for (size_t i = 0; i < m; ++i) {
                ptrs[i] = (char*)c.ntt_io.p + bytes * i;
                H2B_TRY(host_upload(c, ptrs[i], a[mine[g0 + i]], bytes, c.stream, i == 0));
            }
            H2B_TRY(ntt_run_batch(c, ptrs.data(), m, omega, log_n, c.stream));
            for (size_t i = 0; i < m; ++i) H2B_TRY(host_download(c, a[mine[g0 + i]], ptrs[i], bytes, c.stream));
        }
        return H2B_OK;
    };
    return on_devices(first_devices(count < nd ? count : nd), run_device);
}

int h2b_set_msm_precomp(int spacing) {
    if (spacing < -1 || spacing == 1 || spacing > 24) { set_error("h2b_set_msm_precomp: spacing must be -1 (off), 0 (auto) or in [2, 24]"); return H2B_ERR_BAD_ARGUMENT; }
    g_table_policy = spacing;
    return H2B_OK;
}

int h2b_base_set_info(uint64_t handle, uint32_t* n_tables, uint32_t* spacing, uint64_t* device_bytes) {
    H2B_TRY(require_init());
    SetRef bs;
    H2B_TRY(registered_set("h2b_base_set_info", handle, 0, 0, &bs));
    if (n_tables) *n_tables = bs->n_tables;
    if (spacing) *spacing = bs->c0;
    if (device_bytes) { uint64_t m = 0; for (size_t d = 0; d < bs->dev.size(); ++d) m = bs->bytes_on(d) > m ? bs->bytes_on(d) : m; *device_bytes = m; }
    return H2B_OK;
}

int h2b_implicit_cache_stats(uint64_t out[6]) {
    H2B_TRY(require_init());
    if (!out) { set_error("h2b_implicit_cache_stats: null output"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(G.mu);
    uint64_t sets = 0, with_tables = 0;
    for (auto& sp : G.sets.all) if (sp->implicit) { ++sets; if (sp->n_tables > 1) ++with_tables; }
    out[0] = G.implicit_uploads; out[1] = G.implicit_hits; out[2] = G.implicit_stale; out[3] = G.direct_calls; out[4] = sets; out[5] = with_tables;
    return H2B_OK;
}

// One witness / product column through the three steps such a column takes in create_proof ([UP] plonk/prover.rs: commit_lagrange,
// EvaluationDomain::lagrange_to_coeff, EvaluationDomain::coeff_to_extended) with ONE upload and no intermediate round trip
// (SURVEY.md 8f rank 1: the call a patched prover.rs makes per column instead of three host-pointer drop-ins).
int h2b_column_pipeline(int device, const uint64_t* lagrange, uint64_t handle_g_lagrange, uint32_t k, uint32_t extended_k, const uint64_t omega_inv[4],
                        const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], uint64_t out_commitment_jac[12],
                        uint64_t* out_coeff, uint64_t* out_extended, void** d_extended) {
    SetRef bs;      // declared before the device lock: released after it
    const size_t d = (size_t)device;
    return on_device(device, [&]() -> int {
        if (!lagrange || !omega_inv || !ifft_divisor || !extended_omega || !zeta_powers || !out_commitment_jac) { set_error("h2b_column_pipeline: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(extended_k_check("h2b_column_pipeline", k, extended_k));
        const size_t n = (size_t)1 << k;
        H2B_TRY(registered_set("h2b_column_pipeline", handle_g_lagrange, 0, n, &bs));
        if (bs->lo[d] != 0 || bs->rows[d] < n) { set_error("h2b_column_pipeline: device %d does not hold rows [0, %zu) of the set (use a replicated registration)", device, n); return H2B_ERR_BAD_ARGUMENT; }
        return H2B_OK;
    }, [&](DeviceCtx& c) -> int {
        const size_t n = (size_t)1 << k, en = (size_t)1 << extended_k;
        const bool want_ext = out_extended || d_extended;
        void* d_ext = nullptr;
        cudaStream_t st = c.stream;
        H2B_TRY(c.ntt_io.reserve(n * 32));
        H2B_TRY(c.msm_out.reserve(256));
        if (want_ext) {
            if (d_extended) {
                H2B_TRY(dev_malloc(&d_ext, en * 32, "h2b_column_pipeline's extended column"));
            } else {
                H2B_TRY(c.col_ext.reserve(en * 32));
                d_ext = c.col_ext.p;
            }
        }
        int rc = host_upload(c, c.ntt_io.p, lagrange, n * 32, st);
        if (!rc) rc = msm_run(c, c.ntt_io.p, bases_of(*bs, d, 0), n, c.msm_out.p, false, st);
        if (!rc && cudaMemcpyAsync(out_commitment_jac, c.msm_out.p, 96, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = H2B_ERR_CUDA;
        if (!rc) rc = ntt_run(c, c.ntt_io.p, omega_inv, k, st);
        if (!rc) rc = ntt_scale_run(c, c.ntt_io.p, n, ifft_divisor, 1, st);
        if (!rc && want_ext) {
            if (cudaMemcpyAsync(d_ext, c.ntt_io.p, n * 32, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = H2B_ERR_CUDA;
            if (!rc) rc = ntt_scale_run(c, d_ext, n, zeta_powers, 3, st);
            if (!rc && en > n && cudaMemsetAsync((char*)d_ext + n * 32, 0, (en - n) * 32, st) != cudaSuccess) rc = H2B_ERR_CUDA;
            if (!rc) rc = ntt_run(c, d_ext, extended_omega, extended_k, st);
        }
        if (!rc && out_coeff) rc = host_download(c, out_coeff, c.ntt_io.p, n * 32, st);
        if (!rc && out_extended) rc = host_download(c, out_extended, d_ext, en * 32, st);
        if (!rc && cudaStreamSynchronize(st) != cudaSuccess) { set_error("h2b_column_pipeline: %s", cudaGetErrorString(cudaGetLastError())); rc = H2B_ERR_CUDA; }
        if (rc) { if (d_extended && d_ext) cudaFree(d_ext); if (rc == H2B_ERR_CUDA && !*get_error()) set_error("h2b_column_pipeline: CUDA error"); return rc; }
        if (d_extended) *d_extended = d_ext;
        return H2B_OK;
    });
}

}  // extern "C"
