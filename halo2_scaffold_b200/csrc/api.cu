// C ABI of libh2b200 (declared in include/h2b200.h): lifecycle, host-pointer drop-ins for
// best_multiexp / best_fft with device-resident SRS caching and point-range sharding across the
// GPUs of one box, device-pointer entry points, diagnostics.
#include <atomic>
#include <memory>
#include <thread>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/h2b200.h"
#include "common.h"

struct ResidentPk;   // a proving key held on the devices (h2b_pk_create)
struct ShplonkSession;   // a multi-point opening between its two commitments (h2b_shplonk_begin)

namespace h2b {

unsigned long long g_launch_count = 0;
static thread_local std::string t_error;
void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_error = buf;
}
const char* get_error() { return t_error.c_str(); }

// ---- resident point sets --------------------------------------------------------------------------------------------
// An SRS vector (or any base array) resident in device memory, with or without its window tables (msm.cu step 0).
//   replicated: every device holds all n rows  -> any column can run on any device (round-robin columns, SURVEY.md 8e rows 2-3)
//   sharded   : device d holds rows [lo[d], lo[d] + rows[d]) only -> one MSM split by point range (8e row 1) at 1/D of the
//               memory and of the registration time
// Sets are immutable once published and handed out as shared_ptr: a call keeps its set alive while it runs, whatever
// eviction, table builds or h2b_unregister_bases do meanwhile; device memory is released when the last holder lets go.
struct BaseSet {
    uint64_t handle = 0;
    bool implicit = false;            // created by h2b_msm_bn254_g1's cache (not by h2b_register_bases / h2b_srs_read)
    const void* host_ptr = nullptr;   // implicit sets: where the caller's array was when it was uploaded (a hint only)
    size_t n = 0;
    std::vector<uint64_t> digest;     // implicit sets: 128-bit digest of every block of digest_block() points of the uploaded array
    uint64_t last_use = 0, uses = 0;
    uint32_t n_tables = 1;            // 1: points only;  > 1: table j = 2^(c0*j) * P
    uint32_t c0 = 0;
    bool sharded = false;
    std::vector<int> ordinal;         // CUDA ordinal of device d
    std::vector<void*> dev;           // per device: n_tables x rows[d] x 64 bytes
    std::vector<size_t> lo, rows;
    int refs = 1;                     // API references (h2b_register_bases / h2b_srs_read hand-outs); guarded by G.mu
    ~BaseSet() {
        for (size_t d = 0; d < dev.size(); ++d)
            if (dev[d]) { cudaSetDevice(ordinal[d]); cudaFree(dev[d]); }
        cudaGetLastError();
    }
    size_t bytes_on(size_t d) const { return dev[d] ? (size_t)n_tables * rows[d] * 64 : 0; }
};
typedef std::shared_ptr<BaseSet> SetRef;

// files h2b_srs_read has already decoded: the reference re-reads params/kzg_bn254_{k}.srs for every proof
// (src/scaffold.rs:174); a second read of an unchanged file hands out the resident base sets again
struct SrsCacheEntry {
    std::string path;
    int format = 0;
    long long size = 0, mtime_ns = 0;
    uint32_t k = 0;
    uint64_t handle_g = 0, handle_g_lagrange = 0;
    std::vector<unsigned char> g2;
};

struct Global {
    std::mutex mu;
    std::vector<std::unique_ptr<DeviceCtx>> devs;
    std::vector<SetRef> sets;
    std::vector<std::shared_ptr<::ResidentPk>> pks;
    std::vector<std::shared_ptr<::ShplonkSession>> sessions;
    std::vector<SrsCacheEntry> srs_cache;
    uint64_t next_handle = 1;
    uint64_t use_counter = 0;
    std::atomic<unsigned> rr{0};
    std::atomic<unsigned long long> implicit_uploads{0}, implicit_hits{0}, implicit_stale{0}, direct_calls{0};
};
static Global G;

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

static int require_init() {
    if (G.devs.empty()) { set_error("h2b200 is not initialised (call h2b_init)"); return H2B_ERR_NOT_INITIALIZED; }
    return H2B_OK;
}
static int get_ctx(int device, DeviceCtx** out) {
    H2B_TRY(require_init());
    if (device < 0 || (size_t)device >= G.devs.size()) { set_error("device index %d out of range (have %zu)", device, G.devs.size()); return H2B_ERR_BAD_ARGUMENT; }
    *out = G.devs[device].get();
    H2B_CUDA(cudaSetDevice((*out)->device));
    return H2B_OK;
}

static int init_devices(const std::vector<int>& ordinals) {
    std::lock_guard<std::mutex> lk(G.mu);
    if (!G.devs.empty()) return H2B_OK;
    for (int ord : ordinals) {
        std::unique_ptr<DeviceCtx> c(new DeviceCtx());
        c->device = ord;
        H2B_CUDA(cudaSetDevice(ord));
        cudaDeviceProp prop;
        H2B_CUDA(cudaGetDeviceProperties(&prop, ord));
#ifndef H2B_EMU
        if (prop.major < 10) { set_error("device %d (%s, sm_%d%d) is not a Blackwell-class GPU; this library only ships sm_100a code", ord, prop.name, prop.major, prop.minor); G.devs.clear(); return H2B_ERR_NO_DEVICE; }
#endif
        c->sm_count = prop.multiProcessorCount;
        H2B_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        G.devs.push_back(std::move(c));
    }
    // peer access between every pair (NVLink / NVSwitch): table all-gathers and peer copies of decoded SRS vectors go direct
    for (size_t a = 0; a < G.devs.size(); ++a) {
        cudaSetDevice(G.devs[a]->device);
        for (size_t b = 0; b < G.devs.size(); ++b) {
            if (a == b) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, G.devs[a]->device, G.devs[b]->device) == cudaSuccess && can) cudaDeviceEnablePeerAccess(G.devs[b]->device, 0);
        }
    }
    cudaGetLastError();      // "already enabled" is not an error
    return H2B_OK;
}

// pick a device for a single-device call: round robin, preferring one that is idle
static DeviceCtx* pick_device(std::unique_lock<std::mutex>& lock_out, size_t* index = nullptr) {
    size_t nd = G.devs.size();
    unsigned start = G.rr.fetch_add(1);
    for (size_t k = 0; k < nd; ++k) {
        DeviceCtx* c = G.devs[(start + k) % nd].get();
        std::unique_lock<std::mutex> lk(c->mu, std::try_to_lock);
        if (lk.owns_lock()) { lock_out = std::move(lk); if (index) *index = (start + k) % nd; return c; }
    }
    DeviceCtx* c = G.devs[start % nd].get();
    lock_out = std::unique_lock<std::mutex>(c->mu);
    if (index) *index = start % nd;
    return c;
}

// fn(d) for every device index d in `devs`: on the calling thread when there is one, on one thread per device otherwise.  Returns
// the first failure in list order, its message prefixed with "device d: ".
static int on_devices(const std::vector<size_t>& devs, const std::function<int(size_t)>& fn) {
    const size_t m = devs.size();
    std::vector<int> rcs(m, 0);
    std::vector<std::string> errs(m);
    auto run = [&](size_t i) { rcs[i] = fn(devs[i]); if (rcs[i]) errs[i] = get_error(); };
    if (m == 1) {
        run(0);
    } else {
        std::vector<std::thread> th;
        for (size_t i = 0; i < m; ++i) th.emplace_back(run, i);
        for (auto& t : th) t.join();
    }
    for (size_t i = 0; i < m; ++i) if (rcs[i]) { set_error("device %zu: %s", devs[i], errs[i].c_str()); return rcs[i]; }
    return H2B_OK;
}
static std::vector<size_t> first_devices(size_t m) {
    std::vector<size_t> devs(m);
    for (size_t d = 0; d < m; ++d) devs[d] = d;
    return devs;
}

// every device allocation of this file.  A failed cudaMalloc stays the thread's last error, which the next launch check on this
// thread would report as its own: it is cleared here.
static int dev_malloc(void** p, size_t bytes, const char* what) {
    const cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) return H2B_OK;
    cudaGetLastError();
    *p = nullptr;
    set_error("cudaMalloc of %zu bytes for %s failed: %s", bytes, what, cudaGetErrorString(e));
    return H2B_ERR_OOM;
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

static SetRef find_set_locked(uint64_t handle) {
    for (auto& sp : G.sets) if (sp->handle == handle) return sp;
    return SetRef();
}
static SetRef find_set(uint64_t handle) {
    std::lock_guard<std::mutex> lk(G.mu);
    return find_set_locked(handle);
}
// hands a new set out under a fresh handle.  Caller holds G.mu.
static uint64_t publish_new_locked(const SetRef& bs) {
    bs->handle = G.next_handle++;
    bs->last_use = ++G.use_counter;
    G.sets.push_back(bs);
    return bs->handle;
}
static void drop_locked(uint64_t handle) {
    for (size_t i = 0; i < G.sets.size(); ++i) if (G.sets[i]->handle == handle) { G.sets.erase(G.sets.begin() + i); return; }
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
        for (auto& sp : G.sets) {
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
    for (size_t i = 0; i < G.sets.size();) {
        if (G.sets[i]->implicit && G.sets[i]->host_ptr == (const void*)bases) G.sets.erase(G.sets.begin() + i);
        else ++i;
    }
    size_t total_b = 0, free_b = 0;
    cudaSetDevice(G.devs[0]->device);
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); total_b = (size_t)64 << 30; }
    const size_t budget = total_b / 2;
    for (;;) {
        size_t implicit = 0, bytes = 0, victim = (size_t)-1;
        for (size_t i = 0; i < G.sets.size(); ++i) {
            if (!G.sets[i]->implicit) continue;
            ++implicit;
            bytes += G.sets[i]->bytes_on(0);
            if (victim == (size_t)-1 || G.sets[i]->last_use < G.sets[victim]->last_use) victim = i;
        }
        if (victim == (size_t)-1 || (implicit < IMPLICIT_CACHE_MAX_SETS && bytes + n * 64 * 14 <= budget)) break;
        G.sets.erase(G.sets.begin() + victim);
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
static MsmBases bases_of(const BaseSet& bs, size_t d, size_t row /* global row of the first point */) {
    MsmBases b;
    b.tables = bs.dev[d];
    b.n_tables = bs.n_tables;
    b.c0 = bs.c0;
    b.stride = bs.rows[d];
    b.row0 = row - bs.lo[d];
    return b;
}

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

static int msm_host(const uint64_t* scalars, const BaseSet& bs, size_t offset, size_t n, uint64_t out_jac[12]) {
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

}  // namespace h2b

using namespace h2b;

extern "C" {

int h2b_init(int n_devices) {
    if (!G.devs.empty()) return H2B_OK;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        set_error("no usable CUDA device (%s); h2b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return H2B_ERR_NO_DEVICE;
    }
    if (n_devices < 0 || n_devices > count) { set_error("h2b_init(%d): only %d device(s) visible", n_devices, count); return H2B_ERR_BAD_ARGUMENT; }
    if (n_devices == 0) n_devices = count;
    std::vector<int> ords;
    for (int i = 0; i < n_devices; ++i) ords.push_back(i);
    return init_devices(ords);
}

int h2b_init_device(int device) {
    if (!G.devs.empty()) return H2B_OK;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        set_error("no usable CUDA device (%s); h2b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return H2B_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) { set_error("h2b_init_device(%d): only %d device(s) visible", device, count); return H2B_ERR_BAD_ARGUMENT; }
    return init_devices(std::vector<int>{device});
}

void h2b_shutdown(void) {
    std::lock_guard<std::mutex> lk(G.mu);
    G.sets.clear();      // device memory goes when the last holder lets go (now, unless a call is still in flight)
    G.pks.clear();
    G.sessions.clear();
    G.srs_cache.clear();
    for (auto& c : G.devs) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        ntt_release(*c);
        msm_release(*c);
        stager_release(*c);
        c->msm_scalars.release();
        c->msm_out.release();
        c->msm_bases.release();
        c->col_ext.release();
        c->scan_scratch.release();
        evaluate_release(*c);
        c->srs_status.release();
        c->lookup_scratch.release();
        c->srs_io.release();
        c->gen_table.release();
        c->gen_scratch.release();
        c->open_scratch.release();
        c->open_tables.release();
        for (cudaEvent_t e : c->copy_events) cudaEventDestroy(e);
        c->copy_events.clear();
        if (c->copy_stream) { cudaStreamDestroy(c->copy_stream); c->copy_stream = nullptr; }
        cudaStreamDestroy(c->stream);
    }
    G.devs.clear();
}

int h2b_device_count(void) { return (int)G.devs.size(); }
const char* h2b_last_error(void) { return get_error(); }
const char* h2b_version(void) {
#ifdef H2B_EMU
    return "h2b200 0.1 (kernel-logic emulator build: NOT a product library)";
#else
    return "h2b200 0.1 (CUDA sm_100a)";
#endif
}
int h2b_is_emulator(void) {
#ifdef H2B_EMU
    return 1;
#else
    return 0;
#endif
}

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
        if (set->host_ptr == (const void*)bases) drop_locked(set->handle);      // that address holds something else now
        // (a copy uploaded from another address stays: its own array may well be intact); second attempt: the spot check of the
        // remaining candidates runs again, and a miss uploads the array
    }
    return msm_direct(scalars, bases, n, out_jac);      // unreachable in practice: the array changed twice while we looked at it
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

int h2b_register_bases(const uint64_t* bases, size_t n, uint64_t* handle) {
    return register_bases("h2b_register_bases", bases, n, false, handle);
}

int h2b_register_bases_sharded(const uint64_t* bases, size_t n, uint64_t* handle) {
    return register_bases("h2b_register_bases_sharded", bases, n, true, handle);
}

int h2b_unregister_bases(uint64_t handle) {
    H2B_TRY(require_init());
    std::lock_guard<std::mutex> lk(G.mu);
    SetRef bs = find_set_locked(handle);
    if (!bs || bs->implicit) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
    if (--bs->refs > 0) return H2B_OK;
    drop_locked(handle);      // calls still running on the set keep it alive until they return
    return H2B_OK;
}

static int registered_set(const char* who, uint64_t handle, size_t offset, size_t n, SetRef* out) {
    SetRef bs = find_set(handle);
    if (!bs) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
    if (offset > bs->n || n > bs->n - offset) { set_error("%s: range [%zu, %zu) exceeds the registered set of %zu points", who, offset, offset + n, bs->n); return H2B_ERR_BAD_ARGUMENT; }
    *out = bs;
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

// columns short enough to be latency bound share one kernel sequence per device (msm_run_batch): up to MSM_BATCH_MAX columns
// and 2^23 scalars per group; longer columns run one by one (they fill the GPU on their own)
static const size_t BATCH_GROUP_POINTS = (size_t)1 << 23;
static const size_t BATCH_COLUMN_MAX = (size_t)1 << 21;

int h2b_msm_bn254_g1_batch_registered(const uint64_t* const* scalars, const size_t* lens, size_t count, uint64_t handle, uint64_t* out_jac) {
    H2B_TRY(require_init());
    if (count == 0) return H2B_OK;
    if (!scalars || !lens || !out_jac) { set_error("h2b_msm_bn254_g1_batch_registered: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs = find_set(handle);
    if (!bs) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
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

int h2b_ntt_bn254_fr_dev_batch(int device, void* const* d_polys, size_t count, const uint64_t omega[4], uint32_t log_n, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (count == 0) return H2B_OK;
    if (!d_polys || !omega) { set_error("h2b_ntt_bn254_fr_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return ntt_run_batch(*c, d_polys, count, omega, log_n, (cudaStream_t)stream);
}

int h2b_ntt_bn254_fr_dev(int device, void* d_a, const uint64_t omega[4], uint32_t log_n, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!omega) { set_error("h2b_ntt_bn254_fr_dev: null omega"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return ntt_run(*c, d_a, omega, log_n, (cudaStream_t)stream);
}

int h2b_msm_bn254_g1_dev(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_jac, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_out_jac) { set_error("h2b_msm_bn254_g1_dev: null output"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    MsmBases b;
    b.tables = d_bases;
    b.stride = n;
    return msm_run(*c, d_scalars, b, n, d_out_jac, false, (cudaStream_t)stream);
}

int h2b_msm_bn254_g1_dev_partial(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_block, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_out_block) { set_error("h2b_msm_bn254_g1_dev_partial: null output"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    MsmBases b;
    b.tables = d_bases;
    b.stride = n;
    return msm_run(*c, d_scalars, b, n, d_out_block, true, (cudaStream_t)stream);
}

int h2b_msm_bn254_g1_dev_registered(int device, const void* d_scalars, uint64_t handle, size_t offset, size_t n, void* d_out_block, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_out_block) { set_error("h2b_msm_bn254_g1_dev_registered: null output"); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs;      // declared before the device lock: released after it
    H2B_TRY(registered_set("h2b_msm_bn254_g1_dev_registered", handle, offset, n, &bs));
    const size_t d = (size_t)device;
    if (n && (offset < bs->lo[d] || offset + n > bs->lo[d] + bs->rows[d])) {
        set_error("h2b_msm_bn254_g1_dev_registered: device %d holds rows [%zu, %zu) of this sharded set, not [%zu, %zu)", device, bs->lo[d], bs->lo[d] + bs->rows[d], offset, offset + n);
        return H2B_ERR_BAD_ARGUMENT;
    }
    std::lock_guard<std::mutex> lk(c->mu);
    // asynchronous: the set must stay registered until the caller has synchronised `stream`
    return msm_run(*c, d_scalars, bases_of(*bs, d, offset), n, d_out_block, true, (cudaStream_t)stream);
}

int h2b_msm_bn254_g1_dev_batch_registered(int device, const void* const* d_scalars, const size_t* lens, size_t count, uint64_t handle, void* d_out_blocks, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (count == 0) return H2B_OK;
    if (!d_scalars || !lens || !d_out_blocks) { set_error("h2b_msm_bn254_g1_dev_batch_registered: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs = find_set(handle);
    if (!bs) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
    const size_t d = (size_t)device;
    size_t n_max = 0;
    for (size_t j = 0; j < count; ++j) n_max = lens[j] > n_max ? lens[j] : n_max;
    if (bs->lo[d] != 0 || n_max > bs->rows[d]) { set_error("h2b_msm_bn254_g1_dev_batch_registered: device %d does not hold rows [0, %zu) of the set", device, n_max); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    for (size_t j0 = 0; j0 < count; j0 += msm_batch_max()) {
        const size_t m = count - j0 < msm_batch_max() ? count - j0 : msm_batch_max();
        H2B_TRY(msm_run_batch(*c, d_scalars + j0, lens + j0, (uint32_t)m, bases_of(*bs, d, 0), (char*)d_out_blocks + 224 * j0, (cudaStream_t)stream));
    }
    return H2B_OK;
}

int h2b_set_msm_precomp(int spacing) {
    if (spacing < -1 || spacing == 1 || spacing > 24) { set_error("h2b_set_msm_precomp: spacing must be -1 (off), 0 (auto) or in [2, 24]"); return H2B_ERR_BAD_ARGUMENT; }
    g_table_policy = spacing;
    return H2B_OK;
}

int h2b_base_set_info(uint64_t handle, uint32_t* n_tables, uint32_t* spacing, uint64_t* device_bytes) {
    H2B_TRY(require_init());
    SetRef bs = find_set(handle);
    if (!bs) { set_error("unknown base-set handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_HANDLE; }
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
    for (auto& sp : G.sets) if (sp->implicit) { ++sets; if (sp->n_tables > 1) ++with_tables; }
    out[0] = G.implicit_uploads; out[1] = G.implicit_hits; out[2] = G.implicit_stale; out[3] = G.direct_calls; out[4] = sets; out[5] = with_tables;
    return H2B_OK;
}

int h2b_msm_fold_partials(int device, const uint64_t* host_blocks, size_t count, uint64_t out_jac[12]) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!host_blocks || !out_jac || count == 0 || count > 4096) { set_error("h2b_msm_fold_partials: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_TRY(c->msm_scalars.reserve(224 * count));
    H2B_TRY(c->msm_out.reserve(256));
    H2B_CUDA(cudaMemcpyAsync(c->msm_scalars.p, host_blocks, 224 * count, cudaMemcpyHostToDevice, c->stream));
    H2B_TRY(msm_sum_partials_run(*c, c->msm_scalars.p, (uint32_t)count, c->msm_out.p, c->stream));
    H2B_CUDA(cudaMemcpyAsync(out_jac, c->msm_out.p, 96, cudaMemcpyDeviceToHost, c->stream));
    H2B_CUDA(cudaStreamSynchronize(c->stream));
    return H2B_OK;
}

int h2b_msm_fold_partials_dev(int device, const void* d_blocks, size_t count, void* d_out_jac, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_blocks || !d_out_jac || count == 0 || count > 4096) { set_error("h2b_msm_fold_partials_dev: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
    return msm_sum_partials_run(*c, d_blocks, (uint32_t)count, d_out_jac, (cudaStream_t)stream);
}

int h2b_fr_scale_dev(int device, void* d_a, size_t n, const uint64_t* factors, int count, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!factors || (n && !d_a)) { set_error("h2b_fr_scale_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    return ntt_scale_run(*c, d_a, n, factors, count, (cudaStream_t)stream);
}

// ---- EvaluationDomain on the device ([UP] halo2_proofs/src/poly/domain.rs; SURVEY.md row a6) --------------------------
// The column stays in device memory between the scaling, padding and transform steps of each conversion; the constants
// (omega, divisors, zeta) are the caller's: EvaluationDomain::new computes them once per domain on the host.
int h2b_lagrange_to_coeff_dev(int device, void* d_a, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_a || !omega_inv || !ifft_divisor) { set_error("h2b_lagrange_to_coeff_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_TRY(ntt_run(*c, d_a, omega_inv, k, (cudaStream_t)stream));
    return ntt_scale_run(*c, d_a, (size_t)1 << k, ifft_divisor, 1, (cudaStream_t)stream);
}

int h2b_coeff_to_extended_dev(int device, void* d_a, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                              void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_a || !extended_omega || !zeta_powers) { set_error("h2b_coeff_to_extended_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (extended_k < k || extended_k > 28) { set_error("h2b_coeff_to_extended_dev: need k <= extended_k <= 28"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t n = (size_t)1 << k, en = (size_t)1 << extended_k;
    H2B_TRY(ntt_scale_run(*c, d_a, n, zeta_powers, 3, (cudaStream_t)stream));                         // a[i] *= zeta^(i mod 3)
    if (en > n) H2B_CUDA(cudaMemsetAsync((char*)d_a + n * 32, 0, (en - n) * 32, (cudaStream_t)stream));   // zero-pad
    return ntt_run(*c, d_a, extended_omega, extended_k, (cudaStream_t)stream);
}

// The two conversions every witness / product column goes through, for `count` columns at once: the (i)NTT passes and the scaling
// are launched once for the whole batch (polynomial index in blockIdx.y).  d_cols: host array of device pointers.
int h2b_lagrange_to_coeff_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4],
                                    void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (count == 0) return H2B_OK;
    if (!d_cols || !omega_inv || !ifft_divisor) { set_error("h2b_lagrange_to_coeff_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return lagrange_to_coeff_batch_run(*c, d_cols, count, k, omega_inv, ifft_divisor, (cudaStream_t)stream);
}

int h2b_coeff_to_extended_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4],
                                    const uint64_t zeta_powers[12], void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (count == 0) return H2B_OK;
    if (!d_cols || !extended_omega || !zeta_powers) { set_error("h2b_coeff_to_extended_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (extended_k < k || extended_k > 28) { set_error("h2b_coeff_to_extended_dev_batch: need k <= extended_k <= 28"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return coeff_to_extended_batch_run(*c, d_cols, count, k, extended_k, extended_omega, zeta_powers, (cudaStream_t)stream);
}

// One witness / product column through the three steps such a column takes in create_proof ([UP] plonk/prover.rs: commit_lagrange,
// EvaluationDomain::lagrange_to_coeff, EvaluationDomain::coeff_to_extended) with ONE upload and no intermediate round trip
// (SURVEY.md 8f rank 1: the call a patched prover.rs makes per column instead of three host-pointer drop-ins).
int h2b_column_pipeline(int device, const uint64_t* lagrange, uint64_t handle_g_lagrange, uint32_t k, uint32_t extended_k, const uint64_t omega_inv[4],
                        const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], uint64_t out_commitment_jac[12],
                        uint64_t* out_coeff, uint64_t* out_extended, void** d_extended) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!lagrange || !omega_inv || !ifft_divisor || !extended_omega || !zeta_powers || !out_commitment_jac) { set_error("h2b_column_pipeline: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (k > 28 || extended_k < k || extended_k > 28) { set_error("h2b_column_pipeline: need k <= extended_k <= 28"); return H2B_ERR_BAD_ARGUMENT; }
    const size_t n = (size_t)1 << k, en = (size_t)1 << extended_k;
    SetRef bs;
    H2B_TRY(registered_set("h2b_column_pipeline", handle_g_lagrange, 0, n, &bs));
    const size_t d = (size_t)device;
    if (bs->lo[d] != 0 || bs->rows[d] < n) { set_error("h2b_column_pipeline: device %d does not hold rows [0, %zu) of the set (use a replicated registration)", device, n); return H2B_ERR_BAD_ARGUMENT; }
    const bool want_ext = out_extended || d_extended;
    void* d_ext = nullptr;
    std::lock_guard<std::mutex> lk(c->mu);
    cudaStream_t st = c->stream;
    H2B_TRY(c->ntt_io.reserve(n * 32));
    H2B_TRY(c->msm_out.reserve(256));
    if (want_ext) {
        if (d_extended) {
            H2B_TRY(dev_malloc(&d_ext, en * 32, "h2b_column_pipeline's extended column"));
        } else {
            H2B_TRY(c->col_ext.reserve(en * 32));
            d_ext = c->col_ext.p;
        }
    }
    int rc = host_upload(*c, c->ntt_io.p, lagrange, n * 32, st);
    if (!rc) rc = msm_run(*c, c->ntt_io.p, bases_of(*bs, d, 0), n, c->msm_out.p, false, st);
    if (!rc && cudaMemcpyAsync(out_commitment_jac, c->msm_out.p, 96, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = H2B_ERR_CUDA;
    if (!rc) rc = ntt_run(*c, c->ntt_io.p, omega_inv, k, st);
    if (!rc) rc = ntt_scale_run(*c, c->ntt_io.p, n, ifft_divisor, 1, st);
    if (!rc && want_ext) {
        if (cudaMemcpyAsync(d_ext, c->ntt_io.p, n * 32, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = H2B_ERR_CUDA;
        if (!rc) rc = ntt_scale_run(*c, d_ext, n, zeta_powers, 3, st);
        if (!rc && en > n && cudaMemsetAsync((char*)d_ext + n * 32, 0, (en - n) * 32, st) != cudaSuccess) rc = H2B_ERR_CUDA;
        if (!rc) rc = ntt_run(*c, d_ext, extended_omega, extended_k, st);
    }
    if (!rc && out_coeff) rc = host_download(*c, out_coeff, c->ntt_io.p, n * 32, st);
    if (!rc && out_extended) rc = host_download(*c, out_extended, d_ext, en * 32, st);
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess) { set_error("h2b_column_pipeline: %s", cudaGetErrorString(cudaGetLastError())); rc = H2B_ERR_CUDA; }
    if (rc) { if (d_extended && d_ext) cudaFree(d_ext); if (rc == H2B_ERR_CUDA && !*get_error()) set_error("h2b_column_pipeline: CUDA error"); return rc; }
    if (d_extended) *d_extended = d_ext;
    return H2B_OK;
}

int h2b_extended_to_coeff_dev(int device, void* d_a, uint32_t extended_k, const uint64_t extended_omega_inv[4], const uint64_t factors[12], void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_a || !extended_omega_inv || !factors) { set_error("h2b_extended_to_coeff_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_TRY(ntt_run(*c, d_a, extended_omega_inv, extended_k, (cudaStream_t)stream));
    // factors[j] = extended_ifft_divisor * (1, zeta^-1, zeta^-2)[j]: one pass undoes the scaling and the coset
    return ntt_scale_run(*c, d_a, (size_t)1 << extended_k, factors, 3, (cudaStream_t)stream);
}

// ---- grand-product building blocks (SURVEY.md 8f rank 3) ---------------------------------------------------------------
int h2b_fr_batch_invert_dev(int device, void* d_a, size_t n, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return fr_batch_invert_run(*c, d_a, n, (cudaStream_t)stream);
}

int h2b_fr_prefix_product_dev(int device, const void* d_in, void* d_out, size_t n, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return fr_prefix_product_run(*c, d_in, d_out, n, (cudaStream_t)stream);
}

int h2b_fr_eval_polynomial_dev(int device, const void* d_coeffs, size_t n, const uint64_t x[4], void* d_out, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return fr_eval_polynomial_run(*c, d_coeffs, n, x, d_out, (cudaStream_t)stream);
}

int h2b_fr_kate_division_dev(int device, const void* d_a, size_t n, const uint64_t b[4], void* d_q, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return fr_kate_division_run(*c, d_a, n, b, d_q, (cudaStream_t)stream);
}

int h2b_fr_lincomb_dev(int device, const void* const* d_cols, const uint64_t* coeffs, uint32_t m, size_t n, void* d_out, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    return fr_lincomb_run(*c, d_cols, coeffs, m, n, d_out, (cudaStream_t)stream);
}

int h2b_fr_transpose_dev(int device, const void* d_in, void* d_out, uint32_t rows, uint32_t cols, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if ((rows && cols) && (!d_in || !d_out || d_in == d_out)) { set_error("h2b_fr_transpose_dev: null or aliased buffers"); return H2B_ERR_BAD_ARGUMENT; }
    return fr_transpose_run(*c, d_in, d_out, rows, cols, (cudaStream_t)stream);
}

int h2b_permutation_product_dev(int device, const void* const* d_values, const void* const* d_permutations, uint32_t n_columns, size_t n,
                                const uint64_t beta[4], const uint64_t gamma[4], const uint64_t delta[4], const uint64_t deltaomega[4], const uint64_t omega[4],
                                const uint64_t last_z[4], void* d_z, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return permutation_product_run(*c, d_values, d_permutations, n_columns, n, beta, gamma, delta, deltaomega, omega, last_z, d_z, (cudaStream_t)stream);
}

int h2b_lookup_product_dev(int device, const void* d_compressed_input, const void* d_compressed_table, const void* d_permuted_input,
                           const void* d_permuted_table, size_t n, const uint64_t beta[4], const uint64_t gamma[4], void* d_z, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return lookup_product_run(*c, d_compressed_input, d_compressed_table, d_permuted_input, d_permuted_table, n, beta, gamma, d_z, (cudaStream_t)stream);
}

int h2b_lookup_permute_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                           void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return lookup_permute_run(*c, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, nullptr, (cudaStream_t)stream);
}

int h2b_lookup_permute_async_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                                 void* d_status, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_status) { set_error("h2b_lookup_permute_async_dev: null status word"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return lookup_permute_run(*c, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, d_status, (cudaStream_t)stream);
}

// ---- SRS on-disk format (SURVEY.md 8f rank 4) -----------------------------------------------------------------------------
int h2b_g1_decode_dev(int device, const void* d_bytes, size_t n, int format, void* d_out_affine, uint64_t* first_invalid, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return g1_decode_run(*c, d_bytes, n, format, d_out_affine, first_invalid, (cudaStream_t)stream);
}

int h2b_g1_encode_dev(int device, const void* d_affine, size_t n, void* d_out_bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return g1_encode_run(*c, d_affine, n, d_out_bytes, (cudaStream_t)stream);
}

namespace {
struct FileCloser { FILE* f; ~FileCloser() { if (f) fclose(f); } };
}  // namespace

// One point vector made on device 0: `produce` fills n x 64 B on device 0's stream; the points are downloaded to host_out (may be
// null), then registered under *handle as a replicated set with window tables (handle may be null: the points are dropped).
// release_g1gen: the producer runs g1gen.cu kernels whose scratch is given back once they are done.  Errors read "caller: what: ...".
// Caller holds G.mu.
static int device0_points_locked(size_t n, const char* caller, const char* what, bool release_g1gen,
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

// one vector of the file: bytes -> device 0 -> decoded points
static int srs_read_vector(const unsigned char* raw, const char* what, size_t n, int format, uint64_t* host_out, uint64_t* handle) {
    const size_t ps = format == H2B_SERDE_PROCESSED ? 32 : 64;
    std::lock_guard<std::mutex> glk(G.mu);
    return device0_points_locked(n, "h2b_srs_read", what, false, [&](DeviceCtx& c, void* d_pts) -> int {
        H2B_TRY(c.srs_io.reserve(n * ps));
        // the mapping is pageable memory: the staging threads of stage.cu pull it through the page cache in parallel
        H2B_TRY(host_upload(c, c.srs_io.p, raw, n * ps, c.stream));
        uint64_t bad = 0;
        return g1_decode_run(c, c.srs_io.p, n, format, d_pts, &bad, c.stream);
    }, host_out, handle);
}

// one vector of ParamsKZG::setup (which 0: g, 1: g_lagrange)
static int srs_setup_vector(uint32_t k, const uint64_t s[4], int which, uint64_t* host_out, uint64_t* handle) {
    std::lock_guard<std::mutex> glk(G.mu);
    return device0_points_locked((size_t)1 << k, "h2b_srs_setup", which ? "g_lagrange" : "g", true,
                                 [&](DeviceCtx& c, void* d_pts) { return srs_setup_run(c, k, s, which, d_pts, c.stream); }, host_out, handle);
}

namespace {
struct Mapping {
    int fd = -1;
    void* p = MAP_FAILED;
    size_t len = 0;
    ~Mapping() {
        if (p != MAP_FAILED) munmap(p, len);
        if (fd >= 0) close(fd);
    }
};
static bool srs_cache_enabled() {
    const char* e = getenv("H2B_SRS_CACHE");
    return !(e && e[0] == '0');
}
}  // namespace

// points of a resident set (table 0) -> host
static int srs_download_points(uint64_t handle, size_t n, uint64_t* out) {
    SetRef bs = find_set(handle);
    if (!bs || bs->n != n || bs->sharded) { set_error("h2b_srs_read: cached base set vanished"); return H2B_ERR_BAD_HANDLE; }
    const void* src = bs->dev[0];
    DeviceCtx& c = *G.devs[0];
    std::lock_guard<std::mutex> lk(c.mu);
    H2B_CUDA(cudaSetDevice(c.device));
    H2B_TRY(host_download(c, out, src, n * 64, c.stream));
    H2B_CUDA(cudaStreamSynchronize(c.stream));
    return H2B_OK;
}

int h2b_srs_read(const char* path, int format, uint32_t* k, uint64_t* out_g, uint64_t* out_g_lagrange, uint8_t* g2_bytes, size_t g2_cap, size_t* g2_len,
                 uint64_t* handle_g, uint64_t* handle_g_lagrange) {
    H2B_TRY(require_init());
    if (!path || !k) { set_error("h2b_srs_read: null path / k"); return H2B_ERR_BAD_ARGUMENT; }
    if (format < H2B_SERDE_PROCESSED || format > H2B_SERDE_RAW_BYTES_UNCHECKED) { set_error("h2b_srs_read: unknown format %d", format); return H2B_ERR_BAD_ARGUMENT; }
    Mapping m;
    m.fd = open(path, O_RDONLY);
    struct stat sb;
    if (m.fd < 0 || fstat(m.fd, &sb) != 0) { set_error("h2b_srs_read: cannot open %s", path); return H2B_ERR_BAD_ARGUMENT; }
    const long long mtime_ns = (long long)sb.st_mtim.tv_sec * 1000000000ll + sb.st_mtim.tv_nsec;
    // an unchanged file that was decoded before: hand out its resident sets again
    if (srs_cache_enabled()) {
        SrsCacheEntry hit;
        bool found = false;
        {
            std::lock_guard<std::mutex> lk(G.mu);
            for (const SrsCacheEntry& e : G.srs_cache) {
                if (e.path != path || e.format != format || e.size != (long long)sb.st_size || e.mtime_ns != mtime_ns) continue;
                SetRef a = find_set_locked(e.handle_g), b = find_set_locked(e.handle_g_lagrange);
                if (!a || !b) continue;
                if (handle_g) ++a->refs;
                if (handle_g_lagrange) ++b->refs;
                hit = e;
                found = true;
                break;
            }
        }
        if (found) {
            const size_t n = (size_t)1 << hit.k;
            int rc = H2B_OK;
            if (out_g) rc = srs_download_points(hit.handle_g, n, out_g);
            if (!rc && out_g_lagrange) rc = srs_download_points(hit.handle_g_lagrange, n, out_g_lagrange);
            if (rc) {
                if (handle_g) h2b_unregister_bases(hit.handle_g);
                if (handle_g_lagrange) h2b_unregister_bases(hit.handle_g_lagrange);
                return rc;
            }
            *k = hit.k;
            if (handle_g) *handle_g = hit.handle_g;
            if (handle_g_lagrange) *handle_g_lagrange = hit.handle_g_lagrange;
            if (g2_len) *g2_len = hit.g2.size();
            if (g2_bytes) memcpy(g2_bytes, hit.g2.data(), hit.g2.size() < g2_cap ? hit.g2.size() : g2_cap);
            return H2B_OK;
        }
    }
    if (sb.st_size < 4) { set_error("h2b_srs_read: %s is empty", path); return H2B_ERR_BAD_ARGUMENT; }
    m.len = (size_t)sb.st_size;
    m.p = mmap(nullptr, m.len, PROT_READ, MAP_PRIVATE, m.fd, 0);
    if (m.p == MAP_FAILED) { set_error("h2b_srs_read: cannot map %s", path); return H2B_ERR_BAD_ARGUMENT; }
    madvise(m.p, m.len, MADV_SEQUENTIAL);
    const unsigned char* bytes = (const unsigned char*)m.p;
    const uint32_t kk = (uint32_t)bytes[0] | ((uint32_t)bytes[1] << 8) | ((uint32_t)bytes[2] << 16) | ((uint32_t)bytes[3] << 24);
    if (kk > 28) { set_error("h2b_srs_read: k = %u in %s (at most 28)", kk, path); return H2B_ERR_BAD_ARGUMENT; }
    const size_t n = (size_t)1 << kk, ps = format == H2B_SERDE_PROCESSED ? 32 : 64;
    const size_t g2_want = format == H2B_SERDE_PROCESSED ? 128 : 256;      // g2 | s_g2
    if (m.len < 4 + 2 * n * ps) { set_error("h2b_srs_read: %s ends inside %s", path, m.len < 4 + n * ps ? "g" : "g_lagrange"); return H2B_ERR_BAD_ARGUMENT; }
    if (m.len < 4 + 2 * n * ps + g2_want) { set_error("h2b_srs_read: %s ends inside the G2 section", path); return H2B_ERR_BAD_ARGUMENT; }
    // the cache keeps both vectors resident even if the caller only asked for one handle
    const bool cache = srs_cache_enabled();
    uint64_t hg = 0, hl = 0;
    H2B_TRY(srs_read_vector(bytes + 4, "g", n, format, out_g, (handle_g || cache) ? &hg : nullptr));
    int rc = srs_read_vector(bytes + 4 + n * ps, "g_lagrange", n, format, out_g_lagrange, (handle_g_lagrange || cache) ? &hl : nullptr);
    if (rc != H2B_OK) { if (hg) h2b_unregister_bases(hg); return rc; }
    *k = kk;
    if (g2_len) *g2_len = g2_want;
    if (g2_bytes) memcpy(g2_bytes, bytes + 4 + 2 * n * ps, g2_want < g2_cap ? g2_want : g2_cap);
    if (cache) {
        std::lock_guard<std::mutex> lk(G.mu);
        SrsCacheEntry e;
        e.path = path; e.format = format; e.size = (long long)sb.st_size; e.mtime_ns = mtime_ns; e.k = kk;
        e.handle_g = hg; e.handle_g_lagrange = hl;
        e.g2.assign(bytes + 4 + 2 * n * ps, bytes + 4 + 2 * n * ps + g2_want);
        // the cache's own reference is the one srs_read_vector created; each caller that took a handle adds one
        SetRef a = find_set_locked(hg), b = find_set_locked(hl);
        if (a && handle_g) ++a->refs;
        if (b && handle_g_lagrange) ++b->refs;
        // a stale entry for the same path (file rewritten) gives its sets back
        for (size_t i = 0; i < G.srs_cache.size();) {
            if (G.srs_cache[i].path == e.path && G.srs_cache[i].format == e.format) {
                for (uint64_t h : {G.srs_cache[i].handle_g, G.srs_cache[i].handle_g_lagrange}) {
                    for (size_t j = 0; j < G.sets.size(); ++j)
                        if (G.sets[j]->handle == h && --G.sets[j]->refs <= 0) { G.sets.erase(G.sets.begin() + j); break; }
                }
                G.srs_cache.erase(G.srs_cache.begin() + i);
            } else ++i;
        }
        G.srs_cache.push_back(std::move(e));
    }
    if (handle_g) *handle_g = hg;
    if (handle_g_lagrange) *handle_g_lagrange = hl;
    return H2B_OK;
}

int h2b_srs_setup(uint32_t k, const uint64_t s[4], uint64_t* out_g, uint64_t* out_g_lagrange, uint64_t* handle_g, uint64_t* handle_g_lagrange) {
    H2B_TRY(require_init());
    if (!s) { set_error("h2b_srs_setup: null s"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(srs_setup_check(k, s));
    uint64_t hg = 0, hl = 0;
    H2B_TRY(srs_setup_vector(k, s, 0, out_g, handle_g ? &hg : nullptr));
    int rc = srs_setup_vector(k, s, 1, out_g_lagrange, handle_g_lagrange ? &hl : nullptr);
    if (rc != H2B_OK) { if (hg) h2b_unregister_bases(hg); return rc; }
    if (handle_g) *handle_g = hg;
    if (handle_g_lagrange) *handle_g_lagrange = hl;
    return H2B_OK;
}

int h2b_g1_generator_mul_dev(int device, const void* d_scalars, size_t n, void* d_out_affine, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return g1_generator_mul_run(*c, d_scalars, n, d_out_affine, (cudaStream_t)stream);
}

int h2b_g1_to_lagrange_dev(int device, const void* d_g_affine, uint32_t k, void* d_out_affine, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return g1_to_lagrange_run(*c, d_g_affine, k, d_out_affine, (cudaStream_t)stream);
}

int h2b_srs_downsize(uint64_t handle_g, uint32_t k, uint64_t* out_g_lagrange, uint64_t* handle_g_out, uint64_t* handle_g_lagrange_out) {
    H2B_TRY(require_init());
    if (k > 28) { set_error("h2b_srs_downsize: k = %u (at most 28)", k); return H2B_ERR_BAD_ARGUMENT; }
    const size_t n = (size_t)1 << k;
    std::lock_guard<std::mutex> glk(G.mu);
    SetRef src = find_set_locked(handle_g);
    if (!src || src->implicit) { set_error("h2b_srs_downsize: unknown base-set handle %llu", (unsigned long long)handle_g); return H2B_ERR_BAD_ARGUMENT; }
    if (src->sharded) { set_error("h2b_srs_downsize: handle %llu is a sharded set (g must be whole on device 0)", (unsigned long long)handle_g); return H2B_ERR_BAD_ARGUMENT; }
    if (n > src->n) { set_error("h2b_srs_downsize: 2^%u points requested from a set of %zu", k, src->n); return H2B_ERR_BAD_ARGUMENT; }
    uint64_t hg = 0, hl = 0;
    if (handle_g_out)
        H2B_TRY(device0_points_locked(n, "h2b_srs_downsize", "g", false, [&](DeviceCtx& c, void* d_g) -> int {
            H2B_CUDA(cudaMemcpyAsync(d_g, src->dev[0], n * 64, cudaMemcpyDeviceToDevice, c.stream));
            return H2B_OK;
        }, nullptr, &hg));
    if (out_g_lagrange || handle_g_lagrange_out) {
        const int rc = device0_points_locked(n, "h2b_srs_downsize", "g_lagrange", true,
                                             [&](DeviceCtx& c, void* d_gl) { return g1_to_lagrange_run(c, src->dev[0], k, d_gl, c.stream); },
                                             out_g_lagrange, handle_g_lagrange_out ? &hl : nullptr);
        if (rc) {
            if (hg) drop_locked(hg);
            return rc;
        }
    }
    if (handle_g_out) *handle_g_out = hg;
    if (handle_g_lagrange_out) *handle_g_lagrange_out = hl;
    return H2B_OK;
}

// ---- key generation: the permutation argument's sigma columns and keygen_pk's indicator columns ---------------------------------
// ([UP] halo2_proofs/src/plonk/permutation/keygen.rs Assembly::{build_vk, build_pk}, plonk/keygen.rs keygen_pk)
int h2b_permutation_sigma_dev(int device, const void* const* d_mapping, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4],
                              void* const* d_sigma, void* d_status, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (k > 28 || n_columns == 0) { set_error("h2b_permutation_sigma_dev: k = %u, %u columns (need k <= 28 and at least one column)", k, n_columns); return H2B_ERR_BAD_ARGUMENT; }
    if (!d_mapping || !delta || !omega || !d_sigma || !d_status) { set_error("h2b_permutation_sigma_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < n_columns; ++i)
        if (!d_mapping[i] || !d_sigma[i]) { set_error("h2b_permutation_sigma_dev: column %u: null pointer", i); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    const cudaStream_t st = (cudaStream_t)stream;
    H2B_CUDA(cudaMemsetAsync(d_status, 0, 4, st));
    H2B_TRY(permutation_sigma_tables_run(*c, n_columns, k, delta, omega, st));
    return permutation_sigma_run(*c, d_mapping, n_columns, 0, n_columns, k, d_sigma, d_status, st);
}

// the domain arguments of the keygen_pk entry points: the sizes and the constants of the iNTT and the coset NTT
static int domain_check(const char* who, uint32_t k, uint32_t extended_k, const uint64_t* omega_inv, const uint64_t* ifft_divisor,
                        const uint64_t* extended_omega, const uint64_t* zeta_powers) {
    if (extended_k > 28 || extended_k < k) { set_error("%s: need k <= extended_k <= 28 (k = %u, extended_k = %u)", who, k, extended_k); return H2B_ERR_BAD_ARGUMENT; }
    if (!omega_inv || !ifft_divisor || !extended_omega || !zeta_powers) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_keygen_lagrange_indicators_dev(int device, uint32_t k, uint32_t extended_k, uint32_t blinding_factors, const uint64_t omega_inv[4],
                                       const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], void* d_l0,
                                       void* d_l_last, void* d_l_active_row, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    static const char* who = "h2b_keygen_lagrange_indicators_dev";
    H2B_TRY(domain_check(who, k, extended_k, omega_inv, ifft_divisor, extended_omega, zeta_powers));
    if ((uint64_t)blinding_factors + 1 >= ((uint64_t)1 << k)) { set_error("%s: k = %u, %u blinding factors (need bf + 1 < 2^k)", who, k, blinding_factors); return H2B_ERR_BAD_ARGUMENT; }
    if (!d_l0 || !d_l_last || !d_l_active_row) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    void* cols[3] = {d_l0, d_l_last, d_l_active_row};
    return keygen_indicators_run(*c, k, extended_k, blinding_factors, omega_inv, ifft_divisor, extended_omega, zeta_powers, cols, (cudaStream_t)stream);
}

// The combination columns of compress_selectors: combination c's members are the selectors s with combination_of[s] = c, and
// member s writes root_of[s] on its active rows.  Built (and validated) on the host before any device work.
struct SelectorCombinations {
    const uint8_t* const* activations = nullptr;
    uint32_t n_selectors = 0, n_combinations = 0;
    std::vector<std::vector<uint32_t>> members;     // per combination: its selectors, in increasing order
    const uint32_t* root_of = nullptr;
};

// A proving key resident on the devices (h2b_pk_create): one allocation per device, holding per part and form a block of columns.
// Device d's block order is FIXED VALUES | FIXED COEFF | FIXED EXTENDED | PERMUTATION (the same three) | INDICATORS EXTENDED; an
// EXTENDED column there has ext_rows[d] rows (E replicated, the device's slice with its halo sharded).  Immutable in shape once created;
// builds write the columns under `build` and mark them filled.
struct ResidentPk {
    uint64_t handle = 0;
    uint32_t k = 0, extended_k = 0, halo = 0;
    uint32_t count[3] = {0, 0, 3};              // columns per part
    bool sharded = false;
    uint64_t omega[4], omega_inv[4], ifft_divisor[4], extended_omega[4], zeta_powers[12];
    std::vector<int> ordinal;
    std::vector<void*> dev;
    std::vector<size_t> row0, rows, ext_rows;   // per device: the owned extended rows and the slice length with halo
    std::vector<uint8_t> filled[3];             // per part and column: every form written by a completed build
    std::mutex build;                           // one build at a time
    mutable std::mutex filled_mu;               // guards filled[] for the readers
    ~ResidentPk() {
        for (size_t d = 0; d < dev.size(); ++d) {
            if (!dev[d]) continue;
            cudaSetDevice(ordinal[d]);
            cudaDeviceSynchronize();            // work already queued on the device may still read the columns
            cudaFree(dev[d]);
        }
        cudaGetLastError();
    }
    static bool holds(int part, int form) { return part != H2B_PK_INDICATORS || form == H2B_PK_EXTENDED; }
    size_t col_rows(size_t d, int form) const { return form == H2B_PK_EXTENDED ? ext_rows[d] : (size_t)1 << k; }
    size_t bytes_on(size_t d) const {
        size_t b = 0;
        for (int p = 0; p < 3; ++p)
            for (int f = 0; f < 3; ++f) if (holds(p, f)) b += (size_t)count[p] * col_rows(d, f) * 32;
        return b;
    }
    char* ptr(size_t d, int part, int form, uint32_t index) const {
        size_t off = 0;
        for (int p = 0; p < 3; ++p)
            for (int f = 0; f < 3; ++f) {
                if (!holds(p, f)) continue;
                if (p == part && f == form) return (char*)dev[d] + off + (size_t)index * col_rows(d, f) * 32;
                off += (size_t)count[p] * col_rows(d, f) * 32;
            }
        return nullptr;
    }
    // first global row of device d's extended slice
    size_t slice_start(size_t d) const {
        const size_t E = (size_t)1 << extended_k;
        return sharded ? (row0[d] + E - halo) % E : 0;
    }
};
typedef std::shared_ptr<ResidentPk> PkRef;

// Column `index` of (part, form), whole on device d at `src`, into the pk's storage of every device: a plain copy on d, a peer copy
// over NVLink elsewhere; of a sharded EXTENDED column each device receives its slice, in two pieces when it wraps past row E - 1.
// Enqueued on d's stream `st` (the caller synchronises it).
static int pk_place(const ResidentPk& pk, size_t d, cudaStream_t st, const void* src, int part, int form, uint32_t index) {
    DeviceCtx& c = *G.devs[d];
    const size_t E = (size_t)1 << pk.extended_k;
    for (size_t e = 0; e < pk.dev.size(); ++e) {
        char* dst = pk.ptr(e, part, form, index);
        auto copy = [&](char* to, const char* from, size_t bytes) -> int {
            if (to == from || bytes == 0) return H2B_OK;
            if (e == d) H2B_CUDA(cudaMemcpyAsync(to, from, bytes, cudaMemcpyDeviceToDevice, st));
            else H2B_CUDA(cudaMemcpyPeerAsync(to, pk.ordinal[e], from, pk.ordinal[d], bytes, st));
            return H2B_OK;
        };
        if (form != H2B_PK_EXTENDED || !pk.sharded) {
            H2B_TRY(copy(dst, (const char*)src, pk.col_rows(e, form) * 32));
        } else {
            const size_t s = pk.slice_start(e), len = pk.ext_rows[e], head = len < E - s ? len : E - s;
            H2B_TRY(copy(dst, (const char*)src + s * 32, head * 32));
            H2B_TRY(copy(dst + head * 32, (const char*)src, (len - head) * 32));
        }
        c.prof.mark(e == d ? PROF_PK_FORM_COPY : PROF_PK_PLACE, st);
    }
    return H2B_OK;
}

// after the writing pass over columns [first, first + count) of `part`: filled when it succeeded, no longer trusted when it failed midway
static int pk_mark(ResidentPk& pk, int part, uint32_t first, uint32_t count, int rc) {
    std::lock_guard<std::mutex> lk(pk.filled_mu);
    for (uint32_t i = first; i < first + count; ++i) pk.filled[part][i] = rc == H2B_OK;
    return rc;
}

// One build_vk / build_pk pass over the columns [col_begin, col_end); column i runs on device i mod D.  Column i's Lagrange values
// come from, in this order: sigma of mapping[i] for i < n_sigma, the caller's fixed[i - n_sigma] for the next n_fixed, and the
// combination columns of `comb` after those.
struct KeygenJob {
    const uint64_t* const* mapping = nullptr;
    uint32_t n_sigma = 0;
    const uint64_t* const* fixed = nullptr;
    uint32_t n_fixed = 0;
    const SelectorCombinations* comb = nullptr;
    uint32_t k = 0, extended_k = 0, col_begin = 0, col_end = 0;
    const uint64_t *delta = nullptr, *omega = nullptr, *omega_inv = nullptr, *ifft_divisor = nullptr, *extended_omega = nullptr, *zeta_powers = nullptr;
    bool validate_only = false;                 // the columns that can be invalid (sigma, combinations) and the status word only
    const BaseSet* commit_set = nullptr;        // a replicated set: commitments of the columns over its first n points
    uint64_t* commitments = nullptr;            // 12 words (Jacobian) per column, indexed by column
    uint64_t* const* values_out = nullptr;      // per column (indexed by column; an entry may be null), or null
    uint64_t* const* poly_out = nullptr;
    uint64_t* const* coset_out = nullptr;
    ResidentPk* resident = nullptr;             // every form of column i goes to column resident_first + i of resident_part
    int resident_part = 0;
    uint32_t resident_first = 0;
    uint32_t n_columns() const { return n_sigma + n_fixed + (comb ? comb->n_combinations : 0); }
};

// scratch of one device's share, given back on every return path
struct KeygenScratch {
    std::vector<void*> bufs;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    DeviceCtx* ctx = nullptr;
    int alloc(size_t bytes, void** out) {
        H2B_TRY(dev_malloc(out, bytes, "key generation"));
        bufs.push_back(*out);
        return H2B_OK;
    }
    ~KeygenScratch() {
        if (ctx) cudaStreamSynchronize(ctx->stream);
        for (void* p : bufs) cudaFree(p);
        for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
        if (ctx) ctx->keygen_tables.release();
        cudaGetLastError();
    }
};

static const size_t KEYGEN_GROUP_BYTES = (size_t)1 << 31;      // device memory of one group of columns (values / coefficients / cosets)

// Uploads each selector of `sel` (n bytes, pageable) and packs it into d_bits + slot * selector_words(n); the upload of selector t + 1
// goes through the other of the two staging buffers while the pack kernel of selector t runs.
static int keygen_pack_selectors(DeviceCtx& c, KeygenScratch& s, const uint8_t* const* activations, const std::vector<uint32_t>& sel, size_t n,
                                 void* d_bits, cudaStream_t st) {
    if (sel.empty()) return H2B_OK;
    void* d_act[2];
    H2B_TRY(s.alloc(n, &d_act[0]));
    H2B_TRY(s.alloc(n, &d_act[1]));
    for (size_t t = 0; t < sel.size(); ++t) {
        const int slot = (int)(t & 1);
        H2B_CUDA(cudaEventSynchronize(s.ev[slot]));            // the pack kernel that last read this buffer is done
        H2B_TRY(host_upload(c, d_act[slot], activations[sel[t]], n, st, false));
        H2B_TRY(selector_pack_run(c, d_act[slot], n, (uint32_t*)d_bits + t * selector_words(n), st));
        H2B_CUDA(cudaEventRecord(s.ev[slot], st));
    }
    return H2B_OK;
}

// device d's columns of the job, in groups that share the batched MSM / NTT launches.  The mapping of sigma column i + 1 is staged
// while the sigma kernel of column i runs (two mapping buffers); the selectors of this device's combination columns are uploaded and
// packed once, before the first group.  *bad receives the status word of the first group that holds an invalid entry; no output of
// that group or a later one is written.
static int keygen_device(size_t d, const KeygenJob& job, uint32_t* bad) {
    const size_t nd = G.devs.size();
    std::vector<uint32_t> mine;
    for (uint32_t i = job.col_begin; i < job.col_end; ++i) if (i % nd == d) mine.push_back(i);
    if (mine.empty()) return H2B_OK;
    DeviceCtx& c = *G.devs[d];
    std::lock_guard<std::mutex> lk(c.mu);
    H2B_CUDA(cudaSetDevice(c.device));
    const cudaStream_t st = c.stream;
    const uint32_t k = job.k;
    const size_t n = (size_t)1 << k;
    const uint32_t comb0 = job.n_sigma + job.n_fixed;
    const bool want_coset = job.coset_out || job.resident;
    const bool pk = job.poly_out || want_coset;
    const size_t col_bytes = (want_coset && !job.validate_only ? (size_t)1 << job.extended_k : n) * 32;
    size_t group = ntt_batch_max();
    while (group > 1 && group * col_bytes > KEYGEN_GROUP_BYTES) group >>= 1;
    if (job.commit_set && group > msm_batch_max()) group = msm_batch_max();
    KeygenScratch s;
    s.ctx = &c;
    for (cudaEvent_t& e : s.ev) H2B_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    void *d_map[2] = {nullptr, nullptr}, *d_cols, *d_status, *d_blocks, *d_bits = nullptr, *d_members = nullptr;
    const bool any_sigma = mine.front() < job.n_sigma;
    // this device's combinations: the selectors they use get consecutive bitset slots, members become (slot, root) pairs
    std::vector<uint32_t> sel, member_pairs, member_off;
    if (job.comb) {
        std::vector<uint32_t> slot_of(job.comb->n_selectors, UINT32_MAX);
        for (uint32_t i : mine) {
            if (i < comb0) continue;
            member_off.push_back((uint32_t)member_pairs.size() / 2);
            for (uint32_t sidx : job.comb->members[i - comb0]) {
                if (slot_of[sidx] == UINT32_MAX) { slot_of[sidx] = (uint32_t)sel.size(); sel.push_back(sidx); }
                member_pairs.push_back(slot_of[sidx]);
                member_pairs.push_back(job.comb->root_of[sidx]);
            }
        }
        member_off.push_back((uint32_t)member_pairs.size() / 2);
    }
    if (any_sigma) {
        H2B_TRY(s.alloc(n * 16, &d_map[0]));
        H2B_TRY(s.alloc(n * 16, &d_map[1]));
    }
    if (!sel.empty()) {
        H2B_TRY(s.alloc(sel.size() * selector_words(n) * 4, &d_bits));
        H2B_TRY(s.alloc(member_pairs.size() * 4, &d_members));
    }
    H2B_TRY(s.alloc(group * col_bytes, &d_cols));
    H2B_TRY(s.alloc(group * 224 + 32, &d_blocks));
    d_status = (char*)d_blocks + group * 224;
    c.prof.mark(PROF_BEGIN, st);
    H2B_CUDA(cudaMemsetAsync(d_status, 0, 4, st));
    if (any_sigma) H2B_TRY(permutation_sigma_tables_run(c, job.n_sigma, k, job.delta, job.omega, st));
    if (!sel.empty()) {
        H2B_CUDA(cudaMemcpyAsync(d_members, member_pairs.data(), member_pairs.size() * 4, cudaMemcpyHostToDevice, st));
        H2B_TRY(keygen_pack_selectors(c, s, job.comb->activations, sel, n, d_bits, st));
        c.prof.mark(PROF_KEYGEN_PACK, st);
    }
    size_t seq = 0, comb_seq = 0;
    for (size_t g0 = 0; g0 < mine.size(); g0 += group) {
        const size_t m = mine.size() - g0 < group ? mine.size() - g0 : group;
        std::vector<void*> cols(m);
        for (size_t t = 0; t < m; ++t) {
            const uint32_t i = mine[g0 + t];
            cols[t] = (char*)d_cols + t * col_bytes;
            if (i < job.n_sigma) {
                const int slot = (int)(seq++ & 1);
                H2B_CUDA(cudaEventSynchronize(s.ev[slot]));          // the sigma kernel that last read this mapping buffer is done
                H2B_TRY(host_upload(c, d_map[slot], job.mapping[i], n * 16, st, false));
                c.prof.mark(PROF_KEYGEN_UPLOAD, st);
                H2B_TRY(permutation_sigma_run(c, &d_map[slot], 1, i, job.n_sigma, k, &cols[t], d_status, st));
                H2B_CUDA(cudaEventRecord(s.ev[slot], st));
                c.prof.mark(PROF_KEYGEN_SIGMA, st);
            } else if (i < comb0) {
                if (job.validate_only) continue;                     // the caller's values need no check
                H2B_TRY(host_upload(c, cols[t], job.fixed[i - job.n_sigma], n * 32, st, t == 0));
                c.prof.mark(PROF_KEYGEN_FIXED_UPLOAD, st);
            } else {
                const size_t q = comb_seq++;
                H2B_TRY(combination_column_run(c, d_bits, (const uint32_t*)d_members + 2 * (size_t)member_off[q], member_off[q + 1] - member_off[q],
                                               i - comb0, k, cols[t], d_status, st));
                c.prof.mark(PROF_KEYGEN_COMBINATION, st);
            }
        }
        uint32_t status = 0;
        H2B_CUDA(cudaMemcpyAsync(&status, d_status, 4, cudaMemcpyDeviceToHost, st));
        H2B_CUDA(cudaStreamSynchronize(st));
        if (status) { *bad = status; return H2B_OK; }
        if (job.validate_only) continue;
        if (job.commit_set) {
            const MsmBases b = bases_of(*job.commit_set, d, 0);
            if (n > BATCH_COLUMN_MAX) {
                for (size_t t = 0; t < m; ++t) H2B_TRY(msm_run(c, cols[t], b, n, (char*)d_blocks + 224 * t, false, st));
            } else {
                std::vector<size_t> lens(m, n);
                H2B_TRY(msm_run_batch(c, cols.data(), lens.data(), (uint32_t)m, b, d_blocks, st));
            }
            c.prof.mark(PROF_KEYGEN_COMMIT, st);
            std::vector<uint64_t> blocks(28 * m);
            H2B_CUDA(cudaMemcpyAsync(blocks.data(), d_blocks, 224 * m, cudaMemcpyDeviceToHost, st));
            H2B_CUDA(cudaStreamSynchronize(st));
            for (size_t t = 0; t < m; ++t) memcpy(job.commitments + 12 * (size_t)mine[g0 + t], &blocks[28 * t], 96);
        }
        // each form goes to the caller's arrays and into the resident pk before the next in-place transform
        auto emit = [&](int form) -> int {
            uint64_t* const* out = form == H2B_PK_VALUES ? job.values_out : form == H2B_PK_COEFF ? job.poly_out : job.coset_out;
            if (out) {
                for (size_t t = 0; t < m; ++t)
                    if (out[mine[g0 + t]]) H2B_TRY(host_download(c, out[mine[g0 + t]], cols[t], form == H2B_PK_EXTENDED ? col_bytes : n * 32, st));
                c.prof.mark(PROF_KEYGEN_DOWNLOAD, st);
            }
            if (job.resident)
                for (size_t t = 0; t < m; ++t) H2B_TRY(pk_place(*job.resident, d, st, cols[t], job.resident_part, form, job.resident_first + mine[g0 + t]));
            return H2B_OK;
        };
        H2B_TRY(emit(H2B_PK_VALUES));
        if (!pk) continue;
        H2B_TRY(lagrange_to_coeff_batch_run(c, cols.data(), m, k, job.omega_inv, job.ifft_divisor, st));
        c.prof.mark(PROF_KEYGEN_INTT, st);
        H2B_TRY(emit(H2B_PK_COEFF));
        if (want_coset) {
            H2B_TRY(coeff_to_extended_batch_run(c, cols.data(), m, k, job.extended_k, job.extended_omega, job.zeta_powers, st));
            c.prof.mark(PROF_KEYGEN_COSET, st);
            H2B_TRY(emit(H2B_PK_EXTENDED));
        }
        // the next group's uploads into the group buffer must not overtake the copies out of it
        if (job.resident) H2B_CUDA(cudaStreamSynchronize(st));
    }
    return H2B_OK;
}

// every device's share of the job; an invalid mapping entry or two members of a combination on one row fail with H2B_ERR_BAD_ARGUMENT
static int keygen_run(const char* who, const KeygenJob& job) {
    const size_t nd = G.devs.size();
    std::vector<uint32_t> bad(nd, 0);
    H2B_TRY(on_devices(first_devices(nd), [&](size_t d) { return keygen_device(d, job, &bad[d]); }));
    for (size_t d = 0; d < nd; ++d) {
        if (!bad[d]) continue;
        const uint64_t flat = bad[d] - 1, n = (uint64_t)1 << job.k;
        if (job.comb) {
            if (bad[d] == 0xFFFFFFFFu) set_error("%s: two selectors of one combination are active on the same row", who);
            else set_error("%s: two selectors of combination %llu are active on row %llu", who, (unsigned long long)(flat / n), (unsigned long long)(flat % n));
        } else if (bad[d] == 0xFFFFFFFFu) {
            set_error("%s: the mapping holds an entry outside %u columns x 2^%u rows", who, job.n_sigma, job.k);
        } else {
            set_error("%s: mapping[%llu][%llu] is outside %u columns x 2^%u rows", who, (unsigned long long)(flat / n), (unsigned long long)(flat % n),
                      job.n_sigma, job.k);
        }
        return H2B_ERR_BAD_ARGUMENT;
    }
    return H2B_OK;
}

// The build_pk of every column of `job`: a pass that only builds and checks the columns [first_checked, end) -- the ones that can be
// invalid -- then, when the job has an output, the pass that writes it.  So no caller memory and no resident column is written before
// every sigma entry and combination column has been found valid.  The resident columns are marked after the writing pass only: a
// refused build leaves what the pk held readable.
static int keygen_build(const char* who, KeygenJob job, uint32_t first_checked) {
    job.col_begin = 0;
    job.col_end = job.n_columns();
    if (first_checked < job.col_end) {
        KeygenJob check = job;
        check.validate_only = true;
        check.col_begin = first_checked;
        H2B_TRY(keygen_run(who, check));
    }
    if (!job.values_out && !job.poly_out && !job.coset_out && !job.resident) return H2B_OK;
    const int rc = keygen_run(who, job);
    return job.resident ? pk_mark(*job.resident, job.resident_part, job.resident_first, job.col_end, rc) : rc;
}

// commitments of every column of `job` over a registered g_lagrange set (the caller has checked that it holds at least n points)
static int keygen_commit(const char* who, KeygenJob& job, const BaseSet& bs, uint64_t* out_commitments) {
    const size_t n = (size_t)1 << job.k;
    const uint32_t total = job.n_columns();
    std::vector<uint64_t> com((size_t)total * 12);
    if (!bs.sharded) {
        job.commit_set = &bs;
        job.commitments = com.data();
        job.col_begin = 0; job.col_end = total;
        H2B_TRY(keygen_run(who, job));
    } else {
        // a sharded set holds every point on one device only: the columns come back to the host (the caller's fixed columns are
        // there already) and each commitment is split by point range over the devices, as h2b_msm_bn254_g1_batch_registered does
        for (uint32_t i = 0; i < job.n_fixed; ++i) H2B_TRY(msm_host(job.fixed[i], bs, 0, n, com.data() + 12 * (size_t)(job.n_sigma + i)));
        const uint32_t chunk = (uint32_t)ntt_batch_max();
        std::vector<std::vector<uint64_t>> values(chunk, std::vector<uint64_t>(4 * n));
        std::vector<uint64_t*> ptrs(total, nullptr);
        job.values_out = ptrs.data();
        const uint32_t ranges[2][2] = {{0, job.n_sigma}, {job.n_sigma + job.n_fixed, total}};
        for (const auto& r : ranges) {
            for (uint32_t c0 = r[0]; c0 < r[1]; c0 += chunk) {
                const uint32_t c1 = r[1] - c0 < chunk ? r[1] : c0 + chunk;
                for (uint32_t i = c0; i < c1; ++i) ptrs[i] = values[i - c0].data();
                job.col_begin = c0; job.col_end = c1;
                H2B_TRY(keygen_run(who, job));
                for (uint32_t i = c0; i < c1; ++i) H2B_TRY(msm_host(ptrs[i], bs, 0, n, com.data() + 12 * (size_t)i));
            }
        }
    }
    memcpy(out_commitments, com.data(), com.size() * 8);
    return H2B_OK;
}

static int keygen_lookup_set(const char* who, uint64_t handle_g_lagrange, uint32_t k, SetRef* out) {
    *out = find_set(handle_g_lagrange);
    if (!*out) { set_error("%s: unknown base-set handle %llu", who, (unsigned long long)handle_g_lagrange); return H2B_ERR_BAD_ARGUMENT; }
    if (((size_t)1 << k) > (*out)->n) { set_error("%s: 2^%u points requested from a set of %zu", who, k, (*out)->n); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

static int keygen_check(const char* who, const uint64_t* const* mapping, uint32_t n_columns, uint32_t k, const uint64_t* delta, const uint64_t* omega) {
    H2B_TRY(require_init());
    if (k > 28 || n_columns == 0) { set_error("%s: k = %u, %u columns (need k <= 28 and at least one column)", who, k, n_columns); return H2B_ERR_BAD_ARGUMENT; }
    if (!mapping || !delta || !omega) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < n_columns; ++i) if (!mapping[i]) { set_error("%s: mapping column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_permutation_build_vk(const uint64_t* const* mapping, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4],
                             uint64_t handle_g_lagrange, uint64_t* out_commitments) {
    static const char* who = "h2b_permutation_build_vk";
    H2B_TRY(keygen_check(who, mapping, n_columns, k, delta, omega));
    if (!out_commitments) { set_error("%s: null output", who); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs;
    H2B_TRY(keygen_lookup_set(who, handle_g_lagrange, k, &bs));
    KeygenJob job;
    job.mapping = mapping; job.n_sigma = n_columns; job.k = k; job.delta = delta; job.omega = omega;
    return keygen_commit(who, job, *bs, out_commitments);
}

int h2b_permutation_build_pk(const uint64_t* const* mapping, uint32_t n_columns, uint32_t k, uint32_t extended_k, const uint64_t delta[4],
                             const uint64_t omega[4], const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4],
                             const uint64_t zeta_powers[12], uint64_t* const* out_permutations, uint64_t* const* out_polys, uint64_t* const* out_cosets) {
    static const char* who = "h2b_permutation_build_pk";
    H2B_TRY(keygen_check(who, mapping, n_columns, k, delta, omega));
    H2B_TRY(domain_check(who, k, extended_k, omega_inv, ifft_divisor, extended_omega, zeta_powers));
    for (uint64_t* const* outs : {out_permutations, out_polys, out_cosets})
        if (outs)
            for (uint32_t i = 0; i < n_columns; ++i) if (!outs[i]) { set_error("%s: output column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    KeygenJob job;
    job.mapping = mapping; job.n_sigma = n_columns; job.k = k; job.extended_k = extended_k; job.delta = delta; job.omega = omega;
    job.omega_inv = omega_inv; job.ifft_divisor = ifft_divisor; job.extended_omega = extended_omega; job.zeta_powers = zeta_powers;
    job.values_out = out_permutations; job.poly_out = out_polys; job.coset_out = out_cosets;
    return keygen_build(who, job, 0);
}

// ---- key generation: compress_selectors and the fixed columns of keygen_vk / keygen_pk --------------------------------------------
// ([UP] halo2_proofs/src/plonk/circuit/compress_selectors.rs process, plonk/keygen.rs keygen_vk / keygen_pk)
static const uint32_t SELECTORS_MAX = 1u << 14;

static int selectors_check(const char* who, const uint8_t* const* activations, uint32_t n_selectors, uint32_t k) {
    if (k > 28) { set_error("%s: k = %u (need k <= 28)", who, k); return H2B_ERR_BAD_ARGUMENT; }
    if (n_selectors > SELECTORS_MAX) { set_error("%s: %u selectors (at most %u)", who, n_selectors, SELECTORS_MAX); return H2B_ERR_BAD_ARGUMENT; }
    if (n_selectors && !activations) { set_error("%s: null activations", who); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t s = 0; s < n_selectors; ++s) if (!activations[s]) { set_error("%s: activations of selector %u are null", who, s); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_selector_exclusion(const uint8_t* const* activations, uint32_t n_selectors, uint32_t k, uint8_t* out) {
    static const char* who = "h2b_selector_exclusion";
    H2B_TRY(require_init());
    H2B_TRY(selectors_check(who, activations, n_selectors, k));
    if (!out) { set_error("%s: null output", who); return H2B_ERR_BAD_ARGUMENT; }
    if (n_selectors == 0) return H2B_OK;
    const size_t n = (size_t)1 << k, S = n_selectors;
    std::unique_lock<std::mutex> lk;
    size_t d = 0;
    DeviceCtx& c = *pick_device(lk, &d);
    H2B_CUDA(cudaSetDevice(c.device));
    const cudaStream_t st = c.stream;
    KeygenScratch s;
    s.ctx = &c;
    for (cudaEvent_t& e : s.ev) H2B_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    void *d_bits, *d_flags;
    H2B_TRY(s.alloc(S * selector_words(n) * 4, &d_bits));
    H2B_TRY(s.alloc(S * S * 4, &d_flags));
    std::vector<uint32_t> all(S);
    for (uint32_t i = 0; i < S; ++i) all[i] = i;
    c.prof.mark(PROF_BEGIN, st);
    H2B_TRY(keygen_pack_selectors(c, s, activations, all, n, d_bits, st));
    c.prof.mark(PROF_KEYGEN_PACK, st);
    H2B_TRY(selector_exclusion_run(c, d_bits, n_selectors, n, d_flags, st));
    c.prof.mark(PROF_KEYGEN_EXCLUSION, st);
    std::vector<uint32_t> flags(S * S);
    H2B_CUDA(cudaMemcpyAsync(flags.data(), d_flags, S * S * 4, cudaMemcpyDeviceToHost, st));
    H2B_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < S; ++i)
        for (size_t j = 0; j < S; ++j) out[i * S + j] = (uint8_t)(i > j ? flags[i * S + j] != 0 : i < j ? flags[j * S + i] != 0 : 0);
    return H2B_OK;
}

// the arguments both fixed-column entry points take, checked before any device work; *comb receives the members of each combination
static int fixed_keygen_check(const char* who, const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                              const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint32_t k,
                              SelectorCombinations* comb) {
    H2B_TRY(require_init());
    H2B_TRY(selectors_check(who, activations, n_selectors, k));
    if ((uint64_t)n_fixed + n_combinations == 0) { set_error("%s: no fixed and no combination columns", who); return H2B_ERR_BAD_ARGUMENT; }
    if (n_fixed && !fixed) { set_error("%s: null fixed columns", who); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t i = 0; i < n_fixed; ++i) if (!fixed[i]) { set_error("%s: fixed column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    if (n_selectors && (!combination_of || !root_of)) { set_error("%s: null assignment", who); return H2B_ERR_BAD_ARGUMENT; }
    comb->activations = activations;
    comb->n_selectors = n_selectors;
    comb->n_combinations = n_combinations;
    comb->root_of = root_of;
    comb->members.assign(n_combinations, std::vector<uint32_t>());
    for (uint32_t s = 0; s < n_selectors; ++s) {
        if (combination_of[s] >= n_combinations || root_of[s] == 0) {
            set_error("%s: selector %u: combination %u of %u, root %u (need combination < %u and root > 0)", who, s, combination_of[s], n_combinations,
                      root_of[s], n_combinations);
            return H2B_ERR_BAD_ARGUMENT;
        }
        comb->members[combination_of[s]].push_back(s);
    }
    for (uint32_t c = 0; c < n_combinations; ++c)
        if (comb->members[c].empty()) { set_error("%s: combination %u has no selector", who, c); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_keygen_fixed_build_vk(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                              const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint32_t k, uint64_t handle_g_lagrange,
                              uint64_t* out_commitments) {
    static const char* who = "h2b_keygen_fixed_build_vk";
    SelectorCombinations comb;
    H2B_TRY(fixed_keygen_check(who, fixed, n_fixed, activations, n_selectors, combination_of, root_of, n_combinations, k, &comb));
    if (!out_commitments) { set_error("%s: null output", who); return H2B_ERR_BAD_ARGUMENT; }
    SetRef bs;
    H2B_TRY(keygen_lookup_set(who, handle_g_lagrange, k, &bs));
    KeygenJob job;
    job.fixed = fixed; job.n_fixed = n_fixed; job.comb = &comb; job.k = k;
    return keygen_commit(who, job, *bs, out_commitments);
}

int h2b_keygen_fixed_build_pk(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                              const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint32_t k, uint32_t extended_k,
                              const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                              uint64_t* const* out_combination_values, uint64_t* const* out_polys, uint64_t* const* out_cosets) {
    static const char* who = "h2b_keygen_fixed_build_pk";
    SelectorCombinations comb;
    H2B_TRY(fixed_keygen_check(who, fixed, n_fixed, activations, n_selectors, combination_of, root_of, n_combinations, k, &comb));
    H2B_TRY(domain_check(who, k, extended_k, omega_inv, ifft_divisor, extended_omega, zeta_powers));
    const uint32_t total = n_fixed + n_combinations;
    if (out_combination_values)
        for (uint32_t c = 0; c < n_combinations; ++c)
            if (!out_combination_values[c]) { set_error("%s: combination output %u is null", who, c); return H2B_ERR_BAD_ARGUMENT; }
    for (uint64_t* const* outs : {out_polys, out_cosets})
        if (outs)
            for (uint32_t i = 0; i < total; ++i) if (!outs[i]) { set_error("%s: output column %u is null", who, i); return H2B_ERR_BAD_ARGUMENT; }
    std::vector<uint64_t*> values(total, nullptr);
    if (out_combination_values)
        for (uint32_t c = 0; c < n_combinations; ++c) values[n_fixed + c] = out_combination_values[c];
    KeygenJob job;
    job.fixed = fixed; job.n_fixed = n_fixed; job.comb = &comb; job.k = k; job.extended_k = extended_k;
    job.omega_inv = omega_inv; job.ifft_divisor = ifft_divisor; job.extended_omega = extended_omega; job.zeta_powers = zeta_powers;
    job.values_out = out_combination_values ? values.data() : nullptr;
    job.poly_out = out_polys; job.coset_out = out_cosets;
    return keygen_build(who, job, n_fixed);
}

// ---- the proving key resident on the devices ---------------------------------------------------------------------------------------
static int pk_lookup(const char* who, uint64_t handle, PkRef* out) {
    H2B_TRY(require_init());
    std::lock_guard<std::mutex> lk(G.mu);
    for (auto& p : G.pks) if (p->handle == handle) { *out = p; return H2B_OK; }
    set_error("%s: unknown proving-key handle %llu", who, (unsigned long long)handle);
    return H2B_ERR_BAD_ARGUMENT;
}

// a keygen job over the pk's domain, writing into it
static KeygenJob pk_job(ResidentPk& pk, int part, uint32_t first) {
    KeygenJob job;
    job.k = pk.k; job.extended_k = pk.extended_k; job.omega = pk.omega; job.omega_inv = pk.omega_inv; job.ifft_divisor = pk.ifft_divisor;
    job.extended_omega = pk.extended_omega; job.zeta_powers = pk.zeta_powers;
    job.resident = &pk; job.resident_part = part; job.resident_first = first;
    return job;
}

static int pk_range_check(const char* who, const ResidentPk& pk, int part, uint64_t first, uint64_t count) {
    if (first + count > pk.count[part]) {
        set_error("%s: columns %llu .. %llu of a part of %u columns", who, (unsigned long long)first, (unsigned long long)(first + count), pk.count[part]);
        return H2B_ERR_BAD_ARGUMENT;
    }
    return H2B_OK;
}

int h2b_pk_create(uint32_t k, uint32_t extended_k, uint32_t n_fixed, uint32_t n_permutation, int layout, uint32_t halo, const uint64_t omega[4],
                  const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                  uint64_t* handle) {
    static const char* who = "h2b_pk_create";
    H2B_TRY(require_init());
    H2B_TRY(domain_check(who, k, extended_k, omega_inv, ifft_divisor, extended_omega, zeta_powers));
    if (layout != H2B_PK_REPLICATED && layout != H2B_PK_ROW_SHARDED) { set_error("%s: unknown layout %d", who, layout); return H2B_ERR_BAD_ARGUMENT; }
    if (!omega || !handle) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    const size_t nd = G.devs.size(), E = (size_t)1 << extended_k;
    PkRef pk(new ResidentPk());
    pk->k = k; pk->extended_k = extended_k;
    pk->count[H2B_PK_FIXED] = n_fixed; pk->count[H2B_PK_PERMUTATION] = n_permutation;
    pk->sharded = layout == H2B_PK_ROW_SHARDED;
    pk->halo = pk->sharded ? halo : 0;
    memcpy(pk->omega, omega, 32); memcpy(pk->omega_inv, omega_inv, 32); memcpy(pk->ifft_divisor, ifft_divisor, 32);
    memcpy(pk->extended_omega, extended_omega, 32); memcpy(pk->zeta_powers, zeta_powers, 96);
    for (size_t d = 0; d < nd; ++d) {
        const size_t r0 = pk->sharded ? E * d / nd : 0, r1 = pk->sharded ? E * (d + 1) / nd : E;
        pk->row0.push_back(r0);
        pk->rows.push_back(r1 - r0);
        pk->ext_rows.push_back(r1 - r0 + 2 * (size_t)pk->halo);
        if (pk->ext_rows[d] > E) {
            set_error("%s: device %zu holds %zu rows + 2 x %u halo rows of a 2^%u-row coset", who, d, r1 - r0, pk->halo, extended_k);
            return H2B_ERR_BAD_ARGUMENT;
        }
        pk->ordinal.push_back(G.devs[d]->device);
    }
    for (int p = 0; p < 3; ++p) pk->filled[p].assign(pk->count[p], 0);
    pk->dev.assign(nd, nullptr);
    for (size_t d = 0; d < nd; ++d) {
        H2B_CUDA(cudaSetDevice(pk->ordinal[d]));
        H2B_TRY(dev_malloc(&pk->dev[d], pk->bytes_on(d), "the resident proving key"));     // pk's destructor frees what was reserved
    }
    std::lock_guard<std::mutex> lk(G.mu);
    pk->handle = G.next_handle++;
    G.pks.push_back(pk);
    *handle = pk->handle;
    return H2B_OK;
}

int h2b_keygen_fixed_build_pk_resident(const uint64_t* const* fixed, uint32_t n_fixed, const uint8_t* const* activations, uint32_t n_selectors,
                                       const uint32_t* combination_of, const uint32_t* root_of, uint32_t n_combinations, uint64_t handle, uint32_t first_column) {
    static const char* who = "h2b_keygen_fixed_build_pk_resident";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    SelectorCombinations comb;
    H2B_TRY(fixed_keygen_check(who, fixed, n_fixed, activations, n_selectors, combination_of, root_of, n_combinations, pk->k, &comb));
    const uint32_t total = n_fixed + n_combinations;
    H2B_TRY(pk_range_check(who, *pk, H2B_PK_FIXED, first_column, total));
    std::lock_guard<std::mutex> lk(pk->build);
    KeygenJob job = pk_job(*pk, H2B_PK_FIXED, first_column);
    job.fixed = fixed; job.n_fixed = n_fixed; job.comb = &comb;
    return keygen_build(who, job, n_fixed);
}

int h2b_permutation_build_pk_resident(const uint64_t* const* mapping, uint32_t n_columns, const uint64_t delta[4], uint64_t handle) {
    static const char* who = "h2b_permutation_build_pk_resident";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    H2B_TRY(keygen_check(who, mapping, n_columns, pk->k, delta, pk->omega));
    if (n_columns != pk->count[H2B_PK_PERMUTATION]) {
        set_error("%s: %u mapping columns for a pk of %u permutation columns", who, n_columns, pk->count[H2B_PK_PERMUTATION]);
        return H2B_ERR_BAD_ARGUMENT;
    }
    std::lock_guard<std::mutex> lk(pk->build);
    KeygenJob job = pk_job(*pk, H2B_PK_PERMUTATION, 0);
    job.mapping = mapping; job.n_sigma = n_columns; job.delta = delta;
    return keygen_build(who, job, 0);
}

int h2b_keygen_lagrange_indicators_resident(uint64_t handle, uint32_t blinding_factors) {
    static const char* who = "h2b_keygen_lagrange_indicators_resident";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    if ((uint64_t)blinding_factors + 1 >= ((uint64_t)1 << pk->k)) {
        set_error("%s: k = %u, %u blinding factors (need bf + 1 < 2^k)", who, pk->k, blinding_factors);
        return H2B_ERR_BAD_ARGUMENT;
    }
    std::lock_guard<std::mutex> lk(pk->build);
    auto run = [&]() -> int {
        DeviceCtx& c = *G.devs[0];
        std::lock_guard<std::mutex> dlk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        const cudaStream_t st = c.stream;
        KeygenScratch s;
        s.ctx = &c;
        // replicated: straight into device 0's columns, then peer copies; sharded: the whole cosets in scratch, then the slices
        void* cols[3];
        for (uint32_t i = 0; i < 3; ++i) {
            if (pk->sharded) H2B_TRY(s.alloc(((size_t)1 << pk->extended_k) * 32, &cols[i]));
            else cols[i] = pk->ptr(0, H2B_PK_INDICATORS, H2B_PK_EXTENDED, i);
        }
        c.prof.mark(PROF_BEGIN, st);
        H2B_TRY(keygen_indicators_run(c, pk->k, pk->extended_k, blinding_factors, pk->omega_inv, pk->ifft_divisor, pk->extended_omega, pk->zeta_powers, cols,
                                      st));
        for (uint32_t i = 0; i < 3; ++i) H2B_TRY(pk_place(*pk, 0, st, cols[i], H2B_PK_INDICATORS, H2B_PK_EXTENDED, i));
        H2B_CUDA(cudaStreamSynchronize(st));
        return H2B_OK;
    };
    return pk_mark(*pk, H2B_PK_INDICATORS, 0, 3, run());
}

int h2b_pk_put_lagrange(uint64_t handle, int part, uint32_t first, uint32_t count, const uint64_t* const* values) {
    static const char* who = "h2b_pk_put_lagrange";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    if (part != H2B_PK_FIXED && part != H2B_PK_PERMUTATION) {
        set_error("%s: part %d (FIXED or PERMUTATION; the indicators come from h2b_keygen_lagrange_indicators_resident)", who, part);
        return H2B_ERR_BAD_ARGUMENT;
    }
    H2B_TRY(pk_range_check(who, *pk, part, first, count));
    if (count == 0) return H2B_OK;
    if (!values) { set_error("%s: null values", who); return H2B_ERR_BAD_ARGUMENT; }
    for (uint32_t j = 0; j < count; ++j) if (!values[j]) { set_error("%s: values[%u] is null", who, j); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(pk->build);
    KeygenJob job = pk_job(*pk, part, first);
    job.fixed = values; job.n_fixed = count;
    return keygen_build(who, job, count);
}

// the checks every reader of one column makes
static int pk_column_check(const char* who, const ResidentPk& pk, int part, int form, uint32_t index) {
    if (part < 0 || part > 2 || form < 0 || form > 2 || !ResidentPk::holds(part, form)) {
        set_error("%s: part %d does not hold form %d", who, part, form);
        return H2B_ERR_BAD_ARGUMENT;
    }
    if (index >= pk.count[part]) { set_error("%s: column %u of a part of %u columns", who, index, pk.count[part]); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(pk.filled_mu);
    if (!pk.filled[part][index]) { set_error("%s: column %u of part %d was never filled", who, index, part); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_pk_column(uint64_t handle, int device, int part, int form, uint32_t index, void** d_ptr, h2b_eval_shard* shard) {
    static const char* who = "h2b_pk_column";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    if (device < 0 || (size_t)device >= pk->dev.size()) { set_error("%s: device index %d out of range (have %zu)", who, device, pk->dev.size()); return H2B_ERR_BAD_ARGUMENT; }
    if (!d_ptr) { set_error("%s: null output", who); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(pk_column_check(who, *pk, part, form, index));
    *d_ptr = pk->ptr(device, part, form, index);
    if (shard) {
        const bool slice = form == H2B_PK_EXTENDED && pk->sharded;
        shard->row0 = slice ? (uint32_t)pk->row0[device] : 0;
        shard->rows = (uint32_t)(slice ? pk->rows[device] : pk->col_rows(device, form));
        shard->halo = slice ? pk->halo : 0;
    }
    return H2B_OK;
}

int h2b_pk_download(uint64_t handle, int part, int form, uint32_t index, uint64_t* host_out) {
    static const char* who = "h2b_pk_download";
    PkRef pk;
    H2B_TRY(pk_lookup(who, handle, &pk));
    if (!host_out) { set_error("%s: null output", who); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(pk_column_check(who, *pk, part, form, index));
    const bool slices = form == H2B_PK_EXTENDED && pk->sharded;
    for (size_t d = 0; d < (slices ? pk->dev.size() : 1); ++d) {
        DeviceCtx& c = *G.devs[d];
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        // a sharded coset: the rows this device owns sit after its leading halo
        const char* src = pk->ptr(d, part, form, index) + (slices ? (size_t)pk->halo * 32 : 0);
        const size_t row = slices ? pk->row0[d] : 0, rows = slices ? pk->rows[d] : pk->col_rows(d, form);
        H2B_TRY(host_download(c, host_out + 4 * row, src, rows * 32, c.stream));
        H2B_CUDA(cudaStreamSynchronize(c.stream));
    }
    return H2B_OK;
}

int h2b_pk_info(uint64_t handle, uint64_t* per_device_bytes) {
    PkRef pk;
    H2B_TRY(pk_lookup("h2b_pk_info", handle, &pk));
    if (per_device_bytes)
        for (size_t d = 0; d < pk->dev.size(); ++d) per_device_bytes[d] = pk->bytes_on(d);
    return H2B_OK;
}

int h2b_pk_release(uint64_t handle) {
    PkRef drop;      // freed after G.mu is let go (the destructor waits for the devices)
    {
        std::lock_guard<std::mutex> lk(G.mu);
        for (size_t i = 0; i < G.pks.size(); ++i)
            if (G.pks[i]->handle == handle) { drop = G.pks[i]; G.pks.erase(G.pks.begin() + i); break; }
    }
    if (!drop) { set_error("h2b_pk_release: unknown proving-key handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

// ---- the multi-point opening (SHPLONK) -------------------------------------------------------------------------------------------
}  // extern "C"

// One opening between h1 and h2 on one device.  Device memory, one block: the plan's tables | pair values | scalars | h_x | two
// n-coefficient work buffers | the uploaded polynomials of a host-pointer session.  The work buffers hold h' after finish.
struct ShplonkSession {
    uint64_t handle = 0;
    size_t d = 0, n = 0;
    int ordinal = -1;
    h2b::SetRef g;                 // held for the session's life: finish commits over it
    h2b::ShplonkPlan plan;
    void* mem = nullptr;
    size_t tables = 0, evals = 0, scal = 0, hx = 0, a = 0, b = 0, polys = 0;
    bool finished = false;
    std::mutex mu;                 // one call at a time
    char* at(size_t off) const { return (char*)mem + off; }
    ~ShplonkSession() {
        if (!mem) return;
        cudaSetDevice(ordinal);
        cudaDeviceSynchronize();
        cudaFree(mem);
        cudaGetLastError();
    }
};
typedef std::shared_ptr<ShplonkSession> SessionRef;

static int shplonk_n_check(const char* who, size_t n) {
    if (n < 2 || n > ((size_t)1 << 28)) { set_error("%s: n = %zu (2 <= n <= 2^28)", who, n); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

static int session_lookup(const char* who, uint64_t handle, SessionRef* out) {
    H2B_TRY(require_init());
    std::lock_guard<std::mutex> lk(G.mu);
    for (auto& s : G.sessions) if (s->handle == handle) { *out = s; return H2B_OK; }
    set_error("%s: unknown session handle %llu", who, (unsigned long long)handle);
    return H2B_ERR_BAD_ARGUMENT;
}

// the result block of an MSM on the session's device -> host (synchronises the stream)
static int session_commit(DeviceCtx& c, ShplonkSession& s, const void* d_scalars, size_t n, uint64_t out_jac[12]) {
    void* d_jac = (void*)shplonk_tables_jac(s.plan, s.at(s.tables));
    H2B_TRY(msm_run(c, d_scalars, bases_of(*s.g, s.d, 0), n, d_jac, false, c.stream));
    c.prof.mark(PROF_OPEN_MSM, c.stream);
    uint64_t jac[12];
    H2B_CUDA(cudaMemcpyAsync(jac, d_jac, 96, cudaMemcpyDeviceToHost, c.stream));
    uint32_t status = 0;
    H2B_CUDA(cudaMemcpyAsync(&status, shplonk_tables_status(s.plan, s.at(s.tables)), 4, cudaMemcpyDeviceToHost, c.stream));
    H2B_CUDA(cudaStreamSynchronize(c.stream));
    if (status) { set_error("h2b_shplonk_finish: u is a point of T outside S_0 (Z_{T \\ S_0}(u) = 0)"); return H2B_ERR_BAD_ARGUMENT; }
    memcpy(out_jac, jac, 96);
    return H2B_OK;
}

extern "C" {

int h2b_fr_eval_queries_dev(int device, const void* const* d_polys, uint32_t n_polys, size_t n, const h2b_opening_query* queries, uint32_t n_queries,
                            void* d_out, void* stream) {
    static const char* who = "h2b_fr_eval_queries_dev";
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_polys || !d_out) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(shplonk_n_check(who, n));
    ShplonkPlan plan;
    H2B_TRY(shplonk_plan_build(who, queries, n_queries, n_polys, true, &plan));
    for (uint32_t s : plan.used) {
        if (!d_polys[s]) { set_error("%s: polynomial %u is a null pointer", who, s); return H2B_ERR_BAD_ARGUMENT; }
        plan.d_polys.push_back(d_polys[s]);
    }
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t tb = shplonk_tables_bytes(plan);
    H2B_TRY(c->open_tables.reserve(tb + plan.pair_point.size() * 32));
    const cudaStream_t st = (cudaStream_t)stream;
    H2B_TRY(shplonk_tables_upload(plan, plan.d_polys.data(), c->open_tables.p, st));
    return shplonk_eval_queries_run(*c, plan, c->open_tables.p, n, (char*)c->open_tables.p + tb, d_out, st);
}

int h2b_shplonk_begin(int device, const void* const* polys, int polys_on_host, uint32_t n_polys, size_t n, const h2b_opening_query* queries,
                      uint32_t n_queries, uint64_t handle_g, const uint64_t y[4], const uint64_t v[4], uint64_t out_h1_jac[12], uint64_t* session) {
    static const char* who = "h2b_shplonk_begin";
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!polys || !y || !v || !out_h1_jac || !session) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    H2B_TRY(shplonk_n_check(who, n));
    if (!fr_canonical(y) || !fr_canonical(v)) { set_error("%s: a challenge is not below the scalar field modulus", who); return H2B_ERR_BAD_ARGUMENT; }
    SessionRef s(new ShplonkSession());
    H2B_TRY(shplonk_plan_build(who, queries, n_queries, n_polys, true, &s->plan));
    for (uint32_t i = 0; i < n_polys; ++i) if (!polys[i]) { set_error("%s: polynomial %u is a null pointer", who, i); return H2B_ERR_BAD_ARGUMENT; }
    s->g = find_set(handle_g);
    if (!s->g) { set_error("%s: unknown base-set handle %llu", who, (unsigned long long)handle_g); return H2B_ERR_BAD_ARGUMENT; }
    s->d = (size_t)device;
    if (s->g->lo[s->d] != 0 || s->g->rows[s->d] < n) { set_error("%s: device %d does not hold rows [0, %zu) of the set", who, device, n); return H2B_ERR_BAD_ARGUMENT; }
    s->n = n;
    s->ordinal = c->device;
    // the block: tables | pair values | scalars | h_x | a | b | uploaded polynomials
    const ShplonkPlan& p = s->plan;
    const size_t P = p.used.size();
    size_t off = 0;
    s->tables = off; off += shplonk_tables_bytes(p);
    s->evals = off;  off += 32 * p.pair_point.size();
    s->scal = off;   off += 32 * shplonk_scalars_count(p);
    s->hx = off;     off += 32 * n;
    s->a = off;      off += 32 * n;
    s->b = off;      off += 32 * n;
    s->polys = off;  off += polys_on_host ? 32 * n * P : 0;
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_TRY(dev_malloc(&s->mem, off, "the opening session"));     // the session's destructor frees it on every early return
    const cudaStream_t st = c->stream;
    c->prof.mark(PROF_BEGIN, st);
    for (size_t i = 0; i < P; ++i) {
        if (polys_on_host) {
            void* dst = s->at(s->polys + 32 * n * i);
            H2B_TRY(host_upload(*c, dst, polys[p.used[i]], 32 * n, st));
            s->plan.d_polys.push_back(dst);
        } else {
            s->plan.d_polys.push_back(polys[p.used[i]]);
        }
    }
    if (polys_on_host) c->prof.mark(PROF_OPEN_UPLOAD, st);
    H2B_TRY(shplonk_tables_upload(p, p.d_polys.data(), s->at(s->tables), st));
    H2B_TRY(shplonk_begin_run(*c, p, s->at(s->tables), n, y, v, s->at(s->evals), s->at(s->scal), s->at(s->hx), s->at(s->a), s->at(s->b), st));
    uint64_t h1[12];
    H2B_TRY(session_commit(*c, *s, s->at(s->hx), n, h1));
    {
        std::lock_guard<std::mutex> g(G.mu);
        s->handle = G.next_handle++;
        G.sessions.push_back(s);
    }
    memcpy(out_h1_jac, h1, 96);
    *session = s->handle;
    return H2B_OK;
}

int h2b_shplonk_finish(uint64_t session, const uint64_t u[4], uint64_t out_h2_jac[12]) {
    static const char* who = "h2b_shplonk_finish";
    SessionRef s;
    H2B_TRY(session_lookup(who, session, &s));
    if (!u || !out_h2_jac) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    if (!fr_canonical(u)) { set_error("%s: u is not below the scalar field modulus", who); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> sl(s->mu);
    if (s->finished) { set_error("%s: the session is already finished", who); return H2B_ERR_BAD_ARGUMENT; }
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx((int)s->d, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const cudaStream_t st = c->stream;
    c->prof.mark(PROF_BEGIN, st);
    H2B_TRY(shplonk_finish_run(*c, s->plan, s->at(s->tables), s->n, u, s->at(s->evals), s->at(s->scal), s->at(s->hx), s->at(s->a), s->at(s->b), st));
    H2B_TRY(session_commit(*c, *s, s->at(s->b), s->n - 1, out_h2_jac));
    s->finished = true;
    return H2B_OK;
}

int h2b_shplonk_release(uint64_t session) {
    SessionRef drop;      // freed after G.mu is let go (the destructor waits for the device)
    {
        std::lock_guard<std::mutex> lk(G.mu);
        for (size_t i = 0; i < G.sessions.size(); ++i)
            if (G.sessions[i]->handle == session) { drop = G.sessions[i]; G.sessions.erase(G.sessions.begin() + i); break; }
    }
    if (!drop) { set_error("h2b_shplonk_release: unknown session handle %llu", (unsigned long long)session); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_srs_cache_clear(void) {
    H2B_TRY(require_init());
    std::vector<uint64_t> drop;
    {
        std::lock_guard<std::mutex> lk(G.mu);
        for (const SrsCacheEntry& e : G.srs_cache) { drop.push_back(e.handle_g); drop.push_back(e.handle_g_lagrange); }
        G.srs_cache.clear();
    }
    for (uint64_t h : drop) h2b_unregister_bases(h);
    return H2B_OK;
}

int h2b_srs_write(const char* path, int format, uint32_t k, const uint64_t* g, const uint64_t* g_lagrange, const uint8_t* g2_bytes, size_t g2_len) {
    H2B_TRY(require_init());
    if (!path || !g || !g_lagrange || (g2_len && !g2_bytes) || k > 28) { set_error("h2b_srs_write: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
    if (format < H2B_SERDE_PROCESSED || format > H2B_SERDE_RAW_BYTES_UNCHECKED) { set_error("h2b_srs_write: unknown format %d", format); return H2B_ERR_BAD_ARGUMENT; }
    FileCloser fc{fopen(path, "wb")};
    if (!fc.f) { set_error("h2b_srs_write: cannot create %s", path); return H2B_ERR_BAD_ARGUMENT; }
    const unsigned char kb[4] = {(unsigned char)k, (unsigned char)(k >> 8), (unsigned char)(k >> 16), (unsigned char)(k >> 24)};
    const size_t n = (size_t)1 << k;
    bool ok = fwrite(kb, 1, 4, fc.f) == 4;
    for (const uint64_t* v : {g, g_lagrange}) {
        if (!ok) break;
        if (format != H2B_SERDE_PROCESSED) { ok = fwrite(v, 64, n, fc.f) == n; continue; }
        DeviceCtx& c = *G.devs[0];
        std::lock_guard<std::mutex> lk(c.mu);
        H2B_CUDA(cudaSetDevice(c.device));
        H2B_TRY(c.srs_io.reserve(n * 96));
        std::vector<unsigned char> enc(n * 32);
        H2B_TRY(host_upload(c, c.srs_io.p, v, n * 64, c.stream));
        H2B_TRY(g1_encode_run(c, c.srs_io.p, n, (char*)c.srs_io.p + n * 64, c.stream));
        H2B_TRY(host_download(c, enc.data(), (char*)c.srs_io.p + n * 64, n * 32, c.stream));
        H2B_CUDA(cudaStreamSynchronize(c.stream));
        ok = fwrite(enc.data(), 32, n, fc.f) == n;
    }
    if (ok && g2_len) ok = fwrite(g2_bytes, 1, g2_len, fc.f) == g2_len;
    if (!ok) { set_error("h2b_srs_write: short write to %s", path); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

// ---- quotient evaluation (SURVEY.md 8f rank 2) -----------------------------------------------------------------------
int h2b_evaluate_graph_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_graph_run(*c, graph, cols, d_values, size, rot_scale, nullptr, (cudaStream_t)stream);
}
int h2b_evaluate_graph_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                 const h2b_eval_shard* shard, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!shard) { set_error("h2b_evaluate_graph_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_graph_run(*c, graph, cols, d_values, size, rot_scale, shard, (cudaStream_t)stream);
}

int h2b_evaluate_h_permutation_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                   const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                   int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                   const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                   const uint64_t extended_omega[4], void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_h_permutation_run(*c, d_values, size, rot_scale, d_product_cosets, n_sets, d_columns, d_perm_cosets, n_columns, chunk_len, last_rotation,
                                      d_l0, d_l_last, d_l_active_row, beta, gamma, y, delta, zeta, extended_omega, nullptr, (cudaStream_t)stream);
}
int h2b_evaluate_h_permutation_shard_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                         const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                         int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                         const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                         const uint64_t extended_omega[4], const h2b_eval_shard* shard, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!shard) { set_error("h2b_evaluate_h_permutation_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_h_permutation_run(*c, d_values, size, rot_scale, d_product_cosets, n_sets, d_columns, d_perm_cosets, n_columns, chunk_len, last_rotation,
                                      d_l0, d_l_last, d_l_active_row, beta, gamma, y, delta, zeta, extended_omega, shard, (cudaStream_t)stream);
}

int h2b_evaluate_h_lookup_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                              const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                              const void* d_l_last, const void* d_l_active_row, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_h_lookup_run(*c, graph, cols, d_values, size, rot_scale, d_product_coset, d_permuted_input_coset, d_permuted_table_coset, d_l0, d_l_last,
                                 d_l_active_row, nullptr, (cudaStream_t)stream);
}
int h2b_evaluate_h_lookup_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                    const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                                    const void* d_l_last, const void* d_l_active_row, const h2b_eval_shard* shard, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!shard) { set_error("h2b_evaluate_h_lookup_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return evaluate_h_lookup_run(*c, graph, cols, d_values, size, rot_scale, d_product_coset, d_permuted_input_coset, d_permuted_table_coset, d_l0, d_l_last,
                                 d_l_active_row, shard, (cudaStream_t)stream);
}

int h2b_evaluate_graph_info(uint32_t* slots, uint32_t* micro_ops) {
    evaluate_graph_last_info(slots, micro_ops);
    return H2B_OK;
}

int h2b_dev_alloc(int device, size_t bytes, void** out) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!out) { set_error("h2b_dev_alloc: null out"); return H2B_ERR_BAD_ARGUMENT; }
    return dev_malloc(out, bytes ? bytes : 1, "h2b_dev_alloc");
}
int h2b_dev_free(int device, void* p) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    H2B_CUDA(cudaFree(p));
    return H2B_OK;
}
int h2b_memcpy_h2d(int device, void* d_dst, const void* h_src, size_t bytes) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    // pageable sources go through the pinned staging threads (stage.cu); synchronous like cudaMemcpy
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_CUDA(cudaDeviceSynchronize());            // cudaMemcpy semantics: ordered after everything queued on the device
    H2B_TRY(host_upload(*c, d_dst, h_src, bytes, c->stream));
    H2B_CUDA(cudaStreamSynchronize(c->stream));
    return H2B_OK;
}
// Upload that does not wait for the device: d_dst must not be in use by anything in flight.  Work queued on `stream` after the
// call sees the data; the host buffer may be reused on return (pageable sources are consumed by the staging threads, pinned
// ones must stay valid until the stream reaches the copy, as with cudaMemcpyAsync).
int h2b_memcpy_h2d_async(int device, void* d_dst, const void* h_src, size_t bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (bytes && (!d_dst || !h_src)) { set_error("h2b_memcpy_h2d_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return host_upload(*c, d_dst, h_src, bytes, (cudaStream_t)stream, false);
}
int h2b_memcpy_d2d_async(int device, void* d_dst, const void* d_src, size_t bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (bytes && (!d_dst || !d_src)) { set_error("h2b_memcpy_d2d_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_CUDA(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return H2B_OK;
}
int h2b_memset_zero_async(int device, void* d_dst, size_t bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (bytes && !d_dst) { set_error("h2b_memset_zero_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_CUDA(cudaMemsetAsync(d_dst, 0, bytes, (cudaStream_t)stream));
    return H2B_OK;
}
int h2b_memcpy_d2h(int device, void* h_dst, const void* d_src, size_t bytes) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    H2B_CUDA(cudaDeviceSynchronize());
    return host_download(*c, h_dst, d_src, bytes, c->stream);
}
int h2b_dev_sync(int device) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    H2B_CUDA(cudaDeviceSynchronize());
    return H2B_OK;
}

int h2b_gen_points_dev(int device, uint64_t seed, size_t n, void* d_out_affine, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    return gen_points_run(*c, seed, n, d_out_affine, (cudaStream_t)stream);
}
int h2b_gen_scalars_dev(int device, uint64_t seed, size_t n, int kind, void* d_out, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    return gen_scalars_run(*c, seed, n, kind, d_out, (cudaStream_t)stream);
}

int h2b_msm_checksum_dev(int device, const void* d_scalars, uint64_t seed, uint64_t first, size_t n, void* d_out, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!d_out || (n && !d_scalars)) { set_error("h2b_msm_checksum_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return msm_checksum_run(*c, d_scalars, seed, first, n, d_out, (cudaStream_t)stream);
}

static int elementwise_host(int which, int field, int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out, size_t elem_bytes) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(0, &c));
    if (!a || !b || !out) { set_error("elementwise op: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    if (n == 0) return H2B_OK;
    std::lock_guard<std::mutex> lk(c->mu);
    DevBuf da, db, dout;
    int rc = da.reserve(n * elem_bytes);
    if (!rc) rc = db.reserve(n * elem_bytes);
    if (!rc) rc = dout.reserve(n * elem_bytes);
    if (!rc) {
        cudaMemcpyAsync(da.p, a, n * elem_bytes, cudaMemcpyHostToDevice, c->stream);
        cudaMemcpyAsync(db.p, b, n * elem_bytes, cudaMemcpyHostToDevice, c->stream);
        rc = which == 0 ? field_selftest_run(*c, field, op, da.p, db.p, n, dout.p, c->stream) : ec_selftest_run(*c, op, da.p, db.p, n, dout.p, c->stream);
    }
    if (!rc) {
        cudaMemcpyAsync(out, dout.p, n * elem_bytes, cudaMemcpyDeviceToHost, c->stream);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { set_error("elementwise op: %s", cudaGetErrorString(e)); rc = H2B_ERR_CUDA; }
    }
    da.release(); db.release(); dout.release();
    return rc;
}
int h2b_field_op(int field, int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out) {
    if (field < 0 || field > 1 || op < 0 || op > 12) { set_error("h2b_field_op: bad field/op"); return H2B_ERR_BAD_ARGUMENT; }
    return elementwise_host(0, field, op, a, b, n, out, 32);
}
int h2b_ec_op(int op, const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out) {
    if (op < 0 || op > 5) { set_error("h2b_ec_op: bad op"); return H2B_ERR_BAD_ARGUMENT; }
    return elementwise_host(1, 0, op, p, q, n, out, 64);
}

int h2b_imad_bench(int device, int kind, int iters, float* ms_out, double* ops_out) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!ms_out || !ops_out) { set_error("h2b_imad_bench: null output"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    return imad_bench_run(*c, kind, iters, c->sm_count * 8, 256, ms_out, ops_out, c->stream);
}

int h2b_set_msm_window(int c) { return msm_set_window(c); }

unsigned long long h2b_launch_count(void) { return __atomic_load_n(&g_launch_count, __ATOMIC_RELAXED); }

int h2b_profile_enable(int device, int on) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    Profiler& p = c->prof;
    if (on && p.ev.empty()) {
        p.ev.resize(8192);
        p.tag.resize(8192);
        for (auto& e : p.ev) H2B_CUDA(cudaEventCreate(&e));
    }
    p.enabled = on != 0;
    p.used = 0;
    return H2B_OK;
}

int h2b_profile_read(int device, int* tags, float* ms, int cap, int* count) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    if (!tags || !ms || !count) { set_error("h2b_profile_read: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    std::lock_guard<std::mutex> lk(c->mu);
    Profiler& p = c->prof;
    H2B_CUDA(cudaDeviceSynchronize());
    int n = 0;
    for (size_t i = 1; i < p.used && n < cap; ++i) {
        if (p.tag[i] == PROF_BEGIN) continue;
        float t = 0.f;
        H2B_CUDA(cudaEventElapsedTime(&t, p.ev[i - 1], p.ev[i]));
        tags[n] = p.tag[i];
        ms[n] = t;
        ++n;
    }
    *count = n;
    p.used = 0;
    return H2B_OK;
}

}  // extern "C"
