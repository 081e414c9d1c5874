// Internal to the C ABI's host layer (the api*.cu files): what more than one of them uses.  The public interface is include/h2b200.h.
#pragma once
#include <atomic>
#include <memory>

#include "common.h"

namespace h2b {

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

struct ResidentPk;       // a proving key held on the devices (api_keygen.cu: h2b_pk_create)
struct ShplonkSession;   // a multi-point opening between its two commitments (api_open.cu: h2b_shplonk_begin)

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

// The objects of one kind handed out under a handle (base sets, resident proving keys, opening sessions).  Guarded by G.mu; every
// kind draws its handles from G.next_handle.  take() gives the entry back so that its last reference, whose destructor frees device
// memory, can be dropped after G.mu is let go.  The *_locked forms are for callers that hold G.mu.
template <class T> struct Handles {
    std::vector<std::shared_ptr<T>> all;
    std::shared_ptr<T> find_locked(uint64_t handle) const {
        for (auto& p : all) if (p->handle == handle) return p;
        return nullptr;
    }
    std::shared_ptr<T> take_locked(uint64_t handle) {
        for (size_t i = 0; i < all.size(); ++i)
            if (all[i]->handle == handle) { std::shared_ptr<T> p = all[i]; all.erase(all.begin() + i); return p; }
        return nullptr;
    }
    uint64_t publish_locked(const std::shared_ptr<T>& p);
    std::shared_ptr<T> find(uint64_t handle);
    uint64_t publish(const std::shared_ptr<T>& p);
    std::shared_ptr<T> take(uint64_t handle);
};

struct Global {
    std::mutex mu;
    std::vector<std::unique_ptr<DeviceCtx>> devs;
    Handles<BaseSet> sets;
    Handles<ResidentPk> pks;
    Handles<ShplonkSession> sessions;
    std::vector<SrsCacheEntry> srs_cache;
    uint64_t next_handle = 1;
    uint64_t use_counter = 0;
    std::atomic<unsigned> rr{0};
    std::atomic<unsigned long long> implicit_uploads{0}, implicit_hits{0}, implicit_stale{0}, direct_calls{0};
};
extern Global G;   // api.cu

template <class T> uint64_t Handles<T>::publish_locked(const std::shared_ptr<T>& p) {
    p->handle = G.next_handle++;
    all.push_back(p);
    return p->handle;
}
template <class T> std::shared_ptr<T> Handles<T>::find(uint64_t h) { std::lock_guard<std::mutex> lk(G.mu); return find_locked(h); }
template <class T> uint64_t Handles<T>::publish(const std::shared_ptr<T>& p) { std::lock_guard<std::mutex> lk(G.mu); return publish_locked(p); }
template <class T> std::shared_ptr<T> Handles<T>::take(uint64_t h) { std::lock_guard<std::mutex> lk(G.mu); return take_locked(h); }

// ---- the devices --------------------------------------------------------------------------------------------------------------
inline int require_init() {
    if (G.devs.empty()) { set_error("h2b200 is not initialised (call h2b_init)"); return H2B_ERR_NOT_INITIALIZED; }
    return H2B_OK;
}
inline int get_ctx(int device, DeviceCtx** out) {
    H2B_TRY(require_init());
    if (device < 0 || (size_t)device >= G.devs.size()) { set_error("device index %d out of range (have %zu)", device, G.devs.size()); return H2B_ERR_BAD_ARGUMENT; }
    *out = G.devs[device].get();
    H2B_CUDA(cudaSetDevice((*out)->device));
    return H2B_OK;
}

// The lock rule.  A device's context holds scratch buffers and tables that every call on that device shares, so an entry point holds
// the device's lock (DeviceCtx::mu) while it enqueues work there.  An entry point given a device index gets there through on_device.
// The only ones that take no device lock are those that touch no DeviceCtx state: h2b_dev_alloc, h2b_dev_free, h2b_dev_sync,
// h2b_memcpy_d2d_async and h2b_memset_zero_async.
// Lock order: G.mu before any device lock, device locks in index order.  G.mu is never taken while a device lock is held, and no entry
// point calls another entry point while it holds one.

// fn(c) on device `device` with its lock held.  `unlocked()` runs first, without the lock: the argument checks that look a handle up
// under G.mu.  A SetRef it fills belongs to the caller, so it is released after the device lock.
template <class U, class F> int on_device(int device, U&& unlocked, F&& fn) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));
    H2B_TRY(unlocked());
    std::lock_guard<std::mutex> lk(c->mu);
    return fn(*c);
}
template <class F> int on_device(int device, F&& fn) {
    return on_device(device, [] { return H2B_OK; }, fn);
}

// pick a device for a single-device call: round robin, preferring one that is idle
DeviceCtx* pick_device(std::unique_lock<std::mutex>& lock_out, size_t* index = nullptr);
// fn(d) for every device index d in `devs`: on the calling thread when there is one, on one thread per device otherwise.  Returns
// the first failure in list order, its message prefixed with "device d: ".
int on_devices(const std::vector<size_t>& devs, const std::function<int(size_t)>& fn);
std::vector<size_t> first_devices(size_t m);
// every device allocation of the host layer (clears the runtime's error of a failed cudaMalloc)
int dev_malloc(void** p, size_t bytes, const char* what);

// ---- resident sets (api_sets.cu) ----------------------------------------------------------------------------------------------
// One point vector made on device 0: `produce` fills n x 64 B on device 0's stream; the points are downloaded to host_out (may be
// null), then registered under *handle as a replicated set with window tables (handle may be null: the points are dropped).
// release_g1gen: the producer runs g1gen.cu kernels whose scratch is given back once they are done.  Errors read "caller: what: ...".
// Caller holds G.mu.
int device0_points_locked(size_t n, const char* caller, const char* what, bool release_g1gen, const std::function<int(DeviceCtx&, void*)>& produce,
                          uint64_t* host_out, uint64_t* handle);
int registered_set(const char* who, uint64_t handle, size_t offset, size_t n, SetRef* out);
int msm_host(const uint64_t* scalars, const BaseSet& bs, size_t offset, size_t n, uint64_t out_jac[12]);

inline MsmBases bases_of(const BaseSet& bs, size_t d, size_t row /* global row of the first point */) {
    MsmBases b;
    b.tables = bs.dev[d];
    b.n_tables = bs.n_tables;
    b.c0 = bs.c0;
    b.stride = bs.rows[d];
    b.row0 = row - bs.lo[d];
    return b;
}

// columns up to this length share one kernel sequence per device in the batched MSMs; longer columns run one by one
static const size_t BATCH_COLUMN_MAX = (size_t)1 << 21;

// the sizes of a coset conversion
inline int extended_k_check(const char* who, uint32_t k, uint32_t extended_k) {
    if (extended_k < k || extended_k > 28) { set_error("%s: need k <= extended_k <= 28", who); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

}  // namespace h2b
