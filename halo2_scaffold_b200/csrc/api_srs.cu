// C ABI of libh2b200, the SRS: h2b_srs_read / h2b_srs_write (params/kzg_bn254_{k}.srs, with a cache of decoded files),
// ParamsKZG::setup and ParamsKZG::downsize on the device.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "host.h"

namespace h2b {

namespace {
struct FileCloser { FILE* f; ~FileCloser() { if (f) fclose(f); } };
}  // namespace

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
    SetRef bs = G.sets.find(handle);
    if (!bs || bs->n != n || bs->sharded) { set_error("h2b_srs_read: cached base set vanished"); return H2B_ERR_BAD_HANDLE; }
    const void* src = bs->dev[0];
    DeviceCtx& c = *G.devs[0];
    std::lock_guard<std::mutex> lk(c.mu);
    H2B_CUDA(cudaSetDevice(c.device));
    H2B_TRY(host_download(c, out, src, n * 64, c.stream));
    H2B_CUDA(cudaStreamSynchronize(c.stream));
    return H2B_OK;
}

}  // namespace h2b

using namespace h2b;

extern "C" {

// ---- SRS on-disk format (SURVEY.md 8f rank 4) -----------------------------------------------------------------------------
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
                SetRef a = G.sets.find_locked(e.handle_g), b = G.sets.find_locked(e.handle_g_lagrange);
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
        SetRef a = G.sets.find_locked(hg), b = G.sets.find_locked(hl);
        if (a && handle_g) ++a->refs;
        if (b && handle_g_lagrange) ++b->refs;
        // a stale entry for the same path (file rewritten) gives its sets back
        for (size_t i = 0; i < G.srs_cache.size();) {
            if (G.srs_cache[i].path == e.path && G.srs_cache[i].format == e.format) {
                for (uint64_t h : {G.srs_cache[i].handle_g, G.srs_cache[i].handle_g_lagrange}) {
                    SetRef old = G.sets.find_locked(h);
                    if (old && --old->refs <= 0) G.sets.take_locked(h);
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

int h2b_srs_downsize(uint64_t handle_g, uint32_t k, uint64_t* out_g_lagrange, uint64_t* handle_g_out, uint64_t* handle_g_lagrange_out) {
    H2B_TRY(require_init());
    if (k > 28) { set_error("h2b_srs_downsize: k = %u (at most 28)", k); return H2B_ERR_BAD_ARGUMENT; }
    const size_t n = (size_t)1 << k;
    std::lock_guard<std::mutex> glk(G.mu);
    SetRef src = G.sets.find_locked(handle_g);
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
            if (hg) G.sets.take_locked(hg);
            return rc;
        }
    }
    if (handle_g_out) *handle_g_out = hg;
    if (handle_g_lagrange_out) *handle_g_lagrange_out = hl;
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

}  // extern "C"
