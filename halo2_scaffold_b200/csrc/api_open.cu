// C ABI of libh2b200, the multi-point openings: SHPLONK (h2b_fr_eval_queries_dev and the h2b_shplonk_* session) and GWC
// (h2b_gwc_create_proof).
#include "host.h"

namespace h2b {

// One opening between h1 and h2 on one device.  Device memory, one block: the plan's tables | pair values | scalars | h_x | two
// n-coefficient work buffers | the uploaded polynomials of a host-pointer session.  The work buffers hold h' after finish.
struct ShplonkSession {
    uint64_t handle = 0;
    size_t d = 0, n = 0;
    int ordinal = -1;
    SetRef g;                 // held for the session's life: finish commits over it
    ShplonkPlan plan;
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
    *out = G.sessions.find(handle);
    if (*out) return H2B_OK;
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

}  // namespace h2b

using namespace h2b;

extern "C" {

int h2b_fr_eval_queries_dev(int device, const void* const* d_polys, uint32_t n_polys, size_t n, const h2b_opening_query* queries, uint32_t n_queries,
                            void* d_out, void* stream) {
    static const char* who = "h2b_fr_eval_queries_dev";
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_polys || !d_out) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(shplonk_n_check(who, n));
        ShplonkPlan plan;
        H2B_TRY(shplonk_plan_build(who, queries, n_queries, n_polys, true, &plan));
        for (uint32_t s : plan.used) {
            if (!d_polys[s]) { set_error("%s: polynomial %u is a null pointer", who, s); return H2B_ERR_BAD_ARGUMENT; }
            plan.d_polys.push_back(d_polys[s]);
        }
        const size_t tb = shplonk_tables_bytes(plan);
        H2B_TRY(c.open_tables.reserve(tb + plan.pair_point.size() * 32));
        const cudaStream_t st = (cudaStream_t)stream;
        H2B_TRY(shplonk_tables_upload(plan, plan.d_polys.data(), c.open_tables.p, st));
        return shplonk_eval_queries_run(c, plan, c.open_tables.p, n, (char*)c.open_tables.p + tb, d_out, st);
    });
}

int h2b_shplonk_begin(int device, const void* const* polys, int polys_on_host, uint32_t n_polys, size_t n, const h2b_opening_query* queries,
                      uint32_t n_queries, uint64_t handle_g, const uint64_t y[4], const uint64_t v[4], uint64_t out_h1_jac[12], uint64_t* session) {
    static const char* who = "h2b_shplonk_begin";
    SessionRef s(new ShplonkSession());      // released after the device lock: its destructor frees the block on every early return
    uint64_t h1[12];
    H2B_TRY(on_device(device, [&]() -> int {
        if (!polys || !y || !v || !out_h1_jac || !session) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(shplonk_n_check(who, n));
        if (!fr_canonical(y) || !fr_canonical(v)) { set_error("%s: a challenge is not below the scalar field modulus", who); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(shplonk_plan_build(who, queries, n_queries, n_polys, true, &s->plan));
        for (uint32_t i = 0; i < n_polys; ++i) if (!polys[i]) { set_error("%s: polynomial %u is a null pointer", who, i); return H2B_ERR_BAD_ARGUMENT; }
        s->g = G.sets.find(handle_g);
        if (!s->g) { set_error("%s: unknown base-set handle %llu", who, (unsigned long long)handle_g); return H2B_ERR_BAD_ARGUMENT; }
        s->d = (size_t)device;
        if (s->g->lo[s->d] != 0 || s->g->rows[s->d] < n) { set_error("%s: device %d does not hold rows [0, %zu) of the set", who, device, n); return H2B_ERR_BAD_ARGUMENT; }
        return H2B_OK;
    }, [&](DeviceCtx& c) -> int {
        s->n = n;
        s->ordinal = c.device;
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
        H2B_TRY(dev_malloc(&s->mem, off, "the opening session"));
        const cudaStream_t st = c.stream;
        c.prof.mark(PROF_BEGIN, st);
        for (size_t i = 0; i < P; ++i) {
            if (polys_on_host) {
                void* dst = s->at(s->polys + 32 * n * i);
                H2B_TRY(host_upload(c, dst, polys[p.used[i]], 32 * n, st));
                s->plan.d_polys.push_back(dst);
            } else {
                s->plan.d_polys.push_back(polys[p.used[i]]);
            }
        }
        if (polys_on_host) c.prof.mark(PROF_OPEN_UPLOAD, st);
        H2B_TRY(shplonk_tables_upload(p, p.d_polys.data(), s->at(s->tables), st));
        H2B_TRY(shplonk_begin_run(c, p, s->at(s->tables), n, y, v, s->at(s->evals), s->at(s->scal), s->at(s->hx), s->at(s->a), s->at(s->b), st));
        return session_commit(c, *s, s->at(s->hx), n, h1);
    }));
    memcpy(out_h1_jac, h1, 96);
    *session = G.sessions.publish(s);      // after the device lock: G.mu is never taken under one
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
    return on_device((int)s->d, [&](DeviceCtx& c) -> int {
        const cudaStream_t st = c.stream;
        c.prof.mark(PROF_BEGIN, st);
        H2B_TRY(shplonk_finish_run(c, s->plan, s->at(s->tables), s->n, u, s->at(s->evals), s->at(s->scal), s->at(s->hx), s->at(s->a), s->at(s->b), st));
        H2B_TRY(session_commit(c, *s, s->at(s->b), s->n - 1, out_h2_jac));
        s->finished = true;
        return H2B_OK;
    });
}

int h2b_shplonk_release(uint64_t session) {
    SessionRef drop = G.sessions.take(session);      // freed after G.mu is let go (the destructor waits for the device)
    if (!drop) { set_error("h2b_shplonk_release: unknown session handle %llu", (unsigned long long)session); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

int h2b_gwc_create_proof(int device, const void* const* polys, int polys_on_host, uint32_t n_polys, size_t n, const h2b_opening_query* queries,
                         uint32_t n_queries, uint64_t handle_g, const uint64_t v[4], uint64_t* out_w_jac, uint32_t capacity, uint32_t* out_points) {
    static const char* who = "h2b_gwc_create_proof";
    GwcPlan plan;
    SetRef g;      // declared before the device lock: released after it
    H2B_TRY(on_device(device, [&]() -> int {
        if (!polys || !v || !out_w_jac || !out_points) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(shplonk_n_check(who, n));
        if (!fr_canonical(v)) { set_error("%s: v is not below the scalar field modulus", who); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(gwc_plan_build(who, queries, n_queries, n_polys, &plan));
        for (uint32_t i = 0; i < n_polys; ++i) if (!polys[i]) { set_error("%s: polynomial %u is a null pointer", who, i); return H2B_ERR_BAD_ARGUMENT; }
        g = G.sets.find(handle_g);
        if (!g) { set_error("%s: unknown base-set handle %llu", who, (unsigned long long)handle_g); return H2B_ERR_BAD_ARGUMENT; }
        if (g->lo[(size_t)device] != 0 || g->rows[(size_t)device] < n - 1) {
            set_error("%s: device %d does not hold rows [0, %zu) of the set", who, device, n - 1);
            return H2B_ERR_BAD_ARGUMENT;
        }
        if (capacity < plan.n_points()) { set_error("%s: capacity %u < %u distinct points", who, capacity, plan.n_points()); return H2B_ERR_BAD_ARGUMENT; }
        return H2B_OK;
    }, [&](DeviceCtx& c) -> int {
        // the call's block: the work of gwc_run | the uploaded polynomials of a host-pointer call
        const size_t work = gwc_work_bytes(plan, n), upload = polys_on_host ? 32 * n * n_polys : 0;
        struct Block {
            void* p = nullptr;
            ~Block() { if (p) { cudaDeviceSynchronize(); cudaFree(p); cudaGetLastError(); } }
        } mem;
        H2B_TRY(dev_malloc(&mem.p, work + upload, "the GWC opening"));
        const cudaStream_t st = c.stream;
        c.prof.mark(PROF_BEGIN, st);
        std::vector<const void*> d_polys(polys, polys + n_polys);
        if (polys_on_host) {
            for (uint32_t i = 0; i < n_polys; ++i) {
                void* dst = (char*)mem.p + work + 32 * n * i;
                H2B_TRY(host_upload(c, dst, polys[i], 32 * n, st));
                d_polys[i] = dst;
            }
            c.prof.mark(PROF_GWC_UPLOAD, st);
        }
        std::vector<uint64_t> w(12 * (size_t)plan.n_points());
        H2B_TRY(gwc_run(c, plan, d_polys.data(), n, v, bases_of(*g, (size_t)device, 0), mem.p, w.data(), st));
        memcpy(out_w_jac, w.data(), 8 * w.size());
        *out_points = plan.n_points();
        return H2B_OK;
    }));
    return H2B_OK;
}

}  // extern "C"
