// C ABI of libh2b200 (declared in include/h2b200.h): lifecycle and errors, the device-pointer entry points, device memory, synthetic
// workloads, diagnostics and profiling.  The rest of the ABI: api_sets.cu (resident base sets, host-pointer MSM / NTT), api_srs.cu
// (SRS files, setup, downsize), api_keygen.cu (keygen and the resident proving key), api_open.cu (the SHPLONK opening).
#include <thread>

#include "host.h"

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

Global G;

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

DeviceCtx* pick_device(std::unique_lock<std::mutex>& lock_out, size_t* index) {
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

int on_devices(const std::vector<size_t>& devs, const std::function<int(size_t)>& fn) {
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
std::vector<size_t> first_devices(size_t m) {
    std::vector<size_t> devs(m);
    for (size_t d = 0; d < m; ++d) devs[d] = d;
    return devs;
}

// A failed cudaMalloc stays the thread's last error, which the next launch check on this thread would report as its own: it is
// cleared here.
int dev_malloc(void** p, size_t bytes, const char* what) {
    const cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) return H2B_OK;
    cudaGetLastError();
    *p = nullptr;
    set_error("cudaMalloc of %zu bytes for %s failed: %s", bytes, what, cudaGetErrorString(e));
    return H2B_ERR_OOM;
}

// the number of visible devices; h2b200 has no CPU fallback
static int visible_devices(int* count) {
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess || *count <= 0) {
        set_error("no usable CUDA device (%s); h2b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return H2B_ERR_NO_DEVICE;
    }
    return H2B_OK;
}

static int elementwise_host(int which, int field, int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out, size_t elem_bytes) {
    return on_device(0, [&](DeviceCtx& c) -> int {
        if (!a || !b || !out) { set_error("elementwise op: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        if (n == 0) return H2B_OK;
        DevBuf da, db, dout;
        int rc = da.reserve(n * elem_bytes);
        if (!rc) rc = db.reserve(n * elem_bytes);
        if (!rc) rc = dout.reserve(n * elem_bytes);
        if (!rc) {
            cudaMemcpyAsync(da.p, a, n * elem_bytes, cudaMemcpyHostToDevice, c.stream);
            cudaMemcpyAsync(db.p, b, n * elem_bytes, cudaMemcpyHostToDevice, c.stream);
            rc = which == 0 ? field_selftest_run(c, field, op, da.p, db.p, n, dout.p, c.stream) : ec_selftest_run(c, op, da.p, db.p, n, dout.p, c.stream);
        }
        if (!rc) {
            cudaMemcpyAsync(out, dout.p, n * elem_bytes, cudaMemcpyDeviceToHost, c.stream);
            cudaError_t e = cudaStreamSynchronize(c.stream);
            if (e != cudaSuccess) { set_error("elementwise op: %s", cudaGetErrorString(e)); rc = H2B_ERR_CUDA; }
        }
        da.release(); db.release(); dout.release();
        return rc;
    });
}

}  // namespace h2b

using namespace h2b;

extern "C" {

int h2b_init(int n_devices) {
    if (!G.devs.empty()) return H2B_OK;
    int count = 0;
    H2B_TRY(visible_devices(&count));
    if (n_devices < 0 || n_devices > count) { set_error("h2b_init(%d): only %d device(s) visible", n_devices, count); return H2B_ERR_BAD_ARGUMENT; }
    if (n_devices == 0) n_devices = count;
    std::vector<int> ords;
    for (int i = 0; i < n_devices; ++i) ords.push_back(i);
    return init_devices(ords);
}

int h2b_init_device(int device) {
    if (!G.devs.empty()) return H2B_OK;
    int count = 0;
    H2B_TRY(visible_devices(&count));
    if (device < 0 || device >= count) { set_error("h2b_init_device(%d): only %d device(s) visible", device, count); return H2B_ERR_BAD_ARGUMENT; }
    return init_devices(std::vector<int>{device});
}

void h2b_shutdown(void) {
    std::lock_guard<std::mutex> lk(G.mu);
    G.sets.all.clear();      // device memory goes when the last holder lets go (now, unless a call is still in flight)
    G.pks.all.clear();
    G.sessions.all.clear();
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

int h2b_ntt_bn254_fr_dev_batch(int device, void* const* d_polys, size_t count, const uint64_t omega[4], uint32_t log_n, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (count == 0) return H2B_OK;
        if (!d_polys || !omega) { set_error("h2b_ntt_bn254_fr_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        return ntt_run_batch(c, d_polys, count, omega, log_n, (cudaStream_t)stream);
    });
}

int h2b_ntt_bn254_fr_dev(int device, void* d_a, const uint64_t omega[4], uint32_t log_n, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!omega) { set_error("h2b_ntt_bn254_fr_dev: null omega"); return H2B_ERR_BAD_ARGUMENT; }
        return ntt_run(c, d_a, omega, log_n, (cudaStream_t)stream);
    });
}

int h2b_msm_bn254_g1_dev(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_jac, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_out_jac) { set_error("h2b_msm_bn254_g1_dev: null output"); return H2B_ERR_BAD_ARGUMENT; }
        MsmBases b;
        b.tables = d_bases;
        b.stride = n;
        return msm_run(c, d_scalars, b, n, d_out_jac, false, (cudaStream_t)stream);
    });
}

int h2b_msm_bn254_g1_dev_partial(int device, const void* d_scalars, const void* d_bases, size_t n, void* d_out_block, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_out_block) { set_error("h2b_msm_bn254_g1_dev_partial: null output"); return H2B_ERR_BAD_ARGUMENT; }
        MsmBases b;
        b.tables = d_bases;
        b.stride = n;
        return msm_run(c, d_scalars, b, n, d_out_block, true, (cudaStream_t)stream);
    });
}

int h2b_msm_bn254_g1_dev_registered(int device, const void* d_scalars, uint64_t handle, size_t offset, size_t n, void* d_out_block, void* stream) {
    SetRef bs;      // declared before the device lock: released after it
    const size_t d = (size_t)device;
    return on_device(device, [&]() -> int {
        if (!d_out_block) { set_error("h2b_msm_bn254_g1_dev_registered: null output"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(registered_set("h2b_msm_bn254_g1_dev_registered", handle, offset, n, &bs));
        if (n && (offset < bs->lo[d] || offset + n > bs->lo[d] + bs->rows[d])) {
            set_error("h2b_msm_bn254_g1_dev_registered: device %d holds rows [%zu, %zu) of this sharded set, not [%zu, %zu)", device, bs->lo[d], bs->lo[d] + bs->rows[d], offset, offset + n);
            return H2B_ERR_BAD_ARGUMENT;
        }
        return H2B_OK;
    }, [&](DeviceCtx& c) {
        // asynchronous: the set must stay registered until the caller has synchronised `stream`
        return msm_run(c, d_scalars, bases_of(*bs, d, offset), n, d_out_block, true, (cudaStream_t)stream);
    });
}

int h2b_msm_bn254_g1_dev_batch_registered(int device, const void* const* d_scalars, const size_t* lens, size_t count, uint64_t handle, void* d_out_blocks, void* stream) {
    SetRef bs;      // declared before the device lock: released after it
    const size_t d = (size_t)device;
    return on_device(device, [&]() -> int {
        if (count == 0) return H2B_OK;
        if (!d_scalars || !lens || !d_out_blocks) { set_error("h2b_msm_bn254_g1_dev_batch_registered: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(registered_set("h2b_msm_bn254_g1_dev_batch_registered", handle, 0, 0, &bs));
        size_t n_max = 0;
        for (size_t j = 0; j < count; ++j) n_max = lens[j] > n_max ? lens[j] : n_max;
        if (bs->lo[d] != 0 || n_max > bs->rows[d]) { set_error("h2b_msm_bn254_g1_dev_batch_registered: device %d does not hold rows [0, %zu) of the set", device, n_max); return H2B_ERR_BAD_ARGUMENT; }
        return H2B_OK;
    }, [&](DeviceCtx& c) -> int {
        for (size_t j0 = 0; j0 < count; j0 += msm_batch_max()) {
            const size_t m = count - j0 < msm_batch_max() ? count - j0 : msm_batch_max();
            H2B_TRY(msm_run_batch(c, d_scalars + j0, lens + j0, (uint32_t)m, bases_of(*bs, d, 0), (char*)d_out_blocks + 224 * j0, (cudaStream_t)stream));
        }
        return H2B_OK;
    });
}

int h2b_msm_fold_partials(int device, const uint64_t* host_blocks, size_t count, uint64_t out_jac[12]) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!host_blocks || !out_jac || count == 0 || count > 4096) { set_error("h2b_msm_fold_partials: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(c.msm_scalars.reserve(224 * count));
        H2B_TRY(c.msm_out.reserve(256));
        H2B_CUDA(cudaMemcpyAsync(c.msm_scalars.p, host_blocks, 224 * count, cudaMemcpyHostToDevice, c.stream));
        H2B_TRY(msm_sum_partials_run(c, c.msm_scalars.p, (uint32_t)count, c.msm_out.p, c.stream));
        H2B_CUDA(cudaMemcpyAsync(out_jac, c.msm_out.p, 96, cudaMemcpyDeviceToHost, c.stream));
        H2B_CUDA(cudaStreamSynchronize(c.stream));
        return H2B_OK;
    });
}

int h2b_msm_fold_partials_dev(int device, const void* d_blocks, size_t count, void* d_out_jac, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_blocks || !d_out_jac || count == 0 || count > 4096) { set_error("h2b_msm_fold_partials_dev: bad argument"); return H2B_ERR_BAD_ARGUMENT; }
        return msm_sum_partials_run(c, d_blocks, (uint32_t)count, d_out_jac, (cudaStream_t)stream);
    });
}

int h2b_fr_scale_dev(int device, void* d_a, size_t n, const uint64_t* factors, int count, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!factors || (n && !d_a)) { set_error("h2b_fr_scale_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        return ntt_scale_run(c, d_a, n, factors, count, (cudaStream_t)stream);
    });
}

// ---- EvaluationDomain on the device ([UP] halo2_proofs/src/poly/domain.rs; SURVEY.md row a6) --------------------------
// The column stays in device memory between the scaling, padding and transform steps of each conversion; the constants
// (omega, divisors, zeta) are the caller's: EvaluationDomain::new computes them once per domain on the host.
int h2b_lagrange_to_coeff_dev(int device, void* d_a, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4], void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_a || !omega_inv || !ifft_divisor) { set_error("h2b_lagrange_to_coeff_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(ntt_run(c, d_a, omega_inv, k, (cudaStream_t)stream));
        return ntt_scale_run(c, d_a, (size_t)1 << k, ifft_divisor, 1, (cudaStream_t)stream);
    });
}

int h2b_coeff_to_extended_dev(int device, void* d_a, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4], const uint64_t zeta_powers[12],
                              void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_a || !extended_omega || !zeta_powers) { set_error("h2b_coeff_to_extended_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(extended_k_check("h2b_coeff_to_extended_dev", k, extended_k));
        const size_t n = (size_t)1 << k, en = (size_t)1 << extended_k;
        H2B_TRY(ntt_scale_run(c, d_a, n, zeta_powers, 3, (cudaStream_t)stream));                         // a[i] *= zeta^(i mod 3)
        if (en > n) H2B_CUDA(cudaMemsetAsync((char*)d_a + n * 32, 0, (en - n) * 32, (cudaStream_t)stream));   // zero-pad
        return ntt_run(c, d_a, extended_omega, extended_k, (cudaStream_t)stream);
    });
}

// The two conversions every witness / product column goes through, for `count` columns at once: the (i)NTT passes and the scaling
// are launched once for the whole batch (polynomial index in blockIdx.y).  d_cols: host array of device pointers.
int h2b_lagrange_to_coeff_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, const uint64_t omega_inv[4], const uint64_t ifft_divisor[4],
                                    void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (count == 0) return H2B_OK;
        if (!d_cols || !omega_inv || !ifft_divisor) { set_error("h2b_lagrange_to_coeff_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        return lagrange_to_coeff_batch_run(c, d_cols, count, k, omega_inv, ifft_divisor, (cudaStream_t)stream);
    });
}

int h2b_coeff_to_extended_dev_batch(int device, void* const* d_cols, size_t count, uint32_t k, uint32_t extended_k, const uint64_t extended_omega[4],
                                    const uint64_t zeta_powers[12], void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (count == 0) return H2B_OK;
        if (!d_cols || !extended_omega || !zeta_powers) { set_error("h2b_coeff_to_extended_dev_batch: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(extended_k_check("h2b_coeff_to_extended_dev_batch", k, extended_k));
        return coeff_to_extended_batch_run(c, d_cols, count, k, extended_k, extended_omega, zeta_powers, (cudaStream_t)stream);
    });
}

int h2b_extended_to_coeff_dev(int device, void* d_a, uint32_t extended_k, const uint64_t extended_omega_inv[4], const uint64_t factors[12], void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_a || !extended_omega_inv || !factors) { set_error("h2b_extended_to_coeff_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        H2B_TRY(ntt_run(c, d_a, extended_omega_inv, extended_k, (cudaStream_t)stream));
        // factors[j] = extended_ifft_divisor * (1, zeta^-1, zeta^-2)[j]: one pass undoes the scaling and the coset
        return ntt_scale_run(c, d_a, (size_t)1 << extended_k, factors, 3, (cudaStream_t)stream);
    });
}

// ---- grand-product building blocks (SURVEY.md 8f rank 3) ---------------------------------------------------------------
int h2b_fr_batch_invert_dev(int device, void* d_a, size_t n, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return fr_batch_invert_run(c, d_a, n, (cudaStream_t)stream); });
}

int h2b_fr_prefix_product_dev(int device, const void* d_in, void* d_out, size_t n, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return fr_prefix_product_run(c, d_in, d_out, n, (cudaStream_t)stream); });
}

int h2b_fr_eval_polynomial_dev(int device, const void* d_coeffs, size_t n, const uint64_t x[4], void* d_out, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return fr_eval_polynomial_run(c, d_coeffs, n, x, d_out, (cudaStream_t)stream); });
}

int h2b_fr_kate_division_dev(int device, const void* d_a, size_t n, const uint64_t b[4], void* d_q, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return fr_kate_division_run(c, d_a, n, b, d_q, (cudaStream_t)stream); });
}

int h2b_fr_kate_division_batch_dev(int device, const void* d_a, size_t n, const void* d_points, uint32_t count, void* d_q, void* stream) {
    return on_device(device, [&](DeviceCtx& c) {
        return fr_kate_division_batch_run(c, d_a, n, d_points, count, d_q, (cudaStream_t)stream);
    });
}

int h2b_fr_lincomb_dev(int device, const void* const* d_cols, const uint64_t* coeffs, uint32_t m, size_t n, void* d_out, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return fr_lincomb_run(c, d_cols, coeffs, m, n, d_out, (cudaStream_t)stream); });
}

int h2b_fr_transpose_dev(int device, const void* d_in, void* d_out, uint32_t rows, uint32_t cols, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if ((rows && cols) && (!d_in || !d_out || d_in == d_out)) { set_error("h2b_fr_transpose_dev: null or aliased buffers"); return H2B_ERR_BAD_ARGUMENT; }
        return fr_transpose_run(c, d_in, d_out, rows, cols, (cudaStream_t)stream);
    });
}

int h2b_permutation_product_dev(int device, const void* const* d_values, const void* const* d_permutations, uint32_t n_columns, size_t n,
                                const uint64_t beta[4], const uint64_t gamma[4], const uint64_t delta[4], const uint64_t deltaomega[4], const uint64_t omega[4],
                                const uint64_t last_z[4], void* d_z, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        return permutation_product_run(c, d_values, d_permutations, n_columns, n, beta, gamma, delta, deltaomega, omega, last_z, d_z, (cudaStream_t)stream);
    });
}

int h2b_lookup_product_dev(int device, const void* d_compressed_input, const void* d_compressed_table, const void* d_permuted_input,
                           const void* d_permuted_table, size_t n, const uint64_t beta[4], const uint64_t gamma[4], void* d_z, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        return lookup_product_run(c, d_compressed_input, d_compressed_table, d_permuted_input, d_permuted_table, n, beta, gamma, d_z, (cudaStream_t)stream);
    });
}

int h2b_lookup_permute_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                           void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        return lookup_permute_run(c, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, nullptr, (cudaStream_t)stream);
    });
}

int h2b_lookup_permute_async_dev(int device, const void* d_input, const void* d_table, uint32_t usable_rows, void* d_permuted_input, void* d_permuted_table,
                                 void* d_status, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_status) { set_error("h2b_lookup_permute_async_dev: null status word"); return H2B_ERR_BAD_ARGUMENT; }
        return lookup_permute_run(c, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, d_status, (cudaStream_t)stream);
    });
}

int h2b_g1_decode_dev(int device, const void* d_bytes, size_t n, int format, void* d_out_affine, uint64_t* first_invalid, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return g1_decode_run(c, d_bytes, n, format, d_out_affine, first_invalid, (cudaStream_t)stream); });
}

int h2b_g1_encode_dev(int device, const void* d_affine, size_t n, void* d_out_bytes, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return g1_encode_run(c, d_affine, n, d_out_bytes, (cudaStream_t)stream); });
}

int h2b_g1_generator_mul_dev(int device, const void* d_scalars, size_t n, void* d_out_affine, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return g1_generator_mul_run(c, d_scalars, n, d_out_affine, (cudaStream_t)stream); });
}

int h2b_g1_to_lagrange_dev(int device, const void* d_g_affine, uint32_t k, void* d_out_affine, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return g1_to_lagrange_run(c, d_g_affine, k, d_out_affine, (cudaStream_t)stream); });
}

// ---- quotient evaluation (SURVEY.md 8f rank 2) -----------------------------------------------------------------------
int h2b_evaluate_graph_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return evaluate_graph_run(c, graph, cols, d_values, size, rot_scale, nullptr, (cudaStream_t)stream); });
}
int h2b_evaluate_graph_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                 const h2b_eval_shard* shard, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!shard) { set_error("h2b_evaluate_graph_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
        return evaluate_graph_run(c, graph, cols, d_values, size, rot_scale, shard, (cudaStream_t)stream);
    });
}

int h2b_evaluate_h_permutation_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                   const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                   int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                   const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                   const uint64_t extended_omega[4], void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        return evaluate_h_permutation_run(c, d_values, size, rot_scale, d_product_cosets, n_sets, d_columns, d_perm_cosets, n_columns, chunk_len, last_rotation,
                                          d_l0, d_l_last, d_l_active_row, beta, gamma, y, delta, zeta, extended_omega, nullptr, (cudaStream_t)stream);
    });
}
int h2b_evaluate_h_permutation_shard_dev(int device, void* d_values, uint32_t size, int32_t rot_scale, const void* const* d_product_cosets, uint32_t n_sets,
                                         const void* const* d_columns, const void* const* d_perm_cosets, uint32_t n_columns, uint32_t chunk_len,
                                         int32_t last_rotation, const void* d_l0, const void* d_l_last, const void* d_l_active_row, const uint64_t beta[4],
                                         const uint64_t gamma[4], const uint64_t y[4], const uint64_t delta[4], const uint64_t zeta[4],
                                         const uint64_t extended_omega[4], const h2b_eval_shard* shard, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!shard) { set_error("h2b_evaluate_h_permutation_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
        return evaluate_h_permutation_run(c, d_values, size, rot_scale, d_product_cosets, n_sets, d_columns, d_perm_cosets, n_columns, chunk_len, last_rotation,
                                          d_l0, d_l_last, d_l_active_row, beta, gamma, y, delta, zeta, extended_omega, shard, (cudaStream_t)stream);
    });
}

int h2b_evaluate_h_lookup_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                              const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                              const void* d_l_last, const void* d_l_active_row, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        return evaluate_h_lookup_run(c, graph, cols, d_values, size, rot_scale, d_product_coset, d_permuted_input_coset, d_permuted_table_coset, d_l0, d_l_last,
                                     d_l_active_row, nullptr, (cudaStream_t)stream);
    });
}
int h2b_evaluate_h_lookup_shard_dev(int device, const h2b_graph* graph, const h2b_eval_columns* cols, void* d_values, uint32_t size, int32_t rot_scale,
                                    const void* d_product_coset, const void* d_permuted_input_coset, const void* d_permuted_table_coset, const void* d_l0,
                                    const void* d_l_last, const void* d_l_active_row, const h2b_eval_shard* shard, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!shard) { set_error("h2b_evaluate_h_lookup_shard_dev: null shard"); return H2B_ERR_BAD_ARGUMENT; }
        return evaluate_h_lookup_run(c, graph, cols, d_values, size, rot_scale, d_product_coset, d_permuted_input_coset, d_permuted_table_coset, d_l0, d_l_last,
                                     d_l_active_row, shard, (cudaStream_t)stream);
    });
}

int h2b_evaluate_graph_info(uint32_t* slots, uint32_t* micro_ops) {
    evaluate_graph_last_info(slots, micro_ops);
    return H2B_OK;
}

int h2b_dev_alloc(int device, size_t bytes, void** out) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));      // no device lock: touches no DeviceCtx state
    if (!out) { set_error("h2b_dev_alloc: null out"); return H2B_ERR_BAD_ARGUMENT; }
    return dev_malloc(out, bytes ? bytes : 1, "h2b_dev_alloc");
}
int h2b_dev_free(int device, void* p) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));      // no device lock: touches no DeviceCtx state
    H2B_CUDA(cudaFree(p));
    return H2B_OK;
}
int h2b_memcpy_h2d(int device, void* d_dst, const void* h_src, size_t bytes) {
    // pageable sources go through the pinned staging threads (stage.cu); synchronous like cudaMemcpy
    return on_device(device, [&](DeviceCtx& c) -> int {
        H2B_CUDA(cudaDeviceSynchronize());            // cudaMemcpy semantics: ordered after everything queued on the device
        H2B_TRY(host_upload(c, d_dst, h_src, bytes, c.stream));
        H2B_CUDA(cudaStreamSynchronize(c.stream));
        return H2B_OK;
    });
}
// Upload that does not wait for the device: d_dst must not be in use by anything in flight.  Work queued on `stream` after the
// call sees the data; the host buffer may be reused on return (pageable sources are consumed by the staging threads, pinned
// ones must stay valid until the stream reaches the copy, as with cudaMemcpyAsync).
int h2b_memcpy_h2d_async(int device, void* d_dst, const void* h_src, size_t bytes, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (bytes && (!d_dst || !h_src)) { set_error("h2b_memcpy_h2d_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        return host_upload(c, d_dst, h_src, bytes, (cudaStream_t)stream, false);
    });
}
int h2b_memcpy_d2d_async(int device, void* d_dst, const void* d_src, size_t bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));      // no device lock: touches no DeviceCtx state
    if (bytes && (!d_dst || !d_src)) { set_error("h2b_memcpy_d2d_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_CUDA(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return H2B_OK;
}
int h2b_memset_zero_async(int device, void* d_dst, size_t bytes, void* stream) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));      // no device lock: touches no DeviceCtx state
    if (bytes && !d_dst) { set_error("h2b_memset_zero_async: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
    H2B_CUDA(cudaMemsetAsync(d_dst, 0, bytes, (cudaStream_t)stream));
    return H2B_OK;
}
int h2b_memcpy_d2h(int device, void* h_dst, const void* d_src, size_t bytes) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        H2B_CUDA(cudaDeviceSynchronize());
        return host_download(c, h_dst, d_src, bytes, c.stream);
    });
}
int h2b_dev_sync(int device) {
    DeviceCtx* c = nullptr;
    H2B_TRY(get_ctx(device, &c));      // no device lock: touches no DeviceCtx state
    H2B_CUDA(cudaDeviceSynchronize());
    return H2B_OK;
}

int h2b_gen_points_dev(int device, uint64_t seed, size_t n, void* d_out_affine, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return gen_points_run(c, seed, n, d_out_affine, (cudaStream_t)stream); });
}
int h2b_gen_scalars_dev(int device, uint64_t seed, size_t n, int kind, void* d_out, void* stream) {
    return on_device(device, [&](DeviceCtx& c) { return gen_scalars_run(c, seed, n, kind, d_out, (cudaStream_t)stream); });
}

int h2b_msm_checksum_dev(int device, const void* d_scalars, uint64_t seed, uint64_t first, size_t n, void* d_out, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!d_out || (n && !d_scalars)) { set_error("h2b_msm_checksum_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        return msm_checksum_run(c, d_scalars, seed, first, n, d_out, (cudaStream_t)stream);
    });
}

int h2b_field_op(int field, int op, const uint64_t* a, const uint64_t* b, size_t n, uint64_t* out) {
    if (field < 0 || field > 1 || op < 0 || op > 13) { set_error("h2b_field_op: bad field/op"); return H2B_ERR_BAD_ARGUMENT; }
    return elementwise_host(0, field, op, a, b, n, out, 32);
}
int h2b_ec_op(int op, const uint64_t* p, const uint64_t* q, size_t n, uint64_t* out) {
    if (op < 0 || op > 5) { set_error("h2b_ec_op: bad op"); return H2B_ERR_BAD_ARGUMENT; }
    return elementwise_host(1, 0, op, p, q, n, out, 64);
}

int h2b_imad_bench(int device, int kind, int iters, float* ms_out, double* ops_out) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!ms_out || !ops_out) { set_error("h2b_imad_bench: null output"); return H2B_ERR_BAD_ARGUMENT; }
        return imad_bench_run(c, kind, iters, c.sm_count * 8, 256, ms_out, ops_out, c.stream);
    });
}

int h2b_set_msm_window(int c) { return msm_set_window(c); }

unsigned long long h2b_launch_count(void) { return __atomic_load_n(&g_launch_count, __ATOMIC_RELAXED); }

int h2b_profile_enable(int device, int on) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        Profiler& p = c.prof;
        if (on && p.ev.empty()) {
            p.ev.resize(8192);
            p.tag.resize(8192);
            for (auto& e : p.ev) H2B_CUDA(cudaEventCreate(&e));
        }
        p.enabled = on != 0;
        p.used = 0;
        return H2B_OK;
    });
}

int h2b_profile_read(int device, int* tags, float* ms, int cap, int* count) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (!tags || !ms || !count) { set_error("h2b_profile_read: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        Profiler& p = c.prof;
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
    });
}

}  // extern "C"
