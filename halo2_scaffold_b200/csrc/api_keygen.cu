// C ABI of libh2b200, key generation: the permutation argument's sigma columns, compress_selectors and the fixed columns of
// keygen_vk / keygen_pk, keygen_pk's indicator columns, and the proving key held resident on the devices (h2b_pk_*).
#include "host.h"

namespace h2b {

// the domain arguments of the keygen_pk entry points: the sizes and the constants of the iNTT and the coset NTT
static int domain_check(const char* who, uint32_t k, uint32_t extended_k, const uint64_t* omega_inv, const uint64_t* ifft_divisor,
                        const uint64_t* extended_omega, const uint64_t* zeta_powers) {
    if (extended_k > 28 || extended_k < k) { set_error("%s: need k <= extended_k <= 28 (k = %u, extended_k = %u)", who, k, extended_k); return H2B_ERR_BAD_ARGUMENT; }
    if (!omega_inv || !ifft_divisor || !extended_omega || !zeta_powers) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
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
    *out = G.sets.find(handle_g_lagrange);
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

// ---- the proving key resident on the devices ---------------------------------------------------------------------------------------
static int pk_lookup(const char* who, uint64_t handle, PkRef* out) {
    H2B_TRY(require_init());
    *out = G.pks.find(handle);
    if (*out) return H2B_OK;
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

}  // namespace h2b

using namespace h2b;

extern "C" {

// ---- key generation: the permutation argument's sigma columns and keygen_pk's indicator columns ---------------------------------
// ([UP] halo2_proofs/src/plonk/permutation/keygen.rs Assembly::{build_vk, build_pk}, plonk/keygen.rs keygen_pk)
int h2b_permutation_sigma_dev(int device, const void* const* d_mapping, uint32_t n_columns, uint32_t k, const uint64_t delta[4], const uint64_t omega[4],
                              void* const* d_sigma, void* d_status, void* stream) {
    return on_device(device, [&](DeviceCtx& c) -> int {
        if (k > 28 || n_columns == 0) { set_error("h2b_permutation_sigma_dev: k = %u, %u columns (need k <= 28 and at least one column)", k, n_columns); return H2B_ERR_BAD_ARGUMENT; }
        if (!d_mapping || !delta || !omega || !d_sigma || !d_status) { set_error("h2b_permutation_sigma_dev: null pointer"); return H2B_ERR_BAD_ARGUMENT; }
        for (uint32_t i = 0; i < n_columns; ++i)
            if (!d_mapping[i] || !d_sigma[i]) { set_error("h2b_permutation_sigma_dev: column %u: null pointer", i); return H2B_ERR_BAD_ARGUMENT; }
        const cudaStream_t st = (cudaStream_t)stream;
        H2B_CUDA(cudaMemsetAsync(d_status, 0, 4, st));
        H2B_TRY(permutation_sigma_tables_run(c, n_columns, k, delta, omega, st));
        return permutation_sigma_run(c, d_mapping, n_columns, 0, n_columns, k, d_sigma, d_status, st);
    });
}

int h2b_keygen_lagrange_indicators_dev(int device, uint32_t k, uint32_t extended_k, uint32_t blinding_factors, const uint64_t omega_inv[4],
                                       const uint64_t ifft_divisor[4], const uint64_t extended_omega[4], const uint64_t zeta_powers[12], void* d_l0,
                                       void* d_l_last, void* d_l_active_row, void* stream) {
    static const char* who = "h2b_keygen_lagrange_indicators_dev";
    return on_device(device, [&](DeviceCtx& c) -> int {
        H2B_TRY(domain_check(who, k, extended_k, omega_inv, ifft_divisor, extended_omega, zeta_powers));
        if ((uint64_t)blinding_factors + 1 >= ((uint64_t)1 << k)) { set_error("%s: k = %u, %u blinding factors (need bf + 1 < 2^k)", who, k, blinding_factors); return H2B_ERR_BAD_ARGUMENT; }
        if (!d_l0 || !d_l_last || !d_l_active_row) { set_error("%s: null pointer", who); return H2B_ERR_BAD_ARGUMENT; }
        void* cols[3] = {d_l0, d_l_last, d_l_active_row};
        return keygen_indicators_run(c, k, extended_k, blinding_factors, omega_inv, ifft_divisor, extended_omega, zeta_powers, cols, (cudaStream_t)stream);
    });
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
    *handle = G.pks.publish(pk);
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
    PkRef drop = G.pks.take(handle);      // freed after G.mu is let go (the destructor waits for the devices)
    if (!drop) { set_error("h2b_pk_release: unknown proving-key handle %llu", (unsigned long long)handle); return H2B_ERR_BAD_ARGUMENT; }
    return H2B_OK;
}

}  // extern "C"
