// db.cu -- the resident database: construction from host memory (psb_db_create, and the pieces of psb_scan_host),
// its sort and pack chain on the device, the inverse permutation, psb_db_subject and the psb_db_* accessors.  cub's
// kernels are instantiated here only, so the prefix sum the other files need is exclusive_sum below.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"

namespace psb {

__global__ void db_lengths_kernel(const long long *off, long long n, int *len, int *idx) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        len[i] = (int)(off[i + 1] - off[i]);
        idx[i] = (int)i;
    }
}
__global__ void db_wcount_sorted_kernel(const int *len_sorted, long long n, int rpw, long long *wcount) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += stride)
        wcount[i] = i < n ? (len_sorted[i] + rpw - 1) / rpw : 0;
}

int db_io_ensure_ctx(int *device, cudaStream_t *stream) {
    const int rc = ensure_ctx();
    if (rc != PSB_OK) return rc;
    *device = g_ctx.device; *stream = g_ctx.stream;
    return PSB_OK;
}

// Database construction in two phases so that psb_scan_host can overlap the upload of one piece with
// the scan of the previous one.  Phase A (db_begin): one host pass over the offsets (validation,
// longest lengths, packed size), device allocations, and the host->device copies on `up` (the
// caller's stream or the context's copy stream).  Phase B (db_finish): lengths, stable radix sort
// by decreasing length, word offsets (scan), residue mapping + bit packing, all on the compute
// stream and without any host synchronisation.

// Phase A1: the device-side object and the host->device copies (nothing here looks at the individual offsets,
// so psb_scan_host can queue the upload of piece k+1 before it spends host time on piece k)
psb_db *db_upload(DbBuild &B, const uint8_t *cat, const int64_t *off, int64_t n, const HostMatrix &hm, bool use_copy_stream, int force_bits,
                  cudaEvent_t residues_after) {
    Ctx &c = g_ctx;
    if (hm.size > 32) { set_error("psb_db_create: alphabets above 32 letters cannot be 5-bit packed"); return nullptr; }
    if (off[n] <= off[0]) { set_error("psb_db_create: offsets are not increasing"); return nullptr; }
    psb_db *db = new psb_db();
    db->device = c.device; db->stream = c.stream; db->n = n; db->msize = hm.size;
    std::memcpy(db->mapper, hm.mapper, 256);
    // 2 bit for alphabets of up to 4 letters, 3 bit up to 8 (ACGT + wildcard: DNA ships at 3 bit), else 5
    db->bits = force_bits ? force_bits : db_bits_for(hm.size);
    db->residues = off[n] - off[0];
    const size_t n1 = (size_t)n + 1;
    // with the copy stream, the upload must not queue behind whatever scan is already running on the
    // compute stream: its staging blocks are recycled plain allocations (see StageBlock)
    cudaStream_t up = use_copy_stream ? c.copy : c.stream;
    auto fail = [&](const std::string &what) {
        set_error(what);
        cudaStreamSynchronize(up);
        psb_db_free(db);
        return (psb_db *)nullptr;
    };
    if (use_copy_stream) {
        B.st_device = c.device;
        B.st_raw = stage_acquire(c.device, (size_t)db->residues, &B.st_raw_bytes);
        B.st_off = stage_acquire(c.device, n1 * 8, &B.st_off_bytes);
        if (!B.st_raw || !B.st_off) return fail("psb_scan_host: device allocation of the staging blocks failed");
    } else if (B.d_raw.alloc((size_t)db->residues, up) != PSB_OK || B.d_off.alloc(n1 * 8, up) != PSB_OK) {
        return fail(psb_last_error());
    }
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    // offsets first: lengths, sort and word offsets need nothing else, so that whole chain of small launches runs
    // while the residues (the long copy) are still on the link -- under a saturated link each of those launches
    // costs 30-50 us instead of 5 (measured: 0.6 ms for the chain of the first piece, tools/shard_e2e_probe.py)
    ck(upload_h2d(B.offs(), off, n1 * 8, up));
    if (use_copy_stream) {
        ck(cudaEventCreateWithFlags(&B.offs_up, cudaEventDisableTiming));
        ck(cudaEventRecord(B.offs_up, up));
        // a saturated link makes every small launch on the device wait its turn for the command fetch (30-50 us
        // each, measured), so the residues of this piece stay off the link until the previous piece's sort/pack
        // chain has run; they still have that piece's whole scan to land in
        if (residues_after) ck(cudaStreamWaitEvent(up, residues_after, 0));
        ck(cudaEventCreate(&B.res_begin));
        ck(cudaEventRecord(B.res_begin, up));
    }
    ck(upload_h2d(B.raw(), cat + off[0], (size_t)db->residues, up));
    if (use_copy_stream) {
        ck(cudaEventCreate(&B.uploaded));
        ck(cudaEventRecord(B.uploaded, up));
    }
    if (e != cudaSuccess) return fail(std::string("psb_db_create: ") + cudaGetErrorString(e));
    B.db = db; B.raw_base = off[0]; B.up = up;
    fill_lut(B.lut, hm.mapper);
    return db;
}

// words of `rpw` residues that `l` residues occupy; rpw is one of 16 / 10 / 6 (2, 3, 5 bit): constant
// divisors, because a 64-bit division per subject was most of this pass
template <int RPW> static inline long long words_of(long long l) { return (l + RPW - 1) / RPW; }

// Phase A2: one host pass over the offsets (validation, histogram of lengths for the longest few, exact
// packed size) and the remaining device allocations
int db_host_pass(DbBuild &B, const int64_t *off) {
    Ctx &c = g_ctx;
    psb_db *db = B.db;
    const int64_t n = db->n;
    const int rpw = db_residues_per_word(db->bits);
    auto fail = [&](const std::string &what) {
        set_error(what);
        cudaStreamSynchronize(B.up);
        cudaStreamSynchronize(c.stream);
        psb_db_free(db);
        B.db = nullptr;
        return PSB_EINVAL;
    };
    thread_local std::vector<int> hist;
    hist.assign(65537, 0);
    std::vector<int> huge;   // lengths above 65535
    long long words = 0;
    int64_t maxlen = 0, bad = -1;
    auto pass = [&](auto wof) {
        for (int64_t i = 0; i < n; ++i) {
            const int64_t l = off[i + 1] - off[i];
            if (l <= 0 || l > 0x7fffffff) { bad = i; return; }
            words += wof(l);
            if (l > 65535) huge.push_back((int)l); else hist[(size_t)l]++;
            maxlen = l > maxlen ? l : maxlen;
        }
    };
    if (rpw == 6) pass(words_of<6>); else if (rpw == 10) pass(words_of<10>); else if (rpw == 16) pass(words_of<16>);
    else pass([rpw](long long l) { return (l + rpw - 1) / rpw; });
    if (bad >= 0) return fail("psb_db_create: empty or oversized subject " + std::to_string(bad));
    std::sort(huge.begin(), huge.end(), [](int a, int b2) { return a > b2; });
    db->maxlen = (int)maxlen; db->nlong = (int)huge.size(); db->words = words;
    db->top_len = huge;
    if (db->top_len.size() > 4096) db->top_len.resize(4096);
    for (int l = (int)std::min<int64_t>(maxlen, 65535); l >= 1 && db->top_len.size() < 4096; --l)
        for (int t = 0; t < hist[l] && db->top_len.size() < 4096; ++t) db->top_len.push_back(l);

    const size_t n1 = (size_t)n + 1;
    if (B.d_len0.alloc((size_t)n * 4, c.stream) != PSB_OK || B.d_idx0.alloc((size_t)n * 4, c.stream) != PSB_OK ||
        B.d_wcount.alloc(n1 * 8, c.stream) != PSB_OK)
        return fail(psb_last_error());
    cudaError_t e = cudaSuccess;
    auto ck = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    ck(cudaMallocAsync(&db->d_word_off, n1 * 8, c.stream));
    ck(cudaMallocAsync(&db->d_perm, (size_t)n * 4, c.stream));
    ck(cudaMallocAsync(&db->d_len, (size_t)n * 4, c.stream));
    ck(cudaMallocAsync(&db->d_words, (size_t)db->words * 4 + 64, c.stream));
    if (e != cudaSuccess) return fail(std::string("psb_db_create: ") + cudaGetErrorString(e));
    return PSB_OK;
}

static psb_db *db_begin(DbBuild &B, const uint8_t *cat, const int64_t *off, int64_t n, const HostMatrix &hm, bool use_copy_stream, int force_bits = 0) {
    if (!db_upload(B, cat, off, n, hm, use_copy_stream, force_bits)) return nullptr;
    if (db_host_pass(B, off) != PSB_OK) return nullptr;
    return B.db;
}

// `marks`: psb_scan_host's timeline (lengths< >lengths sort> <pack pack>), or nullptr
int db_finish(DbBuild &B, StreamMarks *marks) {
    Ctx &c = g_ctx;
    psb_db *db = B.db;
    const int64_t n = db->n;
    const size_t n1 = (size_t)n + 1;
    const int rpw = db_residues_per_word(db->bits);
    auto mark = [&] { if (marks) marks->mark(c.stream); };
    if (B.offs_up) PSB_CUDA(cudaStreamWaitEvent(c.stream, B.offs_up, 0));
    mark();
    db_lengths_kernel<<<c.sms * 4, 256, 0, c.stream>>>(B.offs(), n, B.d_len0.as<int>(), B.d_idx0.as<int>());
    mark();
    size_t tb = 0, tb2 = 0;
    PSB_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, B.d_len0.as<int>(), db->d_len, B.d_idx0.as<int>(), db->d_perm, (int)n, 0, 32, c.stream));
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb2, B.d_wcount.as<long long>(), db->d_word_off, (int)n1, c.stream));
    PSB_TRY(B.d_tmp.alloc(std::max(tb, tb2), c.stream));
    PSB_CUDA(cub::DeviceRadixSort::SortPairsDescending(B.d_tmp.p, tb, B.d_len0.as<int>(), db->d_len, B.d_idx0.as<int>(), db->d_perm, (int)n, 0, 32, c.stream));
    mark();
    db_wcount_sorted_kernel<<<c.sms * 4, 256, 0, c.stream>>>(db->d_len, n, rpw, B.d_wcount.as<long long>());
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(B.d_tmp.p, tb2, B.d_wcount.as<long long>(), db->d_word_off, (int)n1, c.stream));
    if (B.uploaded) PSB_CUDA(cudaStreamWaitEvent(c.stream, B.uploaded, 0));
    mark();
    launch_pack_db(B, c.sms * 8, 256, 256, c.stream);
    if (B.uploaded) {
        PSB_CUDA(cudaEventCreateWithFlags(&B.packed, cudaEventDisableTiming));
        PSB_CUDA(cudaEventRecord(B.packed, c.stream));
    }
    mark();
    c.launches += 5;
    PSB_CUDA(cudaGetLastError());
    // no synchronisation: later work on this stream is ordered after the packing kernel, and the
    // staging buffers go back to the pool in stream order when B is destroyed
    return PSB_OK;
}

// a database the caller holds in host memory, checked in each entry point's wording; `arg` is the entry point's other
// required pointer.  The host scans (`scan`) report offsets that do not increase as an empty database, before the
// subject count; psb_db_create names them, after it.
int host_db_check(const char *who, const void *arg, const uint8_t *cat, const int64_t *off, int64_t n, bool scan) {
    const std::string w(who);
    if (!arg || !cat || !off || n <= 0 || (scan && off[n] <= off[0])) { set_error(w + ": NULL argument or empty database"); return PSB_EINVAL; }
    if (n > 0x7ffffffe) { set_error(w + ": more than 2^31-2 subjects"); return PSB_EUNSUPPORTED; }
    if (off[n] <= off[0]) { set_error(w + ": offsets are not increasing"); return PSB_EINVAL; }
    return PSB_OK;
}

// what every call that reads a resident database's subjects by caller id checks: the calling thread's device holds it
int db_check(const char *who, const psb_db *db) {
    PSB_TRY(ensure_ctx());
    if (db->device != g_ctx.device) { set_error(std::string(who) + ": database lives on another device"); return PSB_EINVAL; }
    if (db->host_len.empty()) { set_error(std::string(who) + ": the database has no subject lengths on the host"); return PSB_EUNSUPPORTED; }
    return PSB_OK;
}

// The database's inverse permutation, built on first use: the scatter runs on db->stream, behind the sort/pack chain
// psb_db_create queued there (it returns before that chain has finished), and that stream is synchronised before the
// pointer is published.  So whoever sees the pointer -- any host thread, any stream -- also sees finished packed words.
int db_inv_perm(psb_db *db, int *launched) {
    *launched = 0;
    if (db->d_inv_perm) return PSB_OK;
    std::lock_guard<std::mutex> lk(db->mu);
    if (db->d_inv_perm) return PSB_OK;
    int *inv = nullptr;
    PSB_CUDA(cudaMallocAsync(&inv, (size_t)db->n * sizeof(int), db->stream));
    launch_invert_perm(db->d_perm, db->n, inv, (unsigned)std::min<int64_t>((db->n + 255) / 256, (int64_t)g_ctx.sms * 8), 256, db->stream);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(db->stream);
    if (e != cudaSuccess) {
        cudaFreeAsync(inv, db->stream);
        set_error(std::string("psb_db: inverse permutation: ") + cudaGetErrorString(e));
        return PSB_ECUDA;
    }
    db->d_inv_perm = inv;
    *launched = 1;
    return PSB_OK;
}

int exclusive_sum(int *in, long long *out, int n, DevMem &tmp, cudaStream_t stream) {
    size_t tmp_bytes = 0;
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, in, out, n, stream));
    PSB_TRY(tmp.alloc(tmp_bytes, stream));
    PSB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, in, out, n, stream));
    return PSB_OK;
}

}  // namespace psb

using namespace psb;

extern "C" {

psb_db_t *psb_db_create(const uint8_t *cat, const int64_t *off, int64_t n, const parasail_matrix_t *matrix) {
    if (host_db_check("psb_db_create", matrix, cat, off, n, false) != PSB_OK) return nullptr;
    if (ensure_ctx() != PSB_OK) return nullptr;
    HostMatrix hm(matrix);
    // bits per residue from the residues actually present: a DNA database whose residues are all A/C/G/T
    // (no wildcard, which maps to column 4) packs at 2 bit even though its matrix has 5 columns
    int force_bits = 0;
    if (db_bits_for(hm.size) == 3) {
        bool small = true;
        for (int64_t x = off[0]; x < off[n] && small; ++x) small = hm.mapper[cat[x]] < 4;
        if (small) force_bits = 2;
    }
    DbBuild B;
    psb_db *db = db_begin(B, cat, off, n, hm, false, force_bits);
    if (!db) return nullptr;
    // the caller's buffers must be free to go when this returns: wait for the uploads (not for the packing)
    cudaEvent_t up = nullptr;
    if (cudaEventCreateWithFlags(&up, cudaEventDisableTiming) == cudaSuccess) cudaEventRecord(up, g_ctx.stream);
    db->host_len.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) db->host_len[(size_t)i] = (int)(off[i + 1] - off[i]);
    const int rc = db_finish(B);
    if (up) { cudaEventSynchronize(up); cudaEventDestroy(up); } else cudaStreamSynchronize(g_ctx.stream);
    if (rc != PSB_OK) { cudaStreamSynchronize(g_ctx.stream); psb_db_free(db); return nullptr; }
    return db;
}

int64_t psb_db_count(const psb_db_t *db) { return db ? db->n : 0; }
int psb_db_bits(const psb_db_t *db) { return db ? db->bits : 0; }
int64_t psb_db_residues(const psb_db_t *db) { return db ? db->residues : 0; }
int64_t psb_db_device_bytes(const psb_db_t *db) {
    return db ? db->words * 4 + (db->n + 1) * 8 + db->n * 8 : 0;
}

void psb_db_free(psb_db_t *db) {
    if (!db) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(db->device);
    void *ptrs[] = {db->d_words, db->d_word_off, db->d_perm, db->d_len, db->d_res_off, db->d_inv_perm};
    for (void *p : ptrs) if (p) cudaFreeAsync(p, db->stream);
    cudaSetDevice(cur);
    delete db;
}

int64_t psb_db_subject(const psb_db_t *db_c, int64_t id, uint8_t *codes, int64_t cap) {
    if (!db_c || cap < 0 || (cap > 0 && !codes)) { set_error("psb_db_subject: NULL argument or negative capacity"); return PSB_EINVAL; }
    psb_db *db = const_cast<psb_db *>(db_c);
    PSB_TRY(db_check("psb_db_subject", db));
    if (id < 0 || id >= db->n) { set_error("psb_db_subject: id " + std::to_string(id) + " is not a subject of a database of " + std::to_string(db->n)); return PSB_EINVAL; }
    int first_use = 0;
    PSB_TRY(db_inv_perm(db, &first_use));
    const int64_t len = db->host_len[(size_t)id];
    if (cap == 0) return len;
    Ctx &c = g_ctx;
    const int sid = (int)id;
    const long long off[2] = {0, (long long)len};
    DevMem d_id, d_off, d_out;
    PSB_TRY(d_id.alloc(sizeof(int), c.stream));
    PSB_TRY(d_off.alloc(sizeof(off), c.stream));
    PSB_TRY(d_out.alloc((size_t)len, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d_id.p, &sid, sizeof(int), cudaMemcpyHostToDevice, c.stream));
    PSB_CUDA(cudaMemcpyAsync(d_off.p, off, sizeof(off), cudaMemcpyHostToDevice, c.stream));
    launch_unpack_db(db, d_id.as<int>(), db->d_inv_perm, d_off.as<long long>(), d_out.as<uint8_t>(), 1, 1, 32, c.stream);
    PSB_CUDA(cudaGetLastError());
    PSB_CUDA(cudaMemcpyAsync(codes, d_out.p, (size_t)std::min(len, cap), cudaMemcpyDeviceToHost, c.stream));
    PSB_CUDA(cudaStreamSynchronize(c.stream));   // (`sid` / `off` are host temporaries)
    return len;
}
}  // extern "C"
