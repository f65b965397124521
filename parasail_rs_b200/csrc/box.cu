// box.cu -- a resident database sharded over the devices of the box, driven from one process (psb_box_db_*,
// psb_box_scan / psb_box_align / psb_box_search).  The subjects are cut into contiguous caller-id ranges of equal
// residue count (psb_scan_box's cut); shard s is an ordinary psb_db built, scanned and aligned by the resident worker
// of its device.  Every entry point is the single-device one applied per shard, plus a host step that puts the
// shards' rows into caller order: the scan writes each shard's results at its first id, the search merges each
// query's per-shard best rows by the rule of psb_batch_topk.  No kernel of its own and no copy between devices.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"

struct psb_box_db {
    std::vector<psb_db *> shard;
    std::vector<int64_t> first;   // shards + 1 entries: shard s holds caller ids first[s] .. first[s + 1] - 1
    std::vector<int> device;      // shard s lives on device[s]
    int64_t n = 0, residues = 0;
    std::vector<int> len;         // caller-order subject lengths (explicit-width saturation flags)
    int shard_of(int64_t id) const { return (int)(std::upper_bound(first.begin(), first.end(), id) - first.begin()) - 1; }
};

namespace psb {

static const char *kNoDevice = "no CUDA device available: libparasail_b200 has no CPU fallback (needs an sm_100a GPU)";

// The jobs of one call: one per device, each working through that device's shards one after another on the device's
// worker.  The call waits for its own jobs only (a count of its own), so that two host threads can call on one box
// database at once.
struct BoxCall {
    struct Job { int rc = PSB_OK, launches = 0; int shard = -1; double ms = 0.0; std::string err; };
    const psb_box_db *db;
    std::vector<int> devices;     // distinct devices, in order of their first shard
    std::vector<Job> jobs;        // one per entry of `devices`
    std::mutex mu;
    std::condition_variable cv;
    int pending = 0;
    explicit BoxCall(const psb_box_db *d) : db(d) {
        for (int dev : d->device)
            if (std::find(devices.begin(), devices.end(), dev) == devices.end()) devices.push_back(dev);
        jobs.resize(devices.size());
    }
    // runs work(s) for every shard s of every device, on that device's worker with its context bound; a job stops at
    // its first failure.  Each job adds its shards' device time and launches to its own; returns when every job has
    // finished.
    void run(const std::function<int(int)> &work) {
        pending = (int)devices.size();
        for (size_t j = 0; j < devices.size(); ++j) {
            box_worker(devices[j])->submit([this, j, &work] {
                Job &r = jobs[j];
                r.rc = ensure_ctx();
                for (size_t s = 0; s < db->shard.size() && r.rc == PSB_OK; ++s) {
                    if (db->device[s] != devices[j]) continue;
                    g_ctx.last_ms = 0.0; g_ctx.launches = 0;
                    r.shard = (int)s;
                    r.rc = work((int)s);
                    r.ms += g_ctx.last_ms; r.launches += g_ctx.launches;   // one device's shards run one after another
                }
                if (r.rc != PSB_OK) r.err = psb_last_error();
                std::lock_guard<std::mutex> lk(mu);
                --pending;
                cv.notify_all();
            });
        }
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return pending == 0; });
    }
    bool failed() const {
        for (const Job &r : jobs) if (r.rc != PSB_OK) return true;
        return false;
    }
    // the first failure as "who (shard s, device d): ...", and the calling thread's counters: the slowest device's
    // kernel time, the launches of all devices
    int finish(const char *who) {
        int rc = PSB_OK;
        for (const Job &r : jobs)
            if (r.rc != PSB_OK && rc == PSB_OK) {
                rc = r.rc;
                set_error(std::string(who) + " (shard " + std::to_string(r.shard) + ", device " + std::to_string(r.shard >= 0 ? db->device[(size_t)r.shard] : -1) +
                          "): " + r.err);
            }
        Ctx &c = g_ctx;
        c.last_ms = 0.0; c.launches = 0;
        for (const Job &r : jobs) { c.last_ms = std::max(c.last_ms, r.ms); c.launches += r.launches; }
        return rc;
    }
};

static int box_db_check(const char *who, const psb_box_db *db, const parasail_profile_t *profile) {
    if (psb_device_count() <= 0) { set_error(kNoDevice); return PSB_ENODEV; }
    return profile_alphabet_check(who, profile, db->shard[0]);
}

// the alignments of n rows (query row_q[i] against caller id row_id[i]): each shard aligns the rows it holds with
// align_rows, and the rows are gathered in row order.  Adds to `call`'s per-device counters.
static int box_align_rows(const char *who, const FnConfig &cfg, const parasail_profile_t *const *profiles, int64_t nq, const int64_t *row_q,
                          const int64_t *row_id, int64_t n, int open, int gap, BoxCall &call, psb_batch_t **out) {
    const psb_box_db *db = call.db;
    const size_t S = db->shard.size();
    std::vector<std::vector<int64_t>> q(S), id(S);
    std::vector<std::pair<int, int64_t>> src((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        const int s = db->shard_of(row_id[i]);
        src[(size_t)i] = {s, (int64_t)q[(size_t)s].size()};
        q[(size_t)s].push_back(row_q[i]);
        id[(size_t)s].push_back(row_id[i] - db->first[(size_t)s]);
    }
    std::vector<psb_batch_t *> gb(S, nullptr);
    call.run([&](int s) {
        if (q[(size_t)s].empty()) return PSB_OK;
        return align_rows(cfg, profiles, nq, q[(size_t)s].data(), id[(size_t)s].data(), (int64_t)q[(size_t)s].size(), open, gap, db->shard[(size_t)s],
                          &gb[(size_t)s]);
    });
    int rc = call.finish(who);
    // the shards that hold rows, in shard order
    std::vector<psb_batch_t *> held;
    std::vector<int> slot(S, -1);
    for (size_t s = 0; s < S; ++s)
        if (gb[s]) { slot[s] = (int)held.size(); held.push_back(gb[s]); }
    if (rc == PSB_OK && held.size() == 1) { *out = held[0]; return PSB_OK; }   // every row on one shard, in row order
    for (auto &r : src) r.first = slot[(size_t)r.first];
    if (rc == PSB_OK) rc = gather_rows(cfg, held, src, out);
    for (psb_batch_t *b : held) free_batch(b);
    return rc;
}

}  // namespace psb

using namespace psb;

extern "C" {

psb_box_db_t *psb_box_db_create(const uint8_t *cat, const int64_t *off, int64_t n, const parasail_matrix_t *matrix, const int *devices,
                                int n_shards) {
    if (host_db_check("psb_box_db_create", matrix, cat, off, n, false) != PSB_OK) return nullptr;
    const int ndev = psb_device_count();
    if (ndev <= 0) { set_error(kNoDevice); return nullptr; }
    std::vector<int> want;
    if (!devices) {
        for (int d = 0; d < ndev; ++d) want.push_back(d);
    } else {
        if (n_shards <= 0) { set_error("psb_box_db_create: " + std::to_string(n_shards) + " shards"); return nullptr; }
        for (int s = 0; s < n_shards; ++s) {
            if (devices[s] < 0 || devices[s] >= ndev) {
                set_error("psb_box_db_create: devices[" + std::to_string(s) + "] = " + std::to_string(devices[s]) + " is not a device (" +
                          std::to_string(ndev) + " visible)");
                return nullptr;
            }
            want.push_back(devices[s]);
        }
    }
    const int64_t total = off[n] - off[0];
    std::vector<int64_t> targets;
    for (size_t s = 1; s < want.size(); ++s) targets.push_back(total * (int64_t)s / (int64_t)want.size());
    const std::vector<int64_t> cut = cut_subjects(off, n, targets);
    psb_box_db *db = new psb_box_db();
    const size_t S = cut.size() - 1;
    db->shard.assign(S, nullptr);
    db->first = cut;
    db->device.assign(want.begin(), want.begin() + (long)S);
    db->n = n; db->residues = total;
    db->len.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) db->len[(size_t)i] = (int)(off[i + 1] - off[i]);
    BoxCall call(db);
    call.run([&](int s) {
        db->shard[(size_t)s] = psb_db_create(cat, off + cut[(size_t)s], cut[(size_t)s + 1] - cut[(size_t)s], matrix);
        return db->shard[(size_t)s] ? PSB_OK : PSB_ECUDA;
    });
    if (call.finish("psb_box_db_create") != PSB_OK) { psb_box_db_free(db); return nullptr; }
    return db;
}

int64_t psb_box_db_count(const psb_box_db_t *db) { return db ? db->n : 0; }

int psb_box_db_shards(const psb_box_db_t *db, int64_t *first, int *device) {
    if (!db) { set_error("psb_box_db_shards: NULL argument"); return PSB_EINVAL; }
    const int S = (int)db->shard.size();
    for (int s = 0; first && s <= S; ++s) first[s] = db->first[(size_t)s];
    for (int s = 0; device && s < S; ++s) device[s] = db->device[(size_t)s];
    return S;
}

void psb_box_db_free(psb_box_db_t *db) {
    if (!db) return;
    for (psb_db *s : db->shard) psb_db_free(s);
    delete db;
}

int64_t psb_box_db_subject(const psb_box_db_t *db, int64_t id, uint8_t *codes, int64_t cap) {
    if (!db || cap < 0 || (cap > 0 && !codes)) { set_error("psb_box_db_subject: NULL argument or negative capacity"); return PSB_EINVAL; }
    if (id < 0 || id >= db->n) { set_error("psb_box_db_subject: id " + std::to_string(id) + " is not a subject of a database of " + std::to_string(db->n)); return PSB_EINVAL; }
    if (psb_device_count() <= 0) { set_error(kNoDevice); return PSB_ENODEV; }
    if (cap == 0) return db->len[(size_t)id];
    const int s = db->shard_of(id);
    const int64_t local = id - db->first[(size_t)s];
    int64_t len = 0;
    BoxCall call(db);
    call.run([&](int t) {
        if (t != s) return PSB_OK;
        len = psb_db_subject(db->shard[(size_t)s], local, codes, cap);
        return len < 0 ? (int)len : PSB_OK;
    });
    PSB_TRY(call.finish("psb_box_db_subject"));
    return len;
}

int psb_box_scan(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_box_db_t *db, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_box_scan", fn_name, profile, &cfg));
    if (!db || !out) { set_error("psb_box_scan: NULL argument"); return PSB_EINVAL; }
    PSB_TRY(box_db_check("psb_box_scan", db, profile));
    PSB_TRY(ensure_ctx());   // the batch's pinned arrays are allocated by the calling thread
    psb_batch_t *b = new_batch(db->n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    const std::array<int *, 6> hosts = batch_outputs(b);
    std::vector<int64_t> retried(db->shard.size(), 0);
    // each shard's results go straight to its caller-order range of the batch
    BoxCall call(db);
    call.run([&](int s) {
        ScanJob job;
        int rc = scan_enqueue(job, cfg, profile, open, gap, db->shard[(size_t)s], hosts.data(), db->first[(size_t)s]);
        if (rc == PSB_OK) rc = scan_finish(job);
        if (rc != PSB_OK) cudaStreamSynchronize(g_ctx.stream);
        retried[(size_t)s] = job.retried;
        return rc;
    });
    const int rc = call.finish("psb_box_scan");
    if (rc != PSB_OK) { free_batch(b); return rc; }
    for (int64_t r : retried) b->n_retried += r;
    return scan_batch_done(cfg, profile, open, gap, db->residues, [&](int64_t i) { return db->len[(size_t)i]; }, b, out);
}

int psb_box_align(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_box_db_t *db, const int64_t *ids, int64_t n,
                  psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(profile_fn_check("psb_box_align", fn_name, profile, &cfg));
    if (cfg.table || cfg.rowcol) { set_error("psb_box_align: _table/_rowcol outputs exist only on the single-pair API"); return PSB_EUNSUPPORTED; }
    if (!db || !out) { set_error("psb_box_align: NULL argument"); return PSB_EINVAL; }
    PSB_TRY(box_db_check("psb_box_align", db, profile));
    if (n <= 0 || (!ids && n != db->n)) {
        set_error("psb_box_align: " + std::to_string(n) + " ids for a database of " + std::to_string(db->n) + " subjects");
        return PSB_EINVAL;
    }
    std::vector<int64_t> row_id((size_t)n), row_q((size_t)n, 0);
    for (int64_t i = 0; i < n; ++i) {
        const int64_t id = ids ? ids[i] : i;
        if (id < 0 || id >= db->n) {
            set_error("psb_box_align: ids[" + std::to_string(i) + "] = " + std::to_string(id) + " is not a subject of a database of " + std::to_string(db->n));
            return PSB_EINVAL;
        }
        row_id[(size_t)i] = id;
    }
    PSB_TRY(ensure_ctx());
    BoxCall call(db);
    return box_align_rows("psb_box_align", cfg, &profile, 1, row_q.data(), row_id.data(), n, open, gap, call, out);
}

int psb_box_search(const char *fn_name, const parasail_profile_t *const *profiles, int64_t nq, int open, int gap, const psb_box_db_t *db, int k,
                   int64_t *ids_out, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    if (!parse_fn_name(fn_name, &cfg) || !cfg.profile) {
        set_error(std::string("psb_box_search: not a profile function name: ") + (fn_name ? fn_name : "(null)"));
        return PSB_EINVAL;
    }
    if (cfg.table || cfg.rowcol) { set_error("psb_box_search: _table/_rowcol outputs exist only on the single-pair API"); return PSB_EUNSUPPORTED; }
    if (!profiles || !db || !ids_out || !out) { set_error("psb_box_search: NULL argument"); return PSB_EINVAL; }
    if (nq <= 0 || k <= 0) { set_error("psb_box_search: " + std::to_string(nq) + " queries, k = " + std::to_string(k)); return PSB_EINVAL; }
    const int64_t kk = std::min<int64_t>(k, db->n);
    if (nq > INT_MAX / kk) {
        set_error("psb_box_search: " + std::to_string(nq) + " queries x " + std::to_string(kk) + " hits is more than 2^31-1 rows");
        return PSB_EUNSUPPORTED;
    }
    for (int64_t q = 0; q < nq; ++q) {
        const std::string who = "psb_box_search: profiles[" + std::to_string(q) + "]";
        if (!profiles[q]) { set_error(who + " is NULL"); return PSB_EINVAL; }
        PSB_TRY(box_db_check(who.c_str(), db, profiles[q]));
    }
    PSB_TRY(ensure_ctx());
    const size_t S = db->shard.size();
    // (a) on every shard: each query's min(k, n_s) best subjects, shard-local ids
    std::vector<SearchHits> hits(S);
    std::vector<int64_t> kks(S);
    BoxCall call(db);
    call.run([&](int s) {
        kks[(size_t)s] = std::min<int64_t>(k, db->shard[(size_t)s]->n);
        return search_select(cfg, profiles, nq, open, gap, db->shard[(size_t)s], kks[(size_t)s], &hits[(size_t)s]);
    });
    if (call.failed() || (!cfg.trace && !cfg.stats)) PSB_TRY(call.finish("psb_box_search"));
    // the merge: every global top-kk subject is among its own shard's best rows, so per query the kk best of all
    // shards' rows (global ids) by the same rule are the answer
    const int64_t R = nq * kk;
    std::vector<std::pair<int, int64_t>> pick((size_t)R);   // row -> (shard, row in its hits)
    std::vector<std::pair<int, int64_t>> cand;
    for (int64_t q = 0; q < nq; ++q) {
        cand.clear();
        for (size_t s = 0; s < S; ++s)
            for (int64_t r = 0; r < kks[s]; ++r) cand.push_back({(int)s, q * kks[s] + r});
        auto score = [&](const std::pair<int, int64_t> &c) { return hits[(size_t)c.first].score[(size_t)c.second]; };
        auto gid = [&](const std::pair<int, int64_t> &c) { return db->first[(size_t)c.first] + hits[(size_t)c.first].id[(size_t)c.second]; };
        std::partial_sort(cand.begin(), cand.begin() + kk, cand.end(), [&](const std::pair<int, int64_t> &a, const std::pair<int, int64_t> &b) {
            return score(a) != score(b) ? score(a) > score(b) : gid(a) < gid(b);
        });
        for (int64_t r = 0; r < kk; ++r) {
            pick[(size_t)(q * kk + r)] = cand[(size_t)r];
            ids_out[q * kk + r] = gid(cand[(size_t)r]);
        }
    }
    double scan_cells = 0;
    for (int64_t q = 0; q < nq; ++q) scan_cells += (double)profiles[q]->query.size() * (double)db->residues;
    int64_t retried = 0;
    for (const SearchHits &h : hits) retried += h.retried;
    psb_batch_t *b = nullptr;
    if (cfg.trace || cfg.stats) {
        // (b) each kept hit aligned on the device that holds it
        std::vector<int64_t> row_q((size_t)R);
        for (int64_t i = 0; i < R; ++i) row_q[(size_t)i] = i / kk;
        PSB_TRY(box_align_rows("psb_box_search", cfg, profiles, nq, row_q.data(), ids_out, R, open, gap, call, &b));
    } else {
        b = new_batch(R, cfg);
        if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
        for (int64_t i = 0; i < R; ++i) {
            const SearchHits &h = hits[(size_t)pick[(size_t)i].first];
            const size_t j = (size_t)pick[(size_t)i].second;
            b->score[i] = h.score[j]; b->end_query[i] = h.end_query[j]; b->end_ref[i] = h.end_ref[j]; b->saturated[i] = (uint8_t)h.saturated[j];
        }
    }
    b->cells += scan_cells;
    b->n_retried = retried;
    *out = b;
    return PSB_OK;
}

}  // extern "C"
