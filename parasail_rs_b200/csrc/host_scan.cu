// host_scan.cu -- the scan of a database held in host memory: psb_scan_host on the calling thread's device, and
// psb_scan_box over every device of the box, one resident worker thread per device.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

#include "engine.h"

namespace psb {

// The scan of a database that lives in HOST memory, on the calling thread's device: the residues are cut
// into pieces whose upload (copy stream), device-side sort + packing and scan are pipelined, and the
// per-subject results land in hosts[k][base ...] (pinned).  Used by psb_scan_host (one device, base 0) and by
// the per-device workers of psb_scan_box (each with its own range of the caller's arrays).
static uint64_t host_scan_key(const FnConfig &cfg, int lq, int open, int gap, int msize) {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : {(uint64_t)encode_fn(cfg), (uint64_t)lq, (uint64_t)open, (uint64_t)gap, (uint64_t)msize}) { h ^= x + 1; h *= 1099511628211ull; }
    return h | 1;
}
// piece sizes (bytes) for a host scan of `total` residues: geometric with ratio r = 0.85 v/u (every piece lands
// before its predecessor has been scanned), first piece and count chosen to minimise the exposed time
//   (first piece's upload) + (pieces - 1) x boundary,   boundary = sort/pack chain + the scan kernel's ramp and tail
// e.g. C2 on one GPU (362 MB, 52 GB/s, 27 ms of scan): 22 + 76 + 264 MB; a 1/8 shard (45 MB): 10 + 35 MB.
std::vector<int64_t> plan_pieces(int64_t total, double u, double v) {
    const double boundary_ms = 0.35;
    const int64_t cap = (int64_t)1 << 30;   // bounds the device memory of a piece
    // no piece below ~1 ms of scan: the sweep of a piece's longest subjects is serial, so smaller pieces take that
    // long anyway (measured: 8 MB and 11 MB pieces of C2 both scan in 1.2 ms)
    const int64_t min_piece = std::max<int64_t>((int64_t)4 << 20, (int64_t)(1.0 / v));
    // ratio in steps of 1/4 and sizes in steps of 2 MB: the measured rates move a little from call to call, the
    // plan (and with it every allocation size of the pipeline) should not
    const double r = std::min(16.0, std::max(1.25, std::floor(0.85 * v / u * 4.0) / 4.0));
    const double quantum = (double)((int64_t)2 << 20);
    auto cut_up = [&](double s0) {
        std::vector<int64_t> sizes;
        double s = std::max(quantum, std::floor(s0 / quantum) * quantum);
        for (int64_t left = total; left > 0; s *= r) {
            int64_t sz = std::min<int64_t>((int64_t)(std::floor(std::min(s, (double)cap) / quantum) * quantum), left);
            if (left - sz < min_piece) sz = left;
            sizes.push_back(sz);
            left -= sz;
        }
        return sizes;
    };
    std::vector<int64_t> sizes(1, total);
    double best_cost = (double)total * u;
    for (int m = 2; m <= 8; ++m) {
        double s0 = (double)total * (r - 1.0) / (std::pow(r, m) - 1.0);
        const bool floor_hit = s0 < (double)min_piece;
        if (floor_hit) s0 = (double)min_piece;
        if (s0 + (double)min_piece > (double)total) break;
        std::vector<int64_t> cand = cut_up(s0);
        const double cost = (double)cand[0] * u + (double)(cand.size() - 1) * boundary_ms;
        if (cost < best_cost) { best_cost = cost; sizes.swap(cand); }
        if (floor_hit) break;
    }
    return sizes;
}

// subject cuts of the database off[0 .. n] at residue targets (counted from off[0], increasing): 0, then for each target
// the first subject boundary at or past it but at least one subject past the previous cut, then n.  A cut that would
// leave no subject after it ends the list.
static std::vector<int64_t> cut_subjects(const int64_t *off, int64_t n, const std::vector<int64_t> &targets) {
    std::vector<int64_t> cut(1, 0);
    for (const int64_t t : targets) {
        const int64_t at = std::max<int64_t>(std::lower_bound(off, off + n + 1, off[0] + t) - off, cut.back() + 1);
        if (at >= n) break;
        cut.push_back(at);
    }
    cut.push_back(n);
    return cut;
}

// The pieces of a host scan: the upload of piece k+1 (copy stream) runs under the scan of piece k, and nothing on the
// host waits for the GPU until the last piece is queued.  The sizes follow from two measured rates (HostScanState): with
// u = upload time and v = scan time per residue, piece k+1 may be r = 0.85 v/u times piece k and still land before
// piece k has been scanned; the first piece and the number of pieces minimise
// (upload of the first piece) + (pieces - 1) x (cost of a piece boundary).  plan_pieces() above.

struct PiecePlan {
    uint64_t rate_key = 0;              // host_scan_key of the scan
    double u_rate = 0, v_rate = 0;      // upload and scan ms per residue the sizes were planned with
    std::vector<int64_t> cut;           // piece k is subjects cut[k] .. cut[k + 1] - 1
};
// what this thread's host scans are planned from: the measured rates of its device and the previous plan
struct HostScanState {
    double h2d_ms_per_byte = 0;     // residue uploads of >= 4 MB
    uint64_t key = 0;               // the scan (function, query length, penalties) scan_ms_per_byte belongs to
    double scan_ms_per_byte = 0;    // kernel time per database residue of that scan
    int64_t last_total = 0;         // the previous plan: residues, scan and piece sizes
    uint64_t last_key = 0;
    std::vector<int64_t> last_sizes;
    // the rates are exponential averages: a new figure counts half
    static double average(double old, double now) { return old > 0 ? 0.5 * old + 0.5 * now : now; }
    // a finished piece's residue upload (both events have completed by now), counted once
    void note_upload(DbBuild &B) {
        if (!B.res_begin || !B.uploaded || !B.db || B.db->residues < ((int64_t)4 << 20)) return;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, B.res_begin, B.uploaded) != cudaSuccess || ms <= 0.f) { cudaGetLastError(); return; }
        h2d_ms_per_byte = average(h2d_ms_per_byte, (double)ms / (double)B.db->residues);
        cudaEventDestroy(B.res_begin); B.res_begin = nullptr;
    }
    // a host scan of `total` residues whose kernels took `ms`
    void note_scan(uint64_t scan_key, double ms, int64_t total) {
        scan_ms_per_byte = average(key == scan_key ? scan_ms_per_byte : 0, ms / (double)total);
        key = scan_key;
    }
    // the pieces of a call, from the measured rates (defaults for what has not been measured yet)
    PiecePlan plan(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, const int64_t *off, int64_t n) {
        PiecePlan pl;
        const int64_t total = off[n] - off[0];
        pl.rate_key = host_scan_key(cfg, (int)profile->query.size(), open, gap, profile->matrix.size);
        const double u_rate = pl.u_rate = h2d_ms_per_byte > 0 ? h2d_ms_per_byte : 1e3 / 50e9;
        const double v_rate = pl.v_rate = (key == pl.rate_key && scan_ms_per_byte > 0)
                                              ? scan_ms_per_byte
                                              : (double)profile->query.size() * 1e3 / (sw16_wanted(cfg) ? 4.9e12 : 1.5e12);
        std::vector<int64_t> sizes = plan_pieces(total, u_rate, v_rate);
        // hysteresis: the rates are measured and move a little from call to call; a plan that is still within 5 % of
        // the best one is kept, so that a service repeating a scan keeps its allocation sizes (a new size can mean a
        // host-blocking growth of the memory pool)
        auto exposed = [&](const std::vector<int64_t> &sz) {
            double t = (double)sz[0] * u_rate + 0.35 * (double)(sz.size() - 1);
            for (size_t k = 0; k + 1 < sz.size(); ++k) t += std::max(0.0, (double)sz[k + 1] * u_rate - (double)sz[k] * v_rate);
            return t;
        };
        if (last_total == total && last_key == pl.rate_key && !last_sizes.empty() && exposed(last_sizes) <= 1.05 * exposed(sizes) + 0.05) sizes = last_sizes;
        last_total = total; last_key = pl.rate_key; last_sizes = sizes;
        std::vector<int64_t> ends(sizes.size() - 1);   // residues up to the end of every piece but the last
        std::partial_sum(sizes.begin(), sizes.end() - 1, ends.begin());
        pl.cut = cut_subjects(off, n, ends);
        return pl;
    }
};
static thread_local HostScanState g_hs;

// PSB_DEBUG_TIMING on psb_scan_host / psb_scan_box (`on` is false without it): the host's milliseconds since construction
struct HostClock {
    const bool on = debug_timing();
    const std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double ms() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

// piece k's host pass over its offsets and its sort/pack chain.  PSB_DEBUG_TIMING also makes the chain's first mark
// wait for the piece's offsets, so that the timeline shows when they landed.
static int build_piece(HostPiece &p, const int64_t *off, int k, StreamMarks &tl, const HostClock &clk) {
    Ctx &c = g_ctx;
    const double h0 = clk.on ? clk.ms() : 0.0;
    int rc = db_host_pass(p.build, off);
    const double h1 = clk.on ? clk.ms() : 0.0;
    if (clk.on) { cudaStreamWaitEvent(c.stream, p.build.offs_up, 0); tl.mark(c.stream); }
    if (rc == PSB_OK) rc = db_finish(p.build, &tl);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): piece %d host: offsets pass + allocations %.3f ms, chain launches %.3f ms\n", c.device, k, h1 - h0, clk.ms() - h1);
    tl.mark(c.stream);
    return rc;
}

// waits until the piece's results are on the host; its re-runs and its upload time are counted once
static int finish_piece(HostPiece &p, int64_t *n_retried) {
    int rc = PSB_OK;
    if (p.job.ev0 && !p.job.finished) { rc = scan_finish(p.job); *n_retried += p.job.retried; }
    g_hs.note_upload(p.build);
    return rc;
}

// `keep_last`: takes over the last piece once its results are on the host, for a caller with a better moment to give
// its device memory back (psb_scan_box's workers, after they have reported completion)
static int scan_host_into(const FnConfig &cfg, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                          const int64_t *off, int64_t n, int *const hosts[6], int64_t base, int64_t *n_retried,
                          std::unique_ptr<HostPiece> *keep_last = nullptr) {
    Ctx &c = g_ctx;
    const HostClock clk{};
    const PiecePlan pl = g_hs.plan(cfg, profile, open, gap, off, n);
    const std::vector<int64_t> &cut = pl.cut;
    const int npieces = (int)cut.size() - 1;
    const double ms_at_entry = c.last_ms;
    const bool pageable = is_pageable(cat + off[0]);
    if (clk.on) {
        std::string line;
        for (int k = 0; k < npieces; ++k) line += " " + std::to_string((off[cut[k + 1]] - off[cut[k]]) >> 20);
        std::fprintf(stderr, "[psb] scan_host(dev %d): pieces (MB):%s; upload %.1f GB/s, scan %.1f GB/s of residues\n", c.device, line.c_str(),
                     1e-6 / pl.u_rate, 1e-6 / pl.v_rate);
    }
    // a finished piece gives its device memory back, so at most kDepth pieces are resident however large the host
    // database is
    const int kDepth = 4;
    std::vector<std::unique_ptr<HostPiece>> pieces(npieces);
    int rc = PSB_OK;
    auto finish = [&](int k) {
        if (!pieces[k]) return;
        const int r = finish_piece(*pieces[k], n_retried);
        if (rc == PSB_OK) rc = r;
        pieces[k].reset();
    };
    // PSB_DEBUG_TIMING: a device-side timeline (upload landed / packing begins / scan begins / scan ends / results
    // on the host), relative to an event recorded on the idle compute stream at entry
    StreamMarks tl;
    // piece k goes up after piece k - kDepth is finished; its residues wait for piece k-1's chain
    auto upload = [&](int k) {
        if (k >= npieces || rc != PSB_OK) return;
        if (k >= kDepth) finish(k - kDepth);
        if (rc != PSB_OK) return;
        pieces[k].reset(new HostPiece());
        cudaEvent_t gate = k > 0 ? pieces[k - 1]->build.packed : nullptr;
        if (!db_upload(pieces[k]->build, cat, off + cut[k], cut[k + 1] - cut[k], profile->matrix, true, 0, gate)) rc = PSB_ECUDA;
        else tl.mark(c.copy);
    };
    auto scan = [&](int k) {
        if (rc == PSB_OK) rc = scan_enqueue(pieces[k]->job, cfg, profile, open, gap, pieces[k]->build.db, hosts, base + cut[k]);
        tl.mark(c.stream);
    };
    tl.mark(c.stream);
    upload(0);
    if (rc == PSB_OK) rc = prepare_query(cfg, profile, open, gap);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): %d pieces, first upload queued at %.3f ms\n", c.device, npieces, clk.ms());
    for (int k = 0; k < npieces && rc == PSB_OK; ++k) {
        rc = build_piece(*pieces[k], off + cut[k], k, tl, clk);
        // the next upload goes in as soon as its gate (this piece's chain) exists -- unless the caller's memory is
        // pageable: then the upload is a memcpy loop on this thread (upload_h2d) and this piece's scan has to be on the
        // device first
        if (pageable) { scan(k); upload(k + 1); } else { upload(k + 1); scan(k); }
        if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): piece %d queued at %.3f ms\n", c.device, k, clk.ms());
    }
    // everything is queued: the host finishes the earlier pieces while the last ones are still being scanned
    for (int k = 0; k + 1 < npieces; ++k) finish(k);
    cudaStreamSynchronize(c.copy);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): uploads done at %.3f ms\n", c.device, clk.ms());
    if (rc == PSB_OK) rc = finish_piece(*pieces[npieces - 1], n_retried);
    cudaStreamSynchronize(c.stream);
    if (clk.on) std::fprintf(stderr, "[psb] scan_host(dev %d): all done at %.3f ms\n", c.device, clk.ms());
    // order of the marks: entry | upload 0 | per piece k: [upload k+1] upload-k-landed (lengths< >lengths sort> <pack pack>) pack-end results-on-host
    if (clk.on && !tl.ev.empty()) std::fprintf(stderr, "[psb] scan_host(dev %d): device timeline (ms after entry):%s\n", c.device, tl.line().c_str());
    const int64_t total = off[n] - off[0];
    if (rc == PSB_OK && total >= ((int64_t)8 << 20) && c.last_ms > ms_at_entry) g_hs.note_scan(pl.rate_key, c.last_ms - ms_at_entry, total);
    if (keep_last && rc == PSB_OK) *keep_last = std::move(pieces[npieces - 1]);
    for (int k = 0; k < npieces; ++k) finish(k);
    return rc;
}

// the workers of psb_scan_box
static std::mutex g_box_mu;
static std::vector<BoxWorker *> g_box;   // index = device; never destroyed (the threads live as long as the process)
static BoxWorker *box_worker(int device) {
    std::lock_guard<std::mutex> lk(g_box_mu);
    if ((int)g_box.size() <= device) g_box.resize(device + 1, nullptr);
    if (!g_box[device]) g_box[device] = start_worker(device);
    return g_box[device];
}

}  // namespace psb

using namespace psb;

extern "C" {

int psb_scan_host(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                  const int64_t *off, int64_t n, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_scan_host", fn_name, profile, &cfg));
    PSB_TRY(host_db_check("psb_scan_host", out, cat, off, n, true));
    PSB_TRY(ensure_ctx());
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    psb_batch_t *b = new_batch(n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    const int rc = scan_host_into(cfg, profile, open, gap, cat, off, n, batch_outputs(b).data(), 0, &b->n_retried);
    if (rc != PSB_OK) { free_batch(b); return rc; }
    return scan_batch_done(cfg, profile, open, gap, off[n] - off[0], [&](int64_t i) { return span(off, i); }, b, out);
}

// The whole box from one process and one call (SURVEY 8b/8e): the database is cut into n_gpus contiguous
// ranges of equal residue count (contiguous, so every device uploads straight from the caller's arrays and
// writes straight into the caller-order result arrays -- no gather on either side), one resident worker
// thread per device runs the pipelined host scan on its range, and the call returns ONE batch in the
// caller's subject order.  No data-path collective: the ranges are independent.
int psb_scan_box(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                 const int64_t *off, int64_t n, int n_gpus, psb_batch_t **out) {
    if (out) *out = nullptr;
    FnConfig cfg;
    PSB_TRY(scan_check("psb_scan_box", fn_name, profile, &cfg));
    PSB_TRY(host_db_check("psb_scan_box", out, cat, off, n, true));
    const int ndev = psb_device_count();
    if (ndev <= 0) { set_error("no CUDA device available: libparasail_b200 has no CPU fallback (needs an sm_100a GPU)"); return PSB_ENODEV; }
    if (n_gpus <= 0 || n_gpus > ndev) n_gpus = ndev;
    if ((int64_t)n_gpus > n) n_gpus = (int)n;
    const HostClock clk{};
    PSB_TRY(ensure_ctx());   // the batch's pinned arrays are allocated by the calling thread
    psb_batch_t *b = new_batch(n, cfg);
    if (!b) { set_error("pinned host allocation failed"); return PSB_ENOMEM; }
    if (clk.on) std::fprintf(stderr, "[psb] scan_box: batch ready at %.3f ms\n", clk.ms());
    const int64_t total = off[n] - off[0];
    std::vector<int64_t> targets;
    for (int d = 1; d < n_gpus; ++d) targets.push_back(total * d / n_gpus);
    // device d scans range d; the devices past the last range have no work
    const std::vector<int64_t> cut = cut_subjects(off, n, targets);
    const int nranges = (int)cut.size() - 1;
    const std::array<int *, 6> hosts = batch_outputs(b);
    struct DeviceResult { int rc = PSB_OK, launches = 0; int64_t retried = 0; double ms = 0.0; std::string err; };
    std::vector<DeviceResult> res(nranges);
    for (int d = 0; d < nranges; ++d) {
        BoxWorker *w = box_worker(d);
        w->submit([&, d, w] {
            DeviceResult &r = res[d];
            r.rc = ensure_ctx();
            if (r.rc == PSB_OK) {
                g_ctx.last_ms = 0.0; g_ctx.launches = 0;
                r.rc = scan_host_into(cfg, profile, open, gap, cat, off + cut[d], cut[d + 1] - cut[d], hosts.data(), cut[d], &r.retried, &w->left);
                r.ms = g_ctx.last_ms; r.launches = g_ctx.launches;
            }
            if (r.rc != PSB_OK) r.err = psb_last_error();
        });
    }
    int rc = PSB_OK;
    Ctx &c = g_ctx;
    c.last_ms = 0.0; c.launches = 0;
    if (clk.on) std::fprintf(stderr, "[psb] scan_box: %d ranges submitted at %.3f ms\n", n_gpus, clk.ms());
    for (int d = 0; d < nranges; ++d) {
        box_worker(d)->wait();
        if (clk.on) std::fprintf(stderr, "[psb] scan_box: device %d done at %.3f ms\n", d, clk.ms());
        const DeviceResult &r = res[d];
        if (r.rc != PSB_OK && rc == PSB_OK) { rc = r.rc; set_error("psb_scan_box (device " + std::to_string(d) + "): " + r.err); }
        b->n_retried += r.retried;
        c.last_ms = std::max(c.last_ms, r.ms);   // the devices run side by side: the slowest one
        c.launches += r.launches;
    }
    if (rc != PSB_OK) { free_batch(b); return rc; }
    return scan_batch_done(cfg, profile, open, gap, total, [&](int64_t i) { return span(off, i); }, b, out);
}

int psb_host_scan_plan(int64_t total, double upload_ms_per_byte, double scan_ms_per_byte, int64_t *sizes_out, int cap) {
    if (total <= 0 || upload_ms_per_byte <= 0 || scan_ms_per_byte <= 0 || !sizes_out || cap <= 0) { set_error("psb_host_scan_plan: bad argument"); return PSB_EINVAL; }
    const std::vector<int64_t> sizes = plan_pieces(total, upload_ms_per_byte, scan_ms_per_byte);
    for (size_t k = 0; k < sizes.size() && (int)k < cap; ++k) sizes_out[k] = sizes[k];
    return (int)sizes.size();
}
}  // extern "C"
