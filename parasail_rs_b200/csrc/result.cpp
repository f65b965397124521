// result.cpp -- parasail_result_t and its getters, CIGAR and traceback strings, as used by
// parasail-rs's Alignment [REF src/alignment/mod.rs:54-504].  Single-pair results are n = 1
// batches of the GPU path (pairs.cu); this file only reads what the device produced.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "psb_internal.h"

namespace psb {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }

// SURVEY A.8: an explicit 8/16-bit request whose true optimum does not fit that width is
// reported saturated (score/ends zeroed); "sat" and 32/64 return the exact result.
bool saturates(const FnConfig &cfg, const HostMatrix &m, int score, int qlen, int rlen, int open, int gap) {
    if (cfg.width != 8 && cfg.width != 16) return false;
    const long long hi = cfg.width == 8 ? 127 : 32767, lo = -hi - 1;
    if ((long long)score + std::max(m.max, 0) > hi) return true;
    if (cfg.mode != 2) {
        // global-style boundaries reach -(open + (L-1)*gap) along the first row/column
        long long worst = -(long long)open - (long long)(std::max(qlen, rlen) - 1) * gap + std::min(m.min, 0);
        bool bounded_rows = cfg.mode == 0 || !cfg.s1_beg || !cfg.s2_beg;
        if (bounded_rows && worst < lo) return true;
        if ((long long)score + std::min(m.min, 0) < lo) return true;
    }
    return false;
}

parasail_result_t *align_one(const FnConfig &cfg, const HostMatrix &m, const uint8_t *q, int qlen, const uint8_t *r,
                             int rlen, int open, int gap) {
    parasail_result_t *res = (parasail_result_t *)std::calloc(1, sizeof(parasail_result_t));
    if (!res) std::abort();
    res->extra = new psb_result_extra();
    res->flag = cfg.flag();
    if (cfg.width == 0) res->flag |= PARASAIL_FLAG_BITS_32;
    if (m.type == PARASAIL_MATRIX_TYPE_PSSM) qlen = m.length;
    res->extra->qlen = qlen; res->extra->rlen = rlen;
    if (m.size == 0 || !r || rlen <= 0 || qlen <= 0 || (m.type != PARASAIL_MATRIX_TYPE_PSSM && !q)) {
        if (g_error.empty()) set_error("alignment called with an empty sequence");
        res->flag |= PARASAIL_FLAG_SATURATED;
        return res;
    }
    int64_t qoff[2] = {0, qlen}, roff[2] = {0, rlen};
    std::vector<uint8_t> fake_q;
    if (!q) { fake_q.assign((size_t)qlen, 0); q = fake_q.data(); }
    PairsRequest req;
    req.cfg = cfg; req.matrix = &m; req.open = open; req.gap = gap;
    req.q_cat = q; req.q_off = qoff; req.r_cat = r; req.r_off = roff; req.n = 1;
    req.extra = res->extra;
    psb_batch_t *b = nullptr;
    const int rc = run_pairs(req, &b);
    if (rc != PSB_OK || !b) {
        // no CPU fallback: the failure is visible as a saturated, zeroed result + psb_last_error()
        res->flag |= PARASAIL_FLAG_SATURATED;
        std::fprintf(stderr, "libparasail_b200: alignment failed: %s\n", psb_last_error());
        if (b) free_batch(b);
        return res;
    }
    res->score = b->score[0]; res->end_query = b->end_query[0]; res->end_ref = b->end_ref[0];
    if (cfg.stats) { res->extra->matches = b->matches[0]; res->extra->similar = b->similar[0]; res->extra->length = b->length[0]; }
    if (cfg.trace && b->cigar_off) {
        // the trace walk ran on the device (walk_trace_kernel); keep its CIGAR with the result
        res->extra->cigar_ops.assign(b->cigar_ops + b->cigar_off[0], b->cigar_ops + b->cigar_off[1]);
        res->extra->beg_query = b->beg_query[0]; res->extra->beg_ref = b->beg_ref[0];
        if (res->extra->trace_blob.empty()) {
            // the pair ran on the wavefront kernel (a long pair): its flag bytes are fetched only if the caller asks for the
            // trace table [REF src/alignment/mod.rs:291-303], by running the pair once more on the kernel that writes them
            const std::vector<uint8_t> qv(q, q + qlen), rv(r, r + rlen);
            const HostMatrix mc = m;
            res->extra->trace_lazy = [cfg, mc, qv, rv, open, gap](psb_result_extra *x) {
                psb_result_extra tmp;
                tmp.qlen = x->qlen; tmp.rlen = x->rlen;
                const int64_t qo[2] = {0, (int64_t)qv.size()}, ro[2] = {0, (int64_t)rv.size()};
                PairsRequest again;
                again.cfg = cfg; again.matrix = &mc; again.open = open; again.gap = gap;
                again.q_cat = qv.data(); again.q_off = qo; again.r_cat = rv.data(); again.r_off = ro; again.n = 1;
                again.extra = &tmp; again.want_flag_bytes = true;
                psb_batch_t *b2 = nullptr;
                if (run_pairs(again, &b2) == PSB_OK) { x->trace_blob.swap(tmp.trace_blob); x->trace_K = tmp.trace_K; }
                else std::fprintf(stderr, "libparasail_b200: trace table of a long pair: %s\n", psb_last_error());
                if (b2) free_batch(b2);
            };
        }
    }
    free_batch(b);
    if (saturates(cfg, m, res->score, qlen, rlen, open, gap)) {
        res->flag |= PARASAIL_FLAG_SATURATED;
        res->score = 0; res->end_query = 0; res->end_ref = 0;
    }
    return res;
}

}  // namespace psb

extern "C" {

const char *psb_last_error(void) { return psb::g_error.c_str(); }
const char *psb_version(void) { return "parasail_b200 0.1 (sm_100a)"; }

void parasail_result_free(parasail_result_t *result) {
    if (!result) return;
    delete result->extra;
    result->extra = nullptr;
    std::free(result);
}

int parasail_result_get_score(const parasail_result_t *r) { return r->score; }
int parasail_result_get_end_query(const parasail_result_t *r) { return r->end_query; }
int parasail_result_get_end_ref(const parasail_result_t *r) { return r->end_ref; }
int parasail_result_get_matches(const parasail_result_t *r) { return r->extra ? r->extra->matches : 0; }
int parasail_result_get_similar(const parasail_result_t *r) { return r->extra ? r->extra->similar : 0; }
int parasail_result_get_length(const parasail_result_t *r) { return r->extra ? r->extra->length : 0; }

#define PSB_ARRAY_GETTER(NAME)                                                   \
    int *parasail_result_get_##NAME(const parasail_result_t *r) {                \
        return (r->extra && !r->extra->NAME.empty()) ? r->extra->NAME.data() : nullptr; \
    }
PSB_ARRAY_GETTER(score_table) PSB_ARRAY_GETTER(matches_table) PSB_ARRAY_GETTER(similar_table) PSB_ARRAY_GETTER(length_table)
PSB_ARRAY_GETTER(score_row) PSB_ARRAY_GETTER(matches_row) PSB_ARRAY_GETTER(similar_row) PSB_ARRAY_GETTER(length_row)
PSB_ARRAY_GETTER(score_col) PSB_ARRAY_GETTER(matches_col) PSB_ARRAY_GETTER(similar_col) PSB_ARRAY_GETTER(length_col)
#undef PSB_ARRAY_GETTER

// row-major int8 TraceFlags, the layout parasail-rs's TracebackTable reads [REF src/alignment/mod.rs:291-303]
int *parasail_result_get_trace_table(const parasail_result_t *r) {
    return r->extra ? (int *)r->extra->trace_table() : nullptr;
}

int parasail_result_is_nw(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_NW) != 0; }
int parasail_result_is_sg(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_SG) != 0; }
int parasail_result_is_sw(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_SW) != 0; }
int parasail_result_is_saturated(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_SATURATED) != 0; }
int parasail_result_is_banded(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_BANDED) != 0; }
int parasail_result_is_scan(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_SCAN) != 0; }
int parasail_result_is_striped(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_STRIPED) != 0; }
int parasail_result_is_diag(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_DIAG) != 0; }
int parasail_result_is_blocked(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_BLOCKED) != 0; }
int parasail_result_is_stats(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_STATS) != 0; }
int parasail_result_is_table(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_TABLE) != 0; }
int parasail_result_is_rowcol(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_ROWCOL) != 0; }
int parasail_result_is_trace(const parasail_result_t *r) { return (r->flag & PARASAIL_FLAG_TRACE) != 0; }
int parasail_result_is_stats_table(const parasail_result_t *r) {
    return (r->flag & PARASAIL_FLAG_STATS) && (r->flag & PARASAIL_FLAG_TABLE);
}
int parasail_result_is_stats_rowcol(const parasail_result_t *r) {
    return (r->flag & PARASAIL_FLAG_STATS) && (r->flag & PARASAIL_FLAG_ROWCOL);
}

// [REF src/alignment/mod.rs:400-407]  The walk itself ran on the GPU when the pair was aligned
// (walk_trace_kernel + compact_cigar_kernel); this only hands the stored run-length list out.
parasail_cigar_t *parasail_result_get_cigar(parasail_result_t *result, const char *seqA, int lena, const char *seqB,
                                            int lenb, const parasail_matrix_t *matrix) {
    if (!result || !result->extra || !(result->flag & PARASAIL_FLAG_TRACE) || (result->flag & PARASAIL_FLAG_SATURATED) ||
        !seqA || !seqB || !matrix) {
        psb::set_error("parasail_result_get_cigar: result has no trace");
        return nullptr;
    }
    if (lena != result->extra->qlen || lenb != result->extra->rlen) {
        psb::set_error("parasail_result_get_cigar: sequence lengths differ from the aligned pair");
        return nullptr;
    }
    const std::vector<uint32_t> &ops = result->extra->cigar_ops;
    parasail_cigar_t *c = (parasail_cigar_t *)std::calloc(1, sizeof(parasail_cigar_t));
    c->seq = (uint32_t *)std::malloc(sizeof(uint32_t) * std::max<size_t>(ops.size(), 1));
    std::memcpy(c->seq, ops.data(), sizeof(uint32_t) * ops.size());
    c->len = (int)ops.size();
    c->beg_query = result->extra->beg_query; c->beg_ref = result->extra->beg_ref;
    return c;
}

// [REF src/alignment/mod.rs:410] malloc'd: parasail-rs adopts it with CString::from_raw
char *parasail_cigar_decode(parasail_cigar_t *cigar) {
    static const char tab[] = "MIDNSHP=X";
    if (!cigar) return nullptr;
    std::string s;
    for (int k = 0; k < cigar->len; ++k) {
        const uint32_t op = cigar->seq[k] & 0xf;
        s += std::to_string(cigar->seq[k] >> 4);
        s.push_back(op > 8 ? 'M' : tab[op]);
    }
    char *out = (char *)std::malloc(s.size() + 1);
    std::memcpy(out, s.c_str(), s.size() + 1);
    return out;
}

void parasail_cigar_free(parasail_cigar_t *cigar) {
    if (!cigar) return;
    std::free(cigar->seq);
    std::free(cigar);
}

// [REF src/alignment/mod.rs:356-366] three malloc'd strings, adopted by the Rust side.  Pure
// formatting: the device-made CIGAR is expanded over the two sequences.
parasail_traceback_t *parasail_result_get_traceback(parasail_result_t *result, const char *seqA, int lena,
                                                    const char *seqB, int lenb, const parasail_matrix_t *matrix,
                                                    char match, char pos, char neg) {
    if (!result || !result->extra || !(result->flag & PARASAIL_FLAG_TRACE) || (result->flag & PARASAIL_FLAG_SATURATED) ||
        !seqA || !seqB || !matrix) {
        psb::set_error("parasail_result_get_traceback: result has no trace");
        return nullptr;
    }
    if (lena != result->extra->qlen || lenb != result->extra->rlen) return nullptr;
    psb::HostMatrix hm(matrix);
    std::string qs, cs, rs;
    int i = result->extra->beg_query, j = result->extra->beg_ref;
    for (uint32_t w : result->extra->cigar_ops) {
        const int op = (int)(w & 0xf);
        for (uint32_t t = 0; t < (w >> 4); ++t) {
            if (op == 7 || op == 8) {
                const int a = hm.mapper[(uint8_t)seqA[i]], b = hm.mapper[(uint8_t)seqB[j]];
                const int sub = hm.table[(size_t)hm.size * (hm.type == PARASAIL_MATRIX_TYPE_PSSM ? i : a) + b];
                qs.push_back(seqA[i]); rs.push_back(seqB[j]);
                cs.push_back(op == 7 ? match : (sub > 0 ? pos : neg));
                ++i; ++j;
            } else if (op == 1) { qs.push_back(seqA[i]); rs.push_back('-'); cs.push_back(' '); ++i; }
            else { qs.push_back('-'); rs.push_back(seqB[j]); cs.push_back(' '); ++j; }
        }
    }
    auto dup = [](const std::string &s) { char *p = (char *)std::malloc(s.size() + 1); std::memcpy(p, s.c_str(), s.size() + 1); return p; };
    parasail_traceback_t *tb = (parasail_traceback_t *)std::calloc(1, sizeof(parasail_traceback_t));
    tb->query = dup(qs); tb->comp = dup(cs); tb->ref = dup(rs);
    return tb;
}

void parasail_traceback_free(parasail_traceback_t *tb) {
    if (!tb) return;
    std::free(tb->query); std::free(tb->comp); std::free(tb->ref);
    std::free(tb);
}

// [REF src/alignment/mod.rs:324-339] prints the alignment in blocks of `width` columns
void parasail_traceback_generic(const char *seqA, int lena, const char *seqB, int lenb, const char *nameA,
                                const char *nameB, const parasail_matrix_t *matrix, parasail_result_t *result,
                                char match, char pos, char neg, int width, int name_width, int use_stats) {
    parasail_traceback_t *tb = parasail_result_get_traceback(result, seqA, lena, seqB, lenb, matrix, match, pos, neg);
    if (!tb) return;
    parasail_cigar_t *cig = parasail_result_get_cigar(result, seqA, lena, seqB, lenb, matrix);
    const int n = (int)std::strlen(tb->query);
    int qi = cig ? cig->beg_query : 0, ri = cig ? cig->beg_ref : 0;
    int matches = 0, gaps = 0;
    if (width <= 0) width = 80;
    for (int a = 0; a < n; a += width) {
        const int b = std::min(n, a + width);
        int qn = 0, rn = 0;
        for (int k = a; k < b; ++k) { qn += tb->query[k] != '-'; rn += tb->ref[k] != '-'; }
        std::printf("\n%*.*s %8d %.*s %8d\n", name_width, name_width, nameB ? nameB : "", ri + (rn ? 1 : 0), b - a, tb->ref + a, ri + rn);
        std::printf("%*s %8s %.*s\n", name_width, "", "", b - a, tb->comp + a);
        std::printf("%*.*s %8d %.*s %8d\n", name_width, name_width, nameA ? nameA : "", qi + (qn ? 1 : 0), b - a, tb->query + a, qi + qn);
        qi += qn; ri += rn;
    }
    for (int k = 0; k < n; ++k) { matches += tb->comp[k] == match && tb->query[k] != '-' && tb->ref[k] != '-'; gaps += tb->query[k] == '-' || tb->ref[k] == '-'; }
    if (use_stats) {
        std::printf("\nLength: %d\nIdentity: %d/%d\nGaps: %d/%d\nScore: %d\n", n, matches, n, gaps, n, result->score);
    }
    parasail_cigar_free(cig);
    parasail_traceback_free(tb);
}

// ---- side APIs (SURVEY 8f item 4) ----------------------------------------------------------------
// [REF src/aligner/mod.rs:457-489] banded global alignment: the fill is restricted to the diagonal band
// of half-width k (widened by the length difference so that the corner stays reachable); cells outside
// the band are unreachable (-inf).  Runs on the GPU through the general kernel's band mask.
parasail_result_t *parasail_nw_banded(const char *s1, int s1Len, const char *s2, int s2Len, int open, int gap, int k,
                                      const parasail_matrix_t *matrix) {
    psb::FnConfig cfg;
    cfg.mode = 0; cfg.width = 32; cfg.strategy = 0;
    cfg.band = k > 0 ? k : 0;
    psb::HostMatrix hm;
    if (matrix) hm = psb::HostMatrix(matrix);
    parasail_result_t *r = psb::align_one(cfg, hm, (const uint8_t *)s1, s1Len, (const uint8_t *)s2, s2Len, open, gap);
    r->flag &= ~PARASAIL_FLAG_STRIPED;
    r->flag |= PARASAIL_FLAG_BANDED | PARASAIL_FLAG_NOVEC;
    return r;
}

// [REF src/aligner/mod.rs:491-529; src/alignment/mod.rs:507-551] the SSW-compatible call: a local
// alignment with traceback, reported as score + begin/end coordinates + BAM-style CIGAR words.  The fill,
// the walk and the begin coordinates all come from the GPU trace path (sw_trace).  Never NULL: the
// reference dereferences the pointer unconditionally; a failed call returns a zeroed result.
parasail_result_ssw_t *parasail_ssw(const char *s1, int s1Len, const char *s2, int s2Len, int open, int gap,
                                    const parasail_matrix_t *matrix) {
    parasail_result_ssw_t *out = (parasail_result_ssw_t *)std::calloc(1, sizeof(parasail_result_ssw_t));
    if (!out) std::abort();
    if (!matrix || !s1 || !s2 || s1Len <= 0 || s2Len <= 0) { psb::set_error("parasail_ssw: empty sequence or NULL matrix"); return out; }
    psb::FnConfig cfg;
    cfg.mode = 2; cfg.trace = true; cfg.width = 0; cfg.strategy = 0;
    psb::HostMatrix hm(matrix);
    parasail_result_t *r = psb::align_one(cfg, hm, (const uint8_t *)s1, s1Len, (const uint8_t *)s2, s2Len, open, gap);
    if (!(r->flag & PARASAIL_FLAG_SATURATED) && r->extra) {
        out->score1 = (uint16_t)std::min(std::max(r->score, 0), 65535);
        out->ref_end1 = r->end_ref; out->read_end1 = r->end_query;
        out->ref_begin1 = r->extra->beg_ref; out->read_begin1 = r->extra->beg_query;
        const std::vector<uint32_t> &ops = r->extra->cigar_ops;
        out->cigarLen = (int32_t)ops.size();
        out->cigar = (uint32_t *)std::malloc(sizeof(uint32_t) * std::max<size_t>(ops.size(), 1));
        if (out->cigar && !ops.empty()) std::memcpy(out->cigar, ops.data(), sizeof(uint32_t) * ops.size());
    }
    parasail_result_free(r);
    return out;
}
// [REF src/profile/mod.rs:337-358] score_size 0 / 1 / 2 = 8 bit / 16 bit / both upstream; every width is the
// same resident profile here (the kernels pick their own width and re-run on overflow)
parasail_profile_t *parasail_ssw_init(const char *s1, int s1Len, const parasail_matrix_t *matrix, int8_t score_size) {
    (void)score_size;
    return parasail_profile_create_sat(s1, s1Len, matrix);
}
void parasail_result_ssw_free(parasail_result_ssw_t *r) {
    if (!r) return;
    std::free(r->cigar);
    std::free(r);
}

}  // extern "C"
