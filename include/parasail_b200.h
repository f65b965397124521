/*
 * parasail_b200.h -- C ABI of libparasail_b200.so, the B200-native replacement for the
 * slice of the parasail C library that parasail-rs binds through libparasail-sys 0.2.1
 * [REF Cargo.toml:15].  Every function below replaces the upstream parasail symbol of the
 * same name at the reference call site cited beside it; an unmodified parasail-rs linked
 * against this library runs its Gotoh H/E/F fill on the GPU (see INTEGRATION.md).
 *
 * Part 1 mirrors the 105 functions + 7 types imported by the four `use libparasail_sys::{..}`
 * blocks [REF src/aligner/mod.rs:4-7, src/profile/mod.rs:5-32, src/matrix/mod.rs:7-11,
 * src/alignment/mod.rs:6-23].  Part 2 adds the batched entry points named by the north star
 * (one-query-vs-many scan of a resident, packed database; many independent pairs), which have
 * no reference counterpart -- the reference loops over `Aligner::align` per subject
 * [REF src/aligner/mod.rs:397-452].
 *
 * There is no CPU fallback: every alignment entry point needs a CUDA device (sm_100a) and
 * reports failure loudly (see psb_last_error) when none is usable.
 */
#ifndef PARASAIL_B200_H
#define PARASAIL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Part 1a: types.  Field order of parasail_matrix_t follows upstream parasail.h because the
 * Rust side reads .type_, .size, .length and .matrix directly [REF src/matrix/mod.rs:193,
 * 228, 256-258].  Everything else is only reached through getters and is free to differ.
 * ---------------------------------------------------------------------------------------- */

#define PARASAIL_MATRIX_TYPE_SQUARE 0
#define PARASAIL_MATRIX_TYPE_PSSM 1

typedef struct parasail_matrix {
    const char *name;
    const int *matrix;      /* row-major, length x size (square: length == size) */
    const int *mapper;      /* 256 entries: byte -> column index; unknown bytes -> size-1 */
    int size;
    int max;
    int min;
    int *user_matrix;       /* non-NULL iff the matrix is heap-owned and editable */
    int type;               /* PARASAIL_MATRIX_TYPE_* ("type_" in the bindgen output) */
    int length;             /* number of rows */
    const char *alphabet;
    const char *query;      /* pssm built by convert_square_to_pssm: the query it encodes */
} parasail_matrix_t;
typedef struct parasail_matrix parasail_matrix; /* libparasail-sys exports both spellings */

/* result->flag bits (opaque to parasail-rs, which only uses the is_* getters) */
#define PARASAIL_FLAG_NW (1 << 0)
#define PARASAIL_FLAG_SG (1 << 1)
#define PARASAIL_FLAG_SW (1 << 2)
#define PARASAIL_FLAG_SG_S1_BEG (1 << 3)
#define PARASAIL_FLAG_SG_S1_END (1 << 4)
#define PARASAIL_FLAG_SATURATED (1 << 6)
#define PARASAIL_FLAG_BANDED (1 << 7)
#define PARASAIL_FLAG_NOVEC (1 << 8)
#define PARASAIL_FLAG_NOVEC_SCAN (1 << 9)
#define PARASAIL_FLAG_SCAN (1 << 10)
#define PARASAIL_FLAG_STRIPED (1 << 11)
#define PARASAIL_FLAG_DIAG (1 << 12)
#define PARASAIL_FLAG_BLOCKED (1 << 13)
#define PARASAIL_FLAG_SG_S2_BEG (1 << 14)
#define PARASAIL_FLAG_SG_S2_END (1 << 15)
#define PARASAIL_FLAG_STATS (1 << 16)
#define PARASAIL_FLAG_TABLE (1 << 17)
#define PARASAIL_FLAG_ROWCOL (1 << 18)
#define PARASAIL_FLAG_TRACE (1 << 19)
#define PARASAIL_FLAG_BITS_8 (1 << 20)
#define PARASAIL_FLAG_BITS_16 (1 << 21)
#define PARASAIL_FLAG_BITS_32 (1 << 22)
#define PARASAIL_FLAG_BITS_64 (1 << 23)

struct psb_result_extra; /* tables, rows/cols, trace bytes, stats: owned by the result */

typedef struct parasail_result {
    int score;
    int end_query;
    int end_ref;
    int flag;
    struct psb_result_extra *extra;
} parasail_result_t;

typedef struct parasail_cigar_ {
    uint32_t *seq;  /* len<<4 | op, op numbered by "MIDNSHP=X" */
    int len;
    int beg_query;
    int beg_ref;
} parasail_cigar_t;

typedef struct parasail_traceback_ {
    char *query; /* each malloc'd: parasail-rs adopts them with CString::from_raw */
    char *comp;
    char *ref;
} parasail_traceback_t;

typedef struct parasail_profile parasail_profile_t; /* opaque; device-resident */
typedef struct parasail_profile parasail_profile;

typedef struct parasail_result_ssw {
    uint16_t score1;
    int32_t ref_begin1;
    int32_t ref_end1;
    int32_t read_begin1;
    int32_t read_end1;
    uint32_t *cigar;
    int32_t cigarLen;
} parasail_result_ssw_t;

typedef parasail_result_t *parasail_function_t(const char *s1, int s1Len, const char *s2, int s2Len,
                                               int open, int gap, const parasail_matrix_t *matrix);
typedef parasail_result_t *parasail_pfunction_t(const parasail_profile_t *profile, const char *s2,
                                                int s2Len, int open, int gap);

/* ------------------------------------------------------------------------------------------
 * Part 1b: lookup by name.  Name grammar [REF src/aligner/mod.rs:289-331]:
 *   {nw|sg|sw}{_qb|_qe|_qx}{_db|_de|_dx}{_trace}{_stats}{_table|_rowcol}
 *   {_striped|_scan|_diag}{_profile}_{8|16|32|64|sat}
 * with or without a "parasail_" prefix.  NULL for anything else (parasail-rs then panics,
 * [REF src/aligner/mod.rs:353-358]).  s1 = query, s2 = reference, open/gap positive.
 * The returned function never returns NULL; device failures yield a result whose
 * parasail_result_is_saturated() is 1 and psb_last_error() is set.
 * ---------------------------------------------------------------------------------------- */
parasail_function_t *parasail_lookup_function(const char *funcname);   /* REF src/aligner/mod.rs:345 */
parasail_pfunction_t *parasail_lookup_pfunction(const char *funcname); /* REF src/aligner/mod.rs:349 */

/* ------------------------------------------------------------------------------------------
 * Part 1c: matrices [REF src/matrix/mod.rs:40, 62, 140-147, 158, 188-201, 238, 281, 304]
 * ---------------------------------------------------------------------------------------- */
parasail_matrix_t *parasail_matrix_create(const char *alphabet, int match, int mismatch);
const parasail_matrix_t *parasail_matrix_lookup(const char *matrixname); /* static; do not free */
parasail_matrix_t *parasail_matrix_from_file(const char *filename);
parasail_matrix_t *parasail_matrix_pssm_create(const char *alphabet, const int *values, int length);
parasail_matrix_t *parasail_matrix_copy(const parasail_matrix_t *original);
parasail_matrix_t *parasail_matrix_convert_square_to_pssm(const parasail_matrix_t *matrix,
                                                          const char *s1, int s1Len);
void parasail_matrix_set_value(parasail_matrix_t *matrix, int row, int col, int value);
void parasail_matrix_free(parasail_matrix_t *matrix);

/* ------------------------------------------------------------------------------------------
 * Part 1d: query profiles [REF src/profile/mod.rs:5-32, 93-103, 306-333, 384-390].  All 50
 * creators build the same device-resident profile: the ISA/width in the name only selects
 * the width the alignment is reported under.  Query and matrix are deep-copied (upstream
 * borrows them; parasail-rs drops both right after creation, SURVEY Appendix D Q2).
 * ---------------------------------------------------------------------------------------- */
#define PSB_DECL_PROFILE_CREATORS(ISA)                                                                         \
    parasail_profile_t *parasail_profile_create##ISA##_8(const char *s1, int s1Len, const parasail_matrix_t *m);   \
    parasail_profile_t *parasail_profile_create##ISA##_16(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create##ISA##_32(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create##ISA##_64(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create##ISA##_sat(const char *s1, int s1Len, const parasail_matrix_t *m); \
    parasail_profile_t *parasail_profile_create_stats##ISA##_8(const char *s1, int s1Len, const parasail_matrix_t *m);   \
    parasail_profile_t *parasail_profile_create_stats##ISA##_16(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create_stats##ISA##_32(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create_stats##ISA##_64(const char *s1, int s1Len, const parasail_matrix_t *m);  \
    parasail_profile_t *parasail_profile_create_stats##ISA##_sat(const char *s1, int s1Len, const parasail_matrix_t *m);
PSB_DECL_PROFILE_CREATORS()
PSB_DECL_PROFILE_CREATORS(_sse_128)
PSB_DECL_PROFILE_CREATORS(_avx_256)
PSB_DECL_PROFILE_CREATORS(_neon_128)
PSB_DECL_PROFILE_CREATORS(_altivec_128)
#undef PSB_DECL_PROFILE_CREATORS
void parasail_profile_free(parasail_profile_t *profile);

/* ------------------------------------------------------------------------------------------
 * Part 1e: results [REF src/alignment/mod.rs:64-98, 123-307, 390-504]
 * ---------------------------------------------------------------------------------------- */
void parasail_result_free(parasail_result_t *result);
int parasail_result_get_score(const parasail_result_t *result);
int parasail_result_get_end_query(const parasail_result_t *result);
int parasail_result_get_end_ref(const parasail_result_t *result);
int parasail_result_get_matches(const parasail_result_t *result);
int parasail_result_get_similar(const parasail_result_t *result);
int parasail_result_get_length(const parasail_result_t *result);
int *parasail_result_get_score_table(const parasail_result_t *result);
int *parasail_result_get_matches_table(const parasail_result_t *result);
int *parasail_result_get_similar_table(const parasail_result_t *result);
int *parasail_result_get_length_table(const parasail_result_t *result);
int *parasail_result_get_score_row(const parasail_result_t *result);
int *parasail_result_get_matches_row(const parasail_result_t *result);
int *parasail_result_get_similar_row(const parasail_result_t *result);
int *parasail_result_get_length_row(const parasail_result_t *result);
int *parasail_result_get_score_col(const parasail_result_t *result);
int *parasail_result_get_matches_col(const parasail_result_t *result);
int *parasail_result_get_similar_col(const parasail_result_t *result);
int *parasail_result_get_length_col(const parasail_result_t *result);
/* row-major int8 TraceFlags [REF src/alignment/table.rs:127-142].  Built on the first call: the device's flag-byte
 * block is made row-major then; for a long pair (query >= 2048 residues, traced on the whole-GPU wavefront kernel) the
 * block itself is fetched then, by running the pair once more on the kernel that writes flag bytes. */
int *parasail_result_get_trace_table(const parasail_result_t *result);
int parasail_result_is_nw(const parasail_result_t *result);
int parasail_result_is_sg(const parasail_result_t *result);
int parasail_result_is_sw(const parasail_result_t *result);
int parasail_result_is_saturated(const parasail_result_t *result);
int parasail_result_is_banded(const parasail_result_t *result);
int parasail_result_is_scan(const parasail_result_t *result);
int parasail_result_is_striped(const parasail_result_t *result);
int parasail_result_is_diag(const parasail_result_t *result);
int parasail_result_is_blocked(const parasail_result_t *result);
int parasail_result_is_stats(const parasail_result_t *result);
int parasail_result_is_stats_table(const parasail_result_t *result);
int parasail_result_is_stats_rowcol(const parasail_result_t *result);
int parasail_result_is_table(const parasail_result_t *result);
int parasail_result_is_rowcol(const parasail_result_t *result);
int parasail_result_is_trace(const parasail_result_t *result);

parasail_cigar_t *parasail_result_get_cigar(parasail_result_t *result, const char *seqA, int lena,
                                            const char *seqB, int lenb, const parasail_matrix_t *matrix);
char *parasail_cigar_decode(parasail_cigar_t *cigar); /* malloc'd; caller frees with free() */
void parasail_cigar_free(parasail_cigar_t *cigar);
parasail_traceback_t *parasail_result_get_traceback(parasail_result_t *result, const char *seqA, int lena,
                                                    const char *seqB, int lenb, const parasail_matrix_t *matrix,
                                                    char match, char pos, char neg);
void parasail_traceback_free(parasail_traceback_t *traceback);
void parasail_traceback_generic(const char *seqA, int lena, const char *seqB, int lenb, const char *nameA,
                                const char *nameB, const parasail_matrix_t *matrix, parasail_result_t *result,
                                char match, char pos, char neg, int width, int name_width, int use_stats);

/* ------------------------------------------------------------------------------------------
 * Part 1f: side APIs bound by parasail-rs (SURVEY 8f item 4).  parasail_nw_banded fills only the
 * band (half-width k, widened by the length difference) on the GPU's band kernel and sets the BANDED
 * flag; a band that covers the whole table is an ordinary nw fill, a band wider than the band kernel's
 * limit falls back to the masked full-table fill.  parasail_ssw is a local alignment with traceback.
 * ---------------------------------------------------------------------------------------- */
parasail_result_t *parasail_nw_banded(const char *s1, int s1Len, const char *s2, int s2Len, int open, int gap,
                                      int k, const parasail_matrix_t *matrix); /* REF src/aligner/mod.rs:471 */
parasail_result_ssw_t *parasail_ssw(const char *s1, int s1Len, const char *s2, int s2Len, int open, int gap,
                                    const parasail_matrix_t *matrix);          /* REF src/aligner/mod.rs:501 */
parasail_profile_t *parasail_ssw_init(const char *s1, int s1Len, const parasail_matrix_t *matrix,
                                      int8_t score_size);                       /* REF src/profile/mod.rs:345 */
void parasail_result_ssw_free(parasail_result_ssw_t *result);                   /* REF src/alignment/mod.rs:549 */

/* ------------------------------------------------------------------------------------------
 * Part 2: batched entry points (north star; SURVEY 8b "new batched entry points").
 * All return 0 on success or a negative PSB_E* code; psb_last_error() has the text.
 * ---------------------------------------------------------------------------------------- */
#define PSB_OK 0
#define PSB_EINVAL (-1)   /* bad name / NULL argument / empty sequence */
#define PSB_ENODEV (-2)   /* no usable CUDA device (no CPU fallback exists) */
#define PSB_ECUDA (-3)    /* CUDA runtime error */
#define PSB_ENOMEM (-4)
#define PSB_EUNSUPPORTED (-5)

const char *psb_last_error(void);         /* thread-local text of the last failure */
int psb_device_count(void);
int psb_set_device(int device);           /* per host thread; default = current CUDA device */
int psb_set_stream(void *cuda_stream);    /* per host thread; NULL = library-owned stream */
int psb_synchronize(void);

/* Per-pair results of one batch, struct-of-arrays in pinned host memory owned by the batch.
 * Arrays not produced by the requested function are NULL. */
typedef struct psb_batch {
    int64_t n;
    int flag;                 /* PARASAIL_FLAG_* describing every result in the batch */
    int *score, *end_query, *end_ref;
    int *matches, *similar, *length;      /* _stats */
    int64_t *cigar_off;                   /* _trace: n+1 offsets into cigar_ops */
    uint32_t *cigar_ops;                  /* len<<4|op, forward order */
    int *beg_query, *beg_ref;             /* _trace */
    uint8_t *saturated;                   /* 1 where an explicit _8/_16 width overflowed */
    int64_t n_retried;                    /* pairs re-run at 32 bit after 16-bit overflow */
    double cells;                         /* sum of Lq*Lr over the batch */
    void *impl;
} psb_batch_t;
void psb_batch_free(psb_batch_t *batch);

/* many independent pairs, one aligner configuration (configs C1, C3, C4).  q_off/r_off have
 * n+1 entries; sequences are raw residue bytes (not NUL-terminated).  fn_name follows the
 * grammar above without "_profile". */
int psb_align_pairs(const char *fn_name, const parasail_matrix_t *matrix, int open, int gap,
                    const uint8_t *q_cat, const int64_t *q_off, const uint8_t *r_cat, const int64_t *r_off,
                    int64_t n, psb_batch_t **out);

/* banded global alignment of many pairs: cell (i, j) is reachable iff lo <= j - i <= hi with d = rlen - qlen,
 * lo = -k + min(d, 0), hi = k + max(d, 0) (the band of parasail_nw_banded).  Only the band is filled: work per pair
 * is W * (qlen + rlen) cells with W = hi - lo + 1.  fn_name: the psb_align_pairs grammar restricted to nw (with or
 * without _trace / _stats); the batch is the one psb_align_pairs returns for that name, with PARASAIL_FLAG_BANDED in
 * batch->flag.  PSB_EINVAL: sg / sw names, k <= 0, NULL arguments, empty sequences; PSB_EUNSUPPORTED: _table /
 * _rowcol, or a pair whose band neither covers its table nor fits the band kernel (W > 4096). */
int psb_align_pairs_banded(const char *fn_name, const parasail_matrix_t *matrix, int open, int gap, int k,
                           const uint8_t *q_cat, const int64_t *q_off, const uint8_t *r_cat, const int64_t *r_off,
                           int64_t n, psb_batch_t **out);

/* a database resident on the current device: residues mapped through `matrix`'s mapper and
 * bit-packed on the GPU -- 5 bit/residue for protein alphabets, 3 bit for alphabets of up to 8 letters,
 * 2 bit when every residue present maps to one of the first four columns (A/C/G/T without wildcards) --
 * sorted by length, with the permutation kept so results come back in the caller's order.  The caller's
 * buffers may be reused as soon as psb_db_create returns. */
typedef struct psb_db psb_db_t;
psb_db_t *psb_db_create(const uint8_t *cat, const int64_t *off, int64_t n, const parasail_matrix_t *matrix);
int64_t psb_db_count(const psb_db_t *db);
int64_t psb_db_residues(const psb_db_t *db);
int64_t psb_db_device_bytes(const psb_db_t *db);
int psb_db_bits(const psb_db_t *db);      /* bits per packed residue: 2, 3 or 5 */
void psb_db_free(psb_db_t *db);

/* the step before the hot path (SURVEY 8f item 3; no reference counterpart -- parasail-rs callers hand
 * &[u8] to every call): FASTA -> (residues, offsets, names), FASTA -> resident database, and the packed,
 * length-sorted database as one file (layout in csrc/db_io.cu) so that a service does not sort and pack
 * at every start.  psb_db_load checks the file's alphabet against `matrix` when one is given. */
typedef struct psb_fasta psb_fasta_t;
psb_fasta_t *psb_fasta_read(const char *path);
int64_t psb_fasta_count(const psb_fasta_t *fa);
const uint8_t *psb_fasta_residues(const psb_fasta_t *fa);
const int64_t *psb_fasta_offsets(const psb_fasta_t *fa);      /* count + 1 entries */
const char *psb_fasta_name(const psb_fasta_t *fa, int64_t i, int *len);   /* header line of record i, not NUL-terminated */
void psb_fasta_free(psb_fasta_t *fa);
psb_db_t *psb_db_from_fasta(const char *path, const parasail_matrix_t *matrix);
int psb_db_save(const psb_db_t *db, const char *path);
psb_db_t *psb_db_load(const char *path, const parasail_matrix_t *matrix);

/* one resident profile against a resident database (config C2).  fn_name follows the grammar
 * with "_profile".  Every subject's result comes back in the caller's order; psb_batch_topk selects the
 * best k of them on the host. */
int psb_scan(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_db_t *db,
             psb_batch_t **out);
/* the profile's query against selected subjects of a resident database: the alignments behind the hits of a
 * psb_scan (psb_batch_topk gives the ids).  ids: n caller-order subject ids, repeats allowed, any order; or NULL
 * with n == psb_db_count(db) for every subject.  fn_name: the profile grammar ("_profile"), with or without
 * _trace / _stats; _table / _rowcol -> PSB_EUNSUPPORTED.  Result i belongs to ids[i]; the batch's arrays are
 * those psb_align_pairs returns for the same name without "_profile" (cigar_off / cigar_ops / beg_* for _trace).
 * The subjects are read out of the packed store on the device; nothing is uploaded but their ids. */
int psb_db_align(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_db_t *db,
                 const int64_t *ids, int64_t n, psb_batch_t **out);
/* subject `id` of a resident database as matrix column indices (what the kernels align): writes min(len, cap)
 * codes to `codes`, returns the subject's length, or a negative PSB_E* code */
int64_t psb_db_subject(const psb_db_t *db, int64_t id, uint8_t *codes, int64_t cap);
/* many query profiles against a resident database in one call, each query's best hits chosen on the GPU.  Let
 * kk = min(k, psb_db_count(db)).  The batch has nq * kk rows: row q*kk + r holds query q's r-th best subject, and
 * ids_out[q*kk + r] (nq * kk entries, allocated by the caller) is that subject's caller-order id.
 *   - Which subjects: per query, those of a score-only scan under fn_name without _trace and _stats, ordered by score
 *     descending, then by smaller id -- psb_batch_topk applied to that query's psb_scan.  Only the kk rows of each
 *     query leave the device.
 *   - Fields: with _trace or _stats, the rows are the alignments of those hits under fn_name, equal field for field
 *     (CIGAR included) to psb_db_align(fn_name, profiles[q], ..., ids of q, kk); the hits of all queries go through
 *     one pairs pass per group of queries with equal matrices (a PSSM profile has a pass of its own).  With a
 *     score-only name, score / end_query / end_ref are the scan's own values and no second pass runs.  Explicit
 *     _8 / _16 widths flag and zero saturated results as psb_scan and psb_db_align do.
 *   - n_retried: the sum over queries of what psb_scan reports; cells: the nq scans plus the alignment pass.
 *     psb_last_kernel_ms / psb_last_launches cover the whole call.
 *   - PSB_EINVAL: not a profile name, nq <= 0, k <= 0, a NULL argument, a NULL profiles[q] or a profile with
 *     another alphabet than the database (the message names q).  PSB_EUNSUPPORTED: _table / _rowcol, or
 *     nq * kk > 2^31 - 1.  Every check runs before any device work. */
int psb_db_search(const char *fn_name, const parasail_profile_t *const *profiles, int64_t nq, int open, int gap,
                  const psb_db_t *db, int k, int64_t *ids_out, psb_batch_t **out);
/* the same scan for a database that lives in HOST memory (pinned or pageable): the residues are cut
 * into pieces whose upload, device-side packing and scan are pipelined on two streams, so the
 * host-to-device copy hides under the kernels.  Nothing stays resident afterwards. */
int psb_scan_host(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                  const int64_t *off, int64_t n, psb_batch_t **out);
/* the whole box in one call from one process: the host database is cut into n_gpus contiguous ranges of
 * equal residue count, one resident worker thread per device runs the pipelined host scan of its range
 * straight out of / into the caller-order arrays, and ONE batch comes back in the caller's subject order.
 * n_gpus <= 0 means every visible device.  No collective is involved. */
int psb_scan_box(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const uint8_t *cat,
                 const int64_t *off, int64_t n, int n_gpus, psb_batch_t **out);
/* a resident database over the devices of the box, driven from one process.  The subjects are cut into contiguous
 * caller-id ranges of equal residue count (the cut of psb_scan_box); shard s is an ordinary psb_db resident on
 * devices[s], built, scanned and aligned by that device's worker thread.  devices may repeat (the shards of one device
 * are built and scanned one after another); devices == NULL: one shard per visible device, n_shards ignored.  There
 * are fewer shards than asked when there are too few subjects to cut.  NULL + psb_last_error() on failure: the
 * checks of psb_db_create, n_shards <= 0, a device ordinal out of range, no device, or a shard's build
 * ("(shard s, device d): ..."). */
typedef struct psb_box_db psb_box_db_t;
psb_box_db_t *psb_box_db_create(const uint8_t *cat, const int64_t *off, int64_t n, const parasail_matrix_t *matrix,
                                const int *devices, int n_shards);
int64_t psb_box_db_count(const psb_box_db_t *db);
/* the number of shards; fills first[0..shards] (first caller id of each shard, then n) and device[0..shards-1] if
 * non-NULL */
int psb_box_db_shards(const psb_box_db_t *db, int64_t *first, int *device);
int64_t psb_box_db_subject(const psb_box_db_t *db, int64_t id, uint8_t *codes, int64_t cap);   /* as psb_db_subject */
void psb_box_db_free(psb_box_db_t *db);
/* psb_scan, psb_db_align and psb_db_search on a box database: the same ids and rows, field for field, as the
 * single-device function on a psb_db built from the same arrays.  Each shard's work runs on its device's worker, the
 * devices side by side.
 *   - psb_box_scan writes each shard's results at its caller-order range of the batch.
 *   - psb_box_align aligns each id on the device that holds it and gathers the rows in the order of `ids`.
 *   - psb_box_search selects each query's min(k, n_s) best subjects on every shard s, merges them per query by the
 *     same rule (score descending, then smaller caller id) and keeps kk = min(k, n): every global top-kk subject is
 *     among its own shard's best, so the merge is exact.  With _trace / _stats each kept hit is then aligned on the
 *     device that holds it, one pairs pass per device and matrix group for all queries.
 *   - n_retried is the sum over shards.  It can differ from the single-device value: a 16-bit re-run takes the
 *     subject's word partner along, and the partners depend on the cut.
 *   - psb_last_kernel_ms is the slowest device's kernel time, psb_last_launches the sum over devices.
 *   - Errors: the codes and messages of the single-device function under the new name; a failure on a device reads
 *     "(shard s, device d): ...".  Every check runs before any device work.  Two host threads may call on one box
 *     database at once. */
int psb_box_scan(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_box_db_t *db,
                 psb_batch_t **out);
int psb_box_align(const char *fn_name, const parasail_profile_t *profile, int open, int gap, const psb_box_db_t *db,
                  const int64_t *ids, int64_t n, psb_batch_t **out);
int psb_box_search(const char *fn_name, const parasail_profile_t *const *profiles, int64_t nq, int open, int gap,
                   const psb_box_db_t *db, int k, int64_t *ids_out, psb_batch_t **out);
/* indices (caller order) of the k best scores of a scan, ties by smaller index; host-side merge */
int psb_batch_topk(const psb_batch_t *batch, int k, int64_t *idx_out, int *score_out);

/* residue-count balanced sharding of a database across n_shards GPUs (SURVEY 8e): writes
 * shard_of[i] in [0, n_shards) for each of the n sequences. */
int psb_shard_plan(const int64_t *off, int64_t n, int n_shards, int *shard_of);
/* Gives back what the library keeps between calls on the calling thread's device: the decision buffers its
 * pair lanes hold from batch to batch, recycled staging and page-locked blocks, and the unused part of the
 * device's stream-ordered memory pool.  Never needed for correctness; for a process that is done with large
 * batches and wants the memory for something else. */
int psb_trim(void);
/* how psb_scan_host / psb_scan_box cut a host database of `total` residues into pipelined pieces, given the
 * upload time and the scan time per residue (ms per byte; the library measures both while it runs): writes up
 * to `cap` piece sizes (bytes) and returns their number.  Host-only; exported so the plan can be inspected. */
int psb_host_scan_plan(int64_t total, double upload_ms_per_byte, double scan_ms_per_byte, int64_t *sizes_out, int cap);

/* device-time of the kernels of the last batch call on this thread, in milliseconds, and how
 * many kernel launches it issued (bench.py's gpu_launches) */
double psb_last_kernel_ms(void);
int psb_last_launches(void);
const char *psb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PARASAIL_B200_H */
