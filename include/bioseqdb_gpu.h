/* include/bioseqdb_gpu.h -- C ABI of libbioseqdb_gpu.so, the B200 (sm_100a) replacement for the
 * libbwa calls that bioseqdb's bwa adapter makes.  Plain pointers and sizes only; no exceptions, no
 * longjmp; every entry point returns 0 / a handle on success and BSQ_ERR / NULL on failure with the
 * message available from bsq_last_error().
 *
 * Each entry point names the reference interface it replaces (paths relative to the reference repo):
 *   bsq_opts_init        mem_opt_init()                        bioseqdb/bwa.cpp:80
 *   bsq_index_new        BwaIndex::BwaIndex()                  bioseqdb/bwa.cpp:80, bwa.h:34
 *   bsq_index_set_opts   writes to BwaIndex::options           bioseqdb/extension.cpp:220-231
 *   bsq_index_add_ref    BwaIndex::add_ref_sequence            bioseqdb/bwa.cpp:82-105
 *   bsq_index_build      BwaIndex::build (pac2bwt, is_bwt, bwt_bwtupdate_core, bwt_cal_sa)
 *                                                              bioseqdb/bwa.cpp:20-53,107-128
 *   bsq_align_batch      the loop over BwaIndex::align_sequence (mem_align1 + mem_reg2aln per region)
 *                                                              bioseqdb/bwa.cpp:141-181, extension.cpp:362-370
 *   bsq_result_free / bsq_index_free   BwaIndex::~BwaIndex     bioseqdb/bwa.cpp:131-139
 *   bsq_index_save / bsq_index_load    (no reference counterpart: bwa index writes files, bwa mem loads them; the adapter rebuilds)
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef BIOSEQDB_GPU_H
#define BIOSEQDB_GPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSQ_OK 0
#define BSQ_ERR (-1)

/* The 12 fields of the SQL composite bwa_options (bioseqdb--0.0.0.sql:160-173), read by name at
 * extension.cpp:220-231.  Everything else keeps mem_opt_init() defaults; the scoring matrix is NOT
 * refreshed when a/b change (reference behaviour, SURVEY.md B#5). */
typedef struct bsq_opts {
    int32_t min_seed_len, max_occ, a, b, pen_clip3, pen_clip5, zdrop, w, o_del, e_del, o_ins, e_ins;
} bsq_opts;

/* == bntamb1_t (16 bytes), the hole record inside a NUCLSEQ datum (bioseqdb/sequence.h:13-14) */
typedef struct bsq_hole { int64_t offset; int32_t len; char amb; } bsq_hole;

/* One output row (64 bytes) = what BwaMatch is built from (bwa.cpp:151-177: rb, re, qb, qe, rid of the mem_alnreg_t; flag, is_rev, cigar,
 * score of its mem_aln_t) plus MAPQ and NM, which the path computes and the reference never exports (bwa.cpp:158).  rb/re are
 * positions in the doubled (forward+reverse) coordinate; pos is row-relative forward. */
typedef struct bsq_row {
    int64_t rb, re, pos;
    int64_t ref_id;              /* the id column of the reference row (bwa.cpp:160) */
    int32_t qb, qe, rid, score;
    int32_t NM;
    uint32_t cigar_off, n_cigar; /* bwa cigar words (len<<4|op, op: M0 I1 D2 S3) in bsq_result.cigar */
    uint16_t flag;               /* 0x100 = secondary */
    uint8_t mapq, is_rev;
} bsq_row;
/* The remaining mem_alnreg_t fields of a row (48 bytes): only the parity tests and debugging read them, so they travel only when
 * the index carries BSQ_FLAG_ROWS_EXT (bsq_index_set_flags); bsq_result.rows_ext is NULL otherwise. */
typedef struct bsq_row_ext {
    uint64_t hash;
    int32_t truesc, sub, csub, sub_n, w, seedcov, secondary, seedlen0, n_comp;
    float frac_rep;
} bsq_row_ext;

typedef struct bsq_result {
    uint64_t n_reads;
    uint64_t* row_off; /* n_reads + 1 */
    bsq_row* rows;     /* row_off[n_reads] rows, per read in reference order (score desc, hash) */
    uint32_t* cigar;
    uint64_t n_cigar_words;
    bsq_row_ext* rows_ext; /* parallel to rows, or NULL */
} bsq_result;

/* per-stage device timings of the last bsq_align_batch / bsq_align_resident call, milliseconds */
#define BSQ_NOTE_CHUNK_FALLBACK 1u /* bsq_align_batch: the result outgrew the chunk pipeline's estimate, the batch was re-run in one pass */
#define BSQ_NOTE_TABLE_DOWNGRADED 2u /* device memory was short for the batch pools: the seeding prefix table gave up its deepest level */
#define BSQ_NOTE_SA_COMPACTED 4u     /* device memory was short for the inverse SA or the batch pools: the index now keeps every 32nd SA entry
                                      * only (bsq_index_meta.sa_interval = 32) and resolves positions by LF walks; rows are unchanged */
typedef struct bsq_timing {
    float h2d, seed, chain, extend, finalize, d2h, total;
    uint32_t notes;    /* BSQ_NOTE_* bits: things a successful call wants its caller to know (never an error; see bsq_last_error for those) */
    uint64_t launches; /* kernels launched by the call */
    uint64_t h2d_bytes, d2h_bytes;
} bsq_timing;

typedef struct bsq_index bsq_index;

const char* bsq_last_error(void);
int bsq_device_count(void);

void bsq_opts_init(bsq_opts* o);
bsq_index* bsq_index_new(const bsq_opts* o, int device);
int bsq_index_set_opts(bsq_index* h, const bsq_opts* o);
#define BSQ_FLAG_ROWS_EXT 1u   /* results also carry bsq_row_ext records */
#define BSQ_FLAG_TWO_CHUNKS 2u /* bsq_align_batch* cuts a batch into at most two chunks, so that the whole batch is still in HBM when
                                * bsq_result_tuples is called on its result (which then uploads nothing) */
int bsq_index_set_flags(bsq_index* h, uint32_t flags);
int bsq_index_add_ref(bsq_index* h, int64_t id, const uint8_t* pac, uint32_t len, const bsq_hole* holes, uint32_t n_holes);
/* n reference rows in one call: NUCLSEQ datum images as PostgreSQL stores them (sequence.h:18-38), image i at bytes + off[i] --
 * what iterate_nuclseq_table (extension.cpp:157-195) holds after detoasting each row; same semantics as n calls of bsq_index_add_ref */
int bsq_index_add_ref_datums(bsq_index* h, uint64_t n, const int64_t* ids, const uint8_t* bytes, const uint64_t* off);
int bsq_index_build(bsq_index* h);
void bsq_index_free(bsq_index* h);

/* reads: concatenated ASCII (what BwaIndex::align_sequence hands to mem_align1 after to_text_palloc,
 * bwa.cpp:146-149), offs[n+1], ids[n] = the values lrand48() would have returned (SURVEY.md A.10).
 * Large batches run as two chunks whose host<->device copies overlap the other chunk's kernels; that overlap needs PAGE-LOCKED host
 * buffers (cudaHostAlloc / cudaHostRegister).  Pageable buffers are accepted -- the driver then stages every copy synchronously and
 * the call is correct but slower.  The result block itself is always page-locked (the library's own allocation). */
int bsq_align_batch(bsq_index* h, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n, bsq_result** out);
/* The same call with the reads as they sit in the database: n NUCLSEQ datum images (sequence.h:18-38), image i at bytes + off[i],
 * off[n + 1] -- what iterate_nuclseq_table holds for every query row (extension.cpp:362) BEFORE to_text_palloc expands it to one
 * byte per base.  2 bits per base cross the bus; the images are unpacked (holes -> ambiguous code 4) on the device.
 * In both calls ids may be NULL: the library then draws the ids itself, continuing the session's lrand48 stream kept in the handle
 * (one draw per read in call order, starting from glibc's fresh-process state; bsq_session_lrand48 reads / sets it). */
int bsq_align_batch_datums(bsq_index* h, const uint8_t* bytes, const uint64_t* off, const int64_t* ids, uint64_t n, bsq_result** out);
int bsq_session_lrand48(bsq_index* h, int set, uint64_t* state);
void bsq_result_free(bsq_result* r);
int bsq_last_timing(const bsq_index* h, bsq_timing* t);

/* Row materialisation (SURVEY.md 8f-2): the variable-length columns of the bwa_result tuple for every row of `res`, built on the
 * GPU.  Replaces, per row, extract_reference_subseq (bwa.cpp:55-68), cigar_compressed_to_string (bwa.cpp:70-77), the int32
 * ref_match_* arithmetic (bwa.cpp:171-173) and the two nuclseq_from_text calls of build_tuple_bwa (extension.cpp:285,290).
 * For row i: bytes + off[3i] = NUCLSEQ datum image of ref_subseq (varlena length word, holes_num, len, hole records, 2-bit codes;
 * 8-byte aligned, its true size is in the length word), bytes + off[3i+1] = image of query_subseq, bytes + off[3i+2] = the
 * NUL-terminated CIGAR string; ref_match[3i .. 3i+2] = ref_match_begin, ref_match_end, ref_match_len.
 * seqs/offs: the reads `res` was computed from (ASCII, as given to bsq_align_batch).  When `res` is the result of the handle's latest
 * bsq_align_batch* call and that batch is still resident (one or two chunks), rows, CIGARs and reads are taken from HBM: nothing is
 * uploaded and seqs / offs may be NULL. */
typedef struct bsq_tuples {
    uint64_t n_rows;
    uint64_t* off;       /* 3 n_rows + 1 */
    int32_t* ref_match;  /* 3 n_rows */
    uint8_t* bytes;
    uint64_t n_bytes;
    float device_ms;     /* kernels + copies of this call */
} bsq_tuples;
/* flags = 0 reproduces the reference bit for bit, quirks included.  Opt-in fix-ups (SURVEY.md 8f-3) for what the reference leaves as
 * TODO: BSQ_TUPLES_FIX_HOLE_OFFSETS rebases the ambiguity holes of reference row k by that row's offset in the concatenated text
 * (bwa.cpp:100-104 copies them un-rebased, so a hole of any row shadows the same offsets of row 1); BSQ_TUPLES_FIX_REVERSE reports a
 * reverse-strand hit in forward-strand coordinates -- ref_subseq is the forward text it covers, ref_match_begin/end are relative to
 * its row (bwa.cpp:156,172 use the doubled coordinate and read out of bounds).  With both flags ref_subseq is exactly the slice
 * [ref_match_begin, ref_match_end) of the reference row as it was inserted.  MAPQ and NM, computed but never exported by the
 * reference (bwa.cpp:158), are fields of bsq_row. */
#define BSQ_TUPLES_FIX_HOLE_OFFSETS 1u
#define BSQ_TUPLES_FIX_REVERSE 2u
int bsq_result_tuples(bsq_index* h, const bsq_result* res, const char* seqs, const uint64_t* offs, uint32_t flags, bsq_tuples** out);
void bsq_tuples_free(bsq_tuples* t);

/* Bulk text -> NUCLSEQ conversion (SURVEY.md 8f-4): nuclseq_in + nuclseq_from_text (extension.cpp:46-60, sequence.cpp:209-245) for n
 * sequences in one call -- what a bulk loader needs in place of bioseqdb-import's one INSERT (and one server-side nuclseq_in) per
 * FASTA record (bioseqdb-import/main.cpp:52-72).  text: the sequences back to back (upper case, as the importer sends them),
 * offs[n + 1].  Result: image i (datum bytes as in bsq_tuples) at bytes + off[i].  Fails like nuclseq_in: a letter outside
 * "ACGTNWSMKRYBDHV" ("invalid nucleotide in nuclseq_in: 'x'") or a sequence longer than INT32_MAX / 4. */
typedef struct bsq_nuclseqs {
    uint64_t n;
    uint64_t* off;      /* n + 1 */
    uint8_t* bytes;
    uint64_t n_bytes;
    float device_ms;    /* kernels + copies of this call */
} bsq_nuclseqs;
int bsq_nuclseq_from_text_batch(int device, const char* text, const uint64_t* offs, uint64_t n, bsq_nuclseqs** out);
void bsq_nuclseqs_free(bsq_nuclseqs* s);

/* Resident-input variant used by bench.py's `value` leg: upload once, run the kernels with inputs and
 * outputs resident in HBM, download on request. */
int bsq_reads_upload(bsq_index* h, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n);
int bsq_align_resident(bsq_index* h);
int bsq_result_download(bsq_index* h, bsq_result** out);

/* Index inspection (parity tests for SURVEY.md 8a rows a5-a7) and replication (8e: the built index is
 * broadcast to the other GPUs of the box).  what: see BSQ_ARR_*.  Sizes in bytes. */
enum { BSQ_ARR_PAC = 0, BSQ_ARR_OCC = 1, BSQ_ARR_SA = 2, BSQ_ARR_ANN_OFFSET = 3, BSQ_ARR_ANN_LEN = 4, BSQ_ARR_ANN_ID = 5, BSQ_ARR_COUNT = 6 };
typedef struct bsq_index_meta {
    int64_t l_pac; uint64_t seq_len, primary, L2[5]; uint64_t n_anns; uint32_t sa_bytes; /* 4 or 8 per SA entry */
    uint32_t built; uint64_t arr_bytes[BSQ_ARR_COUNT]; double build_ms; uint64_t build_launches;
    uint64_t sort_pass_bytes; /* algorithmic bytes moved by the radix passes of the build */
    /* 1: the full suffix array is resident (arr_bytes[BSQ_ARR_SA] = (seq_len + 1) * sa_bytes).  32: compact -- only SA[0], SA[32], ...
     * ((seq_len + 32) / 32 entries of sa_bytes, entry 0 = seq_len) are held, and there is no inverse SA.  The library compacts an index
     * by itself when the full layout cannot be allocated (BSQ_NOTE_SA_COMPACTED); it is never undone.  Rows are the same either way. */
    uint32_t sa_interval;
    uint32_t reserved;
} bsq_index_meta;
int bsq_index_get_meta(const bsq_index* h, bsq_index_meta* m);
/* Device memory held by the index right now: pac / occ / sa / ann, the derived arrays of the seeding kernel (inverse SA,
 * prefix table) and the batch pools.  What an index cache budgets against (SURVEY.md 8f-1: the reference rebuilds its
 * index on every call, extension.cpp:326,359; a cached handle keeps it resident instead). */
int bsq_index_device_bytes(const bsq_index* h, uint64_t* bytes);
int bsq_index_device_ptr(const bsq_index* h, int what, void** dptr);       /* device pointer of an index array */
int bsq_index_download(const bsq_index* h, int what, void* host_dst, uint64_t bytes);
int bsq_index_alloc_replica(bsq_index* h, const bsq_index_meta* m);        /* allocate arrays to receive a broadcast */
/* Completing a replica: the index also has HOST-side state (the reference rows' ambiguity holes, un-rebased as bwa.cpp:98-104
 * copies them; pac and annotation mirrors).  The source serialises it (size / get), the replica passes the blob to
 * bsq_index_replica_finish once its device arrays have been filled; from then on the replica answers every call -- alignment,
 * bsq_result_tuples with its hole overlay, the adapters' ref_subseq -- exactly like the source. */
int bsq_index_host_state_size(const bsq_index* h, uint64_t* bytes);
int bsq_index_host_state_get(const bsq_index* h, void* buf, uint64_t bytes);
int bsq_index_replica_finish(bsq_index* h, const void* host_state, uint64_t bytes);
int bsq_index_prepare(bsq_index* h, float* ms);   /* build the per-device derived arrays (inverse SA, prefix table) now; *ms = time spent */
/* Index files: build once, load in every process that aligns against the same reference (bwa index / bwa mem).  One file holds pac, Occ,
 * the annotations, the host state and 1/32 of the suffix array; the load rebuilds the full suffix array on the device by LF walks from
 * the samples.  The per-device derived arrays are not stored (bsq_index_prepare builds them).  Layout: bioseqdb_b200/csrc/index_file.cuh.
 * Writes the built index to `path` (written to a temporary name in the same directory, fsync'd, then renamed, so a reader never sees a
 * partial file).  key: 16 opaque bytes stored in the header (the index cache passes its digest), or NULL. */
int bsq_index_save(bsq_index* h, const char* path, const uint8_t* key);
/* Fills a FRESH handle (bsq_index_new, nothing added, not built) from a file written by bsq_index_save: header and sizes checked on the
 * host, sections uploaded and checksummed on the device, full SA rebuilt from its samples, host mirrors restored.  When the full SA
 * cannot be allocated, the index is loaded compact (sa_interval = 32): the samples are kept as they are, after a device check that
 * every one is <= seq_len and sample 0 == seq_len.  A compact index saves the same file it was loaded from.  key != NULL: the
 * file's key must match.  *ms = wall time of the call.  Options and flags are the handle's, as for any index.  On failure the handle is
 * left fresh. */
int bsq_index_load(bsq_index* h, const char* path, const uint8_t* key, float* ms);
/* Where the last successful bsq_index_load of the handle spent its time (file in the page cache or not: whatever the OS gave it). */
typedef struct bsq_index_load_info {
    uint64_t file_bytes;
    float read_ms;       /* wall: file read + upload of every section through the pinned staging buffers */
    float checksum_ms;   /* device: k_section_checksum over the uploaded sections */
    float sa_ms;         /* device: k_sa_from_samples (compact load: the check and narrowing of the samples) */
    float host_ms;       /* wall: host mirrors (pac, annotations, holes) restored */
    float total_ms;      /* wall: the whole call */
    uint64_t lf_steps;   /* LF steps of the suffix-array rebuild (seq_len + 1 for a sound file) */
    uint64_t lane_slots; /* warp iterations x 32 of the rebuild: lf_steps / lane_slots = its lane efficiency */
} bsq_index_load_info;
int bsq_index_last_load(const bsq_index* h, bsq_index_load_info* out);
/* One process, one host thread, several GPUs (SURVEY.md 8b / 8e; reference extension.cpp:346-377 is one backend, one thread): the
 * index of `built` is copied to devices[1..] (peer copies over NVLink + the host-side state), every device derives its own inverse SA /
 * prefix table, and a batch is cut into contiguous blocks of reads, one per device (read i keeps lrand48 id i).  The rows of all
 * devices come back in ONE result in read order.  devices[0] must be the device `built` lives on; `built` stays the caller's (options
 * and flags set on it apply to every device; free it after bsq_multi_free). */
typedef struct bsq_multi bsq_multi;
bsq_multi* bsq_multi_new(bsq_index* built, const int* devices, int n_devices);
void bsq_multi_free(bsq_multi* m);
int bsq_multi_devices(const bsq_multi* m);
int bsq_multi_align_batch(bsq_multi* m, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n, bsq_result** out);
int bsq_multi_align_batch_datums(bsq_multi* m, const uint8_t* bytes, const uint64_t* off, const int64_t* ids, uint64_t n, bsq_result** out);
int bsq_multi_last_timing(const bsq_multi* m, bsq_timing* t);   /* total = the slowest device's time from its first copy to the end of its download;
                                                                 * notes = the BSQ_NOTE_* bits of every device */
/* Row materialisation of a result on every device of `m`: the same tuples, byte for byte, as bsq_result_tuples(built, res, seqs, offs,
 * flags, ...), in one pinned block with the rows in read order, freed by bsq_tuples_free.  The reads are cut into the blocks of
 * bsq_multi_align_batch* (block d = reads [n d / D, n (d + 1) / D)) and device d builds the rows of block d.  A device whose batch still
 * holds that block of `res` (the latest bsq_multi_align_batch* call) takes rows, CIGARs and reads from HBM and uploads nothing; any other
 * device uploads only its block's rows, CIGAR words and reads.  seqs / offs may be NULL only when every device serves its block from HBM.
 * Any result is accepted: a caller-assembled, older or single-device result is staged across all devices.  device_ms = the slowest
 * device's kernels + copies.  An error on any device fails the call. */
int bsq_multi_result_tuples(bsq_multi* m, const bsq_result* res, const char* seqs, const uint64_t* offs, uint32_t flags, bsq_tuples** out);
/* Check of the device index against the text it was built from, by kernels that share no code with the builder or the seeding
 * kernels: SA is a permutation of 0..n (sum / sum of squares over all rows), adjacent suffixes are in order (text comparison), the BWT
 * string is T[SA[k]-1], bwt_invPsi(k) = L2[c] + occ(k, c) lands on the row of SA[k]-1 (what bwt_sa / bwt_extend rely on, libbwa bwt.c
 * behind reference bwa.cpp:149), the Occ checkpoints equal a recount of the blocks, L2 equals the symbol counts of the text.  Rows and
 * blocks are sampled (n_samples draws of each) unless n_samples covers them all.  Every *_bad must be 0 and *_ok 1 for a sound index.
 * On a compact index (sa_interval 32) the checks that need the full SA are not run: sa_permutation_ok and exhaustive are 0 and lf_bad
 * stays 0; sa_out_of_range counts samples > seq_len, order_* compares the suffixes of consecutive samples, rows_checked / bwt_bad check
 * the BWT symbol of sampled rows; Occ and L2 are checked as for a full index. */
typedef struct bsq_index_check {
    uint64_t rows;                 /* n + 1 */
    uint64_t exhaustive;           /* 1: every row and block was checked */
    uint64_t sa_permutation_ok, sa_out_of_range;
    uint64_t order_checked, order_bad, order_undecided;   /* undecided: equal over the comparison limit (64 Ki symbols) */
    uint64_t rows_checked, bwt_bad, lf_bad;
    uint64_t occ_blocks_checked, occ_bad;
    uint64_t l2_ok;
    double ms;
} bsq_index_check;
int bsq_index_verify(bsq_index* h, uint64_t n_samples, uint64_t seed, bsq_index_check* out);
int bsq_index_bwt_plain(const bsq_index* h, uint32_t* out);               /* the u32 stream of bwa.cpp:48-50 */
int bsq_index_sa_sampled(const bsq_index* h, uint64_t* out, uint64_t n_sa); /* bwt_cal_sa(bwt, 32) view */

/* Stage dumps for parity tests (device results copied to host): SMEM intervals after mem_collect_intv,
 * one record = 4 x u64 {x0,x1,x2,info}; cnt[n] = intervals per read, cap = records per read in `out`. */
int bsq_debug_seed(bsq_index* h, const char* seqs, const uint64_t* offs, uint64_t n, uint64_t* out, uint32_t cap, uint32_t* cnt);
/* out[i] = bwt_sa(rows[i]) for rows in [0, seq_len] (row 0 gives seq_len): SA[row] on a full index, the LF walk of the alignment
 * pipeline's position resolve pass on a compact one.  n < 2^31. */
int bsq_debug_sa_lookup(bsq_index* h, const uint64_t* rows, uint64_t n, uint64_t* out);
/* Kernel-level entry points for parity tests of the DP kernels on explicit job lists.
 * ext jobs: query/target are nt4 bytes; out = 6 x int32 per job {score,qle,tle,gtle,gscore,max_off}. */
int bsq_debug_ksw_extend(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                         const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out);
/* the same jobs through the thread-per-extension kernel (one job per thread, query side <= 136 bases); reversed != 0: q holds every
 * query back to front and the kernel's left-extension loader turns it round */
int bsq_debug_ksw_extend_thread(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                                const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out, int reversed);
/* global jobs: out_score[n]; cigar words written at cigar + cig_cap*i with counts in n_cigar[i] */
int bsq_debug_ksw_global(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                         const uint64_t* t_off, const int32_t* w, int32_t* out_score, uint32_t* cigar, uint32_t cig_cap, int32_t* n_cigar);
/* random 64-byte gather microbenchmark over the largest array the seeding kernels read (prefix table / full SA / Occ: at least the
 * size of the index, so that the figure is an HBM number): the seeding roofline denominator, GB/s */
int bsq_bench_gather(bsq_index* h, uint64_t n_loads, int reps, double* gbs);
/* DPX issue microbenchmark (independent __vimax3_s32 / __viaddmax_s32_relu): G instructions per second */
int bsq_bench_dpx(int device, int reps, double* gops);
/* Optional work counters of the last batch (the roofline's algorithmic units, SURVEY.md 8d):
 * out8 = {bwt_extend calls, SA lookups, equal-pos chain events, ksw_extend2 cells, calls, rows, ksw_global2 cells, calls} */
int bsq_set_counters(bsq_index* h, int on);
int bsq_debug_ctl(bsq_index* h, uint32_t* out64);   /* control words of the last batch (queue sizes of the finalize passes at [32..39]) */
int bsq_get_counters(const bsq_index* h, uint64_t* out8);

#ifdef __cplusplus
}
#endif
#endif
