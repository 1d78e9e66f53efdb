// bwa.h -- host C++ mirror of the reference adapter interface (bioseqdb/bwa.h:15-48): BwaMatch and
// BwaIndex{add_ref_sequence, build, align_sequence}, same names and argument meaning, implemented over the
// C ABI of libbioseqdb_gpu.so instead of libbwa.  `options` is the POD the PG glue writes by field
// (extension.cpp:220-231).  Errors surface as std::runtime_error carrying bsq_last_error(); the PG glue
// turns them into ereport(ERROR).
#pragma once
#include <cstdint>
#include <list>
#include <memory>
#include <string>
#include <utility>
#include <vector>
#include "sequence.h"
#include "../../include/bioseqdb_gpu.h"

namespace bioseqdb {

struct BwaMatch {
    int64_t ref_id;
    std::string ref_subseq;
    int32_t ref_match_begin, ref_match_end, ref_match_len;
    std::string query_subseq;
    int32_t query_match_begin, query_match_end, query_match_len;
    bool is_primary, is_secondary, is_reverse;
    std::string cigar;
    int score;
    // computed by the path but not exported by the reference's SQL row (SURVEY.md 8a row a18)
    int mapq, nm;
};

// A batch's rows with their variable-length columns already in PostgreSQL's binary form (SURVEY.md 8f-2): what build_tuple_bwa
// (extension.cpp:282-305) hands to heap_form_tuple, built on the GPU by bsq_result_tuples.  Row k of read i: k in
// [row_begin(i), row_begin(i + 1)).  The datum pointers are 8-byte aligned NUCLSEQ images (the varlena length word is set).
class BwaTupleBatch {
public:
    BwaTupleBatch() = default;
    BwaTupleBatch(bsq_result* r, bsq_tuples* t) : res(r), tup(t) {}
    BwaTupleBatch(BwaTupleBatch&& o) noexcept : res(o.res), tup(o.tup) { o.res = nullptr; o.tup = nullptr; }
    BwaTupleBatch& operator=(BwaTupleBatch&& o) noexcept { release(); res = o.res; tup = o.tup; o.res = nullptr; o.tup = nullptr; return *this; }
    BwaTupleBatch(const BwaTupleBatch&) = delete;
    BwaTupleBatch& operator=(const BwaTupleBatch&) = delete;
    ~BwaTupleBatch() { release(); }
    uint64_t reads() const { return res ? res->n_reads : 0; }
    uint64_t row_begin(uint64_t read) const { return res ? res->row_off[read] : 0; }
    const bsq_row& row(uint64_t k) const { return res->rows[k]; }
    const uint8_t* ref_subseq_datum(uint64_t k) const { return tup->bytes + tup->off[3 * k]; }
    const uint8_t* query_subseq_datum(uint64_t k) const { return tup->bytes + tup->off[3 * k + 1]; }
    const char* cigar(uint64_t k) const { return reinterpret_cast<const char*>(tup->bytes + tup->off[3 * k + 2]); }
    int32_t ref_match_begin(uint64_t k) const { return tup->ref_match[3 * k]; }
    int32_t ref_match_end(uint64_t k) const { return tup->ref_match[3 * k + 1]; }
    int32_t ref_match_len(uint64_t k) const { return tup->ref_match[3 * k + 2]; }
    static size_t datum_size(const uint8_t* datum) { uint32_t w; __builtin_memcpy(&w, datum, 4); return w >> 2; }   // VARSIZE of a 4-byte header
private:
    void release() { if (tup) bsq_tuples_free(tup); if (res) bsq_result_free(res); tup = nullptr; res = nullptr; }
    bsq_result* res = nullptr; bsq_tuples* tup = nullptr;
};

// Bulk text -> NUCLSEQ (SURVEY.md 8f-4): nuclseq_in for a whole batch on the GPU; datum i = bytes of image i.
std::vector<std::vector<uint8_t>> nuclseq_datums_from_texts(const std::vector<std::string>& texts, int device = 0);

class BwaIndex {
public:
    explicit BwaIndex(int device = 0);
    ~BwaIndex();
    BwaIndex(const BwaIndex&) = delete;
    BwaIndex& operator=(const BwaIndex&) = delete;

    std::vector<BwaMatch> align_sequence(const NucleotideSequence& seq);
    // batched form of the per-read loop at extension.cpp:362-370: one GPU pass for all reads
    std::vector<std::vector<BwaMatch>> align_sequences(const std::vector<const NucleotideSequence*>& seqs);
    // the same pass, rows left in binary tuple form (flags: BSQ_TUPLES_FIX_*, 0 = the reference's behaviour)
    BwaTupleBatch align_sequences_tuples(const std::vector<const NucleotideSequence*>& seqs, uint32_t flags = 0);
    void build();
    void add_ref_sequence(int64_t id, const NucleotideSequence& seq);
    // Index files (bsq_index_save / bsq_index_load): build once, load in any process.  key: 16 bytes kept in the file's header, or
    // nullptr.  load() fills a fresh index and refills the host copies extract_reference_subseq reads (pac, row offsets, holes).
    void save(const std::string& path, const uint8_t* key = nullptr) const;
    void load(const std::string& path, const uint8_t* key = nullptr);

    bsq_opts options;            // written by bwa_index_from_query before build()
    size_t ref_count() const { return offsets.size(); }
    uint64_t device_bytes() const;           // bsq_index_device_bytes
    uint64_t& session_lrand_state() { return lrand_state; }

private:
    friend class BwaIndexCache;
    friend class BwaMultiIndex;
    std::vector<uint8_t> pac_forward;      // kept on the host for extract_reference_subseq (bwa.cpp:55-68)
    std::vector<bsq_hole> holes;           // not rebased, as in the reference (bwa.cpp:100-104)
    std::vector<int64_t> offsets;
    bsq_index* index;
    uint64_t lrand_state;                  // glibc lrand48 state: one draw per aligned read (SURVEY.md A.10)
    std::string extract_reference_subseq(int64_t ref_begin, int64_t ref_end) const;
    // the reads as one text with offsets, and their ids: one lrand48 draw per read from the session state
    void batch_of(const std::vector<const NucleotideSequence*>& seqs, std::string& cat, std::vector<uint64_t>& offs, std::vector<int64_t>& ids);
    // the BwaMatch rows of every read of `res`, computed from the reads in cat / offs
    std::vector<std::vector<BwaMatch>> matches_of(const bsq_result* res, const std::string& cat, const std::vector<uint64_t>& offs) const;
};

// Several GPUs behind one backend (bsq_multi_*): the built `ix` replicated to `devices` (devices[0] is the device `ix` lives on; a
// device may repeat).  A batch is cut into one contiguous block of reads per device and its rows come back in read order, with ids
// drawn from ix's session lrand48 state exactly as BwaIndex draws them.  Options and flags are those of `ix`; it must outlive this.
class BwaMultiIndex {
public:
    BwaMultiIndex(BwaIndex& ix, const std::vector<int>& devices);
    ~BwaMultiIndex();
    BwaMultiIndex(const BwaMultiIndex&) = delete;
    BwaMultiIndex& operator=(const BwaMultiIndex&) = delete;

    std::vector<std::vector<BwaMatch>> align_sequences(const std::vector<const NucleotideSequence*>& seqs);
    // each device materialises the tuples of its own block from HBM (bsq_multi_result_tuples)
    BwaTupleBatch align_sequences_tuples(const std::vector<const NucleotideSequence*>& seqs, uint32_t flags = 0);

private:
    BwaIndex& ix;
    bsq_multi* multi = nullptr;            // none while `ix` holds no reference rows: every call then returns no rows, as BwaIndex's
};

// Index cache keyed by the content of the reference rows (SURVEY.md 8f-1).  The reference rebuilds a BwaIndex inside
// every SQL call (bwa_index_from_query, extension.cpp:211-236, called at :326 and :359); the cache keeps built indexes
// resident in HBM, finds them again by a 128-bit digest of (id, length, payload, holes) of every row in cursor order,
// applies the call's options to the cached handle, and evicts least-recently-used indexes beyond `max_bytes`.  It also
// owns the session's lrand48 state (process-wide in the reference), lending it to the index that serves a call.
// With a `directory` a memory miss first looks for `<directory>/<digest hex>.bsqidx` (another backend may have built it) and
// loads it; otherwise it builds and writes the file.  A file that does not load is rebuilt and replaced; a failed write only
// counts in disk_errors.  Empty references are never written.
class BwaIndexCache {
public:
    using Rows = std::vector<std::pair<int64_t, const NucleotideSequence*>>;
    explicit BwaIndexCache(int device = 0, uint64_t max_bytes = 96ull << 30, std::string directory = "");
    BwaIndex& get(const Rows& rows, const bsq_opts& opts);     // built, options applied; owned by the cache
    // align through a cached index with the session's id stream
    std::vector<std::vector<BwaMatch>> align_sequences(BwaIndex& ix, const std::vector<const NucleotideSequence*>& seqs);
    uint64_t hits = 0, misses = 0, evictions = 0;
    uint64_t disk_hits = 0, disk_saves = 0, disk_errors = 0;
    static std::pair<uint64_t, uint64_t> digest(const Rows& rows);
    std::string file_path(const std::pair<uint64_t, uint64_t>& key) const;
private:
    struct Entry { std::pair<uint64_t, uint64_t> key; std::unique_ptr<BwaIndex> index; };
    std::list<Entry> lru;                  // front = most recently used
    int device; uint64_t max_bytes; std::string directory; uint64_t lrand_state = 0;
};

std::string cigar_compressed_to_string(const uint32_t* raw, int len);   // htslib letters on bwa op codes (bwa.cpp:70-77)

}  // namespace bioseqdb
