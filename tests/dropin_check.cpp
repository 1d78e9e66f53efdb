// tests/dropin_check.cpp -- TEST INFRASTRUCTURE.  Compiles the drop-in adapter (integration/bioseqdb/bwa.{h,cpp}) against the
// reference's UNCHANGED sequence.h / sequence.cpp and against the lines of the reference's extension.cpp that use the adapter --
// bwa_index_from_query (extension.cpp:211-236: BwaIndex returned by value, bwa.options->field writes, build()) and the per-read
// loop (extension.cpp:362-370: bwa.align_sequence(*nuclseq) on a const-qualified call, rows read field by field).  The excerpt is
// cut out of the BIOSEQDB_SRC checkout at test time (tests/test_dropin.py) and #included here as dropin_excerpt.inc: nothing of the
// reference is stored in this repository.  Without a checkout, tests/dropin_src supplies a stand-in for sequence.h, sequence.cpp and
// the excerpt.  PostgreSQL is replaced by tests/pg_stub.
#include <algorithm>
#include <cstdio>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>
#include "bwa.h"

// ---- stand-ins for the PostgreSQL glue around the excerpt
typedef void* HeapTupleHeader;
typedef int Portal;
static std::vector<std::pair<int64_t, NucleotideSequence*>> g_rows;
template <class F> Portal iterate_nuclseq_table(const char*, Oid, F f) { for (auto& r : g_rows) f(r.first, r.second); return 0; }
static void SPI_cursor_close(Portal) {}
static int32_t get_opt_or(HeapTupleHeader, const char*, int32_t defval) { return defval; }

#include "dropin_excerpt.inc"     // bwa_index_from_query, verbatim from the reference

static size_t consume(const std::vector<BwaMatch>& aligns) {
    size_t n = 0;
    for (const BwaMatch& row : aligns)      // the fields build_tuple_bwa reads (extension.cpp:282-305)
        n += (size_t)row.ref_id + row.ref_subseq.size() + (size_t)row.ref_match_begin + (size_t)row.ref_match_end + (size_t)row.ref_match_len + row.query_subseq.size() +
             (size_t)row.query_match_begin + (size_t)row.query_match_end + (size_t)row.query_match_len + row.is_primary + row.is_secondary + row.is_reverse + row.cigar.size() + (size_t)row.score;
    return n;
}

int main() {
    std::string ref(3000, 'A');
    uint64_t s = 12345;
    for (auto& c : ref) { s = s * 6364136223846793005ULL + 1442695040888963407ULL; c = "ACGT"[(s >> 33) & 3]; }
    ref.replace(100, 5, "NNNNN");
    g_rows.push_back({7, nuclseq_from_text(ref)});
    const std::string read_text = ref.substr(1000, 150);
    try {
        BwaIndex bwa = bwa_index_from_query("select id, seq from refs", nullptr, 0);
        const BwaIndex& cbwa = bwa;                                   // align_sequence is const in the reference (bwa.h:37)
        const NucleotideSequence* nuclseq = nuclseq_from_text(read_text);
        std::vector<BwaMatch> aligns = cbwa.align_sequence(*nuclseq);
        if (aligns.size() != 1 || aligns[0].cigar != "150M" || aligns[0].ref_id != 7 || aligns[0].ref_match_begin != 1000 || aligns[0].score != 150 ||
            std::string(aligns[0].query_subseq) != read_text || aligns[0].ref_subseq != read_text) { printf("unexpected rows\n"); return 1; }
        printf("dropin ok: %zu row(s), checksum %zu, max_occ %d\n", aligns.size(), consume(aligns), bwa.options->max_occ);
        return 0;
    } catch (const std::runtime_error& e) {
        printf("dropin error: %s\n", e.what());
        return std::string(e.what()).find("no CUDA device") != std::string::npos ? 3 : 1;
    }
}
