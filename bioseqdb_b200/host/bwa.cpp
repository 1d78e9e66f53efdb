// bwa.cpp -- see bwa.h.  Mirrors reference bioseqdb/bwa.cpp:55-181 with libbwa replaced by the C ABI.
#include "bwa.h"
#include <algorithm>
#include <cstring>
#include <stdexcept>
#include <unistd.h>

namespace bioseqdb {

static void fail() { throw std::runtime_error(bsq_last_error()); }

std::string cigar_compressed_to_string(const uint32_t* raw, int len) {
    std::string cigar;
    for (int i = 0; i < len; ++i) {
        cigar += std::to_string(raw[i] >> 4);     // bam_cigar_oplen
        cigar += "MIDNSHP=XB"[raw[i] & 0xf];      // bam_cigar_opchr: bwa's soft clip (3) prints as 'N' (SURVEY.md B#4)
    }
    return cigar;
}

BwaIndex::BwaIndex(int device) : index(nullptr), lrand_state(0) {
    bsq_opts_init(&options);
    index = bsq_index_new(&options, device);
    if (!index) fail();
}

BwaIndex::~BwaIndex() { bsq_index_free(index); }

void BwaIndex::add_ref_sequence(int64_t id, const NucleotideSequence& seq) {
    offsets.push_back((int64_t)pac_forward.size() * 4);
    pac_forward.insert(pac_forward.end(), seq.pac(), seq.pac() + pac_byte_size(seq.len));
    holes.insert(holes.end(), seq.holes(), seq.holes() + seq.holes_num());
    if (bsq_index_add_ref(index, id, seq.pac(), seq.len, seq.holes(), seq.holes_num()) != BSQ_OK) fail();
}

void BwaIndex::build() {
    if (pac_forward.empty()) return;
    if (bsq_index_set_opts(index, &options) != BSQ_OK) fail();
    if (bsq_index_build(index) != BSQ_OK) fail();
}

void BwaIndex::save(const std::string& path, const uint8_t* key) const {
    if (bsq_index_save(index, path.c_str(), key) != BSQ_OK) fail();
}

void BwaIndex::load(const std::string& path, const uint8_t* key) {
    if (bsq_index_load(index, path.c_str(), key, nullptr) != BSQ_OK) fail();
    bsq_index_meta m;
    if (bsq_index_get_meta(index, &m) != BSQ_OK) fail();
    pac_forward.resize(m.arr_bytes[BSQ_ARR_PAC]);
    offsets.resize(m.n_anns);
    if (bsq_index_download(index, BSQ_ARR_PAC, pac_forward.data(), pac_forward.size()) != BSQ_OK) fail();
    if (bsq_index_download(index, BSQ_ARR_ANN_OFFSET, offsets.data(), offsets.size() * 8) != BSQ_OK) fail();
    uint64_t nb = 0;
    if (bsq_index_host_state_size(index, &nb) != BSQ_OK) fail();
    std::vector<uint8_t> st(nb);
    if (bsq_index_host_state_get(index, st.data(), nb) != BSQ_OK) fail();
    uint64_t nh = 0;
    memcpy(&nh, st.data(), 8);
    holes.resize(nh);
    if (nh) memcpy(holes.data(), st.data() + 8, nh * sizeof(bsq_hole));
}

uint64_t BwaIndex::device_bytes() const {
    uint64_t b = 0;
    if (bsq_index_device_bytes(index, &b) != BSQ_OK) fail();
    return b;
}

bool BwaIndex::compact() const {
    bsq_index_meta m;
    if (bsq_index_get_meta(index, &m) != BSQ_OK) fail();
    return m.sa_interval == 32;
}

uint32_t BwaIndex::last_notes() const {
    bsq_timing t;
    if (bsq_last_timing(index, &t) != BSQ_OK) fail();
    return t.notes;
}

// ---- BwaIndexCache
static inline uint64_t mix64(uint64_t h, uint64_t v) {          // splitmix-style accumulate
    h ^= v + 0x9E3779B97F4A7C15ULL + (h << 6) + (h >> 2);
    h *= 0xBF58476D1CE4E5B9ULL; h ^= h >> 31;
    return h;
}
static void digest_bytes(uint64_t& a, uint64_t& b, const void* p, size_t n) {
    const uint8_t* s = static_cast<const uint8_t*>(p);
    for (size_t i = 0; i < n; ++i) { a = (a ^ s[i]) * 0x100000001B3ULL; }                  // FNV-1a
    size_t i = 0;
    for (; i + 8 <= n; i += 8) { uint64_t w; memcpy(&w, s + i, 8); b = mix64(b, w); }
    uint64_t tail = 0; memcpy(&tail, s + i, n - i); b = mix64(b, tail ^ ((uint64_t)(n - i) << 56));
}

std::pair<uint64_t, uint64_t> BwaIndexCache::digest(const Rows& rows) {
    uint64_t a = 0xCBF29CE484222325ULL, b = 0x243F6A8885A308D3ULL;
    for (const auto& r : rows) {
        const int64_t hdr[3] = {r.first, (int64_t)r.second->len, (int64_t)r.second->holes_num()};
        digest_bytes(a, b, hdr, sizeof(hdr));
        digest_bytes(a, b, r.second->pac(), pac_byte_size(r.second->len));
        digest_bytes(a, b, r.second->holes(), (size_t)r.second->holes_num() * sizeof(bsq_hole));
    }
    return {a, b};
}

BwaIndexCache::BwaIndexCache(int device_, uint64_t max_bytes_, std::string directory_)
    : device(device_), max_bytes(max_bytes_), directory(std::move(directory_)) {}

std::string BwaIndexCache::file_path(const std::pair<uint64_t, uint64_t>& key) const {
    char hex[33];
    snprintf(hex, sizeof(hex), "%016llx%016llx", (unsigned long long)key.first, (unsigned long long)key.second);
    return directory + "/" + hex + ".bsqidx";
}

BwaIndex& BwaIndexCache::get(const Rows& rows, const bsq_opts& opts) {
    const auto key = digest(rows);
    for (auto it = lru.begin(); it != lru.end(); ++it)
        if (it->key == key) {
            ++hits;
            lru.splice(lru.begin(), lru, it);
            BwaIndex& ix = *lru.front().index;
            ix.options = opts;
            if (ix.ref_count() && bsq_index_set_opts(ix.index, &ix.options) != BSQ_OK) fail();
            return ix;
        }
    ++misses;
    uint8_t fkey[16];
    memcpy(fkey, &key.first, 8); memcpy(fkey + 8, &key.second, 8);
    bool empty = true;                     // an empty reference builds nothing (bwa.cpp:108-109): nothing to keep on disk
    for (const auto& r : rows) empty = empty && r.second->len == 0;
    const std::string path = directory.empty() || empty ? std::string() : file_path(key);
    std::unique_ptr<BwaIndex> ix;
    if (!path.empty() && access(path.c_str(), F_OK) == 0) {
        ix.reset(new BwaIndex(device));
        try { ix->load(path, fkey); ++disk_hits; }
        catch (const std::runtime_error&) { ++disk_errors; ix.reset(); }   // damaged or foreign: rebuilt and replaced below
    }
    if (ix) {
        ix->options = opts;
        if (bsq_index_set_opts(ix->index, &ix->options) != BSQ_OK) fail();
    } else {
        ix.reset(new BwaIndex(device));
        for (const auto& r : rows) ix->add_ref_sequence(r.first, *r.second);
        ix->options = opts;
        ix->build();
        if (!path.empty()) {
            try { ix->save(path, fkey); ++disk_saves; }
            catch (const std::runtime_error&) { ++disk_errors; }          // this call is served; the next process builds
        }
    }
    lru.push_front(Entry{key, std::move(ix)});
    uint64_t total = 0;
    for (const Entry& e : lru) total += e.index->device_bytes();
    while (lru.size() > 1 && total > max_bytes) {
        total -= lru.back().index->device_bytes();
        lru.pop_back();
        ++evictions;
    }
    return *lru.front().index;
}

std::vector<std::vector<BwaMatch>> BwaIndexCache::align_sequences(BwaIndex& ix, const std::vector<const NucleotideSequence*>& seqs) {
    ix.session_lrand_state() = lrand_state;
    auto out = ix.align_sequences(seqs);
    lrand_state = ix.session_lrand_state();
    return out;
}

std::string BwaIndex::extract_reference_subseq(int64_t rb, int64_t re) const {
    // Forward hits: the reference's arithmetic incl. the un-rebased hole overlay (SURVEY.md B#2).  Reverse hits
    // index past pac_forward in the reference (UB, B#3): defined here as the reverse-strand text.
    const int64_t l_pac = (int64_t)pac_forward.size() * 4;
    std::string subseq((size_t)(re - rb), '?');
    for (int64_t i = 0; i < re - rb; ++i) {
        const int64_t p = rb + i;
        const int c = p < l_pac ? pac_raw_get(pac_forward.data(), (size_t)p) : 3 - pac_raw_get(pac_forward.data(), (size_t)((l_pac << 1) - 1 - p));
        subseq[(size_t)i] = "ACGT"[c];
    }
    for (const bsq_hole& h : holes) {
        const int64_t l = std::max<int64_t>(h.offset, rb), r = std::min<int64_t>(h.offset + h.len, re);
        for (int64_t i = l; i < r; ++i) subseq[(size_t)(i - rb)] = h.amb;
    }
    return subseq;
}

void BwaIndex::batch_of(const std::vector<const NucleotideSequence*>& seqs, std::string& cat, std::vector<uint64_t>& offs, std::vector<int64_t>& ids) {
    offs.assign(seqs.size() + 1, 0);
    ids.resize(seqs.size());
    for (size_t i = 0; i < seqs.size(); ++i) {
        cat += seqs[i]->to_text();
        offs[i + 1] = cat.size();
        lrand_state = (lrand_state * 0x5DEECE66DULL + 0xBULL) & 0xFFFFFFFFFFFFULL;   // id = lrand48()
        ids[i] = (int64_t)(lrand_state >> 17);
    }
}

std::vector<std::vector<BwaMatch>> BwaIndex::matches_of(const bsq_result* res, const std::string& cat, const std::vector<uint64_t>& offs) const {
    std::vector<std::vector<BwaMatch>> out(offs.size() - 1);
    for (size_t i = 0; i < out.size(); ++i) {
        for (uint64_t k = res->row_off[i]; k < res->row_off[i + 1]; ++k) {
            const bsq_row& a = res->rows[k];
            const int64_t ref_offset = offsets[(size_t)a.rid];
            BwaMatch m;
            m.ref_id = a.ref_id;
            m.ref_subseq = extract_reference_subseq(a.rb, a.re);
            m.ref_match_begin = (int32_t)(a.rb - ref_offset);
            m.ref_match_end = (int32_t)(a.re - ref_offset);
            m.ref_match_len = (int32_t)(a.re - a.rb);
            m.query_subseq = cat.substr((size_t)(offs[i] + a.qb), (size_t)(a.qe - a.qb));
            m.query_match_begin = a.qb; m.query_match_end = a.qe; m.query_match_len = a.qe - a.qb;
            m.is_primary = (a.flag & 0x100) == 0; m.is_secondary = (a.flag & 0x100) != 0; m.is_reverse = a.is_rev != 0;
            m.cigar = cigar_compressed_to_string(res->cigar + a.cigar_off, (int)a.n_cigar);
            m.score = a.score; m.mapq = a.mapq; m.nm = a.NM;
            out[i].push_back(std::move(m));
        }
    }
    return out;
}

std::vector<std::vector<BwaMatch>> BwaIndex::align_sequences(const std::vector<const NucleotideSequence*>& seqs) {
    if (pac_forward.empty() || seqs.empty()) return std::vector<std::vector<BwaMatch>>(seqs.size());
    std::string cat; std::vector<uint64_t> offs; std::vector<int64_t> ids;
    batch_of(seqs, cat, offs, ids);
    bsq_result* res = nullptr;
    if (bsq_align_batch(index, cat.data(), offs.data(), ids.data(), seqs.size(), &res) != BSQ_OK) fail();
    auto out = matches_of(res, cat, offs);
    bsq_result_free(res);
    return out;
}

BwaTupleBatch BwaIndex::align_sequences_tuples(const std::vector<const NucleotideSequence*>& seqs, uint32_t flags) {
    if (pac_forward.empty() || seqs.empty()) return BwaTupleBatch();
    std::string cat; std::vector<uint64_t> offs; std::vector<int64_t> ids;
    batch_of(seqs, cat, offs, ids);
    bsq_result* res = nullptr;
    if (bsq_align_batch(index, cat.data(), offs.data(), ids.data(), seqs.size(), &res) != BSQ_OK) fail();
    bsq_tuples* tup = nullptr;
    if (bsq_result_tuples(index, res, cat.data(), offs.data(), flags, &tup) != BSQ_OK) { bsq_result_free(res); fail(); }
    return BwaTupleBatch(res, tup);
}

// ---- BwaMultiIndex
BwaMultiIndex::BwaMultiIndex(BwaIndex& ix_, const std::vector<int>& devices) : ix(ix_) {
    if (ix.pac_forward.empty()) return;
    multi = bsq_multi_new(ix.index, devices.data(), (int)devices.size());
    if (!multi) fail();
}

BwaMultiIndex::~BwaMultiIndex() { bsq_multi_free(multi); }

uint32_t BwaMultiIndex::last_notes() const {
    if (!multi) return 0;
    bsq_timing t;
    if (bsq_multi_last_timing(multi, &t) != BSQ_OK) fail();
    return t.notes;
}

std::vector<std::vector<BwaMatch>> BwaMultiIndex::align_sequences(const std::vector<const NucleotideSequence*>& seqs) {
    if (!multi || seqs.empty()) return std::vector<std::vector<BwaMatch>>(seqs.size());
    std::string cat; std::vector<uint64_t> offs; std::vector<int64_t> ids;
    ix.batch_of(seqs, cat, offs, ids);
    bsq_result* res = nullptr;
    if (bsq_multi_align_batch(multi, cat.data(), offs.data(), ids.data(), seqs.size(), &res) != BSQ_OK) fail();
    auto out = ix.matches_of(res, cat, offs);
    bsq_result_free(res);
    return out;
}

BwaTupleBatch BwaMultiIndex::align_sequences_tuples(const std::vector<const NucleotideSequence*>& seqs, uint32_t flags) {
    if (!multi || seqs.empty()) return BwaTupleBatch();
    std::string cat; std::vector<uint64_t> offs; std::vector<int64_t> ids;
    ix.batch_of(seqs, cat, offs, ids);
    bsq_result* res = nullptr;
    if (bsq_multi_align_batch(multi, cat.data(), offs.data(), ids.data(), seqs.size(), &res) != BSQ_OK) fail();
    bsq_tuples* tup = nullptr;
    if (bsq_multi_result_tuples(multi, res, cat.data(), offs.data(), flags, &tup) != BSQ_OK) { bsq_result_free(res); fail(); }
    return BwaTupleBatch(res, tup);
}

std::vector<std::vector<uint8_t>> nuclseq_datums_from_texts(const std::vector<std::string>& texts, int device) {
    std::string cat;
    std::vector<uint64_t> offs(texts.size() + 1, 0);
    for (size_t i = 0; i < texts.size(); ++i) { cat += texts[i]; offs[i + 1] = cat.size(); }
    bsq_nuclseqs* r = nullptr;
    if (bsq_nuclseq_from_text_batch(device, cat.data(), offs.data(), texts.size(), &r) != BSQ_OK) fail();
    std::vector<std::vector<uint8_t>> out(texts.size());
    for (size_t i = 0; i < texts.size(); ++i) {
        const uint8_t* d = r->bytes + r->off[i];
        out[i].assign(d, d + BwaTupleBatch::datum_size(d));
    }
    bsq_nuclseqs_free(r);
    return out;
}

std::vector<BwaMatch> BwaIndex::align_sequence(const NucleotideSequence& seq) {
    if (pac_forward.empty()) return {};
    return std::move(align_sequences({&seq})[0]);
}

}  // namespace bioseqdb
