// harness.cpp -- PostgreSQL-free replay of the call order of reference bioseqdb/extension.cpp:211-236
// (bwa_index_from_query) and :346-378 (nuclseq_multi_search_bwa): reference rows and query rows come from
// two TSV files "<int id>\t<text>", options from the command line by the bwa_options field names, output is
// the 15-column bwa_result row (bioseqdb--0.0.0.sql:196-212) as TSV, one line per match.
//   harness <reference.tsv> <queries.tsv> [name=value ...]
// With check_tuples=1 the batch is aligned a second time through BwaIndex::align_sequences_tuples (same lrand48 ids) and every
// GPU-built column -- the two NUCLSEQ datums, the CIGAR string, ref_match_* -- is compared with what build_tuple_bwa
// (extension.cpp:282-305) would form from the BwaMatch; with check_bulk=1 the reference rows' texts go through the bulk
// text -> NUCLSEQ conversion and are compared with nuclseq_from_text.  A difference is an error (exit code 1).
// With index_cache=DIR the index comes from a BwaIndexCache with that directory, as a backend's would: the first process builds
// it and writes DIR/<digest>.bsqidx, every later one loads that file.  The counters go to stderr ("index_cache: ...").
// With devices=0,1 the batch is aligned (and, with check_tuples=1, materialised) on those GPUs through BwaMultiIndex, one contiguous
// block of reads per device, as a backend that drives several GPUs would; the output is the same.
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <stdexcept>
#include "bwa.h"

using namespace bioseqdb;

template <class F> static size_t iterate_nuclseq_table(const char* path, F f) {
    std::ifstream in(path);
    if (!in) throw std::runtime_error(std::string("cannot open ") + path);
    std::string line; size_t n = 0;
    while (std::getline(in, line)) {
        if (line.empty()) continue;
        size_t tab = line.find('\t');
        if (tab == std::string::npos) throw std::runtime_error("expected column of integers");   // extension.cpp:173
        if (tab + 1 >= line.size() + 1) continue;
        if (line.compare(0, tab, "NULL") == 0 || line.compare(tab + 1, std::string::npos, "NULL") == 0) continue;   // NULLs skipped (:186)
        int64_t id = std::stoll(line.substr(0, tab));
        f(id, nuclseq_from_text(std::string_view(line).substr(tab + 1)));
        ++n;
    }
    return n;
}

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s reference.tsv queries.tsv [bwa_options name=value ...]\n", argv[0]); return 2; }
    try {
        std::map<std::string, int32_t> opts;
        std::string index_cache;               // string options: taken out before the int options are parsed
        std::vector<int> devices;
        for (int i = 3; i < argc; ++i) {
            if (strncmp(argv[i], "index_cache=", 12) == 0) { index_cache = argv[i] + 12; continue; }
            if (strncmp(argv[i], "devices=", 8) == 0) {
                for (const char* p = argv[i] + 8; *p;) {
                    char* end = nullptr;
                    devices.push_back((int)strtol(p, &end, 10));
                    if (end == p || (*end && *end != ',')) throw std::runtime_error("devices is a comma-separated list of device numbers");
                    p = *end ? end + 1 : end;
                }
                continue;
            }
            const char* eq = strchr(argv[i], '=');
            if (!eq) throw std::runtime_error("options are name=value");
            opts[std::string(argv[i], (size_t)(eq - argv[i]))] = (int32_t)atoi(eq + 1);
        }
        auto get_opt_or = [&](const char* name, int32_t defval) {   // extension.cpp:197-209
            auto it = opts.find(name);
            if (it == opts.end()) return defval;
            if (it->second < 0) throw std::runtime_error(std::string("bwa_opt ") + name + " must be nonnegative");
            return it->second;
        };
        const bool check_tuples = opts.count("check_tuples") && opts["check_tuples"]; opts.erase("check_tuples");
        const bool check_bulk = opts.count("check_bulk") && opts["check_bulk"]; opts.erase("check_bulk");
        std::unique_ptr<BwaIndex> own;
        std::unique_ptr<BwaIndexCache> cache;
        if (index_cache.empty()) own.reset(new BwaIndex());
        else cache.reset(new BwaIndexCache(0, 96ull << 30, index_cache));
        std::vector<NucleotideSequence> ref_rows; std::vector<int64_t> ref_ids;
        size_t count = iterate_nuclseq_table(argv[1], [&](int64_t id, const NucleotideSequence& s) {
            if (own) own->add_ref_sequence(id, s);
            if (check_bulk || cache) { ref_rows.push_back(s); ref_ids.push_back(id); }
        });
        bsq_opts o;
        bsq_opts_init(&o);
        o.max_occ = get_opt_or("max_occ", (int32_t)std::max<size_t>(500, count * 2));
        o.min_seed_len = get_opt_or("min_seed_len", 19);
        o.a = get_opt_or("match_score", 1);
        o.b = get_opt_or("mismatch_penalty", 4);
        o.pen_clip3 = get_opt_or("pen_clip3", 5);
        o.pen_clip5 = get_opt_or("pen_clip5", 5);
        o.zdrop = get_opt_or("zdrop", 100);
        o.w = get_opt_or("bandwidth", 100);
        // defaults as delivered by the SQL function bwa_opts() (positional mix-up, SURVEY.md B#1)
        o.o_del = get_opt_or("o_del", 6);
        o.o_ins = get_opt_or("o_ins", 1);
        o.e_del = get_opt_or("e_del", 6);
        o.e_ins = get_opt_or("e_ins", 1);
        BwaIndex* ix = own.get();
        if (own) {
            own->options = o;
            own->build();
        } else {
            BwaIndexCache::Rows rows;
            for (size_t i = 0; i < ref_rows.size(); ++i) rows.emplace_back(ref_ids[i], &ref_rows[i]);
            ix = &cache->get(rows, o);
            fprintf(stderr, "index_cache: disk_hits=%llu disk_saves=%llu disk_errors=%llu\n", (unsigned long long)cache->disk_hits,
                    (unsigned long long)cache->disk_saves, (unsigned long long)cache->disk_errors);
        }
        BwaIndex& bwa = *ix;
        std::unique_ptr<BwaMultiIndex> multi;
        if (!devices.empty()) multi.reset(new BwaMultiIndex(bwa, devices));
        std::vector<int64_t> qids; std::vector<NucleotideSequence> queries;
        iterate_nuclseq_table(argv[2], [&](int64_t id, NucleotideSequence s) { qids.push_back(id); queries.push_back(std::move(s)); });
        std::vector<const NucleotideSequence*> ptrs;
        for (auto& q : queries) ptrs.push_back(&q);
        const uint64_t ids_at = bwa.session_lrand_state();
        auto all = multi ? multi->align_sequences(ptrs) : bwa.align_sequences(ptrs);
        // the layout of the built index (replicas start in it; a replica that compacts later says so in the multi call's notes)
        const uint32_t notes = multi ? multi->last_notes() : bwa.last_notes();
        fprintf(stderr, "index: layout=%s sa_compacted=%d\n", bwa.compact() ? "compact" : "full", (notes & BSQ_NOTE_SA_COMPACTED) ? 1 : 0);
        auto datum_of = [](const NucleotideSequence& s) {   // the datum as PostgreSQL stores it: length word + varlena payload
            std::vector<uint8_t> pl = s.varlena_payload();
            std::vector<uint8_t> d(4 + pl.size());
            const uint32_t w = (uint32_t)d.size() << 2;
            memcpy(d.data(), &w, 4); memcpy(d.data() + 4, pl.data(), pl.size());
            return d;
        };
        if (check_tuples) {
            bwa.session_lrand_state() = ids_at;
            BwaTupleBatch tb = multi ? multi->align_sequences_tuples(ptrs) : bwa.align_sequences_tuples(ptrs);
            size_t n_rows = 0;
            for (size_t i = 0; i < all.size(); ++i) {
                if (tb.row_begin(i + 1) - tb.row_begin(i) != all[i].size()) throw std::runtime_error("tuples: row count differs");
                for (size_t j = 0; j < all[i].size(); ++j, ++n_rows) {
                    const BwaMatch& m = all[i][j];
                    const uint64_t k = tb.row_begin(i) + j;
                    const std::vector<uint8_t> dr = datum_of(nuclseq_from_text(m.ref_subseq)), dq = datum_of(nuclseq_from_text(m.query_subseq));
                    if (BwaTupleBatch::datum_size(tb.ref_subseq_datum(k)) != dr.size() || memcmp(tb.ref_subseq_datum(k), dr.data(), dr.size())) throw std::runtime_error("tuples: ref_subseq datum differs");
                    if (BwaTupleBatch::datum_size(tb.query_subseq_datum(k)) != dq.size() || memcmp(tb.query_subseq_datum(k), dq.data(), dq.size())) throw std::runtime_error("tuples: query_subseq datum differs");
                    if (m.cigar != tb.cigar(k)) throw std::runtime_error("tuples: cigar differs");
                    if (m.ref_match_begin != tb.ref_match_begin(k) || m.ref_match_end != tb.ref_match_end(k) || m.ref_match_len != tb.ref_match_len(k)) throw std::runtime_error("tuples: ref_match differs");
                }
            }
            fprintf(stderr, "check_tuples: %zu rows identical\n", n_rows);
        }
        if (check_bulk) {
            std::vector<std::string> texts;
            for (const auto& s : ref_rows) texts.push_back(s.to_text());
            const auto datums = nuclseq_datums_from_texts(texts);
            for (size_t i = 0; i < ref_rows.size(); ++i) if (datums[i] != datum_of(ref_rows[i])) throw std::runtime_error("bulk: datum differs");
            fprintf(stderr, "check_bulk: %zu datums identical\n", ref_rows.size());
        }
        for (size_t i = 0; i < all.size(); ++i)
            for (const BwaMatch& m : all[i])
                printf("%lld\t%s\t%d\t%d\t%d\t%lld\t%s\t%d\t%d\t%d\t%s\t%s\t%s\t%s\t%d\n", (long long)m.ref_id, m.ref_subseq.c_str(), m.ref_match_begin,
                       m.ref_match_end, m.ref_match_len, (long long)qids[i], m.query_subseq.c_str(), m.query_match_begin, m.query_match_end,
                       m.query_match_len, m.is_primary ? "t" : "f", m.is_secondary ? "t" : "f", m.is_reverse ? "t" : "f", m.cigar.c_str(), m.score);
    } catch (const std::exception& e) {
        fprintf(stderr, "ERROR:  %s\n", e.what());
        return 1;
    }
    return 0;
}
