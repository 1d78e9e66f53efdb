// seed.cuh -- batched SMEM seeding by FM-index backward/forward search (SURVEY.md A.2, A.4; replaces
// libbwa mem_collect_intv / bwt_smem1a / bwt_seed_strategy1 / bwt_extend reached from reference
// bioseqdb/bwa.cpp:149).  One warp cooperates per read: the two 64-byte Occ blocks of a bwt_extend are
// fetched by one coalesced warp load (lanes 0-15 -> block of k, lanes 16-31 -> block of l), symbol words
// are popcounted per lane and combined with redux.sync (seed.cu).  Bound by random 64-byte HBM/L2 reads.
#pragma once
#include "common.cuh"

struct SeedParams {
    const uint8_t* seqs;      // nt4 codes, concatenated
    const uint64_t* offs;     // n + 1
    uint32_t n_reads;
    Intv* out;                // n_reads x cap
    uint32_t* out_cnt;        // n_reads
    uint32_t cap;
    Intv* scratch;            // per resident warp: 3 lists of list_cap entries
    uint32_t list_cap;
    int lists_in_smem;        // narrow path: the two interval lists of a warp and the read live in shared memory
    uint32_t read_cap;        // bytes reserved per warp for the staged read (>= longest read, multiple of 16)
    const uint4* kmer_tab;    // prefix table: bi-intervals of all t-mers, t <= kmer_k (rows of up to 40 bits), or nullptr
    int kmer_k;
    const uint32_t* kmer_ztab; // sizes-only copy of the prefix table (same indexing), or nullptr
    const void* isa;          // inverse suffix array for the unique-match shortcut (rows as wide as the SA's), or nullptr
    uint32_t* ticket;
    uint32_t* overflow;       // set to 1 when a read needs more than cap intervals
    unsigned long long* n_extend;  // optional counter (roofline units); nullptr in production
    // reads the thread-per-read pass (seed_thread) left for seed_smem; nullptr = seed_smem takes every read
    const uint32_t* todo; const uint32_t* todo_cnt;
    // working arrays of the thread-per-read passes: packed reads (n_reads x seed_thread_words), per-read flags, records / logical
    // extensions after passes 1 and 2
    uint32_t* pk; uint32_t* rflag; uint32_t* cnt12; uint32_t* ext12;
};
// thread-per-read pass: runs before launch_seed when seed_thread_usable() (it needs the inverse SA and the prefix table); appends the
// reads it declines to p.todo
bool seed_thread_usable(const SeedParams& p, const DevOpts& o, uint32_t max_len);
int seed_thread_words(uint32_t max_len);
int launch_seed_thread(const SeedParams& p, const DevIndex& ix, const DevOpts& o, uint32_t max_len, uint32_t* ticket, cudaStream_t st);
void launch_seed(const SeedParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, int* n_warps_out);
int seed_resident_warps();
size_t kmer_table_bytes(int k);
int kmer_table_depth(uint64_t n);
void build_isa(const DevIndex& ix, void* isa, cudaStream_t st, uint64_t* launches);
void build_kmer_table(const DevIndex& ix, void* tab, int k, cudaStream_t st, uint64_t* launches);
void build_kmer_sizes(const void* tab, uint32_t* ztab, int k, cudaStream_t st, uint64_t* launches);
bool seed_lists_fit_smem(uint32_t list_cap, uint32_t read_cap, int sa_bytes);
