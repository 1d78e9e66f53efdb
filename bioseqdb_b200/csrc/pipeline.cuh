// pipeline.cuh -- records passed between the per-read kernels (seed -> chain -> extend -> finalize).
// Names follow libbwa's structs (SURVEY.md A.15): mem_seed_t, mem_chain_t, mem_alnreg_t.
#pragma once
#include "common.cuh"

struct SeedRec { int64_t rbeg; int32_t qbeg, len, score, next; };              // 24 B; `next` links a chain's seeds while chaining
struct ChainRec { int64_t pos; int32_t rid, n_seeds, seed_off, kept; uint32_t w; float frac_rep; };  // 32 B; seed_off is relative to the read's seed block
struct ChainTmp {                                                             // working record while chaining
    int64_t pos, f_rbeg, l_rbeg;
    int32_t f_qbeg, f_len, l_qbeg, l_len, head, tail, n, rid, first, kept;
    uint32_t w, pad;
};
struct RegRec {                                                               // mem_alnreg_t
    int64_t rb, re; uint64_t hash;
    int32_t qb, qe, rid, score, truesc, sub, csub, sub_n, w, seedcov, secondary, seedlen0, n_comp;
    float frac_rep;
};
// per read: where its block lives in the bump-allocated pools
struct ReadBlock { uint32_t base, n_alloc, n_chains, n_seeds; };

struct ChainParams {
    const uint8_t* seqs; const uint64_t* offs; uint32_t n_reads;
    const Intv* intv; const uint32_t* intv_cnt; uint32_t intv_cap;
    // pools (pool_cap records each); a read's block is [base, base + n_alloc) in every pool
    SeedRec* raw; ChainTmp* ctmp; uint32_t* ord; ChainRec* chains; SeedRec* seeds;
    uint32_t pool_cap; uint32_t* pool_top;
    ReadBlock* blocks;
    uint32_t* ticket; uint32_t* overflow;
    unsigned long long* counters;  // optional: [0] = SA lookups, [1] = equal-pos chain events (SURVEY A.5 corner)
    const double* logtab;          // host-libm log(l) for l <= longest read; nullptr when no read is long enough for mem_flt_chained_seeds
    unsigned long long* sw_cells;  // optional: cells of the seed-filter local SW
    uint32_t* todo; uint32_t* todo_cnt;   // reads the thread-per-read pass left for the warp kernel (nullptr = the warp kernel takes every read)
};
void launch_chain_thread(const ChainParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st);
void launch_chain(const ChainParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st);

// Result of one ksw_extend2 call computed ahead of sw_extend by the thread-per-extension kernels (extend_plan.cu).  sw_extend
// uses `out` only when the parameters of the call it is about to make equal the recorded ones (the call is a pure function
// of them), so a plan that guessed wrong costs time, never correctness.
struct ExtMemo {
    int64_t tpos;                      // doubled-coordinate position of target row 0 (rows walk down from it on the left side, up on the right)
    int32_t qlen, tlen, h0, state;     // state: 0 none, 1 planned, 3 planned but h0 waits for the left side's score, 2 done (out valid)
    int32_t out[6];                    // score, qle, tle, gtle, gscore, max_off
};
static_assert(sizeof(ExtMemo) == 48, "ExtMemo layout");
constexpr int EXT_MEMO_MAXQ = 136;     // longest query side the thread kernels take
constexpr int EXT_MEMO_CHAINS = 4;     // chains per read whose first extension is planned; job id = read * EXT_MEMO_CHAINS + chain

struct ExtendParams {
    const uint8_t* seqs; const uint64_t* offs; uint32_t n_reads;
    // thread-per-extension pre-pass (nullptr = off), J = n_reads * EXT_MEMO_CHAINS jobs: memo[0 .. J) left sides, memo[J .. 2J) right
    // sides; key[side * J + job] = query length of the planned job (0 = none); perm[side * J + ...] = jobs sorted by key; hist = 2 x 160 bin counts, then 2 x 160
    // bin starts, then 2 x 160 scatter cursors (zeroed by the host before the launch)
    ExtMemo* memo; uint8_t* memo_key; uint32_t* memo_perm; uint32_t* memo_hist;
    // reads the thread-per-read pass (ext_finish) could not complete, for sw_extend (nullptr = sw_extend takes every read)
    uint32_t* todo; uint32_t* todo_cnt;
    const ReadBlock* blocks; const ChainRec* chains; const SeedRec* seeds; uint64_t* srt;  // srt: one u64 per pooled seed
    RegRec* regs; uint32_t* reg_cnt;       // a read's regions live at regs[blocks[r].base ...], at most n_seeds of them
    uint8_t* scratch; size_t scratch_per_warp; uint32_t max_len, rseq_cap;
    uint32_t* ticket; uint32_t* overflow;
    uint32_t* need_rseq;           // atomicMax of the reference window a read needed when it exceeded rseq_cap (host grows and re-runs)
    unsigned long long* counters;  // optional: [0] = ksw_extend2 cells, [1] = calls, [2] = rows
};
void launch_extend(const ExtendParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st);
void launch_extend_finish(const ExtendParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st);
struct ExtAux { cudaStream_t st[3]; cudaEvent_t ev[4]; };
void launch_extend_memo(const ExtendParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, uint64_t* launches, const ExtAux& aux);
constexpr int EXT_MEMO_BINS = 160;
size_t extend_scratch_per_warp(uint32_t max_len, uint32_t rseq_cap);
int extend_resident_warps();

struct RowDev {  // a row as the finalisation kernels build it (one record per region)
    int64_t rb, re, pos; uint64_t hash;
    int32_t qb, qe, rid, score, truesc, sub, csub, sub_n, w, seedcov, secondary, seedlen0, n_comp;
    float frac_rep;
    int32_t is_rev, mapq, NM, flag;
    uint32_t cigar_off, n_cigar;
    int64_t ref_id;
};
static_assert(sizeof(RowDev) == 120, "RowDev layout");
struct RowPub {  // device image of bsq_row (include/bioseqdb_gpu.h): rows in read order, as they leave the device
    int64_t rb, re, pos, ref_id;
    int32_t qb, qe, rid, score, NM;
    uint32_t cigar_off, n_cigar;
    uint16_t flag; uint8_t mapq, is_rev;
};
static_assert(sizeof(RowPub) == 64, "RowPub must match bsq_row");
struct RowExt {  // device image of bsq_row_ext
    uint64_t hash;
    int32_t truesc, sub, csub, sub_n, w, seedcov, secondary, seedlen0, n_comp;
    float frac_rep;
};
static_assert(sizeof(RowExt) == 48, "RowExt must match bsq_row_ext");

struct FinalizeParams {
    const uint8_t* seqs; const uint64_t* offs; const int64_t* ids; uint32_t n_reads;
    const ReadBlock* blocks; RegRec* regs; const uint32_t* reg_cnt;
    RowDev* rows;                 // same indexing as regs (block base); row_cnt[r] rows valid
    uint32_t* row_cnt;
    uint32_t* cigar_pool; uint32_t cigar_cap; uint32_t* cigar_top;
    uint8_t* scratch; size_t scratch_per_warp; uint32_t max_len, z_cap;
    const int64_t* ann_id;
    // narrow-band regions are queued (read << 32 | row slot) for the thread-per-region kernel; regions that
    // need a wider band on a retry come back through wide_jobs.  narrow_jobs == nullptr disables the split.
    void* narrow_jobs; uint32_t narrow_cap;   // five lists of narrow_cap job records (24 B each): A, B (ping-pong between tries), S (equal-length regions), T4, T8 (tight first tries)
    uint32_t* narrow_cnt;                     // eight consecutive counters: list A, list B, list A (third tries), list S, sink, wide-band hand-over lists of passes 1..3
    uint64_t* wide_jobs; uint32_t* wide_cnt; uint8_t* narrow_z;
    uint32_t* ticket;              // eleven consecutive tickets: finalize, narrow pass 0..3, wide, wide register-band narrow kernel of passes 1..3, the two tight passes
    uint32_t* overflow;
    uint32_t* need_rseq;           // see ExtendParams
    unsigned long long* counters;  // optional: [0] = ksw_global2 cells, [1] = calls
    uint32_t* todo; uint32_t* todo_cnt;   // reads the thread-per-read pass left for regs_finalize (nullptr = no thread pass)
};
struct ExtAux;
// aux (optional): side streams + events; the two kernels of a DP pass (register band / wide register band) then run side by side
void launch_finalize(const FinalizeParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, uint32_t rseq_cap, int n_warps, uint64_t* launches, const ExtAux* aux);
size_t narrow_zbuf_bytes();
size_t finalize_scratch_per_warp(uint32_t max_len, uint32_t rseq_cap, uint32_t* z_cap_out);
int finalize_resident_warps();
