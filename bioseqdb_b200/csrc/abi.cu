// abi.cu -- the extern "C" boundary (include/bioseqdb_gpu.h) and the host-side orchestration of the
// per-batch kernel pipeline: upload -> seed_smem -> chain_build -> sw_extend -> regs_finalize -> compact
// -> download (+ MAPQ, which needs libm's log, SURVEY.md A.12).  Pools are bump-allocated on the device
// and grown by re-running the batch when a kernel raises the overflow flag; there is no CPU fallback for
// any stage.
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <vector>
#include <chrono>
#include <algorithm>
#include <mutex>
#include <memory>
#include "../../include/bioseqdb_gpu.h"
#include "common.cuh"
#include "index_build.cuh"
#include "seed.cuh"
#include "pipeline.cuh"
#include "index_verify.cuh"
#include "tuples.cuh"
#include "loader.cuh"
#include "primitives.cuh"
#include "debug_kernels.cuh"
#include "index_file.cuh"

static thread_local char g_err[1024] = "";
void bsq_set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
// every extern "C" entry point starts with a clean error string: bsq_last_error() after a call describes THAT call
#define BSQ_ENTRY() do { g_err[0] = 0; } while (0)
// CUDA_CHECK with the caller's own prefix: "<what>: <error of the failed call>"
#define CUDA_CHECK_AS(what, x) do { if ((x) != cudaSuccess) { bsq_set_error("%s: %s", what, cudaGetErrorString(cudaGetLastError())); return BSQ_ERR; } } while (0)

static_assert(sizeof(bsq_row) == sizeof(RowPub) && sizeof(bsq_row_ext) == sizeof(RowExt), "bsq_row / RowPub mismatch");
static_assert(sizeof(bsq_hole) == 16, "bsq_hole must match bntamb1_t");

namespace {

// A device buffer that frees itself when its scope ends
template <class T> struct DevBuf {
    T* p = nullptr; size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t n) {      // exactly n elements, the old contents gone
        release();
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n; else p = nullptr;
        return e;
    }
    cudaError_t ensure(size_t n) { return n <= cap ? cudaSuccess : alloc(n + n / 8 + 16); }   // room for n, with slack for the next growth
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    size_t bytes() const { return cap * sizeof(T); }
};

// An event or stream that is destroyed when its scope ends; create it into .h
template <class H, cudaError_t (*Destroy)(H)> struct Owned {
    H h = nullptr;
    Owned() = default;
    Owned(const Owned&) = delete;
    Owned& operator=(const Owned&) = delete;
    ~Owned() { if (h) Destroy(h); }
    operator H() const { return h; }
};
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;

// device scratch of the row materialisation (bsq_result_tuples): a lane's own, or a call's for a result that is not resident
struct TupleScratch { DevBuf<uint64_t> off, tmp; DevBuf<uint32_t> row_read, nholes; DevBuf<int32_t> rm; DevBuf<uint8_t> bytes; };

struct Batch {
    uint64_t n = 0; uint32_t max_len = 0; uint64_t total_bases = 0;
    DevBuf<uint8_t> seqs; DevBuf<uint64_t> offs; DevBuf<int64_t> ids;
    DevBuf<uint8_t> datums; DevBuf<uint64_t> datum_off, scan_tmp64;   // reads handed over as NUCLSEQ datum images (upload_datums)
    DevBuf<uint8_t> ascii;              // the reads as text (what to_text_palloc yields): the row materialisation reads query_subseq from it
    uint64_t res_serial = 0, res_read_base = 0, res_row_base = 0, res_cig_base = 0;   // the result (and the place in it) this batch's rows went to
    DevBuf<uint64_t> row_off64;        // the result's view of row_off: 64-bit, counted from the start of the whole result
    uint64_t cig_rebased = 0;          // what has been added to rows_compact[].cigar_off so far (reset when the rows are written again)
    TupleScratch tup;                  // row materialisation from the resident batch
    DevBuf<Intv> intv; DevBuf<uint32_t> intv_cnt; uint32_t intv_cap = 0;
    DevBuf<Intv> seed_scratch; uint32_t list_cap = 0;
    DevBuf<SeedRec> raw, seeds; DevBuf<ChainTmp> ctmp; DevBuf<uint32_t> ord; DevBuf<ChainRec> chains; DevBuf<uint64_t> srt;
    DevBuf<RegRec> regs; DevBuf<RowDev> rows; DevBuf<RowPub> rows_compact; DevBuf<RowExt> rows_ext; DevBuf<uint32_t> reg_cnt, row_cnt, row_off, scan_tmp;
    DevBuf<ReadBlock> blocks; uint32_t pool_cap = 0;
    DevBuf<uint32_t> cigar; uint32_t cigar_cap = 0;
    DevBuf<double> read_logtab; uint32_t read_logtab_n = 0; uint32_t rseq_cap = 0;
    DevBuf<uint8_t> ext_scratch, fin_scratch, narrow_z, narrow_jobs; DevBuf<uint64_t> wide_jobs;
    DevBuf<ExtMemo> ext_memo; DevBuf<uint8_t> ext_memo_key; DevBuf<uint32_t> ext_memo_perm, ext_memo_hist, ext_todo, chain_todo, fin_todo, seed_todo, seed_pk, seed_u32;   // thread-per-extension pre-pass (extend_plan.cu)
    DevBuf<uint64_t> sa_pos, sa_pos_off;   // compact index: the position resolve pass (sa_resolve.cu), pool_cap slots / n + 1 offsets
    DevBuf<uint32_t> ctl;  // [0..3] tickets, [4] overflow, [5] pool_top, [6] cigar_top, [8..23] counters (u64 x 8), [24] narrow_cnt, [25] wide_cnt, [26..27] tickets, [28..29] LF steps of the resolve pass (u64), [31] its ticket, [51] its error, [54..55] its warp iterations (u64), [56] reads left for sw_extend, [57] reads left for the warp chain kernel, [58] for regs_finalize
    // f(buf) for every DevBuf above: the one list release() frees and device_bytes() counts (BwaIndexCache's eviction budget)
    template <class B, class F> static void each(B& b, F f) {
        f(b.seqs); f(b.offs); f(b.ids); f(b.datums); f(b.datum_off); f(b.scan_tmp64); f(b.ascii); f(b.row_off64);
        f(b.tup.off); f(b.tup.tmp); f(b.tup.row_read); f(b.tup.nholes); f(b.tup.rm); f(b.tup.bytes);
        f(b.intv); f(b.intv_cnt); f(b.seed_scratch); f(b.raw); f(b.seeds); f(b.ctmp); f(b.ord); f(b.chains); f(b.srt);
        f(b.regs); f(b.rows); f(b.rows_compact); f(b.rows_ext); f(b.reg_cnt); f(b.row_cnt); f(b.row_off); f(b.scan_tmp); f(b.blocks); f(b.cigar);
        f(b.read_logtab); f(b.ext_scratch); f(b.fin_scratch); f(b.narrow_z); f(b.narrow_jobs); f(b.wide_jobs);
        f(b.ext_memo); f(b.ext_memo_key); f(b.ext_memo_perm); f(b.ext_memo_hist); f(b.ext_todo); f(b.chain_todo); f(b.fin_todo); f(b.seed_todo); f(b.seed_pk); f(b.seed_u32);
        f(b.sa_pos); f(b.sa_pos_off); f(b.ctl);
    }
    size_t device_bytes() const { size_t n = 0; each(*this, [&](const auto& d) { n += d.bytes(); }); return n; }
    bool resident = false, aligned = false;
    // one batch = one lane of the host pipeline: its stream, the host staging that must outlive the async copies,
    // and the state of the attempt in flight (pipeline_enqueue -> pipeline_check)
    cudaStream_t st = nullptr;
    std::vector<bsq_row_ext> ext_tmp;   // extension records fetched only to finish a MAPQ on the host
    uint32_t* ctl_host = nullptr;       // pinned, 16 words: ctl[0..7], total rows (2 words), host-MAPQ flag, error of the resolve pass
    cudaEvent_t ev[5]; bool ev_ok = false;
    cudaEvent_t ev_x[4]; bool evx_ok = false;   // chunked mode: upload begin/end, download begin/end
    ExtAux ext_aux; bool ext_aux_ok = false;    // side streams of the extension pre-pass
    uint32_t att_rseq_cap = 0; bool idle = true; bool att_compact = false;   // att_compact: the attempt in flight resolved positions (sa_resolve.cu)
    uint64_t out_rows = 0; uint32_t out_cig = 0;
    uint64_t rows_cap = 0;              // capacity of rows_compact (rows of the batch in read order)
    void release() {
        if (ctl_host) { cudaFreeHost(ctl_host); ctl_host = nullptr; }
        if (ev_ok) { for (auto& e : ev) cudaEventDestroy(e); ev_ok = false; }
        if (evx_ok) { for (auto& e : ev_x) cudaEventDestroy(e); evx_ok = false; }
        if (ext_aux_ok) { for (auto& s_ : ext_aux.st) cudaStreamDestroy(s_); for (auto& e : ext_aux.ev) cudaEventDestroy(e); ext_aux_ok = false; }
        each(*this, [](auto& d) { d.release(); });
    }
};

}  // namespace

struct bsq_index {
    int device = 0;
    bsq_opts opts; DevOpts dopts;
    float mapQ_coef_len = 50.f; int mapQ_coef_fac = 0;   // bwamem.h: `float mapQ_coef_len; int mapQ_coef_fac;`
    std::vector<uint8_t> pac; std::vector<int64_t> ann_offset, ann_id; std::vector<int32_t> ann_len; std::vector<bsq_hole> holes; std::vector<uint32_t> hole_ann;   // hole_ann: reference row of every hole
    uint8_t* d_pac = nullptr; uint32_t* d_occ = nullptr; void* d_sa = nullptr; int64_t* d_ann_offset = nullptr; int32_t* d_ann_len = nullptr; int64_t* d_ann_id = nullptr;
    bsq_index_meta meta;
    cudaStream_t stream = nullptr;
    Batch batch, batch2;             // batch2 + stream2: second lane of bsq_align_batch's chunk pipeline
    cudaStream_t stream2 = nullptr;
    bsq_timing timing;
    double* d_logtab = nullptr;
    void* d_isa = nullptr;           // inverse SA for the unique-match shortcut of the seeding kernel (built lazily, rows as wide as the SA's; never on a compact index)
    uint32_t* d_kmer_z = nullptr;    // sizes-only copy of the prefix table
    void* d_kmer = nullptr; int kmer_k = 0;          // k-mer table of the LAST-like seeding pass (built lazily per device index)
    bool collect_counters = false;
    int kmer_k_cap = 15;                   // lowered when the batch pools did not fit beside the table (kmer_downgrade)
    bool alloc_failed = false;             // the last pipeline_enqueue stopped on cudaErrorMemoryAllocation
    int test_pool_oom = getenv("BSQ_TEST_POOL_OOM") ? atoi(getenv("BSQ_TEST_POOL_OOM")) : 0;   // test hook: that many pool allocations "fail"
    int prio_hi = 0, prio_lo = 0;          // stream priorities of the two lanes of the chunked pipeline
    uint32_t flags = 0;              // BSQ_FLAG_*
    uint64_t lrand_state = 0;        // glibc lrand48 state of the session (one draw per aligned read when the caller passes no ids)
    bool replica_pending = false;    // device arrays allocated by bsq_index_alloc_replica, host mirrors not yet rebuilt (bsq_index_replica_finish)
    bsq_index_load_info last_load{};  // the last successful bsq_index_load
    uint64_t counters[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t* tup_host = nullptr;    // pinned, 4 words: byte total [0] and CIGAR span [1..2] of a staged row materialisation piece
};

static void fill_dev_opts(bsq_index* h) {
    const bsq_opts& p = h->opts; DevOpts& o = h->dopts;
    o.a = p.a; o.b = p.b; o.o_del = p.o_del; o.e_del = p.e_del; o.o_ins = p.o_ins; o.e_ins = p.e_ins;
    o.pen_clip5 = p.pen_clip5; o.pen_clip3 = p.pen_clip3; o.w = p.w; o.zdrop = p.zdrop; o.min_seed_len = p.min_seed_len; o.max_occ = p.max_occ;
    o.max_mem_intv = 20; o.split_width = 10;
    o.split_len = (int)(p.min_seed_len * 1.5f + .499);   // (int)(min_seed_len * split_factor + .499), split_factor is a float 1.5
    o.max_chain_gap = 10000; o.max_chain_extend = 1 << 30; o.min_chain_weight = 0;
    o.mask_level = 0.50f; o.drop_ratio = 0.50f; o.mask_level_redun = 0.95f;
    // bwa_fill_scmat(1, 4): filled once by mem_opt_init and never refreshed (SURVEY.md B#5).  This is the only matrix DevOpts ever
    // carries: the register and thread DP kernels (finalize.cu, ksw_thread.cuh) rely on its form -- one match, one mismatch and one
    // ambiguous-base score.
    for (int i = 0; i < 4; ++i) { for (int j = 0; j < 4; ++j) o.mat[i * 5 + j] = i == j ? 1 : -4; o.mat[i * 5 + 4] = -1; }
    for (int j = 0; j < 5; ++j) o.mat[20 + j] = -1;
    o.mat_max = 1;
    h->mapQ_coef_len = 50.f; h->mapQ_coef_fac = (int)log((double)h->mapQ_coef_len);   // mem_opt_init stores log(50) = 3.912 in an int field: 3
}

static int check_opts(const bsq_opts* o) {
    const int32_t* v = &o->min_seed_len;
    static const char* names[12] = {"min_seed_len", "max_occ", "match_score", "mismatch_penalty", "pen_clip3", "pen_clip5", "zdrop", "bandwidth", "o_del", "e_del", "o_ins", "e_ins"};
    for (int i = 0; i < 12; ++i) if (v[i] < 0) { bsq_set_error("bwa_opt %s must be nonnegative", names[i]); return BSQ_ERR; }   // extension.cpp:205-206
    if (o->e_del == 0 || o->e_ins == 0) { bsq_set_error("bwa_opt e_del / e_ins must be positive (libbwa divides by them)"); return BSQ_ERR; }
    if (o->max_occ == 0) { bsq_set_error("bwa_opt max_occ must be positive (libbwa divides by it)"); return BSQ_ERR; }
    return BSQ_OK;
}

namespace { DevIndex make_dev_index(const bsq_index* h); int ensure_kmer_table(bsq_index* h); }

// Test hook BSQ_TEST_COMPACT=1, read each time it could take effect: the allocation of the inverse SA and the allocation of the full SA
// by bsq_index_load "fail" as if device memory were short, so that tests reach the compact layout on references of any size.
static bool test_compact() { const char* v = getenv("BSQ_TEST_COMPACT"); return v && v[0] == '1' && v[1] == 0; }
// the meta of the compact layout of an index: every 32nd SA entry, as wide as the full SA's
static void compact_meta(bsq_index_meta& m) { m.sa_interval = 32; m.arr_bytes[BSQ_ARR_SA] = (m.seq_len + 32) / 32 * m.sa_bytes; }

extern "C" {

const char* bsq_last_error(void) { return g_err; }

int bsq_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

void bsq_opts_init(bsq_opts* o) {
    o->min_seed_len = 19; o->max_occ = 500; o->a = 1; o->b = 4; o->pen_clip3 = 5; o->pen_clip5 = 5; o->zdrop = 100; o->w = 100;
    o->o_del = 6; o->e_del = 1; o->o_ins = 6; o->e_ins = 1;
}

bsq_index* bsq_index_new(const bsq_opts* o, int device) {
    BSQ_ENTRY();
    bsq_opts d;
    if (!o) { bsq_opts_init(&d); o = &d; }
    if (check_opts(o) != BSQ_OK) return nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { bsq_set_error("no CUDA device: libbioseqdb_gpu has no CPU fallback"); return nullptr; }
    if (device < 0 || device >= n) { bsq_set_error("device %d out of range (%d devices)", device, n); return nullptr; }
    CUDA_CHECK_NULL(cudaSetDevice(device));
    bsq_index* h = new bsq_index;
    h->device = device; h->opts = *o;
    memset(&h->meta, 0, sizeof(h->meta)); memset(&h->timing, 0, sizeof(h->timing));
    fill_dev_opts(h);
    // The main stream (and lane 0 of the chunked pipeline) outranks lane 1: two chunks share the SMs, the earlier one gets free ones
    // first and is done -- its result on the way to the host -- while the later one still computes.
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    h->prio_hi = prio_hi; h->prio_lo = prio_lo;
    if (cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) { bsq_set_error("cudaStreamCreate failed"); delete h; return nullptr; }
    h->batch.st = h->stream;
    return h;
}

int bsq_index_set_opts(bsq_index* h, const bsq_opts* o) {
    BSQ_ENTRY();
    if (!h || !o) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (check_opts(o) != BSQ_OK) return BSQ_ERR;
    h->opts = *o; fill_dev_opts(h);
    return BSQ_OK;
}

int bsq_index_set_flags(bsq_index* h, uint32_t flags) {
    BSQ_ENTRY();
    if (!h) { bsq_set_error("null index"); return BSQ_ERR; }
    if (flags & ~(BSQ_FLAG_ROWS_EXT | BSQ_FLAG_TWO_CHUNKS)) { bsq_set_error("unknown flag bits %#x", flags & ~(BSQ_FLAG_ROWS_EXT | BSQ_FLAG_TWO_CHUNKS)); return BSQ_ERR; }
    h->flags = flags;
    return BSQ_OK;
}

// BwaIndex::add_ref_sequence (bwa.cpp:82-105): offset = 4 * bytes so far, byte-rounded append, holes not rebased.  The n_holes
// bsq_hole records at `holes` are read with memcpy: inside a datum they are only 4-byte aligned (SURVEY B#11).
static void append_ref(bsq_index* h, int64_t id, const uint8_t* pac, uint32_t len, const uint8_t* holes, uint32_t n_holes) {
    h->ann_offset.push_back((int64_t)h->pac.size() * 4);
    h->ann_len.push_back((int32_t)len);
    h->ann_id.push_back(id);
    h->pac.insert(h->pac.end(), pac, pac + ((size_t)len + 3) / 4);
    for (uint32_t k = 0; k < n_holes; ++k) {
        bsq_hole hl; memcpy(&hl, holes + (size_t)k * sizeof(bsq_hole), sizeof(bsq_hole));
        h->holes.push_back(hl); h->hole_ann.push_back((uint32_t)h->ann_offset.size() - 1);
    }
}

int bsq_index_add_ref(bsq_index* h, int64_t id, const uint8_t* pac, uint32_t len, const bsq_hole* holes, uint32_t n_holes) {
    BSQ_ENTRY();
    if (!h) { bsq_set_error("null index"); return BSQ_ERR; }
    if (h->meta.built) { bsq_set_error("index already built"); return BSQ_ERR; }
    append_ref(h, id, pac, len, reinterpret_cast<const uint8_t*>(holes), n_holes);
    return BSQ_OK;
}

// Batched form of bsq_index_add_ref: n NUCLSEQ datum images exactly as PostgreSQL hands them to iterate_nuclseq_table after
// detoasting (extension.cpp:157-195; layout sequence.h:18-38: varlena length word, holes_num, len, hole records, pac bytes),
// image i at bytes + off[i].  One call instead of one per reference row (500 k rows in BASELINE configs[4]).
int bsq_index_add_ref_datums(bsq_index* h, uint64_t n, const int64_t* ids, const uint8_t* bytes, const uint64_t* off) {
    BSQ_ENTRY();
    if (!h || (n && (!ids || !bytes || !off))) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (h->meta.built) { bsq_set_error("index already built"); return BSQ_ERR; }
    size_t pac_total = 0, holes_total = 0;
    for (uint64_t i = 0; i < n; ++i) {
        uint32_t hdr[3]; memcpy(hdr, bytes + off[i], 12);
        const uint64_t need = 12 + (uint64_t)hdr[1] * sizeof(bsq_hole) + ((uint64_t)hdr[2] + 3) / 4;
        if ((hdr[0] >> 2) < need) { bsq_set_error("datum %llu is truncated: varlena size %u, header needs %llu", (unsigned long long)i, hdr[0] >> 2, (unsigned long long)need); return BSQ_ERR; }
        pac_total += ((size_t)hdr[2] + 3) / 4; holes_total += hdr[1];
    }
    h->pac.reserve(h->pac.size() + pac_total); h->holes.reserve(h->holes.size() + holes_total); h->hole_ann.reserve(h->hole_ann.size() + holes_total);
    h->ann_offset.reserve(h->ann_offset.size() + n); h->ann_len.reserve(h->ann_len.size() + n); h->ann_id.reserve(h->ann_id.size() + n);
    for (uint64_t i = 0; i < n; ++i) {
        const uint8_t* d = bytes + off[i];
        uint32_t hdr[3]; memcpy(hdr, d, 12);
        append_ref(h, ids[i], d + 12 + (size_t)hdr[1] * sizeof(bsq_hole), hdr[2], d + 12, hdr[1]);
    }
    return BSQ_OK;
}

static void free_index_arrays(bsq_index* h) {
    if (h->d_kmer) { cudaFree(h->d_kmer); h->d_kmer = nullptr; }
    if (h->d_kmer_z) { cudaFree(h->d_kmer_z); h->d_kmer_z = nullptr; }
    if (h->d_isa) { cudaFree(h->d_isa); h->d_isa = nullptr; }
    if (h->d_pac) cudaFree(h->d_pac); if (h->d_occ) cudaFree(h->d_occ); if (h->d_sa) cudaFree(h->d_sa);
    if (h->d_ann_offset) cudaFree(h->d_ann_offset); if (h->d_ann_len) cudaFree(h->d_ann_len); if (h->d_ann_id) cudaFree(h->d_ann_id);
    h->d_pac = nullptr; h->d_occ = nullptr; h->d_sa = nullptr; h->d_ann_offset = nullptr; h->d_ann_len = nullptr; h->d_ann_id = nullptr;
}

static int upload_anns(bsq_index* h) {
    size_t na = h->ann_offset.size();
    CUDA_CHECK(cudaMalloc(&h->d_ann_offset, na * 8 + 8)); CUDA_CHECK(cudaMalloc(&h->d_ann_len, na * 4 + 8)); CUDA_CHECK(cudaMalloc(&h->d_ann_id, na * 8 + 8));
    CUDA_CHECK(cudaMemcpyAsync(h->d_ann_offset, h->ann_offset.data(), na * 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(h->d_ann_len, h->ann_len.data(), na * 4, cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(h->d_ann_id, h->ann_id.data(), na * 8, cudaMemcpyHostToDevice, h->stream));
    return BSQ_OK;
}

int bsq_index_build(bsq_index* h) {
    BSQ_ENTRY();
    if (!h) { bsq_set_error("null index"); return BSQ_ERR; }
    if (h->pac.empty()) return BSQ_OK;   // bwa.cpp:108-109: empty reference => no index, alignments return nothing
    CUDA_CHECK(cudaSetDevice(h->device));
    free_index_arrays(h);
    CUDA_CHECK(cudaMalloc(&h->d_pac, h->pac.size() + 64));
    CUDA_CHECK(cudaMemcpyAsync(h->d_pac, h->pac.data(), h->pac.size(), cudaMemcpyHostToDevice, h->stream));
    if (upload_anns(h) != BSQ_OK) return BSQ_ERR;
    IndexBuild B;
    B.d_pac = h->d_pac; B.l_pac = (int64_t)h->pac.size() * 4;
    { const char* fw = getenv("BSQ_FORCE_WIDE"); B.force_wide = fw && fw[0] == '1'; }   // test hook: 64-bit index path on small inputs
    if (build_index_device(B, h->stream) != BSQ_OK) return BSQ_ERR;
    h->d_occ = B.d_occ; h->d_sa = B.d_sa;
    bsq_index_meta& m = h->meta;
    m.l_pac = B.l_pac; m.seq_len = B.seq_len; m.primary = B.primary; memcpy(m.L2, B.L2, sizeof(m.L2));
    m.n_anns = h->ann_offset.size(); m.sa_bytes = (uint32_t)B.sa_bytes; m.built = 1; m.sa_interval = 1;
    m.arr_bytes[BSQ_ARR_PAC] = h->pac.size(); m.arr_bytes[BSQ_ARR_OCC] = B.occ_bytes; m.arr_bytes[BSQ_ARR_SA] = (B.seq_len + 1) * B.sa_bytes;
    m.arr_bytes[BSQ_ARR_ANN_OFFSET] = m.n_anns * 8; m.arr_bytes[BSQ_ARR_ANN_LEN] = m.n_anns * 4; m.arr_bytes[BSQ_ARR_ANN_ID] = m.n_anns * 8;
    m.build_ms = B.build_ms; m.build_launches = B.launches; m.sort_pass_bytes = B.sort_pass_bytes;
    return BSQ_OK;
}

void bsq_index_free(bsq_index* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    h->batch.release(); h->batch2.release();
    free_index_arrays(h);
    if (h->d_logtab) cudaFree(h->d_logtab);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->stream2) cudaStreamDestroy(h->stream2);
    if (h->tup_host) cudaFreeHost(h->tup_host);
    delete h;
}

int bsq_index_get_meta(const bsq_index* h, bsq_index_meta* m) {
    BSQ_ENTRY();
    if (!h || !m) { bsq_set_error("null argument"); return BSQ_ERR; }
    *m = h->meta;
    return BSQ_OK;
}

int bsq_index_device_bytes(const bsq_index* h, uint64_t* bytes) {
    BSQ_ENTRY();
    if (!h || !bytes) { bsq_set_error("null argument"); return BSQ_ERR; }
    uint64_t b = h->batch.device_bytes() + h->batch2.device_bytes();
    if (h->meta.built) {
        const uint64_t n = h->meta.seq_len;
        b += (h->meta.l_pac + 3) / 4 + ((n + 127) / 128 + 1) * 64 + h->meta.arr_bytes[BSQ_ARR_SA] + h->meta.n_anns * 20;
        if (h->d_isa) b += (n + 1) * (uint64_t)h->meta.sa_bytes + 64;
        if (h->d_kmer) b += kmer_table_bytes(h->kmer_k);
        if (h->d_kmer_z) b += kmer_table_bytes(h->kmer_k) / 4;
    }
    *bytes = b;
    return BSQ_OK;
}

static void* index_array(const bsq_index* h, int what) {
    switch (what) {
        case BSQ_ARR_PAC: return h->d_pac; case BSQ_ARR_OCC: return h->d_occ; case BSQ_ARR_SA: return h->d_sa;
        case BSQ_ARR_ANN_OFFSET: return h->d_ann_offset; case BSQ_ARR_ANN_LEN: return h->d_ann_len; case BSQ_ARR_ANN_ID: return h->d_ann_id;
        default: return nullptr;
    }
}

int bsq_index_device_ptr(const bsq_index* h, int what, void** dptr) {
    BSQ_ENTRY();
    if (!h || !dptr || what < 0 || what >= BSQ_ARR_COUNT) { bsq_set_error("bad argument"); return BSQ_ERR; }
    *dptr = index_array(h, what);
    return BSQ_OK;
}

int bsq_index_download(const bsq_index* h, int what, void* dst, uint64_t bytes) {
    BSQ_ENTRY();
    if (!h || !h->meta.built || what < 0 || what >= BSQ_ARR_COUNT) { bsq_set_error("index not built / bad array"); return BSQ_ERR; }
    if (bytes > h->meta.arr_bytes[what]) { bsq_set_error("download of %llu bytes exceeds array size %llu", (unsigned long long)bytes, (unsigned long long)h->meta.arr_bytes[what]); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    CUDA_CHECK(cudaMemcpy(dst, index_array(h, what), bytes, cudaMemcpyDeviceToHost));
    return BSQ_OK;
}

}  // extern "C"

// The arrays of an index described by *m, to be filled from elsewhere (a peer copy, a file); the handle answers once
// replica_finish has run.  may_compact: when the full SA does not fit, allocate the compact layout instead (h->meta says which).
static int alloc_replica(bsq_index* h, const bsq_index_meta* m, bool may_compact = false) {
    CUDA_CHECK(cudaSetDevice(h->device));
    free_index_arrays(h);
    h->meta = *m;
    h->replica_pending = true;
    CUDA_CHECK(cudaMalloc(&h->d_pac, m->arr_bytes[BSQ_ARR_PAC] + 64));
    CUDA_CHECK(cudaMalloc(&h->d_occ, m->arr_bytes[BSQ_ARR_OCC] + 64));
    cudaError_t e = may_compact && m->sa_interval == 1 && test_compact() ? cudaErrorMemoryAllocation : cudaMalloc(&h->d_sa, m->arr_bytes[BSQ_ARR_SA] + 64);
    if (e == cudaErrorMemoryAllocation && may_compact && m->sa_interval == 1) {
        cudaGetLastError(); h->d_sa = nullptr;
        compact_meta(h->meta);
        e = cudaMalloc(&h->d_sa, h->meta.arr_bytes[BSQ_ARR_SA] + 64);
    }
    CUDA_CHECK(e);
    CUDA_CHECK(cudaMalloc(&h->d_ann_offset, m->arr_bytes[BSQ_ARR_ANN_OFFSET] + 8));
    CUDA_CHECK(cudaMalloc(&h->d_ann_len, m->arr_bytes[BSQ_ARR_ANN_LEN] + 8));
    CUDA_CHECK(cudaMalloc(&h->d_ann_id, m->arr_bytes[BSQ_ARR_ANN_ID] + 8));
    return BSQ_OK;
}

// Host-side state that has no device copy: the ambiguity holes of the reference rows (copied un-rebased, bwa.cpp:98-104) and the
// row each one came from.  Blob = u64 n_holes | n_holes x bsq_hole | n_holes x u32 row.
static uint64_t host_state_bytes(uint64_t n_holes) { return 8 + n_holes * (sizeof(bsq_hole) + 4); }

static void host_state_encode(const bsq_index* h, uint8_t* p) {
    const uint64_t nh = h->holes.size();
    memcpy(p, &nh, 8);
    if (nh) { memcpy(p + 8, h->holes.data(), nh * sizeof(bsq_hole)); memcpy(p + 8 + nh * sizeof(bsq_hole), h->hole_ann.data(), nh * 4); }
}

static int host_state_decode(bsq_index* h, const uint8_t* p, uint64_t bytes) {
    uint64_t nh = 0;
    if (bytes < 8) { bsq_set_error("host-state blob truncated"); return BSQ_ERR; }
    memcpy(&nh, p, 8);
    if (bytes < host_state_bytes(nh)) { bsq_set_error("host-state blob truncated"); return BSQ_ERR; }
    h->holes.resize(nh); h->hole_ann.resize(nh);
    if (nh) { memcpy(h->holes.data(), p + 8, nh * sizeof(bsq_hole)); memcpy(h->hole_ann.data(), p + 8 + nh * sizeof(bsq_hole), nh * 4); }
    for (uint32_t a : h->hole_ann) if (a >= h->meta.n_anns) { bsq_set_error("host-state blob names a reference row the index does not have"); return BSQ_ERR; }
    return BSQ_OK;
}

// After the device arrays of a replica have been filled (broadcast / peer copy / file): rebuild the host mirrors the row
// materialisation and the host adapters read -- pac and the annotation vectors from the device copy, the holes from the
// source's host-state blob -- so that every replica answers exactly like the index it was copied from.
static int replica_finish(bsq_index* h, const void* host_state, uint64_t bytes) {
    CUDA_CHECK(cudaSetDevice(h->device));
    CUDA_CHECK(cudaDeviceSynchronize());
    const bsq_index_meta& m = h->meta;
    h->pac.resize(m.arr_bytes[BSQ_ARR_PAC]); h->ann_offset.resize(m.n_anns); h->ann_len.resize(m.n_anns); h->ann_id.resize(m.n_anns);
    if (!h->pac.empty()) CUDA_CHECK(cudaMemcpy(h->pac.data(), h->d_pac, h->pac.size(), cudaMemcpyDeviceToHost));
    if (m.n_anns) {
        CUDA_CHECK(cudaMemcpy(h->ann_offset.data(), h->d_ann_offset, m.n_anns * 8, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(h->ann_len.data(), h->d_ann_len, m.n_anns * 4, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(h->ann_id.data(), h->d_ann_id, m.n_anns * 8, cudaMemcpyDeviceToHost));
    }
    h->replica_pending = false;
    h->holes.clear(); h->hole_ann.clear();
    return host_state ? host_state_decode(h, static_cast<const uint8_t*>(host_state), bytes) : BSQ_OK;
}

// out[k] = sa[k * stride] for k < n_sa, out_bytes wide: the samples of a full SA (stride 32) or of a compact one (stride 1)
static __global__ void k_sa_sample(const void* sa, int sa_bytes, uint64_t stride, uint64_t n_sa, void* out, int out_bytes) {
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_sa; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t v = sa_bytes == 4 ? (uint64_t)static_cast<const uint32_t*>(sa)[k * stride] : static_cast<const uint64_t*>(sa)[k * stride];
        if (out_bytes == 4) static_cast<uint32_t*>(out)[k] = (uint32_t)v; else static_cast<uint64_t*>(out)[k] = v;
    }
}
// SA[0], SA[32], SA[64], ... of the index, whatever its layout, into out (out_bytes per entry), on h->stream
static void sa_samples_to(const bsq_index* h, void* out, int out_bytes) {
    const uint64_t n_sa = (h->meta.seq_len + 32) / 32;
    k_sa_sample<<<148 * 8, 256, 0, h->stream>>>(h->d_sa, (int)h->meta.sa_bytes, h->meta.sa_interval == 1 ? 32 : 1, n_sa, out, out_bytes);
}

// The compact layout (bsq_index_meta.sa_interval): the index keeps SA[0], SA[32], ... in an array of its SA width and frees the full SA
// and the inverse SA -- 16 bytes per base at 64 bits become a quarter of a byte.  Positions are then resolved by LF walks
// (sa_resolve.cu).  Taken only where the full layout cannot be allocated, and never undone.
static int compact_index(bsq_index* h) {
    bsq_index_meta m = h->meta;
    if (m.sa_interval != 1) return BSQ_OK;
    compact_meta(m);
    void* d = nullptr;
    CUDA_CHECK(cudaMalloc(&d, m.arr_bytes[BSQ_ARR_SA] + 64));
    sa_samples_to(h, d, (int)m.sa_bytes);
    const cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { cudaFree(d); bsq_set_error("compacting the index: %s", cudaGetErrorString(e)); return BSQ_ERR; }
    cudaFree(h->d_sa); h->d_sa = d;   // cudaFree waits for every kernel already queued on the device, so none loses the SA under it
    if (h->d_isa) { cudaFree(h->d_isa); h->d_isa = nullptr; }
    h->meta = m;
    h->timing.notes |= BSQ_NOTE_SA_COMPACTED;
    return BSQ_OK;
}

extern "C" {

int bsq_index_alloc_replica(bsq_index* h, const bsq_index_meta* m) {
    BSQ_ENTRY();
    if (!h || !m || !m->built) { bsq_set_error("bad argument"); return BSQ_ERR; }
    return alloc_replica(h, m);
}

int bsq_index_host_state_size(const bsq_index* h, uint64_t* bytes) {
    BSQ_ENTRY();
    if (!h || !bytes) { bsq_set_error("null argument"); return BSQ_ERR; }
    *bytes = host_state_bytes(h->holes.size());
    return BSQ_OK;
}

int bsq_index_host_state_get(const bsq_index* h, void* buf, uint64_t bytes) {
    BSQ_ENTRY();
    if (!h || !buf) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (bytes < host_state_bytes(h->holes.size())) { bsq_set_error("host-state buffer too small"); return BSQ_ERR; }
    host_state_encode(h, static_cast<uint8_t*>(buf));
    return BSQ_OK;
}

int bsq_index_replica_finish(bsq_index* h, const void* host_state, uint64_t bytes) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("replica not allocated"); return BSQ_ERR; }
    return replica_finish(h, host_state, bytes);
}

int bsq_index_bwt_plain(const bsq_index* h, uint32_t* out) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    std::vector<uint32_t> occ(h->meta.arr_bytes[BSQ_ARR_OCC] / 4);
    if (bsq_index_download(h, BSQ_ARR_OCC, occ.data(), h->meta.arr_bytes[BSQ_ARR_OCC]) != BSQ_OK) return BSQ_ERR;
    uint64_t nw = (h->meta.seq_len + 15) / 16;
    for (uint64_t i = 0; i < nw; ++i) out[i] = occ[(i >> 3 << 4) + 8 + (i & 7)];
    return BSQ_OK;
}

int bsq_index_sa_sampled(const bsq_index* h, uint64_t* out, uint64_t n_sa) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    uint64_t n = h->meta.seq_len;
    if (n_sa != (n + 32) / 32) { bsq_set_error("n_sa must be (seq_len + 32) / 32"); return BSQ_ERR; }
    // rows 0, 32, 64, ... of the SA, gathered on the device (the full array is 50 GB at 3.1 Gbp)
    CUDA_CHECK(cudaSetDevice(h->device));
    DevBuf<uint64_t> d;
    CUDA_CHECK(d.alloc(n_sa));
    sa_samples_to(h, d.p, 8);
    CUDA_CHECK_AS("bsq_index_sa_sampled", cudaMemcpyAsync(out, d.p, n_sa * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK_AS("bsq_index_sa_sampled", cudaStreamSynchronize(h->stream));
    out[0] = (uint64_t)-1;   // bwt_cal_sa: sa[0] = -1 (SURVEY A.3)
    return BSQ_OK;
}

// Builds the arrays the seeding kernel derives from the index on this device (inverse SA, prefix table) now rather than inside
// the first alignment call; *ms = wall time spent (0 when they were already there).  Every replica calls it after the broadcast.
// When the inverse SA does not fit, the index compacts itself first (BSQ_NOTE_SA_COMPACTED in bsq_last_timing's notes).
int bsq_index_prepare(bsq_index* h, float* ms) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    Event e0, e1; cudaEventCreate(&e0.h); cudaEventCreate(&e1.h);
    cudaEventRecord(e0, h->stream);
    const int rc = ensure_kmer_table(h);
    cudaEventRecord(e1, h->stream);
    cudaEventSynchronize(e1);
    if (ms) cudaEventElapsedTime(ms, e0, e1);
    return rc;
}

// Index files (layout and kernels: index_file.cu).  A loaded index is one more replica: allocated and finished by the same code as a
// broadcast's, its arrays filled from the file instead of a peer.
int bsq_index_save(bsq_index* h, const char* path, const uint8_t* key) {
    BSQ_ENTRY();
    if (!h || !path) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (!h->meta.built) { bsq_set_error("bsq_index_save: the index is not built (an empty reference builds nothing)"); return BSQ_ERR; }
    if (h->replica_pending) { bsq_set_error("bsq_index_save: replica without host state"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    std::vector<uint8_t> hs(host_state_bytes(h->holes.size()));
    host_state_encode(h, hs.data());
    const uint64_t n_sa = (h->meta.seq_len + 32) / 32;
    DevBuf<uint64_t> d_samples;
    CUDA_CHECK(d_samples.alloc(n_sa));
    sa_samples_to(h, d_samples.p, 8);   // sample 0 = SA[0] = seq_len
    const IndexFileArrays a{h->d_pac, h->d_occ, h->d_sa, h->d_ann_offset, h->d_ann_len, h->d_ann_id};
    return index_file_save(path, h->meta, a, d_samples.p, h->pac.data(), h->ann_offset.data(), h->ann_len.data(), h->ann_id.data(), hs, key, h->stream);
}

int bsq_index_load(bsq_index* h, const char* path, const uint8_t* key, float* ms) {
    BSQ_ENTRY();
    const auto t0 = std::chrono::steady_clock::now();
    if (!h || !path) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (h->meta.built || !h->ann_offset.empty()) { bsq_set_error("bsq_index_load: the handle already has reference rows or an index (load needs a fresh handle)"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    IndexFileReader r;
    bsq_index_meta m;
    bsq_index_load_info info;
    memset(&info, 0, sizeof(info));
    std::vector<uint8_t> hs;
    int rc = index_file_open(r, path, key, &m);
    if (rc == BSQ_OK) rc = alloc_replica(h, &m, true);   // the compact layout when the full SA does not fit
    if (rc == BSQ_OK) {
        const IndexFileArrays a{h->d_pac, h->d_occ, h->d_sa, h->d_ann_offset, h->d_ann_len, h->d_ann_id};
        rc = index_file_fill(r, a, h->meta.sa_interval != 1, hs, h->device, h->stream, &info);
    }
    info.file_bytes = r.file_bytes;
    index_file_close(r);
    if (rc == BSQ_OK) {
        const auto t1 = std::chrono::steady_clock::now();
        rc = replica_finish(h, hs.data(), hs.size());
        info.host_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t1).count();
    }
    if (rc != BSQ_OK) {   // leave the handle as fresh as it came
        cudaStreamSynchronize(h->stream);
        free_index_arrays(h);
        memset(&h->meta, 0, sizeof(h->meta));
        h->replica_pending = false;
        h->pac.clear(); h->ann_offset.clear(); h->ann_len.clear(); h->ann_id.clear(); h->holes.clear(); h->hole_ann.clear();
        return BSQ_ERR;
    }
    info.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    h->last_load = info;
    if (ms) *ms = info.total_ms;
    return BSQ_OK;
}

int bsq_index_last_load(const bsq_index* h, bsq_index_load_info* out) {
    BSQ_ENTRY();
    if (!h || !out) { bsq_set_error("null argument"); return BSQ_ERR; }
    *out = h->last_load;
    return BSQ_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ batch
namespace {

// the glibc lrand48 state k draws after state x: x_k = A^k x + C (A^k - 1) / (A - 1) mod 2^48 by square-and-multiply on the affine map
__host__ __device__ uint64_t lrand48_advance(uint64_t x, uint64_t k) {
    const uint64_t M = (1ull << 48) - 1;
    uint64_t A = 1, C = 0, ba = 0x5DEECE66DULL, bc = 0xBULL;
    while (k) {
        if (k & 1) { A = (A * ba) & M; C = (C * ba + bc) & M; }
        bc = (bc * ba + bc) & M; ba = (ba * ba) & M;
        k >>= 1;
    }
    return (A * x + C) & M;
}
// ids[i] = the (first + i + 1)-th value glibc lrand48() returns from state x0 (mem_align1 draws one per read, SURVEY A.10): x_k >> 17
__global__ void k_lrand48_ids(uint64_t x0, uint64_t first, uint64_t n, int64_t* ids) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        ids[i] = (int64_t)(lrand48_advance(x0, first + i + 1) >> 17);
}

// NUCLSEQ datum images -> what mem_align1 sees after to_text_palloc + nst_nt4_table (bwa.cpp:146-149): codes 0..3 from the packed
// bases, 4 wherever a hole (an ambiguous letter) covers the base.  Pass 1: lengths; pass 2 (after the scan): one warp per read.
// stats[0] = longest read, stats[1] = index + 1 of a truncated / oversized image (0 = all fine)
__global__ void k_datum_lens(const uint8_t* bytes, const uint64_t* doff, uint64_t base, uint64_t n, uint64_t* lens, uint32_t* stats) {
    uint32_t mx = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t* d = bytes + (doff[i] - base);
        uint32_t hdr[3]; memcpy(hdr, d, 12);
        const uint64_t need = 12 + (uint64_t)hdr[1] * 16 + ((uint64_t)hdr[2] + 3) / 4;
        if ((hdr[0] >> 2) < need || doff[i + 1] < doff[i] + need || hdr[2] > 0x3fffffffu) { atomicMax(stats + 1, (uint32_t)(i + 1)); hdr[2] = 0; }
        lens[i] = hdr[2];
        mx = mx > hdr[2] ? mx : hdr[2];
    }
    mx = __reduce_max_sync(FULL, mx);
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(stats, mx);
    if (blockIdx.x == 0 && threadIdx.x == 0) lens[n] = 0;
}
__global__ void k_datum_unpack(const uint8_t* bytes, const uint64_t* doff, uint64_t base, uint64_t n, const uint64_t* offs, uint8_t* seqs, uint8_t* ascii) {
    const uint64_t gw = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = gw; r < n; r += nw) {
        const uint8_t* d = bytes + (doff[r] - base);
        uint32_t n_holes, len; memcpy(&n_holes, d + 4, 4); memcpy(&len, d + 8, 4);
        const uint8_t* pac = d + 12 + (size_t)n_holes * 16;
        uint8_t* q = seqs + offs[r]; uint8_t* a = ascii + offs[r];
        for (uint32_t i = lane; i < len; i += 32) { const uint32_t c = (pac[i >> 2] >> ((~i & 3u) << 1)) & 3u; q[i] = (uint8_t)c; a[i] = (uint8_t)"ACGT"[c]; }
        __syncwarp();
        for (uint32_t k = 0; k < n_holes; ++k) {   // inplace_to_text (sequence.cpp:71-81): holes in order, later ones overwrite
            int64_t ho; int32_t hl; memcpy(&ho, d + 12 + (size_t)k * 16, 8); memcpy(&hl, d + 12 + (size_t)k * 16 + 8, 4);
            const uint8_t amb = d[12 + (size_t)k * 16 + 12];
            for (int64_t i = ho + lane; i < ho + hl && i < (int64_t)len; i += 32) if (i >= 0) { q[i] = 4; a[i] = amb; }
            __syncwarp();
        }
    }
}

__global__ void k_rebase_offs(uint64_t* offs, uint64_t n, uint64_t base) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) offs[i] -= base;
}

__global__ void k_to_nt4(uint8_t* s, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint8_t c = s[i], v;
        // mem_align1_core: seq[i] < 4 ? seq[i] : nst_nt4_table[seq[i]]
        if (c < 4) v = c;
        else switch (c) {
            case 'A': case 'a': v = 0; break; case 'C': case 'c': v = 1; break; case 'G': case 'g': v = 2; break; case 'T': case 't': v = 3; break;
            case '-': v = 5; break; default: v = 4;
        }
        s[i] = v;
    }
}

// mem_approx_mapq_se (SURVEY A.12) on the device.  The only transcendental is log() of small integers
// (alignment length l and sub_n + 1): both come from a table filled by the HOST libm, so every double
// operation here is an IEEE +,-,*,/ evaluated in the reference's order (the library is compiled with
// --fmad=false).  Rows whose l or sub_n fall outside the table get mapq = -1 and are finished on the host.
constexpr int LOGTAB_N = 65536;   // alignments of up to 65535 bases get their MAPQ on the device
struct MapqParams { int a, b, min_seed_len; float coef_len; double coef_fac; const double* logtab; };

__device__ __forceinline__ int approx_mapq_dev(const MapqParams& M, const RowDev& r) {
    int mapq, l, sub = r.sub ? r.sub : M.min_seed_len * M.a;
    sub = r.csub > sub ? r.csub : sub;
    if (sub >= r.score) return 0;
    l = r.qe - r.qb > r.re - r.rb ? r.qe - r.qb : (int)(r.re - r.rb);
    if (l >= LOGTAB_N || r.sub_n + 1 >= LOGTAB_N || l <= 0) return -1;
    const double identity = 1. - (double)(l * M.a - r.score) / (M.a + M.b) / l;
    if (r.score == 0) mapq = 0;
    else {
        double tmp = l < M.coef_len ? 1. : M.coef_fac / M.logtab[l];
        tmp *= identity * identity;
        mapq = (int)(6.02 * (r.score - sub) / M.a * tmp * tmp + .499);
    }
    if (r.sub_n > 0) mapq -= (int)(4.343 * M.logtab[r.sub_n + 1] + .499);
    if (mapq > 60) mapq = 60;
    if (mapq < 0) mapq = 0;
    mapq = (int)(mapq * (1. - r.frac_rep) + .499);
    return mapq;
}

constexpr int MAPQ_HOST = 255;   // mapq value of a row whose MAPQ the host finishes (l or sub_n outside the device log table)
__global__ void k_compact_rows(const ReadBlock* blocks, const RowDev* rows, const uint32_t* row_cnt, const uint32_t* row_off, uint32_t n_reads,
                               RowPub* out, RowExt* ext, uint32_t out_cap, MapqParams M, uint32_t* host_mapq) {
    // thread per row slot of a read: the 120-byte working record becomes the 64-byte public row (+ the 48-byte extension when asked
    // for).  *host_mapq is raised when a row's MAPQ has to be finished on the host.  Rows beyond out_cap are dropped: the host sees
    // the total from the scan, grows the buffer and runs the batch again.
    // thread per read (a read has one row, rarely a handful)
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += gridDim.x * blockDim.x) {
        const uint32_t c = row_cnt[r];
        if (!c || row_off[r] + c > out_cap) continue;
        const RowDev* srow = rows + blocks[r].base;
        for (uint32_t k = 0; k < c; ++k) {
            const RowDev a = srow[k];
            const int mq = a.secondary < 0 ? approx_mapq_dev(M, a) : 0;
            if (mq < 0) atomicExch(host_mapq, 1u);
            RowPub d;
            d.rb = a.rb; d.re = a.re; d.pos = a.pos; d.ref_id = a.ref_id; d.qb = a.qb; d.qe = a.qe; d.rid = a.rid; d.score = a.score; d.NM = a.NM;
            d.cigar_off = a.cigar_off; d.n_cigar = a.n_cigar; d.flag = (uint16_t)a.flag; d.mapq = (uint8_t)(mq < 0 ? MAPQ_HOST : mq); d.is_rev = (uint8_t)a.is_rev;
            out[row_off[r] + k] = d;
            if (ext) {
                RowExt e;
                e.hash = a.hash; e.truesc = a.truesc; e.sub = a.sub; e.csub = a.csub; e.sub_n = a.sub_n; e.w = a.w; e.seedcov = a.seedcov;
                e.secondary = a.secondary; e.seedlen0 = a.seedlen0; e.n_comp = a.n_comp; e.frac_rep = a.frac_rep;
                ext[row_off[r] + k] = e;
            }
        }
    }
}

DevIndex make_dev_index(const bsq_index* h) {
    DevIndex ix;
    ix.pac = h->d_pac; ix.occ = h->d_occ; ix.sa = h->d_sa; ix.ann_offset = h->d_ann_offset; ix.ann_len = h->d_ann_len;
    ix.l_pac = h->meta.l_pac; ix.seq_len = h->meta.seq_len; ix.primary = h->meta.primary;
    for (int i = 0; i < 5; ++i) ix.L2[i] = h->meta.L2[i];
    ix.n_anns = (int)h->meta.n_anns; ix.sa_bytes = (int)h->meta.sa_bytes;
    return ix;
}

uint32_t rseq_cap_for(const bsq_index* h, uint32_t max_len) { return max_len + 4u * (uint32_t)h->opts.w + 16u; }

// reads longer than this would need mem_flt_chained_seeds' local SW (SURVEY A.6: runs when 5.5 ln L <= 0.05 L)
bool needs_seed_sw(uint32_t len) { return len > 0 && 5.5f * log((double)len) <= 0.05f * (double)len; }

// log(l_query) for mem_flt_chained_seeds' thresholds, for reads of up to max_len bases: host libm values (SURVEY A.6, A.14)
int ensure_read_logtab(Batch& b, uint32_t max_len) {
    if (!needs_seed_sw(max_len) || b.read_logtab_n >= max_len + 1) return BSQ_OK;
    std::vector<double> tab(max_len + 1);
    tab[0] = 0.;
    for (uint32_t i = 1; i <= max_len; ++i) tab[i] = log((double)i);
    CUDA_CHECK(b.read_logtab.ensure(max_len + 1));
    CUDA_CHECK(cudaMemcpy(b.read_logtab.p, tab.data(), (max_len + 1) * sizeof(double), cudaMemcpyHostToDevice));
    b.read_logtab_n = max_len + 1;
    return BSQ_OK;
}

int upload_reads(bsq_index* h, Batch& b, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n, uint64_t id_first = 0) {
    b.resident = false; b.aligned = false; b.res_serial = 0;
    if (n >= 0x7fffffffull) { bsq_set_error("batch too large"); return BSQ_ERR; }
    uint32_t max_len = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (offs[i + 1] < offs[i]) { bsq_set_error("read offsets must be non-decreasing"); return BSQ_ERR; }
        uint64_t l = offs[i + 1] - offs[i];
        if (l > 0x3fffffffull) { bsq_set_error("read too long"); return BSQ_ERR; }
        max_len = std::max<uint32_t>(max_len, (uint32_t)l);
    }
    const uint64_t total = n ? offs[n] - offs[0] : 0;
    b.n = n; b.max_len = max_len; b.total_bases = total;
    if (ensure_read_logtab(b, max_len) != BSQ_OK) return BSQ_ERR;
    CUDA_CHECK(b.seqs.ensure(total + 64)); CUDA_CHECK(b.offs.ensure(n + 1)); CUDA_CHECK(b.ids.ensure(n + 1));
    // the caller's buffers go to the device as they are (pinned buffers make these copies truly asynchronous; pageable ones are staged
    // by the runtime); the offsets are rebased to the batch's first read on the device
    if (total) CUDA_CHECK(cudaMemcpyAsync(b.seqs.p, seqs + offs[0], total, cudaMemcpyHostToDevice, b.st));
    if (n) {
        CUDA_CHECK(cudaMemcpyAsync(b.offs.p, offs, (n + 1) * 8, cudaMemcpyHostToDevice, b.st));
        if (ids) CUDA_CHECK(cudaMemcpyAsync(b.ids.p, ids, n * 8, cudaMemcpyHostToDevice, b.st));
        else { k_lrand48_ids<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 148 * 8), 256, 0, b.st>>>(h->lrand_state, id_first, n, b.ids.p); ++h->timing.launches; }
    } else CUDA_CHECK(cudaMemsetAsync(b.offs.p, 0, 8, b.st));
    if (total) {
        CUDA_CHECK(b.ascii.ensure(total + 64));
        CUDA_CHECK(cudaMemcpyAsync(b.ascii.p, b.seqs.p, total, cudaMemcpyDeviceToDevice, b.st));   // the text stays for the row materialisation
        k_to_nt4<<<(unsigned)std::min<uint64_t>((total + 255) / 256, 148 * 16), 256, 0, b.st>>>(b.seqs.p, total); ++h->timing.launches;
    }
    if (n && offs[0]) { k_rebase_offs<<<(unsigned)std::min<uint64_t>((n + 256) / 256, 148 * 8), 256, 0, b.st>>>(b.offs.p, n + 1, offs[0]); ++h->timing.launches; }
    h->timing.h2d_bytes += total + (n + 1) * 8 + (ids ? n * 8 : 0);
    b.resident = true;
    return BSQ_OK;
}

// The same batch handed over as NUCLSEQ datum images (image i at bytes + doff[i], as PostgreSQL stores the query rows): 2 bits per
// base on the wire instead of 8.  The host reads the headers once (longest read, total bases: the pools are sized from them); the
// images are unpacked on the device.
int upload_datums_begin(bsq_index* h, Batch& b, const uint8_t* bytes, const uint64_t* doff, const int64_t* ids, uint64_t n, uint64_t id_first) {
    b.resident = false; b.aligned = false; b.res_serial = 0;
    if (n >= 0x7fffffffull) { bsq_set_error("batch too large"); return BSQ_ERR; }
    if (n && doff[n] < doff[0]) { bsq_set_error("datum offsets must be non-decreasing"); return BSQ_ERR; }
    const uint64_t nbytes = n ? doff[n] - doff[0] : 0;
    b.n = n; b.max_len = 0; b.total_bases = 0;
    CUDA_CHECK(b.offs.ensure(n + 2)); CUDA_CHECK(b.ids.ensure(n + 1)); CUDA_CHECK(b.ctl.ensure(64));
    CUDA_CHECK(b.datums.ensure(nbytes + 64)); CUDA_CHECK(b.datum_off.ensure(n + 1)); CUDA_CHECK(b.scan_tmp64.ensure(prim::scan_tmp_elems(n + 1) + 16));
    if (!b.ctl_host) CUDA_CHECK(cudaHostAlloc(&b.ctl_host, 16 * 4, cudaHostAllocDefault));
    if (n) {
        // images, their offsets and the ids go down as they are; the headers are read ON THE DEVICE (longest read, total bases, validity:
        // four bytes come back) -- walking a million headers in host memory costs more than the whole copy
        CUDA_CHECK(cudaMemcpyAsync(b.datums.p, bytes + doff[0], nbytes, cudaMemcpyHostToDevice, b.st));
        CUDA_CHECK(cudaMemcpyAsync(b.datum_off.p, doff, (n + 1) * 8, cudaMemcpyHostToDevice, b.st));
        if (ids) CUDA_CHECK(cudaMemcpyAsync(b.ids.p, ids, n * 8, cudaMemcpyHostToDevice, b.st));
        else { k_lrand48_ids<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 148 * 8), 256, 0, b.st>>>(h->lrand_state, id_first, n, b.ids.p); ++h->timing.launches; }
        CUDA_CHECK(cudaMemsetAsync(b.ctl.p + 61, 0, 8, b.st));
        k_datum_lens<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 148 * 8), 256, 0, b.st>>>(b.datums.p, b.datum_off.p, doff[0], n, b.offs.p, b.ctl.p + 61); ++h->timing.launches;
        prim::device_scan<uint64_t, prim::OpSum, false>(b.offs.p, b.offs.p, n + 1, b.scan_tmp64.p, prim::OpSum(), b.st, &h->timing.launches);
        CUDA_CHECK(cudaMemcpyAsync(b.ctl_host + 12, b.ctl.p + 61, 8, cudaMemcpyDeviceToHost, b.st));
        CUDA_CHECK(cudaMemcpyAsync(b.ctl_host + 14, b.offs.p + n, 8, cudaMemcpyDeviceToHost, b.st));
    } else CUDA_CHECK(cudaMemsetAsync(b.offs.p, 0, 8, b.st));
    h->timing.h2d_bytes += nbytes + (n + 1) * 8 + (ids ? n * 8 : 0);
    return BSQ_OK;
}
// second half: waits for the header pass, sizes the text buffers, unpacks the images
int upload_datums_end(bsq_index* h, Batch& b, uint64_t doff0) {
    const uint64_t n = b.n;
    uint64_t total = 0; uint32_t max_len = 0;
    if (n) {
        CUDA_CHECK(cudaStreamSynchronize(b.st));
        if (b.ctl_host[13]) { bsq_set_error("datum %u is truncated or longer than a read may be", b.ctl_host[13] - 1); return BSQ_ERR; }
        max_len = b.ctl_host[12]; memcpy(&total, b.ctl_host + 14, 8);
    }
    b.max_len = max_len; b.total_bases = total;
    if (ensure_read_logtab(b, max_len) != BSQ_OK) return BSQ_ERR;
    CUDA_CHECK(b.seqs.ensure(total + 64)); CUDA_CHECK(b.ascii.ensure(total + 64));
    if (n) { k_datum_unpack<<<(unsigned)std::min<uint64_t>((n + 7) / 8, 148 * 16), 256, 0, b.st>>>(b.datums.p, b.datum_off.p, doff0, n, b.offs.p, b.seqs.p, b.ascii.p); ++h->timing.launches; }
    b.resident = true;
    return BSQ_OK;
}
int upload_datums(bsq_index* h, Batch& b, const uint8_t* bytes, const uint64_t* doff, const int64_t* ids, uint64_t n, uint64_t id_first = 0) {
    if (upload_datums_begin(h, b, bytes, doff, ids, n, id_first) != BSQ_OK) return BSQ_ERR;
    return upload_datums_end(h, b, n ? doff[0] : 0);
}

// k-mer table of the LAST-like seeding pass: built once per device index (also after a broadcast replica).  The inverse SA beside it
// is built only in the full layout; when it cannot be allocated, the index compacts itself and seeds without it.
int ensure_kmer_table(bsq_index* h) {
    DevIndex ix = make_dev_index(h);
    if (ix.seq_len >= (1ull << 40)) return BSQ_OK;   // the table packs rows in 40 bits
    if (!h->d_isa && h->meta.sa_interval == 1) {
        const cudaError_t e = test_compact() ? cudaErrorMemoryAllocation : cudaMalloc(&h->d_isa, (ix.seq_len + 1) * (uint64_t)ix.sa_bytes + 64);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError(); h->d_isa = nullptr;
            if (compact_index(h) != BSQ_OK) return BSQ_ERR;
            ix = make_dev_index(h);
        } else {
            CUDA_CHECK(e);
            build_isa(ix, h->d_isa, h->stream, &h->timing.launches);
            CUDA_CHECK(cudaStreamSynchronize(h->stream));
        }
    }
    if (h->d_kmer || ix.seq_len < (1u << 16)) return BSQ_OK;
    h->kmer_k = kmer_table_depth(ix.seq_len);
    // One level more than ceil(log4 n) where HBM allows it (23 GB at K = 15): a K-mer of the read's own locus then has a second,
    // chance occurrence three times less often, and every such occurrence costs the seeding kernels real bwt_extend steps
    // (measured at 200 M symbols: 13.6 -> 12.3 ms per 1 M reads).  Only for 32-bit indexes; the 64-bit ones keep their HBM for SA + ISA.
    if (h->kmer_k == 14 && ix.seq_len > (1ull << 27)) {
        size_t fr = 0, tot = 0;
        const size_t want = kmer_table_bytes(15) + kmer_table_bytes(15) / 4;     // entries + the size table
        // 32-bit indexes: when the table is a quarter of what is free.  64-bit ones (SA + ISA already hold 16 bytes per symbol): when 40 GB
        // stay free for the batch pools of two lanes (c3: 77 GB free -> 28.6 GB table; measured 28.5 -> 25.9 ms seeding per 1.25 M reads).
        // If the pools do not fit after all, the pipeline drops a level and goes on (kmer_downgrade).
        if (cudaMemGetInfo(&fr, &tot) == cudaSuccess && (ix.sa_bytes == 4 ? fr > 4 * kmer_table_bytes(15) : fr > want + (40ull << 30))) h->kmer_k = 15;
    }
    if (h->kmer_k > h->kmer_k_cap) h->kmer_k = h->kmer_k_cap;
    CUDA_CHECK(cudaMalloc(&h->d_kmer, kmer_table_bytes(h->kmer_k)));
    build_kmer_table(ix, h->d_kmer, h->kmer_k, h->stream, &h->timing.launches);
    if (cudaMalloc(&h->d_kmer_z, kmer_table_bytes(h->kmer_k) / 4) == cudaSuccess) build_kmer_sizes(h->d_kmer, h->d_kmer_z, h->kmer_k, h->stream, &h->timing.launches);
    else { h->d_kmer_z = nullptr; cudaGetLastError(); }
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    return BSQ_OK;
}

// Device memory ran out while sizing a batch's pools: give back the deepest level of the prefix table (three quarters of it) and let
// ensure_kmer_table rebuild the shallower one.  cudaFree waits for everything already queued, so no kernel loses the table under it.
bool kmer_downgrade(bsq_index* h) {
    if (!h->d_kmer || h->kmer_k <= 8) return false;
    cudaFree(h->d_kmer); h->d_kmer = nullptr;
    if (h->d_kmer_z) { cudaFree(h->d_kmer_z); h->d_kmer_z = nullptr; }
    h->kmer_k_cap = h->kmer_k - 1;
    cudaGetLastError();
    return true;
}

// the seeding kernel's view of a batch: inputs, per-read interval slots, the index's derived arrays, control words
SeedParams seed_params(const bsq_index* h, const Batch& b, const DevIndex& ix, uint32_t n, uint32_t cap, uint32_t* ticket, unsigned long long* n_extend) {
    SeedParams P;
    P.seqs = b.seqs.p; P.offs = b.offs.p; P.n_reads = n; P.out = b.intv.p; P.out_cnt = b.intv_cnt.p; P.cap = cap;
    P.kmer_tab = reinterpret_cast<const uint4*>(h->d_kmer); P.kmer_k = h->kmer_k; P.kmer_ztab = h->d_kmer_z; P.isa = h->d_isa;
    P.scratch = b.seed_scratch.p; P.list_cap = b.list_cap;
    // shared-memory bytes per warp for the read: the bases (padded to 16) and their 2-bit packed copy
    P.read_cap = ((b.max_len + 16) & ~15u) + (((b.max_len >> 4) + 3) << 2) + 16 & ~15u;
    P.lists_in_smem = seed_lists_fit_smem(b.list_cap, P.read_cap, ix.sa_bytes);
    P.ticket = ticket; P.overflow = b.ctl.p + 4; P.n_extend = n_extend;
    P.todo = b.seed_todo.p; P.todo_cnt = b.ctl.p + 59;    // reads the thread-per-read passes leave for seed_smem
    P.pk = b.seed_pk.p; P.rflag = b.seed_u32.p; P.cnt12 = b.seed_u32.p ? b.seed_u32.p + n : nullptr; P.ext12 = b.seed_u32.p ? b.seed_u32.p + 2 * (size_t)n : nullptr;
    return P;
}

// One attempt of the kernel pipeline on the batch's stream: size the pools, launch every stage, read the control
// words back asynchronously.  Nothing here waits for the device.
static int pipeline_enqueue_once(bsq_index* h, Batch& b);
int pipeline_enqueue(bsq_index* h, Batch& b) {
    h->alloc_failed = false;
    int rc = pipeline_enqueue_once(h, b);
    for (int tries = 0; rc != BSQ_OK && h->alloc_failed && tries < 2 && kmer_downgrade(h); ++tries) {
        h->alloc_failed = false;
        h->timing.notes |= BSQ_NOTE_TABLE_DOWNGRADED;
        rc = pipeline_enqueue_once(h, b);
        if (rc == BSQ_OK) bsq_set_error("");
    }
    // the last rung: the full SA and the inverse SA give way to the compact layout (at 64 bits, 16 bytes per base)
    if (rc != BSQ_OK && h->alloc_failed && h->meta.sa_interval == 1) {
        if (compact_index(h) != BSQ_OK) return BSQ_ERR;
        h->alloc_failed = false;
        rc = pipeline_enqueue_once(h, b);
        if (rc == BSQ_OK) bsq_set_error("");
    }
    return rc;
}
static int pipeline_enqueue_once(bsq_index* h, Batch& b) {
    if (!b.resident) { bsq_set_error("no reads uploaded"); return BSQ_ERR; }
    const uint32_t n = (uint32_t)b.n;
    bsq_timing& T = h->timing;
    b.idle = true; b.out_rows = 0; b.out_cig = 0;
    if (n == 0 || !h->meta.built) { b.aligned = true; return BSQ_OK; }
    if (ensure_kmer_table(h) != BSQ_OK) return BSQ_ERR;
    const DevIndex ix = make_dev_index(h);
    const DevOpts& o = h->dopts;
    cudaStream_t st = b.st;
    const bool compact = b.att_compact = h->meta.sa_interval != 1;
    const uint32_t max_len = std::max<uint32_t>(b.max_len, 1);
    const uint32_t rseq_cap = b.att_rseq_cap = std::max(rseq_cap_for(h, max_len), b.rseq_cap);
    if (b.intv_cap == 0) b.intv_cap = 48 + max_len / 4;
    b.pool_cap = std::max<uint32_t>(b.pool_cap, (uint32_t)std::min<uint64_t>((uint64_t)n * 24 + 4096, 0x7fffffffull));
    b.cigar_cap = std::max<uint32_t>(b.cigar_cap, (uint32_t)std::min<uint64_t>((uint64_t)n * 8 + 4096, 0x7fffffffull));
    if (!b.ev_ok) { for (auto& e : b.ev) cudaEventCreate(&e); b.ev_ok = true; }
    if (!b.ctl_host) CUDA_CHECK(cudaHostAlloc(&b.ctl_host, 16 * 4, cudaHostAllocDefault));
    cudaEvent_t* ev = b.ev;
    // ---- (re)size pools
    const int seed_warps = seed_resident_warps();
    b.list_cap = std::max<uint32_t>(max_len + 1, b.intv_cap);
    const int ext_warps = extend_resident_warps();
    const size_t ext_per_warp = extend_scratch_per_warp(max_len, rseq_cap);
    uint32_t z_cap = 0;
    const size_t fin_per_warp = finalize_scratch_per_warp(max_len, rseq_cap, &z_cap);
    int fin_warps = finalize_resident_warps();
    {   // bound the traceback scratch to ~8 GB
        size_t budget = (size_t)8 << 30;
        int fit = (int)std::max<size_t>(budget / fin_per_warp, 4 * 148);
        fin_warps = std::min(fin_warps, fit) / 4 * 4;
    }
#define ENS(x) do { cudaError_t e_ = (x); if (e_ == cudaSuccess && h->test_pool_oom > 0) { --h->test_pool_oom; e_ = cudaErrorMemoryAllocation; } \
    if (e_ != cudaSuccess) { if (e_ == cudaErrorMemoryAllocation) h->alloc_failed = true; cudaGetLastError(); bsq_set_error("allocating batch pools: %s", cudaGetErrorString(e_)); return BSQ_ERR; } } while (0)
    ENS(b.intv.ensure((size_t)n * b.intv_cap)); ENS(b.intv_cnt.ensure(n));
    ENS(b.seed_scratch.ensure((size_t)seed_warps * 3 * b.list_cap));
    ENS(b.raw.ensure(b.pool_cap)); ENS(b.seeds.ensure(b.pool_cap)); ENS(b.ctmp.ensure(b.pool_cap)); ENS(b.ord.ensure(b.pool_cap));
    ENS(b.chains.ensure(b.pool_cap)); ENS(b.srt.ensure(b.pool_cap)); ENS(b.regs.ensure(b.pool_cap)); ENS(b.rows.ensure(b.pool_cap));
    ENS(b.reg_cnt.ensure(n)); ENS(b.row_cnt.ensure(n)); ENS(b.row_off.ensure(n + 1)); ENS(b.blocks.ensure(n));
    ENS(b.scan_tmp.ensure(prim::scan_tmp_elems(n + 1) + 16));
    ENS(b.cigar.ensure(b.cigar_cap));
    ENS(b.ext_scratch.ensure((size_t)ext_warps * ext_per_warp)); ENS(b.fin_scratch.ensure((size_t)fin_warps * fin_per_warp));
    ENS(b.narrow_z.ensure(narrow_zbuf_bytes())); ENS(b.narrow_jobs.ensure((size_t)b.pool_cap * 5 * 24)); ENS(b.wide_jobs.ensure(b.pool_cap));
    ENS(b.ctl.ensure(64)); ENS(b.chain_todo.ensure(n)); ENS(b.fin_todo.ensure(n)); ENS(b.seed_todo.ensure(n + 1));
    if (max_len <= 496) { ENS(b.seed_pk.ensure((size_t)n * seed_thread_words(max_len))); ENS(b.seed_u32.ensure(3 * (size_t)n)); }
    if (compact) { ENS(b.sa_pos.ensure(b.pool_cap)); ENS(b.sa_pos_off.ensure((size_t)n + 1)); ENS(b.scan_tmp64.ensure(prim::scan_tmp_elems((size_t)n + 1) + 16)); }
    // the thread-per-extension pre-pass packs column scores in 16 bits: every value it stores is <= l_query * (a + 1)
    // Small batches take the warp-cooperative kernels for the DP stages: the thread-per-extension / thread-per-region kernels are built for
    // throughput (one thread runs a whole DP, ~0.5 ms of latency whatever the batch size), which is what a one-read call of
    // nuclseq_search_bwa would wait for.  BSQ_SMALL_BATCH_READS moves the threshold (0 = thread kernels always; the parity tests use that).
    static const long small_n = getenv("BSQ_SMALL_BATCH_READS") ? atol(getenv("BSQ_SMALL_BATCH_READS")) : 40000;   // measured crossover ~50 k reads (scripts/latency.py)
    const bool small_batch = (long)n < small_n;
    const bool use_memo = !small_batch && max_len <= 512 && (uint64_t)max_len * (uint64_t)(o.a + 1) < 32000 && (uint64_t)n * EXT_MEMO_CHAINS < (1ull << 31);
    if (use_memo) {
        const size_t jobs2 = (size_t)n * EXT_MEMO_CHAINS * 2;
        ENS(b.ext_memo.ensure(jobs2)); ENS(b.ext_memo_key.ensure(jobs2)); ENS(b.ext_memo_perm.ensure(jobs2));
        ENS(b.ext_memo_hist.ensure(6 * EXT_MEMO_BINS)); ENS(b.ext_todo.ensure(n));
    }
    if (!b.ext_aux_ok && !small_batch) {
        for (auto& s_ : b.ext_aux.st) ENS(cudaStreamCreateWithPriority(&s_, cudaStreamNonBlocking, &b == &h->batch ? h->prio_hi : h->prio_lo));
        for (auto& e : b.ext_aux.ev) ENS(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        b.ext_aux_ok = true;
    }
    ENS(cudaMemsetAsync(b.ctl.p, 0, 64 * 4, st));
    unsigned long long* ctr = h->collect_counters ? reinterpret_cast<unsigned long long*>(b.ctl.p + 8) : nullptr;
    cudaEventRecord(ev[0], st);
    {
        SeedParams P = seed_params(h, b, ix, n, b.intv_cap, b.ctl.p + 0, ctr ? ctr + 0 : nullptr);
        // thread per read first (almost every short read); seed_smem, warp per read, takes what it declined
        if (seed_thread_usable(P, o, b.max_len)) T.launches += launch_seed_thread(P, ix, o, b.max_len, b.ctl.p + 60, st);
        else P.todo = nullptr;
        launch_seed(P, ix, o, st, nullptr); ++T.launches;
    }
    cudaEventRecord(ev[1], st);
    if (compact) {   // the text positions of every SA lookup the chain kernels will make, by LF walks from the samples
        SaResolveParams R;
        R.intv = b.intv.p; R.intv_cnt = b.intv_cnt.p; R.intv_cap = b.intv_cap; R.n_reads = n; R.off = b.sa_pos_off.p; R.scan_tmp = b.scan_tmp64.p;
        R.pos = b.sa_pos.p; R.pos_cap = b.pool_cap; R.ticket = b.ctl.p + 31; R.err = b.ctl.p + 51;
        R.lf_steps = reinterpret_cast<unsigned long long*>(b.ctl.p + 28); R.iters = reinterpret_cast<unsigned long long*>(b.ctl.p + 54);
        launch_sa_resolve_batch(R, ix, o, st, &T.launches);
    }
    {
        ChainParams P;
        P.seqs = b.seqs.p; P.offs = b.offs.p; P.n_reads = n; P.intv = b.intv.p; P.intv_cnt = b.intv_cnt.p; P.intv_cap = b.intv_cap;
        P.raw = b.raw.p; P.ctmp = b.ctmp.p; P.ord = b.ord.p; P.chains = b.chains.p; P.seeds = b.seeds.p; P.pool_cap = b.pool_cap; P.pool_top = b.ctl.p + 5;
        P.blocks = b.blocks.p; P.ticket = b.ctl.p + 1; P.overflow = b.ctl.p + 4; P.counters = ctr ? ctr + 1 : nullptr;
        P.logtab = needs_seed_sw(b.max_len) ? b.read_logtab.p : nullptr; P.sw_cells = nullptr;
        // short reads: a thread-per-read pass takes every read with a handful of seed occurrences, the warp kernel the rest
        const bool thread_chain = !P.logtab;
        P.todo = thread_chain ? b.chain_todo.p : nullptr; P.todo_cnt = b.ctl.p + 57;
        P.sa_pos = compact ? b.sa_pos.p : nullptr; P.sa_pos_off = compact ? b.sa_pos_off.p : nullptr;
        if (thread_chain) { launch_chain_thread(P, ix, o, st); ++T.launches; }
        launch_chain(P, ix, o, st); ++T.launches;
    }
    cudaEventRecord(ev[2], st);
    {
        ExtendParams P;
        P.seqs = b.seqs.p; P.offs = b.offs.p; P.n_reads = n; P.blocks = b.blocks.p; P.chains = b.chains.p; P.seeds = b.seeds.p; P.srt = b.srt.p;
        P.regs = b.regs.p; P.reg_cnt = b.reg_cnt.p; P.scratch = b.ext_scratch.p; P.scratch_per_warp = ext_per_warp; P.max_len = max_len; P.rseq_cap = rseq_cap;
        P.ticket = b.ctl.p + 2; P.overflow = b.ctl.p + 4; P.need_rseq = b.ctl.p + 7; P.counters = ctr ? ctr + 3 : nullptr;
        P.memo = use_memo ? b.ext_memo.p : nullptr; P.memo_key = b.ext_memo_key.p; P.memo_perm = b.ext_memo_perm.p; P.memo_hist = b.ext_memo_hist.p;
        P.todo = use_memo ? b.ext_todo.p : nullptr; P.todo_cnt = b.ctl.p + 56;
        launch_extend_memo(P, ix, o, st, &T.launches, b.ext_aux);     // runs only with use_memo, whose !small_batch made the side streams
        if (use_memo) { launch_extend_finish(P, ix, o, st); ++T.launches; }
        launch_extend(P, ix, o, st); ++T.launches;
    }
    cudaEventRecord(ev[3], st);
    {
        FinalizeParams P;
        P.seqs = b.seqs.p; P.offs = b.offs.p; P.ids = b.ids.p; P.n_reads = n; P.blocks = b.blocks.p; P.regs = b.regs.p; P.reg_cnt = b.reg_cnt.p;
        P.rows = b.rows.p; P.row_cnt = b.row_cnt.p; P.cigar_pool = b.cigar.p; P.cigar_cap = b.cigar_cap; P.cigar_top = b.ctl.p + 6;
        P.scratch = b.fin_scratch.p; P.scratch_per_warp = fin_per_warp; P.max_len = max_len; P.z_cap = z_cap; P.ann_id = h->d_ann_id;
        P.narrow_jobs = small_batch ? nullptr : b.narrow_jobs.p; P.narrow_cap = b.pool_cap; P.narrow_cnt = b.ctl.p + 32; P.wide_jobs = b.wide_jobs.p; P.wide_cnt = b.ctl.p + 25;
        P.narrow_z = b.narrow_z.p;
        P.ticket = b.ctl.p + 40; P.overflow = b.ctl.p + 4; P.need_rseq = b.ctl.p + 7; P.counters = ctr ? ctr + 6 : nullptr;
        P.todo = small_batch ? nullptr : b.fin_todo.p; P.todo_cnt = b.ctl.p + 58;
        launch_finalize(P, ix, o, st, rseq_cap, fin_warps, &T.launches, b.ext_aux_ok ? &b.ext_aux : nullptr);
    }
    // compact rows: exclusive scan of row_cnt (n + 1 entries, the last one is a zero pad) -> row_off
    prim::device_scan<uint32_t, prim::OpSum, false>(b.row_cnt.p, b.row_off.p, n, b.scan_tmp.p, prim::OpSum(), st, &T.launches);
    {   // rows in read order + MAPQ (the tail of mem_reg2aln, SURVEY A.12): part of the step, so inside the timed window
        if (!h->d_logtab) {
            std::vector<double> tab(LOGTAB_N);
            tab[0] = 0.;
            for (int i = 1; i < LOGTAB_N; ++i) tab[i] = log((double)i);   // host libm: the values the reference's log() returns
            ENS(cudaMalloc(&h->d_logtab, LOGTAB_N * sizeof(double)));
            ENS(cudaMemcpy(h->d_logtab, tab.data(), LOGTAB_N * sizeof(double), cudaMemcpyHostToDevice));
        }
        b.rows_cap = std::max<uint64_t>(b.rows_cap, (uint64_t)n * 2 + 4096);
        ENS(b.rows_compact.ensure(b.rows_cap));
        // the extension records are always produced on the device: a row the host must finish (MAPQ outside the log table) needs them
        ENS(b.rows_ext.ensure(b.rows_cap));
        MapqParams M; M.a = h->opts.a; M.b = h->opts.b; M.min_seed_len = h->opts.min_seed_len; M.coef_len = h->mapQ_coef_len;
        M.coef_fac = (double)h->mapQ_coef_fac; M.logtab = h->d_logtab;
        b.cig_rebased = 0;
        k_compact_rows<<<(unsigned)std::min<uint32_t>((n + 255) / 256, 148 * 16), 256, 0, st>>>(b.blocks.p, b.rows.p, b.row_cnt.p, b.row_off.p, n, b.rows_compact.p, b.rows_ext.p,
                                                (uint32_t)std::min<uint64_t>(b.rows_cap, 0xffffffffull), M, b.ctl.p + 30); ++T.launches;
    }
    cudaEventRecord(ev[4], st);
    ENS(cudaMemcpyAsync(b.ctl_host, b.ctl.p, 8 * 4, cudaMemcpyDeviceToHost, st));
    ENS(cudaMemcpyAsync(b.ctl_host + 8, b.row_off.p + (n - 1), 4, cudaMemcpyDeviceToHost, st));
    ENS(cudaMemcpyAsync(b.ctl_host + 9, b.row_cnt.p + (n - 1), 4, cudaMemcpyDeviceToHost, st));
    ENS(cudaMemcpyAsync(b.ctl_host + 10, b.ctl.p + 30, 4, cudaMemcpyDeviceToHost, st));
    if (compact) ENS(cudaMemcpyAsync(b.ctl_host + 11, b.ctl.p + 51, 4, cudaMemcpyDeviceToHost, st));
    b.idle = false;
    return BSQ_OK;
#undef ENS
}

// Waits for the attempt in flight and looks at its control words: *again = a pool or a scratch area was too small;
// the capacities have been raised and pipeline_enqueue must run once more.
int pipeline_check(bsq_index* h, Batch& b, bool* again) {
    *again = false;
    if (b.idle) return BSQ_OK;
    bsq_timing& T = h->timing;
    CUDA_CHECK(cudaStreamSynchronize(b.st));
    b.idle = true;
    { cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { bsq_set_error("kernel failure: %s", cudaGetErrorString(e_)); return BSQ_ERR; } }
    const uint32_t* ctl = b.ctl_host;
    if (b.att_compact && ctl[11]) {
        bsq_set_error("compact index: %s (the index is damaged)", ctl[11] == 1 ? "an SA lookup names a row outside [0, seq_len]" : "an LF walk is longer than seq_len");
        return BSQ_ERR;
    }
    cudaEvent_t* ev = b.ev;
    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); T.seed += ms;
    cudaEventElapsedTime(&ms, ev[1], ev[2]); T.chain += ms;
    cudaEventElapsedTime(&ms, ev[2], ev[3]); T.extend += ms;
    cudaEventElapsedTime(&ms, ev[3], ev[4]); T.finalize += ms;
    cudaEventElapsedTime(&ms, ev[0], ev[4]); T.total += ms;
    if (ctl[7] > b.att_rseq_cap && ctl[4] != 2) {   // a reference window was larger than planned: grow the per-warp scratch and run again
        b.rseq_cap = ctl[7] + ctl[7] / 8 + 64;
        *again = true;
        return BSQ_OK;
    }
    if (ctl[4] == 0) {
        if (h->collect_counters) {
            uint64_t c8[8];
            CUDA_CHECK(cudaMemcpy(c8, b.ctl.p + 8, sizeof(c8), cudaMemcpyDeviceToHost));
            for (int i = 0; i < 8; ++i) h->counters[i] += c8[i];
        }
        b.out_rows = (uint64_t)ctl[8] + ctl[9]; b.out_cig = ctl[6];
        if (b.out_rows > b.rows_cap) {   // more rows than the compacted buffer holds: grow it and run the batch again
            b.rows_cap = b.out_rows + b.out_rows / 8 + 4096;
            *again = true;
            return BSQ_OK;
        }
        b.aligned = true;
        return BSQ_OK;
    }
    if (ctl[4] == 2) { bsq_set_error("alignment scratch capacity exceeded (reference window / traceback larger than planned)"); return BSQ_ERR; }
    // a pool was too small: grow everything that can overflow and run the batch again
    if (ctl[5] > b.pool_cap) b.pool_cap = (uint32_t)std::min<uint64_t>((uint64_t)ctl[5] + ctl[5] / 8 + 4096, 0x7fffffffull);
    else if (ctl[6] > b.cigar_cap) b.cigar_cap = (uint32_t)std::min<uint64_t>((uint64_t)ctl[6] + ctl[6] / 8 + 4096, 0x7fffffffull);
    else b.intv_cap *= 2;
    *again = true;
    return BSQ_OK;
}

// finishes the batch: checks the attempt in flight (if any) and re-runs it while capacities have to grow
int pipeline_finish(bsq_index* h, Batch& b) {
    for (int attempt = 0; attempt < 12; ++attempt) {
        bool again = false;
        if (pipeline_check(h, b, &again) != BSQ_OK) return BSQ_ERR;
        if (!again) { if (!b.aligned) break; return BSQ_OK; }
        if (pipeline_enqueue(h, b) != BSQ_OK) return BSQ_ERR;
    }
    bsq_set_error("batch pools kept overflowing");
    return BSQ_ERR;
}

// a call's stage times and counters start from zero (the pipeline adds to them attempt by attempt, chunk by chunk)
void reset_stage_timing(bsq_index* h) {
    bsq_timing& T = h->timing;
    T.seed = T.chain = T.extend = T.finalize = T.total = 0;
    memset(h->counters, 0, sizeof(h->counters));
}

int run_pipeline(bsq_index* h, Batch& b) {
    reset_stage_timing(h);
    if (pipeline_enqueue(h, b) != BSQ_OK) return BSQ_ERR;
    return pipeline_finish(h, b);
}

// mem_approx_mapq_se (SURVEY A.12) on the host: double math with libm log
int approx_mapq(const bsq_index* h, const bsq_row& a, const bsq_row_ext& x) {
    const bsq_opts& o = h->opts;
    int mapq, l, sub = x.sub ? x.sub : o.min_seed_len * o.a;
    double identity;
    sub = x.csub > sub ? x.csub : sub;
    if (sub >= a.score) return 0;
    l = a.qe - a.qb > a.re - a.rb ? a.qe - a.qb : (int)(a.re - a.rb);
    identity = 1. - (double)(l * o.a - a.score) / (o.a + o.b) / l;
    if (a.score == 0) mapq = 0;
    else {   // mapQ_coef_len = 50 > 0
        double tmp;
        tmp = l < h->mapQ_coef_len ? 1. : h->mapQ_coef_fac / log(l);
        tmp *= identity * identity;
        mapq = (int)(6.02 * (a.score - sub) / o.a * tmp * tmp + .499);
    }
    if (x.sub_n > 0) mapq -= (int)(4.343 * log(x.sub_n + 1) + .499);
    if (mapq > 60) mapq = 60;
    if (mapq < 0) mapq = 0;
    mapq = (int)(mapq * (1. - x.frac_rep) + .499);
    return mapq;
}

// A result lives in ONE pinned host block, laid out by capacity: row_off (u64 x (n+1)) | rows (row_cap + 1) |
// cigar (cig_cap + 1) | the device's u32 row offsets (n + 1).  Freed blocks are cached process-wide so that
// steady-state calls do not pay cudaHostAlloc.
struct ResultImpl { bsq_result pub; void* block; size_t bytes; uint64_t row_cap, cig_cap; uint32_t* o32; bsq_row_ext* ext; uint64_t serial; };
// results handed out and not yet freed: bsq_result_tuples recognises its own results (a caller may also pass a bsq_result it assembled)
std::mutex g_live_mu; std::vector<const ResultImpl*> g_live; uint64_t g_result_serial = 0;
struct PinnedCache { void* ptr[4]; size_t bytes[4]; };
PinnedCache g_pinned = {{nullptr, nullptr, nullptr, nullptr}, {0, 0, 0, 0}};
std::mutex g_pinned_mu;

void* pinned_get(size_t need, size_t* got) {
    {
        std::lock_guard<std::mutex> lk(g_pinned_mu);
        for (int i = 0; i < 4; ++i)
            if (g_pinned.ptr[i] && g_pinned.bytes[i] >= need && g_pinned.bytes[i] <= 2 * need + (1 << 20)) {
                void* p = g_pinned.ptr[i]; *got = g_pinned.bytes[i]; g_pinned.ptr[i] = nullptr; g_pinned.bytes[i] = 0; return p;
            }
    }
    void* p = nullptr;
    size_t want = need + need / 8 + 4096;
    if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    *got = want;
    return p;
}
void pinned_put(void* p, size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(g_pinned_mu);
        for (int i = 0; i < 4; ++i) if (!g_pinned.ptr[i]) { g_pinned.ptr[i] = p; g_pinned.bytes[i] = bytes; return; }
    }
    cudaFreeHost(p);
}

// layout by capacity: row_off (u64 x (n+1)) | rows (row_cap + 1) | cigar (cig_cap + 1) | the device's u32 row offsets (n + 1) |
// extension rows (row_cap + 1; only with BSQ_FLAG_ROWS_EXT or when a row's MAPQ was finished on the host)
ResultImpl* result_new(uint64_t n, uint64_t row_cap, uint64_t cig_cap, bool with_ext) {
    const size_t off_rows = ((n + 1) * 8 + 63) & ~(size_t)63;
    const size_t off_cig = (off_rows + (row_cap + 1) * sizeof(bsq_row) + 63) & ~(size_t)63;
    const size_t off_o32 = (off_cig + (cig_cap + 1) * 4 + 63) & ~(size_t)63;
    const size_t off_ext = (off_o32 + (n + 1) * 4 + 63) & ~(size_t)63;
    const size_t need = off_ext + (with_ext ? (row_cap + 1) * sizeof(bsq_row_ext) : 0);
    size_t got = 0;
    void* block = pinned_get(need, &got);
    if (!block) { bsq_set_error("cannot allocate %zu bytes of pinned host memory for the result", need); return nullptr; }
    ResultImpl* R = new ResultImpl;
    R->block = block; R->bytes = got; R->row_cap = row_cap; R->cig_cap = cig_cap;
    R->pub.n_reads = n;
    R->pub.row_off = reinterpret_cast<uint64_t*>(block);
    R->pub.rows = reinterpret_cast<bsq_row*>(static_cast<char*>(block) + off_rows);
    R->pub.cigar = reinterpret_cast<uint32_t*>(static_cast<char*>(block) + off_cig);
    R->pub.n_cigar_words = 0;
    R->o32 = reinterpret_cast<uint32_t*>(static_cast<char*>(block) + off_o32);
    R->ext = with_ext ? reinterpret_cast<bsq_row_ext*>(static_cast<char*>(block) + off_ext) : nullptr;
    R->pub.rows_ext = R->ext;
    { std::lock_guard<std::mutex> lk(g_live_mu); R->serial = ++g_result_serial; g_live.push_back(R); }
    return R;
}

void result_delete(ResultImpl* R) {
    if (!R) return;
    { std::lock_guard<std::mutex> lk(g_live_mu); for (size_t i = 0; i < g_live.size(); ++i) if (g_live[i] == R) { g_live[i] = g_live.back(); g_live.pop_back(); break; } }
    pinned_put(R->block, R->bytes); delete R;
}

// Compacts the aligned batch's rows on the device (+ MAPQ) and starts the copies into the result: the batch's reads are
// reads [read_base, read_base + b.n) of the result, its rows go to row_base, its CIGAR words to cig_base.
// A chunk's place in the whole result, applied on the device ahead of the copy: 64-bit row offsets from the chunk's 32-bit ones, CIGAR
// offsets moved behind the earlier chunks' words (a host loop over a million 64-byte records costs more than the copy itself).
static __global__ void k_result_rebase(const uint32_t* __restrict__ row_off, uint64_t n, uint64_t row_base, uint64_t* __restrict__ row_off64,
                                       RowPub* __restrict__ rows, uint64_t n_rows, uint32_t cig_delta) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t i = t0; i < n; i += stride) row_off64[i] = row_base + row_off[i];
    if (cig_delta) for (uint64_t i = t0; i < n_rows; i += stride) if (rows[i].n_cigar) rows[i].cigar_off += cig_delta;
}

int download_enqueue(bsq_index* h, Batch& b, ResultImpl* R, uint64_t read_base, uint64_t row_base, uint64_t cig_base) {
    const uint64_t n = b.n;
    if (n == 0 || !h->meta.built || !b.aligned) return BSQ_OK;
    const uint64_t total_rows = b.out_rows; const uint32_t cig_top = b.out_cig;
    if (row_base + total_rows > R->row_cap || cig_base + cig_top > R->cig_cap || cig_base + cig_top > 0xffffffffull) { bsq_set_error("result block too small"); return BSQ_ERR; }
    cudaStream_t st = b.st;
    b.res_serial = R->serial; b.res_read_base = read_base; b.res_row_base = row_base; b.res_cig_base = cig_base;
    CUDA_CHECK(b.row_off64.ensure(n + 1));
    k_result_rebase<<<(unsigned)std::min<uint64_t>((std::max<uint64_t>(n, total_rows) + 255) / 256, 148 * 8), 256, 0, st>>>(
        b.row_off.p, n, row_base, b.row_off64.p, b.rows_compact.p, total_rows, (uint32_t)(cig_base - b.cig_rebased));
    ++h->timing.launches;
    b.cig_rebased = cig_base;
    CUDA_CHECK(cudaMemcpyAsync(R->pub.row_off + read_base, b.row_off64.p, n * 8, cudaMemcpyDeviceToHost, st));
    if (total_rows) CUDA_CHECK(cudaMemcpyAsync(R->pub.rows + row_base, b.rows_compact.p, total_rows * sizeof(bsq_row), cudaMemcpyDeviceToHost, st));
    if (total_rows && R->ext) CUDA_CHECK(cudaMemcpyAsync(R->ext + row_base, b.rows_ext.p, total_rows * sizeof(bsq_row_ext), cudaMemcpyDeviceToHost, st));
    else if (total_rows && b.ctl_host[10]) {   // rare: a MAPQ to finish on the host although the caller did not ask for the extension records
        b.ext_tmp.resize(total_rows);
        CUDA_CHECK(cudaMemcpyAsync(b.ext_tmp.data(), b.rows_ext.p, total_rows * sizeof(bsq_row_ext), cudaMemcpyDeviceToHost, st));
    }
    if (cig_top) CUDA_CHECK(cudaMemcpyAsync(R->pub.cigar + cig_base, b.cigar.p, (size_t)cig_top * 4, cudaMemcpyDeviceToHost, st));
    h->timing.d2h_bytes += n * 8 + 12 + total_rows * (sizeof(bsq_row) + (R->ext ? sizeof(bsq_row_ext) : 0)) + (uint64_t)cig_top * 4;
    return BSQ_OK;
}

// after the copies have landed: 64-bit row offsets, and MAPQ of the rows outside the device log table (very long
// alignments).  n reads starting at read_base, n_rows rows starting at row_base.
void download_finish(bsq_index* h, ResultImpl* R, uint64_t n, uint64_t read_base, uint64_t n_rows, uint64_t row_base, bool host_mapq, const bsq_row_ext* ext_tmp) {
    if (!h->meta.built) { for (uint64_t i = 0; i < n; ++i) R->pub.row_off[read_base + i] = row_base; return; }
    if (n_rows && host_mapq) {
        // alignments longer than the device's log table: mem_approx_mapq_se with libm on the host, from the extension records
        const bsq_row_ext* ext = R->ext ? R->ext + row_base : ext_tmp;
        for (uint64_t i = 0; i < n_rows && ext; ++i)
            if (R->pub.rows[row_base + i].mapq == MAPQ_HOST) R->pub.rows[row_base + i].mapq = (uint8_t)approx_mapq(h, R->pub.rows[row_base + i], ext[i]);
    }
}

int download_result(bsq_index* h, Batch& b, bsq_result** out) {
    if (!b.aligned) { bsq_set_error("no aligned batch to download"); return BSQ_ERR; }
    h->timing.d2h_bytes = 0;
    ResultImpl* R = result_new(b.n, b.out_rows, b.out_cig, (h->flags & BSQ_FLAG_ROWS_EXT) != 0);
    if (!R) return BSQ_ERR;
    if (download_enqueue(h, b, R, 0, 0, 0) != BSQ_OK || cudaStreamSynchronize(b.st) != cudaSuccess) { result_delete(R); if (!*bsq_last_error()) bsq_set_error("download failed"); return BSQ_ERR; }
    download_finish(h, R, b.n, 0, b.out_rows, 0, b.ctl_host && b.ctl_host[10], b.ext_tmp.data());
    R->pub.row_off[b.n] = b.out_rows;
    R->pub.n_cigar_words = b.out_cig;
    *out = &R->pub;
    return BSQ_OK;
}

// bsq_align_batch on a large batch: the reads are cut into chunks that alternate between two lanes (batch + stream
// each), so that a chunk's host->device copy and its result's device->host copy run while the other lane computes.
// Chunk c's rows follow chunk c-1's in the result, so downloads are issued in chunk order; a lane takes chunk c+2 as
// soon as chunk c's download has been queued (stream order protects the device buffers), and the host-side completion
// of a download is deferred until the next chunk's work is in the queue.
// chunk size: half of the batch, within [64 K, 1 M] reads.  Measured on B200, 1 M x 150 bp with the slim wire format (64 MB in, 77 MB
// out): one pass 35.2 ms, 2 chunks 31.8, 4 chunks 35.9 (a chunk pays ~40 kernel tails and runs on half-empty persistent grids, so few
// large chunks win once the copies are small).  BSQ_CHUNK_READS overrides it.
constexpr uint64_t CHUNK_MIN = 1u << 16, CHUNK_MAX = 1u << 20;
uint64_t chunk_reads(uint64_t n, bool two = false) {
    if (two) return std::max((n + 1) / 2, CHUNK_MIN);
    if (const char* e = getenv("BSQ_CHUNK_READS")) { const long long x = atoll(e); if (x >= 1024) return (uint64_t)x; }   // read per call: tests set it
    const uint64_t k = std::max<uint64_t>(2, (n + CHUNK_MAX - 1) / CHUNK_MAX);     // as few chunks as the cap allows, at least two
    return std::max((n + k - 1) / k, CHUNK_MIN);
}

// where a batch's reads come from: ASCII + offsets (bsq_align_batch) or NUCLSEQ datum images (bsq_align_batch_datums)
struct ReadSrc { const char* seqs; const uint64_t* offs; const uint8_t* dbytes; const uint64_t* doff; const int64_t* ids; };
int upload_src(bsq_index* h, Batch& b, const ReadSrc& S, uint64_t s0, uint64_t cnt) {
    const int64_t* ids = S.ids ? S.ids + s0 : nullptr;
    return S.dbytes ? upload_datums(h, b, S.dbytes, S.doff + s0, ids, cnt, s0) : upload_reads(h, b, S.seqs, S.offs + s0, ids, cnt, s0);
}

int align_chunked(bsq_index* h, const ReadSrc& S, uint64_t n, bsq_result** out, bool* fell_back) {
    *fell_back = false;
    if (!h->stream2) {
        CUDA_CHECK(cudaStreamCreateWithPriority(&h->stream2, cudaStreamNonBlocking, h->prio_lo));
        h->batch2.st = h->stream2;
    }
    static const bool trace = getenv("BSQ_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto mark = [&](const char* what, uint64_t c) {
        if (trace) fprintf(stderr, "[bsq trace] %8.3f ms  %s %llu\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(), what, (unsigned long long)c);
    };
    Batch* lane[2] = {&h->batch, &h->batch2};
    for (Batch* b : lane) if (!b->evx_ok) { for (auto& e : b->ev_x) cudaEventCreate(&e); b->evx_ok = true; }
    const uint64_t CHUNK_READS = chunk_reads(n, (h->flags & BSQ_FLAG_TWO_CHUNKS) != 0);
    const uint64_t n_chunks = (n + CHUNK_READS - 1) / CHUNK_READS;
    auto start_of = [&](uint64_t c) { return std::min(c * CHUNK_READS, n); };
    auto launch = [&](uint64_t c) -> int {
        Batch& b = *lane[c & 1];
        const uint64_t s0 = start_of(c), cnt = start_of(c + 1) - s0;
        b.intv_cap = std::max(b.intv_cap, lane[(c & 1) ^ 1]->intv_cap);      // capacities learnt by one lane serve the other
        cudaEventRecord(b.ev_x[0], b.st);
        mark("upload begin", c);
        if (upload_src(h, b, S, s0, cnt) != BSQ_OK) return BSQ_ERR;
        mark("upload done (headers back)", c);
        cudaEventRecord(b.ev_x[1], b.st);
        const int rc2 = pipeline_enqueue(h, b);
        mark("pipeline queued", c);
        return rc2;
    };
    struct Pending { bool on = false; uint64_t c = 0, n = 0, n_rows = 0, row_base = 0; bool host_mapq = false; } pend;
    ResultImpl* R = nullptr;
    auto complete = [&](const Pending& q) -> int {       // host side of chunk q.c's download
        Batch& b = *lane[q.c & 1];
        if (cudaEventSynchronize(b.ev_x[3]) != cudaSuccess) { bsq_set_error("result download failed: %s", cudaGetErrorString(cudaGetLastError())); return BSQ_ERR; }
        float ms;
        if (cudaEventElapsedTime(&ms, b.ev_x[2], b.ev_x[3]) == cudaSuccess) h->timing.d2h += ms;
        mark("download arrived", q.c);
        download_finish(h, R, q.n, start_of(q.c), q.n_rows, q.row_base, q.host_mapq, b.ext_tmp.data());
        mark("download finished on the host", q.c);
        return BSQ_OK;
    };
    uint64_t row_base = 0, cig_base = 0;
    int rc = launch(0);
    if (rc == BSQ_OK && n_chunks > 1) rc = launch(1);
    for (uint64_t c = 0; c < n_chunks && rc == BSQ_OK; ++c) {
        Batch& b = *lane[c & 1];
        if ((rc = pipeline_finish(h, b)) != BSQ_OK) break;
        mark("pipeline finished", c);
        { float ms; if (cudaEventElapsedTime(&ms, b.ev_x[0], b.ev_x[1]) == cudaSuccess) h->timing.h2d += ms; }
        if (!R) {
            // capacity of the result from the first chunk's yield
            // (BSQ_TEST_TIGHT_RESULT makes the estimate too small on purpose so that tests reach the one-plain-pass fallback)
            const double scale = (double)n / (double)b.n * (getenv("BSQ_TEST_TIGHT_RESULT") ? 0.4 : 1.2);
            R = result_new(n, (uint64_t)(b.out_rows * scale) + (getenv("BSQ_TEST_TIGHT_RESULT") ? 16 : 65536), (uint64_t)(b.out_cig * scale) + (getenv("BSQ_TEST_TIGHT_RESULT") ? 16 : 65536), (h->flags & BSQ_FLAG_ROWS_EXT) != 0);
            if (!R) { rc = BSQ_ERR; break; }
        }
        if (row_base + b.out_rows > R->row_cap || cig_base + b.out_cig > R->cig_cap) { *fell_back = true; break; }
        cudaEventRecord(b.ev_x[2], b.st);
        if ((rc = download_enqueue(h, b, R, start_of(c), row_base, cig_base)) != BSQ_OK) break;
        cudaEventRecord(b.ev_x[3], b.st);
        mark("download queued", c);
        Pending mine; mine.on = true; mine.c = c; mine.n = b.n; mine.n_rows = b.out_rows; mine.row_base = row_base;
        mine.host_mapq = b.ctl_host[10] != 0;   // read now: the lane's control words are reused by the next chunk it takes
        row_base += b.out_rows; cig_base += b.out_cig;
        if (pend.on) { if ((rc = complete(pend)) != BSQ_OK) break; pend.on = false; }
        // chunk c-1's lane is free on the host side now (its download completed): it already runs chunk c+1.
        // This lane takes chunk c+2 behind its download.
        if (c + 2 < n_chunks) { if ((rc = launch(c + 2)) != BSQ_OK) break; }
        pend = mine;
    }
    if (rc == BSQ_OK && !*fell_back && pend.on) rc = complete(pend);
    if (rc != BSQ_OK || *fell_back) {
        cudaStreamSynchronize(h->stream); cudaStreamSynchronize(h->stream2);
        cudaGetLastError();
        h->batch.idle = h->batch2.idle = true; h->batch.aligned = h->batch2.aligned = false;
        result_delete(R);
        return rc;
    }
    R->pub.row_off[n] = row_base;
    R->pub.n_cigar_words = cig_base;
    *out = &R->pub;
    return BSQ_OK;
}

}  // namespace

extern "C" {

int bsq_reads_upload(bsq_index* h, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n) {
    BSQ_ENTRY();
    if (!h || (n && (!seqs || !offs))) { bsq_set_error("null argument"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    h->timing.launches = 0;
    h->timing.h2d_bytes = 0;
    if (upload_reads(h, h->batch, seqs, offs, ids, n) != BSQ_OK) return BSQ_ERR;
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    return BSQ_OK;
}

int bsq_align_resident(bsq_index* h) {
    BSQ_ENTRY();
    if (!h) { bsq_set_error("null index"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    h->timing.launches = 0;
    return run_pipeline(h, h->batch);
}

int bsq_result_download(bsq_index* h, bsq_result** out) {
    BSQ_ENTRY();
    if (!h || !out) { bsq_set_error("null argument"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    return download_result(h, h->batch, out);
}

static int align_batch_src(bsq_index* h, const ReadSrc& S, uint64_t n, bsq_result** out) {
    CUDA_CHECK(cudaSetDevice(h->device));
    Event e0, e1, e2, e3;
    cudaEventCreate(&e0.h); cudaEventCreate(&e1.h); cudaEventCreate(&e2.h); cudaEventCreate(&e3.h);
    bsq_timing& T = h->timing;
    T.launches = 0; T.h2d_bytes = T.d2h_bytes = 0; T.h2d = T.d2h = 0; T.notes = 0;
    int rc = BSQ_OK;
    bool chunked = n >= 2 * CHUNK_MIN && n > chunk_reads(n, (h->flags & BSQ_FLAG_TWO_CHUNKS) != 0) && h->meta.built;
    cudaEventRecord(e0, h->stream);
    if (chunked) {
        // two lanes, copies overlapped with compute; the stage times are sums over chunks of each lane's stream time
        reset_stage_timing(h);
        bool fell_back = false;
        rc = align_chunked(h, S, n, out, &fell_back);
        if (fell_back) {   // the result outgrew the estimate: one plain pass; the call succeeds and says so in bsq_timing.notes
            T.notes |= BSQ_NOTE_CHUNK_FALLBACK;
            chunked = false; T.h2d_bytes = T.d2h_bytes = 0; T.h2d = T.d2h = 0;
        }
        else { cudaEventRecord(e3, h->stream); cudaEventSynchronize(e3); cudaEventElapsedTime(&T.total, e0, e3); }
    }
    if (!chunked) {
        rc = upload_src(h, h->batch, S, 0, n);
        cudaEventRecord(e1, h->stream);
        if (rc == BSQ_OK) rc = run_pipeline(h, h->batch);
        cudaEventRecord(e2, h->stream);
        if (rc == BSQ_OK) rc = download_result(h, h->batch, out);
        cudaEventRecord(e3, h->stream);
        cudaEventSynchronize(e3);
        cudaEventElapsedTime(&T.h2d, e0, e1); cudaEventElapsedTime(&T.d2h, e2, e3); cudaEventElapsedTime(&T.total, e0, e3);
    }
    if (rc == BSQ_OK && !S.ids) h->lrand_state = lrand48_advance(h->lrand_state, n);   // the session's stream moved on by one draw per read
    return rc;
}

int bsq_align_batch(bsq_index* h, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n, bsq_result** out) {
    BSQ_ENTRY();
    if (!h || !out || (n && (!seqs || !offs))) { bsq_set_error("null argument"); return BSQ_ERR; }
    const ReadSrc S{seqs, offs, nullptr, nullptr, ids};
    return align_batch_src(h, S, n, out);
}

int bsq_align_batch_datums(bsq_index* h, const uint8_t* bytes, const uint64_t* off, const int64_t* ids, uint64_t n, bsq_result** out) {
    BSQ_ENTRY();
    if (!h || !out || (n && (!bytes || !off))) { bsq_set_error("null argument"); return BSQ_ERR; }
    const ReadSrc S{nullptr, nullptr, bytes, off, ids};
    return align_batch_src(h, S, n, out);
}

int bsq_session_lrand48(bsq_index* h, int set, uint64_t* state) {
    BSQ_ENTRY();
    if (!h || !state) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (set) h->lrand_state = *state & 0xFFFFFFFFFFFFULL; else *state = h->lrand_state;
    return BSQ_OK;
}

// ---- row materialisation (SURVEY.md 8f-2)

// row -> read index of a piece from its reads' 64-bit row offsets, counted from row_base (thread per read).  Read 0 starts at row 0
// and the last read ends at n_rows, so every row gets a read whatever offsets a caller-assembled result holds.
static __global__ void k_row_read(const uint64_t* row_off, uint64_t n_reads, uint64_t row_base, uint64_t n_rows, uint32_t* row_read) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t next = r + 1 < n_reads ? row_off[r + 1] - row_base : n_rows, end = next < n_rows ? next : n_rows;
        for (uint64_t k = r ? row_off[r] - row_base : 0; k < end; ++k) row_read[k] = (uint32_t)r;
    }
}
static __global__ void k_add_u64(uint64_t* v, uint64_t n, uint64_t add) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) v[i] += add;
}

static void index_holes_sorted(const bsq_index* h, uint32_t flags, std::vector<TupleHole>& holes, std::vector<int64_t>& maxend) {
    holes.resize(h->holes.size());
    for (size_t i = 0; i < holes.size(); ++i) {
        // reference behaviour: offsets as stored in the row's datum, i.e. relative to its own row (bwa.cpp:100-104); the fix-up rebases them
        const int64_t base = (flags & BSQ_TUPLES_FIX_HOLE_OFFSETS) ? h->ann_offset[h->hole_ann[i]] : 0;
        holes[i].offset = h->holes[i].offset + base; holes[i].end = holes[i].offset + h->holes[i].len; holes[i].idx = (uint32_t)i; holes[i].amb = (uint8_t)h->holes[i].amb;
    }
    std::stable_sort(holes.begin(), holes.end(), [](const TupleHole& a, const TupleHole& b) { return a.offset < b.offset; });
    maxend.resize(holes.size());
    for (size_t i = 0; i < holes.size(); ++i) maxend[i] = i ? std::max(maxend[i - 1], holes[i].end) : holes[i].end;
}

// the tuples handed out: one pinned block from the library's cache, off | ref_match | bytes
struct TuplesImpl { bsq_tuples pub; void* host = nullptr; size_t host_bytes = 0; ~TuplesImpl() { if (host) pinned_put(host, host_bytes); } };

struct StagedResult;

// A piece of a result to materialise on the handle h (its device, pac, annotations and launch counter): device views of the TupleParams
// inputs, the stream it runs on, its scratch, the host word its byte total comes back to and, for a piece that is not resident, the
// uploads that fill those views
struct TuplePiece {
    bsq_index* h;
    const RowPub* rows; uint64_t n_rows; const uint32_t* cigar; const uint8_t* seqs; const uint64_t* offs;
    const uint64_t* row_off; uint64_t n_reads, row_base;    // row offsets of the piece's reads, counted from row_base
    cudaStream_t st; TupleScratch* s; uint64_t* n_bytes;
    StagedResult* stage;
};

// Reads [r0, r0 + n) of a result that is not resident (assembled by the caller, three or more chunks, another call's result, a device
// that has aligned something else since): their rows, row offsets, reads and read offsets go to call-local buffers as they are.  The
// whole result takes every CIGAR word; a part of it takes the span of words its rows use, which the device finds first (k_cigar_span).
struct StagedResult {
    const bsq_result* res = nullptr; const char* seqs = nullptr; const uint64_t* offs = nullptr;
    uint64_t r0 = 0, n = 0, row0 = 0; bool whole = true;
    DevBuf<RowPub> rows; DevBuf<uint32_t> cigar; DevBuf<uint8_t> text; DevBuf<uint64_t> row_off, read_off; DevBuf<unsigned long long> span;
    TupleScratch s;
};

// [first, end) of the CIGAR words that rows with a CIGAR use; span[0] starts at ~0 and span[1] at 0
static __global__ void k_cigar_span(const RowPub* rows, uint64_t n_rows, unsigned long long* span) {
    unsigned long long lo = ~0ull, hi = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (uint64_t)gridDim.x * blockDim.x)
        if (rows[i].n_cigar) { lo = min(lo, (unsigned long long)rows[i].cigar_off); hi = max(hi, (unsigned long long)rows[i].cigar_off + rows[i].n_cigar); }
    for (int o = 16; o; o >>= 1) { lo = min(lo, __shfl_xor_sync(~0u, lo, o)); hi = max(hi, __shfl_xor_sync(~0u, hi, o)); }
    if ((threadIdx.x & 31) == 0) { atomicMin(span, lo); atomicMax(span + 1, hi); }
}

// The piece of reads [r0, r0 + n) of `res` on handle h, with its call-local buffers in S.  A block without rows uploads nothing.
static int stage_block(bsq_index* h, StagedResult& S, const bsq_result* res, const char* seqs, const uint64_t* offs, uint64_t r0, uint64_t n,
                       const char* what, TuplePiece& pc) {
    const uint64_t row0 = r0 ? res->row_off[r0] : 0;
    if (n && res->row_off[r0 + n] < row0) { bsq_set_error("%s: row offsets must be non-decreasing", what); return BSQ_ERR; }
    const uint64_t n_rows = n ? res->row_off[r0 + n] - row0 : 0;
    pc = TuplePiece{h, nullptr, n_rows, nullptr, nullptr, nullptr, nullptr, n, row0, h->stream, &S.s, nullptr, nullptr};
    if (!n_rows) return BSQ_OK;
    CUDA_CHECK_AS(what, cudaSetDevice(h->device));
    if (!h->tup_host && cudaHostAlloc(&h->tup_host, 4 * 8, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError(); h->tup_host = nullptr; bsq_set_error("cannot allocate pinned host memory for the tuples"); return BSQ_ERR;
    }
    S.res = res; S.seqs = seqs; S.offs = offs; S.r0 = r0; S.n = n; S.row0 = row0; S.whole = r0 == 0 && n == res->n_reads;
    CUDA_CHECK_AS(what, S.rows.alloc(n_rows));
    if (S.whole) CUDA_CHECK_AS(what, S.cigar.alloc(res->n_cigar_words + 1)); else CUDA_CHECK_AS(what, S.span.alloc(2));
    CUDA_CHECK_AS(what, S.text.alloc(offs[r0 + n] - offs[r0] + 64));
    CUDA_CHECK_AS(what, S.row_off.alloc(n)); CUDA_CHECK_AS(what, S.read_off.alloc(n + 1));
    pc.rows = S.rows.p; pc.cigar = S.cigar.p; pc.seqs = S.text.p; pc.offs = S.read_off.p; pc.row_off = S.row_off.p;
    pc.n_bytes = h->tup_host; pc.stage = &S;
    return BSQ_OK;
}

// first half of a staged piece's uploads: its rows and, for a part of a result, the span of CIGAR words they use
static int stage_rows(const TuplePiece& pc, const char* what) {
    const StagedResult& S = *pc.stage;
    CUDA_CHECK_AS(what, cudaMemcpyAsync(S.rows.p, S.res->rows + S.row0, pc.n_rows * sizeof(RowPub), cudaMemcpyHostToDevice, pc.st));
    if (!S.whole) {
        CUDA_CHECK_AS(what, cudaMemsetAsync(S.span.p, 0xff, 8, pc.st)); CUDA_CHECK_AS(what, cudaMemsetAsync(S.span.p + 1, 0, 8, pc.st));
        k_cigar_span<<<(unsigned)std::min<uint64_t>((pc.n_rows + 255) / 256, 148 * 8), 256, 0, pc.st>>>(S.rows.p, pc.n_rows, S.span.p); ++pc.h->timing.launches;
        CUDA_CHECK_AS(what, cudaMemcpyAsync(pc.n_bytes + 1, S.span.p, 16, cudaMemcpyDeviceToHost, pc.st));
    }
    return BSQ_OK;
}

// second half, once a part's span has landed: CIGAR words, row offsets, reads and read offsets (rebased to the piece's first read)
static int stage_rest(TuplePiece& pc, const char* what) {
    StagedResult& S = *pc.stage;
    const bsq_result* r = S.res; const uint64_t n = S.n, *offs = S.offs + S.r0, total = offs[n] - offs[0];
    uint64_t lo = 0, hi = r->n_cigar_words;
    if (!S.whole) {
        lo = pc.n_bytes[1]; hi = pc.n_bytes[2];
        if (hi <= lo) lo = hi = 0;   // no row of the piece has a CIGAR
        else if (hi > r->n_cigar_words) { bsq_set_error("%s: a row's CIGAR words lie beyond the result's %llu words", what, (unsigned long long)r->n_cigar_words); return BSQ_ERR; }
        CUDA_CHECK_AS(what, S.cigar.alloc(hi - lo + 1));
        pc.cigar = S.cigar.p - lo;
    }
    if (hi > lo) CUDA_CHECK_AS(what, cudaMemcpyAsync(S.cigar.p, r->cigar + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, pc.st));
    CUDA_CHECK_AS(what, cudaMemcpyAsync(S.row_off.p, r->row_off + S.r0, n * 8, cudaMemcpyHostToDevice, pc.st));
    if (total) CUDA_CHECK_AS(what, cudaMemcpyAsync(S.text.p, S.seqs + offs[0], total, cudaMemcpyHostToDevice, pc.st));
    CUDA_CHECK_AS(what, cudaMemcpyAsync(S.read_off.p, offs, (n + 1) * 8, cudaMemcpyHostToDevice, pc.st));
    if (offs[0]) { k_rebase_offs<<<(unsigned)std::min<uint64_t>((n + 256) / 256, 148 * 8), 256, 0, pc.st>>>(S.read_off.p, n + 1, offs[0]); ++pc.h->timing.launches; }
    return BSQ_OK;
}

// The pieces of `R` still in HBM, in read order: one per lane, its rows in read order (rows_compact), its CIGAR pool and its reads'
// text -- nothing is uploaded again.  0 when the lanes no longer hold the whole result.
static int resident_pieces(bsq_index* h, const ResultImpl* R, TuplePiece* pc) {
    Batch* lanes[2] = {&h->batch, &h->batch2};
    Batch* piece[2]; int np = 0;
    for (Batch* b : lanes) if (b->aligned && b->res_serial == R->serial && b->n) piece[np++] = b;
    if (np == 2 && piece[0]->res_read_base > piece[1]->res_read_base) std::swap(piece[0], piece[1]);
    uint64_t covered = 0;
    for (int k = 0; k < np; ++k) {
        Batch& b = *piece[k];
        if (b.res_read_base != covered) return 0;
        covered += b.n;
        pc[k] = TuplePiece{h, b.rows_compact.p, b.out_rows, b.cigar.p - b.cig_rebased, b.ascii.p, b.offs.p, b.row_off64.p, b.n, b.res_row_base,
                           b.st, &b.tup, reinterpret_cast<uint64_t*>(b.ctl_host + 14), nullptr};
    }
    return covered == R->pub.n_reads ? np : 0;
}

// Row materialisation of the np pieces of a result, in read order, each on its own stream and its handle's device.  Sizes on every
// device, one synchronise, one pinned block for the whole result, then the fill: each piece's byte offsets are moved behind the earlier
// pieces' bytes on its device, and each device copies its rows into the block.  The hole table is sorted once and uploaded once per
// device.  Staged uploads run inside the timed window; device_ms is the slowest device's window.  what: the prefix of the messages.
static int tuples_materialise(TuplePiece* pc, int np, uint32_t flags, const char* what, bsq_tuples** out) {
    std::unique_ptr<TuplesImpl> T(new TuplesImpl());
    std::vector<TupleHole> holes; std::vector<int64_t> maxend;
    index_holes_sorted(pc[0].h, flags, holes, maxend);
    // per device: its hole table, the stream its window starts on, and the event its other streams wait for before they read the holes
    struct DeviceSide { int device = -1; cudaStream_t home = nullptr; DevBuf<TupleHole> holes; DevBuf<int64_t> maxend; Event e0, ready; };
    std::vector<DeviceSide> dv(np); std::vector<int> dev_of(np); std::vector<Event> e1(np); std::vector<uint64_t> nb(np, 0);
    std::vector<TupleParams> P(np);
    int nd = 0;
    for (int k = 0; k < np; ++k) {
        int d = 0;
        while (d < nd && dv[d].device != pc[k].h->device) ++d;
        if (d == nd) { dv[d].device = pc[k].h->device; dv[d].home = pc[k].st; ++nd; }
        dev_of[k] = d;
    }
    // whatever a failed step left queued ends before the buffers above, the pieces' staging and the output block are freed
    struct Drain { const TuplePiece* pc; int np; ~Drain() { for (int k = 0; k < np; ++k) { cudaSetDevice(pc[k].h->device); cudaStreamSynchronize(pc[k].st); } } } drain{pc, np};
    uint64_t n_rows = 0;
    for (int k = 0; k < np; ++k) {
        TupleScratch& s = *pc[k].s; const uint64_t nr = pc[k].n_rows;
        CUDA_CHECK_AS(what, cudaSetDevice(pc[k].h->device));
        CUDA_CHECK_AS(what, cudaEventCreate(&e1[k].h));
        if (cudaSuccess != s.off.ensure(3 * nr + 2) || cudaSuccess != s.tmp.ensure(tuple_scan_tmp_elems(nr)) || cudaSuccess != s.row_read.ensure(nr + 1) ||
            cudaSuccess != s.nholes.ensure(2 * nr + 2) || cudaSuccess != s.rm.ensure(3 * nr + 3)) { bsq_set_error("%s: out of device memory", what); return BSQ_ERR; }
        n_rows += nr;
    }
    for (int d = 0; d < nd; ++d) {
        DeviceSide& v = dv[d];
        CUDA_CHECK_AS(what, cudaSetDevice(v.device));
        CUDA_CHECK_AS(what, cudaEventCreate(&v.e0.h)); CUDA_CHECK_AS(what, cudaEventCreateWithFlags(&v.ready.h, cudaEventDisableTiming));
        CUDA_CHECK_AS(what, v.holes.alloc(holes.size() + 1)); CUDA_CHECK_AS(what, v.maxend.alloc(holes.size() + 1));
        CUDA_CHECK_AS(what, cudaEventRecord(v.e0, v.home));
        if (!holes.empty()) {
            CUDA_CHECK_AS(what, cudaMemcpyAsync(v.holes.p, holes.data(), holes.size() * sizeof(TupleHole), cudaMemcpyHostToDevice, v.home));
            CUDA_CHECK_AS(what, cudaMemcpyAsync(v.maxend.p, maxend.data(), holes.size() * 8, cudaMemcpyHostToDevice, v.home));
        }
        CUDA_CHECK_AS(what, cudaEventRecord(v.ready, v.home));
    }
    bool spans = false;
    for (int k = 0; k < np; ++k) {   // staged uploads; a part of a result stops after its rows until its CIGAR span is known
        TuplePiece& c = pc[k];
        CUDA_CHECK_AS(what, cudaSetDevice(c.h->device));
        if (c.st != dv[dev_of[k]].home) CUDA_CHECK_AS(what, cudaStreamWaitEvent(c.st, dv[dev_of[k]].ready, 0));
        if (!c.stage) continue;
        if (stage_rows(c, what) != BSQ_OK) return BSQ_ERR;
        if (c.stage->whole) { if (stage_rest(c, what) != BSQ_OK) return BSQ_ERR; } else spans = true;
    }
    for (int k = 0; k < np && spans; ++k) {
        TuplePiece& c = pc[k];
        if (!c.stage || c.stage->whole) continue;
        CUDA_CHECK_AS(what, cudaSetDevice(c.h->device)); CUDA_CHECK_AS(what, cudaStreamSynchronize(c.st));
        if (stage_rest(c, what) != BSQ_OK) return BSQ_ERR;
    }
    for (int k = 0; k < np; ++k) {       // sizes of every piece
        const TuplePiece& c = pc[k]; TupleScratch& s = *c.s; const uint64_t nr = c.n_rows; const DeviceSide& v = dv[dev_of[k]];
        TupleParams& q = P[k];
        q.rows = c.rows; q.n_rows = nr; q.row_read = s.row_read.p; q.cigar = c.cigar; q.seqs = c.seqs; q.offs = c.offs;
        q.pac = c.h->d_pac; q.l_pac = c.h->meta.l_pac; q.ann_offset = c.h->d_ann_offset;
        q.holes = v.holes.p; q.hole_maxend = v.maxend.p; q.n_holes = (uint32_t)holes.size();
        q.nholes = s.nholes.p; q.off = s.off.p; q.ref_match = s.rm.p; q.bytes = nullptr; q.fix_reverse = (flags & BSQ_TUPLES_FIX_REVERSE) != 0;
        if (!nr) continue;
        CUDA_CHECK_AS(what, cudaSetDevice(c.h->device));
        k_row_read<<<(unsigned)std::min<uint64_t>((c.n_reads + 255) / 256, 148 * 8), 256, 0, c.st>>>(c.row_off, c.n_reads, c.row_base, nr, s.row_read.p); ++c.h->timing.launches;
        CUDA_CHECK_AS(what, cudaMemsetAsync(s.off.p, 0, (3 * nr + 1) * 8, c.st));
        launch_tuple_sizes(q, s.tmp.p, c.st, &c.h->timing.launches);
        CUDA_CHECK_AS(what, cudaMemcpyAsync(c.n_bytes, s.off.p + 3 * nr, 8, cudaMemcpyDeviceToHost, c.st));
    }
    uint64_t n_bytes = 0;
    for (int k = 0; k < np; ++k) {
        CUDA_CHECK_AS(what, cudaSetDevice(pc[k].h->device)); CUDA_CHECK_AS(what, cudaStreamSynchronize(pc[k].st));
        if (pc[k].n_rows) nb[k] = *pc[k].n_bytes;
        n_bytes += nb[k];
    }
    const size_t off_b = (3 * n_rows + 1) * 8, rm_b = (n_rows * 12 + 7) & ~(size_t)7;
    T->host = pinned_get(off_b + rm_b + n_bytes + 64, &T->host_bytes);
    if (!T->host) { bsq_set_error("cannot allocate pinned host memory for the tuples"); return BSQ_ERR; }
    T->pub.n_rows = n_rows; T->pub.n_bytes = n_bytes; T->pub.device_ms = 0.f;
    T->pub.off = reinterpret_cast<uint64_t*>(T->host);
    T->pub.ref_match = reinterpret_cast<int32_t*>(static_cast<char*>(T->host) + off_b);
    T->pub.bytes = reinterpret_cast<uint8_t*>(static_cast<char*>(T->host) + off_b + rm_b);
    uint64_t row_base = 0, byte_base = 0;
    for (int k = 0; k < np; ++k) {
        const TuplePiece& c = pc[k]; TupleScratch& s = *c.s; const uint64_t nr = c.n_rows;
        CUDA_CHECK_AS(what, cudaSetDevice(c.h->device));
        if (nr) {
            if (cudaSuccess != s.bytes.ensure(nb[k] + 64)) { bsq_set_error("%s: out of device memory", what); return BSQ_ERR; }
            CUDA_CHECK_AS(what, cudaMemsetAsync(s.bytes.p, 0, nb[k] + 64, c.st));
            P[k].bytes = s.bytes.p;
            launch_tuple_fill(P[k], c.st, &c.h->timing.launches);
            if (byte_base) { k_add_u64<<<(unsigned)std::min<uint64_t>((3 * nr + 256) / 256, 148 * 8), 256, 0, c.st>>>(s.off.p, 3 * nr + 1, byte_base); ++c.h->timing.launches; }
            CUDA_CHECK_AS(what, cudaMemcpyAsync(T->pub.off + 3 * row_base, s.off.p, (3 * nr + 1) * 8, cudaMemcpyDeviceToHost, c.st));
            CUDA_CHECK_AS(what, cudaMemcpyAsync(T->pub.ref_match + 3 * row_base, s.rm.p, nr * 12, cudaMemcpyDeviceToHost, c.st));
            CUDA_CHECK_AS(what, cudaMemcpyAsync(T->pub.bytes + byte_base, s.bytes.p, nb[k], cudaMemcpyDeviceToHost, c.st));
        }
        CUDA_CHECK_AS(what, cudaEventRecord(e1[k], c.st));
        row_base += nr; byte_base += nb[k];
    }
    float ms = 0.f;
    for (int k = 0; k < np; ++k) {
        CUDA_CHECK_AS(what, cudaSetDevice(pc[k].h->device)); CUDA_CHECK_AS(what, cudaStreamSynchronize(pc[k].st));
        float t = 0.f;
        CUDA_CHECK_AS(what, cudaEventElapsedTime(&t, dv[dev_of[k]].e0, e1[k]));
        ms = std::max(ms, t);
    }
    CUDA_CHECK_AS(what, cudaGetLastError());
    T->pub.off[3 * n_rows] = n_bytes;
    T->pub.device_ms = ms;
    *out = &T.release()->pub;
    return BSQ_OK;
}

int bsq_result_tuples(bsq_index* h, const bsq_result* res, const char* seqs, const uint64_t* offs, uint32_t flags, bsq_tuples** out) {
    BSQ_ENTRY();
    if (!h || !res || !out) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (h->replica_pending) { bsq_set_error("replica without host state: call bsq_index_replica_finish after filling its arrays (the hole overlay of ref_subseq lives on the host)"); return BSQ_ERR; }
    {   // a result of this library whose batch is still in HBM needs no upload at all
        const ResultImpl* mine = nullptr;
        { std::lock_guard<std::mutex> lk(g_live_mu); for (const ResultImpl* r : g_live) if (&r->pub == res) { mine = r; break; } }
        if (mine && h->meta.built) {
            if (cudaSetDevice(h->device) != cudaSuccess) { bsq_set_error("cudaSetDevice failed"); return BSQ_ERR; }
            TuplePiece pc[2];
            if (const int np = resident_pieces(h, mine, pc)) return tuples_materialise(pc, np, flags, "bsq_result_tuples", out);
        }
    }
    if (!offs) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (!h->meta.built && res->n_reads && res->row_off[res->n_reads]) { bsq_set_error("index not built"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    const uint64_t n_reads = res->n_reads, n_rows = n_reads ? res->row_off[n_reads] : 0;
    if (n_rows && !seqs) { bsq_set_error("null argument"); return BSQ_ERR; }
    StagedResult S; TuplePiece pc;
    if (stage_block(h, S, res, seqs, offs, 0, n_reads, "bsq_result_tuples", pc) != BSQ_OK) return BSQ_ERR;
    return tuples_materialise(&pc, 1, flags, "bsq_result_tuples", out);
}

void bsq_tuples_free(bsq_tuples* t) { delete reinterpret_cast<TuplesImpl*>(t); }

// ---- bulk text -> NUCLSEQ (SURVEY.md 8f-4)
struct NuclseqsImpl { bsq_nuclseqs pub; void* host = nullptr; ~NuclseqsImpl() { if (host) cudaFreeHost(host); } };

int bsq_nuclseq_from_text_batch(int device, const char* text, const uint64_t* offs, uint64_t n, bsq_nuclseqs** out) {
    BSQ_ENTRY();
    if (!offs || !out || (n && !text && offs[n] != offs[0])) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (cudaSetDevice(device) != cudaSuccess) { bsq_set_error("no CUDA device %d (there is no CPU fallback)", device); return BSQ_ERR; }
    std::vector<uint64_t> rel(n + 1), chunk_off(n + 1);
    uint64_t chunks = 0;
    for (uint64_t i = 0; i <= n; ++i) {
        rel[i] = offs[i] - offs[0];
        chunk_off[i] = chunks;
        if (i < n) {
            const uint64_t len = offs[i + 1] - offs[i];
            if (len > (uint64_t)(INT32_MAX / 4)) { bsq_set_error("provided sequence is too long"); return BSQ_ERR; }   // extension.cpp:50
            chunks += (len + 15) >> 4;
        }
    }
    const uint64_t total = rel[n];
    if (chunks >= (1ull << 32) - 2 || total >= (1ull << 32)) { bsq_set_error("batch too large for one call (4 G bases at most: the ranks of ambiguous bases are 32-bit)"); return BSQ_ERR; }
    std::unique_ptr<NuclseqsImpl> S(new NuclseqsImpl());   // declared first, so freed last: the cudaFree of the buffers below waits for the device
    S->pub.n = n; S->pub.off = nullptr; S->pub.bytes = nullptr; S->pub.n_bytes = 0; S->pub.device_ms = 0.f;
    DevBuf<uint8_t> d_text, d_bytes; DevBuf<uint64_t> d_offs, d_chunk_off, d_img, d_tmp64;
    DevBuf<uint32_t> d_amb, d_start, d_holes, d_tmp32; DevBuf<unsigned long long> d_bad;
    Stream st; Event e0, e1;
    const char* me = "bsq_nuclseq_from_text_batch";
    CUDA_CHECK_AS(me, cudaStreamCreateWithFlags(&st.h, cudaStreamNonBlocking)); CUDA_CHECK_AS(me, cudaEventCreate(&e0.h)); CUDA_CHECK_AS(me, cudaEventCreate(&e1.h));
    CUDA_CHECK_AS(me, d_text.alloc(total + 64)); CUDA_CHECK_AS(me, d_offs.alloc(n + 1)); CUDA_CHECK_AS(me, d_chunk_off.alloc(n + 1)); CUDA_CHECK_AS(me, d_img.alloc(n + 2));
    CUDA_CHECK_AS(me, d_amb.alloc(chunks + 2)); CUDA_CHECK_AS(me, d_start.alloc(chunks + 2)); CUDA_CHECK_AS(me, d_holes.alloc(n + 1));
    CUDA_CHECK_AS(me, d_tmp32.alloc(loader_scan_tmp_elems(chunks))); CUDA_CHECK_AS(me, d_tmp64.alloc(loader_scan_tmp_elems(n))); CUDA_CHECK_AS(me, d_bad.alloc(1));
    cudaEventRecord(e0, st);
    if (total) CUDA_CHECK_AS(me, cudaMemcpyAsync(d_text.p, text + offs[0], total, cudaMemcpyHostToDevice, st));
    CUDA_CHECK_AS(me, cudaMemcpyAsync(d_offs.p, rel.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_CHECK_AS(me, cudaMemcpyAsync(d_chunk_off.p, chunk_off.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_CHECK_AS(me, cudaMemsetAsync(d_amb.p, 0, (chunks + 2) * 4, st)); CUDA_CHECK_AS(me, cudaMemsetAsync(d_start.p, 0, (chunks + 2) * 4, st));
    CUDA_CHECK_AS(me, cudaMemsetAsync(d_img.p, 0, (n + 2) * 8, st));
    CUDA_CHECK_AS(me, cudaMemsetAsync(d_bad.p, 0xff, 8, st));
    LoaderParams P;
    P.text = d_text.p; P.offs = d_offs.p; P.n_seqs = n; P.chunk_off = d_chunk_off.p; P.n_chunks = chunks; P.cnt_amb = d_amb.p; P.cnt_start = d_start.p;
    P.holes_num = d_holes.p; P.img_off = d_img.p; P.first_invalid = d_bad.p; P.bytes = nullptr;
    uint64_t launches = 0;
    if (n) launch_loader_scan(P, d_tmp32.p, d_tmp64.p, st, &launches);
    uint64_t n_bytes = 0; unsigned long long bad = ~0ull;
    CUDA_CHECK_AS(me, cudaMemcpyAsync(&n_bytes, d_img.p + n, 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK_AS(me, cudaMemcpyAsync(&bad, d_bad.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK_AS(me, cudaStreamSynchronize(st)); CUDA_CHECK_AS(me, cudaGetLastError());
    if (bad != ~0ull && (bad >> 63)) { bsq_set_error("sequence at text offset %llu needs a datum of 1 GiB or more (too many ambiguity runs): invalid memory alloc request size", (unsigned long long)(bad & ~(1ull << 63))); return BSQ_ERR; }
    if (bad != ~0ull) { bsq_set_error("invalid nucleotide in nuclseq_in: '%c'", text[offs[0] + bad]); return BSQ_ERR; }   // extension.cpp:53-58
    CUDA_CHECK_AS(me, d_bytes.alloc(n_bytes + 64));
    CUDA_CHECK_AS(me, cudaMemsetAsync(d_bytes.p, 0, n_bytes + 64, st));
    P.bytes = d_bytes.p;
    if (n) launch_loader_fill(P, st, &launches);
    const size_t off_b = (n + 1) * 8;
    CUDA_CHECK_AS(me, cudaHostAlloc(&S->host, off_b + n_bytes + 64, cudaHostAllocDefault));
    S->pub.off = reinterpret_cast<uint64_t*>(S->host);
    S->pub.bytes = reinterpret_cast<uint8_t*>(static_cast<char*>(S->host) + off_b);
    S->pub.n_bytes = n_bytes;
    CUDA_CHECK_AS(me, cudaMemcpyAsync(S->pub.off, d_img.p, off_b, cudaMemcpyDeviceToHost, st));
    if (n_bytes) CUDA_CHECK_AS(me, cudaMemcpyAsync(S->pub.bytes, d_bytes.p, n_bytes, cudaMemcpyDeviceToHost, st));
    cudaEventRecord(e1, st);
    CUDA_CHECK_AS(me, cudaStreamSynchronize(st)); CUDA_CHECK_AS(me, cudaGetLastError());
    cudaEventElapsedTime(&S->pub.device_ms, e0, e1);
    *out = &S.release()->pub;
    return BSQ_OK;
}

void bsq_nuclseqs_free(bsq_nuclseqs* s) { delete reinterpret_cast<NuclseqsImpl*>(s); }

void bsq_result_free(bsq_result* r) {
    if (!r) return;
    result_delete(reinterpret_cast<ResultImpl*>(r));   // pub is the first member
}

int bsq_last_timing(const bsq_index* h, bsq_timing* t) {
    BSQ_ENTRY();
    if (!h || !t) { bsq_set_error("null argument"); return BSQ_ERR; }
    *t = h->timing;
    return BSQ_OK;
}

int bsq_set_counters(bsq_index* h, int on) { if (!h) return BSQ_ERR; h->collect_counters = on != 0; return BSQ_OK; }
int bsq_get_counters(const bsq_index* h, uint64_t* out8) { if (!h || !out8) return BSQ_ERR; memcpy(out8, h->counters, sizeof(h->counters)); return BSQ_OK; }

int bsq_index_verify(bsq_index* h, uint64_t n_samples, uint64_t seed, bsq_index_check* out) {
    BSQ_ENTRY();
    if (!h || !out) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (!h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    const DevIndex ix = make_dev_index(h);
    DevBuf<unsigned long long> d; unsigned long long v[IV_WORDS];
    CUDA_CHECK(d.alloc(IV_WORDS));
    Event e0, e1; cudaEventCreate(&e0.h); cudaEventCreate(&e1.h);
    cudaEventRecord(e0, h->stream);
    const uint32_t iv = h->meta.sa_interval;
    launch_index_verify(ix, iv, n_samples, seed, 65536, d.p, h->stream);
    cudaEventRecord(e1, h->stream);
    CUDA_CHECK_AS("bsq_index_verify", cudaMemcpyAsync(v, d.p, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK_AS("bsq_index_verify", cudaStreamSynchronize(h->stream));
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    memset(out, 0, sizeof(*out));
    const uint64_t n = ix.seq_len;
    const unsigned __int128 N = n;
    // sum and sum of squares of 0..n, exact in 128 bits (n < 2^41), compared mod 2^64
    const uint64_t want_sum = (uint64_t)(N * (N + 1) / 2), want_sq = (uint64_t)(N * (N + 1) * (2 * N + 1) / 6);
    out->rows = n + 1;
    out->exhaustive = iv == 1 && n_samples >= n + 1;
    out->sa_permutation_ok = iv == 1 && v[IV_SA_SUM] == want_sum && v[IV_SA_SUMSQ] == want_sq && v[IV_SA_RANGE_BAD] == 0;
    out->sa_out_of_range = v[IV_SA_RANGE_BAD];
    out->order_checked = v[IV_ORDER_CHECKED]; out->order_bad = v[IV_ORDER_BAD]; out->order_undecided = v[IV_ORDER_UNDECIDED];
    out->rows_checked = v[IV_ROWS_CHECKED]; out->bwt_bad = v[IV_BWT_BAD]; out->lf_bad = v[IV_LF_BAD];
    out->occ_blocks_checked = v[IV_OCC_CHECKED]; out->occ_bad = v[IV_OCC_BAD];
    bool l2 = ix.L2[0] == 0;
    for (int c = 0; c < 4; ++c) l2 = l2 && ix.L2[c + 1] - ix.L2[c] == v[IV_TEXT_CNT + c] + v[IV_TEXT_CNT + 3 - c];
    out->l2_ok = l2;
    out->ms = ms;
    return BSQ_OK;
}

// the control words of the last batch's pipeline (queue sizes, tickets; layout at Batch::ctl): read after a call has ended
int bsq_debug_ctl(bsq_index* h, uint32_t* out64) {
    BSQ_ENTRY();
    if (!h || !out64 || !h->batch.ctl.p) { bsq_set_error("no batch"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    CUDA_CHECK(cudaMemcpy(out64, h->batch.ctl.p, 64 * 4, cudaMemcpyDeviceToHost));
    return BSQ_OK;
}

}  // extern "C"
static __global__ void k_sa_gather(DevIndex ix, uint64_t* rows, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) rows[i] = sa_at(ix, rows[i]);
}
extern "C" {

// bwt_sa of explicit rows: on a compact index through the resolve kernel of the alignment pipeline, so that a test can check it on
// every row against a suffix array computed elsewhere
int bsq_debug_sa_lookup(bsq_index* h, const uint64_t* rows, uint64_t n, uint64_t* out) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    if (n && (!rows || !out)) { bsq_set_error("null argument"); return BSQ_ERR; }
    if (n >= (1ull << 31)) { bsq_set_error("bsq_debug_sa_lookup: %llu rows, fewer than 2^31 per call", (unsigned long long)n); return BSQ_ERR; }
    for (uint64_t i = 0; i < n; ++i)
        if (rows[i] > h->meta.seq_len) { bsq_set_error("bsq_debug_sa_lookup: row %llu outside [0, %llu]", (unsigned long long)rows[i], (unsigned long long)h->meta.seq_len); return BSQ_ERR; }
    if (n == 0) return BSQ_OK;
    CUDA_CHECK(cudaSetDevice(h->device));
    const DevIndex ix = make_dev_index(h);
    DevBuf<uint64_t> pos; DevBuf<uint32_t> w;
    CUDA_CHECK(pos.alloc(n + 1)); CUDA_CHECK(w.alloc(2));
    CUDA_CHECK(cudaMemcpyAsync(pos.p, rows, n * 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(pos.p + n, &n, 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_CHECK(cudaMemsetAsync(w.p, 0, 8, h->stream));
    if (h->meta.sa_interval == 1) k_sa_gather<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 148 * 8), 256, 0, h->stream>>>(ix, pos.p, n);
    else launch_sa_resolve(ix, pos.p, pos.p + n, n, w.p, w.p + 1, nullptr, nullptr, h->stream);
    uint32_t err = 0;
    CUDA_CHECK_AS("bsq_debug_sa_lookup", cudaMemcpyAsync(out, pos.p, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK_AS("bsq_debug_sa_lookup", cudaMemcpyAsync(&err, w.p + 1, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK_AS("bsq_debug_sa_lookup", cudaStreamSynchronize(h->stream));
    if (err) { bsq_set_error("bsq_debug_sa_lookup: an LF walk is longer than seq_len (the index is damaged)"); return BSQ_ERR; }
    return BSQ_OK;
}

int bsq_debug_seed(bsq_index* h, const char* seqs, const uint64_t* offs, uint64_t n, uint64_t* out, uint32_t cap, uint32_t* cnt) {
    BSQ_ENTRY();
    if (!h || !h->meta.built) { bsq_set_error("index not built"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    std::vector<int64_t> ids(n, 0);
    if (upload_reads(h, h->batch, seqs, offs, ids.data(), n) != BSQ_OK) return BSQ_ERR;
    Batch& b = h->batch;
    if (ensure_kmer_table(h) != BSQ_OK) return BSQ_ERR;
    const DevIndex ix = make_dev_index(h);
    b.intv_cap = cap;
    b.list_cap = std::max<uint32_t>(b.max_len + 1, cap);
    const int seed_warps = seed_resident_warps();
    CUDA_CHECK(b.intv.ensure((size_t)n * cap)); CUDA_CHECK(b.intv_cnt.ensure(n)); CUDA_CHECK(b.seed_scratch.ensure((size_t)seed_warps * 3 * b.list_cap));
    CUDA_CHECK(b.ctl.ensure(64));
    CUDA_CHECK(cudaMemsetAsync(b.ctl.p, 0, 64 * 4, h->stream));
    CUDA_CHECK(b.seed_todo.ensure(n + 1));
    if (b.max_len <= 496) { CUDA_CHECK(b.seed_pk.ensure((size_t)n * seed_thread_words(b.max_len))); CUDA_CHECK(b.seed_u32.ensure(3 * (size_t)n)); }
    SeedParams P = seed_params(h, b, ix, (uint32_t)n, cap, b.ctl.p, reinterpret_cast<unsigned long long*>(b.ctl.p + 8));
    if (seed_thread_usable(P, h->dopts, b.max_len)) launch_seed_thread(P, ix, h->dopts, b.max_len, b.ctl.p + 60, h->stream);
    else P.todo = nullptr;
    launch_seed(P, ix, h->dopts, h->stream, nullptr);
    uint32_t ctl[8];
    CUDA_CHECK(cudaMemcpyAsync(ctl, b.ctl.p, sizeof(ctl), cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(out, b.intv.p, (size_t)n * cap * sizeof(Intv), cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(cnt, b.intv_cnt.p, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK(cudaMemcpyAsync(h->counters, b.ctl.p + 8, 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    CUDA_CHECK(cudaGetLastError());
    b.intv_cap = 0; b.resident = false;
    if (ctl[4]) { bsq_set_error("interval capacity %u too small", cap); return BSQ_ERR; }
    return BSQ_OK;
}

static int dbg_ksw_extend(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                          const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out, int mode);

int bsq_debug_ksw_extend(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                         const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out) {
    BSQ_ENTRY();
    return dbg_ksw_extend(o, device, n_jobs, q, q_off, t, t_off, w, end_bonus, h0, out, 0);
}

int bsq_debug_ksw_extend_thread(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                                const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out, int reversed) {
    BSQ_ENTRY();
    return dbg_ksw_extend(o, device, n_jobs, q, q_off, t, t_off, w, end_bonus, h0, out, reversed ? 2 : 1);
}

}  // extern "C"

// a scratch index for the debug entry points: options and a stream on the device
using TmpIndex = std::unique_ptr<bsq_index, void (*)(bsq_index*)>;

// mode 0: warp-cooperative kernel; 1 / 2: thread-per-extension kernel, query stored forward / back to front
static int dbg_ksw_extend(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                          const uint64_t* t_off, const int32_t* w, const int32_t* end_bonus, const int32_t* h0, int32_t* out, int mode) {
    TmpIndex h(bsq_index_new(o, device), bsq_index_free);
    if (!h) return BSQ_ERR;
    uint32_t max_q = 0;
    for (uint64_t i = 0; i < n_jobs; ++i) max_q = std::max<uint32_t>(max_q, (uint32_t)(q_off[i + 1] - q_off[i]));
    const int blocks = 148 * 4, warps = blocks * 4;
    const char* me = "debug extend";
    DevBuf<uint8_t> dq, dt; DevBuf<uint64_t> dqo, dto; DevBuf<int> dw, deb, dh0, dout, deh; DevBuf<uint32_t> dtk;
    CUDA_CHECK_AS(me, dq.alloc(q_off[n_jobs] + 16)); CUDA_CHECK_AS(me, dt.alloc(t_off[n_jobs] + 16));
    CUDA_CHECK_AS(me, dqo.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dto.alloc(n_jobs + 1));
    CUDA_CHECK_AS(me, dw.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, deb.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dh0.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dout.alloc(6 * n_jobs + 1));
    CUDA_CHECK_AS(me, deh.alloc((size_t)warps * 2 * (max_q + 2))); CUDA_CHECK_AS(me, dtk.alloc(16));
    CUDA_CHECK_AS(me, cudaMemset(dtk.p, 0, 64));
    CUDA_CHECK_AS(me, cudaMemcpy(dq.p, q, q_off[n_jobs], cudaMemcpyHostToDevice)); CUDA_CHECK_AS(me, cudaMemcpy(dt.p, t, t_off[n_jobs], cudaMemcpyHostToDevice));
    CUDA_CHECK_AS(me, cudaMemcpy(dqo.p, q_off, (n_jobs + 1) * 8, cudaMemcpyHostToDevice)); CUDA_CHECK_AS(me, cudaMemcpy(dto.p, t_off, (n_jobs + 1) * 8, cudaMemcpyHostToDevice));
    CUDA_CHECK_AS(me, cudaMemcpy(dw.p, w, n_jobs * 4, cudaMemcpyHostToDevice)); CUDA_CHECK_AS(me, cudaMemcpy(deb.p, end_bonus, n_jobs * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK_AS(me, cudaMemcpy(dh0.p, h0, n_jobs * 4, cudaMemcpyHostToDevice));
    if (mode == 0) launch_dbg_extend(h->dopts, (uint32_t)n_jobs, dq.p, dqo.p, dt.p, dto.p, dw.p, deb.p, dh0.p, dout.p, deh.p, max_q, dtk.p, nullptr, blocks, h->stream);
    else {
        if (max_q > (uint32_t)EXT_MEMO_MAXQ) { bsq_set_error("debug extend (thread kernel): query longer than %d", EXT_MEMO_MAXQ); return BSQ_ERR; }
        launch_dbg_extend_thread(h->dopts, (uint32_t)n_jobs, dq.p, dqo.p, dt.p, dto.p, dw.p, deb.p, dh0.p, dout.p, mode == 2, h->stream);
    }
    CUDA_CHECK_AS(me, cudaStreamSynchronize(h->stream)); CUDA_CHECK_AS(me, cudaGetLastError());
    CUDA_CHECK_AS(me, cudaMemcpy(out, dout.p, n_jobs * 24, cudaMemcpyDeviceToHost));
    return BSQ_OK;
}

extern "C" {

int bsq_debug_ksw_global(const bsq_opts* o, int device, uint64_t n_jobs, const uint8_t* q, const uint64_t* q_off, const uint8_t* t,
                         const uint64_t* t_off, const int32_t* w, int32_t* out_score, uint32_t* cigar, uint32_t cig_cap, int32_t* n_cigar) {
    BSQ_ENTRY();
    TmpIndex h(bsq_index_new(o, device), bsq_index_free);
    if (!h) return BSQ_ERR;
    uint32_t max_q = 0; size_t z_per_warp = 16;
    for (uint64_t i = 0; i < n_jobs; ++i) {
        uint32_t ql = (uint32_t)(q_off[i + 1] - q_off[i]), tl = (uint32_t)(t_off[i + 1] - t_off[i]);
        max_q = std::max<uint32_t>(max_q, ql);
        size_t ncol = std::min<size_t>(ql, 2 * (size_t)w[i] + 1);
        z_per_warp = std::max<size_t>(z_per_warp, ncol * tl + 16);
    }
    const int blocks = 148 * 2, warps = blocks * 4;
    const char* me = "debug extend";
    DevBuf<uint8_t> dq, dt, dz; DevBuf<uint64_t> dqo, dto; DevBuf<int> dw, dsc, dnc, deh; DevBuf<uint32_t> dtk, dcg;
    CUDA_CHECK_AS(me, dq.alloc(q_off[n_jobs] + 16)); CUDA_CHECK_AS(me, dt.alloc(t_off[n_jobs] + 16));
    CUDA_CHECK_AS(me, dqo.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dto.alloc(n_jobs + 1));
    CUDA_CHECK_AS(me, dw.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dsc.alloc(n_jobs + 1)); CUDA_CHECK_AS(me, dnc.alloc(n_jobs + 1));
    CUDA_CHECK_AS(me, dcg.alloc((size_t)n_jobs * cig_cap + 1));
    CUDA_CHECK_AS(me, deh.alloc((size_t)warps * 2 * (max_q + 2))); CUDA_CHECK_AS(me, dtk.alloc(16)); CUDA_CHECK_AS(me, dz.alloc((size_t)warps * z_per_warp));
    CUDA_CHECK_AS(me, cudaMemset(dtk.p, 0, 64));
    CUDA_CHECK_AS(me, cudaMemcpy(dq.p, q, q_off[n_jobs], cudaMemcpyHostToDevice)); CUDA_CHECK_AS(me, cudaMemcpy(dt.p, t, t_off[n_jobs], cudaMemcpyHostToDevice));
    CUDA_CHECK_AS(me, cudaMemcpy(dqo.p, q_off, (n_jobs + 1) * 8, cudaMemcpyHostToDevice)); CUDA_CHECK_AS(me, cudaMemcpy(dto.p, t_off, (n_jobs + 1) * 8, cudaMemcpyHostToDevice));
    CUDA_CHECK_AS(me, cudaMemcpy(dw.p, w, n_jobs * 4, cudaMemcpyHostToDevice));
    launch_dbg_global(h->dopts, (uint32_t)n_jobs, dq.p, dqo.p, dt.p, dto.p, dw.p, dsc.p, cigar ? dcg.p : nullptr, cig_cap, dnc.p, deh.p, max_q, dz.p, z_per_warp, dtk.p, blocks, h->stream);
    CUDA_CHECK_AS(me, cudaStreamSynchronize(h->stream)); CUDA_CHECK_AS(me, cudaGetLastError());
    CUDA_CHECK_AS(me, cudaMemcpy(out_score, dsc.p, n_jobs * 4, cudaMemcpyDeviceToHost));
    if (cigar) { CUDA_CHECK_AS(me, cudaMemcpy(cigar, dcg.p, (size_t)n_jobs * cig_cap * 4, cudaMemcpyDeviceToHost)); CUDA_CHECK_AS(me, cudaMemcpy(n_cigar, dnc.p, n_jobs * 4, cudaMemcpyDeviceToHost)); }
    return BSQ_OK;
}

int bsq_bench_gather(bsq_index* h, uint64_t n_loads, int reps, double* gbs) {
    BSQ_ENTRY();
    if (!h || !h->meta.built || !gbs) { bsq_set_error("index not built"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(h->device));
    // the table the random 64-byte reads go to: the largest array the seeding kernels gather from (SURVEY 8d asks for a table at least
    // the size of the index, so that the figure is an HBM number, not an L2 one): prefix table, else the full SA, else Occ
    const uint32_t* table = h->d_occ; uint64_t table_bytes = h->meta.arr_bytes[BSQ_ARR_OCC];
    if (h->meta.arr_bytes[BSQ_ARR_SA] > table_bytes) { table = reinterpret_cast<const uint32_t*>(h->d_sa); table_bytes = h->meta.arr_bytes[BSQ_ARR_SA]; }
    if (h->d_kmer && kmer_table_bytes(h->kmer_k) > table_bytes) { table = reinterpret_cast<const uint32_t*>(h->d_kmer); table_bytes = kmer_table_bytes(h->kmer_k); }
    const uint64_t n_blocks = table_bytes / 64;
    const int blocks = 148 * 8;                       // 8 CTAs of 256 threads per SM
    const uint64_t groups = (uint64_t)blocks * 256 / 16;
    uint64_t per_group = std::max<uint64_t>(8, (n_loads / groups) / 8 * 8);
    DevBuf<uint32_t> sink;
    CUDA_CHECK(sink.alloc(16));
    Event e0, e1; cudaEventCreate(&e0.h); cudaEventCreate(&e1.h);
    launch_gather(table, n_blocks, per_group, blocks, sink.p, h->stream);   // warm-up
    float best = 1e30f;
    for (int r = 0; r < reps; ++r) {
        cudaEventRecord(e0, h->stream);
        launch_gather(table, n_blocks, per_group, blocks, sink.p, h->stream);
        cudaEventRecord(e1, h->stream);
        CUDA_CHECK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        best = std::min(best, ms);
    }
    *gbs = (double)(per_group * groups) * 64.0 / (best * 1e-3) / 1e9;
    return BSQ_OK;
}

int bsq_bench_dpx(int device, int reps, double* gops) {
    BSQ_ENTRY();
    if (!gops) { bsq_set_error("null argument"); return BSQ_ERR; }
    CUDA_CHECK(cudaSetDevice(device));
    DevBuf<int> sink;
    CUDA_CHECK(sink.alloc(16));
    Event e0, e1; cudaEventCreate(&e0.h); cudaEventCreate(&e1.h);
    const int blocks = 148 * 8, iters = 4096;
    launch_dpx(iters, blocks, sink.p, 0);
    float best = 1e30f;
    for (int r = 0; r < reps; ++r) {
        cudaEventRecord(e0, 0);
        launch_dpx(iters, blocks, sink.p, 0);
        cudaEventRecord(e1, 0);
        CUDA_CHECK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        best = std::min(best, ms);
    }
    *gops = (double)blocks * 256 * (double)iters * 8.0 / (best * 1e-3) / 1e9;   // DPX instructions (per thread) per second, in G
    return BSQ_OK;
}


// ---------------------------------------------------------------------------------------- one process, several GPUs
// SURVEY.md 8b / 8e: a PostgreSQL backend is one process with one thread.  bsq_multi is that shape: ONE host thread drives every
// device with streams.  The index built on the first device is copied to the others over NVLink (peer copies of pac / Occ / SA /
// annotations + the host-side state), every device derives its own inverse SA and prefix table, a batch is cut into contiguous
// blocks of reads -- read i keeps lrand48 id i -- and the rows of all blocks land in ONE pinned result in read order.
struct bsq_multi {
    std::vector<bsq_index*> ix;      // ix[0] is the caller's (built) handle, the others are replicas owned here
    bsq_timing timing;
};

bsq_multi* bsq_multi_new(bsq_index* built, const int* devices, int n_devices) {
    BSQ_ENTRY();
    if (!built || !built->meta.built || !devices || n_devices < 1) { bsq_set_error("bsq_multi_new: a built index and a device list are needed"); return nullptr; }
    if (devices[0] != built->device) { bsq_set_error("bsq_multi_new: devices[0] must be the device the index was built on (%d)", built->device); return nullptr; }
    bsq_multi* m = new bsq_multi;
    memset(&m->timing, 0, sizeof(m->timing));
    m->ix.push_back(built);
    std::vector<uint8_t> hs(host_state_bytes(built->holes.size()));
    host_state_encode(built, hs.data());
    bool ok = true;
    for (int k = 1; k < n_devices && ok; ++k) {
        bsq_index* r = bsq_index_new(&built->opts, devices[k]);
        if (!r) { ok = false; break; }
        m->ix.push_back(r);
        r->flags = built->flags;
        if (bsq_index_alloc_replica(r, &built->meta) != BSQ_OK) { ok = false; break; }
        int can = 0;   // a repeated device: the peer copies below are device-to-device copies, no peer access to enable
        if (devices[k] != built->device) cudaDeviceCanAccessPeer(&can, devices[k], built->device);
        if (can) { cudaSetDevice(devices[k]); cudaDeviceEnablePeerAccess(built->device, 0); cudaGetLastError(); }
        for (int what = 0; what < BSQ_ARR_COUNT && ok; ++what) {
            const uint64_t nb = built->meta.arr_bytes[what];
            if (nb && cudaMemcpyPeerAsync(index_array(r, what), devices[k], index_array(built, what), built->device, nb, r->stream) != cudaSuccess) {
                bsq_set_error("bsq_multi_new: peer copy to device %d failed: %s", devices[k], cudaGetErrorString(cudaGetLastError())); ok = false;
            }
        }
    }
    for (size_t k = 1; k < m->ix.size() && ok; ++k) {
        if (bsq_index_replica_finish(m->ix[k], hs.data(), hs.size()) != BSQ_OK) { ok = false; break; }
        if (bsq_index_prepare(m->ix[k], nullptr) != BSQ_OK) ok = false;
    }
    if (ok && bsq_index_prepare(built, nullptr) != BSQ_OK) ok = false;
    if (!ok) { char keep[1024]; snprintf(keep, sizeof(keep), "%s", g_err); for (size_t k = 1; k < m->ix.size(); ++k) bsq_index_free(m->ix[k]); delete m; bsq_set_error("%s", keep); return nullptr; }
    return m;
}

void bsq_multi_free(bsq_multi* m) {
    if (!m) return;
    for (size_t k = 1; k < m->ix.size(); ++k) bsq_index_free(m->ix[k]);
    delete m;
}

int bsq_multi_devices(const bsq_multi* m) { return m ? (int)m->ix.size() : 0; }

static int multi_align(bsq_multi* m, const ReadSrc& S, uint64_t n, bsq_result** out) {
    const size_t D = m->ix.size();
    std::vector<uint64_t> lo(D + 1);
    for (size_t d = 0; d <= D; ++d) lo[d] = n * d / D;                       // contiguous blocks, as the oracle's thread sharding
    bsq_index* h0 = m->ix[0];
    const uint64_t session = h0->lrand_state;
    std::vector<Event> e0(D), e1(D);
    int rc = BSQ_OK;
    for (size_t d = 0; d < D; ++d) { cudaSetDevice(m->ix[d]->device); cudaEventCreate(&e0[d].h); cudaEventCreate(&e1[d].h); }
    // phase 1: every device's copies are queued before anything is waited for
    for (size_t d = 0; d < D && rc == BSQ_OK; ++d) {
        bsq_index* h = m->ix[d]; Batch& b = h->batch;
        cudaSetDevice(h->device);
        h->opts = h0->opts; h->dopts = h0->dopts; h->flags = h0->flags; h->lrand_state = session;
        bsq_timing& T = h->timing;
        T.launches = 0; T.h2d_bytes = T.d2h_bytes = 0; T.h2d = T.d2h = 0; T.notes = 0;
        reset_stage_timing(h);
        cudaEventRecord(e0[d], b.st);
        const uint64_t cnt = lo[d + 1] - lo[d];
        const int64_t* ids = S.ids ? S.ids + lo[d] : nullptr;
        rc = S.dbytes ? upload_datums_begin(h, b, S.dbytes, S.doff + lo[d], ids, cnt, lo[d]) : upload_reads(h, b, S.seqs, S.offs + lo[d], ids, cnt, lo[d]);
    }
    // phase 2: the kernel pipelines
    for (size_t d = 0; d < D && rc == BSQ_OK; ++d) {
        bsq_index* h = m->ix[d];
        cudaSetDevice(h->device);
        if (S.dbytes) rc = upload_datums_end(h, h->batch, lo[d + 1] > lo[d] ? S.doff[lo[d]] : 0);
        if (rc == BSQ_OK) rc = pipeline_enqueue(h, h->batch);
    }
    for (size_t d = 0; d < D && rc == BSQ_OK; ++d) { cudaSetDevice(m->ix[d]->device); rc = pipeline_finish(m->ix[d], m->ix[d]->batch); }
    // phase 3: one result, every device's rows behind the previous device's
    ResultImpl* R = nullptr;
    if (rc == BSQ_OK) {
        uint64_t rows = 0, cig = 0;
        for (size_t d = 0; d < D; ++d) { rows += m->ix[d]->batch.out_rows; cig += m->ix[d]->batch.out_cig; }
        if (cig > 0xffffffffull) { bsq_set_error("result has more CIGAR words than a 32-bit offset addresses"); rc = BSQ_ERR; }
        else { cudaSetDevice(h0->device); R = result_new(n, rows, cig, (h0->flags & BSQ_FLAG_ROWS_EXT) != 0); if (!R) rc = BSQ_ERR; }
    }
    if (rc == BSQ_OK) {
        uint64_t row_base = 0, cig_base = 0;
        std::vector<uint64_t> rb(D);
        for (size_t d = 0; d < D && rc == BSQ_OK; ++d) {
            bsq_index* h = m->ix[d]; Batch& b = h->batch;
            cudaSetDevice(h->device);
            rb[d] = row_base;
            rc = download_enqueue(h, b, R, lo[d], row_base, cig_base);
            cudaEventRecord(e1[d], b.st);
            row_base += b.out_rows; cig_base += b.out_cig;
        }
        for (size_t d = 0; d < D && rc == BSQ_OK; ++d) {
            bsq_index* h = m->ix[d]; Batch& b = h->batch;
            cudaSetDevice(h->device);
            if (cudaStreamSynchronize(b.st) != cudaSuccess) { bsq_set_error("device %d: %s", h->device, cudaGetErrorString(cudaGetLastError())); rc = BSQ_ERR; break; }
            download_finish(h, R, b.n, lo[d], b.out_rows, rb[d], b.ctl_host && b.ctl_host[10], b.ext_tmp.data());
        }
        if (rc == BSQ_OK) { R->pub.row_off[n] = row_base; R->pub.n_cigar_words = cig_base; }
    }
    // timing: a device's time runs from its first copy to the end of its download; the call's time is the slowest device's
    bsq_timing& MT = m->timing;
    memset(&MT, 0, sizeof(MT));
    for (size_t d = 0; d < D; ++d) {
        bsq_index* h = m->ix[d];
        cudaSetDevice(h->device);
        float ms = 0;
        if (rc == BSQ_OK && cudaEventElapsedTime(&ms, e0[d], e1[d]) == cudaSuccess) MT.total = std::max(MT.total, ms);
        MT.seed = std::max(MT.seed, h->timing.seed); MT.chain = std::max(MT.chain, h->timing.chain); MT.extend = std::max(MT.extend, h->timing.extend);
        MT.finalize = std::max(MT.finalize, h->timing.finalize);
        MT.launches += h->timing.launches; MT.h2d_bytes += h->timing.h2d_bytes; MT.d2h_bytes += h->timing.d2h_bytes;
        MT.notes |= h->timing.notes;   // what any device had to do differently (a table downgrade, a compaction)
    }
    cudaSetDevice(h0->device);
    if (rc != BSQ_OK) { result_delete(R); return BSQ_ERR; }
    if (!S.ids) h0->lrand_state = lrand48_advance(session, n);
    *out = &R->pub;
    return BSQ_OK;
}

int bsq_multi_align_batch(bsq_multi* m, const char* seqs, const uint64_t* offs, const int64_t* ids, uint64_t n, bsq_result** out) {
    BSQ_ENTRY();
    if (!m || !out || (n && (!seqs || !offs))) { bsq_set_error("null argument"); return BSQ_ERR; }
    const ReadSrc S{seqs, offs, nullptr, nullptr, ids};
    return multi_align(m, S, n, out);
}

int bsq_multi_align_batch_datums(bsq_multi* m, const uint8_t* bytes, const uint64_t* off, const int64_t* ids, uint64_t n, bsq_result** out) {
    BSQ_ENTRY();
    if (!m || !out || (n && (!bytes || !off))) { bsq_set_error("null argument"); return BSQ_ERR; }
    const ReadSrc S{nullptr, nullptr, bytes, off, ids};
    return multi_align(m, S, n, out);
}

int bsq_multi_last_timing(const bsq_multi* m, bsq_timing* t) {
    BSQ_ENTRY();
    if (!m || !t) { bsq_set_error("null argument"); return BSQ_ERR; }
    *t = m->timing;
    return BSQ_OK;
}

int bsq_multi_result_tuples(bsq_multi* m, const bsq_result* res, const char* seqs, const uint64_t* offs, uint32_t flags, bsq_tuples** out) {
    BSQ_ENTRY();
    if (!m || !res || !out) { bsq_set_error("null argument"); return BSQ_ERR; }
    for (const bsq_index* h : m->ix)
        if (h->replica_pending) { bsq_set_error("replica without host state: call bsq_index_replica_finish after filling its arrays (the hole overlay of ref_subseq lives on the host)"); return BSQ_ERR; }
    const ResultImpl* mine = nullptr;
    { std::lock_guard<std::mutex> lk(g_live_mu); for (const ResultImpl* r : g_live) if (&r->pub == res) { mine = r; break; } }
    // block d of the reads, as multi_align cut them: served from device d's batch while that batch still holds exactly it
    const size_t D = m->ix.size(); const uint64_t n = res->n_reads;
    std::vector<uint64_t> lo(D + 1);
    for (size_t d = 0; d <= D; ++d) lo[d] = n * d / D;
    std::vector<char> resident(D);
    bool staged = false, staged_rows = false;
    for (size_t d = 0; d < D; ++d) {
        const Batch& b = m->ix[d]->batch; const uint64_t cnt = lo[d + 1] - lo[d];
        resident[d] = cnt && mine && b.aligned && b.res_serial == mine->serial && b.res_read_base == lo[d] && b.n == cnt;
        if (!resident[d] && cnt) { staged = true; staged_rows |= res->row_off[lo[d + 1]] > (lo[d] ? res->row_off[lo[d]] : 0); }
    }
    if ((staged && !offs) || (staged_rows && !seqs)) { bsq_set_error("null argument"); return BSQ_ERR; }
    std::vector<TuplePiece> pc(D); std::vector<StagedResult> S(D);
    int rc = BSQ_OK;
    for (size_t d = 0; d < D && rc == BSQ_OK; ++d) {
        bsq_index* h = m->ix[d]; Batch& b = h->batch;
        if (resident[d]) pc[d] = TuplePiece{h, b.rows_compact.p, b.out_rows, b.cigar.p - b.cig_rebased, b.ascii.p, b.offs.p, b.row_off64.p, b.n,
                                            b.res_row_base, b.st, &b.tup, reinterpret_cast<uint64_t*>(b.ctl_host + 14), nullptr};
        else rc = stage_block(h, S[d], res, seqs, offs, lo[d], lo[d + 1] - lo[d], "bsq_multi_result_tuples", pc[d]);
    }
    if (rc == BSQ_OK) rc = tuples_materialise(pc.data(), (int)D, flags, "bsq_multi_result_tuples", out);
    cudaSetDevice(m->ix[0]->device);
    return rc;
}

}  // extern "C"
