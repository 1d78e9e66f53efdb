// extend_plan.cu -- thread-per-extension pre-pass of the extension stage (SURVEY.md 8a row a14: mem_chain2aln +
// ksw_extend2, libbwa as reached from reference bioseqdb/bwa.cpp:149).
//
// Almost every ksw_extend2 call of a short-read batch is the left or the right extension of the FIRST seed mem_chain2aln
// visits in a chain (the chain's best seed): its parameters depend on the chain alone, so they are known before the region
// loop runs (whether the seed is skipped as contained in an earlier region is decided later; a skipped plan is just unused).
// The first EXT_MEMO_CHAINS chains of a read are planned -- on a human-size text a read often carries a chance 20-mer hit
// next to its real chain.  `ext_plan` (thread per read) works those parameters out exactly as sw_extend would, the jobs are counting-
// sorted by query length so that the 32 lanes of a warp run extensions of the same shape, and `ext_thread_dp` runs one
// extension per thread (ksw_thread.cuh) -- first all left sides, then all right sides (a right side starts from the left
// side's score).  Results land in ExtMemo records; sw_extend picks a record up only when the call it is about to make has
// the recorded parameters, and computes everything else (further seeds, band retries, long sides) itself.
#include "pipeline.cuh"
#include "ksw_thread.cuh"
#include "launch_cache.cuh"
#include <algorithm>

namespace {

constexpr int PLAN_THREADS = 256;
constexpr int DP_THREADS = 128;
constexpr int PLAN_MAX_SEEDS = 64;      // chains with more seeds are left to sw_extend

__global__ void __launch_bounds__(PLAN_THREADS) ext_plan(ExtendParams P, DevIndex ix, DevOpts o) {
    __shared__ uint32_t hist[2][EXT_MEMO_BINS];
    for (int i = threadIdx.x; i < 2 * EXT_MEMO_BINS; i += PLAN_THREADS) (&hist[0][0])[i] = 0;
    __syncthreads();
    const uint32_t n_reads = P.n_reads;
    const size_t n_jobs = (size_t)n_reads * EXT_MEMO_CHAINS;
    const uint32_t r = blockIdx.x * PLAN_THREADS + threadIdx.x;
    if (r < n_reads) {
        const ReadBlock blk = P.blocks[r];
        const int64_t l_pac = ix.l_pac;
        const int l_query = (int)(P.offs[r + 1] - P.offs[r]);
        for (uint32_t ci = 0; ci < EXT_MEMO_CHAINS; ++ci) {
            const size_t job = (size_t)r * EXT_MEMO_CHAINS + ci;
            int kL = 0, kR = 0;
            ExtMemo mL, mR;
            mL.state = 0; mR.state = 0;
            if (ci < blk.n_chains) {
                const ChainRec c = P.chains[blk.base + ci];
                const SeedRec* seeds = P.seeds + blk.base + c.seed_off;
                const int n = c.n_seeds;
                if (n > 0 && n <= PLAN_MAX_SEEDS) {
                    // the chain's maximal span and its best seed ((score, index) maximal: the first one sw_extend's sorted walk visits)
                    int64_t rmax0 = l_pac << 1, rmax1 = 0;
                    uint64_t best = 0;
                    SeedRec s = seeds[0];
                    const int64_t rbeg0 = s.rbeg;
                    for (int i = 0; i < n; ++i) {
                        const SeedRec t = seeds[i];
                        const int64_t b = t.rbeg - (t.qbeg + cal_max_gap(o, t.qbeg));
                        const int64_t e = t.rbeg + t.len + ((l_query - t.qbeg - t.len) + cal_max_gap(o, l_query - t.qbeg - t.len));
                        rmax0 = rmax0 < b ? rmax0 : b;
                        rmax1 = rmax1 > e ? rmax1 : e;
                        const uint64_t key = (uint64_t)(uint32_t)t.score << 32 | (uint64_t)i;
                        if (key >= best) { best = key; s = t; }
                    }
                    rmax0 = rmax0 > 0 ? rmax0 : 0;
                    rmax1 = rmax1 < (l_pac << 1) ? rmax1 : (l_pac << 1);
                    if (rmax0 < l_pac && l_pac < rmax1) {
                        if (rbeg0 < l_pac) rmax1 = l_pac;
                        else rmax0 = l_pac;
                    }
                    {
                        int is_rev;
                        const int rid = bns_pos2rid(ix, bns_depos(ix, rbeg0, &is_rev));
                        int64_t far_beg = ix.ann_offset[rid], far_end = far_beg + ix.ann_len[rid];
                        if (is_rev) { const int64_t tmp = far_beg; far_beg = (l_pac << 1) - far_end; far_end = (l_pac << 1) - tmp; }
                        rmax0 = rmax0 > far_beg ? rmax0 : far_beg;
                        rmax1 = rmax1 < far_end ? rmax1 : far_end;
                        if (rmax1 < rmax0) rmax1 = rmax0;
                    }
                    const int64_t rlen = rmax1 - rmax0;
                    if (rlen <= (int64_t)P.rseq_cap) {
                        if (s.qbeg > 0 && s.qbeg <= EXT_MEMO_MAXQ) {
                            const int64_t tmp = s.rbeg - rmax0;
                            mL.tpos = s.rbeg - 1; mL.qlen = s.qbeg; mL.tlen = tmp > 0 ? (int)tmp : 0; mL.h0 = s.len * o.a; mL.state = 1;
                            kL = s.qbeg;
                        }
                        const int qe = s.qbeg + s.len;
                        if (qe != l_query && l_query - qe <= EXT_MEMO_MAXQ && (s.qbeg == 0 || kL)) {
                            const int64_t re = s.rbeg + s.len - rmax0;
                            const int64_t tl = rlen - re;
                            mR.tpos = s.rbeg + s.len; mR.qlen = l_query - qe; mR.tlen = tl > 0 ? (int)tl : 0; mR.h0 = s.len * o.a; mR.state = s.qbeg ? 3 : 1;
                            kR = l_query - qe;
                        }
                    }
                }
            }
            if (kL) P.memo[job] = mL; else P.memo[job].state = 0;
            if (kR) P.memo[n_jobs + job] = mR; else P.memo[n_jobs + job].state = 0;
            P.memo_key[job] = (uint8_t)kL;
            P.memo_key[n_jobs + job] = (uint8_t)kR;
            if (kL) atomicAdd(&hist[0][kL], 1u);
            if (kR) atomicAdd(&hist[1][kR], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * EXT_MEMO_BINS; i += PLAN_THREADS) {
        const uint32_t v = (&hist[0][0])[i];
        if (v) atomicAdd(P.memo_hist + i, v);
    }
}

// bin starts (exclusive scan of the counts) and the scatter cursors
__global__ void ext_plan_scan(uint32_t* h) {
    const int side = threadIdx.x;
    if (side >= 2) return;
    const uint32_t* cnt = h + side * EXT_MEMO_BINS;
    uint32_t* start = h + 2 * EXT_MEMO_BINS + side * EXT_MEMO_BINS;
    uint32_t* cur = h + 4 * EXT_MEMO_BINS + side * EXT_MEMO_BINS;
    uint32_t acc = 0;
    for (int k = 0; k < EXT_MEMO_BINS; ++k) { start[k] = acc; cur[k] = acc; acc += cnt[k]; }
}

__global__ void __launch_bounds__(PLAN_THREADS) ext_plan_scatter(ExtendParams P) {
    __shared__ uint32_t cnt[2][EXT_MEMO_BINS], base[2][EXT_MEMO_BINS];
    for (int i = threadIdx.x; i < 2 * EXT_MEMO_BINS; i += PLAN_THREADS) (&cnt[0][0])[i] = 0;
    __syncthreads();
    const uint32_t n = P.n_reads * EXT_MEMO_CHAINS;    // jobs: (read, chain) pairs
    const uint32_t r = blockIdx.x * PLAN_THREADS + threadIdx.x;
    int k0 = 0, k1 = 0; uint32_t my0 = 0, my1 = 0;
    if (r < n) {
        k0 = P.memo_key[r]; k1 = P.memo_key[(size_t)n + r];
        if (k0) my0 = atomicAdd(&cnt[0][k0], 1u);
        if (k1) my1 = atomicAdd(&cnt[1][k1], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * EXT_MEMO_BINS; i += PLAN_THREADS) {
        const uint32_t v = (&cnt[0][0])[i];
        if (v) (&base[0][0])[i] = atomicAdd(P.memo_hist + 4 * EXT_MEMO_BINS + i, v);
    }
    __syncthreads();
    if (k0) P.memo_perm[base[0][k0] + my0] = r;
    if (k1) P.memo_perm[(size_t)n + base[1][k1] + my1] = r;
}

// target rows straight from the 2-bit text: row i is the base at tpos + dir * i of the doubled coordinate
struct PacRows {
    const uint8_t* pac; int64_t a0; int s; uint32_t x;
    __device__ __forceinline__ int operator()(int i) const {
        const int64_t idx = a0 + (int64_t)(s * i);
        return (int)(((pac[idx >> 2] >> ((~idx & 3) << 1)) & 3u) ^ x);
    }
};

template <int NCOL>
__global__ void __launch_bounds__(DP_THREADS) ext_thread_dp(ExtendParams P, DevIndex ix, DevOpts o, int side, int key_lo, int key_hi) {
    extern __shared__ uint32_t dp_smem[];
    constexpr int NT = DP_THREADS;
    uint32_t* eh = dp_smem + threadIdx.x;
    uint32_t* qn = dp_smem + NCOL * NT + threadIdx.x;
    const uint32_t* start = P.memo_hist + 2 * EXT_MEMO_BINS + side * EXT_MEMO_BINS;
    const uint32_t lo = start[key_lo], hi = start[key_hi + 1];
    const uint32_t n = P.n_reads * EXT_MEMO_CHAINS;
    const uint32_t* perm = P.memo_perm + (size_t)side * n;
    ExtMemo* memo = P.memo + (size_t)side * n;
    uint32_t cells = 0, rows = 0;
    for (uint32_t tile = blockIdx.x; lo + tile * NT < hi; tile += gridDim.x) {
        const uint32_t k = tile * NT + threadIdx.x;     // longest jobs of the class first: the short ones fill the tail
        if (k >= hi - lo) continue;
        const uint32_t job = perm[hi - 1 - k];
        const uint32_t r = job / EXT_MEMO_CHAINS;
        ExtMemo m = memo[job];
        if (m.state == 3) {   // right side behind a left side: starts from the left side's score, unless the left side needs its band retry
            const ExtMemo& l = P.memo[job];
            if (l.state != 2 || l.out[5] >= (o.w >> 1) + (o.w >> 2)) { memo[job].state = 0; continue; }
            m.h0 = l.out[0];
        }
        const uint8_t* rq = P.seqs + P.offs[r];
        const int l_query = (int)(P.offs[r + 1] - P.offs[r]);
        int dir;
        if (side == 0) { dir = -1; ksw_thread_load_query<NT>(qn, rq + m.qlen, m.qlen, -1); }
        else { dir = 1; ksw_thread_load_query<NT>(qn, rq + (l_query - m.qlen), m.qlen, 1); }
        PacRows T;
        T.pac = ix.pac;
        if (m.tpos < ix.l_pac) { T.a0 = m.tpos; T.s = dir; T.x = 0; }
        else { T.a0 = (ix.l_pac << 1) - 1 - m.tpos; T.s = -dir; T.x = 3; }
        const ExtOut e = ksw_extend_thread<NT>(o, eh, qn, m.qlen, m.tlen, T, o.w, side == 0 ? o.pen_clip5 : o.pen_clip3, m.h0, cells, rows);
        ExtMemo* d = memo + job;
        d->h0 = m.h0;
        d->out[0] = e.score; d->out[1] = e.qle; d->out[2] = e.tle; d->out[3] = e.gtle; d->out[4] = e.gscore; d->out[5] = e.max_off;
        d->state = 2;
    }
    if (P.counters) {
        unsigned long long c = cells, w = rows;
#pragma unroll
        for (int d = 16; d; d >>= 1) { c += __shfl_xor_sync(FULL, c, d); w += __shfl_xor_sync(FULL, w, d); }
        if (lane_id() == 0 && (c | w)) { atomicAdd(&P.counters[0], c); atomicAdd(&P.counters[2], w); }
    }
}

template <int NCOL>
void launch_dp(const ExtendParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, int side, int key_lo, int key_hi, int sms) {
    constexpr size_t smem = (size_t)(NCOL + (NCOL + 6) / 8) * DP_THREADS * 4;
    const int nb = cached_blocks_per_sm(ext_thread_dp<NCOL>, DP_THREADS, smem);
    const unsigned tiles = (p.n_reads * EXT_MEMO_CHAINS + DP_THREADS - 1) / DP_THREADS;
    const unsigned grid = std::min<unsigned>(tiles, (unsigned)(nb * sms));
    ext_thread_dp<NCOL><<<grid, DP_THREADS, smem, st>>>(p, ix, o, side, key_lo, key_hi);
}

}  // namespace

// aux: three extra streams + eight events (ExtAux, owned by the batch) so that the four length classes of one side run
// concurrently -- each class alone leaves most of the chip idle in its tail.
void launch_extend_memo(const ExtendParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, uint64_t* launches, const ExtAux& aux) {
    if (!p.memo || p.n_reads == 0) return;
    const int sms = cached_sm_count();
    const unsigned blocks = (p.n_reads + PLAN_THREADS - 1) / PLAN_THREADS;
    cudaMemsetAsync(p.memo_hist, 0, 6 * EXT_MEMO_BINS * sizeof(uint32_t), st);
    ext_plan<<<blocks, PLAN_THREADS, 0, st>>>(p, ix, o);
    ext_plan_scan<<<1, 32, 0, st>>>(p.memo_hist);
    ext_plan_scatter<<<(p.n_reads * EXT_MEMO_CHAINS + PLAN_THREADS - 1) / PLAN_THREADS, PLAN_THREADS, 0, st>>>(p);
    for (int side = 0; side < 2; ++side) {
        // fork
        cudaEventRecord(aux.ev[0], st);
        for (int k = 0; k < 3; ++k) cudaStreamWaitEvent(aux.st[k], aux.ev[0], 0);
        launch_dp<97>(p, ix, o, st, side, 65, 96, sms);          // the class with most cells keeps the main stream
        launch_dp<65>(p, ix, o, aux.st[0], side, 33, 64, sms);
        launch_dp<EXT_MEMO_MAXQ + 1>(p, ix, o, aux.st[1], side, 97, EXT_MEMO_MAXQ, sms);
        launch_dp<33>(p, ix, o, aux.st[2], side, 1, 32, sms);
        // join
        for (int k = 0; k < 3; ++k) { cudaEventRecord(aux.ev[1 + k], aux.st[k]); cudaStreamWaitEvent(st, aux.ev[1 + k], 0); }
    }
    if (launches) *launches += 11;
}
