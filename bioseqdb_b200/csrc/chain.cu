// chain.cu -- kernel `chain_build`: SA lookup of every seed occurrence, seed chaining and chain filtering
// (SURVEY.md A.5, A.6; replaces libbwa mem_chain / test_and_merge / mem_chain_weight / mem_chain_flt
// reached from reference bioseqdb/bwa.cpp:149).  One warp per read.  The SA lookups (the only HBM
// random reads here: one 4- or 8-byte load per occurrence when the full SA is resident; on a compact index
// the resolve pass of sa_resolve.cu has put every position in ChainParams::sa_pos) are issued by
// all lanes in parallel; the ordered-insert chaining itself is sequential bookkeeping on a few records.
#include "pipeline.cuh"
#include "ksort_dev.cuh"
#include "launch_cache.cuh"
#include "sa_lookup.cuh"

namespace {

constexpr int CHAIN_THREADS = 128;

// libbwa keeps chains in a B-tree keyed by pos; here: `ord` holds chain indices sorted by pos, the
// newcomer goes after its equals and lookups return the last chain with pos <= key (SURVEY A.5 corner,
// same definition as the oracle).
__device__ __forceinline__ int find_lower(const ChainTmp* ct, const uint32_t* ord, int n, int64_t key) {
    int lo = 0, hi = n;
    while (lo < hi) { int md = (lo + hi) >> 1; if (ct[ord[md]].pos <= key) lo = md + 1; else hi = md; }
    return lo;  // lower = ord[lo - 1] when lo > 0; insertion point = lo
}

__device__ __forceinline__ int chain_weight(const SeedRec* raw, const ChainTmp& c) {
    int64_t end = 0; int w = 0, tmp;
    for (int s = c.head; s >= 0; s = raw[s].next) {
        const SeedRec& q = raw[s];
        if (q.qbeg >= end) w += q.len;
        else if (q.qbeg + q.len > end) w += (int)(q.qbeg + q.len - end);
        end = end > q.qbeg + q.len ? end : q.qbeg + q.len;
    }
    tmp = w; w = 0; end = 0;
    for (int s = c.head; s >= 0; s = raw[s].next) {
        const SeedRec& q = raw[s];
        if (q.rbeg >= end) w += q.len;
        else if (q.rbeg + q.len > end) w += (int)(q.rbeg + q.len - end);
        end = end > q.rbeg + q.len ? end : q.rbeg + q.len;
    }
    w = w < tmp ? w : tmp;
    return w < 1 << 30 ? w : (1 << 30) - 1;
}

constexpr int MEM_SHORT_EXT = 50;
constexpr int MEM_SHORT_LEN = 200;
constexpr int SW_BUF_INTS = 2 * MEM_SHORT_LEN + MEM_SHORT_LEN / 4 + 8;   // boundary H, boundary F, reference window bytes

// Score of ksw_align2 (local SW, affine gaps opening from H, 16-bit kernel => no saturation at these sizes).
// Anti-diagonal wavefront: lane l owns query column 32 b + l of column block b and processes target row
// s - l at step s; H(i,j-1), F(i,j) and H(i-1,j-1) come from the left lane by shuffle, the block's last
// column is parked in shared memory for the next block.  qlen, tlen < 200.
__device__ int ksw_local_warp(const DevOpts& o, const int* smat, int qlen, const uint8_t* q, int tlen, const uint8_t* t, int* bH, int* bF) {
    const int lane = lane_id();
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins, e_del = o.e_del, e_ins = o.e_ins;
    for (int i = lane; i < tlen; i += 32) { bH[i] = 0; bF[i] = 0; }
    __syncwarp();
    int best = 0;
    for (int j0 = 0; j0 < qlen; j0 += 32) {
        const int j = j0 + lane;
        const bool col_ok = j < qlen;
        const int qb = col_ok ? (int)q[j] : 4;
        int h_up = 0, e = 0;          // H(i-1, j), E(i, j) of this lane's column
        int h_cur = 0, h_prev = 0;    // this lane's H at the previous two steps (H(i,j) and H(i-1,j) seen from the right)
        int f_out = 0;                // F(i, j+1) produced by this lane at the previous step
        for (int s = 0; s < tlen + 31; ++s) {
            const int i = s - lane;
            // values from the left neighbour (its state after step s-1): H(i, j-1) = its h_cur, H(i-1, j-1) = its h_prev, F(i, j) = its f_out
            int h_left = __shfl_up_sync(FULL, h_cur, 1), h_diag = __shfl_up_sync(FULL, h_prev, 1), f_in = __shfl_up_sync(FULL, f_out, 1);
            if (lane == 0) {
                const bool in = i >= 0 && i < tlen;
                h_left = in ? bH[i] : 0;
                h_diag = (in && i > 0) ? bH[i - 1] : 0;   // H(i-1, j0-1); the block boundary column still holds the previous block's values
                f_in = in ? bF[i] : 0;
            }
            (void)h_left;
            if (i >= 0 && i < tlen && col_ok) {
                int h = h_diag + smat[(int)t[i] * 5 + qb];
                h = h > e ? h : e;
                h = h > f_in ? h : f_in;
                h = h > 0 ? h : 0;
                best = best > h ? best : h;
                int tt = h - oe_del; tt = tt > 0 ? tt : 0;
                e -= e_del; e = e > tt ? e : tt;
                tt = h - oe_ins; tt = tt > 0 ? tt : 0;
                int f2 = f_in - e_ins; f2 = f2 > tt ? f2 : tt;
                h_prev = h_cur; h_cur = h; f_out = f2; h_up = h;
            } else { h_prev = h_cur; h_cur = 0; f_out = 0; }
            // the last column of the block becomes the next block's left boundary
            if (lane == 31 && i >= 0 && i < tlen) { bH[i] = h_cur; bF[i] = f_out; }
        }
        (void)h_up;
        __syncwarp();
    }
    return __reduce_max_sync(FULL, best);
}

// mem_seed_sw (SURVEY A.6): -1 when the seed or its +-50 bp window is long enough to be trusted
__device__ int mem_seed_sw(const DevIndex& ix, const DevOpts& o, const int* smat, int l_query, const uint8_t* query, const SeedRec& s, int* swbuf,
                           unsigned long long& cells) {
    const int64_t l_pac = ix.l_pac;
    if (s.len >= MEM_SHORT_LEN) return -1;
    int qb = s.qbeg, qe = s.qbeg + s.len;
    int64_t rb = s.rbeg, re = s.rbeg + s.len;
    const int64_t mid = (rb + re) >> 1;
    qb -= MEM_SHORT_EXT; qb = qb > 0 ? qb : 0;
    qe += MEM_SHORT_EXT; qe = qe < l_query ? qe : l_query;
    rb -= MEM_SHORT_EXT; rb = rb > 0 ? rb : 0;
    re += MEM_SHORT_EXT; re = re < (l_pac << 1) ? re : (l_pac << 1);
    if (rb < l_pac && l_pac < re) { if (mid < l_pac) re = l_pac; else rb = l_pac; }
    if (qe - qb >= MEM_SHORT_LEN || re - rb >= MEM_SHORT_LEN) return -1;
    {   // bns_fetch_seq: clamp to the row that holds mid
        int is_rev;
        const int rid = bns_pos2rid(ix, bns_depos(ix, mid, &is_rev));
        int64_t far_beg = ix.ann_offset[rid], far_end = far_beg + ix.ann_len[rid];
        if (is_rev) { const int64_t tmp = far_beg; far_beg = (l_pac << 1) - far_end; far_end = (l_pac << 1) - tmp; }
        rb = rb > far_beg ? rb : far_beg;
        re = re < far_end ? re : far_end;
        if (re < rb) re = rb;
    }
    const int tlen = (int)(re - rb), qlen = qe - qb;
    int* bH = swbuf; int* bF = swbuf + MEM_SHORT_LEN;
    uint8_t* tw = reinterpret_cast<uint8_t*>(swbuf + 2 * MEM_SHORT_LEN);
    __syncwarp();
    for (int i = lane_id(); i < tlen; i += 32) tw[i] = (uint8_t)ref_base(ix, rb + i);
    __syncwarp();
    cells += (unsigned long long)qlen * (unsigned long long)tlen;
    return ksw_local_warp(o, smat, qlen, query + qb, tlen, tw, bH, bF);
}

// ordered-insert chaining of a read's `total` seeds (raw[t].score holds the seed's rid on entry, its length on exit): returns the
// number of chains in ct[], ord[] = chain indices sorted by pos
__device__ __forceinline__ int chain_seeds(SeedRec* raw, ChainTmp* ct, uint32_t* ord, uint32_t total, const DevIndex& ix, const DevOpts& o, unsigned long long& n_dup) {
    int n_ch = 0;
    for (uint32_t t = 0; t < total; ++t) {
        SeedRec s = raw[t];
        int rid = s.score;
        if (rid < 0) continue;
        raw[t].score = s.len;
        bool to_add = true;
        int lo = 0;
        if (n_ch) {
            lo = find_lower(ct, ord, n_ch, s.rbeg);
            if (lo > 0) {
                ChainTmp& c = ct[ord[lo - 1]];
                // test_and_merge
                int64_t qend = c.l_qbeg + c.l_len, rend = c.l_rbeg + c.l_len;
                int res = 0;
                if (rid != c.rid) res = 0;
                else if (s.qbeg >= c.f_qbeg && s.qbeg + s.len <= qend && s.rbeg >= c.f_rbeg && s.rbeg + s.len <= rend) res = 1;
                else if ((c.l_rbeg < ix.l_pac || c.f_rbeg < ix.l_pac) && s.rbeg >= ix.l_pac) res = 0;
                else {
                    int64_t x = s.qbeg - c.l_qbeg, y = s.rbeg - c.l_rbeg;
                    if (y >= 0 && x - y <= o.w && y - x <= o.w && x - c.l_len < o.max_chain_gap && y - c.l_len < o.max_chain_gap) {
                        raw[c.tail].next = (int32_t)t; c.tail = (int32_t)t; ++c.n;
                        c.l_rbeg = s.rbeg; c.l_qbeg = s.qbeg; c.l_len = s.len;
                        res = 1;
                    }
                }
                if (res) to_add = false;
                else if (c.pos == s.rbeg) ++n_dup;
            }
        }
        if (to_add) {
            ChainTmp c;
            c.pos = s.rbeg; c.f_rbeg = c.l_rbeg = s.rbeg; c.f_qbeg = c.l_qbeg = s.qbeg; c.f_len = c.l_len = s.len;
            c.head = c.tail = (int32_t)t; c.n = 1; c.rid = rid; c.first = -1; c.kept = 0; c.w = 0; c.pad = 0;
            ct[n_ch] = c;
            for (int k = n_ch; k > lo; --k) ord[k] = ord[k - 1];
            ord[lo] = (uint32_t)n_ch;
            ++n_ch;
        }
    }
    return n_ch;
}

// mem_chain_flt (SURVEY A.6): ord[] is the chain array `a` in pos order on entry; returns the number of chains that passed
// min_chain_weight, ord[0 .. n) sorted by weight with ct[].kept set
__device__ __forceinline__ int chain_filter(ChainTmp* ct, uint32_t* ord, int n_ch, const DevOpts& o) {
    int n = 0;
    for (int i = 0; i < n_ch; ++i) { uint32_t c = ord[i]; if ((int)ct[c].w >= o.min_chain_weight) ord[n++] = c; }
    if (n == 0) return 0;
    const ChainTmp* ctc = ct;
    ks_introsort_dev(n, ord, [ctc](uint32_t x, uint32_t y) { return ctc[x].w > ctc[y].w; });
    // the kept list lives in ChainTmp.pad (P.ord is n_alloc wide, chains <= seeds, so [n, 2n) may not exist)
    int n_kept = 0;
    ct[ord[0]].kept = 3; ct[n_kept++].pad = 0;
    for (int i = 1; i < n; ++i) {
        ChainTmp& ci = ct[ord[i]];
        int large_ovlp = 0, k;
        int bi = ci.f_qbeg, ei = ci.l_qbeg + ci.l_len;
        for (k = 0; k < n_kept; ++k) {
            int j = (int)ct[k].pad;
            ChainTmp& cj = ct[ord[j]];
            int bj = cj.f_qbeg, ej = cj.l_qbeg + cj.l_len;
            int b_max = bj > bi ? bj : bi, e_min = ej < ei ? ej : ei;
            if (e_min > b_max) {   // is_alt is always 0 on this path (reference bwa.cpp:84-91)
                int li = ei - bi, lj = ej - bj, min_l = li < lj ? li : lj;
                if ((float)(e_min - b_max) >= __fmul_rn((float)min_l, o.mask_level) && min_l < o.max_chain_gap) {
                    large_ovlp = 1;
                    if (cj.first < 0) cj.first = i;
                    if ((float)(int)ci.w < __fmul_rn((float)(int)cj.w, o.drop_ratio) && (int)cj.w - (int)ci.w >= o.min_seed_len << 1) break;
                }
            }
        }
        if (k == n_kept) { ct[n_kept++].pad = (uint32_t)i; ci.kept = large_ovlp ? 2 : 3; }
    }
    for (int k = 0; k < n_kept; ++k) { ChainTmp& c = ct[ord[ct[k].pad]]; if (c.first >= 0) ct[ord[c.first]].kept = 1; }
    int i, k;
    for (i = k = 0; i < n; ++i) {
        int kp = ct[ord[i]].kept;
        if (kp == 0 || kp == 3) continue;
        if (++k >= o.max_chain_extend) break;
    }
    for (; i < n; ++i) if (ct[ord[i]].kept < 3) ct[ord[i]].kept = 0;
    return n;
}

// Thread per read (short reads, no seed filter): the whole of mem_chain + mem_chain_flt for a read whose intervals have at most
// CHAIN_THREAD_MAX_OCC occurrences in total -- a handful of SA reads and a few dozen records of bookkeeping, which a warp would do
// on one lane anyway.  Reads with more occurrences (repeats) are queued for the warp kernel.
constexpr uint32_t CHAIN_THREAD_MAX_OCC = 48;
__global__ void __launch_bounds__(CHAIN_THREADS) chain_build_thread(ChainParams P, DevIndex ix, DevOpts o) {
    const uint32_t r = blockIdx.x * CHAIN_THREADS + threadIdx.x;
    const int lane = lane_id();
    const bool active = r < P.n_reads;
    unsigned long long n_sa = 0, n_dup = 0;
    uint32_t total = 0; int l_rep = 0, n_iv = 0, len = 0;
    const Intv* iv = nullptr;
    if (active) {
        len = (int)(P.offs[r + 1] - P.offs[r]);
        iv = P.intv + (size_t)r * P.intv_cap;
        n_iv = (int)P.intv_cnt[r];
        int b = 0, e = 0;
        for (int i = 0; i < n_iv; ++i) {
            const uint64_t x2 = iv[i].x2;
            total += occ_count(o, x2, nullptr);
            if (x2 > (uint64_t)o.max_occ) {
                const uint64_t info = iv[i].info;
                int sb = (int)(info >> 32), se = (int)(uint32_t)info;
                if (sb > e) { l_rep += e - b; b = sb; e = se; }
                else e = e > se ? e : se;
            }
            if (total > CHAIN_THREAD_MAX_OCC) break;
        }
        l_rep += e - b;
    }
    const bool fast = active && total <= CHAIN_THREAD_MAX_OCC;
    if (active && !fast) P.todo[atomicAdd(P.todo_cnt, 1u)] = r;
    // one pool allocation per warp
    const uint32_t need = fast ? total : 0;
    uint32_t incl = need;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += v; }
    const uint32_t warp_total = __shfl_sync(FULL, incl, 31);
    uint32_t wbase = 0;
    if (lane == 31 && warp_total) wbase = atomicAdd(P.pool_top, warp_total);
    wbase = __shfl_sync(FULL, wbase, 31);
    if (fast) {
        const uint32_t base = wbase + incl - need;
        ReadBlock blk; blk.base = base; blk.n_alloc = total; blk.n_chains = 0; blk.n_seeds = 0;
        // a compact index whose batch has more lookups than position slots resolved none of them: no read chains on that attempt
        if (total == 0 || (uint64_t)base + total > (uint64_t)P.pool_cap || (P.sa_pos && P.sa_pos_off[P.n_reads] > (uint64_t)P.pool_cap)) {
            if (total) atomicExch(P.overflow, 1u);
            blk.n_alloc = 0;
            P.blocks[r] = blk;
        } else {
            SeedRec* raw = P.raw + base; ChainTmp* ct = P.ctmp + base; uint32_t* ord = P.ord + base;
            const uint64_t* pos = P.sa_pos ? P.sa_pos + P.sa_pos_off[r] : nullptr;
            for_each_lookup(iv, n_iv, o, 0u, 1u, [&](uint32_t t, const Intv& p, uint64_t row) {
                const int qb = (int)(p.info >> 32), ql = (int)((uint32_t)p.info - (uint32_t)(p.info >> 32));
                const int64_t rbeg = (int64_t)(pos ? pos[t] : sa_at(ix, row));
                SeedRec sd; sd.rbeg = rbeg; sd.qbeg = qb; sd.len = ql; sd.next = -1;
                sd.score = bns_intv2rid(ix, rbeg, rbeg + ql);
                raw[t] = sd;
            });
            n_sa += total;
            const int n_ch = chain_seeds(raw, ct, ord, total, ix, o, n_dup);
            for (int k = 0; k < n_ch; ++k) ct[k].w = (uint32_t)chain_weight(raw, ct[k]);
            const int n_flt = n_ch ? chain_filter(ct, ord, n_ch, o) : 0;
            int n_out = 0; uint32_t seed_out = 0;
            if (n_flt) {
                ChainRec* co = P.chains + base; SeedRec* so = P.seeds + base;
                const float frac_rep = (float)l_rep / len;
                for (int i = 0; i < n_flt; ++i) {
                    const ChainTmp c = ct[ord[i]];
                    if (c.kept == 0) continue;
                    ChainRec rec; rec.pos = c.pos; rec.rid = c.rid; rec.seed_off = (int32_t)seed_out; rec.kept = c.kept;
                    rec.w = c.w; rec.frac_rep = frac_rep;
                    int kept_seeds = 0;
                    for (int s = c.head; s >= 0; s = raw[s].next) { SeedRec q = raw[s]; q.next = -1; so[seed_out] = q; ++seed_out; ++kept_seeds; }
                    rec.n_seeds = kept_seeds;
                    co[n_out] = rec;
                    ++n_out;
                }
            }
            blk.n_chains = (uint32_t)n_out; blk.n_seeds = seed_out;
            P.blocks[r] = blk;
        }
    }
    if (P.counters) {
#pragma unroll
        for (int d = 16; d; d >>= 1) { n_sa += __shfl_xor_sync(FULL, n_sa, d); n_dup += __shfl_xor_sync(FULL, n_dup, d); }
        if (lane == 0) { if (n_sa) atomicAdd(&P.counters[0], n_sa); if (n_dup) atomicAdd(&P.counters[1], n_dup); }
    }
}

__global__ void __launch_bounds__(CHAIN_THREADS) chain_build(ChainParams P, DevIndex ix, DevOpts o) {
    __shared__ int smat[25];
    __shared__ int sw_smem[CHAIN_THREADS / 32][SW_BUF_INTS];
    if (threadIdx.x < 25) smat[threadIdx.x] = o.mat[threadIdx.x];
    __syncthreads();
    const int lane = lane_id();
    int* swbuf = sw_smem[threadIdx.x >> 5];
    unsigned long long n_sa = 0, n_dup = 0, n_swcells = 0;
    const uint32_t n_todo = P.todo ? *P.todo_cnt : P.n_reads;     // with the thread pass on: only the reads it queued
    for (;;) {
        const uint32_t tk = next_ticket(P.ticket);
        if (tk >= n_todo) break;
        const uint32_t r = P.todo ? P.todo[tk] : tk;
        const int len = (int)(P.offs[r + 1] - P.offs[r]);
        const Intv* iv = P.intv + (size_t)r * P.intv_cap;
        const int n_iv = (int)P.intv_cnt[r];
        // ---- occurrences per interval (count rule of the k/step loop, SURVEY A.5), frac_rep sweep
        uint32_t total = 0;
        int l_rep = 0;
        {
            int b = 0, e = 0;
            for (int i = 0; i < n_iv; ++i) {   // uniform across lanes (broadcast loads)
                uint64_t x2 = iv[i].x2;
                total += occ_count(o, x2, nullptr);
                if (x2 > (uint64_t)o.max_occ) {
                    int sb = (int)(iv[i].info >> 32), se = (int)(uint32_t)iv[i].info;
                    if (sb > e) { l_rep += e - b; b = sb; e = se; }
                    else e = e > se ? e : se;
                }
            }
            l_rep += e - b;
        }
        uint32_t base = 0;
        if (lane == 0 && total) base = atomicAdd(P.pool_top, total);
        base = __shfl_sync(FULL, base, 0);
        ReadBlock blk; blk.base = base; blk.n_alloc = total; blk.n_chains = 0; blk.n_seeds = 0;
        if (total == 0 || (uint64_t)base + total > (uint64_t)P.pool_cap || (P.sa_pos && P.sa_pos_off[P.n_reads] > (uint64_t)P.pool_cap)) {
            if (total && lane == 0) atomicExch(P.overflow, 1u);
            blk.n_alloc = 0;
            if (lane == 0) P.blocks[r] = blk;
            continue;
        }
        SeedRec* raw = P.raw + base; ChainTmp* ct = P.ctmp + base; uint32_t* ord = P.ord + base;
        // ---- SA lookups (one HBM read each).  The occurrences of up to 32 intervals are flattened over the lanes: lane i
        // holds interval i's (x0, step, count, query span), a warp scan gives each interval its slot range, and every lane
        // then looks up the owner of its slot -- a read's handful of mostly unique seeds is fetched in one pass.
        {
            uint32_t t0 = 0;
            for (int i0 = 0; i0 < n_iv; i0 += 32) {
                const int i = i0 + lane;
                uint64_t x0 = 0, step = 1; uint32_t cnt = 0, info_lo = 0, info_hi = 0;
                if (i < n_iv) {
                    const Intv p = iv[i];
                    x0 = p.x0; info_lo = (uint32_t)p.info; info_hi = (uint32_t)(p.info >> 32);
                    cnt = occ_count(o, p.x2, &step);
                }
                uint32_t incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += v; }
                const uint32_t chunk_total = __shfl_sync(FULL, incl, 31);
                for (uint32_t tb = 0; tb < chunk_total; tb += 32) {
                    const uint32_t t = tb + (uint32_t)lane;
                    // owner = number of intervals whose range ends at or before t (binary search over the inclusive sums)
                    int own = 0;
#pragma unroll
                    for (int b = 16; b > 0; b >>= 1) { const uint32_t v = __shfl_sync(FULL, incl, own + b - 1); if (v <= t) own += b; }
                    const uint32_t o_incl = __shfl_sync(FULL, incl, own), o_cnt = __shfl_sync(FULL, cnt, own);
                    const uint64_t o_x0 = __shfl_sync(FULL, x0, own), o_step = __shfl_sync(FULL, step, own);
                    const uint32_t o_lo = __shfl_sync(FULL, info_lo, own), o_hi = __shfl_sync(FULL, info_hi, own);
                    if (t < chunk_total) {
                        const uint32_t c = t - (o_incl - o_cnt);
                        const uint64_t row = lookup_row(o_x0, o_step, c);
                        const int64_t rbeg = (int64_t)(P.sa_pos ? P.sa_pos[P.sa_pos_off[r] + t0 + t] : sa_at(ix, row));
                        SeedRec sd; sd.rbeg = rbeg; sd.qbeg = (int)o_hi; sd.len = (int)(o_lo - o_hi); sd.next = -1;
                        sd.score = bns_intv2rid(ix, rbeg, rbeg + sd.len);   // rid parked in `score` until chaining
                        raw[t0 + t] = sd;
                    }
                }
                t0 += chunk_total;
                n_sa += chunk_total;
            }
        }
        __syncwarp();
        // ---- ordered-insert chaining (lane 0)
        int n_ch = 0;
        if (lane == 0) n_ch = chain_seeds(raw, ct, ord, total, ix, o, n_dup);
        n_ch = __shfl_sync(FULL, n_ch, 0);
        __syncwarp();
        // ---- weights (lanes over chains), min_chain_weight drop
        for (int k = lane; k < n_ch; k += 32) ct[k].w = (uint32_t)chain_weight(raw, ct[k]);
        __syncwarp();
        int n_out = 0, n_flt = 0; uint32_t seed_out = 0;
        if (lane == 0 && n_ch) n_flt = chain_filter(ct, ord, n_ch, o);
        n_flt = __shfl_sync(FULL, n_flt, 0);
        __syncwarp();
        // ---- emit kept chains in order with contiguous seeds; long reads first pass every short seed through
        // mem_seed_sw (local SW of the seed +-50 bp, SURVEY A.6 mem_flt_chained_seeds) on the whole warp
        if (n_flt) {
            ChainRec* co = P.chains + base; SeedRec* so = P.seeds + base;
            const float frac_rep = (float)l_rep / len;
            bool seed_sw = false; int min_HSP = 0;
            if (P.logtab) {
                const double min_l = (double)5.5f * P.logtab[len];            // MEM_MINSC_COEF * log(l_query), min_chain_weight == 0
                seed_sw = !(min_l > (double)__fmul_rn(0.05f, (float)len));   // MEM_SEEDSW_COEF * l_query is a float product
                min_HSP = (int)(o.a * min_l + .499);
            }
            const uint8_t* query = P.seqs + P.offs[r];
            for (int i = 0; i < n_flt; ++i) {
                const ChainTmp c = ct[ord[i]];
                if (c.kept == 0) continue;
                ChainRec rec; rec.pos = c.pos; rec.rid = c.rid; rec.seed_off = (int32_t)seed_out; rec.kept = c.kept;
                rec.w = c.w; rec.frac_rep = frac_rep;
                int kept_seeds = 0;
                for (int s = c.head; s >= 0; s = raw[s].next) {
                    SeedRec q = raw[s]; q.next = -1;
                    bool keep = true;
                    if (seed_sw) {
                        const int sc = mem_seed_sw(ix, o, smat, len, query, q, swbuf, n_swcells);
                        if (sc < 0 || sc >= min_HSP) q.score = sc < 0 ? q.len * o.a : sc;
                        else keep = false;
                    }
                    if (keep) { if (lane == 0) so[seed_out] = q; ++seed_out; ++kept_seeds; }
                }
                rec.n_seeds = kept_seeds;
                if (lane == 0) co[n_out] = rec;
                ++n_out;
            }
        }
        if (lane == 0) { blk.n_chains = (uint32_t)n_out; blk.n_seeds = seed_out; P.blocks[r] = blk; }
    }
    if (P.counters && lane == 0) { if (n_sa) atomicAdd(&P.counters[0], n_sa); if (n_dup) atomicAdd(&P.counters[1], n_dup); }
    if (P.sw_cells && lane == 0 && n_swcells) atomicAdd(P.sw_cells, n_swcells);
}

}  // namespace

void launch_chain_thread(const ChainParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st) {
    if (!p.todo || p.n_reads == 0) return;
    chain_build_thread<<<(p.n_reads + CHAIN_THREADS - 1) / CHAIN_THREADS, CHAIN_THREADS, 0, st>>>(p, ix, o);
}

void launch_chain(const ChainParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st) {
    const int nb = cached_blocks_per_sm(chain_build, CHAIN_THREADS, 0), sms = cached_sm_count();
    chain_build<<<nb * sms, CHAIN_THREADS, 0, st>>>(p, ix, o);
}
