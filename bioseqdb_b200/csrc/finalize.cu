// finalize.cu -- kernel `regs_finalize`: mem_sort_dedup_patch + mem_mark_primary_se (SURVEY.md A.10) and,
// for every surviving region, mem_reg2aln: banded global alignment with traceback (ksw_global2, A.11),
// CIGAR, NM, pos / is_rev (A.12).  Replaces the libbwa calls at reference bioseqdb/bwa.cpp:149 (tail of
// mem_align1) and :158 (mem_reg2aln per region).  One warp per read.  Control flow is evaluated by all
// lanes on the same data (loads broadcast); stores are issued by lane 0 and followed by __syncwarp().
// The DP rows run on the whole warp (ksw_global_warp).  MAPQ needs libm's log() and is finished on the
// host from the fields written here (A.12).
#include "pipeline.cuh"
#include <algorithm>
#include <cstdlib>
#include "ksw_warp.cuh"
#include "ksort_dev.cuh"
#include "launch_cache.cuh"

namespace {

constexpr int FIN_THREADS = 128;
constexpr int FIN_WARPS = FIN_THREADS / 32;
// thread-per-region routing limits (narrow_class): band columns of a first try, target rows, query length
constexpr int NARROW_NC = 64;
constexpr int NARROW_TMAX = 192;
constexpr int NARROW_QMAX = 160;
constexpr int NARROW_THREADS = 128;
constexpr int NARROW_CIG = 48;

struct NarrowJob { uint32_t r, slot; int32_t w2, last_sc, it, score; };   // one pending try of mem_reg2aln's band-doubling loop

struct FScratch { int* ehh; int* ehe; uint8_t* rseq; uint8_t* query; uint8_t* z; uint32_t* cig; };

__device__ __forceinline__ uint64_t hash_64(uint64_t key) {
    key += ~(key << 32); key ^= (key >> 22); key += ~(key << 13); key ^= (key >> 8);
    key += (key << 3); key ^= (key >> 15); key += ~(key << 27); key ^= (key >> 31);
    return key;
}

__device__ __forceinline__ int infer_bw(int l1, int l2, int score, int a, int q, int r) {
    int w;
    if (l1 == l2 && l1 * a - score < (q + r - a) << 1) return 0;
    w = (int)((double)((l1 < l2 ? l1 : l2) * a - score - q) / r + 2.);
    int d = l1 - l2; d = d < 0 ? -d : d;
    if (w < d) w = d;
    return w;
}

struct GenOut { int ok, score, n_cigar, NM; };

// bwa_gen_cigar2 (SURVEY A.11).  Query segment q[0..l_query) (forward orientation in scratch), reference
// [rb, re).  WANT_CIGAR: traceback into S.cig (forward order) and NM.
template <bool WANT_CIGAR>
__device__ GenOut gen_cigar2(const DevIndex& ix, const DevOpts& o, const int* smat, int w_, int l_query, const uint8_t* q, int64_t rb, int64_t re,
                             const FScratch& S, uint32_t rseq_cap, uint32_t z_cap, uint32_t cig_cap, uint32_t* overflow, uint32_t* need_rseq,
                             unsigned long long& cells, unsigned long long& calls) {
    const int lane = lane_id();
    const int64_t l_pac = ix.l_pac;
    GenOut g; g.ok = 0; g.score = 0; g.n_cigar = 0; g.NM = -1;
    if (l_query <= 0 || rb >= re || (rb < l_pac && re > l_pac)) return g;
    // bns_get_seq clamps to [0, 2 l_pac); a clamped fetch makes libbwa bail out (re - rb != rlen)
    if (rb < 0 || re > (l_pac << 1)) return g;
    const int64_t rlen64 = re - rb;
    if (rlen64 > (int64_t)rseq_cap) { if (lane == 0) atomicMax(need_rseq, (uint32_t)(rlen64 < 0x7fffffff ? rlen64 : 0x7fffffff)); return g; }
    const int rlen = (int)rlen64;
    for (int i = lane; i < rlen; i += 32) S.rseq[i] = (uint8_t)ref_base(ix, rb + i);
    __syncwarp();
    // reverse strand: libbwa reverses both sequences so that gaps are left-aligned on the forward strand
    const bool rev = rb >= l_pac;
    const uint8_t* qp = rev ? q + l_query - 1 : q; const int qs = rev ? -1 : 1;
    const uint8_t* tp = rev ? S.rseq + rlen - 1 : S.rseq; const int ts = rev ? -1 : 1;
    g.ok = 1;
    if (l_query == rlen && w_ == 0) {   // no gap: no DP
        int sc = 0;
        for (int i = lane; i < l_query; i += 32) sc += smat[(int)tp[(long)i * ts] * 5 + qp[(long)i * qs]];
        sc = __reduce_add_sync(FULL, sc);
        g.score = sc;
        if (WANT_CIGAR) { if (lane == 0) S.cig[0] = (uint32_t)l_query << 4; g.n_cigar = 1; __syncwarp(); }
    } else {
        int w, max_gap, max_ins, max_del, min_w;
        max_ins = (int)((double)(((l_query + 1) >> 1) * o.mat[0] - o.o_ins) / o.e_ins + 1.);
        max_del = (int)((double)(((l_query + 1) >> 1) * o.mat[0] - o.o_del) / o.e_del + 1.);
        max_gap = max_ins > max_del ? max_ins : max_del;
        max_gap = max_gap > 1 ? max_gap : 1;
        int dl = rlen - l_query; dl = dl < 0 ? -dl : dl;
        w = (max_gap + dl + 1) >> 1;
        w = w < w_ ? w : w_;
        min_w = dl + 3;
        w = w > min_w ? w : min_w;
        const int n_col = l_query < 2 * w + 1 ? l_query : 2 * w + 1;
        uint8_t* z = nullptr;
        if (WANT_CIGAR) {
            if ((uint64_t)n_col * (uint64_t)rlen > (uint64_t)z_cap) { if (lane == 0) atomicExch(overflow, 2u); g.ok = 0; return g; }
            z = S.z;
        }
        ++calls;
        g.score = ksw_global_warp(o, l_query, qp, qs, rlen, tp, ts, w, S.ehh, S.ehe, smat, z, n_col, cells);
        if (WANT_CIGAR) {
            int n_cigar = 0;
            if (lane == 0) {   // traceback: a dependent walk over one byte per step
                int which = 0, i = rlen - 1, k = (i + w + 1 < l_query ? i + w + 1 : l_query) - 1;
                uint32_t* cg = S.cig;   // built backwards, then reversed
                auto push = [&](uint32_t op, uint32_t len) {
                    if (n_cigar == 0 || op != (cg[n_cigar - 1] & 0xf)) { if ((uint32_t)n_cigar < cig_cap) cg[n_cigar] = len << 4 | op; ++n_cigar; }
                    else cg[n_cigar - 1] += len << 4;
                };
                while (i >= 0 && k >= 0) {
                    which = z[(size_t)i * n_col + (k - (i > w ? i - w : 0))] >> (which << 1) & 3;
                    if (which == 0) { push(0, 1); --i; --k; }
                    else if (which == 1) { push(2, 1); --i; }
                    else { push(1, 1); --k; }
                }
                if (i >= 0) push(2, (uint32_t)(i + 1));
                if (k >= 0) push(1, (uint32_t)(k + 1));
                if ((uint32_t)n_cigar > cig_cap) { atomicExch(overflow, 2u); n_cigar = 0; }
                for (int a = 0; a < n_cigar >> 1; ++a) { uint32_t t = cg[a]; cg[a] = cg[n_cigar - 1 - a]; cg[n_cigar - 1 - a] = t; }
            }
            g.n_cigar = __shfl_sync(FULL, n_cigar, 0);
            __syncwarp();
        }
    }
    if (WANT_CIGAR) {   // NM (MD is not exported by the reference adapter)
        int x = 0, y = 0, n_mm = 0, n_gap = 0;
        for (int k = 0; k < g.n_cigar; ++k) {
            const uint32_t cw = S.cig[k];
            const int op = (int)(cw & 0xf), len = (int)(cw >> 4);
            if (op == 0) {
                for (int i = lane; i < len; i += 32) n_mm += qp[(long)(x + i) * qs] != tp[(long)(y + i) * ts];
                x += len; y += len;
            } else if (op == 2) {
                if (k > 0 && k < g.n_cigar - 1) n_gap += len;
                y += len;
            } else if (op == 1) { x += len; n_gap += len; }
        }
        n_mm = __reduce_add_sync(FULL, n_mm);
        g.NM = n_mm + n_gap;
    }
    return g;
}

// mem_patch_reg (SURVEY A.10); a = earlier region, b = later region
__device__ int patch_reg(const DevIndex& ix, const DevOpts& o, const int* smat, const uint8_t* query, const RegRec& a, const RegRec& b, int* _w,
                         const FScratch& S, uint32_t rseq_cap, uint32_t* overflow, uint32_t* need_rseq, unsigned long long& cells, unsigned long long& calls) {
    int w, score, q_s, r_s;
    double r;
    if (a.rb < ix.l_pac && b.rb >= ix.l_pac) return 0;
    if (a.qb >= b.qb || a.qe >= b.qe || a.re >= b.re) return 0;
    w = (int)((a.re - b.rb) - (a.qe - b.qb));
    w = w > 0 ? w : -w;
    r = (double)(a.re - b.rb) / (double)(b.re - a.rb) - (double)(a.qe - b.qb) / (double)(b.qe - a.qb);
    r = r > 0. ? r : -r;
    if (a.re < b.rb || a.qe < b.qb) {
        if (w > o.w << 1 || r >= (double)0.05f) return 0;
    } else if (w > o.w << 2 || r >= (double)(0.05f * 2)) return 0;
    w += a.w + b.w;
    w = w < o.w << 2 ? w : o.w << 2;
    GenOut g = gen_cigar2<false>(ix, o, smat, w, b.qe - a.qb, query + a.qb, a.rb, b.re, S, rseq_cap, 0, 0, overflow, need_rseq, cells, calls);
    score = g.score;
    q_s = (int)((double)(b.qe - a.qb) / (double)((b.qe - b.qb) + (a.qe - a.qb)) * (double)(b.score + a.score) + .499);
    r_s = (int)((double)(b.re - a.rb) / (double)((b.re - b.rb) + (a.re - a.rb)) * (double)(b.score + a.score) + .499);
    if ((double)score / (double)(q_s > r_s ? q_s : r_s) < (double)0.90f) return 0;
    *_w = w;
    return score;
}

__device__ __forceinline__ RowDev row_from_reg(const RegRec& ar, const int64_t* ann_id) {
    RowDev row;
    row.rb = ar.rb; row.re = ar.re; row.pos = 0; row.hash = ar.hash; row.qb = ar.qb; row.qe = ar.qe; row.rid = ar.rid; row.score = ar.score;
    row.truesc = ar.truesc; row.sub = ar.sub; row.csub = ar.csub; row.sub_n = ar.sub_n; row.w = ar.w; row.seedcov = ar.seedcov;
    row.secondary = ar.secondary; row.seedlen0 = ar.seedlen0; row.n_comp = ar.n_comp; row.frac_rep = ar.frac_rep;
    row.is_rev = 0; row.mapq = 0;   // mapq is filled on the host (mem_approx_mapq_se needs libm log)
    row.NM = -1; row.flag = ar.secondary >= 0 ? 0x100 : 0; row.cigar_off = 0; row.n_cigar = 0;
    row.ref_id = ann_id[ar.rid];
    return row;
}

__device__ __forceinline__ int reg2aln_w2(const DevOpts& o, const RegRec& ar) {
    const int qb = ar.qb, qe = ar.qe; const int64_t rb = ar.rb, re = ar.re;
    int tmpw = infer_bw(qe - qb, (int)(re - rb), ar.truesc, o.a, o.o_del, o.e_del);
    int w2 = infer_bw(qe - qb, (int)(re - rb), ar.truesc, o.a, o.o_ins, o.e_ins);
    w2 = w2 > tmpw ? w2 : tmpw;
    if (w2 > o.w) w2 = w2 < ar.w ? w2 : ar.w;
    return w2;
}

// effective band of bwa_gen_cigar2 for a requested w_ (SURVEY A.11)
__device__ __forceinline__ int gen_cigar_band(const DevOpts& o, int l_query, int rlen, int w_) {
    int max_ins = (int)((double)(((l_query + 1) >> 1) * o.mat[0] - o.o_ins) / o.e_ins + 1.);
    int max_del = (int)((double)(((l_query + 1) >> 1) * o.mat[0] - o.o_del) / o.e_del + 1.);
    int max_gap = max_ins > max_del ? max_ins : max_del;
    max_gap = max_gap > 1 ? max_gap : 1;
    int dl = rlen - l_query; dl = dl < 0 ? -dl : dl;
    int w = (max_gap + dl + 1) >> 1;
    w = w < w_ ? w : w_;
    const int min_w = dl + 3;
    return w > min_w ? w : min_w;
}

// A job list holds both classes of thread-per-region work so that the lanes of a warp do similar work: regions whose band
// fits the register window (w <= REG_WT) grow from the front, wider ones (the wide register kernel, w <= REG_WT2) from the back.
constexpr int REG_WT = 16;
// tight first tries: MODE 4 runs a 9-column window, MODE 3 a 17-column one; a result is accepted only when no path that leaves
// the window can reach the score found inside it (lists T4 -> T8 -> A)
constexpr uint32_t NARROW_SHORT_LIST = 1024;
constexpr int REG_WT3 = 8;
constexpr int REG_WT4 = 4;
constexpr int NARROW_T4_CNT = 20, NARROW_T8_CNT = 21;   // counters of lists T4 / T8 behind narrow_cnt (ctl words 52, 53)
constexpr int REG_WT2 = 32;   // second register kernel: bands of half-width 17..32 (65 columns of H and E in registers, 2 CTAs per SM)
__device__ __forceinline__ bool narrow_is_big(const DevOpts& o, int lq, int rlen, int w2) {
    w2 = w2 < o.w << 2 ? w2 : o.w << 2;
    return gen_cigar_band(o, lq, rlen, w2) > REG_WT;
}
// the tight pass takes a region when the register kernels can score it and the end cell lies inside the tight window
__device__ __forceinline__ bool narrow_is_tight(const DevOpts& o, int lq, int rlen, int wt = REG_WT3) {
    const int dl = lq - rlen;
    return (dl < 0 ? -dl : dl) <= wt && o.o_del >= 0 && o.e_del >= 0 && o.o_ins >= 0 && o.e_ins >= 0 && o.mat_max > 0;
}
// 0: align on the warp here; 1: thread-per-region narrow-band DP; 2: thread-per-region, no DP (equal lengths, zero band).
// A region whose band is wider than any thread kernel's still gets its first try there when the tight passes can take it (their
// proof does not care how wide the band asked for is; a region they cannot settle travels on to the exact-band lists, whose
// kernels hand a band they do not hold to the warp-cooperative one).
__device__ __forceinline__ int narrow_class(const DevOpts& o, const RegRec& ar, uint32_t max_len) {
    const int lq = ar.qe - ar.qb; const int64_t rl = ar.re - ar.rb;
    if (max_len > NARROW_QMAX || lq <= 0 || rl <= 0 || rl > NARROW_TMAX) return 0;
    int w2 = reg2aln_w2(o, ar);
    w2 = w2 < o.w << 2 ? w2 : o.w << 2;
    if (lq == rl) return 2;   // equal lengths: first a thread checks whether the gap-free diagonal is provably the unique optimum
    if (2 * gen_cigar_band(o, lq, (int)rl, w2) + 1 <= NARROW_NC) return 1;
    return narrow_is_tight(o, lq, (int)rl) ? 1 : 0;
}
__device__ __forceinline__ void push_narrow(NarrowJob* list, uint32_t cap, uint32_t* cnt_reg, uint32_t* cnt_big, const NarrowJob& jb, bool big) {
    if (big) list[cap - 1u - atomicAdd(cnt_big, 1u)] = jb;
    else list[atomicAdd(cnt_reg, 1u)] = jb;
}

// mem_reg2aln (SURVEY A.12) for one region on the whole warp; completes *out (NM, pos, is_rev, CIGAR)
__device__ void reg2aln_warp(const FinalizeParams& P, const DevIndex& ix, const DevOpts& o, const int* smat, const FScratch& S, uint32_t cig_cap,
                             uint32_t rseq_cap, int l_query, const RegRec& ar, RowDev* out, unsigned long long& cells, unsigned long long& calls) {
    const int lane = lane_id();
    const int qb = ar.qb, qe = ar.qe; const int64_t rb = ar.rb, re = ar.re;
    int w2 = reg2aln_w2(o, ar);
    int it = 0, score = 0, last_sc = -(1 << 30);
    GenOut g;
    do {
        w2 = w2 < o.w << 2 ? w2 : o.w << 2;
        g = gen_cigar2<true>(ix, o, smat, w2, qe - qb, S.query + qb, rb, re, S, rseq_cap, P.z_cap, cig_cap - 2, P.overflow, P.need_rseq, cells, calls);
        if (g.ok) score = g.score;
        if (score == last_sc || w2 == o.w << 2) break;
        last_sc = score;
        w2 <<= 1;
    } while (++it < 3 && score < ar.truesc - o.a);
    int is_rev;
    int64_t pos = bns_depos(ix, rb < ix.l_pac ? rb : re - 1, &is_rev);
    // squeeze out a leading or trailing deletion, add soft clips, publish the CIGAR
    int n_cigar = g.n_cigar, first = 0;
    if (n_cigar > 0) {
        if ((S.cig[0] & 0xf) == 2) { pos += S.cig[0] >> 4; first = 1; --n_cigar; }
        else if ((S.cig[g.n_cigar - 1] & 0xf) == 2) --n_cigar;
    }
    int clip5 = 0, clip3 = 0;
    if (qb != 0 || qe != l_query) { clip5 = is_rev ? l_query - qe : qb; clip3 = is_rev ? qb : l_query - qe; }
    const int n_out = n_cigar + (clip5 ? 1 : 0) + (clip3 ? 1 : 0);
    uint32_t coff = 0;
    if (lane == 0 && n_out) coff = atomicAdd(P.cigar_top, (uint32_t)n_out);
    coff = __shfl_sync(FULL, coff, 0);
    uint32_t r_off = 0, r_n = 0;
    if ((uint64_t)coff + (uint64_t)n_out > (uint64_t)P.cigar_cap) { if (lane == 0) atomicExch(P.overflow, 1u); }
    else {
        r_off = coff; r_n = (uint32_t)n_out;
        if (lane == 0) {
            uint32_t* dst = P.cigar_pool + coff;
            int k = 0;
            if (clip5) dst[k++] = (uint32_t)clip5 << 4 | 3;
            for (int c = 0; c < n_cigar; ++c) dst[k++] = S.cig[first + c];
            if (clip3) dst[k++] = (uint32_t)clip3 << 4 | 3;
        }
    }
    const int rid = bns_pos2rid(ix, pos);
    if (lane == 0) {
        out->NM = g.NM; out->is_rev = is_rev; out->cigar_off = r_off; out->n_cigar = r_n;
        out->pos = pos - ix.ann_offset[rid < 0 ? 0 : rid];
    }
    __syncwarp();
}

// Thread per read: the phase-1 work of a read with ONE region that the thread-per-region kernels can align (no dedup / patch to
// do; mem_mark_primary_se of a single region is three assignments) -- the common case of a short-read batch.  Every other read
// is queued for regs_finalize.  Job-list slots are claimed once per warp and list.
__global__ void __launch_bounds__(128) regs_finalize_thread(FinalizeParams P, DevIndex ix, DevOpts o) {
    const uint32_t r = blockIdx.x * 128 + threadIdx.x;
    const int lane = lane_id();
    int cat = 0;      // 0 nothing to push, 1 register-band DP job, 2 wide-band DP job, 3 no-DP job, 4 / 5 tight first try (9 / 17 columns)
    NarrowJob jb; jb.r = r; jb.slot = 0; jb.w2 = 0; jb.last_sc = -(1 << 30); jb.it = 0; jb.score = 0;
    if (r < P.n_reads) {
        const ReadBlock blk = P.blocks[r];
        const int n = blk.n_alloc ? (int)P.reg_cnt[r] : 0;
        bool done = false;
        if (n == 0) { P.row_cnt[r] = 0; done = true; }
        else if (n == 1) {
            RegRec ar = P.regs[blk.base];
            const int ncls = narrow_class(o, ar, P.max_len);
            if (ncls != 0) {
                ar.sub = 0; ar.secondary = -1; ar.hash = hash_64((uint64_t)P.ids[r]);      // mem_mark_primary_se, n == 1
                P.regs[blk.base] = ar;
                P.rows[blk.base] = row_from_reg(ar, P.ann_id);
                jb.slot = blk.base; jb.w2 = reg2aln_w2(o, ar);
                if (ncls == 1) {
                    if (narrow_is_tight(o, ar.qe - ar.qb, (int)(ar.re - ar.rb))) cat = narrow_is_tight(o, ar.qe - ar.qb, (int)(ar.re - ar.rb), REG_WT4) ? 4 : 5;
                    else cat = narrow_is_big(o, ar.qe - ar.qb, (int)(ar.re - ar.rb), jb.w2) ? 2 : 1;
                } else cat = 3;
                P.row_cnt[r] = 1;
                done = true;
            }
        }
        if (!done) P.todo[atomicAdd(P.todo_cnt, 1u)] = r;
    }
    NarrowJob* lists = reinterpret_cast<NarrowJob*>(P.narrow_jobs);
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int c = 1; c <= 5; ++c) {
        const uint32_t mask = __ballot_sync(FULL, cat == c);
        if (!mask) continue;
        uint32_t base = 0;
        if (lane == __ffs(mask) - 1) base = atomicAdd(P.narrow_cnt + (c == 1 ? 0 : (c == 2 ? 5 : (c == 3 ? 3 : (c == 4 ? NARROW_T4_CNT : NARROW_T8_CNT)))), (uint32_t)__popc(mask));
        base = __shfl_sync(FULL, base, __ffs(mask) - 1);
        if (cat == c) {
            const uint32_t k = base + (uint32_t)__popc(mask & lt);
            if (c == 1) lists[k] = jb;
            else if (c == 2) lists[P.narrow_cap - 1u - k] = jb;
            else if (c == 3) lists[2u * P.narrow_cap + k] = jb;
            else lists[(c == 4 ? 3u : 4u) * P.narrow_cap + k] = jb;
        }
    }
}

template <bool SMEM>
__global__ void __launch_bounds__(FIN_THREADS, 6) regs_finalize(FinalizeParams P, DevIndex ix, DevOpts o, uint32_t cig_cap, uint32_t rseq_cap) {
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    __shared__ int smat[25];
    if (threadIdx.x < 25) smat[threadIdx.x] = o.mat[threadIdx.x];
    __syncthreads();
    const int lane = lane_id();
    const uint32_t gwarp = (blockIdx.x * FIN_THREADS + threadIdx.x) >> 5;
    FScratch S;
    {
        // fast part (DP rows, sequences) optionally in shared memory; z and the cigar buffer stay in global scratch
        const size_t fast = ((size_t)(P.max_len + 2) * 8 + rseq_cap + P.max_len + 15) & ~(size_t)15;
        uint8_t* gbase = P.scratch + (size_t)gwarp * P.scratch_per_warp;
        uint8_t* fbase = SMEM ? dyn_smem + (size_t)(threadIdx.x >> 5) * fast : gbase;
        S.ehh = reinterpret_cast<int*>(fbase);
        S.ehe = S.ehh + (P.max_len + 2);
        S.rseq = reinterpret_cast<uint8_t*>(S.ehe + (P.max_len + 2));
        S.query = S.rseq + rseq_cap;
        S.cig = reinterpret_cast<uint32_t*>(gbase + fast);
        S.z = reinterpret_cast<uint8_t*>(S.cig + cig_cap);
    }
    unsigned long long cells = 0, calls = 0;
    const uint32_t n_todo = P.todo ? *P.todo_cnt : P.n_reads;     // with the thread pass on: only the reads it queued
    for (;;) {
        const uint32_t tk = next_ticket(P.ticket);
        if (tk >= n_todo) break;
        const uint32_t r = P.todo ? P.todo[tk] : tk;
        const ReadBlock blk = P.blocks[r];
        int n = blk.n_alloc ? (int)P.reg_cnt[r] : 0;
        if (n == 0) { if (lane == 0) P.row_cnt[r] = 0; continue; }
        const int l_query = (int)(P.offs[r + 1] - P.offs[r]);
        {
            const uint8_t* qg = P.seqs + P.offs[r];
            for (int i = lane; i < l_query; i += 32) S.query[i] = qg[i];
        }
        RegRec* a = P.regs + blk.base;
        __syncwarp();
        // ---------------- mem_sort_dedup_patch
        if (n > 1) {
            if (lane == 0) {
                ks_introsort_dev(n, a, [](const RegRec& x, const RegRec& y) { return x.re < y.re; });
                for (int i = 0; i < n; ++i) a[i].n_comp = 1;
            }
            __syncwarp();
            for (int i = 1; i < n; ++i) {
                if (a[i].rid != a[i - 1].rid || a[i].rb >= a[i - 1].re + o.max_chain_gap) continue;
                for (int j = i - 1; j >= 0 && a[i].rid == a[j].rid && a[i].rb < a[j].re + o.max_chain_gap; --j) {
                    const RegRec p = a[i], q = a[j];
                    int64_t orr, oq, mr, mq;
                    int score, w;
                    if (q.qe == q.qb) continue;
                    orr = q.re - p.rb;
                    oq = q.qb < p.qb ? q.qe - p.qb : p.qe - q.qb;
                    mr = q.re - q.rb < p.re - p.rb ? q.re - q.rb : p.re - p.rb;
                    mq = q.qe - q.qb < p.qe - p.qb ? q.qe - q.qb : p.qe - p.qb;
                    if ((float)orr > __fmul_rn(o.mask_level_redun, (float)mr) && (float)oq > __fmul_rn(o.mask_level_redun, (float)mq)) {
                        if (p.score < q.score) {
                            if (lane == 0) a[i].qe = p.qb;
                            __syncwarp();
                            break;
                        } else {
                            if (lane == 0) a[j].qe = q.qb;
                            __syncwarp();
                        }
                    } else if (q.rb < p.rb && (score = patch_reg(ix, o, smat, S.query, q, p, &w, S, rseq_cap, P.overflow, P.need_rseq, cells, calls)) > 0) {
                        if (lane == 0) {
                            RegRec& pp = a[i];
                            pp.n_comp += q.n_comp + 1;
                            pp.seedcov = p.seedcov > q.seedcov ? p.seedcov : q.seedcov;
                            pp.sub = p.sub > q.sub ? p.sub : q.sub;
                            pp.csub = p.csub > q.csub ? p.csub : q.csub;
                            pp.qb = q.qb; pp.rb = q.rb;
                            pp.truesc = pp.score = score;
                            pp.w = w;
                            a[j].qb = q.qe;
                        }
                        __syncwarp();
                    }
                }
            }
            int m = 0;
            if (lane == 0) {
                for (int i = 0; i < n; ++i)
                    if (a[i].qe > a[i].qb) { if (m != i) a[m++] = a[i]; else ++m; }
                n = m;
                ks_introsort_dev(n, a, [](const RegRec& x, const RegRec& y) {
                    return x.score > y.score || (x.score == y.score && (x.rb < y.rb || (x.rb == y.rb && x.qb < y.qb)));
                });
                for (int i = 1; i < n; ++i)
                    if (a[i].score == a[i - 1].score && a[i].rb == a[i - 1].rb && a[i].qb == a[i - 1].qb) a[i].qe = a[i].qb;
                m = n < 1 ? 0 : 1;
                for (int i = 1; i < n; ++i)
                    if (a[i].qe > a[i].qb) { if (m != i) a[m++] = a[i]; else ++m; }
            }
            n = __shfl_sync(FULL, m, 0);
            __syncwarp();
        }
        // ---------------- mem_mark_primary_se
        if (lane == 0 && n > 0) {
            const int64_t id = P.ids[r];
            for (int i = 0; i < n; ++i) { a[i].sub = 0; a[i].secondary = -1; a[i].hash = hash_64((uint64_t)(id + i)); }
            ks_introsort_dev(n, a, [](const RegRec& x, const RegRec& y) { return x.score > y.score || (x.score == y.score && x.hash < y.hash); });
            int tmp = o.a + o.b;
            tmp = o.o_del + o.e_del > tmp ? o.o_del + o.e_del : tmp;
            tmp = o.o_ins + o.e_ins > tmp ? o.o_ins + o.e_ins : tmp;
            // z list: indices of non-secondary regions, kept in the (not yet used) n_comp-free field `secondary` of ...
            // simple: the list is a prefix-ordered subset; store it in the csub field of slot k (csub is 0 on this path
            // except after a patch merge, so keep a copy and restore)
            int nz = 0;
            // use the cigar scratch as the z list (free at this point)
            uint32_t* zl = S.cig;
            zl[nz++] = 0;
            for (int i = 1; i < n; ++i) {
                int k;
                for (k = 0; k < nz; ++k) {
                    const int j = (int)zl[k];
                    const int b_max = a[j].qb > a[i].qb ? a[j].qb : a[i].qb;
                    const int e_min = a[j].qe < a[i].qe ? a[j].qe : a[i].qe;
                    if (e_min > b_max) {
                        const int li = a[i].qe - a[i].qb, lj = a[j].qe - a[j].qb;
                        const int min_l = li < lj ? li : lj;
                        if ((float)(e_min - b_max) >= __fmul_rn((float)min_l, o.mask_level)) {
                            if (a[j].sub == 0) a[j].sub = a[i].score;
                            if (a[j].score - a[i].score <= tmp) ++a[j].sub_n;
                            break;
                        }
                    }
                }
                if (k == nz) { if ((uint32_t)nz < cig_cap) zl[nz] = (uint32_t)i; ++nz; }
                else a[i].secondary = (int)zl[k];
            }
            if ((uint32_t)nz > cig_cap) atomicExch(P.overflow, 2u);
        }
        __syncwarp();
        // ---------------- mem_reg2aln per region (reference bwa.cpp:151-177 calls it for every region):
        // narrow-band regions are queued for the thread-per-region kernel, the rest run here on the warp
        RowDev* rows = P.rows + blk.base;
        for (int i = 0; i < n; ++i) {
            const RegRec ar = a[i];
            RowDev row = row_from_reg(ar, P.ann_id);
            const int ncls = P.narrow_jobs != nullptr ? narrow_class(o, ar, P.max_len) : 0;
            const bool narrow = ncls != 0;
            if (lane == 0) {
                rows[i] = row;
                if (narrow) {
                    // DP regions and no-DP regions go to separate lists so that the lanes of a warp do similar work
                    NarrowJob jb; jb.r = r; jb.slot = blk.base + i; jb.w2 = reg2aln_w2(o, ar); jb.last_sc = -(1 << 30); jb.it = 0; jb.score = 0;
                    NarrowJob* lists = reinterpret_cast<NarrowJob*>(P.narrow_jobs);
                    if (ncls == 1 && narrow_is_tight(o, ar.qe - ar.qb, (int)(ar.re - ar.rb))) {
                        if (narrow_is_tight(o, ar.qe - ar.qb, (int)(ar.re - ar.rb), REG_WT4)) lists[3u * P.narrow_cap + atomicAdd(P.narrow_cnt + NARROW_T4_CNT, 1u)] = jb;
                        else lists[4u * P.narrow_cap + atomicAdd(P.narrow_cnt + NARROW_T8_CNT, 1u)] = jb;
                    }
                    else if (ncls == 1) push_narrow(lists, P.narrow_cap, P.narrow_cnt, P.narrow_cnt + 5, jb, narrow_is_big(o, ar.qe - ar.qb, (int)(ar.re - ar.rb), jb.w2));
                    else lists[2u * P.narrow_cap + atomicAdd(P.narrow_cnt + 3, 1u)] = jb;
                }
            }
            __syncwarp();
            if (!narrow) reg2aln_warp(P, ix, o, smat, S, cig_cap, rseq_cap, l_query, ar, rows + i, cells, calls);
        }
        if (lane == 0) P.row_cnt[r] = (uint32_t)n;
    }
    if (P.counters && lane == 0) { atomicAdd(&P.counters[0], cells); atomicAdd(&P.counters[1], calls); }
}

// ---------------------------------------------------------------------------------------------------
// ksw_global2 on ONE thread with the band in registers.  In diagonal coordinates kk = j - i + WT a cell's three
// inputs are: the diagonal H(i-1, j-1) at the SAME kk, E from (i-1, j) at kk + 1, F from (i, j-1) at kk - 1 -- so
// with the kk loop fully unrolled the whole band state (Hd[], Ep[]) is a register file, nothing is indexed
// dynamically and no shared memory is needed.  A region's own band [i - w, i + w] (w <= WT) is a sub-range of the
// window: cells outside [beg, end) are computed but masked where it matters (their E and F outputs are -inf, as
// ksw_global2 has it for cells it never computes; their H is never consumed).  The query travels in a nibble
// window that slides one base per row; scores come from the three distinct values of bwa_fill_scmat.
// Z (traceback): one byte per cell, [row][kk / 4][lane] words.  Returns eh[qlen].h.
// TIGHT (the tight passes): rows whose whole window lies inside the matrix and the band (w == WT, WT < i, i + WT < lq) take a leaner
// cell -- no validity masks, no first-column case, match / mismatch from one XOR of the window with the row's base.  That cell
// scores an ambiguous query base as a mismatch, so the caller must discard the result when *amb has a bit above the low two.
template <int WT, bool TIGHT>
__device__ __forceinline__ int global_dp_reg(const uint8_t* __restrict__ qg, int lq, bool rev, const uint8_t* __restrict__ pac, int64_t tbase,
                                             int rlen, int w, int sA, int sB, int sN, int o_del, int e_del, int o_ins, int e_ins,
                                             uint32_t* __restrict__ Z, unsigned long long& cells, uint32_t* amb_out = nullptr) {
    uint32_t amb = 0;
    constexpr int W = 2 * WT + 1, NW = (W + 7) / 8, ZW = (W + 3) / 4;
    const int oe_del = o_del + e_del, oe_ins = o_ins + e_ins;
    int Hd[W], Ep[W + 1];
    uint32_t win[NW];
#pragma unroll
    for (int kk = 0; kk < W; ++kk) {
        const int j = kk - WT;                     // row 0: eh[j].h = H(-1, j-1) = -(o_ins + e_ins j) for 1 <= j <= w
        Hd[kk] = (j >= 1 && j <= w) ? -(o_ins + e_ins * j) : KSW_NEG_INF;
        Ep[kk] = KSW_NEG_INF;
    }
    Ep[W] = KSW_NEG_INF;
#pragma unroll
    for (int x = 0; x < NW; ++x) win[x] = 0xffffffffu;
#pragma unroll
    for (int kk = WT; kk < W; ++kk) {
        const int j = kk - WT;
        if (j < lq) {
            const uint32_t b = rev ? qg[lq - 1 - j] : qg[j];
            amb |= b;
            win[kk >> 3] = (win[kk >> 3] & ~(15u << ((kk & 7) * 4))) | (b << ((kk & 7) * 4));
        }
    }
    int tb = rev ? 3 - (int)pac_get(pac, tbase) : (int)pac_get(pac, tbase);
    for (int i = 0; i < rlen; ++i) {
        const int beg = i > w ? i - w : 0;
        const int end = i + w + 1 < lq ? i + w + 1 : lq;
        const int ioff = i - WT - beg;                  // kk + ioff = j - beg
        const unsigned span = (unsigned)(end - beg);
        const int tz = beg == 0 ? 0 : 0x7fffffff;      // j == 0 (first column): the diagonal input is H(i-1, -1)
        const int colm1 = i == 0 ? 0 : -(o_del + e_del * i);
        cells += span;
        // next row's inputs: reference base, query base entering the window
        int tb_next = 0; uint32_t nb = 15u;
        if (i + 1 < rlen) tb_next = rev ? 3 - (int)pac_get(pac, tbase + i + 1) : (int)pac_get(pac, tbase + i + 1);
        { const int jn = i + 1 + WT; if (jn < lq) { nb = rev ? qg[lq - 1 - jn] : qg[jn]; amb |= nb; } }
        int f = KSW_NEG_INF;
        uint32_t zpack = 0;
        uint32_t* zi = Z + (size_t)i * ZW * 32;
        if (TIGHT && w == WT && i > WT && i + WT + 1 <= lq) {
            uint32_t xw[NW];
#pragma unroll
            for (int x = 0; x < NW; ++x) xw[x] = win[x] ^ ((uint32_t)tb * 0x11111111u);
#pragma unroll
            for (int kk = 0; kk < W; ++kk) {
                const bool mis = ((xw[kk >> 3] >> ((kk & 7) * 4)) & 15u) != 0;
                const int m = Hd[kk] + (mis ? sB : sA);
                int e = Ep[kk + 1];
                int d = m >= e ? 0 : 1;
                int h = m >= e ? m : e;
                d = h >= f ? d : 2;
                h = h >= f ? h : f;
                Hd[kk] = h;
                int tt = m - oe_del;
                e -= e_del;
                d |= e > tt ? 1 << 2 : 0;
                Ep[kk] = e > tt ? e : tt;
                tt = m - oe_ins;
                f -= e_ins;
                d |= f > tt ? 2 << 4 : 0;
                f = f > tt ? f : tt;
                zpack |= (uint32_t)d << ((kk & 3) * 8);
                if ((kk & 3) == 3 || kk == W - 1) { zi[(kk >> 2) * 32] = zpack; zpack = 0; }
            }
        } else
#pragma unroll
        for (int kk = 0; kk < W; ++kk) {
            const int t = ioff + kk;
            const bool valid = (unsigned)t < span;
            const int qb = (int)((win[kk >> 3] >> ((kk & 7) * 4)) & 15u);
            const int sc = qb == tb ? sA : (qb < 4 ? sB : sN);
            int m = (t == tz ? colm1 : Hd[kk]) + sc;
            int e = Ep[kk + 1];
            int d = m >= e ? 0 : 1;
            int h = m >= e ? m : e;
            d = h >= f ? d : 2;
            h = h >= f ? h : f;
            Hd[kk] = h;
            int tt = m - oe_del;
            e -= e_del;
            d |= e > tt ? 1 << 2 : 0;
            e = e > tt ? e : tt;
            Ep[kk] = valid ? e : KSW_NEG_INF;
            tt = m - oe_ins;
            int f2 = f - e_ins;
            d |= f2 > tt ? 2 << 4 : 0;
            f2 = f2 > tt ? f2 : tt;
            f = valid ? f2 : f;
            zpack |= (uint32_t)d << ((kk & 3) * 8);
            if ((kk & 3) == 3 || kk == W - 1) { zi[(kk >> 2) * 32] = zpack; zpack = 0; }
        }
        // slide the query window by one base
#pragma unroll
        for (int x = 0; x + 1 < NW; ++x) win[x] = __funnelshift_r(win[x], win[x + 1], 4);
        win[NW - 1] = ((win[NW - 1] >> 4) & ~(15u << (((W - 1) & 7) * 4))) | (nb << (((W - 1) & 7) * 4));
        tb = tb_next;
    }
    // eh[qlen].h after the last row = H(rlen-1, lq-1): diagonal offset lq - rlen + WT
    const int ks = lq - rlen + WT;
    int score = KSW_NEG_INF;
#pragma unroll
    for (int kk = 0; kk < W; ++kk) if (kk == ks) score = Hd[kk];
    if (TIGHT && amb_out) *amb_out = amb;
    return score;
}

// 16 bases pac[f .. f+16), first base in the top bits (pac is padded, f >= 0)
__device__ __forceinline__ uint32_t pac_win16(const uint8_t* pac, int64_t f) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(pac) + (f >> 4);
    return __funnelshift_l(__byte_perm(w[1], 0, 0x0123), __byte_perm(w[0], 0, 0x0123), (int)(f & 15) << 1);
}
// Mismatches on the gap-free diagonal of a region with lq == rlen, 16 bases per step: the query bytes (codes 0..3) are packed to two
// bits and XORed with a pac window.  Pairs are (q[j], pac[tbase + j]) on the forward strand and (q[j], 3 - pac[tbase + lq - 1 - j])
// on the reverse one (libbwa reverses both sequences there; a count does not care about the order).  *ok = false when the query
// holds a code above 3 (the caller then scores base by base with the matrix).
__device__ __forceinline__ int diag_mismatches(const uint8_t* qg, int lq, bool rev, const uint8_t* pac, int64_t tbase, bool* ok) {
    const uint32_t* qa = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(qg) & ~(uintptr_t)3);
    const int sh = (int)(reinterpret_cast<uintptr_t>(qg) & 3) * 8;
    uint32_t prev = qa[0], amb = 0;
    int mm = 0, j0 = 0;
    for (; j0 + 16 <= lq; j0 += 16) {
        uint32_t Q = 0;                                   // base j0 + k at bits 2k
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t nx = qa[(j0 >> 2) + k + 1];   // the read buffer is padded: the word behind the last base exists
            const uint32_t x = __funnelshift_r(prev, nx, sh);
            prev = nx;
            amb |= x;
            Q |= ((x | x >> 6 | x >> 12 | x >> 18) & 0xffu) << (8 * k);
        }
        uint32_t v;
        if (rev) v = ~pac_win16(pac, tbase + lq - 16 - j0);   // position tbase + lq - 1 - (j0 + k) sits at bits 2k of the window
        else {
            const uint32_t r = __brev(pac_win16(pac, tbase + j0));             // base order reversed, and the two bits of each base
            v = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);
        }
        const uint32_t d = Q ^ v;
        mm += __popc((d | d >> 1) & 0x55555555u);
    }
    for (int j = j0; j < lq; ++j) {
        const uint32_t q = qg[j];
        amb |= q;
        mm += q != (rev ? 3u - pac_get(pac, tbase + lq - 1 - j) : pac_get(pac, tbase + j));
    }
    *ok = (amb & 0xfcfcfcfcu) == 0;
    return mm;
}

// ---------------------------------------------------------------------------------------------------
// Thread-per-region mem_reg2aln for narrow bands (the common case for 150 bp reads: w = 6..31).
// One thread runs the ksw_global2 recurrence with the band in registers (global_dp_reg), reference bases are
// decoded from pac once per row, traceback bytes go to a per-warp global buffer laid out [cell][lane]
// (coalesced while lanes run in step).  A region whose band the kernel does not hold is handed to
// regs_cigar_wide (warp-cooperative rows).
struct NarrowParams {
    const uint8_t* seqs; const uint64_t* offs; const RegRec* regs; RowDev* rows;
    const NarrowJob* jobs; int job_stride; const uint32_t* n_jobs;      // jobs[k * job_stride]: a list's front (+1) or back (-1) section
    NarrowJob* requeue; uint32_t requeue_cap; uint32_t* requeue_cnt; uint32_t* requeue_big_cnt; uint64_t* wide_jobs; uint32_t* wide_cnt;
    uint32_t* cigar_pool; uint32_t cigar_cap; uint32_t* cigar_top;
    uint8_t* zbuf; uint32_t* ticket; uint32_t* overflow; unsigned long long* counters;
    NarrowJob* tight; uint32_t* tight_cnt;   // the next tight list: T4 for the diagonal pass (MODE 5), T8 for MODE 4
    uint32_t short_list;   // lists of at most this many regions are handed to the warp-cooperative kernel (BSQ_FIN_SHORT_LIST)
};

// MODE 5: the diagonal pass only (no DP code, few registers: the pass is a chain of dependent loads per region and lives on occupancy).
// MODE 1: the band in registers (global_dp_reg, w <= REG_WT); MODE 2: the same for w <= REG_WT2 (2 CTAs per SM); MODE 4 / 3: the
// tight passes.  Scores come from the three values of bwa_fill_scmat, the only matrix DevOpts carries (fill_dev_opts).
template <int MODE>
__global__ void __launch_bounds__(NARROW_THREADS, MODE == 5 ? 10 : (MODE >= 3 ? 6 : (MODE == 1 ? 4 : 2))) regs_cigar_narrow(NarrowParams P, DevIndex ix, DevOpts o) {
    __shared__ int smat[25];
    if (threadIdx.x < 25) smat[threadIdx.x] = o.mat[threadIdx.x];
    __syncthreads();
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t gwarp = (blockIdx.x * NARROW_THREADS + tid) >> 5;
    // traceback bytes, 4 cells per 32-bit store, laid out [row][4-cell group][lane]: a warp store is 128 contiguous bytes
    constexpr int WTM = MODE == 2 ? REG_WT2 : (MODE == 3 ? REG_WT3 : (MODE == 4 ? REG_WT4 : REG_WT));                                // half-width of the register window
    constexpr int ZROW = (2 * WTM + 1 + 3) / 4;                                      // words per row and lane
    uint32_t* Z = reinterpret_cast<uint32_t*>(P.zbuf + (size_t)gwarp * NARROW_TMAX * ZROW * 4 * 32) + lane;
    int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins, e_del = o.e_del, e_ins = o.e_ins;
    // keep the four gap constants in registers: left to itself the compiler re-reads them from the constant bank per cell
    asm volatile("" : "+r"(oe_del), "+r"(oe_ins), "+r"(e_del), "+r"(e_ins));
    const int64_t l_pac = ix.l_pac;
    const uint32_t n_jobs = *P.n_jobs;
    // A short list is a latency problem for one thread per region (a launch lasts as long as ONE region's DP, hundreds of
    // microseconds): its regions go to the warp-cooperative kernel, which runs a row's cells side by side.
    // MODE 5 (the diagonal pass): equal-length regions -- finish the ones whose diagonal is provably optimal, hand the rest to the DP list
    constexpr bool diag_pass = MODE == 5;
    const bool short_list = !diag_pass && n_jobs <= P.short_list;
    unsigned long long cells = 0, calls = 0;
    for (;;) {
        uint32_t t = next_ticket(P.ticket);
        if ((uint64_t)t * 32 >= n_jobs) break;
        const uint32_t j_id = t * 32 + lane;
        uint32_t cg[NARROW_CIG];
        // what the lane has to write into the CIGAR pool (one allocation per warp, behind the region's work)
        int e_nc = 0, e_first = 0, e_clip5 = 0, e_clip3 = 0, e_n = 0;
        uint32_t e_slot = 0; bool e_on = false;
        if (j_id < n_jobs) {
            const NarrowJob jb = P.jobs[(long)j_id * P.job_stride];
            const uint32_t r = jb.r, slot = jb.slot;
            const uint64_t job = (uint64_t)r << 32 | slot;
            const RegRec ar = P.regs[slot];
            const int l_read = (int)(P.offs[r + 1] - P.offs[r]);
            const int qb = ar.qb, qe = ar.qe, lq = qe - qb;
            const int64_t rb = ar.rb, re = ar.re;
            const int rlen = (int)(re - rb);
            const bool rev = rb >= l_pac;
            const bool reject = lq <= 0 || rb >= re || (rb < l_pac && re > l_pac) || rb < 0 || re > (l_pac << 1);
            // libbwa reverses query and reference on the reverse strand; both then read pac ascending
            const int64_t tbase = rev ? (l_pac << 1) - re : rb;
            const uint8_t* qg = P.seqs + P.offs[r] + qb;
            auto qat = [&](int j) -> int { return (int)(rev ? qg[lq - 1 - j] : qg[j]); };
            // ONE try of the band-doubling loop per pass; a region that needs another try is re-queued so that the
            // lanes of a warp stay balanced (the loop state travels in the job record)
            int n_cigar = 0, NM = -1, score = jb.score;
            int w2 = jb.w2 < o.w << 2 ? jb.w2 : o.w << 2;
            bool go_wide = false, again = false;
            do {
                n_cigar = 0; NM = -1;
                if (short_list && !reject) { go_wide = true; break; }
                int nm_known = -1;       // mismatches of a gap-free row, when the packed comparison has counted them already
                if (!reject) {
                    bool diagonal = lq == rlen && w2 == 0;   // bwa_gen_cigar2's own no-DP case
                    if (diag_pass && lq == rlen) {
                        // Equal lengths: any alignment other than the gap-free diagonal has >= 1 insertion and >= 1 deletion and at
                        // most lq - 1 aligned pairs, so it scores <= (lq - 1) max(mat) - oe_ins - oe_del.  If the diagonal beats that
                        // bound it is the UNIQUE optimum of ksw_global2 for every band (the diagonal lies inside any band), so the
                        // traceback is lq M and the score is band-independent: the DP and the band-doubling retries are skipped.
                        int sc = 0;
                        bool fast = false;
                        const int mm = diag_mismatches(qg, lq, rev, ix.pac, tbase, &fast);
                        if (fast) { sc = smat[0] * (lq - mm) + smat[1] * mm; nm_known = mm; }
                        else for (int i = 0; i < lq; ++i) {
                            const int tb = rev ? 3 - (int)pac_get(ix.pac, tbase + i) : (int)pac_get(ix.pac, tbase + i);
                            sc += smat[tb * 5 + qat(i)];
                        }
                        if (diagonal || sc > (lq - 1) * o.mat_max - oe_ins - oe_del) { score = sc; cg[0] = (uint32_t)lq << 4; n_cigar = 1; diagonal = true; }
                        else {   // needs the DP: over to the tight pass or the DP list, same try
                            if (narrow_is_tight(o, lq, rlen)) P.tight[atomicAdd(P.tight_cnt, 1u)] = jb;
                            else push_narrow(P.requeue, P.requeue_cap, P.requeue_cnt, P.requeue_big_cnt, jb, narrow_is_big(o, lq, rlen, jb.w2));
                            again = true; break;
                        }
                    } else if (diagonal) {
                        int sc = 0;
                        for (int i = 0; i < lq; ++i) {
                            const int tb = rev ? 3 - (int)pac_get(ix.pac, tbase + i) : (int)pac_get(ix.pac, tbase + i);
                            sc += smat[tb * 5 + qat(i)];
                        }
                        score = sc; cg[0] = (uint32_t)lq << 4; n_cigar = 1;
                    }
                    if (MODE != 5 && !diagonal) {
                        const int wx = gen_cigar_band(o, lq, rlen, w2);
                        // MODE 3 / 4 run the band min(w, WTM).  A path that leaves that band reaches a diagonal k = wr + 1 away from the
                        // main one and has to come back to the end cell: at least k gap bases on one side and k -+ (lq - rlen) on the other,
                        // so it scores at most ub.  If the score found inside the tight band beats ub, every decision along the traceback
                        // sees the same winner as under the band bwa_gen_cigar2 asks for (an alternative through outside cells, continued
                        // along the same suffix, would be a full path scoring >= the optimum): score and CIGAR are those of band w.
                        const int w = MODE >= 3 ? (wx < WTM ? wx : WTM) : wx;
                        if (MODE >= 3 && (!narrow_is_tight(o, lq, rlen, WTM) || rlen > NARROW_TMAX)) {
                            push_narrow(P.requeue, P.requeue_cap, P.requeue_cnt, P.requeue_big_cnt, jb, narrow_is_big(o, lq, rlen, jb.w2));
                            again = true; break;
                        }
                        if (MODE < 3 && (w > WTM || rlen > NARROW_TMAX)) { go_wide = true; break; }
                        ++calls;
                        uint32_t amb = 0;
                        score = global_dp_reg<WTM, (MODE >= 3)>(qg, lq, rev, ix.pac, tbase, rlen, w, smat[0], smat[1], smat[4], o.o_del, e_del, o.o_ins, e_ins, Z, cells, &amb);
                        if (MODE >= 3 && (amb & ~3u)) {            // an ambiguous base in the query: the exact-band kernels score it
                            push_narrow(P.requeue, P.requeue_cap, P.requeue_cnt, P.requeue_big_cnt, jb, narrow_is_big(o, lq, rlen, jb.w2));
                            again = true; break;
                        }
                        if (MODE >= 3 && w < wx) {
                            const int k = w + 1, dl = lq - rlen;
                            const int ubp = o.mat_max * (lq - k) - (o.o_ins + e_ins * k) - (o.o_del + e_del * (k - dl));
                            const int ubm = o.mat_max * (rlen - k) - (o.o_del + e_del * k) - (o.o_ins + e_ins * (k + dl));
                            if (score <= (ubp > ubm ? ubp : ubm)) {    // not provable: the next wider window, or the band bwa asks for; same try
                                if (MODE == 4) P.tight[atomicAdd(P.tight_cnt, 1u)] = jb;
                                else push_narrow(P.requeue, P.requeue_cap, P.requeue_cnt, P.requeue_big_cnt, jb, narrow_is_big(o, lq, rlen, jb.w2));
                                again = true; break;
                            }
                        }
                        // traceback
                        {
                            int which = 0, i = rlen - 1, k = (i + w + 1 < lq ? i + w + 1 : lq) - 1;
                            bool full = false;
                            auto push = [&](uint32_t op, uint32_t len) {
                                if (n_cigar == 0 || op != (cg[n_cigar - 1] & 0xf)) { if (n_cigar < NARROW_CIG) cg[n_cigar++] = len << 4 | op; else full = true; }
                                else cg[n_cigar - 1] += len << 4;
                            };
                            while (i >= 0 && k >= 0) {
                                const int jj = k - i + WTM;
                                which = (int)(Z[((size_t)i * ZROW + (jj >> 2)) * 32] >> ((jj & 3) << 3) & 0xff) >> (which << 1) & 3;
                                if (which == 0) { push(0, 1); --i; --k; }
                                else if (which == 1) { push(2, 1); --i; }
                                else { push(1, 1); --k; }
                            }
                            if (i >= 0) push(2, (uint32_t)(i + 1));
                            if (k >= 0) push(1, (uint32_t)(k + 1));
                            if (full) { go_wide = true; break; }
                            for (int a = 0; a < n_cigar >> 1; ++a) { uint32_t x = cg[a]; cg[a] = cg[n_cigar - 1 - a]; cg[n_cigar - 1 - a] = x; }
                        }
                    }
                    // NM
                    int x = 0, y = 0, n_mm = 0, n_gap = 0;
                    if (nm_known >= 0 && n_cigar == 1) n_mm = nm_known;
                    else for (int k = 0; k < n_cigar; ++k) {
                        const int op = (int)(cg[k] & 0xf), len = (int)(cg[k] >> 4);
                        if (op == 0) {
                            bool fast = false;
                            int mm = 0;
                            // a run of M: q[x .. x+len) against the reference from y on -- the packed comparison of the diagonal pass
                            if (len >= 16) mm = diag_mismatches(rev ? qg + (lq - x - len) : qg + x, len, rev, ix.pac, tbase + y, &fast);
                            if (fast) n_mm += mm;
                            else for (int i = 0; i < len; ++i) {
                                const int tb = rev ? 3 - (int)pac_get(ix.pac, tbase + y + i) : (int)pac_get(ix.pac, tbase + y + i);
                                n_mm += qat(x + i) != tb;
                            }
                            x += len; y += len;
                        } else if (op == 2) { if (k > 0 && k < n_cigar - 1) n_gap += len; y += len; }
                        else if (op == 1) { x += len; n_gap += len; }
                    }
                    NM = n_mm + n_gap;
                }
                if (score == jb.last_sc || w2 == o.w << 2) break;
                if (diag_pass && !reject && lq == rlen && !(lq == rlen && w2 == 0)) break;   // band-independent result (see above)
                if (jb.it + 1 < 3 && score < ar.truesc - o.a) {
                    again = true;
                    NarrowJob nx; nx.r = r; nx.slot = slot; nx.w2 = w2 << 1; nx.last_sc = score; nx.it = jb.it + 1; nx.score = score;
                    push_narrow(P.requeue, P.requeue_cap, P.requeue_cnt, P.requeue_big_cnt, nx, narrow_is_big(o, lq, rlen, nx.w2));
                }
            } while (false);
            if (go_wide) {
                uint32_t k = atomicAdd(P.wide_cnt, 1u);
                P.wide_jobs[k] = job;
            } else if (!again) {
                int is_rev;
                int64_t pos = bns_depos(ix, rb < l_pac ? rb : re - 1, &is_rev);
                int nc = n_cigar, first = 0;
                if (nc > 0) {
                    if ((cg[0] & 0xf) == 2) { pos += cg[0] >> 4; first = 1; --nc; }
                    else if ((cg[n_cigar - 1] & 0xf) == 2) --nc;
                }
                int clip5 = 0, clip3 = 0;
                if (qb != 0 || qe != l_read) { clip5 = is_rev ? l_read - qe : qb; clip3 = is_rev ? qb : l_read - qe; }
                e_nc = nc; e_first = first; e_clip5 = clip5; e_clip3 = clip3; e_n = nc + (clip5 ? 1 : 0) + (clip3 ? 1 : 0);
                e_slot = slot; e_on = true;
                RowDev* out = P.rows + slot;
                const int rid = bns_pos2rid(ix, pos);
                out->NM = NM; out->is_rev = is_rev; out->pos = pos - ix.ann_offset[rid < 0 ? 0 : rid];
            }
        }
        __syncwarp();
        {   // pool space for the warp's CIGARs: one atomic (a million single-lane atomics on one word are a stage of their own)
            uint32_t incl = (uint32_t)e_n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t up = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += up; }
            uint32_t base = 0;
            if (lane == 31 && incl) base = atomicAdd(P.cigar_top, incl);
            base = __shfl_sync(FULL, base, 31);
            if (e_on) {
                const uint32_t coff = base + incl - (uint32_t)e_n;
                RowDev* out = P.rows + e_slot;
                if ((uint64_t)coff + (uint64_t)e_n > (uint64_t)P.cigar_cap) { atomicExch(P.overflow, 1u); }
                else {
                    uint32_t* dst = P.cigar_pool + coff;
                    int k = 0;
                    if (e_clip5) dst[k++] = (uint32_t)e_clip5 << 4 | 3;
                    for (int c = 0; c < e_nc; ++c) dst[k++] = cg[e_first + c];
                    if (e_clip3) dst[k++] = (uint32_t)e_clip3 << 4 | 3;
                    out->cigar_off = coff; out->n_cigar = (uint32_t)e_n;
                }
            }
        }
        __syncwarp();
    }
    if (P.counters) {
        cells = __reduce_add_sync(FULL, (unsigned)(cells & 0xffffffffu)) + ((unsigned long long)__reduce_add_sync(FULL, (unsigned)(cells >> 32)) << 32);
        calls = __reduce_add_sync(FULL, (unsigned)calls);
        if (lane == 0) { atomicAdd(&P.counters[0], cells); atomicAdd(&P.counters[1], calls); }
    }
}

// regions handed over by the narrow kernel: warp-cooperative mem_reg2aln, one warp per job
template <bool SMEM>
__global__ void __launch_bounds__(FIN_THREADS) regs_cigar_wide(FinalizeParams P, DevIndex ix, DevOpts o, uint32_t cig_cap, uint32_t rseq_cap) {
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    __shared__ int smat[25];
    if (threadIdx.x < 25) smat[threadIdx.x] = o.mat[threadIdx.x];
    __syncthreads();
    const int lane = lane_id();
    const uint32_t gwarp = (blockIdx.x * FIN_THREADS + threadIdx.x) >> 5;
    FScratch S;
    {
        const size_t fast = ((size_t)(P.max_len + 2) * 8 + rseq_cap + P.max_len + 15) & ~(size_t)15;
        uint8_t* gbase = P.scratch + (size_t)gwarp * P.scratch_per_warp;
        uint8_t* fbase = SMEM ? dyn_smem + (size_t)(threadIdx.x >> 5) * fast : gbase;
        S.ehh = reinterpret_cast<int*>(fbase);
        S.ehe = S.ehh + (P.max_len + 2);
        S.rseq = reinterpret_cast<uint8_t*>(S.ehe + (P.max_len + 2));
        S.query = S.rseq + rseq_cap;
        S.cig = reinterpret_cast<uint32_t*>(gbase + fast);
        S.z = reinterpret_cast<uint8_t*>(S.cig + cig_cap);
    }
    unsigned long long cells = 0, calls = 0;
    const uint32_t n_jobs = *P.wide_cnt;
    for (;;) {
        uint32_t t = next_ticket(P.ticket);
        if (t >= n_jobs) break;
        const uint64_t job = P.wide_jobs[t];
        const uint32_t r = (uint32_t)(job >> 32), slot = (uint32_t)job;
        const int l_query = (int)(P.offs[r + 1] - P.offs[r]);
        const uint8_t* qg = P.seqs + P.offs[r];
        for (int i = lane; i < l_query; i += 32) S.query[i] = qg[i];
        __syncwarp();
        const RegRec ar = P.regs[slot];
        reg2aln_warp(P, ix, o, smat, S, cig_cap, rseq_cap, l_query, ar, P.rows + slot, cells, calls);
    }
    if (P.counters && lane == 0) { atomicAdd(&P.counters[0], cells); atomicAdd(&P.counters[1], calls); }
}

}  // namespace

static size_t fin_fast_bytes(uint32_t max_len, uint32_t rseq_cap) { return ((size_t)(max_len + 2) * 8 + rseq_cap + max_len + 15) & ~(size_t)15; }
static uint32_t fin_cig_cap(uint32_t max_len, uint32_t rseq_cap) { return max_len + rseq_cap + 8; }

size_t finalize_scratch_per_warp(uint32_t max_len, uint32_t rseq_cap, uint32_t* z_cap_out) {
    // traceback matrix: n_col <= min(qlen, 2w+1) with w <= 4 * opt.w handled by the caller through rseq_cap;
    // worst case qlen x tlen for short reads, band-limited for long ones
    uint64_t z = (uint64_t)max_len * (uint64_t)rseq_cap;
    const uint64_t z_band = (uint64_t)rseq_cap * 1024;   // 2w+1 <= 801 columns when w = 4 * 100
    if (z > z_band) z = z_band;
    if (z_cap_out) *z_cap_out = (uint32_t)z;
    size_t b = fin_fast_bytes(max_len, rseq_cap) + (size_t)fin_cig_cap(max_len, rseq_cap) * 4 + (size_t)z;
    return (b + 255) & ~(size_t)255;
}

static bool fin_use_smem(uint32_t max_len, uint32_t rseq_cap) { return fin_fast_bytes(max_len, rseq_cap) * FIN_WARPS <= 40 * 1024; }

int finalize_resident_warps() {
    return cached_blocks_per_sm(regs_finalize<false>, FIN_THREADS, 0) * cached_sm_count() * FIN_WARPS;
}

// resident CTAs of a thread-per-region kernel on the whole chip (a launch fills it once; the kernel takes jobs by ticket)
template <int MODE> static int narrow_blocks() { return cached_blocks_per_sm(regs_cigar_narrow<MODE>, NARROW_THREADS, 0) * cached_sm_count(); }
// traceback buffer of a kernel whose register window has half-width wt
static size_t narrow_z_bytes(int blocks, int wt) { return (size_t)blocks * (NARROW_THREADS / 32) * NARROW_TMAX * ((2 * wt + 1 + 3) / 4) * 4 * 32; }
// The two kernels of a DP pass run side by side, so each has its own traceback buffer: MODE 1's first (the tight passes run alone
// and share it), MODE 2's behind it.
static size_t narrow_z_front() {
    return std::max(narrow_z_bytes(narrow_blocks<1>(), REG_WT), std::max(narrow_z_bytes(narrow_blocks<3>(), REG_WT3), narrow_z_bytes(narrow_blocks<4>(), REG_WT4)));
}

size_t narrow_zbuf_bytes() { return narrow_z_front() + narrow_z_bytes(narrow_blocks<2>(), REG_WT2); }

void launch_finalize(const FinalizeParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, uint32_t rseq_cap, int n_warps, uint64_t* launches, const ExtAux* aux) {
    const uint32_t cig_cap = fin_cig_cap(p.max_len, rseq_cap);
    int blocks = n_warps / FIN_WARPS;
    if (blocks < 1) blocks = 1;
    const bool smem_ok = fin_use_smem(p.max_len, rseq_cap);
    const size_t smem = smem_ok ? fin_fast_bytes(p.max_len, rseq_cap) * FIN_WARPS : 0;
    // phase 1: dedup / patch / primary marking; wide regions aligned inline, narrow ones queued.  Single-region reads first, thread per read.
    if (p.todo && p.narrow_jobs && p.n_reads) {
        regs_finalize_thread<<<(p.n_reads + 127) / 128, 128, 0, st>>>(p, ix, o);
        if (launches) ++*launches;
    }
    if (smem_ok) regs_finalize<true><<<blocks, FIN_THREADS, smem, st>>>(p, ix, o, cig_cap, rseq_cap);
    else regs_finalize<false><<<blocks, FIN_THREADS, 0, st>>>(p, ix, o, cig_cap, rseq_cap);
    if (launches) ++*launches;
    if (!p.narrow_jobs) return;
    // phase 2: thread-per-region narrow-band mem_reg2aln, one try of the band-doubling loop per pass (<= 3 tries)
    {
        NarrowJob* listA = reinterpret_cast<NarrowJob*>(p.narrow_jobs);
        NarrowJob* listB = listA + p.narrow_cap;
        NarrowJob* listS = listA + 2 * (size_t)p.narrow_cap;
        NarrowJob* listT4 = listA + 3 * (size_t)p.narrow_cap;
        NarrowJob* listT8 = listA + 4 * (size_t)p.narrow_cap;
        for (int pass = 0; pass < 4; ++pass) {
            // pass 0: equal-length regions (list S): diagonal proof, the rest joins list A; pass 1: DP regions (A -> re-queue B);
            // pass 2: second tries (B -> A); pass 3: third tries (A).  A DP pass is two launches: the register-band kernel on
            // the front section of the list, the wide register-band kernel on the back section (bands wider than REG_WT).
            // counters: 0 A front, 1 B front, 2 A front (third tries), 3 S, 4 sink, 5 A back, 6 B back, 7 A back (third tries)
            NarrowParams q;
            q.seqs = p.seqs; q.offs = p.offs; q.regs = p.regs; q.rows = p.rows;
            NarrowJob* in = pass == 0 ? listS : (pass == 2 ? listB : listA);
            q.requeue = (pass == 0 || pass == 2) ? listA : listB; q.requeue_cap = p.narrow_cap;
            q.requeue_cnt = p.narrow_cnt + (pass == 0 ? 0 : (pass == 1 ? 1 : (pass == 2 ? 2 : 4)));   // pass 3 never re-queues
            q.requeue_big_cnt = p.narrow_cnt + (pass == 0 ? 5 : (pass == 1 ? 6 : (pass == 2 ? 7 : 4)));
            q.wide_jobs = p.wide_jobs; q.wide_cnt = p.wide_cnt; q.cigar_pool = p.cigar_pool; q.cigar_cap = p.cigar_cap; q.cigar_top = p.cigar_top;
            q.zbuf = p.narrow_z; q.overflow = p.overflow; q.counters = p.counters;
            q.tight = listT4; q.tight_cnt = p.narrow_cnt + NARROW_T4_CNT;
            { static const uint32_t sl = getenv("BSQ_FIN_SHORT_LIST") ? (uint32_t)atoi(getenv("BSQ_FIN_SHORT_LIST")) : NARROW_SHORT_LIST; q.short_list = sl; }
            q.jobs = in; q.job_stride = 1; q.ticket = p.ticket + 1 + pass;
            q.n_jobs = p.narrow_cnt + (pass == 0 ? 3 : (pass == 1 ? 0 : (pass == 2 ? 1 : 2)));
            if (pass == 0) {
                // the diagonal proof needs no band state: a build of the kernel without the DP (12 CTAs per SM)
                regs_cigar_narrow<5><<<narrow_blocks<5>(), NARROW_THREADS, 0, st>>>(q, ix, o);
                // passes T4, T8: every first try whose end cell fits the tight window; what T4 cannot prove goes to T8, what T8
                // cannot prove joins list A -- always the same try
                q.jobs = listT4; q.n_jobs = p.narrow_cnt + NARROW_T4_CNT; q.ticket = p.ticket + 9;
                q.tight = listT8; q.tight_cnt = p.narrow_cnt + NARROW_T8_CNT;
                regs_cigar_narrow<4><<<narrow_blocks<4>(), NARROW_THREADS, 0, st>>>(q, ix, o);
                q.jobs = listT8; q.n_jobs = p.narrow_cnt + NARROW_T8_CNT; q.ticket = p.ticket + 10;
                regs_cigar_narrow<3><<<narrow_blocks<3>(), NARROW_THREADS, 0, st>>>(q, ix, o);
                if (launches) *launches += 3;
            } else {
                // the two kernels of a DP pass work on disjoint sections of the list: side by side when a side stream is there
                cudaStream_t s2 = aux ? aux->st[0] : st;
                if (aux) { cudaEventRecord(aux->ev[0], st); cudaStreamWaitEvent(s2, aux->ev[0], 0); }
                regs_cigar_narrow<1><<<narrow_blocks<1>(), NARROW_THREADS, 0, st>>>(q, ix, o);
                q.jobs = in + p.narrow_cap - 1; q.job_stride = -1; q.ticket = p.ticket + 5 + pass;      // tickets 6..8
                q.n_jobs = p.narrow_cnt + (pass == 1 ? 5 : (pass == 2 ? 6 : 7));
                q.zbuf = p.narrow_z + narrow_z_front();
                regs_cigar_narrow<2><<<narrow_blocks<2>(), NARROW_THREADS, 0, s2>>>(q, ix, o);
                if (aux) { cudaEventRecord(aux->ev[1], s2); cudaStreamWaitEvent(st, aux->ev[1], 0); }
                if (launches) *launches += 2;
            }
        }
    }
    // phase 3: whatever needed a wider band on a retry
    {
        FinalizeParams w = p;
        w.ticket = p.ticket + 5;
        if (smem_ok) regs_cigar_wide<true><<<blocks, FIN_THREADS, smem, st>>>(w, ix, o, cig_cap, rseq_cap);
        else regs_cigar_wide<false><<<blocks, FIN_THREADS, 0, st>>>(w, ix, o, cig_cap, rseq_cap);
        if (launches) ++*launches;
    }
}
