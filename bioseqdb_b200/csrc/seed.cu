// seed.cu -- kernel `seed_smem`: the three seeding passes of mem_collect_intv (SURVEY.md A.4), one warp
// per read, persistent warps with an atomic ticket.  All control flow is warp-uniform: every lane holds
// the same interval registers; the lanes split the two 64-byte Occ blocks of a bwt_extend (one coalesced
// warp load: lanes 0-15 -> block of row k, lanes 16-31 -> block of row l).
//
// Only the child interval of the ONE base being extended is ever needed, and it is a few sums over the 32
// lanes --
//     x2' = sum_l eq - sum_k eq,   S = sum_l gt - sum_k gt (symbols > c, for the cumulative side),   tk[c] = sum_k eq
// where a lane contributes its checkpoint word (lanes holding the checkpoint of symbol c) or the popcount of
// its masked symbol word.  Each sum is ONE redux.sync (warp reduce hardware): a bwt_extend costs one load,
// two popcounts and three reductions per lane.  Texts of 2^32 rows or more keep row indices in 64 bits; x2'
// and S still fit 32 bits (they are bounded by the parent interval), only tk[c] needs its checkpoint's two
// halves, i.e. two more single-contributor reductions.  Interval lists and the read live in shared memory.
#include "seed.cuh"
#include "seed_thread.cuh"
#include "launch_cache.cuh"
#include <algorithm>

namespace {

constexpr int SEED_THREADS = 256;
constexpr int SEED_WARPS = SEED_THREADS / 32;
// prefix table: bi-intervals of every t-mer, t = 1..K, levels back to back.  K is chosen per index, about log4 of the text
// length, so that a K-mer has a handful of occurrences at most: 12 -> 358 MB, 13 -> 1.4 GB, 14 -> 5.7 GB (of 180 GB HBM)
constexpr int KMER_K_MAX = 14;      // choice by text length; ensure_kmer_table goes to 15 (23 GB) where HBM allows
__host__ __device__ constexpr uint32_t kmer_level_off(int t) { return (0x55555555u >> (32 - 2 * t)) - 1u; }   // first entry of level t = (4^t - 4) / 3, 1 <= t <= 16

template <class IdxT> struct IvT { IdxT x0, x1; uint32_t x2, info; };   // info = end of the match on the query
// prefix-table entry {x0 low word, x1 low word, x2, hi}: hi = bits 32..39 of x0 | bits 32..39 of x1 << 8 (zero while rows fit 32 bits)
template <class IdxT> __device__ __forceinline__ IdxT tab_x0(const uint4& e) {
    return sizeof(IdxT) == 4 ? (IdxT)e.x : (IdxT)((unsigned long long)(e.w & 0xffu) << 32 | e.x);
}
template <class IdxT> __device__ __forceinline__ IdxT tab_x1(const uint4& e) {
    return sizeof(IdxT) == 4 ? (IdxT)e.y : (IdxT)((unsigned long long)((e.w >> 8) & 0xffu) << 32 | e.y);
}
__host__ __device__ __forceinline__ uint4 tab_entry(unsigned long long x0, unsigned long long x1, uint32_t x2) {
    return make_uint4((uint32_t)x0, (uint32_t)x1, x2, (uint32_t)((x0 >> 32) & 0xffu) | (uint32_t)((x1 >> 32) & 0xffu) << 8);
}
template <> struct __align__(16) IvT<uint32_t> { uint32_t x0, x1, x2, info; };

// warp-private context: everything the extend needs without indexing the kernel parameter block dynamically
// (a dynamically indexed parameter array is spilled to local memory)
template <class IdxT> struct Ctx {
    const uint32_t* occ;
    const IdxT* sL2;         // shared memory: L2[0..4]
    const uint4* kmer_tab;   // prefix table (x0, x1, x2, -) of all t-mers, t <= kk; nullptr when absent
    int kk;                  // depth of the prefix table
    int lane;                // the thread's lane, read from the special register ONCE (the compiler otherwise re-issues S2R in hot loops)
    // unique-match shortcut: full SA, inverse SA and the 2-bit text; isa == nullptr disables it
    const IdxT* sa; const IdxT* isa; const uint8_t* pac; IdxT l_pac, n;
    IdxT primary;
    uint32_t sym_base;       // first symbol covered by this lane's word (symbol lanes), 1 << 20 for checkpoint lanes
    int cnt_sym;             // symbol whose checkpoint LOW word this lane holds, -1 otherwise
    int cnt_hi;              // symbol whose checkpoint HIGH word this lane holds, -1 otherwise
    bool lhalf;              // lanes 16-31 read the block of row l
};

// child interval of `ik` for base c.  IS_BACK selects which of x0/x1 plays "k" (SURVEY A.2 bwt_extend).
template <class IdxT, int IS_BACK>
__device__ __forceinline__ IvT<IdxT> extend1(const Ctx<IdxT>& C, const IvT<IdxT>& ik, int c) {
    const IdxT xo = IS_BACK ? ik.x0 : ik.x1, xb = IS_BACK ? ik.x1 : ik.x0;
    IdxT pos = xo - 1 + (C.lhalf ? (IdxT)ik.x2 : (IdxT)0);
    pos -= (pos >= C.primary);
    const uint32_t word = __ldg(C.occ + ((size_t)(pos >> 7) << 4) + (C.lane & 15));
    // symbol lanes: count symbols == c and > c among the first nsym symbols of the word (branch-free)
    int nsym = (int)(pos & 127) + 1 - (int)C.sym_base;
    nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
    const uint32_t keep = __funnelshift_rc(0u, 0x55555555u, 2 * nsym);   // low bit of each of the top nsym symbols
    const uint32_t C1 = 0u - (uint32_t)(c >> 1), C0 = 0u - (uint32_t)(c & 1);
    const uint32_t hx = ~((word >> 1) ^ C1);          // hi bit equals c's hi bit
    const uint32_t eqm = hx & ~(word ^ C0) & keep;
    const uint32_t gtm = (((word >> 1) & ~C1) | (hx & word & ~C0)) & keep;
    const int pop_eq = __popc(eqm);
    int eq = pop_eq, gt = __popc(gtm);
    if (C.cnt_sym >= 0) { eq = C.cnt_sym == c ? (int)word : 0; gt = C.cnt_sym > c ? (int)word : 0; }
    const int sz = __reduce_add_sync(FULL, C.lhalf ? eq : -eq);
    const int S = __reduce_add_sync(FULL, C.lhalf ? gt : -gt);
    IdxT tk;
    if (sizeof(IdxT) == 4) tk = (IdxT)(uint32_t)__reduce_add_sync(FULL, C.lhalf ? 0 : eq);
    else {   // exactly one lane contributes to each of the two halves of the 64-bit checkpoint
        const uint32_t lo = __reduce_add_sync(FULL, (!C.lhalf && C.cnt_sym == c) ? word : 0u);
        const uint32_t hi = __reduce_add_sync(FULL, (!C.lhalf && C.cnt_hi == c) ? word : 0u);
        const uint32_t pp = __reduce_add_sync(FULL, (!C.lhalf && C.cnt_sym < 0) ? (uint32_t)pop_eq : 0u);
        tk = (IdxT)(((unsigned long long)hi << 32 | lo) + pp);
    }
    const IdxT no = C.sL2[c] + 1 + tk;
    const IdxT nb = xb + (IdxT)(xo <= C.primary && xo + ik.x2 - 1 >= C.primary) + (IdxT)(uint32_t)S;
    IvT<IdxT> ok;
    ok.x0 = IS_BACK ? no : nb; ok.x1 = IS_BACK ? nb : no; ok.x2 = (uint32_t)sz; ok.info = ik.info;
    return ok;
}

// Four backward extensions per warp step: lane group g = lane / 8 extends its own list entry with the same base c
// (the entries of a backward step are independent).  Inside a group lanes 0-3 read the block of row k and lanes
// 4-7 the block of row l, 16 bytes each (lane 0: checkpoints A,C; lane 1: G,T; lanes 2,3: 64 symbols each), so a
// warp load touches 8 cache lines for 4 extensions; the three sums are 3-step xor-shuffle reductions confined to
// the group.  Every lane of a group returns the group's child interval.
template <class IdxT>
__device__ __forceinline__ IvT<IdxT> extend4_back(const Ctx<IdxT>& C, const IvT<IdxT>& ik, int c, bool valid) {
    const int t = C.lane & 7;
    const bool lside = (t & 4) != 0;
    const IdxT xo = ik.x0, xb = ik.x1;
    IdxT pos = xo - 1 + (lside ? (IdxT)ik.x2 : (IdxT)0);
    pos -= (pos >= C.primary);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (valid) v = __ldg(reinterpret_cast<const uint4*>(C.occ + ((size_t)(pos >> 7) << 4)) + (t & 3));
    // symbol lanes (t & 2): 4 words = 64 symbols starting at 64 (t & 1); checkpoint lanes get rem = 0 => nothing counted
    const uint32_t C1 = 0u - (uint32_t)(c >> 1), C0 = 0u - (uint32_t)(c & 1);
    const int rem = (t & 2) ? (int)(pos & 127) + 1 - ((t & 1) << 6) : 0;
    int eq = 0, gt = 0;
    const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int nsym = rem - (k << 4);
        nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
        const uint32_t keep = __funnelshift_rc(0u, 0x55555555u, 2 * nsym);
        const uint32_t word = w4[k];
        const uint32_t hx = ~((word >> 1) ^ C1);
        eq += __popc(hx & ~(word ^ C0) & keep);
        gt += __popc((((word >> 1) & ~C1) | (hx & word & ~C0)) & keep);
    }
    uint32_t tk_hi = 0;
    if ((t & 2) == 0) {   // checkpoint lanes: symbols a = 2 (t & 1) and a + 1; u64 checkpoints = (.x,.y) and (.z,.w)
        const int a = (t & 1) << 1;
        eq = c == a ? (int)v.x : (c == a + 1 ? (int)v.z : 0);
        gt = (a > c ? (int)v.x : 0) + (a + 1 > c ? (int)v.z : 0);
        if (sizeof(IdxT) == 8 && !lside) tk_hi = c == a ? v.y : (c == a + 1 ? v.w : 0u);
    }
    int sz = lside ? eq : -eq, S = lside ? gt : -gt;
    // tk: the checkpoint's low word and the popcounts are summed separately so that a 64-bit checkpoint cannot lose a carry
    uint32_t tk_lo = (!lside && (t & 2) == 0) ? (uint32_t)eq : 0u, tk_pop = (!lside && (t & 2) != 0) ? (uint32_t)eq : 0u;
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
        sz += __shfl_xor_sync(FULL, sz, d); S += __shfl_xor_sync(FULL, S, d);
        tk_lo += __shfl_xor_sync(FULL, tk_lo, d); tk_pop += __shfl_xor_sync(FULL, tk_pop, d);
        if (sizeof(IdxT) == 8) tk_hi += __shfl_xor_sync(FULL, tk_hi, d);
    }
    const IdxT tk = sizeof(IdxT) == 8 ? (IdxT)(((unsigned long long)tk_hi << 32 | tk_lo) + tk_pop) : (IdxT)(tk_lo + tk_pop);
    IvT<IdxT> ok;
    ok.x0 = C.sL2[c] + 1 + tk;
    ok.x1 = xb + (IdxT)(xo <= C.primary && xo + ik.x2 - 1 >= C.primary) + (IdxT)(uint32_t)S;
    ok.x2 = (uint32_t)sz; ok.info = ik.info;
    return ok;
}

// ---- unique-match shortcut --------------------------------------------------------------------------
// An interval of size 1 is ONE occurrence of the match at text position pos = SA[x0].  Extending it can only keep
// it (the next text base equals the read base) or kill it, so the FM-index need not be consulted: the warp
// compares read and text directly, 32 bases per step, and the rows of the extended match come from the inverse
// suffix array -- x0 = ISA[start], x1 = ISA[n - start - length] (T is its own reverse complement).  The result
// is the bi-interval bwt_extend would have produced, because the bi-interval of a string is unique.
template <class IdxT> __device__ __forceinline__ uint32_t text_base(const Ctx<IdxT>& C, IdxT p) {
    return p < C.l_pac ? pac_get(C.pac, (int64_t)p) : 3u - pac_get(C.pac, (int64_t)2 * (int64_t)C.l_pac - 1 - (int64_t)p);
}
// number of consecutive k in [0, maxlen) with q[qpos + k] an ACGT base equal to T[tpos + k]
template <class IdxT> __device__ __forceinline__ int match_run_fwd(const Ctx<IdxT>& C, IdxT tpos, const uint8_t* q, int qpos, int maxlen) {
    const int lane = C.lane;
    for (int base = 0; base < maxlen; base += 32) {
        const int k = base + lane;
        bool ok = k < maxlen;
        if (ok) { const IdxT p = tpos + (IdxT)k; const uint32_t b = q[qpos + k]; ok = p < C.n && b < 4 && text_base(C, p) == b; }
        const uint32_t bad = __ballot_sync(FULL, !ok);
        if (bad) { const int r = base + __ffs(bad) - 1; return r < maxlen ? r : maxlen; }
    }
    return maxlen;
}
// backwards: number of consecutive k in [0, maxlen) with q[qpos - k] == T[tpos - 1 - k]
template <class IdxT> __device__ __forceinline__ int match_run_bwd(const Ctx<IdxT>& C, IdxT tpos, const uint8_t* q, int qpos, int maxlen) {
    const int lane = C.lane;
    for (int base = 0; base < maxlen; base += 32) {
        const int k = base + lane;
        bool ok = k < maxlen;
        if (ok) { const uint32_t b = q[qpos - k]; ok = (IdxT)k < tpos && b < 4 && text_base(C, (IdxT)(tpos - 1 - (IdxT)k)) == b; }
        const uint32_t bad = __ballot_sync(FULL, !ok);
        if (bad) { const int r = base + __ffs(bad) - 1; return r < maxlen ? r : maxlen; }
    }
    return maxlen;
}

// 16 bases of the read starting at x, 2 bits each, first base in the top bits; false when one of the first K is ambiguous.
// pk = 2-bit packed copy of the read (shared-memory mode), has_n = the read holds an ambiguous base somewhere.
__device__ __forceinline__ bool kmer_word(const uint8_t* q, const uint32_t* pk, bool has_n, int x, int K, uint32_t& w) {
    if (pk != nullptr && !has_n) { w = __funnelshift_l(pk[(x >> 4) + 1], pk[x >> 4], (x & 15) << 1); return true; }
    uint32_t idx = 0; bool acgt = true;
    for (int t = 0; t < K; ++t) { const uint32_t b = q[x + t]; acgt = acgt && b < 4; idx = idx << 2 | (b & 3); }
    w = idx << (32 - 2 * K);
    return acgt;
}

template <class IdxT> __device__ __forceinline__ IvT<IdxT> set_intv(const Ctx<IdxT>& C, int c) {
    IvT<IdxT> ik;
    ik.x0 = C.sL2[c] + 1; ik.x1 = C.sL2[3 - c] + 1; ik.x2 = (uint32_t)(C.sL2[c + 1] - C.sL2[c]); ik.info = 0;
    return ik;
}

struct Out { Intv* out; uint32_t n, cap; bool ovf; int lane; };

template <class IdxT> __device__ __forceinline__ void emit(Out& O, const IvT<IdxT>& p, uint32_t start, uint32_t end) {
    if (O.n < O.cap) {
        if (O.lane == 0) { Intv v; v.x0 = p.x0; v.x1 = p.x1; v.x2 = p.x2; v.info = (uint64_t)start << 32 | end; O.out[O.n] = v; }
    } else O.ovf = true;
    ++O.n;
}

// bwt_smem1a with max_intv == 0 (the only way this path calls it).  la/lb: two interval lists of list_cap entries.
template <class IdxT>
__device__ __forceinline__ int smem1(const Ctx<IdxT>& C, const DevOpts& o, int len, const uint8_t* q, int x, uint32_t min_intv, IvT<IdxT>* la,
                                     IvT<IdxT>* lb, uint32_t list_cap, Out& O, unsigned long long& n_ext, const uint32_t* pk, bool has_n, IvT<IdxT>* hand) {
    if (q[x] > 3) return x + 1;
    if (min_intv < 1) min_intv = 1;
    const int KK = C.kk;
    const int lane = C.lane;
    IvT<IdxT> ik = set_intv(C, q[x]);
    ik.info = (uint32_t)(x + 1);
    IvT<IdxT>* curr = la; IvT<IdxT>* prev = lb;
    uint32_t n_curr = 0;
    int i = x + 1;
    bool fwd_done = false;
    if (C.kmer_tab && x + KK <= len) {
        // The first KK - 1 forward steps from the prefix table: lane t fetches the interval of q[x .. x+t]; the step
        // that appends base t+1 records lane t's interval when the size changes and stops the walk when it falls below
        // min_intv -- the same decisions the scalar loop takes, evaluated for all steps at once.
        uint32_t w;
        if (kmer_word(q, pk, has_n, x, KK, w)) {
            uint4 e = make_uint4(0, 0, 0, 0);
            if (lane < KK) e = __ldg(C.kmer_tab + kmer_level_off(lane + 1) + (w >> (30 - 2 * lane)));
            const uint32_t x2n = __shfl_down_sync(FULL, e.z, 1);
            const bool change = lane < KK - 1 && x2n != e.z;
            const uint32_t brk = __ballot_sync(FULL, change && x2n < min_intv);
            const int steps = brk ? __ffs(brk) : KK - 1;
            const bool push = change && lane < steps;
            const uint32_t pmask = __ballot_sync(FULL, push);
            if (push) { IvT<IdxT> pv; pv.x0 = tab_x0<IdxT>(e); pv.x1 = tab_x1<IdxT>(e); pv.x2 = e.z; pv.info = (uint32_t)(x + lane + 1); curr[__popc(pmask & ((1u << lane) - 1u))] = pv; }
            n_curr = (uint32_t)__popc(pmask);
            n_ext += (unsigned long long)steps;
            if (brk) { fwd_done = true; i = x + steps; }
            else {
                uint4 ek;
                ek.x = __shfl_sync(FULL, e.x, KK - 1); ek.y = __shfl_sync(FULL, e.y, KK - 1); ek.z = __shfl_sync(FULL, e.z, KK - 1);
                ek.w = sizeof(IdxT) == 8 ? __shfl_sync(FULL, e.w, KK - 1) : 0u;
                ik.x0 = tab_x0<IdxT>(ek); ik.x1 = tab_x1<IdxT>(ek); ik.x2 = ek.z; ik.info = (uint32_t)(x + KK);
                i = x + KK;
            }
        }
    }
    if (!fwd_done)
    for (; i < len; ++i) {
        if (C.isa && ik.x2 == 1 && min_intv == 1) {
            // unique match q[x .. i): walk to the first base that does not match (or the end of the read) in one go
            const IdxT pos = C.sa[ik.x0];
            const int run = match_run_fwd(C, (IdxT)(pos + (IdxT)(i - x)), q, i, len - i);
            if (run > 0) { i += run; ik.x1 = C.isa[C.n - pos - (IdxT)(i - x)]; ik.info = (uint32_t)i; n_ext += (unsigned long long)run; }
            if (i == len) break;                               // matched to the end: recorded after the loop
            if (q[i] < 4) ++n_ext;                             // the extension the scalar code tries next: it empties the interval
            if (n_curr < list_cap) { if (lane == 0) curr[n_curr] = ik; } else O.ovf = true;
            ++n_curr;
            break;
        }
        const int b = q[i];
        if (b < 4) {
            IvT<IdxT> ok = extend1<IdxT, 0>(C, ik, 3 - b); ++n_ext;
            if (ok.x2 != ik.x2) {
                if (n_curr < list_cap) { if (lane == 0) curr[n_curr] = ik; } else O.ovf = true;
                ++n_curr;
                if (ok.x2 < min_intv) break;
            }
            ik = ok; ik.info = (uint32_t)(i + 1);
        } else {
            if (n_curr < list_cap) { if (lane == 0) curr[n_curr] = ik; } else O.ovf = true;
            ++n_curr;
            break;
        }
    }
    if (i == len) { if (n_curr < list_cap) { if (lane == 0) curr[n_curr] = ik; } else O.ovf = true; ++n_curr; }
    if (n_curr > list_cap) n_curr = list_cap;
    __syncwarp();
    const int ret = (int)curr[n_curr - 1].info;     // the list is consumed backwards (longest match first)
    { IvT<IdxT>* t = curr; curr = prev; prev = t; }
    uint32_t n_prev = n_curr; bool reversed = true;
    const uint32_t out_first = O.n;
    bool have_mem = false; uint32_t last_mem_start = 0;
    if (n_prev <= 32) {
        // Lane k keeps entry k of the list (longest match first) in registers for the whole backward walk.  Every
        // entry walks on its own -- the interval of q[i .. e_k) does not depend on the other entries -- and the list
        // logic of bwt_smem1a reduces to two masks per step: an entry stays in the list iff it survives
        // (size >= min_intv) and its size differs from the nearest surviving longer entry's (an entry with the size
        // of a longer one IS that longer one's occurrence set from here on); a MEM is emitted exactly when the
        // first entry of the list dies (longer matches die first, so nothing survives ahead of it, and its start
        // i + 1 is below every start emitted before).
        const bool own = (uint32_t)lane < n_prev;
        IvT<IdxT> p; p.x0 = 1; p.x1 = 1; p.x2 = 0; p.info = 0;
        if (own) p = prev[n_prev - 1 - (uint32_t)lane];
        uint32_t present = __ballot_sync(FULL, own);
        const uint32_t lt = (1u << lane) - 1u;
        const bool can_uq = C.isa != nullptr && min_intv == 1;
        const bool tab_ok = pk != nullptr;
        const bool fast_ok = tab_ok && !has_n && o.min_seed_len > KK;
        // unique first entry: its walk is one text comparison (uq_stop = the index i at which it dies, uq_x0 = its row then)
        bool uq = false; int uq_stop = 0; IdxT uq_x0 = 0;
        uint32_t ne = 0;
        for (i = x - 1; i >= -1; --i) {
            const int first = __ffs(present) - 1;
            if (can_uq && !uq) {
                const uint32_t fx2 = __shfl_sync(FULL, p.x2, first);
                if (fx2 == 1) {
                    const IdxT fx0 = __shfl_sync(FULL, p.x0, first);
                    const IdxT pos = C.sa[fx0];
                    const int run = match_run_bwd(C, pos, q, i, i + 1);
                    uq = true; uq_stop = i - run; uq_x0 = run > 0 ? C.isa[pos - (IdxT)run] : fx0;
                }
            }
            if (uq && (present & (present - 1)) == 0 && i > uq_stop) { ne += (uint32_t)(i - uq_stop); i = uq_stop; }   // alone: jump
            // Fast steps: while every entry other than a unique first one is short enough for the prefix table (and the read
            // has no ambiguous base, and no entry that dies here can be long enough to be emitted) a step is one table read
            // plus the two masks -- no base test, no Occ hand-off, no emission logic.
            if (fast_ok) {
                bool done = false;
                while (i >= 0 && !(uq && i <= uq_stop)) {
                    const int fst = __ffs(present) - 1;
                    const bool actf = (present >> lane) & 1u;
                    const bool is_uqf = uq && lane == fst;
                    const int lq = (int)p.info - i;
                    if (__any_sync(FULL, actf && !is_uqf && lq > KK)) break;
                    if (!uq && can_uq && __shfl_sync(FULL, p.x2, fst) == 1) break;            // a new unique first entry: general step converts it
                    uint4 e = make_uint4(0u, 0u, 1u, 0u);      // a unique first entry keeps its interval (size 1)
                    if (actf && !is_uqf) {
                        const uint32_t w = __funnelshift_l(pk[(i >> 4) + 1], pk[i >> 4], (i & 15) << 1);
                        e = __ldg(C.kmer_tab + kmer_level_off(lq) + (w >> (32 - 2 * lq)));
                    }
                    const bool alivef = actf && e.z >= min_intv;
                    const uint32_t amask = __ballot_sync(FULL, alivef);
                    const uint32_t bef = amask & lt;
                    const uint32_t psz = __shfl_sync(FULL, e.z, 31 - __clz(bef));
                    const bool keepf = alivef && (bef == 0 || e.z != psz);
                    ne += (uint32_t)__popc(present);
                    present = __ballot_sync(FULL, keepf);
                    if (keepf && !is_uqf) { p.x0 = tab_x0<IdxT>(e); p.x1 = tab_x1<IdxT>(e); p.x2 = e.z; }
                    if (!present) { done = true; break; }
                    --i;
                }
                if (done) break;
                if (uq && (present & (present - 1)) == 0 && i > uq_stop) { ne += (uint32_t)(i - uq_stop); i = uq_stop; }
            }
            const int first2 = __ffs(present) - 1;
            int c = -1;
            if (i >= 0) { c = q[i]; if (c > 3) c = -1; }
            const bool act = (present >> lane) & 1u;
            IdxT nx0 = p.x0, nx1 = p.x1; uint32_t sz = 0;
            if (c >= 0) {
                const bool is_uq = uq && lane == first2;
                if (is_uq) sz = i > uq_stop ? 1u : 0u;
                const int lq = (int)p.info - i;                      // length of the match after prepending q[i]
                // a match of at most KK bases needs no Occ access: its bi-interval is in the prefix table
                const bool by_table = act && !is_uq && tab_ok && lq <= KK;
                if (by_table) {
                    const uint32_t w = __funnelshift_l(pk[(i >> 4) + 1], pk[i >> 4], (i & 15) << 1);
                    const uint4 e = __ldg(C.kmer_tab + kmer_level_off(lq) + (w >> (32 - 2 * lq)));
                    nx0 = tab_x0<IdxT>(e); nx1 = tab_x1<IdxT>(e); sz = e.z;
                }
                uint32_t todo = __ballot_sync(FULL, act && !is_uq && !by_table);
                ne += (uint32_t)__popc(present);
                while (todo) {
                    // the four lowest pending entries go through the warp's hand-off slots: group g (lanes 8g..8g+7)
                    // extends the entry in slot g and its leader writes the result back
                    const int rank = __popc(todo & lt);
                    const bool mine = ((todo >> lane) & 1u) && rank < 4;
                    if (mine) hand[rank] = p;
                    __syncwarp();
                    const int g = lane >> 3;
                    const bool gv = g < __popc(todo);
                    IvT<IdxT> pg = hand[g];
                    const IvT<IdxT> og = extend4_back(C, pg, c, gv);
                    __syncwarp();
                    if ((lane & 7) == 0) hand[g] = og;
                    __syncwarp();
                    if (mine) { const IvT<IdxT> r = hand[rank]; nx0 = r.x0; nx1 = r.x1; sz = r.x2; }
                    __syncwarp();
                    todo &= todo - 1; todo &= todo - 1; todo &= todo - 1; todo &= todo - 1;
                }
            }
            const bool alive = act && sz >= min_intv;
            const uint32_t alive_mask = __ballot_sync(FULL, alive);
            if (!((alive_mask >> first2) & 1u)) {
                const uint32_t pinfo = __shfl_sync(FULL, p.info, first2);
                if ((int)pinfo - (i + 1) >= o.min_seed_len) {
                    if (O.n < O.cap) {
                        if (lane == first2) { Intv v; v.x0 = uq ? uq_x0 : p.x0; v.x1 = p.x1; v.x2 = p.x2; v.info = (uint64_t)(uint32_t)(i + 1) << 32 | p.info; O.out[O.n] = v; }
                    } else O.ovf = true;
                    ++O.n;
                }
                uq = false;
            }
            const uint32_t before = alive_mask & lt;                         // surviving entries ahead of mine
            const uint32_t prev_sz = __shfl_sync(FULL, sz, 31 - __clz(before));   // (lane 31 when there is none: unused)
            const bool keep = alive && (before == 0 || sz != prev_sz);
            present = __ballot_sync(FULL, keep);
            if (keep) { p.x0 = nx0; p.x1 = nx1; p.x2 = sz; }
            if (!present) break;
        }
        n_ext += ne;
    } else
    for (i = x - 1; i >= -1; --i) {
        // more entries than lanes (highly repetitive reads): the list logic of bwt_smem1a, one entry at a time
        const int c = i < 0 ? -1 : (q[i] < 4 ? q[i] : -1);
        n_curr = 0;
        uint32_t last_x2 = 0;
        for (uint32_t j = 0; j < n_prev; ++j) {
            const IvT<IdxT> p = prev[reversed ? n_prev - 1 - j : j];
            IvT<IdxT> ok; ok.x2 = 0;
            if (c >= 0) { ok = extend1<IdxT, 1>(C, p, c); ++n_ext; }
            if (c < 0 || ok.x2 < min_intv) {
                if (n_curr == 0) {
                    if (!have_mem || (uint32_t)(i + 1) < last_mem_start) {
                        const int slen = (int)p.info - (i + 1);
                        if (slen >= o.min_seed_len) emit(O, p, (uint32_t)(i + 1), p.info);
                        have_mem = true; last_mem_start = (uint32_t)(i + 1);
                    }
                }
            } else if (n_curr == 0 || ok.x2 != last_x2) {
                if (lane == 0) curr[n_curr] = ok;    // n_curr < n_prev <= list_cap
                ++n_curr; last_x2 = ok.x2;
            }
        }
        if (n_curr == 0) break;
        __syncwarp();
        { IvT<IdxT>* t = curr; curr = prev; prev = t; }
        n_prev = n_curr; reversed = false;
    }
    // emitted in decreasing start order: reverse the appended segment
    __syncwarp();
    {
        const uint32_t hi = O.n < O.cap ? O.n : O.cap;
        if (hi > out_first + 1) {
            const uint32_t cnt = hi - out_first;
            for (uint32_t k = lane; k < cnt / 2; k += 32) {
                Intv a = O.out[out_first + k], b = O.out[hi - 1 - k];
                O.out[out_first + k] = b; O.out[hi - 1 - k] = a;
            }
            __syncwarp();
        }
    }
    return ret;
}

template <class IdxT>
__device__ __forceinline__ int seed_strategy1(const Ctx<IdxT>& C, int len, const uint8_t* q, int x, int min_len, uint32_t max_intv, Out& O,
                                              unsigned long long& n_ext, const uint32_t* pk, bool has_n) {
    if (q[x] > 3) return x + 1;
    IvT<IdxT> ik = set_intv(C, q[x]);
    int i = x + 1;
    // The first kk - 1 extensions can neither emit (i - x < min_len) nor be observed: take their result from the
    // k-mer table when the next kk bases are all ACGT (an ambiguous base ends the walk, which the plain loop handles)
    if (C.kmer_tab && min_len >= C.kk && x + C.kk <= len) {
        uint32_t w;
        if (kmer_word(q, pk, has_n, x, C.kk, w)) {
            const uint4 e = __ldg(C.kmer_tab + kmer_level_off(C.kk) + (w >> (32 - 2 * C.kk)));
            ik.x0 = tab_x0<IdxT>(e); ik.x1 = tab_x1<IdxT>(e); ik.x2 = e.z;
            i = x + C.kk; n_ext += C.kk - 1;   // the roofline unit stays the reference's count of bwt_extend calls
        }
    }
    for (; i < len; ++i) {
        if (C.isa && ik.x2 == 1 && max_intv > 1 && i - x <= min_len) {
            // unique match q[x .. i): the walk ends at j = x + min_len (emit iff still matching), at an ambiguous base
            // (nothing emitted), or at the end of the read
            const int stop = x + min_len;                       // index of the base whose extension triggers the emission test
            const int lim = (stop < len ? stop + 1 : len) - i;  // bases q[i .. i + lim) are looked at
            const int lane = C.lane;
            bool isn = false;
            if (lane < lim) isn = q[i + lane] > 3;              // lim <= min_len + 1 - (i - x) <= 32 for min_seed_len <= 31
            const uint32_t nmask = __ballot_sync(FULL, isn);
            const IdxT pos = C.sa[ik.x0];
            const int run = match_run_fwd(C, (IdxT)(pos + (IdxT)(i - x)), q, i, lim);
            if (nmask) { const int jn = i + __ffs(nmask) - 1; n_ext += (unsigned long long)(jn - i); return jn + 1; }
            n_ext += (unsigned long long)lim;
            if (stop >= len) return len;
            if (run == lim) {
                IvT<IdxT> ok = ik;
                ok.x1 = C.isa[C.n - pos - (IdxT)(stop + 1 - x)]; ok.x2 = 1;
                emit(O, ok, (uint32_t)x, (uint32_t)(stop + 1));
            }
            return stop + 1;
        }
        const int b = q[i];
        if (b < 4) {
            IvT<IdxT> ok = extend1<IdxT, 0>(C, ik, 3 - b); ++n_ext;
            if (ok.x2 < max_intv && i - x >= min_len) {
                if (ok.x2 > 0) emit(O, ok, (uint32_t)x, (uint32_t)(i + 1));
                return i + 1;
            }
            ik = ok;
        } else return i + 1;
    }
    return len;
}

// the three passes of mem_collect_intv for one read
template <class IdxT>
__device__ __forceinline__ void collect_intv(const Ctx<IdxT>& C, const DevOpts& o, int len, const uint8_t* q, IvT<IdxT>* la, IvT<IdxT>* lb,
                                             uint32_t list_cap, Out& O, unsigned long long& n_ext, const uint32_t* pk, bool has_n, IvT<IdxT>* hand) {
    // passes 1 and 2 share ONE inlined copy of smem1 (the kernel's largest function): a two-state loop feeds it
    // first every SMEM start (pass 1), then the middle of each long, rare SMEM of pass 1 (pass 2: re-seeding)
    int x = 0;
    uint32_t old_n = 0, k = 0;
    bool pass2 = false;
    for (;;) {
        int sx; uint32_t mi;
        if (!pass2) {
            while (x < len && q[x] > 3) ++x;
            if (x >= len) { pass2 = true; old_n = O.n < O.cap ? O.n : O.cap; k = 0; continue; }
            sx = x; mi = 1;
        } else {
            bool found = false;
            for (; k < old_n; ++k) {
                const Intv p = O.out[k];
                const int start = (int)(p.info >> 32), end = (int)(uint32_t)p.info;
                if (end - start < o.split_len || p.x2 > (uint64_t)o.split_width) continue;
                sx = (start + end) >> 1; mi = (uint32_t)p.x2 + 1; found = true; ++k;
                break;
            }
            if (!found) break;
        }
        const int r = smem1(C, o, len, q, sx, mi, la, lb, list_cap, O, n_ext, pk, has_n, hand);
        if (!pass2) x = r;
    }
    if (o.max_mem_intv > 0) {                // pass 3: LAST-like
        x = 0;
        const int min_len = o.min_seed_len, L = min_len + 1;    // a seed of this pass is the first L-mer with < max_mem_intv occurrences
        // The walk x -> f(x) is sequential, but f is a pure function of x and almost always returns x + L.  Lane t therefore
        // evaluates f(x + t L) on its own -- K-mer from the prefix table, then (unique K-mer) one text comparison of the
        // remaining L - K bases -- so the dependent loads of up to 32 starts are in flight together; the chain then consumes
        // the results in order for as long as each start is the predicted one and was decidable without Occ.
        const bool spec_ok = C.kmer_tab != nullptr && pk != nullptr && !has_n &&
                             min_len >= C.kk && o.max_mem_intv > 1 && L <= 32;
        const int lane = C.lane;
        while (x < len) {
            if (spec_ok) {
                if (x + L > len) { n_ext += (unsigned long long)(len - 1 - x); break; }   // too short to emit: only the extension count remains
                const int xs = x + L * lane;
                int state = 0;                     // 0 undecided (needs Occ) or out of range, 1 no seed, 2 seed
                IdxT r0 = 0, r1 = 0;
                if (xs + L <= len) {
                    const uint32_t w = __funnelshift_l(pk[(xs >> 4) + 1], pk[xs >> 4], (xs & 15) << 1);
                    const uint4 e = __ldg(C.kmer_tab + kmer_level_off(C.kk) + (w >> (32 - 2 * C.kk)));
                    if (e.z == 0) state = 1;
                    else if (e.z == 1) {
                        const IdxT pos = C.sa[tab_x0<IdxT>(e)];
                        bool ok = pos + (IdxT)L <= C.n;
                        for (int k = C.kk; ok && k < L; ++k) ok = text_base(C, (IdxT)(pos + (IdxT)k)) == (uint32_t)q[xs + k];
                        state = ok ? 2 : 1;
                        if (ok) { r0 = tab_x0<IdxT>(e); r1 = C.isa[C.n - pos - (IdxT)L]; }
                    }
                }
                const uint32_t decided = __ballot_sync(FULL, state != 0);
                const int run = decided == 0xffffffffu ? 32 : __ffs(~decided) - 1;   // leading starts that are decided (0 => lane 0 needs the general walk)
                if (run > 0) {
                    const uint32_t runmask = run >= 32 ? 0xffffffffu : ((1u << run) - 1u);
                    const uint32_t em = __ballot_sync(FULL, state == 2) & runmask;
                    if (state == 2 && lane < run) {
                        const uint32_t k = O.n + (uint32_t)__popc(em & ((1u << lane) - 1u));
                        if (k < O.cap) { Intv v; v.x0 = r0; v.x1 = r1; v.x2 = 1; v.info = (uint64_t)(uint32_t)xs << 32 | (uint32_t)(xs + L); O.out[k] = v; }
                    }
                    if (O.n + (uint32_t)__popc(em) > O.cap) O.ovf = true;
                    O.n += (uint32_t)__popc(em);
                    n_ext += (unsigned long long)run * (unsigned long long)min_len;
                    x += run * L;
                    continue;
                }
            }
            if (q[x] < 4) x = seed_strategy1(C, len, q, x, min_len, (uint32_t)o.max_mem_intv, O, n_ext, pk, has_n);
            else ++x;
        }
    }
}

// ---------------------------------------------------------------- k-mer table of the LAST-like pass
// Level-by-level: the 4^t intervals of level t come from one forward bwt_extend of each level t-1 interval
// (all four children at once, scalar Occ4 per thread).  Entry of k-mer b0 b1 .. b_{K-1} sits at index sum b_t 4^{K-1-t}.
template <class IdxT>
__device__ __forceinline__ void occ4_scalar(const uint32_t* occ, IdxT primary, IdxT k, IdxT cnt[4]) {
    k -= (k >= primary);
    const uint4* blk = reinterpret_cast<const uint4*>(occ + ((size_t)(k >> 7) << 4));
    const uint4 ca = __ldg(blk), cb = __ldg(blk + 1), s0 = __ldg(blk + 2), s1 = __ldg(blk + 3);
    if (sizeof(IdxT) == 4) { cnt[0] = (IdxT)ca.x; cnt[1] = (IdxT)ca.z; cnt[2] = (IdxT)cb.x; cnt[3] = (IdxT)cb.z; }
    else {
        cnt[0] = (IdxT)((unsigned long long)ca.y << 32 | ca.x); cnt[1] = (IdxT)((unsigned long long)ca.w << 32 | ca.z);
        cnt[2] = (IdxT)((unsigned long long)cb.y << 32 | cb.x); cnt[3] = (IdxT)((unsigned long long)cb.w << 32 | cb.z);
    }
    const int within = (int)(k & 127) + 1;
    const uint32_t w8[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        int nsym = within - (w << 4);
        nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
        const uint32_t keep = __funnelshift_rc(0u, 0x55555555u, 2 * nsym);
        const uint32_t lo = w8[w] & keep, hi = (w8[w] >> 1) & keep, nlo = ~w8[w] & keep, nhi = ~(w8[w] >> 1) & keep;
        cnt[0] += __popc(nhi & nlo); cnt[1] += __popc(nhi & lo); cnt[2] += __popc(hi & nlo); cnt[3] += __popc(hi & lo);
    }
}

template <class IdxT> struct L2Vals { IdxT v[5]; };

template <class IdxT>
__global__ void k_kmer_level(const uint4* __restrict__ parent, uint4* __restrict__ child, uint32_t n_parent, const uint32_t* __restrict__ occ,
                             IdxT primary, L2Vals<IdxT> L2) {
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_parent; p += gridDim.x * blockDim.x) {
        const uint4 ik = parent[p];   // x0, x1, x2
        const IdxT ix0 = tab_x0<IdxT>(ik), ix1 = tab_x1<IdxT>(ik);
        IdxT tk[4], tl[4];
        occ4_scalar<IdxT>(occ, primary, ix1 - 1, tk);
        occ4_scalar<IdxT>(occ, primary, ix1 - 1 + ik.z, tl);
        IdxT x1[4], x0[4]; uint32_t sz[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { x1[c] = L2.v[c] + 1 + tk[c]; sz[c] = (uint32_t)(tl[c] - tk[c]); }
        x0[3] = ix0 + (IdxT)(ix1 <= primary && ix1 + ik.z - 1 >= primary);
        x0[2] = x0[3] + sz[3]; x0[1] = x0[2] + sz[2]; x0[0] = x0[1] + sz[1];
#pragma unroll
        for (int b = 0; b < 4; ++b) {   // appending base b = taking ok[3 - b] of a forward extension (SURVEY A.2)
            const int c = 3 - b;
            child[(size_t)p * 4 + b] = tab_entry(x0[c], x1[c], ik.z ? sz[c] : 0u);
        }
    }
}
template <class IdxT>
__global__ void k_kmer_level0(uint4* out, L2Vals<IdxT> L2) {
    const int c = threadIdx.x;
    if (c < 4) out[c] = tab_entry(L2.v[c] + 1, L2.v[3 - c] + 1, (uint32_t)(L2.v[c + 1] - L2.v[c]));
}

template <class IdxT>
__global__ void k_build_isa(const IdxT* __restrict__ sa, uint64_t rows, IdxT* __restrict__ isa) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (uint64_t)gridDim.x * blockDim.x) isa[sa[r]] = (IdxT)r;
}

// sort a read's intervals by info (ties are bit-identical records, so any correct sort equals ks_introsort's result)
__device__ void sort_by_info(Intv* out, uint32_t n_out, Intv* tmp, uint32_t tmp_cap, uint32_t* overflow) {
    const int lane = lane_id();
    if (n_out <= 1) return;
    if (n_out <= 32) {   // one record per lane, ranks by shuffle
        Intv me; me.x0 = me.x1 = me.x2 = 0; me.info = ~0ull;
        if ((uint32_t)lane < n_out) me = out[lane];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n_out; ++j) {
            uint64_t oi = __shfl_sync(FULL, me.info, (int)j);
            rank += (oi < me.info) || (oi == me.info && j < (uint32_t)lane);
        }
        __syncwarp();
        if ((uint32_t)lane < n_out) out[rank] = me;
        __syncwarp();
        return;
    }
    if (n_out > tmp_cap) { if (lane == 0) atomicExch(overflow, 1u); return; }
    for (uint32_t base = 0; base < n_out; base += 32) {
        uint32_t k = base + lane;
        if (k < n_out) {
            Intv me = out[k];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < n_out; ++j) {
                uint64_t oi = out[j].info;
                rank += (oi < me.info) || (oi == me.info && j < k);
            }
            tmp[rank] = me;
        }
    }
    __syncwarp();
    for (uint32_t k = lane; k < n_out; k += 32) out[k] = tmp[k];
    __syncwarp();
}

// IdxT = uint32_t while the text has fewer than 2^32 rows; SMEM: interval lists and the read staged in shared
// memory (otherwise in the per-warp global scratch: reads too long for shared memory)
template <class IdxT, bool SMEM, int MINB>
__global__ void __launch_bounds__(SEED_THREADS, MINB) seed_smem(SeedParams P, DevIndex ix, DevOpts o) {
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    __shared__ IdxT sL2[8];
    __shared__ IvT<IdxT> s_hand[SEED_WARPS][4];   // hand-off slots of the grouped backward extensions
    // lane / warp index: read the special register once and make the values opaque, otherwise the compiler re-issues S2R
    // (a long-scoreboard instruction) wherever they are used inside the hot loops
    int tid = threadIdx.x;
    asm volatile("" : "+r"(tid));
    const int warp_in_cta = tid >> 5;
    IvT<IdxT>* hand = s_hand[warp_in_cta];
    const IdxT* sL2p = sL2;
    asm volatile("" : "+l"(hand), "+l"(sL2p));      // formed once: re-deriving a generic address of shared memory costs an S2UR each time
    if (tid < 5) sL2[tid] = (IdxT)ix.L2[tid];
    __syncthreads();
    using Iv = IvT<IdxT>;
    const int lane = tid & 31;
    const uint32_t gwarp = (blockIdx.x * SEED_THREADS + (uint32_t)tid) >> 5;
    Intv* gl = P.scratch + (size_t)gwarp * 3 * P.list_cap;     // global scratch: lists of long reads, big-sort buffer
    unsigned long long n_ext = 0;
    Ctx<IdxT> C;
    C.occ = ix.occ; C.sL2 = sL2p; C.primary = (IdxT)ix.primary; C.kmer_tab = P.kmer_tab; C.kk = P.kmer_k; C.lane = lane;
    C.sa = reinterpret_cast<const IdxT*>(ix.sa); C.isa = reinterpret_cast<const IdxT*>(P.isa); C.pac = ix.pac; C.l_pac = (IdxT)ix.l_pac; C.n = (IdxT)ix.seq_len;
    {
        const int idx = lane & 15;
        C.sym_base = idx >= 8 ? (uint32_t)((idx - 8) << 4) : (1u << 20);
        C.cnt_sym = (idx < 8 && !(idx & 1)) ? (idx >> 1) : -1;
        C.cnt_hi = (idx < 8 && (idx & 1)) ? (idx >> 1) : -1;
        C.lhalf = (lane & 16) != 0;
        // lanes holding the high half of a checkpoint act as symbol lanes with zero symbols: they contribute 0 to eq / gt
    }
    Iv* la; Iv* lb; uint8_t* sq = nullptr;
    if (SMEM) {
        la = reinterpret_cast<Iv*>(dyn_smem) + (size_t)warp_in_cta * 2 * P.list_cap; lb = la + P.list_cap;
        sq = dyn_smem + (size_t)SEED_WARPS * 2 * P.list_cap * sizeof(Iv) + (size_t)warp_in_cta * P.read_cap;
    } else { la = reinterpret_cast<Iv*>(gl); lb = la + P.list_cap; }
    const uint32_t n_todo = P.todo ? *P.todo_cnt : P.n_reads;     // with the thread pass on: only the reads it queued
    for (;;) {
        const uint32_t tk = next_ticket(P.ticket);
        if (tk >= n_todo) break;
        const uint32_t r = P.todo ? P.todo[tk] : tk;
        const uint8_t* q = P.seqs + P.offs[r];
        const int len = (int)(P.offs[r + 1] - P.offs[r]);
        Out O; O.out = P.out + (size_t)r * P.cap; O.n = 0; O.cap = P.cap; O.ovf = false; O.lane = lane;
        if (len >= o.min_seed_len) {   // mem_chain returns before seeding otherwise (SURVEY A.5)
            if (SMEM) {
                __syncwarp();
                bool amb = false;
                for (int i = lane; i < len; i += 32) { const uint8_t b = q[i]; sq[i] = b; amb = amb || b > 3; }
                const bool has_n = __any_sync(FULL, amb);
                __syncwarp();
                // 2-bit packed copy of the read (16 bases per word, MSB first) for k-mer indices of arbitrary substrings
                uint32_t* pk = nullptr;
                if (C.kmer_tab) {
                    pk = reinterpret_cast<uint32_t*>(sq + ((len + 15) & ~15));
                    for (int w = lane; w <= (len >> 4) + 1; w += 32) {
                        uint32_t v = 0;
                        for (int k = 0; k < 16; ++k) { const int pos = (w << 4) + k; v = v << 2 | (pos < len ? (sq[pos] & 3u) : 0u); }
                        pk[w] = v;
                    }
                    __syncwarp();
                }
                collect_intv(C, o, len, sq, la, lb, P.list_cap, O, n_ext, pk, has_n, hand);
            } else collect_intv(C, o, len, q, la, lb, P.list_cap, O, n_ext, (const uint32_t*)nullptr, true, hand);
            __syncwarp();
        }
        uint32_t n_out = O.n;
        if (O.ovf || n_out > P.cap) { if (lane == 0) atomicExch(P.overflow, 1u); n_out = n_out < P.cap ? n_out : P.cap; }
        sort_by_info(O.out, n_out, gl, 3 * P.list_cap, P.overflow);
        if (lane == 0) P.out_cnt[r] = n_out;
    }
    if (P.n_extend && lane == 0 && n_ext) atomicAdd(P.n_extend, n_ext);
}

// ---------------------------------------------------------------- thread-per-read passes (seed_thread.cuh)
// Three kernels.  seed_pack turns every read into its 2-bit packed copy (16 bases per word) and flags the reads the thread code does
// not take.  seed_calls runs passes 1 and 2 of mem_collect_intv -- every bwt_smem1a call -- with PERSISTENT LANES: a lane works
// through the calls of its read and fetches the next read as soon as it has none left, so that in every round all 32 lanes of a
// warp carry a call (reads differ a lot in how many calls they need: one per sequencing error); inside a round the lanes walk the
// list entry by list entry, loop counters being warp votes (seed_thread.cuh).  seed_last, thread per read, runs the LAST-like
// pass, ranks the read's intervals by `info` and writes them in order; reads the thread code declined go to `todo` for seed_smem.
// The reads' packed copies and the P(b) arrays live in shared memory laid out [word][thread] (bank = lane); intervals are staged
// unsorted in the upper half of the read's output slots.
constexpr int ST_THREADS = 128;
constexpr uint32_t ST_FAIL = 0xffffffffu;
enum { STF_FALLBACK = 1, STF_EMPTY = 2 };      // read flags: not for the thread code (ambiguous base / too long); shorter than a seed

__global__ void seed_pack(SeedParams P, int min_seed_len, int words) {
    const uint64_t total = (uint64_t)P.n_reads * (uint32_t)words;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)(t / (uint32_t)words); const int w = (int)(t % (uint32_t)words);
        const uint64_t off = P.offs[r];
        const int len = (int)(P.offs[r + 1] - off);
        uint32_t v = 0, amb = 0;
        const int b0 = w << 4;
        if ((len >> 4) + 3 <= words && b0 < len) {
            const uint8_t* q = P.seqs + off + b0;
            const int nb = len - b0 < 16 ? len - b0 : 16;
            for (int k = 0; k < nb; ++k) { const uint32_t c = q[k]; amb |= c; v |= (c & 3u) << (30 - 2 * k); }
        }
        P.pk[t] = v;
        uint32_t f = amb > 3 ? (uint32_t)STF_FALLBACK : 0u;
        if (w == 0) { if (len < min_seed_len) f |= STF_EMPTY; else if ((len >> 4) + 3 > words) f |= STF_FALLBACK; }
        if (f) atomicOr(P.rflag + r, f);
    }
}

template <class IdxT> __device__ __forceinline__ seedt::Index<IdxT> st_index(const SeedParams& P, const DevIndex& ix) {
    seedt::Index<IdxT> X;
    X.occ = ix.occ; X.tab = reinterpret_cast<const seedt::U4*>(P.kmer_tab); X.kk = P.kmer_k; X.ztab = P.kmer_ztab;
    X.sa = reinterpret_cast<const IdxT*>(ix.sa); X.isa = reinterpret_cast<const IdxT*>(P.isa); X.pac = ix.pac;
    X.l_pac = (IdxT)ix.l_pac; X.n = (IdxT)ix.seq_len; X.primary = (IdxT)ix.primary;
#pragma unroll
    for (int c = 0; c < 5; ++c) X.L2[c] = (IdxT)ix.L2[c];
    return X;
}

template <class IdxT>
__global__ void __launch_bounds__(ST_THREADS) seed_calls(SeedParams P, DevIndex ix, DevOpts o, uint32_t* ticket, int words) {
    extern __shared__ __align__(16) uint32_t st_pk[];      // [words][ST_THREADS] packed reads, then [PCAP][ST_THREADS] P(b) arrays
    uint32_t* st_pc = st_pk + (size_t)words * ST_THREADS;
    const int tid = threadIdx.x, lane = tid & 31;
    const seedt::Index<IdxT> X = st_index<IdxT>(P, ix);
    seedt::Opts so; so.min_seed_len = o.min_seed_len; so.split_len = o.split_len; so.split_width = o.split_width; so.max_mem_intv = o.max_mem_intv;
    const uint32_t half = P.cap / 2;                 // sorted records go to slots [0, half), the staging is [cap - half, cap)
    const uint32_t stage_cap = half < (uint32_t)seedt::PCAP ? half : (uint32_t)seedt::PCAP;
    seedt::Read R; R.pk = st_pk + tid; R.stride = ST_THREADS; R.len = 0;
    seedt::Work<IdxT> W;
    seedt::work_init(W, (seedt::IntvOut*)nullptr, stage_cap, st_pc + tid, ST_THREADS);
    seedt::Calls C; seedt::calls_init(C);
    uint32_t r = ST_FAIL;                            // the lane's read (ST_FAIL = none)
    bool dry = false;                                // the queue of reads is exhausted
    for (;;) {
        // ---- every lane gets a call: the next one of its read, or the first one of a new read
        int x = 0; uint32_t mi = 1; bool has = false;
        for (;;) {
            if (r != ST_FAIL && !has) {
                has = seedt::next_call(C, so, R, W, &x, &mi);
                if (!has) {                           // passes 1 and 2 of this read are done
                    P.cnt12[r] = W.fail ? ST_FAIL : W.n_out; P.ext12[r] = (uint32_t)W.n_ext;
                    r = ST_FAIL;
                }
            }
            const bool need = r == ST_FAIL && !dry;
            const uint32_t nm = __ballot_sync(FULL, need);
            if (!nm) break;
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(ticket, (uint32_t)__popc(nm));
            base = __shfl_sync(FULL, base, 0);
            if (need) {
                const uint32_t rr = base + (uint32_t)__popc(nm & ((1u << lane) - 1u));
                if (rr >= P.n_reads) dry = true;
                else if (P.rflag[rr] == 0) {
                    r = rr;
                    const uint32_t* src = P.pk + (size_t)rr * (uint32_t)words;
                    for (int w = 0; w < words; ++w) st_pk[w * ST_THREADS + tid] = src[w];
                    R.len = (int)(P.offs[rr + 1] - P.offs[rr]);
                    seedt::work_init(W, reinterpret_cast<seedt::IntvOut*>(P.out + (size_t)rr * P.cap + (P.cap - half)), stage_cap, st_pc + tid, ST_THREADS);
                    seedt::calls_init(C);
                }
            }
        }
        if (!__any_sync(FULL, has)) break;
        // ---- one bwt_smem1a call per lane: forward walk, then the backward walk entry by entry
        if (has) seedt::smem_forward(X, R, x, mi, W);
        const int ncol = has && !W.fail ? W.n : 0;
        for (int k = 0; __any_sync(FULL, k < ncol); ++k) seedt::smem_column(X, so, R, k, W, k < ncol && !W.fail);
        if (has && C.pass == 1) C.next_x = W.ret;
    }
}

template <class IdxT>
__global__ void __launch_bounds__(ST_THREADS) seed_last(SeedParams P, DevIndex ix, DevOpts o, int words) {
    extern __shared__ __align__(16) uint32_t st_pk[];
    uint32_t* st_pc = st_pk + (size_t)words * ST_THREADS;
    const int tid = threadIdx.x, lane = tid & 31;
    const seedt::Index<IdxT> X = st_index<IdxT>(P, ix);
    seedt::Opts so; so.min_seed_len = o.min_seed_len; so.split_len = o.split_len; so.split_width = o.split_width; so.max_mem_intv = o.max_mem_intv;
    const uint32_t half = P.cap / 2;
    const uint32_t stage_cap = half < (uint32_t)seedt::PCAP ? half : (uint32_t)seedt::PCAP;
    unsigned long long n_ext_sum = 0;
    for (uint32_t base = blockIdx.x * ST_THREADS; base < P.n_reads; base += gridDim.x * ST_THREADS) {
        const uint32_t r = base + (uint32_t)tid;
        bool fail = false;
        if (r < P.n_reads) {
            const uint32_t fl = P.rflag[r], c12 = P.cnt12[r];
            if (fl & STF_EMPTY) P.out_cnt[r] = 0;                                   // mem_chain returns before seeding (SURVEY A.5)
            else if (fl || c12 == ST_FAIL) fail = true;
            else {
                const uint32_t* src = P.pk + (size_t)r * (uint32_t)words;
                for (int w = 0; w < words; ++w) st_pk[w * ST_THREADS + tid] = src[w];
                seedt::Read R; R.pk = st_pk + tid; R.stride = ST_THREADS; R.len = (int)(P.offs[r + 1] - P.offs[r]);
                Intv* slots = P.out + (size_t)r * P.cap;
                seedt::Work<IdxT> W;
                seedt::work_init(W, reinterpret_cast<seedt::IntvOut*>(slots + (P.cap - half)), stage_cap, st_pc + tid, ST_THREADS);
                W.n_out = c12;
                seedt::last_like_pass(X, so, R, W);
                fail = W.fail;
                if (!fail) {
                    // rank by info: key = start | end | staging index (9 + 9 + 6 bits; reads of at most 496 bases, at most 64 records);
                    // the keys live in the lane's P(b) array, which is free here
                    uint32_t* key = st_pc + tid;
                    const uint32_t n = W.n_out;
                    for (uint32_t k = 0; k < n; ++k) {
                        const uint64_t info = W.out[k].info;
                        uint32_t kk = (uint32_t)(info >> 32) << 15 | ((uint32_t)info & 0x1ffu) << 6 | k;
                        uint32_t j = k;
                        while (j > 0 && key[(j - 1) * ST_THREADS] > kk) { key[j * ST_THREADS] = key[(j - 1) * ST_THREADS]; --j; }
                        key[j * ST_THREADS] = kk;
                    }
                    for (uint32_t k = 0; k < n; ++k) slots[k] = reinterpret_cast<const Intv*>(W.out)[key[k * ST_THREADS] & 63u];
                    P.out_cnt[r] = n;
                    n_ext_sum += W.n_ext + P.ext12[r];
                }
            }
        }
        const uint32_t fm = __ballot_sync(FULL, fail);
        if (fm) {
            uint32_t at = 0;
            if (lane == 0) at = atomicAdd(const_cast<uint32_t*>(P.todo_cnt), (uint32_t)__popc(fm));
            at = __shfl_sync(FULL, at, 0);
            if (fail) const_cast<uint32_t*>(P.todo)[at + (uint32_t)__popc(fm & ((1u << lane) - 1u))] = r;
        }
    }
    if (P.n_extend) {
#pragma unroll
        for (int d = 16; d; d >>= 1) n_ext_sum += __shfl_xor_sync(FULL, n_ext_sum, d);
        if (lane == 0 && n_ext_sum) atomicAdd(P.n_extend, n_ext_sum);
    }
}

template <class IdxT> size_t lists_bytes(uint32_t list_cap, uint32_t read_cap) {
    return (size_t)SEED_WARPS * (2 * (size_t)list_cap * sizeof(IvT<IdxT>) + read_cap);
}

template <class IdxT, bool SMEM, int MINB> void launch_mode(const SeedParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, size_t smem, int* n_warps_out) {
    const int sms = cached_sm_count();
    int nb = cached_blocks_per_sm(seed_smem<IdxT, SMEM, MINB>, SEED_THREADS, smem);
    if (nb * SEED_WARPS > 64) nb = 64 / SEED_WARPS;
    if (n_warps_out) *n_warps_out = nb * sms * SEED_WARPS;
    seed_smem<IdxT, SMEM, MINB><<<nb * sms, SEED_THREADS, smem, st>>>(p, ix, o);
}

}  // namespace

size_t kmer_table_bytes(int k) { return (size_t)kmer_level_off(k + 1) * sizeof(uint4); }

static __global__ void k_kmer_sizes(const uint4* __restrict__ tab, uint32_t* __restrict__ ztab, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) ztab[i] = tab[i].z;
}
// the sizes-only copy of the prefix table (kmer_table_bytes(k) / 4 bytes)
void build_kmer_sizes(const void* tab, uint32_t* ztab, int k, cudaStream_t st, uint64_t* launches) {
    const uint64_t n = kmer_level_off(k + 1);
    k_kmer_sizes<<<148 * 16, 256, 0, st>>>(reinterpret_cast<const uint4*>(tab), ztab, n);
    if (launches) ++*launches;
}

// depth of the prefix table for a text of n symbols: ceil(log4 n), within [8, KMER_K_MAX]
int kmer_table_depth(uint64_t n) {
    int k = 8;
    while (k < KMER_K_MAX && (1ull << (2 * k)) < n) ++k;
    return k;
}

// builds levels 1..k of the prefix table into `tab` (kmer_table_bytes(k)); rows of up to 40 bits
template <class IdxT>
static void build_kmer_table_t(const DevIndex& ix, void* tab, int k, cudaStream_t st, uint64_t* launches) {
    uint4* base = reinterpret_cast<uint4*>(tab);
    L2Vals<IdxT> L2;
    for (int c = 0; c < 5; ++c) L2.v[c] = (IdxT)ix.L2[c];
    k_kmer_level0<IdxT><<<1, 32, 0, st>>>(base + kmer_level_off(1), L2);
    if (launches) ++*launches;
    uint32_t n = 4;
    for (int t = 2; t <= k; ++t) {
        const unsigned blocks = (unsigned)std::min<uint32_t>((n + 255) / 256, 148u * 16u);
        k_kmer_level<IdxT><<<blocks ? blocks : 1, 256, 0, st>>>(base + kmer_level_off(t - 1), base + kmer_level_off(t), n, ix.occ, (IdxT)ix.primary, L2);
        if (launches) ++*launches;
        n *= 4;
    }
}
void build_kmer_table(const DevIndex& ix, void* tab, int k, cudaStream_t st, uint64_t* launches) {
    if (ix.sa_bytes == 8) build_kmer_table_t<uint64_t>(ix, tab, k, st, launches);
    else build_kmer_table_t<uint32_t>(ix, tab, k, st, launches);
}

// inverse suffix array: isa[SA[r]] = r for the n + 1 rows; `isa` holds n + 1 entries of ix.sa_bytes bytes
void build_isa(const DevIndex& ix, void* isa, cudaStream_t st, uint64_t* launches) {
    const uint64_t rows = ix.seq_len + 1;
    const unsigned blocks = (unsigned)std::min<uint64_t>((rows + 255) / 256, 148ull * 16);
    if (ix.sa_bytes == 8) k_build_isa<uint64_t><<<blocks, 256, 0, st>>>(reinterpret_cast<const uint64_t*>(ix.sa), rows, reinterpret_cast<uint64_t*>(isa));
    else k_build_isa<uint32_t><<<blocks, 256, 0, st>>>(reinterpret_cast<const uint32_t*>(ix.sa), rows, reinterpret_cast<uint32_t*>(isa));
    if (launches) ++*launches;
}

int seed_resident_warps() {
    // upper bound used to size the per-warp global scratch: 64 warps per SM
    return 64 * cached_sm_count();
}

bool seed_lists_fit_smem(uint32_t list_cap, uint32_t read_cap, int sa_bytes) {
    const size_t b = sa_bytes == 8 ? lists_bytes<uint64_t>(list_cap, read_cap) : lists_bytes<uint32_t>(list_cap, read_cap);
    return b <= 72 * 1024;
}

void launch_seed(const SeedParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, int* n_warps_out) {
    const bool wide = ix.sa_bytes == 8;   // 64-bit row indices
    if (wide) {
        if (p.lists_in_smem) launch_mode<uint64_t, true, 3>(p, ix, o, st, lists_bytes<uint64_t>(p.list_cap, p.read_cap), n_warps_out);
        else launch_mode<uint64_t, false, 1>(p, ix, o, st, 0, n_warps_out);
    } else {
        if (p.lists_in_smem) launch_mode<uint32_t, true, 4>(p, ix, o, st, lists_bytes<uint32_t>(p.list_cap, p.read_cap), n_warps_out);
        else launch_mode<uint32_t, false, 1>(p, ix, o, st, 0, n_warps_out);
    }
}

// The thread-per-read pass takes a batch when the prefix table (and with it the inverse SA) exists, seeds are longer than the table
// is deep (so that an emitted match always carries its rows) and the reads fit its packed shared-memory copy and 9-bit sort key.
bool seed_thread_usable(const SeedParams& p, const DevOpts& o, uint32_t max_len) {
    return p.kmer_tab && p.todo && p.pk && o.min_seed_len > p.kmer_k && o.max_mem_intv > 1 && max_len <= 496 && p.cap / 2 >= 16 && p.cap / 2 <= 64;
}

int seed_thread_words(uint32_t max_len) { return (int)(max_len >> 4) + 3; }

// seed_pack -> seed_calls -> seed_last on `st`; returns the number of launches
int launch_seed_thread(const SeedParams& p, const DevIndex& ix, const DevOpts& o, uint32_t max_len, uint32_t* ticket, cudaStream_t st) {
    const int words = seed_thread_words(max_len);
    const size_t smem = (size_t)(words + seedt::PCAP) * ST_THREADS * 4;
    const int sms = cached_sm_count();
    cudaMemsetAsync(p.rflag, 0, (size_t)p.n_reads * 4, st);
    const uint64_t total = (uint64_t)p.n_reads * (uint32_t)words;
    seed_pack<<<(unsigned)std::min<uint64_t>((total + 255) / 256, (uint64_t)sms * 16), 256, 0, st>>>(p, o.min_seed_len, words);
    const unsigned last_blocks = (unsigned)std::min<uint64_t>(((uint64_t)p.n_reads + ST_THREADS - 1) / ST_THREADS, (uint64_t)sms * 8);
    if (ix.sa_bytes == 8) {
        const int nb = cached_blocks_per_sm(seed_calls<uint64_t>, ST_THREADS, smem);
        seed_calls<uint64_t><<<nb * sms, ST_THREADS, smem, st>>>(p, ix, o, ticket, words);
        seed_last<uint64_t><<<last_blocks, ST_THREADS, smem, st>>>(p, ix, o, words);
    } else {
        const int nb = cached_blocks_per_sm(seed_calls<uint32_t>, ST_THREADS, smem);
        seed_calls<uint32_t><<<nb * sms, ST_THREADS, smem, st>>>(p, ix, o, ticket, words);
        seed_last<uint32_t><<<last_blocks, ST_THREADS, smem, st>>>(p, ix, o, words);
    }
    return 3;
}
