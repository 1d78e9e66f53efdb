// seed_thread.cuh -- mem_collect_intv (SURVEY.md A.4) with ONE THREAD PER READ.
//
// The warp-per-read kernel (seed.cu) keeps one dependent chain of loads in flight per warp and runs its control flow on all 32
// lanes; on short reads almost every bwt_extend is a 16-byte prefix-table read or a text comparison (seed.cu header), i.e. scalar
// work.  Here a thread runs the reference's scalar algorithm for its own read -- the forward walk, the backward list logic of
// bwt_smem1a, re-seeding and the LAST-like pass -- with the same three shortcuts, so that a warp carries 32 independent chains
// (32x the memory-level parallelism per warp, ~1/20 of the warp instructions per read):
//   * a match of at most K bases is a prefix-table entry: interval = one 16-byte load indexed by the k-mer (no Occ);
//   * a match with ONE occurrence is extended by comparing read and text 16 bases per step (2-bit packed words), its rows
//     recovered from the inverse suffix array;
//   * everything else (longer repeats) is a real bwt_extend by the thread: the two 64-byte Occ blocks as 16-byte loads.
// List entries of at most K bases carry no rows at all (they are re-read from the table when needed).  Reads the thread cannot
// take (an ambiguous base, more list entries / intervals than its fixed buffers hold) are queued for the warp kernel, which
// starts them from scratch: results do not depend on which kernel took a read.
//
// The logical bwt_extend count (n_ext, the roofline unit of SURVEY 8d) is accumulated exactly as the reference would execute it.
//
// The file compiles for the device (seed.cu) and for the HOST: tests/seed_thread_check.cpp runs the same code on a CPU copy of
// the index and compares intervals and counters with the oracle's mem_collect_intv.  That host build is test infrastructure; the
// product library only contains the device instantiation.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define ST_HD __host__ __device__ __forceinline__
#else
#define ST_HD inline
#endif

namespace seedt {

struct U4 { uint32_t x, y, z, w; };          // == uint4 (prefix-table entry, Occ quarter block)
struct IntvOut { uint64_t x0, x1, x2, info; };  // == Intv (common.cuh)

#if defined(__CUDA_ARCH__)
ST_HD U4 ld_u4(const U4* p) { const uint4 v = __ldg(reinterpret_cast<const uint4*>(p)); U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r; }
ST_HD uint32_t ld_u32(const uint32_t* p) { return __ldg(p); }
template <class T> ST_HD T ld_idx(const T* p) { return __ldg(p); }
ST_HD int popc32(uint32_t v) { return __popc(v); }
ST_HD int clz32(uint32_t v) { return __clz(v); }
ST_HD int ctz32(uint32_t v) { return __ffs(v) - 1; }
ST_HD uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
ST_HD uint32_t brev32(uint32_t v) { return __brev(v); }
#else
ST_HD U4 ld_u4(const U4* p) { return *p; }
ST_HD uint32_t ld_u32(const uint32_t* p) { return *p; }
template <class T> ST_HD T ld_idx(const T* p) { return *p; }
ST_HD int popc32(uint32_t v) { return __builtin_popcount(v); }
ST_HD int clz32(uint32_t v) { return v ? __builtin_clz(v) : 32; }
ST_HD int ctz32(uint32_t v) { return v ? __builtin_ctz(v) : -1; }
ST_HD uint32_t bswap32(uint32_t v) { return __builtin_bswap32(v); }
ST_HD uint32_t brev32(uint32_t v) { uint32_t r = 0; for (int i = 0; i < 32; ++i) r |= ((v >> i) & 1u) << (31 - i); return r; }
#endif

ST_HD uint32_t level_off(int t) { return (0x55555555u >> (32 - 2 * t)) - 1u; }   // first entry of level t = (4^t - 4) / 3, 1 <= t <= 15
// funnel shift left of hi:lo by s in [0, 32): the top 32 bits
ST_HD uint32_t fsl(uint32_t lo, uint32_t hi, int s) { return s ? (hi << s) | (lo >> (32 - s)) : hi; }

template <class IdxT> struct Index {
    const uint32_t* occ; const U4* tab; int kk;
    const uint32_t* ztab;    // sizes only (the .z of every table entry, same indexing): what the walks compare; 4 bytes per entry, so the
                             // levels that stay in L2 reach two levels deeper than with the 16-byte entries (nullptr: read tab)
    const IdxT* sa; const IdxT* isa; const uint8_t* pac;    // the inverse SA is always there: the pass runs only beside the prefix table
    IdxT l_pac, n, primary; IdxT L2[5];
};
struct Opts { int min_seed_len, split_len, split_width, max_mem_intv; };

template <class IdxT> ST_HD IdxT tab_x0(const U4& e) { return sizeof(IdxT) == 4 ? (IdxT)e.x : (IdxT)((unsigned long long)(e.w & 0xffu) << 32 | e.x); }
template <class IdxT> ST_HD IdxT tab_x1(const U4& e) { return sizeof(IdxT) == 4 ? (IdxT)e.y : (IdxT)((unsigned long long)((e.w >> 8) & 0xffu) << 32 | e.y); }

// ---- the read: 2 bits per base, 16 bases per word, first base in the top bits; word w of the read at pk[w * stride]
// (stride = threads per CTA in shared memory, 1 on the host); two zero words follow the last base
struct Read { const uint32_t* pk; int stride; int len; };
ST_HD uint32_t rd_word(const Read& R, int w) { return R.pk[w * R.stride]; }
// 16 bases starting at s (0 <= s <= len), top-aligned; bases beyond the read are zero
ST_HD uint32_t rd_window(const Read& R, int s) { return fsl(rd_word(R, (s >> 4) + 1), rd_word(R, s >> 4), (s & 15) << 1); }
ST_HD int rd_base(const Read& R, int i) { return (int)(rd_word(R, i >> 4) >> (30 - ((i & 15) << 1))) & 3; }

// ---- the text T = fwd(l_pac) | revcomp(l_pac), 2 bits per base in pac (MSB first inside a byte)
template <class IdxT> ST_HD uint32_t text_base(const Index<IdxT>& X, IdxT p) {
    if (p < X.l_pac) return (X.pac[p >> 2] >> ((~(uint32_t)p & 3u) << 1)) & 3u;
    const IdxT f = (IdxT)(2 * X.l_pac - 1 - p);
    return 3u - ((X.pac[f >> 2] >> ((~(uint32_t)f & 3u) << 1)) & 3u);
}
// 16 forward bases pac[f .. f+16), top-aligned (f + 16 <= l_pac; the array is readable 4 bytes past its end)
template <class IdxT> ST_HD uint32_t pac_window(const Index<IdxT>& X, IdxT f) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(X.pac) + (f >> 4);
    return fsl(bswap32(ld_u32(w + 1)), bswap32(ld_u32(w)), (int)(f & 15) << 1);
}
// 16 bases T[p .. p+16), top-aligned; *ok = false when the window crosses l_pac or the end of the text (caller goes base by base)
template <class IdxT> ST_HD uint32_t text_window(const Index<IdxT>& X, IdxT p, bool* ok) {
    *ok = true;
    if (p + 16 <= X.l_pac) return pac_window(X, p);
    if (p >= X.l_pac && p + 16 <= X.n) {
        // T[p + k] = 3 - pac[2 l - 1 - p - k]: the forward window [2l - 16 - p, 2l - p) reversed and complemented
        const uint32_t v = pac_window(X, (IdxT)(2 * X.l_pac - 16 - p));
        const uint32_t r = brev32(v);                                    // reverses bases AND the two bits of each base
        return ~(((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1));    // swap the bit pairs back, complement
    }
    *ok = false;
    return 0;
}
// number of consecutive k in [0, maxlen) with q[qpos + k] == T[tpos + k] (tpos + k < n)
template <class IdxT> ST_HD int match_run_fwd(const Index<IdxT>& X, const Read& R, IdxT tpos, int qpos, int maxlen) {
    int k = 0;
    while (k < maxlen) {
        const int m = maxlen - k < 16 ? maxlen - k : 16;
        bool ok;
        const uint32_t tw = text_window(X, (IdxT)(tpos + (IdxT)k), &ok);
        if (ok) {
            uint32_t diff = tw ^ rd_window(R, qpos + k);
            if (m < 16) diff &= ~(0xffffffffu >> (2 * m));
            if (diff) return k + (clz32(diff) >> 1);
            k += m;
        } else {
            for (int j = 0; j < m; ++j, ++k) {
                const IdxT p = (IdxT)(tpos + (IdxT)k);
                if (!(p < X.n) || text_base(X, p) != (uint32_t)rd_base(R, qpos + k)) return k;
            }
        }
    }
    return maxlen;
}
// number of consecutive k in [0, maxlen) with k < tpos and q[qpos - k] == T[tpos - 1 - k]
template <class IdxT> ST_HD int match_run_bwd(const Index<IdxT>& X, const Read& R, IdxT tpos, int qpos, int maxlen) {
    int k = 0;
    while (k < maxlen) {
        const int m = maxlen - k < 16 ? maxlen - k : 16;
        bool ok = false;
        uint32_t tw = 0;
        // window of 16 ending just before tpos - k on the text, ending at qpos - k (inclusive) on the read
        if (tpos >= (IdxT)(k + 16) && qpos - k >= 15) tw = text_window(X, (IdxT)(tpos - (IdxT)k - 16), &ok);
        if (ok) {
            uint32_t diff = tw ^ rd_window(R, qpos - k - 15);
            if (m < 16) diff &= (1u << (2 * m)) - 1u;
            if (diff) return k + (ctz32(diff) >> 1);
            k += m;
        } else {
            for (int j = 0; j < m; ++j, ++k) {
                if (!((IdxT)k < tpos) || qpos - k < 0) return k;
                if (text_base(X, (IdxT)(tpos - 1 - (IdxT)k)) != (uint32_t)rd_base(R, qpos - k)) return k;
            }
        }
    }
    return maxlen;
}

// size of table entry `idx` (all levels share one index space)
template <class IdxT> ST_HD uint32_t tab_size(const Index<IdxT>& X, uint32_t idx) {
    return X.ztab ? ld_u32(X.ztab + idx) : ld_u32(reinterpret_cast<const uint32_t*>(X.tab + idx) + 2);
}
// ---- prefix table: entry of the t-mer starting at read position s (1 <= t <= kk, s + t <= len)
template <class IdxT> ST_HD U4 tab_get(const Index<IdxT>& X, const Read& R, int s, int t) {
    return ld_u4(X.tab + level_off(t) + (rd_window(R, s) >> (32 - 2 * t)));
}

// ---- bwt_extend by one thread (SURVEY A.2): child interval of `ik` for base c
template <class IdxT> struct Iv { IdxT x0, x1; uint32_t x2; };
// eq = #c, gt = #symbols > c in B[0 .. pos] (pos already shifted for the primary row): checkpoint + popcounts of the block's symbols
template <class IdxT> ST_HD void occ_eq_gt(const Index<IdxT>& X, IdxT pos, int c, IdxT& eq, IdxT& gt) {
    const U4* blk = reinterpret_cast<const U4*>(X.occ + ((size_t)(pos >> 7) << 4));
    const U4 ca = ld_u4(blk), cb = ld_u4(blk + 1);
    IdxT cp[4];
    if (sizeof(IdxT) == 4) { cp[0] = (IdxT)ca.x; cp[1] = (IdxT)ca.z; cp[2] = (IdxT)cb.x; cp[3] = (IdxT)cb.z; }
    else {
        cp[0] = (IdxT)((unsigned long long)ca.y << 32 | ca.x); cp[1] = (IdxT)((unsigned long long)ca.w << 32 | ca.z);
        cp[2] = (IdxT)((unsigned long long)cb.y << 32 | cb.x); cp[3] = (IdxT)((unsigned long long)cb.w << 32 | cb.z);
    }
    eq = cp[c]; gt = 0;
    for (int a = 3; a > c; --a) gt += cp[a];
    const int within = (int)(pos & 127) + 1;
    const uint32_t C1 = 0u - (uint32_t)(c >> 1), C0 = 0u - (uint32_t)(c & 1);
    int ne = 0, ng = 0;
    const U4 s0 = ld_u4(blk + 2);
    const uint32_t w0[4] = {s0.x, s0.y, s0.z, s0.w};
    for (int w = 0; w < 4; ++w) {
        int nsym = within - (w << 4); nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
        const uint32_t keep = nsym ? (uint32_t)(0x5555555500000000ull >> (2 * nsym)) : 0u;
        const uint32_t word = w0[w], hx = ~((word >> 1) ^ C1);
        ne += popc32(hx & ~(word ^ C0) & keep);
        ng += popc32((((word >> 1) & ~C1) | (hx & word & ~C0)) & keep);
    }
    if (within > 64) {
        const U4 s1 = ld_u4(blk + 3);
        const uint32_t w1[4] = {s1.x, s1.y, s1.z, s1.w};
        for (int w = 0; w < 4; ++w) {
            int nsym = within - 64 - (w << 4); nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
            const uint32_t keep = nsym ? (uint32_t)(0x5555555500000000ull >> (2 * nsym)) : 0u;
            const uint32_t word = w1[w], hx = ~((word >> 1) ^ C1);
            ne += popc32(hx & ~(word ^ C0) & keep);
            ng += popc32((((word >> 1) & ~C1) | (hx & word & ~C0)) & keep);
        }
    }
    eq += (IdxT)ne; gt += (IdxT)ng;
}
template <class IdxT, int IS_BACK> ST_HD Iv<IdxT> extend_one(const Index<IdxT>& X, const Iv<IdxT>& ik, int c) {
    const IdxT xo = IS_BACK ? ik.x0 : ik.x1, xb = IS_BACK ? ik.x1 : ik.x0;
    IdxT pk = xo - 1; pk -= (pk >= X.primary);
    IdxT pl = xo - 1 + (IdxT)ik.x2; pl -= (pl >= X.primary);
    IdxT eqk, gtk, eql, gtl;
    occ_eq_gt(X, pk, c, eqk, gtk);
    occ_eq_gt(X, pl, c, eql, gtl);
    const IdxT no = X.L2[c] + 1 + eqk;
    const IdxT nb = xb + (IdxT)(xo <= X.primary && xo + ik.x2 - 1 >= X.primary) + (gtl - gtk);
    Iv<IdxT> ok;
    ok.x0 = IS_BACK ? no : nb; ok.x1 = IS_BACK ? nb : no; ok.x2 = (uint32_t)(eql - eqk);
    return ok;
}

// ---- per-read working state
// bwt_smem1a's backward phase, COLUMN-WISE.  The reference walks the list of forward matches step by step (i = x-1, x-2, ...), all
// entries per step.  The same result follows from walking ONE ENTRY AT A TIME through all of its steps (its "column" of the
// (step, entry) table), longest match first, because an entry interacts with the others only through
//   P(b) = the size, at step b, of the nearest longer entry that is still in the list at step b (0 when there is none):
// an entry leaves the list when its size drops below min_intv (it "dies"; sizes only shrink, and a longer match never outlives a
// shorter one) or when its size equals P(b) (it has become the same occurrence set as that longer entry and from then on lives
// and dies with it).  A MEM is emitted when an entry dies at a step where no longer entry is left (P(b) == 0).  The number of
// bwt_extend calls the reference makes is the number of (entry, step) pairs visited, which is what the column walk counts.
// A column is a tight loop of prefix-table lookups with one comparison against P(b) -- the same loop for every thread of a warp --
// followed, when the match outgrows the table, by a tail of real extensions or (one occurrence) a text comparison.
// P lives in a small per-thread array pc[] (steps a non-unique entry was kept) plus one implicit range (the steps the unique
// entry is alive).
constexpr int RCAP = 8;                       // forward entries longer than the table (they carry their rows)
constexpr int TAB_UNROLL = 4;                 // prefix-table lookups a thread keeps in flight in a column walk
constexpr int PCAP = 32;                      // steps a non-unique entry may be kept (table depth + a few real extensions)
template <class IdxT> struct RowsEnt { IdxT x0, x1; uint32_t x2; int end; };

// The forward entries of a call need no array: an entry of at most K bases is fully described by its length (its size is a table
// entry), so the table part of the list is a BIT MASK over lengths 1..K; only the few entries longer than the table are stored.
template <class IdxT> struct Work {
    // the call in flight: bwt_smem1a(x, min_intv)
    int x, ret, n, n_rows; uint32_t min_intv;
    uint32_t mask, top_z;                     // bit L set: the match q[x .. x+L) is a list entry; top_z = size of the longest of them
    int nvalid, uq_lo, uq_hi, last_mem_start; bool have_mem;
    uint32_t* pc; int pc_stride;             // pc[b * pc_stride], b < PCAP
    RowsEnt<IdxT> re[RCAP];
    // results
    IntvOut* out; uint32_t n_out, cap; bool fail; unsigned long long n_ext;
};

template <class IdxT> ST_HD void emit(Work<IdxT>& W, IdxT x0, IdxT x1, uint32_t x2, int start, int end) {
    if (W.n_out >= W.cap) { W.fail = true; return; }
    IntvOut v; v.x0 = x0; v.x1 = x1; v.x2 = x2; v.info = (uint64_t)(uint32_t)start << 32 | (uint32_t)end;
    W.out[W.n_out++] = v;
}
template <class IdxT> ST_HD bool push_rows(Work<IdxT>& W, IdxT x0, IdxT x1, uint32_t x2, int end) {
    if (W.n_rows >= RCAP) { W.fail = true; return false; }
    RowsEnt<IdxT>& d = W.re[W.n_rows++]; d.x0 = x0; d.x1 = x1; d.x2 = x2; d.end = end;
    return true;
}

// forward walk of bwt_smem1a(x, min_intv): records the list entries (mask + rows entries); W.ret = end of the longest match
template <class IdxT>
ST_HD void smem_forward(const Index<IdxT>& X, const Read& R, int x, uint32_t min_intv, Work<IdxT>& W) {
    const int len = R.len, K = X.kk;
    if (min_intv < 1) min_intv = 1;
    W.x = x; W.min_intv = min_intv; W.n = 0; W.n_rows = 0; W.mask = 0; W.top_z = 0; W.ret = len;
    W.nvalid = 0; W.uq_lo = W.uq_hi = 0; W.have_mem = false; W.last_mem_start = 0;
    // matches of up to K bases: the prefix table.  The K lookups are independent: all in flight together.
    const int maxt = len - x < K ? len - x : K;
    const uint32_t w0 = rd_window(R, x);
    uint32_t zs[16];
#pragma unroll
    for (int t = 1; t <= 15; ++t) zs[t] = t <= maxt ? tab_size(X, level_off(t) + (w0 >> (32 - 2 * t))) : 0u;
    uint32_t cur_x2 = zs[1], n_ext = 0, mask = 0, top_z = 0;
    int i = x + 1; bool stopped = false;
#pragma unroll
    for (int t = 2; t <= 15; ++t) {              // appending q[i], i = x + t - 1
        if (t <= maxt && !stopped) {
            const uint32_t sz = zs[t];
            ++n_ext;
            if (sz != cur_x2) {
                mask |= 1u << (t - 1); top_z = cur_x2;
                if (sz < min_intv) stopped = true;
            }
            if (!stopped) { cur_x2 = sz; ++i; }
        }
    }
    W.n_ext += n_ext;
    if (!stopped) {
        const U4 e = ld_u4(X.tab + level_off(maxt) + (w0 >> (32 - 2 * maxt)));
        Iv<IdxT> ik; ik.x0 = tab_x0<IdxT>(e); ik.x1 = tab_x1<IdxT>(e); ik.x2 = cur_x2;
        for (; i < len; ++i) {
            if (ik.x2 == 1 && min_intv == 1) {
                // unique match q[x .. i): walk to the first base that does not match (or the end of the read) by text comparison
                const IdxT pos = ld_idx(X.sa + ik.x0);
                const int run = match_run_fwd(X, R, (IdxT)(pos + (IdxT)(i - x)), i, len - i);
                if (run > 0) { i += run; ik.x1 = ld_idx(X.isa + (X.n - pos - (IdxT)(i - x))); W.n_ext += (unsigned long long)run; }
                if (i == len) break;
                ++W.n_ext;                       // the extension the scalar code tries next empties the interval
                if (i - x <= K) { mask |= 1u << (i - x); top_z = 1; }
                else if (!push_rows(W, ik.x0, ik.x1, 1u, i)) return;
                stopped = true;
                break;
            }
            const Iv<IdxT> ok = extend_one<IdxT, 0>(X, ik, 3 - rd_base(R, i));
            ++W.n_ext;
            if (ok.x2 != ik.x2) {
                if (i - x <= K) { mask |= 1u << (i - x); top_z = ik.x2; }
                else if (!push_rows(W, ik.x0, ik.x1, ik.x2, i)) return;
                if (ok.x2 < min_intv) { stopped = true; break; }
            }
            ik = ok;
        }
        if (!stopped) {                          // reached the end of the read: the last interval is recorded too
            if (len - x <= K) { mask |= 1u << (len - x); top_z = ik.x2; }
            else if (!push_rows(W, ik.x0, ik.x1, ik.x2, len)) return;
        }
    }
    W.mask = mask; W.top_z = top_z;
    W.n = W.n_rows + popc32(mask);
    W.ret = W.n_rows ? W.re[W.n_rows - 1].end : x + (31 - clz32(mask));
}

// the entry with rows (x0, x1, x2) dies at step i (it is the match q[i+1 .. end)): bwt_smem1a's emission rule
template <class IdxT>
ST_HD void entry_dies(const Opts& o, Work<IdxT>& W, bool longer_left, int i, int end, IdxT x0, IdxT x1, uint32_t x2) {
    if (!longer_left && (!W.have_mem || i + 1 < W.last_mem_start)) {
        if (end - (i + 1) >= o.min_seed_len) emit(W, x0, x1, x2, i + 1, end);   // such a match is longer than K: its rows are known
        W.have_mem = true; W.last_mem_start = i + 1;
    }
}

// backward walk of list entry k (0 = longest match) of the call set up by smem_forward.  On the device ALL lanes of the warp call
// this together (`live` = this lane really has an entry k): the two loops are driven by warp votes and have a single exit, so the
// lanes that are in the table loop step together, and so do the lanes in the tail.
#if defined(__CUDA_ARCH__)
#define ST_ANY(p) __any_sync(0xffffffffu, (p))
#else
#define ST_ANY(p) (p)
#endif
template <class IdxT>
ST_HD void smem_column(const Index<IdxT>& X, const Opts& o, const Read& R, int k, Work<IdxT>& W, bool live) {
    const int K = X.kk, x = W.x;
    const uint32_t min_intv = W.min_intv;
    const bool can_uq = min_intv == 1;
    int end = 0, b = 0, i = x - 1, nb = 0;
    uint32_t cur = 0; IdxT x0 = 0, x1 = 0; bool rows = false;
    if (live) {
        if (k < W.n_rows) { const RowsEnt<IdxT>& p = W.re[W.n_rows - 1 - k]; end = p.end; cur = p.x2; x0 = p.x0; x1 = p.x1; rows = true; }
        else {
            // the longest table entry not walked yet; its size is only needed when it is 1 (the longest entry of the list) --
            // every other entry has at least 2 occurrences, and the exact number is read again if the walk outgrows the table
            const int L = 31 - clz32(W.mask);
            cur = (k == W.n_rows) ? W.top_z : 2u;
            W.mask ^= 1u << L; end = x + L;
        }
        if (!(can_uq && cur == 1)) nb = i + 1 < K - (end - x) ? i + 1 : K - (end - x);     // steps with i >= 0 and end - i <= K
        if (nb < 0) nb = 0;
    }
    // ---- steps inside the prefix table: one lookup and one comparison with P(b) each.  The address of a step's lookup does not
    // depend on the previous step's result (only whether the walk goes on does), so TAB_UNROLL lookups are issued together
    // (loads in flight per thread), then consumed in order; the lookups past the end of the walk are simply not used.
    uint32_t n_ext = 0;
    while (ST_ANY(live && b < nb)) {
        if (live && b < nb) {
            const int w = i >> 4;
            const uint32_t wc = rd_word(R, w > 0 ? w - 1 : 0), wa = rd_word(R, w), wb = rd_word(R, w + 1);
            uint32_t sv[TAB_UNROLL];
#pragma unroll
            for (int u = 0; u < TAB_UNROLL; ++u) {
                sv[u] = 0;
                const int iu = i - u;
                if (b + u < nb) {
                    const int sh = (iu & 15) << 1, lq = end - iu;
                    const uint32_t win = (iu >> 4) == w ? fsl(wb, wa, sh) : fsl(wa, wc, sh);
                    sv[u] = tab_size(X, level_off(lq) + (win >> (32 - 2 * lq)));
                }
            }
#pragma unroll
            for (int u = 0; u < TAB_UNROLL; ++u) {
                if (live && b < nb) {
                    const uint32_t s = sv[u];
                    ++n_ext;
                    const uint32_t P = b < W.nvalid ? W.pc[b * W.pc_stride] : (b >= W.uq_lo && b < W.uq_hi ? 1u : 0u);
                    if (s < min_intv) { entry_dies(o, W, P != 0, i, end, x0, x1, cur); live = false; }
                    else if (s == P) live = false;                        // same occurrences as a longer entry from here on
                    else {
                        W.pc[b * W.pc_stride] = s; if (W.nvalid <= b) W.nvalid = b + 1;
                        cur = s; rows = false; ++b; --i;
                        if (can_uq && s == 1) nb = b;                     // one occurrence left: the tail takes it
                    }
                }
            }
        }
    }
    W.n_ext += n_ext;
    // ---- tail: one occurrence => text comparison; otherwise real extensions
    while (ST_ANY(live)) {
        if (live) {
            if (can_uq && cur == 1) {
                if (!rows) { const U4 f = tab_get(X, R, i + 1, end - (i + 1)); x0 = tab_x0<IdxT>(f); x1 = tab_x1<IdxT>(f); }
                const IdxT pos = ld_idx(X.sa + x0);
                const int run = match_run_bwd(X, R, pos, i, i + 1);
                const int stop = i - run;                                 // the step at which it dies
                W.n_ext += (unsigned long long)run + (stop >= 0 ? 1u : 0u);
                W.uq_lo = b; W.uq_hi = b + run;                           // alive (size 1) at steps [b, b + run)
                // nothing longer is left when an entry has one occurrence (a longer one would have the same size and have absorbed it)
                entry_dies(o, W, false, stop, end, run > 0 ? ld_idx(X.isa + (pos - (IdxT)run)) : x0, x1, 1u);
                live = false;
            } else {
                const uint32_t P = b < W.nvalid ? W.pc[b * W.pc_stride] : (b >= W.uq_lo && b < W.uq_hi ? 1u : 0u);
                if (i < 0) { entry_dies(o, W, P != 0, i, end, x0, x1, cur); live = false; }   // start of the read: what is left dies, nothing is extended
                else {
                    const int lq = end - i;
                    uint32_t s; IdxT nx0 = x0, nx1 = x1; bool nrows = false;
                    if (lq <= K) s = tab_get(X, R, i, lq).z;
                    else {
                        if (!rows) { const U4 f = tab_get(X, R, i + 1, lq - 1); x0 = tab_x0<IdxT>(f); x1 = tab_x1<IdxT>(f); cur = f.z; }
                        Iv<IdxT> pi; pi.x0 = x0; pi.x1 = x1; pi.x2 = cur;
                        const Iv<IdxT> ok = extend_one<IdxT, 1>(X, pi, rd_base(R, i));
                        s = ok.x2; nx0 = ok.x0; nx1 = ok.x1; nrows = true;
                    }
                    ++W.n_ext;
                    if (s < min_intv) { entry_dies(o, W, P != 0, i, end, x0, x1, cur); live = false; }
                    else if (s == P) live = false;
                    else if (b >= PCAP) { W.fail = true; live = false; }
                    else {
                        W.pc[b * W.pc_stride] = s; if (W.nvalid <= b) W.nvalid = b + 1;
                        cur = s; x0 = nx0; x1 = nx1; rows = nrows; ++b; --i;
                    }
                }
            }
        }
    }
}

// bwt_seed_strategy1(x, min_len, max_intv): the first match from x with fewer than max_intv occurrences and more than min_len bases
template <class IdxT>
ST_HD int seed_strategy1(const Index<IdxT>& X, const Opts& o, const Read& R, int x, Work<IdxT>& W) {
    const int len = R.len, K = X.kk, min_len = o.min_seed_len;
    const uint32_t max_intv = (uint32_t)o.max_mem_intv;
    // the first K - 1 extensions can neither emit (i - x < min_len) nor be observed: their result is the K-mer's table entry
    const U4 e = tab_get(X, R, x, K);
    Iv<IdxT> ik; ik.x0 = tab_x0<IdxT>(e); ik.x1 = tab_x1<IdxT>(e); ik.x2 = e.z;
    W.n_ext += (unsigned long long)(K - 1);
    int i = x + K;
    if (ik.x2 == 0) {
        // an empty interval stays empty: the walk ends at the first i with i - x >= min_len (nothing emitted) or at the end of the read
        const int stop = x + min_len;
        if (stop < len) { W.n_ext += (unsigned long long)(stop + 1 - i); return stop + 1; }
        W.n_ext += (unsigned long long)(len - i);
        return len;
    }
    for (; i < len; ++i) {
        if (ik.x2 == 1 && max_intv > 1 && i - x <= min_len) {
            // unique match q[x .. i): the walk ends at j = x + min_len (emit iff still matching) or at the end of the read
            const int stop = x + min_len;
            const int lim = (stop < len ? stop + 1 : len) - i;       // bases q[i .. i + lim) are looked at
            const IdxT pos = ld_idx(X.sa + ik.x0);
            const int run = match_run_fwd(X, R, (IdxT)(pos + (IdxT)(i - x)), i, lim);
            W.n_ext += (unsigned long long)lim;
            if (stop >= len) return len;
            if (run == lim) emit(W, ik.x0, ld_idx(X.isa + (X.n - pos - (IdxT)(stop + 1 - x))), 1u, x, stop + 1);
            return stop + 1;
        }
        const Iv<IdxT> ok = extend_one<IdxT, 0>(X, ik, 3 - rd_base(R, i));
        ++W.n_ext;
        if (ok.x2 < max_intv && i - x >= min_len) {
            if (ok.x2 > 0) emit(W, ok.x0, ok.x1, ok.x2, x, i + 1);
            return i + 1;
        }
        ik = ok;
    }
    return len;
}

// pass 3: the LAST-like pass.  The walk x -> f(x) is sequential, but f is a pure function of x and almost always returns x + L
// (L = min_seed_len + 1: the first match with fewer than max_mem_intv occurrences is the L-mer itself).  LAST_BATCH predicted starts are
// therefore evaluated together -- K-mer entries, then (one occurrence) SA rows, text words, ISA rows: each group of loads in flight at
// once -- and consumed in order for as long as each start is the predicted one and was decidable without Occ.
constexpr int LAST_BATCH = 8;
constexpr int MWL = 4;                       // K-mer occurrences the LAST-like pass settles by text comparison
template <class IdxT> ST_HD void last_like_pass(const Index<IdxT>& X, const Opts& o, const Read& R, Work<IdxT>& W) {
    if (o.max_mem_intv <= 0) return;
    const int len = R.len, K = X.kk, min_len = o.min_seed_len, L = min_len + 1;
    const bool spec_ok = o.max_mem_intv > 1 && min_len >= K;
    int x = 0;
    while (x < len && !W.fail) {
        const int nb = spec_ok ? ((len - x) / L < LAST_BATCH ? (len - x) / L : LAST_BATCH) : 0;   // starts whose whole L-mer lies in the read
        if (nb > 0) {
            U4 e[LAST_BATCH]; IdxT pos[LAST_BATCH], r1[LAST_BATCH]; bool hit[LAST_BATCH];
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) if (k < nb) e[k] = tab_get(X, R, x + k * L, K);
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) { pos[k] = 0; if (k < nb && e[k].z == 1) pos[k] = ld_idx(X.sa + tab_x0<IdxT>(e[k])); }
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) {
                hit[k] = false;
                if (k < nb && e[k].z == 1) hit[k] = match_run_fwd(X, R, (IdxT)(pos[k] + (IdxT)K), x + k * L + K, L - K) == L - K;
            }
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) { r1[k] = 0; if (hit[k]) r1[k] = ld_idx(X.isa + (X.n - pos[k] - (IdxT)L)); }
            int done = 0;
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) {
                if (k == done && k < nb && e[k].z <= 1) {            // decided without Occ: no seed, or the unique L-mer
                    if (hit[k]) emit(W, tab_x0<IdxT>(e[k]), r1[k], 1u, x + k * L, x + k * L + L);
                    W.n_ext += (unsigned long long)min_len;
                    ++done;
                }
            }
            x += done * L;
            if (done == nb || W.fail) continue;
            // The start at x stopped the batch.  A K-mer with a handful of occurrences (fewer than max_mem_intv) is decided the same way
            // as the unique one, from the text: the L-mer's occurrences are those of the K-mer whose next L - K bases match the read;
            // they are consecutive rows of the K-mer's interval (the longer pattern's interval lies inside the shorter one's), and the
            // reverse-strand row is the smallest row of their reverse-complement occurrences.  No Occ block is touched.
            U4 em; em.x = em.y = em.z = em.w = 0;
#pragma unroll
            for (int k = 0; k < LAST_BATCH; ++k) if (k == done) em = e[k];
            if (em.z >= 2u && em.z <= (uint32_t)MWL && em.z < (uint32_t)o.max_mem_intv) {
                const IdxT b0 = tab_x0<IdxT>(em);
                IdxT pp[MWL]; bool hh[MWL];
#pragma unroll
                for (int t = 0; t < MWL; ++t) pp[t] = t < (int)em.z ? ld_idx(X.sa + b0 + (IdxT)t) : (IdxT)0;
#pragma unroll
                for (int t = 0; t < MWL; ++t) hh[t] = t < (int)em.z && match_run_fwd(X, R, (IdxT)(pp[t] + (IdxT)K), x + K, L - K) == L - K;
                uint32_t cnt = 0; int tfirst = 0;
#pragma unroll
                for (int t = MWL - 1; t >= 0; --t) if (hh[t]) { ++cnt; tfirst = t; }
                if (cnt) {
                    IdxT rr[MWL];
#pragma unroll
                    for (int t = 0; t < MWL; ++t) rr[t] = hh[t] ? ld_idx(X.isa + (X.n - pp[t] - (IdxT)L)) : (IdxT)0;
                    IdxT rmin = 0; bool have = false;
#pragma unroll
                    for (int t = 0; t < MWL; ++t) if (hh[t] && (!have || rr[t] < rmin)) { rmin = rr[t]; have = true; }
                    emit(W, (IdxT)(b0 + (IdxT)tfirst), rmin, cnt, x, x + L);
                }
                W.n_ext += (unsigned long long)min_len;
                x += L;
                continue;
            }
        }
        if (x + K > len) {
            // fewer than K bases left: no table entry; the walk cannot emit (i - x < min_len), only its extensions count
            W.n_ext += (unsigned long long)(len - 1 - x);
            break;
        }
        x = seed_strategy1(X, o, R, x, W);
    }
}

// The calls of passes 1 and 2 in order: pass 1 starts a call where the previous longest match ended; pass 2 re-seeds from the
// middle of every long, rare SMEM of pass 1.  Returns false when there is no further call.
struct Calls { int pass, next_x; uint32_t k2, old_n; };
ST_HD void calls_init(Calls& C) { C.pass = 1; C.next_x = 0; C.k2 = 0; C.old_n = 0; }
template <class IdxT> ST_HD bool next_call(Calls& C, const Opts& o, const Read& R, const Work<IdxT>& W, int* x, uint32_t* min_intv) {
    if (W.fail) return false;
    if (C.pass == 1) {
        if (C.next_x < R.len) { *x = C.next_x; *min_intv = 1; return true; }
        C.pass = 2; C.k2 = 0; C.old_n = W.n_out;
    }
    for (; C.k2 < C.old_n; ++C.k2) {
        const IntvOut p = W.out[C.k2];
        const int start = (int)(p.info >> 32), end = (int)(uint32_t)p.info;
        if (end - start < o.split_len || p.x2 > (uint64_t)o.split_width) continue;
        *x = (start + end) >> 1; *min_intv = (uint32_t)p.x2 + 1u; ++C.k2;
        return true;
    }
    return false;
}

template <class IdxT> ST_HD void work_init(Work<IdxT>& W, IntvOut* out, uint32_t cap, uint32_t* pc, int pc_stride) {
    W.out = out; W.n_out = 0; W.cap = cap; W.fail = false; W.n_ext = 0; W.n = 0; W.pc = pc; W.pc_stride = pc_stride;
}

// mem_collect_intv for ONE read on the host (tests); the device kernel runs the same calls warp-wide, column by column
template <class IdxT> ST_HD void collect(const Index<IdxT>& X, const Opts& o, const Read& R, Work<IdxT>& W) {
    Calls C; calls_init(C);
    int x; uint32_t mi;
    while (next_call(C, o, R, W, &x, &mi)) {
        smem_forward(X, R, x, mi, W);
        for (int k = 0; k < W.n && !W.fail; ++k) smem_column(X, o, R, k, W, true);
        if (C.pass == 1) C.next_x = W.ret;
    }
    if (!W.fail) last_like_pass(X, o, R, W);
}

}  // namespace seedt
