// sa_lookup.cuh -- what the SA lookups of mem_chain are, and one LF step over the Occ blocks.
//
// The lookups of a read (SURVEY A.5, the k/step loop of mem_chain): interval by interval in the order seeding stored them, and within
// an interval the rows x0, x0 + step, x0 + 2 step, ... (occ_count of them).  Lookup t of a read is the t-th row of that sequence.  The
// chain kernels (chain.cu) and the position resolve pass of a compact index (sa_resolve.cu) both enumerate it with these functions, so
// the position the resolve pass puts in slot t is the one the chain kernels expect there.
#pragma once
#include "common.cuh"

// occurrences an interval contributes (the k/step loop of mem_chain, SURVEY A.5) and the stride between them
__device__ __forceinline__ uint32_t occ_count(const DevOpts& o, uint64_t x2, uint64_t* step_out) {
    uint64_t step = 1, cnt = x2;
    if (x2 > (uint64_t)o.max_occ) {
        step = x2 / (uint64_t)o.max_occ;
        cnt = (x2 + step - 1) / step;
        if (cnt > (uint64_t)o.max_occ) cnt = (uint64_t)o.max_occ;
    }
    if (step_out) *step_out = step;
    return (uint32_t)cnt;
}

// the row of occurrence c of an interval
__device__ __forceinline__ uint64_t lookup_row(uint64_t x0, uint64_t step, uint32_t c) { return x0 + (uint64_t)c * step; }

// f(t, interval, row) for the lookups t = first, first + stride, ... of the read's intervals iv[0 .. n_iv); returns their count
template <class F>
__device__ __forceinline__ uint32_t for_each_lookup(const Intv* iv, int n_iv, const DevOpts& o, uint32_t first, uint32_t stride, F f) {
    uint32_t t = 0;
    for (int i = 0; i < n_iv; ++i) {
        const Intv p = iv[i];
        uint64_t step;
        const uint32_t cnt = occ_count(o, p.x2, &step);
        for (uint32_t c = first; c < cnt; c += stride) f(t + c, p, lookup_row(p.x0, step, c));
        t += cnt;
    }
    return t;
}

// The Occ view an LF walk needs
struct LfView {
    const uint32_t* occ;
    uint64_t n, primary, L0, L1, L2, L3;     // L2[0..3] of the index
};

// bwt_invPsi (libbwa bwt.h) for a row j in [0, n]: 0 for the primary row, else L2[c] + occ(j, c) with c = B0[j - (j > primary)] and occ
// the count of c in B0[0 .. j - (j >= primary)] -- the checkpoint of j's 128-symbol block plus the popcounts of its symbols up to j.
// P: any record with the fields of LfView.
template <class P>
__device__ __forceinline__ uint64_t lf(const P& V, uint64_t j) {
    if (j == V.primary) return 0;
    const uint64_t x = j - (j > V.primary);
    const uint4* blk = reinterpret_cast<const uint4*>(V.occ + ((size_t)(x >> 7) << 4));
    const uint4 ca = __ldg(blk), cb = __ldg(blk + 1), s0 = __ldg(blk + 2), s1 = __ldg(blk + 3);
    const uint32_t w8[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
    const int wi = (int)((x >> 4) & 7);
    uint32_t word = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) word = w == wi ? w8[w] : word;
    const uint32_t c = (word >> ((15 - (uint32_t)(x & 15)) << 1)) & 3u;
    const uint32_t rep = c * 0x55555555u;
    const int within = (int)(x & 127) + 1;
    uint32_t cnt = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        int nsym = within - (w << 4);
        nsym = nsym < 0 ? 0 : (nsym > 16 ? 16 : nsym);
        const uint32_t keep = __funnelshift_rc(0u, 0x55555555u, 2 * nsym);   // the first nsym symbols of the word (MSB first)
        const uint32_t t = ~(w8[w] ^ rep);                                     // 11 where a symbol equals c
        cnt += __popc(t & (t >> 1) & keep);
    }
    const uint64_t ck = c == 0 ? ((uint64_t)ca.y << 32 | ca.x) : c == 1 ? ((uint64_t)ca.w << 32 | ca.z)
                      : c == 2 ? ((uint64_t)cb.y << 32 | cb.x) : ((uint64_t)cb.w << 32 | cb.z);
    const uint64_t base = c == 0 ? V.L0 : c == 1 ? V.L1 : c == 2 ? V.L2 : V.L3;
    return base + ck + cnt;
}
