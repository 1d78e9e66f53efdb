// sa_resolve.cu -- text positions of the SA lookups of a batch on a compact index (1/32 of the suffix array in HBM).
//
//   k_sa_count    thread per read: cnt[r] = the read's lookups (sa_lookup.cuh); an exclusive scan turns the counts into offsets
//   k_sa_rows     warp per read: pos[off[r] + t] = the row of lookup t, in the order the chain kernels consume them
//   k_sa_resolve  every row in place -> its text position: bwa's bwt_sa.  Walk bwt_invPsi (one 64-byte Occ block per step) until the
//                 row is a multiple of 32; the position is (sample + steps) mod (n + 1).  Sample 0 holds n, so a walk through the
//                 primary row (LF = 0) gives steps - 1, bwa's sa[0] = -1 convention.  Walks are the gaps between sampled suffixes in
//                 text order: 32 steps on average with a long tail, so lanes are persistent and take the next lookup as soon as theirs
//                 ends, from a pool of 32 per warp refilled with one atomic ticket (the shape of k_sa_from_samples, index_file.cu).
// A row outside [0, n] or a walk longer than n (a damaged index: LF is one cycle over the n + 1 rows) stops that walk and is reported
// in err; no out-of-range row is ever read.
#include <algorithm>
#include "pipeline.cuh"
#include "primitives.cuh"
#include "sa_lookup.cuh"
#include "launch_cache.cuh"

namespace {

constexpr int RS_THREADS = 256;

__global__ void k_sa_count(const Intv* intv, const uint32_t* intv_cnt, uint32_t intv_cap, uint32_t n, DevOpts o, uint64_t* cnt) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += gridDim.x * blockDim.x) {
        uint64_t c = 0;
        if (r < n) {
            const Intv* iv = intv + (size_t)r * intv_cap;
            const int n_iv = (int)intv_cnt[r];
            for (int i = 0; i < n_iv; ++i) c += occ_count(o, iv[i].x2, nullptr);
        }
        cnt[r] = c;
    }
}

__global__ void k_sa_rows(const Intv* intv, const uint32_t* intv_cnt, uint32_t intv_cap, uint32_t n, DevOpts o, const uint64_t* off,
                          uint64_t* pos, uint64_t cap) {
    const uint32_t lane = threadIdx.x & 31, nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += nw) {
        const uint64_t base = off[r];
        if (off[r + 1] > cap) continue;      // the chain pool overflows too: the batch is run again with both grown
        uint64_t* out = pos + base;
        for_each_lookup(intv + (size_t)r * intv_cap, (int)intv_cnt[r], o, lane, 32u, [&](uint32_t t, const Intv&, uint64_t row) { out[t] = row; });
    }
}

__device__ __forceinline__ void resolve_fail(uint32_t* err, uint32_t code) { atomicCAS(err, 0u, code); }

template <class SaT>
__global__ void __launch_bounds__(RS_THREADS) k_sa_resolve(LfView V, const SaT* __restrict__ samples, uint64_t* pos, const uint64_t* total_p,
                                                            uint64_t cap, uint32_t* ticket, uint32_t* err, unsigned long long* lf_steps,
                                                            unsigned long long* n_iters) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const uint64_t total = *total_p <= cap ? *total_p : 0;   // more lookups than slots: the batch runs again, with more slots
    bool active = false, dry = false;
    uint64_t j = 0, slot = 0, steps = 0, all_steps = 0, iters = 0;
    uint32_t pool = 0, used = 32;          // the warp's current block of 32 lookups [pool, pool + 32), `used` of them handed out
    for (;;) {
        const bool need = !active && !dry;
        const uint32_t nm = __ballot_sync(FULL, need);
        if (nm) {                          // idle lanes take the next lookups of the pool, a new block when it runs dry
            const uint32_t k = __popc(nm), avail = 32 - used;
            uint32_t fresh = 0;
            if (k > avail) {
                if (lane == 0) fresh = atomicAdd(ticket, 32u);
                fresh = __shfl_sync(FULL, fresh, 0);
            }
            if (need) {
                const uint32_t r = __popc(nm & lt);
                const uint64_t s = r < avail ? (uint64_t)pool + used + r : (uint64_t)fresh + (r - avail);
                if (s >= total) dry = true;
                else {
                    slot = s; j = pos[s]; steps = 0;
                    if (j > V.n) { resolve_fail(err, 1u); dry = true; }
                    else active = true;
                }
            }
            if (k > avail) { pool = fresh; used = k - avail; } else used += k;
        }
        if (!__any_sync(FULL, active)) { if (__all_sync(FULL, dry)) break; continue; }
        ++iters;
        if (active) {
            if ((j & 31) == 0) {           // a sampled row: this lookup is done
                uint64_t p = (uint64_t)samples[j >> 5] + steps;
                if (p > V.n) p -= V.n + 1;
                pos[slot] = p;
                active = false;
            } else {
                j = lf(V, j); ++steps; ++all_steps;
                if (j > V.n || steps > V.n) { resolve_fail(err, 2u); active = false; dry = true; }
            }
        }
        if ((iters & 63) == 0 && __shfl_sync(FULL, *(volatile uint32_t*)err, 0)) break;   // another warp found damage
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) all_steps += __shfl_xor_sync(FULL, all_steps, o);
    if (lane == 0 && lf_steps) { atomicAdd(lf_steps, (unsigned long long)all_steps); atomicAdd(n_iters, (unsigned long long)iters); }
}

}  // namespace

void launch_sa_resolve(const DevIndex& ix, uint64_t* pos, const uint64_t* total, uint64_t cap, uint32_t* ticket, uint32_t* err,
                       unsigned long long* lf_steps, unsigned long long* iters, cudaStream_t st) {
    LfView V;
    V.occ = ix.occ; V.n = ix.seq_len; V.primary = ix.primary; V.L0 = ix.L2[0]; V.L1 = ix.L2[1]; V.L2 = ix.L2[2]; V.L3 = ix.L2[3];
    const int sms = cached_sm_count();
    if (ix.sa_bytes == 4) {
        const int nb = cached_blocks_per_sm(k_sa_resolve<uint32_t>, RS_THREADS, 0);
        k_sa_resolve<uint32_t><<<nb * sms, RS_THREADS, 0, st>>>(V, static_cast<const uint32_t*>(ix.sa), pos, total, cap, ticket, err, lf_steps, iters);
    } else {
        const int nb = cached_blocks_per_sm(k_sa_resolve<uint64_t>, RS_THREADS, 0);
        k_sa_resolve<uint64_t><<<nb * sms, RS_THREADS, 0, st>>>(V, static_cast<const uint64_t*>(ix.sa), pos, total, cap, ticket, err, lf_steps, iters);
    }
}

void launch_sa_resolve_batch(const SaResolveParams& p, const DevIndex& ix, const DevOpts& o, cudaStream_t st, uint64_t* launches) {
    const uint32_t n = p.n_reads;
    const unsigned g1 = (unsigned)std::min<uint64_t>(((uint64_t)n + 256) / 256, 148 * 8), g2 = (unsigned)std::min<uint64_t>(((uint64_t)n + 7) / 8, 148 * 16);
    k_sa_count<<<g1, 256, 0, st>>>(p.intv, p.intv_cnt, p.intv_cap, n, o, p.off);
    prim::device_scan<uint64_t, prim::OpSum, false>(p.off, p.off, (size_t)n + 1, p.scan_tmp, prim::OpSum(), st, launches);
    k_sa_rows<<<g2, 256, 0, st>>>(p.intv, p.intv_cnt, p.intv_cap, n, o, p.off, p.pos, p.pos_cap);
    launch_sa_resolve(ix, p.pos, p.off + n, p.pos_cap, p.ticket, p.err, p.lf_steps, p.iters, st);
    if (launches) *launches += 3;
}
