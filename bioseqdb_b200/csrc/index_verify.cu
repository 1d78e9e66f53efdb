// index_verify.cu -- checks a device FM-index against the TEXT it was built from, without any code of the builder or of the
// seeding kernels (VERDICT r1 item 1c: "so the 6.2 G-row index is checked by something other than itself").  What is checked:
//   * SA is a permutation of 0..n          -- sum and sum of squares of every entry (mod 2^64) against the closed forms (all rows);
//   * SA is sorted                          -- suffix SA[k] < suffix SA[k+1] by direct comparison of the text T = fwd || revcomp
//                                              (the suffix that runs into the end of the text is the smaller one), sampled rows;
//   * the BWT string is the text seen through SA -- B0[k'] == T[SA[k] - 1] for sampled rows k != primary, SA[primary] == 0;
//   * Occ / L2 give LF                      -- bwt_invPsi(k) = L2[c] + occ(k, c) lands on the row of suffix SA[k] - 1, sampled rows
//                                              (reference call sites: bwt_sa / bwt_extend behind bwa.cpp:149);
//   * the Occ checkpoints                   -- counts of block b+1 == counts of block b + a recount of the block's symbols, sampled
//                                              blocks; first record zero; trailing record == L2 differences;
//   * L2                                    -- L2[c+1] - L2[c] == occurrences of c in T, counted from pac (all bases).
// "Sampled" means every row / block when n_samples covers them (small indexes, tests), else rows drawn by splitmix64.
// A compact index (SA interval 32) holds SA[32 k] only: the sums, range and LF checks cover nothing it does not hold, order compares
// consecutive samples, the BWT check runs on the sampled rows; Occ and L2 are checked as for a full index.
#include <cstdint>
#include <cuda_runtime.h>
#include "common.cuh"
#include "index_verify.cuh"

namespace {

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}
// the i-th of m samples over [0, range): all of them when m >= range
__device__ __forceinline__ uint64_t sample_of(uint64_t i, uint64_t m, uint64_t range, uint64_t seed) {
    return m >= range ? i : splitmix64(seed ^ (i * 0x2545f4914f6cdd1dull)) % range;
}
__device__ __forceinline__ uint32_t text_at(const DevIndex& ix, uint64_t p) { return ref_base(ix, (int64_t)p); }

// symbol x of the $-less BWT string, read straight from the interleaved blocks
__device__ __forceinline__ uint32_t b0_at(const DevIndex& ix, uint64_t x) {
    const uint32_t w = ix.occ[((x >> 7) << 4) + 8 + ((x & 127) >> 4)];
    return (w >> ((15 - (x & 15)) << 1)) & 3u;
}
__device__ __forceinline__ uint64_t block_count(const DevIndex& ix, uint64_t b, int c) {
    return reinterpret_cast<const unsigned long long*>(ix.occ + (b << 4))[c];
}
// occurrences of c in B0[0 .. x] (x inclusive), one symbol at a time from the block's checkpoint
__device__ uint64_t occ_upto(const DevIndex& ix, uint64_t x, uint32_t c) {
    const uint64_t b = x >> 7;
    uint64_t cnt = block_count(ix, b, (int)c);
    for (uint64_t j = b << 7; j <= x; ++j) cnt += b0_at(ix, j) == c;
    return cnt;
}

// out: see IV_* in index_verify.cuh
__global__ void k_verify_sa_sums(DevIndex ix, uint64_t rows, unsigned long long* out) {
    unsigned long long s = 0, q = 0;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < rows; k += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long v = sa_at(ix, k);
        s += v; q += v * v;
        if (v > ix.seq_len) atomicAdd(out + IV_SA_RANGE_BAD, 1ull);
    }
    for (int d = 16; d; d >>= 1) { s += __shfl_xor_sync(FULL, s, d); q += __shfl_xor_sync(FULL, q, d); }
    if ((threadIdx.x & 31) == 0) { atomicAdd(out + IV_SA_SUM, s); atomicAdd(out + IV_SA_SUMSQ, q); }
}

__global__ void k_verify_text_counts(DevIndex ix, unsigned long long* out) {
    unsigned long long c4[4] = {0, 0, 0, 0};
    const uint64_t l = (uint64_t)ix.l_pac;
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < l; p += (uint64_t)gridDim.x * blockDim.x) ++c4[pac_get(ix.pac, (int64_t)p)];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        unsigned long long v = c4[c];
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(out + IV_TEXT_CNT + c, v);
    }
}

// entries k of ix.sa stand for rows k * iv; nk = entries held
__global__ void k_verify_rows(DevIndex ix, uint32_t iv, uint64_t m, uint64_t seed, uint64_t max_lcp, unsigned long long* out) {
    const uint64_t n = ix.seq_len, nk = (n + iv) / iv;
    unsigned long long ord_bad = 0, ord_und = 0, bwt_bad = 0, lf_bad = 0, n_ord = 0, n_row = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        // ---- order: entries k, k + 1 (k in [0, nk - 1))
        {
            const uint64_t k = sample_of(i, m, nk - 1, seed);
            if (k < nk - 1) {
                const uint64_t a = sa_at(ix, k), b = sa_at(ix, k + 1);
                ++n_ord;
                if (a > n || b > n || a == b) ++ord_bad;
                else {
                    uint64_t t = 0; int verdict = 0;          // -1: a < b (good), +1: a > b, 0: undecided
                    for (; t < max_lcp; ++t) {
                        if (a + t >= n) { verdict = -1; break; }      // a ran into the end first (it is the shorter one or both end: a != b)
                        if (b + t >= n) { verdict = +1; break; }
                        const uint32_t ca = text_at(ix, a + t), cb = text_at(ix, b + t);
                        if (ca != cb) { verdict = ca < cb ? -1 : +1; break; }
                    }
                    if (verdict > 0) ++ord_bad; else if (verdict == 0) ++ord_und;
                }
            }
        }
        // ---- BWT symbol and LF of row k (entry e in [0, nk))
        {
            const uint64_t e = sample_of(i, m, nk, seed ^ 0x5bd1e995u);
            if (e < nk) {
                const uint64_t k = e * iv;
                ++n_row;
                const uint64_t s = sa_at(ix, e);
                if (k == ix.primary) { if (s != 0) { ++bwt_bad; lf_bad += iv == 1; } }
                else if (s == 0 || s > n) { ++bwt_bad; lf_bad += iv == 1; }
                else {
                    const uint64_t x = k - (k > ix.primary);
                    const uint32_t c = b0_at(ix, x);
                    if (c != text_at(ix, s - 1)) ++bwt_bad;
                    if (iv != 1) continue;
                    // bwt_invPsi: L2[c] + occ(k, c), occ counting B0[0 .. k - (k >= primary)]
                    const uint64_t r = ix.L2[c] + occ_upto(ix, k - (k >= ix.primary), c);
                    if (r > n || sa_at(ix, r) + 1 != s) ++lf_bad;
                }
            }
        }
    }
    unsigned long long v[6] = {n_ord, ord_bad, ord_und, n_row, bwt_bad, lf_bad};
    const int slot[6] = {IV_ORDER_CHECKED, IV_ORDER_BAD, IV_ORDER_UNDECIDED, IV_ROWS_CHECKED, IV_BWT_BAD, IV_LF_BAD};
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        unsigned long long x = v[j];
        for (int d = 16; d; d >>= 1) x += __shfl_xor_sync(FULL, x, d);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(out + slot[j], x);
    }
}

__global__ void k_verify_blocks(DevIndex ix, uint64_t m, uint64_t seed, unsigned long long* out) {
    const uint64_t n = ix.seq_len, n_blocks = (n + 127) >> 7;
    unsigned long long bad = 0, checked = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t b = sample_of(i, m, n_blocks, seed ^ 0xc2b2ae35u);
        if (b >= n_blocks) continue;
        ++checked;
        uint64_t c4[4] = {0, 0, 0, 0};
        const uint64_t end = ((b + 1) << 7) < n ? ((b + 1) << 7) : n;
        for (uint64_t j = b << 7; j < end; ++j) ++c4[b0_at(ix, j)];
        bool ok = true;
        for (int c = 0; c < 4; ++c) ok = ok && block_count(ix, b + 1, c) == block_count(ix, b, c) + c4[c];
        // bits a partial last block leaves unused must be zero (bwa's own blocks are)
        if (b == 0) for (int c = 0; c < 4; ++c) ok = ok && block_count(ix, 0, c) == 0;
        if (b == n_blocks - 1) for (int c = 0; c < 4; ++c) ok = ok && block_count(ix, n_blocks, c) == ix.L2[c + 1] - ix.L2[c];
        if (!ok) ++bad;
    }
    for (int d = 16; d; d >>= 1) { bad += __shfl_xor_sync(FULL, bad, d); checked += __shfl_xor_sync(FULL, checked, d); }
    if ((threadIdx.x & 31) == 0) { if (bad) atomicAdd(out + IV_OCC_BAD, bad); if (checked) atomicAdd(out + IV_OCC_CHECKED, checked); }
}

}  // namespace

void launch_index_verify(const DevIndex& ix, uint32_t iv, uint64_t n_samples, uint64_t seed, uint64_t max_lcp, unsigned long long* d_out, cudaStream_t st) {
    cudaMemsetAsync(d_out, 0, IV_WORDS * 8, st);
    const unsigned grid = 148 * 8;
    const uint64_t rows = (ix.seq_len + iv) / iv, blocks = (ix.seq_len + 127) >> 7;
    k_verify_sa_sums<<<grid, 256, 0, st>>>(ix, rows, d_out);
    k_verify_text_counts<<<grid, 256, 0, st>>>(ix, d_out);
    const uint64_t m_rows = n_samples >= rows ? rows : n_samples, m_blk = n_samples >= blocks ? blocks : n_samples;
    k_verify_rows<<<grid, 256, 0, st>>>(ix, iv, m_rows, seed, max_lcp, d_out);
    k_verify_blocks<<<grid, 256, 0, st>>>(ix, m_blk, seed, d_out);
}
