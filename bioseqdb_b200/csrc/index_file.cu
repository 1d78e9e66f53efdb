// index_file.cu -- writing a built index to one file and reading it back (layout: index_file.cuh).
//
//   k_section_checksum   the per-section checksum, one grid-stride pass + warp sums + one atomic per warp (a plain sum: deterministic)
//   k_sa_from_samples    the full suffix array from its 1/32 samples.  LF is one cycle over the n + 1 rows and row 0 (SA = n) is a
//                        sample, so the chains that start at the sampled rows and walk LF until the next sampled row cover every other
//                        row exactly once:  row j = 32 s, p = sample[s]: SA[j] = p; loop { j = LF(j); if (j % 32 == 0) break; SA[j] = --p; }
//                        Chains are the gaps between sampled suffixes in text order (32 on average, with a long tail); lanes are
//                        persistent and take the next sample as soon as their chain ends, from a pool of 32 samples per warp refilled
//                        with one atomic ticket.  Every step reads one 64-byte Occ block at a random row and scatters one SA entry.
// A file that got past its checksums can still be wrong: a row outside [0, n], a sample above n or a chain longer than n stops the walk
// and is reported, and no index the kernel computes is used before it has been range-checked.
#include <cerrno>
#include <cstddef>
#include <chrono>
#include <cstring>
#include <string>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include "index_file.cuh"
#include "common.cuh"

const char* const kSectionName[SEC_COUNT] = {"pac", "occ", "sa_samples", "ann_offset", "ann_len", "ann_id", "host_state"};

uint64_t checksum_host(const void* p, uint64_t bytes) {
    const uint8_t* s = static_cast<const uint8_t*>(p);
    const uint64_t nw = bytes / 8;
    uint64_t sum = 0;
    for (uint64_t i = 0; i < nw; ++i) { uint64_t w; memcpy(&w, s + i * 8, 8); sum += checksum_term(w, i); }
    if (bytes & 7) { uint64_t w = 0; memcpy(&w, s + nw * 8, bytes & 7); sum += checksum_term(w, nw); }
    return sum;
}

namespace {

constexpr int CK_THREADS = 256, SA_THREADS = 256;

// out += checksum of bytes [0, bytes) of p (p 8-byte aligned: every section sits at the start of its own cudaMalloc)
__global__ void __launch_bounds__(CK_THREADS) k_section_checksum(const uint8_t* __restrict__ p, uint64_t bytes, unsigned long long* out) {
    const uint64_t nw = bytes >> 3;
    uint64_t s = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (uint64_t)gridDim.x * blockDim.x)
        s += checksum_term(__ldg(reinterpret_cast<const unsigned long long*>(p) + i), i);
    if (blockIdx.x == 0 && threadIdx.x == 0 && (bytes & 7)) {
        uint64_t w = 0;
        for (uint64_t b = nw << 3; b < bytes; ++b) w |= (uint64_t)p[b] << ((b & 7) << 3);
        s += checksum_term(w, nw);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, (unsigned long long)s);
}

struct SaRebuild {
    const uint32_t* occ; const uint64_t* samples;
    uint64_t n, primary, L0, L1, L2, L3;     // L2[0..3] of the index
    uint32_t n_samples;
    unsigned int* ticket;
    unsigned long long* stats;               // [0] error code, [1] where, [2] rows written, [3] LF steps, [4] warp iterations
};
enum { SA_ERR_SAMPLE = 1, SA_ERR_ROW = 2, SA_ERR_CHAIN = 3 };

__device__ __forceinline__ void sa_fail(const SaRebuild& P, unsigned long long code, unsigned long long where) {
    if (atomicCAS(P.stats, 0ull, code) == 0ull) atomicExch(P.stats + 1, where);
}

// bwt_invPsi (libbwa bwt.h) for a row j in [0, n]: 0 for the primary row, else L2[c] + occ(j, c) with c = B0[j - (j > primary)] and occ
// the count of c in B0[0 .. j - (j >= primary)] -- the checkpoint of j's 128-symbol block plus the popcounts of its symbols up to j.
__device__ __forceinline__ uint64_t lf(const SaRebuild& P, uint64_t j) {
    if (j == P.primary) return 0;
    const uint64_t x = j - (j > P.primary);
    const uint4* blk = reinterpret_cast<const uint4*>(P.occ + ((size_t)(x >> 7) << 4));
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
    const uint64_t base = c == 0 ? P.L0 : c == 1 ? P.L1 : c == 2 ? P.L2 : P.L3;
    return base + ck + cnt;
}

template <class SaT>
__global__ void __launch_bounds__(SA_THREADS) k_sa_from_samples(SaRebuild P, SaT* __restrict__ sa) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    bool active = false, dry = false;
    uint64_t j = 0, p = 0, len = 0, written = 0, steps = 0, iters = 0;
    uint32_t pool = 0, used = 32;          // the warp's current block of 32 samples [pool, pool + 32), `used` of them handed out
    for (;;) {
        const bool need = !active && !dry;
        const uint32_t nm = __ballot_sync(FULL, need);
        if (nm) {                          // idle lanes take the next samples of the pool, a new block when it runs dry
            const uint32_t k = __popc(nm), avail = 32 - used;
            uint32_t fresh = 0;
            if (k > avail) {
                if (lane == 0) fresh = atomicAdd(P.ticket, 32u);
                fresh = __shfl_sync(FULL, fresh, 0);
            }
            if (need) {
                const uint32_t r = __popc(nm & lt);
                const uint32_t s = r < avail ? pool + used + r : fresh + (r - avail);
                if (s >= P.n_samples) dry = true;
                else {
                    j = (uint64_t)s * 32; p = __ldg(P.samples + s); len = 0;
                    if (p > P.n) { sa_fail(P, SA_ERR_SAMPLE, s); dry = true; }
                    else { sa[j] = (SaT)p; ++written; active = true; }
                }
            }
            if (k > avail) { pool = fresh; used = k - avail; } else used += k;
        }
        if (!__any_sync(FULL, active)) break;
        ++iters;
        if (active) {
            const uint64_t nj = lf(P, j);
            ++steps;
            if (nj > P.n) { sa_fail(P, SA_ERR_ROW, j); active = false; dry = true; }
            else if ((nj & 31) == 0) active = false;                   // reached the next sampled row: this chain is done
            else if (p == 0 || ++len > P.n) { sa_fail(P, SA_ERR_CHAIN, j); active = false; dry = true; }
            else { j = nj; sa[j] = (SaT)--p; ++written; }
        }
        if ((iters & 63) == 0 && __shfl_sync(FULL, *(volatile unsigned long long*)P.stats, 0)) break;   // another warp found damage
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { written += __shfl_xor_sync(FULL, written, o); steps += __shfl_xor_sync(FULL, steps, o); }
    if (lane == 0) { atomicAdd(P.stats + 2, (unsigned long long)written); atomicAdd(P.stats + 3, (unsigned long long)steps); atomicAdd(P.stats + 4, (unsigned long long)iters); }
}

// two pinned buffers: the file read of one chunk overlaps the copy of the other
struct Staging {
    static constexpr size_t CAP = 16u << 20;
    void* buf[2] = {nullptr, nullptr}; cudaEvent_t ev[2] = {nullptr, nullptr};
    int init() {
        for (int k = 0; k < 2; ++k) {
            CUDA_CHECK(cudaHostAlloc(&buf[k], CAP, cudaHostAllocDefault));
            CUDA_CHECK(cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming));
        }
        return BSQ_OK;
    }
    ~Staging() { for (int k = 0; k < 2; ++k) { if (ev[k]) cudaEventSynchronize(ev[k]), cudaEventDestroy(ev[k]); if (buf[k]) cudaFreeHost(buf[k]); } }
};

struct DevScratch {   // device buffers of one call, freed on every way out
    void* p[3] = {nullptr, nullptr, nullptr};
    ~DevScratch() { for (void* q : p) if (q) cudaFree(q); }
};

int io_error(const char* what, const char* path) { bsq_set_error("%s %s: %s", what, path, strerror(errno)); return BSQ_ERR; }

int write_full(int fd, const void* p, uint64_t n, const char* path) {
    const uint8_t* s = static_cast<const uint8_t*>(p);
    while (n) {
        const ssize_t w = write(fd, s, n < (1ull << 30) ? n : (1ull << 30));
        if (w < 0) { if (errno == EINTR) continue; return io_error("bsq_index_save: cannot write", path); }
        s += w; n -= (uint64_t)w;
    }
    return BSQ_OK;
}

int read_full(int fd, void* p, uint64_t n, uint64_t off, const char* path) {
    uint8_t* d = static_cast<uint8_t*>(p);
    while (n) {
        const ssize_t r = pread(fd, d, n < (1ull << 30) ? n : (1ull << 30), (off_t)off);
        if (r < 0) { if (errno == EINTR) continue; return io_error("bsq_index_load: cannot read", path); }
        if (r == 0) { bsq_set_error("bsq_index_load: %s ends inside a section", path); return BSQ_ERR; }
        d += r; n -= (uint64_t)r; off += (uint64_t)r;
    }
    return BSQ_OK;
}

// device bytes -> file, chunk i + 1 copied while chunk i is written
int download_to_file(Staging& S, int fd, const void* dsrc, uint64_t bytes, cudaStream_t st, const char* path) {
    const uint8_t* s = static_cast<const uint8_t*>(dsrc);
    const uint64_t n_chunks = (bytes + Staging::CAP - 1) / Staging::CAP;
    auto enqueue = [&](uint64_t i) -> cudaError_t {
        const uint64_t at = i * Staging::CAP, c = bytes - at < Staging::CAP ? bytes - at : Staging::CAP;
        cudaError_t e = cudaMemcpyAsync(S.buf[i & 1], s + at, c, cudaMemcpyDeviceToHost, st);
        return e == cudaSuccess ? cudaEventRecord(S.ev[i & 1], st) : e;
    };
    if (n_chunks) CUDA_CHECK(enqueue(0));
    for (uint64_t i = 0; i < n_chunks; ++i) {
        if (i + 1 < n_chunks) CUDA_CHECK(enqueue(i + 1));
        CUDA_CHECK(cudaEventSynchronize(S.ev[i & 1]));
        const uint64_t at = i * Staging::CAP, c = bytes - at < Staging::CAP ? bytes - at : Staging::CAP;
        if (write_full(fd, S.buf[i & 1], c, path) != BSQ_OK) return BSQ_ERR;
    }
    return BSQ_OK;
}

// file -> device bytes, the read of chunk i + 1 overlapping the copy of chunk i
int upload_from_file(Staging& S, int fd, uint64_t off, uint64_t bytes, void* ddst, cudaStream_t st, const char* path, int& k) {
    uint8_t* d = static_cast<uint8_t*>(ddst);
    for (uint64_t done = 0; done < bytes; k ^= 1) {
        const uint64_t c = bytes - done < Staging::CAP ? bytes - done : Staging::CAP;
        CUDA_CHECK(cudaEventSynchronize(S.ev[k]));          // the last copy out of this buffer has finished
        if (read_full(fd, S.buf[k], c, off + done, path) != BSQ_OK) return BSQ_ERR;
        CUDA_CHECK(cudaMemcpyAsync(d + done, S.buf[k], c, cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaEventRecord(S.ev[k], st));
        done += c;
    }
    return BSQ_OK;
}

// sums[s] = checksum of the device section s, for the six sections that live on the device
int launch_checksums(const void* const sec[SEC_HOST_STATE], const uint64_t* bytes, unsigned long long* d_sums, cudaStream_t st) {
    CUDA_CHECK(cudaMemsetAsync(d_sums, 0, SEC_HOST_STATE * 8, st));
    for (int s = 0; s < SEC_HOST_STATE; ++s) {
        const uint64_t g = (bytes[s] / 8 + CK_THREADS - 1) / CK_THREADS;
        const unsigned grid = (unsigned)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
        k_section_checksum<<<grid, CK_THREADS, 0, st>>>(static_cast<const uint8_t*>(sec[s]), bytes[s], d_sums + s);
    }
    CUDA_CHECK(cudaGetLastError());
    return BSQ_OK;
}

uint64_t align_up(uint64_t v) { return (v + IDX_FILE_ALIGN - 1) & ~(IDX_FILE_ALIGN - 1); }

// the sizes every section must have for the index the header describes (host_state: only its minimum)
void section_sizes(const IndexFileHeader& h, uint64_t out[SEC_COUNT]) {
    const uint64_t n = h.seq_len;
    out[SEC_PAC] = (uint64_t)h.l_pac / 4; out[SEC_OCC] = ((n + 127) / 128 + 1) * 64; out[SEC_SA_SAMPLES] = (n + IDX_FILE_SA_INTERVAL) / IDX_FILE_SA_INTERVAL * 8;
    out[SEC_ANN_OFFSET] = h.n_anns * 8; out[SEC_ANN_LEN] = h.n_anns * 4; out[SEC_ANN_ID] = h.n_anns * 8; out[SEC_HOST_STATE] = 8;
}

}  // namespace

int index_file_save(const char* path, const bsq_index_meta& m, const IndexFileArrays& d, const uint64_t* d_samples, const uint8_t* pac,
                    const int64_t* ann_offset, const int32_t* ann_len, const int64_t* ann_id, const std::vector<uint8_t>& host_state,
                    const uint8_t* key, cudaStream_t st) {
    IndexFileHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "BSQIDX\0\0", 8);
    h.version = IDX_FILE_VERSION; h.byte_order = IDX_FILE_BYTE_ORDER;
    h.l_pac = m.l_pac; h.seq_len = m.seq_len; h.primary = m.primary; memcpy(h.L2, m.L2, sizeof(h.L2)); h.n_anns = m.n_anns;
    h.sa_bytes = m.sa_bytes; h.sa_interval = IDX_FILE_SA_INTERVAL;
    h.build_ms = m.build_ms; h.build_launches = m.build_launches; h.sort_pass_bytes = m.sort_pass_bytes;
    if (key) memcpy(h.key, key, 16);
    uint64_t sizes[SEC_COUNT];
    section_sizes(h, sizes);
    sizes[SEC_HOST_STATE] = host_state.size();
    uint64_t off = IDX_FILE_HEADER_BYTES;
    for (int s = 0; s < SEC_COUNT; ++s) { h.sec[s].offset = off; h.sec[s].bytes = sizes[s]; off = align_up(off + sizes[s]); }

    // ---- the device checksums
    DevScratch D;
    unsigned long long* d_sums = nullptr;
    CUDA_CHECK(cudaMalloc(&D.p[0], SEC_COUNT * 8)); d_sums = static_cast<unsigned long long*>(D.p[0]);
    const void* dev_sec[SEC_HOST_STATE] = {d.pac, d.occ, d_samples, d.ann_offset, d.ann_len, d.ann_id};
    if (launch_checksums(dev_sec, sizes, d_sums, st) != BSQ_OK) return BSQ_ERR;
    uint64_t sums[SEC_COUNT];
    CUDA_CHECK(cudaMemcpyAsync(sums, d_sums, SEC_HOST_STATE * 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    sums[SEC_HOST_STATE] = checksum_host(host_state.data(), host_state.size());
    for (int s = 0; s < SEC_COUNT; ++s) h.sec[s].checksum = sums[s];
    h.header_checksum = checksum_host(&h, offsetof(IndexFileHeader, header_checksum));

    Staging S;
    if (S.init() != BSQ_OK) return BSQ_ERR;
    // ---- write to a temporary name in the same directory, fsync, rename: readers see the old file or the whole new one
    std::string tmp = std::string(path) + ".tmp.XXXXXX";
    const int fd = mkstemp(&tmp[0]);
    if (fd < 0) return io_error("bsq_index_save: cannot create a file next to", path);
    fchmod(fd, 0644);
    auto body = [&]() -> int {
        static const uint8_t zeros[IDX_FILE_HEADER_BYTES] = {};
        if (write_full(fd, &h, sizeof(h), path) != BSQ_OK || write_full(fd, zeros, IDX_FILE_HEADER_BYTES - sizeof(h), path) != BSQ_OK) return BSQ_ERR;
        const void* host_sec[SEC_COUNT] = {pac, nullptr, nullptr, ann_offset, ann_len, ann_id, host_state.data()};
        for (int s = 0; s < SEC_COUNT; ++s) {
            const int rc = host_sec[s] || sizes[s] == 0 ? write_full(fd, host_sec[s], sizes[s], path)
                                                        : download_to_file(S, fd, s == SEC_OCC ? (const void*)d.occ : (const void*)d_samples, sizes[s], st, path);
            if (rc != BSQ_OK) return BSQ_ERR;
            const uint64_t pad = (s + 1 < SEC_COUNT ? h.sec[s + 1].offset : align_up(h.sec[s].offset + sizes[s])) - (h.sec[s].offset + sizes[s]);
            if (write_full(fd, zeros, pad, path) != BSQ_OK) return BSQ_ERR;
        }
        if (fsync(fd) != 0) return io_error("bsq_index_save: cannot fsync", path);
        return BSQ_OK;
    };
    int rc = body();
    if (close(fd) != 0 && rc == BSQ_OK) rc = io_error("bsq_index_save: cannot close", path);
    if (rc == BSQ_OK && rename(tmp.c_str(), path) != 0) rc = io_error("bsq_index_save: cannot rename the temporary file to", path);
    if (rc != BSQ_OK) { unlink(tmp.c_str()); return BSQ_ERR; }
    // the rename itself is durable once the directory is synced
    std::string dir(path);
    const size_t slash = dir.find_last_of('/');
    dir = slash == std::string::npos ? "." : (slash == 0 ? "/" : dir.substr(0, slash));
    const int dfd = open(dir.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
    if (dfd >= 0) { fsync(dfd); close(dfd); }
    return BSQ_OK;
}

int index_file_open(IndexFileReader& r, const char* path, const uint8_t* key, bsq_index_meta* m) {
    r.path = path;
    r.fd = open(path, O_RDONLY | O_CLOEXEC);
    if (r.fd < 0) return io_error("bsq_index_load: cannot open", path);
    struct stat sb;
    if (fstat(r.fd, &sb) != 0) return io_error("bsq_index_load: cannot stat", path);
    r.file_bytes = (uint64_t)sb.st_size;
    if (r.file_bytes < IDX_FILE_HEADER_BYTES) { bsq_set_error("bsq_index_load: %s is %llu bytes, shorter than the %llu-byte header", path, (unsigned long long)r.file_bytes, (unsigned long long)IDX_FILE_HEADER_BYTES); return BSQ_ERR; }
    IndexFileHeader& h = r.hdr;
    if (read_full(r.fd, &h, sizeof(h), 0, path) != BSQ_OK) return BSQ_ERR;
    if (memcmp(h.magic, "BSQIDX\0\0", 8) != 0) { bsq_set_error("bsq_index_load: %s is not an index file (wrong magic)", path); return BSQ_ERR; }
    if (h.byte_order != IDX_FILE_BYTE_ORDER) { bsq_set_error("bsq_index_load: %s: byte-order word %#x, this host reads %#x", path, h.byte_order, IDX_FILE_BYTE_ORDER); return BSQ_ERR; }
    if (h.version != IDX_FILE_VERSION) { bsq_set_error("bsq_index_load: %s: format version %u, this library reads version %u", path, h.version, IDX_FILE_VERSION); return BSQ_ERR; }
    if (checksum_host(&h, offsetof(IndexFileHeader, header_checksum)) != h.header_checksum) { bsq_set_error("bsq_index_load: %s: checksum mismatch in section 'header'", path); return BSQ_ERR; }
    typedef unsigned long long ull;
    const uint64_t n = h.seq_len;
    if (h.sa_interval != IDX_FILE_SA_INTERVAL) { bsq_set_error("bsq_index_load: %s: SA sample interval %u, expected %u", path, h.sa_interval, IDX_FILE_SA_INTERVAL); return BSQ_ERR; }
    if (h.l_pac <= 0 || h.l_pac % 4 || n != 2 * (uint64_t)h.l_pac || n >= (1ull << 33)) { bsq_set_error("bsq_index_load: %s: seq_len %llu inconsistent with l_pac %lld", path, (ull)n, (long long)h.l_pac); return BSQ_ERR; }
    if (h.sa_bytes != 4 && h.sa_bytes != 8) { bsq_set_error("bsq_index_load: %s: SA entry width %u", path, h.sa_bytes); return BSQ_ERR; }
    if (h.sa_bytes == 4 && n + 1 >= (1ull << 32)) { bsq_set_error("bsq_index_load: %s: 4-byte SA entries for %llu rows (2^32 or more need 8)", path, (ull)(n + 1)); return BSQ_ERR; }
    if (h.n_anns == 0 || h.n_anns >= (1ull << 31)) { bsq_set_error("bsq_index_load: %s: n_anns %llu", path, (ull)h.n_anns); return BSQ_ERR; }
    if (h.primary == 0 || h.primary > n) { bsq_set_error("bsq_index_load: %s: primary %llu outside [1, seq_len %llu]", path, (ull)h.primary, (ull)n); return BSQ_ERR; }
    if (h.L2[0] != 0 || h.L2[4] != n || h.L2[1] < h.L2[0] || h.L2[2] < h.L2[1] || h.L2[3] < h.L2[2] || h.L2[4] < h.L2[3]) { bsq_set_error("bsq_index_load: %s: L2 inconsistent with seq_len %llu", path, (ull)n); return BSQ_ERR; }
    uint64_t want[SEC_COUNT];
    section_sizes(h, want);
    uint64_t off = IDX_FILE_HEADER_BYTES;
    for (int s = 0; s < SEC_COUNT; ++s) {
        const IndexFileSection& q = h.sec[s];
        const bool size_ok = s == SEC_HOST_STATE ? q.bytes >= 8 && (q.bytes - 8) % (sizeof(bsq_hole) + 4) == 0 : q.bytes == want[s];
        if (!size_ok) { bsq_set_error("bsq_index_load: %s: section '%s' has %llu bytes, the index needs %llu", path, kSectionName[s], (ull)q.bytes, (ull)want[s]); return BSQ_ERR; }
        if (q.offset != off) { bsq_set_error("bsq_index_load: %s: section '%s' at offset %llu, expected %llu", path, kSectionName[s], (ull)q.offset, (ull)off); return BSQ_ERR; }
        off = align_up(off + q.bytes);
    }
    const uint64_t end = h.sec[SEC_HOST_STATE].offset + h.sec[SEC_HOST_STATE].bytes;
    if (r.file_bytes < end) { bsq_set_error("bsq_index_load: %s is %llu bytes, shorter than its section table (%llu)", path, (ull)r.file_bytes, (ull)end); return BSQ_ERR; }
    if (key && memcmp(key, h.key, 16) != 0) { bsq_set_error("bsq_index_load: %s: key mismatch (the file holds the index of other content)", path); return BSQ_ERR; }
    memset(m, 0, sizeof(*m));
    m->l_pac = h.l_pac; m->seq_len = n; m->primary = h.primary; memcpy(m->L2, h.L2, sizeof(m->L2)); m->n_anns = h.n_anns; m->sa_bytes = h.sa_bytes;
    m->built = 1;
    m->arr_bytes[BSQ_ARR_PAC] = want[SEC_PAC]; m->arr_bytes[BSQ_ARR_OCC] = want[SEC_OCC]; m->arr_bytes[BSQ_ARR_SA] = (n + 1) * h.sa_bytes;
    m->arr_bytes[BSQ_ARR_ANN_OFFSET] = want[SEC_ANN_OFFSET]; m->arr_bytes[BSQ_ARR_ANN_LEN] = want[SEC_ANN_LEN]; m->arr_bytes[BSQ_ARR_ANN_ID] = want[SEC_ANN_ID];
    m->build_ms = h.build_ms; m->build_launches = h.build_launches; m->sort_pass_bytes = h.sort_pass_bytes;
    return BSQ_OK;
}

void index_file_close(IndexFileReader& r) { if (r.fd >= 0) close(r.fd); r.fd = -1; }

int index_file_fill(IndexFileReader& r, const IndexFileArrays& d, std::vector<uint8_t>& host_state, int device, cudaStream_t st,
                    bsq_index_load_info* info) {
    typedef unsigned long long ull;
    const IndexFileHeader& h = r.hdr;
    const char* path = r.path.c_str();
    const auto t0 = std::chrono::steady_clock::now();
    const uint64_t n = h.seq_len, n_samples = h.sec[SEC_SA_SAMPLES].bytes / 8;
    DevScratch D;
    uint64_t* d_samples = nullptr; ull* d_sums = nullptr; ull* d_stats = nullptr;
    CUDA_CHECK(cudaMalloc(&D.p[0], n_samples * 8 + 8)); d_samples = static_cast<uint64_t*>(D.p[0]);
    CUDA_CHECK(cudaMalloc(&D.p[1], SEC_COUNT * 8)); d_sums = static_cast<ull*>(D.p[1]);
    CUDA_CHECK(cudaMalloc(&D.p[2], 8 * 8)); d_stats = static_cast<ull*>(D.p[2]);
    // ---- read + upload
    {
        Staging S;
        if (S.init() != BSQ_OK) return BSQ_ERR;
        void* dst[SEC_HOST_STATE] = {d.pac, d.occ, d_samples, d.ann_offset, d.ann_len, d.ann_id};
        int k = 0;
        for (int s = 0; s < SEC_HOST_STATE; ++s)
            if (upload_from_file(S, r.fd, h.sec[s].offset, h.sec[s].bytes, dst[s], st, path, k) != BSQ_OK) return BSQ_ERR;
        host_state.resize(h.sec[SEC_HOST_STATE].bytes);
        if (read_full(r.fd, host_state.data(), host_state.size(), h.sec[SEC_HOST_STATE].offset, path) != BSQ_OK) return BSQ_ERR;
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
    const auto t1 = std::chrono::steady_clock::now();
    info->read_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
    // ---- checksums, before any kernel reads the sections
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 4; ++i) if (e[i]) cudaEventDestroy(e[i]); } } eg{ev};
    for (auto& e : ev) CUDA_CHECK(cudaEventCreate(&e));
    CUDA_CHECK(cudaEventRecord(ev[0], st));
    const void* dev_sec[SEC_HOST_STATE] = {d.pac, d.occ, d_samples, d.ann_offset, d.ann_len, d.ann_id};
    uint64_t sizes[SEC_COUNT];
    for (int s = 0; s < SEC_COUNT; ++s) sizes[s] = h.sec[s].bytes;
    if (launch_checksums(dev_sec, sizes, d_sums, st) != BSQ_OK) return BSQ_ERR;
    CUDA_CHECK(cudaEventRecord(ev[1], st));
    uint64_t sums[SEC_COUNT];
    CUDA_CHECK(cudaMemcpyAsync(sums, d_sums, SEC_HOST_STATE * 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    sums[SEC_HOST_STATE] = checksum_host(host_state.data(), host_state.size());
    for (int s = 0; s < SEC_COUNT; ++s)
        if (sums[s] != h.sec[s].checksum) { bsq_set_error("bsq_index_load: checksum mismatch in section '%s'", kSectionName[s]); return BSQ_ERR; }
    CUDA_CHECK(cudaEventElapsedTime(&info->checksum_ms, ev[0], ev[1]));
    // ---- the full suffix array from its samples
    SaRebuild P;
    P.occ = d.occ; P.samples = d_samples; P.n = n; P.primary = h.primary; P.L0 = h.L2[0]; P.L1 = h.L2[1]; P.L2 = h.L2[2]; P.L3 = h.L2[3];
    P.n_samples = (uint32_t)n_samples; P.ticket = reinterpret_cast<unsigned int*>(d_stats + 5); P.stats = d_stats;
    CUDA_CHECK(cudaMemsetAsync(d_stats, 0, 8 * 8, st));
    int sms = 0, per_sm = 0;
    CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (h.sa_bytes == 4) CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sa_from_samples<uint32_t>, SA_THREADS, 0));
    else CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sa_from_samples<uint64_t>, SA_THREADS, 0));
    uint64_t grid = (uint64_t)sms * (per_sm > 0 ? per_sm : 1);
    const uint64_t need = (n_samples + SA_THREADS - 1) / SA_THREADS;   // no more lanes than samples
    if (grid > need) grid = need ? need : 1;
    CUDA_CHECK(cudaEventRecord(ev[2], st));
    if (h.sa_bytes == 4) k_sa_from_samples<uint32_t><<<(unsigned)grid, SA_THREADS, 0, st>>>(P, static_cast<uint32_t*>(d.sa));
    else k_sa_from_samples<uint64_t><<<(unsigned)grid, SA_THREADS, 0, st>>>(P, static_cast<uint64_t*>(d.sa));
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaEventRecord(ev[3], st));
    ull stats[5];
    CUDA_CHECK(cudaMemcpyAsync(stats, d_stats, sizeof(stats), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    CUDA_CHECK(cudaEventElapsedTime(&info->sa_ms, ev[2], ev[3]));
    info->lf_steps = stats[3]; info->lane_slots = stats[4] * 32;
    switch (stats[0]) {
        case 0: break;
        case SA_ERR_SAMPLE: bsq_set_error("bsq_index_load: SA sample %llu is larger than seq_len %llu", stats[1], (ull)n); return BSQ_ERR;
        case SA_ERR_ROW: bsq_set_error("bsq_index_load: the LF walk from row %llu left the rows [0, %llu]", stats[1], (ull)n); return BSQ_ERR;
        default: bsq_set_error("bsq_index_load: the LF chain through row %llu does not reach a sampled row", stats[1]); return BSQ_ERR;
    }
    if (stats[2] != n + 1) { bsq_set_error("bsq_index_load: the LF chains wrote %llu of the %llu suffix-array rows", stats[2], (ull)(n + 1)); return BSQ_ERR; }
    return BSQ_OK;
}
