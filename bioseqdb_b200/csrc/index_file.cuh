// index_file.cuh -- the on-disk form of a built index (bsq_index_save / bsq_index_load, index_file.cu).
//
// One little-endian file: a 320-byte header, then seven sections, each starting at a 64-byte boundary, in this order:
//   pac          the forward 2-bit text as the index holds it (byte-rounded rows)
//   occ          the device Occ array verbatim: 64-byte blocks {4 x u64 counts, 8 x u32 of 16 symbols} + the trailing count record
//   sa_samples   SA[0], SA[32], SA[64], ... as u64, (seq_len + 32) / 32 entries; entry 0 holds seq_len
//   ann_offset, ann_len, ann_id
//   host_state   the blob of bsq_index_host_state_get (ambiguity holes and their rows)
// The full suffix array (49.6 of 53.5 GB at 3.1 Gbp) is not stored: the load rebuilds it on the device from the samples by LF walks
// (k_sa_from_samples), or keeps only the samples when it does not fit (the compact layout, bsq_index_meta.sa_interval = 32; saving such
// an index writes the same file).  Neither are the per-device derived arrays (inverse SA, prefix table): bsq_index_prepare builds them.
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/bioseqdb_gpu.h"

constexpr uint32_t IDX_FILE_VERSION = 1;
constexpr uint32_t IDX_FILE_BYTE_ORDER = 0x01020304u;   // read back as 0x04030201 on a big-endian host
constexpr uint32_t IDX_FILE_SA_INTERVAL = 32;
constexpr uint64_t IDX_FILE_ALIGN = 64;
constexpr uint64_t IDX_FILE_HEADER_BYTES = 320;

enum { SEC_PAC = 0, SEC_OCC, SEC_SA_SAMPLES, SEC_ANN_OFFSET, SEC_ANN_LEN, SEC_ANN_ID, SEC_HOST_STATE, SEC_COUNT };
extern const char* const kSectionName[SEC_COUNT];

struct IndexFileSection { uint64_t offset, bytes, checksum; };
struct IndexFileHeader {
    char magic[8];                       // "BSQIDX\0\0"
    uint32_t version, byte_order;
    int64_t l_pac; uint64_t seq_len, primary, L2[5], n_anns;
    uint32_t sa_bytes, sa_interval;
    double build_ms; uint64_t build_launches, sort_pass_bytes;   // the builder's figures, kept verbatim
    uint8_t key[16];                     // opaque caller key (the index caches store their content digest), zeros without one
    IndexFileSection sec[SEC_COUNT];
    uint64_t header_checksum;            // section_checksum over every byte above
};
static_assert(sizeof(IndexFileHeader) == 312 && sizeof(IndexFileHeader) <= IDX_FILE_HEADER_BYTES, "header layout");

// The checksum of a section: its bytes as u64 words w_i (the tail zero-padded), sum of splitmix64(w_i ^ i * golden) mod 2^64.  A plain
// sum of position-keyed terms: order-sensitive, and a GPU reduction of it is deterministic.
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t checksum_term(uint64_t w, uint64_t i) { return splitmix64(w ^ (i * 0x9e3779b97f4a7c15ull)); }
uint64_t checksum_host(const void* p, uint64_t bytes);

// Device arrays of an index, as the file is written from / read into them.
struct IndexFileArrays {
    uint8_t* pac; uint32_t* occ; void* sa; int64_t* ann_offset; int32_t* ann_len; int64_t* ann_id;
};

// Save: every device section (d_samples: rows 0, 32, 64, ... of the full SA) hashed on the device; pac and the annotations are written
// from the host mirrors, Occ and the samples through pinned staging.  The file appears under `path` only when complete (temporary name,
// fsync, rename).
int index_file_save(const char* path, const bsq_index_meta& m, const IndexFileArrays& d, const uint64_t* d_samples, const uint8_t* pac,
                    const int64_t* ann_offset, const int32_t* ann_len, const int64_t* ann_id, const std::vector<uint8_t>& host_state,
                    const uint8_t* key, cudaStream_t st);

// Load, step 1: open the file, check the header against itself, the file size and `key`; *m = the meta of the index it holds.
struct IndexFileReader { int fd = -1; uint64_t file_bytes = 0; IndexFileHeader hdr; std::string path; };
int index_file_open(IndexFileReader& r, const char* path, const uint8_t* key, bsq_index_meta* m);
// Load, step 2 (arrays allocated for *m): sections uploaded, checksummed on the device, full SA rebuilt -- or, compact, d.sa = the
// samples, checked and as wide as the index's SA entries; host_state = the blob.
int index_file_fill(IndexFileReader& r, const IndexFileArrays& d, bool compact, std::vector<uint8_t>& host_state, int device, cudaStream_t st,
                    bsq_index_load_info* info);
void index_file_close(IndexFileReader& r);
