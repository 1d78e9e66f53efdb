// tests/dropin_src/sequence.h -- TEST INFRASTRUCTURE: stand-in for the reference's bioseqdb/sequence.h, reduced to the surface that the
// drop-in adapter (integration/bioseqdb/bwa.{h,cpp}) and tests/dropin_check.cpp use: the NUCLSEQ varlena {vl_len[4], u32 holes_num,
// u32 len, bntamb1_t holes[], u8 pac[]} (SURVEY.md section 2, component 2), pac_byte_size, pac_raw_get, nuclseq_from_text and
// to_text_palloc.  The codec behind it is the repository's host mirror (bioseqdb_b200/host/sequence.cpp).
#pragma once
#include <cstddef>
#include <cstdint>
#include <string_view>

#include "postgres.h"
extern "C" {
#include <bwa/bwt.h>
#include <bwa/bwamem.h>
}

struct NucleotideSequence {
    char vl_len_[4];
    uint32_t holes_num;
    uint32_t len;

    const bntamb1_t* holes() const { return reinterpret_cast<const bntamb1_t*>(reinterpret_cast<const char*>(this) + 12); }
    const ubyte_t* pac() const { return reinterpret_cast<const ubyte_t*>(holes() + holes_num); }
    char* to_text_palloc() const;
};

static inline size_t pac_byte_size(size_t x) { return x / 4 + (x % 4 != 0 ? 1 : 0); }
static inline uint8_t pac_raw_get(const ubyte_t* pac, size_t index) { return pac[index >> 2] >> ((~index & 3) << 1) & 3; }
NucleotideSequence* nuclseq_from_text(std::string_view text);
