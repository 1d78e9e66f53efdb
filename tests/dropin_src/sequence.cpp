// tests/dropin_src/sequence.cpp -- TEST INFRASTRUCTURE: see sequence.h.  The datum is the host mirror's varlena payload behind a 4-byte
// length word, in palloc'ed memory as the reference's nuclseq_from_text returns it.
#include "sequence.h"

#include <cstring>
#include <vector>

#include "../../bioseqdb_b200/host/sequence.h"

NucleotideSequence* nuclseq_from_text(std::string_view text) {
    const std::vector<uint8_t> payload = bioseqdb::nuclseq_from_text(text).varlena_payload();
    char* datum = static_cast<char*>(palloc0(VARHDRSZ + payload.size()));
    SET_VARSIZE(datum, VARHDRSZ + payload.size());
    memcpy(datum + VARHDRSZ, payload.data(), payload.size());
    return reinterpret_cast<NucleotideSequence*>(datum);
}

char* NucleotideSequence::to_text_palloc() const {
    char* text = static_cast<char*>(palloc(len + 1));
    for (uint32_t i = 0; i < len; ++i) text[i] = "ACGT"[pac_raw_get(pac(), i)];
    for (uint32_t k = 0; k < holes_num; ++k) {
        bntamb1_t h;
        memcpy(&h, holes() + k, sizeof(h));       // hole records start 4 bytes past an 8-byte boundary
        memset(text + h.offset, h.amb, (size_t)h.len);
    }
    text[len] = 0;
    return text;
}
