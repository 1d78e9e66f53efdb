// index_verify.cuh -- device-side check of an FM-index against its text (index_verify.cu)
#pragma once
#include "common.cuh"
enum { IV_SA_SUM = 0, IV_SA_SUMSQ, IV_SA_RANGE_BAD, IV_TEXT_CNT /* 4 words */, IV_ORDER_CHECKED = 7, IV_ORDER_BAD, IV_ORDER_UNDECIDED,
       IV_ROWS_CHECKED, IV_BWT_BAD, IV_LF_BAD, IV_OCC_CHECKED, IV_OCC_BAD, IV_WORDS = 16 };
// iv: the index's SA interval -- 1 (full SA) or 32 (compact: ix.sa holds SA[0], SA[32], ...; the checks that need the full SA are skipped)
void launch_index_verify(const DevIndex& ix, uint32_t iv, uint64_t n_samples, uint64_t seed, uint64_t max_lcp, unsigned long long* d_out, cudaStream_t st);
