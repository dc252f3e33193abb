// filters.cuh -- launch interface of the post-scan filters (filters.cu) and the record sort
// (radix_sort.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "lines.cuh"
#include "scan.cuh"

namespace olm {

// Bytes of scratch both filters need for n records.
size_t filter_scratch_bytes(uint64_t n);

// Greedy no-overlap over n sorted records: kept records are written to `out` (must not alias
// `in`), their count to *d_total (device).  matcher.c:570-584.  Records that start before `floor`
// are dropped and the chain starts at the first record at or past it: the chain of a stream whose
// earlier records ended their last kept match at `floor` (0: the plain filter).  With `in_pos`, the
// line positions of the records (lines.cuh, one per record) are compacted with the same keep flags
// into `out_pos`.
cudaError_t no_overlap_launch(const Record *in, uint64_t n, Record *out, void *scratch,
                              unsigned long long *d_total, cudaStream_t st, uint32_t *launches, uint64_t floor = 0,
                              const LinePos *in_pos = nullptr, LinePos *out_pos = nullptr);

// Longest-only over n sorted records (first record of every offset).  matcher.c:564-579.
cudaError_t longest_launch(const Record *in, uint64_t n, Record *out, void *scratch,
                           unsigned long long *d_total, cudaStream_t st, uint32_t *launches);

// LSD radix sort of records by (offset ascending, length descending); matcher.c:258-325.
// `tmp` holds n records; the sorted data ends up in `data`.
size_t sort_scratch_bytes(uint64_t n);
cudaError_t sort_records_launch(Record *data, Record *tmp, uint64_t n, void *scratch, cudaStream_t st,
                                uint32_t *launches);

} // namespace olm
