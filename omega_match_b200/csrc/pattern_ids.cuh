// pattern_ids.cuh -- launch interface of the pattern-id pass (pattern_ids.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "scan.cuh"

namespace olm {

// The device copy of a store's catalogue (store.h PatternCatalog).
struct PatternIdTables {
  const uint2 *table = nullptr;      // {id, fingerprint}, table_mask + 1 entries
  uint32_t table_mask = 0;
  const uint2 *refs = nullptr;       // per id {offset, len}
  const uint8_t *store = nullptr;    // DeviceStore::store: bytes of the long patterns
  const uint8_t *short_bytes = nullptr;
  uint32_t store_flags = 0;          // kFlagIgnoreCase | kFlagIgnorePunct | kFlagElideSpace
  uint32_t count = 0;                // catalogue size: ids are 0 .. count - 1
};

// Writes the id of each record's pattern into Record::_pad.  `buf` holds the global haystack
// bytes [buf_begin, ...) (the buffer the records were matched in).  A record whose bytes name no
// pattern gets kNoPatternId and is counted into *d_missing.
cudaError_t pattern_ids_launch(Record *records, uint64_t n, const uint8_t *buf, uint64_t buf_begin,
                               const PatternIdTables &t, unsigned long long *d_missing, int sms,
                               cudaStream_t stream, uint32_t *launches);

// Adds to counts[id] (count entries) the number of records [0, n) whose pattern is id.  With `buf`
// the ids are resolved from the haystack as pattern_ids_launch does (the pads are not written);
// with buf == nullptr they are read from the records' pad words.  A record whose bytes name no
// pattern, or whose pad holds an id >= t.count, is not counted but counted into *d_missing.
// `block_table` selects the histogram with a per-block shared-memory table of ids
// (pattern_counts_block_table() is the rule the engine uses).
cudaError_t pattern_counts_launch(const Record *records, uint64_t n, const uint8_t *buf, uint64_t buf_begin,
                                  const PatternIdTables &t, bool block_table, unsigned long long *counts,
                                  unsigned long long *d_missing, int sms, cudaStream_t stream, uint32_t *launches);
// Whether n records over the catalogue of `t` repeat ids enough for the block table to pay.
bool pattern_counts_block_table(uint64_t n, const PatternIdTables &t);

} // namespace olm
