// lines.cuh -- launch interface of the line passes (lines.cu): where the newlines of a byte range
// are, the line of every record, and the matching lines of a call (include/olm_b200.h "lines").
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "scan.cuh"

namespace olm {

// olm_line_pos_t / olm_line_t / olm_newline_facts_t of include/olm_b200.h
struct LinePos {
  unsigned long long line, begin, end;
};
struct LineEntry {
  unsigned long long line, begin, end, records;
};
struct NewlineFacts {
  unsigned long long newlines, first, last;
};
struct LineOrigin {
  uint64_t line, begin, next_newline;
};
constexpr unsigned long long kNoNewline = ~0ull;
// bytes per tile of the newline facts (one bitmap of a tile fits a block's shared memory)
constexpr uint32_t kLineTileBytes = 64 * 1024;

// Device scratch of the newline facts of `len` bytes: per tile {count, first, last} and the scan of
// the tiles (newlines before, last newline before, first newline after), per record-block starts.
size_t line_tiles_bytes(uint64_t len);

// Pass 1 over bytes[0, len) (16-byte aligned): the tiles' facts and their scan into `tiles`
// (line_tiles_bytes(len)), the facts of the whole range into *d_facts (positions relative to bytes).
cudaError_t newline_facts_launch(const uint8_t *bytes, uint64_t len, void *tiles, NewlineFacts *d_facts,
                                 cudaStream_t st, uint32_t *launches);

// Pass 2, after newline_facts_launch on the same bytes and tiles: the position of each of the n records
// (offset order; global offsets, bytes[0] is the byte at global offset bytes_begin).  A record whose
// offset lies outside [bytes_begin, bytes_begin + len) is counted into *d_outside and not written.
// `origin.next_newline` == kNoNewline leaves the end of the records on the range's last line at
// kNoNewline (a later range resolves it).
cudaError_t line_positions_launch(const Record *rec, uint64_t n, const uint8_t *bytes, uint64_t bytes_begin,
                                  uint64_t len, void *tiles, const LineOrigin &origin, LinePos *out,
                                  unsigned long long *d_outside, cudaStream_t st, uint32_t *launches);

// Run-length encoding of n positions (line order) by line: the entries go to `out` (n at most),
// their number to *d_count.  `scratch`: matching_lines_scratch_bytes(n).
size_t matching_lines_scratch_bytes(uint64_t n);
cudaError_t matching_lines_launch(const LinePos *pos, uint64_t n, LineEntry *out, void *scratch,
                                  unsigned long long *d_count, cudaStream_t st, uint32_t *launches);

} // namespace olm
