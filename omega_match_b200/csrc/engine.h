// engine.h -- one matcher on one GPU: the uploaded store, work buffers, and the sequence of
// kernels that make up a match call.  Plain C++ interface; api.cpp puts the C ABI on top.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/olm_b200.h"
#include "store.h"

namespace olm {

struct MatchFlags {
  bool no_overlap = false, longest_only = false, word_boundary = false, word_prefix = false,
       word_suffix = false, line_start = false, line_end = false;
};

// What part of which haystack a call scans (SURVEY 8e).
struct ScanRange {
  const void *dev = nullptr;   // device bytes of [slice_begin, slice_begin + slice_len)
  uint64_t slice_begin = 0, slice_len = 0;
  uint64_t own_begin = 0, own_end = 0; // start positions reported by this call
  uint64_t global_size = 0;
  uint64_t match_ptr_base = 0;
  uint64_t floor = 0;     // no_overlap: records before it are dropped, the chain starts there (filters.cuh)
  uint64_t out_front = 0; // records left free in front of the call's output (no_overlap off)
};

// Byte-range shards of one haystack (SURVEY 8e): a shard OWNS the start positions [own_begin,
// own_end) and needs the bytes [slice_begin, slice_end).
struct Shard {
  uint64_t own_begin = 0, own_end = 0, slice_begin = 0, slice_end = 0;
};
// The shard that owns [own_begin, own_end) of `size` bytes: 16 bytes in front (alignment + the previous
// byte) and the longest pattern + 1 behind.  Stores with a transform flag shard on multiples of the
// 4 MiB source window and need no halo.  The whole haystack is shard_of(0, size, size, ...).
inline Shard shard_of(uint64_t own_begin, uint64_t own_end, uint64_t size, uint32_t largest, bool windowed) {
  if (windowed) return Shard{own_begin, own_end, own_begin, own_end};
  return Shard{own_begin, own_end, own_begin >= 16 ? own_begin - 16 : 0, std::min<uint64_t>(size, own_end + largest + 1)};
}
// The range a call scans for shard `s`; dev: the device bytes of its slice (nullptr: a host slice)
inline ScanRange scan_range(const Shard &s, uint64_t size, uint64_t match_ptr_base, const void *dev = nullptr) {
  return ScanRange{dev, s.slice_begin, s.slice_end - s.slice_begin, s.own_begin, s.own_end, size, match_ptr_base};
}

struct EngineImpl;

// One stream (include/olm_b200.h "Streams"): the haystack arrives in pushes; `carry` holds the device
// bytes [carry_begin, received) the next push scans again (halo, or the incomplete 4 MiB window).
struct StreamState {
  MatchFlags f;
  uint64_t match_ptr_base = 0;
  uint64_t received = 0, settled = 0;
  uint64_t floor = 0; // no_overlap: the end of the last kept record
  bool finished = false, failed = false;
  void *carry = nullptr;
  size_t carry_cap = 0;
  uint64_t carry_begin = 0;
};

// What olm_cuda_match_lines / olm_cuda_matching_lines return.
struct LinesResult {
  omega_match_results_t *results = nullptr; // records (not for lines_only)
  olm_line_pos_t *positions = nullptr;      // one per record
  olm_line_t *lines = nullptr;              // lines_only
  uint64_t n_lines = 0, total = 0;          // total: the call's record count
};
// Result arrays of the host API (cuda_util.cu): pinned from 1 MiB, freed by host_result_free.
// host_results: an omega_match_results_t of `count` records (nullptr when out of memory).
void *host_result_alloc(size_t bytes);
void host_result_free(void *p);
omega_match_results_t *host_results(uint64_t count);

class Engine {
public:
  // Parses + re-stages the mapped store and uploads it.  On failure returns nullptr and
  // fills *err.
  static Engine *create(const uint8_t *file, size_t size, int device, std::string *err);
  ~Engine();

  int device() const;
  const Header &header() const;

  // Device-resident input, device-resident output (records stay in the engine's buffer).  With
  // `dev_counts` (the pattern tables loaded: load_pattern_tables) the call adds the count of its
  // final records per pattern to dev_counts[id] instead of writing ids, whether ids are on or off.
  int match_device(const ScanRange &r, const MatchFlags &f, olm_cuda_results_t *out, void *dev_counts = nullptr);
  // Host input/output: H2D, match_device, D2H into a host_results array.  One GPU, or
  // OLM_HOST_SPAN_BYTES spans (host_spans).
  omega_match_results_t *match_host(const uint8_t *haystack, size_t n, const MatchFlags &f);
  // A byte range (range.dev is ignored) whose slice lies in HOST memory: segmented H2D overlapped
  // with the scan, device-resident records.
  int match_shard_host(const uint8_t *host_slice, const ScanRange &range, const MatchFlags &f, olm_cuda_results_t *out,
                       void *dev_counts = nullptr);

  // "offset:bytes\n" for every record (the CLI's listing, main.c:89-133) as one device text buffer;
  // dev_haystack = device address of the haystack byte with offset `offset0`
  int format_records(const void *dev_records, uint64_t count, const void *dev_haystack, uint64_t offset0,
                     void **dev_text, uint64_t *text_bytes);
  // (with dev_positions: the records' line positions are compacted with them)
  // (floor: see ScanRange::floor)
  int64_t no_overlap_inplace(void *dev_records, uint64_t count, void *dev_positions = nullptr, uint64_t floor = 0);
  int sort_records(void *dev_records, uint64_t count);

  // for the multi-GPU layer (multi.cpp)
  bool needs_window_tails() const;           // transforming store with 2..4 byte patterns (SURVEY H6, transform.cu)
  void *ghost_image() const;                 // device image of the reference's scratch buffer (kWindowBytes + 1 bytes) or nullptr
  void *stream() const;                      // the matcher's cudaStream_t
  void *gather_buffer(size_t bytes, size_t *cap = nullptr); // device memory for gathered records (kept until a larger request); *cap = its size
  int sync();                                // waits for stream()

  const olm_cuda_timing_t &timing() const;
  void collect_stats(omega_match_stats_t *accum); // adds the counters of the last call
  // While on, every call also runs stats_kernel (stats.cuh) so that collect_stats() reports the
  // reference's counters exactly; off (default): the scan's own counters, no extra kernel.
  void set_exact_stats(bool on);
  // host threads that stage PAGEABLE haystacks through pinned memory (omega_matcher_set_num_threads)
  void set_host_threads(int n);
  // While on, every call writes the id of each final record's pattern into its pad word
  // (pattern_ids.cuh); off (default): the pad stays 0.  The first switch on uploads the catalogue's
  // lookup table (`cat`, the catalogue of this engine's store; not needed to switch off).
  int set_pattern_ids(bool on, const PatternCatalog *cat);
  bool pattern_ids() const;
  // Uploads the catalogue's lookup table once (set_pattern_ids does when switching on; the counts
  // need it without switching ids on).  0 when it is there already.
  int load_pattern_tables(const PatternCatalog *cat);
  uint64_t pattern_count() const; // of the loaded tables

  // Pattern counts (include/olm_b200.h): counts[id] += the final records of pattern id, *total = their
  // number; the records stay on the device.  Host counts: one device scratch array per call, copied
  // back once.  count_records reads ids from the records' pads (-1 for an id out of range).
  int count_host(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t *counts, uint64_t *total);
  int count_shard_host(const uint8_t *host_slice, const ScanRange &range, const MatchFlags &f, uint64_t *counts,
                       uint64_t *total);
  int count_records(const void *dev_records, uint64_t count, void *dev_counts);
  int count_records_to_host(const void *dev_records, uint64_t count, uint64_t *counts); // counts[id] += ...

  // Lines (include/olm_b200.h "lines", lines.cuh).  newline_facts: the facts of the device bytes
  // [0, len); the tile scan it leaves serves a following line_positions(..., tiles_ready = true) on the
  // same bytes.  line_positions: one LinePos per device record (offsets in [bytes_begin, bytes_begin +
  // len), dev_bytes the byte at bytes_begin).  matching_lines: run-length by line into a matcher-owned
  // device array.  Each adds its time to timing().total_ms.
  int newline_facts(const void *dev_bytes, uint64_t len, olm_newline_facts_t *out);
  int line_positions(const void *dev_records, uint64_t count, const void *dev_bytes, uint64_t bytes_begin, uint64_t len,
                     const olm_line_origin_t &origin, void *dev_positions, bool tiles_ready = false);
  int matching_lines(const void *dev_positions, uint64_t count, void **dev_lines, uint64_t *n_lines);
  // Host haystack: the records of match_host and their positions, or (lines_only) only the matching
  // lines; the arrays are host_result_alloc'ed.  One GPU, or OLM_HOST_SPAN_BYTES spans (host_spans).
  int lines_host(const uint8_t *haystack, size_t n, const MatchFlags &f, bool lines_only, LinesResult *out);
  // device records + positions -> host arrays, or (lines_only) their matching lines
  int lines_to_host(const void *dev_records, const void *dev_positions, uint64_t count, bool lines_only,
                    LinesResult *out);
  // Streams: one push of `n` bytes (host or device memory) -> the records it settles, on the device
  // (valid until the next call), or with `counts`: counts[id] += the records of pattern id (the tables
  // loaded).  The piece is not referenced after the call.  stream_release frees the carried bytes.
  int stream_push(StreamState &s, const void *bytes, size_t n, bool on_device, bool last, olm_cuda_results_t *out,
                  uint64_t *counts = nullptr);
  void stream_release(StreamState &s);

  const void *resident_haystack() const;           // the device copy of the last host haystack or slice
  void *positions_buffer(size_t bytes, int which); // device buffers for positions: 0 = a call's, 1 = gathered
  int copy_to_host(void *host_dst, const void *dev_src, size_t bytes); // asynchronous, on stream()

private:
  Engine() = default;
  // (dst_off: where the bytes go in the haystack buffer, which may be reallocated to dst_off + n bytes)
  int stage_host(const uint8_t *src, size_t n, size_t dst_off = 0);
  int stage_pageable(const uint8_t *src, size_t n, uint64_t nseg, size_t dst_off);
  int finish_staging();
  // step(span, its device records, several spans)
  using SpanStep = std::function<int(const Shard &, const olm_cuda_results_t &, bool)>;
  int host_spans(const uint8_t *haystack, size_t n, const MatchFlags &f, void *dev_counts, const SpanStep &step);
  unsigned long long *zeroed_counts();
  int add_counts_to_host(uint64_t *counts);
  EngineImpl *impl_ = nullptr;
};

// Pattern ids on for `engines` (their tables loaded) while the guard lives, for a call that needs ids in
// the pads whatever the caller chose; every engine's own setting comes back on every exit path.
class PatternIdsOn {
public:
  explicit PatternIdsOn(const std::vector<Engine *> &engines, bool on = true) {
    if (!on) return;
    for (Engine *e : engines) {
      saved_.emplace_back(e, e->pattern_ids());
      e->set_pattern_ids(true, nullptr);
    }
  }
  ~PatternIdsOn() {
    for (auto &s : saved_) s.first->set_pattern_ids(s.second, nullptr);
  }
  PatternIdsOn(const PatternIdsOn &) = delete;
  PatternIdsOn &operator=(const PatternIdsOn &) = delete;

private:
  std::vector<std::pair<Engine *, bool>> saved_;
};

} // namespace olm
