// engine.h -- one matcher on one GPU: the uploaded store, work buffers, and the sequence of
// kernels that make up a match call.  Plain C++ interface; api.cpp puts the C ABI on top.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>

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
};

// Large result arrays of the host API (cuda_util.cu): pinned, recycled across calls.
void *pinned_result_alloc(size_t bytes);
bool pinned_result_release(void *p); // false: not one of ours (plain malloc)
constexpr size_t kPinnedResultMin = size_t(1) << 20;

struct EngineImpl;

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
  // Host input/output: H2D, match_device, D2H into a malloc'ed array.
  omega_match_results_t *match_host(const uint8_t *haystack, size_t n, const MatchFlags &f);
  // A byte range (range.dev is ignored) whose slice lies in HOST memory: segmented H2D overlapped
  // with the scan, device-resident records.
  int match_shard_host(const uint8_t *host_slice, const ScanRange &range, const MatchFlags &f, olm_cuda_results_t *out,
                       void *dev_counts = nullptr);

  // "offset:bytes\n" for every record (the CLI's listing, main.c:89-133) as one device text buffer;
  // dev_haystack = device address of the haystack byte with offset `offset0`
  int format_records(const void *dev_records, uint64_t count, const void *dev_haystack, uint64_t offset0,
                     void **dev_text, uint64_t *text_bytes);
  int64_t no_overlap_inplace(void *dev_records, uint64_t count);
  int sort_records(void *dev_records, uint64_t count);

  // for the multi-GPU layer (multi.cpp)
  bool needs_window_tails() const;           // transforming store with 2..4 byte patterns (SURVEY H6, transform.cu)
  void *ghost_image() const;                 // device image of the reference's scratch buffer (kWindowBytes + 1 bytes) or nullptr
  void *stream() const;                      // the matcher's cudaStream_t
  void *gather_buffer(size_t bytes, size_t *cap = nullptr); // device memory for gathered records (kept until a larger request); *cap = its size
  int records_to_host(void *host_dst, const void *dev_records, uint64_t count); // asynchronous, on stream()
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

private:
  Engine() = default;
  int stage_host(const uint8_t *src, size_t n);
  int stage_pageable(const uint8_t *src, size_t n, uint64_t nseg);
  int finish_staging();
  omega_match_results_t *match_host_spans(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t span);
  int count_host_spans(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t span, uint64_t *counts,
                       uint64_t *total);
  unsigned long long *zeroed_counts();
  int add_counts_to_host(uint64_t *counts);
  EngineImpl *impl_ = nullptr;
};

} // namespace olm
