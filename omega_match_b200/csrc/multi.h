// multi.h -- several GPUs behind the C ABI: one process driving N GPUs (MultiMatcher) and the
// NCCL gather of a one-process-per-GPU job (Comm).  See multi.cpp.
#pragma once
#include <cstddef>
#include <cstdint>
#include <functional>
#include <string>
#include <vector>

#include "engine.h"

namespace olm {

// "0,1,2", "0-3", "all" -> device indices (sorted, unique); empty on a malformed list or an index
// that does not exist
std::vector<int> parse_device_list(const char *spec, int n_devices);

// Byte-range shards of one haystack (SURVEY 8e, shard_of): rank r owns the r-th of `world` runs of
// 4 KiB units (stores with a transform flag: 4 MiB windows).
std::vector<Shard> plan_shards(uint64_t size, int world, uint32_t largest_pattern, bool windowed);

class MultiMatcher {
public:
  static MultiMatcher *create(const uint8_t *file, size_t size, const std::vector<int> &devices, std::string *err);
  ~MultiMatcher();
  omega_match_results_t *match_host(const uint8_t *haystack, size_t n, const MatchFlags &f);
  // Engine::count_host over the GPUs (the pattern tables loaded on every engine)
  int count_host(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t *counts, uint64_t *total);
  // Engine::lines_host over the GPUs: every GPU takes the newline facts of its own range, the host
  // combines them into each GPU's origin, and every GPU resolves its records with it
  int lines_host(const uint8_t *haystack, size_t n, const MatchFlags &f, bool lines_only, LinesResult *out);
  void collect_stats(omega_match_stats_t *accum);
  void set_exact_stats(bool on);
  int set_pattern_ids(bool on, const PatternCatalog *cat); // every engine (Engine::set_pattern_ids)
  int load_pattern_tables(const PatternCatalog *cat);      // every engine
  const olm_cuda_timing_t &timing() const { return last_; }
  Engine *first() const { return engines_.front(); }
  int size() const { return (int)engines_.size(); }

private:
  bool first_alone(const uint8_t *haystack, size_t n, const MatchFlags &f, const std::function<int()> &call, int *rc);
  void sync_ghost(int from);
  int run_shards(const uint8_t *haystack, size_t n, const std::function<int(int, const uint8_t *, const ScanRange &)> &scan);
  int64_t gather_no_overlap(const std::vector<olm_cuda_results_t> &res, uint64_t total, const void **dst,
                            const std::vector<void *> *positions = nullptr, void **pos_dst = nullptr);
  int copy_out(const std::vector<olm_cuda_results_t> &res, omega_match_result_t *dst,
               const std::vector<void *> *positions = nullptr, olm_line_pos_t *pos_dst = nullptr);
  std::vector<Engine *> engines_;
  std::vector<bool> scanned_; // engines that took part in the last call
  olm_cuda_timing_t last_{};
};

struct Comm;
int comm_unique_id(void *id, size_t bytes);
Comm *comm_create(Engine *engine, const void *id, int rank, int world);
void comm_destroy(Comm *c);
int comm_gather(Comm *c, const void *dev_records, uint64_t count, int root, bool no_overlap, olm_cuda_results_t *out);

} // namespace olm
