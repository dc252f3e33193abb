// api.cpp -- the C ABI of libomega_match.so (declarations and reference citations:
// include/olm_b200.h).  Thin: argument checking, file handling, and calls into Engine.
#include <unistd.h>

#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <memory>
#include <string>
#include <thread>

#include "../../include/olm_b200.h"
#include "engine.h"
#include "host_util.h"
#include "lines.cuh"
#include "multi.h"
#include "store.h"

#ifndef OLM_B200_VERSION
#define OLM_B200_VERSION "0.1.0"
#endif

struct olm_cuda_comm {
  olm::Comm *comm = nullptr;
};

struct omega_list_matcher_struct {
  olm::Engine *engine = nullptr;          // the (first) GPU's engine
  olm::MultiMatcher *multi = nullptr;     // several GPUs in this process (owns `engine` then)
  uint8_t *file = nullptr; // mapped store
  size_t file_size = 0;
  char *temp_path = nullptr; // set when the store was compiled on the fly (matcher.c:458-481)
  omega_match_stats_t *stats = nullptr;
  bool exact_stats = false; // olm_cuda_set_exact_stats / OLM_EXACT_STATS=1
  int threads = 1;
  int chunk = 4096;
  // pattern ids: the store's catalogue, built on first use (olm_pattern_count & co. are const)
  mutable std::unique_ptr<olm::PatternCatalog> catalog;
  mutable std::string catalog_err;
};

static_assert(sizeof(olm_line_pos_t) == sizeof(olm::LinePos) && sizeof(olm_line_t) == sizeof(olm::LineEntry) &&
                  sizeof(olm_line_pos_t) == sizeof(omega_match_result_t),
              "the line structs are lines.cuh's, and a position is as large as a record");
static_assert(sizeof(olm_result_with_id_t) == sizeof(omega_match_result_t) &&
                  offsetof(olm_result_with_id_t, offset) == offsetof(omega_match_result_t, offset) &&
                  offsetof(olm_result_with_id_t, len) == offsetof(omega_match_result_t, len) &&
                  offsetof(olm_result_with_id_t, pattern_id) == offsetof(omega_match_result_t, len) + 4 &&
                  offsetof(olm_result_with_id_t, match) == offsetof(omega_match_result_t, match),
              "olm_result_with_id_t is omega_match_result_t with its pad named");

namespace {

int g_default_device = -1;

int default_device() {
  if (g_default_device >= 0) return g_default_device;
  if (const char *e = std::getenv("OLM_CUDA_DEVICE")) return std::atoi(e);
  return 0;
}

int max_host_threads() {
  const unsigned n = std::thread::hardware_concurrency();
  return n ? int(n) : 1;
}

// 1234567 -> "1,234,567" (what the reference's header line prints, util.h:28-58)
std::string with_commas(uint64_t v) {
  std::string s = std::to_string(v);
  for (int i = int(s.size()) - 3; i > 0; i -= 3) s.insert(size_t(i), ",");
  return s;
}

olm::MatchFlags to_flags(int no_overlap, int longest_only, int word_boundary, int word_prefix, int word_suffix,
                         int line_start, int line_end) {
  olm::MatchFlags f;
  f.no_overlap = no_overlap != 0;
  f.longest_only = longest_only != 0;
  f.word_boundary = word_boundary != 0;
  f.word_prefix = word_prefix != 0;
  f.word_suffix = word_suffix != 0;
  f.line_start = line_start != 0;
  f.line_end = line_end != 0;
  return f;
}

} // namespace

extern "C" {

const char *omega_match_version(void) { return OLM_B200_VERSION; }

namespace {
// devices == nullptr: the default device, or the GPUs listed in OLM_CUDA_DEVICES
omega_list_matcher_t *create_on(const char *path, int case_insensitive, int ignore_punctuation, int elide_whitespace,
                                omega_match_pattern_store_stats_t *stats, const std::vector<int> *devices);
} // namespace

omega_list_matcher_t *omega_list_matcher_create(const char *path, int case_insensitive, int ignore_punctuation,
                                                int elide_whitespace, omega_match_pattern_store_stats_t *stats) {
  return create_on(path, case_insensitive, ignore_punctuation, elide_whitespace, stats, nullptr);
}

omega_list_matcher_t *olm_cuda_matcher_create_multi(const char *path, const int *devices, int n_devices) {
  if (!path || !devices || n_devices < 1) return nullptr;
  std::vector<int> d(devices, devices + n_devices);
  return create_on(path, 0, 0, 0, nullptr, &d);
}

namespace {
omega_list_matcher_t *create_on(const char *path, int case_insensitive, int ignore_punctuation, int elide_whitespace,
                                omega_match_pattern_store_stats_t *stats, const std::vector<int> *devices) {
  if (!path) return nullptr;
  std::string load = path;
  char *temp_path = nullptr;
  if (!omega_list_matcher_is_compiled(path)) {
    char tmp[] = "/tmp/oa_matcher_XXXXXX";
    const int fd = mkstemp(tmp);
    if (fd < 0) {
      std::perror("mkstemp");
      return nullptr;
    }
    close(fd);
    if (omega_list_matcher_compile_patterns_filename(tmp, path, case_insensitive, ignore_punctuation,
                                                     elide_whitespace, stats) != 0) {
      unlink(tmp);
      return nullptr;
    }
    temp_path = strdup(tmp);
    load = tmp;
  }
  auto *m = new omega_list_matcher_struct();
  m->temp_path = temp_path;
  m->file = olm::map_whole_file(load.c_str(), &m->file_size, false);
  std::string err = "cannot map file";
  std::vector<int> devs;
  if (devices) {
    devs = *devices;
  } else if (const char *spec = std::getenv("OLM_CUDA_DEVICES")) {
    devs = olm::parse_device_list(spec, olm_cuda_device_count());
    if (devs.empty() && *spec) err = "OLM_CUDA_DEVICES names no usable GPU";
  }
  try { // no exception crosses the C ABI: a store that asks for absurd allocations is a bad file
    if (m->file && devs.size() > 1) {
      m->multi = olm::MultiMatcher::create(m->file, m->file_size, devs, &err);
      if (m->multi) m->engine = m->multi->first();
    } else if (m->file && !(devices == nullptr && std::getenv("OLM_CUDA_DEVICES") && *std::getenv("OLM_CUDA_DEVICES") && devs.empty())) {
      m->engine = olm::Engine::create(m->file, m->file_size, devs.size() == 1 ? devs[0] : default_device(), &err);
    }
  } catch (const std::exception &ex) {
    m->engine = nullptr;
    err = std::string("malformed store (") + ex.what() + ")";
  }
  if (!m->engine) {
    std::fprintf(stderr, "libomega_match(b200): cannot create matcher from %s: %s\n", path, err.c_str());
    omega_list_matcher_destroy(m);
    return nullptr;
  }
  omega_matcher_set_num_threads(m, 0); // matcher.c:509-511
  omega_matcher_set_chunk_size(m, 0);
  return m;
}

// the matcher's catalogue, built when first asked for; nullptr (and a message on stderr) for a
// store the catalogue rejects
const olm::PatternCatalog *catalog_of(const omega_list_matcher_t *m) {
  if (!m || !m->file) return nullptr;
  if (!m->catalog && m->catalog_err.empty()) {
    olm::StoreView v;
    std::string err = olm::parse_store(m->file, m->file_size, &v);
    auto c = std::make_unique<olm::PatternCatalog>();
    try {
      if (err.empty()) err = olm::build_catalog(v, c.get());
    } catch (const std::exception &ex) {
      err = std::string("malformed store (") + ex.what() + ")";
    }
    if (err.empty()) m->catalog = std::move(c);
    else m->catalog_err = err;
  }
  if (!m->catalog) std::fprintf(stderr, "libomega_match(b200): no pattern catalogue: %s\n", m->catalog_err.c_str());
  return m->catalog.get();
}

// the device haystack [0, n) at `dev` as one range
olm::ScanRange whole_haystack(const omega_list_matcher_t *m, const void *dev, uint64_t n, const void *match_ptr_base) {
  const olm::Header &h = m->engine->header();
  return olm::scan_range(olm::shard_of(0, n, n, h.largest, h.flags & olm::kFlagAnyTransform), n,
                         reinterpret_cast<uint64_t>(match_ptr_base), dev);
}
} // namespace

omega_list_matcher_t *omega_list_matcher_create_from_buffer(const char *compiled_file, const uint8_t *patterns_buffer,
                                                            uint64_t patterns_buffer_size, int case_insensitive,
                                                            int ignore_punctuation, int elide_whitespace,
                                                            omega_match_pattern_store_stats_t *stats) {
  if (!patterns_buffer || patterns_buffer_size == 0) return nullptr;
  if (omega_list_matcher_compile_patterns(compiled_file, patterns_buffer, patterns_buffer_size, case_insensitive,
                                          ignore_punctuation, elide_whitespace, stats) != 0)
    return nullptr;
  return omega_list_matcher_create(compiled_file, case_insensitive, ignore_punctuation, elide_whitespace, stats);
}

int omega_list_matcher_add_stats(omega_list_matcher_t *m, omega_match_stats_t *stats) {
  if (!m || !stats) return -1;
  m->stats = stats;
  const char *ex = std::getenv("OLM_EXACT_STATS");
  if (ex && ex[0] == '1') m->exact_stats = true;
  if (m->multi) m->multi->set_exact_stats(m->exact_stats);
  else m->engine->set_exact_stats(m->exact_stats);
  return 0;
}

int omega_list_matcher_destroy(omega_list_matcher_t *m) {
  if (!m) return -1;
  if (m->multi) delete m->multi; // (owns the engines)
  else delete m->engine;
  if (m->file) olm::unmap(m->file, m->file_size);
  if (m->temp_path) {
    unlink(m->temp_path);
    std::free(m->temp_path);
  }
  delete m;
  return 0;
}

int omega_list_matcher_emit_header_info(const omega_list_matcher_t *m, FILE *fp) {
  if (!m || !m->engine || !fp) return -1;
  const olm::Header &h = m->engine->header();
  std::fprintf(fp,
               "Header v%d stats: total_patterns=%s, smallest_pattern_length=%s, largest_pattern_length=%s,"
               " case_insensitive_support=%s, string_store_size=%s, bloom_filter_size=%s, num_occupied_buckets=%s,"
               " table_size=%s, min_bucket_size=%s, max_bucket_size=%s, load_factor=%.2f, avg_bucket_size=%.2f\n",
               int(h.version), with_commas(h.stored_patterns).c_str(), with_commas(h.smallest).c_str(),
               with_commas(h.largest).c_str(), (h.flags & olm::kFlagIgnoreCase) ? "yes" : "no",
               with_commas(h.store_bytes).c_str(), with_commas(h.bloom_bytes).c_str(),
               with_commas(h.occupied).c_str(), with_commas(h.table_size).c_str(), with_commas(h.min_bucket).c_str(),
               with_commas(h.max_bucket).c_str(), h.load_factor, h.avg_bucket);
  return 0;
}

omega_match_results_t *omega_list_matcher_match(const omega_list_matcher_t *m, const uint8_t *haystack,
                                                size_t haystack_size, int no_overlap, int longest_only,
                                                int word_boundary, int word_prefix, int word_suffix, int line_start,
                                                int line_end) {
  if (!m || !m->engine) return nullptr;
  const olm::MatchFlags f = to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end);
  if (m->multi) { // byte-range shards over the matcher's GPUs (multi.cpp)
    omega_match_results_t *r = m->multi->match_host(haystack, haystack_size, f);
    if (r && m->stats) m->multi->collect_stats(m->stats);
    return r;
  }
  omega_match_results_t *r = m->engine->match_host(haystack, haystack_size, f);
  if (r && m->stats) m->engine->collect_stats(m->stats);
  return r;
}

void omega_match_results_destroy(omega_match_results_t *results) {
  if (!results) return;
  olm::host_result_free(results->matches);
  results->matches = nullptr;
  results->count = 0;
  std::free(results);
}

int omega_matcher_set_num_threads(omega_list_matcher_t *m, int threads) {
  if (!m) return -1;
  const int mx = max_host_threads();
  if (threads == 0) threads = mx;
  else if (threads < 0 || threads > mx) return -1;
  m->threads = threads;
  if (m->engine && !m->multi) m->engine->set_host_threads(threads); // staging of pageable haystacks (engine.cu Stager)
  return 0;
}
int omega_matcher_get_num_threads(const omega_list_matcher_t *m) { return m ? m->threads : -1; }

int omega_matcher_set_chunk_size(omega_list_matcher_t *m, int chunk) {
  if (!m) return -1;
  if (chunk == 0) chunk = 4096;
  else if (chunk < 1) return -1;
  else if (chunk & (chunk - 1)) chunk = int(olm::next_pow2_u32(uint32_t(chunk)));
  m->chunk = chunk;
  return 0;
}
int omega_matcher_get_chunk_size(const omega_list_matcher_t *m) { return m ? m->chunk : -1; }

/* ------------------------------------------------------------------ B200 extensions */

int olm_cuda_set_default_device(int device) {
  if (device < 0) return -1;
  g_default_device = device;
  return 0;
}
int olm_cuda_matcher_device(const omega_list_matcher_t *m) { return (m && m->engine) ? m->engine->device() : -1; }

int olm_cuda_match_device(const omega_list_matcher_t *m, const void *dev_haystack, size_t n,
                          const void *match_ptr_base, int no_overlap, int longest_only, int word_boundary,
                          int word_prefix, int word_suffix, int line_start, int line_end, olm_cuda_results_t *out) {
  if (!m || !m->engine || !out) return -1;
  const int rc = m->engine->match_device(
      whole_haystack(m, dev_haystack, n, match_ptr_base), to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), out);
  if (rc == 0 && m->stats) m->engine->collect_stats(m->stats);
  return rc;
}

int olm_cuda_match_shard(const omega_list_matcher_t *m, const void *dev_slice, uint64_t slice_begin,
                         uint64_t slice_len, uint64_t own_begin, uint64_t own_end, uint64_t global_size,
                         const void *match_ptr_base, int longest_only, int word_boundary, int word_prefix,
                         int word_suffix, int line_start, int line_end, olm_cuda_results_t *out) {
  if (!m || !m->engine || !out) return -1;
  olm::ScanRange r;
  r.dev = dev_slice;
  r.slice_begin = slice_begin;
  r.slice_len = slice_len;
  r.own_begin = own_begin;
  r.own_end = own_end;
  r.global_size = global_size;
  r.match_ptr_base = reinterpret_cast<uint64_t>(match_ptr_base);
  const int rc = m->engine->match_device(
      r, to_flags(0, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), out);
  if (rc == 0 && m->stats) m->engine->collect_stats(m->stats);
  return rc;
}

int olm_cuda_match_shard_host(const omega_list_matcher_t *m, const void *host_slice, uint64_t slice_begin,
                              uint64_t slice_len, uint64_t own_begin, uint64_t own_end, uint64_t global_size,
                              const void *match_ptr_base, int longest_only, int word_boundary, int word_prefix,
                              int word_suffix, int line_start, int line_end, olm_cuda_results_t *out) {
  if (!m || !m->engine || !out || !host_slice) return -1;
  olm::ScanRange r;
  r.dev = nullptr;
  r.slice_begin = slice_begin;
  r.slice_len = slice_len;
  r.own_begin = own_begin;
  r.own_end = own_end;
  r.global_size = global_size;
  r.match_ptr_base = reinterpret_cast<uint64_t>(match_ptr_base);
  const int rc = m->engine->match_shard_host(
      static_cast<const uint8_t *>(host_slice), r,
      to_flags(0, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), out);
  if (rc == 0 && m->stats) m->engine->collect_stats(m->stats);
  return rc;
}

int64_t olm_cuda_no_overlap(const omega_list_matcher_t *m, void *dev_records, uint64_t count) {
  if (!m || !m->engine) return -1;
  return m->engine->no_overlap_inplace(dev_records, count);
}

int olm_cuda_format_records(const omega_list_matcher_t *m, const void *dev_records, uint64_t count,
                            const void *dev_haystack, uint64_t haystack_offset0, void **dev_text, uint64_t *text_bytes) {
  if (!m || !m->engine || !dev_text || !text_bytes || (count && (!dev_records || !dev_haystack))) return -1;
  return m->engine->format_records(dev_records, count, dev_haystack, haystack_offset0, dev_text, text_bytes);
}

int olm_cuda_sort_records(const omega_list_matcher_t *m, void *dev_records, uint64_t count) {
  if (!m || !m->engine) return -1;
  return m->engine->sort_records(dev_records, count);
}

int olm_cuda_set_exact_stats(omega_list_matcher_t *m, int on) {
  if (!m || !m->engine) return -1;
  m->exact_stats = on != 0;
  if (m->multi) m->multi->set_exact_stats(m->exact_stats && m->stats);
  else m->engine->set_exact_stats(m->exact_stats && m->stats); // the kernel runs only for an attached struct
  return 0;
}

int olm_cuda_set_pattern_ids(omega_list_matcher_t *m, int on) {
  if (!m || !m->engine) return -1;
  const olm::PatternCatalog *c = nullptr;
  if (on && !(c = catalog_of(m))) return -1;
  return m->multi ? m->multi->set_pattern_ids(on != 0, c) : m->engine->set_pattern_ids(on != 0, c);
}

int64_t olm_pattern_count(const omega_list_matcher_t *m) {
  const olm::PatternCatalog *c = catalog_of(m);
  return c ? int64_t(c->size()) : -1;
}

int olm_pattern_bytes(const omega_list_matcher_t *m, uint64_t id, const uint8_t **bytes, uint32_t *len) {
  if (!bytes || !len) return -1;
  const olm::PatternCatalog *c = catalog_of(m);
  if (!c || id >= c->size()) return -1;
  *bytes = c->bytes(id);
  *len = c->refs[id].y;
  return 0;
}

namespace {
// the catalogue's lookup table on every GPU of the matcher (ids stay as they are); -1 on a malformed store
int load_pattern_tables(const omega_list_matcher_t *m) {
  const olm::PatternCatalog *c = catalog_of(m);
  if (!c) return -1;
  return m->multi ? m->multi->load_pattern_tables(c) : m->engine->load_pattern_tables(c);
}
} // namespace

int olm_cuda_count_patterns(const omega_list_matcher_t *m, const uint8_t *haystack, size_t size, int no_overlap,
                            int longest_only, int word_boundary, int word_prefix, int word_suffix, int line_start,
                            int line_end, uint64_t *counts, uint64_t *total) {
  if (!m || !m->engine || !counts || !total || (!haystack && size) || load_pattern_tables(m)) return -1;
  const olm::MatchFlags f = to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end);
  if (m->multi) {
    const int rc = m->multi->count_host(haystack, size, f, counts, total);
    if (rc == 0 && m->stats) m->multi->collect_stats(m->stats);
    return rc;
  }
  const int rc = m->engine->count_host(haystack, size, f, counts, total);
  if (rc == 0 && m->stats) m->engine->collect_stats(m->stats);
  return rc;
}

int olm_cuda_count_patterns_device(const omega_list_matcher_t *m, const void *dev_haystack, size_t size,
                                   int no_overlap, int longest_only, int word_boundary, int word_prefix,
                                   int word_suffix, int line_start, int line_end, void *dev_counts, uint64_t *total) {
  if (!m || !m->engine || !dev_counts || !total || load_pattern_tables(m)) return -1;
  olm_cuda_results_t res;
  const int rc = m->engine->match_device(
      whole_haystack(m, dev_haystack, size, dev_haystack), to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), &res,
      dev_counts);
  if (rc != 0) return rc;
  if (m->stats) m->engine->collect_stats(m->stats);
  *total = res.count;
  return 0;
}

int olm_cuda_count_records(const omega_list_matcher_t *m, const void *dev_records, uint64_t count, void *dev_counts) {
  if (!m || !m->engine || !dev_counts || (count && !dev_records) || load_pattern_tables(m)) return -1;
  return m->engine->count_records(dev_records, count, dev_counts);
}

namespace {
// olm_cuda_match_lines / olm_cuda_matching_lines: one GPU, spans or several GPUs; nothing is kept on failure
int lines_call(const omega_list_matcher_t *m, const uint8_t *haystack, size_t size, const olm::MatchFlags &f,
               bool lines_only, olm::LinesResult *r) {
  const int rc = m->multi ? m->multi->lines_host(haystack, size, f, lines_only, r)
                          : m->engine->lines_host(haystack, size, f, lines_only, r);
  if (rc != 0) {
    omega_match_results_destroy(r->results);
    olm::host_result_free(r->positions);
    olm::host_result_free(r->lines);
    *r = olm::LinesResult{};
    return -1;
  }
  if (m->stats) {
    if (m->multi) m->multi->collect_stats(m->stats);
    else m->engine->collect_stats(m->stats);
  }
  return 0;
}
bool null_output(const char *what) {
  std::fprintf(stderr, "libomega_match(b200): %s: an output pointer is NULL\n", what);
  return true;
}
} // namespace

int olm_cuda_match_lines(const omega_list_matcher_t *m, const uint8_t *haystack, size_t size, int no_overlap,
                         int longest_only, int word_boundary, int word_prefix, int word_suffix, int line_start,
                         int line_end, omega_match_results_t **results, olm_line_pos_t **positions) {
  if (!m || !m->engine || (!haystack && size)) return -1;
  if ((!results || !positions) && null_output("olm_cuda_match_lines")) return -1;
  *results = nullptr;
  *positions = nullptr;
  olm::LinesResult r;
  if (lines_call(m, haystack, size,
                 to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), false,
                 &r) != 0)
    return -1;
  *results = r.results;
  *positions = r.positions;
  return 0;
}

int olm_cuda_matching_lines(const omega_list_matcher_t *m, const uint8_t *haystack, size_t size, int no_overlap,
                            int longest_only, int word_boundary, int word_prefix, int word_suffix, int line_start,
                            int line_end, olm_line_t **lines, uint64_t *n_lines, uint64_t *total_records) {
  if (!m || !m->engine || (!haystack && size)) return -1;
  if ((!lines || !n_lines || !total_records) && null_output("olm_cuda_matching_lines")) return -1;
  *lines = nullptr;
  *n_lines = *total_records = 0;
  olm::LinesResult r;
  if (lines_call(m, haystack, size,
                 to_flags(no_overlap, longest_only, word_boundary, word_prefix, word_suffix, line_start, line_end), true,
                 &r) != 0)
    return -1;
  *lines = r.lines;
  *n_lines = r.n_lines;
  *total_records = r.total;
  return 0;
}

void olm_lines_free(void *p) { olm::host_result_free(p); }

int olm_cuda_line_positions(const omega_list_matcher_t *m, const void *dev_records, uint64_t count, const void *dev_bytes,
                            uint64_t bytes_begin, uint64_t bytes_len, const olm_line_origin_t *origin,
                            void *dev_positions) {
  if (!m || !m->engine) return -1;
  if (count && (!dev_positions || !dev_records) && null_output("olm_cuda_line_positions")) return -1;
  if (!origin && bytes_begin != 0) {
    std::fprintf(stderr, "libomega_match(b200): olm_cuda_line_positions: without an origin the bytes start at offset 0\n");
    return -1;
  }
  const olm_line_origin_t o = origin ? *origin : olm_line_origin_t{0, 0, bytes_len};
  return m->engine->line_positions(dev_records, count, dev_bytes, bytes_begin, bytes_len, o, dev_positions);
}

int olm_cuda_newline_facts(const omega_list_matcher_t *m, const void *dev_bytes, uint64_t len, olm_newline_facts_t *out) {
  if (!m || !m->engine) return -1;
  if (!out && null_output("olm_cuda_newline_facts")) return -1;
  return m->engine->newline_facts(dev_bytes, len, out);
}

int olm_cuda_matching_lines_device(const omega_list_matcher_t *m, const void *dev_positions, uint64_t count,
                                   void **dev_lines, uint64_t *n_lines) {
  if (!m || !m->engine) return -1;
  if ((!dev_lines || !n_lines || (count && !dev_positions)) && null_output("olm_cuda_matching_lines_device")) return -1;
  return m->engine->matching_lines(dev_positions, count, dev_lines, n_lines);
}

int olm_cuda_last_timing(const omega_list_matcher_t *m, olm_cuda_timing_t *out) {
  if (!m || !m->engine || !out) return -1;
  *out = m->multi ? m->multi->timing() : m->engine->timing();
  return 0;
}

int olm_cuda_matcher_device_count(const omega_list_matcher_t *m) { return !m || !m->engine ? -1 : (m->multi ? m->multi->size() : 1); }

int olm_shard_plan(uint32_t largest_pattern, int windowed, uint64_t global_size, int world, int rank, olm_shard_t *out) {
  if (!out || world < 1 || rank < 0 || rank >= world) return -1;
  const olm::Shard s = olm::plan_shards(global_size, world, largest_pattern, windowed != 0)[size_t(rank)];
  out->own_begin = s.own_begin;
  out->own_end = s.own_end;
  out->slice_begin = s.slice_begin;
  out->slice_end = s.slice_end;
  return 0;
}

int olm_cuda_shard_plan(const omega_list_matcher_t *m, uint64_t global_size, int world, int rank, olm_shard_t *out) {
  if (!m || !m->engine) return -1;
  const olm::Header &h = m->engine->header();
  return olm_shard_plan(h.largest, (h.flags & olm::kFlagAnyTransform) != 0, global_size, world, rank, out);
}

int olm_cuda_comm_unique_id(void *id, size_t id_bytes) { return olm::comm_unique_id(id, id_bytes); }

olm_cuda_comm_t *olm_cuda_comm_create(const omega_list_matcher_t *m, const void *id, int rank, int world) {
  if (!m || !m->engine || m->multi) return nullptr;
  olm::Comm *c = olm::comm_create(m->engine, id, rank, world);
  if (!c) return nullptr;
  auto *h = new olm_cuda_comm();
  h->comm = c;
  return h;
}

int olm_cuda_comm_destroy(olm_cuda_comm_t *c) {
  if (!c) return -1;
  olm::comm_destroy(c->comm);
  delete c;
  return 0;
}

int olm_cuda_gather_records(olm_cuda_comm_t *c, const void *dev_records, uint64_t count, int root, int no_overlap,
                            olm_cuda_results_t *out) {
  if (!c || !c->comm) return -1;
  return olm::comm_gather(c->comm, dev_records, count, root, no_overlap != 0, out);
}

int olm_store_inspect(const char *compiled_file, olm_store_info_t *out) {
  if (!compiled_file || !out) return -1;
  size_t n = 0;
  uint8_t *f = olm::map_whole_file(compiled_file, &n, false);
  if (!f) return -1;
  olm::StoreView v;
  const std::string err = olm::parse_store(f, n, &v);
  int rc = -1;
  if (err.empty()) try {
    olm::StagedStore s;
    olm::FilterBudget b;
    const std::string e2 = olm::stage_store(v, b, &s);
    olm::StagedStats ss; // (and the tables of the exact statistics: everything create() stages)
    if (e2.empty() && olm::check_staged_store(v, s) == 0 && olm::stage_stats(v, &ss).empty()) {
      out->flags = v.hdr.flags;
      out->smallest = v.hdr.smallest;
      out->largest = v.hdr.largest;
      out->stored_patterns = v.hdr.stored_patterns;
      out->table_size = v.hdr.table_size;
      out->occupied_buckets = v.hdr.occupied;
      out->len1 = v.n1;
      out->len2 = v.n2;
      out->len3 = v.n3;
      out->len4 = v.n4;
      out->store_bytes = v.hdr.store_bytes;
      out->file_bytes = n;
      out->gram_keys = s.n_keys;
      out->key_bytes = s.params.key_bytes;
      out->key_buckets = s.params.key_mask + 1;
      out->g4_bits = s.params.g4_words * 32;
      out->class_run = s.params.cls.run;
      out->class_and_mask = s.params.cls.and_mask;
      out->class_ranges = s.params.cls.n_ranges;
      for (int i = 0; i < 2; ++i) {
        out->class_lo[i] = s.params.cls.lo[i];
        out->class_hi[i] = s.params.cls.hi[i];
      }
      rc = 0;
    } else {
      std::fprintf(stderr, "libomega_match(b200): %s: %s\n", compiled_file, e2.empty() ? "self check failed" : e2.c_str());
    }
  } catch (const std::exception &ex) {
    std::fprintf(stderr, "libomega_match(b200): %s: malformed store (%s)\n", compiled_file, ex.what());
    rc = -1;
  } else {
    std::fprintf(stderr, "libomega_match(b200): %s: %s\n", compiled_file, err.c_str());
  }
  olm::unmap(f, n);
  return rc;
}

} // extern "C"
