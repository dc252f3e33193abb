// multi.cpp -- several GPUs behind the C ABI (SURVEY 8e): byte-range shards, ownership rule, one
// gather.  Two ways to use more than one GPU, both without anything but C/C++, CUDA and NCCL:
//
//  (1) ONE PROCESS, N GPUS -- `MultiMatcher`.  A matcher created while OLM_CUDA_DEVICES lists
//      several GPUs (or through olm_cuda_matcher_create_multi) owns one engine per GPU.
//      omega_list_matcher_match(host haystack) then is: N host threads, each driving its GPU's
//      engine over its byte range (its own PCIe link: segmented H2D overlapped with the scan),
//      the per-GPU totals give every shard its place in the one result array, and the records are
//      copied out by all GPUs at once, each into its range of that (pinned) array.  `no_overlap`
//      -- the one filter that crosses shards -- first gathers the records on the first GPU over
//      NVLink (peer copies, final order = shard order) and runs once there.
//
//  (2) ONE PROCESS PER GPU -- `olm_cuda_comm_t`.  Every rank scans its shard
//      (olm_cuda_match_shard[_host]); olm_cuda_gather_records() exchanges the counts
//      (ncclAllGather of 8 bytes) and moves the records to the root's HBM with one group of
//      ncclSend / ncclRecv on the matcher's stream (NVLink / NVSwitch), then applies `no_overlap`
//      there.  NCCL is opened with dlopen() the first time a communicator is made, so the library
//      has no link-time dependency on it and single-GPU users never load it.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "multi.h"
#include "scan.cuh"

namespace olm {

namespace {

#define OLM_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      std::fprintf(stderr, "libomega_match(b200): %s failed: %s (%s:%d)\n", #expr,              \
                   cudaGetErrorString(_e), __FILE__, __LINE__);                                 \
      return -1;                                                                                \
    }                                                                                           \
  } while (0)

// ---- NCCL, loaded on demand ------------------------------------------------------------------
struct Nccl {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};

Nccl &nccl() {
  static Nccl n = [] {
    Nccl x;
    // a copy that is already in the process (e.g. the one a host framework brought along) wins
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
      x.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (x.lib) break;
    }
    if (!x.lib) {
      std::fprintf(stderr, "libomega_match(b200): cannot load NCCL (%s)\n", dlerror());
      return x;
    }
    auto sym = [&](const char *s) { return dlsym(x.lib, s); };
    x.GetUniqueId = reinterpret_cast<decltype(x.GetUniqueId)>(sym("ncclGetUniqueId"));
    x.CommInitRank = reinterpret_cast<decltype(x.CommInitRank)>(sym("ncclCommInitRank"));
    x.CommDestroy = reinterpret_cast<decltype(x.CommDestroy)>(sym("ncclCommDestroy"));
    x.AllGather = reinterpret_cast<decltype(x.AllGather)>(sym("ncclAllGather"));
    x.Send = reinterpret_cast<decltype(x.Send)>(sym("ncclSend"));
    x.Recv = reinterpret_cast<decltype(x.Recv)>(sym("ncclRecv"));
    x.GroupStart = reinterpret_cast<decltype(x.GroupStart)>(sym("ncclGroupStart"));
    x.GroupEnd = reinterpret_cast<decltype(x.GroupEnd)>(sym("ncclGroupEnd"));
    x.GetErrorString = reinterpret_cast<decltype(x.GetErrorString)>(sym("ncclGetErrorString"));
    x.ok = x.GetUniqueId && x.CommInitRank && x.CommDestroy && x.AllGather && x.Send && x.Recv && x.GroupStart &&
           x.GroupEnd && x.GetErrorString;
    if (!x.ok) std::fprintf(stderr, "libomega_match(b200): the NCCL library lacks a symbol this library needs\n");
    return x;
  }();
  return n;
}

#define OLM_NCCL(expr)                                                                          \
  do {                                                                                          \
    ncclResult_t _r = (expr);                                                                   \
    if (_r != ncclSuccess) {                                                                    \
      std::fprintf(stderr, "libomega_match(b200): %s failed: %s (%s:%d)\n", #expr,              \
                   nccl().GetErrorString(_r), __FILE__, __LINE__);                              \
      return -1;                                                                                \
    }                                                                                           \
  } while (0)

} // namespace

// ================================ (1) one process, N GPUs =========================================

std::vector<int> parse_device_list(const char *spec, int n_devices) {
  std::vector<int> out;
  if (!spec || !*spec) return out;
  std::string s(spec);
  if (s == "all") {
    for (int i = 0; i < n_devices; ++i) out.push_back(i);
    return out;
  }
  size_t at = 0;
  while (at < s.size()) {
    size_t end = s.find(',', at);
    if (end == std::string::npos) end = s.size();
    const std::string tok = s.substr(at, end - at);
    const size_t dash = tok.find('-');
    char *e1 = nullptr;
    if (dash == std::string::npos) {
      const long v = std::strtol(tok.c_str(), &e1, 10);
      if (tok.empty() || *e1 || v < 0 || v >= n_devices) return {};
      out.push_back((int)v);
    } else {
      const std::string a = tok.substr(0, dash), b = tok.substr(dash + 1);
      char *e2 = nullptr;
      const long lo = std::strtol(a.c_str(), &e1, 10), hi = std::strtol(b.c_str(), &e2, 10);
      if (a.empty() || b.empty() || *e1 || *e2 || lo < 0 || hi < lo || hi >= n_devices) return {};
      for (long v = lo; v <= hi; ++v) out.push_back((int)v);
    }
    at = end + 1;
  }
  std::sort(out.begin(), out.end());
  out.erase(std::unique(out.begin(), out.end()), out.end());
  return out;
}

std::vector<Shard> plan_shards(uint64_t size, int world, uint32_t largest_pattern, bool windowed) {
  std::vector<Shard> shards;
  const uint64_t unit = windowed ? kWindowBytes : 4096;
  const uint64_t units = (size + unit - 1) / unit;
  for (int r = 0; r < world; ++r) {
    Shard s;
    s.own_begin = std::min<uint64_t>(size, units * (uint64_t)r / (uint64_t)world * unit);
    s.own_end = r + 1 < world ? std::min<uint64_t>(size, units * (uint64_t)(r + 1) / (uint64_t)world * unit) : size;
    if (windowed) { // windows are independent: no halo at all
      s.slice_begin = s.own_begin;
      s.slice_end = s.own_end;
    } else { // 16 bytes in front (alignment + the previous byte), the longest pattern + 1 behind
      s.slice_begin = s.own_begin >= 16 ? s.own_begin - 16 : 0;
      s.slice_end = std::min<uint64_t>(size, s.own_end + largest_pattern + 1);
    }
    shards.push_back(s);
  }
  return shards;
}

MultiMatcher *MultiMatcher::create(const uint8_t *file, size_t size, const std::vector<int> &devices, std::string *err) {
  auto *m = new MultiMatcher();
  for (int d : devices) {
    Engine *e = Engine::create(file, size, d, err);
    if (!e) {
      delete m;
      return nullptr;
    }
    m->engines_.push_back(e);
  }
  // peer access towards the first GPU: the no_overlap gather copies over NVLink
  for (size_t g = 1; g < m->engines_.size(); ++g) {
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, m->engines_[g]->device(), m->engines_[0]->device()) == cudaSuccess && can) {
      cudaSetDevice(m->engines_[g]->device());
      if (cudaDeviceEnablePeerAccess(m->engines_[0]->device(), 0) != cudaSuccess) cudaGetLastError(); // (already enabled: fine)
      cudaSetDevice(m->engines_[0]->device());
      if (cudaDeviceEnablePeerAccess(m->engines_[g]->device(), 0) != cudaSuccess) cudaGetLastError();
    }
  }
  return m;
}

MultiMatcher::~MultiMatcher() {
  for (Engine *e : engines_) delete e;
}

omega_match_results_t *MultiMatcher::match_host(const uint8_t *haystack, size_t n, const MatchFlags &f) {
  const int N = (int)engines_.size();
  auto *results = static_cast<omega_match_results_t *>(std::malloc(sizeof(omega_match_results_t)));
  if (!results) return nullptr;
  results->count = 0;
  results->matches = static_cast<omega_match_result_t *>(std::malloc(sizeof(omega_match_result_t)));
  last_ = olm_cuda_timing_t{};
  scanned_.assign(N, false);
  if (n == 0 || !haystack) return results;
  auto bail = [&]() -> omega_match_results_t * {
    if (!pinned_result_release(results->matches)) std::free(results->matches);
    std::free(results);
    return nullptr;
  };
  // The stale-tail bytes of SURVEY H6 (2..4 byte patterns of a transforming store under word_boundary)
  // depend on the windows in front of a window -- which a shard does not see.  Such calls run on the
  // first GPU alone; all other calls shard, and afterwards every engine gets the scratch-buffer image
  // of the engine that scanned the haystack's last windows.
  const bool tails = engines_[0]->needs_window_tails();
  if (tails && f.word_boundary) {
    scanned_[0] = true;
    std::free(results->matches);
    std::free(results);
    omega_match_results_t *r = engines_[0]->match_host(haystack, n, f);
    last_ = engines_[0]->timing();
    if (r) sync_ghost(0);
    return r;
  }
  MatchFlags fs = f;
  fs.no_overlap = false; // crosses shards: once, on the gathered records
  std::vector<olm_cuda_results_t> res(N);
  for (int g = 0; g < N; ++g) res[g] = olm_cuda_results_t{0, nullptr, engines_[g]->device()};
  if (run_shards(haystack, n, [&](int g, const uint8_t *slice, const ScanRange &r) {
        return engines_[g]->match_shard_host(slice, r, fs, &res[g]);
      }) != 0)
    return bail();
  uint64_t total = 0;
  std::vector<uint64_t> off(N, 0);
  for (int g = 0; g < N; ++g) {
    off[g] = total;
    total += res[g].count;
  }
  if (total == 0) return results;

  Engine *E0 = engines_[0];
  const void *src0 = nullptr; // records that leave through the first GPU (no_overlap)
  uint64_t kept = total;
  if (f.no_overlap && total > 1) {
    const int64_t k = gather_no_overlap(res, total, &src0);
    if (k < 0) return bail();
    kept = (uint64_t)k;
  }
  std::free(results->matches);
  const size_t rbytes = std::max<uint64_t>(kept, 1) * sizeof(omega_match_result_t);
  results->matches = nullptr;
  if (rbytes >= kPinnedResultMin) results->matches = static_cast<omega_match_result_t *>(pinned_result_alloc(rbytes));
  if (!results->matches) results->matches = static_cast<omega_match_result_t *>(std::malloc(rbytes));
  if (!results->matches) {
    std::free(results);
    return nullptr;
  }
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  cudaSetDevice(E0->device());
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  cudaEventRecord(e0, static_cast<cudaStream_t>(E0->stream()));
  bool ok = true;
  if (src0) {
    ok = E0->records_to_host(results->matches, src0, kept) == 0;
  } else { // every GPU copies its records into its range of the one array, all links at once
    for (int g = 0; g < N && ok; ++g)
      if (res[g].count) ok = engines_[g]->records_to_host(results->matches + off[g], res[g].records, res[g].count) == 0;
  }
  for (int g = 0; g < N; ++g)
    if (engines_[g]->sync() != 0) ok = false;
  cudaSetDevice(E0->device());
  cudaEventRecord(e1, static_cast<cudaStream_t>(E0->stream()));
  cudaEventSynchronize(e1);
  cudaEventElapsedTime(&last_.d2h_ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (!ok) return bail();
  results->count = kept;
  return results;
}

// Runs scan(g, slice, range) for every GPU's shard of the host haystack, one host thread per GPU,
// then takes the call's timing from the engines and, for stores whose windows leave stale tails,
// gives every engine the scratch-buffer image of the engine that scanned the last windows.
int MultiMatcher::run_shards(const uint8_t *haystack, size_t n,
                             const std::function<int(int, const uint8_t *, const ScanRange &)> &scan) {
  const int N = (int)engines_.size();
  const Header &h = engines_[0]->header();
  const std::vector<Shard> plan = plan_shards(n, N, h.largest, h.flags & kFlagAnyTransform);
  std::vector<int> rc(N, 0);
  {
    std::vector<std::thread> th;
    for (int g = 0; g < N; ++g) {
      const Shard &s = plan[g];
      if (s.own_end <= s.own_begin) continue;
      scanned_[g] = true;
      th.emplace_back([&, g]() {
        const Shard &sh = plan[g];
        ScanRange r;
        r.slice_begin = sh.slice_begin;
        r.slice_len = sh.slice_end - sh.slice_begin;
        r.own_begin = sh.own_begin;
        r.own_end = sh.own_end;
        r.global_size = n;
        r.match_ptr_base = reinterpret_cast<uint64_t>(haystack);
        rc[g] = scan(g, haystack + sh.slice_begin, r);
      });
    }
    for (auto &t : th) t.join();
  }
  for (int g = 0; g < N; ++g) {
    if (rc[g] != 0) return -1;
    const olm_cuda_timing_t &t = engines_[g]->timing();
    last_.scan_ms = std::max(last_.scan_ms, t.scan_ms);
    last_.transform_ms = std::max(last_.transform_ms, t.transform_ms);
    last_.total_ms = std::max(last_.total_ms, t.total_ms);
    last_.h2d_ms = std::max(last_.h2d_ms, t.h2d_ms);
    last_.scan_launches += t.scan_launches;
    last_.kernel_launches += t.kernel_launches;
    last_.matches_before_filter += t.matches_before_filter;
  }
  if (engines_[0]->needs_window_tails()) {
    int last = 0;
    for (int g = 0; g < N; ++g)
      if (scanned_[g]) last = g;
    sync_ghost(last);
  }
  return 0;
}

// The shards' records (res, `total` in all) gathered on the first GPU over NVLink in shard order, and
// no_overlap applied there; returns the number kept (*dst: where they are), -1 on failure.
// With `positions` (per GPU, one per record) they travel with their records and are compacted with the
// same keep flags (*pos_dst: where they are).
int64_t MultiMatcher::gather_no_overlap(const std::vector<olm_cuda_results_t> &res, uint64_t total, const void **dst,
                                        const std::vector<void *> *positions, void **pos_dst) {
  Engine *E0 = engines_[0];
  void *buf = E0->gather_buffer(total * sizeof(Record));
  void *pbuf = positions ? E0->positions_buffer(total * sizeof(Record), 1) : nullptr;
  if (!buf || (positions && !pbuf)) return -1;
  cudaStream_t s0 = static_cast<cudaStream_t>(E0->stream());
  uint64_t off = 0;
  for (size_t g = 0; g < res.size(); off += res[g].count, ++g) {
    if (!res[g].count) continue;
    if (cudaMemcpyPeerAsync(static_cast<uint8_t *>(buf) + off * sizeof(Record), E0->device(), res[g].records,
                            engines_[g]->device(), res[g].count * sizeof(Record), s0) != cudaSuccess)
      return -1;
    if (positions && cudaMemcpyPeerAsync(static_cast<uint8_t *>(pbuf) + off * sizeof(olm_line_pos_t), E0->device(),
                                         (*positions)[g], engines_[g]->device(), res[g].count * sizeof(olm_line_pos_t),
                                         s0) != cudaSuccess)
      return -1;
  }
  if (cudaStreamSynchronize(s0) != cudaSuccess) return -1;
  const int64_t k = E0->no_overlap_inplace(buf, total, pbuf);
  last_.filter_ms = E0->timing().filter_ms;
  *dst = buf;
  if (pos_dst) *pos_dst = pbuf;
  return k;
}

int MultiMatcher::lines_host(const uint8_t *haystack, size_t n, const MatchFlags &f, bool lines_only, LinesResult *out) {
  const int N = (int)engines_.size();
  *out = LinesResult{};
  last_ = olm_cuda_timing_t{};
  scanned_.assign(N, false);
  if (n == 0 || !haystack) return engines_[0]->lines_host(haystack, n, f, lines_only, out);
  if (engines_[0]->needs_window_tails() && f.word_boundary) { // (as match_host)
    scanned_[0] = true;
    const int rc = engines_[0]->lines_host(haystack, n, f, lines_only, out);
    last_ = engines_[0]->timing();
    if (rc == 0) sync_ghost(0);
    return rc;
  }
  MatchFlags fs = f;
  fs.no_overlap = false;
  std::vector<olm_cuda_results_t> res(N);
  std::vector<olm_newline_facts_t> facts(N, olm_newline_facts_t{0, ~0ull, ~0ull});
  std::vector<uint64_t> own_begin(N, 0), own_end(N, 0), slice_begin(N, 0);
  for (int g = 0; g < N; ++g) res[g] = olm_cuda_results_t{0, nullptr, engines_[g]->device()};
  if (run_shards(haystack, n, [&](int g, const uint8_t *slice, const ScanRange &r) {
        own_begin[g] = r.own_begin;
        own_end[g] = r.own_end;
        slice_begin[g] = r.slice_begin;
        if (engines_[g]->match_shard_host(slice, r, fs, &res[g]) != 0) return -1;
        const uint8_t *own = static_cast<const uint8_t *>(engines_[g]->resident_haystack()) + (r.own_begin - r.slice_begin);
        return engines_[g]->newline_facts(own, r.own_end - r.own_begin, &facts[g]);
      }) != 0)
    return -1;
  // every GPU's origin from the facts of the ranges before and after it (shard order = byte order)
  std::vector<olm_line_origin_t> origin(N);
  uint64_t line = 0, begin = 0;
  for (int g = 0; g < N; ++g) {
    origin[g].line = line;
    origin[g].begin = begin;
    line += facts[g].newlines;
    if (facts[g].newlines) begin = own_begin[g] + facts[g].last + 1;
  }
  uint64_t next = n;
  for (int g = N - 1; g >= 0; --g) {
    origin[g].next_newline = next;
    if (facts[g].newlines) next = own_begin[g] + facts[g].first;
  }
  std::vector<void *> pos(N, nullptr);
  std::vector<int> rc(N, 0);
  {
    std::vector<std::thread> th;
    for (int g = 0; g < N; ++g) {
      if (!res[g].count) continue;
      th.emplace_back([&, g]() {
        Engine *e = engines_[g];
        const uint8_t *own = static_cast<const uint8_t *>(e->resident_haystack()) + (own_begin[g] - slice_begin[g]);
        pos[g] = e->positions_buffer(res[g].count * sizeof(olm_line_pos_t), 0);
        rc[g] = !pos[g] || e->line_positions(res[g].records, res[g].count, own, own_begin[g], own_end[g] - own_begin[g],
                                             origin[g], pos[g], true) != 0;
      });
    }
    for (auto &t : th) t.join();
  }
  uint64_t total = 0;
  std::vector<uint64_t> off(N, 0);
  for (int g = 0; g < N; ++g) {
    if (rc[g]) return -1;
    off[g] = total;
    total += res[g].count;
    last_.total_ms = std::max(last_.total_ms, engines_[g]->timing().total_ms);
  }
  Engine *E0 = engines_[0];
  if (f.no_overlap && total > 1) { // the records and their positions on the first GPU, filtered once
    const void *recs = nullptr;
    void *p0 = nullptr;
    const int64_t k = gather_no_overlap(res, total, &recs, &pos, &p0);
    if (k < 0) return -1;
    return E0->lines_to_host(recs, p0, uint64_t(k), lines_only, out);
  }
  out->total = total;
  if (lines_only) { // per GPU, then one entry for a line that continues on the next GPU
    std::vector<olm_line_t> all;
    for (int g = 0; g < N; ++g) {
      if (!res[g].count) continue;
      void *dl = nullptr;
      uint64_t m = 0;
      if (engines_[g]->matching_lines(pos[g], res[g].count, &dl, &m) != 0) return -1;
      const size_t at = all.size();
      all.resize(at + m);
      if (engines_[g]->copy_to_host(all.data() + at, dl, m * sizeof(olm_line_t)) != 0 || engines_[g]->sync() != 0) return -1;
      if (at && m && all[at - 1].line == all[at].line) {
        all[at - 1].records += all[at].records;
        all.erase(all.begin() + at);
      }
    }
    out->lines = static_cast<olm_line_t *>(host_result_alloc(all.size() * sizeof(olm_line_t)));
    if (!out->lines) return -1;
    if (!all.empty()) std::memcpy(out->lines, all.data(), all.size() * sizeof(olm_line_t));
    out->n_lines = all.size();
    return 0;
  }
  out->results = static_cast<omega_match_results_t *>(std::malloc(sizeof(omega_match_results_t)));
  if (!out->results) return -1;
  out->results->count = total;
  out->results->matches = static_cast<omega_match_result_t *>(host_result_alloc(total * sizeof(omega_match_result_t)));
  out->positions = static_cast<olm_line_pos_t *>(host_result_alloc(total * sizeof(olm_line_pos_t)));
  if (!out->results->matches || !out->positions) return -1;
  bool ok = true; // every GPU copies into its range of the arrays, all links at once
  for (int g = 0; g < N && ok; ++g)
    if (res[g].count)
      ok = engines_[g]->records_to_host(out->results->matches + off[g], res[g].records, res[g].count) == 0 &&
           engines_[g]->copy_to_host(out->positions + off[g], pos[g], res[g].count * sizeof(olm_line_pos_t)) == 0;
  for (int g = 0; g < N; ++g)
    if (engines_[g]->sync() != 0) ok = false;
  return ok ? 0 : -1;
}

// match_host() counting (include/olm_b200.h olm_cuda_count_patterns).  Without no_overlap every GPU
// counts its shard and the counts are summed on the host: no record moves.  With it the shards write
// ids, the gather and the filter run as in match_host, and the first GPU counts the pads.
int MultiMatcher::count_host(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t *counts, uint64_t *total) {
  const int N = (int)engines_.size();
  last_ = olm_cuda_timing_t{};
  scanned_.assign(N, false);
  *total = 0;
  if (n == 0 || !haystack) return 0;
  if (engines_[0]->needs_window_tails() && f.word_boundary) { // (as match_host)
    scanned_[0] = true;
    const int rc = engines_[0]->count_host(haystack, n, f, counts, total);
    last_ = engines_[0]->timing();
    if (rc == 0) sync_ghost(0);
    return rc;
  }
  MatchFlags fs = f;
  fs.no_overlap = false;
  const uint64_t P = engines_[0]->pattern_count();
  if (!f.no_overlap) {
    std::vector<std::vector<uint64_t>> part(N);
    std::vector<uint64_t> tot(N, 0);
    if (run_shards(haystack, n, [&](int g, const uint8_t *slice, const ScanRange &r) {
          part[g].assign(P, 0);
          return engines_[g]->count_shard_host(slice, r, fs, part[g].data(), &tot[g]);
        }) != 0)
      return -1;
    for (int g = 0; g < N; ++g) {
      if (!scanned_[g]) continue;
      for (uint64_t i = 0; i < P; ++i) counts[i] += part[g][i];
      *total += tot[g];
      last_.d2h_ms = std::max(last_.d2h_ms, engines_[g]->timing().d2h_ms);
    }
    return 0;
  }
  std::vector<olm_cuda_results_t> res(N);
  std::vector<bool> ids_were(N);
  for (int g = 0; g < N; ++g) {
    res[g] = olm_cuda_results_t{0, nullptr, engines_[g]->device()};
    ids_were[g] = engines_[g]->pattern_ids();
    engines_[g]->set_pattern_ids(true, nullptr); // (the tables are loaded)
  }
  int rc = run_shards(haystack, n, [&](int g, const uint8_t *slice, const ScanRange &r) {
    return engines_[g]->match_shard_host(slice, r, fs, &res[g]);
  });
  for (int g = 0; g < N; ++g) engines_[g]->set_pattern_ids(ids_were[g], nullptr);
  if (rc != 0) return -1;
  uint64_t all = 0;
  for (const olm_cuda_results_t &r : res) all += r.count;
  if (all > 1) {
    const void *recs = nullptr;
    const int64_t k = gather_no_overlap(res, all, &recs);
    if (k < 0 || engines_[0]->count_records_to_host(recs, uint64_t(k), counts) != 0) return -1;
    all = uint64_t(k);
    last_.d2h_ms = engines_[0]->timing().d2h_ms;
  } else {
    for (int g = 0; g < N; ++g) // (one record at most: nothing to filter)
      if (res[g].count && engines_[g]->count_records_to_host(res[g].records, res[g].count, counts) != 0) return -1;
  }
  *total = all;
  return 0;
}

// every engine's image of the reference's scratch buffer <- the one of engine `from`
void MultiMatcher::sync_ghost(int from) {
  Engine *src = engines_[size_t(from)];
  if (!src->ghost_image()) return;
  cudaStream_t st = static_cast<cudaStream_t>(src->stream());
  for (size_t g = 0; g < engines_.size(); ++g)
    if ((int)g != from && engines_[g]->ghost_image())
      cudaMemcpyPeerAsync(engines_[g]->ghost_image(), engines_[g]->device(), src->ghost_image(), src->device(),
                          size_t(kWindowBytes) + 1, st);
  cudaSetDevice(src->device());
  cudaStreamSynchronize(st);
}

void MultiMatcher::collect_stats(omega_match_stats_t *s) {
  for (size_t g = 0; g < engines_.size(); ++g)
    if (g < scanned_.size() && scanned_[g]) engines_[g]->collect_stats(s);
}
void MultiMatcher::set_exact_stats(bool on) {
  for (Engine *e : engines_) e->set_exact_stats(on);
}
int MultiMatcher::set_pattern_ids(bool on, const PatternCatalog *cat) {
  for (Engine *e : engines_)
    if (e->set_pattern_ids(on, cat) != 0) return -1;
  return 0;
}
int MultiMatcher::load_pattern_tables(const PatternCatalog *cat) {
  for (Engine *e : engines_)
    if (e->load_pattern_tables(cat) != 0) return -1;
  return 0;
}

// ================================ (2) one process per GPU =========================================

// Per-rank entry of the exchange that opens every gather: the rank's record count and -- meaningful
// for the root only -- where its gather buffer is, how large, which buffer the other ranks have mapped,
// and the buffer's IPC handle.
struct alignas(16) GatherHello {
  unsigned long long count;
  unsigned long long buf;      // root: its gather buffer as it is now (0 = none)
  unsigned long long cap;      // root: bytes of that buffer
  unsigned long long exported; // root: the buffer the handle below belongs to
  unsigned long long ok;       // this rank can use the window (0: it failed to map it once -> NCCL send/recv from now on)
  unsigned long long _pad;
  unsigned char handle[64];    // cudaIpcMemHandle_t of `exported`
};
static_assert(sizeof(GatherHello) == 112 && sizeof(cudaIpcMemHandle_t) == 64, "exchange layout");

struct Comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  Engine *engine = nullptr;
  GatherHello *d_hello = nullptr; // world entries
  std::vector<GatherHello> h_hello;
  // the root's gather buffer as a window the other ranks write their records into (CUDA IPC + NVLink)
  bool use_window = true;          // OLM_GATHER_WINDOW=0, or a rank that could not map it: NCCL send/recv instead
  unsigned long long exported = 0; // root: the buffer whose handle is current
  cudaIpcMemHandle_t handle{};     // root: that handle
  unsigned long long mapped = 0;   // other ranks: root buffer (its address there) that is mapped here ...
  void *window = nullptr;          // ... and where
};

Comm *comm_create(Engine *engine, const void *id, int rank, int world) {
  if (!engine || !id || world < 1 || rank < 0 || rank >= world || !nccl().ok) return nullptr;
  if (cudaSetDevice(engine->device()) != cudaSuccess) return nullptr;
  auto *c = new Comm();
  c->rank = rank;
  c->world = world;
  c->engine = engine;
  c->h_hello.assign(world, GatherHello{});
  if (const char *e = std::getenv("OLM_GATHER_WINDOW")) c->use_window = std::atoi(e) != 0;
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof uid);
  if (cudaMalloc(&c->d_hello, (sizeof(GatherHello) + 8) * world) != cudaSuccess ||
      nccl().CommInitRank(&c->comm, world, uid, rank) != ncclSuccess) {
    std::fprintf(stderr, "libomega_match(b200): cannot create the NCCL communicator (rank %d of %d)\n", rank, world);
    if (c->d_hello) cudaFree(c->d_hello);
    delete c;
    return nullptr;
  }
  return c;
}

void comm_destroy(Comm *c) {
  if (!c) return;
  cudaSetDevice(c->engine->device());
  if (c->window) cudaIpcCloseMemHandle(c->window);
  if (c->comm) nccl().CommDestroy(c->comm);
  if (c->d_hello) cudaFree(c->d_hello);
  delete c;
}

int comm_unique_id(void *id, size_t bytes) {
  if (!id || bytes < sizeof(ncclUniqueId) || !nccl().ok) return -1;
  ncclUniqueId uid;
  OLM_NCCL(nccl().GetUniqueId(&uid));
  std::memcpy(id, &uid, sizeof uid);
  return 0;
}

namespace {
// every rank contributes its entry of h_hello; afterwards all entries are on every rank's host
int exchange_hello(Comm *c, cudaStream_t st) {
  OLM_CUDA(cudaMemcpyAsync(c->d_hello + c->rank, &c->h_hello[c->rank], sizeof(GatherHello), cudaMemcpyHostToDevice, st));
  OLM_NCCL(nccl().AllGather(c->d_hello + c->rank, c->d_hello, sizeof(GatherHello), ncclUint8, c->comm, st));
  OLM_CUDA(cudaMemcpyAsync(c->h_hello.data(), c->d_hello, sizeof(GatherHello) * c->world, cudaMemcpyDeviceToHost, st));
  OLM_CUDA(cudaStreamSynchronize(st));
  return 0;
}
} // namespace

// Gather of the per-rank record arrays (each in final order, shards ordered by rank) on `root`.
// One exchange tells every rank all counts, hence where its records go.  Then
//   * window path (default): the root's gather buffer is mapped into the other ranks (CUDA IPC, set up
//     when the buffer is first made or grows) and every rank COPIES its records to their final place
//     over NVLink with its copy engines -- all ranks at once, no kernel on any SM, nothing staged; a
//     closing 8-byte collective on the same streams tells the root that all copies have landed;
//   * fallback (OLM_GATHER_WINDOW=0, or a rank that cannot map the window): one group of ncclSend /
//     ncclRecv (measured: ~290 GB/s into the root whatever the number of senders; the window path is
//     bound by the root's NVLink ingest).
int comm_gather(Comm *c, const void *dev_records, uint64_t count, int root, bool no_overlap, olm_cuda_results_t *out) {
  if (!c || !out || root < 0 || root >= c->world) return -1;
  Engine *E = c->engine;
  OLM_CUDA(cudaSetDevice(E->device()));
  cudaStream_t st = static_cast<cudaStream_t>(E->stream());
  out->count = 0;
  out->records = nullptr;
  out->device = E->device();
  const bool is_root = c->rank == root;

  GatherHello &me = c->h_hello[c->rank];
  me = GatherHello{};
  me.count = count;
  me.ok = c->use_window ? 1 : 0;
  if (is_root) {
    size_t cap_now = 0;
    void *cur = E->gather_buffer(0, &cap_now); // (the buffer as it is: nothing is allocated here)
    me.buf = reinterpret_cast<unsigned long long>(cur);
    me.cap = cap_now;
    me.exported = c->exported;
    std::memcpy(me.handle, &c->handle, sizeof c->handle);
  }
  if (exchange_hello(c, st)) return -1;
  uint64_t total = 0;
  std::vector<uint64_t> off(c->world, 0);
  bool window = true;
  for (int r = 0; r < c->world; ++r) {
    off[r] = total;
    total += c->h_hello[r].count;
    window = window && c->h_hello[r].ok != 0;
  }
  const uint64_t need = total * sizeof(Record);
  uint8_t *buf = nullptr; // root: the gather buffer

  if (window && total) {
    const GatherHello root_now = c->h_hello[root];
    // (Re)open the window when the root's buffer is too small or is not the one whose handle went round.
    if (need > root_now.cap || root_now.buf == 0 || root_now.buf != root_now.exported) {
      // the other ranks let go of the old mapping before the root frees the memory behind it
      if (c->window) { // (also a rank that is the root now and was not before)
        cudaIpcCloseMemHandle(c->window);
        c->window = nullptr;
        c->mapped = 0;
      }
      me = GatherHello{};
      me.ok = 1;
      if (exchange_hello(c, st)) return -1; // (barrier: every mapping is closed)
      me = GatherHello{};
      me.ok = 1;
      if (is_root) {
        size_t cap = 0;
        // (with room to grow; at least a few MiB, so that the allocation is one of its own: the handle
        // describes a whole allocation)
        void *p = E->gather_buffer(need + need / 4 + (size_t(4) << 20), &cap);
        if (p && cudaIpcGetMemHandle(&c->handle, p) == cudaSuccess) {
          c->exported = reinterpret_cast<unsigned long long>(p);
          me.buf = me.exported = c->exported;
          me.cap = cap;
          std::memcpy(me.handle, &c->handle, sizeof c->handle);
        } else {
          cudaGetLastError();
          me.ok = 0;
        }
      }
      if (exchange_hello(c, st)) return -1; // the new handle
      if (!is_root && c->h_hello[root].ok) {
        cudaIpcMemHandle_t h;
        std::memcpy(&h, c->h_hello[root].handle, sizeof h);
        if (cudaIpcOpenMemHandle(&c->window, h, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess) {
          c->mapped = c->h_hello[root].buf;
        } else {
          cudaGetLastError();
          c->window = nullptr;
          me.ok = 0;
        }
      }
      me.count = 0;
      if (exchange_hello(c, st)) return -1; // did everybody get it?
      for (int r = 0; r < c->world; ++r) window = window && c->h_hello[r].ok != 0;
      if (!window) {
        if (c->use_window && c->rank == 0)
          std::fprintf(stderr, "libomega_match(b200): the gather window could not be mapped on every rank; using ncclSend/ncclRecv\n");
        c->use_window = false;
        if (!is_root && c->window) {
          cudaIpcCloseMemHandle(c->window);
          c->window = nullptr;
          c->mapped = 0;
        }
      }
    }
  }

  if (window && total) {
    if (is_root) {
      buf = static_cast<uint8_t *>(E->gather_buffer(need, nullptr));
      if (!buf || reinterpret_cast<unsigned long long>(buf) != c->exported) return -1;
    }
    uint8_t *dst = is_root ? buf : static_cast<uint8_t *>(c->window);
    if (count)
      OLM_CUDA(cudaMemcpyAsync(dst + off[c->rank] * sizeof(Record), dev_records, count * sizeof(Record), cudaMemcpyDeviceToDevice, st));
    // every rank's copy precedes its part of this collective in stream order: when it completes on the
    // root, all records are in the root's memory
    uint8_t *sync = reinterpret_cast<uint8_t *>(c->d_hello + c->world); // world x 8 bytes behind the entries
    OLM_NCCL(nccl().AllGather(sync + 8 * c->rank, sync, 8, ncclUint8, c->comm, st));
    OLM_CUDA(cudaStreamSynchronize(st));
    if (!is_root) return 0;
  } else {
    if (!is_root) { // shards are ordered: the root lays the ranks' records out in rank order
      if (count) OLM_NCCL(nccl().Send(dev_records, count * sizeof(Record), ncclUint8, root, c->comm, st));
      OLM_CUDA(cudaStreamSynchronize(st));
      return 0;
    }
    if (total) {
      buf = static_cast<uint8_t *>(E->gather_buffer(need, nullptr));
      if (!buf) return -1;
      if (count)
        OLM_CUDA(cudaMemcpyAsync(buf + off[root] * sizeof(Record), dev_records, count * sizeof(Record), cudaMemcpyDeviceToDevice, st));
      OLM_NCCL(nccl().GroupStart());
      for (int r = 0; r < c->world; ++r)
        if (r != root && c->h_hello[r].count)
          OLM_NCCL(nccl().Recv(buf + off[r] * sizeof(Record), c->h_hello[r].count * sizeof(Record), ncclUint8, r, c->comm, st));
      OLM_NCCL(nccl().GroupEnd());
      OLM_CUDA(cudaStreamSynchronize(st));
    }
  }
  uint64_t kept = total;
  if (no_overlap && total > 1) {
    const int64_t k = E->no_overlap_inplace(buf, total);
    if (k < 0) return -1;
    kept = (uint64_t)k;
  }
  out->count = kept;
  out->records = buf;
  return 0;
}

} // namespace olm
