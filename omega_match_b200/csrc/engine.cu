// engine.cu -- sequencing of one match call on one GPU.
//
//   no transform flag in the store (matcher.c:939-943):
//       scan -> prefix -> place -> redo over the owned byte range (one launch group; the host
//       path runs one group per 256 MiB segment while later segments are still being copied)
//       -> (no_overlap filter)
//   transform flag (matcher.c:945-1018): for every batch of <= kBatchWindows source windows
//       (window descriptors, only where a launch needs them: transform.cu) -> scan -> prefix ->
//       place -> redo over the SOURCE bytes of the windows -- the scan normalises chunk by chunk
//       in shared memory and reports source coordinates; the running match total carries over
//       from batch to batch, so the records of all windows come out in one ordered array
//       -> (no_overlap filter)
//
// place_kernel / redo_kernel write final records; the only host synchronisation of a call is the
// read-back of the record count (needed to size the D2H copy / to detect a too small result or
// temp buffer, in which case the buffers are grown to the exact size and the call repeated).
#include "engine.h"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "filters.cuh"
#include "format.cuh"
#include "lines.cuh"
#include "pattern_ids.cuh"
#include "scan.cuh"
#include "stats.cuh"
#include "transform.cuh"

namespace olm {

namespace {

constexpr uint32_t kBatchWindows = 64;                 // stores with a transform flag: 256 MiB of source per launch group
constexpr uint32_t kTilesPerWindow = kWindowBytes / kTileBytes;
constexpr uint32_t kMaxBatches = 1u << 16;
constexpr uint64_t kSegmentBytes = uint64_t(kBatchWindows) * kWindowBytes; // host path: H2D/scan pipeline unit (256 MiB)
constexpr uint64_t kPipelineMin = 2 * kSegmentBytes;                       // shorter haystacks: one copy, one scan

#define OLM_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      std::fprintf(stderr, "libomega_match(b200): %s failed: %s (%s:%d)\n", #expr,              \
                   cudaGetErrorString(_e), __FILE__, __LINE__);                                 \
      return -1;                                                                                \
    }                                                                                           \
  } while (0)

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  int ensure(size_t n, bool keep = false) {
    if (n <= cap) return 0;
    size_t want = (n + (size_t(1) << 20)) & ~((size_t(1) << 20) - 1);
    void *q = nullptr;
    OLM_CUDA(cudaMalloc(&q, want));
    if (keep && p && cap) OLM_CUDA(cudaMemcpy(q, p, cap, cudaMemcpyDeviceToDevice));
    if (p) cudaFree(p);
    p = q;
    cap = want;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

template <typename T>
int upload(DevBuf &b, const std::vector<T> &v, const T **out) {
  const size_t bytes = std::max<size_t>(16, v.size() * sizeof(T));
  if (b.ensure(bytes)) return -1;
  OLM_CUDA(cudaMemset(b.p, 0, bytes));
  if (!v.empty()) OLM_CUDA(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = static_cast<const T *>(b.p);
  return 0;
}

} // namespace

// Pageable host haystacks (main.c maps the file, the cffi wrapper copies into ordinary memory): a
// plain cudaMemcpyAsync from such memory is a synchronous, single-threaded staged copy with no
// overlap.  Instead worker threads copy 4 MiB pieces into the engine's own pinned slots and issue
// the H2D copies from there, so that the CPU copy of one piece, the DMA of others and the scan of
// the segments that are complete all run at once.  Up to kStageThreadsMax threads (a thread's
// memcpy runs at a few GB/s; the PCIe link takes ~55).
constexpr size_t kPieceBytes = size_t(4) << 20;
constexpr int kStageThreadsMax = 16;
struct Stager {
  std::vector<std::thread> workers;
  std::vector<uint8_t *> slots;          // 2 per worker, pinned
  std::vector<uint8_t *> slabs;          // the pinned allocations the slots lie in
  std::vector<cudaEvent_t> slot_events;  // the slot's last copy has finished
  std::unique_ptr<std::atomic<int>[]> seg_left; // pieces of a segment not issued yet
  std::atomic<uint64_t> next_piece{0};
  std::atomic<int> failed{0};
  std::mutex mu;
  std::condition_variable cv;
  std::vector<char> recorded;            // seg_events[i] has been recorded (guarded by mu)
  bool active = false;
};

struct EngineImpl {
  int device = 0, sms = 0;
  int host_threads = 4;
  Stager stager;
  size_t smem_limit = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  // host path: the haystack arrives in segments; seg_events[i] fires when bytes
  // [0, (i+1) * seg_bytes) are in HBM (empty = everything is resident already)
  std::vector<cudaEvent_t> seg_events;
  uint64_t seg_bytes = 0;
  uint64_t seg_off = 0;  // bytes of the slice in front of the staged ones (a stream's carried bytes)
  size_t seg_waited = 0; // segment events of this call the stream already waits for
  bool streaming = false; // set by match_host around its call of match_device
  Header hdr;
  DeviceStore ds;
  ScanGeometry geo;
  bool has_short_234 = false;
  DevBuf d_keys, d_slots, d_recs, d_store, d_g4, d_p23, d_set3, d_bitmap2, d_sx;
  DevBuf hay, out, out2, chunk_desc, span_base, temp, tfblocks, tfvisible, tfplan, tfextent, misc, windows, ghost, ghost_start, fscratch, gather, text;
  cudaEvent_t ev[8] = {};
  olm_cuda_timing_t last{};
  uint64_t out_hint = 0;
  unsigned long long counters[8] = {};
  uint64_t attempts_last = 0;
  // exact statistics (stats.cuh): tables uploaded at create(), the kernel runs only while a stats
  // struct is attached to the matcher
  DevBuf d_bloom, d_smap, d_slens;
  StatsTables stats;
  bool want_stats = false, stats_valid = false;
  unsigned long long stat_counters[5] = {};
  // host haystacks scanned in spans (OLM_HOST_SPAN_BYTES, opt-in): bytes per span (0 = off) and the
  // statistics of the spans before the last one (collect_stats adds them to the last call's)
  uint64_t host_span = 0;
  omega_match_stats_t span_acc{};
  // pattern ids (pattern_ids.cuh): tables uploaded when first switched on
  bool want_ids = false;
  PatternIdTables ids;
  DevBuf d_id_table, d_id_refs, d_id_short;
  // pattern counts of the host path: device scratch, zeroed per call, and its pinned host copy
  DevBuf d_counts;
  uint64_t *h_counts = nullptr;
  size_t h_counts_cap = 0;
  int count_table = -1; // OLM_COUNT_TABLE=0 / 1 (include/olm_b200.h): forces a counting histogram
  // lines (lines.cuh): tile facts and scan, positions of a call (and compacted / gathered), matching
  // lines and their scratch
  DevBuf d_tiles, d_pos, d_pos2, d_pos_gather, d_lines, d_lscratch;
};

namespace {
// The words behind the batch tickets and redo flags of the misc buffer.  Every scan clears `scan`
// with one memset; the other words belong to the passes that use them.
struct MiscWords {
  struct {
    unsigned long long total, filter_total, counters[8], temp_count;
    unsigned long long stats[5]; // stats_kernel (stats.cuh)
  } scan;
  unsigned long long missing_ids; // records without a pattern of the catalogue (ids, counts)
  unsigned long long unused17[3];
  unsigned long long records_outside; // line positions: records outside their bytes
  unsigned long long matching_lines;
  unsigned long long unused22[2];
  NewlineFacts newline_facts;
};
static_assert(sizeof(MiscWords) <= 256, "the misc words fit the 256 bytes behind the tickets");

// misc: [0, kMaxBatches) u32 tickets | [kMaxBatches, 2 kMaxBatches) u32 redo flags | MiscWords
MiscWords *misc_words(EngineImpl &E) {
  if (E.misc.ensure(size_t(kMaxBatches) * 8 + 256)) return nullptr;
  return reinterpret_cast<MiscWords *>(static_cast<uint8_t *>(E.misc.p) + size_t(kMaxBatches) * 8);
}
// index of the event after which the first `bytes` bytes of the slice are in HBM
size_t seg_event_for(const EngineImpl &E, uint64_t bytes) {
  bytes = bytes > E.seg_off ? bytes - E.seg_off : 0;
  if (E.seg_events.size() <= 1 || E.seg_bytes == 0 || bytes == 0) return 0;
  return std::min<size_t>(E.seg_events.size() - 1, size_t((bytes - 1) / E.seg_bytes));
}
// The stream may only wait on a segment event that HAS been recorded: with staging threads at work
// the host first waits until the segment's last piece has been issued.
// (Staged pieces are issued by several threads: a later segment's event does not imply the earlier
// ones, so every segment up to idx is waited for once.)
int wait_segment(EngineImpl &E, size_t idx) {
  Stager &S = E.stager;
  for (size_t j = std::min(E.seg_waited, idx); j <= idx; ++j) {
    if (S.active) {
      std::unique_lock<std::mutex> lk(S.mu);
      S.cv.wait(lk, [&] { return S.recorded[j] || S.failed.load(); });
      if (S.failed.load()) return -1;
    }
    if (cudaStreamWaitEvent(E.stream, E.seg_events[j], 0) != cudaSuccess) return -1;
  }
  E.seg_waited = std::max(E.seg_waited, idx + 1);
  return 0;
}
bool count_block_table(const EngineImpl &E, uint64_t n) {
  return E.count_table >= 0 ? E.count_table != 0 : pattern_counts_block_table(n, E.ids);
}
} // namespace

Engine *Engine::create(const uint8_t *file, size_t size, int device, std::string *err) {
  auto fail = [&](const std::string &m) -> Engine * {
    if (err) *err = m;
    return nullptr;
  };
  StoreView view;
  std::string e = parse_store(file, size, &view);
  if (!e.empty()) return fail(e);

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("no CUDA device: this library has no CPU matching path");
  if (device < 0 || device >= ndev) return fail("CUDA device index out of range");
  if (cudaSetDevice(device) != cudaSuccess) return fail("cudaSetDevice failed");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail("cudaGetDeviceProperties failed");
  if (prop.major < 10) return fail("this build contains sm_100a code only (needs a B200 class GPU)");

  auto *impl = new EngineImpl();
  Engine *eng = new Engine();
  eng->impl_ = impl;
  impl->device = device;
  impl->sms = prop.multiProcessorCount;
  impl->smem_limit = prop.sharedMemPerBlockOptin;
  impl->hdr = view.hdr;

  StagedStore staged;
  FilterBudget budget;
  const bool has_p23 = view.n1 || view.n2 || view.n3;
  // (stores with a transform flag scan in private chunk buffers: less room for the filter)
  budget.g4_max_log2 = (has_p23 || (view.hdr.flags & kFlagAnyTransform)) ? 19 : OLM_G4_MAX_LOG2;
  budget.p23_max_log2 = 18;
  e = stage_store(view, budget, &staged);
  if (e.empty() && check_staged_store(view, staged) != 0) e = "internal error: staged store failed its self check";
  if (!e.empty()) {
    delete eng;
    return fail(e);
  }
  impl->has_short_234 = view.n2 || view.n3 || view.n4;
  impl->ds = staged.params;
  bool ok = true;
  ok = ok && upload(impl->d_keys, staged.keys, &impl->ds.keys) == 0;
  ok = ok && upload(impl->d_slots, staged.slots, &impl->ds.slots) == 0;
  ok = ok && upload(impl->d_recs, staged.recs, &impl->ds.recs) == 0;
  ok = ok && upload(impl->d_store, staged.store, &impl->ds.store) == 0;
  ok = ok && upload(impl->d_g4, staged.g4, &impl->ds.g4) == 0;
  ok = ok && upload(impl->d_p23, staged.p23, &impl->ds.p23) == 0;
  if (impl->ds.sx_words) ok = ok && upload(impl->d_sx, staged.sx, &impl->ds.sx) == 0;
  ok = ok && upload(impl->d_set3, staged.set3, &impl->ds.set3) == 0;
  ok = ok && upload(impl->d_bitmap2, staged.bitmap2, &impl->ds.bitmap2) == 0;
  if (const char *sp = std::getenv("OLM_HOST_SPAN_BYTES")) {
    const unsigned long long v = std::strtoull(sp, nullptr, 10);
    impl->host_span = (v + kWindowBytes - 1) / kWindowBytes * kWindowBytes; // whole 4 MiB windows
  }
  if (const char *ct = std::getenv("OLM_COUNT_TABLE")) impl->count_table = std::atoi(ct) != 0;
  {
    StagedStats ss;
    e = stage_stats(view, &ss);
    if (!e.empty()) {
      delete eng;
      return fail(e);
    }
    impl->stats.bloom_mask = ss.bloom_mask;
    impl->stats.map_shift = ss.map_shift;
    impl->stats.map_mask = ss.map_mask;
    impl->stats.largest = view.hdr.largest;
    ok = ok && upload(impl->d_bloom, ss.bloom, &impl->stats.bloom) == 0;
    ok = ok && upload(impl->d_smap, ss.map, &impl->stats.map) == 0;
    ok = ok && upload(impl->d_slens, ss.lens, &impl->stats.lens) == 0;
  }
  ok = ok && cudaStreamCreateWithFlags(&impl->stream, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&impl->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
  for (auto &ev : impl->ev) ok = ok && cudaEventCreate(&ev) == cudaSuccess;
  ok = ok && scan_configure(impl->smem_limit) == cudaSuccess;
  impl->geo = scan_pick_geometry(impl->ds, impl->smem_limit);
  if (impl->ds.sx_words) {
    // The short candidates' second look (DeviceStore::sx) lives in shared memory beside the filters.
    // It pays where p23 is the weak filter -- the direct two-byte bitmap of stores with 1-byte
    // patterns: 366 vs 339 GB/s on BASELINE configs[3] -- and costs a little where p23 is the hashed
    // three-byte bitmap (names.txt 326 vs 339, census 89 vs 92); and it must not take the room of the
    // tile ring or of the staging areas (census with all transform flags: chunk capacity 168 -> 64,
    // dense chunks redone, 14.5 vs 40 GB/s).  OLM_SHORT_LOOK=0 / 1 overrides the first condition.
    DeviceStore plain = impl->ds;
    plain.sx_words = 0;
    const ScanGeometry g0 = scan_pick_geometry(plain, impl->smem_limit);
    const char *env = std::getenv("OLM_SHORT_LOOK");
    // (the kernels with the second look exist for plain stores without the cooperative compare)
    const bool plain_store = !(impl->hdr.flags & kFlagAnyTransform) && !impl->ds.coop;
    const bool weak_p23 = plain_store && (env ? std::atoi(env) != 0 : impl->ds.p23_mul == 1);
    const bool room = impl->geo.stages != 0 && (impl->geo.stages >= g0.stages || impl->geo.stages >= 8) &&
                      impl->geo.chunk_cap >= std::min<uint32_t>(g0.chunk_cap, 256);
    if (!weak_p23 || !room) {
      impl->ds.sx_words = 0;
      impl->geo = g0;
    }
  }
  if (impl->hdr.flags & kFlagAnyTransform) {
    ok = impl->ghost.ensure(kWindowBytes + 64) == 0 && cudaMemset(impl->ghost.p, 0, impl->ghost.cap) == cudaSuccess;
    if (!ok) {
      delete eng;
      return fail("CUDA allocation failed");
    }
  }
  return eng;
}

Engine::~Engine() {
  if (!impl_) return;
  cudaSetDevice(impl_->device);
  for (DevBuf *b : {&impl_->d_keys, &impl_->d_slots, &impl_->d_recs, &impl_->d_store, &impl_->d_g4, &impl_->d_p23, &impl_->d_sx, &impl_->d_set3,
                    &impl_->d_bitmap2, &impl_->hay, &impl_->out, &impl_->out2, &impl_->chunk_desc, &impl_->span_base, &impl_->temp, &impl_->tfblocks, &impl_->tfvisible, &impl_->tfplan, &impl_->tfextent, &impl_->misc,
                    &impl_->windows, &impl_->gather, &impl_->text, &impl_->ghost, &impl_->ghost_start, &impl_->fscratch, &impl_->d_bloom, &impl_->d_smap,
                    &impl_->d_slens, &impl_->d_id_table, &impl_->d_id_refs, &impl_->d_id_short, &impl_->d_counts,
                    &impl_->d_tiles, &impl_->d_pos, &impl_->d_pos2, &impl_->d_pos_gather, &impl_->d_lines, &impl_->d_lscratch})
    b->release();
  if (impl_->h_counts) cudaFreeHost(impl_->h_counts);
  for (auto &ev : impl_->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &ev : impl_->seg_events) cudaEventDestroy(ev);
  for (auto &ev : impl_->stager.slot_events) cudaEventDestroy(ev);
  for (uint8_t *p : impl_->stager.slabs) cudaFreeHost(p);
  if (impl_->stream) cudaStreamDestroy(impl_->stream);
  if (impl_->copy_stream) cudaStreamDestroy(impl_->copy_stream);
  delete impl_;
}

int Engine::device() const { return impl_->device; }
const Header &Engine::header() const { return impl_->hdr; }
const olm_cuda_timing_t &Engine::timing() const { return impl_->last; }

int Engine::match_device(const ScanRange &r, const MatchFlags &f, olm_cuda_results_t *res, void *dev_counts) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  // device-resident input may have been produced on any stream of the caller
  if (!E.streaming) OLM_CUDA(cudaDeviceSynchronize());
  res->count = 0;
  res->records = nullptr;
  res->device = E.device;
  E.last = olm_cuda_timing_t{};
  std::memset(E.counters, 0, sizeof E.counters);
  std::memset(E.stat_counters, 0, sizeof E.stat_counters);
  E.attempts_last = 0;
  E.stats_valid = false; // (an empty range adds nothing to an attached stats struct, like the reference)

  const bool windowed = E.hdr.flags & kFlagAnyTransform;
  if (r.own_end < r.own_begin || r.own_end > r.global_size || r.own_begin < r.slice_begin ||
      r.own_end > r.slice_begin + r.slice_len || (reinterpret_cast<uintptr_t>(r.dev) & 15) ||
      ((r.own_begin - r.slice_begin) & 15)) {
    std::fprintf(stderr, "libomega_match(b200): invalid scan range / unaligned device buffer\n");
    return -1;
  }
  if (windowed && ((r.own_begin % kWindowBytes) != 0)) {
    std::fprintf(stderr, "libomega_match(b200): shards of a transforming store must start on a 4 MiB window\n");
    return -1;
  }
  if (!windowed && r.own_end > r.own_begin) {
    // the kernel reads one byte in front of the first owned position (start predicates; staged as a
    // 16-byte front halo) and the longest pattern + 1 bytes behind the last one (SURVEY 8e)
    const bool front_ok = r.own_begin == 0 || r.own_begin - r.slice_begin >= 16;
    const uint64_t need_end = std::min<uint64_t>(r.global_size, r.own_end + E.hdr.largest + 1);
    if (!front_ok || r.slice_begin + r.slice_len < need_end) {
      std::fprintf(stderr, "libomega_match(b200): shard slice lacks its halo (16 bytes in front of own_begin, "
                           "largest pattern + 1 bytes behind own_end)\n");
      return -1;
    }
  }
  if (r.out_front && f.no_overlap) {
    std::fprintf(stderr, "libomega_match(b200): internal error: room in front of a filtered output\n");
    return -1;
  }
  const uint64_t n_own = r.own_end - r.own_begin;
  if (n_own == 0) return 0;

  // ---- plan
  const uint64_t n_windows = windowed ? (n_own + kWindowBytes - 1) / kWindowBytes : 0;
  const uint64_t tiles = windowed ? n_windows * kTilesPerWindow : (n_own + kTileBytes - 1) / kTileBytes;
  // plain stores: one launch, or one per segment while the host path streams the bytes in
  const uint64_t seg = (!windowed && E.streaming && E.seg_bytes) ? E.seg_bytes : 0;
  const uint64_t n_batches =
      windowed ? (n_windows + kBatchWindows - 1) / kBatchWindows : (seg ? (n_own + seg - 1) / seg : 1);
  if (tiles >= 0xFFFFFFF0ull || n_batches > kMaxBatches) {
    std::fprintf(stderr, "libomega_match(b200): haystack too large for one call\n");
    return -1;
  }
  MiscWords *w = misc_words(E);
  if (!w) return -1;
  unsigned int *d_tickets = static_cast<unsigned int *>(E.misc.p);
  unsigned int *d_redo_flags = d_tickets + kMaxBatches;
  const uint64_t tiles_per_launch =
      windowed ? uint64_t(kBatchWindows) * kTilesPerWindow : (seg ? (seg + kTileBytes - 1) / kTileBytes : tiles);
  const uint64_t chunks_per_launch = tiles_per_launch * kTileChunks;
  if (E.chunk_desc.ensure((chunks_per_launch + 1) * sizeof(ChunkDesc))) return -1;
  if (E.span_base.ensure((chunks_per_launch / kPrefixSpan + 2) * 8)) return -1;
  unsigned long long *d_total = &w->scan.total;
  unsigned long long *d_counters = w->scan.counters;
  unsigned long long *d_temp_count = &w->scan.temp_count;
  unsigned long long *d_stats = w->scan.stats;
  E.stats_valid = false;

  const bool identity_map = windowed && !(E.hdr.flags & (kFlagIgnorePunct | kFlagElideSpace));
  // window descriptors: case-folding-only stores need the trimmed window lengths, stores with
  // 2..4 byte patterns the stale-tail bytes (transform.cu)
  // The stale-tail bytes are read only under word_boundary (matcher.c:812-848), but the image of the
  // scratch buffer has to follow EVERY call.  Stores that drop bytes: with word_boundary the
  // descriptors are computed before the scan (one more pass over the source); without, the scan
  // counts the window extents as it goes and only the image is updated afterwards.
  const bool need_tails = windowed && E.has_short_234;
  const bool ghost_after = need_tails && !identity_map && !f.word_boundary;
  const bool need_desc = windowed && (identity_map || (need_tails && !ghost_after));
  if (need_desc || ghost_after) {
    const uint64_t bw = std::min<uint64_t>(n_windows, kBatchWindows);
    if (need_desc && E.windows.ensure(n_windows * sizeof(WindowDesc))) return -1;
    if (!identity_map) {
      if (E.tfblocks.ensure(bw * kTfBlocksPerWindow * sizeof(TfBlock))) return -1;
      if (E.tfvisible.ensure(bw * sizeof(uint2))) return -1;
      if (E.tfplan.ensure(bw * sizeof(uint4))) return -1;
      if (E.tfextent.ensure(bw * sizeof(uint32_t))) return -1;
    }
  }

  const uint64_t front = r.out_front;
  uint64_t cap = std::max<uint64_t>(E.out_hint, n_own / 64 + 4096);
  if (E.out.cap / sizeof(Record) >= cap + front) cap = E.out.cap / sizeof(Record) - front;

  uint32_t fl = 0;
  if (f.word_boundary) fl |= kWordBoundary;
  if (f.word_prefix) fl |= kWordPrefix;
  if (f.word_suffix) fl |= kWordSuffix;
  if (f.line_start) fl |= kLineStart;
  if (f.line_end) fl |= kLineEnd;
  if (f.longest_only) fl |= kLongestOnly;
  if (windowed) fl |= kWindowMode;
  if (identity_map) fl |= kIdentityMap;
  if (E.want_stats) fl |= kCountAll;

  // Stores that drop bytes, under word_boundary: every launch group reads its stale tails from the
  // image and then writes its windows into it (transform.cu window_descs_launch).  A second attempt
  // has to read the image the call started with, not the one the first attempt left behind.
  const bool keep_ghost = need_desc && !identity_map;
  if (keep_ghost) {
    if (E.ghost_start.ensure(kWindowBytes + 64)) return -1;
    OLM_CUDA(cudaMemcpyAsync(E.ghost_start.p, E.ghost.p, kWindowBytes + 64, cudaMemcpyDeviceToDevice, E.stream));
  }

  unsigned long long total = 0, temp_used = 0;
  uint64_t temp_extra = 0; // grows when the block allocator of temp[] wasted more than the slack
  for (int attempt = 0; attempt < 4; ++attempt) {
    if (keep_ghost && attempt > 0)
      OLM_CUDA(cudaMemcpyAsync(E.ghost.p, E.ghost_start.p, kWindowBytes + 64, cudaMemcpyDeviceToDevice, E.stream));
    if (E.out.ensure((cap + front) * sizeof(Record))) return -1;
    cap = E.out.cap / sizeof(Record) - front;
    const uint64_t temp_cap = cap + cap / 2 + temp_slack_entries(E.sms) * n_batches + temp_extra;
    if (temp_cap > 0xFFFFFFF0ull) { // chunk descriptors index temp[] with 32 bits
      std::fprintf(stderr, "libomega_match(b200): too many matches for one call\n");
      return -1;
    }
    if (E.temp.ensure(temp_cap * 4)) return -1;
    OLM_CUDA(cudaMemsetAsync(d_tickets, 0, n_batches * 4, E.stream));
    OLM_CUDA(cudaMemsetAsync(d_redo_flags, 0, n_batches * 4, E.stream));
    OLM_CUDA(cudaMemsetAsync(&w->scan, 0, sizeof w->scan, E.stream));
    uint32_t launches = 0, scan_launches = 0;
    uint64_t tf_batches = 0;
    OLM_CUDA(cudaEventRecord(E.ev[0], E.stream));

    ScanParams P{};
    P.st = E.ds;
    P.chunk_desc = static_cast<ChunkDesc *>(E.chunk_desc.p);
    P.span_base = static_cast<unsigned long long *>(E.span_base.p);
    P.temp = static_cast<uint32_t *>(E.temp.p);
    P.temp_cap = temp_cap;
    P.temp_count = d_temp_count;
    P.out = static_cast<Record *>(E.out.p) + front;
    P.out_cap = cap;
    P.match_ptr_base = r.match_ptr_base;
    P.total = d_total;
    P.counters = d_counters;
    P.flags = fl;
    P.stages = E.geo.stages;
    P.chunk_cap = E.geo.chunk_cap;
    P.store_flags = E.hdr.flags;
    P.tail_byte = 0;

    if (!windowed) {
      P.buf = static_cast<const uint8_t *>(r.dev);
      P.buf_len = (r.slice_len + 15) & ~uint64_t(15);
      P.seg_buf_off = -(int64_t)r.slice_begin;
      P.seg_len = r.global_size;
      for (uint64_t b = 0; b < n_batches; ++b) {
        P.scan_begin = r.own_begin + (seg ? b * seg : 0);
        P.scan_end = seg ? std::min<uint64_t>(r.own_end, P.scan_begin + seg) : r.own_end;
        P.num_tiles = (uint32_t)((P.scan_end - P.scan_begin + kTileBytes - 1) / kTileBytes);
        P.ticket = d_tickets + b;
        P.redo_flag = d_redo_flags + b;
        if (E.streaming) { // the scan reads a halo past its positions: the copy has to be that far
          const uint64_t upto = std::min<uint64_t>(r.slice_len, P.scan_end - r.slice_begin + kTileHalo + 16);
          if (wait_segment(E, seg_event_for(E, upto))) return -1;
        }
        OLM_CUDA(scan_launch(P, E.sms, E.stream, &launches));
        if (E.want_stats) OLM_CUDA(stats_launch(P, E.stats, d_stats, E.sms, E.stream, &launches));
        ++scan_launches;
      }
    } else {
      for (uint64_t b = 0; b < n_batches; ++b) {
        const uint64_t w0 = b * kBatchWindows;
        const uint32_t nw = (uint32_t)std::min<uint64_t>(kBatchWindows, n_windows - w0);
        if (E.streaming) { // source bytes of this batch of windows
          const uint64_t src_end = std::min<uint64_t>(n_own, (w0 + nw) * uint64_t(kWindowBytes));
          if (wait_segment(E, seg_event_for(E, (r.own_begin - r.slice_begin) + src_end))) return -1;
        }
        P.buf = static_cast<const uint8_t *>(r.dev);
        P.buf_len = (r.slice_len + 15) & ~uint64_t(15);
        P.win_buf_off = (r.own_begin - r.slice_begin) + w0 * kWindowBytes;
        P.win_src_base = r.own_begin + w0 * kWindowBytes;
        P.win_src_len = std::min<uint64_t>(uint64_t(nw) * kWindowBytes, n_own - w0 * kWindowBytes);
        P.windows = nullptr;
        P.win_extent = nullptr;
        TransformParams T{};
        T.src = P.buf;
        T.src_off = P.win_buf_off;
        T.src_len = P.win_src_len;
        T.windows = need_desc ? static_cast<WindowDesc *>(E.windows.p) + w0 : nullptr;
        T.blocks = static_cast<TfBlock *>(E.tfblocks.p);
        T.visible = static_cast<uint2 *>(E.tfvisible.p);
        T.plan = static_cast<uint4 *>(E.tfplan.p);
        T.ghost = static_cast<uint8_t *>(E.ghost.p);
        T.flags = E.hdr.flags;
        if (ghost_after) {
          P.win_extent = static_cast<uint32_t *>(E.tfextent.p);
          OLM_CUDA(cudaMemsetAsync(P.win_extent, 0, nw * sizeof(uint32_t), E.stream));
        }
        if (need_desc) {
          OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
          OLM_CUDA(window_descs_launch(T, nw, need_tails, E.sms, E.stream, &launches));
          OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
          P.windows = T.windows;
          tf_batches = b + 1;
        }
        P.tiles_per_win = kTilesPerWindow;
        P.num_tiles = nw * kTilesPerWindow;
        P.ticket = d_tickets + b;
        P.redo_flag = d_redo_flags + b;
        OLM_CUDA(scan_launch(P, E.sms, E.stream, &launches));
        if (ghost_after) OLM_CUDA(ghost_update_launch(T, nw, P.win_extent, E.sms, E.stream, &launches));
        if (E.want_stats) OLM_CUDA(stats_launch(P, E.stats, d_stats, E.sms, E.stream, &launches));
        ++scan_launches;
      }
    }
    OLM_CUDA(cudaEventRecord(E.ev[1], E.stream));
    if (E.want_stats)
      OLM_CUDA(cudaMemcpyAsync(E.stat_counters, d_stats, sizeof E.stat_counters, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaMemcpyAsync(&total, d_total, sizeof total, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaMemcpyAsync(&temp_used, d_temp_count, sizeof temp_used, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaMemcpyAsync(E.counters, d_counters, sizeof E.counters, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    E.last.kernel_launches = launches;
    E.last.scan_launches = scan_launches;
    E.last.transform_ms = 0.f;
    if (tf_batches) { // (the last batch's descriptor kernels; all batches of a call are alike)
      float t = 0.f;
      cudaEventElapsedTime(&t, E.ev[2], E.ev[3]);
      E.last.transform_ms = t * float(tf_batches);
    }
    if (total <= cap && temp_used <= temp_cap) break;
    if (temp_used > temp_cap) temp_extra += temp_used - temp_cap + temp_used / 8;
    if (attempt == 3) {
      std::fprintf(stderr, "libomega_match(b200): result buffer still too small after retry\n");
      return -1;
    }
    if (total > cap) cap = total + total / 16 + 4096; // exact count is known now
  }
  E.out_hint = std::max<uint64_t>(E.out_hint, total + total / 8);
  E.stats_valid = E.want_stats;
  E.last.matches_before_filter = total;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, E.ev[0], E.ev[1]);
  E.last.scan_ms = ms;
  E.last.total_ms = ms;

  void *final_records = static_cast<Record *>(E.out.p) + front;
  if (f.no_overlap && total > (r.floor ? 0 : 1)) {
    if (E.out2.ensure(total * sizeof(Record))) return -1;
    if (E.fscratch.ensure(filter_scratch_bytes(total))) return -1;
    uint32_t launches = 0;
    OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
    OLM_CUDA(no_overlap_launch(static_cast<const Record *>(E.out.p), total, static_cast<Record *>(E.out2.p),
                               E.fscratch.p, &w->scan.filter_total, E.stream, &launches, r.floor));
    OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
    OLM_CUDA(cudaMemcpyAsync(&total, &w->scan.filter_total, sizeof total, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    cudaEventElapsedTime(&ms, E.ev[2], E.ev[3]);
    E.last.filter_ms = ms;
    E.last.total_ms += ms;
    E.last.kernel_launches += launches;
    std::swap(E.out, E.out2);
    final_records = E.out.p;
  }
  if ((E.want_ids || dev_counts) && total) {
    unsigned long long *d_missing = &w->missing_ids;
    unsigned long long missing = 0;
    uint32_t launches = 0;
    // (the host path: a record may end in a segment the scan did not have to wait for)
    if (E.streaming && !E.seg_events.empty() && wait_segment(E, E.seg_events.size() - 1)) return -1;
    OLM_CUDA(cudaMemsetAsync(d_missing, 0, sizeof missing, E.stream));
    OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
    if (dev_counts) // instead of the ids: the count of the records per pattern
      OLM_CUDA(pattern_counts_launch(static_cast<const Record *>(final_records), total, static_cast<const uint8_t *>(r.dev),
                                     r.slice_begin, E.ids, count_block_table(E, total),
                                     static_cast<unsigned long long *>(dev_counts), d_missing, E.sms, E.stream, &launches));
    else
      OLM_CUDA(pattern_ids_launch(static_cast<Record *>(final_records), total, static_cast<const uint8_t *>(r.dev),
                                  r.slice_begin, E.ids, d_missing, E.sms, E.stream, &launches));
    OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
    OLM_CUDA(cudaMemcpyAsync(&missing, d_missing, sizeof missing, cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    cudaEventElapsedTime(&ms, E.ev[2], E.ev[3]);
    E.last.total_ms += ms;
    E.last.kernel_launches += launches;
    if (missing) {
      std::fprintf(stderr, "libomega_match(b200): %llu records matched no pattern of the catalogue (internal error)\n",
                   missing);
      return -1;
    }
  }
  // statistics that do not need a kernel: long-path attempts without word_boundary
  if (E.hdr.largest >= 5 && !f.word_boundary && !windowed) {
    const uint64_t lim = r.global_size >= 3 ? r.global_size - 3 : 0;
    const uint64_t hi = std::min<uint64_t>(r.own_end, lim);
    E.attempts_last = hi > r.own_begin ? hi - r.own_begin : 0;
  }
  res->count = total;
  res->records = final_records;
  return 0;
}

// H2D of `n` host bytes into the engine's haystack buffer: long inputs arrive in 256 MiB segments
// on the copy stream while earlier segments are being scanned (match_device waits on the segment
// events); short ones in one copy.  ev[4]/ev[5] bracket the copies.
int Engine::stage_host(const uint8_t *src, size_t n, size_t dst_off) {
  EngineImpl &E = *impl_;
  const size_t padded = ((dst_off + n + 15) & ~size_t(15)) + 256;
  if (E.hay.ensure(padded)) return -1;
  const uint64_t nseg = n >= kPipelineMin ? (n + kSegmentBytes - 1) / kSegmentBytes : 1;
  while (E.seg_events.size() < nseg) {
    cudaEvent_t ev;
    OLM_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    E.seg_events.push_back(ev);
  }
  while (E.seg_events.size() > nseg) { // seg_event_for() indexes by size: keep exactly nseg
    cudaEventDestroy(E.seg_events.back());
    E.seg_events.pop_back();
  }
  E.seg_bytes = nseg > 1 ? kSegmentBytes : 0;
  E.seg_off = dst_off;
  E.seg_waited = 0;
  OLM_CUDA(cudaEventRecord(E.ev[4], E.copy_stream));
  {
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess &&
                        (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (!pinned && n >= 4 * kPieceBytes) return stage_pageable(src, n, nseg, dst_off);
  }
  for (uint64_t i = 0; i < nseg; ++i) {
    const uint64_t b = i * kSegmentBytes, e = nseg > 1 ? std::min<uint64_t>(n, b + kSegmentBytes) : n;
    OLM_CUDA(cudaMemcpyAsync(static_cast<uint8_t *>(E.hay.p) + dst_off + b, src + b, e - b, cudaMemcpyHostToDevice,
                             E.copy_stream));
    OLM_CUDA(cudaEventRecord(E.seg_events[i], E.copy_stream));
  }
  OLM_CUDA(cudaEventRecord(E.ev[5], E.copy_stream));
  return 0;
}

// Pageable memory: see Stager.  Returns after the workers have been started; match_device() waits
// for a segment's event to be recorded before it lets the stream wait on it, finish_staging() joins.
int Engine::stage_pageable(const uint8_t *src, size_t n, uint64_t nseg, size_t dst_off) {
  EngineImpl &E = *impl_;
  Stager &S = E.stager;
  const uint64_t n_pieces = (n + kPieceBytes - 1) / kPieceBytes;
  const uint64_t per_seg = nseg > 1 ? kSegmentBytes / kPieceBytes : n_pieces;
  const int T = (int)std::max<uint64_t>(1, std::min<uint64_t>({(uint64_t)E.host_threads, (uint64_t)kStageThreadsMax, n_pieces}));
  if (S.slots.size() < size_t(2 * T)) { // (one pinned allocation for all the slots that are missing)
    const size_t more = size_t(2 * T) - S.slots.size();
    uint8_t *slab = nullptr;
    OLM_CUDA(cudaHostAlloc(&slab, more * kPieceBytes, cudaHostAllocDefault));
    S.slabs.push_back(slab);
    for (size_t i = 0; i < more; ++i) {
      cudaEvent_t ev;
      OLM_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      S.slots.push_back(slab + i * kPieceBytes);
      S.slot_events.push_back(ev);
    }
  }
  S.seg_left.reset(new std::atomic<int>[nseg]);
  for (uint64_t i = 0; i < nseg; ++i) {
    const uint64_t first = i * per_seg, last = std::min<uint64_t>(n_pieces, first + per_seg);
    S.seg_left[i].store((int)(last - first));
  }
  S.recorded.assign(nseg, 0);
  S.next_piece.store(0);
  S.failed.store(0);
  S.active = true;
  uint8_t *dst = static_cast<uint8_t *>(E.hay.p) + dst_off;
  for (int t = 0; t < T; ++t) {
    S.workers.emplace_back([&E, &S, src, dst, n, n_pieces, per_seg, nseg, t]() {
      if (cudaSetDevice(E.device) != cudaSuccess) S.failed.store(1);
      for (uint32_t use = 0; !S.failed.load(); ++use) {
        const uint64_t p = S.next_piece.fetch_add(1);
        if (p >= n_pieces) break;
        const size_t slot = size_t(2 * t) + (use & 1u);
        const uint64_t b = p * kPieceBytes, len = std::min<uint64_t>(kPieceBytes, n - b);
        bool ok = cudaEventSynchronize(S.slot_events[slot]) == cudaSuccess; // (never recorded: returns at once)
        if (ok) {
          std::memcpy(S.slots[slot], src + b, len);
          ok = cudaMemcpyAsync(dst + b, S.slots[slot], len, cudaMemcpyHostToDevice, E.copy_stream) == cudaSuccess &&
               cudaEventRecord(S.slot_events[slot], E.copy_stream) == cudaSuccess;
        }
        const uint64_t seg = std::min<uint64_t>(nseg - 1, p / per_seg);
        if (ok && S.seg_left[seg].fetch_sub(1) == 1) { // the segment's last piece: every copy of it has been issued
          ok = cudaEventRecord(E.seg_events[seg], E.copy_stream) == cudaSuccess;
          if (ok && seg == nseg - 1) ok = cudaEventRecord(E.ev[5], E.copy_stream) == cudaSuccess;
          std::lock_guard<std::mutex> lk(S.mu);
          S.recorded[seg] = 1;
          S.cv.notify_all();
        }
        if (!ok) {
          S.failed.store(1);
          std::lock_guard<std::mutex> lk(S.mu);
          S.cv.notify_all();
        }
      }
    });
  }
  return 0;
}

int Engine::finish_staging() {
  Stager &S = impl_->stager;
  if (!S.active) return 0;
  for (auto &t : S.workers) t.join();
  S.workers.clear();
  S.active = false;
  return S.failed.load() ? -1 : 0;
}

void Engine::set_host_threads(int n) { impl_->host_threads = n < 1 ? 1 : n; }

namespace {
struct StreamingScope { // the device-resident entry points never see segments
  EngineImpl &E;
  explicit StreamingScope(EngineImpl &e) : E(e) { E.streaming = true; }
  ~StreamingScope() { E.streaming = false; }
};
} // namespace

// One rank's byte range from HOST memory: the slice is copied in segments while the scan of the
// earlier segments runs; the records stay on the device (like match_device with a shard range).
int Engine::match_shard_host(const uint8_t *host_slice, const ScanRange &range, const MatchFlags &f,
                             olm_cuda_results_t *out, void *dev_counts) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (!host_slice || range.slice_len == 0) return -1;
  if (stage_host(host_slice, range.slice_len)) return -1;
  StreamingScope scope(E);
  ScanRange r = range;
  r.dev = E.hay.p;
  const int rc = match_device(r, f, out, dev_counts);
  if (finish_staging() != 0 || rc != 0) return -1;
  float ms = 0.f;
  OLM_CUDA(cudaStreamSynchronize(E.copy_stream));
  cudaEventElapsedTime(&ms, E.ev[4], E.ev[5]);
  E.last.h2d_ms = ms;
  return 0;
}

// ---- streams (include/olm_b200.h "Streams")
//
// A push scans the owned positions [settled before, settled after) as a byte-range shard of the whole
// stream (SURVEY 8e) with global_size = received, so no predicate sees the end early.  The bytes it
// needs in front of the piece are the carried ones: [settled - 16, received) of a plain store, the
// incomplete window of a transforming one.  Host pieces are staged behind the carried bytes in the
// haystack buffer and scanned in one call.  Device pieces of a plain store are scanned in place: only
// the seam -- the positions up to the piece's 16th byte -- is scanned from the carried bytes and the
// piece's first largest + 17 bytes; its records go in front of the bulk's.  Other device pieces are
// copied behind the carried bytes.  no_overlap runs on the push's records with the stream's floor.

namespace {
void add_timing(olm_cuda_timing_t &t, const olm_cuda_timing_t &a) {
  t.total_ms += a.total_ms;
  t.transform_ms += a.transform_ms;
  t.scan_ms += a.scan_ms;
  t.filter_ms += a.filter_ms;
  t.h2d_ms += a.h2d_ms;
  t.d2h_ms += a.d2h_ms;
  t.scan_launches += a.scan_launches;
  t.kernel_launches += a.kernel_launches;
  t.matches_before_filter += a.matches_before_filter;
}
} // namespace

void Engine::stream_release(StreamState &s) {
  if (s.carry) {
    cudaSetDevice(impl_->device);
    cudaFree(s.carry);
  }
  s.carry = nullptr;
  s.carry_cap = 0;
}

int Engine::stream_push(StreamState &s, const void *bytes, size_t n, bool on_device, bool last,
                        olm_cuda_results_t *out, uint64_t *counts) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  out->count = 0;
  out->records = nullptr;
  out->device = E.device;
  if (s.finished || s.failed || (n && !bytes)) {
    std::fprintf(stderr, "libomega_match(b200): stream push %s\n",
                 s.failed ? "after a failed push" : s.finished ? "after the last push" : "of NULL bytes");
    return -1;
  }
  s.failed = true; // until the push has succeeded
  if (on_device) OLM_CUDA(cudaDeviceSynchronize()); // the piece may come from any stream of the caller
  E.span_acc = omega_match_stats_t{};
  const bool windowed = E.hdr.flags & kFlagAnyTransform;
  const uint64_t R = s.received, recv = R + n, largest = E.hdr.largest;
  uint64_t settled = recv;
  if (!last && windowed) {
    settled = recv / kWindowBytes * kWindowBytes;
  } else if (!last) { // (a shard starts at 0 or has 16 bytes in front: below 16 nothing settles)
    const uint64_t k = recv > largest + 1 ? recv - largest - 1 : 0;
    settled = std::max<uint64_t>(s.settled, k >= 16 ? k : 0);
  }
  const uint64_t carried = R - s.carry_begin; // bytes in front of the piece
  unsigned long long *d_counts = nullptr;
  if (counts && !(d_counts = zeroed_counts())) return -1;
  MatchFlags fs = s.f;
  const uint8_t *piece = static_cast<const uint8_t *>(bytes);
  // plain store, aligned device piece with positions past its 16th byte to settle: in place
  const bool in_place =
      on_device && !counts && !windowed && !(reinterpret_cast<uintptr_t>(bytes) & 15) && settled > R + 16;
  olm_cuda_results_t res{};
  if (!in_place) { // carried bytes + piece in the haystack buffer, one call
    if (on_device) {
      if (E.hay.ensure(((carried + n + 15) & ~size_t(15)) + 256)) return -1;
      if (n) OLM_CUDA(cudaMemcpyAsync(static_cast<uint8_t *>(E.hay.p) + carried, piece, n, cudaMemcpyDeviceToDevice, E.stream));
    } else if (n && stage_host(piece, n, carried)) {
      return -1;
    } else if (!n && E.hay.ensure(((carried + 15) & ~size_t(15)) + 256)) {
      return -1;
    }
    if (carried) OLM_CUDA(cudaMemcpyAsync(E.hay.p, s.carry, carried, cudaMemcpyDeviceToDevice, E.stream));
    ScanRange r{E.hay.p, s.carry_begin, recv - s.carry_begin, s.settled, settled, recv, s.match_ptr_base, s.floor, 0};
    int rc;
    {
      const bool staged = !on_device && n;
      if (staged) E.streaming = true;
      rc = match_device(r, fs, &res, d_counts);
      // the new carried bytes are copied out of the buffer below: all of the piece has to be there
      if (staged) {
        E.streaming = false;
        if (rc == 0 && !E.seg_events.empty() && wait_segment(E, E.seg_events.size() - 1)) rc = -1;
        if (finish_staging() != 0) rc = -1;
        float ms = 0.f;
        OLM_CUDA(cudaStreamSynchronize(E.copy_stream));
        cudaEventElapsedTime(&ms, E.ev[4], E.ev[5]);
        E.last.h2d_ms = ms;
      }
    }
    if (rc != 0) return -1;
  } else { // seam from the haystack buffer, then the bulk in the caller's buffer
    const uint64_t seam_bytes = std::min<uint64_t>(n, largest + 17);
    if (E.hay.ensure(((carried + seam_bytes + 15) & ~size_t(15)) + 256)) return -1;
    if (carried) OLM_CUDA(cudaMemcpyAsync(E.hay.p, s.carry, carried, cudaMemcpyDeviceToDevice, E.stream));
    OLM_CUDA(cudaMemcpyAsync(static_cast<uint8_t *>(E.hay.p) + carried, piece, seam_bytes, cudaMemcpyDeviceToDevice, E.stream));
    fs.no_overlap = false; // (once, on the concatenation)
    const ScanRange seam{E.hay.p, s.carry_begin, carried + seam_bytes, s.settled, R + 16, recv, s.match_ptr_base, 0, 0};
    if (match_device(seam, fs, &res)) return -1;
    const olm_cuda_timing_t t_seam = E.last;
    { // the seam's statistics are collected with the bulk's (as host_spans does with its spans)
      omega_match_stats_t acc{};
      collect_stats(&acc);
      E.span_acc = acc;
    }
    const uint64_t n_seam = res.count;
    if (n_seam && E.gather.ensure(n_seam * sizeof(Record))) return -1;
    if (n_seam) OLM_CUDA(cudaMemcpyAsync(E.gather.p, res.records, n_seam * sizeof(Record), cudaMemcpyDeviceToDevice, E.stream));
    const ScanRange bulk{piece, R, n, R + 16, settled, recv, s.match_ptr_base, 0, n_seam};
    if (match_device(bulk, fs, &res)) return -1;
    add_timing(E.last, t_seam);
    if (n_seam) OLM_CUDA(cudaMemcpyAsync(E.out.p, E.gather.p, n_seam * sizeof(Record), cudaMemcpyDeviceToDevice, E.stream));
    res.records = E.out.p;
    res.count += n_seam;
    if (s.f.no_overlap && res.count) {
      const int64_t kept = no_overlap_inplace(E.out.p, res.count, nullptr, s.floor);
      if (kept < 0) return -1;
      res.count = uint64_t(kept);
    }
  }
  // the floor of the next push: the end of the last kept record
  if (s.f.no_overlap && res.count) {
    Record lastrec;
    OLM_CUDA(cudaMemcpyAsync(&lastrec, static_cast<const Record *>(res.records) + (res.count - 1), sizeof lastrec,
                             cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    s.floor = lastrec.offset + lastrec.len;
  }
  if (counts && add_counts_to_host(counts)) return -1;
  // carry [next_begin, recv): what lies before the piece from the haystack buffer, the rest from the
  // buffer too unless the piece was scanned in place
  const uint64_t next_begin = last ? recv : windowed ? settled : (settled >= 16 ? settled - 16 : 0);
  const uint64_t keep = recv - next_begin;
  if (keep > s.carry_cap) {
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    if (s.carry) cudaFree(s.carry);
    s.carry = nullptr;
    s.carry_cap = 0;
    const size_t want = std::max<size_t>(keep, 4096);
    OLM_CUDA(cudaMalloc(&s.carry, want));
    s.carry_cap = want;
  }
  const uint8_t *hay = static_cast<const uint8_t *>(E.hay.p);
  uint8_t *dst = static_cast<uint8_t *>(s.carry);
  if (in_place) {
    const uint64_t a = std::min(next_begin, R); // [a, R) from the carried bytes in front of the seam
    if (R > a) OLM_CUDA(cudaMemcpyAsync(dst, hay + (a - s.carry_begin), R - a, cudaMemcpyDeviceToDevice, E.stream));
    const uint64_t b = std::max(next_begin, R);
    if (recv > b) OLM_CUDA(cudaMemcpyAsync(dst + (b - next_begin), piece + (b - R), recv - b, cudaMemcpyDeviceToDevice, E.stream));
  } else if (keep) {
    OLM_CUDA(cudaMemcpyAsync(dst, hay + (next_begin - s.carry_begin), keep, cudaMemcpyDeviceToDevice, E.stream));
  }
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  s.carry_begin = next_begin;
  s.received = recv;
  s.settled = settled;
  s.finished = last;
  s.failed = false;
  *out = res;
  out->device = E.device;
  return 0;
}

// A host haystack in consecutive spans of host_span start positions (opt-in: OLM_HOST_SPAN_BYTES; for
// haystacks that should not be resident in HBM all at once), or in one span of all n bytes.  Every span
// is a byte-range shard of the whole (SURVEY 8e: same ownership rule, halo and global-size predicates
// as the multi-GPU path), scanned from host memory with the copy overlapped; step(span, its records,
// several) runs after each.  With several spans, `no_overlap` -- the one filter that crosses span
// edges -- is left to the caller, to run once on the concatenation, and nothing is counted into
// dev_counts (counts follow the filter).  Returns the number of spans, -1 on failure.
int Engine::host_spans(const uint8_t *haystack, size_t n, const MatchFlags &f, void *dev_counts, const SpanStep &step) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  E.span_acc = omega_match_stats_t{};
  if (n == 0 || !haystack) { // nothing scanned: collect_stats() and timing() must not report the previous call
    std::memset(E.counters, 0, sizeof E.counters);
    std::memset(E.stat_counters, 0, sizeof E.stat_counters);
    E.attempts_last = 0;
    E.stats_valid = false;
    E.last = olm_cuda_timing_t{};
    return 0;
  }
  const uint64_t span = E.host_span && n > E.host_span ? E.host_span : n;
  const bool several = span < n;
  MatchFlags fs = f;
  if (several && f.no_overlap) {
    fs.no_overlap = false;
    dev_counts = nullptr;
  }
  int spans = 0;
  for (uint64_t b = 0; b < n; b += span, ++spans) {
    const Shard s = shard_of(b, std::min<uint64_t>(n, b + span), n, E.hdr.largest, E.hdr.flags & kFlagAnyTransform);
    olm_cuda_results_t d;
    if (match_shard_host(haystack + s.slice_begin, scan_range(s, n, reinterpret_cast<uint64_t>(haystack)), fs, &d,
                         dev_counts) != 0 ||
        step(s, d, several) != 0)
      return -1;
    if (s.own_end < n) { // the last span's counters are collected by the caller, like those of a plain call
      omega_match_stats_t acc = E.span_acc;
      E.span_acc = omega_match_stats_t{};
      collect_stats(&acc);
      E.span_acc = acc;
    }
  }
  return spans;
}

omega_match_results_t *Engine::match_host(const uint8_t *haystack, size_t n, const MatchFlags &f) {
  EngineImpl &E = *impl_;
  static_assert(sizeof(Record) == sizeof(omega_match_result_t), "records are copied out verbatim");
  omega_match_results_t *results = nullptr; // one span: its records, straight from the device
  std::vector<Record> all;                  // several: their records, concatenated on the host
  const int spans = host_spans(haystack, n, f, nullptr, [&](const Shard &, const olm_cuda_results_t &d, bool several) {
    if (several) {
      if (!d.count) return 0;
      const size_t at = all.size();
      all.resize(at + d.count);
      return copy_to_host(all.data() + at, d.records, d.count * sizeof(Record)) == 0 && sync() == 0 ? 0 : -1;
    }
    if (!(results = host_results(d.count))) return -1;
    if (!d.count) return 0;
    float ms = 0.f;
    cudaEventRecord(E.ev[6], E.stream);
    OLM_CUDA(cudaMemcpyAsync(results->matches, d.records, d.count * sizeof(Record), cudaMemcpyDeviceToHost, E.stream));
    cudaEventRecord(E.ev[7], E.stream);
    OLM_CUDA(cudaStreamSynchronize(E.stream));
    cudaEventElapsedTime(&ms, E.ev[6], E.ev[7]);
    E.last.d2h_ms = ms;
    return 0;
  });
  if (spans < 0) {
    omega_match_results_destroy(results);
    return nullptr;
  }
  if (results) return results;
  uint64_t total = all.size();
  if (f.no_overlap && total > 1) { // several spans: the filter once, on the device
    if (E.out.ensure(total * sizeof(Record))) return nullptr;
    if (cudaMemcpyAsync(E.out.p, all.data(), total * sizeof(Record), cudaMemcpyHostToDevice, E.stream) != cudaSuccess) return nullptr;
    const int64_t kept = no_overlap_inplace(E.out.p, total);
    if (kept < 0) return nullptr;
    total = uint64_t(kept);
    if (cudaMemcpyAsync(all.data(), E.out.p, total * sizeof(Record), cudaMemcpyDeviceToHost, E.stream) != cudaSuccess ||
        cudaStreamSynchronize(E.stream) != cudaSuccess)
      return nullptr;
  }
  if (!(results = host_results(total))) return nullptr;
  if (total) std::memcpy(results->matches, all.data(), total * sizeof(Record));
  return results;
}

int Engine::format_records(const void *dev_records, uint64_t count, const void *dev_haystack, uint64_t offset0,
                           void **dev_text, uint64_t *text_bytes) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  *dev_text = nullptr;
  *text_bytes = 0;
  if (count == 0) return 0;
  OLM_CUDA(cudaDeviceSynchronize()); // records and haystack may come from any stream of the caller
  if (E.fscratch.ensure(format_scratch_bytes(count))) return -1;
  MiscWords *w = misc_words(E);
  if (!w) return -1;
  unsigned long long *d_total = &w->scan.filter_total;
  uint32_t launches = 0;
  unsigned long long total = 0;
  const Record *rec = static_cast<const Record *>(dev_records);
  const uint8_t *hay = static_cast<const uint8_t *>(dev_haystack);
  OLM_CUDA(format_lengths_launch(rec, count, hay, offset0, E.fscratch.p, d_total, E.stream, &launches));
  OLM_CUDA(cudaMemcpyAsync(&total, d_total, sizeof total, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  if (E.text.ensure(total + 16)) return -1;
  OLM_CUDA(format_write_launch(rec, count, hay, offset0, E.fscratch.p, static_cast<uint8_t *>(E.text.p), total, E.stream, &launches));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  *dev_text = E.text.p;
  *text_bytes = total;
  return 0;
}

int64_t Engine::no_overlap_inplace(void *dev_records, uint64_t count, void *dev_positions, uint64_t floor) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (count < (floor ? 1 : 2)) return (int64_t)count;
  // the records may have been produced on any stream of the caller (a gather, a copy): the
  // matcher's stream is non-blocking and would not wait for them (same contract as match_device)
  OLM_CUDA(cudaDeviceSynchronize());
  if (E.out2.ensure(count * sizeof(Record))) return -1;
  if (E.fscratch.ensure(filter_scratch_bytes(count))) return -1;
  MiscWords *w = misc_words(E);
  if (!w) return -1;
  unsigned long long *d_ftotal = &w->scan.filter_total;
  uint32_t launches = 0;
  unsigned long long total = 0;
  if (dev_positions && E.d_pos2.ensure(count * sizeof(LinePos))) return -1;
  OLM_CUDA(no_overlap_launch(static_cast<const Record *>(dev_records), count, static_cast<Record *>(E.out2.p),
                             E.fscratch.p, d_ftotal, E.stream, &launches, floor, static_cast<const LinePos *>(dev_positions),
                             static_cast<LinePos *>(E.d_pos2.p)));
  OLM_CUDA(cudaMemcpyAsync(&total, d_ftotal, sizeof total, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  OLM_CUDA(cudaMemcpyAsync(dev_records, E.out2.p, total * sizeof(Record), cudaMemcpyDeviceToDevice, E.stream));
  if (dev_positions)
    OLM_CUDA(cudaMemcpyAsync(dev_positions, E.d_pos2.p, total * sizeof(LinePos), cudaMemcpyDeviceToDevice, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  return (int64_t)total;
}

int Engine::sort_records(void *dev_records, uint64_t count) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (count < 2) return 0;
  OLM_CUDA(cudaDeviceSynchronize()); // see no_overlap_inplace
  if (E.out2.ensure(count * sizeof(Record))) return -1;
  if (E.fscratch.ensure(sort_scratch_bytes(count))) return -1;
  uint32_t launches = 0;
  OLM_CUDA(sort_records_launch(static_cast<Record *>(dev_records), static_cast<Record *>(E.out2.p), count,
                               E.fscratch.p, E.stream, &launches));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  return 0;
}

void *Engine::stream() const { return impl_->stream; }
bool Engine::needs_window_tails() const { return (impl_->hdr.flags & kFlagAnyTransform) && impl_->has_short_234; }
void *Engine::ghost_image() const { return impl_->ghost.p; }

void *Engine::gather_buffer(size_t bytes, size_t *cap) {
  if (cudaSetDevice(impl_->device) != cudaSuccess) return nullptr;
  // (bytes == 0 with `cap`: the buffer as it is, nothing allocated)
  if ((bytes || !cap) && impl_->gather.ensure(bytes ? bytes : 16)) return nullptr;
  if (cap) *cap = impl_->gather.cap;
  return impl_->gather.p;
}

int Engine::sync() {
  OLM_CUDA(cudaSetDevice(impl_->device));
  OLM_CUDA(cudaStreamSynchronize(impl_->stream));
  return 0;
}

void Engine::set_exact_stats(bool on) { impl_->want_stats = on; }

int Engine::load_pattern_tables(const PatternCatalog *cat) {
  EngineImpl &E = *impl_;
  if (E.ids.table) return 0;
  if (!cat) return -1;
  OLM_CUDA(cudaSetDevice(E.device));
  PatternIdTables t;
  if (upload(E.d_id_table, cat->table, &t.table) || upload(E.d_id_refs, cat->refs, &t.refs) ||
      upload(E.d_id_short, cat->short_bytes, &t.short_bytes))
    return -1;
  t.table_mask = cat->table_mask;
  t.store = E.ds.store;
  t.store_flags = E.hdr.flags;
  t.count = uint32_t(cat->size());
  E.ids = t;
  return 0;
}

int Engine::set_pattern_ids(bool on, const PatternCatalog *cat) {
  if (on && load_pattern_tables(cat)) return -1;
  impl_->want_ids = on;
  return 0;
}

bool Engine::pattern_ids() const { return impl_->want_ids; }
uint64_t Engine::pattern_count() const { return impl_->ids.count; }

// ---- pattern counts (include/olm_b200.h): the tables are loaded (load_pattern_tables) before any
// of these runs

int Engine::count_records(const void *dev_records, uint64_t count, void *dev_counts) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (!E.ids.table) return -1;
  if (count == 0) return 0;
  OLM_CUDA(cudaDeviceSynchronize()); // see no_overlap_inplace
  MiscWords *w = misc_words(E);
  if (!w) return -1;
  unsigned long long *d_missing = &w->missing_ids;
  unsigned long long missing = 0;
  uint32_t launches = 0;
  OLM_CUDA(cudaMemsetAsync(d_missing, 0, sizeof missing, E.stream));
  OLM_CUDA(pattern_counts_launch(static_cast<const Record *>(dev_records), count, nullptr, 0, E.ids,
                                 count_block_table(E, count), static_cast<unsigned long long *>(dev_counts), d_missing,
                                 E.sms, E.stream, &launches));
  OLM_CUDA(cudaMemcpyAsync(&missing, d_missing, sizeof missing, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  if (missing) {
    std::fprintf(stderr, "libomega_match(b200): %llu records hold no pattern id of the catalogue (%u patterns)\n",
                 missing, E.ids.count);
    return -1;
  }
  return 0;
}

// the device scratch counts of the host path, zeroed on the stream
unsigned long long *Engine::zeroed_counts() {
  EngineImpl &E = *impl_;
  const size_t bytes = std::max<size_t>(1, E.ids.count) * sizeof(uint64_t);
  if (E.d_counts.ensure(bytes) || cudaMemsetAsync(E.d_counts.p, 0, bytes, E.stream) != cudaSuccess) return nullptr;
  return static_cast<unsigned long long *>(E.d_counts.p);
}

// counts[] += the device scratch counts: one D2H of 8 bytes per pattern (d2h_ms)
int Engine::add_counts_to_host(uint64_t *counts) {
  EngineImpl &E = *impl_;
  const size_t n = E.ids.count;
  if (E.h_counts_cap < n) {
    if (E.h_counts) cudaFreeHost(E.h_counts);
    E.h_counts = nullptr;
    E.h_counts_cap = 0;
    OLM_CUDA(cudaHostAlloc(&E.h_counts, n * sizeof(uint64_t), cudaHostAllocDefault));
    E.h_counts_cap = n;
  }
  float ms = 0.f;
  OLM_CUDA(cudaEventRecord(E.ev[6], E.stream));
  OLM_CUDA(cudaMemcpyAsync(E.h_counts, E.d_counts.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaEventRecord(E.ev[7], E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  cudaEventElapsedTime(&ms, E.ev[6], E.ev[7]);
  E.last.d2h_ms = ms;
  for (size_t i = 0; i < n; ++i) counts[i] += E.h_counts[i];
  return 0;
}

int Engine::count_shard_host(const uint8_t *host_slice, const ScanRange &range, const MatchFlags &f, uint64_t *counts,
                             uint64_t *total) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  unsigned long long *d = zeroed_counts();
  olm_cuda_results_t res;
  if (!d || match_shard_host(host_slice, range, f, &res, d) != 0 || add_counts_to_host(counts) != 0) return -1;
  *total = res.count;
  return 0;
}

// Without no_overlap, or in one span, every span counts on the device into one scratch array.  Several
// spans under no_overlap write ids instead (their haystacks are gone when the filter runs): their
// records are concatenated on the device, filtered once, and counted from the pads.
int Engine::count_host(const uint8_t *haystack, size_t n, const MatchFlags &f, uint64_t *counts, uint64_t *total) {
  EngineImpl &E = *impl_;
  *total = 0;
  OLM_CUDA(cudaSetDevice(E.device));
  unsigned long long *d = zeroed_counts();
  if (!d) return -1;
  PatternIdsOn ids({this}, f.no_overlap); // (a span that counts into d writes no ids)
  uint64_t all = 0; // records concatenated in E.gather (several spans under no_overlap)
  const int spans = host_spans(haystack, n, f, d, [&](const Shard &, const olm_cuda_results_t &res, bool several) {
    const uint64_t at = all;
    all += res.count;
    if (!several || !f.no_overlap || !res.count) return 0;
    // grown geometrically (each growth copies what is there; it is not ordered after the stream's copies)
    const size_t need = all * sizeof(Record);
    if (need > E.gather.cap &&
        (cudaStreamSynchronize(E.stream) != cudaSuccess || E.gather.ensure(std::max(need, 2 * E.gather.cap), true)))
      return -1;
    OLM_CUDA(cudaMemcpyAsync(static_cast<Record *>(E.gather.p) + at, res.records, res.count * sizeof(Record),
                             cudaMemcpyDeviceToDevice, E.stream));
    return 0;
  });
  if (spans <= 0) return spans;
  if (f.no_overlap && spans > 1 && all) {
    const int64_t kept = no_overlap_inplace(E.gather.p, all);
    if (kept < 0 || count_records_to_host(E.gather.p, uint64_t(kept), counts) != 0) return -1;
    *total = uint64_t(kept);
    return 0;
  }
  if (add_counts_to_host(counts) != 0) return -1;
  *total = all;
  return 0;
}

int Engine::count_records_to_host(const void *dev_records, uint64_t count, uint64_t *counts) {
  OLM_CUDA(cudaSetDevice(impl_->device));
  unsigned long long *d = zeroed_counts();
  if (!d || count_records(dev_records, count, d) != 0) return -1;
  return add_counts_to_host(counts);
}

// ---- lines (lines.cuh, include/olm_b200.h "lines")

namespace {
// the pass between ev[2] and ev[3] is part of the call's device time
void add_pass_time(EngineImpl &E, uint32_t launches) {
  float ms = 0.f;
  cudaEventElapsedTime(&ms, E.ev[2], E.ev[3]);
  E.last.total_ms += ms;
  E.last.kernel_launches += launches;
}
bool bytes_unaligned(const void *p) {
  if (!(reinterpret_cast<uintptr_t>(p) & 15)) return false;
  std::fprintf(stderr, "libomega_match(b200): the device bytes of a line pass must be 16-byte aligned\n");
  return true;
}
} // namespace

const void *Engine::resident_haystack() const { return impl_->hay.p; }

void *Engine::positions_buffer(size_t bytes, int which) {
  DevBuf &b = which ? impl_->d_pos_gather : impl_->d_pos;
  if (cudaSetDevice(impl_->device) != cudaSuccess || b.ensure(std::max<size_t>(bytes, 16))) return nullptr;
  return b.p;
}

int Engine::copy_to_host(void *host_dst, const void *dev_src, size_t bytes) {
  OLM_CUDA(cudaSetDevice(impl_->device));
  if (bytes) OLM_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, impl_->stream));
  return 0;
}

int Engine::newline_facts(const void *dev_bytes, uint64_t len, olm_newline_facts_t *out) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (!out || (len && !dev_bytes) || bytes_unaligned(dev_bytes)) return -1;
  OLM_CUDA(cudaDeviceSynchronize()); // the bytes may come from any stream (see no_overlap_inplace)
  MiscWords *w = misc_words(E);
  if (!w || E.d_tiles.ensure(line_tiles_bytes(len))) return -1;
  uint32_t launches = 0;
  NewlineFacts f{};
  OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
  OLM_CUDA(newline_facts_launch(static_cast<const uint8_t *>(dev_bytes), len, E.d_tiles.p, &w->newline_facts, E.stream,
                                &launches));
  OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
  OLM_CUDA(cudaMemcpyAsync(&f, &w->newline_facts, sizeof f, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  add_pass_time(E, launches);
  *out = olm_newline_facts_t{f.newlines, f.first, f.last};
  return 0;
}

int Engine::line_positions(const void *dev_records, uint64_t count, const void *dev_bytes, uint64_t bytes_begin,
                           uint64_t len, const olm_line_origin_t &origin, void *dev_positions, bool tiles_ready) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (count == 0) return 0;
  if (!dev_records || !dev_positions || (len && !dev_bytes) || bytes_unaligned(dev_bytes)) return -1;
  if (!tiles_ready) {
    olm_newline_facts_t f;
    if (newline_facts(dev_bytes, len, &f) != 0) return -1;
  } else {
    OLM_CUDA(cudaDeviceSynchronize());
  }
  MiscWords *w = misc_words(E);
  if (!w) return -1;
  uint32_t launches = 0;
  unsigned long long outside = 0;
  OLM_CUDA(cudaMemsetAsync(&w->records_outside, 0, sizeof outside, E.stream));
  OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
  OLM_CUDA(line_positions_launch(static_cast<const Record *>(dev_records), count, static_cast<const uint8_t *>(dev_bytes),
                                 bytes_begin, len, E.d_tiles.p, LineOrigin{origin.line, origin.begin, origin.next_newline},
                                 static_cast<LinePos *>(dev_positions), &w->records_outside, E.stream, &launches));
  OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
  OLM_CUDA(cudaMemcpyAsync(&outside, &w->records_outside, sizeof outside, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  add_pass_time(E, launches);
  if (outside) {
    std::fprintf(stderr, "libomega_match(b200): line positions: records outside the bytes [%llu, %llu) (or not in offset order)\n",
                 (unsigned long long)bytes_begin, (unsigned long long)(bytes_begin + len));
    return -1;
  }
  return 0;
}

int Engine::matching_lines(const void *dev_positions, uint64_t count, void **dev_lines, uint64_t *n_lines) {
  EngineImpl &E = *impl_;
  OLM_CUDA(cudaSetDevice(E.device));
  if (!dev_lines || !n_lines || (count && !dev_positions)) return -1;
  *dev_lines = nullptr;
  *n_lines = 0;
  OLM_CUDA(cudaDeviceSynchronize());
  MiscWords *w = misc_words(E);
  if (!w || E.d_lines.ensure(std::max<uint64_t>(count, 1) * sizeof(LineEntry)) ||
      E.d_lscratch.ensure(matching_lines_scratch_bytes(count)))
    return -1;
  uint32_t launches = 0;
  unsigned long long m = 0;
  OLM_CUDA(cudaEventRecord(E.ev[2], E.stream));
  OLM_CUDA(matching_lines_launch(static_cast<const LinePos *>(dev_positions), count, static_cast<LineEntry *>(E.d_lines.p),
                                 E.d_lscratch.p, &w->matching_lines, E.stream, &launches));
  OLM_CUDA(cudaEventRecord(E.ev[3], E.stream));
  OLM_CUDA(cudaMemcpyAsync(&m, &w->matching_lines, sizeof m, cudaMemcpyDeviceToHost, E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  add_pass_time(E, launches);
  *dev_lines = E.d_lines.p;
  *n_lines = m;
  return 0;
}

// device records + positions -> host arrays (out->results / positions), or only their matching lines
int Engine::lines_to_host(const void *dev_records, const void *dev_positions, uint64_t count, bool lines_only,
                          LinesResult *out) {
  EngineImpl &E = *impl_;
  out->total = count;
  void *dl = nullptr;
  uint64_t m = 0;
  if (lines_only && count && matching_lines(dev_positions, count, &dl, &m) != 0) return -1;
  if (lines_only) {
    out->lines = static_cast<olm_line_t *>(host_result_alloc(m * sizeof(olm_line_t)));
    out->n_lines = m;
  } else {
    out->results = host_results(count);
    out->positions = static_cast<olm_line_pos_t *>(host_result_alloc(count * sizeof(olm_line_pos_t)));
  }
  if (lines_only ? !out->lines : (!out->results || !out->positions)) return -1;
  if (lines_only ? m == 0 : count == 0) return 0;
  float ms = 0.f;
  OLM_CUDA(cudaEventRecord(E.ev[6], E.stream));
  if (lines_only) {
    OLM_CUDA(cudaMemcpyAsync(out->lines, dl, m * sizeof(olm_line_t), cudaMemcpyDeviceToHost, E.stream));
  } else {
    OLM_CUDA(cudaMemcpyAsync(out->results->matches, dev_records, count * sizeof(Record), cudaMemcpyDeviceToHost, E.stream));
    OLM_CUDA(cudaMemcpyAsync(out->positions, dev_positions, count * sizeof(LinePos), cudaMemcpyDeviceToHost, E.stream));
  }
  OLM_CUDA(cudaEventRecord(E.ev[7], E.stream));
  OLM_CUDA(cudaStreamSynchronize(E.stream));
  cudaEventElapsedTime(&ms, E.ev[6], E.ev[7]);
  E.last.d2h_ms = ms;
  return 0;
}

// match_host with positions.  Several spans: a span's line and line start carry in from the spans before
// it; the records on its last line get their end from the first later span that holds a '\n' (or n).
// With no_overlap, or for the matching lines, their concatenation goes back to the device.
int Engine::lines_host(const uint8_t *haystack, size_t n, const MatchFlags &f, bool lines_only, LinesResult *out) {
  EngineImpl &E = *impl_;
  *out = LinesResult{};
  std::vector<Record> all; // several spans: records and positions concatenated on the host
  std::vector<LinePos> pos;
  uint64_t line = 0, begin = 0;
  size_t pending = 0; // pos[pending, size()) lie on a line no span so far has ended
  const int spans = host_spans(haystack, n, f, nullptr, [&](const Shard &s, const olm_cuda_results_t &d, bool several) {
    const uint8_t *own = static_cast<const uint8_t *>(E.hay.p) + (s.own_begin - s.slice_begin);
    const uint64_t len = s.own_end - s.own_begin;
    olm_newline_facts_t nf{}; // (one span: line_positions takes the facts itself, and only for records)
    if (several && newline_facts(own, len, &nf) != 0) return -1;
    void *dp = nullptr;
    const olm_line_origin_t origin{line, begin, s.own_end == n ? n : kNoNewline};
    if (d.count && (!(dp = positions_buffer(d.count * sizeof(LinePos), 0)) ||
                    line_positions(d.records, d.count, own, s.own_begin, len, origin, dp, several) != 0))
      return -1;
    if (!several) return lines_to_host(d.records, dp, d.count, lines_only, out);
    const size_t at = all.size();
    if (d.count) {
      all.resize(at + d.count);
      pos.resize(at + d.count);
      if (copy_to_host(all.data() + at, d.records, d.count * sizeof(Record)) != 0 ||
          copy_to_host(pos.data() + at, dp, d.count * sizeof(LinePos)) != 0 || sync() != 0)
        return -1;
    }
    if (nf.newlines) {
      for (size_t i = pending; i < at; ++i) pos[i].end = s.own_begin + nf.first;
      pending = pos.size();
      while (pending > at && pos[pending - 1].end == kNoNewline) --pending;
      line += nf.newlines;
      begin = s.own_begin + nf.last + 1;
    }
    return 0;
  });
  if (spans < 0) return -1;
  if (spans == 1) return 0;
  for (size_t i = pending; i < pos.size(); ++i) pos[i].end = n;
  uint64_t total = all.size();
  if ((f.no_overlap && total > 1) || (lines_only && total)) {
    void *dp = positions_buffer(total * sizeof(LinePos), 0);
    if (!dp || E.out.ensure(total * sizeof(Record))) return -1;
    OLM_CUDA(cudaMemcpyAsync(E.out.p, all.data(), total * sizeof(Record), cudaMemcpyHostToDevice, E.stream));
    OLM_CUDA(cudaMemcpyAsync(dp, pos.data(), total * sizeof(LinePos), cudaMemcpyHostToDevice, E.stream));
    if (f.no_overlap && total > 1) {
      const int64_t kept = no_overlap_inplace(E.out.p, total, dp);
      if (kept < 0) return -1;
      total = uint64_t(kept);
    }
    return lines_to_host(E.out.p, dp, total, lines_only, out);
  }
  if (lines_only) return lines_to_host(nullptr, nullptr, 0, true, out);
  out->total = total;
  out->results = host_results(total);
  out->positions = static_cast<olm_line_pos_t *>(host_result_alloc(total * sizeof(olm_line_pos_t)));
  if (!out->results || !out->positions) return -1;
  if (total) {
    std::memcpy(out->results->matches, all.data(), total * sizeof(Record));
    std::memcpy(out->positions, pos.data(), total * sizeof(LinePos));
  }
  return 0;
}

void Engine::collect_stats(omega_match_stats_t *s) {
  if (!s) return;
  EngineImpl &E = *impl_;
  { // spans of a host haystack before the last one (host_spans); normally all zero
    s->total_attempts += E.span_acc.total_attempts;
    s->total_filtered += E.span_acc.total_filtered;
    s->total_misses += E.span_acc.total_misses;
    s->total_hits += E.span_acc.total_hits;
    s->total_comparisons += E.span_acc.total_comparisons;
    E.span_acc = omega_match_stats_t{};
  }
  // counters written by the scan: [0] hits (key slots found + short matches accepted)
  // [1] misses (short candidates rejected by a predicate)  [2] comparisons  [3] key slots found
  if (E.stats_valid) {
    // exact (stats.cuh): the long path as core_match() counts it (matcher.c:783-799, :210),
    // the short matcher's hits and misses (:818-877) from the scan
    s->total_attempts += E.stat_counters[kStatAttempts];
    s->total_filtered += E.stat_counters[kStatFiltered];
    s->total_misses += E.stat_counters[kStatLongMisses] + E.counters[1];
    s->total_hits += E.stat_counters[kStatLongHits] + (E.counters[0] - E.counters[3]);
    s->total_comparisons += E.stat_counters[kStatComparisons];
    return;
  }
  s->total_hits += E.counters[0];
  s->total_misses += E.counters[1];
  s->total_comparisons += E.counters[2];
  s->total_attempts += E.attempts_last;
  const uint64_t long_hits = E.counters[3];
  s->total_filtered += E.attempts_last > long_hits ? E.attempts_last - long_hits : 0;
}

} // namespace olm
