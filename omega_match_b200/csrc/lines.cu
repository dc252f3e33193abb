// lines.cu -- the line passes: newline facts of a byte range, the line of every record, and the
// matching lines of a call (include/olm_b200.h "lines").
//
// A line ends at a '\n' byte and at nothing else.  The range is cut into 64 KiB tiles.
//   newline_tiles_kernel      one block per tile reads it once (16-byte streaming loads) and keeps
//                             {count, first, last} of its '\n' bytes (byte compares, popc/ffs/clz).
//   newline_scan_*_kernel     three-phase scan over the tiles (block_scan.cuh): newlines before the
//                             tile (sum), the last '\n' before it (max), the first '\n' after it
//                             (min, from the right); the top phase also gives the range's facts.
//   tile_starts_kernel        one thread per tile edge: the first record at or after it (binary
//                             search; the records are in offset order).
//   line_positions_kernel     one block per tile that holds records.  A tile without '\n' answers
//                             its records from the scan alone.  Otherwise the block reads the tile
//                             again into a shared-memory bitmap (one bit per byte) with, per 32-bit
//                             word, the newlines before it, the last '\n' before it and the first
//                             after it (block scans), and answers every record in O(1): popc for the
//                             line, clz for its start, ffs for its end, the tile scan for what lies
//                             outside the tile.  A long line costs nothing per byte of its length.
//   matching_lines_*          run-length encoding of the positions by line: head flags, a scan of
//                             their count and a compaction, then the records per entry from the
//                             distance between heads.
// The second read touches only tiles that hold records and contain a '\n'.
#include "lines.cuh"

#include <algorithm>

#include "block_scan.cuh"

namespace olm {

namespace {

constexpr uint32_t kLineTileWords = kLineTileBytes / 32;     // 32 bytes per bitmap word
constexpr uint32_t kWordsPerThread = kLineTileWords / kFThreads;
constexpr uint32_t kNone32 = 0xFFFFFFFFu;
static_assert(kWordsPerThread * kFThreads == kLineTileWords, "a block covers its tile");

struct TileFacts { // in-tile byte positions; `last` is the position + 1 (0: none), `first` kNone32: none
  uint32_t count, first, last;
};
struct TileScan { // positions relative to the range
  unsigned long long before;     // '\n' bytes in the tiles before
  unsigned long long last1;      // last '\n' before the tile + 1, 0: none
  unsigned long long next_first; // first '\n' after the tile, kNoNewline: none
};
using TileAgg = TileScan; // per block of kFBlock tiles: {sum, max last1, min first}, then their scan

struct TileLayout {
  TileFacts *facts;
  TileScan *scan;
  TileAgg *agg;
  unsigned long long *starts; // tiles + 1 entries
};

__host__ __device__ inline uint64_t align256(uint64_t x) { return (x + 255) & ~uint64_t(255); }
__host__ __device__ inline uint64_t n_tiles(uint64_t len) { return (len + kLineTileBytes - 1) / kLineTileBytes; }
__host__ __device__ inline uint64_t n_tile_blocks(uint64_t tiles) { return (tiles + kFBlock - 1) / kFBlock; }

TileLayout layout(void *p, uint64_t len) {
  const uint64_t t = n_tiles(len);
  uint8_t *b = static_cast<uint8_t *>(p);
  TileLayout L;
  L.facts = reinterpret_cast<TileFacts *>(b);
  b += align256(t * sizeof(TileFacts));
  L.scan = reinterpret_cast<TileScan *>(b);
  b += align256(t * sizeof(TileScan));
  L.agg = reinterpret_cast<TileAgg *>(b);
  b += align256(n_tile_blocks(t) * sizeof(TileAgg));
  L.starts = reinterpret_cast<unsigned long long *>(b);
  return L;
}

// bit k: byte k of the word x is '\n'
__device__ __forceinline__ uint32_t nl_bits4(uint32_t x) {
  const uint32_t m = __vcmpeq4(x, 0x0A0A0A0Au);
  return ((m & 0x01010101u) * 0x01020408u) >> 24;
}
__device__ __forceinline__ uint32_t nl_bits16(uint4 v) {
  return nl_bits4(v.x) | nl_bits4(v.y) << 4 | nl_bits4(v.z) << 8 | nl_bits4(v.w) << 12;
}

// The bitmap words w = threadIdx.x + k * kFThreads of the tile at t0: bit j of word w is byte
// t0 + 32 w + j; bytes at or past len read as no '\n'.
__device__ __forceinline__ void load_tile_words(const uint8_t *__restrict__ bytes, uint64_t len, uint64_t t0,
                                                uint32_t (&m)[kWordsPerThread]) {
  if (t0 + kLineTileBytes <= len) {
    const uint4 *q = reinterpret_cast<const uint4 *>(bytes + t0);
    uint4 v[2 * kWordsPerThread];
#pragma unroll
    for (uint32_t k = 0; k < kWordsPerThread; ++k) {
      const uint32_t w = threadIdx.x + k * kFThreads;
      v[2 * k] = __ldcs(q + 2 * w);
      v[2 * k + 1] = __ldcs(q + 2 * w + 1);
    }
#pragma unroll
    for (uint32_t k = 0; k < kWordsPerThread; ++k) m[k] = nl_bits16(v[2 * k]) | nl_bits16(v[2 * k + 1]) << 16;
    return;
  }
  for (uint32_t k = 0; k < kWordsPerThread; ++k) {
    const uint64_t p = t0 + 32ull * (threadIdx.x + k * kFThreads);
    uint32_t w = 0;
    if (p + 32 <= len) {
      const uint4 *q = reinterpret_cast<const uint4 *>(bytes + p);
      w = nl_bits16(__ldcs(q)) | nl_bits16(__ldcs(q + 1)) << 16;
    } else {
      for (uint32_t j = 0; p + j < len && j < 32; ++j) w |= uint32_t(bytes[p + j] == '\n') << j;
    }
    m[k] = w;
  }
}

__global__ void __launch_bounds__(kFThreads) newline_tiles_kernel(const uint8_t *__restrict__ bytes, uint64_t len,
                                                                  TileFacts *facts) {
  __shared__ uint32_t s_red[3][kFThreads / 32];
  const uint64_t t0 = uint64_t(blockIdx.x) * kLineTileBytes;
  uint32_t m[kWordsPerThread];
  load_tile_words(bytes, len, t0, m);
  uint32_t cnt = 0, first = kNone32, last = 0;
#pragma unroll
  for (uint32_t k = 0; k < kWordsPerThread; ++k) {
    if (!m[k]) continue;
    const uint32_t w = threadIdx.x + k * kFThreads;
    cnt += __popc(m[k]);
    first = min(first, 32 * w + __ffs(m[k]) - 1);
    last = max(last, 32 * w + 32 - __clz(m[k])); // position + 1
  }
  cnt = __reduce_add_sync(kFull, cnt);
  first = __reduce_min_sync(kFull, first);
  last = __reduce_max_sync(kFull, last);
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    s_red[0][warp] = cnt;
    s_red[1][warp] = first;
    s_red[2][warp] = last;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    TileFacts f{0, kNone32, 0};
    for (int w = 0; w < kFThreads / 32; ++w) {
      f.count += s_red[0][w];
      f.first = min(f.first, s_red[1][w]);
      f.last = max(f.last, s_red[2][w]);
    }
    facts[blockIdx.x] = f;
  }
}

// a tile's facts in range coordinates: {count, last + 1 (0: none), first (kNoNewline: none)}
__device__ __forceinline__ TileScan tile_values(const TileFacts *facts, uint64_t t) {
  const TileFacts f = facts[t];
  const unsigned long long t0 = t * kLineTileBytes;
  return TileScan{f.count, f.last ? t0 + f.last : 0ull, f.first != kNone32 ? t0 + f.first : kNoNewline};
}

// Exclusive scans of one value per thread over the block: sum and max in thread order, min in
// reverse thread order (over the threads after this one).  Totals -> *total.
__device__ TileScan block_scan3(const TileScan &v, TileScan *total) {
  __shared__ unsigned long long s_rev[kFThreads];
  TileScan r, t;
  r.before = block_exclusive_scan<SumOp>(v.before, &t.before);
  r.last1 = block_exclusive_scan<MaxOp>(v.last1, &t.last1);
  s_rev[kFThreads - 1 - threadIdx.x] = v.next_first;
  __syncthreads();
  const unsigned long long ex = block_exclusive_scan<MinOp>(s_rev[threadIdx.x], &t.next_first);
  __syncthreads();
  s_rev[kFThreads - 1 - threadIdx.x] = ex;
  __syncthreads();
  r.next_first = s_rev[threadIdx.x];
  __syncthreads();
  *total = t;
  return r;
}

// phase 1: per block of kFBlock tiles, {sum, max, min}
__global__ void __launch_bounds__(kFThreads) newline_scan_aggregate_kernel(const TileFacts *facts, uint64_t tiles,
                                                                           TileAgg *agg) {
  const uint64_t base = uint64_t(blockIdx.x) * kFBlock + uint64_t(threadIdx.x) * kFItems;
  TileScan a{0, 0, kNoNewline};
  for (int k = 0; k < kFItems; ++k) {
    if (base + k >= tiles) break;
    const TileScan v = tile_values(facts, base + k);
    a.before += v.before;
    a.last1 = max(a.last1, v.last1);
    a.next_first = min(a.next_first, v.next_first);
  }
  TileScan total;
  block_scan3(a, &total);
  if (threadIdx.x == 0) agg[blockIdx.x] = total;
}

// phase 2 (one block): the aggregates' exclusive scans, in place; the range's facts
__global__ void __launch_bounds__(kFThreads) newline_scan_top_kernel(TileAgg *agg, uint64_t nb, NewlineFacts *d_facts) {
  unsigned long long sum = 0, last1 = 0, first = kNoNewline;
  for (uint64_t base = 0; base < nb; base += kFThreads) { // forward: sum, max
    const uint64_t i = base + threadIdx.x;
    const TileScan v = i < nb ? agg[i] : TileScan{0, 0, kNoNewline};
    unsigned long long ts, tl;
    const unsigned long long es = block_exclusive_scan<SumOp>(v.before, &ts);
    const unsigned long long el = block_exclusive_scan<MaxOp>(v.last1, &tl);
    if (i < nb) {
      agg[i].before = sum + es;
      agg[i].last1 = max(last1, el);
    }
    sum += ts;
    last1 = max(last1, tl);
    __syncthreads();
  }
  for (uint64_t base = 0; base < nb; base += kFThreads) { // backward: min
    const uint64_t j = base + threadIdx.x;
    const uint64_t i = nb - 1 - j;
    const unsigned long long v = j < nb ? agg[i].next_first : kNoNewline;
    unsigned long long tf;
    const unsigned long long ef = block_exclusive_scan<MinOp>(v, &tf);
    if (j < nb) agg[i].next_first = min(first, ef);
    first = min(first, tf);
    __syncthreads();
  }
  if (threadIdx.x == 0) *d_facts = NewlineFacts{sum, first, last1 ? last1 - 1 : kNoNewline};
}

// phase 3: per tile
__global__ void __launch_bounds__(kFThreads) newline_scan_finish_kernel(const TileFacts *facts, uint64_t tiles,
                                                                        const TileAgg *agg, TileScan *scan) {
  const uint64_t base = uint64_t(blockIdx.x) * kFBlock + uint64_t(threadIdx.x) * kFItems;
  TileScan v[kFItems];
  TileScan a{0, 0, kNoNewline};
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    v[k] = base + k < tiles ? tile_values(facts, base + k) : TileScan{0, 0, kNoNewline};
    a.before += v[k].before;
    a.last1 = max(a.last1, v[k].last1);
    a.next_first = min(a.next_first, v[k].next_first);
  }
  TileScan total;
  TileScan ex = block_scan3(a, &total);
  const TileAgg c = agg[blockIdx.x];
  unsigned long long before = c.before + ex.before, last1 = max(c.last1, ex.last1);
  unsigned long long first = min(c.next_first, ex.next_first);
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    if (base + k < tiles) scan[base + k] = TileScan{before, last1, 0};
    before += v[k].before;
    last1 = max(last1, v[k].last1);
  }
#pragma unroll
  for (int k = kFItems - 1; k >= 0; --k) {
    if (base + k < tiles) scan[base + k].next_first = first;
    first = min(first, v[k].next_first);
  }
}

// starts[t] = the first record with offset >= bytes_begin + t * tile (t < tiles), starts[tiles] = the
// first with offset >= bytes_begin + len.  Records before the range or behind it -> *d_outside.
__global__ void __launch_bounds__(kFThreads) tile_starts_kernel(const Record *rec, uint64_t n, uint64_t bytes_begin,
                                                                uint64_t len, uint64_t tiles,
                                                                unsigned long long *starts,
                                                                unsigned long long *d_outside) {
  const uint64_t t = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t > tiles) return;
  const uint64_t key = bytes_begin + (t < tiles ? t * kLineTileBytes : len);
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = lo + ((hi - lo) >> 1);
    if (rec[mid].offset < key) lo = mid + 1;
    else hi = mid;
  }
  starts[t] = lo;
  if ((t == 0 && lo != 0) || (t == tiles && lo != n)) atomicAdd(d_outside, t == 0 ? lo : n - lo);
}

__global__ void __launch_bounds__(kFThreads) line_positions_kernel(const Record *__restrict__ rec,
                                                                   const uint8_t *__restrict__ bytes,
                                                                   uint64_t bytes_begin, uint64_t len,
                                                                   TileLayout L, LineOrigin origin, LinePos *out,
                                                                   unsigned long long *d_outside) {
  __shared__ uint32_t s_bm[kLineTileWords], s_pre[kLineTileWords], s_last1[kLineTileWords], s_first[kLineTileWords];
  const uint64_t t = blockIdx.x;
  const uint64_t r0 = L.starts[t], r1 = L.starts[t + 1];
  if (r1 <= r0) return;
  const uint64_t t0 = t * kLineTileBytes;
  const TileScan s = L.scan[t];
  const unsigned long long line0 = origin.line + s.before;
  const unsigned long long begin_in = s.last1 ? bytes_begin + s.last1 : origin.begin;
  const unsigned long long end_out = s.next_first != kNoNewline ? bytes_begin + s.next_first : origin.next_newline;
  const unsigned long long tile_g = bytes_begin + t0; // global offset of the tile's first byte
  if (L.facts[t].count == 0) {
    for (uint64_t i = r0 + threadIdx.x; i < r1; i += kFThreads) {
      const uint64_t p = rec[i].offset - tile_g;
      if (p >= kLineTileBytes) { // (records out of order)
        atomicAdd(d_outside, 1ull);
        continue;
      }
      out[i] = LinePos{line0, begin_in, end_out};
    }
    return;
  }
  {
    uint32_t m[kWordsPerThread];
    load_tile_words(bytes, len, t0, m);
#pragma unroll
    for (uint32_t k = 0; k < kWordsPerThread; ++k) s_bm[threadIdx.x + k * kFThreads] = m[k];
  }
  __syncthreads();
  // thread i: words [8 i, 8 i + 8)
  const uint32_t w0 = threadIdx.x * kWordsPerThread;
  TileScan a{0, 0, kNoNewline};
#pragma unroll
  for (uint32_t k = 0; k < kWordsPerThread; ++k) {
    const uint32_t x = s_bm[w0 + k];
    if (!x) continue;
    a.before += __popc(x);
    a.last1 = max(a.last1, (unsigned long long)(32 * (w0 + k) + 32 - __clz(x)));
    a.next_first = min(a.next_first, (unsigned long long)(32 * (w0 + k) + __ffs(x) - 1));
  }
  TileScan total;
  const TileScan ex = block_scan3(a, &total);
  {
    uint32_t before = uint32_t(ex.before), last1 = uint32_t(ex.last1);
    uint32_t first = ex.next_first == kNoNewline ? kNone32 : uint32_t(ex.next_first);
#pragma unroll
    for (uint32_t k = 0; k < kWordsPerThread; ++k) {
      const uint32_t x = s_bm[w0 + k];
      s_pre[w0 + k] = before;
      s_last1[w0 + k] = last1;
      before += __popc(x);
      if (x) last1 = 32 * (w0 + k) + 32 - __clz(x);
    }
#pragma unroll
    for (int k = kWordsPerThread - 1; k >= 0; --k) {
      const uint32_t x = s_bm[w0 + k];
      s_first[w0 + k] = first;
      if (x) first = 32 * (w0 + k) + __ffs(x) - 1;
    }
  }
  __syncthreads();
  for (uint64_t i = r0 + threadIdx.x; i < r1; i += kFThreads) {
    const uint64_t p = rec[i].offset - tile_g;
    if (p >= kLineTileBytes) {
      atomicAdd(d_outside, 1ull);
      continue;
    }
    const uint32_t w = uint32_t(p >> 5), b = uint32_t(p & 31);
    const uint32_t x = s_bm[w];
    const uint32_t below = x & ((1u << b) - 1u), from = x & ~((1u << b) - 1u);
    LinePos q;
    q.line = line0 + s_pre[w] + __popc(below);
    if (below) q.begin = tile_g + 32 * w + 32 - __clz(below);
    else q.begin = s_last1[w] ? tile_g + s_last1[w] : begin_in;
    if (from) q.end = tile_g + 32 * w + __ffs(from) - 1;
    else q.end = s_first[w] != kNone32 ? tile_g + s_first[w] : end_out;
    out[i] = q;
  }
}

// ---- matching lines

__device__ __forceinline__ bool line_head(const LinePos *pos, uint64_t i) {
  return i == 0 || pos[i].line != pos[i - 1].line;
}

__global__ void __launch_bounds__(kFThreads) line_heads_aggregate_kernel(const LinePos *pos, uint64_t n,
                                                                         unsigned long long *agg) {
  block_aggregate<SumOp>(n, agg, [&](uint64_t i) { return (unsigned long long)line_head(pos, i); });
}

// heads -> out[k] = {line, begin, end, -}, head_at[k] = the head's record index
__global__ void __launch_bounds__(kFThreads) matching_lines_kernel(const LinePos *pos, uint64_t n,
                                                                   const unsigned long long *agg, LineEntry *out,
                                                                   unsigned long long *head_at) {
  const uint64_t base = uint64_t(blockIdx.x) * kFBlock + uint64_t(threadIdx.x) * kFItems;
  bool h[kFItems];
  unsigned long long a = 0;
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    h[k] = base + k < n && line_head(pos, base + k);
    a += h[k];
  }
  unsigned long long total;
  unsigned long long o = agg[blockIdx.x] + block_exclusive_scan<SumOp>(a, &total);
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    if (!h[k]) continue;
    const LinePos q = pos[base + k];
    out[o] = LineEntry{q.line, q.begin, q.end, 0};
    head_at[o++] = base + k;
  }
}

__global__ void __launch_bounds__(kFThreads) line_records_kernel(LineEntry *out, const unsigned long long *head_at,
                                                                 uint64_t n, const unsigned long long *d_count) {
  const uint64_t k = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t m = *d_count;
  if (k < m) out[k].records = (k + 1 < m ? head_at[k + 1] : n) - head_at[k];
}

} // namespace

size_t line_tiles_bytes(uint64_t len) {
  const uint64_t t = n_tiles(len);
  return align256(t * sizeof(TileFacts)) + align256(t * sizeof(TileScan)) + align256(n_tile_blocks(t) * sizeof(TileAgg)) +
         (t + 1) * sizeof(unsigned long long) + 256;
}

cudaError_t newline_facts_launch(const uint8_t *bytes, uint64_t len, void *tiles, NewlineFacts *d_facts,
                                 cudaStream_t st, uint32_t *launches) {
  if (len == 0) { // {0, none, none}
    const cudaError_t e = cudaMemsetAsync(d_facts, 0, sizeof *d_facts, st);
    return e != cudaSuccess ? e : cudaMemsetAsync(&d_facts->first, 0xFF, 2 * sizeof(unsigned long long), st);
  }
  const uint64_t t = n_tiles(len), nb = n_tile_blocks(t);
  const TileLayout L = layout(tiles, len);
  newline_tiles_kernel<<<(unsigned)t, kFThreads, 0, st>>>(bytes, len, L.facts);
  newline_scan_aggregate_kernel<<<(unsigned)nb, kFThreads, 0, st>>>(L.facts, t, L.agg);
  newline_scan_top_kernel<<<1, kFThreads, 0, st>>>(L.agg, nb, d_facts);
  newline_scan_finish_kernel<<<(unsigned)nb, kFThreads, 0, st>>>(L.facts, t, L.agg, L.scan);
  *launches += 4;
  return cudaGetLastError();
}

cudaError_t line_positions_launch(const Record *rec, uint64_t n, const uint8_t *bytes, uint64_t bytes_begin,
                                  uint64_t len, void *tiles, const LineOrigin &origin, LinePos *out,
                                  unsigned long long *d_outside, cudaStream_t st, uint32_t *launches) {
  if (n == 0) return cudaSuccess;
  if (len == 0) return cudaMemsetAsync(d_outside, 0xFF, sizeof *d_outside, st); // every record lies outside
  const uint64_t t = n_tiles(len);
  const TileLayout L = layout(tiles, len);
  tile_starts_kernel<<<(unsigned)((t + kFThreads) / kFThreads), kFThreads, 0, st>>>(rec, n, bytes_begin, len, t, L.starts,
                                                                                   d_outside);
  line_positions_kernel<<<(unsigned)t, kFThreads, 0, st>>>(rec, bytes, bytes_begin, len, L, origin, out, d_outside);
  *launches += 2;
  return cudaGetLastError();
}

size_t matching_lines_scratch_bytes(uint64_t n) {
  return align256(n * sizeof(unsigned long long)) + (n_tile_blocks(n) + 2) * sizeof(unsigned long long) + 256;
}

cudaError_t matching_lines_launch(const LinePos *pos, uint64_t n, LineEntry *out, void *scratch,
                                  unsigned long long *d_count, cudaStream_t st, uint32_t *launches) {
  if (n == 0) return cudaMemsetAsync(d_count, 0, sizeof *d_count, st);
  const uint64_t blocks = n_tile_blocks(n);
  unsigned long long *head_at = static_cast<unsigned long long *>(scratch);
  unsigned long long *agg = reinterpret_cast<unsigned long long *>(static_cast<uint8_t *>(scratch) +
                                                                   align256(n * sizeof(unsigned long long)));
  line_heads_aggregate_kernel<<<(unsigned)blocks, kFThreads, 0, st>>>(pos, n, agg);
  aggregate_scan_kernel<SumOp><<<1, kFThreads, 0, st>>>(agg, blocks, d_count);
  matching_lines_kernel<<<(unsigned)blocks, kFThreads, 0, st>>>(pos, n, agg, out, head_at);
  line_records_kernel<<<(unsigned)((n + kFThreads - 1) / kFThreads), kFThreads, 0, st>>>(out, head_at, n, d_count);
  *launches += 4;
  return cudaGetLastError();
}

} // namespace olm
