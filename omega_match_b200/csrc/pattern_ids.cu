// pattern_ids.cu -- the pattern-id pass: which catalogue pattern (store.h PatternCatalog) each final
// record matched; and the counting pass, which adds up the records per pattern instead.
//
// One thread per record, grid-stride; records are in offset order, so neighbouring threads read
// neighbouring haystack bytes.  A thread normalises the record's source span on the fly (fold case,
// skip punctuation, collapse a whitespace run to one space -- transform_apply, transform_table.c:
// 36-88, WITHOUT its trailing-space trim, which belongs to the end of a window, not to a match),
// hashes the bytes, probes the lookup table and confirms a fingerprint hit by normalising the span
// once more against the catalogue's bytes.  The span's first and last source bytes are kept bytes
// (matcher.c:986-997) and the whitespace-run state in front of a kept byte is "not in a run", so
// the span normalises in isolation to exactly the bytes the window produced.  The walk costs one
// step per source byte: spans that hold long runs of skipped bytes cost in proportion.
#include "pattern_ids.cuh"

#include <algorithm>

#include "olm_classes.h"
#include "store.h"

namespace olm {

namespace {

constexpr int kIdThreads = 256;

// Normalises src[0, len) and hands every produced byte to `emit(index, byte)`; returns the number of
// bytes produced, or kNoPatternId as soon as `emit` returns false.
template <typename Emit>
__device__ __forceinline__ uint32_t normalise_span(const uint8_t *__restrict__ src, uint32_t len, bool ci, bool ip,
                                                   bool ew, Emit &&emit) {
  uint32_t n = 0;
  bool in_space = false;
  for (uint32_t i = 0; i < len; ++i) {
    uint32_t m;
    const ByteAction a = classify_byte(__ldg(src + i), ci, ip, ew, &m);
    if (a == kSkip) continue;
    if (a == kSpace) {
      if (in_space) continue;
      in_space = true;
    } else {
      in_space = false;
    }
    if (!emit(n, m)) return kNoPatternId;
    ++n;
  }
  return n;
}

// The id of the pattern the record at src[0, len) matched, or kNoPatternId.
__device__ __forceinline__ uint32_t resolve_pattern_id(const uint8_t *__restrict__ src, uint32_t len,
                                                       const PatternIdTables &T, bool ci, bool ip, bool ew) {
  uint64_t h = kPatternHashSeed;
  const uint32_t nlen = normalise_span(src, len, ci, ip, ew, [&](uint32_t, uint32_t m) {
    h = pattern_hash_step(h, m);
    return true;
  });
  h = pattern_hash_final(h, nlen);
  const uint32_t fp = pattern_fingerprint(h);
  for (uint32_t s = pattern_home(h, T.table_mask);; s = (s + 1) & T.table_mask) {
    const uint2 e = T.table[s];
    if (e.x == kNoPatternId) break;
    if (e.y != fp) continue;
    const uint2 r = T.refs[e.x];
    if (r.y != nlen) continue;
    const uint8_t *p = (r.y >= 5 ? T.store : T.short_bytes) + r.x;
    if (normalise_span(src, len, ci, ip, ew, [&](uint32_t j, uint32_t m) { return p[j] == m; }) == nlen) return e.x;
  }
  return kNoPatternId;
}

__global__ void __launch_bounds__(kIdThreads) pattern_id_kernel(Record *rec, uint64_t n, const uint8_t *buf,
                                                                 uint64_t buf_begin, PatternIdTables T,
                                                                 unsigned long long *d_missing) {
  const bool ci = T.store_flags & kFlagIgnoreCase, ip = T.store_flags & kFlagIgnorePunct,
             ew = T.store_flags & kFlagElideSpace;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const uint32_t id = resolve_pattern_id(buf + (rec[i].offset - buf_begin), rec[i].len, T, ci, ip, ew);
    rec[i]._pad = id;
    if (id == kNoPatternId) atomicAdd(d_missing, 1ull);
  }
}

// ---- counting: counts[id] += records of pattern id
//
// Each block takes one contiguous range of records, a block-wide step at a time, so that a warp's
// 32 records are neighbours in the text.  A warp first groups its lanes by id (MATCH.ANY) and the
// lowest lane of each group adds the group's size: one add per distinct id per warp step.  With the
// block table, that add goes to a per-block open-addressing table of ids in shared memory (32-bit
// counts, flushed with one global add per occupied slot when the block ends); an id that finds no
// slot within kCountProbes, like every add without the table, is a non-returning 64-bit global add.
// The table pays when ids repeat within a block's range (few patterns, many records); with about
// as many patterns as records it only adds work (pattern_counts_launch chooses).
constexpr int kCountThreads = 256;
constexpr int kCountTableLog2 = 11;
constexpr uint32_t kCountSlots = 1u << kCountTableLog2;
constexpr int kCountProbes = 8;
// records per catalogue pattern from which a call counts through the block table
constexpr uint64_t kCountTableMinRepeat = 64;

__device__ __forceinline__ void table_add(uint32_t *keys, uint32_t *cnt, uint32_t id, uint32_t c,
                                          unsigned long long *counts) {
  uint32_t s = (id * 0x9E3779B1u) >> (32 - kCountTableLog2);
  for (int p = 0; p < kCountProbes; ++p, s = (s + 1) & (kCountSlots - 1)) {
    uint32_t k = static_cast<volatile uint32_t *>(keys)[s]; // (a key once set never changes)
    if (k == kNoPatternId) k = atomicCAS(keys + s, kNoPatternId, id);
    if (k == kNoPatternId || k == id) {
      atomicAdd(cnt + s, c);
      return;
    }
  }
  atomicAdd(counts + id, (unsigned long long)c);
}

// kResolve: ids resolved from the haystack (buf, buf_begin as for pattern_id_kernel); else read
// from the pad words.  An id the catalogue does not have is counted into *d_missing, not into counts.
template <bool kResolve, bool kTable>
__global__ void __launch_bounds__(kCountThreads) pattern_count_kernel(const Record *__restrict__ rec, uint64_t n,
                                                                      uint64_t per_block, const uint8_t *buf,
                                                                      uint64_t buf_begin, PatternIdTables T,
                                                                      unsigned long long *counts,
                                                                      unsigned long long *d_missing) {
  __shared__ uint32_t keys[kTable ? kCountSlots : 1], cnt[kTable ? kCountSlots : 1];
  if (kTable) {
    for (uint32_t s = threadIdx.x; s < kCountSlots; s += blockDim.x) {
      keys[s] = kNoPatternId;
      cnt[s] = 0;
    }
    __syncthreads();
  }
  const bool ci = T.store_flags & kFlagIgnoreCase, ip = T.store_flags & kFlagIgnorePunct,
             ew = T.store_flags & kFlagElideSpace;
  const unsigned lane = threadIdx.x & 31;
  const uint64_t begin = uint64_t(blockIdx.x) * per_block, end = min(n, begin + per_block);
  for (uint64_t base = begin; base < end; base += blockDim.x) { // (block-uniform: every lane takes each step)
    const uint64_t i = base + threadIdx.x;
    uint32_t id = kNoPatternId;
    if (i < end) {
      id = kResolve ? resolve_pattern_id(buf + (rec[i].offset - buf_begin), rec[i].len, T, ci, ip, ew) : rec[i]._pad;
      if (id >= T.count) {
        atomicAdd(d_missing, 1ull);
        id = kNoPatternId;
      }
    }
    const unsigned same = __match_any_sync(0xFFFFFFFFu, id);
    if (id != kNoPatternId && lane == unsigned(__ffs(same) - 1)) {
      if (kTable) table_add(keys, cnt, id, __popc(same), counts);
      else atomicAdd(counts + id, (unsigned long long)__popc(same));
    }
  }
  if (kTable) {
    __syncthreads();
    for (uint32_t s = threadIdx.x; s < kCountSlots; s += blockDim.x)
      if (cnt[s]) atomicAdd(counts + keys[s], (unsigned long long)cnt[s]);
  }
}

} // namespace

cudaError_t pattern_ids_launch(Record *records, uint64_t n, const uint8_t *buf, uint64_t buf_begin,
                               const PatternIdTables &t, unsigned long long *d_missing, int sms,
                               cudaStream_t stream, uint32_t *launches) {
  if (n == 0) return cudaSuccess;
  const uint64_t blocks = std::min<uint64_t>((n + kIdThreads - 1) / kIdThreads, uint64_t(sms) * 16);
  pattern_id_kernel<<<(unsigned)blocks, kIdThreads, 0, stream>>>(records, n, buf, buf_begin, t, d_missing);
  ++*launches;
  return cudaGetLastError();
}

bool pattern_counts_block_table(uint64_t n, const PatternIdTables &t) {
  return n >= kCountTableMinRepeat * t.count;
}

cudaError_t pattern_counts_launch(const Record *records, uint64_t n, const uint8_t *buf, uint64_t buf_begin,
                                  const PatternIdTables &t, bool block_table, unsigned long long *counts,
                                  unsigned long long *d_missing, int sms, cudaStream_t stream, uint32_t *launches) {
  if (n == 0) return cudaSuccess;
  // one range per block; a block's table counts in 32 bits, so no range holds 2^31 records or more
  uint64_t blocks = std::min<uint64_t>((n + kCountThreads - 1) / kCountThreads, uint64_t(sms) * 16);
  blocks = std::max<uint64_t>(blocks, (n >> 31) + 1);
  const uint64_t per_block = (n + blocks - 1) / blocks;
  blocks = (n + per_block - 1) / per_block;
  auto kernel = buf ? (block_table ? pattern_count_kernel<true, true> : pattern_count_kernel<true, false>)
                    : (block_table ? pattern_count_kernel<false, true> : pattern_count_kernel<false, false>);
  kernel<<<(unsigned)blocks, kCountThreads, 0, stream>>>(records, n, per_block, buf, buf_begin, t, counts, d_missing);
  ++*launches;
  return cudaGetLastError();
}

} // namespace olm
