// pattern_ids.cu -- the pattern-id pass: which catalogue pattern (store.h PatternCatalog) each final
// record matched.
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

__global__ void __launch_bounds__(kIdThreads) pattern_id_kernel(Record *rec, uint64_t n, const uint8_t *buf,
                                                                 uint64_t buf_begin, PatternIdTables T,
                                                                 unsigned long long *d_missing) {
  const bool ci = T.store_flags & kFlagIgnoreCase, ip = T.store_flags & kFlagIgnorePunct,
             ew = T.store_flags & kFlagElideSpace;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
    const uint8_t *src = buf + (rec[i].offset - buf_begin);
    const uint32_t len = rec[i].len;
    uint64_t h = kPatternHashSeed;
    const uint32_t nlen = normalise_span(src, len, ci, ip, ew, [&](uint32_t, uint32_t m) {
      h = pattern_hash_step(h, m);
      return true;
    });
    h = pattern_hash_final(h, nlen);
    const uint32_t fp = pattern_fingerprint(h);
    uint32_t id = kNoPatternId;
    for (uint32_t s = pattern_home(h, T.table_mask);; s = (s + 1) & T.table_mask) {
      const uint2 e = T.table[s];
      if (e.x == kNoPatternId) break;
      if (e.y != fp) continue;
      const uint2 r = T.refs[e.x];
      if (r.y != nlen) continue;
      const uint8_t *p = (r.y >= 5 ? T.store : T.short_bytes) + r.x;
      if (normalise_span(src, len, ci, ip, ew, [&](uint32_t j, uint32_t m) { return p[j] == m; }) == nlen) {
        id = e.x;
        break;
      }
    }
    rec[i]._pad = id;
    if (id == kNoPatternId) atomicAdd(d_missing, 1ull);
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

} // namespace olm
