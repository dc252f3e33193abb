// filters.cu -- the post-scan filters on sorted device records (kernels K6/K7 of SURVEY 2.1).
//
// Reference: apply_filter / filter_longest / filter_no_overlap / finalize_match_results
// (omega_match/src/matcher.c:552-623), which walk the sorted match vector serially.
//
//   longest-only : "keep a record iff its offset differs from the previous KEPT record".
//                  On the single-GPU path this is fused into the scan (a position stops after
//                  its first accepted match); longest_flags_kernel is the stand-alone form,
//                  used on gathered shard results and by tests.
//   no-overlap   : "keep a record iff offset >= end of the previous KEPT record" -- a greedy
//                  chain.  With a floor, records that start before it are dropped and the chain
//                  starts at the first record at or past it (the records are sorted, so those are
//                  a prefix: one test per record finds it).  Parallel form (SURVEY H4): with E_i = max end over records < i,
//                  record i is a CERTAIN START iff E_i <= offset_i (nothing earlier reaches
//                  it, so it is kept whatever the chain did before).  Chains between certain
//                  starts are independent; each is walked by one thread with a galloping
//                  search for "first record starting at or after my end".  A chain never
//                  jumps over a certain start (its end is <= that start's offset).
//   compaction   : exclusive sum scan of the keep flags + scatter.
//
// The two scans (prefix max, prefix sum) are three-phase block scans: per-block aggregate,
// one-block scan of the aggregates, per-block finish.
#include "filters.cuh"

#include "block_scan.cuh"

namespace olm {

namespace {

__device__ __forceinline__ unsigned long long rec_end(const Record &r) { return r.offset + r.len; }

// (records below the floor reach nothing: their end counts as 0, the identity of the max)
__global__ void __launch_bounds__(kFThreads) end_max_aggregate_kernel(const Record *r, uint64_t n, uint64_t floor,
                                                                      unsigned long long *agg) {
  block_aggregate<MaxOp>(n, agg, [&](uint64_t i) { return r[i].offset >= floor ? rec_end(r[i]) : 0ull; });
}
__global__ void __launch_bounds__(kFThreads) keep_sum_aggregate_kernel(const uint8_t *keep, uint64_t n, unsigned long long *agg) {
  block_aggregate<SumOp>(n, agg, [&](uint64_t i) { return (unsigned long long)keep[i]; });
}

// phase 3 (prefix max): certain-start flags
__global__ void __launch_bounds__(kFThreads) certain_start_kernel(const Record *r, uint64_t n, uint64_t floor,
                                                                  const unsigned long long *agg, uint8_t *start) {
  const uint64_t base = (uint64_t)blockIdx.x * kFBlock + (uint64_t)threadIdx.x * kFItems;
  unsigned long long ends[kFItems], offs[kFItems];
  unsigned long long a = 0;
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    ends[k] = offs[k] = 0;
    if (base + k < n) {
      const Record x = r[base + k];
      offs[k] = x.offset;
      ends[k] = x.offset >= floor ? x.offset + x.len : 0;
      a = a > ends[k] ? a : ends[k];
    }
  }
  unsigned long long total;
  unsigned long long run = MaxOp::apply(agg[blockIdx.x], block_exclusive_scan<MaxOp>(a, &total));
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    if (base + k < n) {
      start[base + k] = (offs[k] >= floor && run <= offs[k]) ? 1 : 0;
      run = run > ends[k] ? run : ends[k];
    }
  }
}

// Walk one chain per certain start (matcher.c:552-561 restricted to the chain).
__global__ void __launch_bounds__(kFThreads) chain_walk_kernel(const Record *r, uint64_t n, const uint8_t *start,
                                                               uint8_t *keep) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !start[i]) return;
  uint64_t j = i;
  while (true) {
    keep[j] = 1;
    const unsigned long long e = r[j].offset + r[j].len;
    // first k > j with offset_k >= e: gallop, then bisect
    uint64_t lo = j + 1, step = 1;
    if (lo >= n) return;
    uint64_t hi = lo;
    while (hi < n && r[hi].offset < e) {
      lo = hi + 1;
      hi += step;
      step <<= 1;
    }
    if (hi > n) hi = n;
    while (lo < hi) { // invariant: answer in [lo, hi]
      const uint64_t mid = lo + ((hi - lo) >> 1);
      if (r[mid].offset < e) lo = mid + 1;
      else hi = mid;
    }
    if (lo >= n || start[lo]) return;
    j = lo;
  }
}

__global__ void __launch_bounds__(kFThreads) longest_flags_kernel(const Record *r, uint64_t n, uint8_t *keep) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) keep[i] = (i == 0 || r[i].offset != r[i - 1].offset) ? 1 : 0;
}

// phase 3 (prefix sum): scatter kept records (or the items of an array parallel to them)
template <typename T>
__global__ void __launch_bounds__(kFThreads) compact_kernel(const T *in, uint64_t n, const uint8_t *keep,
                                                            const unsigned long long *agg, T *out) {
  const uint64_t base = (uint64_t)blockIdx.x * kFBlock + (uint64_t)threadIdx.x * kFItems;
  uint32_t k8[kFItems];
  unsigned long long a = 0;
#pragma unroll
  for (int k = 0; k < kFItems; ++k) {
    k8[k] = (base + k < n) ? keep[base + k] : 0;
    a += k8[k];
  }
  unsigned long long total;
  unsigned long long o = agg[blockIdx.x] + block_exclusive_scan<SumOp>(a, &total);
#pragma unroll
  for (int k = 0; k < kFItems; ++k)
    if (k8[k]) out[o++] = in[base + k];
}

} // namespace

size_t filter_scratch_bytes(uint64_t n) {
  const uint64_t blocks = (n + kFBlock - 1) / kFBlock;
  // start flags + keep flags + block aggregates + total
  return size_t(n) * 2 + (blocks + 2) * sizeof(unsigned long long) + 64;
}

static cudaError_t compact(const Record *in, uint64_t n, const uint8_t *keep, unsigned long long *agg,
                           unsigned long long *d_total, Record *out, cudaStream_t st, uint32_t *launches) {
  const uint32_t blocks = uint32_t((n + kFBlock - 1) / kFBlock);
  keep_sum_aggregate_kernel<<<blocks, kFThreads, 0, st>>>(keep, n, agg);
  aggregate_scan_kernel<SumOp><<<1, kFThreads, 0, st>>>(agg, blocks, d_total);
  compact_kernel<<<blocks, kFThreads, 0, st>>>(in, n, keep, agg, out);
  *launches += 3;
  return cudaGetLastError();
}

cudaError_t no_overlap_launch(const Record *in, uint64_t n, Record *out, void *scratch,
                              unsigned long long *d_total, cudaStream_t st, uint32_t *launches, uint64_t floor,
                              const LinePos *in_pos, LinePos *out_pos) {
  if (n == 0) return cudaSuccess;
  const uint32_t blocks = uint32_t((n + kFBlock - 1) / kFBlock);
  uint8_t *start = static_cast<uint8_t *>(scratch);
  uint8_t *keep = start + n;
  unsigned long long *agg = reinterpret_cast<unsigned long long *>((reinterpret_cast<uintptr_t>(keep + n) + 63) & ~uintptr_t(63));
  cudaError_t e = cudaMemsetAsync(keep, 0, n, st);
  if (e != cudaSuccess) return e;
  end_max_aggregate_kernel<<<blocks, kFThreads, 0, st>>>(in, n, floor, agg);
  aggregate_scan_kernel<MaxOp><<<1, kFThreads, 0, st>>>(agg, blocks, nullptr);
  certain_start_kernel<<<blocks, kFThreads, 0, st>>>(in, n, floor, agg, start);
  chain_walk_kernel<<<uint32_t((n + kFThreads - 1) / kFThreads), kFThreads, 0, st>>>(in, n, start, keep);
  *launches += 4;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = compact(in, n, keep, agg, d_total, out, st, launches)) != cudaSuccess || !in_pos) return e;
  // the positions of the records: the same keep flags, the block offsets compact() left in agg
  compact_kernel<<<blocks, kFThreads, 0, st>>>(in_pos, n, keep, agg, out_pos);
  *launches += 1;
  return cudaGetLastError();
}

cudaError_t longest_launch(const Record *in, uint64_t n, Record *out, void *scratch,
                           unsigned long long *d_total, cudaStream_t st, uint32_t *launches) {
  if (n == 0) return cudaSuccess;
  uint8_t *keep = static_cast<uint8_t *>(scratch) + n;
  unsigned long long *agg = reinterpret_cast<unsigned long long *>((reinterpret_cast<uintptr_t>(keep + n) + 63) & ~uintptr_t(63));
  longest_flags_kernel<<<uint32_t((n + kFThreads - 1) / kFThreads), kFThreads, 0, st>>>(in, n, keep);
  *launches += 1;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return compact(in, n, keep, agg, d_total, out, st, launches);
}

} // namespace olm
