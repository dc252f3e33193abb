// block_scan.cuh -- the block-wide scans of the post-scan passes (filters.cu, lines.cu): a
// 256-thread exclusive scan under any associative operator, and the three-phase scan over many
// blocks -- per-block aggregate, one-block scan of the aggregates, per-block finish.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace olm {

namespace {

constexpr int kFThreads = 256;
constexpr int kFItems = 8;
constexpr int kFBlock = kFThreads * kFItems; // items per block
constexpr uint32_t kFull = 0xFFFFFFFFu;

struct MaxOp {
  __device__ static unsigned long long identity() { return 0ull; }
  __device__ static unsigned long long apply(unsigned long long a, unsigned long long b) { return a > b ? a : b; }
};
struct SumOp {
  __device__ static unsigned long long identity() { return 0ull; }
  __device__ static unsigned long long apply(unsigned long long a, unsigned long long b) { return a + b; }
};
struct MinOp {
  __device__ static unsigned long long identity() { return ~0ull; }
  __device__ static unsigned long long apply(unsigned long long a, unsigned long long b) { return a < b ? a : b; }
};

template <typename Op>
__device__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long *total) {
  __shared__ unsigned long long s_w[kFThreads / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long t = __shfl_up_sync(kFull, incl, d);
    if (lane >= (uint32_t)d) incl = Op::apply(incl, t);
  }
  unsigned long long excl = __shfl_up_sync(kFull, incl, 1);
  if (lane == 0) excl = Op::identity();
  __syncthreads();
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  unsigned long long pre = Op::identity(), all = Op::identity();
#pragma unroll
  for (int w = 0; w < kFThreads / 32; ++w) {
    if ((uint32_t)w < warp) pre = Op::apply(pre, s_w[w]);
    all = Op::apply(all, s_w[w]);
  }
  *total = all;
  return Op::apply(pre, excl);
}

// phase 1 of a scan: per-block aggregate of value(i)
template <typename Op, typename F>
__device__ void block_aggregate(uint64_t n, unsigned long long *agg, F value) {
  const uint64_t base = (uint64_t)blockIdx.x * kFBlock + (uint64_t)threadIdx.x * kFItems;
  unsigned long long a = Op::identity();
#pragma unroll
  for (int k = 0; k < kFItems; ++k)
    if (base + k < n) a = Op::apply(a, value(base + k));
  unsigned long long total;
  block_exclusive_scan<Op>(a, &total);
  if (threadIdx.x == 0) agg[blockIdx.x] = total;
}

// phase 2: exclusive scan of the block aggregates by ONE block (in place); total -> *out_total
template <typename Op>
__global__ void __launch_bounds__(kFThreads) aggregate_scan_kernel(unsigned long long *agg, uint64_t n_blocks,
                                                                   unsigned long long *out_total) {
  unsigned long long carry = Op::identity();
  for (uint64_t base = 0; base < n_blocks; base += kFThreads) {
    const uint64_t i = base + threadIdx.x;
    const unsigned long long v = i < n_blocks ? agg[i] : Op::identity();
    unsigned long long total;
    const unsigned long long excl = block_exclusive_scan<Op>(v, &total);
    if (i < n_blocks) agg[i] = Op::apply(carry, excl);
    carry = Op::apply(carry, total);
    __syncthreads();
  }
  if (threadIdx.x == 0 && out_total) *out_total = carry;
}

} // namespace

} // namespace olm
