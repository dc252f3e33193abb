// cuda_util.cu -- small CUDA-facing entry points of the C ABI that do not belong to a matcher.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "../../include/olm_b200.h"
#include "engine.h"

namespace olm {

// Result arrays of the host API live in pinned memory when they are large: a D2H copy into
// freshly malloc'ed pageable memory runs at ~2 GB/s (page faults under the DMA), into pinned
// memory at PCIe speed.  Pinning is slow, so released blocks are kept for the next call;
// omega_match_results_destroy() hands them back here (it cannot know the matcher).
namespace {
struct PinnedBlock {
  void *p;
  size_t cap;
  bool busy;
};
std::mutex g_pin_mu;
std::vector<PinnedBlock> g_pin;
constexpr size_t kMaxIdleBlocks = 4;
constexpr size_t kPinnedResultMin = size_t(1) << 20;

void *pinned_result_alloc(size_t bytes) {
  std::lock_guard<std::mutex> lk(g_pin_mu);
  PinnedBlock *best = nullptr;
  for (auto &b : g_pin)
    if (!b.busy && b.cap >= bytes && (!best || b.cap < best->cap)) best = &b;
  if (best) {
    best->busy = true;
    return best->p;
  }
  void *p = nullptr;
  const size_t cap = bytes + bytes / 4 + (size_t(1) << 20);
  if (cudaHostAlloc(&p, cap, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  g_pin.push_back(PinnedBlock{p, cap, true});
  return p;
}

// false: not one of ours (plain malloc)
bool pinned_result_release(void *p) {
  std::lock_guard<std::mutex> lk(g_pin_mu);
  size_t idle = 0;
  PinnedBlock *mine = nullptr;
  for (auto &b : g_pin) {
    if (b.p == p) mine = &b;
    else if (!b.busy) ++idle;
  }
  if (!mine) return false;
  mine->busy = false;
  if (idle >= kMaxIdleBlocks) { // too many cached: give this one back to the driver
    cudaFreeHost(mine->p);
    *mine = g_pin.back();
    g_pin.pop_back();
  }
  return true;
}
} // namespace

void *host_result_alloc(size_t bytes) {
  void *p = bytes >= kPinnedResultMin ? pinned_result_alloc(bytes) : nullptr;
  return p ? p : std::malloc(std::max<size_t>(bytes, 1));
}

void host_result_free(void *p) {
  if (p && !pinned_result_release(p)) std::free(p);
}

omega_match_results_t *host_results(uint64_t count) {
  auto *r = static_cast<omega_match_results_t *>(std::malloc(sizeof(omega_match_results_t)));
  if (!r) return nullptr;
  r->count = count;
  r->matches = static_cast<omega_match_result_t *>(host_result_alloc(count * sizeof(omega_match_result_t)));
  if (!r->matches) {
    std::free(r);
    return nullptr;
  }
  return r;
}

} // namespace olm

extern "C" {

int olm_cuda_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

void *olm_cuda_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
  return p;
}

void olm_cuda_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

} // extern "C"
