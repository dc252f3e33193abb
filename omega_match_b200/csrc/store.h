// store.h -- host view of a compiled store and the builder of its HBM layout.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "device_tables.h"
#include "olm_format.h"

namespace olm {

// Parsed (not copied) view of a mapped .olm file.  Reference reader: matcher.c:329-432.
struct StoreView {
  const uint8_t *base = nullptr;
  size_t size = 0;
  Header hdr;
  const uint8_t *patterns = nullptr; // hdr.store_bytes
  uint32_t bloom_bits = 0;
  const uint8_t *bloom = nullptr; // hdr.bloom_bytes
  const uint8_t *index = nullptr; // hdr.table_size * 4
  const uint8_t *blob = nullptr;  // hdr.blob_bytes
  const uint8_t *bitmap1 = nullptr, *bitmap2 = nullptr;
  uint32_t n1 = 0, n2 = 0, n3 = 0, n4 = 0;
  const uint8_t *arr3 = nullptr, *arr4 = nullptr;
};

// Returns an empty string on success, else what is wrong with the file.
std::string parse_store(const uint8_t *file, size_t size, StoreView *out);

// Host-side image of the device tables (device_tables.h), ready to be uploaded verbatim.
struct StagedStore {
  std::vector<uint4> keys;  // buckets of four grams
  std::vector<Slot> slots;  // 4 per bucket
  std::vector<Rec> recs;
  std::vector<uint8_t> store;
  std::vector<uint32_t> g4, p23, set3, bitmap2, sx;
  DeviceStore params; // pointer members are filled in after upload
  uint32_t n_keys = 0;
};

// Limits for the two shared-memory filters, in log2(bits).
struct FilterBudget {
#ifndef OLM_G4_MAX_LOG2
#define OLM_G4_MAX_LOG2 20
#endif
  uint32_t g4_max_log2 = OLM_G4_MAX_LOG2;  // 128 KiB
  uint32_t p23_max_log2 = 18; // 32 KiB
};

std::string stage_store(const StoreView &v, const FilterBudget &budget, StagedStore *out);

// Host image of the tables behind the exact statistics (stats.cuh): the file's Bloom bits as
// 64-bit words, its gram -> bucket map as an open-addressing table, the pattern lengths per bucket.
struct StagedStats {
  std::vector<unsigned long long> bloom;
  uint32_t bloom_mask = 0;
  std::vector<uint2> map; // {gram, 1 + index into lens} or {0, 0}
  uint32_t map_shift = 32, map_mask = 0;
  std::vector<uint32_t> lens; // per bucket: count, lengths (file order: longest first)
};
std::string stage_stats(const StoreView &v, StagedStats *out);

// Walks every pattern of the file through the staged tables exactly as the scan kernel would
// probe them; returns the number of patterns that are NOT reachable (0 = tables are sound).
// Used by CPU-only tests; it does not match haystacks.
uint64_t check_staged_store(const StoreView &v, const StagedStore &s);

// ---- pattern ids (include/olm_b200.h): the catalogue of a store and its lookup table
//
// Id i names the i-th distinct normalised pattern of the file: the long patterns (>= 5 bytes) in
// order of their offset in the pattern store -- the order in which each first appeared in the
// compile input -- then the 1-, 2-, 3- and 4-byte patterns, each length in ascending byte order
// (bitmap1 bit order, bitmap2 bit order b0<<8|b1, arr3 order, arr4 order).  The catalogue is
// defined by the .olm file alone and is built on the host when first asked for.
//
// The lookup table is open addressing over a 64-bit hash of (length, bytes): one 8-byte entry
// {id, fingerprint} per pattern, load <= 0.5; the id pass (pattern_ids.cuh) probes it with the
// hash of a record's normalised bytes and confirms a fingerprint hit with a full byte compare.
struct PatternCatalog {
  uint32_t n_long = 0;
  std::vector<uint2> refs;          // per id: {offset, len}; offset into the pattern store (len >= 5) or into short_bytes
  std::vector<uint8_t> short_bytes; // bytes of the 1..4 byte patterns, concatenated
  const uint8_t *patterns = nullptr; // StoreView::patterns (the mapped file outlives the catalogue)
  std::vector<uint2> table;         // {id, fingerprint}; id kNoPatternId = empty
  uint32_t table_mask = 0;
  uint64_t size() const { return refs.size(); }
  const uint8_t *bytes(uint64_t id) const {
    return refs[id].y >= 5 ? patterns + refs[id].x : short_bytes.data() + refs[id].x;
  }
};
constexpr uint32_t kNoPatternId = 0xFFFFFFFFu;
std::string build_catalog(const StoreView &v, PatternCatalog *out);

// Hash of a pattern's normalised bytes, fed one byte at a time (the device feeds it while it
// normalises a record's source span), then finished with the length.  FNV-1a 64 + a murmur3 finaliser.
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint64_t pattern_hash_step(uint64_t h, uint32_t byte) { return (h ^ byte) * 0x100000001B3ull; }
constexpr uint64_t kPatternHashSeed = 0xCBF29CE484222325ull;
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint64_t pattern_hash_final(uint64_t h, uint32_t len) {
  h ^= uint64_t(len) * 0x9E3779B97F4A7C15ull;
  h ^= h >> 33;
  h *= 0xFF51AFD7ED558CCDull;
  h ^= h >> 33;
  h *= 0xC4CEB9FE1A85EC53ull;
  h ^= h >> 33;
  return h;
}
// home slot of a hash / its fingerprint
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint32_t pattern_home(uint64_t h, uint32_t mask) { return uint32_t(h >> 32) & mask; }
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint32_t pattern_fingerprint(uint64_t h) { return uint32_t(h); }

// host mirror of the device hashing (scan.cu uses the same expressions)
inline uint32_t key_home(const DeviceStore &d, uint32_t key) { return key >> d.key_shift; }
inline uint32_t g4_bit(const DeviceStore &d, uint32_t key) { return key >> d.g4_shift; }
constexpr uint32_t kSx3Off = 2048; // words of sx in front of its hashed part
// bit of a 3-byte pattern (key3 = b0<<16|b1<<8|b2) in the hashed part of sx
inline uint32_t sx3_bit(const DeviceStore &d, uint32_t key3) { return (key3 * kHashMul) >> d.sx3_shift; }
inline uint32_t p23_bit(const DeviceStore &d, uint32_t gram) {
  return ((gram & d.p23_and) * d.p23_mul) >> d.p23_shift;
}
// byte-class prefilter as the kernel evaluates it (device_tables.h ByteClass)
inline bool class_has(const ByteClass &c, uint32_t b) {
  if (b >= 0x80) return false;
  const uint32_t t = b & c.and_mask;
  for (uint32_t i = 0; i < c.n_ranges; ++i)
    if (t >= c.lo[i] && t <= c.hi[i]) return true;
  return false;
}
inline uint32_t set3_home(const DeviceStore &d, uint32_t key3) { return (key3 * kHashMul >> 8) & d.set3_mask; }

} // namespace olm
