// store.cpp -- parse a compiled store and re-stage it for HBM (kernel K1 of SURVEY 2.1).
//
// parse_store() follows the section walk of the reference loader (omega_match/src/matcher.c:
// 329-432) with explicit bounds checks.  stage_store() then builds the device layout that
// device_tables.h describes.  The index array of the file is ignored: the bucket blob is
// walked record by record, which yields every (gram -> patterns) pair without depending on
// how unused index slots were written (SURVEY F8).
#include "store.h"

#include <algorithm>
#include <cstdlib>

#include "host_util.h"

// buckets of the key table = 2^OLM_KEY_EXTRA_LOG2 x the smallest power of two >= #keys.  With 1 a
// probe meets a full bucket (and has to look at the next one) 0.2 % of the time instead of 1.6 %;
// as a warp takes that path when ANY of its 32 probes does, this is 5 % instead of 40 % of the
// rounds (measured: +4 % throughput at 1 M patterns; the table -- 32 MiB -- still lives in L2).
#ifndef OLM_KEY_EXTRA_LOG2
#define OLM_KEY_EXTRA_LOG2 1
#endif
namespace olm {

std::string parse_store(const uint8_t *f, size_t size, StoreView *v) {
  *v = StoreView{};
  if (!f || size < kHeaderBytes) return "file shorter than the 72-byte header";
  if (std::memcmp(f, kMagicHeader, 8) != 0) return "header magic mismatch";
  Header &h = v->hdr;
  h.version = rd32(f + 8);
  h.flags = rd32(f + 12);
  h.store_bytes = rd64(f + 16);
  h.stored_patterns = rd32(f + 24);
  h.smallest = rd32(f + 28);
  h.largest = rd32(f + 32);
  h.bloom_bytes = rd32(f + 36);
  h.blob_bytes = rd32(f + 40);
  h.table_size = rd32(f + 44);
  h.occupied = rd32(f + 48);
  h.min_bucket = rd32(f + 52);
  h.max_bucket = rd32(f + 56);
  h.short_bytes = rd32(f + 60);
  std::memcpy(&h.load_factor, f + 64, 4);
  std::memcpy(&h.avg_bucket, f + 68, 4);
  v->base = f;
  v->size = size;

  uint64_t off = kHeaderBytes;
  auto need = [&](uint64_t n) { return off <= size && n <= size - off; }; // (no wrap-around for huge n)
  if (!need(h.store_bytes)) return "pattern store runs past the end of the file";
  v->patterns = f + off;
  off += h.store_bytes;
  if (!need(12) || std::memcmp(f + off, kMagicBloom, 8) != 0) return "bloom magic mismatch";
  off += 8;
  v->bloom_bits = rd32(f + off);
  off += 4;
  if (!need(h.bloom_bytes)) return "bloom filter runs past the end of the file";
  v->bloom = f + off;
  off += h.bloom_bytes;
  if (!need(8) || std::memcmp(f + off, kMagicHash, 8) != 0) return "hash table magic mismatch";
  off += 8;
  if (!need(uint64_t(h.table_size) * 4)) return "index array runs past the end of the file";
  v->index = f + off;
  off += uint64_t(h.table_size) * 4;
  if (!need(h.blob_bytes)) return "bucket data runs past the end of the file";
  v->blob = f + off;
  off += h.blob_bytes;
  if (off > size || h.short_bytes != size - off) return "short matcher size mismatch"; // matcher.c:425
  if (h.short_bytes) {
    if (h.short_bytes < 8 + 32 + 8192 + 16 || std::memcmp(f + off, kMagicShort, 8) != 0)
      return "short matcher magic mismatch";
    const uint8_t *p = f + off + 8;
    v->bitmap1 = p;
    v->bitmap2 = p + 32;
    p += 32 + 8192;
    v->n1 = rd32(p);
    v->n2 = rd32(p + 4);
    v->n3 = rd32(p + 8);
    v->n4 = rd32(p + 12);
    p += 16;
    if (uint64_t(8 + 32 + 8192 + 16) + 4ull * v->n3 + 4ull * v->n4 != h.short_bytes)
      return "short matcher arrays do not fit their section";
    v->arr3 = p;
    v->arr4 = p + 4ull * v->n3;
  }
  return "";
}

namespace {

uint32_t ceil_log2(uint64_t v) {
  uint32_t l = 0;
  while ((1ull << l) < v) ++l;
  return l;
}

struct BucketRef {
  uint32_t gram;
  uint32_t count;
  const uint8_t *recs; // count x 16 bytes in the blob
};

} // namespace

std::string stage_store(const StoreView &v, const FilterBudget &budget, StagedStore *s) {
  *s = StagedStore{};
  const Header &h = v.hdr;
  if (h.store_bytes >= 0xFFFFFFF0ull) return "pattern store of 4 GiB or more is not supported";

  // ---- walk the bucket blob: [u32 gram][u32 count][{u64 off,u32 len,u32 0} x count]
  std::vector<BucketRef> buckets;
  buckets.reserve(size_t(std::min<uint64_t>(h.occupied, h.blob_bytes / (8 + kBucketRecordBytes)))); // (the header is not trusted)
  uint64_t n_recs_multi = 0, n_long = 0;
  for (uint64_t p = 0; p < h.blob_bytes;) {
    if (p + 8 > h.blob_bytes) return "truncated bucket header";
    BucketRef b{rd32(v.blob + p), rd32(v.blob + p + 4), v.blob + p + 8};
    if (b.count == 0 || p + 8 + uint64_t(b.count) * kBucketRecordBytes > h.blob_bytes)
      return "bucket runs past the bucket data";
    for (uint32_t j = 0; j < b.count; ++j) {
      const uint64_t po = rd64(b.recs + 16ull * j);
      const uint32_t pl = rd32(b.recs + 16ull * j + 8);
      if (pl < 5 || pl > kSlotValueMask || po > h.store_bytes || pl > h.store_bytes - po) return "pattern record out of range";
      if (rd32(v.patterns + po) != __builtin_bswap32(b.gram)) return "pattern does not start with its bucket gram";
    }
    n_long += b.count;
    if (b.count > 1) n_recs_multi += b.count;
    buckets.push_back(b);
    p += 8 + uint64_t(b.count) * kBucketRecordBytes;
  }
  (void)n_recs_multi;

  // ---- pattern bytes, padded for unaligned 4-byte reads
  s->store.assign(size_t(h.store_bytes) + 16, 0);
  if (h.store_bytes) std::memcpy(s->store.data(), v.patterns, size_t(h.store_bytes));

  // ---- keys + slots.  A key covers the first K bytes of a pattern (device_tables.h).
  uint32_t min_long = 0xFFFFFFFFu, max_long = 0;
  for (const BucketRef &b : buckets)
    for (uint32_t j = 0; j < b.count; ++j) {
      min_long = std::min(min_long, rd32(b.recs + 16ull * j + 8));
      max_long = std::max(max_long, rd32(b.recs + 16ull * j + 8));
    }
  // (shard halos are sized from the header's longest pattern: it must not understate the records)
  if (max_long > h.largest) return "header understates the longest pattern";
  DeviceStore &d = s->params;
  // (stores with 1..4 byte patterns keep 4-byte keys: the 4-byte patterns are keys themselves, and
  // the kernels for short-pattern stores hash four bytes only)
  d.key_bytes = (v.n1 || v.n2 || v.n3 || v.n4 || buckets.empty()) ? 4u : std::min<uint32_t>(8u, min_long);
  d.tail_mask = d.key_bytes >= 8 ? 0xFFFFFFFFu : ((1u << (8 * (d.key_bytes - 4))) - 1u);

  auto word_of = [&](uint64_t off, uint32_t len, uint32_t from) {
    uint32_t w = 0;
    for (uint32_t i = 0; i < 4 && from + i < len; ++i) w |= uint32_t(s->store[off + from + i]) << (8 * i);
    return w;
  };
  // every long pattern with its key, grouped by key in order of first appearance
  struct Pat {
    uint32_t key, len;
    uint64_t off;
  };
  std::vector<Pat> pats;
  pats.reserve(n_long);
  for (const BucketRef &b : buckets)
    for (uint32_t j = 0; j < b.count; ++j) {
      const uint64_t po = rd64(b.recs + 16ull * j);
      const uint32_t pl = rd32(b.recs + 16ull * j + 8);
      pats.push_back(Pat{key_hash(b.gram, word_of(po, pl, 4) & d.tail_mask), pl, po});
    }
  std::vector<uint32_t> all; // distinct keys (patterns and 4-byte grams)
  all.reserve(pats.size() + v.n4);
  for (const Pat &p : pats) all.push_back(p.key);
  for (uint32_t i = 0; i < v.n4; ++i) all.push_back(key_hash(rd32(v.arr4 + 4ull * i), 0));
  std::sort(all.begin(), all.end());
  all.erase(std::unique(all.begin(), all.end()), all.end());
  const uint64_t n_keys_total = all.size();
  // buckets of four places; #buckets >= 2 x #keys, i.e. load <= 0.125
  uint32_t lg_buckets = std::max<uint32_t>(3, ceil_log2(std::max<uint64_t>(1, n_keys_total)) + OLM_KEY_EXTRA_LOG2);
  if (lg_buckets > 27) return "too many distinct keys";
  const uint32_t n_buckets = 1u << lg_buckets;
  d.key_shift = 32 - lg_buckets;
  d.key_mask = n_buckets - 1;
  {
    uint32_t e = 0xFFFFFFFFu; // a value that is no key marks unused places
    while (std::binary_search(all.begin(), all.end(), e)) --e;
    d.empty_key = e;
  }
  s->keys.assign(n_buckets, make_uint4(d.empty_key, d.empty_key, d.empty_key, d.empty_key));
  s->slots.assign(size_t(n_buckets) * 4, Slot{0, 0, 0, 0});

  // returns the slot index of `key`, claiming the first free place from its home bucket on
  auto find_or_claim = [&](uint32_t key, bool *fresh) -> size_t {
    for (uint32_t b = key_home(d, key);; b = (b + 1) & d.key_mask) {
      uint32_t *k = reinterpret_cast<uint32_t *>(&s->keys[b]);
      for (uint32_t j = 0; j < 4; ++j) {
        if (k[j] == key || k[j] == d.empty_key) {
          *fresh = k[j] != key;
          k[j] = key;
          return 4 * size_t(b) + j;
        }
      }
    }
  };
  // patterns per slot, in order of appearance; then single slots inline, the rest through recs[]
  std::vector<std::vector<uint32_t>> members; // indices into pats, per claimed slot (dense ids)
  std::vector<size_t> slot_of_group;
  {
    std::vector<uint32_t> group_of_slot(s->slots.size(), 0xFFFFFFFFu);
    for (uint32_t i = 0; i < pats.size(); ++i) {
      bool fresh = false;
      const size_t si = find_or_claim(pats[i].key, &fresh);
      if (group_of_slot[si] == 0xFFFFFFFFu) {
        group_of_slot[si] = uint32_t(members.size());
        members.emplace_back();
        slot_of_group.push_back(si);
      }
      members[group_of_slot[si]].push_back(i);
    }
  }
  uint64_t n_multi = 0;
  for (const auto &m : members)
    if (m.size() > 1) n_multi += m.size();
  if (n_multi > kSlotValueMask) return "too many patterns";
  s->recs.reserve(n_multi);
  for (size_t g = 0; g < members.size(); ++g) {
    Slot &sl = s->slots[slot_of_group[g]];
    const auto &m = members[g];
    if (m.size() == 1) {
      const Pat &p = pats[m[0]];
      sl.meta = p.len;
      sl.ref = uint32_t(p.off);
      sl.w0 = word_of(p.off, p.len, 0);
      sl.w1 = word_of(p.off, p.len, 4);
    } else {
      sl.meta = kSlotMulti | uint32_t(m.size());
      d.max_recs = std::max<uint32_t>(d.max_recs, uint32_t(m.size()));
      sl.ref = uint32_t(s->recs.size());
      const size_t first = s->recs.size();
      for (uint32_t i : m) {
        const Pat &p = pats[i];
        s->recs.push_back(Rec{word_of(p.off, p.len, 0), p.len, uint32_t(p.off), word_of(p.off, p.len, 4)});
      }
      // the scan emits a slot's matches in record order and relies on "longest first"
      // (compiler.c:271 sorts a bucket that way; patterns that can match at the same position
      // share their first K bytes, hence their slot)
      std::stable_sort(s->recs.begin() + first, s->recs.end(), [](const Rec &x, const Rec &y) { return x.len > y.len; });
      // Which bytes follow the key in the slot's patterns: bit (b & 31) of w0 for byte K, of w1 for byte
      // K + 1 (all ones when a pattern ends before that byte, or the byte lies outside the 8 bytes the
      // scan holds of a position).  A position whose next byte is in neither set cannot match any of the
      // records: the scan skips them all (census surnames behind 4-byte keys: 5.3 records per key).
      const uint32_t K = d.key_bytes;
      uint32_t m0 = 0, m1 = 0;
      bool all0 = K < 8, all1 = K + 1 < 8;
      for (uint32_t i : m) {
        const Pat &p = pats[i];
        if (p.len > K) m0 |= 1u << (s->store[p.off + K] & 31);
        else all0 = false;
        if (p.len > K + 1) m1 |= 1u << (s->store[p.off + K + 1] & 31);
        else all1 = false;
      }
      sl.w0 = all0 ? m0 : 0xFFFFFFFFu;
      sl.w1 = all1 ? m1 : 0xFFFFFFFFu;
    }
  }
  for (uint32_t i = 0; i < v.n4; ++i) {
    bool fresh = false;
    Slot &sl = s->slots[find_or_claim(key_hash(rd32(v.arr4 + 4ull * i), 0), &fresh)];
    sl.meta |= kSlotShort4;
  }
  s->n_keys = uint32_t(n_keys_total);
  // Keys with many patterns behind them are compared by the whole warp (scan.cu, COOP kernels).  That
  // pays when such keys are the rule -- census surnames: 5.6 patterns per 4-byte key, 90 vs 73 GB/s
  // on text -- and costs a little when they are the exception (names.txt: 2.4 per key, 327 vs 335).
  d.coop = d.max_recs >= kCoopMinRecs && n_long >= 4 * n_keys_total ? 1u : 0u;
  if (s->recs.empty()) s->recs.push_back(Rec{0, 0, 0, 0}); // never dereferenced; keeps the upload non-empty

  // ---- g4: one bit per gram, >= 16 bits per key while it fits the shared-memory budget
  if (s->n_keys) {
    const uint32_t n_keys = s->n_keys;
    const uint32_t lg = std::min(budget.g4_max_log2, std::max<uint32_t>(10, ceil_log2(uint64_t(n_keys) * 16)));
    d.g4_shift = 32 - lg;
    d.g4_words = (1u << lg) / 32;
    s->g4.assign(d.g4_words, 0);
    for (const uint4 &kb : s->keys)
      for (uint32_t k : {kb.x, kb.y, kb.z, kb.w})
        if (k != d.empty_key) {
          const uint32_t b = g4_bit(d, k); // k is a key already
          s->g4[b >> 5] |= 1u << (b & 31);
        }
  }

  // ---- p23: candidates for the 1..3 byte patterns
  d.n1 = v.n1;
  d.n2 = v.n2;
  d.n3 = v.n3;
  d.n4 = v.n4;
  if (v.n1 || v.n2 || v.n3) {
    const uint64_t hashed_entries = uint64_t(v.n3) + uint64_t(v.n2) * 256;
    const bool hashed = v.n1 == 0 && hashed_entries * 16 <= (1ull << budget.p23_max_log2);
    if (hashed) { // index = hash of the first three bytes; 2-byte patterns cover all third bytes
      const uint32_t lg = std::min(budget.p23_max_log2, std::max<uint32_t>(10, ceil_log2(hashed_entries * 16)));
      d.p23_and = 0xFFFFFF00u;
      d.p23_mul = kHashMul;
      d.p23_shift = 32 - lg;
      d.p23_words = (1u << lg) / 32;
    } else { // index = the first two bytes; exact for 2-byte patterns, a prefix test for the rest
      d.p23_and = 0xFFFF0000u;
      d.p23_mul = 1;
      d.p23_shift = 16;
      d.p23_words = 65536 / 32;
    }
    s->p23.assign(d.p23_words, 0);
    auto set_bit = [&](uint32_t gram) {
      const uint32_t b = p23_bit(d, gram);
      s->p23[b >> 5] |= 1u << (b & 31);
    };
    for (uint32_t i = 0; i < v.n3; ++i) set_bit(rd32(v.arr3 + 4ull * i) << 8);
    for (uint32_t w = 0; w < 65536; ++w) {
      if (!(v.bitmap2[w >> 3] & (1u << (w & 7)))) continue;
      if (hashed)
        for (uint32_t c = 0; c < 256; ++c) set_bit((w << 16) | (c << 8));
      else
        set_bit(w << 16);
    }
    if (!hashed)
      for (uint32_t b0 = 0; b0 < 256; ++b0)
        if (v.bitmap1[b0 >> 3] & (1u << (b0 & 7)))
          for (uint32_t b1 = 0; b1 < 256; ++b1) set_bit((b0 << 24) | (b1 << 16));
  }

  // ---- exact sets for the short lengths
  {
    const uint32_t lg = std::max<uint32_t>(4, ceil_log2(std::max<uint64_t>(1, uint64_t(v.n3) * 2)));
    d.set3_mask = (1u << lg) - 1;
    s->set3.assign(size_t(1) << lg, 0);
    for (uint32_t i = 0; i < v.n3; ++i) {
      const uint32_t k = rd32(v.arr3 + 4ull * i);
      uint32_t j = set3_home(d, k);
      while (s->set3[j] != 0 && s->set3[j] != k + 1) j = (j + 1) & d.set3_mask;
      s->set3[j] = k + 1;
    }
    s->bitmap2.assign(2048, 0);
    if (v.bitmap2) std::memcpy(s->bitmap2.data(), v.bitmap2, 8192);
    if (v.bitmap1) std::memcpy(d.bitmap1, v.bitmap1, 32);
  }
  // ---- sx: the short candidates' second look (device_tables.h)
  if (v.n1 || v.n2 || v.n3) {
    s->sx.assign(kSx3Off, 0);
    if (v.n2) std::copy(s->bitmap2.begin(), s->bitmap2.end(), s->sx.begin());
    for (uint32_t b0 = 0; b0 < 256 && v.n1; ++b0)
      if (d.bitmap1[b0 >> 5] >> (b0 & 31) & 1)
        for (uint32_t w = 0; w < 8; ++w) s->sx[b0 * 8 + w] = 0xFFFFFFFFu; // every second byte
    if (v.n3) {
      const uint32_t lg = std::min<uint32_t>(17, std::max<uint32_t>(10, ceil_log2(uint64_t(v.n3) * 64)));
      d.sx3_shift = 32 - lg;
      s->sx.resize(kSx3Off + (size_t(1) << lg) / 32, 0);
      for (uint32_t i = 0; i < v.n3; ++i) {
        const uint32_t b = sx3_bit(d, rd32(v.arr3 + 4ull * i));
        s->sx[kSx3Off + (b >> 5)] |= 1u << (b & 31);
      }
    }
    d.sx_words = uint32_t(s->sx.size()); // (a multiple of 4: copied to shared memory 16 bytes at a time)
  }
  // ---- byte-class prefilter (device_tables.h): only when every pattern has >= 4 bytes
  if (v.n1 == 0 && v.n2 == 0 && v.n3 == 0 && (n_long || v.n4)) {
    uint32_t run = v.n4 ? 4 : std::min<uint32_t>(8, h.smallest);
    if (run == 7) run = 6;
    bool used[256] = {false};
    for (const BucketRef &b : buckets)
      for (uint32_t j = 0; j < b.count; ++j) {
        const uint64_t po = rd64(b.recs + 16ull * j);
        for (uint32_t i = 0; i < run; ++i) used[v.patterns[po + i]] = true;
      }
    for (uint32_t i = 0; i < v.n4; ++i) {
      const uint32_t g = rd32(v.arr4 + 4ull * i);
      for (uint32_t k = 0; k < 4; ++k) used[(g >> (8 * k)) & 0xFF] = true;
    }
    bool ascii = true;
    for (uint32_t b = 0x80; b < 256; ++b) ascii = ascii && !used[b];
    if (ascii && run >= 4) {
      // best cover of the used values by <= 2 ranges, with and without folding bit 5
      ByteClass best;
      uint32_t best_cost = 1u << 30;
      for (uint32_t mask : {0x7Fu, 0x5Fu}) {
        bool u[128] = {false};
        for (uint32_t b = 0; b < 128; ++b)
          if (used[b]) u[b & mask] = true;
        uint32_t first = 128, last = 0;
        for (uint32_t t = 0; t < 128; ++t)
          if (u[t]) {
            first = std::min(first, t);
            last = t;
          }
        if (first > last) continue;
        // widest gap inside [first, last] splits the cover in two
        uint32_t gap_lo = 0, gap_len = 0, run_start = first;
        for (uint32_t t = first; t <= last; ++t)
          if (u[t]) {
            if (t > run_start && t - run_start > gap_len) {
              gap_len = t - run_start;
              gap_lo = run_start;
            }
            run_start = t + 1;
          }
        ByteClass c;
        c.run = run;
        c.and_mask = mask;
        if (gap_len) {
          c.n_ranges = 2;
          c.lo[0] = first;
          c.hi[0] = gap_lo - 1;
          c.lo[1] = gap_lo + gap_len;
          c.hi[1] = last;
        } else {
          c.n_ranges = 1;
          c.lo[0] = first;
          c.hi[0] = last;
        }
        // cost = byte values (0..255) the class lets through
        uint32_t cost = 0;
        for (uint32_t b = 0; b < 256; ++b) cost += class_has(c, b);
        cost = cost * 4 + c.n_ranges; // fewer values first, then fewer ranges
        if (cost < best_cost) {
          best_cost = cost;
          best = c;
        }
      }
      // worth its instructions only when it lets through a minority of the byte values
      if (best.run && best_cost / 4 <= 96) {
        best.and4 = best.and_mask * 0x01010101u;
        for (uint32_t i = 0; i < 2; ++i) {
          best.addlo[i] = (0x80u - best.lo[i]) * 0x01010101u;
          best.addhi[i] = (0x7Fu - best.hi[i]) * 0x01010101u;
        }
        d.cls = best;
      }
    }
  }

  d.n_long = uint32_t(n_long);
  d.smallest = h.smallest;
  d.largest = h.largest;
  d.flags = h.flags;
  return "";
}

std::string stage_stats(const StoreView &v, StagedStats *s) {
  *s = StagedStats{};
  const Header &h = v.hdr;
  if (v.bloom_bits == 0 || (v.bloom_bits & (v.bloom_bits - 1)) || uint64_t(v.bloom_bits) / 8 > h.bloom_bytes)
    return "bloom filter size is not a power of two that fits its section";
  s->bloom.assign(std::max<size_t>(1, v.bloom_bits / 64), 0);
  std::memcpy(s->bloom.data(), v.bloom, std::min<size_t>(s->bloom.size() * 8, h.bloom_bytes));
  s->bloom_mask = v.bloom_bits - 1;
  // (sized by the buckets the bucket data really holds, not by the header's count: a wrong count
  // must neither exhaust memory nor leave the open-addressing insert below without a free place)
  uint64_t n_buckets = 0;
  for (uint64_t p = 0; p < h.blob_bytes; ++n_buckets) {
    if (p + 8 > h.blob_bytes) return "truncated bucket header";
    const uint32_t count = rd32(v.blob + p + 4);
    if (count == 0 || p + 8 + uint64_t(count) * kBucketRecordBytes > h.blob_bytes) return "bucket runs past the bucket data";
    p += 8 + uint64_t(count) * kBucketRecordBytes;
  }
  const uint32_t lg = std::max<uint32_t>(4, ceil_log2(std::max<uint64_t>(1, n_buckets) * 2));
  if (lg > 30) return "too many buckets";
  s->map.assign(size_t(1) << lg, make_uint2(0, 0));
  s->map_shift = 32 - lg;
  s->map_mask = (1u << lg) - 1;
  for (uint64_t p = 0; p < h.blob_bytes;) { // (validated by stage_store)
    if (p + 8 > h.blob_bytes) return "truncated bucket header";
    const uint32_t gram = rd32(v.blob + p), count = rd32(v.blob + p + 4);
    if (count == 0 || p + 8 + uint64_t(count) * kBucketRecordBytes > h.blob_bytes) return "bucket runs past the bucket data";
    if (s->lens.size() + count + 1 >= 0xFFFFFFF0ull) return "too many patterns";
    const uint32_t at = uint32_t(s->lens.size());
    s->lens.push_back(count);
    for (uint32_t j = 0; j < count; ++j) s->lens.push_back(rd32(v.blob + p + 8 + 16ull * j + 8));
    for (uint32_t i = (gram * kHashMul) >> s->map_shift;; i = (i + 1) & s->map_mask)
      if (s->map[i].y == 0) {
        s->map[i] = make_uint2(gram, at + 1);
        break;
      }
    p += 8 + uint64_t(count) * kBucketRecordBytes;
  }
  if (s->lens.empty()) s->lens.push_back(0);
  return "";
}

std::string build_catalog(const StoreView &v, PatternCatalog *c) {
  *c = PatternCatalog{};
  const Header &h = v.hdr;
  if (h.store_bytes >= 0xFFFFFFF0ull) return "pattern store of 4 GiB or more is not supported";
  c->patterns = v.patterns;
  // ---- long patterns: every bucket record, in order of store_off
  for (uint64_t p = 0; p < h.blob_bytes;) {
    if (p + 8 > h.blob_bytes) return "truncated bucket header";
    const uint32_t count = rd32(v.blob + p + 4);
    if (count == 0 || p + 8 + uint64_t(count) * kBucketRecordBytes > h.blob_bytes) return "bucket runs past the bucket data";
    for (uint32_t j = 0; j < count; ++j) {
      const uint64_t po = rd64(v.blob + p + 8 + 16ull * j);
      const uint32_t pl = rd32(v.blob + p + 8 + 16ull * j + 8);
      if (pl < 5 || po > h.store_bytes || pl > h.store_bytes - po) return "pattern record out of range";
      c->refs.push_back(make_uint2(uint32_t(po), pl));
    }
    p += 8 + uint64_t(count) * kBucketRecordBytes;
  }
  std::sort(c->refs.begin(), c->refs.end(), [](const uint2 &a, const uint2 &b) { return a.x < b.x; });
  for (size_t i = 1; i < c->refs.size(); ++i)
    if (c->refs[i].x == c->refs[i - 1].x) return "two pattern records share a store offset";
  c->n_long = uint32_t(c->refs.size());
  // ---- short patterns, each length in ascending byte order
  auto add_short = [&](uint32_t be, uint32_t len) { // be = the bytes packed big endian
    c->refs.push_back(make_uint2(uint32_t(c->short_bytes.size()), len));
    for (uint32_t k = len; k-- > 0;) c->short_bytes.push_back(uint8_t(be >> (8 * k)));
  };
  for (uint32_t b = 0; b < 256 && v.bitmap1; ++b)
    if (v.bitmap1[b >> 3] & (1u << (b & 7))) add_short(b, 1);
  for (uint32_t w = 0; w < 65536 && v.bitmap2; ++w)
    if (v.bitmap2[w >> 3] & (1u << (w & 7))) add_short(w, 2);
  for (uint32_t i = 0; i < v.n3; ++i) add_short(rd32(v.arr3 + 4ull * i) & 0xFFFFFFu, 3);
  for (uint32_t i = 0; i < v.n4; ++i) add_short(rd32(v.arr4 + 4ull * i), 4);
  if (c->refs.size() >= kNoPatternId) return "too many patterns";

  // ---- lookup table; of two ids with the same bytes (a hand-made file) the lower one is kept
  const uint32_t lg = std::max<uint32_t>(4, ceil_log2(uint64_t(c->refs.size()) * 2));
  c->table.assign(size_t(1) << lg, make_uint2(kNoPatternId, 0));
  c->table_mask = (1u << lg) - 1;
  for (uint32_t id = 0; id < c->refs.size(); ++id) {
    const uint8_t *b = c->bytes(id);
    const uint32_t len = c->refs[id].y;
    uint64_t hv = kPatternHashSeed;
    for (uint32_t k = 0; k < len; ++k) hv = pattern_hash_step(hv, b[k]);
    hv = pattern_hash_final(hv, len);
    const uint32_t fp = pattern_fingerprint(hv);
    for (uint32_t i = pattern_home(hv, c->table_mask);; i = (i + 1) & c->table_mask) {
      uint2 &e = c->table[i];
      if (e.x == kNoPatternId) {
        e = make_uint2(id, fp);
        break;
      }
      if (e.y == fp && c->refs[e.x].y == len && std::memcmp(c->bytes(e.x), b, len) == 0) break;
    }
  }
  return "";
}

uint64_t check_staged_store(const StoreView &v, const StagedStore &s) {
  const DeviceStore &d = s.params;
  uint64_t bad = 0;
  // the probe of the scan kernel: bitmap, then the key buckets from the key's home on
  auto probe = [&](uint32_t key) -> const Slot * {
    if (!s.g4.empty()) {
      const uint32_t b = g4_bit(d, key);
      if (!(s.g4[b >> 5] >> (b & 31) & 1)) return nullptr;
    }
    for (uint32_t b = key_home(d, key);; b = (b + 1) & d.key_mask) {
      const uint32_t *k = reinterpret_cast<const uint32_t *>(&s.keys[b]);
      for (uint32_t j = 0; j < 4; ++j)
        if (k[j] == key) return key == d.empty_key ? nullptr : &s.slots[4 * size_t(b) + j];
      if (k[3] == d.empty_key) return nullptr;
    }
  };
  auto in_class = [&](const uint8_t *p) {
    for (uint32_t i = 0; i < d.cls.run; ++i)
      if (!class_has(d.cls, p[i])) return false;
    return true;
  };
  auto le_word = [&](uint64_t po, uint32_t pl, uint32_t from) {
    uint32_t w = 0;
    for (uint32_t i = 0; i < 4 && from + i < pl; ++i) w |= uint32_t(v.patterns[po + from + i]) << (8 * i);
    return w;
  };
  for (uint64_t p = 0; p < v.hdr.blob_bytes;) {
    const uint32_t gram = rd32(v.blob + p), count = rd32(v.blob + p + 4);
    for (uint32_t j = 0; j < count; ++j) {
      const uint64_t po = rd64(v.blob + p + 8 + 16ull * j);
      const uint32_t pl = rd32(v.blob + p + 8 + 16ull * j + 8);
      const uint32_t w0 = le_word(po, pl, 0), w1 = le_word(po, pl, 4);
      bool ok = pl >= d.key_bytes;
      const Slot *sl = ok ? probe(key_hash(gram, w1 & d.tail_mask)) : nullptr;
      ok = sl != nullptr;
      if (ok && !(sl->meta & kSlotMulti)) {
        ok = (sl->meta & kSlotValueMask) == pl && sl->ref == po && sl->w0 == w0 && sl->w1 == w1;
      } else if (ok) {
        const uint32_t n = sl->meta & kSlotValueMask;
        bool found = false;
        for (uint32_t q = 0; q < n; ++q) {
          const Rec &rc = s.recs[sl->ref + q];
          if (q > 0 && s.recs[sl->ref + q - 1].len < rc.len) ok = false; // longest first
          if (rc.len == pl && rc.store_off == po) found = rc.w0 == w0 && rc.w1 == w1;
        }
        ok = ok && found;
        // the slot's next-byte sets never rule this pattern out (scan.cu next_bytes_ok)
        const uint32_t K = d.key_bytes;
        if (K < 8) ok = ok && (pl > K ? (sl->w0 >> (v.patterns[po + K] & 31) & 1) != 0 : sl->w0 == 0xFFFFFFFFu);
        if (K + 1 < 8) ok = ok && (pl > K + 1 ? (sl->w1 >> (v.patterns[po + K + 1] & 31) & 1) != 0 : sl->w1 == 0xFFFFFFFFu);
      }
      ok = ok && std::memcmp(s.store.data() + po, v.patterns + po, pl) == 0 && in_class(v.patterns + po);
      bad += !ok;
    }
    p += 8 + 16ull * count;
  }
  for (uint32_t i = 0; i < v.n4; ++i) {
    const uint32_t g4v = rd32(v.arr4 + 4ull * i);
    const Slot *sl = d.key_bytes == 4 ? probe(key_hash(g4v, 0)) : nullptr;
    const uint8_t g4b[4] = {uint8_t(g4v >> 24), uint8_t(g4v >> 16), uint8_t(g4v >> 8), uint8_t(g4v)};
    bad += !(sl && (sl->meta & kSlotShort4) && (d.cls.run == 0 || (d.cls.run == 4 && in_class(g4b))));
  }
  auto p23_ok = [&](uint32_t gram) {
    const uint32_t b = p23_bit(d, gram);
    return !s.p23.empty() && (s.p23[b >> 5] >> (b & 31) & 1);
  };
  for (uint32_t i = 0; i < v.n3; ++i) {
    const uint32_t k = rd32(v.arr3 + 4ull * i);
    bool found = false;
    for (uint32_t j = set3_home(d, k); s.set3[j] != 0; j = (j + 1) & d.set3_mask)
      if (s.set3[j] == k + 1) {
        found = true;
        break;
      }
    for (uint32_t c = 0; c < 256; c += 51) bad += !p23_ok((k << 8) | c);
    bad += !found;
    if (d.sx_words) { // the second look never drops a 3-byte pattern
      const uint32_t b = sx3_bit(d, k);
      bad += !(s.sx[kSx3Off + (b >> 5)] >> (b & 31) & 1);
    }
  }
  for (uint32_t w = 0; w < 65536 && v.bitmap2; ++w)
    if (v.bitmap2[w >> 3] & (1u << (w & 7))) {
      bad += !(s.bitmap2[w >> 5] >> (w & 31) & 1);
      if (d.sx_words) bad += !(s.sx[w >> 5] >> (w & 31) & 1);
      for (uint32_t c = 0; c < 65536; c += 4099) bad += !p23_ok((w << 16) | c);
    }
  for (uint32_t b = 0; b < 256 && v.bitmap1; ++b)
    if (v.bitmap1[b >> 3] & (1u << (b & 7))) {
      bad += !(d.bitmap1[b >> 5] >> (b & 31) & 1);
      if (d.sx_words) bad += !(s.sx[b * 8] & 1);
      for (uint32_t c = 0; c < (1u << 24); c += 65521) bad += !p23_ok((b << 24) | c);
    }
  return bad;
}

} // namespace olm
