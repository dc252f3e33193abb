/* olm_b200.h -- C ABI of libomega_match.so (B200 build).
 *
 * Part 1 is the drop-in boundary: the 22 entry points and 4 POD structs of the reference's
 * public header (omega_match/include/omega/list_matcher.h), same names, argument order and
 * return conventions, so that main.c:400-464 and the cffi wrapper
 * (bindings/python/omega_match/omega_match.py:14-330 cdef, :409-420 OMEGA_MATCH_LIB_PATH)
 * bind to this library unchanged.  Each prototype cites the reference declaration it
 * replaces as  [ref list_matcher.h:LINE -> implementation FILE:LINE].
 *
 * Part 2 (olm_cuda_*) is new: device-resident input/output, byte-range shards for multi-GPU,
 * device timing.  Nothing in this header mentions torch, CUDA types or C++.
 */
#ifndef OLM_B200_H
#define OLM_B200_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- Part 1: reference ABI */

typedef struct omega_list_matcher_struct omega_list_matcher_t;                   /* [ref :16] */
typedef struct omega_list_matcher_compiler_struct omega_list_matcher_compiler_t; /* [ref :13] */

typedef struct { /* [ref :19-23] 24 bytes; `match` aliases the caller's haystack */
  size_t offset;
  uint32_t len;
  const uint8_t *match;
} omega_match_result_t;

typedef struct { /* [ref :26-29] */
  size_t count;
  omega_match_result_t *matches;
} omega_match_results_t;

typedef struct { /* [ref :32-40] */
  uint64_t total_input_bytes;
  uint64_t total_stored_bytes;
  uint32_t stored_pattern_count;
  uint32_t short_pattern_count;
  uint32_t duplicate_patterns;
  uint32_t smallest_pattern_length;
  uint32_t largest_pattern_length;
} omega_match_pattern_store_stats_t;

typedef struct { /* [ref :43-49] accumulated into (+=) by every match call */
  uint64_t total_hits;
  uint64_t total_misses;
  uint64_t total_filtered;
  uint64_t total_attempts;
  uint64_t total_comparisons;
} omega_match_stats_t;

/* -- the hot path ------------------------------------------------------------------- */

/* [ref :201-206 -> matcher.c:934-1019]  Scan `haystack` (HOST memory) for every pattern of
 * the store.  Result order: offset ascending, then length descending; `longest_only` and
 * `no_overlap` are applied in that order afterwards.  Returns a heap object owned by the
 * caller until omega_match_results_destroy(); NULL only on a CUDA failure. */
omega_match_results_t *omega_list_matcher_match(const omega_list_matcher_t *matcher,
                                                const uint8_t *haystack, size_t haystack_size,
                                                int no_overlap, int longest_only,
                                                int word_boundary, int word_prefix,
                                                int word_suffix, int line_start, int line_end);

/* [ref :212 -> matcher.c:1022-1028] */
void omega_match_results_destroy(omega_match_results_t *results);

/* -- matcher life cycle --------------------------------------------------------------- */

/* [ref :169-173 -> matcher.c:451-513]  `path` is a compiled store or a newline separated
 * pattern file (then compiled to /tmp/oa_matcher_XXXXXX with the three flags and removed on
 * destroy).  The store is mmapped, re-staged and uploaded to HBM once.  NULL on failure
 * (bad file, no CUDA device). */
omega_list_matcher_t *omega_list_matcher_create(const char *compiled_or_patterns_file,
                                                int case_insensitive, int ignore_punctuation,
                                                int elide_whitespace,
                                                omega_match_pattern_store_stats_t *stats);

/* [ref :155-158 -> matcher.c:434-448] compile `patterns_buffer` into `compiled_file`, then create. */
omega_list_matcher_t *omega_list_matcher_create_from_buffer(
    const char *compiled_file, const uint8_t *patterns_buffer, uint64_t patterns_buffer_size,
    int case_insensitive, int ignore_punctuation, int elide_whitespace,
    omega_match_pattern_store_stats_t *stats);

/* [ref :181-182 -> matcher.c:516-523] attach caller-owned counters. */
int omega_list_matcher_add_stats(omega_list_matcher_t *matcher, omega_match_stats_t *stats);

/* [ref :189 -> matcher.c:526-545] */
int omega_list_matcher_destroy(omega_list_matcher_t *matcher);

/* [ref :106-107 -> matcher.c:176-179, common.c:6-40] one "Header v1 stats: ..." line. */
int omega_list_matcher_emit_header_info(const omega_list_matcher_t *matcher, FILE *fp);

/* [ref :250-277 -> matcher.c:135-173]  Kept for source compatibility.  On the GPU build the
 * thread count is the number of host staging threads and the chunk size is informational;
 * validation and defaults are the reference's (0 -> max / 4096, chunk rounded to 2^k, -1 on
 * negative or too large values). */
int omega_matcher_set_num_threads(omega_list_matcher_t *matcher, int threads);
int omega_matcher_get_num_threads(const omega_list_matcher_t *matcher);
int omega_matcher_set_chunk_size(omega_list_matcher_t *matcher, int chunk);
int omega_matcher_get_chunk_size(const omega_list_matcher_t *matcher);

/* -- pattern compiler (writes the .olm store; host side) ------------------------------ */

/* [ref :59-63 -> compiler.c:132-195] */
omega_list_matcher_compiler_t *omega_list_matcher_compiler_create(const char *compiled_file,
                                                                  int case_insensitive,
                                                                  int ignore_punctuation,
                                                                  int elide_whitespace);
/* [ref :71-73 -> compiler.c:197-229]  Returns 0, or -1 when the pattern is empty after
 * normalisation (the reference aborts the process there, compiler.c:126-127). */
int omega_list_matcher_compiler_add_pattern(omega_list_matcher_compiler_t *compiler,
                                            const uint8_t *pattern, uint32_t len);
/* [ref :80-82 -> compiler.c:231-239] */
const omega_match_pattern_store_stats_t *omega_list_matcher_compiler_get_pattern_store_stats(
    const omega_list_matcher_compiler_t *compiler);
/* [ref :89-90 -> compiler.c:241-380] finalises and writes the file. */
int omega_list_matcher_compiler_destroy(omega_list_matcher_compiler_t *compiler);
/* [ref :120-124 -> compiler.c:382-425] one pattern per line, a trailing \r is dropped. */
int omega_list_matcher_compile_patterns(const char *compiled_file, const uint8_t *patterns_buf,
                                        uint64_t patterns_buf_size, int case_insensitive,
                                        int ignore_punctuation, int elide_whitespace,
                                        omega_match_pattern_store_stats_t *pattern_store_stats);
/* [ref :136-139 -> compiler.c:427-463] */
int omega_list_matcher_compile_patterns_filename(
    const char *compiled_file, const char *patterns_file, int case_insensitive,
    int ignore_punctuation, int elide_whitespace,
    omega_match_pattern_store_stats_t *pattern_store_stats);
/* [ref :97 -> compiler.c:466-476] 1 when the file starts with the store magic. */
int omega_list_matcher_is_compiled(const char *compiled_file);

/* -- file mapping helpers and version -------------------------------------------------- */

/* [ref :221-222, :231-233, :241 -> util.c:207-250] */
uint8_t *omega_matcher_map_file(FILE *file, size_t *size, int prefetch_sequential);
uint8_t *omega_matcher_map_filename(const char *filename, size_t *size, int prefetch_sequential);
int omega_matcher_unmap_file(const uint8_t *addr, size_t size);
/* [ref :283 -> version.c:6] "MAJOR.MINOR.PATCH" */
const char *omega_match_version(void);

/* ---------------------------------------------------------------- Part 2: B200 extensions */

/* Results that stay in HBM: `records` is a DEVICE pointer to `count` omega_match_result_t
 * (24 bytes each, final order, filters applied). */
typedef struct {
  uint64_t count;
  void *records;   /* device memory owned by the matcher; valid until the next match call */
  int device;
} olm_cuda_results_t;

/* Device-side timings of the most recent match call on this matcher, in milliseconds
 * (CUDA events on the matcher's stream). */
typedef struct {
  float total_ms;     /* first kernel start -> last kernel end (no H2D/D2H) */
  float transform_ms; /* normalisation kernels (stores with a transform flag), else 0 */
  float scan_ms;      /* the scan kernel(s) */
  float filter_ms;    /* no-overlap filter + compaction, else 0 */
  float h2d_ms, d2h_ms;
  uint64_t scan_launches, kernel_launches;
  uint64_t matches_before_filter;
} olm_cuda_timing_t;

/* Environment variables read at omega_list_matcher_create():
 *   OLM_CUDA_DEVICE=<i>       default GPU (see olm_cuda_set_default_device)
 *   OLM_CUDA_DEVICES=<list>   "0,1,2,3", "0-7" or "all": the matcher owns one engine per listed GPU
 *                             and omega_list_matcher_match() shards every host haystack by byte
 *                             range over them (see olm_cuda_matcher_create_multi)
 *   OLM_EXACT_STATS=1         see olm_cuda_set_exact_stats
 *   OLM_HOST_SPAN_BYTES=<n>   omega_list_matcher_match scans host haystacks longer than n bytes in
 *                             spans of n bytes (bounded device memory; same results)
 *   OLM_SHORT_LOOK=0|1        never / whenever there is room: the second look at candidates of the
 *                             1..3 byte patterns (default: for stores with 1-byte patterns)
 *   OLM_COUNT_TABLE=0|1       the histogram of the pattern counts without / with its per-block
 *                             table of ids (default: with it from 64 records per catalogue pattern;
 *                             same counts either way).  For tests and measurements of both.
 * and at olm_cuda_comm_create():
 *   OLM_GATHER_WINDOW=0       gather with ncclSend/ncclRecv instead of the IPC window */
int olm_cuda_device_count(void);
/* Choose the GPU a matcher lives on BEFORE create (process wide default: device 0 or
 * $OLM_CUDA_DEVICE). */
int olm_cuda_set_default_device(int device);
int olm_cuda_matcher_device(const omega_list_matcher_t *matcher);

/* Same as omega_list_matcher_match() but the haystack is DEVICE memory on the matcher's GPU
 * (16-byte aligned, readable up to the next multiple of 16) and the results stay there.  The
 * kernels run on a stream owned by the matcher; the call first waits for all work queued on the
 * device (so bytes produced on any other stream are complete) and returns after its own kernels
 * have finished.
 * `match_ptr_base` is the address written into record.match (+offset); pass the device
 * pointer itself or the host address the bytes came from.  Returns 0, or -1 on a CUDA error. */
int olm_cuda_match_device(const omega_list_matcher_t *matcher, const void *dev_haystack,
                          size_t haystack_size, const void *match_ptr_base, int no_overlap,
                          int longest_only, int word_boundary, int word_prefix, int word_suffix,
                          int line_start, int line_end, olm_cuda_results_t *out);

/* Byte-range shard of a larger haystack (multi-GPU, SURVEY 8e).  `dev_slice` holds the global
 * bytes [slice_begin, slice_begin+slice_len); starts in [own_begin, own_end) are reported
 * with GLOBAL offsets; end-of-buffer predicates use `global_size`.  For stores with a
 * transform flag own_begin and slice_begin must be multiples of 4 MiB.  `no_overlap` is NOT
 * applied here (it crosses shards): call olm_cuda_no_overlap() on the gathered records (or let
 * olm_cuda_gather_records() do it).  Other stores: the slice must hold the shard's halo -- 16 bytes
 * in front of own_begin (unless it is 0) and the longest pattern + 1 bytes behind own_end (up to
 * global_size); the call fails otherwise.  One deviation from a single call over the whole haystack:
 * the stale-tail bytes of the reference's scratch buffer (2..4 byte patterns of a transforming store
 * under word_boundary at the very end of a 4 MiB window) are resolved against the shard's own
 * windows and this matcher's earlier calls only -- a shard does not see the windows in front of it. */
int olm_cuda_match_shard(const omega_list_matcher_t *matcher, const void *dev_slice,
                         uint64_t slice_begin, uint64_t slice_len, uint64_t own_begin,
                         uint64_t own_end, uint64_t global_size, const void *match_ptr_base,
                         int longest_only, int word_boundary, int word_prefix, int word_suffix,
                         int line_start, int line_end, olm_cuda_results_t *out);

/* olm_cuda_match_shard() for a slice that lies in HOST memory (pinned memory copies fastest): the
 * slice goes to the GPU in 256 MiB segments while the scan of the earlier segments runs -- the
 * host-pointer efficiency of omega_list_matcher_match() (matcher.c:934-1019 takes host memory)
 * for one rank of a multi-GPU job.  The records stay on the device. */
int olm_cuda_match_shard_host(const omega_list_matcher_t *matcher, const void *host_slice,
                              uint64_t slice_begin, uint64_t slice_len, uint64_t own_begin,
                              uint64_t own_end, uint64_t global_size, const void *match_ptr_base,
                              int longest_only, int word_boundary, int word_prefix, int word_suffix,
                              int line_start, int line_end, olm_cuda_results_t *out);

/* ---- several GPUs (SURVEY 8e) ------------------------------------------------------------------
 * (1) One process, N GPUs.  The matcher owns one engine per GPU; omega_list_matcher_match() on it
 * shards the host haystack by byte range (ownership rule: a match belongs to the shard that owns
 * its start; stores with a transform flag shard on 4 MiB windows), runs every shard on its GPU
 * from its own host thread (H2D over that GPU's link overlapped with its scan), and delivers ONE
 * result array in final order: the records are copied out by all GPUs at once, each into its
 * range of the array; with no_overlap they are first gathered on the first GPU over NVLink and
 * filtered there.  The olm_cuda_* device entry points of such a matcher address its first GPU. */
omega_list_matcher_t *olm_cuda_matcher_create_multi(const char *compiled_file, const int *devices,
                                                    int n_devices);
int olm_cuda_matcher_device_count(const omega_list_matcher_t *matcher);

/* The byte range rank `rank` of `world` owns and the bytes it has to hold (its slice: 16 bytes in
 * front, the longest pattern + 1 behind; none for stores with a transform flag, which shard on
 * 4 MiB windows).  olm_shard_plan() needs no GPU (largest pattern length and transform flags as
 * olm_store_inspect() reports them). */
typedef struct {
  uint64_t own_begin, own_end, slice_begin, slice_end;
} olm_shard_t;
int olm_shard_plan(uint32_t largest_pattern, int windowed, uint64_t global_size, int world, int rank,
                   olm_shard_t *out);
int olm_cuda_shard_plan(const omega_list_matcher_t *matcher, uint64_t global_size, int world, int rank,
                        olm_shard_t *out);

/* (2) One process per GPU.  Every rank scans its shard (olm_cuda_match_shard[_host]) and the ranks
 * gather the per-rank sorted records on `root` over NVLink: one ncclAllGather tells every rank all
 * counts, hence where its records go (rank order = global order); the root's gather buffer is
 * mapped into the other ranks' address spaces (CUDA IPC, set up when the buffer is made or grows)
 * and every rank copies its records to their final place with its copy engines, all ranks at once;
 * a closing 8-byte collective tells the root that everything has landed.  Then -- if asked -- the
 * no_overlap filter once on the whole.  OLM_GATHER_WINDOW=0 (or a rank that cannot map the window)
 * selects one group of ncclSend/ncclRecv instead.  Rank 0 makes the id (128 bytes) and hands it to
 * the other ranks by whatever means the job has.  NCCL is opened with dlopen("libnccl.so.2") on
 * first use.  Collective: every rank calls olm_cuda_gather_records(). */
typedef struct olm_cuda_comm olm_cuda_comm_t;
int olm_cuda_comm_unique_id(void *id, size_t id_bytes);
olm_cuda_comm_t *olm_cuda_comm_create(const omega_list_matcher_t *matcher, const void *id, int rank,
                                      int world);
int olm_cuda_comm_destroy(olm_cuda_comm_t *comm);
/* `out` is filled on the root only (device records, valid until the root's next gather). */
int olm_cuda_gather_records(olm_cuda_comm_t *comm, const void *dev_records, uint64_t count, int root,
                            int no_overlap, olm_cuda_results_t *out);

/* The greedy no-overlap filter (matcher.c:570-584) over `count` sorted device records, in
 * place; returns the kept count or -1.  The records may have been produced on any stream: the
 * call first waits for all work queued on the device (like olm_cuda_match_device). */
int64_t olm_cuda_no_overlap(const omega_list_matcher_t *matcher, void *dev_records, uint64_t count);

/* The result listing of the reference's CLI -- one line "offset:matched bytes\n" per record, exactly
 * what omega_match/main.c:89-133 prints (snprintf "%zu:%.*s\n": a line's bytes stop at the first NUL
 * of the match) -- formatted on the GPU from device records and the device-resident haystack
 * (`dev_haystack` = device address of the haystack byte with offset `haystack_offset0`).  *dev_text is
 * device memory owned by the matcher (valid until the next format call), *text_bytes its length. */
int olm_cuda_format_records(const omega_list_matcher_t *matcher, const void *dev_records, uint64_t count,
                            const void *dev_haystack, uint64_t haystack_offset0, void **dev_text,
                            uint64_t *text_bytes);

/* Sort device records by (offset ascending, length descending) -- the order of
 * radix_sort_matches(), matcher.c:258-325 -- with the library's LSD radix sort. */
int olm_cuda_sort_records(const omega_list_matcher_t *matcher, void *dev_records, uint64_t count);

int olm_cuda_last_timing(const omega_list_matcher_t *matcher, olm_cuda_timing_t *out);

/* Statistics (omega_match_stats_t, list_matcher.h:43-49, filled as matcher.c:783-799, :818-877,
 * :210 do).  Default: the counters the scan produces by itself -- hits, misses and comparisons of
 * ITS tables, attempts, filtered = attempts - hits -- at no cost.  With exact statistics on, every
 * match call of a matcher that has a stats struct attached also runs one kernel that evaluates
 * the reference's 3-probe Bloom filter (bloom.c:51-64) and gram -> bucket map
 * (hash_table.c:91-109) for every position, and the five counters equal the reference's.
 * Also switched on for all matchers by the environment variable OLM_EXACT_STATS=1. */
int olm_cuda_set_exact_stats(omega_list_matcher_t *matcher, int on);

/* Pattern ids: which pattern of the store produced each match.
 *
 * The catalogue of a store is the list of its distinct normalised patterns, defined by the
 * compiled file alone (stores written by the reference and by this library behave the same):
 *   ids 0 .. n_long-1   the patterns of 5 or more bytes, in order of their offset in the file's
 *                       pattern store, which is the order in which each distinct pattern first
 *                       appeared in the compile input;
 *   the next ids        the 1-byte, then 2-, 3- and 4-byte patterns, each length in ascending
 *                       byte order.
 * The bytes of an id are the pattern as stored: normalised when the store has a transform flag
 * (`o-malley` in a haystack matches the stored `OMALLEY` of an ignore-case + ignore-punctuation
 * store, and its id names `OMALLEY`).
 *
 * With ids on, omega_list_matcher_match, olm_cuda_match_device, olm_cuda_match_shard and
 * olm_cuda_match_shard_host return records whose 4 pad bytes (after `len`) hold the id
 * (olm_result_with_id_t names them); the records are otherwise byte for byte those of a call with
 * ids off, where the pad bytes are 0.  The ids are resolved on the GPU after the filters, one more
 * kernel per call, included in olm_cuda_timing_t.total_ms; sorting, no_overlap and the gathers
 * move whole records, so ids follow their records.  Switching on first builds the catalogue and
 * uploads a lookup table (about 24 bytes per pattern of device memory); it returns -1 for a store
 * whose pattern records are malformed (out of range, or two at one offset).  A call fails (-1 /
 * NULL, with a message on stderr) rather than return a record without its id. */
typedef struct {
  size_t offset;
  uint32_t len;
  uint32_t pattern_id;
  const uint8_t *match;
} olm_result_with_id_t; /* omega_match_result_t with the pad named (same layout) */
int olm_cuda_set_pattern_ids(omega_list_matcher_t *matcher, int on); /* default off */
/* Catalogue size, or -1 on a malformed store.  No GPU work. */
int64_t olm_pattern_count(const omega_list_matcher_t *matcher);
/* The bytes of pattern `id` (valid for the matcher's lifetime); -1 for an id out of range. */
int olm_pattern_bytes(const omega_list_matcher_t *matcher, uint64_t id, const uint8_t **bytes,
                      uint32_t *len);

/* Pattern counts: how often each pattern of the store occurs, without returning the records.
 *
 * A count call takes the haystack and the seven match flags of the match call it mirrors and adds to
 * counts[id] one for every record that call would have returned (longest_only and no_overlap
 * applied) whose pattern is `id` (the id defined above).  `counts` has olm_pattern_count() entries.
 * The counts are ADDED (+=), as omega_match_stats_t is, so calls, spans, shards and GPUs sum without
 * more API; *total receives the number of records this call counted, the `count` of the equivalent
 * match call.
 *   - Pattern ids may be on or off; a count call leaves that setting as it was (a later match call
 *     with ids off still returns zero pads).  The first count call builds the catalogue and uploads
 *     its lookup table, as olm_cuda_set_pattern_ids does.
 *   - The records never leave the GPU; only the counts (8 bytes per pattern) are copied.
 *   - A record whose bytes name no pattern of the catalogue, and a malformed store, fail the call
 *     (-1, message on stderr); the contents of `counts` are then unspecified.
 *   - The counting pass is part of olm_cuda_timing_t.total_ms, the copy of the counts of d2h_ms.
 * On the device the ids of a call's final records are resolved as with ids on and added into a
 * histogram; records in offset order repeat ids within a warp and a block, which the histogram
 * aggregates before it adds to global memory. */
/* host haystack -> host counts: the one-GPU path, OLM_HOST_SPAN_BYTES spans, multi-GPU matchers */
int olm_cuda_count_patterns(const omega_list_matcher_t *matcher, const uint8_t *haystack, size_t size,
                            int no_overlap, int longest_only, int word_boundary, int word_prefix,
                            int word_suffix, int line_start, int line_end, uint64_t *counts, uint64_t *total);
/* device haystack (the contract of olm_cuda_match_device) -> counts in device memory of the
 * matcher's (first) GPU */
int olm_cuda_count_patterns_device(const omega_list_matcher_t *matcher, const void *dev_haystack, size_t size,
                                   int no_overlap, int longest_only, int word_boundary, int word_prefix,
                                   int word_suffix, int line_start, int line_end, void *dev_counts,
                                   uint64_t *total);
/* Records in device memory of the matcher's (first) GPU whose pad words hold ids (made with ids on:
 * shards, olm_cuda_gather_records) -> device counts.  One process per GPU counts each rank's shard
 * and sums the ranks' counts by its own means, or gathers the records (no_overlap included) and
 * counts on the root.  An id >= olm_pattern_count() fails the call (-1). */
int olm_cuda_count_records(const omega_list_matcher_t *matcher, const void *dev_records, uint64_t count,
                           void *dev_counts);

/* Pinned host memory helpers (so callers can hand DMA-able buffers to _match). */
void *olm_cuda_host_alloc(size_t bytes);
void olm_cuda_host_free(void *p);

/* Store facts without touching a GPU (used by tools and CPU-only tests). */
typedef struct {
  uint32_t flags, smallest, largest, stored_patterns, table_size, occupied_buckets;
  uint32_t len1, len2, len3, len4;
  uint64_t store_bytes, file_bytes;
  /* how the store is staged for the GPU (device_tables.h) */
  uint32_t gram_keys;      /* distinct keys in the key table */
  uint32_t key_buckets;    /* 16-byte buckets of that table */
  uint32_t g4_bits;        /* bits of the shared-memory gram bitmap */
  uint32_t class_run;      /* byte-class prefilter: leading pattern bytes tested (0 = off) */
  uint32_t class_and_mask; /* 0x7f, or 0x5f when bit 5 is folded (case) */
  uint32_t class_ranges;   /* 1 or 2 */
  uint32_t class_lo[2], class_hi[2];
  uint32_t key_bytes;      /* leading pattern bytes a key covers (4..8) */
} olm_store_info_t;
int olm_store_inspect(const char *compiled_file, olm_store_info_t *out);

#ifdef __cplusplus
}
#endif
#endif /* OLM_B200_H */
