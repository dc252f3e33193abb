"""Byte-range sharding of one haystack over several GPUs (SURVEY 8e), one process per GPU.

Host logic only -- which rank scans what, and how per-rank results become the single ordered
result -- on top of `torch.distributed` (NCCL on GPUs; the same code runs on gloo/CPU tensors
in the tests, with the scan itself supplied by the caller).

* No transform flag: rank r OWNS the start positions [own_begin, own_end); it needs the bytes
  [own_begin-16, own_end + largest_pattern_length] (previous byte for the word/line predicates,
  the match body, and the byte after the match).  A match is reported by the rank that owns its
  start -> no duplicates, nothing to reconcile.  End-of-buffer tests use the GLOBAL size.
* Transform flag: shards are multiples of the 4 MiB source window (matcher.c:946-947); windows
  are independent (SURVEY F4), so there is no halo at all.
* Per-rank results are sorted and shards are ordered by offset, so the global order is the
  concatenation in rank order.  `longest_only` never crosses shards; `no_overlap` can (the
  chain's last kept match of shard r may overlap the first of r+1), so it is applied once on the
  gathered array.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

WINDOW = 4 * 1024 * 1024
ALIGN = 16
RECORD_BYTES = 24
NO_NEWLINE = 2**64 - 1  # olm_newline_facts_t first / last of a range without '\n'


@dataclass(frozen=True)
class Shard:
    rank: int
    own_begin: int
    own_end: int
    slice_begin: int
    slice_end: int

    @property
    def own_len(self) -> int:
        return self.own_end - self.own_begin


def shard_plan(size: int, world: int, largest_pattern: int, windowed: bool) -> List[Shard]:
    """Split [0, size) into `world` contiguous ownership ranges plus the bytes each rank must hold:
    the library's own plan (include/olm_b200.h olm_shard_plan), the one its multi-GPU matcher uses."""
    if world < 1:
        raise ValueError("world must be >= 1")
    import ctypes as C

    from . import _lib
    lib = _lib.load()
    shards = []
    for r in range(world):
        sh = _lib.ShardC()
        if lib.olm_shard_plan(largest_pattern, int(bool(windowed)), size, world, r, C.byref(sh)) != 0:
            raise RuntimeError("olm_shard_plan failed")
        shards.append(Shard(r, sh.own_begin, sh.own_end, sh.slice_begin, sh.slice_end))
    return shards


def line_origins(facts, own_ranges, global_size: int) -> List[Tuple[int, int, int]]:
    """Every shard's line origin (include/olm_b200.h olm_line_origin_t: line, begin, next_newline) from
    the newline facts of all shards.  `facts[k]` = (newlines, first, last) of shard k's OWN range
    (olm_cuda_newline_facts: positions relative to the range; first / last None or 2**64-1 when it has no
    '\n'), `own_ranges[k]` = (own_begin, own_end); the ranges lie in byte order and cover
    [0, global_size) without gaps.  Pure host logic: a one-process-per-GPU job exchanges the facts (3
    words per rank) by its own means and calls this on every rank."""
    if len(facts) != len(own_ranges):
        raise ValueError("one facts entry per range")
    at = 0
    for b, e in own_ranges:
        if b != at or e < b:
            raise ValueError("the own ranges must cover [0, global_size) in order without gaps")
        at = e
    if at != global_size:
        raise ValueError("the own ranges must cover [0, global_size) in order without gaps")

    def none(v):
        return v is None or v == NO_NEWLINE

    out = []
    line = begin = 0
    for (count, first, last), (b, _) in zip(facts, own_ranges):
        out.append([line, begin, 0])
        line += int(count)
        if count:
            begin = b + int(last) + 1
    nxt = global_size
    for k in range(len(facts) - 1, -1, -1):
        out[k][2] = nxt
        count, first, _ = facts[k]
        if count and not none(first):
            nxt = own_ranges[k][0] + int(first)
    return [tuple(o) for o in out]


def gather_records(local, dist, dst: int = 0, group=None):
    """Variable-length gather of per-rank record tensors (shape [count, 3] int64 = 24-byte
    records) to rank `dst`, concatenated in rank order.  Returns the tensor on dst, None elsewhere."""
    import torch
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    counts = [torch.zeros(1, dtype=torch.int64, device=local.device) for _ in range(world)]
    dist.all_gather(counts, torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device), group=group)
    counts = [int(c.item()) for c in counts]
    if rank == dst:
        out = torch.empty((sum(counts), 3), dtype=torch.int64, device=local.device)
        reqs, at = [], 0
        for r, c in enumerate(counts):
            if r == dst:
                out[at:at + c].copy_(local)
            elif c:
                reqs.append(dist.irecv(out[at:at + c], src=r, group=group))
            at += c
        for q in reqs:
            q.wait()
        return out
    if local.shape[0]:
        dist.send(local.contiguous(), dst=dst, group=group)
    return None
