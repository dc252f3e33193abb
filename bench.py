#!/usr/bin/env python3
"""bench.py -- haystack GB/s of the matching hot path (BASELINE.json metric).

Workload of the line (`cfg5`, BASELINE.json configs[4]): a 16 GiB synthetic haystack (SURVEY 8d
generator, one planted pattern per 4 KiB) x 1,000,000 compiled patterns (length 6-24 over
a-zA-Z), byte-range sharded over N GPUs of one node, one process per GPU.  Weak scaling: every GPU
owns a 16 GiB byte range of an N x 16 GiB haystack.  The path has no exchange step; the one
collective is the gather of the per-rank sorted records to rank 0, done by the LIBRARY (C, NCCL:
olm_cuda_gather_records) -- torch.distributed only starts the job and carries the NCCL id.

A step = one pass of the hot path over the whole haystack:
  value    -- inputs already resident in HBM: every rank scans the start positions it owns
              (olm_cuda_match_shard), the records are gathered on rank 0.  K steps bracketed by
              barrier + cuda synchronize, max over ranks.
  e2e      -- the same from HOST memory through the C ABI: N=1 omega_list_matcher_match(pinned host
              pointer) = H2D + kernels + D2H of the records; N>1 every rank's slice from pinned host
              memory (olm_cuda_match_shard_host), gather on rank 0, D2H of the merged records there.
              `e2e.pageable` (N=1): the same call on ordinary (pageable) memory.
  roofline -- algorithmic bytes (1 byte per haystack byte, SURVEY 8d) / CUDA-event duration of the
              scan kernels, against the measured HBM copy bandwidth (MEASURED_PEAKS.json).
  cpu_baseline -- the unmodified reference library (oracle/_ref) with all host threads on a bounded
              prefix of the same haystack (SURVEY F8 puts the full size out of reach).
  strong   -- (N>1) the SAME 16 GiB split N ways, as BASELINE configs[4] words it.
  parity   -- (N>1) on 256 MiB per rank: the N-rank gathered record stream equals rank 0 scanning
              the whole buffer alone, record by record, for several flag sets and a transforming
              store; a mismatch fails the run.
  other_workloads -- (N=1) BASELINE configs[0..3] (names.txt / census on KJV-like text with their
              flags, the short-pattern store on its synthetic haystack), each from a process of its
              own (`--leg`), each with its own roofline and CPU baseline.

`--impl reference` times only the reference's CPU implementation on the same workload definition.
`--dump-outputs DIR` writes the records of the last timed step as .npy files (see dump_records), so
that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import os

os.environ.pop("OMP_NUM_THREADS", None)  # torchrun exports 1: the CPU baseline is to use every host core

import argparse
import json
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import inputs  # noqa: E402

GIB = 1 << 30
MIB = 1 << 20
METRIC = "haystack_throughput"
UNIT = "GB/s"
REF_PREFIX_BYTES = 8 * MIB  # --impl reference: the same prefix for every N
FLAG_ORDER = ("no_overlap", "longest_only", "word_boundary", "word_prefix", "word_suffix", "line_start", "line_end")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner there)
# must not get in between: fd 1 is pointed at stderr for the whole run and the line is
# written to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_traffic(workload: str):
    """ncu dram bytes of one scan launch of this workload (profiles/traffic.json), or None."""
    try:
        d = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        if workload in d:
            return d[workload]
        return d if workload == "cfg5" and "dram_bytes_per_launch" in d else None
    except Exception:
        return None


# ---------------------------------------------------------------------------------- workloads

def kjv_text(n: int, seed: int) -> np.ndarray:
    """KJV-like text: the pseudo-KJV haystack the reference's goldens are pinned on (SURVEY 8c)
    between stretches of punctuation / whitespace rich word salad."""
    pk = np.frombuffer(inputs.pseudo_kjv(), dtype=np.uint8)
    parts, size, i = [], 0, 0
    while size < n:
        t = inputs.text_haystack(MIB + 4099 * (i + 1), seed + i)
        parts += [pk, t]
        size += pk.size + t.size
        i += 1
    return np.concatenate(parts)[:n].copy()


TEXT_BASE_BYTES = 24 * MIB  # text haystacks: this much generated on the host, tiled on the device

WORKLOADS = {
    # name: (description, pattern set, store flags, match flags, haystack kind)
    "cfg5": ("BASELINE configs[4]: synthetic haystack x 1M compiled patterns, byte-range sharded", "synth_long", (0, 0, 0), {},
             "synth5"),
    "cfg4": ("BASELINE configs[3]: tlds.txt + generated 1-4 byte patterns x planted synthetic haystack", "short", (0, 0, 0), {},
             "synth4"),
    "names": ("BASELINE configs[0]: names.txt, baseline flags x KJV-like text", "names", (0, 0, 0), {}, "text"),
    "census-c": ("BASELINE configs[1]: surnames_us_census.txt, ignore-case + word_boundary x KJV-like text", "census",
                 (1, 0, 0), {"word_boundary": True}, "text"),
    "census-cpw": ("BASELINE configs[2]: census, ignore-case + ignore-punct + elide-whitespace + no_overlap + longest x "
                   "KJV-like text", "census", (1, 1, 1), {"no_overlap": True, "longest_only": True}, "text"),
    "names-synth": ("names.txt x synthetic haystack (round-1 leg)", "names", (0, 0, 0), {}, "synth5"),
    "names-cpw-synth": ("names.txt with all transform flags x synthetic haystack (round-1 leg)", "names", (1, 1, 1), {},
                        "synth5"),
}


def workload_patterns(name: str, n_patterns: int):
    _, pset, sflags, mflags, hay = WORKLOADS[name]
    if pset == "synth_long":
        pats = inputs.synth_long_patterns(n_patterns)
    elif pset == "short":
        pats = list(inputs._pattern_set("tlds")) + inputs.synth_short_patterns()
    else:
        pats = [p for p in inputs.case_patterns(dict(patterns=pset, store_flags=sflags)).split(b"\n") if p]
    return pats, sflags, dict(mflags), hay


def host_sample(hay_kind: str, n: int, pats) -> np.ndarray:
    """The first n bytes of a workload's haystack on the host (+ 64 spare bytes)."""
    if hay_kind == "text":
        h = kjv_text(max(n, TEXT_BASE_BYTES), 0x51)[:n] if n > TEXT_BASE_BYTES else kjv_text(TEXT_BASE_BYTES, 0x51)[:n]
    else:
        seed = inputs.SEED_H5 if hay_kind == "synth5" else inputs.SEED_H4
        h = inputs.plant(inputs.synth_haystack(n, seed), pats, seed ^ 0x77)
    buf = np.zeros(n + 64, dtype=np.uint8)
    buf[:n] = h[:n]
    return buf


def device_haystack(torch, synth_torch, hay_kind: str, pats, begin: int, end: int, dev):
    """Bytes [begin, end) of a workload's haystack, generated on the GPU (text: a host base tiled)."""
    if hay_kind == "text":
        base = torch.from_numpy(kjv_text(TEXT_BASE_BYTES, 0x51)).to(dev)
        reps = (end - begin + base.numel() - 1) // base.numel() + 1
        off = begin % base.numel()
        return base.repeat(reps)[off:off + (end - begin)].contiguous(), 0
    seed = inputs.SEED_H5 if hay_kind == "synth5" else inputs.SEED_H4
    gen_b = (begin // 4096) * 4096
    gen_e = ((end + 4095) // 4096) * 4096
    gen = synth_torch.synth_haystack_torch(gen_e - gen_b, seed, start=gen_b, device=dev)
    pb, pl = synth_torch.pack_patterns(pats, dev)
    planted = synth_torch.plant_torch(gen, pb, pl, seed ^ 0x77, start=gen_b)
    return gen[begin - gen_b:end - gen_b], planted


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


class DevArray:
    """Zero-copy torch view of library-owned device memory (24-byte records as [n,3] int64)."""

    def __init__(self, ptr: int, count: int):
        self.__cuda_array_interface__ = {"shape": (count, 3), "typestr": "<i8", "data": (ptr, False), "version": 2}


DUMP_MAX_RECORDS = 1 << 21  # three float64 arrays of this length: 48 MiB


def dump_records(out_dir: str, torch, dev, rec_ptr: int, count: int):
    """The records a caller of the timed path receives, as out_dir/<name>.npy (float64):
    count.npy   [1]  the number of records,
    index.npy   [k]  which records are stored: all of them, or for more than DUMP_MAX_RECORDS a
                     fixed seeded sample (sorted), so that the files stay under 64 MB,
    offset.npy  [k]  their offsets (exact: below 2**53), length.npy [k] their lengths.
    (A record's `match` pointer is match_ptr_base + offset, with base 0 here: nothing to add.)"""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    if count > DUMP_MAX_RECORDS:
        idx = np.sort(np.random.default_rng(20261020).choice(count, DUMP_MAX_RECORDS, replace=False))
    else:
        idx = np.arange(count, dtype=np.int64)
    rec = np.zeros((0, 3), dtype=np.int64)
    if count:
        rec = torch.as_tensor(DevArray(rec_ptr, count), device=dev)[torch.from_numpy(idx).to(dev)].cpu().numpy()
    np.save(d / "count.npy", np.array([count], dtype=np.float64))
    np.save(d / "index.npy", idx.astype(np.float64))
    np.save(d / "offset.npy", rec[:, 0].astype(np.float64))
    np.save(d / "length.npy", (rec[:, 1] & 0xFFFFFFFF).astype(np.float64))
    log(f"[bench] wrote {idx.size} of {count} records of the last timed step to {d}")


# ---------------------------------------------------------------------------------- CPU baseline

def cpu_reference_setup(pattern_buf: bytes, store_flags):
    """The unmodified reference (oracle/_ref) with every host core, else the oracle port on one."""
    from oracle.oracle import Oracle, RefLib, ref_available
    tmp = tempfile.NamedTemporaryFile(suffix=".olm", delete=False)
    tmp.close()
    if ref_available():
        RefLib.compile(tmp.name, pattern_buf, *store_flags)
        ref = RefLib(tmp.name)  # create() = set_num_threads(0) = all cores (matcher.c:509)
        return "reference", ref, ref.threads(), tmp.name
    o = Oracle.from_patterns(pattern_buf, *store_flags)
    return "port", o, 1, tmp.name


def cpu_match_timed(kind, obj, sample: np.ndarray, n: int, mflags):
    if kind == "reference":
        return obj.match_timed(sample, n, **mflags)
    t0 = time.perf_counter()
    m = obj.match(sample[:n], **mflags)
    return m.size, time.perf_counter() - t0


def cpu_baseline_for(pats, sflags, mflags, hay_kind, matcher, budget_s: float, max_bytes: int):
    """Times the reference on a prefix sized for ~budget_s seconds and checks the CUDA path on the same bytes."""
    pbuf = b"\n".join(pats) + b"\n"
    kind, obj, cores, tmpname = cpu_reference_setup(pbuf, sflags)
    try:
        n = MIB
        sample = host_sample(hay_kind, max_bytes if hay_kind == "text" else n, pats)
        _, dt = cpu_match_timed(kind, obj, sample, n, mflags)
        want = int(min(max_bytes, max(n, n * budget_s / max(dt, 1e-4)))) & ~4095
        if want > n:
            n = want
            if hay_kind != "text":
                sample = host_sample(hay_kind, n, pats)
        cnt, dt = cpu_match_timed(kind, obj, sample, n, mflags)
        ref_m = obj.match(sample[:n], **mflags) if kind == "port" else obj.match(sample[:n].tobytes(), **mflags)
        got = matcher.match_arrays(sample[:n], **mflags)
        same = got.size == ref_m.size and bool((got["offset"] == ref_m["offset"]).all()) and bool(
            (got["len"] == ref_m["len"]).all())
        return {"value": n / dt / 1e9, "unit": UNIT, "cores": cores, "kind": kind,
                "sample": f"first {n} bytes of the same haystack, {cnt} matches, {dt:.2f}s; "
                          f"CUDA result on the same bytes identical: {same}"}
    finally:
        os.unlink(tmpname)


def run_reference(args):
    """--impl reference: the reference's CPU implementation on a bounded prefix per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    pats, sflags, mflags, hay_kind = workload_patterns(args.workload, args.patterns)
    kind, obj, cores, tmpname = cpu_reference_setup(b"\n".join(pats) + b"\n", sflags)
    n = REF_PREFIX_BYTES
    sample = host_sample(hay_kind, n, pats)
    for _ in range(args.warmup):
        cpu_match_timed(kind, obj, sample, n, mflags)
    t, cnt = 0.0, 0
    for _ in range(args.steps):
        cnt, dt = cpu_match_timed(kind, obj, sample, n, mflags)
        t += dt
    val = n * args.steps / t / 1e9
    os.unlink(tmpname)
    emit({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
          "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
          "config": workload_config(args, n_bytes=n, note="bounded prefix of the workload per step (the same for every N)"),
          "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                           "sample": f"first {n} bytes of the haystack, {cnt} matches"},
          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0})


def workload_config(args, n_bytes=None, note=None):
    c = {"workload": WORKLOADS[args.workload][0],
         "haystack_bytes": int(n_bytes if n_bytes is not None else args.size_gib * GIB * args.gpus),
         "haystack_bytes_per_gpu": int(n_bytes if n_bytes is not None else args.size_gib * GIB),
         "patterns": args.patterns if args.workload == "cfg5" else None,
         "match_flags": sorted(WORKLOADS[args.workload][3]), "l2": "haystack is far larger than the 126 MB L2, no flush needed",
         "parallelism": f"byte-range shards x{args.gpus}, one process per GPU, records gathered by the library over NCCL"}
    if note:
        c["note"] = note
    return c


# ---------------------------------------------------------------------------------- our arm

def run_ours(args):
    import torch
    import torch.distributed as dist
    import synth_torch
    from omega_match_b200 import Compiler, Matcher, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def reduce_max_sum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world == 1:
            return t.tolist(), t.tolist()
        mx, sm = t.clone(), t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        return mx.tolist(), sm.tolist()

    def new_comm(matcher):  # the library's own communicator; torch only carries the 128-byte id
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(Matcher.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        matcher.comm_init(idt.cpu().numpy().tobytes(), rank, world)

    pats, sflags, mflags, hay_kind = workload_patterns(args.workload, args.patterns)
    pbuf = b"\n".join(pats) + b"\n"
    olm = f"/tmp/olm_bench_{os.getuid()}_{args.workload}_{len(pats)}.olm"
    t0 = time.time()
    if local == 0:
        st = Compiler.compile_from_buffer(olm + ".tmp", pbuf, *map(bool, sflags))
        os.replace(olm + ".tmp", olm)
        log(f"[bench] compiled {len(pats)} patterns in {time.time() - t0:.1f}s: {st}")
    barrier()
    m = Matcher(olm, device=local)
    if world > 1:
        new_comm(m)

    total = int(args.size_gib * GIB) * world  # weak scaling: size_gib per GPU
    own_b, own_e, sl_b, sl_e = m.shard_plan(total, world, rank)
    t0 = time.time()
    gen, planted = device_haystack(torch, synth_torch, hay_kind, pats, sl_b, sl_e, dev)
    hay = torch.empty(((sl_e - sl_b + 15) // 16) * 16 + 256, dtype=torch.uint8, device=dev)  # 16-byte aligned slice
    hay[:sl_e - sl_b] = gen
    del gen
    torch.cuda.synchronize()
    log(f"[bench] rank {rank}: slice [{sl_b},{sl_e}) own [{own_b},{own_e}) generated in {time.time() - t0:.1f}s, {planted} planted")
    shard_flags = {k: v for k, v in mflags.items() if k != "no_overlap"}
    no_overlap = bool(mflags.get("no_overlap"))

    def step():
        cnt, ptr = m.match_shard(hay.data_ptr(), sl_b, sl_e - sl_b, own_b, own_e, total, 0, **shard_flags)
        t = m.last_timing()
        tot = cnt
        if world > 1:
            tot, ptr = m.gather_records(ptr, cnt, 0, no_overlap)
        elif no_overlap:
            tot = m.no_overlap_device(ptr, cnt)
        return cnt, tot, t, ptr

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    scan_ms, launches, cnt, merged_total, rec_ptr = 0.0, 0, 0, 0, 0
    for _ in range(args.steps):
        cnt, merged_total, t, rec_ptr = step()
        scan_ms += t["scan_ms"]
        launches += int(t["kernel_launches"])
    torch.cuda.synchronize()
    barrier()
    dt = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    mx, sm = reduce_max_sum([dt, scan_ms / args.steps, float(cnt), float(launches)])
    dt, scan_ms_step, total_matches, launches = mx[0], mx[1], int(sm[2]), int(sm[3])
    value = total * args.steps / dt / 1e9
    if args.dump_outputs and rank == 0:  # before the e2e calls below reuse the matcher's record buffer
        dump_records(args.dump_outputs, torch, dev, rec_ptr, merged_total)

    # ---- e2e: host buffers, H2D + kernels (+ gather) + D2H inside the timed region
    own_len = sl_e - sl_b
    host = torch.empty(own_len + 64, dtype=torch.uint8, pin_memory=True)
    host[:own_len].copy_(hay[:own_len])
    torch.cuda.synchronize()
    lib = _lib.load()
    e2e_steps = max(1, min(args.steps, 3))
    d2h = [0]
    rec_host = [None]
    h2d_ms = [0.0]
    flag_ints = [int(bool(mflags.get(k))) for k in FLAG_ORDER]

    def e2e_step():
        if world == 1:
            res = lib.omega_list_matcher_match(m._matcher, host.data_ptr(), total, *flag_ints)
            if not res:
                raise SystemExit("omega_list_matcher_match failed")
            d2h[0] = int(res.contents.count) * 24
            lib.omega_match_results_destroy(res)
            h2d_ms[0] = max(h2d_ms[0], m.last_timing()["h2d_ms"])
            return
        # this rank's slice from pinned host memory (segmented H2D overlapped with the scan), the library's
        # gather to rank 0, and the merged records to rank 0's host memory: the result a caller would hold
        c, ptr_ = m.match_shard_host(host.data_ptr(), sl_b, own_len, own_b, own_e, total, 0, **shard_flags)
        h2d_ms[0] = max(h2d_ms[0], m.last_timing()["h2d_ms"])
        tot, gptr = m.gather_records(ptr_, c, 0, no_overlap)
        if rank == 0 and tot:
            rec = torch.as_tensor(DevArray(gptr, tot), device=dev)
            if rec_host[0] is None or rec_host[0].numel() < rec.numel():  # pinned, recycled (as the host API does)
                rec_host[0] = torch.empty(rec.numel() + rec.numel() // 8, dtype=rec.dtype, pin_memory=True)
            rec_host[0][:rec.numel()].view_as(rec).copy_(rec, non_blocking=True)
            d2h[0] = rec.numel() * 8
        torch.cuda.synchronize()

    e2e_step()
    if rank == 0:
        log(f"[bench] e2e call breakdown (device events, ms): {m.last_timing()}")
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    barrier()
    e2e_dt = time.perf_counter() - t0
    mx, sm = reduce_max_sum([e2e_dt, float(own_len), float(d2h[0]), h2d_ms[0]])
    e2e = {"value": total * e2e_steps / mx[0] / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(sm[1]),
           "d2h_bytes_per_step": int(sm[2]), "steps": e2e_steps, "h2d_ms_max_over_ranks": mx[3],
           "api": "omega_list_matcher_match(pinned host ptr)" if world == 1 else
           "per rank: pinned host slice -> olm_cuda_match_shard_host; olm_cuda_gather_records to rank 0; merged records D2H on rank 0"}
    if world == 1 and not args.no_extra:
        # the same call on ordinary memory, as main.c's mmap and the cffi wrapper's copy hand it over
        n_pg = min(total, 4 * GIB)
        pageable = np.empty(n_pg + 64, dtype=np.uint8)
        pageable[:n_pg] = host[:n_pg].numpy()
        pg = []
        for _ in range(3):  # (the first call also allocates the library's pinned staging slots)
            t0 = time.perf_counter()
            res = lib.omega_list_matcher_match(m._matcher, pageable.ctypes.data, n_pg, *flag_ints)
            pg.append(time.perf_counter() - t0)
            if res:
                lib.omega_match_results_destroy(res)
        if res:
            e2e["pageable"] = {"value": n_pg / min(pg[1:]) / 1e9, "first_call": n_pg / pg[0] / 1e9, "unit": UNIT, "bytes": n_pg,
                               "host_threads": int(lib.omega_matcher_get_num_threads(m._matcher)),
                               "note": "haystack in ordinary (pageable) host memory; best of two calls after the first"}
        del pageable
    del host

    # ---- N>1: strong scaling of the stated config and parity of the gathered stream
    strong = parity = None
    if world > 1:
        strong = strong_block(args, m, hay, total // world, world, rank, barrier, torch, reduce_max_sum)
        parity = parity_block(m, pats, hay_kind, world, rank, local, dev, barrier, torch, synth_torch, new_comm)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    own_bytes = own_e - own_b
    achieved = own_bytes / (scan_ms_step * 1e-3) / 1e9 if scan_ms_step > 0 else 0.0
    traffic = kernel_traffic(args.workload)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args),
            "matches_per_step": total_matches, "records_on_rank0": merged_total,
            "roofline": {"bound": "hbm", "kernel": "scan_kernel (+ prefix/place/redo, 5 launches per step and rank)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": own_bytes, "kernel_ms": scan_ms_step,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch")},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
    if strong:
        line["strong"] = strong
    if parity:
        line["parity"] = parity
    if world == 1 and not args.no_cpu:
        try:
            line["cpu_baseline"] = cpu_baseline_for(pats, sflags, mflags, hay_kind, m, 10.0, 256 * MIB)
        except Exception as e:  # the baseline is reported, never required
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)}
    if world == 1 and args.workload == "cfg5" and not args.no_extra:
        del hay
        m.destroy()
        torch.cuda.empty_cache()
        line["other_workloads"] = {w: run_leg(w, args) for w in ("cfg4", "names", "census-c", "census-cpw")}
    emit(line)
    if parity and not parity["ok"]:
        raise SystemExit("bench: the gathered multi-GPU stream differs from the single-GPU stream")
    if world > 1:
        dist.destroy_process_group()


def strong_block(args, m, hay, size, world, rank, barrier, torch, reduce_max_sum):
    """BASELINE configs[4] as worded: ONE haystack of size_gib, byte-range sharded over the N GPUs.  Rank r
    scans start positions [r*size/N, (r+1)*size/N) -- the bytes come from the front of its resident buffer
    (whose byte 0 stands for the first byte of that rank's slice)."""
    own_b, own_e, sl_b, sl_e = m.shard_plan(size, world, rank)
    steps = max(1, min(args.steps, 3))

    def step():
        cnt, ptr = m.match_shard(hay.data_ptr(), sl_b, sl_e - sl_b, own_b, own_e, size, 0)
        m.gather_records(ptr, cnt, 0, False)
        return m.last_timing()["scan_ms"]

    step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    k_ms = 0.0
    for _ in range(steps):
        k_ms += step()
    torch.cuda.synchronize()
    barrier()
    dt = time.perf_counter() - t0
    mx, _ = reduce_max_sum([dt, k_ms / steps])
    return {"value": size * steps / mx[0] / 1e9, "unit": UNIT, "haystack_bytes": int(size), "steps": steps,
            "ms_per_step": mx[0] / steps * 1e3, "kernel_ms_max_over_ranks": mx[1],
            "note": "the same haystack size as N=1, split N ways; gather included"}


def parity_block(m, pats, hay_kind, world, rank, local, dev, barrier, torch, synth_torch, new_comm):
    """1-GPU vs N-GPU streams on the same bytes (SURVEY 8d 'large-scale parity (ii)'): 256 MiB per rank; every
    rank scans its shard, the library gathers; rank 0 also scans the whole buffer alone; the two record arrays
    must be identical (offset, len, order).  Plain store with three flag sets, then a transforming store."""
    from omega_match_b200 import Compiler, Matcher
    per = 256 * MIB
    size = per * world
    out = {"haystack_bytes": size, "cases": [], "ok": True}
    olm2 = f"/tmp/olm_bench_{os.getuid()}_parity_cw.olm"
    if local == 0:
        sub = pats[:20000] + [b"zq", b"The", b"of", b"a b"]
        Compiler.compile_from_buffer(olm2 + ".tmp", b"\n".join(sub) + b"\n", True, False, True)
        os.replace(olm2 + ".tmp", olm2)
    barrier()
    m2 = Matcher(olm2, device=local)
    new_comm(m2)
    flagsets = [{}, {"no_overlap": True}, {"longest_only": True, "word_boundary": True}]
    empty = torch.empty((0, 2), dtype=torch.int64, device=dev)
    for label, mm in (("plain", m), ("ignore-case + elide-whitespace", m2)):
        own_b, own_e, sl_b, sl_e = mm.shard_plan(size, world, rank)
        gen, _ = device_haystack(torch, synth_torch, hay_kind, pats, sl_b, sl_e, dev)
        sl = torch.zeros(((sl_e - sl_b + 15) // 16) * 16 + 256, dtype=torch.uint8, device=dev)
        sl[:sl_e - sl_b] = gen
        whole = None
        if rank == 0:
            g2, _ = device_haystack(torch, synth_torch, hay_kind, pats, 0, size, dev)
            whole = torch.zeros(size + 256, dtype=torch.uint8, device=dev)
            whole[:size] = g2
            del g2
        del gen
        torch.cuda.synchronize()
        for fs in flagsets:
            sf = {k: v for k, v in fs.items() if k != "no_overlap"}
            cnt, ptr = mm.match_shard(sl.data_ptr(), sl_b, sl_e - sl_b, own_b, own_e, size, 0, **sf)
            tot, gptr = mm.gather_records(ptr, cnt, 0, bool(fs.get("no_overlap")))
            if rank == 0:
                got = torch.as_tensor(DevArray(gptr, tot), device=dev)[:, :2].clone() if tot else empty
                c1, p1 = mm.match_device(whole.data_ptr(), size, 0, **fs)
                ref = torch.as_tensor(DevArray(p1, c1), device=dev)[:, :2].clone() if c1 else empty
                got[:, 1] &= 0xFFFFFFFF
                ref[:, 1] &= 0xFFFFFFFF
                same = bool(tot == c1 and torch.equal(got, ref))
                out["cases"].append({"store": label, "flags": sorted(fs), "records": int(c1), "gathered": int(tot),
                                     "identical": same})
                out["ok"] = out["ok"] and same
            barrier()
        del sl, whole
        torch.cuda.empty_cache()
    m2.destroy()
    return out


# ---------------------------------------------------------------------------------- other workloads (N=1)

_EXTRA_DEADLINE = [None]


def run_leg(name: str, args):
    """One workload in a process of its own (`bench.py --leg name`) -> its dict, or {"error": ...}."""
    if _EXTRA_DEADLINE[0] is None:
        _EXTRA_DEADLINE[0] = time.time() + 300.0
    tmo = min(110.0, _EXTRA_DEADLINE[0] - time.time())
    if tmo < 25.0:
        return {"error": "skipped: the extra legs' time budget is used up"}
    try:
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--leg", name] + (["--no-cpu"] if args.no_cpu else []),
                           capture_output=True, text=True, timeout=tmo)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": (r.stderr or r.stdout)[-400:]}
        return json.loads(lines[-1])
    except Exception as e:
        return {"error": repr(e)[:300]}


def leg_main(args):
    """BASELINE configs[0..3]: device-timed GB/s on a resident haystack, roofline, CPU baseline on a slice."""
    import torch
    import synth_torch
    from omega_match_b200 import Compiler, Matcher
    name = args.leg
    pats, sflags, mflags, hay_kind = workload_patterns(name, args.patterns)
    olm = f"/tmp/olm_bench_{os.getuid()}_leg_{name}.olm"
    Compiler.compile_from_buffer(olm, b"\n".join(pats) + b"\n", *map(bool, sflags))
    n = int((4 if hay_kind != "text" else 2) * GIB)
    dev = torch.device("cuda", 0)
    gen, _ = device_haystack(torch, synth_torch, hay_kind, pats, 0, n, dev)
    hay = torch.zeros(n + 256, dtype=torch.uint8, device=dev)
    hay[:n] = gen
    del gen
    torch.cuda.synchronize()
    out = {"workload": WORKLOADS[name][0], "haystack_bytes": n, "match_flags": sorted(mflags)}
    with Matcher(olm) as m:
        best, launches, cnt, t_best = None, 0, 0, None
        for i in range(4):
            cnt, _ = m.match_device(hay.data_ptr(), n, **mflags)
            t = m.last_timing()
            if i and (best is None or t["total_ms"] < best):
                best, t_best = t["total_ms"], t
            launches = int(t["kernel_launches"])
        peak, peak_src = measured_peak()
        achieved = n / (best * 1e-3) / 1e9
        traffic = kernel_traffic(name)
        out.update({"value": achieved, "unit": UNIT, "matches_per_step": cnt, "gpu_launches_per_step": launches,
                    "roofline": {"bound": "hbm", "kernel": "all kernels of one call: window descriptors, scan, prefix/place/redo, filter",
                                 "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                 "peak_source": peak_src, "algorithmic_bytes_per_launch": n, "kernel_ms": best,
                                 "scan_ms": t_best["scan_ms"], "transform_ms": t_best["transform_ms"],
                                 "filter_ms": t_best["filter_ms"],
                                 "traffic": (traffic or {}).get("dram_bytes_per_launch")}})
        if not args.no_cpu:
            try:
                out["cpu_baseline"] = cpu_baseline_for(pats, sflags, mflags, hay_kind, m, 4.0, TEXT_BASE_BYTES)
            except Exception as e:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)}
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS))
    ap.add_argument("--size-gib", type=float, default=16.0)
    ap.add_argument("--patterns", type=int, default=1_000_000)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extra", "--no-experimental", dest="no_extra", action="store_true",
                    help="skip other_workloads and the pageable e2e figure (N=1)")
    ap.add_argument("--leg", default=None, choices=sorted(WORKLOADS), help="internal: one other_workloads leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step to DIR/<name>.npy (float64, at most 48 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times match counts only)")
    if args.leg:
        return leg_main(args)
    if args.warmup < 3 and args.impl == "ours":
        log("[bench] note: fewer than 3 warm-up steps requested")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
