#!/usr/bin/env python3
"""stream_bench.py -- what scanning a haystack as a stream of pieces costs (include/olm_b200.h "Streams").

For each workload (bench.py's WORKLOADS, patterns and device-resident haystacks, imported from there):
  device  wall ms (host clock; every call ends synchronised) of one match_device over the whole buffer
          against device streams of 64 MiB, 256 MiB and 1 GiB pieces pushed from the same buffer,
          alternating after warm-up.
  host    cfg5 only: from pinned host memory, one omega_list_matcher_match against a stream of 1 GiB
          host pushes.
  check   the stream's records, piece by piece, equal the single call's.
One JSON line on stdout, with the card's name and power limit read in the same run.

  python tools/stream_bench.py [--workloads cfg5,names,census-cpw] [--rounds 5] [--warmup 1]
"""
from __future__ import annotations

import argparse
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402  (points fd 1 at stderr; the result line goes out through bench.emit)
from pattern_ids_bench import N_PATTERNS, SIZES, card  # noqa: E402

MIB = 1 << 20
PIECES = {"64MiB": 64 * MIB, "256MiB": 256 * MIB, "1GiB": 1024 * MIB}


def run_workload(torch, synth_torch, name: str, tmp: str, args, dev) -> dict:
    from omega_match_b200 import Compiler, Matcher
    pats, sflags, mflags, hay_kind = bench.workload_patterns(name, N_PATTERNS.get(name, 0))
    n = SIZES[name]
    olm = str(Path(tmp) / f"stream_{name}.olm")
    Compiler.compile_from_buffer(olm, b"\n".join(pats) + b"\n", *map(bool, sflags))
    gen, _ = bench.device_haystack(torch, synth_torch, hay_kind, pats, 0, n, dev)
    hay = torch.empty(n + 256, dtype=torch.uint8, device=dev)
    hay[:n] = gen
    hay[n:] = 0
    del gen
    torch.cuda.synchronize()
    m = Matcher(olm, device=dev.index)
    base = hay.data_ptr()

    def one_call():
        t = time.perf_counter()
        cnt, ptr = m.match_device(base, n, **mflags)
        return (time.perf_counter() - t) * 1e3, cnt, ptr

    def stream(piece, check=None):
        at, t = 0, time.perf_counter()
        with m.stream(match_ptr_base=base, **mflags) as s:
            for b in range(0, n, piece):
                ptr, c = s.push_device(base + b, min(piece, n - b), last=b + piece >= n)
                if check is not None:
                    part = torch.as_tensor(bench.DevArray(ptr, c), device=dev) if c else None
                    if c and not torch.equal(part, check[at:at + c]):
                        raise SystemExit(f"{name}: stream of {piece} byte pieces differs at record {at}")
                at += c
        return (time.perf_counter() - t) * 1e3, at

    calls = {"one_call": lambda: one_call()[0]}
    for k, p in PIECES.items():
        calls[f"stream_{k}"] = lambda p=p: stream(p)[0]
    for _ in range(args.warmup):
        for f in calls.values():
            f()
    ms = {k: [] for k in calls}
    for _ in range(args.rounds):
        for k, f in calls.items():
            ms[k].append(f())
    med = {k: float(np.median(v)) for k, v in ms.items()}
    _, cnt, ptr = one_call()
    whole = torch.as_tensor(bench.DevArray(ptr, cnt), device=dev).clone() if cnt else torch.empty((0, 3), dtype=torch.int64, device=dev)
    for p in PIECES.values():
        _, got = stream(p, whole)
        if got != cnt:
            raise SystemExit(f"{name}: stream of {p} byte pieces returned {got} records, one call {cnt}")
    res = {"bytes": n, "records": int(cnt), "match_flags": sorted(mflags), "records_identical": True}
    for k in calls:
        res[f"ms_{k}"] = round(med[k], 2)
        res[f"gbps_{k}"] = round(n / med[k] / 1e6, 1)
        if k != "one_call":
            res[f"{k}_over_one_call"] = round(med[k] / med["one_call"], 4)
    res["ms_all"] = {k: [round(x, 2) for x in v] for k, v in ms.items()}
    del whole

    if name == "cfg5":  # host pushes from pinned memory against one host call
        host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        host.copy_(hay[:n])
        hnp = host.numpy()
        del hay
        torch.cuda.empty_cache()

        def host_call():
            t = time.perf_counter()
            r = m.match_arrays(hnp, **mflags)
            return (time.perf_counter() - t) * 1e3, r

        def host_stream():
            t, parts = time.perf_counter(), []
            with m.stream(**mflags) as s:
                for b in range(0, n, 1024 * MIB):
                    parts.append(s.push(hnp[b:b + 1024 * MIB], last=b + 1024 * MIB >= n))
            return (time.perf_counter() - t) * 1e3, np.concatenate(parts)

        host_call(), host_stream()
        wall = {"host_call": [], "host_stream_1GiB": []}
        for _ in range(args.host_rounds):
            t1, r1 = host_call()
            t2, r2 = host_stream()
            wall["host_call"].append(t1)
            wall["host_stream_1GiB"].append(t2)
        if not (np.array_equal(r1["offset"], r2["offset"]) and np.array_equal(r1["len"], r2["len"])):
            raise SystemExit("cfg5: host stream records differ from one host call")
        for k, v in wall.items():
            res[f"ms_{k}"] = round(float(np.median(v)), 1)
            res[f"gbps_{k}"] = round(n / float(np.median(v)) / 1e6, 1)
        res["host_stream_over_host_call"] = round(res["ms_host_stream_1GiB"] / res["ms_host_call"], 4)
        res["host_ms_all"] = {k: [round(x, 1) for x in v] for k, v in wall.items()}
        del host, hnp
    m.destroy()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg5,names,census-cpw")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--host-rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import synth_torch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = {"tool": "stream_bench", "gpu": card(0),
            "unit_ms": "wall ms per haystack (host clock around calls that end synchronised); GB/s = bytes / that",
            "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for w in args.workloads.split(","):
            res = run_workload(torch, synth_torch, w, tmp, args, dev)
            line["workloads"][w] = res
            bench.log(f"[stream] {w}: {res}")
    bench.emit(line)


if __name__ == "__main__":
    main()
