#!/usr/bin/env python3
"""line_positions_bench.py -- what the line passes cost (include/olm_b200.h "lines").

For each workload (bench.py's WORKLOADS, patterns and device-resident haystacks, imported from there):
  device  median olm_cuda_timing_t.total_ms, alternating after warm-up, of
            match         match_device, ids off;
            positions     match_device + line_positions_device (newline facts + positions);
            lines         match_device + line_positions_device + matching_lines_device.
          The line passes add their time to the call's total_ms, so the differences are their cost.
  host    wall time from pinned host memory of matching_lines() and match_lines(), against
          match_arrays() + the numpy reference (searchsorted over flatnonzero(hay == 10)).
  check   every device position against a torch reference on the device (searchsorted over
          nonzero(hay == 10)); a seeded sample of 100 000 host positions against numpy; the records of
          match_lines() equal those of match_arrays(); the matching lines sum to the record count.
One JSON line on stdout, with the card's name and power limit read in the same run.

  python tools/line_positions_bench.py [--workloads cfg5,names,census-cpw] [--rounds 5] [--warmup 2]
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
from pattern_ids_bench import N_PATTERNS, SAMPLE, SIZES, card  # noqa: E402

GIB = 1 << 30


def numpy_positions(hay: np.ndarray, offsets: np.ndarray) -> np.ndarray:
    """The reference a caller would write without the library (test_lines_cpu.positions), its
    newline list built in 1 GiB pieces."""
    nl = np.concatenate([np.flatnonzero(hay[b:b + GIB] == 10) + b for b in range(0, hay.size, GIB)] or
                        [np.zeros(0, dtype=np.int64)]).astype(np.int64)
    i = np.searchsorted(nl, offsets.astype(np.int64))
    pad = np.concatenate([[-1], nl, [hay.size]])
    return np.stack([i, pad[i] + 1, pad[i + 1]], axis=1).astype(np.uint64)


def run_workload(torch, synth_torch, name: str, tmp: str, args, dev) -> dict:
    from omega_match_b200 import Compiler, Matcher
    pats, sflags, mflags, hay_kind = bench.workload_patterns(name, N_PATTERNS.get(name, 0))
    n = SIZES[name]
    olm = str(Path(tmp) / f"lines_{name}.olm")
    t0 = time.time()
    Compiler.compile_from_buffer(olm, b"\n".join(pats) + b"\n", *map(bool, sflags))
    gen, _ = bench.device_haystack(torch, synth_torch, hay_kind, pats, 0, n, dev)
    hay = torch.empty(n + 256, dtype=torch.uint8, device=dev)
    hay[:n] = gen
    hay[n:] = 0
    del gen
    torch.cuda.synchronize()
    newlines = int((hay[:n] == 10).sum().item())
    bench.log(f"[lines] {name}: {len(pats)} patterns, {n} bytes, {newlines} newlines, set up in {time.time() - t0:.1f}s")
    m = Matcher(olm, device=dev.index)
    pos = None

    def positions():
        nonlocal pos
        cnt, ptr = m.match_device(hay.data_ptr(), n, **mflags)
        if pos is None or pos.shape[0] < cnt:
            pos = torch.empty((max(cnt, 1), 3), dtype=torch.int64, device=dev)
        m.line_positions_device(ptr, cnt, hay.data_ptr(), 0, n, pos.data_ptr())
        return cnt, ptr

    def lines():
        cnt, _ = positions()
        return m.matching_lines_device(pos.data_ptr(), cnt)

    def total(f):
        f()
        return m.last_timing()["total_ms"]

    calls = {"match": lambda: total(lambda: m.match_device(hay.data_ptr(), n, **mflags)),
             "positions": lambda: total(positions), "lines": lambda: total(lines)}
    for _ in range(args.warmup):
        for f in calls.values():
            f()
    ms = {k: [] for k in calls}
    for _ in range(args.rounds):
        for k, f in calls.items():
            ms[k].append(f())
    med = {k: float(np.median(v)) for k, v in ms.items()}

    # check on the device: every position against searchsorted over the haystack's '\n' bytes
    cnt, ptr = positions()
    rec = torch.as_tensor(bench.DevArray(ptr, cnt), device=dev).clone()
    nl = torch.nonzero(hay[:n] == 10).flatten()
    i = torch.searchsorted(nl, rec[:, 0].contiguous())
    pad = torch.cat([torch.tensor([-1], device=dev), nl, torch.tensor([n], device=dev)])
    p = pos[:cnt]
    if not (bool((p[:, 0] == i).all()) and bool((p[:, 1] == pad[i] + 1).all()) and bool((p[:, 2] == pad[i + 1]).all())):
        raise SystemExit(f"{name}: device positions differ from the torch reference")
    n_lines, _ = m.matching_lines_device(pos.data_ptr(), cnt)
    want_lines = int(torch.unique_consecutive(i).numel())
    if n_lines != want_lines:
        raise SystemExit(f"{name}: {n_lines} matching lines, the reference has {want_lines}")
    del rec, nl, i, pad, p, pos

    # host path from pinned memory
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    host.copy_(hay[:n])
    hnp = host.numpy()
    del hay
    torch.cuda.empty_cache()

    def timed(f):
        t = time.perf_counter()
        r = f()
        return (time.perf_counter() - t) * 1e3, r

    host_calls = {"matching_lines": lambda: m.matching_lines(hnp, **mflags),
                  "match_lines": lambda: m.match_lines(hnp, **mflags),
                  "match_arrays_numpy": lambda: numpy_positions(hnp, m.match_arrays(hnp, **mflags)["offset"])}
    for f in host_calls.values():  # warm-up
        f()
    wall = {k: [] for k in host_calls}
    res = {}
    for _ in range(args.host_rounds):
        for k, f in host_calls.items():
            t, res[k] = timed(f)
            wall[k].append(t)
    got, ref_all = res["match_lines"], res["match_arrays_numpy"]
    arr = m.match_arrays(hnp, **mflags)
    if got.size != cnt or not (got["offset"] == arr["offset"]).all() or not (got["len"] == arr["len"]).all():
        raise SystemExit(f"{name}: match_lines records differ from match_arrays")
    rng = np.random.default_rng(20261021)
    pick = np.sort(rng.choice(got.size, size=min(SAMPLE, got.size), replace=False))
    sample_ref = numpy_positions(hnp, got["offset"][pick])
    mine = np.stack([got["line"][pick], got["line_begin"][pick], got["line_end"][pick]], axis=1)
    if not (mine == sample_ref).all() or not (ref_all[pick] == sample_ref).all():
        raise SystemExit(f"{name}: host positions differ from numpy")
    ml = res["matching_lines"]
    if ml.size != want_lines or int(ml["records"].sum()) != cnt:
        raise SystemExit(f"{name}: host matching lines differ")
    m.destroy()
    del host, hnp
    out = {"bytes": n, "patterns": len(pats), "records": int(cnt), "newlines": newlines, "matching_lines": n_lines,
           "match_flags": sorted(mflags)}
    for k in calls:
        out[f"ms_{k}"] = round(med[k], 3)
    out["positions_over_match"] = round(med["positions"] / med["match"], 4)
    out["lines_over_match"] = round(med["lines"] / med["match"], 4)
    for k, v in wall.items():
        out[f"host_ms_{k}"] = round(float(np.median(v)), 1)
    out["device_ms_all"] = {k: [round(x, 3) for x in v] for k, v in ms.items()}
    out["host_ms_all"] = {k: [round(x, 1) for x in v] for k, v in wall.items()}
    out["checked"] = {"device_positions": int(cnt), "host_sample": int(pick.size)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg5,names,census-cpw")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-rounds", type=int, default=2)
    args = ap.parse_args()
    import torch
    import synth_torch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = {"tool": "line_positions_bench", "gpu": card(0),
            "unit_ms": "device ms per call (olm_cuda_timing_t.total_ms); host: wall ms per call from pinned memory",
            "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for w in args.workloads.split(","):
            res = run_workload(torch, synth_torch, w, tmp, args, dev)
            line["workloads"][w] = res
            bench.log(f"[lines] {w}: {res}")
    bench.emit(line)


if __name__ == "__main__":
    main()
