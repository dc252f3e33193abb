#!/usr/bin/env python3
"""pattern_ids_bench.py -- what the pattern-id pass costs (include/olm_b200.h "pattern ids").

For each workload (bench.py's WORKLOADS, patterns and device-resident haystacks, imported from
there) one matcher scans the haystack with ids off and on, alternating, after warm-up, and the
device time of every call (olm_cuda_timing_t.total_ms: scan + filter + id pass) is recorded.
Reported per workload: median device ms and GB/s off and on, their difference (the id pass), the
record count.  Checked per workload: the ids-on records have exactly the offsets, lengths and
match pointers of the ids-off records, and a seeded sample of records has ids whose catalogue
bytes equal the record's normalised source span.  One JSON line on stdout, with the card's name
and power limit read in the same run.

  python tools/pattern_ids_bench.py [--workloads cfg5,names,census-cpw] [--rounds 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import bench  # noqa: E402  (points fd 1 at stderr; the result line goes out through bench.emit)

GIB = 1 << 30
# workload -> haystack bytes
SIZES = {"cfg5": 16 * GIB, "names": 2 * GIB, "census-cpw": 2 * GIB}
N_PATTERNS = {"cfg5": 1_000_000}
SAMPLE = 100_000


def card(index: int) -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                         capture_output=True, text=True).stdout.strip()
    name, _, power = out.partition(",")
    return {"name": name.strip(), "power_limit": power.strip()}


def check_sample(torch, m, hay, rec, sflags, seed: int) -> int:
    """Ids of a seeded sample of records against the catalogue; returns the sample size."""
    from oracle.oracle import Oracle
    count = rec.shape[0]
    k = min(count, SAMPLE)
    g = torch.Generator(device=rec.device).manual_seed(seed)
    pick = torch.randperm(count, device=rec.device, generator=g)[:k].sort().values
    r = rec[pick]
    off, ln, pid = r[:, 0], r[:, 1] & 0xFFFFFFFF, (r[:, 1] >> 32) & 0xFFFFFFFF
    width = int(ln.max().item())
    idx = (off[:, None] + torch.arange(width, device=rec.device)[None, :]).clamp_(max=hay.numel() - 1)
    spans = hay[idx].cpu().numpy()
    ln, pid = ln.cpu().numpy(), pid.cpu().numpy()
    cat = {}
    for i in range(k):
        span = spans[i, :ln[i]].tobytes()
        norm = Oracle.transform(span + b"Q", *sflags)[0][:-1] if any(sflags) else span
        p = int(pid[i])
        if p not in cat:
            cat[p] = m.pattern(p)
        if cat[p] != norm:
            raise SystemExit(f"record {int(off[i])}+{int(ln[i])}: id {p} names {cat[p]!r}, span normalises to {norm!r}")
    return k


def run_workload(torch, synth_torch, name: str, tmp: str, args, dev) -> dict:
    from omega_match_b200 import Compiler, Matcher
    pats, sflags, mflags, hay_kind = bench.workload_patterns(name, N_PATTERNS.get(name, 0))
    n = SIZES[name]
    olm = str(Path(tmp) / f"ids_{name}.olm")
    t0 = time.time()
    Compiler.compile_from_buffer(olm, b"\n".join(pats) + b"\n", *map(bool, sflags))
    gen, _ = bench.device_haystack(torch, synth_torch, hay_kind, pats, 0, n, dev)
    hay = torch.empty(n + 256, dtype=torch.uint8, device=dev)
    hay[:n] = gen
    hay[n:] = 0
    del gen
    torch.cuda.synchronize()
    bench.log(f"[ids] {name}: {len(pats)} patterns, {n} bytes, set up in {time.time() - t0:.1f}s")
    m = Matcher(olm, device=dev.index)

    def call(ids: bool):
        m.set_pattern_ids(ids)
        cnt, ptr = m.match_device(hay.data_ptr(), n, **mflags)
        return cnt, ptr, m.last_timing()["total_ms"]

    for _ in range(args.warmup):
        call(False)
        call(True)
    off_ms, on_ms = [], []
    for _ in range(args.rounds):
        off_ms.append(call(False)[2])
        on_ms.append(call(True)[2])
    # the records of both modes, compared on the device
    cnt_off, ptr, _ = call(False)
    rec_off = torch.as_tensor(bench.DevArray(ptr, cnt_off), device=dev).clone()
    cnt_on, ptr, _ = call(True)
    rec_on = torch.as_tensor(bench.DevArray(ptr, cnt_on), device=dev)
    same = cnt_on == cnt_off and bool((rec_on[:, 0] == rec_off[:, 0]).all()) and bool(
        ((rec_on[:, 1] & 0xFFFFFFFF) == rec_off[:, 1]).all()) and bool((rec_on[:, 2] == rec_off[:, 2]).all())
    if not same:
        raise SystemExit(f"{name}: the ids-on records differ from the ids-off records")
    del rec_off
    checked = check_sample(torch, m, hay, rec_on, sflags, seed=0x1D5)
    m.set_pattern_ids(False)
    m.destroy()
    del hay, rec_on
    torch.cuda.empty_cache()
    off, on = float(np.median(off_ms)), float(np.median(on_ms))
    return {"bytes": n, "patterns": len(pats), "records": int(cnt_on), "match_flags": sorted(mflags),
            "ms_off": round(off, 3), "ms_on": round(on, 3), "id_pass_ms": round(on - off, 3),
            "id_pass_share": round((on - off) / off, 4), "gbs_off": round(n / off / 1e6, 1), "gbs_on": round(n / on / 1e6, 1),
            "ms_off_all": [round(x, 3) for x in off_ms], "ms_on_all": [round(x, 3) for x in on_ms],
            "records_equal": True, "ids_checked": checked}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg5,names,census-cpw")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    import synth_torch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = {"tool": "pattern_ids_bench", "gpu": card(0), "unit_ms": "device ms per call (olm_cuda_timing_t.total_ms)",
            "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for w in args.workloads.split(","):
            res = run_workload(torch, synth_torch, w, tmp, args, dev)
            line["workloads"][w] = res
            bench.log(f"[ids] {w}: {res}")
    bench.emit(line)


if __name__ == "__main__":
    main()
