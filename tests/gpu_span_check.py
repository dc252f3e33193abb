#!/usr/bin/env python3
"""GPU-box checker for the opt-in span path of the host entry point (OLM_HOST_SPAN_BYTES;
engine.cu `host_spans`): a host haystack scanned as consecutive byte-range shards, records
concatenated, `no_overlap` once on the whole.  Not collected by pytest.

  python tests/gpu_span_check.py        # spans of 4 MiB over 9..21 MiB haystacks vs the oracle
"""
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
os.environ["OLM_HOST_SPAN_BYTES"] = str(4 << 20)

import numpy as np  # noqa: E402

import inputs  # noqa: E402
from gpu_quick import run  # noqa: E402

FS = [(), ("no_overlap",), ("longest_only", "no_overlap"), ("word_boundary",), ("line_end", "longest_only", "no_overlap"),
      ("word_prefix",), ("word_suffix", "no_overlap")]


def main() -> int:
    bad = 0
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    for n in ((4 << 20) + 1, (8 << 20), (9 << 20) + 12345, (21 << 20) + 7):
        hay = inputs.text_haystack(n, 7 + n)
        # matches across every span edge: a long name written over each 4 MiB boundary
        for edge in range(4 << 20, n - 6, 4 << 20):
            hay[edge - 5:edge + 6] = np.frombuffer(b"Christopher", dtype=np.uint8)
        bad += run(f"names-spans-n{n}", names, (0, 0, 0), hay, FS)
        bad += run(f"names-cpw-spans-n{n}", names, (1, 1, 1), hay, FS[:3])
    pats = b"\n".join(inputs.synth_long_patterns(3000))
    hay = inputs.plant(inputs.synth_haystack((13 << 20) + 5, 99), inputs.synth_long_patterns(3000), 5, block=512)
    bad += run("synth3000-spans", pats, (0, 0, 0), hay, FS[:3])
    print("TOTAL BAD", bad)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
