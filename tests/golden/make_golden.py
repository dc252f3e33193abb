#!/usr/bin/env python3
"""Regenerates tests/golden/ from the reference checkout (run in the build container only).

  OLM_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden.py

1. data/*.xz      -- the reference's own pattern lists, haystacks and expected-output files
                     (reference data/, byte-identical, xz-compressed), so that the tests
                     never read the reference checkout.
2. vectors.json   -- results of the UNMODIFIED reference library (oracle/_ref, built by
                     `make -C oracle ref`) on seeded synthetic inputs over the flag matrix of
                     perf_test.py:69-91 plus word-prefix/word-suffix: match count and an
                     order-sensitive digest of the (offset,len) stream.  Inputs are
                     regenerated from the seeds by tests/inputs.py.

The script re-executes itself with MALLOC_PERTURB_=255 (glibc then hands out zero-filled
memory).  Reason: with a transform flag the reference's short-matcher word-boundary test reads
scratch[M_w] (matcher.c:812,:830,:848 on the re-used buffer of transform_table.c:40-51); for a
window longer than everything normalised before, that byte was never written and is
uninitialised heap memory.  Observed here: `census-text-cpw` + word_boundary returned 139148
or 139149 matches depending on what the process had freed before.  Zero-filled allocations are
what a fresh process gets from the kernel and what the oracle and the CUDA path assume.
"""
import json
import lzma
import os
import sys
from pathlib import Path

if os.environ.get("MALLOC_PERTURB_") != "255":
    os.execve(sys.executable, [sys.executable] + sys.argv, dict(os.environ, MALLOC_PERTURB_="255"))

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

if not os.environ.get("OLM_REFERENCE_DIR"):
    sys.exit("usage: OLM_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden.py "
             "(oracle/_ref built from the same checkout: make -C oracle ref)")
REF_DATA = Path(os.environ["OLM_REFERENCE_DIR"]) / "data"  # the checkout oracle/_ref was built from
FILES = ["names.txt", "surnames_us_census.txt", "tlds.txt", "usernames.txt", "haystack_email.txt",
         "line_anchor_haystack.txt", "line_anchor_patterns.txt", "line_exact_match_haystack.txt",
         "line_exact_match_patterns.txt", "line_exact_haystack.txt", "line_exact_patterns.txt",
         "punct_haystack.txt", "small_hay.txt", "small_pats.txt",
         "expected_word_prefix.txt", "expected_word_suffix.txt", "expected_line_start.txt",
         "expected_line_end.txt", "expected_line_start_word_boundary.txt", "expected_line_exact_match.txt",
         "matcher_found.txt", "grep_found.txt"]


def main():
    (HERE / "data").mkdir(exist_ok=True)
    for name in FILES:
        raw = (REF_DATA / name).read_bytes()
        (HERE / "data" / (name + ".xz")).write_bytes(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME))
        print(f"{name}: {len(raw)} bytes")

    import inputs  # tests/inputs.py
    from oracle.oracle import Oracle, RefLib

    vectors = []
    tmp = Path("/tmp/olm_golden.olm")
    for case in inputs.vector_cases():
        pats = inputs.case_patterns(case)
        RefLib.compile(tmp, pats, *case["store_flags"])
        ref = RefLib(tmp)
        hay = inputs.case_haystack(case)
        for mf in inputs.MATCH_FLAG_SETS:
            m = ref.match(hay, **{k: True for k in mf})
            vectors.append({"case": case["name"], "flags": list(mf), "count": int(m.size),
                            "digest": f"{Oracle.stream_digest(m):016x}"})
        ref.close()
        print(case["name"], "done")
    (HERE / "vectors.json").write_text(json.dumps({"generator": "tests/golden/make_golden.py",
                                                    "reference": "oracle/_ref/libomega_match_ref.so",
                                                    "vectors": vectors}, indent=1))
    print(len(vectors), "vectors")


if __name__ == "__main__":
    main()
