"""BASELINE.json configs[0..3] at 64 MiB and more through the C ABI, record by record against the
oracle (SURVEY 8d "Flag matrix for parity"), and the span path of the host entry point -- needs a
B200.

  configs[0]  names.txt, baseline flags                       pseudo-KJV tiled + text
  configs[1]  surnames_us_census.txt, ignore-case              + word_boundary
  configs[2]  census, ignore-case + ignore-punct + elide-ws    + no_overlap + longest_only
  configs[3]  tlds.txt + the generated 1..4 byte patterns      4 KiB-planted synthetic haystack
"""
import numpy as np
import pytest

import inputs
from conftest import describe_diff, same_matches
from omega_match_b200 import Matcher
from oracle.oracle import Oracle

pytestmark = pytest.mark.gpu

MIB = 1 << 20


def kjv_tiled(n: int, seed: int) -> np.ndarray:
    """pseudo-KJV copies with stretches of punctuation / whitespace rich text between them, so that
    copies start at varying offsets relative to the 4 MiB windows and the 4 KiB tiles."""
    pk = np.frombuffer(inputs.pseudo_kjv(), dtype=np.uint8)
    parts, size, i = [], 0, 0
    while size < n:
        t = inputs.text_haystack(MIB + 4099 * (i + 1), seed + i)
        parts += [pk, t]
        size += pk.size + t.size
        i += 1
    return np.concatenate(parts)[:n].copy()


def _check(m, o, hay, **kw):
    got = m.match_arrays(hay, **kw)
    want = o.match(hay, **kw)
    assert same_matches(got, want), f"{kw}: " + describe_diff(got, want)
    return got


CONFIGS = {
    "cfg1-names-baseline": ("names", (0, 0, 0), [{}, {"longest_only": True, "no_overlap": True}]),
    "cfg2-census-ci-wb": ("census", (1, 0, 0), [{"word_boundary": True}]),
    "cfg3-census-cpw-nol": ("census", (1, 1, 1), [{"no_overlap": True, "longest_only": True},
                                                   {"word_boundary": True}]),
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_baseline_text_configs_at_64mib(store_cache, name):
    kind, sf, flagsets = CONFIGS[name]
    pats = inputs.case_patterns(dict(patterns=kind, store_flags=sf))
    path = store_cache(f"cfg-{kind}", pats, sf)
    hay = kjv_tiled(64 * MIB + 54321, 0x51 + sum(sf))
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for kw in flagsets:
            got = _check(m, o, hay, **kw)
            assert got.size > 100_000


def test_short_matcher_config_at_64mib(store_cache):
    """configs[3]: tlds.txt + 4/64/1024/8192 patterns of 1/2/3/4 bytes over the planted synthetic
    haystack (SURVEY 8d), a 64 MiB slice that does not start at 0 (shard-style generation)."""
    pats = list(inputs._pattern_set("tlds")) + inputs.synth_short_patterns()
    path = store_cache("cfg4-short", b"\n".join(pats) + b"\n")
    start = 3 * 4096 * 1000
    hay = inputs.plant(inputs.synth_haystack(64 * MIB + 4096, inputs.SEED_H4, start=start), pats, inputs.SEED_H4 ^ 0x77,
                       start=start)[:64 * MIB + 777]
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for kw in ({}, {"longest_only": True, "no_overlap": True}, {"word_boundary": True}, {"word_suffix": True}):
            _check(m, o, hay, **kw)


def test_perf_matrix_on_census_at_16mib(store_cache):
    """Every variant of perf_test.py:69-91 (+ word-prefix / word-suffix) with the census list on 16 MiB of
    pseudo-KJV + text: four 4 MiB windows, every store-flag set of the matrix."""
    hay = kjv_tiled(16 * MIB + 999, 0x77)
    for sf in sorted({v[1] for v in inputs.PERF_VARIANTS}):
        pats = inputs.case_patterns(dict(patterns="census", store_flags=sf))
        path = store_cache("cfg-census", pats, sf)
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            for _, vsf, mf in inputs.PERF_VARIANTS:
                if vsf == sf:
                    _check(m, o, hay, **{k: True for k in mf})


def test_host_span_path(store_cache, monkeypatch):
    """OLM_HOST_SPAN_BYTES: omega_list_matcher_match scans a host haystack as consecutive byte-range
    shards of that many start positions (engine.cu host_spans): matches written across every
    span edge, plain and transforming stores, no_overlap across span edges, exact statistics summed."""
    monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(4 * MIB))
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    flagsets = [{}, {"no_overlap": True}, {"longest_only": True, "no_overlap": True}, {"word_boundary": True},
                {"line_end": True, "longest_only": True, "no_overlap": True}, {"word_prefix": True}]
    for sf in ((0, 0, 0), (1, 1, 1)):
        path = store_cache("span-names", names, sf)
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            for n in (4 * MIB + 1, 9 * MIB + 12345, 21 * MIB + 7):
                hay = inputs.text_haystack(n, 7 + n)
                for edge in range(4 * MIB, n - 6, 4 * MIB):
                    hay[edge - 5:edge + 6] = np.frombuffer(b"Christopher", dtype=np.uint8)
                for kw in flagsets[:3] if any(sf) else flagsets:
                    _check(m, o, hay, **kw)
