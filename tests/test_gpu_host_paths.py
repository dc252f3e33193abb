"""The host entry points alike on every host path -- one GPU, OLM_HOST_SPAN_BYTES spans, several
engines (engine.cu host_spans, multi.cpp first_alone) -- needs a B200."""
import pytest

import inputs
from omega_match_b200 import Matcher
from test_gpu_multi import _devices

pytestmark = pytest.mark.gpu

MIB = 1 << 20


@pytest.mark.parametrize("kind", ["one", "spans", "multi"])
def test_empty_call_reports_zero_timing(store_cache, monkeypatch, kind):
    """After an empty host call, last_timing() reports that call -- all zeros -- not the call before."""
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    path = store_cache("span-names", names, (0, 0, 0))
    hay = inputs.text_haystack(9 * MIB + 7, 3).tobytes()
    if kind == "spans":
        monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(4 * MIB))
    with Matcher(path, devices=_devices(2) if kind == "multi" else None) as m:
        calls = {"match": m.match_arrays, "pattern_counts": m.pattern_counts, "match_lines": m.match_lines,
                 "matching_lines": m.matching_lines}
        for name, call in calls.items():
            call(hay)
            assert m.last_timing()["kernel_launches"] > 0, f"{kind} {name}"
            got = call(b"")
            assert got.sum() == 0 if name == "pattern_counts" else got.size == 0, f"{kind} {name}"
            t = m.last_timing()
            assert all(v == 0 for v in t.values()), f"{kind} {name}: {t}"
