"""omega_match_b200 -- the matching hot path of OmegaMatch (omega_list_matcher_match) on B200.

The product is `lib/libomega_match.so` (hand-written sm_100a CUDA behind the reference's C
ABI, see include/olm_b200.h); this package is the host-side mirror of the reference's Python
binding plus the device-resident / sharded entry points.
"""
from .omega_match import (Compiler, Matcher, MatchResult, MatchStats, PatternStoreStats, get_library_info,
                          get_version, MATCH_DTYPE, MATCH_IDS_DTYPE, RECORD_DTYPE, FLAG_NAMES)

__all__ = ["Compiler", "Matcher", "MatchResult", "MatchStats", "PatternStoreStats", "get_version",
           "get_library_info", "MATCH_DTYPE", "MATCH_IDS_DTYPE", "RECORD_DTYPE", "FLAG_NAMES"]
