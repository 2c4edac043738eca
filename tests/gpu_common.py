"""Shared helpers of the GPU parity tests: run a batch through the C ABI (CUDA) and
through the oracle, and compare field by field (bit-exact)."""
from __future__ import annotations

import numpy as np

import bdx_b200 as bdx
from bdx_b200 import capi
import orc


def has_gpu() -> bool:
    try:
        return capi.load_library().bdx_device_count() > 0
    except Exception:
        return False


def run_cuda(cfg, reads, want_stats=False, details=True, debug=0):
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=max(len(reads), 1), max_bytes=max(int(off[-1]), 16),
                     want_stats=want_stats, debug=debug) as eng:
        if details:
            eng.stream.enable_details(True)
        out = eng.classify_packed(blob, off, want_details=details)
        counters = (eng.stream.stats(), eng.stream.stats_overflow()) if want_stats else None
        layout = eng.config.layout
    if details:
        return out[0], out[1], counters, layout
    return out, None, counters, layout


def compare(cfg, reads, want_stats=False, label="", debug=0):
    """debug: BDX_DEBUG_* flags of the CUDA run (single pipeline stages switched off)."""
    res, det, counters, layout = run_cuda(cfg, reads, want_stats=want_stats, debug=debug)
    ref = orc.Oracle(cfg, want_stats=want_stats).classify_reads(reads)
    n = len(reads)
    for f in ("status", "bc1", "bc2", "keep_start", "keep_end"):
        bad = np.nonzero(res[f] != ref[f])[0]
        assert bad.size == 0, (f"{label}: field {f} differs at read {bad[0]} ({reads[bad[0]]!r}): "
                               f"cuda={res[bad[0]]} oracle={ref[bad[0]]}")
    for p in (0, 1):
        rp = ref["passes"][:, p]
        dp = det[p]
        bad = np.nonzero(dp["status"] != rp["status"])[0]
        assert bad.size == 0, f"{label}: pass {p} status differs at {bad[0]}: {dp[bad[0]]} vs {rp[bad[0]]}"
        m = rp["status"] == 0
        for f, g in (("bc", "bc"), ("start", "start"), ("end", "end")):
            bad = np.nonzero(m & (dp[f] != rp[g]))[0]
            assert bad.size == 0, (f"{label}: pass {p} {f} differs at read {bad[0]} ({reads[bad[0]]!r}): "
                                   f"cuda={dp[bad[0]]} oracle={rp[bad[0]]}")
        score = np.full(n, np.inf)
        score[m] = dp["dist"][m].astype(np.float64) / dp["norm"][m].astype(np.float64)
        bad = np.nonzero(m & (score != rp["score"]))[0]
        assert bad.size == 0, f"{label}: pass {p} score differs at {bad[0]}: {score[bad[0]]} vs {rp['score'][bad[0]]}"
    if want_stats:
        from bdx_b200.stats import stats_from_counters, stats_from_passes
        got = stats_from_counters(counters[0], layout, cfg, counters[1])
        passes = [[tuple(ref["passes"][i, p][k] for k in ("status", "bc", "start", "end", "score")) for p in (0, 1)]
                  for i in range(n)]
        want = stats_from_passes(ref["status"], ref["bc1"], ref["bc2"], passes, cfg)
        assert got == want, f"{label}: DemuxStats differ"
    return res, ref
