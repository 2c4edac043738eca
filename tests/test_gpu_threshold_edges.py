"""Every deciding kernel at the floating-point edges of the acceptance and min_delta rules (tests/threshold_edges.py):
each case runs at the edge value and one ulp either side, bit-exact against the oracle (results, pass details,
DemuxStats), with proof that the kernel the case is for decided reads."""
import math

import pytest

import bdx_b200 as bdx
from bdx_b200 import capi
import threshold_edges as te
from gpu_common import compare

pytestmark = pytest.mark.gpu

_WORK = {"prefilter": 0, "seed": 1, "automaton": 2}      # work_counters()


def _compare_counted(cfg, reads, debug, step, counter, label, check_plan=True):
    """compare() bit-exact against the oracle; then (check_plan) one profiled run of the same batch: the plan names
    `step` and the counter (work_counters or the launches of a profiling stage) shows that its kernel did the work."""
    compare(cfg, reads, want_stats=bool(cfg.summary), label=label, debug=debug)
    if not check_plan:
        return
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=len(reads), max_bytes=max(int(off[-1]), 16), debug=debug) as eng:
        plan = [ln for p in range(2) for ln in eng.config.describe(p).splitlines() if ln.startswith("plan:")]
        eng.stream.profile(True)
        eng.stream.work_counters(reset=True)
        eng.classify_packed(blob, off)
        work = eng.stream.work_counters()
        stages = {stage: n for stage, (_, n) in eng.stream.profile_read_stages().items()}
        eng.stream.profile(False)
        text = eng.config.describe(0)
    if step:
        assert step in plan[0].split("=")[1].split(","), (label, plan)
    _check_depths(text, cfg, label)
    if counter in _WORK:
        assert work[_WORK[counter]] > 0, (label, counter, work)
    else:
        assert stages[counter] > 0, (label, counter, stages)
    if step in ("k_seed@2", "k_seed_deep"):
        # the seed counter sums every seed stage.  The k_seed levels in front of `step` decide at most the reads
        # their rules allow (te.seed_level_decides, from every barcode's distance read back from the oracle); what
        # k_prefilter takes first is a verbatim barcode with min_delta = 0, which those levels would decide too.  More
        # reads decided by k_prefilter and the seed stages together than that bound prove that `step` decided reads
        levels = [int(ln.split("K=")[1].split()[0]) for ln in text.splitlines() if ln.startswith("k_seed level")]
        before = levels[:1] if step == "k_seed@2" else levels
        m = len(cfg.bc_seqs[0])
        bound = 0
        for r in reads:
            ds = [te.oracle_distance(b, r) for b in cfg.bc_seqs]
            bound += any(te.seed_level_decides(ds, m, k, i == len(levels) - 1, cfg.max_error_rate, cfg.min_delta)
                         for i, k in enumerate(before))
        assert work[_WORK["seed"]] + work[_WORK["prefilter"]] > bound, (label, step, bound, work)


def _check_depths(text, cfg, label):
    """The depths the host derived for the kernels that ran agree with floor(fl(thr * m)) in Python: no k_seed level
    deeper than the allowed distance, a complete k_seed_var level exactly at it, k_hamming_scan at it."""
    allowed = [te.allowed(cfg.max_error_rate, len(b)) for b in cfg.bc_seqs]
    for ln in text.splitlines():
        f = dict(x.split("=", 1) for x in ln.split(": ", 1)[-1].split() if "=" in x)
        if ln.startswith("k_seed level"):
            assert int(f["K"]) <= min(allowed), (label, ln)
        elif ln.startswith("k_seed_var level") and f["complete"] == "1":
            assert f["K"] == f"{min(allowed)}..{max(allowed)}", (label, ln)
        elif ln.startswith("k_hamming_scan"):
            assert int(f["allowed"]) == allowed[0], (label, ln)


@pytest.mark.parametrize("side", ["below", "edge", "above"])
@pytest.mark.parametrize("name", sorted(te.EDGE_CASES))
def test_edge(name, side):
    edge, build, debug, step, counter = te.EDGE_CASES[name]
    value = dict(zip(("below", "edge", "above"), te.neighbours(edge)))[side]
    cfg, reads = build(value)
    # one ulp off the edge the seed depths may differ, and with them the plan: the kernel is pinned at the edge
    _compare_counted(cfg, reads, debug, step, counter, f"{name} {side} ({value!r})", check_plan=side == "edge")


@pytest.mark.parametrize("thr", [0.0, -0.0, 5e-324, -5e-324], ids=repr)
def test_exact_zero_thresholds(thr):
    """:exact with thresholds at and next to zero: a verbatim occurrence scores 0 and is accepted for 0.0, -0.0 and
    5e-324 (0 <= thr, floor(thr * m) = 0), for -5e-324 nothing is; k_prefilter<1> generates the candidates."""
    cfg, reads = te.extreme_case("exact", thr, 0.0, seed=70)
    if thr >= 0:
        _compare_counted(cfg, reads, 0, "k_prefilter", "k_prefilter", f"exact thr={thr!r}")
    else:
        compare(cfg, reads, label=f"exact thr={thr!r}")


@pytest.mark.parametrize("thr", te.EXTREME_THR, ids=repr)
@pytest.mark.parametrize("algorithm", te.EXTREME_ALGORITHMS)
def test_extreme_thresholds(algorithm, thr):
    cfg, reads = te.extreme_case(algorithm, thr, 0.0)
    if thr == float("inf") and algorithm != "exact":
        with pytest.raises(capi.BdxError, match="outside Int64"):     # as the reference raises
            capi.Config(cfg)
        return
    compare(cfg, reads, label=f"{algorithm} thr={thr!r}")
    cfg.trim_side = 3
    compare(cfg, reads, want_stats=True, label=f"{algorithm} thr={thr!r} trim 3, stats")


@pytest.mark.parametrize("min_delta", te.EXTREME_MIN_DELTA, ids=repr)
@pytest.mark.parametrize("algorithm", te.EXTREME_ALGORITHMS)
def test_extreme_min_delta(algorithm, min_delta):
    """min_delta = 5e-324 turns the identical pair (barcodes 2 and 5) ambiguous where 0 gives barcode 2; inf makes
    every read with an accepted runner-up ambiguous; -0.0 is 0."""
    cfg, reads = te.extreme_case(algorithm, 0.2, min_delta)
    compare(cfg, reads, label=f"{algorithm} min_delta={min_delta!r}")
    cfg.trim_side = 3
    compare(cfg, reads, want_stats=True, label=f"{algorithm} min_delta={min_delta!r} trim 3, stats")
    if min_delta == 5e-324:
        import orc
        ref = orc.Oracle(cfg).classify_reads(reads[:2])
        assert (ref["status"] != 0).all(), ref        # the identical pair: exact tie, now ambiguous


@pytest.mark.parametrize("side", ["edge", "above"])
def test_seed_var_sigma_bound(side):
    """k_seed_var's unseen-runner-up bound decides a read exactly when fl(sigma - s1) >= min_delta: at min_delta =
    sigma every verbatim read is decided by the level itself, one ulp above none of them is (they go on to k_filter)."""
    cfg, _ = te.sigma_case(0.1)
    config = capi.Config(cfg)
    try:
        line = [ln for ln in config.describe(0).splitlines() if ln.startswith("k_seed_var level 1")][0]
    finally:
        config.close()
    assert "complete=0" in line, line
    q = int(line.split("q=")[1].split()[0])
    sigma = te.sigma_of(cfg.bc_seqs, cfg.max_error_rate, q)
    value = sigma if side == "edge" else math.nextafter(sigma, math.inf)
    cfg, reads = te.sigma_case(value)
    compare(cfg, reads, label=f"sigma {side}")
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=len(reads), max_bytes=int(off[-1])) as eng:
        eng.stream.work_counters(reset=True)
        eng.classify_packed(blob, off)
        work = eng.stream.work_counters()
    if side == "edge":
        assert work[_WORK["seed"]] == len(reads) and work[_WORK["automaton"]] == 0, work
    else:
        assert work[_WORK["automaton"]] > 0, work
