"""The floating-point edges of the acceptance and min_delta rules (tests/threshold_edges.py), the edge cases the
GPU tests run, and the host's seed depths at edge and extreme thresholds -- no GPU."""
import math
from fractions import Fraction

import numpy as np
import pytest

from bdx_b200 import capi
import orc
import threshold_edges as te


@pytest.fixture(scope="module")
def lib():
    capi.build_library()
    return capi.load_library()


def test_edge_enumeration_agrees_with_fractions():
    """Every (m, d) up to 256 is classified once in doubles and once in exact rationals (both checks evaluated as
    the correctly rounded results of the exact operations); the enumerators find exactly the disagreements."""
    up, down = set(), set()
    for m in range(1, 257):
        for d in range(1, m + 1):
            t_up = math.nextafter(d / m, 0.0)
            floor_up = math.floor(Fraction(float(Fraction(t_up) * m)))
            if floor_up == d and Fraction(float(Fraction(d, m))) > Fraction(t_up):
                up.add((m, d))
            t_dn = d / m
            if math.floor(Fraction(float(Fraction(t_dn) * m))) < d:
                down.add((m, d))
    got_up = {(m, d) for m, d, _ in te.round_up_edges(range(1, 257), 256)}
    got_down = {(m, d) for m, d, _ in te.round_down_edges(range(1, 257), 256)}
    assert got_up == up and got_down == down
    assert len(up) == 2483 and len(down) == 1087
    for pair in ((25, 5), (24, 5), (26, 3), (13, 3), (13, 5), (13, 6)):
        assert pair in up, pair
    assert (22, 15) in down
    # the round thresholds of the other tests never sit on an edge
    for thr in (0.05, 0.1, 0.13, 0.2, 0.25, 0.3, 0.34, 0.5):
        for m in range(1, 257):
            for d in range(0, m + 1):
                assert (d <= te.allowed(thr, m)) == (d / m <= thr), (thr, m, d)


def test_round_up_edge_values():
    m, d, thr = next(e for e in te.round_up_edges([25], 5) if e[1] == 5)
    assert thr == 0.19999999999999998 == math.nextafter(0.2, 0.0)
    assert te.allowed(thr, m) == 5 and not te.accepts(5, 25, thr) and te.accepts(5, 25, 0.2)
    _, _, thr = next(e for e in te.round_down_edges([22], 15) if e[1] == 15)
    assert thr == 15 / 22 and te.allowed(thr, 22) == 14 and not te.accepts(15, 22, thr)


def test_min_delta_edges():
    """fl(fl(d2/m2) - fl(d1/m1)) on one length and across two; one ulp either side is a different double."""
    pairs = [(0, 25, 4, 25), (0, 24, 4, 24), (1, 20, 3, 25), (2, 17, 5, 28), (0, 26, 3, 26)]
    for d1, m1, d2, m2, (lo, md, hi) in te.min_delta_edges(pairs):
        delta = d2 / m2 - d1 / m1
        assert Fraction(md) == Fraction(float(Fraction(float(Fraction(d2, m2))) - Fraction(float(Fraction(d1, m1)))))
        assert not (delta < md) and delta < hi and not (delta < lo)
        assert lo < md < hi


def test_extreme_allowed():
    """The depth the host and device derive at the extreme thresholds: clamped, never NaN or an overflow."""
    for thr in te.EXTREME_THR:
        for m in (1, 13, 26, 64, 256):
            a = te.allowed(thr, m)
            assert -(1 << 28) <= a <= (1 << 28)
            if thr >= 0:
                assert a >= 0
    assert te.allowed(math.inf, 24) == 1 << 28 and te.allowed(-5e-324, 24) == -1 and te.allowed(-0.0, 24) == 0


def test_planted_pair_distances():
    """The 96 x 26 pair: barcode 41 = barcode 11 at columns 3, 10, 17 breaks every segment of depth 2 and leaves
    segment 3 of depth 3 intact; the oracle puts each planted read at the distance it was built for."""
    assert te.intact_segments(26, 2, (3, 10, 17)) == []
    assert te.intact_segments(26, 3, (3, 10, 17)) == [3]
    bcs = te._pair_set(26, (3, 10, 17), 26)
    rng = np.random.default_rng(0)
    read = te.planted(rng, bcs, bcs[11], {11: 0, 41: 3})
    assert te.oracle_distance(bcs[41], read) == 3 and te.oracle_distance(bcs[11], read) == 0
    cfg, reads = te.EDGE_CASES["k_seed_26_trim3"][1](te.EDGE_CASES["k_seed_26_trim3"][0])
    got = te.oracle_pass_distances(cfg, reads[:12])
    assert got[0] == (0, 12, 0) and got[1] == (0, 42, 0), got[:2]


@pytest.mark.parametrize("name", sorted(te.EDGE_CASES))
def test_edge_case_is_real(lib, name):
    """Each GPU case sits on a boundary: the oracle's verdict for its reads changes between the edge value and
    its neighbour one ulp away, and its plan runs the kernel the case is for."""
    edge, build, debug, step, _ = te.EDGE_CASES[name]
    verdicts = []
    for v in te.neighbours(edge):
        cfg, reads = build(v)
        ref = orc.Oracle(cfg).classify_reads(reads)
        verdicts.append([(int(r["status"]), int(r["bc1"]), int(r["bc2"])) for r in ref])
    assert verdicts[1] != verdicts[0] or verdicts[1] != verdicts[2], name
    cfg, _ = build(edge)
    if step:
        config = capi.Config(cfg, debug=debug)
        try:
            plan = [ln for ln in config.describe(0).splitlines() if ln.startswith("plan:")][0]
        finally:
            config.close()
        assert step in plan.split("=")[1].split(","), (name, plan)


def _describe(cfg, debug=0):
    config = capi.Config(cfg, debug=debug)
    try:
        return config.describe(0)
    finally:
        config.close()


def _levels(text, kernel):
    out = []
    for ln in text.splitlines():
        if ln.startswith(kernel + " level"):
            out.append({k: v for k, v in (f.split("=", 1) for f in ln.split(": ", 1)[1].split())})
    return out


def test_seed_depths_at_round_up_edge(lib):
    """96 x 26 at thr one ulp below fl(3/26): floor(fl(thr * 26)) = 3, so k_seed's deep level is K = 3 and
    k_seed_var's level is complete at K = 3; one ulp lower the depth is 2."""
    bcs = te._pair_set(26, (3, 10, 17), 26)
    thr = math.nextafter(3 / 26, 0.0)
    assert te.allowed(thr, 26) == 3 and te.allowed(math.nextafter(thr, 0.0), 26) == 2
    for t, want in ((thr, 3), (math.nextafter(thr, 0.0), 2), (3 / 26, 3)):
        text = _describe(te._cfg(bcs, max_error_rate=t, min_delta=0.12, trim_side=3))
        sd = _levels(text, "k_seed")
        assert int(sd[-1]["K"]) == min(want, 7), (t, text)
        sv = _levels(text, "k_seed_var")
        q = int(sv[0]["q"])
        k = min(26 // q - 1, want)
        assert sv[0]["K"] == f"{k}..{k}" and int(sv[0]["complete"]) == int(k == want), (t, text)


def test_seed_var_depths_at_round_down_edge(lib):
    """Lengths 45..49 at thr = fl(4/49): fl(thr * 49) rounds below 4, so the depth of the 49-nt barcodes is 3, as
    for the shorter ones; the complete level reads K = 3..3 (exact arithmetic would give 3..4)."""
    thr = 4 / 49
    assert (49, 4, thr) in te.round_down_edges([49], 4)
    bcs = te._barcodes(60, 96, 45, 49)
    assert max(len(b) for b in bcs) == 49
    text = _describe(te._cfg(bcs, max_error_rate=thr))
    sv = _levels(text, "k_seed_var")
    want = [te.allowed(thr, len(b)) for b in bcs]
    q = int(sv[0]["q"])
    ks = [min(len(b) // q - 1, a) for b, a in zip(bcs, want)]
    assert sv[0]["K"] == f"{min(ks)}..{max(ks)}" == "3..3", text
    assert int(sv[0]["complete"]) == int(all(k == a for k, a in zip(ks, want))) == 1, text


@pytest.mark.parametrize("thr", te.EXTREME_THR, ids=repr)
@pytest.mark.parametrize("lengths", [(24, 24), (16, 28), (13, 13)], ids=lambda x: f"{x[0]}..{x[1]}")
def test_seed_depths_at_extremes(lib, thr, lengths):
    """At the extreme thresholds every depth the host prints is the Python floor(fl(thr * m)) bounded as its
    builder bounds it; thr >= 1 and inf never reach the byte-wide depth tables with a value above 255."""
    bcs = te._barcodes(61, 96, *lengths)
    if math.isinf(thr):
        with pytest.raises(capi.BdxError, match="outside Int64"):
            _describe(te._cfg(bcs, max_error_rate=thr))
        text = _describe(te._cfg(bcs, max_error_rate=thr, matching_algorithm="exact"))
        assert "plan: steps=k_prefilter,k_literal@cand" in text, text
        return
    text = _describe(te._cfg(bcs, max_error_rate=thr))
    allowed = [te.allowed(thr, len(b)) for b in bcs]
    for lv in _levels(text, "k_seed_var"):
        q = int(lv["q"])
        lo, hi = (int(x) for x in lv["K"].split(".."))
        assert 0 <= lo <= hi <= 255, text
        # a single-length level cuts min(m / q - 1, allowed) segments, a complete level allowed + 1
        ks = [min(len(b) // q - 1, a) for b, a in zip(bcs, allowed)]
        assert (lo, hi) in ((min(ks), max(ks)), (min(allowed), max(allowed))), (thr, text)
    if thr < 0:
        assert not _levels(text, "k_seed_var"), text
    for lv in _levels(text, "k_seed"):
        assert 1 <= int(lv["K"]) <= min(7, min(allowed)), text
    if thr >= 1.0:
        assert min(allowed) >= lengths[0]


_T63 = 9223372036854775808.0 / 20      # thr * 20 = 2^63 exactly: floor(Int, .) just beyond typemax(Int64)


@pytest.mark.parametrize("thr,fits", [(math.inf, False), (-math.inf, False), (1e300, False), (-1e300, False),
                                      (_T63, False), (math.nextafter(_T63, 0.0), True), (-_T63, True),
                                      (math.nextafter(-_T63, -math.inf), False), (1.5, True)], ids=repr)
@pytest.mark.parametrize("algorithm", ["semiglobal", "hamming", "exact"])
def test_threshold_outside_int64(lib, algorithm, thr, fits):
    """floor(Int, thr * m) raises InexactError in the reference (:254, :567) unless the product's floor fits Int64
    (-2^63 does, 2^63 does not): such a config is refused for :semiglobal and :hamming; :exact never takes that
    floor and accepts every threshold."""
    assert (thr * 20 >= -2.0 ** 63 and thr * 20 < 2.0 ** 63) == fits
    cfg = te._cfg(te._barcodes(63, 8, 20), max_error_rate=thr, matching_algorithm=algorithm)
    if fits or algorithm == "exact":
        _describe(cfg)
    else:
        with pytest.raises(capi.BdxError, match="outside Int64"):
            _describe(cfg)


@pytest.mark.parametrize("m,d", [(13, 3), (24, 5), (25, 5), (26, 3)])
def test_hamming_depth_at_round_up_edge(lib, m, d):
    """k_hamming_scan's allowed distance is floor(fl(thr * m)) at the round-up edge, d, not d - 1."""
    thr = math.nextafter(d / m, 0.0)
    text = _describe(te._cfg(te._barcodes(62, 96, m), max_error_rate=thr, matching_algorithm="hamming"))
    assert f"k_hamming_scan: m={m} allowed={d} segments={d + 1}" in text, text
