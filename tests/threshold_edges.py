"""Floating-point edges of the acceptance and min_delta rules (classification.jl:254, :567, :658, :666, :696,
:711), and reads planted at known distances from chosen barcodes (TEST INFRASTRUCTURE, no GPU).

A barcode at distance d of normalisation length m is accepted under threshold thr only if both
  * d <= floor(fl(thr * m))       -- the distance the DP allows, and
  * fl(d / m) <= thr              -- the score test.
A read is ambiguous when fl(sub_min - min_score) < min_delta.  At most thresholds the two acceptance checks
agree; the edges below are where they do not:
  * round-up edge:   thr = nextafter(fl(d / m), 0): the DP allows d, the score test rejects it;
  * round-down edge: thr = fl(d / m): the score test accepts d, the DP allows less than d.
Each edge is confirmed with exact rational arithmetic (fractions.Fraction), not only with doubles.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

import orc

# extreme option values every rule has to survive
EXTREME_THR = (0.0, -0.0, 5e-324, -5e-324, -0.1, 1.0, 1.5, math.inf)
EXTREME_MIN_DELTA = (-0.0, 5e-324, -0.1, math.inf)

_CLAMP = 1 << 28       # host_allowed / allowed_from clamp (beyond any reachable distance)


def allowed(thr: float, m: int) -> int:
    """floor(Int, thr * m) as an IEEE double product, clamped like the library (tables.cu, literal.cuh)."""
    x = thr * float(m)
    if not (x < _CLAMP):
        return _CLAMP
    return max(math.floor(x), -_CLAMP)


def accepts(d: int, m: int, thr: float) -> bool:
    """Both acceptance checks of the reference for a barcode at distance d, normalisation length m."""
    return d <= allowed(thr, m) and d / m <= thr


def _fl_product_floor(thr: float, m: int) -> int:
    """floor(fl(thr * m)) from the exact product rounded once to the nearest double (Fraction -> float is
    correctly rounded), independent of the float multiply."""
    return math.floor(Fraction(float(Fraction(thr) * m)))


def _fl_quotient(d: int, m: int) -> Fraction:
    """fl(d / m) as an exact rational."""
    return Fraction(float(Fraction(d, m)))


def round_up_edges(lengths, d_max: int):
    """[(m, d, thr)] with thr = nextafter(fl(d/m), 0), floor(fl(thr*m)) = d and fl(d/m) > thr, confirmed exactly."""
    out = []
    for m in lengths:
        for d in range(1, min(d_max, m) + 1):
            thr = math.nextafter(d / m, 0.0)
            if allowed(thr, m) == d and d / m > thr:
                assert _fl_product_floor(thr, m) == d and _fl_quotient(d, m) > Fraction(thr), (m, d, thr)
                out.append((m, d, thr))
    return out


def round_down_edges(lengths, d_max: int):
    """[(m, d, thr)] with thr = fl(d/m): fl(d/m) <= thr but floor(fl(thr*m)) < d, confirmed exactly."""
    out = []
    for m in lengths:
        for d in range(1, min(d_max, m) + 1):
            thr = d / m
            if allowed(thr, m) < d:
                assert _fl_product_floor(thr, m) < d and _fl_quotient(d, m) <= Fraction(thr), (m, d, thr)
                out.append((m, d, thr))
    return out


def neighbours(x: float):
    """(one ulp below, x, one ulp above)."""
    return math.nextafter(x, -math.inf), x, math.nextafter(x, math.inf)


def min_delta_edge(d1: int, m1: int, d2: int, m2: int) -> float:
    """min_delta = fl(fl(d2/m2) - fl(d1/m1)): a best at d1 / m1 and a runner-up at d2 / m2 are unambiguous at
    this value and ambiguous one ulp above it (the rule is `delta < min_delta`)."""
    md = d2 / m2 - d1 / m1
    assert Fraction(md) == Fraction(float(_fl_quotient(d2, m2) - _fl_quotient(d1, m1)))
    return md


def min_delta_edges(pairs):
    """[(d1, m1, d2, m2, (below, edge, above))] for each (d1, m1, d2, m2)."""
    return [(d1, m1, d2, m2, neighbours(min_delta_edge(d1, m1, d2, m2))) for d1, m1, d2, m2 in pairs]


def pigeonhole_segments(m: int, k: int):
    """The k + 1 segments [o, o + len) k_seed's level of depth k cuts a barcode of length m into (tables.cu)."""
    seg = m // (k + 1)
    return [(i * seg, i * seg + seg) for i in range(k + 1)]


def near_neighbour(src: str, columns, alphabet="ACGT") -> str:
    """`src` with a substitution at each of `columns` (0-based): the next letter of the alphabet, so the result
    is deterministic and differs from src at exactly those columns."""
    s = list(src)
    for c in columns:
        s[c] = alphabet[(alphabet.index(s[c]) + 1) % len(alphabet)]
    return "".join(s)


def intact_segments(m: int, k: int, columns):
    """Indices of the depth-k pigeonhole segments that no column of `columns` touches."""
    return [i for i, (a, b) in enumerate(pigeonhole_segments(m, k)) if not any(a <= c < b for c in columns)]


def flank(rng, n: int) -> bytes:
    return bytes(rng.choice(list(b"ACGT"), size=n).astype(np.uint8))


def plant(rng, bc: str, left: int = 30, right: int = 40) -> bytes:
    """`bc` verbatim between random flanks."""
    return flank(rng, left) + bc.encode() + flank(rng, right)


def oracle_distance(bc: str, read: bytes) -> int:
    """The reference's semiglobal distance of `bc` in `read` (unit costs, whole read),
    read back from its score x length."""
    m = len(bc)
    score = orc.semiglobal(bc, read, 1.0)
    if math.isinf(score):
        return 1 << 30
    d = round(score * m)
    assert d / m == score, (bc, read, score)
    return d


def oracle_pass_distances(cfg, reads, p: int = 0):
    """Per read: (status, barcode, distance) of pass p, the distance read back from the oracle's score x norm."""
    ref = orc.Oracle(cfg).classify_reads(reads)
    out = []
    for r in ref:
        ps = r["passes"][p]
        if ps["status"] != 0:
            out.append((int(ps["status"]), 0, None))
            continue
        b = int(ps["bc"])
        seqs = cfg.bc_seqs if p == 0 else cfg.bc_seqs2
        norms = cfg.bc_lengths_no_N if p == 0 else cfg.bc_lengths_no_N2
        norm = norms[b - 1] if cfg.nindel is not None else len(seqs[b - 1])
        d = round(float(ps["score"]) * norm)
        assert d / norm == ps["score"], (r, norm)
        out.append((0, b, d))
    return out


def seed_level_decides(ds, norm: int, K: int, last: bool, thr: float, min_delta: float) -> bool:
    """Whether a k_seed level of depth K can decide a read whose barcodes lie at distances `ds` (seed.cu): it knows
    exactly the barcodes within K; with min_delta it needs the runner-up known or provably far."""
    order = sorted(ds)
    best = order[0]
    if best > K:
        return last and K >= allowed(thr, norm)          # nothing acceptable
    if not accepts(best, norm, thr):
        return False
    if min_delta == 0.0:
        return True
    if len(order) > 1 and order[1] <= K:
        return True
    if accepts(K + 1, norm, thr):
        return not ((K + 1) / norm - best / norm < min_delta)
    return True


def hamming_distance(bc: str, read: bytes) -> int:
    """The reference's :hamming distance of `bc` in `read` (best start anywhere), read back from its score."""
    m = len(bc)
    score, _, _ = orc.hamming(bc, read, 1.0, (1, len(read)), len(read), 1)
    if math.isinf(score):
        return 1 << 30
    d = round(score * m)
    assert d / m == score, (bc, read, score)
    return d


def planted(rng, bcs, core: str, want: dict, dist=oracle_distance, left=30, right=40, tries=200) -> bytes:
    """A read of random flanks around `core` in which barcode b (0-based) lies at distance want[b] for every b of
    `want` and every other barcode lies farther than all of them -- every distance read back from the oracle."""
    far = max(want.values())
    for _ in range(tries):
        read = flank(rng, left) + core.encode() + flank(rng, right)
        ds = [dist(b, read) for b in bcs]
        if all(ds[b] == d for b, d in want.items()) and all(x > far for i, x in enumerate(ds) if i not in want):
            return read
    raise AssertionError(f"no flanks give distances {want} for {core}")


# ---- the cases the GPU tests run: each is a small batch of planted and random reads under one config, with the
# option that sits on an edge.  A case is built for a value of that option: the edge itself or a neighbour. ----

def _cfg(bcs, bcs2=None, **kw):
    import bdx_b200 as bdx
    c = bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[len(x) for x in bcs], ids=[f"a{i}" for i in range(len(bcs))], **kw)
    if bcs2:
        c.is_dual = True
        c.bc_seqs2, c.bc_lengths_no_N2, c.ids2 = bcs2, [len(x) for x in bcs2], [f"b{i}" for i in range(len(bcs2))]
    return c


def _barcodes(seed, n, lo, hi=None):
    import synth
    return synth.random_barcodes(np.random.default_rng(seed), n, lo, hi or lo)


def _random_reads(seed, bcs, n=150, bcs2=None, **kw):
    import synth
    return synth.random_reads(np.random.default_rng(seed), n, bcs, barcodes2=bcs2, min_len=100, max_len=130, **kw)


def _pair_set(m, cols, seed):
    """96 barcodes of length m; barcode 41 is barcode 11 with substitutions at `cols`."""
    bcs = _barcodes(seed, 96, m)
    bcs[41] = near_neighbour(bcs[11], cols)
    return bcs


def _pair_reads(rng, bcs, d, extra=()):
    """Barcodes 11 and 41 verbatim (the other at distance d), plus reads with one of them mutated at `extra`."""
    reads = []
    for _ in range(6):
        reads.append(planted(rng, bcs, bcs[11], {11: 0, 41: d}))
        reads.append(planted(rng, bcs, bcs[41], {41: 0, 11: d}))
    for cols, want in extra:
        reads.append(planted(rng, bcs, near_neighbour(bcs[11], cols), want))
    return reads


def _spread_reads(rng, bcs, ks, per=3, cols_of=None, dist=oracle_distance):
    """For several barcodes b and each k of `ks`: b with k substitutions (columns cols_of(m, k)), planted so that
    b is the nearest barcode, at distance k."""
    reads = []
    for b in range(0, len(bcs), max(1, len(bcs) // 16)):
        m = len(bcs[b])
        for k in ks:
            cols = cols_of(m, k) if cols_of else [round((i + 0.5) * m / k) - 1 for i in range(k)]
            for _ in range(per):
                try:
                    reads.append(planted(rng, bcs, near_neighbour(bcs[b], cols), {b: k}, dist=dist))
                except AssertionError:
                    pass      # another barcode happens to lie as near: left out
    return reads


def _seed26(value, seed, **kw):
    """The 96 x 26 case: barcode 41 = barcode 11 at columns 3, 10, 17 (no depth-2 segment intact, depth-3
    segment 3 intact), threshold one ulp below fl(3/26) unless `value` replaces it."""
    rng = np.random.default_rng(seed)
    bcs = _pair_set(26, (3, 10, 17), seed)
    reads = _pair_reads(rng, bcs, 3, extra=[((3,), {11: 1, 41: 2}), ((3, 10), {11: 2, 41: 1})])
    reads += _spread_reads(rng, bcs, (2, 3), cols_of=lambda m, k: (3, 10, 17)[:k])
    return _cfg(bcs, max_error_rate=value, **kw), reads + _random_reads(seed, bcs)


def _bound(m, value, seed, thr):
    """96 x m, K < allowed: barcode 41 = barcode 11 at K + 1 = 4 columns, min_delta on the edge of
    fl(4/m) - 0 (best verbatim, runner-up unseen by the seed level at K + 1)."""
    rng = np.random.default_rng(seed)
    bcs = _pair_set(m, (2, 8, 14, 20), seed)
    reads = _pair_reads(rng, bcs, 4, extra=[((2,), {11: 1, 41: 3})])
    return _cfg(bcs, max_error_rate=thr, min_delta=value, trim_side=3), reads + _random_reads(seed, bcs)


def _small(m, d, cols, value, seed, n_bc=5, trim=3):
    """n_bc barcodes of length m, a read set around distance d on the round-up edge of (m, d), trimmed on `trim`."""
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, n_bc, m)
    reads = _spread_reads(rng, bcs, (d - 1, d), per=6, cols_of=lambda mm, k: cols[:k])
    return _cfg(bcs, max_error_rate=value, trim_side=trim), reads + _random_reads(seed, bcs, max_edits=d + 1)


def _varlen(value, seed, option="thr", geometry=None):
    """200 barcodes of 16..28 nt, score-only, min_delta.  option "thr": thr = one ulp below 0.2, on a round-up
    edge for 25 nt (d = 5) only; option "min_delta": reads with a 20-nt barcode at d = 1 and a 25-nt one at d = 3
    next to each other, min_delta on the edge of fl(3/25) - fl(1/20)."""
    import bdx_b200 as bdx
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, 200, 16, 28)
    for i, m in enumerate((20, 25, 25, 26, 24, 20)):          # lengths the cases plant
        bcs[i] = _barcodes(seed + 1 + i, 1, m)[0]
    thr, md = (value, 0.05) if option == "thr" else (math.nextafter(0.2, 0.0), value)
    kw = dict(max_error_rate=thr, min_delta=md)
    if geometry == "config3":
        R = bdx.parse_dynamic_range
        kw.update(ref_search_range=R("1:40"), barcode_start_range=R("1:6"))
        geo = dict(left=2, right=70)

        def dist(bc, read):
            score = orc.semiglobal(bc, read, 1.0, rng=(1, min(40, len(read))), max_start_pos=6)
            return 1 << 30 if math.isinf(score) else round(score * len(bc))
    else:
        geo, dist = {}, oracle_distance
    reads = []
    if option == "thr":
        for b in (1, 2, 3, 4):
            m = len(bcs[b])
            for k in (4, 5):
                for _ in range(4):
                    try:
                        cols = [round((i + 0.5) * m / k) - 1 for i in range(k)]
                        reads.append(planted(rng, bcs, near_neighbour(bcs[b], cols), {b: k}, dist=dist, tries=20, **geo))
                    except AssertionError:
                        pass
    else:
        for _ in range(8):
            core = near_neighbour(bcs[0], (9,)) + flank(rng, 6).decode() + near_neighbour(bcs[1], (3, 11, 19))
            reads.append(planted(rng, bcs, core, {0: 1, 1: 3}))
    return _cfg(bcs, **kw), reads + _random_reads(seed, bcs, start_hi=5 if geometry else None)


def _weighted(value, seed):
    """96 x 24, mismatch 2, indel 3: reads at weighted distance 4 and 5 on the round-up edge of (24, 5)."""
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, 96, 24)
    costs = dict(mismatch=2, indel=3)

    def dist(bc, read):
        score = orc.semiglobal(bc, read, 1.0, mismatch=2, indel=3)
        return 1 << 30 if math.isinf(score) else round(score * len(bc))
    reads = []
    for b in range(0, 96, 8):
        for core, d in ((near_neighbour(bcs[b], (5, 17)), 4), (near_neighbour(bcs[b], (5,))[:15] + bcs[b][16:], 5),
                        (near_neighbour(bcs[b], (5,)), 2)):
            try:
                reads.append(planted(rng, bcs, core, {b: d}, dist=dist))
            except AssertionError:
                pass
    return _cfg(bcs, max_error_rate=value, **costs), reads + _random_reads(seed, bcs)


def _hamming(m, d, trim, value, seed):
    """96 x m :hamming at the round-up edge of (m, d), min_delta 0.25 (above fl(d/m)): barcode 41 = barcode 11 at d
    columns, so the runner-up sits exactly on the edge."""
    rng = np.random.default_rng(seed)
    cols = [round((i + 0.5) * m / d) - 1 for i in range(d)]
    bcs = _pair_set(m, cols, seed)
    reads = []
    for _ in range(6):
        reads.append(planted(rng, bcs, bcs[11], {11: 0, 41: d}, dist=hamming_distance))
        reads.append(planted(rng, bcs, bcs[41], {41: 0, 11: d}, dist=hamming_distance))
    reads += _spread_reads(rng, bcs, (d - 1, d), per=2, dist=hamming_distance)
    cfg = _cfg(bcs, max_error_rate=value, min_delta=0.25, matching_algorithm="hamming", trim_side=trim)
    return cfg, reads + _random_reads(seed, bcs, max_edits=0)


def _dual(value, seed):
    """Dual: 96 x 24 on pass 1, 96 x 26 on pass 2 with the round-up edge of (26, 3) -- reads with a verbatim
    pass-1 barcode in front and a pass-2 barcode at 2 or 3 substitutions at the end."""
    rng = np.random.default_rng(seed)
    b1, b2 = _barcodes(seed, 96, 24), _barcodes(seed + 1, 96, 26)
    reads = []
    for b in range(0, 96, 6):
        for cols in ((3, 10, 17), (3, 10)):
            r2 = planted(rng, b2, near_neighbour(b2[b], cols), {b: len(cols)}, left=40, right=3)
            reads.append(flank(rng, 5) + b1[b].encode() + r2)
    return _cfg(b1, b2, max_error_rate=value), reads + _random_reads(seed, b1, bcs2=b2)


def _one_level(value, seed):
    """16 x 26: a single k_seed level at K = allowed = 3 that decides score-only passes itself (no k_literal
    re-alignment behind it); reads at 2 and 3 substitutions."""
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, 16, 26)
    reads = _spread_reads(rng, bcs, (2, 3), per=4, cols_of=lambda m, k: (3, 10, 17)[:k])
    return _cfg(bcs, max_error_rate=value), reads + _random_reads(seed, bcs, max_edits=3)


def _round_down(m, d, n_bc, value, seed, **kw):
    """n_bc x m at the round-down edge thr = fl(d/m): the score test accepts d, the DP allows d - 1."""
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, n_bc, m)
    reads = _spread_reads(rng, bcs, (d - 1, d), per=3)
    return _cfg(bcs, max_error_rate=value, **kw), reads + _random_reads(seed, bcs, max_edits=d)


_T26, _T25, _T24 = math.nextafter(3 / 26, 0.0), math.nextafter(5 / 25, 0.0), math.nextafter(5 / 24, 0.0)
_NS_NP = 4 | 2          # BDX_DEBUG_NO_SEEDS | BDX_DEBUG_NO_PREFILTER

# name: (edge value, builder(value) -> (cfg, reads), BDX_DEBUG_* flags, plan step that has to run, counter that
# proves it decided reads: "seed" / "prefilter" / "automaton" (work_counters) or a profiling stage name)
EDGE_CASES = {
    "k_seed_26_trim3": (_T26, lambda v: _seed26(v, 26, min_delta=0.12, trim_side=3), 0, "k_seed@2", "seed"),
    "k_seed_26_summary": (_T26, lambda v: _seed26(v, 27, min_delta=0.12, summary=True), 0, "k_seed@2", "seed"),
    "k_seed_26_score_only": (_T26, lambda v: _seed26(v, 28, min_delta=0.12), 0, "k_seed_var@1", "seed"),
    "k_seed_26_nodelta_trim3": (_T26, lambda v: _seed26(v, 29, trim_side=3), 0, "k_seed@2", "seed"),
    "k_seed_var_26_nodelta": (_T26, lambda v: _seed26(v, 30), 0, "k_seed_var@1", "seed"),
    "k_seed_25_bound": (min_delta_edge(0, 25, 4, 25), lambda v: _bound(25, v, 31, _T25), 0, "k_seed@2", "seed"),
    "k_seed_24_bound": (min_delta_edge(0, 24, 4, 24), lambda v: _bound(24, v, 32, _T24), 0, "k_seed@2", "seed"),
    "k_seed_deep_24": (_T24, lambda v: _small(24, 5, (1, 5, 9, 13, 17), v, 33), 0, "k_seed_deep", "seed"),
    # score-only: k_seed_deep's verdicts are final (no k_literal behind it); columns 1, 7, 13, 19 break every
    # segment of k_seed's level (K = 3), column 20 in addition leaves only the depth-5 segment [8, 12) intact
    "k_seed_deep_24_score_only": (_T24, lambda v: _small(24, 5, (1, 7, 13, 19, 20), v, 49, n_bc=8, trim=0), 0,
                                  "k_seed_deep", "seed"),
    "k_seed_deep_13": (math.nextafter(3 / 13, 0.0), lambda v: _small(13, 3, (1, 5, 9), v, 34), 0, "k_literal@rest", "seed"),
    "k_seed_small_26": (_T26, lambda v: _small(26, 3, (3, 10, 17), v, 35), 0, "k_literal@rest", "seed"),
    "k_seed_var_thr": (_T25, lambda v: _varlen(v, 36), 0, "k_seed_var@1", "seed"),
    "k_seed_var_min_delta": (min_delta_edge(1, 20, 3, 25), lambda v: _varlen(v, 37, option="min_delta"), 0,
                             "k_seed_var@1", "seed"),
    "k_seed_var_config3": (_T25, lambda v: _varlen(v, 38, geometry="config3"), 0, "k_seed_var@1", "seed"),
    "k_filter_26_delta": (_T26, lambda v: _seed26(v, 39, min_delta=0.12), _NS_NP, "k_filter", "automaton"),
    "k_filter_26_nodelta": (_T26, lambda v: _seed26(v, 40), _NS_NP, "k_filter", "automaton"),
    "k_filter_varlen_min_delta": (min_delta_edge(1, 20, 3, 25), lambda v: _varlen(v, 41, option="min_delta"), _NS_NP,
                                  "k_filter", "automaton"),
    "weighted_24": (_T24, lambda v: _weighted(v, 42), 0, "k_literal@full", "k_literal"),
    "k_seed_one_level_26": (_T26, lambda v: _one_level(v, 45), 0, "k_seed@1", "seed"),
    "round_down_47": (3 / 47, lambda v: _round_down(47, 3, 96, v, 46), 0, "k_seed@1", "seed"),
    "round_down_47_trim3": (3 / 47, lambda v: _round_down(47, 3, 96, v, 47, trim_side=3), 0, "k_literal@full",
                            "k_literal"),
    "round_down_98_literal": (2 / 98, lambda v: _round_down(98, 2, 16, v, 48), 0, "k_literal@all", "k_literal"),
    "dual_pass2_26": (_T26, lambda v: _dual(v, 43), 0, None, "seed"),
}
for _m, _d in ((13, 3), (24, 5), (25, 5), (26, 3)):
    for _trim in (3, 5):
        EDGE_CASES[f"k_hamming_scan_{_m}_trim{_trim}"] = (
            math.nextafter(_d / _m, 0.0), (lambda m, d, t, s: lambda v: _hamming(m, d, t, v, s))(_m, _d, _trim, 44 + _m + _trim),
            0, "k_hamming_scan", "k_hamming_scan")

EXTREME_ALGORITHMS = ("semiglobal", "hamming", "exact")


def sigma_case(value, seed=90):
    """200 barcodes of 16..28 nt, thr 0.2, k_seed_var's level 1 incomplete: verbatim reads, whose runner-ups the
    level does not see, are decided by its bound sigma - s1 >= min_delta with s1 = 0.  Returns (cfg, reads, sigma)
    with sigma = min over b of fl((K_b + 1) / m_b), K_b = min(m_b / q - 1, allowed_b) (tables.cu)."""
    rng = np.random.default_rng(seed)
    bcs = _barcodes(seed, 200, 16, 28)
    reads = [planted(rng, bcs, bcs[b], {b: 0}) for b in range(0, 200, 5)]
    return _cfg(bcs, max_error_rate=0.2, min_delta=value), reads


def sigma_of(bcs, thr, q):
    return min((min(len(b) // q - 1, allowed(thr, len(b))) + 1) / len(b) for b in bcs)


def extreme_case(algorithm, thr, min_delta, seed=50):
    """96 x 24 with an identical pair (barcodes 2 and 5) and a pair one substitution apart (11, 41)."""
    rng = np.random.default_rng(seed)
    bcs = _pair_set(24, (7,), seed)
    bcs[5] = bcs[2]
    reads = [flank(rng, 20) + bcs[b].encode() + flank(rng, 30) for b in (2, 5, 11, 41, 0, 1)]
    reads += [flank(rng, 20) + near_neighbour(bcs[b], (4,)).encode() + flank(rng, 30) for b in (2, 11, 0)]
    reads += _random_reads(seed, bcs, max_edits=3) + [b"", b"ACGT"]
    return _cfg(bcs, max_error_rate=thr, min_delta=min_delta, matching_algorithm=algorithm), reads
