"""Search-window input, host side (bdx_window_spans / bdx_window_reads): the spans agree with a derivation of their
own from the reference's range semantics, and the rule is sound -- on the oracle, replacing every read byte outside
the spans changes no result, pass detail or DemuxStats entry -- and tight enough that shrinking a span by one column
is caught."""
import numpy as np
import pytest

import orc
import windows_cases as wc
from bdx_b200 import capi
from bdx_b200.ranges import resolve
from bdx_b200.stats import stats_from_passes


@pytest.fixture(scope="module")
def lib():
    capi.build_library()
    return capi.load_library()


def py_spans(cfg, n, shrink=None):
    """The window rule from the reference's resolve() and match_barcode_pass prologue.  shrink: a deliberately
    too small window -- "sg" (end_j - 1), "no_tail" (:hamming / :exact without the max_m - 1 columns)."""
    sets = [(cfg.ref_search_range, cfg.barcode_start_range, cfg.barcode_end_range, cfg.bc_seqs)]
    if cfg.is_dual:
        sets.append((cfg.ref_search_range2, cfg.barcode_start_range2, cfg.barcode_end_range2, cfg.bc_seqs2))
    spans = []
    for rs, bs, be, bcs in sets:
        rf, rl = resolve(rs, n)
        bf, bl = resolve(bs, n)
        ef, el = resolve(be, n)
        start, end = max(rf, bf, 1), min(rl, el, n)
        if start > end or start > bl or end < ef:
            continue
        if cfg.matching_algorithm == "semiglobal":
            hi = end - (shrink == "sg")
        else:
            hi = min(n, min(end, bl) + (0 if shrink == "no_tail" else max(len(b) for b in bcs) - 1))
        if hi >= start:
            spans.append([start, hi])
    spans.sort()
    if len(spans) == 2 and spans[1][0] <= spans[0][1] + 1:
        spans = [[spans[0][0], max(spans[0][1], spans[1][1])]]
    return [tuple(s) for s in spans]


def c_spans(config, n):
    (lo1, hi1, lo2, hi2), total = config.window_spans(n)
    out = [(lo, hi) for lo, hi in ((lo1, hi1), (lo2, hi2)) if hi >= lo]
    assert total == sum(hi - lo + 1 for lo, hi in out)
    if len(out) == 2:
        assert out[0][1] + 1 < out[1][0]          # sorted, not touching
    assert (lo2, hi2) == (1, 0) or len(out) == 2   # an absent second span reads (1, 0)
    return out


@pytest.mark.parametrize("name", sorted(wc.CASES))
def test_spans_match_the_reference_ranges(lib, name):
    cfg, _, _ = wc.make_case(name, np.random.default_rng(sum(map(ord, name))))
    config = capi.Config(cfg)
    for n in range(0, 401):
        assert c_spans(config, n) == py_spans(cfg, n), (name, n)
    config.close()


def test_spans_of_the_long_read_geometries(lib):
    """1:120 and end-119:end on a 3 kb read: 240 of 3004 bytes."""
    cfg, _, _ = wc.make_case("sg_dual", np.random.default_rng(1))
    cfg.ref_search_range, cfg.ref_search_range2 = wc.R("1:120"), wc.R("end-119:end")
    config = capi.Config(cfg)
    assert config.window_spans(3004) == ((1, 120, 2885, 3004), 240)
    assert config.window_spans(200) == ((1, 200, 1, 0), 200)      # the two ranges overlap: one span
    assert config.window_spans(240) == ((1, 240, 1, 0), 240)      # they touch
    assert config.window_spans(0) == ((1, 0, 1, 0), 0)
    config.close()


def scrambled(reads, spans_of, rng, alphabet):
    """The reads with every byte outside spans_of(len) replaced: random bytes of `alphabet`, or the filler."""
    out = []
    for r in reads:
        x = bytearray(alphabet[rng.integers(0, len(alphabet), len(r))].tobytes()) if len(alphabet) > 1 \
            else bytearray(bytes(alphabet) * len(r))
        for lo, hi in spans_of(len(r)):
            x[lo - 1:hi] = r[lo - 1:hi]
        out.append(bytes(x))
    return out


def differences(cfg, reads, spans_of, seed):
    """Fields in which the oracle's results on scrambled reads differ from those on the originals."""
    o = orc.Oracle(cfg)
    want = o.classify_reads(reads)
    rng = np.random.default_rng(seed)
    alphabets = [np.frombuffer(b"ACGTN", np.uint8), np.zeros(1, np.uint8)]    # barcode bytes; the filler (0)
    found = set()
    for alpha in alphabets:
        got = o.classify_reads(scrambled(reads, spans_of, rng, alpha))
        for f in ("status", "bc1", "bc2", "keep_start", "keep_end"):
            if (got[f] != want[f]).any():
                found.add(f)
        for f in ("status", "bc", "start", "end", "score"):
            if (got["passes"][f] != want["passes"][f]).any():
                found.add("pass " + f)
        if cfg.summary and not found:
            def stats(r):
                passes = [[tuple(r["passes"][i, p][k] for k in ("status", "bc", "start", "end", "score"))
                           for p in (0, 1)] for i in range(len(r))]
                return stats_from_passes(r["status"], r["bc1"], r["bc2"], passes, cfg)
            if stats(got) != stats(want):
                found.add("stats")
    return found


@pytest.mark.parametrize("name", sorted(wc.CASES))
def test_bytes_outside_the_windows_change_nothing(lib, name):
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    cfg, b1, b2 = wc.make_case(name, rng)
    reads = wc.make_reads(rng, b1, b2, 3000)
    config = capi.Config(cfg)
    cache = {}

    def spans_of(n):
        if n not in cache:
            cache[n] = c_spans(config, n)
        return cache[n]

    assert differences(cfg, reads, spans_of, seed=5) == set(), name
    config.close()


@pytest.mark.parametrize("shrink,algos", [("sg", ("semiglobal",)), ("no_tail", ("hamming", "exact"))])
def test_a_window_one_column_short_is_caught(lib, shrink, algos):
    """The soundness check above has teeth: with a span cut short it finds a difference for some config."""
    caught = []
    for name in sorted(wc.CASES):
        if wc.CASES[name][2].get("matching_algorithm", "semiglobal") not in algos:
            continue
        rng = np.random.default_rng(sum(map(ord, name)) + 1)
        cfg, b1, b2 = wc.make_case(name, rng)
        reads = wc.make_reads(rng, b1, b2, 3000)
        if differences(cfg, reads, lambda n: py_spans(cfg, n, shrink), seed=5):
            caught.append(name)
    assert caught, shrink


def test_window_reads_layout_and_refusals(lib):
    rng = np.random.default_rng(9)
    cfg, b1, b2 = wc.make_case("sg_dual", rng)
    reads = wc.make_reads(rng, b1, b2, 400)
    config = capi.Config(cfg)
    seq, off = orc.pack_reads(reads)
    win, win_off = config.window_reads(seq, off)
    want = [b"".join(r[lo - 1:hi] for lo, hi in c_spans(config, len(r))) for r in reads]
    assert win_off[0] == 0 and (np.diff(win_off) == [len(w) for w in want]).all()
    assert win.tobytes() == b"".join(want)
    # sizing call: win_bytes = NULL fills only the offsets
    L = config.lib
    off32 = off.astype(np.int32)
    sized = np.full(len(reads) + 1, -7, np.int32)
    assert L.bdx_window_reads(config.handle, None, off32.ctypes.data, len(reads), None, sized.ctypes.data) == 0
    assert (sized == win_off).all()
    # refusals
    bad_off = off32.copy()
    bad_off[3] = bad_off[4] + 1
    first = off32.copy()
    first[0] = 1
    for args in ((seq.ctypes.data, bad_off.ctypes.data, len(reads), None, sized.ctypes.data),
                 (seq.ctypes.data, first.ctypes.data, len(reads), None, sized.ctypes.data),
                 (seq.ctypes.data, off32.ctypes.data, -1, None, sized.ctypes.data),
                 (seq.ctypes.data, off32.ctypes.data, len(reads), None, None),
                 (None, off32.ctypes.data, len(reads), win.ctypes.data, sized.ctypes.data)):
        assert L.bdx_window_reads(config.handle, *args) == capi.BDX_ERR_INVALID, args
    assert L.bdx_window_spans(config.handle, -1, sized.ctypes.data) == capi.BDX_ERR_INVALID
    assert L.bdx_window_spans(None, 10, sized.ctypes.data) == capi.BDX_ERR_INVALID
    empty_off = np.zeros(1, np.int32)
    assert config.window_reads(np.zeros(0, np.uint8), empty_off)[1].tolist() == [0]
    config.close()
