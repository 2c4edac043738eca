"""k_prefilter<0> with a sampled table (csrc/filter.cu, pf_scan): the q-mer of every stride-th column against the q-mers
at offsets 0 .. stride - 1 of every barcode.  Verbatim occurrences at every residue mod stride, at both ends of the
search range and one column outside it, competing occurrences of different and of the same barcode, internal repeats,
duplicate sequences, N bytes, mixed lengths and config 4's adapter pass -- bit-exact against the oracle (results, pass
details, DemuxStats), with proof that k_prefilter ran at the stride the case is for and decided reads."""
import numpy as np
import pytest

import bdx_b200 as bdx
from bdx_b200 import capi
import synth
from gpu_common import compare

pytestmark = pytest.mark.gpu
R = bdx.parse_dynamic_range
ADAPTER = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"
READ_LEN = 150


def _cfg(bcs, **kw):
    return bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[len(b) for b in bcs], ids=[f"bc{i}" for i in range(len(bcs))],
                           **kw)


def _flank(rng, n):
    return bytes(synth.BASES[rng.integers(0, 4, n)])


def _plant(rng, items, length=READ_LEN):
    """A random read of `length` bases with each (start, bytes) of `items` written over it (0-based starts)."""
    r = bytearray(_flank(rng, length))
    for s, b in items:
        r[s:s + len(b)] = b
    return bytes(r[:length])


def _stride(cfg, pass_=0):
    text = capi.Config(cfg).describe(pass_)
    line = [ln for ln in text.splitlines() if ln.startswith("prefilter:")][0]
    return int(line.split("stride=")[1].split()[0])


def _prefilter_reads(cfg, reads, want_stats=False):
    """(plan of pass 1, reads k_prefilter decided) of one run of the batch"""
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=len(reads), max_bytes=max(int(off[-1]), 16), want_stats=want_stats) as eng:
        plan = [ln for ln in eng.config.describe(0).splitlines() if ln.startswith("plan:")][0]
        eng.stream.work_counters(reset=True)
        eng.classify_packed(blob, off)
        return plan, eng.stream.work_counters()[0]


def _check(cfg, reads, label, stride, want_stats=False):
    assert _stride(cfg) == stride, label
    compare(cfg, reads, want_stats=want_stats, label=label)
    plan, decided = _prefilter_reads(cfg, reads, want_stats)
    assert "k_prefilter" in plan, (label, plan)
    assert decided > 0, label
    return decided


def _set_96x24(seed=11):
    return synth.random_barcodes(np.random.default_rng(seed), 96, 24)


def _every_start_reads(rng, bcs, starts, length=READ_LEN):
    return [_plant(rng, [(s, bcs[(s * 7 + k) % len(bcs)].encode())], length) for s in starts for k in range(3)]


@pytest.mark.parametrize("opts", [dict(), dict(trim_side=5), dict(trim_side=3), dict(stats=True)],
                         ids=["score", "trim5", "trim3", "stats"])
def test_every_residue_and_both_ends(opts):
    """Occurrences at every start 0 .. 126 of a 150-column range (every residue mod 13, the first and the last start
    the range allows), and reads cut one column short at either end."""
    rng = np.random.default_rng(1)
    bcs = _set_96x24()
    opts = dict(opts)
    stats = opts.pop("stats", False)
    reads = _every_start_reads(rng, bcs, range(READ_LEN - 24 + 1))
    reads += [bcs[3].encode()[1:] + _flank(rng, 100), _flank(rng, 100) + bcs[4].encode()[:-1]]
    reads += [bcs[3].encode(), bcs[5].encode() + bcs[6].encode()]
    decided = _check(_cfg(bcs, **opts), reads, f"every start {opts}", 13, want_stats=stats)
    assert decided >= 3 * (READ_LEN - 24 + 1)


@pytest.mark.parametrize("rs", ["1:40", "end-39:end"])
@pytest.mark.parametrize("trim", [0, 3, 5])
def test_search_range_edges(rs, trim):
    """A 40-column search range: every start inside it, and occurrences that begin or end one column outside."""
    rng = np.random.default_rng(2)
    bcs = _set_96x24()
    lo = 0 if rs == "1:40" else READ_LEN - 40
    reads = _every_start_reads(rng, bcs, range(lo, lo + 40 - 24 + 1))
    reads += _every_start_reads(rng, bcs, [lo - 1, lo + 40 - 24 + 1] if lo else [lo + 40 - 24 + 1])
    opts = dict(ref_search_range=R(rs))
    if trim:
        opts["trim_side"] = trim
    _check(_cfg(bcs, **opts), reads, f"range {rs} trim {trim}", 13)


@pytest.mark.parametrize("trim", [0, 3, 5])
def test_competing_occurrences(trim):
    """Two different barcodes (the lower index wins wherever it is), and the same barcode twice: far apart, a stride
    apart and less than a stride apart (leftmost, or rightmost with trim_side 3)."""
    rng = np.random.default_rng(3)
    bcs = _set_96x24()
    reads = []
    for _ in range(150):
        a, b = sorted(rng.choice(96, 2, replace=False))
        s1 = int(rng.integers(0, 50))
        s2 = int(rng.integers(s1 + 24, READ_LEN - 24 + 1))
        reads.append(_plant(rng, [(s1, bcs[a].encode()), (s2, bcs[b].encode())]))
        reads.append(_plant(rng, [(s1, bcs[b].encode()), (s2, bcs[a].encode())]))
        reads.append(_plant(rng, [(s1, bcs[a].encode()), (s2, bcs[a].encode())]))
    # a period-6 barcode: occurrences 6 columns apart share a stride window and its q-mers at offsets 0, 6 and 12
    # are one table key
    periodic = "ACGTTG" * 4
    bcs2 = bcs[:10] + [periodic] + bcs[10:]
    for s in range(0, 40):
        reads.append(_plant(rng, [(s, ("ACGTTG" * 5).encode())]))
        reads.append(_plant(rng, [(s, ("ACGTTG" * 6).encode())]))
        reads.append(_plant(rng, [(s, periodic.encode()), (s + 13, periodic.encode())]))
        reads.append(_plant(rng, [(s, periodic.encode()), (s + 30, periodic.encode())]))
        reads.append(_plant(rng, [(s, bcs[s].encode()), (s + 24, bcs[s].encode())]))
    opts = dict(trim_side=trim) if trim else {}
    _check(_cfg(bcs2, **opts), reads, f"competing trim {trim}", 13)


def test_internal_repeats_and_duplicates():
    """Barcodes whose q-mers repeat inside them or across barcodes, and identical sequences (the lowest index
    wins)."""
    rng = np.random.default_rng(4)
    base = _set_96x24()
    rep = ["ACGTACGTACGTACGTACGTACGT", "AAAAAAAAAAAAAAAAAAAAAAAA", "ACGTTGCAACGTTGCAACGTTGCA",
           base[0][:12] * 2, base[1][:13] + base[1][:11]]
    # base[2]'s 12-mer at offset 5 is base[3]'s at offset 0: one key, two entries
    shared = base[3][:12]
    b2 = base[2][:5] + shared + base[2][17:]
    bcs = base[:2] + [b2] + base[3:20] + rep + [base[7], base[3], b2] + base[20:]
    reads = []
    for b in range(len(bcs)):
        for s in (0, 7, 13, 51, READ_LEN - 24):
            reads.append(_plant(rng, [(s, bcs[b].encode())]))
    for s in range(0, 30):
        reads.append(_plant(rng, [(s, ("ACGT" * 12).encode())]))
        reads.append(_plant(rng, [(s, ("A" * 40).encode())]))
    reads += [b"A" * READ_LEN, b"ACGT" * 37, (bcs[2] + bcs[3]).encode() * 3]
    _check(_cfg(bcs), reads, "repeats and duplicates", 13)
    _check(_cfg(bcs, trim_side=3), reads, "repeats and duplicates trim 3", 13, want_stats=True)


def test_n_inside_occurrences():
    """An N anywhere inside an occurrence makes it not verbatim; N bytes next to one do not."""
    rng = np.random.default_rng(5)
    bcs = _set_96x24()
    reads = []
    for s in (0, 13, 26, 60, READ_LEN - 24):
        for i in range(24):
            b = bytearray(bcs[(s + i) % 96].encode())
            b[i] = ord("N")
            reads.append(_plant(rng, [(s, bytes(b))]))
        r = bytearray(_plant(rng, [(s, bcs[s % 96].encode())]))
        if s > 0:
            r[s - 1] = ord("N")
        if s + 24 < READ_LEN:
            r[s + 24] = ord("N")
        reads.append(bytes(r))
    _check(_cfg(bcs), reads, "N bytes", 13)
    _check(_cfg(bcs, trim_side=5), reads, "N bytes trim 5", 13, want_stats=True)


def test_mixed_lengths():
    """Barcodes of 24 .. 31 nt (stride 13 from the shortest): the longer ones are found through their first 24 bases,
    including barcodes that extend or contain others."""
    rng = np.random.default_rng(6)
    bcs = synth.random_barcodes(rng, 80, 24, 31)
    short = [b for b in bcs if len(b) == 24][:4]
    bcs += [short[0] + "ACGTAC", "TT" + short[1], short[2] + short[2][:7], short[3][:24]]
    assert min(len(b) for b in bcs) == 24
    reads = []
    for b in range(len(bcs)):
        m = len(bcs[b])
        for s in (0, 5, 13, 40, READ_LEN - m):
            reads.append(_plant(rng, [(s, bcs[b].encode())]))
    for trim in (0, 3, 5):
        opts = dict(trim_side=trim) if trim else {}
        _check(_cfg(bcs, **opts), reads, f"mixed lengths trim {trim}", 13)


def test_config4_adapter_pass():
    """Config 4: 96 barcodes (1:32, trim 5') in front of the 33-nt adapter (trim 3'), whose pass samples every 22nd
    column: the adapter at every start, twice, and cut short by the read's end."""
    rng = np.random.default_rng(7)
    bcs = _set_96x24()
    cfg = _cfg(bcs, ref_search_range=R("1:32"), trim_side=5)
    cfg.is_dual = True
    cfg.bc_seqs2, cfg.bc_lengths_no_N2, cfg.ids2, cfg.trim_side2 = [ADAPTER], [len(ADAPTER)], ["adapter"], 3
    assert _stride(cfg, 1) == 22
    a = ADAPTER.encode()
    reads = []
    for s in range(24, READ_LEN - len(a) + 1):
        reads.append(_plant(rng, [(s % 8, bcs[s % 96].encode()), (s, a)]))
    for s in range(24, 60, 3):
        reads.append(_plant(rng, [(1, bcs[s].encode()), (s, a), (s + 40, a)]))
        reads.append(_plant(rng, [(1, bcs[s].encode()), (s, a), (s + 20, a)]))
    reads.append(_plant(rng, [(0, bcs[1].encode()), (READ_LEN - 20, a)]))
    compare(cfg, reads, want_stats=True, label="config 4")
    compare(cfg, reads, label="config 4")


# reads k_prefilter decided on the batch of test_config2_decided_reads with the per-column prefix scan, before the
# sampled table (measured on one NVIDIA B200): sampling must not lose any
PREFIX_SCAN_DECIDED = 6489


def config2_batch(n=20000):
    """bench.py's workload (96 x 24 nt, 90 % planted with up to 5 edits, 0.5 % N) at a test's size"""
    rng = np.random.default_rng(8)
    bcs = synth.random_barcodes(rng, 96, 24)
    reads = synth.random_reads(rng, n, bcs, min_len=READ_LEN, plant=0.9, start_hi=119, n_prob=0.005)
    return _cfg(bcs), reads


def test_config2_decided_reads():
    cfg, reads = config2_batch()
    decided = _check(cfg, reads, "config 2 batch", 13)
    assert decided >= PREFIX_SCAN_DECIDED, (decided, PREFIX_SCAN_DECIDED)
