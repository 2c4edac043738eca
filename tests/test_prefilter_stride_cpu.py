"""The sampled table of k_prefilter<0> (csrc/tables.cu build_prefilter, csrc/filter.cu pf_scan) on the CPU: the
arithmetic that makes sampling exact for verbatim occurrences, and the stride and table sizes the host chooses for the
benchmark configs and for other sets (bdx_config_describe's `prefilter:` line)."""
import numpy as np
import pytest

import bdx_b200 as bdx
from bdx_b200 import capi
import synth

R = bdx.parse_dynamic_range
ADAPTER = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"


def _cover_counts(ncols, q, stride):
    """For every start s: the (sampled column, table offset) pairs that name s -- the scan hashes the q-mer at every
    column P = 0, stride, 2 stride, ... with P + q <= ncols and turns a table entry of offset o into the start P - o"""
    hits = [[] for _ in range(ncols)]
    for p in range(0, ncols - q + 1, stride):
        for o in range(stride):
            if p - o >= 0:
                hits[p - o].append((p, o))
    return hits


@pytest.mark.parametrize("q", [6, 7, 9, 12])
def test_every_start_is_named_once(q):
    """Every occurrence start s of a barcode of length m >= m_min that fits the scanned columns is named by exactly
    one (sampled column, offset) pair, whose q-mer lies inside the barcode's first m_min bases; for every stride up to
    m_min - q + 1, and m_min from q (stride 1) upwards."""
    for m_min in range(q, q + 30):
        lengths = sorted({m_min, m_min + 1, m_min + 7, m_min + 30})
        for stride in sorted({1, 2, (m_min - q + 2) // 2, m_min - q + 1}):
            if stride < 1 or stride > m_min - q + 1:
                continue
            for ncols in (m_min, m_min + 1, 150, 401):
                hits = _cover_counts(ncols, q, stride)
                for m in lengths:
                    for s in range(0, 401):
                        if s + m > ncols:
                            break
                        assert len(hits[s]) == 1, (q, m_min, stride, ncols, m, s, hits[s])
                        p, o = hits[s][0]
                        assert o + q <= m_min and p + q <= ncols, (q, m_min, stride, m, s, p, o)


def _describe(cfg, pass_=0):
    text = capi.Config(cfg).describe(pass_)
    line = [ln for ln in text.splitlines() if ln.startswith("prefilter:")][0]
    return {k: int(v) for k, v in (x.split("=") for x in line.split(": ", 1)[1].split())}


def _smem(log2, bm_log2):
    """k_prefilter's dynamic shared memory (filter.cu prefilter_smem_bytes): read staging, keys + values, bitmap"""
    return 48 * 1024 + 16 + (8 << log2) + (4 << (bm_log2 - 5))


def _blocks(smem):
    """resident 256-thread blocks an sm_100 SM holds at that shared memory (228 KB, 1 KB reserved per block)"""
    return min(8, 228 * 1024 // (smem + 1024))


def _prefix_log2(n_bc):
    lg = 4
    while (1 << lg) < 2 * n_bc:
        lg += 1
    return lg


def _expected(n_bc, min_m, semiglobal=True):
    """(stride, log2, bitmap_log2) by the host's rule: the largest stride in 4 .. min_m - q + 1 whose table (load
    <= 3/4) keeps the prefix table's resident blocks, else 1"""
    q = min(min_m, 12)
    bl = 13
    while bl < 18 and (1 << bl) < 512 * n_bc:
        bl += 1
    blocks = max(1, _blocks(_smem(_prefix_log2(n_bc), bl)))
    for s in range(min_m - q + 1 if semiglobal else 1, 3, -1):
        lg = 4
        while 3 * (1 << lg) < 4 * n_bc * s:
            lg += 1
        if _blocks(_smem(lg, bl)) >= blocks:
            return s, lg, bl
    return 1, _prefix_log2(n_bc), bl


def _cfg(bcs, **kw):
    return bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[len(b) for b in bcs], ids=[f"b{i}" for i in range(len(bcs))],
                           **kw)


def test_benchmark_configs():
    """Config 2 and config 4's barcodes sample every 13th column, config 4's adapter every 22nd; none of them loses a
    resident block of k_prefilter against the prefix table.  Config 5's 1536 barcodes would fit stride 2 only, below
    the minimum: they keep the rolling scan."""
    rng = np.random.default_rng(0x42444D58)
    b96 = synth.random_barcodes(rng, 96, 24)
    b1536 = synth.random_barcodes(rng, 1536, 24)
    cfg4 = _cfg(b96, ref_search_range=R("1:32"), trim_side=5)
    cfg4.is_dual = True
    cfg4.bc_seqs2, cfg4.bc_lengths_no_N2, cfg4.ids2, cfg4.trim_side2 = [ADAPTER], [len(ADAPTER)], ["adapter"], 3
    cases = [(_cfg(b96), 0, 96, 24, 13), (cfg4, 0, 96, 24, 13), (cfg4, 1, 1, 33, 22), (_cfg(b1536), 0, 1536, 24, 1)]
    for cfg, pass_, n_bc, m, stride in cases:
        d = _describe(cfg, pass_)
        assert d["seed"] == 12 and d["stride"] == stride, d
        assert (d["stride"], d["log2"], d["bitmap_log2"]) == _expected(n_bc, m), d
        assert 4 * n_bc * stride <= 3 * (1 << d["log2"]), d
        assert _blocks(_smem(d["log2"], d["bitmap_log2"])) >= _blocks(_smem(_prefix_log2(n_bc), d["bitmap_log2"])), d
    # config 2: three resident blocks of 256 threads, as with the prefix table
    d = _describe(_cfg(b96))
    assert _blocks(_smem(d["log2"], d["bitmap_log2"])) == 3


def test_other_sets_and_algorithms():
    """Random sets: the stride rule above; :hamming and :exact keep the prefix table; sets whose shortest barcode
    has 14 nt or less (stride <= 3) have stride 1."""
    rng = np.random.default_rng(5)
    for n_bc, lo, hi in ((1, 6, 6), (3, 12, 12), (8, 13, 13), (40, 16, 28), (200, 20, 40), (700, 30, 30),
                         (1000, 24, 24), (2000, 14, 50), (5000, 24, 24)):
        bcs = synth.random_barcodes(rng, n_bc, lo, hi)
        min_m = min(len(b) for b in bcs)
        d = _describe(_cfg(bcs))
        assert (d["stride"], d["log2"], d["bitmap_log2"]) == _expected(n_bc, min_m), (n_bc, lo, hi, d)
        if min_m <= 14:
            assert d["stride"] == 1
        for algo in ("hamming", "exact"):
            d = _describe(_cfg(bcs, matching_algorithm=algo))
            assert (d["stride"], d["log2"]) == (1, _prefix_log2(n_bc)), (algo, d)
