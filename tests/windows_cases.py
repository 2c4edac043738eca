"""Configs and reads shared by the search-window input tests (bdx_window_spans / bdx_submit_windows): every kind of
range geometry the window rule distinguishes, for all three algorithms, single and dual sets."""
from __future__ import annotations

import numpy as np

import bdx_b200 as bdx
import synth

R = bdx.parse_dynamic_range

# name -> (barcode lengths (set 1, set 2 or None), DemuxConfig keywords)
CASES = {
    "sg_full": ((24, 24), None, dict()),
    "sg_start": ((16, 28), None, dict(ref_search_range=R("1:40"), barcode_start_range=R("1:6"), min_delta=0.1,
                                      trim_side=5, max_error_rate=0.3)),
    "sg_end_stats": ((16, 28), None, dict(ref_search_range=R("end-39:end"), barcode_end_range=R("end-5:end"),
                                          trim_side=3, summary=True)),
    "sg_weighted_sub": ((20, 24), None, dict(ref_search_range=R("3:45"), barcode_end_range=R("20:end"), mismatch=2,
                                             indel=3, max_error_rate=0.3, trim_side=3, summary=True)),
    "sg_nindel": ((20, 26), None, dict(ref_search_range=R("1:50"), nindel=1, max_error_rate=0.3, n_frac=0.15)),
    "sg_longer_than_reads": ((24, 24), None, dict(ref_search_range=R("1:500"), trim_side=5)),
    "sg_invalid_rs": ((12, 18), None, dict(ref_search_range=R("10:5"))),
    "sg_invalid_bs": ((12, 18), None, dict(barcode_start_range=R("end+3:end"), trim_side=3)),
    "sg_invalid_be": ((12, 18), None, dict(barcode_end_range=R("end+1:end"))),
    "sg_dual": ((16, 28), (16, 28), dict(ref_search_range=R("1:40"), ref_search_range2=R("end-39:end"),
                                         trim_side=5, trim_side2=3, min_delta=0.05, summary=True)),
    "sg_dual_overlap": ((20, 24), (20, 24), dict(ref_search_range=R("1:80"), ref_search_range2=R("60:end-10"),
                                                 trim_side=5)),
    "ham_start": ((24, 24), None, dict(matching_algorithm="hamming", ref_search_range=R("1:60"), trim_side=3)),
    "ham_var_bs": ((6, 12), None, dict(matching_algorithm="hamming", barcode_start_range=R("1:30"),
                                       barcode_end_range=R("10:end"), trim_side=5, min_delta=0.1,
                                       max_error_rate=0.34)),
    "ham_end_stats": ((16, 20), None, dict(matching_algorithm="hamming", ref_search_range=R("end-49:end"),
                                           trim_side=3, summary=True, max_error_rate=0.15)),
    "ham_dual": ((16, 16), (20, 20), dict(matching_algorithm="hamming", ref_search_range=R("1:30"),
                                          ref_search_range2=R("end-29:end"), trim_side=5, trim_side2=3)),
    "exact_trim3": ((4, 8), None, dict(matching_algorithm="exact", ref_search_range=R("5:70"), trim_side=3)),
    "exact_end5": ((10, 14), None, dict(matching_algorithm="exact", ref_search_range=R("end-50:end"), trim_side=5)),
    "exact_bs3": ((6, 10), None, dict(matching_algorithm="exact", barcode_start_range=R("1:20"), trim_side=3,
                                      summary=True)),
    "exact_dual": ((8, 12), (8, 12), dict(matching_algorithm="exact", ref_search_range=R("1:30"),
                                          ref_search_range2=R("end-29:end"), trim_side=5, trim_side2=3)),
}


def make_case(name, rng, n_bc=40):
    (lo1, hi1), set2, kw = CASES[name]
    kw = dict(kw)
    n_frac = kw.pop("n_frac", 0.0)
    b1 = synth.random_barcodes(rng, n_bc, lo1, hi1, n_frac=n_frac)
    cfg = bdx.DemuxConfig(bc_seqs=b1, bc_lengths_no_N=[sum(c != "N" for c in b) for b in b1],
                          ids=[f"a{i}" for i in range(n_bc)], **kw)
    b2 = None
    if set2:
        b2 = synth.random_barcodes(rng, n_bc, set2[0], set2[1])
        cfg.is_dual, cfg.bc_seqs2, cfg.bc_lengths_no_N2 = True, b2, [len(b) for b in b2]
        cfg.ids2 = [f"b{i}" for i in range(n_bc)]
    return cfg, b1, b2


def make_reads(rng, b1, b2, n):
    """Short, medium and long reads with barcodes planted near both ends, where the search windows begin and end."""
    reads = synth.random_reads(rng, n // 2, b1, barcodes2=b2, min_len=0, max_len=160, start_hi=60, max_edits=2)
    reads += synth.random_reads(rng, n // 4, b1, barcodes2=b2, min_len=100, max_len=400, start_hi=90, max_edits=2)
    for r in synth.random_reads(rng, n - len(reads), b1, min_len=30, max_len=90, start_hi=40, max_edits=1):
        reads.append(bytes(synth.BASES[rng.integers(0, 4, int(rng.integers(0, 300)))]) + r)   # barcodes near the end
    reads += [b"", b"A", b"ACGT"]
    return reads
