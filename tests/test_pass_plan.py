"""The kernel sequence of each pass (csrc/plan.cu) for a matrix of configs: on the CPU the `plan:` line of
bdx_config_describe, on the GPU the launches a profiled batch really makes, stage by stage."""
import numpy as np
import pytest

import bdx_b200 as bdx
from bdx_b200 import capi
import synth

R = bdx.parse_dynamic_range
ADAPTER = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"

# barcode sets: seed, count, shortest, longest, alphabet
SETS = {
    "96x24": (1, 96, 24, 24, b"ACGT"),
    "384x16..28": (2, 384, 16, 28, b"ACGT"),
    "384x16..28'": (3, 384, 16, 28, b"ACGT"),
    "1536x24": (4, 1536, 24, 24, b"ACGT"),
    "5x12": (5, 5, 12, 12, b"ACGT"),
    "96x16N": (6, 96, 16, 16, b"ACGTN"),
    "16x70": (7, 16, 70, 70, b"ACGT"),
    "9000x10": (8, 9000, 10, 10, b"ACGT"),
}
CONFIG3 = dict(ref_search_range=R("1:40"), barcode_start_range=R("1:6"), ref_search_range2=R("end-39:end"),
               barcode_end_range2=R("end-5:end"), min_delta=0.1)
CONFIG4 = dict(ref_search_range=R("1:32"), trim_side=5, trim_side2=3)

# id: (set of pass 0, set of pass 1 or None, DemuxConfig options, BDX_DEBUG_* flags, steps of each pass)
CASES = {
    "config2": ("96x24", None, {}, 0, ["k_prefilter,k_seed@1,k_seed_var@2,k_filter"]),
    "config2_trim5": ("96x24", None, dict(trim_side=5), 0,
                      ["k_prefilter,k_seed@1,k_seed@2,k_filter,k_literal@win,k_literal@full"]),
    "config2_summary": ("96x24", None, dict(summary=True), 0,
                        ["k_prefilter,k_seed@1,k_seed@2,k_filter,k_literal@win,k_literal@full"]),
    "config2_min_delta": ("96x24", None, dict(min_delta=0.1), 0, ["k_seed@1,k_seed_var@2,k_filter"]),
    "config2_indel2": ("96x24", None, dict(indel=2), 0, ["k_prefilter,k_filter,k_literal@full"]),
    "config2_prefer_seed_var": ("96x24", None, {}, capi.DEBUG_PREFER_SEED_VAR,
                                ["k_prefilter,k_seed_var@1,k_seed_var@2,k_filter"]),
    "config2_no_filter": ("96x24", None, {}, capi.DEBUG_NO_FILTER, ["k_literal@all"]),
    "config3": ("384x16..28", "384x16..28'", CONFIG3, 0,
                ["k_seed_var@1,k_seed_var@2,k_filter,k_literal@full"] * 2),
    "config4": ("96x24", "adapter", CONFIG4, 0,
                ["k_prefilter,k_seed@1,k_seed@2,k_filter,k_literal@win,k_literal@full",
                 "k_prefilter,k_seed@1,k_seed_deep,k_mark_pending,k_literal@win,k_literal@rest"]),
    "config5_semiglobal": ("1536x24", None, {}, 0, ["k_prefilter,k_seed@1,k_seed@2,k_filter"]),
    "config5_hamming": ("1536x24", None, dict(matching_algorithm="hamming"), 0, ["k_hamming_scan,k_literal@cand"]),
    "config5_exact": ("1536x24", None, dict(matching_algorithm="exact"), 0, ["k_prefilter,k_literal@cand"]),
    # fewer than 8 barcodes: no filter kernel; k_seed_var's level 1 is the complete level behind k_seed
    "small_set": ("5x12", None, {}, 0,
                  ["k_prefilter,k_seed@1,k_seed_var@1,k_mark_pending,k_literal@win,k_literal@rest"]),
    "hamming_with_N": ("96x16N", None, dict(matching_algorithm="hamming"), 0, ["k_filter,k_literal@full"]),
    "match_minus_1": ("96x24", None, dict(match=-1), 0, ["k_literal@all"]),
    "barcodes_over_64nt": ("16x70", None, {}, 0, ["k_literal@all"]),
    # k_prefilter's hash table needs 256 KB of shared memory, more than a block can have: the tables are built,
    # but neither k_prefilter nor the k_seed levels behind it run
    "prefilter_over_smem_limit": ("9000x10", None, {}, 0, ["k_filter"]),
}


def _barcodes(name):
    if name == "adapter":
        return [ADAPTER]
    seed, n, lo, hi, alphabet = SETS[name]
    return synth.random_barcodes(np.random.default_rng(seed), n, lo, hi, alphabet=alphabet)


def _case(case_id):
    """(DemuxConfig, debug flags, expected steps per pass, barcodes of both sets) of a CASES entry."""
    s1, s2, kw, debug, steps = CASES[case_id]
    b1, b2 = _barcodes(s1), _barcodes(s2) if s2 else None
    cfg = bdx.DemuxConfig(bc_seqs=b1, bc_lengths_no_N=[len(x) for x in b1], ids=[f"a{i}" for i in range(len(b1))], **kw)
    if b2:
        cfg.is_dual = True
        cfg.bc_seqs2, cfg.bc_lengths_no_N2, cfg.ids2 = b2, [len(x) for x in b2], [f"b{i}" for i in range(len(b2))]
    return cfg, debug, steps, b1, b2


@pytest.fixture(scope="module")
def lib():
    capi.build_library()
    return capi.load_library()


@pytest.mark.parametrize("case_id", list(CASES))
def test_plan_line(lib, case_id):
    """bdx_config_describe's `plan:` line (computed against sm_100's shared-memory limit) for each pass."""
    cfg, debug, steps, _, _ = _case(case_id)
    config = capi.Config(cfg, debug=debug)
    try:
        for p, want in enumerate(steps):
            lines = [ln for ln in config.describe(p).splitlines() if ln.startswith("plan:")]
            assert lines == [f"plan: steps={want}"], (case_id, p, lines)
        if len(steps) == 1:
            assert config.describe(1) == ""
    finally:
        config.close()


def _launches(steps_per_pass):
    """Launches per profiling stage (capi.Stream.STAGES) that the steps of every pass make, plus one k_finalize."""
    stage_of = {"k_prefilter": "k_prefilter", "k_seed": "k_seed", "k_seed_deep": "k_seed_deep", "k_filter": "k_filter",
                "k_literal": "k_literal", "k_hamming_scan": "k_hamming_scan", "k_mark_pending": "other"}
    want = dict.fromkeys(capi.Stream.STAGES, 0)
    for steps in steps_per_pass:
        after_k_seed = False
        for step in steps.split(","):
            kernel, _, level = step.partition("@")
            if kernel == "k_seed_var":
                # level 1 of a k_seed_var run is a "k_seed" stage; its later levels and the complete level behind
                # k_seed's levels are "k_seed_deep"
                want["k_seed" if level == "1" and not after_k_seed else "k_seed_deep"] += 1
            else:
                want[stage_of[kernel]] += 1
            after_k_seed |= kernel == "k_seed"
    want["k_finalize"] += 1
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", list(CASES))
def test_launches_follow_the_plan(lib, case_id):
    """One profiled batch of 4 000 reads launches, per stage, exactly the kernels the expected steps name."""
    cfg, debug, steps, b1, b2 = _case(case_id)
    reads = synth.random_reads(np.random.default_rng(11), 4000, b1, b2, min_len=150)
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=len(reads), max_bytes=int(off[-1]), debug=debug) as eng:
        eng.stream.profile(True)
        eng.classify_packed(blob, off)
        got = {stage: n for stage, (_, n) in eng.stream.profile_read_stages().items()}
        eng.stream.profile(False)
    assert got == _launches(steps), case_id
