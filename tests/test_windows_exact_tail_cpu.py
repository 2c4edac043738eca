"""The :hamming and :exact halves of the search-window rule are each load-bearing: with a span that stops at
min(end_j, max_start_pos) instead of reaching max_m - 1 columns further, the oracle's results on reads scrambled
outside the span differ for some config of each algorithm on its own."""
import numpy as np
import pytest

import windows_cases as wc
from test_windows_cpu import differences, lib, py_spans  # noqa: F401  (lib: the module fixture)


@pytest.mark.parametrize("algo", ["hamming", "exact"])
def test_the_max_m_tail_is_needed_per_algorithm(lib, algo):
    caught = []
    for name in sorted(wc.CASES):
        if wc.CASES[name][2].get("matching_algorithm", "semiglobal") != algo:
            continue
        rng = np.random.default_rng(sum(map(ord, name)) + 1)
        cfg, b1, b2 = wc.make_case(name, rng)
        reads = wc.make_reads(rng, b1, b2, 3000)
        if differences(cfg, reads, lambda n: py_spans(cfg, n, "no_tail"), seed=5):
            caught.append(name)
    assert caught, algo
